// BiFPN kernels: resolved (pointer-level) argument structs, tile geometry and the shared fused input loader.
//
// Data flow (see DESIGN.md):  every tensor between nodes is stored ONCE, pre-BatchNorm ("raw"), together with a
// 4*C float vector (scale, shift, mean, invstd).  Consumers apply y = scale*x + shift while loading, resample on
// the fly (nearest x2 / 3x3-s2 zero-padded max) and fuse the weighted sum + swish, so the reference's padded
// copies, upsampled / pooled tensors, fused sums and normalised outputs never exist in HBM.
#pragma once
#include "common.cuh"

namespace mmd {

constexpr int kThreads = 256;
constexpr int kTileP = 128;    // output positions per tile == rows of the pointwise GEMM
constexpr int kHaloMax = 180;  // (TH+2)*(TW+2) upper bound, e.g. (8+2)*(16+2)

struct TensorP {
  const void* data;
  const float* bn;  // nullptr: final values
  int H, W;
};

struct TileGeom {
  int H, W, B;
  int TH, TW, tiles_x, tiles_y, ntiles;
};

inline TileGeom make_geom(int B, int H, int W) {
  TileGeom g;
  g.H = H; g.W = W; g.B = B;
  // widest divisor of W that is <= 16 (falls back to min(W,16) with masked partial tiles)
  int tw = W < 16 ? W : 16;
  for (int t = tw; t >= 8 && t * 2 > tw; --t)
    if (W % t == 0) { tw = t; break; }
  int th = kTileP / tw;
  if (th > H) th = H;
  while ((th + 2) * (tw + 2) > kHaloMax) --th;
  for (int t = th; t * 2 > th && t >= 1; --t)
    if (H % t == 0) { th = t; break; }
  g.TH = th; g.TW = tw;
  g.tiles_x = (W + tw - 1) / tw;
  g.tiles_y = (H + th - 1) / th;
  g.ntiles = B * g.tiles_x * g.tiles_y;
  return g;
}

// Algorithmic HBM bytes of one fusion node (SURVEY.md 8d): every input read once at its own resolution, the output
// written once.  The backward pair (node_bwd_a + node_bwd_b) is charged twice this (the "fwd+bwd = 3x fwd" convention).
inline double node_algo_bytes(const TensorP* in, int n_in, const TileGeom& g, int C, size_t esize) {
  double pos = (double)g.H * g.W;
  for (int i = 0; i < n_in; ++i) pos += (double)in[i].H * in[i].W;
  return pos * g.B * C * (double)esize;
}

// Input-channel chunking of the tensor-core projection backward (bifpn_bwd_v4.cu): chunk width NC in {48, 128, 176}
// (accumulator columns in TMEM and operand tiles in shared memory bound it), n chunks cover Cin.
struct ProjChunks {
  int NC, n;
};
inline ProjChunks proj_chunks(int Cin) {
  ProjChunks c;
  c.NC = Cin <= 48 ? 48 : (Cin <= 128 ? 128 : 176);
  c.n = (Cin + c.NC - 1) / c.NC;
  return c;
}

// Layout of one op's packed parameter block (include/mmd.h, written by prep.cu).
struct PackedLayout {
  int Kp;              // K of the forward GEMM, padded to a multiple of 16
  int offBias, offTaps, offBwd, fwdBytes, bytes;
};
inline PackedLayout packed_layout(int kind, int Cin, int C) {
  PackedLayout L;
  const bool node = (kind == MMD_OP_NODE_FWD || kind == MMD_OP_NODE_BWD);
  if (node) Cin = C;
  L.Kp = (Cin + 15) / 16 * 16;
  L.offBias = (L.Kp * C * 2 + 127) / 128 * 128;
  L.offTaps = L.offBias + C * 4;
  L.fwdBytes = node ? L.offTaps + 9 * C * 4 : L.offTaps;   // what the forward kernel copies into shared memory
  L.offBwd = (L.fwdBytes + 127) / 128 * 128;
  if (node) {
    L.bytes = L.offBwd + (C * C * 2 + 127) / 128 * 128;
  } else {   // projection backward operand: [chunk][C/8][NC][8] bf16, element (o, i) = W[o][chunk*NC + i] (zero padded)
    const ProjChunks pc = proj_chunks(Cin);
    L.bytes = L.offBwd + (pc.n * (C / 8) * pc.NC * 16 + 127) / 128 * 128;
  }
  return L;
}

// Where the BatchNorm vector (scale, shift) of a deferred-BN input can be rebuilt from when its producer leaves the
// finalisation to bn_finalize_all_kernel (see NodeFwdP::defer_bn): the producer's raw statistics.
struct BnSrc {
  const double* stats;   // double[MMD_STATS_REPLICAS][2*C] sums / sums of squares; nullptr: read TensorP::bn
  const float* gamma;
  const float* beta;
  double n;              // B * H * W of the producer's output
  float eps;
};

struct NodeFwdP {
  TensorP in[3];
  int mode[3];
  int n_in, swish, train, Cin;
  const float* fw;
  float fw_eps;
  const float *dw_w, *pw_w, *pw_b, *bn_w, *bn_b;
  float *bn_rm, *bn_rv;
  long long* bn_nbt;
  void* out;
  float* out_bn;
  void* save_d;
  const unsigned char* packed;  // packed parameter block (nullptr: convert in the kernel)
  unsigned char* pidx[3];
  double* stats;
  unsigned* counter;
  float bn_eps, bn_mom;
  TileGeom g;
  int fw_n;        // 0: `fw` has n_in entries, input i uses entry i
  int fw_idx[3];   // entry of `fw` weighing input i; -1: weight 1 (operand produced by a POOLFUSE pre-pass)
  // Deferred BatchNorm finalisation (training, bf16 path).  A producer with defer_bn = 1 only accumulates its statistics
  // and returns: no fence, no ticket, no last-CTA pass at the end of the launch.  Its forward consumers rebuild
  // (scale, shift) from the sums in their prologue (bnsrc[i].stats != nullptr, same arithmetic as the finaliser), and
  // ONE bn_finalize_all launch at the end of the forward writes every out_bn vector for the backward, updates the running
  // statistics and clears the accumulators.
  BnSrc bnsrc[3];
  int defer_bn;
  // Frozen BatchNorm (MmdOp::frozen_bn): out_bn already holds the running-statistics vector (frozen_bn_vector, written by
  // mmd_bifpn_prep); the producer accumulates no statistics, finalises nothing and never touches the running statistics.
  int frozen_bn;
};

// out_bn of a frozen BatchNorm (the layer is in eval() inside a training forward): PyTorch's eval-mode normalisation
// y = gamma * (x - running_mean) / sqrt(running_var + eps) + beta as the (scale, shift, mean, invstd) vector the consumers
// apply on load and the backward reads.
template <int C>
__device__ __forceinline__ void frozen_bn_vector(int c, const float* gamma, const float* beta, const float* rm, const float* rv,
                                                 float eps, float* out_bn) {
  const float invstd = (float)(1.0 / sqrt((double)rv[c] + (double)eps));
  const float scale = gamma[c] * invstd;
  out_bn[c] = scale;
  out_bn[C + c] = beta[c] - rm[c] * scale;
  out_bn[2 * C + c] = rm[c];
  out_bn[3 * C + c] = invstd;
}

// (scale, shift) of channel c of input `t`: from the finalised vector, or rebuilt from the producer's statistics
template <int C>
__device__ __forceinline__ void bn_coef(const TensorP& t, const BnSrc& b, int c, float& scale, float& shift) {
  if (b.stats == nullptr) {
    scale = t.bn ? t.bn[c] : 1.f;
    shift = t.bn ? t.bn[C + c] : 0.f;
    return;
  }
  double sum = 0.0, sq = 0.0;
#pragma unroll
  for (int r = 0; r < MMD_STATS_REPLICAS; ++r) {
    sum += __ldcg(b.stats + r * (2 * C) + c);
    sq += __ldcg(b.stats + r * (2 * C) + C + c);
  }
  const double mean = sum / b.n;
  double var = sq / b.n - mean * mean;
  if (var < 0.0) var = 0.0;
  const float invstd = (float)(1.0 / sqrt(var + (double)b.eps));
  scale = b.gamma[c] * invstd;
  shift = b.beta[c] - (float)mean * scale;
}

// one entry of the deferred finalisation launch
struct BnFinalEntry {
  double* stats;
  const float *gamma, *beta;
  float *rm, *rv, *out_bn;
  long long* nbt;
  double n;
  float eps, mom;
};
constexpr int kBnFinalPerLaunch = 24;
struct BnFinalBatch {
  BnFinalEntry e[kBnFinalPerLaunch];
};
int launch_bn_finalize_all(const BnFinalEntry* entries, int n, int C, cudaStream_t s);
bool bn_deferral_enabled();

// up to 4 networks (student + teachers) run the same node in ONE launch: blockIdx.y selects the network
constexpr int kMaxBatchNets = 4;
struct NodeFwdBatch {
  NodeFwdP p[kMaxBatchNets];
  // 1-D grids (node_fwd_v4 / poolfuse): network k owns CTAs [cta_begin[k], cta_begin[k+1]) — a train-mode network
  // (statistics, saved tensors, arg-max records) gets a larger share than a frozen one, see batch_shares()
  int cta_begin[kMaxBatchNets + 1];
  // node_fwd_v4 with the POOLFUSE pre-pass folded in (small pyramid levels, see launch_node_fwd_v4_pre): the pre-pass op
  // of every network; its output tile is built in shared memory by the node kernel itself
  NodeFwdP pre[kMaxBatchNets];
};
static_assert(sizeof(NodeFwdBatch) <= 4096, "kernel parameter space (4 KB without the large-parameter opt-in)");
// split `budget` CTAs over the n networks of a lockstep launch: weight `train_w` for networks with p.train != 0, 1 for
// the others; at least 1 and at most `max_per_net` CTAs each
void batch_shares(NodeFwdBatch& batch, int n, int budget, int max_per_net, float train_w);
float env_float(const char* name, float dflt);

struct ConsP {
  const void* du;
  int H, W;  // consumer resolution
  int mode;
  int fw_k, fw_n;
  float fw_eps;
  const float* fw;
  const double* slot;
  const unsigned char* pidx;
};

struct NodeBwdP {
  // forward description (inputs are re-read to rebuild the fused sum)
  TensorP in[3];
  int mode[3];
  int n_in, swish, Cin, accumulate_dx;
  const float* fw;
  float fw_eps;
  const float *dw_w, *pw_w, *bn_w;
  const float* in_bn_w[3];
  const float* in_bn_b[3];
  const void* out;      // raw forward output of this op
  const float* out_bn;  // its scale/shift/mean/invstd
  const void* save_d;
  const unsigned char* packed;   // packed parameter block of the forward op (nullptr: convert in the kernel)
  const unsigned char* pidx[3];  // arg-max indices written by the forward for pooled inputs
  const void* aux;               // bf16 nodes with a pooled input: the POOLFUSE operand (final values) ...
  const void* praw;              // ... and the raw pooled-input value at each arg-max
  int n_cons;
  ConsP cons[3];
  void* du;
  void* dd;
  double* in_slot[3];
  void* dx;
  float *g_dw, *g_pw, *g_pb, *g_bn_w, *g_bn_b, *g_fw;
  unsigned* counter;
  TileGeom g;
  int defer_fw;   // 1: node_bwd_b4 leaves the fusion-weight gradient to fwgrad_kernel (one launch per backward)
  int frozen_bn;  // 1: the BatchNorm of `out` normalised with its running statistics (see bn_bwd_coefs)
};

// Deferred fusion-weight gradients: the slots (sum du, sum du * xhat per input edge) of every node are complete when the
// backward's last kernel has run, so ONE launch turns them into all g_fw vectors instead of a fence + ticket +
// last-CTA epilogue at the end of each of the 40 part-B launches.
struct FwGradEntry {
  const double* slot[3];
  const float* in_bn_w[3];
  const float* in_bn_b[3];   // nullptr: the input was final (the slot holds sum du * x)
  const float* fw;
  float* g_fw;
  float fw_eps;
  int n_in;
};
constexpr int kFwGradPerLaunch = 24;
struct FwGradBatch {
  FwGradEntry e[kFwGradPerLaunch];
};
int launch_fwgrad(const FwGradEntry* entries, int n, int C, cudaStream_t s);
bool fwgrad_deferral_enabled();

// fusion weight of kernel input i (ops fed by a POOLFUSE pre-pass see only part of the node's inputs)
__device__ __forceinline__ float in_weight(const NodeFwdP& P, int i) {
  if (P.fw == nullptr) return 1.f;
  const int n = P.fw_n > 0 ? P.fw_n : P.n_in;
  const int k = P.fw_n > 0 ? P.fw_idx[i] : i;
  if (k < 0) return 1.f;
  return fusion_weight(P.fw, n, k, P.fw_eps);
}

// ---- fused input loader -------------------------------------------------------------------------------------
// Loads 4 channels of input `t` as seen by an output position (y, x) of a node:
//   SAME : t[b, y, x]            UP2 : t[b, y>>1, x>>1]   (nn.Upsample nearest x2, YetAnotherEfficientDet.py:223-226)
//   POOL : max over the 3x3 stride-2 window of the zero-padded, ALREADY NORMALISED tensor
//          (MaxPool2dStaticSamePadding, YetAnotherEfficientNet.py:90-104; first maximum in row-major order wins).
// `val` = normalised value (scale*raw+shift), `raw` = the stored element it came from, `arg` = 4 packed
// window indices (0..8, 9 = padding) for POOL.
template <typename T, int C>
__device__ __forceinline__ void load_input(const TensorP& t, int mode, int b, int y, int x, int q, float4 sc, float4 sh,
                                           float4& val, float4& raw, unsigned& arg) {
  const T* base = reinterpret_cast<const T*>(t.data);
  arg = 0u;
  if (mode != MMD_IN_POOL) {
    const int sy = (mode == MMD_IN_UP2) ? (y >> 1) : y;
    const int sx = (mode == MMD_IN_UP2) ? (x >> 1) : x;
    raw = ld4<T>(base + (((long long)b * t.H + sy) * t.W + sx) * C + 4 * q);
    val = f4_fma(raw, sc, sh);
    return;
  }
  const int top = pool_pad_before(t.H), left = pool_pad_before(t.W);
  float m[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
  float r[4] = {0.f, 0.f, 0.f, 0.f};
  unsigned a[4] = {9u, 9u, 9u, 9u};
#pragma unroll
  for (int wy = 0; wy < 3; ++wy) {
    const int fy = 2 * y - top + wy;
#pragma unroll
    for (int wx = 0; wx < 3; ++wx) {
      const int fx = 2 * x - left + wx;
      const bool inside = (fy >= 0) && (fy < t.H) && (fx >= 0) && (fx < t.W);
      float4 rv = f4_zero(), vv = f4_zero();
      if (inside) {
        rv = ld4<T>(base + (((long long)b * t.H + fy) * t.W + fx) * C + 4 * q);
        vv = f4_fma(rv, sc, sh);
      }
      const unsigned id = inside ? (unsigned)(wy * 3 + wx) : 9u;
      if (vv.x > m[0]) { m[0] = vv.x; r[0] = rv.x; a[0] = id; }
      if (vv.y > m[1]) { m[1] = vv.y; r[1] = rv.y; a[1] = id; }
      if (vv.z > m[2]) { m[2] = vv.z; r[2] = rv.z; a[2] = id; }
      if (vv.w > m[3]) { m[3] = vv.w; r[3] = rv.w; a[3] = id; }
    }
  }
  val = make_float4(m[0], m[1], m[2], m[3]);
  raw = make_float4(r[0], r[1], r[2], r[3]);
  arg = a[0] | (a[1] << 8) | (a[2] << 16) | (a[3] << 24);
}

// independent small ops of ONE network (the 5 output BNAPPLYs of a training stack, the 5 SLOT ops that open its
// backward) share a launch: blockIdx.y selects the op, every op keeps its own geometry
constexpr int kMaxGroupOps = 6;
struct NodeFwdGroup {
  NodeFwdP p[kMaxGroupOps];
};
struct NodeBwdGroup {
  NodeBwdP p[kMaxGroupOps];
};
static_assert(sizeof(NodeFwdGroup) <= 4096 && sizeof(NodeBwdGroup) <= 4096, "kernel parameter space");
int launch_bnapply_group(const NodeFwdP* p, int n, int C, int dtype, cudaStream_t s);
// streaming fast paths of the bf16 SAME-mode groups (bifpn_fwd_v4.cu / bifpn_bwd_v4.cu)
bool bnapply_same_bf16_usable(const NodeFwdP* p, int n);
int launch_bnapply_same_bf16(const NodeFwdP* p, int n, cudaStream_t s);
bool slot_same_bf16_usable(const NodeBwdP* p, int n);
int launch_slot_same_bf16(const NodeBwdP* p, int n, cudaStream_t s);
int launch_slot_group(const NodeBwdP* p, int n, int C, int dtype, cudaStream_t s);

// kernels' host launchers (defined in bifpn_fwd.cu / bifpn_bwd.cu)
int launch_node_fwd(const NodeFwdP& p, int C, int dtype, cudaStream_t s);
int launch_node_fwd_tc(const NodeFwdP& p, int C, cudaStream_t s);       // bf16, tcgen05 pointwise conv
// bf16, compile-time tile geometry (bifpn_fwd_v4.cu); `n` networks share one launch
bool fwd_v4_usable(const NodeFwdP& p);
int launch_node_fwd_v4(const NodeFwdP* p, int n, int C, cudaStream_t s);
int launch_poolfuse(const NodeFwdP* p, int n, int C, cudaStream_t s);
// POOLFUSE + NODE_FWD of a small level (<= 24x24) as ONE launch: `pre[i]` is the pre-pass whose output is node[i].in[1]
bool fwd_v4_pre_usable(const NodeFwdP& pre, const NodeFwdP& node);
bool fwd_v4_pre_fusable(const NodeFwdP& pre, const NodeFwdP& node);   // the same without the MMD_INLINE_POOL switch
int launch_node_fwd_v4_pre(const NodeFwdP* node, const NodeFwdP* pre, int n, int C, cudaStream_t s);
// Persistent small-level chain (bifpn_fwd_v4.cu: chain_fwd_kernel): consecutive P5-P7 nodes of all lockstep networks in ONE
// launch, separated by grid barriers.  One host-side step = the same node of n networks (+ its folded POOLFUSE pre-pass).
constexpr int kMaxChainStepsH = 6;
struct ChainStepH {
  NodeFwdP node[kMaxBatchNets];
  NodeFwdP pre[kMaxBatchNets];
  int has_pre;
};
bool chain_fwd_enabled();                                          // MMD_CHAIN=1 / mmd_set_option("chain_fwd", 1); off by default
void set_chain_fwd(int on);
bool chain_fwd_step_usable(const NodeFwdP& node, const NodeFwdP* pre);   // small level, v4 body, deferred BN when training
int launch_chain_fwd(const ChainStepH* steps, int n_steps, int n_nets, int C, cudaStream_t s);
// bf16 backward, compile-time tile geometry (bifpn_bwd_v4.cu)
bool bwd_v4_usable(const NodeBwdP& p);
int launch_node_bwd_v4(const NodeBwdP& p, int C, cudaStream_t s);
bool proj_bwd_v4_usable(const NodeBwdP& p);
int launch_proj_bwd_v4(const NodeBwdP& p, int C, cudaStream_t s);
int launch_proj_fwd_tc(const NodeFwdP& p, int C, cudaStream_t s);      // bf16, tcgen05 projection Cin -> C
int launch_proj_fwd_tc_multi(const NodeFwdP* p, int n, int C, cudaStream_t s);   // n networks in one launch
// warp-specialised tensor-map TMA pipeline for the same op (bifpn_proj_tma.cu); launch_proj_fwd_tc_multi prefers it
bool proj_fwd_tma_usable(const NodeFwdP* p, int n);
int launch_proj_fwd_tma(const NodeFwdP* p, int n, int C, cudaStream_t s);
void set_proj_tma(int on);
int launch_node_bwd_a_tc(const NodeBwdP& p, int C, cudaStream_t s);     // bf16, tcgen05 dgrad + wgrad
bool tc_disabled();  // MMD_NO_TC=1: debugging aid, runs the bf16 path on the CUDA-core kernels instead
int launch_proj_fwd(const NodeFwdP& p, int C, int dtype, cudaStream_t s);
int launch_bnapply(const NodeFwdP& p, int C, int dtype, cudaStream_t s);
int launch_bnapply_multi(const NodeFwdP* p, int n, int C, int dtype, cudaStream_t s);   // n networks in one launch
int launch_node_bwd(const NodeBwdP& p, int C, int dtype, cudaStream_t s);
int launch_proj_bwd(const NodeBwdP& p, int C, int dtype, cudaStream_t s);
int launch_pull(const NodeBwdP& p, int C, int dtype, cudaStream_t s);
int launch_slot(const NodeBwdP& p, int C, int dtype, cudaStream_t s);
// detection-head glue (heads.cu)
int launch_act_fwd(const void* x, void* y, long long n, int dtype, cudaStream_t s);
int launch_act_bwd(const void* x, const void* g, void* dx, long long n, int dtype, cudaStream_t s);
int launch_head_move(int scatter, const void* const* in, void* const* dst, void* out, const void* gout, int B, int HW, int C, int K,
                     int tot, int off, int act, int dtype, cudaStream_t s);
int launch_copy_f32(const float* src, float* dst, long long n, cudaStream_t s);

}  // namespace mmd
