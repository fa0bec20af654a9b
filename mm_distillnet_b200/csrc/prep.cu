// mmd_bifpn_prep: build the packed parameter blocks (include/mmd.h) of every NODE / PROJ op of a stack in one or two
// launches.  The per-tile kernels then fetch their B operands / bias / depthwise taps with ONE bulk copy into shared
// memory instead of every CTA re-reading and re-formatting ~50 KB of fp32 parameters.
//
//   forward B operand : bf16 [Kp/8][C][8], W[n][k] (eval: BatchNorm scale folded: src/YetAnotherEfficientDet.py:176 with
//                       running statistics), zero padded in k up to Kp = ceil16(Cin)
//   bias              : fp32 [C] (eval: folded)
//   taps              : fp32 [9][C] (depthwise [C,1,3,3] transposed to tap-major)
//   backward B operand: bf16 [C/8][C][8], element (o, i) of W stored at [o/8][i][o%8]  (dL/dd = dy * W)
//
// It also writes the BatchNorm vector of every frozen layer (MmdOp::frozen_bn) from gamma, beta and the running
// statistics: every training forward, since gamma and beta move every step.  bf16 plans do it in the packing launch,
// fp32 plans (no packed blocks) in one frozen_bn_kernel launch.
#include "bifpn.cuh"

namespace mmd {

struct PrepDesc {
  const float *pw_w, *pw_b, *bn_w, *bn_b, *bn_rm, *bn_rv, *dw_w;
  unsigned char* dst;
  float* frozen_bn;   // non-null: out.bn of a frozen BatchNorm, written from bn_w / bn_b / bn_rm / bn_rv
  int Cin, Kp, train, node, NC, nchunks, bwd;
  int offBias, offTaps, offBwd;
  float eps;
};
constexpr int kPrepMax = 24;   // descriptors per launch (kernel parameter space is 4 KB)
struct PrepArgs {
  PrepDesc d[kPrepMax];
};

__device__ __forceinline__ uint32_t prep_pack2(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

template <int C>
__global__ void __launch_bounds__(256) prep_kernel(const __grid_constant__ PrepArgs A) {
  const PrepDesc& D = A.d[blockIdx.x];
  const int tid = blockIdx.y * blockDim.x + threadIdx.x, nthr = gridDim.y * blockDim.x;
  const int KG = D.Kp / 8;
  // forward B operand: one 16-byte chunk (kg, n) per item
  for (int item = tid; item < KG * C; item += nthr) {
    const int kg = item / C, n = item - kg * C;
    float w[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = 8 * kg + j;
      w[j] = (k < D.Cin) ? D.pw_w[(long long)n * D.Cin + k] : 0.f;
    }
    if (!D.train) {
      const float sc = D.bn_w[n] * rsqrtf(D.bn_rv[n] + D.eps);
#pragma unroll
      for (int j = 0; j < 8; ++j) w[j] *= sc;
    }
    uint4 r;
    r.x = prep_pack2(w[0], w[1]); r.y = prep_pack2(w[2], w[3]);
    r.z = prep_pack2(w[4], w[5]); r.w = prep_pack2(w[6], w[7]);
    *reinterpret_cast<uint4*>(D.dst + ((size_t)kg * C + n) * 16) = r;
  }
  if (blockIdx.y == 0 && threadIdx.x < C) {
    const int c = threadIdx.x;
    float bia = D.pw_b[c];
    if (!D.train) {
      const float sc = D.bn_w[c] * rsqrtf(D.bn_rv[c] + D.eps);
      bia = (bia - D.bn_rm[c]) * sc + D.bn_b[c];
    }
    reinterpret_cast<float*>(D.dst + D.offBias)[c] = bia;
    if (D.frozen_bn) frozen_bn_vector<C>(c, D.bn_w, D.bn_b, D.bn_rm, D.bn_rv, D.eps, D.frozen_bn);
  }
  if (!D.node) {
    if (!D.bwd) return;
    // projection backward operand: chunk (ch, og, i) holds W[8*og + j][ch*NC + i], j = 0..7 (zero beyond Cin)
    for (int item = tid; item < D.nchunks * (C / 8) * D.NC; item += nthr) {
      const int i = item % D.NC, og = (item / D.NC) % (C / 8), ch = item / (D.NC * (C / 8));
      const int ci = ch * D.NC + i;
      float w[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) w[j] = (ci < D.Cin) ? D.pw_w[(long long)(8 * og + j) * D.Cin + ci] : 0.f;
      uint4 r;
      r.x = prep_pack2(w[0], w[1]); r.y = prep_pack2(w[2], w[3]);
      r.z = prep_pack2(w[4], w[5]); r.w = prep_pack2(w[6], w[7]);
      *reinterpret_cast<uint4*>(D.dst + D.offBwd + (size_t)item * 16) = r;
    }
    return;
  }
  float* taps = reinterpret_cast<float*>(D.dst + D.offTaps);
  for (int idx = tid; idx < 9 * C; idx += nthr) {
    const int tap = idx / C, c = idx - tap * C;
    taps[idx] = D.dw_w[c * 9 + tap];
  }
  if (!D.bwd) return;
  // backward B operand: chunk (og, i) holds W[8*og + j][i], j = 0..7
  for (int item = tid; item < (C / 8) * C; item += nthr) {
    const int og = item / C, i = item - og * C;
    float w[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) w[j] = D.pw_w[(long long)(8 * og + j) * C + i];
    uint4 r;
    r.x = prep_pack2(w[0], w[1]); r.y = prep_pack2(w[2], w[3]);
    r.z = prep_pack2(w[4], w[5]); r.w = prep_pack2(w[6], w[7]);
    *reinterpret_cast<uint4*>(D.dst + D.offBwd + ((size_t)og * C + i) * 16) = r;
  }
}

// fp32 plans: the frozen BatchNorm vectors on their own, one CTA per layer
struct FrozenBnDesc {
  const float *gamma, *beta, *rm, *rv;
  float* out_bn;
  float eps;
};
constexpr int kFrozenMax = 64;
struct FrozenBnArgs {
  FrozenBnDesc d[kFrozenMax];
};
static_assert(sizeof(FrozenBnArgs) <= 4096 && sizeof(PrepArgs) <= 4096, "kernel parameter space");

template <int C>
__global__ void __launch_bounds__(128) frozen_bn_kernel(const __grid_constant__ FrozenBnArgs A) {
  const FrozenBnDesc& D = A.d[blockIdx.x];
  if (threadIdx.x < C) frozen_bn_vector<C>(threadIdx.x, D.gamma, D.beta, D.rm, D.rv, D.eps, D.out_bn);
}

}  // namespace mmd

using namespace mmd;

extern "C" size_t mmd_packed_bytes(int32_t kind, int32_t Cin, int32_t C) {
  if (kind != MMD_OP_NODE_FWD && kind != MMD_OP_PROJ_FWD) return 0;
  return (size_t)packed_layout(kind, Cin, C).bytes;
}

extern "C" int mmd_bifpn_prep(const MmdOp* ops, int32_t n_ops, void* const* bases, int32_t n_bases, int32_t C,
                              int32_t dtype, mmd_stream_t stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  MMD_CHECK_ARG(ops != nullptr && n_ops >= 0 && bases != nullptr, "mmd_bifpn_prep: null arguments");
  MMD_CHECK_ARG(C == 112, "mmd_bifpn_prep: kernels are built for C=112 (EfficientDet-D2), got %d", C);
  for (int i = 0; i < n_ops; ++i)     // staging copies of zero-padded header parameters: before anything reads them
    if (ops[i].kind == MMD_OP_COPY) {
      const int rc = launch_copy_f32(ops[i].copy_src, ops[i].copy_dst, (long long)ops[i].copy_n, stream);
      if (rc) return rc;
    }
  Bases B{bases, n_bases};
  // frozen BatchNorm vectors that no packing launch writes (fp32 plans, ops without a packed block)
  FrozenBnArgs fargs;
  int nf = 0;
  for (int i = 0; i < n_ops; ++i) {
    const MmdOp& op = ops[i];
    if (!op.frozen_bn || (op.kind != MMD_OP_NODE_FWD && op.kind != MMD_OP_PROJ_FWD)) continue;
    MMD_CHECK_ARG(op.train && op.bn_w && op.bn_b && op.bn_rm && op.bn_rv && B.get<float>(op.out.bn) != nullptr,
                  "prep: frozen op %d misses its BatchNorm parameters or vector", i);
    if (dtype == MMD_BF16 && B.get<unsigned char>(op.packed) != nullptr) continue;   // prep_kernel writes it
    MMD_CHECK_ARG(nf < kFrozenMax, "prep: more than %d frozen BatchNorm layers in one op list", kFrozenMax);
    fargs.d[nf++] = FrozenBnDesc{op.bn_w, op.bn_b, op.bn_rm, op.bn_rv, B.get<float>(op.out.bn), op.bn_eps};
  }
  if (nf > 0) {
    frozen_bn_kernel<112><<<nf, 128, 0, stream>>>(fargs);
    MMD_LAUNCH_CHECK();
    pdl_fence_next();
  }
  if (dtype != MMD_BF16) return 0;   // the fp32 parity kernels read the fp32 parameters directly
  PrepArgs args;
  int n = 0;
  auto flush = [&]() -> int {
    if (n == 0) return 0;
    prep_kernel<112><<<dim3(n, 4), 256, 0, stream>>>(args);
    MMD_LAUNCH_CHECK();
    n = 0;
    return 0;
  };
  for (int i = 0; i < n_ops; ++i) {
    const MmdOp& op = ops[i];
    if (op.kind != MMD_OP_NODE_FWD && op.kind != MMD_OP_PROJ_FWD) continue;
    unsigned char* dst = B.get<unsigned char>(op.packed);
    if (dst == nullptr) continue;
    const bool node = op.kind == MMD_OP_NODE_FWD;
    MMD_CHECK_ARG(op.pw_w && op.pw_b && op.bn_w && op.bn_b && op.bn_rm && op.bn_rv, "prep: op %d misses parameters", i);
    MMD_CHECK_ARG(!node || op.dw_w != nullptr, "prep: node op %d has no depthwise weight", i);
    const int Cin = node ? C : op.Cin;
    MMD_CHECK_ARG(Cin >= 4, "prep: op %d has Cin=%d", i, Cin);
    const PackedLayout L = packed_layout(op.kind, Cin, C);
    PrepDesc& D = args.d[n++];
    D.pw_w = op.pw_w; D.pw_b = op.pw_b; D.bn_w = op.bn_w; D.bn_b = op.bn_b;
    D.bn_rm = op.bn_rm; D.bn_rv = op.bn_rv; D.dw_w = op.dw_w;
    D.dst = dst;
    D.frozen_bn = op.frozen_bn ? B.get<float>(op.out.bn) : nullptr;
    D.Cin = Cin; D.Kp = L.Kp; D.train = op.train; D.node = node ? 1 : 0;
    D.bwd = (op.train || op.save_d.base >= 0) ? 1 : 0;
    D.offBias = L.offBias; D.offTaps = L.offTaps; D.offBwd = L.offBwd;
    D.eps = op.bn_eps;
    const ProjChunks pc = proj_chunks(Cin);
    D.NC = pc.NC; D.nchunks = pc.n;
    if (n == kPrepMax) {
      int rc = flush();
      if (rc) return rc;
    }
  }
  const int rc = flush();
  pdl_fence_next();   // the next forward kernel reads these blocks in its prologue, before its griddepcontrol.wait
  return rc;
}
