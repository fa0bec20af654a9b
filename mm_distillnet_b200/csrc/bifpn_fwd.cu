// BiFPN forward kernels (sm_100a).
//
//   node_fwd_kernel   one fusion node of a BiFPN cell (src/YetAnotherEfficientDet.py:338-341 and its 7 siblings
//                     + SeparableConvBlock.forward :182-192) as ONE kernel per node:
//                       prologue : BN-on-load of every input, nearest-x2 / 3x3-s2 same-pad max resampling, fast
//                                  normalised weighted sum, swish  ->  (TH+2)x(TW+2) halo tile in shared memory
//                       depthwise: 3x3, zero padding = the halo                        -> [128][C] A tile (smem)
//                       pointwise: [128 x C] x [C x C] (+bias, eval: BatchNorm folded into W and bias)
//                       epilogue : raw output written once; train: per-channel sum / sum-of-squares -> double
//                                  atomics; the last CTA turns them into scale/shift/mean/invstd and updates the
//                                  running statistics (momentum 0.01, unbiased variance) and num_batches_tracked.
//   proj_fwd_kernel   first-cell 1x1 projections Cin -> C (+bias, BN) (:237-266), same epilogue.
//   bnapply_kernel    materialises [pool](scale*x+shift): P6/P7 synthesis (:324-325) and the stack outputs.
//
// This file is the fp32-exact CUDA-core path (FFMA GEMM from shared memory); see DESIGN.md for the roofline.
#include <stdlib.h>

#include "bifpn.cuh"

namespace mmd {

template <int C>
struct FwdSmem {
  static constexpr int LDD = C + 4;  // padded row of the GEMM A tile (bank-conflict-free broadcast reads)
  static constexpr int kV = kHaloMax * C;
  static constexpr int kD = kTileP * LDD;
  static constexpr int kW = C * C;
  static constexpr int kK = 9 * C;
  static constexpr int kBias = C;
  static constexpr int kInSc = 3 * 2 * C;
  static constexpr int kFloats = kV + kD + kW + kK + kBias + kInSc;
};

// ---- shared epilogue: acc (8 rows x 7 cols per thread) -> +bias -> smem staging -> stats + coalesced store -----
template <typename T, int C>
__device__ __forceinline__ void tile_epilogue(float (&acc)[8][C / 16], const float* s_bias, float* s_y, T* out,
                                              const TileGeom& g, int b, int ty0, int tx0, int th, int tw, bool train,
                                              double& st_sum, double& st_sq) {
  constexpr int NJ = C / 16;
  const int tid = threadIdx.x, tn = tid & 15, tm = tid >> 4;
#pragma unroll
  for (int r = 0; r < 8; ++r)
#pragma unroll
    for (int j = 0; j < NJ; ++j) s_y[(tm + 16 * r) * C + tn + 16 * j] = acc[r][j] + s_bias[tn + 16 * j];
  __syncthreads();
  if (train && tid < C) {
    // double accumulation: with eps = 1e-3 and var << eps an fp32 partial sum would show up at the 1e-4 level
    double s = 0.0, q = 0.0;
    for (int ty = 0; ty < th; ++ty)
      for (int tx = 0; tx < tw; ++tx) {
        const double v = (double)s_y[(ty * g.TW + tx) * C + tid];
        s += v;
        q = fma(v, v, q);
      }
    st_sum += s;
    st_sq += q;
  }
  constexpr int NQ = C / 4;
  for (int idx = tid; idx < g.TH * g.TW * NQ; idx += kThreads) {
    const int p = idx / NQ, q = idx - p * NQ;
    const int ty = p / g.TW, tx = p - ty * g.TW;
    if (ty < th && tx < tw) {
      float4 v = *reinterpret_cast<const float4*>(s_y + p * C + 4 * q);
      st4<T>(out + (((long long)b * g.H + ty0 + ty) * g.W + tx0 + tx) * C + 4 * q, v);
    }
  }
  __syncthreads();
}

// ---- BatchNorm finalisation by the last CTA -----------------------------------------------------------------
template <int C>
__device__ __forceinline__ void bn_finalize(const NodeFwdP& P, double st_sum, double st_sq, int* s_flag) {
  if (P.frozen_bn) return;   // running-statistics vector written by mmd_bifpn_prep; nothing to accumulate or update
  const int tid = threadIdx.x;
  if (tid < C) {
    atomicAdd(P.stats + tid, st_sum);
    atomicAdd(P.stats + C + tid, st_sq);
  }
  __threadfence();
  __syncthreads();
  if (tid == 0) {
    unsigned ticket = atomicAdd(P.counter, 1u);
    *s_flag = (ticket == gridDim.x - 1) ? 1 : 0;
  }
  __syncthreads();
  if (*s_flag == 0) return;
  __threadfence();
  if (tid < C) {
    const double n = (double)P.g.B * P.g.H * P.g.W;
    const double mean = __ldcg(P.stats + tid) / n;
    double var = __ldcg(P.stats + C + tid) / n - mean * mean;
    if (var < 0.0) var = 0.0;
    const float invstd = (float)(1.0 / sqrt(var + (double)P.bn_eps));
    const float scale = P.bn_w[tid] * invstd;
    P.out_bn[tid] = scale;
    P.out_bn[C + tid] = P.bn_b[tid] - (float)mean * scale;
    P.out_bn[2 * C + tid] = (float)mean;
    P.out_bn[3 * C + tid] = invstd;
    const double unbiased = var * (n / (n > 1.0 ? n - 1.0 : 1.0));
    P.bn_rm[tid] = (1.f - P.bn_mom) * P.bn_rm[tid] + P.bn_mom * (float)mean;
    P.bn_rv[tid] = (1.f - P.bn_mom) * P.bn_rv[tid] + P.bn_mom * (float)unbiased;
    P.stats[tid] = 0.0;  // leave the accumulators clean for the next use of this plan
    P.stats[C + tid] = 0.0;
  }
  if (tid == 0) {
    *P.counter = 0u;
    if (P.bn_nbt) *P.bn_nbt += 1;
  }
}

// ---- fusion node ---------------------------------------------------------------------------------------------
template <typename T, int C>
__global__ void __launch_bounds__(kThreads, 1) node_fwd_kernel(const __grid_constant__ NodeFwdP P) {
  using S = FwdSmem<C>;
  constexpr int NQ = C / 4, NJ = C / 16, LDD = S::LDD;
  extern __shared__ __align__(16) float smem[];
  float* s_v = smem;
  float* s_d = s_v + S::kV;
  float* s_w = s_d + S::kD;
  float* s_k = s_w + S::kW;
  float* s_bias = s_k + S::kK;
  float* s_insc = s_bias + S::kBias;
  __shared__ int s_flag;

  const int tid = threadIdx.x;
  const TileGeom g = P.g;
  const bool train = P.train != 0;

  // ---- per-CTA constants: fusion weights, depthwise taps (tap-major), pointwise weights transposed to [k][n]
  float wgt[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) wgt[i] = (i < P.n_in) ? in_weight(P, i) : 0.f;
  for (int idx = tid; idx < 9 * C; idx += kThreads) {
    const int c = idx / 9, tap = idx - c * 9;
    s_k[tap * C + c] = P.dw_w[idx];
  }
  for (int idx = tid; idx < C * C; idx += kThreads) {
    const int n = idx / C, k = idx - n * C;
    float w = P.pw_w[idx];
    if (!train) w *= P.bn_w[n] * rsqrtf(P.bn_rv[n] + P.bn_eps);  // fold eval-mode BatchNorm into the 1x1 conv
    s_w[k * C + n] = w;
  }
  if (tid < C) {
    float bia = P.pw_b[tid];
    if (!train) {
      const float sc = P.bn_w[tid] * rsqrtf(P.bn_rv[tid] + P.bn_eps);
      bia = (bia - P.bn_rm[tid]) * sc + P.bn_b[tid];
    }
    s_bias[tid] = bia;
  }
  for (int idx = tid; idx < 3 * C; idx += kThreads) {
    const int i = idx / C, c = idx - i * C;
    const float* bn = (i < P.n_in) ? P.in[i].bn : nullptr;
    s_insc[(2 * i) * C + c] = bn ? bn[c] : 1.f;
    s_insc[(2 * i + 1) * C + c] = bn ? bn[C + c] : 0.f;
  }
  __syncthreads();

  double st_sum = 0.0, st_sq = 0.0;
  const int tn = tid & 15, tm = tid >> 4;
  const int HW2 = g.TW + 2;

  for (int tile = blockIdx.x; tile < g.ntiles; tile += gridDim.x) {
    const int b = tile / (g.tiles_x * g.tiles_y);
    const int rem = tile - b * (g.tiles_x * g.tiles_y);
    const int ty0 = (rem / g.tiles_x) * g.TH, tx0 = (rem % g.tiles_x) * g.TW;
    const int th = min(g.TH, g.H - ty0), tw = min(g.TW, g.W - tx0);

    // ---- prologue: v = swish(sum_i w_i * resample_i(bn_i(x_i))) on the halo tile; zero outside the image
    const int nh = (g.TH + 2) * HW2;
    for (int idx = tid; idx < nh * NQ; idx += kThreads) {
      const int hp = idx / NQ, q = idx - hp * NQ;
      const int hy = hp / HW2, hx = hp - hy * HW2;
      const int y = ty0 - 1 + hy, x = tx0 - 1 + hx;
      float4 u = f4_zero();
      if (y >= 0 && y < g.H && x >= 0 && x < g.W) {
        const bool center = (hy >= 1 && hy <= th && hx >= 1 && hx <= tw);
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          if (i < P.n_in) {
            const float4 sc = *reinterpret_cast<const float4*>(s_insc + (2 * i) * C + 4 * q);
            const float4 sh = *reinterpret_cast<const float4*>(s_insc + (2 * i + 1) * C + 4 * q);
            float4 val, raw;
            unsigned arg;
            load_input<T, C>(P.in[i], P.mode[i], b, y, x, q, sc, sh, val, raw, arg);
            u = f4_axpy(wgt[i], val, u);
            if (center && P.mode[i] == MMD_IN_POOL && P.pidx[i] != nullptr)
              *reinterpret_cast<unsigned*>(P.pidx[i] + (((long long)b * g.H + y) * g.W + x) * C + 4 * q) = arg;
          }
        }
        if (P.swish) {
          u.x *= sigmoidf_(u.x); u.y *= sigmoidf_(u.y); u.z *= sigmoidf_(u.z); u.w *= sigmoidf_(u.w);
        }
      }
      *reinterpret_cast<float4*>(s_v + hp * C + 4 * q) = u;
    }
    __syncthreads();

    // ---- depthwise 3x3 (stride 1, SAME = zero halo)
    for (int idx = tid; idx < kTileP * NQ; idx += kThreads) {
      const int p = idx / NQ, q = idx - p * NQ;
      const int ty = p / g.TW, tx = p - ty * g.TW;
      float4 d = f4_zero();
      if (ty < th && tx < tw) {
#pragma unroll
        for (int dy = 0; dy < 3; ++dy)
#pragma unroll
          for (int dx = 0; dx < 3; ++dx) {
            const float4 v = *reinterpret_cast<const float4*>(s_v + ((ty + dy) * HW2 + tx + dx) * C + 4 * q);
            const float4 k = *reinterpret_cast<const float4*>(s_k + (dy * 3 + dx) * C + 4 * q);
            d = f4_fma(v, k, d);
          }
        if (P.save_d != nullptr)
          st4<T>(reinterpret_cast<T*>(P.save_d) + (((long long)b * g.H + ty0 + ty) * g.W + tx0 + tx) * C + 4 * q, d);
      }
      *reinterpret_cast<float4*>(s_d + p * LDD + 4 * q) = d;
    }
    __syncthreads();

    // ---- pointwise 1x1: acc[r][j] = sum_k d[tm+16r][k] * W[k][tn+16j]
    float acc[8][NJ];
#pragma unroll
    for (int r = 0; r < 8; ++r)
#pragma unroll
      for (int j = 0; j < NJ; ++j) acc[r][j] = 0.f;
#pragma unroll 4
    for (int k = 0; k < C; ++k) {
      float a[8], w[NJ];
#pragma unroll
      for (int r = 0; r < 8; ++r) a[r] = s_d[(tm + 16 * r) * LDD + k];
#pragma unroll
      for (int j = 0; j < NJ; ++j) w[j] = s_w[k * C + tn + 16 * j];
#pragma unroll
      for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int j = 0; j < NJ; ++j) acc[r][j] = fmaf(a[r], w[j], acc[r][j]);
    }
    tile_epilogue<T, C>(acc, s_bias, s_v, reinterpret_cast<T*>(P.out), g, b, ty0, tx0, th, tw, train, st_sum, st_sq);
  }
  if (train) bn_finalize<C>(P, st_sum, st_sq, &s_flag);
}

// ---- first-cell projection Cin -> C ------------------------------------------------------------------------
constexpr int kProjKC = 32;
template <int C>
struct ProjSmem {
  static constexpr int LDA = kProjKC + 4;
  static constexpr int kA = kTileP * LDA;
  static constexpr int kW = kProjKC * C;
  static constexpr int kY = kTileP * C;
  static constexpr int kFloats = kA + kW + kY + C;
};

template <typename T, int C>
__global__ void __launch_bounds__(kThreads, 2) proj_fwd_kernel(const __grid_constant__ NodeFwdP P) {
  using S = ProjSmem<C>;
  constexpr int NJ = C / 16, LDA = S::LDA, KC = kProjKC;
  extern __shared__ __align__(16) float smem[];
  float* s_a = smem;
  float* s_w = s_a + S::kA;
  float* s_y = s_w + S::kW;
  float* s_bias = s_y + S::kY;
  __shared__ int s_flag;

  const int tid = threadIdx.x, tn = tid & 15, tm = tid >> 4;
  const TileGeom g = P.g;
  const bool train = P.train != 0;
  const int Cin = P.Cin;
  const T* __restrict__ xin = reinterpret_cast<const T*>(P.in[0].data);

  if (tid < C) {
    float bia = P.pw_b[tid];
    if (!train) {
      const float sc = P.bn_w[tid] * rsqrtf(P.bn_rv[tid] + P.bn_eps);
      bia = (bia - P.bn_rm[tid]) * sc + P.bn_b[tid];
    }
    s_bias[tid] = bia;
  }
  double st_sum = 0.0, st_sq = 0.0;

  for (int tile = blockIdx.x; tile < g.ntiles; tile += gridDim.x) {
    const int b = tile / (g.tiles_x * g.tiles_y);
    const int rem = tile - b * (g.tiles_x * g.tiles_y);
    const int ty0 = (rem / g.tiles_x) * g.TH, tx0 = (rem % g.tiles_x) * g.TW;
    const int th = min(g.TH, g.H - ty0), tw = min(g.TW, g.W - tx0);
    float acc[8][NJ];
#pragma unroll
    for (int r = 0; r < 8; ++r)
#pragma unroll
      for (int j = 0; j < NJ; ++j) acc[r][j] = 0.f;

    for (int k0 = 0; k0 < Cin; k0 += KC) {
      __syncthreads();  // previous chunk fully consumed (also orders s_bias on the first pass)
      for (int idx = tid; idx < kTileP * (KC / 4); idx += kThreads) {
        const int p = idx / (KC / 4), kq = idx - p * (KC / 4);
        const int ty = p / g.TW, tx = p - ty * g.TW;
        float4 v = f4_zero();
        if (ty < th && tx < tw && k0 + 4 * kq < Cin)
          v = ld4<T>(xin + (((long long)b * g.H + ty0 + ty) * g.W + tx0 + tx) * Cin + k0 + 4 * kq);
        *reinterpret_cast<float4*>(s_a + p * LDA + 4 * kq) = v;
      }
      for (int idx = tid; idx < C * KC; idx += kThreads) {
        const int n = idx / KC, kk = idx - n * KC;
        float w = 0.f;
        if (k0 + kk < Cin) {
          w = P.pw_w[(long long)n * Cin + k0 + kk];
          if (!train) w *= P.bn_w[n] * rsqrtf(P.bn_rv[n] + P.bn_eps);
        }
        s_w[kk * C + n] = w;
      }
      __syncthreads();
#pragma unroll 4
      for (int kk = 0; kk < KC; ++kk) {
        float a[8], w[NJ];
#pragma unroll
        for (int r = 0; r < 8; ++r) a[r] = s_a[(tm + 16 * r) * LDA + kk];
#pragma unroll
        for (int j = 0; j < NJ; ++j) w[j] = s_w[kk * C + tn + 16 * j];
#pragma unroll
        for (int r = 0; r < 8; ++r)
#pragma unroll
          for (int j = 0; j < NJ; ++j) acc[r][j] = fmaf(a[r], w[j], acc[r][j]);
      }
    }
    tile_epilogue<T, C>(acc, s_bias, s_y, reinterpret_cast<T*>(P.out), g, b, ty0, tx0, th, tw, train, st_sum, st_sq);
  }
  if (train) bn_finalize<C>(P, st_sum, st_sq, &s_flag);
}

// ---- materialise [pool](scale*x + shift) -------------------------------------------------------------------
template <typename T, int C>
__device__ __forceinline__ void bnapply_body(const NodeFwdP& P);

template <typename T, int C>
__global__ void __launch_bounds__(kThreads) bnapply_kernel(const __grid_constant__ NodeFwdP P) {
  bnapply_body<T, C>(P);
}
// the same op of up to 4 networks (student + teachers) in one launch: blockIdx.y selects the network
template <typename T, int C>
__global__ void __launch_bounds__(kThreads) bnapply_multi_kernel(const __grid_constant__ NodeFwdBatch BATCH) {
  bnapply_body<T, C>(BATCH.p[blockIdx.y]);
}

// several independent ops of one network in one launch: blockIdx.y selects the op (each with its own geometry)
template <typename T, int C>
__global__ void __launch_bounds__(kThreads) bnapply_group_kernel(const __grid_constant__ NodeFwdGroup GROUP) {
  bnapply_body<T, C>(GROUP.p[blockIdx.y]);
}

template <typename T, int C>
__device__ __forceinline__ void bnapply_body(const NodeFwdP& P) {
  constexpr int NQ = C / 4;
  const TileGeom g = P.g;
  const long long total = (long long)g.B * g.H * g.W * NQ;
  // (scale, shift) of the source, staged once per block (rebuilt from the producer's statistics when its BatchNorm
  // finalisation is deferred, see NodeFwdP::defer_bn)
  __shared__ __align__(16) float s_bn[2 * C];
  if ((long long)blockIdx.x * blockDim.x >= total) return;
  if (threadIdx.x < C) {
    float sc1, sh1;
    bn_coef<C>(P.in[0], P.bnsrc[0], threadIdx.x, sc1, sh1);
    s_bn[threadIdx.x] = sc1;
    s_bn[C + threadIdx.x] = sh1;
  }
  __syncthreads();
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int q = (int)(idx % NQ);
    long long pos = idx / NQ;
    const int x = (int)(pos % g.W);
    pos /= g.W;
    const int y = (int)(pos % g.H);
    const int b = (int)(pos / g.H);
    const float4 sc = *reinterpret_cast<const float4*>(s_bn + 4 * q);
    const float4 sh = *reinterpret_cast<const float4*>(s_bn + C + 4 * q);
    float4 val, raw;
    unsigned arg;
    load_input<T, C>(P.in[0], P.mode[0], b, y, x, q, sc, sh, val, raw, arg);
    st4<T>(reinterpret_cast<T*>(P.out) + (((long long)b * g.H + y) * g.W + x) * C + 4 * q, val);
    if (P.mode[0] == MMD_IN_POOL && P.pidx[0] != nullptr)
      *reinterpret_cast<unsigned*>(P.pidx[0] + (((long long)b * g.H + y) * g.W + x) * C + 4 * q) = arg;
  }
}

// ---- host launchers ----------------------------------------------------------------------------------------
static int num_sms() { return device_sm_count(); }

template <typename T>
static int launch_node_fwd_t(const NodeFwdP& p, cudaStream_t s) {
  constexpr int C = 112;
  const size_t smem = FwdSmem<C>::kFloats * sizeof(float);
  MMD_SMEM((node_fwd_kernel<T, C>), smem);
  int grid = p.g.ntiles < num_sms() ? p.g.ntiles : num_sms();
  ProfScope prof(PK_NODE_FWD, node_algo_bytes(p.in, p.n_in, p.g, C, sizeof(T)), s);
  node_fwd_kernel<T, C><<<grid, kThreads, smem, s>>>(p);
  MMD_LAUNCH_CHECK();
  return 0;
}

template <typename T>
static int launch_proj_fwd_t(const NodeFwdP& p, cudaStream_t s) {
  constexpr int C = 112;
  const size_t smem = ProjSmem<C>::kFloats * sizeof(float);
  MMD_SMEM((proj_fwd_kernel<T, C>), smem);
  int grid = p.g.ntiles < 2 * num_sms() ? p.g.ntiles : 2 * num_sms();
  ProfScope prof(PK_PROJ_FWD, (double)p.g.B * p.g.H * p.g.W * (p.Cin + C) * sizeof(T), s);
  proj_fwd_kernel<T, C><<<grid, kThreads, smem, s>>>(p);
  MMD_LAUNCH_CHECK();
  return 0;
}

template <typename T>
static int launch_bnapply_multi_t(const NodeFwdP* p, int n, cudaStream_t s) {
  constexpr int C = 112;
  NodeFwdBatch batch;
  double bytes = 0.0;
  for (int i = 0; i < kMaxBatchNets; ++i) batch.p[i] = p[i < n ? i : 0];
  for (int i = 0; i < n; ++i) bytes += node_algo_bytes(p[i].in, 1, p[i].g, C, sizeof(T));
  long long total = (long long)p[0].g.B * p[0].g.H * p[0].g.W * (C / 4);
  long long grid = (total + kThreads - 1) / kThreads;
  if (grid > 8LL * num_sms() / n) grid = 8LL * num_sms() / n;
  if (grid < 1) grid = 1;
  ProfScope prof(PK_BNAPPLY, bytes, s);
  bnapply_multi_kernel<T, C><<<dim3((unsigned)grid, n), kThreads, 0, s>>>(batch);
  MMD_LAUNCH_CHECK();
  return 0;
}

template <typename T>
static int launch_bnapply_group_t(const NodeFwdP* p, int n, cudaStream_t s) {
  constexpr int C = 112;
  NodeFwdGroup group;
  double bytes = 0.0;
  long long maxtotal = 0;
  for (int i = 0; i < kMaxGroupOps; ++i) group.p[i] = p[i < n ? i : 0];
  for (int i = 0; i < n; ++i) {
    bytes += node_algo_bytes(p[i].in, 1, p[i].g, C, sizeof(T));
    const long long total = (long long)p[i].g.B * p[i].g.H * p[i].g.W * (C / 4);
    if (total > maxtotal) maxtotal = total;
  }
  long long grid = (maxtotal + kThreads - 1) / kThreads;
  if (grid > 8LL * num_sms()) grid = 8LL * num_sms();
  if (grid < 1) grid = 1;
  ProfScope prof(PK_BNAPPLY, bytes, s);
  bnapply_group_kernel<T, C><<<dim3((unsigned)grid, n), kThreads, 0, s>>>(group);
  MMD_LAUNCH_CHECK();
  return 0;
}

template <typename T>
static int launch_bnapply_t(const NodeFwdP& p, cudaStream_t s) {
  constexpr int C = 112;
  long long total = (long long)p.g.B * p.g.H * p.g.W * (C / 4);
  long long grid = (total + kThreads - 1) / kThreads;
  if (grid > 8LL * num_sms()) grid = 8LL * num_sms();
  ProfScope prof(PK_BNAPPLY, node_algo_bytes(p.in, 1, p.g, C, sizeof(T)), s);
  bnapply_kernel<T, C><<<(unsigned)grid, kThreads, 0, s>>>(p);
  MMD_LAUNCH_CHECK();
  return 0;
}

#define MMD_DISPATCH(fn)                                                             \
  MMD_CHECK_ARG(C == 112, "BiFPN kernels are built for C=112 (EfficientDet-D2), got %d", C); \
  if (dtype == MMD_F32) return fn<float>(p, s);                                      \
  if (dtype == MMD_BF16) return fn<__nv_bfloat16>(p, s);                             \
  set_error("unsupported dtype %d", dtype);                                          \
  return MMD_E_ARG;

bool tc_disabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("MMD_NO_TC");
    v = (e && e[0] == '1') ? 1 : 0;
  }
  return v == 1;
}

int launch_node_fwd(const NodeFwdP& p, int C, int dtype, cudaStream_t s) {
  if (dtype == MMD_BF16 && !tc_disabled()) return launch_node_fwd_tc(p, C, s);
  MMD_DISPATCH(launch_node_fwd_t)
}
int launch_proj_fwd(const NodeFwdP& p, int C, int dtype, cudaStream_t s) {
  if (dtype == MMD_BF16 && !tc_disabled() && p.Cin % 8 == 0) return launch_proj_fwd_tc(p, C, s);
  MMD_DISPATCH(launch_proj_fwd_t)
}
int launch_bnapply(const NodeFwdP& p, int C, int dtype, cudaStream_t s) { MMD_DISPATCH(launch_bnapply_t) }
int launch_bnapply_group(const NodeFwdP* p, int n, int C, int dtype, cudaStream_t s) {
  MMD_CHECK_ARG(C == 112, "BiFPN kernels are built for C=112 (EfficientDet-D2), got %d", C);
  MMD_CHECK_ARG(n >= 1 && n <= kMaxGroupOps, "bnapply group of %d ops", n);
  if (dtype == MMD_F32) return launch_bnapply_group_t<float>(p, n, s);
  if (dtype == MMD_BF16 && !tc_disabled() && bnapply_same_bf16_usable(p, n)) return launch_bnapply_same_bf16(p, n, s);
  if (dtype == MMD_BF16) return launch_bnapply_group_t<__nv_bfloat16>(p, n, s);
  set_error("unsupported dtype %d", dtype);
  return MMD_E_ARG;
}
int launch_bnapply_multi(const NodeFwdP* p, int n, int C, int dtype, cudaStream_t s) {
  MMD_CHECK_ARG(C == 112, "BiFPN kernels are built for C=112 (EfficientDet-D2), got %d", C);
  MMD_CHECK_ARG(n >= 1 && n <= kMaxBatchNets, "bnapply: %d networks in one launch", n);
  if (dtype == MMD_F32) return launch_bnapply_multi_t<float>(p, n, s);
  if (dtype == MMD_BF16) return launch_bnapply_multi_t<__nv_bfloat16>(p, n, s);
  set_error("unsupported dtype %d", dtype);
  return MMD_E_ARG;
}

}  // namespace mmd
