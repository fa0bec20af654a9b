// BiFPN fusion node, forward, bf16 storage: the pointwise 1x1 convolution runs on the 5th-generation tensor cores
// (tcgen05.mma kind::f16, bf16 operands staged in shared memory, fp32 accumulator in TMEM).
//
// Per 128-position tile (one CTA, 256 threads, two CTAs per SM):
//   prologue  : BN-on-load + resample + weighted fusion + swish -> (TH+2)x(TW+2) halo tile v (bf16, smem)
//   depthwise : 3x3 in fp32 registers -> d (bf16) written straight into the UMMA A-operand layout (smem) and, in
//               training, to HBM for the backward
//   pointwise : ONE elected thread issues 7 x tcgen05.mma (M=128, N=112, K=16): D[128x112] = d[128x112] * W^T,
//               W (bf16, BatchNorm folded in eval mode) resident in smem for the life of the CTA; completion is
//               signalled through tcgen05.commit -> mbarrier
//   epilogue  : all 8 warps read the accumulator with tcgen05.ld (32 lanes x 8 columns at a time), add the bias, round
//               to bf16 into a staging tile; then per-channel sum / sum-of-squares (train) and 16-byte coalesced stores.
#include <stdlib.h>

#include "bifpn.cuh"
#include "tc.cuh"

namespace mmd {

typedef __nv_bfloat16 bf16;

template <int C>
struct FwdTcSmem {
  static constexpr int kVBytes = kHaloMax * C * 2;              // halo tile v (bf16); reused as the output staging tile
  static constexpr int LDS = C + 8;                             // staging row (bf16 elements), 16-byte aligned rows
  static constexpr int kABytes = kTileP * C * 2;                // A operand: [C/8][128][8] bf16
  static constexpr int kBBytes = C * C * 2;                     // B operand: [C/8][C][8] bf16
  static constexpr int kKBytes = 9 * C * 4;
  static constexpr int kBiasBytes = C * 4;
  static constexpr int kInScBytes = 3 * 2 * C * 4;
  static constexpr int offV = 0;
  static constexpr int offA = offV + ((kVBytes + 127) / 128) * 128;
  static constexpr int offB = offA + kABytes;
  static constexpr int offK = offB + ((kBBytes + 127) / 128) * 128;
  static constexpr int offBias = offK + kKBytes;
  static constexpr int offInSc = offBias + kBiasBytes;
  static constexpr int offBar = offInSc + kInScBytes;
  static constexpr int kBytes = offBar + 16;
  static_assert(kTileP * LDS * 2 <= kVBytes, "staging tile must fit in the halo tile");
};


// ---- shared epilogue: TMEM accumulator -> +bias -> bf16 staging tile -> stats + 16-byte coalesced stores -------------
template <int C>
__device__ __forceinline__ void tile_epilogue_tc(uint32_t tmem_base, const float* s_bias, bf16* s_y, bf16* out,
                                                 const TileGeom& g, int b, int ty0, int tx0, int th, int tw, bool train,
                                                 double& st_sum, double& st_sq) {
  constexpr int NG = C / 8, LDS = C + 8;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  {
    const int row = 32 * (warp & 3) + lane;          // TMEM lane == tile position
    const int col0 = (warp >> 2) * (C / 2);          // warps 0-3: columns [0,56), warps 4-7: [56,112)
    const uint32_t taddr = tmem_base + ((uint32_t)(32 * (warp & 3)) << 16) + (uint32_t)col0;
    float acc[C / 16][8];
#pragma unroll
    for (int j = 0; j < C / 16; ++j) tc::tmem_ld8(taddr + 8 * j, acc[j]);
    tc::tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < C / 16; ++j) {
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[j][e] += s_bias[col0 + 8 * j + e];
      *reinterpret_cast<uint4*>(s_y + row * LDS + col0 + 8 * j) = tc::pack8_bf16(acc[j]);
    }
  }
  tc::fence_before_sync();   // order the TMEM reads before the next tile's MMAs
  __syncthreads();
  if (train && tid < C) {
    // fp32 partial sums over one tile row (<= 16 values), accumulated in double across rows / tiles
    for (int ty = 0; ty < th; ++ty) {
      float s = 0.f, q = 0.f;
      for (int tx = 0; tx < tw; ++tx) {
        const float v = __bfloat162float(s_y[(ty * g.TW + tx) * LDS + tid]);
        s += v;
        q = fmaf(v, v, q);
      }
      st_sum += (double)s;
      st_sq += (double)q;
    }
  }
  for (int idx = tid; idx < g.TH * g.TW * NG; idx += kThreads) {
    const int p = idx / NG, gq = idx - p * NG;
    const int ty = p / g.TW, tx = p - ty * g.TW;
    if (ty < th && tx < tw)
      *reinterpret_cast<uint4*>(out + (((long long)b * g.H + ty0 + ty) * g.W + tx0 + tx) * C + 8 * gq) =
          *reinterpret_cast<const uint4*>(s_y + p * LDS + 8 * gq);
  }
  __syncthreads();
}

template <int C>
__device__ __forceinline__ void bn_finalize_tc(const NodeFwdP& P, double st_sum, double st_sq, int* s_flag) {
  if (P.frozen_bn) return;   // running-statistics vector written by mmd_bifpn_prep; nothing to accumulate or update
  const int tid = threadIdx.x;
  const TileGeom& g = P.g;
  if (tid < C) {
    double* rep = P.stats + (blockIdx.x & (MMD_STATS_REPLICAS - 1)) * (2 * C);   // spread the same-address atomics
    atomicAdd(rep + tid, st_sum);
    atomicAdd(rep + C + tid, st_sq);
  }
  if (P.defer_bn) return;   // see NodeFwdP::defer_bn
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
    const double n = (double)g.B * g.H * g.W;
    double sum = 0.0, sq = 0.0;
#pragma unroll
    for (int r = 0; r < MMD_STATS_REPLICAS; ++r) {
      sum += __ldcg(P.stats + r * (2 * C) + tid);
      sq += __ldcg(P.stats + r * (2 * C) + C + tid);
    }
    const double mean = sum / n;
    double var = sq / n - mean * mean;
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
#pragma unroll
    for (int r = 0; r < MMD_STATS_REPLICAS; ++r) {
      P.stats[r * (2 * C) + tid] = 0.0;
      P.stats[r * (2 * C) + C + tid] = 0.0;
    }
  }
  if (tid == 0) {
    *P.counter = 0u;
    if (P.bn_nbt) *P.bn_nbt += 1;
  }
}

__device__ __forceinline__ float4 ld4_smem_bf16(const bf16* p) { return ld4<bf16>(p); }

template <int C>
__global__ void __launch_bounds__(kThreads, 2) node_fwd_tc_kernel(const __grid_constant__ NodeFwdP P) {
  using S = FwdTcSmem<C>;
  constexpr int NQ = C / 4, NG = C / 8, LDS = S::LDS;
  constexpr uint32_t kTmemCols = 128;
  constexpr uint32_t kIdesc = tc::make_idesc_bf16(128, C, false, false);
  extern __shared__ __align__(128) unsigned char smem_raw[];
  bf16* s_v = reinterpret_cast<bf16*>(smem_raw + S::offV);
  bf16* s_y = s_v;  // staging aliases the halo tile (dead after the depthwise stage)
  bf16* s_a = reinterpret_cast<bf16*>(smem_raw + S::offA);
  bf16* s_b = reinterpret_cast<bf16*>(smem_raw + S::offB);
  float* s_k = reinterpret_cast<float*>(smem_raw + S::offK);
  float* s_bias = reinterpret_cast<float*>(smem_raw + S::offBias);
  float* s_insc = reinterpret_cast<float*>(smem_raw + S::offInSc);
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem_raw + S::offBar);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem_raw + S::offBar + 8);
  __shared__ int s_flag;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const TileGeom g = P.g;
  const bool train = P.train != 0;
  bf16* __restrict__ out = reinterpret_cast<bf16*>(P.out);

  // ---- per-CTA setup ----------------------------------------------------------------------------------------
  if (warp == 0) tc::tmem_alloc(s_tmem, kTmemCols);
  if (tid == 32) {
    tc::mbar_init(s_bar, 1);
    tc::fence_mbar_init();
  }
  float wgt[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) wgt[i] = (i < P.n_in) ? in_weight(P, i) : 0.f;
  for (int idx = tid; idx < 9 * C; idx += kThreads) {
    const int c = idx / 9, tap = idx - c * 9;
    s_k[tap * C + c] = P.dw_w[idx];
  }
  // B operand: W[n][k] (native [out][in]) -> bf16 [k/8][n][k%8]; eval: fold the BatchNorm scale of channel n
#pragma unroll 7
  for (int idx = tid; idx < C * C; idx += kThreads) {
    const int n = idx / C, k = idx - n * C;
    float w = P.pw_w[idx];
    if (!train) w *= P.bn_w[n] * rsqrtf(P.bn_rv[n] + P.bn_eps);
    s_b[(k >> 3) * (C * 8) + n * 8 + (k & 7)] = __float2bfloat16_rn(w);
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
  tc::fence_async_smem();       // s_b is read by the async proxy
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem_base = *s_tmem;
  const uint32_t a_addr = tc::smem_u32(s_a), b_addr = tc::smem_u32(s_b);

  double st_sum = 0.0, st_sq = 0.0;
  const int HW2 = g.TW + 2;
  uint32_t phase = 0;

  for (int tile = blockIdx.x; tile < g.ntiles; tile += gridDim.x) {
    const int b = tile / (g.tiles_x * g.tiles_y);
    const int rem = tile - b * (g.tiles_x * g.tiles_y);
    const int ty0 = (rem / g.tiles_x) * g.TH, tx0 = (rem % g.tiles_x) * g.TW;
    const int th = min(g.TH, g.H - ty0), tw = min(g.TW, g.W - tx0);

    // ---- prologue: fused input halo tile (bf16)
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
            load_input<bf16, C>(P.in[i], P.mode[i], b, y, x, q, sc, sh, val, raw, arg);
            u = f4_axpy(wgt[i], val, u);
            if (center && P.mode[i] == MMD_IN_POOL && P.pidx[i] != nullptr)
              *reinterpret_cast<unsigned*>(P.pidx[i] + (((long long)b * g.H + y) * g.W + x) * C + 4 * q) = arg;
          }
        }
        if (P.swish) {
          u.x *= sigmoidf_(u.x); u.y *= sigmoidf_(u.y); u.z *= sigmoidf_(u.z); u.w *= sigmoidf_(u.w);
        }
      }
      st4<bf16>(s_v + hp * C + 4 * q, u);
    }
    __syncthreads();

    // ---- depthwise 3x3 -> A operand (bf16, [c/8][p][c%8])
    for (int idx = tid; idx < kTileP * NQ; idx += kThreads) {
      const int p = idx / NQ, q = idx - p * NQ;
      const int ty = p / g.TW, tx = p - ty * g.TW;
      float4 d = f4_zero();
      if (ty < th && tx < tw) {
#pragma unroll
        for (int dy = 0; dy < 3; ++dy)
#pragma unroll
          for (int dx = 0; dx < 3; ++dx) {
            const float4 v = ld4_smem_bf16(s_v + ((ty + dy) * HW2 + tx + dx) * C + 4 * q);
            const float4 k = *reinterpret_cast<const float4*>(s_k + (dy * 3 + dx) * C + 4 * q);
            d = f4_fma(v, k, d);
          }
        if (P.save_d != nullptr)
          st4<bf16>(reinterpret_cast<bf16*>(P.save_d) + (((long long)b * g.H + ty0 + ty) * g.W + tx0 + tx) * C + 4 * q, d);
      }
      st4<bf16>(s_a + (q >> 1) * (kTileP * 8) + p * 8 + (q & 1) * 4, d);
    }
    tc::fence_async_smem();  // the A tile was written through the generic proxy
    __syncthreads();

    // ---- pointwise 1x1 on the tensor cores: one thread issues, the accumulator lives in TMEM
    if (tid == 0) {
      tc::fence_after_sync();
#pragma unroll
      for (int j = 0; j < C / 16; ++j) {
        const uint64_t adesc = tc::make_desc(a_addr + j * 2 * (kTileP * 16), kTileP * 16, 128);
        const uint64_t bdesc = tc::make_desc(b_addr + j * 2 * (C * 16), C * 16, 128);
        tc::umma_bf16(tmem_base, adesc, bdesc, kIdesc, j > 0 ? 1u : 0u);
      }
      tc::umma_commit(s_bar);
    }
    tc::mbar_wait(s_bar, phase);
    phase ^= 1u;
    tc::fence_after_sync();

    tile_epilogue_tc<C>(tmem_base, s_bias, s_y, out, g, b, ty0, tx0, th, tw, train, st_sum, st_sq);
  }

  // ---- teardown + BatchNorm finalisation (last CTA)
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tmem_base, kTmemCols);
  if (!train) return;
  bn_finalize_tc<C>(P, st_sum, st_sq, &s_flag);
}


// =====================================================================================================================
// v2: same data flow, restructured CUDA-core phases (the tensor-core GEMM made them the critical path).
//   phase 1: a thread owns (8-channel group, halo column) and walks the halo rows: 16-byte loads, BatchNorm scale/shift
//            pre-multiplied by the fusion weight (one FMA per element and input), swish via one MUFU.TANH, no div/mod.
//   phase 2: a thread owns (4-channel quad, column) and walks the rows with three rolling accumulators: every halo
//            element is read from shared memory once per column instead of three times, taps live in registers.
// =====================================================================================================================
__device__ __forceinline__ void unpack8(const uint4& r, float (&f)[8]) {
  f[0] = __uint_as_float(r.x << 16); f[1] = __uint_as_float(r.x & 0xffff0000u);
  f[2] = __uint_as_float(r.y << 16); f[3] = __uint_as_float(r.y & 0xffff0000u);
  f[4] = __uint_as_float(r.z << 16); f[5] = __uint_as_float(r.z & 0xffff0000u);
  f[6] = __uint_as_float(r.w << 16); f[7] = __uint_as_float(r.w & 0xffff0000u);
}
__device__ __forceinline__ void unpack4(const uint2& r, float (&f)[4]) {
  f[0] = __uint_as_float(r.x << 16); f[1] = __uint_as_float(r.x & 0xffff0000u);
  f[2] = __uint_as_float(r.y << 16); f[3] = __uint_as_float(r.y & 0xffff0000u);
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float swish_fast(float x) {   // x * sigmoid(x) = 0.5 x (1 + tanh(x/2))
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.5f * x));
  const float h = 0.5f * x;
  return fmaf(h, t, h);
}

template <int C>
__global__ void __launch_bounds__(kThreads, 2) node_fwd_tc2_kernel(const __grid_constant__ NodeFwdP P) {
  using S = FwdTcSmem<C>;
  constexpr int NQ = C / 4, NG = C / 8;
  constexpr uint32_t kTmemCols = 128;
  constexpr uint32_t kIdesc = tc::make_idesc_bf16(128, C, false, false);
  extern __shared__ __align__(128) unsigned char smem_raw[];
  bf16* s_v = reinterpret_cast<bf16*>(smem_raw + S::offV);
  bf16* s_y = s_v;
  bf16* s_a = reinterpret_cast<bf16*>(smem_raw + S::offA);
  bf16* s_b = reinterpret_cast<bf16*>(smem_raw + S::offB);
  float* s_k = reinterpret_cast<float*>(smem_raw + S::offK);
  float* s_bias = reinterpret_cast<float*>(smem_raw + S::offBias);
  float* s_insc = reinterpret_cast<float*>(smem_raw + S::offInSc);   // [input][scale*w | shift*w][C] (pool: unweighted)
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem_raw + S::offBar);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem_raw + S::offBar + 8);
  __shared__ int s_flag;

  const int tid = threadIdx.x, warp = tid >> 5;
  const TileGeom g = P.g;
  const bool train = P.train != 0;
  bf16* __restrict__ out = reinterpret_cast<bf16*>(P.out);

  if (warp == 0) tc::tmem_alloc(s_tmem, kTmemCols);
  if (tid == 32) {
    tc::mbar_init(s_bar, 1);
    tc::fence_mbar_init();
  }
  float wgt[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) wgt[i] = (i < P.n_in) ? in_weight(P, i) : 0.f;
  for (int idx = tid; idx < 9 * C; idx += kThreads) {
    const int c = idx / 9, tap = idx - c * 9;
    s_k[tap * C + c] = P.dw_w[idx];
  }
#pragma unroll 7
  for (int idx = tid; idx < C * C; idx += kThreads) {
    const int n = idx / C, k = idx - n * C;
    float w = P.pw_w[idx];
    if (!train) w *= P.bn_w[n] * rsqrtf(P.bn_rv[n] + P.bn_eps);
    s_b[(k >> 3) * (C * 8) + n * 8 + (k & 7)] = __float2bfloat16_rn(w);
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
    const float w = (i < P.n_in && P.mode[i] != MMD_IN_POOL) ? wgt[i] : 1.f;   // pool: the weight is applied after the max
    s_insc[(2 * i) * C + c] = (bn ? bn[c] : 1.f) * w;
    s_insc[(2 * i + 1) * C + c] = (bn ? bn[C + c] : 0.f) * w;
  }
  for (int idx = tid; idx < kTileP * C / 8; idx += kThreads) reinterpret_cast<uint4*>(s_a)[idx] = make_uint4(0u, 0u, 0u, 0u);
  tc::fence_async_smem();
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem_base = *s_tmem;
  const uint32_t a_addr = tc::smem_u32(s_a), b_addr = tc::smem_u32(s_b);

  double st_sum = 0.0, st_sq = 0.0;
  const int HW2 = g.TW + 2, HH2 = g.TH + 2;
  uint32_t phase = 0;

  for (int tile = blockIdx.x; tile < g.ntiles; tile += gridDim.x) {
    const int b = tile / (g.tiles_x * g.tiles_y);
    const int rem = tile - b * (g.tiles_x * g.tiles_y);
    const int ty0 = (rem / g.tiles_x) * g.TH, tx0 = (rem % g.tiles_x) * g.TW;
    const int th = min(g.TH, g.H - ty0), tw = min(g.TW, g.W - tx0);

    // ---- phase 1: fused inputs -> halo tile v (bf16)
    for (int item = tid; item < NG * HW2; item += kThreads) {
      const int col = item / NG, cg = item - col * NG;
      const int x = tx0 - 1 + col;
      const bool col_in = (x >= 0) && (x < g.W);
      const bool col_center = (col >= 1) && (col <= tw);
      for (int hy = 0; hy < HH2; ++hy) {
        const int y = ty0 - 1 + hy;
        uint4 packed = make_uint4(0u, 0u, 0u, 0u);
        if (col_in && y >= 0 && y < g.H) {
          float u[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) u[e] = 0.f;
#pragma unroll
          for (int i = 0; i < 3; ++i) {
            if (i >= P.n_in) break;
            const TensorP& t = P.in[i];
            const bf16* base = reinterpret_cast<const bf16*>(t.data);
            float sc[8], sh[8];
            *reinterpret_cast<float4*>(sc) = *reinterpret_cast<const float4*>(s_insc + (2 * i) * C + 8 * cg);
            *reinterpret_cast<float4*>(sc + 4) = *reinterpret_cast<const float4*>(s_insc + (2 * i) * C + 8 * cg + 4);
            *reinterpret_cast<float4*>(sh) = *reinterpret_cast<const float4*>(s_insc + (2 * i + 1) * C + 8 * cg);
            *reinterpret_cast<float4*>(sh + 4) = *reinterpret_cast<const float4*>(s_insc + (2 * i + 1) * C + 8 * cg + 4);
            if (P.mode[i] != MMD_IN_POOL) {
              const int sy = (P.mode[i] == MMD_IN_UP2) ? (y >> 1) : y;
              const int sx = (P.mode[i] == MMD_IN_UP2) ? (x >> 1) : x;
              const uint4 r = *reinterpret_cast<const uint4*>(base + (((long long)b * t.H + sy) * t.W + sx) * C + 8 * cg);
              float f[8];
              unpack8(r, f);
#pragma unroll
              for (int e = 0; e < 8; ++e) u[e] += fmaf(f[e], sc[e], sh[e]);
            } else {
              const int top = pool_pad_before(t.H), left = pool_pad_before(t.W);
              float m[8];
              unsigned a[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) { m[e] = -INFINITY; a[e] = 9u; }
#pragma unroll
              for (int wy = 0; wy < 3; ++wy) {
                const int fy = 2 * y - top + wy;
#pragma unroll
                for (int wx = 0; wx < 3; ++wx) {
                  const int fx = 2 * x - left + wx;
                  const bool inside = (fy >= 0) && (fy < t.H) && (fx >= 0) && (fx < t.W);
                  float vv[8];
#pragma unroll
                  for (int e = 0; e < 8; ++e) vv[e] = 0.f;
                  if (inside) {
                    const uint4 r = *reinterpret_cast<const uint4*>(base + (((long long)b * t.H + fy) * t.W + fx) * C + 8 * cg);
                    float f[8];
                    unpack8(r, f);
#pragma unroll
                    for (int e = 0; e < 8; ++e) vv[e] = fmaf(f[e], sc[e], sh[e]);
                  }
                  const unsigned id = inside ? (unsigned)(wy * 3 + wx) : 9u;
#pragma unroll
                  for (int e = 0; e < 8; ++e)
                    if (vv[e] > m[e]) { m[e] = vv[e]; a[e] = id; }
                }
              }
#pragma unroll
              for (int e = 0; e < 8; ++e) u[e] = fmaf(wgt[i], m[e], u[e]);
              if (col_center && hy >= 1 && hy <= th && P.pidx[i] != nullptr) {
                uint2 pk;
                pk.x = a[0] | (a[1] << 8) | (a[2] << 16) | (a[3] << 24);
                pk.y = a[4] | (a[5] << 8) | (a[6] << 16) | (a[7] << 24);
                *reinterpret_cast<uint2*>(P.pidx[i] + (((long long)b * g.H + y) * g.W + x) * C + 8 * cg) = pk;
              }
            }
          }
          if (P.swish) {
#pragma unroll
            for (int e = 0; e < 8; ++e) u[e] = swish_fast(u[e]);
          }
          packed.x = pack2(u[0], u[1]); packed.y = pack2(u[2], u[3]);
          packed.z = pack2(u[4], u[5]); packed.w = pack2(u[6], u[7]);
        }
        *reinterpret_cast<uint4*>(s_v + (hy * HW2 + col) * C + 8 * cg) = packed;
      }
    }
    __syncthreads();

    // ---- phase 2: depthwise 3x3 with rolling accumulators -> A operand
    for (int item = tid; item < NQ * g.TW; item += kThreads) {
      const int c = item / NQ, q = item - c * NQ;
      float4 wk[9];
#pragma unroll
      for (int t9 = 0; t9 < 9; ++t9) wk[t9] = *reinterpret_cast<const float4*>(s_k + t9 * C + 4 * q);
      float4 acc0 = f4_zero(), acc1 = f4_zero(), acc2 = f4_zero();
      const bf16* vcol = s_v + c * C + 4 * q;
      const int a_off = (q >> 1) * (kTileP * 8) + (q & 1) * 4;
      bf16* dsave = (P.save_d != nullptr)
                        ? reinterpret_cast<bf16*>(P.save_d) + (((long long)b * g.H + ty0) * g.W + tx0 + c) * C + 4 * q
                        : nullptr;
      auto row_step = [&](int r, float4& a_new, float4& a_mid, float4& a_old) {
        // input halo row r: tap row 0 of output r (a_new), tap row 1 of output r-1 (a_mid), tap row 2 of output r-2 (a_old)
        float4 v[3];
#pragma unroll
        for (int dx = 0; dx < 3; ++dx) {
          const uint2 raw = *reinterpret_cast<const uint2*>(vcol + (r * HW2 + dx) * C);
          float f[4];
          unpack4(raw, f);
          v[dx] = make_float4(f[0], f[1], f[2], f[3]);
        }
        a_new = f4_mul(v[0], wk[0]);
        a_new = f4_fma(v[1], wk[1], a_new);
        a_new = f4_fma(v[2], wk[2], a_new);
#pragma unroll
        for (int dx = 0; dx < 3; ++dx) {
          a_mid = f4_fma(v[dx], wk[3 + dx], a_mid);
          a_old = f4_fma(v[dx], wk[6 + dx], a_old);
        }
        const int ty = r - 2;
        if (ty >= 0 && ty < th && c < tw) {
          uint2 pk;
          pk.x = pack2(a_old.x, a_old.y);
          pk.y = pack2(a_old.z, a_old.w);
          *reinterpret_cast<uint2*>(s_a + a_off + (ty * g.TW + c) * 8) = pk;
          if (dsave) *reinterpret_cast<uint2*>(dsave + (long long)ty * g.W * C) = pk;
        }
      };
      for (int r0 = 0; r0 < HH2; r0 += 3) {
        row_step(r0, acc0, acc2, acc1);
        if (r0 + 1 < HH2) row_step(r0 + 1, acc1, acc0, acc2);
        if (r0 + 2 < HH2) row_step(r0 + 2, acc2, acc1, acc0);
      }
    }
    tc::fence_async_smem();
    __syncthreads();

    if (tid == 0) {
      tc::fence_after_sync();
#pragma unroll
      for (int j = 0; j < C / 16; ++j) {
        const uint64_t adesc = tc::make_desc(a_addr + j * 2 * (kTileP * 16), kTileP * 16, 128);
        const uint64_t bdesc = tc::make_desc(b_addr + j * 2 * (C * 16), C * 16, 128);
        tc::umma_bf16(tmem_base, adesc, bdesc, kIdesc, j > 0 ? 1u : 0u);
      }
      tc::umma_commit(s_bar);
    }
    tc::mbar_wait(s_bar, phase);
    phase ^= 1u;
    tc::fence_after_sync();
    tile_epilogue_tc<C>(tmem_base, s_bias, s_y, out, g, b, ty0, tx0, th, tw, train, st_sum, st_sq);
  }

  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tmem_base, kTmemCols);
  if (!train) return;
  bn_finalize_tc<C>(P, st_sum, st_sq, &s_flag);
}

int launch_node_fwd_tc(const NodeFwdP& p, int C, cudaStream_t s) {
  MMD_CHECK_ARG(C == 112, "BiFPN kernels are built for C=112 (EfficientDet-D2), got %d", C);
  constexpr int CC = 112;
  static int no_v4 = -1;
  if (no_v4 < 0) {
    const char* e = getenv("MMD_NO_V4");
    no_v4 = (e && e[0] == '1') ? 1 : 0;
  }
  if (!no_v4 && fwd_v4_usable(p)) return launch_node_fwd_v4(&p, 1, C, s);
  const size_t smem = FwdTcSmem<CC>::kBytes;
  static int use_v1 = -1;
  if (use_v1 < 0) {
    const char* e = getenv("MMD_FWD_V1");
    use_v1 = (e && e[0] == '1') ? 1 : 0;
  }
  MMD_SMEM((node_fwd_tc_kernel<CC>), smem);
  MMD_SMEM((node_fwd_tc2_kernel<CC>), smem);
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int grid = p.g.ntiles < 2 * sms ? p.g.ntiles : 2 * sms;
  ProfScope prof(PK_NODE_FWD, node_algo_bytes(p.in, p.n_in, p.g, C, 2), s);
  if (use_v1) node_fwd_tc_kernel<CC><<<grid, kThreads, smem, s>>>(p);
  else node_fwd_tc2_kernel<CC><<<grid, kThreads, smem, s>>>(p);
  MMD_LAUNCH_CHECK();
  return 0;
}


// ---- first-cell projection Cin -> C on the tensor cores ------------------------------------------------------------
// A = the input tile itself: a 16-byte global chunk (position p, channels 8k..8k+7) IS one row of core matrix k, so the
// NHWC -> UMMA layout change costs nothing.  K is padded to a multiple of 16 with zero chunks (Cin = 120 -> 128).
template <int C>
__global__ void __launch_bounds__(kThreads, 1) proj_fwd_tc_kernel(const __grid_constant__ NodeFwdBatch BATCH, int Kp, int packed_off_bias) {
  const NodeFwdP& P = BATCH.p[blockIdx.y];   // blockIdx.y = network (student / teachers share the launch)
  constexpr int LDS = C + 8;
  constexpr uint32_t kTmemCols = 128;
  constexpr uint32_t kIdesc = tc::make_idesc_bf16(128, C, false, false);
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int KG = Kp / 8;
  bf16* s_a = reinterpret_cast<bf16*>(smem_raw);                                   // [KG][128][8]
  bf16* s_b = reinterpret_cast<bf16*>(smem_raw + KG * kTileP * 16);                // [KG][C][8]
  unsigned char* tail = smem_raw + KG * kTileP * 16 + ((KG * C * 16 + 127) / 128) * 128;
  bf16* s_y = reinterpret_cast<bf16*>(tail);                                       // [128][LDS]
  float* s_bias = reinterpret_cast<float*>(tail + kTileP * LDS * 2);
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(tail + kTileP * LDS * 2 + C * 4);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(tail + kTileP * LDS * 2 + C * 4 + 8);
  __shared__ int s_flag;

  const int tid = threadIdx.x, warp = tid >> 5;
  const TileGeom g = P.g;
  const bool train = P.train != 0;
  const int Cin = P.Cin;
  const bf16* __restrict__ xin = reinterpret_cast<const bf16*>(P.in[0].data);
  bf16* __restrict__ out = reinterpret_cast<bf16*>(P.out);

  if (warp == 0) tc::tmem_alloc(s_tmem, kTmemCols);
  if (tid == 32) {
    tc::mbar_init(s_bar, 1);
    tc::fence_mbar_init();
  }
  uint64_t* s_bar_w = s_bar + 2;
  if (P.packed == nullptr) pdl_wait();   // slow path reads parameters that a preceding kernel may have produced
  if (P.packed != nullptr) {   // B operand + bias prepared by mmd_bifpn_prep: two bulk copies
    if (tid == 32) {
      tc::mbar_init(s_bar_w, 1);
      tc::fence_mbar_init();
      tc::mbar_expect_tx(s_bar_w, (uint32_t)(Kp * C * 2 + C * 4));
      tc::bulk_g2s(s_b, P.packed, (uint32_t)(Kp * C * 2), s_bar_w);
      tc::bulk_g2s(s_bias, P.packed + packed_off_bias, C * 4, s_bar_w);
    }
  } else {
#pragma unroll 8
    for (int idx = tid; idx < C * Kp; idx += kThreads) {
      const int n = idx / Kp, k = idx - n * Kp;
      float w = 0.f;
      if (k < Cin) {
        w = P.pw_w[(long long)n * Cin + k];
        if (!train) w *= P.bn_w[n] * rsqrtf(P.bn_rv[n] + P.bn_eps);
      }
      s_b[(k >> 3) * (C * 8) + n * 8 + (k & 7)] = __float2bfloat16_rn(w);
    }
    if (tid < C) {
      float bia = P.pw_b[tid];
      if (!train) {
        const float sc = P.bn_w[tid] * rsqrtf(P.bn_rv[tid] + P.bn_eps);
        bia = (bia - P.bn_rm[tid]) * sc + P.bn_b[tid];
      }
      s_bias[tid] = bia;
    }
  }
  pdl_wait();
  pdl_trigger();
  tc::fence_async_smem();
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem_base = *s_tmem;
  const uint32_t a_addr = tc::smem_u32(s_a), b_addr = tc::smem_u32(s_b);
  double st_sum = 0.0, st_sq = 0.0;
  uint32_t phase = 0;
  bool first_tile = true;

  for (int tile = blockIdx.x; tile < g.ntiles; tile += gridDim.x) {
    const int b = tile / (g.tiles_x * g.tiles_y);
    const int rem = tile - b * (g.tiles_x * g.tiles_y);
    const int ty0 = (rem / g.tiles_x) * g.TH, tx0 = (rem % g.tiles_x) * g.TW;
    const int th = min(g.TH, g.H - ty0), tw = min(g.TW, g.W - tx0);
    for (int idx = tid; idx < kTileP * KG; idx += kThreads) {
      const int p = idx / KG, kg = idx - p * KG;
      const int ty = p / g.TW, tx = p - ty * g.TW;
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (ty < th && tx < tw && 8 * kg < Cin)
        v = *reinterpret_cast<const uint4*>(xin + (((long long)b * g.H + ty0 + ty) * g.W + tx0 + tx) * Cin + 8 * kg);
      *reinterpret_cast<uint4*>(s_a + kg * (kTileP * 8) + p * 8) = v;
    }
    tc::fence_async_smem();
    __syncthreads();
    if (first_tile && P.packed != nullptr) tc::mbar_wait(s_bar_w, 0u);   // weights + bias have landed
    first_tile = false;
    if (tid == 0) {
      tc::fence_after_sync();
      for (int j = 0; j < Kp / 16; ++j) {
        const uint64_t adesc = tc::make_desc(a_addr + j * 2 * (kTileP * 16), kTileP * 16, 128);
        const uint64_t bdesc = tc::make_desc(b_addr + j * 2 * (C * 16), C * 16, 128);
        tc::umma_bf16(tmem_base, adesc, bdesc, kIdesc, j > 0 ? 1u : 0u);
      }
      tc::umma_commit(s_bar);
    }
    tc::mbar_wait(s_bar, phase);
    phase ^= 1u;
    tc::fence_after_sync();
    tile_epilogue_tc<C>(tmem_base, s_bias, s_y, out, g, b, ty0, tx0, th, tw, train, st_sum, st_sq);
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tmem_base, kTmemCols);
  if (!train) return;
  bn_finalize_tc<C>(P, st_sum, st_sq, &s_flag);
}

int launch_proj_fwd_tc_multi(const NodeFwdP* ps, int n, int C, cudaStream_t s) {
  const NodeFwdP& p = ps[0];
  MMD_CHECK_ARG(C == 112, "BiFPN kernels are built for C=112 (EfficientDet-D2), got %d", C);
  MMD_CHECK_ARG(p.Cin % 8 == 0, "bf16 projection needs Cin %% 8 == 0, got %d", p.Cin);
  MMD_CHECK_ARG(n >= 1 && n <= kMaxBatchNets, "proj_fwd: %d networks in one launch", n);
  if (proj_fwd_tma_usable(ps, n)) return launch_proj_fwd_tma(ps, n, C, s);
  constexpr int CC = 112;
  const int Kp = (p.Cin + 15) / 16 * 16, KG = Kp / 8;
  const size_t smem = (size_t)KG * kTileP * 16 + ((KG * CC * 16 + 127) / 128) * 128 + kTileP * (CC + 8) * 2 + CC * 4 + 32;
  MMD_CHECK_ARG(smem <= 227 * 1024, "projection with Cin=%d does not fit in shared memory", p.Cin);
  MMD_SMEM((proj_fwd_tc_kernel<CC>), smem);
  NodeFwdBatch batch;
  for (int i = 0; i < kMaxBatchNets; ++i) batch.p[i] = ps[i < n ? i : 0];
  for (int i = 1; i < n; ++i)
    MMD_CHECK_ARG(ps[i].Cin == p.Cin && ps[i].g.H == p.g.H && ps[i].g.W == p.g.W && ps[i].g.B == p.g.B,
                  "proj_fwd: batched networks must share the shape");
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int per_sm = smem <= 110 * 1024 ? 2 : 1;
  int cap = per_sm * sms / n;
  if (cap < 1) cap = 1;
  const int grid = p.g.ntiles < cap ? p.g.ntiles : cap;
  ProfScope prof(PK_PROJ_FWD, (double)n * p.g.B * p.g.H * p.g.W * (p.Cin + C) * 2, s);
  MMD_CUDA(launch_pdl(proj_fwd_tc_kernel<CC>, dim3(grid, n), dim3(kThreads), smem, s, batch, Kp,
                      packed_layout(MMD_OP_PROJ_FWD, p.Cin, C).offBias));
  MMD_LAUNCH_CHECK();
  return 0;
}

int launch_proj_fwd_tc(const NodeFwdP& p, int C, cudaStream_t s) { return launch_proj_fwd_tc_multi(&p, 1, C, s); }

}  // namespace mmd
