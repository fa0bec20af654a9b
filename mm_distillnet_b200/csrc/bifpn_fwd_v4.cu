// BiFPN fusion node, forward, bf16 storage — v4 (sm_100a): compile-time tile geometry.
//
// Same fusion as the earlier bf16 kernels (BN-on-load + nearest-x2 resampling + fast-normalised weighted sum + swish ->
// depthwise 3x3 -> pointwise 1x1 on tcgen05 with the accumulator in TMEM -> bias / BatchNorm statistics), but
//   * the tile shape <TW, TH> is a template parameter and only full tiles exist (W % TW == 0, H % TH == 0): the ncu source
//     view of v3 showed ~60 executed instructions per output element, 85 % of them runtime index arithmetic, divisions and
//     bounds checks.  Here every shared-memory offset is a constant, both CUDA-core phases are fully unrolled straight-line
//     code (out-of-image halo positions are computed and then replaced by zero with a select), so the compiler interleaves
//     the rows of one thread;
//   * a node stages at most TWO inputs by bulk copies: pooled inputs (3x3 stride-2 windows over a tensor with 4x the
//     positions, impossible to stage) are folded, together with a third same-resolution input, into one operand by the
//     streaming pre-pass poolfuse_kernel below (MMD_OP_POOLFUSE);
//   * the output tile leaves through bulk shared->global copies (one per tile row, a tile row of an NHWC tensor is
//     contiguous) from a dense staging tile: no per-element store instructions;
//   * the raw input tiles of the NEXT tile are requested as soon as their shared-memory regions are free (input 1 right
//     after the MMA has consumed the A operand, input 0 after the output tile has been read by the bulk store);
//   * up to four networks (student + the three teachers) run the same node in one launch (blockIdx.y): the small pyramid
//     levels have fewer tiles than the GPU has SMs.
// Shared memory (2 CTAs / SM):  region 0 = raw input 0 -> v (in place) -> output staging;  region 1 = raw input 1 -> UMMA
// A operand;  packed parameter block (B operand in UMMA layout, bias, taps: one bulk copy);  folded BN/fusion coefficients.
#include <stdlib.h>

#include "bifpn.cuh"
#include "tc.cuh"

namespace mmd {
namespace v4 {

typedef __nv_bfloat16 bf16;
using tc::add2;
using tc::bf2_to_f2;
using tc::f2_to_bf2;
using tc::fma2;
using tc::mul2;

constexpr int C = 112, NG = C / 8, NQ = C / 4, POS = C * 2;
constexpr int M1_NONE = 0, M1_SAME = 1, M1_UP2 = 2;

constexpr int cmax(int a, int b) { return a > b ? a : b; }
constexpr int up128(int a) { return (a + 127) / 128 * 128; }

// Shared-memory layout.  The mbarriers and the TMEM base address sit at FIXED offsets at the front (the same for every tile
// shape): a persistent kernel that runs nodes of several shapes one after the other (chain_fwd_kernel) initialises them
// once and carries their phases from node to node.
constexpr int kOffBar = 0;          // bar_pack | bar_in0 | bar_in1 | bar_mma | tmem address   (64 bytes reserved)
constexpr int kOffFlag = 64;        // int: "this CTA finalises" flag of the non-deferred BatchNorm epilogue
constexpr int kFront = 128;

template <int TW, int TH>
struct Cfg {
  static_assert(TW % 2 == 0 && TH % 2 == 0, "nearest-x2 inputs need even tiles");
  static constexpr int HW2 = TW + 2, HH2 = TH + 2, NH = HW2 * HH2, NP = TW * TH;
  static constexpr int UW = TW / 2 + 2, UH = TH / 2 + 2;      // staged source rectangle of a nearest-x2 input
  static constexpr int kAStride = 128 * 16 + 16;               // bytes between channel groups of the A operand (padded)
  static constexpr int kABytes = NG * kAStride;                // 28 896
  static constexpr int kStage = 128 * POS;                     // dense output staging tile (rows >= NP unused)
  static constexpr int kR0 = up128(cmax(NH * POS, kStage));
  // region 1: raw input 1 (a full halo tile, or the (TH/2+2) x (TW/2+2) source rectangle of a nearest-x2 input) -> UMMA A
  // operand.  Nodes with a nearest-x2 input also stage their OUTPUT tile here, behind the next tile's input-1 rectangle
  // (the A operand is dead once the MMA has completed): region 0 is then free right after phase 2 and the next tile's
  // input 0 is requested a whole MMA + epilogue + store earlier (ncu source view: 18 % of the forward kernel's stall
  // samples sat in the mbarrier wait for the input tiles).
  static constexpr int kUp2Bytes = UH * UW * POS;
  static constexpr int kR1 = up128(cmax(cmax(NH * POS, kABytes), kUp2Bytes + kStage));
  static constexpr int kWBytes = C * C * 2;
  static constexpr int kPackBytes = kWBytes + C * 4 + 9 * C * 4;   // 29 568
  static constexpr int offR0 = kFront, offR1 = offR0 + kR0, offPack = offR1 + kR1, offCoef = offPack + kPackBytes;
  static constexpr int offPc = offCoef + 3 * C * 4;            // pre-pass coefficients (PRE kernels only)
  static constexpr int kBytes = offPc;
  static constexpr int kBytesPre = offPc + 4 * C * 4;
  static constexpr int kP1Threads = NG * HW2, kP2Threads = NQ * (TW / 2);
  static_assert(NP <= 128 && kP1Threads <= kThreads && kP2Threads <= kThreads && HH2 <= 32, "tile too large");
  static_assert(offPack % 128 == 0 && offCoef % 16 == 0 && offPc % 16 == 0, "alignment");
  static_assert(2 * (kBytes + 1024) <= 233472, "two CTAs per SM");
};

__device__ __forceinline__ void bulk_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(__cvta_generic_to_global(dst_gmem)),
               "r"(tc::smem_u32(src_smem)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

struct TilePos {
  int b, ty0, tx0;
};
// tile -> (sample, first row, first column).  The two divisions are by loop-invariant small numbers: ncu's source view
// charged ~5 % of the forward kernel's instructions to them, so they are multiply-high by precomputed reciprocals
// (exact for tile * divisor < 2^32).
struct TileDiv {
  int per, tiles_x;
  uint32_t m_per, m_tx;
};
__device__ __forceinline__ TileDiv make_tile_div(int tiles_x, int tiles_y) {
  TileDiv d;
  d.per = tiles_x * tiles_y;
  d.tiles_x = tiles_x;
  d.m_per = 0xFFFFFFFFu / (uint32_t)d.per + 1u;
  d.m_tx = 0xFFFFFFFFu / (uint32_t)tiles_x + 1u;
  return d;
}
__device__ __forceinline__ TilePos tile_pos(int tile, const TileDiv& d, int TW, int TH) {
  TilePos t;
  t.b = (d.per == 1) ? tile : (int)__umulhi((uint32_t)tile, d.m_per);
  const int rem = tile - t.b * d.per;
  const int ry = (d.tiles_x == 1) ? rem : (int)__umulhi((uint32_t)rem, d.m_tx);
  t.ty0 = ry * TH;
  t.tx0 = (rem - ry * d.tiles_x) * TW;
  return t;
}

// ---- bulk row copies of one raw input tile (executed by one warp, one row per lane) ------------------------------
// SAME inputs land at their halo coordinates; a nearest-x2 input lands as its (TH/2+2) x (TW/2+2) source rectangle.
// Rows / columns outside the image are simply not copied (the consumer replaces those positions by zero).
template <int TW, int TH>
__device__ __forceinline__ void issue_input(unsigned char* dst, const bf16* src, bool up2, const TilePos t, int H, int W,
                                            int lane, uint64_t* bar) {
  using S = Cfg<TW, TH>;
  int rows_lo, rows_hi, col_lo, col_hi, pitch, gy0, gx0, SH, SW;
  if (!up2) {
    rows_lo = (t.ty0 == 0) ? 1 : 0;
    rows_hi = (t.ty0 + TH >= H) ? S::HH2 - 2 : S::HH2 - 1;
    col_lo = (t.tx0 == 0) ? 1 : 0;
    col_hi = (t.tx0 + TW >= W) ? S::HW2 - 2 : S::HW2 - 1;
    pitch = S::HW2;
    gy0 = t.ty0 - 1; gx0 = t.tx0 - 1; SH = H; SW = W;
  } else {
    SH = H >> 1; SW = W >> 1;
    rows_lo = (t.ty0 == 0) ? 1 : 0;
    rows_hi = ((t.ty0 >> 1) + TH / 2 >= SH) ? S::UH - 2 : S::UH - 1;
    col_lo = (t.tx0 == 0) ? 1 : 0;
    col_hi = ((t.tx0 >> 1) + TW / 2 >= SW) ? S::UW - 2 : S::UW - 1;
    pitch = S::UW;
    gy0 = (t.ty0 >> 1) - 1; gx0 = (t.tx0 >> 1) - 1;
  }
  const uint32_t rb = (uint32_t)(col_hi - col_lo + 1) * POS;
  const int nrows = rows_hi - rows_lo + 1;
  if (lane == 0) tc::mbar_expect_tx(bar, (uint32_t)nrows * rb);
  __syncwarp();
  if (lane < nrows) {
    const int r = rows_lo + lane;
    tc::bulk_g2s(dst + (r * pitch + col_lo) * POS, src + (((long long)t.b * SH + gy0 + r) * SW + gx0 + col_lo) * C, rb, bar);
  }
}

// ---- phase 1: v = swish(a0 * x0 + a1 * resample(x1) + shift), written in place over raw input 0 ------------------
template <int TW, int TH, int M1, bool SW>
__device__ __forceinline__ void phase1(unsigned char* r0, const unsigned char* r1, const float* s_coef, int tid,
                                       const TilePos t, int H, int W) {
  using S = Cfg<TW, TH>;
  if (tid >= S::kP1Threads) return;
  const int cg = tid % NG, hx = tid / NG;
  float2 a0[4], a1[4], sh[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    a0[e] = *reinterpret_cast<const float2*>(s_coef + 8 * cg + 2 * e);
    a1[e] = *reinterpret_cast<const float2*>(s_coef + C + 8 * cg + 2 * e);
    sh[e] = *reinterpret_cast<const float2*>(s_coef + 2 * C + 8 * cg + 2 * e);
  }
  const int x = t.tx0 - 1 + hx;
  const bool x_ok = (x >= 0) && (x < W);
  const bool top_ok = t.ty0 > 0, bot_ok = t.ty0 + TH < H;
  unsigned char* cell = r0 + hx * POS + cg * 16;
  const unsigned char* src1 = r1 + ((M1 == M1_UP2) ? ((hx + 1) >> 1) : hx) * POS + cg * 16;
  uint4 s1 = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
  for (int hy = 0; hy < S::HH2; ++hy) {
    const bool ok = x_ok && (hy == 0 ? top_ok : (hy == S::HH2 - 1 ? bot_ok : true));
    const uint4 r = *reinterpret_cast<const uint4*>(cell + hy * (S::HW2 * POS));
    float2 u[4];
    u[0] = fma2(bf2_to_f2(r.x), a0[0], sh[0]);
    u[1] = fma2(bf2_to_f2(r.y), a0[1], sh[1]);
    u[2] = fma2(bf2_to_f2(r.z), a0[2], sh[2]);
    u[3] = fma2(bf2_to_f2(r.w), a0[3], sh[3]);
    if (M1 != M1_NONE) {
      if (M1 == M1_SAME) {
        s1 = *reinterpret_cast<const uint4*>(src1 + hy * (S::HW2 * POS));
      } else if (hy == 0 || (hy & 1)) {   // halo rows 2k-1 and 2k share source row k
        s1 = *reinterpret_cast<const uint4*>(src1 + ((hy + 1) >> 1) * (S::UW * POS));
      }
      u[0] = fma2(bf2_to_f2(s1.x), a1[0], u[0]);
      u[1] = fma2(bf2_to_f2(s1.y), a1[1], u[1]);
      u[2] = fma2(bf2_to_f2(s1.z), a1[2], u[2]);
      u[3] = fma2(bf2_to_f2(s1.w), a1[3], u[3]);
    }
    if (SW) {
#pragma unroll
      for (int e = 0; e < 4; ++e) u[e] = tc::swish2(u[e]);
    }
    uint4 pk;
    pk.x = ok ? f2_to_bf2(u[0]) : 0u;
    pk.y = ok ? f2_to_bf2(u[1]) : 0u;
    pk.z = ok ? f2_to_bf2(u[2]) : 0u;
    pk.w = ok ? f2_to_bf2(u[3]) : 0u;
    *reinterpret_cast<uint4*>(cell + hy * (S::HW2 * POS)) = pk;
  }
}

// ---- phase 2: depthwise 3x3 over the v halo tile -> UMMA A operand (+ the saved depthwise output in training) ------
template <int TW, int TH>
__device__ __forceinline__ void phase2(const unsigned char* r0, unsigned char* r1, const float* s_k, int tid, bf16* dsave,
                                       int W) {
  using S = Cfg<TW, TH>;
  if (tid >= S::kP2Threads) return;
  const int q = tid % NQ, c0 = 2 * (tid / NQ);
  float2 wk[9][2];
#pragma unroll
  for (int t9 = 0; t9 < 9; ++t9) {
    const float4 k4 = *reinterpret_cast<const float4*>(s_k + t9 * C + 4 * q);
    wk[t9][0] = make_float2(k4.x, k4.y);
    wk[t9][1] = make_float2(k4.z, k4.w);
  }
  const unsigned char* vcol = r0 + c0 * POS + q * 8;
  unsigned char* arow = r1 + (q >> 1) * S::kAStride + (q & 1) * 8 + c0 * 16;
  if (dsave != nullptr) dsave += c0 * C + 4 * q;
  float2 acc[3][2][2];   // [output row mod 3][column][channel pair]
#pragma unroll
  for (int r = 0; r < S::HH2; ++r) {
    float2 v[4][2];
#pragma unroll
    for (int dx = 0; dx < 4; ++dx) {
      const uint2 raw = *reinterpret_cast<const uint2*>(vcol + (r * S::HW2 + dx) * POS);
      v[dx][0] = bf2_to_f2(raw.x);
      v[dx][1] = bf2_to_f2(raw.y);
    }
    // halo row r is tap row 0 of output row r, tap row 1 of r-1, tap row 2 of r-2
#pragma unroll
    for (int c = 0; c < 2; ++c)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        if (r < TH) {
          float2 a = mul2(v[c][h], wk[0][h]);
          a = fma2(v[c + 1][h], wk[1][h], a);
          acc[r % 3][c][h] = fma2(v[c + 2][h], wk[2][h], a);
        }
        if (r >= 1 && r - 1 < TH) {
          float2 a = acc[(r + 2) % 3][c][h];
          a = fma2(v[c][h], wk[3][h], a);
          a = fma2(v[c + 1][h], wk[4][h], a);
          acc[(r + 2) % 3][c][h] = fma2(v[c + 2][h], wk[5][h], a);
        }
        if (r >= 2) {
          float2 a = acc[(r + 1) % 3][c][h];
          a = fma2(v[c][h], wk[6][h], a);
          a = fma2(v[c + 1][h], wk[7][h], a);
          acc[(r + 1) % 3][c][h] = fma2(v[c + 2][h], wk[8][h], a);
        }
      }
    if (r >= 2) {
      const int o = r - 2;
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint2 pk;
        pk.x = f2_to_bf2(acc[(r + 1) % 3][c][0]);
        pk.y = f2_to_bf2(acc[(r + 1) % 3][c][1]);
        *reinterpret_cast<uint2*>(arow + (o * TW + c) * 16) = pk;
        if (dsave != nullptr) *reinterpret_cast<uint2*>(dsave + ((long long)o * W + c) * C) = pk;
      }
    }
  }
}

// ---- inline pooling pre-pass (small levels): the POOLFUSE operand of one tile (+ halo) built straight in region 1 ------
// out = w_a * maxpool3x3s2(bn_a(src)) [+ w_b * bn_b(same)], rounded to bf16 exactly as poolfuse_kernel stores it.  Window
// scan in row-major order, strict '>' (first maximum wins), zero padding takes part with index 9 (MaxPool2dStaticSamePadding,
// src/YetAnotherEfficientNet.py:90-104) — the comparison form of load_input().  In training the operand, the arg-max bytes
// and the raw value at the arg-max of the tile's own positions also go to HBM for the backward.
template <int TW, int TH>
__device__ __forceinline__ void inline_pool_tile(const NodeFwdP& Q, const float* s_pc, unsigned char* r1, const TilePos t,
                                                 const int H, const int W, const int tid, const float wa) {
  using S = Cfg<TW, TH>;
  const bf16* __restrict__ src = reinterpret_cast<const bf16*>(Q.in[0].data);
  const bf16* __restrict__ same = (Q.n_in >= 2) ? reinterpret_cast<const bf16*>(Q.in[1].data) : nullptr;
  const int SH = Q.in[0].H, SWd = Q.in[0].W;
  bf16* __restrict__ aux = reinterpret_cast<bf16*>(Q.out);
  unsigned char* __restrict__ pidx = Q.pidx[0];
  bf16* __restrict__ praw = reinterpret_cast<bf16*>(Q.save_d);
  const bool record = (pidx != nullptr) || (praw != nullptr);
  const int top = pool_pad_before(SH), left = pool_pad_before(SWd);
  for (int item = tid; item < S::NH * NG; item += kThreads) {
    const int hp = item / NG, cg = item - hp * NG;
    const int hy = hp / S::HW2, hx = hp - hy * S::HW2;
    const int y = t.ty0 - 1 + hy, x = t.tx0 - 1 + hx;
    if (y < 0 || y >= H || x < 0 || x >= W) continue;   // phase 1 replaces out-of-image positions by zero
    float sc[8], sh[8], best[8], braw[8];
    uint32_t bid[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      sc[e] = s_pc[8 * cg + e];
      sh[e] = s_pc[C + 8 * cg + e];
      best[e] = -INFINITY;
      braw[e] = 0.f;
      bid[e] = 9u;
    }
#pragma unroll
    for (int wy = 0; wy < 3; ++wy) {
      const int fy = 2 * y - top + wy;
#pragma unroll
      for (int wx = 0; wx < 3; ++wx) {
        const int fx = 2 * x - left + wx;
        const bool inside = (fy >= 0) && (fy < SH) && (fx >= 0) && (fx < SWd);
        uint4 r = make_uint4(0u, 0u, 0u, 0u);
        if (inside) r = __ldcg(reinterpret_cast<const uint4*>(src + (((long long)t.b * SH + fy) * SWd + fx) * C + 8 * cg));
        const uint32_t w[4] = {r.x, r.y, r.z, r.w};
        const uint32_t id = inside ? (uint32_t)(wy * 3 + wx) : 9u;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 raw = bf2_to_f2(w[e]);
          const float v0 = inside ? fmaf(raw.x, sc[2 * e], sh[2 * e]) : 0.f;
          const float v1 = inside ? fmaf(raw.y, sc[2 * e + 1], sh[2 * e + 1]) : 0.f;
          if (v0 > best[2 * e]) { best[2 * e] = v0; braw[2 * e] = raw.x; bid[2 * e] = id; }
          if (v1 > best[2 * e + 1]) { best[2 * e + 1] = v1; braw[2 * e + 1] = raw.y; bid[2 * e + 1] = id; }
        }
      }
    }
    float u[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) u[e] = wa * best[e];
    const long long oo = (((long long)t.b * H + y) * W + x) * C + 8 * cg;
    if (same != nullptr) {
      const uint4 r = __ldcg(reinterpret_cast<const uint4*>(same + oo));
      const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 f = bf2_to_f2(w[e]);
        u[2 * e] += fmaf(f.x, s_pc[2 * C + 8 * cg + 2 * e], s_pc[3 * C + 8 * cg + 2 * e]);
        u[2 * e + 1] += fmaf(f.y, s_pc[2 * C + 8 * cg + 2 * e + 1], s_pc[3 * C + 8 * cg + 2 * e + 1]);
      }
    }
    uint4 pk;
    pk.x = f2_to_bf2(make_float2(u[0], u[1]));
    pk.y = f2_to_bf2(make_float2(u[2], u[3]));
    pk.z = f2_to_bf2(make_float2(u[4], u[5]));
    pk.w = f2_to_bf2(make_float2(u[6], u[7]));
    *reinterpret_cast<uint4*>(r1 + hp * POS + cg * 16) = pk;
    if (record && hy >= 1 && hy <= TH && hx >= 1 && hx <= TW) {   // the tile's own positions: what the backward reads
      *reinterpret_cast<uint4*>(aux + oo) = pk;
      if (pidx != nullptr) {
        uint2 ip;
        ip.x = bid[0] | (bid[1] << 8) | (bid[2] << 16) | (bid[3] << 24);
        ip.y = bid[4] | (bid[5] << 8) | (bid[6] << 16) | (bid[7] << 24);
        *reinterpret_cast<uint2*>(pidx + oo) = ip;
      }
      if (praw != nullptr) {
        uint4 rp;
        rp.x = f2_to_bf2(make_float2(braw[0], braw[1]));
        rp.y = f2_to_bf2(make_float2(braw[2], braw[3]));
        rp.z = f2_to_bf2(make_float2(braw[4], braw[5]));
        rp.w = f2_to_bf2(make_float2(braw[6], braw[7]));
        *reinterpret_cast<uint4*>(praw + oo) = rp;
      }
    }
  }
}

// Per-CTA state that outlives one node: where TMEM is, and the phase of every mbarrier (each is used a different number of
// times per node — bar_in1 only by nodes that stage a second input, bar_pack once per node — so each carries its own bit).
struct FwdCtx {
  uint32_t tmem_base;
  uint32_t ph_pack, ph_in0, ph_in1, ph_mma;
};

// One fusion node for the CTAs [0, nctas) of one network.  Called by every thread of the CTA; all barriers inside are
// CTA-wide.  `pdl`: this is the first node of its kernel, do the griddepcontrol handshake where the prologue allows.
template <int TW, int TH, bool PRE>
__device__ __forceinline__ void node_fwd_body(const NodeFwdP& P, const NodeFwdP& Q, const int cta, const int nctas,
                                              unsigned char* smem, FwdCtx& X, const bool pdl) {
  using S = Cfg<TW, TH>;
  constexpr uint32_t kIdesc = tc::make_idesc_bf16(128, C, false, false);
  unsigned char* r0 = smem + S::offR0;
  unsigned char* r1 = smem + S::offR1;
  unsigned char* s_pack = smem + S::offPack;
  const float* s_bias = reinterpret_cast<const float*>(s_pack + S::kWBytes);
  const float* s_k = s_bias + C;
  float* s_coef = reinterpret_cast<float*>(smem + S::offCoef);
  float* s_pc = reinterpret_cast<float*>(smem + S::offPc);   // PRE: the pre-pass coefficients (as poolfuse_kernel's s_c)
  uint64_t* bar_pack = reinterpret_cast<uint64_t*>(smem + kOffBar);
  uint64_t* bar_in0 = bar_pack + 1;
  uint64_t* bar_in1 = bar_pack + 2;
  uint64_t* bar_mma = bar_pack + 3;
  int* s_flag = reinterpret_cast<int*>(smem + kOffFlag);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int H = P.g.H, W = P.g.W;
  const int tiles_x = W / TW, tiles_y = H / TH, ntiles = P.g.B * tiles_x * tiles_y;
  const TileDiv tdiv = make_tile_div(tiles_x, tiles_y);
  const bool train = P.train != 0;
  const int m1 = (P.n_in < 2) ? M1_NONE : (P.mode[1] == MMD_IN_UP2 ? M1_UP2 : M1_SAME);
  const bool sw = P.swish != 0;
  bf16* __restrict__ out = reinterpret_cast<bf16*>(P.out);
  const bf16* __restrict__ in0 = reinterpret_cast<const bf16*>(P.in[0].data);
  const bf16* __restrict__ in1 = reinterpret_cast<const bf16*>(P.in[1].data);

  // ---- per-node setup ---------------------------------------------------------------------------------------------
  if (tid == 32) {   // the packed parameter block: B operand, bias, depthwise taps (one bulk copy)
    tc::mbar_expect_tx(bar_pack, S::kPackBytes);
    tc::bulk_g2s(s_pack, P.packed, S::kPackBytes, bar_pack);
  }
  if (pdl) {
    pdl_wait();      // everything above overlaps the previous kernel; its outputs (inputs / BN vectors here) are visible now
    pdl_trigger();
  }
  // first tile's inputs: requested before the coefficient set-up below, whose dependent global loads (fusion weights,
  // BatchNorm vectors) would otherwise delay them by a full round trip (warp 1 owns the barriers)
  int tile = cta;
  if (warp == 1) {
    __syncwarp();
    if (tile < ntiles) {
      const TilePos t = tile_pos(tile, tdiv, TW, TH);
      issue_input<TW, TH>(r0, in0, false, t, H, W, lane, bar_in0);
      if (!PRE && m1 != M1_NONE) issue_input<TW, TH>(r1, in1, m1 == M1_UP2, t, H, W, lane, bar_in1);
    }
  }
  float pre_wa = 0.f;
  if (PRE) {
    pre_wa = in_weight(Q, 0);
    if (tid < C) {
      const float wb = (Q.n_in >= 2) ? in_weight(Q, 1) : 0.f;
      float qs0, qh0, qs1 = 1.f, qh1 = 0.f;
      bn_coef<C>(Q.in[0], Q.bnsrc[0], tid, qs0, qh0);
      if (Q.n_in >= 2) bn_coef<C>(Q.in[1], Q.bnsrc[1], tid, qs1, qh1);
      s_pc[tid] = qs0;
      s_pc[C + tid] = qh0;
      s_pc[2 * C + tid] = qs1 * wb;
      s_pc[3 * C + tid] = qh1 * wb;
    }
  }
  if (tid < C) {
    const float w0 = in_weight(P, 0), w1 = (P.n_in >= 2) ? in_weight(P, 1) : 0.f;
    float sc0, sh0, sc1 = 1.f, sh1 = 0.f;
    bn_coef<C>(P.in[0], P.bnsrc[0], tid, sc0, sh0);
    if (P.n_in >= 2) bn_coef<C>(P.in[1], P.bnsrc[1], tid, sc1, sh1);
    s_coef[tid] = sc0 * w0;
    s_coef[C + tid] = sc1 * w1;
    s_coef[2 * C + tid] = fmaf(sh1, w1, sh0 * w0);
  }
  __syncthreads();
  const uint32_t tmem_base = X.tmem_base;
  const uint32_t a_addr = tc::smem_u32(r1), b_addr = tc::smem_u32(s_pack);

  // statistics role: channel pair sp of row slice ss (32 staging rows)
  const int sp = tid % (C / 2), ss = tid / (C / 2);
  double st[4] = {0.0, 0.0, 0.0, 0.0};
  bool pack_ready = false;

  for (; tile < ntiles; tile += nctas) {
    const TilePos t = tile_pos(tile, tdiv, TW, TH);
    const int next = tile + nctas;

    // ---- (0) PRE: build the pooled operand of this tile in region 1 (free: the previous tile's MMA has completed)
    if (PRE) {
      inline_pool_tile<TW, TH>(Q, s_pc, r1, t, H, W, tid, pre_wa);
      __syncthreads();
    }

    // ---- (1) raw inputs have landed
    tc::mbar_wait(bar_in0, X.ph_in0);
    X.ph_in0 ^= 1u;
    if (!PRE && m1 != M1_NONE) {
      tc::mbar_wait(bar_in1, X.ph_in1);
      X.ph_in1 ^= 1u;
    }

    // ---- (2) phase 1
    if (sw) {
      if (m1 == M1_UP2) phase1<TW, TH, M1_UP2, true>(r0, r1, s_coef, tid, t, H, W);
      else if (m1 == M1_SAME) phase1<TW, TH, M1_SAME, true>(r0, r1, s_coef, tid, t, H, W);
      else phase1<TW, TH, M1_NONE, true>(r0, r1, s_coef, tid, t, H, W);
    } else {
      if (m1 == M1_UP2) phase1<TW, TH, M1_UP2, false>(r0, r1, s_coef, tid, t, H, W);
      else if (m1 == M1_SAME) phase1<TW, TH, M1_SAME, false>(r0, r1, s_coef, tid, t, H, W);
      else phase1<TW, TH, M1_NONE, false>(r0, r1, s_coef, tid, t, H, W);
    }
    __syncthreads();
    if (!pack_ready) {   // taps / bias / B operand have landed (first tile only)
      tc::mbar_wait(bar_pack, X.ph_pack);
      pack_ready = true;
    }

    // ---- (3) phase 2
    {
      bf16* dsave = (P.save_d != nullptr)
                        ? reinterpret_cast<bf16*>(P.save_d) + (((long long)t.b * H + t.ty0) * W + t.tx0) * C
                        : nullptr;
      phase2<TW, TH>(r0, r1, s_k, tid, dsave, W);
    }
    tc::fence_async_smem();   // the A operand was written through the generic proxy (and region 0 has been read)
    __syncthreads();
    const bool early0 = !PRE && (m1 == M1_UP2);   // output staged in region 1: region 0 is free from here on
    if (early0 && warp == 1 && next < ntiles) {
      const TilePos tn = tile_pos(next, tdiv, TW, TH);
      issue_input<TW, TH>(r0, in0, false, tn, H, W, lane, bar_in0);
    }
    // ---- (4) pointwise 1x1 on the tensor cores
    if (tid == 0) {
      tc::fence_after_sync();
#pragma unroll
      for (int j = 0; j < C / 16; ++j) {
        const uint64_t adesc = tc::make_desc(a_addr + j * 2 * S::kAStride, S::kAStride, 128);
        const uint64_t bdesc = tc::make_desc(b_addr + j * 2 * (C * 16), C * 16, 128);
        tc::umma_bf16(tmem_base, adesc, bdesc, kIdesc, j > 0 ? 1u : 0u);
      }
      tc::umma_commit(bar_mma);
    }
    tc::mbar_wait(bar_mma, X.ph_mma);
    X.ph_mma ^= 1u;
    tc::fence_after_sync();
    // region 1 is free: request the next tile's input 1 while the epilogue runs
    if (!PRE && warp == 1 && next < ntiles && m1 != M1_NONE) {
      const TilePos tn = tile_pos(next, tdiv, TW, TH);
      issue_input<TW, TH>(r1, in1, m1 == M1_UP2, tn, H, W, lane, bar_in1);
    }

    // ---- (5) epilogue: TMEM -> +bias -> dense bf16 staging tile (region 0; region 1 behind the input-1 rectangle for
    //      nodes with a nearest-x2 input)
    unsigned char* stg = early0 ? (r1 + S::kUp2Bytes) : r0;
    bf16* s_y = reinterpret_cast<bf16*>(stg);
    {
      const int row = 32 * (warp & 3) + lane;
      const int col0 = (warp >> 2) * (C / 2);
      const uint32_t taddr = tmem_base + ((uint32_t)(32 * (warp & 3)) << 16) + (uint32_t)col0;
      float acc[C / 16][8];
      tc::tmem_ld56(taddr, acc);
      if (row < S::NP) {
#pragma unroll
        for (int j = 0; j < C / 16; ++j) {
          const float4 b0 = *reinterpret_cast<const float4*>(s_bias + col0 + 8 * j);
          const float4 b1 = *reinterpret_cast<const float4*>(s_bias + col0 + 8 * j + 4);
          uint4 pk;
          pk.x = f2_to_bf2(add2(make_float2(acc[j][0], acc[j][1]), make_float2(b0.x, b0.y)));
          pk.y = f2_to_bf2(add2(make_float2(acc[j][2], acc[j][3]), make_float2(b0.z, b0.w)));
          pk.z = f2_to_bf2(add2(make_float2(acc[j][4], acc[j][5]), make_float2(b1.x, b1.y)));
          pk.w = f2_to_bf2(add2(make_float2(acc[j][6], acc[j][7]), make_float2(b1.z, b1.w)));
          *reinterpret_cast<uint4*>(s_y + row * C + col0 + 8 * j) = pk;
        }
      }
    }
    tc::fence_before_sync();   // order the TMEM reads before the next tile's MMAs
    tc::fence_async_smem();    // staging tile -> visible to the bulk store engine
    __syncthreads();

    // ---- (6) output tile: one bulk copy per tile row; BatchNorm statistics from the staging tile
    if (warp == 1) {
      if (lane < TH)
        bulk_s2g(out + (((long long)t.b * H + t.ty0 + lane) * W + t.tx0) * C, stg + lane * (TW * POS), TW * POS);
      bulk_commit();
    }
    if (train && ss < 4) {
      constexpr int NP = S::NP;
      const int p0 = ss * 32, p1 = (p0 + 32 < NP) ? p0 + 32 : NP;
      float2 s = make_float2(0.f, 0.f), q = make_float2(0.f, 0.f);
      const bf16* colp = s_y + 2 * sp;
#pragma unroll 8
      for (int p = p0; p < p1; ++p) {
        const float2 v = bf2_to_f2(*reinterpret_cast<const uint32_t*>(colp + p * C));
        s = add2(s, v);
        q = fma2(v, v, q);
      }
      st[0] += (double)s.x; st[1] += (double)s.y; st[2] += (double)q.x; st[3] += (double)q.y;
    }
    tc::fence_async_smem();   // generic accesses to region 0 are ordered before the next tile's bulk copies
    __syncthreads();
    if (warp == 1) {
      bulk_wait_read0();      // the bulk stores have read the staging tile
      __syncwarp();
      if (!early0 && next < ntiles) {
        const TilePos tn = tile_pos(next, tdiv, TW, TH);
        issue_input<TW, TH>(r0, in0, false, tn, H, W, lane, bar_in0);
      }
    }
  }
  if (!pack_ready) tc::mbar_wait(bar_pack, X.ph_pack);   // a CTA without tiles still consumes this node's pack phase
  X.ph_pack ^= 1u;

  // ---- BatchNorm statistics (+ finalisation by the last CTA of this network unless it is deferred; none when frozen)
  tc::fence_before_sync();
  __syncthreads();
  if (!train || P.frozen_bn) return;
  double* s_red = reinterpret_cast<double*>(r1);   // [4 slices][C/2 pairs][4]
  if (ss < 4) {
#pragma unroll
    for (int e = 0; e < 4; ++e) s_red[(ss * (C / 2) + sp) * 4 + e] = st[e];
  }
  __syncthreads();
  if (tid < C && cta < ntiles) {
    double s = 0.0, q = 0.0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      s += s_red[(k * (C / 2) + (tid >> 1)) * 4 + (tid & 1)];
      q += s_red[(k * (C / 2) + (tid >> 1)) * 4 + 2 + (tid & 1)];
    }
    double* rep = P.stats + (cta & (MMD_STATS_REPLICAS - 1)) * (2 * C);   // spread the same-address atomics
    atomicAdd(rep + tid, s);
    atomicAdd(rep + C + tid, q);
  }
  if (P.defer_bn) return;   // consumers rebuild (scale, shift) from the sums; bn_finalize_all does the rest
  __threadfence();
  __syncthreads();
  if (tid == 0) {
    const unsigned ticket = atomicAdd(P.counter, 1u);
    *s_flag = (ticket == (unsigned)nctas - 1u) ? 1 : 0;
  }
  __syncthreads();
  if (*s_flag == 0) return;
  __threadfence();
  if (tid < C) {
    const double n = (double)P.g.B * H * W;
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

// per-CTA one-time setup shared by the single-node kernel and the chain kernel: TMEM allocation, mbarrier init
__device__ __forceinline__ void fwd_ctx_init(unsigned char* smem, FwdCtx& X, const uint32_t tmem_cols) {
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + kOffBar);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bar + 4);
  const int tid = threadIdx.x, warp = tid >> 5;
  if (warp == 0) tc::tmem_alloc(s_tmem, tmem_cols);
  if (tid == 32) {
    tc::mbar_init(bar + 0, 1);
    tc::mbar_init(bar + 1, 1);
    tc::mbar_init(bar + 2, 1);
    tc::mbar_init(bar + 3, 1);
    tc::fence_mbar_init();
  }
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  X.tmem_base = *s_tmem;
  X.ph_pack = X.ph_in0 = X.ph_in1 = X.ph_mma = 0u;
}

template <int TW, int TH, bool PRE>
__global__ void __launch_bounds__(kThreads, 2) node_fwd_v4_kernel(const __grid_constant__ NodeFwdBatch BATCH) {
  constexpr uint32_t kTmemCols = 128;
  int net = 0;
#pragma unroll
  for (int k = 1; k < kMaxBatchNets; ++k)
    if ((int)blockIdx.x >= BATCH.cta_begin[k]) net = k;
  const int cta = (int)blockIdx.x - BATCH.cta_begin[net], nctas = BATCH.cta_begin[net + 1] - BATCH.cta_begin[net];
  extern __shared__ __align__(128) unsigned char smem[];
  FwdCtx X;
  fwd_ctx_init(smem, X, kTmemCols);
  node_fwd_body<TW, TH, PRE>(BATCH.p[net], BATCH.pre[net], cta, nctas, smem, X, true);
  tc::fence_before_sync();
  __syncthreads();
  if ((threadIdx.x >> 5) == 0) tc::tmem_dealloc(X.tmem_base, kTmemCols);
}

// ---- persistent small-level chain ---------------------------------------------------------------------------------------
// The P5 - P7 nodes hold 6 % of the bytes of a cell but took 26 % of the step as separate launches: every launch costs
// 12 - 20 us whatever it moves (launch -> prologue -> dependent parameter loads -> first tile -> drain).  Between two
// blocks of large-level work the small nodes form a strict chain (p5_out, p6_out, p7_out of cell k, then p6_up, p5_up of
// cell k + 1: src/YetAnotherEfficientDet.py:338-390), each needing its predecessor's complete output (tile halos, and in
// training the batch-global BatchNorm sums).  chain_fwd_kernel runs such a chain — for all lockstep networks — as ONE
// launch: the node bodies are the device functions above (TMEM allocated once, mbarrier phases carried from node to node,
// pooled inputs built inline) separated by a grid barrier.  All CTAs are co-resident (grid <= 2 x SM count, 2 CTAs / SM).
constexpr int kMaxChainSteps = 6;
struct ChainStep {
  NodeFwdP p[kMaxBatchNets];      // the node of every network
  NodeFwdP pre[kMaxBatchNets];    // its POOLFUSE pre-pass (has_pre): folded into the node body
  int cta_begin[kMaxBatchNets + 1];
  int geom;                       // pick_geom() code of the node's tile shape: 1 <12,8>, 3 <12,6>, 4 <6,6>
  int has_pre;
};
struct ChainFwd {
  ChainStep step[kMaxChainSteps];
  int n_steps;
  unsigned* sync;                 // [0] barrier arrivals, [1] exit tickets; zero on entry, re-zeroed by the last CTA to leave
  unsigned long long* dbg;        // MMD_CHAIN_DEBUG=1: [step][4] = min start, max body end, max barrier end, sum body ns (globaltimer)
};
static_assert(sizeof(ChainFwd) <= 32000, "kernel parameter space (32 764 bytes since CUDA 12.1)");

__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// Barrier over all CTAs of the grid.  Before arriving, everything this CTA wrote to global memory is made visible device
// wide: bulk shared->global stores are complete (wait_group 0 by the issuing warp), generic and async-proxy accesses are
// ordered against each other (the next node reads through bulk copies what this one wrote through generic stores, e.g.
// the inline-pooled operand, and vice versa), __threadfence.  A CTA that waits longer than ~1 s traps (a grid that is
// not co-resident would otherwise hang the GPU): the launch then fails loudly with a sticky CUDA error.
__device__ __forceinline__ void grid_barrier(unsigned* sync, const unsigned nctas, unsigned& epoch) {
  if ((threadIdx.x >> 5) == 1) bulk_wait_all();
  asm volatile("fence.proxy.async;" ::: "memory");
  __threadfence();
  __syncthreads();
  epoch += 1u;
  if (threadIdx.x == 0) {
    const unsigned target = epoch * nctas;
    atomicAdd(sync, 1u);
    unsigned seen, spins = 0u;
    while (true) {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(sync) : "memory");
      if (seen >= target) break;
      __nanosleep(64);
      if (++spins > (1u << 23)) __trap();
    }
    __threadfence();
  }
  __syncthreads();
  asm volatile("fence.proxy.async;" ::: "memory");
}

__device__ __forceinline__ unsigned long long gtimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

__global__ void __launch_bounds__(kThreads, 2) chain_fwd_kernel(const __grid_constant__ ChainFwd CH) {
  constexpr uint32_t kTmemCols = 128;
  extern __shared__ __align__(128) unsigned char smem[];
  FwdCtx X;
  fwd_ctx_init(smem, X, kTmemCols);
  unsigned epoch = 0u;
  for (int s = 0; s < CH.n_steps; ++s) {
    unsigned long long t0 = 0ull;
    if (CH.dbg != nullptr && threadIdx.x == 0) {
      t0 = gtimer();
      atomicMin(CH.dbg + 4 * s, t0);
    }
    const ChainStep& S = CH.step[s];
    int net = 0;
#pragma unroll
    for (int k = 1; k < kMaxBatchNets; ++k)
      if ((int)blockIdx.x >= S.cta_begin[k]) net = k;
    const int cta = (int)blockIdx.x - S.cta_begin[net], nctas = S.cta_begin[net + 1] - S.cta_begin[net];
    const bool active = (int)blockIdx.x < S.cta_begin[kMaxBatchNets];
    const bool pdl = (s == 0);
    if (active) {
      const NodeFwdP& P = S.p[net];
      const NodeFwdP& Q = S.pre[net];
      if (S.has_pre) {
        if (S.geom == 1) node_fwd_body<12, 8, true>(P, Q, cta, nctas, smem, X, pdl);
        else if (S.geom == 3) node_fwd_body<12, 6, true>(P, Q, cta, nctas, smem, X, pdl);
        else node_fwd_body<6, 6, true>(P, Q, cta, nctas, smem, X, pdl);
      } else {
        if (S.geom == 1) node_fwd_body<12, 8, false>(P, Q, cta, nctas, smem, X, pdl);
        else if (S.geom == 3) node_fwd_body<12, 6, false>(P, Q, cta, nctas, smem, X, pdl);
        else node_fwd_body<6, 6, false>(P, Q, cta, nctas, smem, X, pdl);
      }
    } else if (pdl) {
      pdl_wait();
      pdl_trigger();
    }
    if (CH.dbg != nullptr && threadIdx.x == 0) {
      const unsigned long long t1 = gtimer();
      atomicMax(CH.dbg + 4 * s + 1, t1);
      atomicAdd(CH.dbg + 4 * s + 3, t1 - t0);
    }
    if (s + 1 < CH.n_steps) grid_barrier(CH.sync, gridDim.x, epoch);
    if (CH.dbg != nullptr && threadIdx.x == 0) atomicMax(CH.dbg + 4 * s + 2, gtimer());
  }
  // ---- teardown: the last CTA to leave re-arms the barrier words for the next launch
  tc::fence_before_sync();
  __syncthreads();
  if ((threadIdx.x >> 5) == 0) tc::tmem_dealloc(X.tmem_base, kTmemCols);
  if (threadIdx.x == 0 && CH.n_steps > 1) {
    const unsigned ticket = atomicAdd(CH.sync + 1, 1u);
    if (ticket == gridDim.x - 1u) {
      CH.sync[0] = 0u;
      CH.sync[1] = 0u;
      __threadfence();
    }
  }
}

// ---- pooling pre-pass ------------------------------------------------------------------------------------------------
// out = w_a * maxpool3x3s2(bn_a(in[0]))  [+ w_b * bn_b(in[1])]   (final bf16 values at the node's resolution)
// MaxPool2dStaticSamePadding (src/YetAnotherEfficientNet.py:90-104): the zero padding takes part in the max of the
// NORMALISED values.  scale*x+shift is monotonic in x, so the window is searched on the raw bf16 values (sign flipped
// where the scale is negative): each value is expanded to fp32 with a 5-bit position tag in its lowest mantissa bits
// (those bits are zero after the expansion), so ONE fmaxf per element yields the maximum AND its position (larger tag =
// earlier in the row-major scan, so the first maximum wins for positive values).  A thread produces two horizontally
// adjacent outputs: their windows share a column, the 3 x 5 raw vectors are loaded and tagged once.
constexpr int kPoolThreads = 224;   // 16 output pairs x 14 channel groups
constexpr int kPoolLanes = kPoolThreads / NG;

template <bool NEG>
__device__ __forceinline__ void pool_key8(const uint4 r, const uint32_t tag, const uint32_t (&sgn)[8], float (&key)[8]) {
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    uint32_t lo = __byte_perm(w[e], tag, 0x1054);
    uint32_t hi = (w[e] & 0xffff0000u) | tag;
    if (NEG) { lo ^= sgn[2 * e]; hi ^= sgn[2 * e + 1]; }
    key[2 * e] = __uint_as_float(lo);
    key[2 * e + 1] = __uint_as_float(hi);
  }
}

// one output pair; BORDER: some window entries fall outside the source (zero padding)
template <bool NEG, bool BORDER>
__device__ __forceinline__ void pool_pair(const bf16* __restrict__ src, const int SH, const int SWd, const long long img,
                                          const int fy0, const int fx0, const int cg, const uint32_t (&sgn)[8],
                                          float (&bestA)[8], float (&bestB)[8], bool& padA, bool& padB) {
#pragma unroll
  for (int e = 0; e < 8; ++e) bestA[e] = bestB[e] = -INFINITY;
  padA = padB = false;
#pragma unroll
  for (int wy = 0; wy < 3; ++wy) {
    const int fy = fy0 + wy;
    const bool rok = !BORDER || (fy >= 0 && fy < SH);
    const bf16* row = src + (img + (long long)(BORDER ? min(max(fy, 0), SH - 1) : fy) * SWd) * C + 8 * cg;
#pragma unroll
    for (int cc = 0; cc < 5; ++cc) {
      const int fx = fx0 + cc;
      const bool ok = rok && (!BORDER || (fx >= 0 && fx < SWd));
      const uint4 r = __ldg(reinterpret_cast<const uint4*>(row + (long long)(BORDER ? min(max(fx, 0), SWd - 1) : fx) * C));
      float key[8];
      pool_key8<NEG>(r, 31u - (uint32_t)(wy * 5 + cc), sgn, key);
      if (BORDER && !ok) {
#pragma unroll
        for (int e = 0; e < 8; ++e) key[e] = -INFINITY;
        if (cc <= 2) padA = true;
        if (cc >= 2) padB = true;
      }
      if (cc <= 2) {
#pragma unroll
        for (int e = 0; e < 8; ++e) bestA[e] = fmaxf(bestA[e], key[e]);
      }
      if (cc >= 2) {
#pragma unroll
        for (int e = 0; e < 8; ++e) bestB[e] = fmaxf(bestB[e], key[e]);
      }
    }
  }
}

// Fast path for a pooled input that holds FINAL values and needs no arg-max record (frozen teachers: BatchNorm is folded
// into the 1x1 weights, nothing is saved for a backward): the window maximum is taken on the packed bf16 pairs directly
// (HMNMX2.BF16, one instruction per two channels, no expansion / tagging).
__device__ __forceinline__ uint32_t bfmax2(uint32_t a, uint32_t b) {
  __nv_bfloat162 r = __hmax2(*reinterpret_cast<const __nv_bfloat162*>(&a), *reinterpret_cast<const __nv_bfloat162*>(&b));
  return *reinterpret_cast<uint32_t*>(&r);
}
template <bool BORDER>
__device__ __forceinline__ void pool_pair_final(const bf16* __restrict__ src, const int SH, const int SWd, const long long img,
                                                const int fy0, const int fx0, const int cg, uint32_t (&bestA)[4],
                                                uint32_t (&bestB)[4], bool& padA, bool& padB) {
#pragma unroll
  for (int e = 0; e < 4; ++e) bestA[e] = bestB[e] = 0xff80ff80u;   // (-inf, -inf)
  padA = padB = false;
#pragma unroll
  for (int wy = 0; wy < 3; ++wy) {
    const int fy = fy0 + wy;
    const bool rok = !BORDER || (fy >= 0 && fy < SH);
    const bf16* row = src + (img + (long long)(BORDER ? min(max(fy, 0), SH - 1) : fy) * SWd) * C + 8 * cg;
#pragma unroll
    for (int cc = 0; cc < 5; ++cc) {
      const int fx = fx0 + cc;
      const bool ok = rok && (!BORDER || (fx >= 0 && fx < SWd));
      uint4 r = __ldg(reinterpret_cast<const uint4*>(row + (long long)(BORDER ? min(max(fx, 0), SWd - 1) : fx) * C));
      if (BORDER && !ok) {
        r = make_uint4(0xff80ff80u, 0xff80ff80u, 0xff80ff80u, 0xff80ff80u);
        if (cc <= 2) padA = true;
        if (cc >= 2) padB = true;
      }
      if (cc <= 2) {
        bestA[0] = bfmax2(bestA[0], r.x); bestA[1] = bfmax2(bestA[1], r.y);
        bestA[2] = bfmax2(bestA[2], r.z); bestA[3] = bfmax2(bestA[3], r.w);
      }
      if (cc >= 2) {
        bestB[0] = bfmax2(bestB[0], r.x); bestB[1] = bfmax2(bestB[1], r.y);
        bestB[2] = bfmax2(bestB[2], r.z); bestB[3] = bfmax2(bestB[3], r.w);
      }
    }
  }
}

// ---- what a thread does with the window maxima of its output pair (shared by poolfuse_kernel and poolfuse_tiled_kernel) ----
// frozen network: packed bf16 maxima -> w_a * max [+ second input] -> operand
__device__ __forceinline__ void emit_pair_final(const uint32_t (&bA)[4], const uint32_t (&bB)[4], const bool pA, const bool pB,
                                                const bool second, const long long oo0, const int cg, const float wa,
                                                const float* s_c, const bf16* __restrict__ same, bf16* __restrict__ out) {
#pragma unroll
  for (int o = 0; o < 2; ++o) {
    if (o == 1 && !second) break;
    const uint32_t* best = o ? bB : bA;
    const bool has_pad = o ? pB : pA;
    const long long oo = oo0 + (long long)o * C;
    uint4 sm = make_uint4(0u, 0u, 0u, 0u);
    if (same != nullptr) sm = __ldg(reinterpret_cast<const uint4*>(same + oo));
    const uint32_t sw[4] = {sm.x, sm.y, sm.z, sm.w};
    uint32_t pk[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const uint32_t m = has_pad ? bfmax2(best[e], 0u) : best[e];   // the zero padding takes part in the maximum
      float2 u = mul2(bf2_to_f2(m), make_float2(wa, wa));
      if (same != nullptr) {
        const float2 f = bf2_to_f2(sw[e]);
        u.x += fmaf(f.x, s_c[2 * C + 8 * cg + 2 * e], s_c[3 * C + 8 * cg + 2 * e]);
        u.y += fmaf(f.y, s_c[2 * C + 8 * cg + 2 * e + 1], s_c[3 * C + 8 * cg + 2 * e + 1]);
      }
      pk[e] = f2_to_bf2(u);
    }
    *reinterpret_cast<uint4*>(out + oo) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
  }
}

// training network: tagged fp32 keys -> value, window index (9 = padding), raw value at the arg-max; operand, arg-max bytes and
// raw values go to HBM
__device__ __forceinline__ void emit_pair_train(const float (&bestA)[8], const float (&bestB)[8], const bool padA, const bool padB,
                                                const bool pad_first, const bool second, const long long oo0, const int cg,
                                                const float wa, const float (&sc)[8], const float (&sh)[8], const uint32_t (&sgn)[8],
                                                const float* s_c, const bf16* __restrict__ same, bf16* __restrict__ out,
                                                unsigned char* __restrict__ pidx, bf16* __restrict__ praw) {
#pragma unroll
  for (int o = 0; o < 2; ++o) {
    if (o == 1 && !second) break;
    const float* best = o ? bestB : bestA;
    const bool has_pad = o ? padB : padA;
    float u[8];
    uint32_t idx[8], rawb[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const uint32_t bits = __float_as_uint(best[e]);
      const uint32_t t = 31u - (bits & 31u);
      const uint32_t wy = (t * 52u) >> 8;            // t / 5 for t < 32
      idx[e] = wy * 3u + (t - wy * 5u) - (o ? 2u : 0u);
      rawb[e] = (bits ^ sgn[e]) & 0xffff0000u;
      float val = fmaf(__uint_as_float(rawb[e]), sc[e], sh[e]);
      if (has_pad && (pad_first ? (0.f >= val) : (0.f > val))) {
        val = 0.f;
        idx[e] = 9u;
        rawb[e] = 0u;
      }
      u[e] = wa * val;
    }
    const long long oo = oo0 + (long long)o * C;
    if (same != nullptr) {
      const uint4 r = __ldg(reinterpret_cast<const uint4*>(same + oo));
      const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 f = bf2_to_f2(w[e]);
        u[2 * e] += fmaf(f.x, s_c[2 * C + 8 * cg + 2 * e], s_c[3 * C + 8 * cg + 2 * e]);
        u[2 * e + 1] += fmaf(f.y, s_c[2 * C + 8 * cg + 2 * e + 1], s_c[3 * C + 8 * cg + 2 * e + 1]);
      }
    }
    uint4 pk;
    pk.x = f2_to_bf2(make_float2(u[0], u[1]));
    pk.y = f2_to_bf2(make_float2(u[2], u[3]));
    pk.z = f2_to_bf2(make_float2(u[4], u[5]));
    pk.w = f2_to_bf2(make_float2(u[6], u[7]));
    *reinterpret_cast<uint4*>(out + oo) = pk;
    if (pidx != nullptr) {
      uint2 ip;
      ip.x = idx[0] | (idx[1] << 8) | (idx[2] << 16) | (idx[3] << 24);
      ip.y = idx[4] | (idx[5] << 8) | (idx[6] << 16) | (idx[7] << 24);
      *reinterpret_cast<uint2*>(pidx + oo) = ip;
    }
    if (praw != nullptr) {
      uint4 rp;
      rp.x = (rawb[0] >> 16) | rawb[1];
      rp.y = (rawb[2] >> 16) | rawb[3];
      rp.z = (rawb[4] >> 16) | rawb[5];
      rp.w = (rawb[6] >> 16) | rawb[7];
      *reinterpret_cast<uint4*>(praw + oo) = rp;
    }
  }
}

template <int MINB>
__global__ void __launch_bounds__(kPoolThreads, MINB) poolfuse_kernel(const __grid_constant__ NodeFwdBatch BATCH) {
  int net = 0;
#pragma unroll
  for (int k = 1; k < kMaxBatchNets; ++k)
    if ((int)blockIdx.x >= BATCH.cta_begin[k]) net = k;
  const NodeFwdP& P = BATCH.p[net];
  const int cta = (int)blockIdx.x - BATCH.cta_begin[net], nctas = BATCH.cta_begin[net + 1] - BATCH.cta_begin[net];
  __shared__ __align__(16) float s_c[4 * C];   // pooled input: scale | shift ; second input: w_b*scale | w_b*shift
  const int cg = threadIdx.x % NG, pl = threadIdx.x / NG;
  const int H = P.g.H, W = P.g.W, SH = P.in[0].H, SWd = P.in[0].W;
  const int WP = (W + 1) >> 1;                  // output pairs per row
  const int npairs = P.g.B * H * WP;
  const bf16* __restrict__ src = reinterpret_cast<const bf16*>(P.in[0].data);
  const bf16* __restrict__ same = (P.n_in >= 2) ? reinterpret_cast<const bf16*>(P.in[1].data) : nullptr;
  bf16* __restrict__ out = reinterpret_cast<bf16*>(P.out);
  bf16* __restrict__ praw = reinterpret_cast<bf16*>(P.save_d);
  unsigned char* __restrict__ pidx = P.pidx[0];

  pdl_wait();
  pdl_trigger();
  const float wa = in_weight(P, 0);
  if (threadIdx.x < C) {
    const int c = threadIdx.x;
    const float wb = (P.n_in >= 2) ? in_weight(P, 1) : 0.f;
    float ps0, ph0, ps1 = 1.f, ph1 = 0.f;
    bn_coef<C>(P.in[0], P.bnsrc[0], c, ps0, ph0);
    if (P.n_in >= 2) bn_coef<C>(P.in[1], P.bnsrc[1], c, ps1, ph1);
    s_c[c] = ps0;
    s_c[C + c] = ph0;
    s_c[2 * C + c] = ps1 * wb;
    s_c[3 * C + c] = ph1 * wb;
  }
  __syncthreads();
  float sc[8], sh[8];
  uint32_t sgn[8];
  bool anyneg = false;
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    sc[e] = s_c[8 * cg + e];
    sh[e] = s_c[C + 8 * cg + e];
    sgn[e] = (sc[e] < 0.f) ? 0x80000000u : 0u;
    anyneg = anyneg || (sc[e] < 0.f);
  }
  const int top = pool_pad_before(SH), left = pool_pad_before(SWd);
  const bool final_in = (P.in[0].bn == nullptr) && (pidx == nullptr) && (praw == nullptr);

  for (int pp = cta * kPoolLanes + pl; pp < npairs; pp += nctas * kPoolLanes) {
    const int b = pp / (H * WP);
    const int rem = pp - b * (H * WP);
    const int y = rem / WP, xp = rem - y * WP;
    const int x0 = 2 * xp;
    const bool second = (x0 + 1 < W);
    const int fy0 = 2 * y - top, fx0 = 2 * x0 - left;
    const long long img = (long long)b * SH * SWd;
    const bool border = (fy0 < 0) || (fy0 + 2 >= SH) || (fx0 < 0) || (fx0 + 4 >= SWd);
    if (final_in) {
      uint32_t bA[4], bB[4];
      bool pA, pB;
      if (!border) pool_pair_final<false>(src, SH, SWd, img, fy0, fx0, cg, bA, bB, pA, pB);
      else pool_pair_final<true>(src, SH, SWd, img, fy0, fx0, cg, bA, bB, pA, pB);
      emit_pair_final(bA, bB, pA, pB, second, (((long long)b * H + y) * W + x0) * C + 8 * cg, cg, wa, s_c, same, out);
      continue;
    }
    float bestA[8], bestB[8];
    bool padA, padB;
    if (!border) {
      if (anyneg) pool_pair<true, false>(src, SH, SWd, img, fy0, fx0, cg, sgn, bestA, bestB, padA, padB);
      else pool_pair<false, false>(src, SH, SWd, img, fy0, fx0, cg, sgn, bestA, bestB, padA, padB);
    } else {
      pool_pair<true, true>(src, SH, SWd, img, fy0, fx0, cg, sgn, bestA, bestB, padA, padB);
    }
    const bool pad_first = (fy0 < 0) || (fx0 < 0);   // left / top padding precedes the real elements in scan order
    emit_pair_train(bestA, bestB, padA, padB, pad_first, second, (((long long)b * H + y) * W + x0) * C + 8 * cg, cg, wa, sc, sh, sgn,
                    s_c, same, out, pidx, praw);
  }
}

// ---- pooling pre-pass, shared-memory tiled (large levels: P3 -> P4, P4 -> P5) -------------------------------------------
// poolfuse_kernel reads every source element ~1.9 times through L1 / L2 (3 x 5 window loads per output pair, rows shared
// with the pair below) and is bound by the latency of those loads (ncu: 12.9 warps stalled on the long scoreboard per issue,
// DRAM traffic 1.27 x the algorithmic bytes).  Here a CTA walks a strip of kPtRows output rows x kPtCols output columns of one
// image top to bottom and keeps the source rows it needs in a RING of shared-memory row slots filled by bulk asynchronous
// copies (one per source row, mbarrier completion) kPtSlots - 3 source rows ahead of the compute: every source element is
// read from HBM once per strip (+ one halo row per strip and one halo column) and the window scan reads shared memory.
// Work item = (image, row strip, column strip); thread = (output pair, channel group) as in poolfuse_kernel, whose scan
// (tagged keys for the training network, packed bf16 maxima for frozen ones) and emit code it shares.
// Even source sizes only (no top / left padding): the D2 pyramid.
constexpr int kPtCols = 24;                       // output columns per strip  -> 49 source columns per row slot
constexpr int kPtRows = 8;                        // output rows per strip     -> 17 source rows
constexpr int kPtSlots = 9;                       // ring slots (source rows)
constexpr int kPtSlotBytes = up128((2 * kPtCols + 1) * POS);   // 11 008
constexpr int kPtRowThreads = (kPtCols / 2) * NG; // 168: 12 output pairs x 14 channel groups = one output row of the strip
constexpr int kPtRowsPerStep = 2;                 // output rows computed concurrently (2 x 168 threads: more warps per SM)
constexpr int kPtThreads = kPtRowsPerStep * kPtRowThreads;
constexpr int kPtSmem = kPtSlots * kPtSlotBytes + 4 * C * 4 + kPtSlots * 8 + 16;

__global__ void __launch_bounds__(kPtThreads, 2) poolfuse_tiled_kernel(const __grid_constant__ NodeFwdBatch BATCH) {
  int net = 0;
#pragma unroll
  for (int k = 1; k < kMaxBatchNets; ++k)
    if ((int)blockIdx.x >= BATCH.cta_begin[k]) net = k;
  const NodeFwdP& P = BATCH.p[net];
  const int cta = (int)blockIdx.x - BATCH.cta_begin[net], nctas = BATCH.cta_begin[net + 1] - BATCH.cta_begin[net];
  extern __shared__ __align__(128) unsigned char smem[];
  float* s_c = reinterpret_cast<float*>(smem + kPtSlots * kPtSlotBytes);   // scale | shift | w_b*scale_b | w_b*shift_b
  uint64_t* bar = reinterpret_cast<uint64_t*>(s_c + 4 * C);                // [kPtSlots] slot filled
  const int tid = threadIdx.x, rg = tid / kPtRowThreads, tl = tid - rg * kPtRowThreads;   // row group, thread inside it
  const int cg = tl % NG, pl = tl / NG;
  const int H = P.g.H, W = P.g.W, SH = P.in[0].H, SWd = P.in[0].W;
  const bf16* __restrict__ src = reinterpret_cast<const bf16*>(P.in[0].data);
  const bf16* __restrict__ same = (P.n_in >= 2) ? reinterpret_cast<const bf16*>(P.in[1].data) : nullptr;
  bf16* __restrict__ out = reinterpret_cast<bf16*>(P.out);
  bf16* __restrict__ praw = reinterpret_cast<bf16*>(P.save_d);
  unsigned char* __restrict__ pidx = P.pidx[0];
  if (tid == 0) {
    for (int i = 0; i < kPtSlots; ++i) tc::mbar_init(bar + i, 1);
    tc::fence_mbar_init();
  }
  pdl_wait();
  pdl_trigger();
  const float wa = in_weight(P, 0);
  if (tid < C) {
    const float wb = (P.n_in >= 2) ? in_weight(P, 1) : 0.f;
    float ps0, ph0, ps1 = 1.f, ph1 = 0.f;
    bn_coef<C>(P.in[0], P.bnsrc[0], tid, ps0, ph0);
    if (P.n_in >= 2) bn_coef<C>(P.in[1], P.bnsrc[1], tid, ps1, ph1);
    s_c[tid] = ps0;
    s_c[C + tid] = ph0;
    s_c[2 * C + tid] = ps1 * wb;
    s_c[3 * C + tid] = ph1 * wb;
  }
  __syncthreads();
  float sc[8], sh[8];
  uint32_t sgn[8];
  bool anyneg = false;
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    sc[e] = s_c[8 * cg + e];
    sh[e] = s_c[C + 8 * cg + e];
    sgn[e] = (sc[e] < 0.f) ? 0x80000000u : 0u;
    anyneg = anyneg || (sc[e] < 0.f);
  }
  const bool final_in = (P.in[0].bn == nullptr) && (pidx == nullptr) && (praw == nullptr);

  const int strips_y = (H + kPtRows - 1) / kPtRows, strips_x = W / kPtCols;
  const int nitems = P.g.B * strips_y * strips_x;
  uint32_t phases = 0u;   // bit i: parity the next wait on slot i expects
  for (int item = cta; item < nitems; item += nctas) {
    const int b = item / (strips_y * strips_x);
    const int rem = item - b * (strips_y * strips_x);
    const int y0 = (rem / strips_x) * kPtRows, xs0 = (rem % strips_x) * kPtCols;
    const int ny = min(kPtRows, H - y0);
    const int sy0 = 2 * y0, sx0 = 2 * xs0;
    const int nsrc = min(2 * ny + 1, SH - sy0);                 // source rows of this strip that exist
    const int ncol = min(2 * kPtCols + 1, SWd - sx0);           // source columns that exist (49, or 48 at the right border)
    const bf16* src0 = src + (((long long)b * SH + sy0) * SWd + sx0) * C;
    auto issue_row = [&](int r) {   // source row r of the strip -> slot r % kPtSlots   (thread 0)
      const int sl = r % kPtSlots;
      tc::mbar_expect_tx(bar + sl, (uint32_t)ncol * POS);
      tc::bulk_g2s(smem + sl * kPtSlotBytes, src0 + (long long)r * SWd * C, (uint32_t)ncol * POS, bar + sl);
    };
    if (tid == 0)
      for (int r = 0; r < min(nsrc, kPtSlots); ++r) issue_row(r);
    int waited = 0;   // source rows [0, waited) of this strip have landed and been observed by this thread
    for (int ys = 0; ys < ny; ys += kPtRowsPerStep) {
      const int yy = ys + rg;                      // this row group's output row of the step
      const int need = min(2 * (ys + kPtRowsPerStep - 1) + 3, nsrc);
      for (; waited < need; ++waited) {
        const int sl = waited % kPtSlots;
        tc::mbar_wait(bar + sl, (phases >> sl) & 1u);
        phases ^= (1u << sl);
      }
      if (yy < ny) {
      const int y = y0 + yy;
      const int x0 = xs0 + 2 * pl;
      const long long oo0 = (((long long)b * H + y) * W + x0) * C + 8 * cg;
      // the three window rows of this output row (a row beyond the image is the zero padding: any readable slot will do)
      const unsigned char* rows[3];
      bool rok[3];
#pragma unroll
      for (int wy = 0; wy < 3; ++wy) {
        const int r = 2 * yy + wy;
        rok[wy] = r < nsrc;
        rows[wy] = smem + ((rok[wy] ? r : 2 * yy) % kPtSlots) * kPtSlotBytes + (4 * pl) * POS + cg * 16;
      }
      const int cols_ok = ncol - 4 * pl;   // valid source columns from this thread's first one (>= 5 unless at the right border)
      const bool border = !rok[2] || cols_ok < 5;
      if (final_in) {
        uint32_t bA[4], bB[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) bA[e] = bB[e] = 0xff80ff80u;   // (-inf, -inf)
        bool pA = false, pB = false;
#pragma unroll
        for (int wy = 0; wy < 3; ++wy) {
#pragma unroll
          for (int cc = 0; cc < 5; ++cc) {
            uint4 r = *reinterpret_cast<const uint4*>(rows[wy] + (cc < cols_ok ? cc : 0) * POS);
            if (border && !(rok[wy] && cc < cols_ok)) {
              r = make_uint4(0xff80ff80u, 0xff80ff80u, 0xff80ff80u, 0xff80ff80u);
              if (cc <= 2) pA = true;
              if (cc >= 2) pB = true;
            }
            if (cc <= 2) {
              bA[0] = bfmax2(bA[0], r.x); bA[1] = bfmax2(bA[1], r.y); bA[2] = bfmax2(bA[2], r.z); bA[3] = bfmax2(bA[3], r.w);
            }
            if (cc >= 2) {
              bB[0] = bfmax2(bB[0], r.x); bB[1] = bfmax2(bB[1], r.y); bB[2] = bfmax2(bB[2], r.z); bB[3] = bfmax2(bB[3], r.w);
            }
          }
        }
        emit_pair_final(bA, bB, pA, pB, true, oo0, cg, wa, s_c, same, out);
      } else {
        float bestA[8], bestB[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) bestA[e] = bestB[e] = -INFINITY;
        bool padA = false, padB = false;
#pragma unroll
        for (int wy = 0; wy < 3; ++wy) {
#pragma unroll
          for (int cc = 0; cc < 5; ++cc) {
            const uint4 r = *reinterpret_cast<const uint4*>(rows[wy] + (cc < cols_ok ? cc : 0) * POS);
            float key[8];
            if (anyneg) pool_key8<true>(r, 31u - (uint32_t)(wy * 5 + cc), sgn, key);
            else pool_key8<false>(r, 31u - (uint32_t)(wy * 5 + cc), sgn, key);
            if (border && !(rok[wy] && cc < cols_ok)) {
#pragma unroll
              for (int e = 0; e < 8; ++e) key[e] = -INFINITY;
              if (cc <= 2) padA = true;
              if (cc >= 2) padB = true;
            }
            if (cc <= 2) {
#pragma unroll
              for (int e = 0; e < 8; ++e) bestA[e] = fmaxf(bestA[e], key[e]);
            }
            if (cc >= 2) {
#pragma unroll
              for (int e = 0; e < 8; ++e) bestB[e] = fmaxf(bestB[e], key[e]);
            }
          }
        }
        emit_pair_train(bestA, bestB, padA, padB, false, true, oo0, cg, wa, sc, sh, sgn, s_c, same, out, pidx, praw);
      }
      }
      // the first 2 * kPtRowsPerStep source rows of the step are dead: their slots take the rows kPtSlots further down
      // (generic reads -> async-proxy writes)
      tc::fence_async_smem();
      __syncthreads();
      if (tid == 0) {
        for (int r = 2 * ys + kPtSlots; r < min(nsrc, 2 * ys + 2 * kPtRowsPerStep + kPtSlots); ++r) issue_row(r);
      }
    }
    // drain: rows of this strip that were loaded but never needed (none: need == nsrc at the last output row), and make sure
    // every thread has observed every landed row before the next strip re-arms the barriers
    for (; waited < nsrc; ++waited) {
      const int sl = waited % kPtSlots;
      tc::mbar_wait(bar + sl, (phases >> sl) & 1u);
      phases ^= (1u << sl);
    }
    __syncthreads();
  }
}

template <int TW, int TH, bool PRE = false>
static int launch_geom(const NodeFwdBatch& batch, int n, cudaStream_t s) {
  using S = Cfg<TW, TH>;
  MMD_SMEM((node_fwd_v4_kernel<TW, TH, PRE>), (PRE ? S::kBytesPre : S::kBytes));
  const int sms = device_sm_count();
  const NodeFwdP& p = batch.p[0];
  const int ntiles = p.g.B * (p.g.H / TH) * (p.g.W / TW);
  static const float train_w = env_float("MMD_FWD_TRAIN_SHARE", 1.0f);
  NodeFwdBatch b2 = batch;
  batch_shares(b2, n, 2 * sms, ntiles, train_w);
  MMD_CUDA(launch_pdl(node_fwd_v4_kernel<TW, TH, PRE>, dim3(b2.cta_begin[n]), dim3(kThreads), PRE ? S::kBytesPre : S::kBytes, s, b2));
  MMD_LAUNCH_CHECK();
  return 0;
}

// tile shapes, tried in this order (exact fits only; anything else runs on the generic kernel of bifpn_fwd_tc.cu)
static int pick_geom(int H, int W) {
  if (W % 16 == 0 && H % 8 == 0) return 0;
  if (W % 12 == 0 && H % 8 == 0) return 1;
  if (W % 8 == 0 && H % 8 == 0) return 2;
  if (W % 12 == 0 && H % 6 == 0) return 3;
  if (W % 6 == 0 && H % 6 == 0) return 4;
  return -1;
}

}  // namespace v4

namespace v4 {
// ---- deferred BatchNorm finalisation: one block per train-mode op of the forward ------------------------------------
// Same arithmetic as the in-kernel finaliser (and as bn_coef()): out_bn = scale | shift | mean | invstd, running statistics
// (momentum update with the unbiased variance, src/YetAnotherEfficientDet.py:176 semantics of nn.BatchNorm2d),
// num_batches_tracked, accumulators cleared for the next forward.
__global__ void __launch_bounds__(128) bn_finalize_all_kernel(const __grid_constant__ BnFinalBatch BATCH) {
  const BnFinalEntry& E = BATCH.e[blockIdx.x];
  const int tid = threadIdx.x;
  pdl_wait();
  if (tid < C) {
    double sum = 0.0, sq = 0.0;
#pragma unroll
    for (int r = 0; r < MMD_STATS_REPLICAS; ++r) {
      sum += __ldcg(E.stats + r * (2 * C) + tid);
      sq += __ldcg(E.stats + r * (2 * C) + C + tid);
    }
    const double n = E.n;
    const double mean = sum / n;
    double var = sq / n - mean * mean;
    if (var < 0.0) var = 0.0;
    const float invstd = (float)(1.0 / sqrt(var + (double)E.eps));
    const float scale = E.gamma[tid] * invstd;
    E.out_bn[tid] = scale;
    E.out_bn[C + tid] = E.beta[tid] - (float)mean * scale;
    E.out_bn[2 * C + tid] = (float)mean;
    E.out_bn[3 * C + tid] = invstd;
    const double unbiased = var * (n / (n > 1.0 ? n - 1.0 : 1.0));
    E.rm[tid] = (1.f - E.mom) * E.rm[tid] + E.mom * (float)mean;
    E.rv[tid] = (1.f - E.mom) * E.rv[tid] + E.mom * (float)unbiased;
#pragma unroll
    for (int r = 0; r < MMD_STATS_REPLICAS; ++r) {
      E.stats[r * (2 * C) + tid] = 0.0;
      E.stats[r * (2 * C) + C + tid] = 0.0;
    }
  }
  if (tid == 0 && E.nbt) *E.nbt += 1;
}
}  // namespace v4


// ---- streaming BNAPPLY (bf16, SAME mode): the 5 stack outputs of a training forward -----------------------------------
// out = scale * x + shift over the flat tensor.  The generic kernel (bifpn_fwd.cu) handles 4 channels per thread with
// three 64-bit divisions per element and one 8-byte load in flight: ~0.2 of the HBM rate.  Here a block is 16 positions x
// 14 channel groups (one 16-byte vector per thread, the thread's channel group never changes, so its 8 + 8 coefficients
// live in registers), four position blocks per iteration in flight.  blockIdx.y = op of the group.
namespace v4 {
constexpr int kBnThreads = 224;   // 16 positions x 14 channel groups
__global__ void __launch_bounds__(kBnThreads) bnapply_same_bf16_kernel(const __grid_constant__ NodeFwdGroup GROUP) {
  const NodeFwdP& P = GROUP.p[blockIdx.y];
  __shared__ __align__(16) float s_bn[2 * C];
  const long long npos = (long long)P.g.B * P.g.H * P.g.W;
  const long long nblk = (npos + 15) / 16;
  if ((long long)blockIdx.x >= nblk) return;
  pdl_wait();
  pdl_trigger();
  if (threadIdx.x < C) {
    float sc1, sh1;
    bn_coef<C>(P.in[0], P.bnsrc[0], threadIdx.x, sc1, sh1);
    s_bn[threadIdx.x] = sc1;
    s_bn[C + threadIdx.x] = sh1;
  }
  __syncthreads();
  const int cg = threadIdx.x % NG, pl = threadIdx.x / NG;
  float2 sc[4], sh[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    sc[e] = *reinterpret_cast<const float2*>(s_bn + 8 * cg + 2 * e);
    sh[e] = *reinterpret_cast<const float2*>(s_bn + C + 8 * cg + 2 * e);
  }
  const uint4* __restrict__ src = reinterpret_cast<const uint4*>(P.in[0].data);
  uint4* __restrict__ dst = reinterpret_cast<uint4*>(P.out);
  constexpr int U = 4;
  for (long long blk = blockIdx.x; blk < nblk; blk += (long long)U * gridDim.x) {
    uint4 r[U];
    long long pos[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      pos[u] = (blk + (long long)u * gridDim.x) * 16 + pl;
      r[u] = make_uint4(0u, 0u, 0u, 0u);
      if (pos[u] < npos) r[u] = __ldg(src + pos[u] * NG + cg);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (pos[u] >= npos) continue;
      uint4 o;
      o.x = f2_to_bf2(fma2(bf2_to_f2(r[u].x), sc[0], sh[0]));
      o.y = f2_to_bf2(fma2(bf2_to_f2(r[u].y), sc[1], sh[1]));
      o.z = f2_to_bf2(fma2(bf2_to_f2(r[u].z), sc[2], sh[2]));
      o.w = f2_to_bf2(fma2(bf2_to_f2(r[u].w), sc[3], sh[3]));
      dst[pos[u] * NG + cg] = o;
    }
  }
}
}  // namespace v4

bool bnapply_same_bf16_usable(const NodeFwdP* p, int n) {
  for (int i = 0; i < n; ++i) {
    if (p[i].mode[0] != MMD_IN_SAME || p[i].pidx[0] != nullptr) return false;
    if ((((uintptr_t)p[i].in[0].data | (uintptr_t)p[i].out) & 15u) != 0) return false;
  }
  return true;
}

int launch_bnapply_same_bf16(const NodeFwdP* p, int n, cudaStream_t s) {
  NodeFwdGroup group;
  double bytes = 0.0;
  long long maxblk = 1;
  for (int i = 0; i < kMaxGroupOps; ++i) group.p[i] = p[i < n ? i : 0];
  for (int i = 0; i < n; ++i) {
    bytes += node_algo_bytes(p[i].in, 1, p[i].g, 112, 2);
    const long long nblk = ((long long)p[i].g.B * p[i].g.H * p[i].g.W + 15) / 16;
    if (nblk > maxblk) maxblk = nblk;
  }
  long long grid = (maxblk + 3) / 4;
  const long long cap = 8LL * device_sm_count();
  if (grid > cap) grid = cap;
  ProfScope prof(PK_BNAPPLY, bytes, s);
  MMD_CUDA(launch_pdl(v4::bnapply_same_bf16_kernel, dim3((unsigned)grid, n), dim3(v4::kBnThreads), 0, s, group));
  MMD_LAUNCH_CHECK();
  return 0;
}

bool bn_deferral_enabled() {
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("MMD_NO_DEFER_BN");
    const char* v = getenv("MMD_NO_V4");   // the generic node kernels read the finalised vectors only
    on = ((e && e[0] == '1') || (v && v[0] == '1')) ? 0 : 1;
  }
  return on == 1;
}

int launch_bn_finalize_all(const BnFinalEntry* entries, int n, int C, cudaStream_t s) {
  MMD_CHECK_ARG(C == 112, "BiFPN kernels are built for C=112 (EfficientDet-D2), got %d", C);
  for (int i0 = 0; i0 < n; i0 += kBnFinalPerLaunch) {
    const int m = (n - i0 < kBnFinalPerLaunch) ? n - i0 : kBnFinalPerLaunch;
    BnFinalBatch batch;
    for (int k = 0; k < kBnFinalPerLaunch; ++k) batch.e[k] = entries[i0 + (k < m ? k : 0)];
    MMD_CUDA(launch_pdl(v4::bn_finalize_all_kernel, dim3(m), dim3(128), 0, s, batch));
    MMD_LAUNCH_CHECK();
  }
  return 0;
}

float env_float(const char* name, float dflt) {
  const char* e = getenv(name);
  if (e == nullptr || *e == 0) return dflt;
  const float v = (float)atof(e);
  return v > 0.f ? v : dflt;
}

void batch_shares(NodeFwdBatch& batch, int n, int budget, int max_per_net, float train_w) {
  float wsum = 0.f;
  for (int i = 0; i < n; ++i) wsum += batch.p[i].train ? train_w : 1.f;
  int begin = 0;
  for (int i = 0; i < kMaxBatchNets; ++i) {
    batch.cta_begin[i] = begin;
    if (i < n) {
      int c = (int)((float)budget * (batch.p[i].train ? train_w : 1.f) / wsum);
      if (c > max_per_net) c = max_per_net;
      if (c < 1) c = 1;
      begin += c;
    }
  }
  batch.cta_begin[kMaxBatchNets] = begin;
  for (int i = n; i <= kMaxBatchNets; ++i) batch.cta_begin[i] = begin;
}

bool fwd_v4_usable(const NodeFwdP& p) {
  if (p.packed == nullptr || p.n_in < 1 || p.n_in > 2 || p.mode[0] != MMD_IN_SAME) return false;
  if (p.n_in == 2 && p.mode[1] == MMD_IN_POOL) return false;
  if (p.n_in == 2 && p.mode[1] == MMD_IN_UP2 && (2 * p.in[1].H != p.g.H || 2 * p.in[1].W != p.g.W)) return false;
  for (int i = 0; i < p.n_in; ++i)
    if (((uintptr_t)p.in[i].data & 15u) != 0) return false;
  if (((uintptr_t)p.out & 15u) != 0) return false;
  return v4::pick_geom(p.g.H, p.g.W) >= 0;
}

int launch_node_fwd_v4(const NodeFwdP* p, int n, int C, cudaStream_t s) {
  MMD_CHECK_ARG(C == 112, "BiFPN kernels are built for C=112 (EfficientDet-D2), got %d", C);
  MMD_CHECK_ARG(n >= 1 && n <= kMaxBatchNets, "node_fwd_v4: %d networks in one launch", n);
  NodeFwdBatch batch;
  double bytes = 0.0;
  for (int i = 0; i < n; ++i) {
    batch.p[i] = p[i];
    MMD_CHECK_ARG(p[i].g.H == p[0].g.H && p[i].g.W == p[0].g.W && p[i].g.B == p[0].g.B,
                  "node_fwd_v4: batched networks must share the geometry");
    // a node fed by a POOLFUSE pre-pass: the reads of its pooled / third input are charged to the pre-pass
    const bool aux = p[i].fw_n > 0 && p[i].n_in == 2 && p[i].fw_idx[1] < 0;
    bytes += node_algo_bytes(p[i].in, aux ? 1 : p[i].n_in, p[i].g, C, 2);
  }
  for (int i = n; i < kMaxBatchNets; ++i) batch.p[i] = p[0];
  const int geom = v4::pick_geom(p[0].g.H, p[0].g.W);
  ProfScope prof(geom == 0 ? PK_NODE_FWD_16x8 : PK_NODE_FWD, bytes, s);
  switch (geom) {
    case 0: return v4::launch_geom<16, 8>(batch, n, s);
    case 1: return v4::launch_geom<12, 8>(batch, n, s);
    case 2: return v4::launch_geom<8, 8>(batch, n, s);
    case 3: return v4::launch_geom<12, 6>(batch, n, s);
    case 4: return v4::launch_geom<6, 6>(batch, n, s);
  }
  set_error("node_fwd_v4: no tile shape fits %dx%d", p[0].g.H, p[0].g.W);
  return MMD_E_ARG;
}

bool fwd_v4_pre_usable(const NodeFwdP& pre, const NodeFwdP& node) {
  // Off unless MMD_INLINE_POOL=1.  Measured (B=16, 4 lockstep networks): 15 launches per step fewer and -0.31 ms of
  // poolfuse time, but +0.33 ms in the node kernels — every thread walks ~8 (position, channel group) items of nine
  // dependent L2 loads each per tile — i.e. break-even; kept as the starting point of the persistent small-level kernels.
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("MMD_INLINE_POOL");
    on = (e && e[0] == '1') ? 1 : 0;
  }
  if (!on) return false;
  return fwd_v4_pre_fusable(pre, node);
}

// conditions under which the node body can build the pre-pass operand inline (PRE = true instantiations)
bool fwd_v4_pre_fusable(const NodeFwdP& pre, const NodeFwdP& node) {
  if (!fwd_v4_usable(node) || node.n_in != 2 || node.mode[1] != MMD_IN_SAME) return false;
  if (node.in[1].data != pre.out || pre.out == nullptr) return false;                     // the node consumes the pre-pass
  if (pre.mode[0] != MMD_IN_POOL || (pre.n_in == 2 && pre.mode[1] != MMD_IN_SAME) || pre.n_in > 2) return false;
  if (pre.g.H != node.g.H || pre.g.W != node.g.W || node.g.H * node.g.W > 24 * 24) return false;   // P5 and smaller
  const int geom = v4::pick_geom(node.g.H, node.g.W);
  if (geom != 1 && geom != 3 && geom != 4) return false;
  for (int i = 0; i < pre.n_in; ++i)
    if (((uintptr_t)pre.in[i].data & 15u) != 0) return false;
  return (((uintptr_t)pre.out | (uintptr_t)pre.pidx[0] | (uintptr_t)pre.save_d) & 15u) == 0;
}

// Off by default.  Measured on B200 (profiles/r2_chain_fwd.md): the chain of one cell boundary (5 nodes, 4 lockstep
// networks, B = 16) takes 120 - 160 us against 110 - 143 us for the same nodes as separate PDL launches — the time of a
// small-level node is the latency of ONE tile through the body (parameter block + coefficient round trips, two CUDA-core
// phases, MMA, epilogue, store drain: ~10 us), which a grid barrier (2.5 - 3 us incl. the bulk-store drain) does not
// shorten compared with a PDL launch boundary.  MMD_CHAIN=1 or mmd_set_option("chain_fwd", 1) turns it on.
static int g_chain_fwd = -1;
void set_chain_fwd(int on) { g_chain_fwd = on ? 1 : 0; }
bool chain_fwd_enabled() {
  if (g_chain_fwd < 0) {
    const char* e = getenv("MMD_CHAIN");
    g_chain_fwd = (e && e[0] == '1') ? 1 : 0;
  }
  return g_chain_fwd == 1;
}

bool chain_fwd_step_usable(const NodeFwdP& node, const NodeFwdP* pre) {
  if (!fwd_v4_usable(node) || node.g.H * node.g.W > 24 * 24) return false;
  const int geom = v4::pick_geom(node.g.H, node.g.W);
  if (geom != 1 && geom != 3 && geom != 4) return false;
  if (node.train && !node.defer_bn) return false;     // the in-kernel finaliser is per launch, not per chain step
  if (pre != nullptr && !fwd_v4_pre_fusable(*pre, node)) return false;
  return true;
}

int launch_chain_fwd(const ChainStepH* steps, int n_steps, int n_nets, int C, cudaStream_t s) {
  MMD_CHECK_ARG(C == 112, "BiFPN kernels are built for C=112 (EfficientDet-D2), got %d", C);
  MMD_CHECK_ARG(n_steps >= 1 && n_steps <= v4::kMaxChainSteps && n_nets >= 1 && n_nets <= kMaxBatchNets,
                "chain_fwd: %d steps, %d networks", n_steps, n_nets);
  static_assert(kMaxChainStepsH == v4::kMaxChainSteps, "host / device chain length");
  unsigned* sync = steps[0].node[0].counter;
  MMD_CHECK_ARG(sync != nullptr, "chain_fwd: the first node carries no counter storage (barrier words)");
  // shared memory: the largest layout any step needs; all CTAs must be co-resident
  size_t smem = 0;
  int max_tiles = 1;
  double bytes = 0.0;
  for (int k = 0; k < n_steps; ++k) {
    const NodeFwdP& p0 = steps[k].node[0];
    const int geom = v4::pick_geom(p0.g.H, p0.g.W);
    size_t need = 0;
    int tiles = 0;
    switch (geom) {
      case 1: need = steps[k].has_pre ? v4::Cfg<12, 8>::kBytesPre : v4::Cfg<12, 8>::kBytes; tiles = p0.g.B * (p0.g.H / 8) * (p0.g.W / 12); break;
      case 3: need = steps[k].has_pre ? v4::Cfg<12, 6>::kBytesPre : v4::Cfg<12, 6>::kBytes; tiles = p0.g.B * (p0.g.H / 6) * (p0.g.W / 12); break;
      case 4: need = steps[k].has_pre ? v4::Cfg<6, 6>::kBytesPre : v4::Cfg<6, 6>::kBytes; tiles = p0.g.B * (p0.g.H / 6) * (p0.g.W / 6); break;
      default: set_error("chain_fwd: step %d has no small-level tile shape (%dx%d)", k, p0.g.H, p0.g.W); return MMD_E_ARG;
    }
    smem = need > smem ? need : smem;
    max_tiles = tiles * n_nets > max_tiles ? tiles * n_nets : max_tiles;
    for (int i = 0; i < n_nets; ++i) {
      const NodeFwdP& p = steps[k].node[i];
      MMD_CHECK_ARG(p.g.H == p0.g.H && p.g.W == p0.g.W && p.g.B == p0.g.B, "chain_fwd: lockstep networks must share the geometry");
      bytes += node_algo_bytes(p.in, steps[k].has_pre ? 1 : p.n_in, p.g, C, 2);
      if (steps[k].has_pre) {
        const NodeFwdP& q = steps[k].pre[i];
        for (int j = 0; j < q.n_in; ++j) bytes += (double)q.g.B * q.in[j].H * q.in[j].W * C * 2.0;
      }
    }
  }
  MMD_SMEM(v4::chain_fwd_kernel, smem);
  int per_sm = 0;
  MMD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, v4::chain_fwd_kernel, kThreads, smem));
  if (per_sm > 2) per_sm = 2;
  MMD_CHECK_ARG(per_sm >= 1, "chain_fwd: the kernel does not fit on an SM (%zu bytes of shared memory)", smem);
  int grid = per_sm * device_sm_count();
  if (grid > max_tiles) grid = max_tiles;
  v4::ChainFwd ch;
  ch.n_steps = n_steps;
  ch.sync = sync;
  ch.dbg = nullptr;
  static int dbg_on = -1;
  static unsigned long long* dbg_buf = nullptr;
  if (dbg_on < 0) {
    const char* e = getenv("MMD_CHAIN_DEBUG");
    dbg_on = (e && e[0] == '1') ? 1 : 0;
    if (dbg_on) cudaMalloc(&dbg_buf, 4 * v4::kMaxChainSteps * sizeof(unsigned long long));
  }
  if (dbg_on && dbg_buf != nullptr) {
    unsigned long long init[4 * v4::kMaxChainSteps];
    for (int k = 0; k < v4::kMaxChainSteps; ++k) { init[4 * k] = ~0ull; init[4 * k + 1] = init[4 * k + 2] = init[4 * k + 3] = 0ull; }
    cudaMemcpyAsync(dbg_buf, init, sizeof(init), cudaMemcpyHostToDevice, s);
    cudaStreamSynchronize(s);
    ch.dbg = dbg_buf;
  }
  for (int k = 0; k < v4::kMaxChainSteps; ++k) {
    const ChainStepH& src = steps[k < n_steps ? k : 0];
    v4::ChainStep& d = ch.step[k];
    NodeFwdBatch tmp;
    for (int i = 0; i < kMaxBatchNets; ++i) {
      d.p[i] = src.node[i < n_nets ? i : 0];
      d.pre[i] = src.pre[i < n_nets ? i : 0];
      tmp.p[i] = d.p[i];
    }
    const NodeFwdP& p0 = src.node[0];
    d.geom = v4::pick_geom(p0.g.H, p0.g.W);
    d.has_pre = src.has_pre;
    const int tiles = (d.geom == 1) ? p0.g.B * (p0.g.H / 8) * (p0.g.W / 12)
                                    : (d.geom == 3 ? p0.g.B * (p0.g.H / 6) * (p0.g.W / 12) : p0.g.B * (p0.g.H / 6) * (p0.g.W / 6));
    batch_shares(tmp, n_nets, grid, tiles, 1.0f);
    for (int i = 0; i <= kMaxBatchNets; ++i) d.cta_begin[i] = tmp.cta_begin[i];
  }
  ProfScope prof(PK_CHAIN_FWD, bytes, s);
  // cooperative launch: the driver guarantees that all CTAs are co-resident (or refuses the launch), also when other
  // streams keep SMs busy; programmatic dependent launch on top when the driver accepts the combination
  static int coop_pdl = -1;   // -1: not probed yet, 1: both attributes, 0: cooperative only
  static int no_coop = -1;
  if (no_coop < 0) {
    const char* e = getenv("MMD_CHAIN_NOCOOP");   // debugging aid: plain (PDL) launch; safe only while nothing else runs
    no_coop = (e && e[0] == '1') ? 1 : 0;
  }
  if (no_coop) {
    MMD_CUDA(launch_pdl(v4::chain_fwd_kernel, dim3(grid), dim3(kThreads), smem, s, ch));
    MMD_LAUNCH_CHECK();
    return 0;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeCooperative;
  attr[0].val.cooperative = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = pdl_take() ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = (coop_pdl == 0) ? 1 : 2;
  cudaError_t e = cudaLaunchKernelEx(&cfg, v4::chain_fwd_kernel, ch);
  if (e != cudaSuccess && cfg.numAttrs == 2 && coop_pdl < 0) {   // the combination is not supported: cooperative only
    cudaGetLastError();
    coop_pdl = 0;
    cfg.numAttrs = 1;
    e = cudaLaunchKernelEx(&cfg, v4::chain_fwd_kernel, ch);
  } else if (e == cudaSuccess && coop_pdl < 0) {
    coop_pdl = 1;
  }
  MMD_CUDA(e);
  MMD_LAUNCH_CHECK();
  if (dbg_on && dbg_buf != nullptr) {
    unsigned long long h[4 * v4::kMaxChainSteps];
    cudaStreamSynchronize(s);
    cudaMemcpy(h, dbg_buf, sizeof(h), cudaMemcpyDeviceToHost);
    fprintf(stderr, "[chain_fwd] grid %d, coop_pdl %d, %d steps:", grid, coop_pdl, n_steps);
    for (int k = 0; k < n_steps; ++k)
      fprintf(stderr, "  [%dx%d%s start +%.1f body %.1f (avg %.1f) barrier %.1f us]", steps[k].node[0].g.H, steps[k].node[0].g.W,
              steps[k].has_pre ? " pre" : "", (double)(h[4 * k] - h[0]) * 1e-3, (double)(h[4 * k + 1] - h[4 * k]) * 1e-3,
              (double)h[4 * k + 3] * 1e-3 / grid, (double)(h[4 * k + 2] - h[4 * k + 1]) * 1e-3);
    fprintf(stderr, "\n");
  }
  return 0;
}

int launch_node_fwd_v4_pre(const NodeFwdP* node, const NodeFwdP* pre, int n, int C, cudaStream_t s) {
  MMD_CHECK_ARG(C == 112, "BiFPN kernels are built for C=112 (EfficientDet-D2), got %d", C);
  MMD_CHECK_ARG(n >= 1 && n <= kMaxBatchNets, "node_fwd_v4_pre: %d networks in one launch", n);
  NodeFwdBatch batch;
  double bytes = 0.0;
  for (int i = 0; i < n; ++i) {
    batch.p[i] = node[i];
    batch.pre[i] = pre[i];
    MMD_CHECK_ARG(node[i].g.H == node[0].g.H && node[i].g.W == node[0].g.W && node[i].g.B == node[0].g.B,
                  "node_fwd_v4_pre: batched networks must share the geometry");
    bytes += node_algo_bytes(node[i].in, 1, node[i].g, C, 2);   // input 0 + output; the pre-pass inputs:
    for (int k = 0; k < pre[i].n_in; ++k) bytes += (double)pre[i].g.B * pre[i].in[k].H * pre[i].in[k].W * C * 2.0;
  }
  for (int i = n; i < kMaxBatchNets; ++i) {
    batch.p[i] = node[0];
    batch.pre[i] = pre[0];
  }
  ProfScope prof(PK_NODE_FWD, bytes, s);
  switch (v4::pick_geom(node[0].g.H, node[0].g.W)) {
    case 1: return v4::launch_geom<12, 8, true>(batch, n, s);
    case 3: return v4::launch_geom<12, 6, true>(batch, n, s);
    case 4: return v4::launch_geom<6, 6, true>(batch, n, s);
  }
  set_error("node_fwd_v4_pre: no tile shape fits %dx%d", node[0].g.H, node[0].g.W);
  return MMD_E_ARG;
}

int launch_poolfuse(const NodeFwdP* p, int n, int C, cudaStream_t s) {
  MMD_CHECK_ARG(C == 112, "BiFPN kernels are built for C=112 (EfficientDet-D2), got %d", C);
  MMD_CHECK_ARG(n >= 1 && n <= kMaxBatchNets, "poolfuse: %d networks in one launch", n);
  NodeFwdBatch batch;
  double bytes = 0.0;
  for (int i = 0; i < n; ++i) {
    batch.p[i] = p[i];
    MMD_CHECK_ARG(p[i].g.H == p[0].g.H && p[i].g.W == p[0].g.W && p[i].g.B == p[0].g.B,
                  "poolfuse: batched networks must share the geometry");
    MMD_CHECK_ARG(p[i].mode[0] == MMD_IN_POOL && (p[i].n_in == 1 || (p[i].n_in == 2 && p[i].mode[1] == MMD_IN_SAME)),
                  "poolfuse: inputs must be (POOL[, SAME])");
    // algorithmic bytes of the node's pooled + third input (each read once at its own resolution)
    for (int k = 0; k < p[i].n_in; ++k) bytes += (double)p[i].g.B * p[i].in[k].H * p[i].in[k].W * C * 2.0;
  }
  for (int i = n; i < kMaxBatchNets; ++i) batch.p[i] = p[0];
  // large levels (P3 -> P4, P4 -> P5): the shared-memory tiled kernel
  static const int no_tiled = getenv("MMD_NO_POOL_TILED") ? 1 : 0;
  bool tiled = !no_tiled && p[0].g.W % v4::kPtCols == 0 && p[0].in[0].H == 2 * p[0].g.H && p[0].in[0].W == 2 * p[0].g.W;
  for (int i = 0; i < n && tiled; ++i)
    tiled = (((uintptr_t)p[i].in[0].data | (uintptr_t)p[i].out | (uintptr_t)p[i].in[1].data | (uintptr_t)p[i].pidx[0] |
              (uintptr_t)p[i].save_d) & 15u) == 0;
  if (tiled) {
    const int items = p[0].g.B * ((p[0].g.H + v4::kPtRows - 1) / v4::kPtRows) * (p[0].g.W / v4::kPtCols);
    static const float tiled_train_w = env_float("MMD_POOL_TILED_TRAIN_SHARE", 2.0f);   // measured: 1.0 -> +0.3 ms, 1.5 .. 2.5 flat
    batch_shares(batch, n, 2 * device_sm_count(), items, tiled_train_w);
    MMD_SMEM(v4::poolfuse_tiled_kernel, v4::kPtSmem);
    ProfScope prof(PK_POOLFUSE, bytes, s);
    MMD_CUDA(launch_pdl(v4::poolfuse_tiled_kernel, dim3(batch.cta_begin[n]), dim3(v4::kPtThreads), v4::kPtSmem, s, batch));
    MMD_LAUNCH_CHECK();
    return 0;
  }
  const int npairs = p[0].g.B * p[0].g.H * ((p[0].g.W + 1) / 2);
  const int gx = (npairs + v4::kPoolLanes - 1) / v4::kPoolLanes;
  // ~2 resident CTAs per SM and 2 waves over all networks; a training network (tagged arg-max search, two extra
  // outputs) costs several times a frozen one (packed bf16 maxima)
  static const float train_w = env_float("MMD_POOL_TRAIN_SHARE", 3.0f);
  static const float waves = env_float("MMD_POOL_WAVES", 2.0f);
  static const int minb = (int)env_float("MMD_POOL_MINB", 4.0f);   // resident CTAs per SM the kernel is compiled for
  batch_shares(batch, n, (int)(148 * minb * waves), gx, train_w);
  ProfScope prof(PK_POOLFUSE, bytes, s);
  if (minb >= 4) MMD_CUDA(launch_pdl(v4::poolfuse_kernel<4>, dim3(batch.cta_begin[n]), dim3(v4::kPoolThreads), 0, s, batch));
  else if (minb == 3) MMD_CUDA(launch_pdl(v4::poolfuse_kernel<3>, dim3(batch.cta_begin[n]), dim3(v4::kPoolThreads), 0, s, batch));
  else MMD_CUDA(launch_pdl(v4::poolfuse_kernel<2>, dim3(batch.cta_begin[n]), dim3(v4::kPoolThreads), 0, s, batch));
  MMD_LAUNCH_CHECK();
  return 0;
}

}  // namespace mmd
