// Device helpers shared by the backward kernels: gradient gather ("pull"), consumer weights, BatchNorm-backward
// coefficients.  See bifpn_bwd.cu for the formulation.
#pragma once
#include "bifpn.cuh"

namespace mmd {

// ---- gradient gather ----------------------------------------------------------------------------------------
template <typename T, int C>
__device__ __forceinline__ float4 pull_grad(const NodeBwdP& P, const float (&cw)[3], int b, int y, int x, int q) {
  float4 G = f4_zero();
  const int H = P.g.H, W = P.g.W;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    if (c >= P.n_cons) break;
    const ConsP& cs = P.cons[c];
    const T* du = reinterpret_cast<const T*>(cs.du);
    if (cs.mode == MMD_CONS_SAME) {
      G = f4_axpy(cw[c], ld4<T>(du + (((long long)b * cs.H + y) * cs.W + x) * C + 4 * q), G);
    } else if (cs.mode == MMD_CONS_UP2) {
      float4 s = f4_zero();
#pragma unroll
      for (int dy = 0; dy < 2; ++dy)
#pragma unroll
        for (int dx = 0; dx < 2; ++dx) {
          const int fy = 2 * y + dy, fx = 2 * x + dx;
          if (fy < cs.H && fx < cs.W) s = f4_add(s, ld4<T>(du + (((long long)b * cs.H + fy) * cs.W + fx) * C + 4 * q));
        }
      G = f4_axpy(cw[c], s, G);
    } else {
      const int top = pool_pad_before(H), left = pool_pad_before(W);
#pragma unroll
      for (int wy = 0; wy < 3; ++wy) {
        const int ny = y + top - wy;
        if (ny < 0 || (ny & 1)) continue;
        const int i = ny >> 1;
        if (i >= cs.H) continue;
#pragma unroll
        for (int wx = 0; wx < 3; ++wx) {
          const int nx = x + left - wx;
          if (nx < 0 || (nx & 1)) continue;
          const int j = nx >> 1;
          if (j >= cs.W) continue;
          const long long off = (((long long)b * cs.H + i) * cs.W + j) * C + 4 * q;
          const unsigned packed = *reinterpret_cast<const unsigned*>(cs.pidx + off);
          const float4 g = ld4<T>(du + off);
          const unsigned id = (unsigned)(wy * 3 + wx);
          if ((packed & 0xffu) == id) G.x = fmaf(cw[c], g.x, G.x);
          if (((packed >> 8) & 0xffu) == id) G.y = fmaf(cw[c], g.y, G.y);
          if (((packed >> 16) & 0xffu) == id) G.z = fmaf(cw[c], g.z, G.z);
          if (((packed >> 24) & 0xffu) == id) G.w = fmaf(cw[c], g.w, G.w);
        }
      }
    }
  }
  return G;
}

__device__ __forceinline__ void cons_weights(const NodeBwdP& P, float (&cw)[3]) {
#pragma unroll
  for (int c = 0; c < 3; ++c)
    cw[c] = (c < P.n_cons) ? fusion_weight(P.cons[c].fw, P.cons[c].fw_n, P.cons[c].fw_k, P.cons[c].fw_eps) : 0.f;
}

// BN backward coefficients per channel: dL/dx_raw = A*G + Bc*x_raw + Cc  (SURVEY.md A.3), from the consumers' slots.
// A frozen BatchNorm (eval-mode layer in a training forward) normalised with constants: A = gamma*invstd_r, Bc = Cc = 0;
// the slots still give dL/dbeta = S1 and dL/dgamma = S2 (their xhat is taken against the running statistics of out_bn).
template <int C>
__device__ __forceinline__ void bn_bwd_coefs(const NodeBwdP& P, const float (&cw)[3], float* s_coef) {
  const int tid = threadIdx.x;
  if (tid < C) {
    double S1 = 0.0, S2 = 0.0;
    for (int c = 0; c < P.n_cons; ++c) {
      S1 += (double)cw[c] * P.cons[c].slot[tid];
      S2 += (double)cw[c] * P.cons[c].slot[C + tid];
    }
    const double n = (double)P.g.B * P.g.H * P.g.W;
    const float gamma = P.bn_w[tid], mean = P.out_bn[2 * C + tid], invstd = P.out_bn[3 * C + tid];
    const float A = gamma * invstd;
    const float Bc = P.frozen_bn ? 0.f : (float)(-(double)gamma * invstd * invstd * S2 / n);
    const float Cc = P.frozen_bn ? 0.f : (float)(-(double)A * S1 / n - (double)Bc * mean);
    s_coef[tid] = A;
    s_coef[C + tid] = Bc;
    s_coef[2 * C + tid] = Cc;
    if (blockIdx.x == 0 && blockIdx.y == 0) {
      if (P.g_bn_w) P.g_bn_w[tid] = (float)S2;
      if (P.g_bn_b) P.g_bn_b[tid] = (float)S1;
    }
  }
}

}  // namespace mmd
