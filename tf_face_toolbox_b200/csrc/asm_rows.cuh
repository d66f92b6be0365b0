// Per-row pieces shared by the single-shard kernels (asm_prep.cu) and the kernels that fold the
// NVLink exchange into them (asm_p2p.cu).
#pragma once
#include "asm_common.cuh"
#include "asm_kernels.cuh"

namespace asmh {

// One lane per row, after the row's global (max M, sum-exp Z, target logit f_y) are known:
//   lse = M + log Z, loss_i = lse - f_y, the exp2 offset of the backward, and the target-column
//   gradient coefficients
//   g_y = (e^{f_y - lse} - 1)/B,  G'_y = g_y (lambda + psi')/(1 + lambda),
//   r   = g_y (psi - t psi') / ((1 + lambda) n)            (SURVEY.md 8a, row a3)
// or, for the additive margin, G'_y = g_y phi'(t) with t = s_y / s, and r = 0 (the projection of
// dx_finish_rows_margin replaces the r_i x_i term).
// A row whose label lies outside [0, C_total) (ylocal == -2) has no defined loss: it gets NaN,
// as the reference's sparse_softmax_cross_entropy does on the GPU (nets/sphere.py:109).
//
// Focal loss (s.ls.kind == 1, DESIGN.md section 2.2): with ce = lse - f_y, p = e^{-ce}, u = 1 - p,
//   loss_i = gamma u^alpha ce,   d loss_i / d f_ij = w_i (softmax_ij - delta_{j,y_i}),
//   w_i = gamma (u^alpha + alpha p (ce / u) u^alpha)        (ce / u := 1 at u == 0)
// so the row's whole gradient is the cross-entropy one times w_i: log2 w_i joins the exp2 offset,
// G'_y and r are multiplied by it.  w_i depends only on the global (M, Z, f_y), so every class
// shard computes the same value.  w_i = 0 (ce == 0, alpha > 0) gives negoff = -inf, which the
// recompute kernels turn into exp2(-inf) = 0.
__device__ __forceinline__ void focal_row(const LossParams& ls, float ce, float& w, float& loss) {
  const float c = fmaxf(ce, 0.f);                // rounding can leave lse a hair below f_y
  const float p = expf(-c);
  const float u = -expm1f(-c);                   // 1 - p without cancellation
  const float ua = powf(u, ls.alpha);            // powf(u, 0) == 1: alpha = 0 gives w = gamma exactly
  const float cu = u > 0.f ? c / u : 1.0f;
  w = ls.gamma * (ua + ls.alpha * p * cu * ua);
  loss = ls.gamma * ua * ce;
}

__device__ __forceinline__ void row_epilogue(const Step& s, int row, float m, float z, float fy,
                                             int yl_row, float tgt_f_row, float tgt_s_row,
                                             float inv_n_row) {
  const bool owned = yl_row >= 0;
  const float lse = m + logf(z);
  s.lse[row] = lse;
  const float gB = s.invB * s.gscale;            // every gradient carries 1/B and the caller's scale
  float negoff = -lse * 1.4426950408889634f + log2f(gB);
  float loss = lse - fy, w = 1.0f;
  const bool focal = s.ls.kind != 0;
  if (focal) {
    focal_row(s.ls, loss, w, loss);
    negoff += log2f(w);
  }
  s.negoff[row] = negoff;
  s.rowgrad[row] = focal ? gB * w : gB;
  s.rowloss[row] = yl_row == -2 ? __int_as_float(0x7fc00000) : loss;
  float gt = 0.f, r = 0.f;
  if (owned && s.mg.kind != 0) {                 // additive: G'_y = g_y phi'(t), r = 0
    float phi, dphi;
    phi_eval(tgt_s_row * s.mg.inv_s, s.mg, phi, dphi);
    gt = (expf(tgt_f_row - lse) - 1.0f) * gB * dphi;
  } else if (owned) {
    float psi, dpsi;
    const float t = fminf(1.f, fmaxf(-1.f, tgt_s_row * inv_n_row));
    psi_eval(t, s.m, psi, dpsi);
    const float gy = (expf(tgt_f_row - lse) - 1.0f) * gB;
    const float lam = step_lambda(s.lambda, s.lambda_dev);
    const float il = 1.0f / (1.0f + lam);
    gt = gy * (lam + dpsi) * il;
    r = gy * (psi - t * dpsi) * il * inv_n_row;
  }
  if (focal) {
    gt *= w;
    r *= w;
  }
  s.gtarget[row] = gt;
  s.rcoef[row] = r;
}

// dX = sum_z dx_part[z] + r_i * x_i for the float4 elements  vb*nt + t, stepping by nb*nt
// (float4 along D; D % 4 == 0).  KS_T > 0: all KS_T partial loads are issued before the first
// add (one memory round trip); KS_T == 0: generic loop in batches of four.  Summation order
// z = 0..KS-1 either way.
// Four elements  4i .. 4i+3  of the step's embeddings X [B, D] (fp32, or bf16 when x_bf16).
__device__ __forceinline__ float4 load_x4(const Step& s, size_t i) {
  if (s.x_bf16) {                                   // embeddings handed over as bf16
    const uint2 h = __ldg(reinterpret_cast<const uint2*>(s.X) + i);
    const __nv_bfloat162 a2 = *reinterpret_cast<const __nv_bfloat162*>(&h.x);
    const __nv_bfloat162 b2 = *reinterpret_cast<const __nv_bfloat162*>(&h.y);
    return make_float4(__low2float(a2), __high2float(a2), __low2float(b2), __high2float(b2));
  }
  return __ldg(reinterpret_cast<const float4*>(s.X) + i);
}

template <int KS_T>
__device__ __forceinline__ void dx_finish_rows(const Step& s, float* dxo, unsigned vb, unsigned nb) {
  const size_t total4 = (size_t)s.B * s.D / 4;
  const size_t stride4 = total4;
  for (size_t i = vb * (size_t)blockDim.x + threadIdx.x; i < total4; i += (size_t)nb * blockDim.x) {
    const int row = (int)((i * 4) / s.D);
    const float4* p = reinterpret_cast<const float4*>(s.dx_part) + i;
    const float r = s.rcoef[row];
    const float4 x = load_x4(s, i);
    float4 a = make_float4(r * x.x, r * x.y, r * x.z, r * x.w);
    if (KS_T > 0) {
      float4 v[KS_T > 0 ? KS_T : 1];
#pragma unroll
      for (int z = 0; z < KS_T; ++z) v[z] = __ldcg(p + (size_t)z * stride4);
#pragma unroll
      for (int z = 0; z < KS_T; ++z) { a.x += v[z].x; a.y += v[z].y; a.z += v[z].z; a.w += v[z].w; }
    } else {
      int z = 0;
      for (; z + 4 <= s.KS; z += 4) {
        const float4 v0 = __ldcg(p + (size_t)(z + 0) * stride4);
        const float4 v1 = __ldcg(p + (size_t)(z + 1) * stride4);
        const float4 v2 = __ldcg(p + (size_t)(z + 2) * stride4);
        const float4 v3 = __ldcg(p + (size_t)(z + 3) * stride4);
        a.x += v0.x; a.y += v0.y; a.z += v0.z; a.w += v0.w;
        a.x += v1.x; a.y += v1.y; a.z += v1.z; a.w += v1.w;
        a.x += v2.x; a.y += v2.y; a.z += v2.z; a.w += v2.w;
        a.x += v3.x; a.y += v3.y; a.z += v3.z; a.w += v3.w;
      }
      for (; z < s.KS; ++z) {
        const float4 v = __ldcg(p + (size_t)z * stride4);
        a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
      }
    }
    reinterpret_cast<float4*>(dxo)[i] = a;
  }
}

// Additive margin, row by row (256 threads: 128 per row, two rows per block and trip, rows
// 2vb, 2vb+1, then 2(vb+nb), ...):  v_i = sum_z dx_part[z][i] (z = 0..KS-1 in order), then
//   dX_i = (s/n_i) (v_i - (x_i.v_i)/n_i^2 x_i)
// the gradient through x_i -> s x_i/n_i.  Up to four float4 per thread (D <= 2048) stay in
// registers between the dot product and the projection; beyond that v goes through dxo.
// `red` is [8] floats of shared memory.  The projection is linear in v, so a class shard can
// project its own partial sum (dx_finish_margin_p2p_kernel).
__device__ __forceinline__ void dx_finish_rows_margin(const Step& s, float* dxo, unsigned vb, unsigned nb,
                                                      float* red) {
  const int half = threadIdx.x >> 7, t = threadIdx.x & 127, w = threadIdx.x >> 5;
  const int d4 = s.D / 4;
  const size_t stride4 = (size_t)s.B * s.D / 4;
  auto vsum = [&](size_t i) {
    const float4* p = reinterpret_cast<const float4*>(s.dx_part) + i;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    int z = 0;
    for (; z + 4 <= s.KS; z += 4) {
      const float4 v0 = __ldcg(p + (size_t)(z + 0) * stride4);
      const float4 v1 = __ldcg(p + (size_t)(z + 1) * stride4);
      const float4 v2 = __ldcg(p + (size_t)(z + 2) * stride4);
      const float4 v3 = __ldcg(p + (size_t)(z + 3) * stride4);
      a.x += v0.x; a.y += v0.y; a.z += v0.z; a.w += v0.w;
      a.x += v1.x; a.y += v1.y; a.z += v1.z; a.w += v1.w;
      a.x += v2.x; a.y += v2.y; a.z += v2.z; a.w += v2.w;
      a.x += v3.x; a.y += v3.y; a.z += v3.z; a.w += v3.w;
    }
    for (; z < s.KS; ++z) {
      const float4 v = __ldcg(p + (size_t)z * stride4);
      a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
    }
    return a;
  };
  for (int r0 = 2 * (int)vb; r0 < s.B; r0 += 2 * (int)nb) {     // same trip count in the whole block
    const int row = r0 + half;
    const bool rv = row < s.B;
    const size_t base = (size_t)row * d4;
    float4 keep[4];
    float dot = 0.f;
    if (rv) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int k = t + 128 * u;
        if (k < d4) {
          keep[u] = vsum(base + k);
          const float4 x = load_x4(s, base + k);
          dot += x.x * keep[u].x + x.y * keep[u].y + x.z * keep[u].z + x.w * keep[u].w;
        }
      }
      for (int k = t + 512; k < d4; k += 128) {
        const float4 a = vsum(base + k);
        const float4 x = load_x4(s, base + k);
        dot += x.x * a.x + x.y * a.y + x.z * a.z + x.w * a.w;
        reinterpret_cast<float4*>(dxo)[base + k] = a;
      }
    }
    dot = warp_sum(dot);
    if ((threadIdx.x & 31) == 0) red[w] = dot;
    __syncthreads();
    dot = (red[4 * half] + red[4 * half + 1]) + (red[4 * half + 2] + red[4 * half + 3]);
    __syncthreads();                                             // red is reused by the next trip
    if (!rv) continue;
    const float in = s.inv_n[row];
    const float av = s.mg.s * in;                                // s / n
    const float ax = -av * dot * in * in;                        // -(s/n) (x.v) / n^2
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int k = t + 128 * u;
      if (k < d4) {
        const float4 x = load_x4(s, base + k);
        const float4 v = keep[u];
        reinterpret_cast<float4*>(dxo)[base + k] =
            make_float4(fmaf(av, v.x, ax * x.x), fmaf(av, v.y, ax * x.y), fmaf(av, v.z, ax * x.z),
                        fmaf(av, v.w, ax * x.w));
      }
    }
    for (int k = t + 512; k < d4; k += 128) {                    // this thread wrote v there itself
      const float4 x = load_x4(s, base + k);
      const float4 v = reinterpret_cast<const float4*>(dxo)[base + k];
      reinterpret_cast<float4*>(dxo)[base + k] =
          make_float4(fmaf(av, v.x, ax * x.x), fmaf(av, v.y, ax * x.y), fmaf(av, v.z, ax * x.z),
                      fmaf(av, v.w, ax * x.w));
    }
  }
}

// Fixed-order mean of the per-row losses by the last block of a grid to get here (deterministic).
__device__ __forceinline__ void last_block_loss(const Step& s, float* red /* [256] shared */, bool* is_last) {
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) *is_last = (atomicAdd(s.counter, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!*is_last) return;
  __threadfence();
  float acc = 0.f;
  for (int i = threadIdx.x; i < s.B; i += 256) acc += __ldcg(s.rowloss + i);
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    if (s.loss) *s.loss = red[0] * s.invB;
    *s.counter = 0u;
  }
}

}  // namespace asmh
