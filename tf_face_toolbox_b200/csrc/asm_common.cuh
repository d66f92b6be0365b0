// Shared device helpers for the A-softmax head kernels (sm_100a).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

namespace asmh {

constexpr int kRowTile = 128;      // batch-row tile used for the q_part column-sum partials

// ---------------------------------------------------------------------------------------
// psi(theta) = (-1)^k cos(m theta) - 2k on the target column (SURVEY.md 8a, row a1').
// k is found by comparing t = cos(theta) against cos(l*pi/m), l = 1..m-1 (no acosf).
// Returns psi and d(psi)/dt; k / sign are piecewise constants.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void psi_eval(float t, int m, float& psi, float& dpsi) {
  t = fminf(1.0f, fmaxf(-1.0f, t));
  float T, dT;
  int k = 0;
  const float t2 = t * t;
  if (m == 4) {
    T = fmaf(8.0f * t2, t2 - 1.0f, 1.0f);            // 8t^4 - 8t^2 + 1
    dT = t * fmaf(32.0f, t2, -16.0f);                // 32t^3 - 16t
    k = (t <= 0.70710678118654752f) + (t <= 0.0f) + (t <= -0.70710678118654752f);
  } else if (m == 3) {
    T = t * fmaf(4.0f, t2, -3.0f);
    dT = fmaf(12.0f, t2, -3.0f);
    k = (t <= 0.5f) + (t <= -0.5f);
  } else if (m == 2) {
    T = fmaf(2.0f, t2, -1.0f);
    dT = 4.0f * t;
    k = (t <= 0.0f);
  } else {
    T = t;
    dT = 1.0f;
  }
  const float sgn = (k & 1) ? -1.0f : 1.0f;
  psi = fmaf(sgn, T, -2.0f * (float)k);
  dpsi = sgn * dT;
}

// ---------------------------------------------------------------------------------------
// Additive margin on L2-normalised embeddings (asm_set_margin, DESIGN.md section 2.1).  The
// GEMMs then see s * x_i / n_i, so a raw logit is s * cos(theta) and t = logit / s.
//   t >= tau = cos(pi - m2):  phi = cos(theta + m2) - m3,  phi' = cos m2 + t sin m2 / sin(theta)
//   otherwise:                phi = t - m2 sin m2 - m3,    phi' = 1
// (the usual non-"easy-margin" fallback; phi jumps at tau).  kind == 0: A-softmax instead;
// kind == 3: the plain linear classifier f_ij = x_i.w_j (DESIGN.md section 2.3), no margin at all.
// ---------------------------------------------------------------------------------------
constexpr int kMarginAdditive = 1;
constexpr int kMarginLinear = 3;
struct Margin {
  int kind;                  // 0 = A-softmax (psi, lambda), 1 = additive (s, m2, m3), 3 = linear
  float s, inv_s;            // scale and 1/s
  float cm, sm;              // cos m2, sin m2
  float tau;                 // cos(pi - m2)
  float fb;                  // m2 sin m2 + m3: offset of the fallback branch
  float m3;
};

__device__ __forceinline__ void phi_eval(float t, const Margin& g, float& phi, float& dphi) {
  t = fminf(1.0f, fmaxf(-1.0f, t));
  if (t >= g.tau) {
    const float st = sqrtf(fmaxf(1.0f - t * t, 1e-12f));
    phi = t * g.cm - st * g.sm - g.m3;
    dphi = g.cm + t * g.sm / st;
  } else {
    phi = t - g.fb;
    dphi = 1.0f;
  }
}

// The norm kernel copies the step's Margin into the workspace slot of kMarginRecordFloats floats
// that directly precedes tgt_s (asm_api.cu, make_layout), where the forward GEMM's out-of-line
// target patch finds it without an argument of its own.
constexpr int kMarginRecordFloats = 64;
static_assert(sizeof(Margin) <= kMarginRecordFloats * sizeof(float), "margin record slot");
__device__ __forceinline__ const Margin* margin_record(const float* tgt_s) {
  return reinterpret_cast<const Margin*>(tgt_s - kMarginRecordFloats);
}

// f_{i,y} = s * phi(s_y / s)
__device__ __forceinline__ float additive_logit(float sv, const Margin& g) {
  float phi, dphi;
  phi_eval(sv * g.inv_s, g, phi, dphi);
  return g.s * phi;
}

// f_{i,y} = (lambda * s + n * psi(s/n)) / (1 + lambda)
__device__ __forceinline__ float target_logit(float s, float n, float inv_n, int m, float lambda) {
  float psi, dpsi;
  psi_eval(s * inv_n, m, psi, dpsi);
  return (lambda * s + n * psi) / (1.0f + lambda);
}

// lambda of this step: a by-value kernel argument, or (for CUDA-graph replay, where kernel
// arguments are frozen) a device scalar the host updates between replays
__device__ __forceinline__ float step_lambda(float by_value, const float* dev) {
  return dev ? __ldg(dev) : by_value;
}

// Programmatic dependent launch (PDL).  pdl_trigger(): the next kernel in the stream may
// start launching (its CTAs become resident as SMs free up and run their prologue).
// pdl_wait(): blocks until the previous kernel has completed and its writes are visible --
// required before touching anything a predecessor produced.  Both are no-ops for a kernel
// that was launched without the programmatic-serialization attribute.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// Online-softmax pair combine: (m, z) <- (m, z) (+) (m2, z2)
__device__ __forceinline__ void ms_combine(float& m, float& z, float m2, float z2) {
  const float mn = fmaxf(m, m2);
  if (mn == -INFINITY) { m = mn; z = 0.f; return; }
  z = z * __expf(m - mn) + z2 * __expf(m2 - mn);
  m = mn;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace asmh
