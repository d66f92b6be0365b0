// fp32 mode: CUDA-core (FFMA) contractions with the fused A-softmax epilogues.
//
// One register-tiled kernel template (128x128x8 block tile, 8x8 per thread, register
// prefetch + double-buffered shared memory) instantiated for the four contractions of the
// head; operands are read in place from the reference layouts (X [B,D], W [D,C]) with
// fully predicated loads, so there is no padding or alignment requirement in fp32 mode.
//   FWD  : S = X . W            epilogue: scale by 1/c_j, margin on the target column,
//                               per-row (max, sumexp) partial per column tile (+ logits)
//   BWDG : S recomputed         epilogue: G'' = G' / c_j  (fp32, [B,Cp]; the non-target G'
//                               carries the per-row factor rowgrad = gscale w_i / B) and the column
//                               sums q_j = sum_i G'_ij s_ij per 128-row tile
//   DW   : dWhat'' = X^T . G''  epilogue: dW = dWhat'' - W * q_j / c_j^2
//   DX   : dX partial = G'' . W^T over a K-split of the classes
// This path is exact fp32 (loss within 1e-5 relative of the float64 oracle) and doubles as
// the on-device reference the tcgen05 path is validated against.
#include "asm_common.cuh"
#include "asm_kernels.cuh"

namespace asmh {

namespace {
constexpr int BM = 128, BN = 128, BK = 8;
enum { K_FWD = 0, K_BWDG = 1, K_DW = 2, K_DX = 3 };

__device__ __forceinline__ int sub_index(int t, int a) {   // a in [0,8): two groups of four
  return (a < 4) ? (t * 4 + a) : (64 + t * 4 + (a - 4));
}
}  // namespace

template <int KIND>
__global__ void __launch_bounds__(256) simt_kernel(Step s, int k_per_split) {
  __shared__ __align__(16) float As[2][BK][BM];
  __shared__ __align__(16) float Bs[2][BK][BN];
  __shared__ float red[16][BN];

  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;

  // problem mapping
  int M, N, K;
  if (KIND == K_FWD || KIND == K_BWDG) { M = s.B; N = s.C; K = s.D; }
  else if (KIND == K_DW)               { M = s.D; N = s.C; K = s.B; }
  else                                 { M = s.B; N = s.D; K = s.C; }
  int kbeg = 0, kend = K;
  if (KIND == K_DX) {
    kbeg = blockIdx.z * k_per_split;
    kend = min(K, kbeg + k_per_split);
  }
  const float* G = reinterpret_cast<const float*>(s.G);

  auto loadA = [&](int k0, float (&r)[4]) {
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      const int idx = tid + l * 256;
      float v = 0.f;
      if (KIND == K_DW) {                     // A(d, i) = X[i*D + d]   (m-contiguous)
        const int mm = m0 + (idx & 127), kk = k0 + (idx >> 7);
        if (mm < M && kk < kend) v = __ldg(s.X + (size_t)kk * s.D + mm);
      } else if (KIND == K_DX) {              // A(i, j) = G[i*Cp + j]  (k-contiguous)
        const int mm = m0 + (idx >> 3), kk = k0 + (idx & 7);
        if (mm < M && kk < kend) v = G[(size_t)mm * s.Cp + kk];
      } else {                                // A(i, d) = X[i*D + d]   (k-contiguous)
        const int mm = m0 + (idx >> 3), kk = k0 + (idx & 7);
        if (mm < M && kk < kend) v = __ldg(s.X + (size_t)mm * s.D + kk);
      }
      r[l] = v;
    }
  };
  auto storeA = [&](int buf, const float (&r)[4]) {
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      const int idx = tid + l * 256;
      if (KIND == K_DW) As[buf][idx >> 7][idx & 127] = r[l];
      else              As[buf][idx & 7][idx >> 3] = r[l];
    }
  };
  auto loadB = [&](int k0, float (&r)[4]) {
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      const int idx = tid + l * 256;
      float v = 0.f;
      if (KIND == K_DW) {                     // B(i, j) = G[i*Cp + j]  (n-contiguous)
        const int nn = n0 + (idx & 127), kk = k0 + (idx >> 7);
        if (nn < N && kk < kend) v = G[(size_t)kk * s.Cp + nn];
      } else if (KIND == K_DX) {              // B(j, d) = W[d*C + j]   (k-contiguous)
        const int nn = n0 + (idx >> 3), kk = k0 + (idx & 7);
        if (nn < N && kk < kend) v = __ldg(s.W + (size_t)nn * s.C + kk);
      } else {                                // B(d, j) = W[d*C + j]   (n-contiguous)
        const int nn = n0 + (idx & 127), kk = k0 + (idx >> 7);
        if (nn < N && kk < kend) v = __ldg(s.W + (size_t)kk * s.C + nn);
      }
      r[l] = v;
    }
  };
  auto storeB = [&](int buf, const float (&r)[4]) {
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      const int idx = tid + l * 256;
      if (KIND == K_DX) Bs[buf][idx & 7][idx >> 3] = r[l];
      else              Bs[buf][idx >> 7][idx & 127] = r[l];
    }
  };

  float acc[8][8];
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int b = 0; b < 8; ++b) acc[a][b] = 0.f;

  float ra[4], rb[4];
  const int nk = (kend - kbeg + BK - 1) / BK;
  if (nk > 0) {
    loadA(kbeg, ra);
    loadB(kbeg, rb);
    storeA(0, ra);
    storeB(0, rb);
  }
  __syncthreads();
  int cur = 0;
  for (int kt = 0; kt < nk; ++kt) {
    const bool more = kt + 1 < nk;
    if (more) {
      loadA(kbeg + (kt + 1) * BK, ra);
      loadB(kbeg + (kt + 1) * BK, rb);
    }
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[cur][k][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[cur][k][64 + ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Bs[cur][k][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs[cur][k][64 + tx * 4]);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int a = 0; a < 8; ++a)
#pragma unroll
        for (int b = 0; b < 8; ++b) acc[a][b] = fmaf(av[a], bv[b], acc[a][b]);
    }
    if (more) {
      storeA(cur ^ 1, ra);
      storeB(cur ^ 1, rb);
    }
    __syncthreads();
    cur ^= 1;
  }

  // ------------------------------------------------------------------ epilogues
  if (KIND == K_FWD) {
    float ic[8];
#pragma unroll
    for (int b = 0; b < 8; ++b) {
      const int j = n0 + sub_index(tx, b);
      ic[b] = j < s.C ? s.inv_c[j] : 0.f;
    }
#pragma unroll
    for (int a = 0; a < 8; ++a) {
      const int i = m0 + sub_index(ty, a);
      const bool rv = i < s.B;
      const int yl = rv ? s.ylocal[i] : -1;
      float f[8];
      float mx = -INFINITY;
#pragma unroll
      for (int b = 0; b < 8; ++b) {
        const int j = n0 + sub_index(tx, b);
        float v = acc[a][b] * ic[b];
        if (rv && j == yl) {
          s.tgt_s[i] = v;
          if (s.mg.kind == kMarginAdditive) v = additive_logit(v, s.mg);
          else if (s.mg.kind != kMarginLinear)
            v = target_logit(v, s.n[i], s.inv_n[i], s.m, step_lambda(s.lambda, s.lambda_dev));
          s.tgt_f[i] = v;
        }
        if (j >= s.C) v = -INFINITY;
        f[b] = v;
        mx = fmaxf(mx, v);
      }
      if (rv && s.logits) {
#pragma unroll
        for (int b = 0; b < 8; ++b) {
          const int j = n0 + sub_index(tx, b);
          if (j < s.C) s.logits[(size_t)i * s.C + j] = f[b];
        }
      }
      float z = 0.f;
      if (mx > -INFINITY) {
#pragma unroll
        for (int b = 0; b < 8; ++b) z += __expf(f[b] - mx);
      }
#pragma unroll
      for (int o = 1; o < 16; o <<= 1) {
        const float m2 = __shfl_xor_sync(0xffffffffu, mx, o);
        const float z2 = __shfl_xor_sync(0xffffffffu, z, o);
        ms_combine(mx, z, m2, z2);
      }
      if (rv && tx == 0) s.part[(size_t)i * s.NT + blockIdx.x] = make_float2(mx, z);
    }
  } else if (KIND == K_BWDG) {
    float ic[8], cs[8];
#pragma unroll
    for (int b = 0; b < 8; ++b) {
      const int j = n0 + sub_index(tx, b);
      ic[b] = j < s.C ? s.inv_c[j] : 0.f;
      cs[b] = 0.f;
    }
    float* Gw = reinterpret_cast<float*>(s.G);
#pragma unroll
    for (int a = 0; a < 8; ++a) {
      const int i = m0 + sub_index(ty, a);
      if (i < s.B) {
        const int yl = s.ylocal[i];
        const float lse = s.lse[i];
        const float gt = s.gtarget[i];
        const float gB = s.rowgrad[i];        // invB * gscale * w_i (exactly invB for CE at gscale 1)
#pragma unroll
        for (int b = 0; b < 8; ++b) {
          const int j = n0 + sub_index(tx, b);
          if (j < s.Cp) {
            const float sv = acc[a][b] * ic[b];
            float gp = 0.f;
            if (j < s.C) gp = (j == yl) ? gt : __expf(sv - lse) * gB;
            cs[b] = fmaf(gp, sv, cs[b]);
            Gw[(size_t)i * s.Cp + j] = gp * ic[b];
          }
        }
      }
    }
#pragma unroll
    for (int b = 0; b < 8; ++b) red[ty][sub_index(tx, b)] = cs[b];
    __syncthreads();
    if (tid < BN) {
      float q = 0.f;
#pragma unroll
      for (int r = 0; r < 16; ++r) q += red[r][tid];
      const int j = n0 + tid;
      if (j < s.Cp) s.q_part[(size_t)blockIdx.y * s.Cp + j] = q;
    }
  } else if (KIND == K_DW) {
#pragma unroll
    for (int b = 0; b < 8; ++b) {
      const int j = n0 + sub_index(tx, b);
      if (j >= s.C) continue;
      float q = 0.f;
      for (int t = 0; t < s.MT; ++t) q += s.q_part[(size_t)t * s.Cp + j];
      const float ic = s.wcorr[j];
      const float coef = q * ic * ic;
#pragma unroll
      for (int a = 0; a < 8; ++a) {
        const int d = m0 + sub_index(ty, a);
        if (d < s.D) {
          const size_t o = (size_t)d * s.C + j;
          if (s.opt.kind == 0) {
            s.dW[o] = acc[a][b] - __ldg(s.W + o) * (coef - s.wd_g);
          } else {                              // fused optimizer: W updated in place
            float w = s.Wmut[o], s0 = s.opt_s0[o], s1 = s.opt.kind == 2 ? s.opt_s1[o] : 0.f;
            opt_apply(s.opt, acc[a][b] - w * coef, w, s0, s1);
            s.Wmut[o] = w;
            s.opt_s0[o] = s0;
            if (s.opt.kind == 2) s.opt_s1[o] = s1;
          }
        }
      }
    }
  } else {
    float* out = s.dx_part + (size_t)blockIdx.z * s.B * s.D;
#pragma unroll
    for (int a = 0; a < 8; ++a) {
      const int i = m0 + sub_index(ty, a);
      if (i >= s.B) continue;
#pragma unroll
      for (int b = 0; b < 8; ++b) {
        const int d = n0 + sub_index(tx, b);
        if (d < s.D) out[(size_t)i * s.D + d] = acc[a][b];
      }
    }
  }
}

int simt_forward_tiles(int C) { return (C + BN - 1) / BN; }

int simt_dx_splits(int B, int D, int Cp) {
  const int tiles = ((B + BM - 1) / BM) * ((D + BN - 1) / BN);
  int ks = (2 * 148 + tiles - 1) / tiles;
  const int maxks = (Cp + 255) / 256;
  if (ks > maxks) ks = maxks;
  if (ks < 1) ks = 1;
  if (ks > 64) ks = 64;
  return ks;
}

void launch_simt_forward(const Step& s, cudaStream_t st) {
  dim3 grd((s.C + BN - 1) / BN, (s.B + BM - 1) / BM);
  simt_kernel<K_FWD><<<grd, 256, 0, st>>>(s, 0);
}

void launch_simt_bwdg(const Step& s, cudaStream_t st) {
  dim3 g1((s.Cp + BN - 1) / BN, (s.B + BM - 1) / BM);
  simt_kernel<K_BWDG><<<g1, 256, 0, st>>>(s, 0);
}

void launch_simt_dw(const Step& s, cudaStream_t st) {
  dim3 g2((s.C + BN - 1) / BN, (s.D + BM - 1) / BM);
  simt_kernel<K_DW><<<g2, 256, 0, st>>>(s, 0);
}

void launch_simt_dx(const Step& s, cudaStream_t st) {
  int kper = (s.C + s.KS - 1) / s.KS;
  kper = (kper + BK - 1) / BK * BK;
  dim3 g3((s.D + BN - 1) / BN, (s.B + BM - 1) / BM, s.KS);
  simt_kernel<K_DX><<<g3, 256, 0, st>>>(s, kper);
}

void simt_preload_kernels() {
  cudaFuncAttributes a;
  cudaFuncGetAttributes(&a, simt_kernel<K_FWD>);
  cudaFuncGetAttributes(&a, simt_kernel<K_BWDG>);
  cudaFuncGetAttributes(&a, simt_kernel<K_DW>);
  cudaFuncGetAttributes(&a, simt_kernel<K_DX>);
}

}  // namespace asmh
