// HBM-bound kernels of the A-softmax head: norms (+ bf16 operand copies), stats combine,
// dX finish.  See DESIGN.md "Kernels" for the per-kernel roofline and algorithmic bytes.
#include <stdlib.h>

#include "asm_common.cuh"
#include "asm_kernels.cuh"
#include "asm_p2p.cuh"
#include "asm_rows.cuh"

namespace asmh {

// ---------------------------------------------------------------------------------------
// prep: one launch, two roles (block = TX column pairs x TY row groups).
//   blocks [0, nwb): W role. Block (32 x 8) owns 64 columns; thread (tx, ty) owns the column
//     pair 2*(blk*32+tx) and the rows ty, ty+8, ...  Loads are coalesced along C (a warp
//     reads 256 contiguous bytes per row), the bf16 copy is written with the same mapping
//     (128 B per warp per row) into the padded pitch Cp, and the 8 row groups are reduced
//     through shared memory into inv_c[j] = 1/||w_j||.  W is read exactly once.
//   blocks [nwb, ...): X role. One warp per embedding row: n_i, 1/n_i, bf16 copy, and the
//     label -> local-class-index translation with the range check.
// With the NVLink transport (p.world > 1) the launch starts with npub PUBLISH blocks that copy
// this rank's rows into its symmetric block and raise its phase-0 flag on every peer, and the X
// role reads each row from the symmetric block of the rank that owns it (waiting for that
// rank's flag) while it normalises it -- the all-gather of X costs no launch of its own, and
// the W role, which depends on nobody, runs meanwhile.  Publish blocks come first in the grid
// so that they are dispatched before any block that waits for a peer.
// ---------------------------------------------------------------------------------------
// Per-row results of the X role (lane 0 of the row's warp): norm, 1/norm, local label.
__device__ __forceinline__ void prep_row_tail(const Step& s, int row, float acc, long long y) {
  const float nn = sqrtf(acc);
  s.n[row] = nn;
  s.inv_n[row] = nn > 0.f ? 1.0f / nn : 0.f;
  // -1: owned by another shard; -2: outside [0, C_total) (reported by asm_check_labels, and
  // the row's loss becomes NaN; both mean "no target column here" to the GEMM kernels, so a
  // bad label never faults)
  const long long yl = y - s.class_offset;
  s.ylocal[row] = (y < 0 || y >= s.C_total) ? -2 : ((yl >= 0 && yl < s.C) ? (int)yl : -1);
  s.tgt_s[row] = 0.f;
  s.tgt_f[row] = 0.f;
}

// X role for the additive margin (one warp per row): the operand copies hold fl(x * (s/n)), so
// n must be known before the first plane is written.  Pass 1 reads the row (and, on the NVLink
// path, stores the gathered copy Xg) and reduces |x|^2; pass 2 writes the PL bf16 planes of the
// scaled row, or with PL == 0 (CUDA-core fp32 path) the fp32 copy Xs.  A row of up to 128
// 16-byte pieces (D <= 512 fp32, D <= 1024 bf16) stays in registers; a longer one is read again
// (from Xg on the NVLink path: this lane wrote those pieces itself).  n / inv_n stay the true norm.
template <int PL>
__device__ __forceinline__ void prep_row_scaled(const Step& s, const char* x, char* xg, int esz, bool gather,
                                                int row, long long y) {
  const int tx = threadIdx.x & 31;
  const float4* x4 = reinterpret_cast<const float4*>(x);
  const int n16 = s.D * esz / 16;
  const int epp = 16 / esz;
  auto sq16 = [&](const float4& v) {
    if (esz == 2) {
      const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&v);
      float a = 0.f;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float l = __low2float(h2[q]), h = __high2float(h2[q]);
        a = fmaf(l, l, a);
        a = fmaf(h, h, a);
      }
      return a;
    }
    return fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, v.w * v.w)));
  };
  float4 v[4];
  float acc = 0.f;
  for (int i0 = 0; i0 < n16; i0 += 128) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * 32 + tx;
      v[u] = i < n16 ? (gather ? __ldcv(x4 + i) : __ldg(x4 + i)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * 32 + tx;
      if (i < n16) {
        if (gather) reinterpret_cast<float4*>(xg)[i] = v[u];
        acc += sq16(v[u]);
      }
    }
  }
  acc = warp_sum(acc);
  const float nn = sqrtf(acc);
  const float sc = nn > 0.f ? s.mg.s / nn : 0.f;
  auto put = [&](int d, float e) {
    const float u = e * sc;
    if (PL > 0) {
      __nv_bfloat16* dst = s.Xb + (size_t)row * PL * s.D + d;
      float r = u;
#pragma unroll
      for (int p2 = 0; p2 < PL; ++p2) {
        const __nv_bfloat16 hv = __float2bfloat16_rn(r);
        dst[(size_t)p2 * s.D] = hv;
        r -= __bfloat162float(hv);
      }
    } else {
      s.Xs[(size_t)row * s.D + d] = u;
    }
  };
  auto put16 = [&](int e0, const float4& w) {
    if (esz == 2) {
      const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&w);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        put(e0 + 2 * q, __low2float(h2[q]));
        put(e0 + 2 * q + 1, __high2float(h2[q]));
      }
    } else {
      put(e0, w.x); put(e0 + 1, w.y); put(e0 + 2, w.z); put(e0 + 3, w.w);
    }
  };
  const float4* again = gather ? reinterpret_cast<const float4*>(xg) : x4;
  for (int i0 = 0; i0 < n16; i0 += 128) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * 32 + tx;
      if (i < n16) put16(i * epp, n16 <= 128 ? v[u] : again[i]);
    }
  }
  if (tx == 0) prep_row_tail(s, row, acc, y);
}

// vblock: the block index this call plays (blockIdx.x).  ADD: the additive-margin X role
// (prep_row_scaled), a separate instantiation so that it costs the A-softmax kernels no registers.
template <bool VEC2, int PL, int TX, int TY, int U, bool ADD>
__device__ __forceinline__ void prep_block(const Step& s, const void* labels, int label_bytes,
                                           int nwb, int npub, const P2P& p, const int vblock,
                                           float (*red)[2 * TX]) {
  static_assert(TX * TY == 256, "256 threads");
  const int tid = threadIdx.x;
  if (vblock < npub) {
    const unsigned cur = p2p_current_step(p);
    float4* xs = reinterpret_cast<float4*>(p.x(p.rank, cur & 1));
    int* ys = p.y(p.rank, cur & 1);
    const size_t n4 = (size_t)p.b_local * p.D * (s.x_bf16 ? 2 : 4) / 16;     // 16-byte pieces of my rows
    for (size_t i = vblock * (size_t)256 + tid; i < n4; i += (size_t)npub * 256)
      xs[i] = __ldg(reinterpret_cast<const float4*>(p.x_local) + i);
    for (int i = vblock * 256 + tid; i < p.b_local; i += npub * 256)
      ys[i] = p.y_bytes == 8 ? (int)reinterpret_cast<const long long*>(p.y_local)[i]
                             : reinterpret_cast<const int*>(p.y_local)[i];
    if (block_ticket(p.tickets + 0, (unsigned)npub) == (unsigned)npub - 1 && tid == 0)
      p2p_publish(p, 0, cur);
    return;
  }
  const int bid = vblock - npub;
  if (bid < nwb) {
    const int tx = tid % TX, ty = tid / TX;
    const int j0 = (bid * TX + tx) * 2;
    float a0 = 0.f, a1 = 0.f;
    if (j0 < s.Cp) {
      const bool v0 = j0 < s.C, v1 = j0 + 1 < s.C;
      const float* w = s.W + j0;
      constexpr bool BF16 = PL > 0;                 // PL: bf16 planes written (0, 1 or 3)
      // bf16 copy, COLUMN-BLOCKED [plane][Cp/64][D][64]: the GEMM kernels' 64-class TMA boxes are
      // contiguous in memory (asm_umma_gemm.cu, wb_row)
      __nv_bfloat16* wb = BF16 ? s.Wb + (size_t)(j0 >> 6) * s.D * 64 + (j0 & 63) : nullptr;
      const size_t plane = (size_t)s.D * s.Cp;
      // U rows per trip: all loads are issued before the first use so that U x 8 B per
      // thread are in flight (the bf16 stores would otherwise serialise the loads).
      for (int d0 = ty; d0 < s.D; d0 += TY * U) {
        float x0[U], x1[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int d = d0 + TY * u;
          x0[u] = 0.f; x1[u] = 0.f;
          if (d < s.D) {
            if (VEC2) {
              if (v1) {
                // the fp32 master weights are read once per step: evict-first keeps the bf16
                // copy written below (what the GEMM kernels read next) resident in L2 instead
                const float2* wp = reinterpret_cast<const float2*>(w + (size_t)d * s.C);
                const float2 v = s.l2_hints ? __ldcs(wp) : __ldg(wp);
                x0[u] = v.x; x1[u] = v.y;
              } else if (v0) {
                x0[u] = __ldg(w + (size_t)d * s.C);
              }
            } else {
              if (v0) x0[u] = __ldg(w + (size_t)d * s.C);
              if (v1) x1[u] = __ldg(w + (size_t)d * s.C + 1);
            }
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int d = d0 + TY * u;
          a0 = fmaf(x0[u], x0[u], a0);
          a1 = fmaf(x1[u], x1[u], a1);
          if (BF16 && d < s.D) {
            __nv_bfloat162* dst = reinterpret_cast<__nv_bfloat162*>(wb + (size_t)d * 64);
            float r0 = x0[u], r1 = x1[u];
#pragma unroll
            for (int p = 0; p < PL; ++p) {             // exact split: residual after each plane
              const __nv_bfloat162 hv = __floats2bfloat162_rn(r0, r1);
              dst[(size_t)p * (plane / 2)] = hv;
              r0 -= __low2float(hv);
              r1 -= __high2float(hv);
            }
          }
        }
      }
    }
    red[ty][tx * 2] = a0;
    red[ty][tx * 2 + 1] = a1;
    __syncthreads();
    for (int t = tid; t < 2 * TX; t += 256) {
      float acc = 0.f;
#pragma unroll
      for (int r = 0; r < TY; ++r) acc += red[r][t];
      const int j = bid * 2 * TX + t;
      if (j < s.Cp) s.inv_c[j] = (j < s.C && acc > 0.f) ? rsqrtf(acc) : 0.f;
      if (s.reg_out) red[0][t] = j < s.C ? acc : 0.f;
    }
    if (s.reg_out) {
      // reg_loss = wd/2 * sum_j c_j^2 (nets/net_base.py:103-107) falls out of the column sums:
      // one partial per block, totalled in a fixed order by the last W-role block to finish
      __syncthreads();
      if (tid == 0) {
        float tot = 0.f;
        for (int t = 0; t < 2 * TX; ++t) tot += red[0][t];
        s.wsq_part[bid] = tot;
      }
      if (block_ticket(s.wsq_ticket, (unsigned)nwb) == (unsigned)nwb - 1) {
        __shared__ float wred[256];
        float acc = 0.f;
        for (int i = tid; i < nwb; i += 256) acc += __ldcg(s.wsq_part + i);
        wred[tid] = acc;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
          if (tid < o) wred[tid] += wred[tid + o];
          __syncthreads();
        }
        if (tid == 0) *s.reg_out = s.reg_scale * wred[0];
      }
    }
  } else {
    const int tx = tid & 31;
    const int row = (bid - nwb) * 8 + (tid >> 5);
    if (row >= s.B) return;
    // embeddings arrive as fp32 or (bf16 mode, asm_set_embedding_dtype) as bf16: `esz` bytes each
    const int esz = s.x_bf16 ? 2 : 4;
    const char* x = reinterpret_cast<const char*>(s.X) + (size_t)row * s.D * esz;
    char* xg = nullptr;
    long long y;
    if (npub > 0) {
      // gathered batch: row `row` lives in the symmetric block of rank row / b_local
      const unsigned cur = p2p_current_step(p);
      const int src = row / p.b_local, lr = row - src * p.b_local;
      if (tx == 0) p2p_wait(p, 0, src, cur);
      __syncwarp();
      x = reinterpret_cast<const char*>(p.x(src, cur & 1)) + (size_t)lr * s.D * esz;
      xg = reinterpret_cast<char*>(p.Xg) + (size_t)row * s.D * esz;   // copy for the r_i x_i term of dX
      y = (long long)__ldcv(p.y(src, cur & 1) + lr);
    } else {
      y = label_bytes == 8 ? reinterpret_cast<const long long*>(labels)[row]
                           : (long long)reinterpret_cast<const int*>(labels)[row];
    }
    if (ADD) {
      prep_row_scaled<PL>(s, x, xg, esz, npub > 0, row, y);
      return;
    }
    float acc = 0.f;
    auto emit = [&](int d, float v) {               // one element: norm, bf16 planes
      acc = fmaf(v, v, acc);
      if (PL > 0) {
        __nv_bfloat16* dst = s.Xb + (size_t)row * PL * s.D + d;
        float r = v;
#pragma unroll
        for (int p2 = 0; p2 < PL; ++p2) {
          const __nv_bfloat16 hv = __float2bfloat16_rn(r);
          dst[(size_t)p2 * s.D] = hv;
          r -= __bfloat162float(hv);
        }
      }
    };
    auto emit16 = [&](int e0, const float4& v) {    // one 16-byte piece: 4 fp32 or 8 bf16 elements
      if (s.x_bf16) {
        const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          emit(e0 + 2 * q, __low2float(h2[q]));
          emit(e0 + 2 * q + 1, __high2float(h2[q]));
        }
      } else {
        emit(e0, v.x); emit(e0 + 1, v.y); emit(e0 + 2, v.z); emit(e0 + 3, v.w);
      }
    };
    {
      // 16-byte pieces of the row, up to 4 per lane requested back to back (for a peer's row every
      // load is an NVLink round trip: nothing is used before all of them are in flight)
      const float4* x4 = reinterpret_cast<const float4*>(x);
      const int n16 = s.D * esz / 16;                // D % 16 == 0
      const int epp = 16 / esz;                      // elements per piece
      for (int i0 = 0; i0 < n16; i0 += 128) {
        float4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int i = i0 + u * 32 + tx;
          v[u] = i < n16 ? (npub > 0 ? __ldcv(x4 + i) : __ldg(x4 + i)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int i = i0 + u * 32 + tx;
          if (i < n16) {
            if (npub > 0) reinterpret_cast<float4*>(xg)[i] = v[u];
            emit16(i * epp, v[u]);
          }
        }
      }
    }
    acc = warp_sum(acc);
    if (tx == 0) prep_row_tail(s, row, acc, y);
  }
}

template <bool VEC2, int PL, int TX, int TY, int U, bool ADD>
__global__ void __launch_bounds__(256) prep_kernel(Step s, const void* labels, int label_bytes,
                                                   int nwb, int npub, P2P p) {
  pdl_trigger();            // first kernel of the step: nothing to wait for
  __shared__ float red[TY][2 * TX];
  if (blockIdx.x == 0 && threadIdx.x == 0) *const_cast<Margin*>(margin_record(s.tgt_s)) = s.mg;
  prep_block<VEC2, PL, TX, TY, U, ADD>(s, labels, label_bytes, nwb, npub, p, (int)blockIdx.x, red);
}

template <int TX, int TY, int U, bool ADD>
static void launch_prep_t(const Step& s, const void* labels, int label_bytes, cudaStream_t st, const P2P* p) {
  const int nwb = (s.Cp + 2 * TX - 1) / (2 * TX);
  const int nxb = (s.B + 7) / 8;
  int npub = 0;
  P2P pp{};
  if (p != nullptr && p->world > 1) {
    pp = *p;
    npub = (int)(((size_t)p->b_local * p->D / 4 + 2047) / 2048);     // 8 float4 per thread
    if (npub < 1) npub = 1;
    if (npub > 32) npub = 32;
  }
  const bool vec2 = (s.C % 2 == 0) && ((reinterpret_cast<uintptr_t>(s.W) & 7) == 0);
  dim3 grd(npub + nwb + nxb);
  if (s.x3) {
    if (vec2) prep_kernel<true, 3, TX, TY, U, ADD><<<grd, 256, 0, st>>>(s, labels, label_bytes, nwb, npub, pp);
    else prep_kernel<false, 3, TX, TY, U, ADD><<<grd, 256, 0, st>>>(s, labels, label_bytes, nwb, npub, pp);
  } else if (s.mode == 1) {
    if (vec2) prep_kernel<true, 1, TX, TY, U, ADD><<<grd, 256, 0, st>>>(s, labels, label_bytes, nwb, npub, pp);
    else prep_kernel<false, 1, TX, TY, U, ADD><<<grd, 256, 0, st>>>(s, labels, label_bytes, nwb, npub, pp);
  } else {
    if (vec2) prep_kernel<true, 0, TX, TY, U, ADD><<<grd, 256, 0, st>>>(s, labels, label_bytes, nwb, npub, pp);
    else prep_kernel<false, 0, TX, TY, U, ADD><<<grd, 256, 0, st>>>(s, labels, label_bytes, nwb, npub, pp);
  }
}

template <int TX, int TY, int U>
static void launch_prep_t(const Step& s, const void* labels, int label_bytes, cudaStream_t st, const P2P* p) {
  if (s.mg.kind != 0) launch_prep_t<TX, TY, U, true>(s, labels, label_bytes, st, p);
  else launch_prep_t<TX, TY, U, false>(s, labels, label_bytes, st, p);
}

void launch_prep(const Step& s, const void* labels, int label_bytes, cudaStream_t st, const P2P* p) {
  // Block shape (column pairs x row groups) and loads in flight per thread.  Measured at
  // cfg 3 (263.9 MB): 32x8/U=4 51.7 us (5.1 TB/s), 16x16/U=8 51.7, 32x8/U=8 53.2,
  // 32x8/U=16 59.8, 32x8/U=32 94, 32x8/U=2 65, 128x2/U=16 73: occupancy beats unroll depth,
  // and wider per-block column spans do not help.  ASM_PREP_SHAPE selects the alternatives.
  static int shape = -1, small_auto = -1;
  if (shape < 0) {
    const char* e = getenv("ASM_PREP_SHAPE");
    shape = e ? atoi(e) : 0;
    // ASM_PREP_AUTO=1 (opt-in until measured): shards below 32 k classes have too few 64-column
    // blocks to fill the SMs, so they take the 16x16 shape (32 columns per block, twice the
    // blocks, half the dependent trips) -- DESIGN.md section 9.
    e = getenv("ASM_PREP_AUTO");
    small_auto = (e && atoi(e) != 0) ? 1 : 0;
  }
  if (shape == 0 && small_auto && s.Cp <= 32768) {
    launch_prep_t<16, 16, 8>(s, labels, label_bytes, st, p);
    return;
  }
  if (shape == 1) launch_prep_t<32, 8, 16>(s, labels, label_bytes, st, p);
  else if (shape == 2) launch_prep_t<16, 16, 8>(s, labels, label_bytes, st, p);
  else if (shape == 3) launch_prep_t<128, 2, 16>(s, labels, label_bytes, st, p);
  else launch_prep_t<32, 8, 4>(s, labels, label_bytes, st, p);
}

// ---------------------------------------------------------------------------------------
// combine_local: one warp per row reduces the per-column-tile (max, sumexp) partials.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) combine_local_kernel(Step s) {
  pdl_trigger();
  pdl_wait();
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= s.B) return;
  float m = -INFINITY, z = 0.f;
  const float2* p = s.part + (size_t)row * s.NT;
  for (int t = lane; t < s.NT; t += 32) {
    const float2 v = p[t];
    ms_combine(m, z, v.x, v.y);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float m2 = __shfl_xor_sync(0xffffffffu, m, o);
    const float z2 = __shfl_xor_sync(0xffffffffu, z, o);
    ms_combine(m, z, m2, z2);
  }
  if (lane == 0) {
    float* st = s.stats_local;
    st[row] = m;
    st[s.B + row] = z;
    st[2 * s.B + row] = s.ylocal[row] >= 0 ? s.tgt_f[row] : 0.f;
  }
}

void launch_combine_local(const Step& s, cudaStream_t st) {
  launch_pdl(combine_local_kernel, dim3((s.B + 7) / 8), dim3(256), 0, st, s.pdl != 0, 1, s);
}

// ---------------------------------------------------------------------------------------
// combine: one warp per batch row.
//   FUSED (single shard): reduce the row's (max, sum-exp) partials, publish stats_local and
//     continue straight to the global quantities.
//   otherwise: reduce the [n_shards, 3, B] statistics gathered from all class shards.
// Per row: M = max_g m_g, Z = sum_g z_g e^{m_g - M}, lse = M + log Z, loss_i = lse - f_y, the
// exp2 offset of the backward, and the target-column gradient coefficients
//   g_y = (e^{f_y - lse} - 1)/B,  G'_y = g_y (lambda + psi')/(1 + lambda),
//   r   = g_y (psi - t psi') / ((1 + lambda) n)            (SURVEY.md 8a, row a3)
// The mean loss is summed in a fixed order by the last block to finish (deterministic).
// ---------------------------------------------------------------------------------------
template <bool FUSED>
__global__ void __launch_bounds__(256) combine_kernel(Step s, const float* stats_all, int n_shards) {
  __shared__ float red[256];
  __shared__ bool is_last;
  pdl_trigger();
  pdl_wait();
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row < s.B) {
    float m = -INFINITY, z = 0.f, fy = 0.f;
    // per-row scalars of the epilogue below: issued up front (warp-uniform addresses) so that
    // they travel together with the partials instead of adding a second memory round trip
    const int yl_row = s.ylocal[row];
    const float tgt_f_row = s.tgt_f[row], tgt_s_row = s.tgt_s[row], inv_n_row = s.inv_n[row];
    if (FUSED) {
      const float2* p = s.part + (size_t)row * s.NT;
      for (int t = lane; t < s.NT; t += 32) {
        const float2 v = p[t];
        ms_combine(m, z, v.x, v.y);
      }
    } else {
      for (int g = lane; g < n_shards; g += 32) {
        const float* sg = stats_all + (size_t)g * 3 * s.B;
        ms_combine(m, z, sg[row], sg[s.B + row]);
        fy += sg[2 * s.B + row];
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float m2 = __shfl_xor_sync(0xffffffffu, m, o);
      const float z2 = __shfl_xor_sync(0xffffffffu, z, o);
      ms_combine(m, z, m2, z2);
      fy += __shfl_xor_sync(0xffffffffu, fy, o);
    }
    if (lane == 0) {
      if (FUSED) {
        fy = yl_row >= 0 ? tgt_f_row : 0.f;
        s.stats_local[row] = m;
        s.stats_local[s.B + row] = z;
        s.stats_local[2 * s.B + row] = fy;
      }
      row_epilogue(s, row, m, z, fy, yl_row, tgt_f_row, tgt_s_row, inv_n_row);
    }
  }
  // With gradients the backward kernels do not need the mean loss: its reduction is deferred
  // to an idle warp of the dX kernel so that the recompute kernel can start right away.
  if (s.defer_loss) return;
  last_block_loss(s, red, &is_last);
}

void launch_combine_global(const Step& s, const float* stats_all, int n_shards, cudaStream_t st) {
  launch_pdl(combine_kernel<false>, dim3((s.B + 7) / 8), dim3(256), 0, st, false, 1, s, stats_all, n_shards);
}

void launch_combine_fused(const Step& s, cudaStream_t st) {
  launch_pdl(combine_kernel<true>, dim3((s.B + 7) / 8), dim3(256), 0, st, s.pdl != 0, 1, s,
             static_cast<const float*>(nullptr), 1);
}

// ---------------------------------------------------------------------------------------
// dx_finish: dX = sum_z dx_part[z] + r_i * x_i   (float4 along D; D % 4 == 0)
// additive margin: dX_i = (s/n_i) (v_i - (x_i.v_i)/n_i^2 x_i),  v_i = sum_z dx_part[z][i]
// ---------------------------------------------------------------------------------------
template <int KS_T>
__global__ void __launch_bounds__(256) dx_finish_kernel(Step s) {
  pdl_trigger();
  pdl_wait();
  dx_finish_rows<KS_T>(s, s.dX, blockIdx.x, gridDim.x);
}

// additive margin: the same sum, then each row projected onto the tangent space of x_i (two rows per block)
__global__ void __launch_bounds__(256) dx_finish_margin_kernel(Step s) {
  __shared__ float red[8];
  pdl_trigger();
  pdl_wait();
  dx_finish_rows_margin(s, s.dX, blockIdx.x, gridDim.x, red);
}

void launch_dx_finish(const Step& s, cudaStream_t st) {
  if (s.mg.kind != 0) {
    int blocks = (s.B + 1) / 2;
    if (blocks > 148 * 8) blocks = 148 * 8;
    launch_pdl(dx_finish_margin_kernel, dim3(blocks), dim3(256), 0, st, s.pdl != 0, 1, s);
    return;
  }
  const size_t total4 = (size_t)s.B * s.D / 4;
  int blocks = (int)((total4 + 255) / 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  switch (s.KS) {
    case 18: launch_pdl(dx_finish_kernel<18>, dim3(blocks), dim3(256), 0, st, s.pdl != 0, 1, s); break;
    case 9:  launch_pdl(dx_finish_kernel<9>, dim3(blocks), dim3(256), 0, st, s.pdl != 0, 1, s); break;
    case 4:  launch_pdl(dx_finish_kernel<4>, dim3(blocks), dim3(256), 0, st, s.pdl != 0, 1, s); break;
    default: launch_pdl(dx_finish_kernel<0>, dim3(blocks), dim3(256), 0, st, s.pdl != 0, 1, s); break;
  }
}

// ---------------------------------------------------------------------------------------
// opt_stream: the classifier update as ONE streaming pass over (dW, W, state) after the plain
// dW kernel -- the alternative to the fused dW epilogue (ASM_OPT_STREAM=1, DESIGN.md section 9
// item 4).  Same opt_apply arithmetic; fully sequential 16-byte accesses.
// ---------------------------------------------------------------------------------------
template <int V>
__global__ void __launch_bounds__(256) opt_stream_kernel(const float* __restrict__ dW, float* W, float* s0,
                                                         float* s1, size_t n, OptParams op) {
  pdl_trigger();
  pdl_wait();
  const size_t stride = (size_t)gridDim.x * blockDim.x * V;
  for (size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * V; i < n; i += stride) {
    float g[V], w[V], a[V], b[V];
    if (V == 4) {
      const float4 gv = __ldcs(reinterpret_cast<const float4*>(dW + i));
      const float4 wv = *reinterpret_cast<const float4*>(W + i);
      const float4 av = *reinterpret_cast<const float4*>(s0 + i);
      const float4 bv = op.kind == 2 ? *reinterpret_cast<const float4*>(s1 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
      g[0] = gv.x; g[1] = gv.y; g[2] = gv.z; g[3] = gv.w;
      w[0] = wv.x; w[1] = wv.y; w[2] = wv.z; w[3] = wv.w;
      a[0] = av.x; a[1] = av.y; a[2] = av.z; a[3] = av.w;
      b[0] = bv.x; b[1] = bv.y; b[2] = bv.z; b[3] = bv.w;
    } else {
      g[0] = dW[i]; w[0] = W[i]; a[0] = s0[i]; b[0] = op.kind == 2 ? s1[i] : 0.f;
    }
#pragma unroll
    for (int v = 0; v < V; ++v) opt_apply(op, g[v], w[v], a[v], b[v]);
    if (V == 4) {
      *reinterpret_cast<float4*>(W + i) = make_float4(w[0], w[1], w[2], w[3]);
      *reinterpret_cast<float4*>(s0 + i) = make_float4(a[0], a[1], a[2], a[3]);
      if (op.kind == 2) *reinterpret_cast<float4*>(s1 + i) = make_float4(b[0], b[1], b[2], b[3]);
    } else {
      W[i] = w[0]; s0[i] = a[0];
      if (op.kind == 2) s1[i] = b[0];
    }
  }
}

void launch_opt_stream(const Step& s, const float* dW, cudaStream_t st) {
  const size_t n = (size_t)s.D * s.C;
  const uintptr_t al = reinterpret_cast<uintptr_t>(dW) | reinterpret_cast<uintptr_t>(s.Wmut) |
                       reinterpret_cast<uintptr_t>(s.opt_s0) | reinterpret_cast<uintptr_t>(s.opt_s1);
  if (n % 4 == 0 && (al & 15) == 0) {
    size_t blocks = (n / 4 + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    launch_pdl(opt_stream_kernel<4>, dim3((unsigned)blocks), dim3(256), 0, st, false, 1, dW, s.Wmut, s.opt_s0,
               s.opt_s1, n, s.opt);
  } else {
    size_t blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    launch_pdl(opt_stream_kernel<1>, dim3((unsigned)blocks), dim3(256), 0, st, false, 1, dW, s.Wmut, s.opt_s0,
               s.opt_s1, n, s.opt);
  }
}

template <int TX, int TY, int U, bool ADD>
static void preload_prep_t() {
  cudaFuncAttributes a;
  cudaFuncGetAttributes(&a, prep_kernel<true, 3, TX, TY, U, ADD>);
  cudaFuncGetAttributes(&a, prep_kernel<false, 3, TX, TY, U, ADD>);
  cudaFuncGetAttributes(&a, prep_kernel<true, 1, TX, TY, U, ADD>);
  cudaFuncGetAttributes(&a, prep_kernel<false, 1, TX, TY, U, ADD>);
  cudaFuncGetAttributes(&a, prep_kernel<true, 0, TX, TY, U, ADD>);
  cudaFuncGetAttributes(&a, prep_kernel<false, 0, TX, TY, U, ADD>);
}
template <int TX, int TY, int U>
static void preload_prep_t() {
  preload_prep_t<TX, TY, U, false>();
  preload_prep_t<TX, TY, U, true>();
}
void prep_preload_kernels() {
  preload_prep_t<16, 16, 8>();
  preload_prep_t<32, 8, 16>();
  preload_prep_t<128, 2, 16>();
  preload_prep_t<32, 8, 4>();
  cudaFuncAttributes a;
  cudaFuncGetAttributes(&a, combine_local_kernel);
  cudaFuncGetAttributes(&a, combine_kernel<true>);
  cudaFuncGetAttributes(&a, combine_kernel<false>);
  cudaFuncGetAttributes(&a, dx_finish_kernel<0>);
  cudaFuncGetAttributes(&a, dx_finish_margin_kernel);
  cudaFuncGetAttributes(&a, opt_stream_kernel<4>);
  cudaFuncGetAttributes(&a, opt_stream_kernel<1>);
}

}  // namespace asmh
