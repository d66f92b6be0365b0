// Class-sharded step over NVLink peer memory: the three collectives of the sharded head
// (all-gather X / labels, all-gather of the [3,B] softmax statistics, reduce-scatter of dX)
// done INSIDE the head's own kernels with P2P loads from the peers' symmetric buffers and
// release/acquire flags -- no NCCL launch and no transport-only launch anywhere in the step:
//
//   prep_kernel           publish my rows (phase 0)  |  W norms  |  gather + normalise all rows
//   umma_kernel<FWD>      (unchanged)
//   combine_p2p_kernel    my [3,B] statistics -> my block (phase 1), wait, global combine
//   umma_kernel<BWDG>, <DW>, <DX>   (unchanged)
//   dx_finish_p2p_kernel  my dX contribution -> my block (phase 2), wait, sum of MY rows
//
// i.e. 7 launches per step (15 before the fold).  Every rank owns one symmetric block
// (peer-mapped by the host, e.g. torch symmetric memory):
//   x   [2][b_max, D] fp32   this rank's embeddings, double-buffered by step parity
//   y   [2][b_max]    int32  this rank's labels
//   st  [2][3, B_max] fp32   this shard's (max, sum-exp, target logit) statistics
//   dx  [2][B_max, D] fp32   this shard's dX contribution for ALL rows
//   fl  [3][16]       u32    flags[phase][src rank] = last step that rank published
// Producers write only their OWN block and then push their step number into every peer's
// flag word (st.release.sys); consumers spin on their local flag words (ld.acquire.sys) and
// read the peers' data with L1-bypassing loads.  Parity double-buffering is sufficient
// because a rank can run at most one step ahead of its slowest peer (it needs that peer's
// step-s statistics and dX before it can finish step s).  Ranks must therefore stay in
// lock-step; a peer that does not arrive within the configured time is reported through
// asm_p2p_status(), not by a trap.
#include "asm_common.cuh"
#include "asm_kernels.cuh"
#include "asm_p2p.cuh"
#include "asm_rows.cuh"

namespace asmh {

// ---- phase 1: statistics of this shard out, everybody's in, global combine -----------------
// One warp per batch row (as combine_kernel).  The local half reduces the forward kernel's
// per-CTA (max, sum-exp) partials and writes the row's three statistics to this rank's block;
// the last block to finish raises the phase-1 flag on every peer.  The global half then waits
// for each peer's flag (lane g waits for rank g) and reads that rank's three floats for the row
// straight from its block: M = max_g m_g, Z = sum_g z_g e^{m_g - M}, f_y = sum_g f_y,g.
__global__ void __launch_bounds__(256) combine_p2p_kernel(Step s, P2P p) {
  __shared__ float red[256];
  pdl_trigger();
  pdl_wait();
  const unsigned cur = p2p_current_step(p);
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const bool rv = row < s.B;
  if (rv) {
    float m = -INFINITY, z = 0.f;
    const int yl_row = s.ylocal[row];
    const float tgt_f_row = s.tgt_f[row];
    const float2* pt = s.part + (size_t)row * s.NT;
    for (int t = lane; t < s.NT; t += 32) {
      const float2 v = pt[t];
      ms_combine(m, z, v.x, v.y);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float m2 = __shfl_xor_sync(0xffffffffu, m, o);
      const float z2 = __shfl_xor_sync(0xffffffffu, z, o);
      ms_combine(m, z, m2, z2);
    }
    if (lane == 0) {
      float* st = p.st(p.rank, cur & 1);
      st[row] = m;
      st[s.B + row] = z;
      st[2 * s.B + row] = yl_row >= 0 ? tgt_f_row : 0.f;
    }
  }
  const unsigned n = gridDim.x;
  const unsigned tk = block_ticket(p.tickets + 1, n);
  if (tk == n - 1 && threadIdx.x == 0) p2p_publish(p, 1, cur);
  // only the last `waiters` blocks stay for the exchange (all of them by default): the number of
  // blocks that can ever spin on a peer is bounded, which matters when ranks share a GPU
  const unsigned nred = n < (unsigned)p.waiters ? n : (unsigned)p.waiters;
  if (tk < n - nred) return;
  const unsigned vb = tk - (n - nred);
  for (int r2 = (int)vb * 8 + (threadIdx.x >> 5); r2 < s.B; r2 += (int)nred * 8) {
    float m = -INFINITY, z = 0.f, fy = 0.f;
    if (lane < p.world) {
      p2p_wait(p, 1, lane, cur);
      const float* sg = p.st(lane, cur & 1);
      m = __ldcv(sg + r2);
      z = __ldcv(sg + s.B + r2);
      fy = __ldcv(sg + 2 * s.B + r2);
    }
    // fixed combination order (butterfly over the lanes): identical bits on every rank
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float m2 = __shfl_xor_sync(0xffffffffu, m, o);
      const float z2 = __shfl_xor_sync(0xffffffffu, z, o);
      ms_combine(m, z, m2, z2);
      fy += __shfl_xor_sync(0xffffffffu, fy, o);
    }
    if (lane == 0) row_epilogue(s, r2, m, z, fy, s.ylocal[r2], s.tgt_f[r2], s.tgt_s[r2], s.inv_n[r2]);
  }
  if (s.defer_loss) return;
  // mean loss, summed in a fixed order by the last of the remaining blocks
  if (block_ticket(p.tickets + 3, nred) != nred - 1) return;
  float acc = 0.f;
  for (int i = threadIdx.x; i < s.B; i += 256) acc += __ldcg(s.rowloss + i);
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0 && s.loss) *s.loss = red[0] * s.invB;
}

void launch_combine_p2p(const Step& s, const P2P& p, cudaStream_t st) {
  launch_pdl(combine_p2p_kernel, dim3((s.B + 7) / 8), dim3(256), 0, st, s.pdl != 0, 1, s, p);
}

// ---- phase 2: dX contribution of this shard out, everybody's in, sum of this rank's rows -----
// All blocks finish dX = sum_z dx_part[z] + r_i x_i for ALL rows into this rank's block.  The last
// block to finish raises the phase-2 flag and closes the step (the step counter advances: every
// kernel of the step, this one included, has read it by then).  Only the last kReducers blocks
// stay for the exchange (p.waiters: so at most that many blocks ever spin on a peer), wait for every
// rank's flag and sum this rank's rows over the shards in rank order (deterministic).
__device__ __forceinline__ void dx_exchange(const Step& s, const P2P& p, unsigned cur) {
  const unsigned n = gridDim.x;
  const unsigned tk = block_ticket(p.tickets + 2, n);
  if (tk == n - 1 && threadIdx.x == 0) {
    p2p_publish(p, 2, cur);
    *p.step_dev = cur;
  }
  const unsigned cap = (unsigned)p.waiters < 32u ? (unsigned)p.waiters : 32u;
  const unsigned nred = n < cap ? n : cap;
  if (tk < n - nred) return;
  const unsigned vb = tk - (n - nred);
  if (threadIdx.x < (unsigned)p.world) p2p_wait(p, 2, threadIdx.x, cur);
  __syncthreads();
  const size_t n4 = (size_t)p.b_local * s.D / 4;
  const size_t row0 = (size_t)p.rank * p.b_local * s.D / 4;
  for (size_t i = vb * (size_t)256 + threadIdx.x; i < n4; i += (size_t)nred * 256) {
    // all peers' contributions are requested before the first add: one NVLink round trip per
    // element instead of one per peer; the sum still runs in rank order (deterministic)
    float4 v[kMaxPeers];
#pragma unroll
    for (int g = 0; g < kMaxPeers; ++g)
      v[g] = g < p.world ? __ldcv(reinterpret_cast<const float4*>(p.dx(g, cur & 1)) + row0 + i)
                         : make_float4(0.f, 0.f, 0.f, 0.f);
    float4 a = v[0];
#pragma unroll
    for (int g = 1; g < kMaxPeers; ++g) {
      if (g < p.world) { a.x += v[g].x; a.y += v[g].y; a.z += v[g].z; a.w += v[g].w; }
    }
    reinterpret_cast<float4*>(p.dx_local)[i] = a;
  }
}

template <int KS_T>
__global__ void __launch_bounds__(256) dx_finish_p2p_kernel(Step s, P2P p) {
  pdl_trigger();
  pdl_wait();
  const unsigned cur = p2p_current_step(p);
  dx_finish_rows<KS_T>(s, p.dx(p.rank, cur & 1), blockIdx.x, gridDim.x);
  dx_exchange(s, p, cur);
}

// additive margin: this shard projects its own partial sum of every row before it publishes it
// (the projection is linear in v); the rank-order sum of the exchange is unchanged
__global__ void __launch_bounds__(256) dx_finish_margin_p2p_kernel(Step s, P2P p) {
  __shared__ float red[8];
  pdl_trigger();
  pdl_wait();
  const unsigned cur = p2p_current_step(p);
  dx_finish_rows_margin(s, p.dx(p.rank, cur & 1), blockIdx.x, gridDim.x, red);
  dx_exchange(s, p, cur);
}

void launch_dx_finish_p2p(const Step& s, const P2P& p, cudaStream_t st) {
  if (s.mg.kind != 0) {
    int blocks = (s.B + 1) / 2;
    if (blocks > 148 * 2) blocks = 148 * 2;
    launch_pdl(dx_finish_margin_p2p_kernel, dim3(blocks), dim3(256), 0, st, s.pdl != 0, 1, s, p);
    return;
  }
  const size_t total4 = (size_t)s.B * s.D / 4;
  int blocks = (int)((total4 + 255) / 256);
  if (blocks > 148 * 2) blocks = 148 * 2;
  switch (s.KS) {
    case 18: launch_pdl(dx_finish_p2p_kernel<18>, dim3(blocks), dim3(256), 0, st, s.pdl != 0, 1, s, p); break;
    case 9:  launch_pdl(dx_finish_p2p_kernel<9>, dim3(blocks), dim3(256), 0, st, s.pdl != 0, 1, s, p); break;
    case 4:  launch_pdl(dx_finish_p2p_kernel<4>, dim3(blocks), dim3(256), 0, st, s.pdl != 0, 1, s, p); break;
    default: launch_pdl(dx_finish_p2p_kernel<0>, dim3(blocks), dim3(256), 0, st, s.pdl != 0, 1, s, p); break;
  }
}

// With lazy module loading the first launch of a kernel may synchronise the context.  A rank whose
// earlier kernel is already spinning on a peer must never get into that situation (several ranks
// can share one process, and then one GPU context), so the transport's kernels are loaded up front.
void p2p_preload_kernels() {
  cudaFuncAttributes a;
  cudaFuncGetAttributes(&a, combine_p2p_kernel);
  cudaFuncGetAttributes(&a, dx_finish_p2p_kernel<18>);
  cudaFuncGetAttributes(&a, dx_finish_p2p_kernel<9>);
  cudaFuncGetAttributes(&a, dx_finish_p2p_kernel<4>);
  cudaFuncGetAttributes(&a, dx_finish_p2p_kernel<0>);
  cudaFuncGetAttributes(&a, dx_finish_margin_p2p_kernel);
  prep_preload_kernels();
  simt_preload_kernels();
  cudaGetLastError();
}

}  // namespace asmh
