// bf16 mode: the four contractions of the A-softmax head as tcgen05 / TMEM tensor-core
// GEMMs fed by TMA, with the head's epilogues fused (hand-written for sm_100a).
//
// One persistent, warp-specialised kernel template (CTA tile 128 x 256 x 64, 4-stage
// TMA->smem ring, 2 accumulator stages of 256 TMEM columns so the epilogue of tile t
// overlaps the MMAs of tile t+1), 384 threads (640 in the paired forward / recompute kernels):
//   warp 0  : TMA producer (one elected lane)      warp 1 : tcgen05.mma issuer (one lane)
//   warp 2  : TMEM allocator; in the paired dW kernel also the issuer of the dW TMA stores
//   warp 3  : dW: weight-chunk producer; dX: deferred loss sum
//   warps 4-11 (4-19 with sixteen epilogue warps) : epilogue; warp w owns TMEM lanes
//             32*(w%4).. and the column group (w-4)/4 of the 256-column accumulator
//
//   KIND   D (lanes x columns)          A (M x K)                  B (N x K)
//   FWD    S   [batch x classes] K=D    Xb [B,D]   K-major         Wb (below) MN-major
//   BWDG   S^T [classes x batch] K=D    Wb         MN-major        Xb [B,D]   K-major
//   DW     dW^T[classes x d]     K=B    G''[Cp,Bp] K-major         Xb [B,D]   MN-major
//   DX     dX  [batch x d]       K=C    G''[Cp,Bp] MN-major        Wb         K-major (split-K)
// G'' = G' diag(1/c) is kept CLASS-major ([Cp, Bp], batch contiguous): the recompute kernel's
// threads own a class each, so their 32 batch values of a chunk are 64 contiguous bytes -- four
// 16-byte shared-memory stores into a 64B-swizzled staging block that one TMA store writes out.
// The orientation is chosen per kernel so that every reduction is thread-local and every
// global store is coalesced: in FWD a thread owns a batch row (online max / sum-exp over the
// classes in its registers); in BWDG and DW a thread owns a class (the column sums q_j and
// the 1/c_j scaling are per-thread constants, and for a fixed batch row / fixed d the 32
// lanes of a warp write 32 consecutive classes of G'' / dW).  The bf16 copy of W keeps the
// reference's orientation (d outer, classes inner: no transpose anywhere) but is stored
// column-blocked, [Cp/64][D][64], so that every 64-class TMA box is one contiguous piece;
// every operand is read by TMA with 128-byte swizzle, and nothing but [B]-sized statistics
// leaves the forward kernel.
#include <type_traits>

#include "asm_common.cuh"
#include "asm_kernels.cuh"
#include "asm_umma.cuh"

// Bring-up knobs (ASM_UMMA_DEBUG bits: skip the epilogue math, experimental kernel variants)
// exist only in a -DASM_BRINGUP build; the default library cannot be told to skip work.
#ifdef ASM_BRINGUP
#define ASM_DBG(flags, bit) ((flags) & (bit))
#else
#define ASM_DBG(flags, bit) 0
#endif

namespace asmh {

namespace {
constexpr int BM = 128, BN = 256, BK = 64, STAGES = 4;
constexpr int BN_FULL = BN;                   // widest tile: sizes the per-tile vectors and the TMEM stage stride
constexpr int A_BYTES = BM * BK * 2;           // 16 KB
constexpr int B_BYTES = BN * BK * 2;           // 32 KB
constexpr int STAGE_BYTES = A_BYTES + B_BYTES; // 48 KB
// threads per CTA: 4 role warps + the epilogue warps of the instantiation (Geo::NTHREADS: 384 or 640)
constexpr int AUX_BARS = 512;                  // barriers + tmem ptr
constexpr int AUX_VEC = 3 * 2 * BN * 4;        // per-tile vectors: 3 arrays x 2 stages x 256
constexpr int STG_HALF = 32 * 128 * 2;         // G'' staging per column half: 128 classes x 32 batch rows (bf16)
constexpr int AUX_STG = 2 * STG_HALF;          // 16 KB
constexpr int WB_BUF = 32 * 128 * 2;           // DW: one [32 d x 128 classes] bf16 weight chunk
constexpr int AUX_WB = 2 * 2 * WB_BUF;         // 2 column halves x 2 buffers = 32 KB
constexpr int DSTG = 32 * 128 * 4;             // DW: one [32 d x 128 classes] fp32 staging block of dW (16 KB)
// the region after the barriers holds vec + stg (FWD / BWDG) or the weight-chunk ring (DW)
constexpr int AUX_REGION = (AUX_VEC + AUX_STG) > AUX_WB ? (AUX_VEC + AUX_STG) : AUX_WB;
constexpr float LOG2E = 1.4426950408889634f;

// U_FWDR is an experimental forward kernel with the CTA's 128-row block of Xb RESIDENT in
// shared memory (D <= 512): only the weight tiles stream (32-deep K stages, 5 of them), which
// cuts the L2 -> SM operand traffic by a third.  Measured SLOWER than the streaming kernel
// (55 vs 48 us at cfg 3): the pipeline is bound by bytes in flight (80 KB vs 192 KB), not by
// L2 bandwidth.  Kept behind ASM_UMMA_DEBUG bit 2 as the record of that experiment.
// U_DWOPT is the dW kernel with the classifier optimizer fused into its epilogue.
// U_DWF is the dW kernel of the fp32 (x3) path: the correction term reads the fp32 weights.
// U_BWDG1 is BWDG with the earlier geometry (6 operand stages, one staging buffer, two named
// barriers per chunk), selectable with ASM_UMMA_DEBUG bit 3 for same-box A/B timing.
enum { U_FWD = 0, U_BWDG = 1, U_DW = 2, U_DX = 3, U_FWDR = 4, U_DWOPT = 5, U_DWF = 6, U_BWDG1 = 7 };

// pipeline geometry per kernel kind
// CG = 2: a CTA pair (cluster of 2, cta_group::2) computes one 256 x 256 tile; each CTA
// stages its own 128 A rows and HALF of the B tile, so a stage is 32 KB and the ring is 6 deep.
// BNT: tile width along N (256, or 128 for shards whose unit count does not fill the pairs)
#ifndef ASM_FWD_EPI16
#define ASM_FWD_EPI16 1
#endif
constexpr bool FWD_EPI16 = ASM_FWD_EPI16 != 0;
#ifndef ASM_BWDG_EPI16
#define ASM_BWDG_EPI16 1
#endif
constexpr bool BWDG_EPI16 = ASM_BWDG_EPI16 != 0;
template <int KIND, int CG = 1, int BNT = BN_FULL> struct Geo {
  static constexpr bool RES = (KIND == U_FWDR);
  // Epilogue warps.  The epilogues, not the MMAs, bound these kernels (the light dX epilogue
  // reaches 83 % of the tensor pipe, the forward one 62 %): each scheduler hosts only two
  // epilogue warps, which spend ~8 cycles per issued instruction on dependency and queue
  // latencies.  The forward and the recompute kernel of a CTA pair therefore run SIXTEEN
  // epilogue warps -- four per TMEM lane quarter, 64 accumulator columns each -- with
  // single-buffered TMEM loads (and, in the recompute kernel, one G'' staging block per warp) to
  // stay inside 96 registers and the shared memory.
  static constexpr int EPIW = ((KIND == U_FWD && FWD_EPI16) || (KIND == U_BWDG && BWDG_EPI16)) && CG == 2 && BNT == 256 ? 16 : 8;
  static constexpr int NTHREADS = 128 + 32 * EPIW;
  static constexpr int KB = (RES && CG == 1) ? 32 : BK;    // K elements per pipeline stage
  // weight-chunk buffers per column half (4 buffers paid for with one of the dW kernel's four
  // operand stages measured SLOWER: 83 vs 78 us at config 3)
  static constexpr int NWB = 2;
  // the dW kernel of a CTA pair stages its output in shared memory and leaves through TMA
  // stores (two [32 d x 128 classes] fp32 buffers per column half), paid for with two operand stages
  static constexpr bool DW_TMA = (KIND == U_DW && CG == 2);
  // the BWDG kernel of a CTA pair trades its 6th operand stage for double-buffered G'' staging
  static constexpr int NSB = (KIND == U_BWDG && CG == 2) ? 2 : 1;   // G'' staging buffers per column half
  static constexpr int NST = RES ? 5 : (CG == 2 ? (DW_TMA ? 4 : (KIND == U_BWDG ? 5 : 6)) : STAGES);   // pipeline depth
  static constexpr int A_ST = RES ? 0 : BM * KB * 2;       // A bytes per stage
  static constexpr int B_ST = BNT * KB * 2 / CG;           // B bytes per stage (per CTA)
  static constexpr int ST_B = A_ST + B_ST;
  static constexpr int RES_B = RES ? 8 * A_BYTES : 0;      // resident A block (K <= 512)
  static constexpr int CH_B = 64 * KB * 2;                 // one 64-wide MN-major chunk
  static constexpr int PIPE_B = RES_B + NST * ST_B;
  static constexpr int AUX_R = (RES || KIND == U_FWD) ? AUX_VEC       // forward: the per-tile vectors only
                               : (KIND == U_DW ? 2 * NWB * WB_BUF + (DW_TMA ? 4 * DSTG : 0)
                                               : (NSB == 2 ? AUX_VEC + 2 * AUX_STG + (EPIW == 16 ? 2048 : 0) : AUX_REGION));
  static constexpr int SMEM = PIPE_B + AUX_BARS + AUX_R + 1024;
  static_assert(SMEM <= 232448, "exceeds the 227 KB shared memory of an sm_100 CTA");
};

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ float fast_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// (i == k) ? a : b as one setp + selp (keeps dynamic-index selects out of branch trees)
__device__ __forceinline__ float sel_eq(int i, int k, float a, float b) {
  float r;
  asm("{\n\t.reg .pred p;\n\tsetp.eq.s32 p, %1, %2;\n\tselp.f32 %0, %3, %4, p;\n\t}\n"
      : "=f"(r)
      : "r"(i), "r"(k), "f"(a), "f"(b));
  return r;
}
// Rare paths of the forward epilogue, kept out of line so the hot loop stays small.
// The margin comes from the record the norm kernel stored in front of tgt_s: an extra argument
// would change the register allocation of the forward kernel's hot loop.
__device__ __noinline__ float fwd_target(float* tgt_s, float* tgt_f, const float* n,
                                         const float* inv_n, int m, float lambda, int row,
                                         float sv) {
  tgt_s[row] = sv;
  const Margin mg = *margin_record(tgt_s);
  const float fv = mg.kind != 0 ? additive_logit(sv, mg) : target_logit(sv, n[row], inv_n[row], m, lambda);
  tgt_f[row] = fv;
  return fv;
}
}  // namespace

template <int KIND, int CG = 1, int BNT = BN_FULL>
__global__ void __launch_bounds__((Geo<KIND, CG, BNT>::NTHREADS), 1)
umma_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
            const __grid_constant__ CUtensorMap mapC, const __grid_constant__ CUtensorMap mapD,
            const __grid_constant__ CUtensorMap mapE, Step s, UmmaArgs g) {
  using G_ = Geo<KIND, CG, BNT>;
  constexpr int BN = BNT;                 // tile width of this instantiation (shadows the default)
  constexpr int EPIW = G_::EPIW;          // epilogue warps (8, or 16 in the paired forward kernel)
  constexpr int NQ = EPIW / 4;            // column groups ("halves" below): 2, or 4
  constexpr int HC = BN / NQ;             // accumulator columns per column group
  constexpr int EPI_THREADS = 32 * EPIW;
  static_assert(BNT == 256 || BNT == 128, "tile width");
  static_assert(BNT == 256 || (KIND != U_FWDR && KIND != U_BWDG1), "narrow tiles: main kinds only");
  pdl_trigger();      // the next kernel's CTAs may take over SMs as this grid's tail drains
  // CTA pair: rank within the cluster, work is distributed over PAIRS
  const int crank = CG == 2 ? (int)ptx::cluster_ctarank() : 0;
  const int pair_id = (int)blockIdx.x / CG;
  const int npairs = (int)gridDim.x / CG;
  constexpr bool IS_FWD = (KIND == U_FWD || KIND == U_FWDR);
  constexpr bool RES = G_::RES;
  constexpr int KB = G_::KB, NST = G_::NST, A_ST = G_::A_ST, ST_B = G_::ST_B;
  constexpr int RES_B = G_::RES_B, CH_B = G_::CH_B, PIPE_B = G_::PIPE_B;
  constexpr bool IS_DW = (KIND == U_DW || KIND == U_DWOPT || KIND == U_DWF);
  constexpr bool IS_BWDG = (KIND == U_BWDG || KIND == U_BWDG1);
  constexpr bool A_MN = (IS_BWDG || KIND == U_DX);
  constexpr bool B_MN = (IS_FWD || IS_DW);
  constexpr bool N_FAST = (IS_BWDG || IS_DW);   // tile order: n index fastest
  extern __shared__ uint8_t smem_raw[];
  // align to 1024 B (SWIZZLE_128B atoms) by adding an integer offset, so that the compiler
  // keeps the shared address space (ld.shared, not generic loads) for everything below
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* pipe = smem + RES_B;                                       // stage ring
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + PIPE_B);        // [8] (NST used)
  uint64_t* empty = full + 8;                                         // [8]
  uint64_t* tfull = empty + 8;                                        // [2]
  uint64_t* tempty = tfull + 2;                                       // [2]
  uint64_t* wfull = tempty + 2;                                       // DW: [half][buf]; FWDR: [0] = X resident
  uint64_t* wempty = wfull + 8;                                       // DW: [half][buf]
  uint64_t* sfull = wempty + 8;                                       // DW (pairs): [half][2] staging buffer filled
  uint64_t* sempty = sfull + 4;                                       // DW (pairs): [half][2] ... drained by its TMA store
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(sempty + 4);
  constexpr int NWB = G_::NWB;
  float* vec0 = reinterpret_cast<float*>(smem + PIPE_B + AUX_BARS);   // [2][BN_FULL]
  float* vec1 = vec0 + 2 * BN_FULL;
  float* vec2 = vec1 + 2 * BN_FULL;
  uint8_t* stg = smem + PIPE_B + AUX_BARS + AUX_VEC;                  // BWDG: [2 halves][NSB][STG_HALF]
  constexpr int NSB = G_::NSB;
  uint8_t* wbuf = smem + PIPE_B + AUX_BARS;                           // DW: [2][2][WB_BUF]
  uint8_t* dstg = wbuf + 2 * NWB * WB_BUF;                            // DW (pairs): [2 halves][2][DSTG]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && ptx::elect_one()) {
    ptx::prefetch_tmap(&mapA);
    ptx::prefetch_tmap(&mapB);
    if (IS_BWDG || KIND == U_DW || KIND == U_DX) ptx::prefetch_tmap(&mapC);
    if (G_::DW_TMA) { ptx::prefetch_tmap(&mapD); ptx::prefetch_tmap(&mapE); }
    if (IS_BWDG) ptx::prefetch_tmap(&mapD);
  }
  if (warp == 1 && ptx::elect_one()) {
    for (int i = 0; i < NST; ++i) {
      ptx::mbar_init(&full[i], 1);
      ptx::mbar_init(&empty[i], 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&tfull[a], 1);
      ptx::mbar_init(&tempty[a], EPIW * CG);                 // one arrival per epilogue warp
    }
    for (int i = 0; i < 8; ++i) {
      ptx::mbar_init(&wfull[i], 1);
      ptx::mbar_init(&wempty[i], 128);
    }
    for (int i = 0; i < 4; ++i) {
      ptx::mbar_init(&sfull[i], 4);                          // one arrival per epilogue warp of the half
      ptx::mbar_init(&sempty[i], 1);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    if (CG == 2) { ptx::tmem_alloc_cg2(tmem_ptr, 512); ptx::tmem_relinquish_cg2(); }
    else         { ptx::tmem_alloc(tmem_ptr, 512); ptx::tmem_relinquish(); }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (CG == 2) ptx::cluster_sync_all();       // the peer's barriers exist before anyone signals
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  // prologue done (barriers, TMEM, descriptor prefetch overlapped the predecessor's tail);
  // from here on the kernel reads what earlier kernels wrote
  pdl_wait();

  const int tiles_mn = g.mt * g.nt;
  const int total = tiles_mn * g.ks;
  auto decode = [&](int u, int& z, int& m_idx, int& n_idx) {
    z = u / tiles_mn;
    const int t = u - z * tiles_mn;
    if (N_FAST) { m_idx = t / g.nt; n_idx = t - m_idx * g.nt; }
    else        { n_idx = t / g.mt; m_idx = t - n_idx * g.mt; }
    // class tiles in descending order: consecutive kernels of a step sweep the classes in
    // opposite directions, so each starts on what its predecessor left in L2
    if (g.rev) { if (N_FAST) m_idx = g.mt - 1 - m_idx; else n_idx = g.nt - 1 - n_idx; }
  };
  // K blocks of split z.  Contiguous ranges [z kb_per, (z+1) kb_per) by default; with
  // g.kstride (dX: K = classes) split z takes blocks z, z + ks, z + 2 ks, ... so that ALL CTAs
  // sweep the class range together (descending when g.rev) -- the sweep starts on the classes
  // the preceding kernel touched last, which are still in L2.
  auto kcount = [&](int z) {
    if (g.kstride) return (g.kb_total - z + g.ks - 1) / g.ks;
    const int kb0 = z * g.kb_per;
    return min(g.kb_total, kb0 + g.kb_per) - kb0;
  };
  auto kblock = [&](int z, int i) {
    if (g.kstride) return g.rev ? g.kb_total - 1 - (z + i * g.ks) : z + i * g.ks;
    return z * g.kb_per + i;
  };

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (ptx::elect_one()) {
      uint32_t it = 0;
      if (RES && pair_id < total) {
        // the CTA's 128 batch rows of Xb, all of K, loaded once (grid % mt == 0)
        const int nblk = (s.D + 63) / 64;
        const int mrow = ((pair_id % g.mt) * CG + crank) * BM;
        if (CG == 2) {
          // both CTAs' blocks are counted on the leader's barrier (the leader issues the MMAs)
          if (crank == 0) ptx::mbar_expect_tx(&wfull[0], 2 * nblk * A_BYTES);
          for (int i = 0; i < nblk; ++i)
            ptx::tma_load_2d_cg2(smem + i * A_BYTES, &mapA, &wfull[0], i * 64, mrow);
        } else {
          ptx::mbar_expect_tx(&wfull[0], nblk * A_BYTES);
          for (int i = 0; i < nblk; ++i)
            ptx::tma_load_2d(smem + i * A_BYTES, &mapA, &wfull[0], i * 64, mrow);
        }
      }
      for (int u = pair_id; u < total; u += npairs) {
        int z, m_idx, n_idx;
        decode(u, z, m_idx, n_idx);
        const int m0 = (m_idx * CG + crank) * BM, n0 = n_idx * BN;
        const int nk = kcount(z);
        for (int ki = 0; ki < nk; ++ki, ++it) {
          const int kb = kblock(z, ki);
          const int st = it % NST;
          const uint32_t ph = (it / NST) & 1;
          ptx::mbar_wait(&empty[st], ph ^ 1);
          uint8_t* sA = pipe + st * ST_B;
          uint8_t* sB = sA + A_ST;
          int k0 = kb * KB, oa = 0, ob = 0;
          if (g.nseg > 1) {
            // x3: plane-pair segment of this K block; the plane offset goes to the INNER
            // coordinate of each operand's tensor (K for K-major loads, M/N for MN-major)
            const int seg = kb / g.kb_seg;
            k0 = (kb - seg * g.kb_seg) * KB;
            oa = g.segA[seg];
            ob = g.segB[seg];
          }
          const int kA = A_MN ? k0 : k0 + oa, mA = A_MN ? m0 + oa : m0;
          const int kB = B_MN ? k0 : k0 + ob, nB = B_MN ? n0 + ob : n0;
          // The bf16 weights are stored COLUMN-BLOCKED, [plane][Cp/64][D][64]: the 64 classes x rows
          // box of any weight operand is one contiguous piece of memory (8 KB for 64 rows), not 64
          // rows a whole weight-matrix pitch apart.  Box coordinate: (0, row of the 2-D view
          // [planes * Cp/64 * D, 64]); for weight operands oa / ob hold the PLANE, not an offset.
          auto wb_row = [&](int cls0, int d0, int plane) { return (plane * (s.Cp >> 6) + (cls0 >> 6)) * s.D + d0; };
          if (CG == 2) {
            // both CTAs load their A rows and their half of B; all bytes are counted on the
            // leader's full barrier, which only the leader arms
            if (crank == 0) ptx::mbar_expect_tx(&full[st], 2 * ST_B);
            if (RES) {
              // A is resident
            } else if (A_MN) {
#pragma unroll
              for (int c = 0; c < BM / 64; ++c) {
                if (IS_BWDG) ptx::tma_load_2d_cg2(sA + c * CH_B, &mapA, &full[st], 0, wb_row(m0 + c * 64, k0, oa));
                else ptx::tma_load_2d_cg2(sA + c * CH_B, &mapA, &full[st], mA + c * 64, kA);
              }
            } else {
              ptx::tma_load_2d_cg2(sA, &mapA, &full[st], kA, mA);
            }
            if (B_MN) {
#pragma unroll
              for (int c = 0; c < BN / 128; ++c) {
                if (IS_FWD) ptx::tma_load_2d_cg2(sB + c * CH_B, &mapB, &full[st], 0,
                                                 wb_row(n0 + (crank * (BN / 128) + c) * 64, k0, ob));
                else ptx::tma_load_2d_cg2(sB + c * CH_B, &mapB, &full[st], nB + (crank * (BN / 128) + c) * 64, kB);
              }
            } else if (KIND == U_DX) {
              ptx::tma_load_2d_cg2(sB, &mapB, &full[st], 0, wb_row(k0, n0 + crank * (BN / 2), ob));
            } else {
              ptx::tma_load_2d_cg2(sB, &mapB, &full[st], kB, nB + crank * (BN / 2));
            }
            continue;
          }
          ptx::mbar_expect_tx(&full[st], ST_B);
          if (RES) {
            // A is resident
          } else if (A_MN) {
#pragma unroll
            for (int c = 0; c < BM / 64; ++c) {
              if (IS_BWDG) ptx::tma_load_2d(sA + c * CH_B, &mapA, &full[st], 0, wb_row(m0 + c * 64, k0, oa));
              else ptx::tma_load_2d(sA + c * CH_B, &mapA, &full[st], mA + c * 64, kA);
            }
          } else {
            ptx::tma_load_2d(sA, &mapA, &full[st], kA, mA);
          }
          if (B_MN) {
#pragma unroll
            for (int c = 0; c < BN / 64; ++c) {
              if (IS_FWD) ptx::tma_load_2d(sB + c * CH_B, &mapB, &full[st], 0, wb_row(n0 + c * 64, k0, ob));
              else ptx::tma_load_2d(sB + c * CH_B, &mapB, &full[st], nB + c * 64, kB);
            }
          } else if (KIND == U_DX) {
            ptx::tma_load_2d(sB, &mapB, &full[st], 0, wb_row(k0, n0, ob));
          } else {
            ptx::tma_load_2d(sB, &mapB, &full[st], kB, nB);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    if ((CG == 1 || crank == 0) && ptx::elect_one()) {   // CTA pair: the leader issues for both
      const uint32_t idesc = ptx::make_idesc_bf16(BM * CG, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
      const uint64_t hiA = A_MN ? g.desc_hi_mn : g.desc_hi_k;
      const uint64_t hiB = B_MN ? g.desc_hi_mn : g.desc_hi_k;
      const uint32_t stepA = A_MN ? g.kstep_mn : 32u;
      const uint32_t stepB = B_MN ? g.kstep_mn : 32u;
      uint32_t it = 0, lt = 0;
      if (RES && pair_id < total) ptx::mbar_wait(&wfull[0], 0);   // resident Xb landed
#ifdef ASM_TIMING
      long long t_tempty = 0, t_full = 0, t_all = clock64();
#endif
      for (int u = pair_id; u < total; u += npairs, ++lt) {
        const int z = u / tiles_mn;
        const int nk = kcount(z);
        const uint32_t a = lt & 1, aph = (lt >> 1) & 1;
#ifdef ASM_TIMING
        long long t0 = clock64();
#endif
        ptx::mbar_wait(&tempty[a], aph ^ 1);
#ifdef ASM_TIMING
        t_tempty += clock64() - t0;
#endif
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + a * BN_FULL;
        for (int ki = 0; ki < nk; ++ki, ++it) {
          const int kb = RES ? kblock(z, ki) : 0;     // only the resident-A variant addresses by kb
          const int st = it % NST;
          const uint32_t ph = (it / NST) & 1;
#ifdef ASM_TIMING
          long long t1 = clock64();
#endif
          ptx::mbar_wait(&full[st], ph);
#ifdef ASM_TIMING
          t_full += clock64() - t1;
#endif
          ptx::tc_fence_after();
          // resident A: 64-wide K blocks of 16 KB; stage kb covers K = [32 kb, 32 kb + 32)
          const uint32_t aA = RES ? ptx::smem_u32(smem + ((kb * KB) >> 6) * A_BYTES) + ((kb * KB) & 63) * 2u
                                  : ptx::smem_u32(pipe + st * ST_B);
          const uint32_t aB = ptx::smem_u32(pipe + st * ST_B) + A_ST;
#pragma unroll
          for (int kk = 0; kk < KB / 16; ++kk) {
            if (CG == 2)
              ptx::umma_bf16_cg2(d_tmem, ptx::smem_desc(hiA, aA + kk * stepA),
                                 ptx::smem_desc(hiB, aB + kk * stepB), idesc,
                                 (ki > 0 || kk > 0) ? 1u : 0u);
            else
              ptx::umma_bf16(d_tmem, ptx::smem_desc(hiA, aA + kk * stepA),
                             ptx::smem_desc(hiB, aB + kk * stepB), idesc,
                             (ki > 0 || kk > 0) ? 1u : 0u);
          }
          // frees the smem slot (in both CTAs of a pair) when these MMAs retire
          if (CG == 2) ptx::umma_commit_cg2(&empty[st]); else ptx::umma_commit(&empty[st]);
        }
        // accumulator ready for the epilogue (of both CTAs of a pair)
        if (CG == 2) ptx::umma_commit_cg2(&tfull[a]); else ptx::umma_commit(&tfull[a]);
      }
#ifdef ASM_TIMING
      if (pair_id == 0 || pair_id == npairs / 2)
        printf("TIMING kind %d pair %d tiles %u: mma warp total %lld cyc, wait tempty %lld, wait full %lld\n", KIND,
               pair_id, lt, clock64() - t_all, t_tempty, t_full);
#endif
    }
  } else if (warp == 2) {
    // ------------------------------------------------------------ DW (pairs): dW store issuer
    // One thread per column half takes the staged [32 d x 128 classes] chunks off the epilogue
    // warps' hands: it waits for a staging buffer to be full, issues its two TMA stores (even /
    // odd d rows), waits until they have READ the buffer and hands it back.  The epilogue
    // warps never wait for a store, only -- two chunks later -- for the buffer.
    if (G_::DW_TMA && g.dw_tma && lane < 2 && !ASM_DBG(g.debug_flags, 1)) {
      const int half = lane;
      const int dw_sh = g.dw_shift;
      // nothing reads dW inside the step: mark its lines evict-first so that they do not push
      // the operands the next kernels read (G'', the bf16 weights) out of L2
      uint64_t store_policy = 0;
      if (g.store_evict_first) store_policy = ptx::policy_evict_first();
      uint32_t cc = 0;
      for (int u = pair_id; u < total; u += npairs) {
        int z, m_idx, n_idx;
        decode(u, z, m_idx, n_idx);
        const int m0 = (m_idx * CG + crank) * BM, n0 = n_idx * BN;
        for (int c = 0; c < BN / 64; ++c, ++cc) {
          const uint32_t sb = cc & 1, sph = (cc >> 1) & 1;
          ptx::mbar_wait(&sfull[half * 2 + sb], sph);
          const int db = n0 + half * HC + c * 32;             // first d of the chunk
          if (db < s.D) {                                     // D % 32 == 0 in bf16 mode
            const uint8_t* src = dstg + half * 2 * DSTG + sb * DSTG;
            if (g.store_evict_first) {
              ptx::tma_store_2d_hint(&mapD, src, m0, db >> 1, store_policy);                            // even d
              ptx::tma_store_2d_hint(&mapE, src + DSTG / 2, s.C + m0 + dw_sh, db >> 1, store_policy);   // odd d
            } else {
              ptx::tma_store_2d(&mapD, src, m0, db >> 1);
              ptx::tma_store_2d(&mapE, src + DSTG / 2, s.C + m0 + dw_sh, db >> 1);
            }
            ptx::bulk_commit();
            ptx::bulk_wait_read0();
          }
          ptx::mbar_arrive(&sempty[half * 2 + sb]);
        }
      }
      ptx::bulk_wait0();
    }
  } else if (warp == 3) {
    // ------------------------------------------------------------ DW: weight-chunk producer
    // Streams the bf16 weight block of each tile ([256 d x 128 classes], needed by the
    // normalisation-Jacobian correction in the epilogue) through a 2-deep ring per column
    // half, so the epilogue never waits on a global load.
    if (KIND == U_DW && !ASM_DBG(g.debug_flags, 1) && ptx::elect_one()) {
      uint32_t cc = 0;
      for (int u = pair_id; u < total; u += npairs) {
        int z, m_idx, n_idx;
        decode(u, z, m_idx, n_idx);
        m_idx = m_idx * CG + crank;
        for (int c = 0; c < BN / 64; ++c, ++cc) {
          const uint32_t buf = cc % NWB, ph = (cc / NWB) & 1;
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            ptx::mbar_wait(&wempty[h * NWB + buf], ph ^ 1);
            ptx::mbar_expect_tx(&wfull[h * NWB + buf], WB_BUF);
            const int d0 = n_idx * BN + h * HC + c * 32;
#pragma unroll
            for (int qb = 0; qb < 2; ++qb)          // column-blocked weights: [2 blocks][32 d][64 classes]
              ptx::tma_load_2d(wbuf + (h * NWB + buf) * WB_BUF + qb * (WB_BUF / 2), &mapC, &wfull[h * NWB + buf], 0,
                               ((m_idx * BM + qb * 64) >> 6) * s.D + d0);
          }
        }
      }
    }
    if (KIND == U_DX && s.defer_loss && blockIdx.x == 0) {
      // Deferred mean loss.  One warp reproduces, bit for bit, the fixed-order reduction of
      // combine_kernel's last block: 256 strided partial sums, then the pairwise tree
      // (offsets 128, 64, 32 stay inside a lane, 16..1 go through shuffles).
      float part[8];
#pragma unroll
      for (int v = 0; v < 8; ++v) {
        float acc = 0.f;
        for (int i = v * 32 + lane; i < s.B; i += 256) acc += __ldcg(s.rowloss + i);
        part[v] = acc;
      }
#pragma unroll
      for (int o = 4; o > 0; o >>= 1)
#pragma unroll
        for (int v = 0; v < o; ++v) part[v] += part[v + o];
      float r = part[0];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) r += __shfl_down_sync(0xffffffffu, r, o);
      if (lane == 0 && s.loss) *s.loss = r * s.invB;
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------ epilogue (EPIW warps)
    const int q4 = warp & 3;                  // TMEM lane quarter this warp may access
    const int half = (warp - 4) >> 2;         // column group: which HC of the 256 accumulator columns (0..NQ-1)
    const int et = threadIdx.x - 128;         // 0 .. 32 EPIW - 1
    const int lane_row = q4 * 32 + lane;      // row of the tile owned by this thread
    const int col0 = half * HC;
    uint32_t lt = 0;
    // per-tile vectors are fetched one tile ahead into registers (pre0..2) and published to
    // shared memory at the start of their tile, so no global-load latency is exposed
    float pre0 = 0.f, pre1 = 0.f, pre2 = 0.f, pre3 = 0.f, pre4 = 0.f, pre5 = 0.f;
    // FWD: the grid is a multiple of the number of row tiles, so a CTA always works on the
    // same 128 batch rows and keeps ONE running (max, sum-exp) per thread over all its tiles
    float run_m = -INFINITY, run_z = 0.f;
    int fwd_row = -1;
    auto prefetch_tile = [&](int pu) {
      if (pu >= total) return;
      int pz, pm, pn;
      decode(pu, pz, pm, pn);
      pm = pm * CG + crank;
      if (IS_FWD) pre0 = s.inv_c[pn * BN + (et & (BN - 1))];
      if (IS_BWDG) {
        const int i = pn * BN + (et & (BN - 1));
        const bool iv = i < s.B;
        pre0 = iv ? s.negoff[i] : -INFINITY;                  // -(lse_i log2e) + log2(1/B)
        pre1 = iv ? __int_as_float(s.ylocal[i]) : __int_as_float(-1);
        pre2 = iv ? s.gtarget[i] : 0.f;
        pre3 = s.inv_c[pm * BM + lane_row];                    // 1/c of the class this thread owns next
      }
      if (IS_DW) {
        // raw loads only (no arithmetic here, so nothing waits on them until the next tile)
        const int pj = pm * BM + lane_row;
        const float* qp = s.q_part + pj;
        pre0 = qp[0];
        pre1 = s.MT > 1 ? qp[(size_t)s.Cp] : 0.f;
        pre2 = s.inv_c[pj];
        pre3 = s.MT > 2 ? qp[(size_t)2 * s.Cp] : 0.f;
        pre4 = s.MT > 3 ? qp[(size_t)3 * s.Cp] : 0.f;
        pre5 = 0.f;
        for (int t = 4; t < s.MT; ++t) pre5 += qp[(size_t)t * s.Cp];   // batches > 512 rows
      }
    };
    prefetch_tile(pair_id);
    // accumulator stage released: one arrival per warp on the (leader's) tmem-empty barrier
    auto release_acc = [&](uint32_t a) {
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (CG == 2 && crank != 0) ptx::mbar_arrive_cluster(&tempty[a], 0);
        else ptx::mbar_arrive(&tempty[a]);
      }
    };
#ifdef ASM_TIMING
    long long e_all = clock64(), e_wait = 0;
#endif
    // recompute kernel with sixteen epilogue warps: q_j of the previous tile, written one tile late
    float q_prev = 0.f;
    int q_prev_a = 0;
    long long q_prev_idx = -1;
    float* qx = reinterpret_cast<float*>(stg + 16 * 2048);   // [2 stages][2 column-group pairs][128 classes]
    for (int u = pair_id; u < total; u += npairs, ++lt) {
      int z, m_idx, n_idx;
      decode(u, z, m_idx, n_idx);
      m_idx = m_idx * CG + crank;
      const int m0 = m_idx * BM, n0 = n_idx * BN;
      const uint32_t a = lt & 1, aph = (lt >> 1) & 1;
#ifdef ASM_TIMING
      {   // time this warp would wait for the accumulator (measured before the real waits below)
        long long t0 = clock64();
        ptx::mbar_wait(&tfull[a], aph);
        e_wait += clock64() - t0;
      }
#endif
      const uint32_t taddr =
          tmem_base + (static_cast<uint32_t>(q4 * 32) << 16) + a * BN_FULL + col0;
      float* v0 = vec0 + a * BN_FULL;
      float* v1 = vec1 + a * BN_FULL;
      float* v2 = vec2 + a * BN_FULL;
      uint32_t r0[32], r1[32];
      if (ASM_DBG(g.debug_flags, 1)) {        // bring-up knob: mainloop only, no epilogue math
        ptx::mbar_wait(&tfull[a], aph);
        ptx::tc_fence_after();
        release_acc(a);
        continue;
      }

      // The four 32-column chunks of this thread's half are read with the TMEM load of
      // chunk c+1 in flight while chunk c is processed; the accumulator stage is released
      // to the MMA warp as soon as the last chunk is in registers.  The chunk body is
      // instantiated twice only (r0 / r1) to keep the kernel inside the instruction cache.
#define ASM_EPILOGUE_CHUNKS(process)                       \
      if (EPIW == 16) {                                    \
        /* two chunks per warp, one register buffer */    \
        ptx::tmem_ld32(taddr, r0);                         \
        ptx::tmem_ld_wait_dep(r0);                         \
        process(r0, 0);                                    \
        ptx::tmem_ld32(taddr + 32, r0);                    \
        ptx::tmem_ld_wait_dep(r0);                         \
        release_acc(a);                                    \
        process(r0, 1);                                    \
      } else {                                             \
      ptx::tmem_ld32(taddr, r0);                           \
      _Pragma("unroll 1")                                  \
      for (int cp = 0; cp < HC / 64; ++cp) {               \
        ptx::tmem_ld_wait_dep(r0);                         \
        ptx::tmem_ld32(taddr + cp * 64 + 32, r1);          \
        process(r0, cp * 2);                               \
        ptx::tmem_ld_wait_dep(r1);                         \
        if (cp + 1 < HC / 64) {                            \
          ptx::tmem_ld32(taddr + 64, r0);                  \
        } else {                                           \
          release_acc(a);                                  \
        }                                                  \
        process(r1, cp * 2 + 1);                           \
      }                                                    \
      }

      if (IS_FWD) {
        // ---- thread = batch row, columns = classes.  Stage 1/c_j for the tile in smem.
        if (et < BN) v0[et] = pre0;
        prefetch_tile(u + npairs);
        const int row = m0 + lane_row;
        const bool rv = row < s.B;
        const int yl = rv ? s.ylocal[row] : -1;
        const bool last_tile = n0 + BN > s.C;
        named_bar_sync(1, EPI_THREADS);
        ptx::mbar_wait(&tfull[a], aph);
        ptx::tc_fence_after();
        fwd_row = rv ? row : -1;
        auto process = [&](const uint32_t (&r)[32], int c) {
          const int cb = col0 + c * 32;              // column offset inside the tile
          const int jb = n0 + cb;
          float v[32];
#pragma unroll
          for (int b4 = 0; b4 < 8; ++b4) {
            const float4 ic = *reinterpret_cast<const float4*>(v0 + cb + b4 * 4);
            v[b4 * 4 + 0] = __uint_as_float(r[b4 * 4 + 0]) * ic.x;
            v[b4 * 4 + 1] = __uint_as_float(r[b4 * 4 + 1]) * ic.y;
            v[b4 * 4 + 2] = __uint_as_float(r[b4 * 4 + 2]) * ic.z;
            v[b4 * 4 + 3] = __uint_as_float(r[b4 * 4 + 3]) * ic.w;
          }
          // rare paths (last class tile, target column, logits requested) are kept compact
          if (last_tile) {
#pragma unroll
            for (int b = 0; b < 32; ++b)
              if (jb + b >= s.C) v[b] = -INFINITY;
          }
          const int bsel = yl - jb;
          if (bsel >= 0 && bsel < 32) {             // straight-line selects (no branch tree)
            float sv = 0.f;
#pragma unroll
            for (int b = 0; b < 32; ++b) sv = sel_eq(b, bsel, v[b], sv);
            const float fv = fwd_target(s.tgt_s, s.tgt_f, s.n, s.inv_n, s.m,
                                        step_lambda(s.lambda, s.lambda_dev), row, sv);
#pragma unroll
            for (int b = 0; b < 32; ++b) v[b] = sel_eq(b, bsel, fv, v[b]);
          }
          if (s.logits != nullptr && rv) {
            float* dst = s.logits + (size_t)row * s.C + jb;
#pragma unroll
            for (int b = 0; b < 32; ++b)
              if (jb + b < s.C) dst[b] = v[b];
          }
          float cm0 = fmaxf(v[0], v[1]), cm1 = fmaxf(v[2], v[3]);
#pragma unroll
          for (int b = 4; b < 32; b += 2) {
            cm0 = fmaxf(cm0, v[b]);
            cm1 = fmaxf(cm1, v[b + 1]);
          }
          const float cm = fmaxf(cm0, cm1);
          if (cm > -INFINITY) {
            const float nm = fmaxf(run_m, cm);
            const float nml = nm * LOG2E;
            float z0 = 0.f, z1 = 0.f, z2 = 0.f, z3 = 0.f;
#pragma unroll
            for (int b = 0; b < 32; b += 4) {
              z0 += fast_ex2(fmaf(v[b], LOG2E, -nml));
              z1 += fast_ex2(fmaf(v[b + 1], LOG2E, -nml));
              z2 += fast_ex2(fmaf(v[b + 2], LOG2E, -nml));
              z3 += fast_ex2(fmaf(v[b + 3], LOG2E, -nml));
            }
            run_z = run_z * fast_ex2((run_m - nm) * LOG2E) + ((z0 + z1) + (z2 + z3));
            run_m = nm;
          }
        };
        ASM_EPILOGUE_CHUNKS(process)
      } else if (IS_BWDG) {
        // ---- thread = class j (row m), columns = batch rows i.  Stage the per-row terms.
        if (et < BN) {
          v0[et] = pre0;
          v1[et] = pre1;
          v2[et] = pre2;
        }
        const float ic = pre3;                                // fetched one tile ahead
        prefetch_tile(u + npairs);
        const int j = m0 + lane_row;                          // class (< Cp always)
        const float icl = ic * LOG2E;
        // G'' leaves through shared memory: the four warps of a column half stage a
        // [32 rows x 128 classes] bf16 block and one thread issues a TMA store (rows >= B are
        // clipped by the hardware), so the hot loop has no global address arithmetic at all.
        // With two staging buffers per half (CTA pairs) a chunk costs ONE named barrier: the
        // leader confirms, before the barrier of chunk c, that the store of chunk c-1 has
        // drained its buffer -- the buffer chunk c+1 writes after that barrier.
        uint8_t* stg_half = stg + half * NSB * STG_HALF;
        const bool leader = (threadIdx.x == 128 + half * 128);
        named_bar_sync(1, EPI_THREADS);
        if (EPIW == 16 && q_prev_idx >= 0 && (half & 1) == 0) {
          // sixteen warps: the q_j partial of the PREVIOUS tile, own 64 columns + the neighbouring
          // column group's (left in shared memory before the barrier above): two partials per
          // batch tile as with eight warps, so the dW kernel sums the same number of them
          s.q_part[q_prev_idx] = q_prev + qx[(q_prev_a * 2 + (half >> 1)) * 128 + lane_row];
        }
        ptx::mbar_wait(&tfull[a], aph);
        ptx::tc_fence_after();
        float q0 = 0.f, q1 = 0.f, q2 = 0.f, q3 = 0.f;         // sum_i G'_ij * acc_ij  (x ic later)
        const int jw0 = m0 + q4 * 32;                         // first class of this warp
        auto process = [&](const uint32_t (&r)[32], int c) {
          const int cb = col0 + c * 32;
          const int ib = n0 + cb;                             // first batch row of the chunk
          float gq[32];
          // Target column G'_{i,y}: at most one element per batch row, and only when that row's
          // label is one of this warp's 32 classes.  A ballot makes the test warp-uniform, so the
          // hot variant of the loop carries no per-element compare at all; the patching variant
          // (same arithmetic as before, the target replaced BEFORE it enters q_j) runs rarely.
          const int ylane = __float_as_int(v1[cb + lane]);    // local class index of row ib + lane
          const bool hit = __ballot_sync(0xffffffffu, static_cast<unsigned>(ylane - jw0) < 32u) != 0u;
          auto body = [&](auto patch_tag) {
            constexpr bool PATCH = decltype(patch_tag)::value;
            // three passes over the chunk's 32 elements (exponent arguments, exponentials, products)
            // instead of one fused pass: 32 independent MUFU operations issue back to back
#pragma unroll
            for (int b4 = 0; b4 < 8; ++b4) {
              const float4 no = *reinterpret_cast<const float4*>(v0 + cb + b4 * 4);
              gq[b4 * 4 + 0] = fmaf(__uint_as_float(r[b4 * 4 + 0]), icl, no.x);
              gq[b4 * 4 + 1] = fmaf(__uint_as_float(r[b4 * 4 + 1]), icl, no.y);
              gq[b4 * 4 + 2] = fmaf(__uint_as_float(r[b4 * 4 + 2]), icl, no.z);
              gq[b4 * 4 + 3] = fmaf(__uint_as_float(r[b4 * 4 + 3]), icl, no.w);
            }
#pragma unroll
            for (int b = 0; b < 32; ++b) gq[b] = fast_ex2(gq[b]);    // softmax prob / B
            if (PATCH) {
#pragma unroll
              for (int b4 = 0; b4 < 8; ++b4) {
                const int4 yy = *reinterpret_cast<const int4*>(v1 + cb + b4 * 4);
                if (yy.x == j) gq[b4 * 4 + 0] = v2[cb + b4 * 4 + 0];   // target column: G'_{i,y}
                if (yy.y == j) gq[b4 * 4 + 1] = v2[cb + b4 * 4 + 1];
                if (yy.z == j) gq[b4 * 4 + 2] = v2[cb + b4 * 4 + 2];
                if (yy.w == j) gq[b4 * 4 + 3] = v2[cb + b4 * 4 + 3];
              }
            }
#pragma unroll
            for (int b = 0; b < 32; b += 4) {
              q0 = fmaf(gq[b + 0], __uint_as_float(r[b + 0]), q0);
              q1 = fmaf(gq[b + 1], __uint_as_float(r[b + 1]), q1);
              q2 = fmaf(gq[b + 2], __uint_as_float(r[b + 2]), q2);
              q3 = fmaf(gq[b + 3], __uint_as_float(r[b + 3]), q3);
            }
#pragma unroll
            for (int b = 0; b < 32; ++b) gq[b] *= ic;
          };
          if (hit) body(std::true_type{}); else body(std::false_type{});
          // x3: G'' leaves as two bf16 planes (value, then the rounding residual), side by side
          // along the batch dimension.  The thread's 32 batch values of this chunk are one 64-byte
          // row of the class-major staging block [128 classes][32 batch]: four 16-byte stores, the
          // 16-byte chunks XOR-swizzled by the row (CU_TENSOR_MAP_SWIZZLE_64B) so that the eight
          // lanes of a store phase hit eight different bank groups.
          const int npl = s.x3 ? 2 : 1;
#pragma unroll 1
          for (int pl = 0; pl < npl; ++pl) {
            uint32_t pk[16];
            if (NSB == 2) {
              // CTA pairs: every WARP owns two [32 classes x 32 batch] staging blocks and issues its
              // own TMA store, so the epilogue warps never wait for each other: one
              // __syncwarp per chunk instead of a 128-thread barrier.  Before block (c & 1) is
              // rewritten, lane 0 confirms that the store before last has drained it.
              // (sixteen warps: ONE block per warp -- the store before has had a whole chunk of
              //  arithmetic to drain it)
              uint8_t* sbuf = stg + (EPIW == 16 ? (warp - 4) : (warp - 4) * 2 + ((c * npl + pl) & 1)) * 2048;
              uint4* rowp = reinterpret_cast<uint4*>(sbuf + lane * 64);
              const int rsw = (lane >> 1) & 3;
              if (lane == 0) { if (EPIW == 16) ptx::bulk_wait_read0(); else ptx::bulk_wait_read1(); }
              __syncwarp();
#pragma unroll
              for (int b = 0; b < 16; ++b) {
                const __nv_bfloat162 hv = __floats2bfloat162_rn(gq[2 * b], gq[2 * b + 1]);
                pk[b] = *reinterpret_cast<const uint32_t*>(&hv);
                if (npl > 1) {
                  gq[2 * b] -= __low2float(hv);
                  gq[2 * b + 1] -= __high2float(hv);
                }
              }
#pragma unroll
              for (int qd = 0; qd < 4; ++qd)
                rowp[qd ^ rsw] = make_uint4(pk[4 * qd], pk[4 * qd + 1], pk[4 * qd + 2], pk[4 * qd + 3]);
              ptx::fence_proxy_async();                       // generic writes -> async proxy
              __syncwarp();
              if (lane == 0 && ib < s.Bp) {                   // chunks past the padded batch hold nothing
                ptx::tma_store_2d(&mapD, sbuf, ib + pl * s.Bp, m0 + q4 * 32);
                ptx::bulk_commit();
              }
            } else {
              const int rsw = (lane_row >> 1) & 3;
              uint8_t* sbuf = stg_half;
              uint4* rowp = reinterpret_cast<uint4*>(sbuf + lane_row * 64);
              if (leader) ptx::bulk_wait_read0();             // the earlier store has drained the block
              named_bar_sync(2 + half, 128);
#pragma unroll
              for (int b = 0; b < 16; ++b) {
                const __nv_bfloat162 hv = __floats2bfloat162_rn(gq[2 * b], gq[2 * b + 1]);
                pk[b] = *reinterpret_cast<const uint32_t*>(&hv);
                if (npl > 1) {
                  gq[2 * b] -= __low2float(hv);
                  gq[2 * b + 1] -= __high2float(hv);
                }
              }
#pragma unroll
              for (int qd = 0; qd < 4; ++qd)
                rowp[qd ^ rsw] = make_uint4(pk[4 * qd], pk[4 * qd + 1], pk[4 * qd + 2], pk[4 * qd + 3]);
              ptx::fence_proxy_async();
              named_bar_sync(2 + half, 128);
              if (leader && ib < s.Bp) {
                ptx::tma_store_2d(&mapC, sbuf, ib + pl * s.Bp, m0);
                ptx::bulk_commit();
              }
            }
          }
        };
        ASM_EPILOGUE_CHUNKS(process)
        if (EPIW == 16) {
          const float qv = ((q0 + q1) + (q2 + q3)) * ic;
          if (half & 1) qx[(a * 2 + (half >> 1)) * 128 + lane_row] = qv;
          q_prev = qv;
          q_prev_a = (int)a;
          q_prev_idx = (long long)(n_idx * 2 + (half >> 1)) * s.Cp + j;
        } else {
          s.q_part[(size_t)(n_idx * 2 + half) * s.Cp + j] = ((q0 + q1) + (q2 + q3)) * ic;
        }
      } else if (KIND == U_DW) {
        // ---- thread = class j, columns = d.  dW[d][j] = acc - Wb[d][j] * q_j / c_j^2
        // The q_j partials and 1/c_j were fetched one tile ahead; the bf16 weight chunks
        // arrive through the TMA ring filled by warp 3.  CTA pairs stage each
        // [32 d x 128 classes] fp32 block in shared memory (even d rows first, then the odd
        // ones) and one thread writes it with two TMA stores on the [D/2, 2C] view of the
        // caller's dW (row pitch 8C bytes is a multiple of 16 for even C: row d -> view row
        // d/2, column (d & 1) C + j); columns >= C are clipped by the tensor extent.
        const int j = m0 + lane_row;
        const bool jv = j < s.C;
        const float coef = fmaf(-(((pre0 + pre1) + (pre3 + pre4)) + pre5) * pre2, pre2, s.wd_g);   // + gscale * wd * W
        prefetch_tile(u + npairs);
        const int d_first = n0 + col0;
        const bool dw_tma = G_::DW_TMA && g.dw_tma;
        const int dw_sh = g.dw_shift;                         // 0, or 2 when C % 4 == 2
        const int dw_op = 128 - 2 * dw_sh;                    // classes per odd-row box
        const bool dw_edge = dw_sh != 0 && (lane_row < dw_sh || lane_row >= 128 - dw_sh);
        uint8_t* dstg_half = dstg + half * 2 * DSTG;
        ptx::mbar_wait(&tfull[a], aph);
        ptx::tc_fence_after();
        auto process = [&](const uint32_t (&r)[32], int c) {
          const uint32_t cc = lt * (BN / 64) + c;             // chunk counter of this half
          const uint32_t buf = cc % NWB, ph = (cc / NWB) & 1;
          const unsigned short* wsm =
              reinterpret_cast<const unsigned short*>(wbuf + (half * NWB + buf) * WB_BUF) +
              (lane_row >> 6) * (32 * 64) + (lane_row & 63);       // [2 blocks of 64 classes][32 d][64]
          ptx::mbar_wait(&wfull[half * NWB + buf], ph);
          float o[32];
#pragma unroll
          for (int b = 0; b < 32; ++b)
            o[b] = fmaf(__uint_as_float(static_cast<uint32_t>(wsm[b * 64]) << 16), coef,
                        __uint_as_float(r[b]));
          ptx::mbar_arrive(&wempty[half * NWB + buf]);       // chunk consumed (values in o[])
          const int db = d_first + c * 32;                    // first d of the chunk
          if (dw_tma) {
            // the staging buffer is free again once the stores of chunk c-2 have read it
            // (warp 2 hands it back)
            ptx::mbar_wait(&sempty[half * 2 + (cc & 1)], ((cc >> 1) & 1) ^ 1);
            float* sbe = reinterpret_cast<float*>(dstg_half + (c & 1) * DSTG) + lane_row;
            float* sbo = reinterpret_cast<float*>(dstg_half + (c & 1) * DSTG + DSTG / 2) + (lane_row - dw_sh);
#pragma unroll
            for (int b = 0; b < 32; b += 2) sbe[(b >> 1) * 128] = o[b];
            if (!dw_edge) {
#pragma unroll
              for (int b = 1; b < 32; b += 2) sbo[(b >> 1) * dw_op] = o[b];
            } else if (jv && db < s.D) {
              // odd rows start 8 bytes off a 16-byte boundary when C % 4 == 2 and a TMA store
              // must start on one: their box is shifted by two classes, and the two classes on
              // either end of the CTA's 128 are written directly by the threads that own them
              float* dst = s.dW + (size_t)(db + 1) * s.C + j;
#pragma unroll
              for (int b = 1; b < 32; b += 2) {
                *dst = o[b];
                dst += 2 * (size_t)s.C;
              }
            }
            if (dw_sh != 0 && jv && j >= s.C - 2 && db < s.D) {
              // ... and the even rows END 8 bytes off one: a box clipped there shares its last
              // 16-byte granule with classes 0 and 1 of the next (odd) row and was seen to
              // clobber them, so the even-row extent stops two classes early (umma_build_dw_maps)
              // and the last two classes are written by their owners
              float* dst = s.dW + (size_t)db * s.C + j;
#pragma unroll
              for (int b = 0; b < 32; b += 2) {
                *dst = o[b];
                dst += 2 * (size_t)s.C;
              }
            }
            ptx::fence_proxy_async();                         // generic writes -> async proxy
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&sfull[half * 2 + (cc & 1)]);    // warp 2 issues the stores
          } else if (jv && db < s.D) {
            float* dst = s.dW + (size_t)db * s.C + j;
#pragma unroll
            for (int b = 0; b < 32; ++b) {
              *dst = o[b];
              dst += s.C;
            }
          }
        };
        ASM_EPILOGUE_CHUNKS(process)
      } else if (KIND == U_DWF) {
        // ---- fp32 (x3) path: thread = class j, columns = d.  dW[d][j] = acc - W[d][j] q_j / c_j^2
        // with the fp32 weights read straight from global memory (coalesced along j).
        const int j = m0 + lane_row;
        const bool jv = j < s.C;
        const float coef = fmaf(-(((pre0 + pre1) + (pre3 + pre4)) + pre5) * pre2, pre2, s.wd_g);   // + gscale * wd * W
        prefetch_tile(u + npairs);
        const int d_first = n0 + col0;
        ptx::mbar_wait(&tfull[a], aph);
        ptx::tc_fence_after();
        auto process = [&](const uint32_t (&r)[32], int c) {
          const int db = d_first + c * 32;
          if (!jv || db >= s.D) return;
          const size_t base = (size_t)db * s.C + j;
          float w[32];
#pragma unroll
          for (int b = 0; b < 32; ++b) w[b] = __ldg(s.W + base + (size_t)b * s.C);
#pragma unroll
          for (int b = 0; b < 32; ++b)
            s.dW[base + (size_t)b * s.C] = fmaf(w[b], coef, __uint_as_float(r[b]));
        };
        ASM_EPILOGUE_CHUNKS(process)
      } else if (KIND == U_DWOPT) {
        // ---- fused optimizer: thread = class j, columns = d.  The gradient element
        // dW[d][j] = acc - W[d][j] q_j / c_j^2 (fp32 master weight) is consumed on the spot:
        // W and the optimizer state are read, updated and written back, dW never exists.
        const int j = m0 + lane_row;
        const bool jv = j < s.C;
        const float coef = -(((pre0 + pre1) + (pre3 + pre4)) + pre5) * pre2 * pre2;
        prefetch_tile(u + npairs);
        const int d_first = n0 + col0;
        const OptParams op = s.opt;
        // The weights and optimizer state are read with plain (register) loads, 16 columns at
        // a time, which alone cannot keep enough bytes in flight to HBM.  So the 128 threads of
        // a column half pull the NEXT 32-column chunk of W / state into L2 (one prefetch per
        // 128-byte line) before working on the current one: the loads that follow hit L2.
        const int ht = et & 127;
        auto prefetch_chunk = [&](int pm0, int pdb) {
          if (ASM_DBG(g.debug_flags, 16)) return;              // A/B knob: no prefetch
          // [32 d x 128 classes] fp32 per array: 4 lines per row (+1 when the row is not
          // line-aligned, covered by the first 32 threads)
          const int row = ht >> 2;
          if (pdb + row < s.D) {
            const size_t e0 = (size_t)(pdb + row) * s.C + pm0 + (ht & 3) * 32;
            if (pm0 + (ht & 3) * 32 < s.C) {
              ptx::prefetch_l2(s.Wmut + e0);
              ptx::prefetch_l2(s.opt_s0 + e0);
              if (op.kind == 2) ptx::prefetch_l2(s.opt_s1 + e0);
            }
          }
          if (ht < 32 && pdb + ht < s.D && pm0 + 127 < s.C) {
            const size_t e1 = (size_t)(pdb + ht) * s.C + pm0 + 127;
            ptx::prefetch_l2(s.Wmut + e1);
            ptx::prefetch_l2(s.opt_s0 + e1);
            if (op.kind == 2) ptx::prefetch_l2(s.opt_s1 + e1);
          }
        };
        if (lt == 0) prefetch_chunk(m0, d_first);
        int nm0 = -1, nd_first = 0;                           // first chunk of this CTA's next tile
        if (u + npairs < total) {
          int nz, nmi, nni;
          decode(u + npairs, nz, nmi, nni);
          nm0 = (nmi * CG + crank) * BM;
          nd_first = nni * BN + col0;
        }
        ptx::mbar_wait(&tfull[a], aph);
        ptx::tc_fence_after();
        auto process = [&](const uint32_t (&r)[32], int c) {
          const int db = d_first + c * 32;
          if (c < BN / 64 - 1) prefetch_chunk(m0, db + 32);
          else if (nm0 >= 0) prefetch_chunk(nm0, nd_first);
          if (!jv || db >= s.D) return;
#pragma unroll
          for (int hf = 0; hf < 2; ++hf) {                   // 16 columns at a time
            const size_t base = (size_t)(db + hf * 16) * s.C + j;
            float w[16], s0[16], s1[16];
#pragma unroll
            for (int b = 0; b < 16; ++b) {
              w[b] = s.Wmut[base + (size_t)b * s.C];
              s0[b] = s.opt_s0[base + (size_t)b * s.C];
              s1[b] = op.kind == 2 ? s.opt_s1[base + (size_t)b * s.C] : 0.f;
            }
#pragma unroll
            for (int b = 0; b < 16; ++b) {
              const float grad = fmaf(w[b], coef, __uint_as_float(r[hf * 16 + b]));
              opt_apply(op, grad, w[b], s0[b], s1[b]);
              s.Wmut[base + (size_t)b * s.C] = w[b];
              s.opt_s0[base + (size_t)b * s.C] = s0[b];
              if (op.kind == 2) s.opt_s1[base + (size_t)b * s.C] = s1[b];
            }
          }
        };
        ASM_EPILOGUE_CHUNKS(process)
      } else {  // U_DX: thread = batch row, columns = d; split-K partial
        const int row = m0 + lane_row;
        const bool rv = row < s.B;
        float* out = s.dx_part + ((size_t)z * s.B + row) * s.D + n0 + col0;
        // A thread owns a row, so a direct store instruction would write 32 separate 16-byte pieces
        // 2 KB apart.  Instead the four warps of a column half stage [128 rows x 32 d] fp32 in the
        // (otherwise unused) auxiliary region, 16-byte chunks XOR-swizzled by the row as
        // CU_TENSOR_MAP_SWIZZLE_128B expects, and one TMA store writes the block; rows past B are
        // clipped per split by the 3-D extent {D, B, KS}.
        uint8_t* dstage = smem + PIPE_B + AUX_BARS + half * (128 * 128);
        const bool leader = (threadIdx.x == 128 + half * 128);
        ptx::mbar_wait(&tfull[a], aph);
        ptx::tc_fence_after();
        auto process = [&](const uint32_t (&r)[32], int c) {
          if (g.dx_tma) {
            float4* rowp = reinterpret_cast<float4*>(dstage + lane_row * 128);
            const int sw = (ptx::smem_u32(rowp) >> 7) & 7;
#pragma unroll
            for (int qd = 0; qd < 8; ++qd)
              rowp[qd ^ sw] = make_float4(__uint_as_float(r[4 * qd]), __uint_as_float(r[4 * qd + 1]),
                                          __uint_as_float(r[4 * qd + 2]), __uint_as_float(r[4 * qd + 3]));
            ptx::fence_proxy_async();
            named_bar_sync(2 + half, 128);
            if (leader) {
              if (n0 + col0 + c * 32 < s.D) {
                ptx::tma_store_3d(&mapC, dstage, n0 + col0 + c * 32, m0, z);
                ptx::bulk_commit();
              }
              ptx::bulk_wait_read0();                          // the block is reused by the next chunk
            }
            named_bar_sync(2 + half, 128);
          } else if (rv && n0 + col0 + c * 32 < s.D) {
#pragma unroll
            for (int b = 0; b < 32; b += 4)
              *reinterpret_cast<float4*>(out + c * 32 + b) =
                  make_float4(__uint_as_float(r[b]), __uint_as_float(r[b + 1]),
                              __uint_as_float(r[b + 2]), __uint_as_float(r[b + 3]));
          }
        };
        ASM_EPILOGUE_CHUNKS(process)
      }
#undef ASM_EPILOGUE_CHUNKS
    }
    if (IS_BWDG && EPIW == 16 && lt > 0) {
      named_bar_sync(1, EPI_THREADS);                        // the last tile's neighbour partials are in place
      if (q_prev_idx >= 0 && (half & 1) == 0)
        s.q_part[q_prev_idx] = q_prev + qx[(q_prev_a * 2 + (half >> 1)) * 128 + lane_row];
    }
#ifdef ASM_TIMING
    if ((pair_id == 0 || pair_id == npairs / 2) && crank == 0 && lane == 0 && (warp == 4 || warp == 11))
      printf("TIMING kind %d pair %d warp %d: epilogue total %lld cyc, wait tfull %lld\n", KIND, pair_id, warp,
             clock64() - e_all, e_wait);
#endif
    if (IS_FWD && fwd_row >= 0)
      s.part[(size_t)fwd_row * s.NT + (pair_id / g.mt) * NQ + half] = make_float2(run_m, run_z);
  }

  if ((IS_BWDG || KIND == U_DX) && warp >= 4 && lane == 0) ptx::bulk_wait0();
  ptx::tc_fence_before();
  __syncthreads();
  if (CG == 2) ptx::cluster_sync_all();       // the peer may still be read / signalled by the leader
  if (warp == 2) {
    if (CG == 2) ptx::tmem_dealloc_cg2(tmem_base, 512); else ptx::tmem_dealloc(tmem_base, 512);
  }
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
namespace {
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) !=
          cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

// bf16 row-major [outer, inner] tensor with `pitch` elements per row; box = {box_inner, box_outer}
bool encode_map(CUtensorMap* m, const void* base, uint64_t inner, uint64_t outer, uint64_t pitch,
                uint32_t box_inner, uint32_t box_outer, bool swizzle128 = true, bool f32 = false,
                bool swizzle64 = false) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return false;
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {pitch * (f32 ? 4 : 2)};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  return fn(m, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
            const_cast<void*>(base), dims, strides, box,
            estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B
                       : (swizzle64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE),
            CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
}  // namespace

// FWD grid: a multiple of the number of 128-row tiles so each CTA keeps one set of rows
// cg = 1: one CTA per tile; cg = 2: CTA pairs (cta_group::2) on 256-row tiles.  The pair kernels
// are used per kernel kind when the M extent has at least two 128-row tiles.
static int fwd_cg(int B, int cg) { return (cg == 2 && B > BM) ? 2 : 1; }

// Tile width along N of FWD (classes), BWDG (batch rows) and DW (d): 256, or 128 when the
// tuning asks for it and the kernel runs as CTA pairs.  (Narrow tiles double the number of
// work units; see DESIGN.md section 9, wave quantisation on small shards.)
int umma_tile_width(const UmmaTuning& tu, int cg, long long units256, int num_sms) {
  if (cg != 2) return BN_FULL;                 // narrow tiles exist for the CTA-pair kernels only
  if (tu.bn == 128) return 128;
  if (tu.bn == 256) return BN_FULL;
  // auto: rounds x width over the CTA pairs, with 128-wide rounds charged 15 % extra (half the
  // operand reuse, twice the per-tile overhead -- measured: at 670 units the 256-wide tiles win
  // by 9 %, at 84 units (a 1/8 shard of config 3) the 128-wide ones do)
  const long long pairs = num_sms / 2;
  const long long r256 = (units256 + pairs - 1) / pairs * 256;
  const long long r128 = (2 * units256 + pairs - 1) / pairs * 128;
  return (double)r128 * 1.15 < (double)r256 ? 128 : BN_FULL;
}

// FWD grid: a multiple of the number of row tiles so each CTA keeps one set of rows
int umma_forward_grid(int B, int Cp, int num_sms, int cg, int bn) {
  cg = fwd_cg(B, cg);
  const int mt = ((B + BM - 1) / BM + cg - 1) / cg;      // row tiles of 128*cg rows
  const int total = mt * (Cp / bn);
  const int units = num_sms / cg;                          // CTAs or CTA pairs
  if (mt > units) return 0;
  const int g = (units / mt) * mt;
  return (g < total ? g : total) * cg;
}
// (max, sum-exp) partials per row written by FWD: one per column half per CTA of that row tile
int umma_forward_tiles(int B, int Cp, int num_sms, int cg, int bn) {
  const int c = fwd_cg(B, cg);
  const int mt = ((B + BM - 1) / BM + c - 1) / c;
  // one (max, sum-exp) partial per column group of a CTA: 2, or 4 with sixteen epilogue warps
  const int nq = (c == 2 && bn == 256 ? Geo<U_FWD, 2, 256>::EPIW : 8) / 4;
  return nq * (umma_forward_grid(B, Cp, num_sms, cg, bn) / c / mt);
}
// two q_j partials per batch tile (sixteen epilogue warps add theirs up pairwise in shared memory)
int umma_q_parts(int B, int bn, int cg) {
  (void)cg;
  return 2 * ((B + bn - 1) / bn);
}

int umma_dx_splits(int B, int D, int Cp, int num_sms, int cg) {
  const int c = fwd_cg(B, cg);
  const int tiles = (((B + BM - 1) / BM + c - 1) / c) * ((D + BN - 1) / BN);
  int ks = (num_sms / c) / tiles;
  const int kb_total = (Cp + BK - 1) / BK;
  if (ks > kb_total) ks = kb_total;
  if (ks < 1) ks = 1;
  const int kb_per = (kb_total + ks - 1) / ks;
  return (kb_total + kb_per - 1) / kb_per;       // every split non-empty
}

// fp32 [d2][d1][d0] tensor with 128-byte-swizzled boxes {32, 128, 1} (the dX partials)
static bool encode_map3_f32(CUtensorMap* m, const void* base, uint64_t d0, uint64_t d1, uint64_t d2) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return false;
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {d0 * 4, d0 * d1 * 4};
  cuuint32_t box[3] = {32, 128, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  return fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(base), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

bool umma_build_maps(UmmaMaps* m, const Step& s) {
  bool ok = true;
  // x3: the bf16 planes of each operand lie side by side along the inner dimension
  const uint64_t xd = (uint64_t)(s.x3 ? 3 : 1) * s.D;      // Xb [B, D] or [B, 3D]
  const uint64_t gp = (uint64_t)(s.x3 ? 2 : 1) * s.Bp;     // G'' pitch: [Cp, Bp] or [Cp, 2Bp] (two planes)
  const uint64_t gi = s.x3 ? gp : (uint64_t)s.B;           // inner extent (batch): clipped at B, planes at Bp
  ok &= encode_map(&m->xb_k, s.Xb, xd, s.B, xd, 64, 128);     // A of FWD  (K-major, M = batch)
  ok &= encode_map(&m->xb_k256, s.Xb, xd, s.B, xd, 64, 256);  // B of BWDG (K-major, N = batch)
  ok &= encode_map(&m->xb_mn, s.Xb, xd, s.B, xd, 64, 64);     // B of DW   (MN-major, N = d)
  // the bf16 weights, column-blocked [planes * Cp/64 * D rows][64 classes]: every box is contiguous
  const uint64_t wrows = (uint64_t)(s.x3 ? 3 : 1) * (s.Cp / 64) * s.D;
  ok &= encode_map(&m->wb_mn, s.Wb, 64, wrows, 64, 64, 64);     // B of FWD / A of BWDG (MN-major)
  ok &= encode_map(&m->wb_mn32, s.Wb, 64, wrows, 64, 64, 32);   // B of FWDR (32-deep K stages)
  ok &= encode_map(&m->wb_k, s.Wb, 64, wrows, 64, 64, 256);     // B of DX   (K-major, N = d)
  ok &= encode_map(&m->wb_k128, s.Wb, 64, wrows, 64, 64, 128);  // B half of DX in a CTA pair
  ok &= encode_map(&m->g_k, s.G, gi, s.Cp, gp, 64, 128);      // A of DW   (K-major: K = batch, M = class)
  ok &= encode_map(&m->g_mn, s.G, gi, s.Cp, gp, 64, 64);      // A of DX   (MN-major: M = batch, K = class)
  ok &= encode_map(&m->g_st, s.G, gi, s.Cp, gp, 32, 128, false, false, true);   // BWDG store (64B swizzle)
  ok &= encode_map(&m->g_st32, s.G, gi, s.Cp, gp, 32, 32, false, false, true);  // ... one warp's 32 classes
  ok &= encode_map(&m->wb_box, s.Wb, 64, wrows, 64, 64, 32, false); // DW weight chunks (two per 128 classes)
  // dX partials [KS][B][D] fp32 (D % 4 == 0, so every stride is a multiple of 16 bytes)
  m->dx_ok = encode_map3_f32(&m->dx_st, s.dx_part, (uint64_t)s.D, (uint64_t)s.B, (uint64_t)(s.KS > 0 ? s.KS : 1)) ? 1 : 0;
  return ok;
}

void umma_build_dw_maps(UmmaMaps* m, const Step& s) {
  if (m->dw_ptr == s.dW && m->dw_ptr != nullptr) return;
  m->dw_ptr = s.dW;
  m->dw_ok = 0;
  // [D/2, 2C] view: needs an even C (pitch 8C bytes % 16 == 0), an even D and a 16-byte base
  if (s.dW == nullptr || (s.C & 1) || (s.D & 1) || (reinterpret_cast<uintptr_t>(s.dW) & 15)) return;
  const uint64_t C = (uint64_t)s.C, rows = (uint64_t)s.D / 2;
  // a TMA store must start on a 16-byte boundary: odd rows begin 4C bytes into a view row, so
  // for C % 4 == 2 their box starts two classes later and is four classes narrower
  const uint32_t odd_box = (s.C & 3) ? 124 : 128;
  // ... and must not be CLIPPED off one either (see the dW epilogue): even rows stop at C - 2
  bool ok = encode_map(&m->dw_even, s.dW, (s.C & 3) ? C - 2 : C, rows, 2 * C, 128, 16, false, true);
  ok &= encode_map(&m->dw_odd, s.dW, 2 * C, rows, 2 * C, odd_box, 16, false, true);
  m->dw_ok = ok ? 1 : 0;
}

// x3 segment tables.  A contraction of two fp32 operands split as a = a0 + a1 + a2 (bf16
// planes, |a_p| <= 2^-8p |a|) keeps the plane pairs with p + q <= 2: what is dropped is below
// 2^-24 relative, the fp32 rounding level.  G'' carries two planes (its own error budget is the
// 2e-3 / cosine bar on gradients; 2^-16 is far inside it).  Segments are accumulated smallest
// term first.
static int x3_segments() {
  static int n = -1;
  if (n < 0) {
    const char* e = getenv("ASM_X3_SEGS");     // 3: (0,0),(0,1),(1,0) only (~2^-16)
    n = e ? atoi(e) : 6;
    if (n < 1) n = 1;
    if (n > 6) n = 6;
  }
  return n;
}
// pa/pb: plane of operand A / B per segment; strideA/strideB: elements per plane
static void set_segments(UmmaArgs& g, bool on, int kb_seg, const int* pa, const int* pb, int n,
                         int strideA, int strideB) {
  g.kb_seg = kb_seg;
  g.nseg = 1;
  g.segA[0] = g.segB[0] = 0;
  if (on) {
    g.nseg = n;
    for (int i = 0; i < n; ++i) {             // reversed: small terms first
      g.segA[i] = pa[n - 1 - i] * strideA;
      g.segB[i] = pb[n - 1 - i] * strideB;
    }
  }
  g.kb_total = g.nseg * kb_seg;
  g.kb_per = g.kb_total;
}
static const int kSegHi[6] = {0, 0, 1, 1, 0, 2};   // three-plane operand pairs: (x, w)
static const int kSegLo[6] = {0, 1, 0, 1, 2, 0};
static const int kSegG[5] = {0, 0, 1, 1, 0};       // two-plane G'' against a three-plane operand
static const int kSegO[5] = {0, 1, 0, 1, 2};

static UmmaArgs base_args(const UmmaTuning& tu) {
  UmmaArgs g{};
  g.desc_hi_k = ptx::make_smem_desc_hi(16, 1024);
  g.desc_hi_mn = ptx::make_smem_desc_hi(tu.mn_lbo, tu.mn_sbo);
  g.kstep_mn = tu.mn_kstep;
  g.debug_flags = tu.debug_flags;
  g.ks = 1;
  return g;
}

namespace {
template <int KIND, int CG, int BNT = BN_FULL>
cudaError_t set_smem() {
  return cudaFuncSetAttribute(umma_kernel<KIND, CG, BNT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              Geo<KIND, CG, BNT>::SMEM);
}
// launch with `units` work units (CTAs, or CTA pairs as clusters of 2)
template <int KIND, int CG, int BNT = BN_FULL>
void launch_k(int units, const CUtensorMap& a, const CUtensorMap& b, const CUtensorMap& c,
              const Step& s, const UmmaArgs& g, cudaStream_t st, const CUtensorMap* d = nullptr,
              const CUtensorMap* e = nullptr) {
  if (units <= 0) return;
  // DW follows an event record (the dX fork), everything else follows a kernel directly
  const bool pdl = s.pdl != 0 && KIND != U_DW && KIND != U_DWOPT && KIND != U_DWF;
  launch_pdl(umma_kernel<KIND, CG, BNT>, dim3(units * CG), dim3(Geo<KIND, CG, BNT>::NTHREADS), Geo<KIND, CG, BNT>::SMEM, st,
             pdl, CG, a, b, c, d ? *d : c, e ? *e : c, s, g);
}
}  // namespace

cudaError_t umma_configure() {
  cudaError_t e;
  if ((e = set_smem<U_FWD, 1>()) != cudaSuccess) return e;
  if ((e = set_smem<U_FWD, 2>()) != cudaSuccess) return e;
#ifdef ASM_BRINGUP
  if ((e = set_smem<U_FWDR, 1>()) != cudaSuccess) return e;
  if ((e = set_smem<U_FWDR, 2>()) != cudaSuccess) return e;
  if ((e = set_smem<U_BWDG1, 2>()) != cudaSuccess) return e;
#endif
  if ((e = set_smem<U_BWDG, 1>()) != cudaSuccess) return e;
  if ((e = set_smem<U_BWDG, 2>()) != cudaSuccess) return e;
  if ((e = set_smem<U_DW, 1>()) != cudaSuccess) return e;
  if ((e = set_smem<U_DW, 2>()) != cudaSuccess) return e;
  if ((e = set_smem<U_DWOPT, 1>()) != cudaSuccess) return e;
  if ((e = set_smem<U_DWOPT, 2>()) != cudaSuccess) return e;
  if ((e = set_smem<U_DWF, 1>()) != cudaSuccess) return e;
  if ((e = set_smem<U_DWF, 2>()) != cudaSuccess) return e;
  if ((e = set_smem<U_DX, 1>()) != cudaSuccess) return e;
  if ((e = set_smem<U_DX, 2>()) != cudaSuccess) return e;
  // 128-wide tiles (UmmaTuning::bn, ASM_UMMA_BN=128): CTA-pair kernels only
  if ((e = set_smem<U_FWD, 2, 128>()) != cudaSuccess) return e;
  if ((e = set_smem<U_BWDG, 2, 128>()) != cudaSuccess) return e;
  if ((e = set_smem<U_DW, 2, 128>()) != cudaSuccess) return e;
  if ((e = set_smem<U_DWOPT, 2, 128>()) != cudaSuccess) return e;
  return set_smem<U_DWF, 2, 128>();
}

void launch_umma_forward(const Step& s, const UmmaMaps& m, const UmmaTuning& tu, int num_sms,
                         cudaStream_t st) {
  UmmaArgs g = base_args(tu);   // S = Xb Wb: lanes = batch rows, columns = classes
  const int cg = fwd_cg(s.B, (tu.cg_mask & 1) ? 2 : 1);
  g.mt = ((s.B + BM - 1) / BM + cg - 1) / cg;
  const int bn = umma_tile_width(tu, cg, (long long)g.mt * (s.Cp / BN_FULL), num_sms);
  g.nt = s.Cp / bn;
  const int units = umma_forward_grid(s.B, s.Cp, num_sms, cg, bn) / cg;
  if (bn == 128) {              // narrow tiles: more units for shards that do not fill the pairs
    set_segments(g, s.x3 != 0, (s.D + BK - 1) / BK, kSegHi, kSegLo, x3_segments(), s.D, 1);
    launch_k<U_FWD, 2, 128>(units, m.xb_k, m.wb_mn, m.wb_mn, s, g, st);
    return;
  }
#ifdef ASM_BRINGUP
  if (s.D <= 512 && (tu.debug_flags & 4) && cg == 2 && !s.x3) {
    // opt-in: Xb row tiles resident in both CTAs of a pair, only the weight halves stream
    g.kb_total = (s.D + BK - 1) / BK;
    g.kb_per = g.kb_total;
    launch_k<U_FWDR, 2>(units, m.xb_k, m.wb_mn, m.wb_mn, s, g, st);
    return;
  }
  if (s.D <= 512 && (tu.debug_flags & 4) && cg == 1 && !s.x3) {   // opt-in: measured slower (55 vs 48 us)
    // Xb row tile resident in shared memory, weights stream in 32-deep K stages
    g.kb_total = (s.D + 31) / 32;
    g.kb_per = g.kb_total;
    g.desc_hi_mn = ptx::make_smem_desc_hi(Geo<U_FWDR>::CH_B, tu.mn_sbo);   // chunk stride 4 KB
    launch_k<U_FWDR, 1>(units, m.xb_k, m.wb_mn32, m.wb_mn32, s, g, st);
    return;
  }
#endif
  set_segments(g, s.x3 != 0, (s.D + BK - 1) / BK, kSegHi, kSegLo, x3_segments(), s.D, 1);
  if (cg == 2) launch_k<U_FWD, 2>(units, m.xb_k, m.wb_mn, m.wb_mn, s, g, st);
  else launch_k<U_FWD, 1>(units, m.xb_k, m.wb_mn, m.wb_mn, s, g, st);
}

void launch_umma_bwdg(const Step& s, const UmmaMaps& m, const UmmaTuning& tu, int num_sms,
                      cudaStream_t st) {
  UmmaArgs g = base_args(tu);   // recompute S^T -> G'' (bf16) + q_part: lanes = classes
  const int cg = (tu.cg_mask & 2) ? 2 : 1;
  g.mt = s.Cp / (BM * cg);
  const int bn = umma_tile_width(tu, cg, (long long)g.mt * ((s.B + BN_FULL - 1) / BN_FULL), num_sms);
  g.nt = (s.B + bn - 1) / bn;
  // A = weights, B = embeddings: the same plane pairs with the roles swapped
  set_segments(g, s.x3 != 0, (s.D + BK - 1) / BK, kSegLo, kSegHi, x3_segments(), 1, s.D);
  g.rev = tu.l2_order ? 1 : 0;  // the forward kernel swept the classes upwards: start where it stopped
  const int units = min(g.mt * g.nt, num_sms / cg);
  if (bn == 128) launch_k<U_BWDG, 2, 128>(units, m.wb_mn, m.xb_mn, m.g_st, s, g, st, &m.g_st32);   // X box: 64 rows per CTA
#ifdef ASM_BRINGUP
  else if (cg == 2 && (tu.debug_flags & 8)) launch_k<U_BWDG1, 2>(units, m.wb_mn, m.xb_k, m.g_st, s, g, st);
#endif
  else if (cg == 2) launch_k<U_BWDG, 2>(units, m.wb_mn, m.xb_k, m.g_st, s, g, st, &m.g_st32);
  else launch_k<U_BWDG, 1>(units, m.wb_mn, m.xb_k256, m.g_st, s, g, st);
}

void launch_umma_dw(const Step& s, const UmmaMaps& m, const UmmaTuning& tu, int num_sms,
                    cudaStream_t st) {
  UmmaArgs g = base_args(tu);   // dW^T = G''^T Xb - correction: lanes = classes, columns = d
  const int cg = (tu.cg_mask & 4) ? 2 : 1;
  g.mt = s.Cp / (BM * cg);
  const int bn = umma_tile_width(tu, cg, (long long)g.mt * ((s.D + BN_FULL - 1) / BN_FULL), num_sms);
  g.nt = (s.D + bn - 1) / bn;
  set_segments(g, s.x3 != 0, (s.B + BK - 1) / BK, kSegG, kSegO, x3_segments() < 5 ? x3_segments() : 5,
               s.Bp, s.D);
  const int units = min(g.mt * g.nt, num_sms / cg);
  // upwards again (BWDG went down): the first class tiles are the ones BWDG wrote last
  g.dw_tma = (tu.dw_tma && cg == 2 && s.opt.kind == 0 && !s.x3 && m.dw_ok && m.dw_ptr == s.dW) ? 1 : 0;
  g.dw_shift = (s.C & 3) ? 2 : 0;
  g.store_evict_first = (tu.l2_hints & 2) ? 1 : 0;
  if (bn == 128) {
    if (s.opt.kind != 0) launch_k<U_DWOPT, 2, 128>(units, m.g_k, m.xb_mn, m.wb_box, s, g, st);
    else if (s.x3) launch_k<U_DWF, 2, 128>(units, m.g_k, m.xb_mn, m.wb_box, s, g, st);
    else launch_k<U_DW, 2, 128>(units, m.g_k, m.xb_mn, m.wb_box, s, g, st, &m.dw_even, &m.dw_odd);
    return;
  }
  if (s.opt.kind == 0 && s.x3) {
    if (cg == 2) launch_k<U_DWF, 2>(units, m.g_k, m.xb_mn, m.wb_box, s, g, st);
    else launch_k<U_DWF, 1>(units, m.g_k, m.xb_mn, m.wb_box, s, g, st);
    return;
  }
  if (s.opt.kind != 0) {
    if (cg == 2) launch_k<U_DWOPT, 2>(units, m.g_k, m.xb_mn, m.wb_box, s, g, st);
    else launch_k<U_DWOPT, 1>(units, m.g_k, m.xb_mn, m.wb_box, s, g, st);
  } else {
    if (cg == 2) launch_k<U_DW, 2>(units, m.g_k, m.xb_mn, m.wb_box, s, g, st, &m.dw_even, &m.dw_odd);
    else launch_k<U_DW, 1>(units, m.g_k, m.xb_mn, m.wb_box, s, g, st);
  }
}

void launch_umma_dx(const Step& s, const UmmaMaps& m, const UmmaTuning& tu, int num_sms,
                    cudaStream_t st) {
  UmmaArgs g = base_args(tu);   // dX partials = G'' Wb^T, split over the classes
  const int cg = fwd_cg(s.B, (tu.cg_mask & 8) ? 2 : 1);
  g.mt = ((s.B + BM - 1) / BM + cg - 1) / cg;
  g.nt = (s.D + BN - 1) / BN;
  set_segments(g, s.x3 != 0, (s.Cp + BK - 1) / BK, kSegG, kSegO, x3_segments() < 5 ? x3_segments() : 5,
               s.Bp, 1);
  g.ks = s.KS;
  g.kb_per = (g.kb_total + g.ks - 1) / g.ks;
  if (tu.l2_order && !s.x3) {   // all splits sweep the classes together, downwards (DW went up) --
    g.kstride = 1;              // or upwards WITH it when the two kernels share the SMs (num_sms < all)
    g.rev = tu.side_by_side ? 0 : 1;
  }
  const int units = min(g.mt * g.nt * g.ks, num_sms / cg);
  g.dx_tma = (tu.dw_tma && m.dx_ok) ? 1 : 0;
  if (cg == 2) launch_k<U_DX, 2>(units, m.g_mn, m.wb_k128, m.dx_st, s, g, st);
  else launch_k<U_DX, 1>(units, m.g_mn, m.wb_k, m.dx_st, s, g, st);
}

}  // namespace asmh
