// Kernel launchers shared between translation units of libasoftmax_b200.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "asm_common.cuh"

namespace asmh {

// Everything one step needs; filled by the host API (asm_api.cu), passed by value.
// Fused classifier optimizer (asm_set_optimizer): the update the reference applies with
// MomentumOptimizer(lr, 0.9) / AdamOptimizer(lr, beta1=0.5, beta2=0.999)
// (data_parallel.py:186-196) to the L2-regularised gradient (nets/sphere.py:88), executed in
// the epilogue of the dW kernel so that dW never goes to HBM.
struct OptParams {
  int kind;                  // 0 = off, 1 = momentum, 2 = adam
  float lr;                  // momentum: lr; adam: lr * sqrt(1 - b2^t) / (1 - b1^t)
  float mu, b1, b2, eps, wd;
};
__host__ __device__ inline void opt_apply(const OptParams& o, float grad, float& w, float& s0,
                                          float& s1) {
  const float g = grad + o.wd * w;               // + d(reg_loss)/dw = wd * w
  if (o.kind == 1) {
    s0 = o.mu * s0 + g;                          // accum = momentum * accum + grad
    w -= o.lr * s0;                              // var  -= lr * accum
  } else {
    s0 = o.b1 * s0 + (1.0f - o.b1) * g;
    s1 = o.b2 * s1 + (1.0f - o.b2) * g * g;
#ifdef __CUDA_ARCH__
    w -= o.lr * s0 / (sqrtf(s1) + o.eps);
#else
    w -= o.lr * s0 / (sqrtf(s1) + o.eps);
#endif
  }
}

// Loss on the logits (asm_set_loss): kind 0 = softmax cross-entropy, 1 = the reference's focal
// loss gamma (1 - p_y)^alpha CE (gamma the multiplier, alpha the exponent; DESIGN.md section 2.2).
struct LossParams {
  int kind;
  float gamma, alpha;
};

// NVLink peer-memory transport of the class-sharded step (asm_p2p.cu)
constexpr int kMaxPeers = 8;
constexpr int kFlagStride = 16;        // flag words per phase
struct P2P {
  int rank, world, b_local, b_max, B_max, D;
  unsigned* step_dev;                  // device counter: steps this rank has COMPLETED
  unsigned* err_dev;                   // 0, or 0x80000000 | phase << 8 | src of the first wait that timed out
  unsigned* tickets;                   // [4] last-block-done tickets of the producing kernels
  int waiters;                         // blocks per exchange kernel that may wait for peers (ASM_P2P_WAITERS)
  unsigned long long timeout_ns;       // per-wait limit (0 = wait for ever)
  char* base[kMaxPeers];               // every rank's symmetric block (own included)
  size_t off_x, off_y, off_st, off_dx, off_fl;
  // per step (caller buffers of this rank)
  const float* x_local;                // [b_local, D]
  const void* y_local;                 // [b_local]
  int y_bytes;
  float* dx_local;                     // [b_local, D]
  float* Xg;                           // [B, D] gathered embeddings (workspace; dx_finish reads them)
  __host__ __device__ float* x(int r, int par) const {
    return reinterpret_cast<float*>(base[r] + off_x) + (size_t)par * b_max * D;
  }
  __host__ __device__ int* y(int r, int par) const {
    return reinterpret_cast<int*>(base[r] + off_y) + (size_t)par * b_max;
  }
  __host__ __device__ float* st(int r, int par) const {
    return reinterpret_cast<float*>(base[r] + off_st) + (size_t)par * 3 * B_max;
  }
  __host__ __device__ float* dx(int r, int par) const {
    return reinterpret_cast<float*>(base[r] + off_dx) + (size_t)par * B_max * D;
  }
  __host__ __device__ unsigned* flags_of(int r) const {
    return reinterpret_cast<unsigned*>(base[r] + off_fl);
  }
  __host__ __device__ unsigned* flags_local() const { return flags_of(rank); }
};

// Launch with the programmatic-stream-serialization attribute when `pdl` is set (never while
// the stream is being captured into a graph): the kernel may start while its predecessor
// drains, and orders itself with pdl_wait().
template <typename... KArgs, typename... Args>
inline void launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                       bool pdl, int cluster, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int n = 0;
  if (cluster > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = cluster;
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    ++n;
  }
  if (pdl) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n;
  cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

constexpr int kRowTileHost = 128;   // == asmh::kRowTile (asm_common.cuh)

struct Step {
  // problem
  int B, D, C, Cp, C_total, class_offset, m, mode;
  float lambda, invB;
  const float* lambda_dev;   // optional device scalar overriding `lambda` (CUDA-graph replay)
  // gradient transform (asm_set_gradient_transform): dX, dW come out as
  // gscale * (d loss / d.) and dW additionally carries gscale * weight_decay * W -- what
  // tf.gradients(cross_entropy + reg_loss) * mult_lr / num_gpus yields (data_parallel.py:32-38)
  float gscale;              // 1 by default
  float wd_g;                // gscale * weight_decay (0 by default)
  float reg_scale;           // 0.5 * weight_decay: reg_loss = reg_scale * ||W||^2 (contrib l2_regularizer)
  float* reg_out;            // device scalar receiving reg_loss of this shard's classes, or null
  float* wsq_part;           // [W-role blocks of the norm kernel] partial sums of w^2
  unsigned int* wsq_ticket;  // [1]
  // caller buffers (device)
  const float* X;            // [B, D] fp32, or bf16 when x_bf16 (bf16 mode only)
  int x_bf16;
  const float* W;            // [D, C]
  float* logits;             // [B, C] or null
  float* dX;                 // [B, D]
  float* dW;                 // [D, C]
  float* loss;               // scalar
  // workspace (device)
  int* ylocal;               // [B]   y - class_offset if owned, -1 if another shard's, -2 if out of range
  int* flags;                // [1]   (unused)
  float* n;                  // [B]
  float* inv_n;              // [B]
  float* inv_c;              // [Cp]  1/||w_j|| (0 on pad columns)
  float* tgt_s;              // [B]   s_{i,y} (owner shard only)
  float* tgt_f;              // [B]   f_{i,y}
  float2* part;              // [B, NT] per-column-tile (max, sumexp)
  int NT;                    // number of column tiles of the forward kernel
  float* stats_local;        // [3, B]
  float* lse;                // [B]   M_i + log Z_i (global)
  float* negoff;             // [B]   -(lse_i * log2 e) + log2(gscale/B) (+ log2 w_i, focal): exp2 offset of the backward
  float* gtarget;            // [B]   G'_{i,y_i}
  float* rcoef;              // [B]   r_i  (0 if not owned)
  float* rowloss;            // [B]   lse_i - f_{i,y}  (focal: gamma (1 - p_iy)^alpha (lse_i - f_{i,y}))
  unsigned int* counter;     // [1]   last-block-done ticket of the combine kernel
  float* q_part;             // [MT, Cp] column sums  sum_i G'_ij s_ij per 128-row group
  int MT;
  void* G;                   // G'' = G' * inv_c: tcgen05 paths bf16 CLASS-major [Cp, Bp] ([Cp, 2Bp] when x3); CUDA-core path fp32 [B, Cp]
  int Bp;                    // batch pitch of the class-major G'': B rounded up to 64
  float* dx_part;            // [KS, B, D] split-K partials of dX
  int KS;
  __nv_bfloat16* Xb;         // [B, D]    bf16 mode;  [B, 3D]  (three planes side by side) when x3
  __nv_bfloat16* Wb;         // bf16 mode: column-blocked [planes][Cp/64][D][64], planes = 3 when x3
  // x3 = 1: fp32 mode on the tensor cores.  Every fp32 operand is split exactly into bf16
  // planes (v = p0 + p1 + p2, p0 = bf16(v), p1 = bf16(v - p0), ...) stored side by side along
  // the inner dimension; a contraction runs as a chain of plane-pair segments accumulated in
  // the same fp32 TMEM tile.  G'' then has two planes: [B, 2Cp] bf16.
  int x3;
  OptParams opt;             // fused optimizer (kind 0 = off: dW is written instead)
  float* Wmut;               // [D, C]  W, updated in place when opt.kind != 0
  float* opt_s0;             // [D, C]  momentum accumulator / adam m
  float* opt_s1;             // [D, C]  adam v
  int l2_hints;              // evict-first on single-use streams (the fp32 W read of the norm kernel)
  int pdl;                   // launch dependents programmatically (eager, non-captured streams)
  int defer_loss;            // the mean-loss reduction runs in an idle warp of the dX kernel, not in combine
  // margin of the target logit (asm_set_margin).  Additive kind: the norm kernel writes the operand
  // copies of s * x_i / n_i (n, inv_n and X stay the true embeddings, for dx_finish), the forward
  // patches s * phi(t) in, combine sets G'_y = g_y phi'(t) and r = 0, dx_finish projects each row.
  Margin mg;
  float* Xs;                 // [B, D] fp32 s * x_i / n_i: what the CUDA-core kernels read in place of X (additive kind)
  // loss on the logits (asm_set_loss).  Read by the combine kernels only (row_epilogue): focal
  // loss multiplies every row's softmax gradient by one scalar w_i, which rides in negoff, gtarget,
  // rcoef and rowgrad, so no GEMM kernel sees it.
  LossParams ls;
  float* rowgrad;            // [B]   invB * gscale * w_i: the CUDA-core recompute's per-row gradient factor
  // [Cp] per-class scale of the normalisation term of dW: coef_j = -q_j wcorr_j^2 + wd_g.  inv_c for
  // A-softmax and the additive margin; an all-zero array for the linear kind, whose dW has no such term.
  const float* wcorr;
};

// prep: column norms of W (+ bf16 copy), row norms of X (+ bf16 copy), label localisation.
// With a transport (p != null): the same launch also publishes this rank's rows to its peers
// and its embedding role gathers every rank's rows over NVLink as it normalises them.
void launch_prep(const Step& s, const void* labels, int label_bytes, cudaStream_t st, const P2P* p = nullptr);
// NVLink transport: statistics of this shard -> symmetric block, exchange, global combine (one launch)
void launch_combine_p2p(const Step& s, const P2P& p, cudaStream_t st);
// NVLink transport: dX contribution of this shard -> symmetric block, exchange, sum of this rank's rows (one launch)
void launch_dx_finish_p2p(const Step& s, const P2P& p, cudaStream_t st);
// combine per-tile (max,sumexp) partials into stats_local [3,B]
void launch_combine_local(const Step& s, cudaStream_t st);
// combine [n_shards,3,B] stats into lse / loss / target coefficients
void launch_combine_global(const Step& s, const float* stats_all, int n_shards, cudaStream_t st);
// single shard: both of the above in one launch (partials -> stats_local, lse, loss, ...)
void launch_combine_fused(const Step& s, cudaStream_t st);
// dX = sum_z dx_part[z] + r_i x_i; additive kind: dX_i = (s/n_i)(v_i - (x_i.v_i)/n_i^2 x_i), v_i = sum_z dx_part[z]
void launch_dx_finish(const Step& s, cudaStream_t st);
// streaming classifier update from a dW buffer (alternative to the fused dW epilogue)
void launch_opt_stream(const Step& s, const float* dW, cudaStream_t st);

// force the lazy loading of every kernel the NVLink-transport step can launch (asm_p2p_attach)
void p2p_preload_kernels();
void prep_preload_kernels();
void simt_preload_kernels();

// fp32 (CUDA-core) contractions with fused epilogues
void launch_simt_forward(const Step& s, cudaStream_t st);
void launch_simt_bwdg(const Step& s, cudaStream_t st);   // recompute S -> G'' + q_part
void launch_simt_dw(const Step& s, cudaStream_t st);
void launch_simt_dx(const Step& s, cudaStream_t st);
int simt_forward_tiles(int C);                               // NT for the fp32 path
int simt_dx_splits(int B, int D, int Cp);

// bf16 (tcgen05 / TMEM / TMA) contractions with fused epilogues
struct UmmaMaps {            // TMA descriptors over the bf16 workspace operands
  CUtensorMap xb_k, xb_k256, xb_mn, wb_mn, wb_k, wb_k128, g_k, g_mn, g_st, g_st32, wb_box;
  // the caller's dW [D, C] fp32 seen as [D/2, 2C] (row pitch 8C bytes): even rows through a
  // tensor of extent {C, D/2}, odd rows through one of extent {2C, D/2} at column offset C
  CUtensorMap dw_even, dw_odd;
  CUtensorMap dx_st;         // the dX split-K partials [KS][B][D] fp32 as a 3-D tensor (store, 128B swizzle)
  int dx_ok;
  const void* dw_ptr;        // buffer the two maps above were encoded for (re-encoded when it changes)
  int dw_ok;                 // 0: dW cannot be addressed by TMA (odd C, misaligned base): direct stores
};
struct UmmaTuning {          // schedule of the tcgen05 kernels, per handle (defaults in asm_head, overridden by ASM_* knobs)
  uint32_t cg_mask;          // CTA pairs (cta_group::2) per kernel: bit0 FWD, bit1 BWDG, bit2 DW, bit3 DX
  uint32_t bn;               // tile width along N of FWD / BWDG / DW: 0 = chosen per launch from the unit count, 128, 256 (ASM_UMMA_BN)
  uint32_t l2_order;         // consecutive kernels sweep the classes in opposite directions (ASM_L2_ORDER=0 disables)
  uint32_t dw_tma;           // dW leaves through shared memory + TMA stores (ASM_DW_TMA=0: direct stores)
  uint32_t side_by_side;     // per step: dW and dX run concurrently on disjoint SMs (ASM_DW_PAIRS)
  uint32_t l2_hints;         // evict-first on single-use streams: bit0 the fp32 W read of the norm kernel, bit1 the dW stores (ASM_L2_HINTS)
};
struct UmmaArgs {
  int mt, nt, ks, kb_total, kb_per;
  // plane-pair segments of the K loop (x3): K block kb belongs to segment kb / kb_seg, whose
  // operands start segA / segB elements further along the inner dimension of their tensors
  int nseg, kb_seg;
  int segA[6], segB[6];
  uint64_t desc_hi_k, desc_hi_mn;
  uint32_t kstep_mn;
  int rev;                   // class tiles (or, with kstride, K blocks) in descending order
  int kstride;               // split-K: split z takes K blocks z, z + ks, ... instead of a contiguous range
  int dw_tma;                // DW: staged TMA stores (maps D / E valid)
  int dx_tma;                // DX: staged TMA stores of the split-K partials (map C valid)
  int dw_shift;              // DW: class offset of the odd-row boxes (2 when C % 4 == 2, else 0)
  int store_evict_first;     // DW: the dW stores carry an evict-first L2 policy
};
cudaError_t umma_configure();
bool umma_build_maps(UmmaMaps* m, const Step& s);
// (re-)encode the dW store maps for this step's output buffer; sets m->dw_ok
void umma_build_dw_maps(UmmaMaps* m, const Step& s);
// tile width along N of a CTA-pair kernel with `units256` 256-wide work units (0 / auto, 128 or 256 by tu.bn)
int umma_tile_width(const UmmaTuning& tu, int cg, long long units256, int num_sms);
int umma_forward_tiles(int B, int Cp, int num_sms, int cg, int bn = 256);
int umma_forward_grid(int B, int Cp, int num_sms, int cg, int bn = 256);
int umma_q_parts(int B, int bn, int cg);
int umma_dx_splits(int B, int D, int Cp, int num_sms, int cg);
void launch_umma_forward(const Step& s, const UmmaMaps& m, const UmmaTuning& tu, int num_sms,
                         cudaStream_t st);
void launch_umma_bwdg(const Step& s, const UmmaMaps& m, const UmmaTuning& tu, int num_sms,
                      cudaStream_t st);
void launch_umma_dw(const Step& s, const UmmaMaps& m, const UmmaTuning& tu, int num_sms,
                    cudaStream_t st);   // dW, or the fused optimizer update when s.opt.kind != 0
void launch_umma_dx(const Step& s, const UmmaMaps& m, const UmmaTuning& tu, int num_sms,
                    cudaStream_t st);

}  // namespace asmh
