/*
 * asoftmax_b200.h -- C ABI of the B200-native A-softmax (SphereFace angular-margin) head.
 *
 * Drop-in boundary for the classifier-FC + softmax-CE slot of medivhna/TF_Face_Toolbox.
 * The reference has no C/FFI boundary (SURVEY.md section 8b): its boundary is the Python
 * method contract between the tower wrapper and the Network object.  Each entry point
 * below names the reference interface it replaces:
 *
 *   asm_create / asm_destroy     the `classifier/fc_classifier` variable scope + graph build
 *                                of the head        nets/sphere.py:84-90, data_parallel.py:215-224
 *   asm_forward_backward         forward(images, labels, num_classes=..) -> logits,
 *                                loss_function(scope, labels, **logits) -> losses,
 *                                tf.gradients(total_loss, params)
 *                                                   data_parallel.py:220, :223, :32-38
 *   asm_forward                  the forward half only (loss + optional logits)
 *                                                   nets/sphere.py:78-95, :103-118
 *   asm_forward_partial /        one class shard's share of the same step; they replace the
 *   asm_backward_partial         replicated-FC gradient all-reduce nccl.all_sum(grads)
 *                                                   data_parallel.py:175-181
 *   asm_lambda                   the lambda-annealing schedule driven by global_step
 *                                                   train.py:157, data_parallel.py:252-253
 *
 * Conventions: every function returns 0 (ASM_OK) or a negative asm_status; nothing throws
 * or aborts.  All buffers are DEVICE pointers, caller-owned and borrowed for the duration
 * of the stream-ordered work.  Calls are asynchronous on `cuda_stream` (a cudaStream_t
 * passed as void*); the caller synchronises.  One handle per (device, shard); a handle is
 * not thread-safe, distinct handles are independent.  Layouts follow the reference:
 * X [B, D] row-major fp32, W / dW [D, C_local] row-major fp32 (tf fully_connected [in,out],
 * nets/sphere.py:86), labels [B] int32 (data.py:259) or int64.
 */
#ifndef ASOFTMAX_B200_H_
#define ASOFTMAX_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct asm_head asm_head; /* opaque */

typedef enum {
  ASM_OK = 0,
  ASM_ERR_INVALID_ARG = -1,   /* bad shape / NULL pointer / unsupported m or mode */
  ASM_ERR_CUDA = -2,          /* a CUDA runtime / driver call failed (see asm_last_error) */
  ASM_ERR_NO_DEVICE = -3,     /* no sm_100 device: there is NO CPU fallback */
  ASM_ERR_LABEL_RANGE = -4,   /* a label was outside [0, C_total) (asm_check_labels) */
  ASM_ERR_ALLOC = -5,
  ASM_ERR_PEER_TIMEOUT = -6   /* NVLink transport: a peer did not publish in time (asm_p2p_status) */
} asm_status;

enum { ASM_MODE_FP32 = 0, ASM_MODE_BF16 = 1 };

typedef struct {
  int32_t D;             /* embedding dim (512 in every BASELINE config)            */
  int32_t C_total;       /* num_classes (data.py:54)                                */
  int32_t C_local;       /* classes owned by this shard                             */
  int32_t class_offset;  /* shard owns [class_offset, class_offset + C_local)       */
  int32_t B_max;         /* largest (global) batch this handle will see             */
  int32_t m;             /* margin, 1..4                                            */
  int32_t mode;          /* ASM_MODE_BF16: X, W rounded to bf16 (RNE), fp32 accumulate (D % 64 == 0).
                            ASM_MODE_FP32: all 24 significand bits of X and W are used -- on the
                            tensor cores through an exact three-plane bf16 split when D % 64 == 0,
                            on CUDA cores otherwise (D % 16 == 0). */
  int32_t rank, world;   /* informational; world == 1 -> single shard               */
  void*   nccl_comm;     /* reserved, must be NULL: collectives are issued by the
                            host between asm_forward_partial / asm_backward_partial */
} asm_config;

/* Bytes of device workspace asm_create will allocate for cfg (0 on invalid cfg). */
size_t asm_workspace_bytes(const asm_config* cfg);

int asm_create(asm_head** out, const asm_config* cfg);
int asm_destroy(asm_head* h);

/* Last error text for this handle (or for a failed asm_create when h == NULL). */
const char* asm_last_error(const asm_head* h);

/* lambda(it) = max(lambda_min, base * (1 + gamma*it)^(-power)), it counted from 1. */
float asm_lambda(int64_t iteration, float base, float gamma, float power, float lambda_min);

/*
 * Whole step on one shard that owns every class (world == 1).
 *   X        [B, D] fp32                       labels [B] int32 (label_bytes 4) or int64 (8)
 *   W        [D, C_local] fp32 master weights  lambda  host scalar (asm_lambda)
 *   loss_out device float: mean over the batch of softmax-CE on the margin logits
 *   logits_out_or_null  [B, C_local] fp32 margin-modified logits f, or NULL (bench path:
 *                       the logit matrix is never written to HBM)
 *   dX [B, D] fp32, dW [D, C_local] fp32  (gradients of loss_out)
 */
int asm_forward_backward(asm_head* h, const float* X, int32_t B,
                         const void* labels, int32_t label_bytes, const float* W,
                         float lambda, float* loss_out, float* logits_out_or_null,
                         float* dX, float* dW, void* cuda_stream);

/* Forward only: loss (+ optional logits). world == 1. */
int asm_forward(asm_head* h, const float* X, int32_t B, const void* labels,
                int32_t label_bytes, const float* W, float lambda, float* loss_out,
                float* logits_out_or_null, void* cuda_stream);

/*
 * Class-sharded step, phase 1.  X / labels are the GATHERED global batch (all B rows);
 * W is this shard's [D, C_local] slice.  Writes stats_out [3, B] fp32:
 *   row 0: local max_j f_ij   row 1: local sum_j exp(f_ij - max)   row 2: f_{i,y_i} if this
 *   shard owns class y_i else 0.
 * The host all-gathers stats_out over the shards ([world, 3, B]) and calls phase 2.
 */
int asm_forward_partial(asm_head* h, const float* X, int32_t B, const void* labels,
                        int32_t label_bytes, const float* W, float lambda,
                        float* stats_out, float* logits_out_or_null, void* cuda_stream);

/*
 * Phase 2.  stats_all [n_shards, 3, B] fp32 (this shard's own stats included).  Must
 * follow asm_forward_partial on the same handle / stream with the same X, labels, W.
 *   loss_out   device float, global-batch mean loss (identical on every shard)
 *   dX_partial [B, D] fp32: this shard's contribution; sum over shards (reduce-scatter)
 *              gives dX.  The r_i * x_i term is added by the shard that owns class y_i.
 *   dW         [D, C_local] fp32: complete for this shard -- no collective on dW.
 */
int asm_backward_partial(asm_head* h, const float* stats_all, int32_t n_shards,
                         float* loss_out, float* dX_partial, float* dW, void* cuda_stream);

/* Synchronises `cuda_stream` and reports whether the last step saw a label outside
 * [0, C_total): ASM_OK or ASM_ERR_LABEL_RANGE.  (Out-of-range labels never fault the
 * kernels: the row is treated as having no target on this shard.) */
int asm_check_labels(asm_head* h, void* cuda_stream);

/* Number of kernels the last asm_* step call launched on its stream (for bench.py). */
int asm_last_launch_count(const asm_head* h);

/*
 * Fused classifier optimizer (SURVEY.md section 8f rank 1).  Replaces, for the classifier
 * variable, `opt.apply_gradients(grads)` of data_parallel.py:186-196 --
 * MomentumOptimizer(lr, momentum=0.9) or AdamOptimizer(lr, beta1=0.5, beta2=0.999) -- applied to
 * the gradient of cross_entropy + reg_loss (L2 regulariser wd * 0.5 * |W|^2, nets/sphere.py:88).
 * While an optimizer is armed (kind != ASM_OPT_NONE) every step call UPDATES `W` IN PLACE in the
 * epilogue of the dW kernel (the `const` on W is waived), `dW` is not written and may be NULL,
 * and state0 / state1 ([D, C_local] fp32, caller-owned, zero-initialised by the caller) hold the
 * momentum accumulator, or Adam's m and v.  Pass opt == NULL or kind == ASM_OPT_NONE to disarm.
 *   momentum: accum = momentum*accum + g;  W -= lr*accum              (g = dW + wd*W)
 *   adam:     m = b1*m + (1-b1)*g;  v = b2*v + (1-b2)*g*g;
 *             W -= lr*sqrt(1-b2^t)/(1-b1^t) * m/(sqrt(v)+eps),  t = opt->step (from 1)
 */
enum { ASM_OPT_NONE = 0, ASM_OPT_MOMENTUM = 1, ASM_OPT_ADAM = 2 };
typedef struct {
  int32_t kind;
  float   lr, momentum, beta1, beta2, epsilon, weight_decay;
  int64_t step;
} asm_optimizer;
int asm_set_optimizer(asm_head* h, const asm_optimizer* opt, float* state0, float* state1);

/*
 * Center loss (loss.py:29-45; SURVEY.md section 8f rank 2), sharded by class like W.
 *   loss      = mean(square(features - centers[labels]))   over B*D, with the PRE-update centers
 *   centers   = scatter_sub(centers, labels, (1 - alpha) * (centers[labels] - features))
 *               (duplicate labels accumulate), updated in place
 *   dX_accum += weight * 2 (features - centers[labels]) / (B*D)       (optional, may be NULL)
 * A shard only touches rows whose label lies in [class_offset, class_offset + C_local); its
 * loss_out is that shard's partial sum / (B*D) (sum the shards' values).  `scratch` is a
 * caller-owned device buffer of asm_center_scratch_bytes(B) bytes (3 B + 4 words: row losses, the
 * label-sorted row order, segment lengths, a ticket) that is ZERO on first use.  B <= 4096,
 * D % 4 == 0.  Two launches: a one-block shared-memory sort of (label, row) that turns duplicate
 * labels into contiguous segments, and one block per segment that reads its center row once, every
 * member row once, and writes the center row once.  Deterministic (no float atomics; duplicates
 * are summed in row order).  Stateless: no handle needed.
 */
size_t asm_center_scratch_bytes(int32_t B);
int asm_center_loss(const float* X, int32_t B, int32_t D, const void* labels, int32_t label_bytes,
                    float* centers, int32_t C_local, int32_t class_offset, float alpha,
                    float weight, float* loss_out, float* dX_accum_or_null, float* scratch,
                    void* cuda_stream);

/*
 * NVLink peer-memory transport of the class-sharded step: the whole step of one rank --
 * gather of X / labels, statistics exchange, dX reduce-scatter included -- in ONE call, with
 * no NCCL launch: the head's kernels read the peers' symmetric buffers over NVLink (P2P loads)
 * and synchronise with release/acquire flags.  Replaces asm_forward_partial + host
 * collectives + asm_backward_partial (and with them nccl.all_sum, data_parallel.py:175-181).
 *   asm_p2p_bytes   bytes of peer-mapped ("symmetric") device memory every rank must provide
 *                   for cfg (B_max = largest GLOBAL batch; cfg->world ranks)
 *   asm_p2p_attach  peer_bases[world]: the device address, valid on THIS rank, of every rank's
 *                   block (own rank included).  The blocks must be zero-filled before the
 *                   first step of any rank (e.g. zero + barrier on the host).
 *   asm_step_p2p    X_local [b_local, D] / labels_local [b_local]: this rank's rows (every
 *                   rank passes the same b_local; global batch = b_local * world);
 *                   W / dW: this shard's [D, C_local]; loss_out: global mean loss;
 *                   dX_local [b_local, D]: the complete gradient of this rank's rows.
 * Asynchronous on cuda_stream and capturable into a CUDA graph (the step counter lives on the
 * device).  Seven kernel launches per step, none of them transport-only: the norm kernel publishes
 * and gathers the rows, the statistics exchange rides in the combine kernel, the dX exchange in
 * the dX-finish kernel.  Ranks must stay in lock-step (every rank calls asm_step_p2p once per
 * step).  A wait for a peer gives up after the configured time (default 60 s, env
 * ASM_P2P_TIMEOUT_MS or asm_p2p_set_timeout; 0 = wait for ever): nothing traps and the CUDA
 * context stays usable, but that step's results are undefined and asm_p2p_status -- which
 * synchronises the stream -- returns ASM_ERR_PEER_TIMEOUT from then on.
 */
size_t asm_p2p_bytes(const asm_config* cfg);
int asm_p2p_attach(asm_head* h, void* const* peer_bases);
int asm_step_p2p(asm_head* h, const float* X_local, int32_t b_local, const void* labels_local,
                 int32_t label_bytes, const float* W, float lambda, float* loss_out,
                 float* dX_local, float* dW, void* cuda_stream);
int asm_p2p_set_timeout(asm_head* h, int32_t milliseconds);
int asm_p2p_status(asm_head* h, void* cuda_stream);

/*
 * Gradient transform and regularisation loss, at no extra pass over [D, C].  The reference's
 * towers differentiate total_loss = cross_entropy + reg_loss and scale every gradient by
 * mult_lr / num_gpus (data_parallel.py:32-38, :224; reg_loss = wd/2 |W|^2 from the contrib
 * l2_regularizer, nets/sphere.py:88, nets/net_base.py:103-107).  Once set, every step call
 * returns  dX := grad_scale * dX,  dW := grad_scale * (dW + weight_decay * W)  (the scale rides in
 * the softmax-gradient offset, the weight-decay term in the dW epilogue's per-class coefficient)
 * and, when reg_loss_out is not NULL, writes  weight_decay/2 * sum over this shard's classes of
 * |w_j|^2  to that device float (the column sums of squares are a by-product of the norm kernel;
 * deterministic).  loss_out stays the unscaled loss (asm_set_loss).  Defaults: 1, 0, NULL.  With a
 * fused optimizer armed the optimizer's own weight_decay applies instead of this one.
 */
int asm_set_gradient_transform(asm_head* h, float grad_scale, float weight_decay, float* reg_loss_out);

/*
 * Element type of the embeddings handed to the step calls: 4 = fp32 (default, what the reference's
 * backbones emit), 2 = bf16 (ASM_MODE_BF16 only).  With 2, every X / X_local pointer is a bf16
 * [B, D] array: the norm kernel skips the rounding it would do itself, the r_i x_i term of dX reads
 * the bf16 rows, and the NVLink transport publishes and gathers half the bytes.  dX stays fp32.
 */
int asm_set_embedding_dtype(asm_head* h, int32_t bytes_per_element);

/*
 * Margin of the target logit, per handle; it applies to every step call (asm_forward_backward,
 * asm_forward, asm_forward_partial / asm_backward_partial, asm_step_p2p) and, like the other
 * per-handle settings, is captured with them into a CUDA graph.
 *   ASM_MARGIN_ASOFTMAX (default)  SphereFace: f_y = (lambda s_y + n psi(t)) / (1 + lambda) on the
 *                                  raw embeddings, margin cfg.m.
 *   ASM_MARGIN_ADDITIVE            L2-normalised embeddings, fixed scale s:  s_ij = s x_i.w_j / (n_i c_j),
 *                                  t = s_iy / s,  f_y = s phi(t),  every other logit s_ij, where
 *                                  phi(t) = cos(theta + m2) - m3        if t >= cos(pi - m2)
 *                                         = t - m2 sin(m2) - m3          otherwise (no "easy margin").
 *                                  m2 = 0: CosFace (s (cos theta - m3)); m3 = 0: ArcFace
 *                                  (s cos(theta + m2)).  lambda and cfg.m are ignored.
 * margin == NULL restores the default.  s must be finite and > 0, m2 in [0, pi/2], m3 finite and
 * >= 0; anything else returns ASM_ERR_INVALID_ARG and changes nothing.
 */
enum { ASM_MARGIN_ASOFTMAX = 0, ASM_MARGIN_ADDITIVE = 1 };
typedef struct {
  int32_t kind;
  float   s, m2, m3;
} asm_margin;
int asm_set_margin(asm_head* h, const asm_margin* margin);

/*
 * Loss applied to the head's logits f (the margin logits of whichever margin is set), per handle;
 * like the margin it applies to every step call and is captured with them into a CUDA graph.
 *   ASM_LOSS_SOFTMAX_CE (default)  L = mean_i (lse_i - f_iy), the softmax cross-entropy.
 *   ASM_LOSS_FOCAL                 L = mean_i gamma (1 - p_iy)^alpha (lse_i - f_iy),
 *                                  p_iy = softmax(f_i)_{y_i}: the reference's focal_loss (loss.py).
 *                                  The names follow the reference, not Lin et al.: gamma is the
 *                                  multiplier and alpha the exponent.  The gradient differentiates
 *                                  through (1 - p)^alpha (no stop-gradient): every row's softmax
 *                                  gradient is multiplied by
 *                                  w_i = gamma ((1 - p)^alpha + alpha p (1 - p)^(alpha - 1) ce_i).
 * loss_out (asm_forward included) receives the loss selected here; grad_scale, weight_decay and
 * reg_loss_out (asm_set_gradient_transform) apply to it as to the cross-entropy.  loss == NULL
 * restores the default.  gamma must be finite and > 0, alpha finite and >= 0; anything else returns
 * ASM_ERR_INVALID_ARG and changes nothing.
 */
enum { ASM_LOSS_SOFTMAX_CE = 0, ASM_LOSS_FOCAL = 1 };
typedef struct {
  int32_t kind;
  float   gamma, alpha;
} asm_loss;
int asm_set_loss(asm_head* h, const asm_loss* loss);

/* CUDA-graph support.  Kernel arguments are frozen when a step is captured into a graph, so
 * lambda (which anneals per step) can instead be read from a caller-owned DEVICE float:
 * once set (non-NULL) it overrides the by-value `lambda` argument of every step call; NULL
 * restores the by-value behaviour.  All step calls are capturable (no synchronisation, no
 * allocation) as long as asm_check_labels / profiling are not used inside the capture. */
int asm_set_lambda_device(asm_head* h, const float* lambda_dev);

/* Per-kernel device timing for bench.py's roofline: when enabled (1) every kernel of a step is
 * bracketed by CUDA events on the step's stream, which also puts them all on that one stream,
 * one after the other.  enable == 2 records events only between PHASES -- norm kernel, forward
 * kernel, combine, recompute kernel, then the dW kernel next to the dX branch as one phase -- and
 * leaves the real schedule (side stream, dW and dX on disjoint CTA pairs) in place.  asm_get_profile synchronises on the last
 * event and writes up to max_n durations (ms) and 32-byte NUL-terminated kernel names;
 * returns the number written (>= 0) or a negative asm_status. */
int asm_set_profiling(asm_head* h, int enable);
int asm_get_profile(asm_head* h, int32_t max_n, float* ms_out, char* names_out);

/* Version / build info string, e.g. "asoftmax_b200 0.1 sm_100a". */
const char* asm_version(void);

#ifdef __cplusplus
}
#endif
#endif /* ASOFTMAX_B200_H_ */
