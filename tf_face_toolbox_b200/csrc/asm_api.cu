// C ABI of libasoftmax_b200 (see include/asoftmax_b200.h): handle, workspace carving and
// the stream-ordered launch sequence of one A-softmax head step.  No CPU fallback: without
// an sm_100 device asm_create fails with ASM_ERR_NO_DEVICE.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>
#include <vector>

#include "../../include/asoftmax_b200.h"
#include "asm_kernels.cuh"

using namespace asmh;

struct asm_head {
  asm_config cfg;
  int device = 0;
  int num_sms = 148;
  int Cp = 0;
  int NT = 0;
  char* ws = nullptr;            // single device allocation
  size_t ws_bytes = 0;
  Step st{};                     // pointers into ws + per-step state
  size_t dx_part_capacity = 0;   // floats
  UmmaMaps maps{};
  int maps_B = -1;               // (B, KS) the maps were encoded for: dx_st's extent is {D, B, KS}
  int maps_KS = -1;
  bool opt_stream = false;       // ASM_OPT_STREAM=1: dW kernel + streaming update instead of the fused epilogue (opt-in)
  float* dw_scratch = nullptr;   // [D, C_local] fp32, allocated on first use of opt_stream
  bool defer_loss = true;        // ASM_DEFER_LOSS=0: combine reduces the loss itself (A/B knob)
  bool tc = false;               // tcgen05 kernels (bf16 mode, or fp32 mode through bf16 planes)
  UmmaTuning tune{15, 0, 1, 1, 0, 3};   // CTA pairs on all four kernels (ASM_UMMA_CG=0: single-CTA)
  bool fwd_valid = false;
  // dX branch of the backward (DX + dx_finish) runs on a second stream so that it fills the
  // SMs the DW kernel's tail leaves idle; both only depend on G'' from the BWDG kernel
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  bool overlap = true;           // ASM_NO_OVERLAP=1 disables
  int dw_pairs = 0;              // > 0: the dW kernel runs on this many CTA pairs and the dX kernel, concurrently, on the
                                 // remaining ones (ASM_DW_PAIRS): both read G'' and the bf16 weights, class tile by class tile
  bool pdl = true;               // programmatic dependent launch between the step's kernels (ASM_PDL=0 disables)
  // NVLink peer-memory transport (asm_p2p_attach / asm_step_p2p)
  P2P p2p{};
  bool p2p_ready = false;
  float* Xg = nullptr;           // [B_max, D] gathered embeddings
  float* wzero = nullptr;        // [Cp] zeros (workspace): Step::wcorr of the linear kind
  int launches = 0;
  // optional per-kernel timing (asm_set_profiling): event i is recorded before kernel i
  bool profiling = false;
  bool phase_profiling = false;  // asm_set_profiling(h, 2): events only where the main stream serialises anyway, so the
                                 // real schedule (side stream, dW next to dX) is what gets timed
  static constexpr int kMaxMarks = 16;
  cudaEvent_t ev[kMaxMarks + 1] = {};
  const char* mark_name[kMaxMarks] = {};
  int n_marks = 0;
  char err[512];
};

namespace {
thread_local char g_create_err[512] = "";

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct Layout {
  size_t ylocal, flags, n, inv_n, inv_c, margin, tgt_s, tgt_f, part, stats_local, lse, negoff, gtarget, rcoef, rowloss, rowgrad, counter,
      q_part, G, dx_part, Xb, Wb, Xs, Xg, step_dev, wsq_part, wsq_ticket, wzero, total;
  int Cp, NT, MT;
  size_t dx_capacity;
};

bool valid_cfg(const asm_config* c) {
  if (!c) return false;
  if (c->D <= 0 || c->D % 16 != 0) return false;
  if (c->C_total <= 0 || c->C_local <= 0 || c->class_offset < 0) return false;
  if ((long long)c->class_offset + c->C_local > c->C_total) return false;
  if (c->B_max <= 0 || c->m < 1 || c->m > 4) return false;
  if (c->mode != ASM_MODE_FP32 && c->mode != ASM_MODE_BF16) return false;
  if (c->mode == ASM_MODE_BF16 && c->D % 64 != 0) return false;
  if (c->world < 1 || c->rank < 0 || c->rank >= c->world) return false;
  if (c->nccl_comm != nullptr) return false;
  return true;
}

// fp32 mode runs on the tensor cores (operands split into bf16 planes, "x3") whenever the
// tcgen05 tiling applies; ASM_FP32_SIMT=1 forces the CUDA-core kernels.
bool use_x3(const asm_config& c) {
  if (c.mode != ASM_MODE_FP32 || c.D % 64 != 0) return false;
  const char* e = getenv("ASM_FP32_SIMT");
  return !(e && atoi(e) != 0);
}
bool use_tc(const asm_config& c) { return c.mode == ASM_MODE_BF16 || use_x3(c); }

Layout make_layout(const asm_config& c, int num_sms) {
  Layout L{};
  const bool tc = use_tc(c);
  const size_t planes = use_x3(c) ? 3 : 1;
  const size_t B = c.B_max, D = c.D;
  L.Cp = (int)align_up(c.C_local, 256);
  L.NT = (L.Cp + 127) / 128;
  if (L.NT < 2 * num_sms) L.NT = 2 * num_sms;   // tcgen05 forward: 2 partials per CTA
  L.MT = 2 * (int)((B + 127) / 128);      // two per batch tile, down to 128-row tiles
  if (L.MT < 4 * (int)((B + 255) / 256)) L.MT = 4 * (int)((B + 255) / 256);   // four per 256-row tile (sixteen epilogue warps)
  // dX split-K partial capacity: the larger of both paths at B_max, but never less than
  // what a single 128-row tile would use (KS grows when B shrinks).
  const int ks_simt = simt_dx_splits(c.B_max, c.D, L.Cp);
  const int ks_umma = umma_dx_splits(c.B_max, c.D, L.Cp, num_sms, 1);
  const int ks_one = tc ? umma_dx_splits(128, c.D, L.Cp, num_sms, 1)
                        : simt_dx_splits(128, c.D, L.Cp);
  const size_t cap_full = (size_t)(tc ? ks_umma : ks_simt) * B * D;
  const size_t cap_one = (size_t)ks_one * (B < 128 ? B : 128) * D;
  L.dx_capacity = cap_full > cap_one ? cap_full : cap_one;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  L.ylocal = take(B * 4);
  L.flags = take(256);
  L.n = take(B * 4);
  L.inv_n = take(B * 4);
  L.inv_c = take((size_t)L.Cp * 4);
  L.margin = take(kMarginRecordFloats * 4);   // must directly precede tgt_s (margin_record)
  L.tgt_s = take(B * 4);
  L.tgt_f = take(B * 4);
  L.part = take(B * (size_t)L.NT * 8);
  L.stats_local = take(3 * B * 4);
  L.lse = take(B * 4);
  L.negoff = take(B * 4);
  L.gtarget = take(B * 4);
  L.rcoef = take(B * 4);
  L.rowloss = take(B * 4);
  L.counter = take(256);
  L.wsq_part = take(((size_t)L.Cp / 32 + 16) * 4);    // one partial per W-role block of the norm kernel
  L.wsq_ticket = take(256);
  L.q_part = take((size_t)L.MT * L.Cp * 4);
  L.G = take(align_up(B, 64) * (size_t)L.Cp * (c.mode == ASM_MODE_BF16 ? 2 : 4));   // fp32 mode: two bf16 planes, or fp32 on the CUDA-core path
  L.dx_part = take(L.dx_capacity * 4);
  if (tc) {
    L.Xb = take(planes * B * D * 2);
    L.Wb = take(planes * D * (size_t)L.Cp * 2);
  } else {
    L.Xs = take(B * D * 4);   // the CUDA-core kernels' scaled, normalised copy of X (additive margin)
  }
  if (c.world > 1) {
    L.Xg = take(B * D * 4);
    L.step_dev = take(256);
  }
  L.rowgrad = take(B * 4);   // last: every buffer before it keeps the offset it had without it
  L.wzero = take((size_t)L.Cp * 4);   // zeroed once, never written: the linear kind's dW correction scale
  L.total = off;
  return L;
}

int fail(asm_head* h, int code, const char* fmt, const char* detail) {
  char* dst = h ? h->err : g_create_err;
  snprintf(dst, 512, fmt, detail ? detail : "");
  return code;
}

#define CU_TRY(h, expr)                                                         \
  do {                                                                          \
    cudaError_t e__ = (expr);                                                   \
    if (e__ != cudaSuccess) return fail(h, ASM_ERR_CUDA, #expr ": %s", cudaGetErrorString(e__)); \
  } while (0)

// Counts a kernel launch and, when profiling, records the event that precedes it.
void mark(asm_head* h, const char* name, cudaStream_t stream, bool phase_start = true) {
  h->launches += 1;
  if (h->phase_profiling && !phase_start) return;      // inside a phase: no event
  if (h->profiling && h->n_marks < asm_head::kMaxMarks) {
    cudaEventRecord(h->ev[h->n_marks], stream);
    h->mark_name[h->n_marks] = name;
    h->n_marks += 1;
  }
}
void mark_end(asm_head* h, cudaStream_t stream) {
  if (h->profiling) cudaEventRecord(h->ev[h->n_marks], stream);
}

int check_launch(asm_head* h, const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    snprintf(h->err, 512, "%s: %s", what, cudaGetErrorString(e));
    return ASM_ERR_CUDA;
  }
  return ASM_OK;
}

// SMs given to the dW and to the dX kernel (all of them to each unless the two are meant to run
// side by side: dX forked to the side stream AND a pair split configured)
bool split_active(const asm_head* h) {
  return h->dw_pairs > 0 && h->overlap && (!h->profiling || h->phase_profiling) && h->side != nullptr && h->tc &&
         (h->tune.cg_mask & 12) == 12;
}
int dw_sms(const asm_head* h) { return split_active(h) ? 2 * h->dw_pairs : h->num_sms; }
int dx_sms(const asm_head* h) { return split_active(h) ? h->num_sms - 2 * h->dw_pairs : h->num_sms; }

// The CUDA-core kernels read their embedding operand from s.X in place: with the additive margin
// that operand is the scaled, normalised copy Xs the norm kernel wrote.
Step simt_step(const Step& s) {
  Step t = s;
  if (s.mg.kind == kMarginAdditive) t.X = s.Xs;
  return t;
}

// forward half up to stats_local; shared by every entry point
int run_forward(asm_head* h, const float* X, int B, const void* labels, int label_bytes,
                const float* W, float lambda, float* logits, bool want_local_stats,
                cudaStream_t stream, const P2P* tp = nullptr) {
  if (!h) return ASM_ERR_INVALID_ARG;
  if (!X || !labels || !W) return fail(h, ASM_ERR_INVALID_ARG, "null input pointer%s", "");
  if (B <= 0 || B > h->cfg.B_max) return fail(h, ASM_ERR_INVALID_ARG, "B out of range%s", "");
  if (label_bytes != 4 && label_bytes != 8)
    return fail(h, ASM_ERR_INVALID_ARG, "label_bytes must be 4 or 8%s", "");
  if (!(lambda >= 0.f)) return fail(h, ASM_ERR_INVALID_ARG, "lambda must be >= 0%s", "");
  Step& s = h->st;
  s.B = B;
  s.lambda = lambda;
  s.invB = 1.0f / (float)B;
  s.Bp = (int)align_up((size_t)B, 64);
  s.X = X;
  s.W = W;
  s.logits = logits;
  s.l2_hints = (h->tune.l2_hints & 1) ? 1 : 0;
  {
    // BWDG geometry: class tiles of 256 (per CTA pair) x batch tiles; it writes one q partial per
    // column half of a batch tile
    const int bcg = (h->tune.cg_mask & 2) ? 2 : 1;
    const long long bunits = (long long)(s.Cp / (128 * bcg)) * ((B + 255) / 256);
    s.MT = h->tc ? umma_q_parts(B, umma_tile_width(h->tune, bcg, bunits, h->num_sms), bcg)
                 : (B + kRowTileHost - 1) / kRowTileHost;
  }
  h->launches = 0;
  h->n_marks = 0;
  {
    // no programmatic edges inside a graph capture, none while per-kernel events are recorded
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(stream, &cs);
    s.pdl = (h->pdl && !h->profiling && cs == cudaStreamCaptureStatusNone) ? 1 : 0;
  }
  h->fwd_valid = false;
  if (h->tc) {
    if ((B + 127) / 128 > h->num_sms)
      return fail(h, ASM_ERR_INVALID_ARG, "batch too large for the tcgen05 forward grid%s", "");
    {
      const int fcg = (h->tune.cg_mask & 1) ? 2 : 1;
      // narrow tiles only with CTA pairs, and the forward pairs need at least two row tiles
      const int ecg = (fcg == 2 && B > 128) ? 2 : 1;
      const long long funits = (long long)(((B + 127) / 128 + ecg - 1) / ecg) * (s.Cp / 256);
      s.NT = umma_forward_tiles(B, s.Cp, h->num_sms, fcg, umma_tile_width(h->tune, ecg, funits, h->num_sms));
    }
    s.KS = umma_dx_splits(B, s.D, s.Cp, dx_sms(h), (h->tune.cg_mask & 8) ? 2 : 1);
    while (s.KS > 1 && (size_t)s.KS * B * s.D > h->dx_part_capacity) --s.KS;
    // KS changes at a fixed B when profiling toggles the dW / dX split (dx_sms): a stale dx_st
    // extent would drop the stores of the splits past the old KS without an error
    if (h->maps_B != B || h->maps_KS != s.KS) {
      if (!umma_build_maps(&h->maps, s))
        return fail(h, ASM_ERR_CUDA, "cuTensorMapEncodeTiled failed%s", "");
      h->maps_B = B;
      h->maps_KS = s.KS;
    }
  } else {
    s.NT = simt_forward_tiles(s.C);
    s.KS = simt_dx_splits(B, s.D, s.Cp);
  }
  while (s.KS > 1 && (size_t)s.KS * B * s.D > h->dx_part_capacity) --s.KS;
  mark(h, "prep_norms", stream);
  launch_prep(s, labels, label_bytes, stream, tp);
  mark(h, "fwd_logits_stats", stream);
  if (h->tc) launch_umma_forward(s, h->maps, h->tune, h->num_sms, stream);
  else launch_simt_forward(simt_step(s), stream);
  if (want_local_stats) {
    mark(h, "combine_local", stream);
    launch_combine_local(s, stream);
  }
  mark_end(h, stream);
  int rc = check_launch(h, "forward launch");
  if (rc == ASM_OK) h->fwd_valid = true;
  return rc;
}

int run_backward(asm_head* h, const float* stats_all, int n_shards, float* loss_out,
                 float* dX, float* dW, bool grads, cudaStream_t stream, const P2P* tp = nullptr) {
  Step& s = h->st;
  s.loss = loss_out;
  s.dX = dX;
  s.dW = dW;
  s.Wmut = const_cast<float*>(s.W);       // only written when an optimizer is armed
  const bool tc = h->tc;
  s.defer_loss = (grads && tc && h->defer_loss) ? 1 : 0;   // the tcgen05 dX kernel reduces the loss
  if (tp) {
    mark(h, "combine_exchange", stream);
    launch_combine_p2p(s, *tp, stream);
  } else if (stats_all) {
    // profiling: the gap between the two halves is the host-side statistics all-gather
    if (h->profiling && h->n_marks > 0 && h->n_marks < asm_head::kMaxMarks)
      h->mark_name[h->n_marks++] = "stats_exchange_host";
    mark(h, "combine_global", stream);
    launch_combine_global(s, stats_all, n_shards, stream);
  } else {
    mark(h, "combine_stats", stream);
    launch_combine_fused(s, stream);
  }
  if (grads) {
    h->tune.side_by_side = split_active(h) ? 1 : 0;
    mark(h, "bwd_recompute_g", stream);
    if (tc) launch_umma_bwdg(s, h->maps, h->tune, h->num_sms, stream);
    else launch_simt_bwdg(simt_step(s), stream);
    // The CUDA-core dX kernel reads the fp32 master weights, which a fused optimizer rewrites in
    // the dW kernel: in that combination dX runs first, on the same stream (the tcgen05 kernels
    // read the bf16 copy, which the update never touches, so they may overlap).
    const bool dx_first = !tc && s.opt.kind != 0;
    // the per-kernel profile needs one stream; otherwise fork the dX branch
    const bool fork = h->overlap && (!h->profiling || h->phase_profiling) && h->side != nullptr && !dx_first;
    cudaStream_t sx = stream;
    if (fork) {
      cudaEventRecord(h->ev_fork, stream);
      cudaStreamWaitEvent(h->side, h->ev_fork, 0);
      sx = h->side;
    }
    auto run_dx = [&]() {
      mark(h, "dx_gemm", sx, !h->phase_profiling);
      if (tc) launch_umma_dx(s, h->maps, h->tune, dx_sms(h), sx);
      else launch_simt_dx(simt_step(s), sx);
      const bool add = s.mg.kind == kMarginAdditive;
      mark(h, tp ? (add ? "dx_finish_margin_exchange" : "dx_finish_exchange") : (add ? "dx_finish_margin" : "dx_finish"), sx,
           !h->phase_profiling);
      if (tp) launch_dx_finish_p2p(s, *tp, sx);
      else launch_dx_finish(s, sx);
    };
    if (dx_first) run_dx();
    mark(h, h->phase_profiling ? "dw+dx+dx_finish (side by side)" : "dw_gemm", stream);
    if (tc && s.opt.kind != 0 && h->opt_stream) {
      // opt-in alternative to the fused epilogue: plain dW into a scratch buffer, then one
      // streaming pass over (dW, W, state)
      if (!h->dw_scratch &&
          cudaMalloc(&h->dw_scratch, (size_t)s.D * h->cfg.C_local * sizeof(float)) != cudaSuccess) {
        cudaGetLastError();
        h->dw_scratch = nullptr;
        return fail(h, ASM_ERR_ALLOC, "cudaMalloc(dW scratch for ASM_OPT_STREAM)%s", "");
      }
      Step t = s;
      t.opt.kind = 0;
      t.dW = h->dw_scratch;
      launch_umma_dw(t, h->maps, h->tune, h->num_sms, stream);
      mark(h, "opt_stream", stream);
      launch_opt_stream(s, h->dw_scratch, stream);
    } else if (tc) {
      if (s.opt.kind == 0 && !s.x3 && h->tune.dw_tma) umma_build_dw_maps(&h->maps, s);
      launch_umma_dw(s, h->maps, h->tune, dw_sms(h), stream);
    } else launch_simt_dw(simt_step(s), stream);
    if (!dx_first) run_dx();
    if (fork) {
      cudaEventRecord(h->ev_join, h->side);
      cudaStreamWaitEvent(stream, h->ev_join, 0);
    }
  }
  mark_end(h, stream);
  return check_launch(h, "backward launch");
}
}  // namespace

extern "C" {

const char* asm_version(void) { return "asoftmax_b200 0.3 sm_100a"; }

float asm_lambda(int64_t iteration, float base, float gamma, float power, float lambda_min) {
  const double v = (double)base * pow(1.0 + (double)gamma * (double)iteration, -(double)power);
  return (float)(v > (double)lambda_min ? v : (double)lambda_min);
}

size_t asm_workspace_bytes(const asm_config* cfg) {
  if (!valid_cfg(cfg)) return 0;
  return make_layout(*cfg, 148).total;
}

int asm_create(asm_head** out, const asm_config* cfg) {
  if (!out) return fail(nullptr, ASM_ERR_INVALID_ARG, "out is NULL%s", "");
  *out = nullptr;
  if (!valid_cfg(cfg)) return fail(nullptr, ASM_ERR_INVALID_ARG, "invalid asm_config%s", "");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(nullptr, ASM_ERR_NO_DEVICE, "no CUDA device (this library has no CPU fallback)%s", "");
  }
  int dev = 0, major = 0, sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess)
    return fail(nullptr, ASM_ERR_CUDA, "cudaGetDevice failed%s", "");
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (major != 10)
    return fail(nullptr, ASM_ERR_NO_DEVICE, "device is not sm_100 (Blackwell B200) %s", "");
  asm_head* h = new (std::nothrow) asm_head();
  if (!h) return fail(nullptr, ASM_ERR_ALLOC, "host allocation failed%s", "");
  h->cfg = *cfg;
  h->device = dev;
  h->num_sms = sms > 0 ? sms : 148;
  h->err[0] = 0;
  const char* e;
  if ((e = getenv("ASM_L2_ORDER"))) h->tune.l2_order = atoi(e) != 0;
  if ((e = getenv("ASM_DW_TMA"))) h->tune.dw_tma = atoi(e) != 0;
  if ((e = getenv("ASM_L2_HINTS"))) h->tune.l2_hints = (uint32_t)atoi(e);
  if ((e = getenv("ASM_UMMA_CG"))) h->tune.cg_mask = (uint32_t)atoi(e);
  if ((e = getenv("ASM_UMMA_BN"))) h->tune.bn = (uint32_t)atoi(e);   // 128 / 256: force the tile width
  if ((e = getenv("ASM_NO_OVERLAP")) && atoi(e)) h->overlap = false;
  // default: 57 % of the CTA pairs to the (HBM-bound) dW kernel, the rest to the (tensor-bound) dX
  // kernel -- measured at config 3: 252.8 us per step one after the other, 235.5 us side by side
  h->dw_pairs = (h->num_sms / 2) * 42 / 74;
  if ((e = getenv("ASM_DW_PAIRS"))) h->dw_pairs = atoi(e);
  if (h->dw_pairs < 0 || h->dw_pairs >= h->num_sms / 2) h->dw_pairs = 0;
  if ((e = getenv("ASM_PDL"))) h->pdl = atoi(e) != 0;
  if ((e = getenv("ASM_DEFER_LOSS"))) h->defer_loss = atoi(e) != 0;
  if ((e = getenv("ASM_OPT_STREAM"))) h->opt_stream = atoi(e) != 0;
  if (cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming) != cudaSuccess) {
    cudaGetLastError();
    h->side = nullptr;
  }
  const Layout L = make_layout(*cfg, h->num_sms);
  cudaError_t ce = cudaMalloc(&h->ws, L.total);
  if (ce != cudaSuccess) {
    fail(nullptr, ASM_ERR_ALLOC, "cudaMalloc(workspace): %s", cudaGetErrorString(ce));
    delete h;
    return ASM_ERR_ALLOC;
  }
  h->ws_bytes = L.total;
  cudaMemset(h->ws, 0, L.total);
  h->tc = use_tc(*cfg);
  if (h->tc) {
    ce = umma_configure();
    if (ce != cudaSuccess) {
      fail(nullptr, ASM_ERR_CUDA, "cudaFuncSetAttribute(smem): %s", cudaGetErrorString(ce));
      cudaFree(h->ws);
      delete h;
      return ASM_ERR_CUDA;
    }
  }
  Step& s = h->st;
  s.D = cfg->D;
  s.C = cfg->C_local;
  s.Cp = L.Cp;
  s.C_total = cfg->C_total;
  s.class_offset = cfg->class_offset;
  s.m = cfg->m;
  s.mode = cfg->mode;
  s.x3 = use_x3(*cfg) ? 1 : 0;
  char* w = h->ws;
  s.ylocal = (int*)(w + L.ylocal);
  s.flags = (int*)(w + L.flags);
  s.n = (float*)(w + L.n);
  s.inv_n = (float*)(w + L.inv_n);
  s.inv_c = (float*)(w + L.inv_c);
  s.tgt_s = (float*)(w + L.tgt_s);
  s.tgt_f = (float*)(w + L.tgt_f);
  s.part = (float2*)(w + L.part);
  s.stats_local = (float*)(w + L.stats_local);
  s.lse = (float*)(w + L.lse);
  s.negoff = (float*)(w + L.negoff);
  s.gtarget = (float*)(w + L.gtarget);
  s.rcoef = (float*)(w + L.rcoef);
  s.rowloss = (float*)(w + L.rowloss);
  s.rowgrad = (float*)(w + L.rowgrad);
  h->wzero = (float*)(w + L.wzero);
  s.wcorr = s.inv_c;
  s.counter = (unsigned int*)(w + L.counter);
  s.q_part = (float*)(w + L.q_part);
  s.wsq_part = (float*)(w + L.wsq_part);
  s.wsq_ticket = (unsigned int*)(w + L.wsq_ticket);
  s.gscale = 1.0f;
  s.wd_g = 0.0f;
  s.reg_scale = 0.0f;
  s.reg_out = nullptr;
  s.G = (void*)(w + L.G);
  s.dx_part = (float*)(w + L.dx_part);
  h->dx_part_capacity = L.dx_capacity;
  if (h->tc) {
    s.Xb = (__nv_bfloat16*)(w + L.Xb);
    s.Wb = (__nv_bfloat16*)(w + L.Wb);
  } else {
    s.Xs = (float*)(w + L.Xs);
  }
  s.mg.kind = 0;
  s.ls = LossParams{0, 1.0f, 0.0f};
  if (cfg->world > 1) {
    h->Xg = (float*)(w + L.Xg);
    h->p2p.step_dev = (unsigned*)(w + L.step_dev);     // zeroed with the workspace
    h->p2p.err_dev = h->p2p.step_dev + 1;
    h->p2p.tickets = h->p2p.step_dev + 2;
  }
  h->Cp = L.Cp;
  *out = h;
  return ASM_OK;
}

int asm_destroy(asm_head* h) {
  if (!h) return ASM_ERR_INVALID_ARG;
  if (h->ws) cudaFree(h->ws);
  if (h->dw_scratch) cudaFree(h->dw_scratch);
  if (h->side) cudaStreamDestroy(h->side);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  if (h->ev[0])
    for (int i = 0; i <= asm_head::kMaxMarks; ++i) cudaEventDestroy(h->ev[i]);
  delete h;
  return ASM_OK;
}

const char* asm_last_error(const asm_head* h) { return h ? h->err : g_create_err; }

int asm_last_launch_count(const asm_head* h) { return h ? h->launches : 0; }

int asm_forward_partial(asm_head* h, const float* X, int32_t B, const void* labels,
                        int32_t label_bytes, const float* W, float lambda, float* stats_out,
                        float* logits_out_or_null, void* cuda_stream) {
  cudaStream_t stream = (cudaStream_t)cuda_stream;
  int rc = run_forward(h, X, B, labels, label_bytes, W, lambda, logits_out_or_null, true, stream);
  if (rc != ASM_OK) return rc;
  if (!stats_out) return fail(h, ASM_ERR_INVALID_ARG, "stats_out is NULL%s", "");
  CU_TRY(h, cudaMemcpyAsync(stats_out, h->st.stats_local, (size_t)3 * B * sizeof(float),
                            cudaMemcpyDeviceToDevice, stream));
  return ASM_OK;
}

int asm_backward_partial(asm_head* h, const float* stats_all, int32_t n_shards, float* loss_out,
                         float* dX_partial, float* dW, void* cuda_stream) {
  if (!h) return ASM_ERR_INVALID_ARG;
  if (!h->fwd_valid)
    return fail(h, ASM_ERR_INVALID_ARG, "asm_backward_partial without asm_forward_partial%s", "");
  if (!stats_all || n_shards < 1 || !dX_partial || (!dW && h->st.opt.kind == 0))
    return fail(h, ASM_ERR_INVALID_ARG, "null pointer / bad n_shards%s", "");
  return run_backward(h, stats_all, n_shards, loss_out, dX_partial, dW, true,
                      (cudaStream_t)cuda_stream);
}

int asm_forward_backward(asm_head* h, const float* X, int32_t B, const void* labels,
                         int32_t label_bytes, const float* W, float lambda, float* loss_out,
                         float* logits_out_or_null, float* dX, float* dW, void* cuda_stream) {
  cudaStream_t stream = (cudaStream_t)cuda_stream;
  if (h && h->cfg.C_local != h->cfg.C_total)
    return fail(h, ASM_ERR_INVALID_ARG,
                "asm_forward_backward needs a shard that owns every class; use the partial calls%s", "");
  int rc = run_forward(h, X, B, labels, label_bytes, W, lambda, logits_out_or_null, false, stream);
  if (rc != ASM_OK) return rc;
  if (!loss_out || !dX || (!dW && h->st.opt.kind == 0))
    return fail(h, ASM_ERR_INVALID_ARG, "null output pointer%s", "");
  return run_backward(h, nullptr, 1, loss_out, dX, dW, true, stream);
}

int asm_forward(asm_head* h, const float* X, int32_t B, const void* labels, int32_t label_bytes,
                const float* W, float lambda, float* loss_out, float* logits_out_or_null,
                void* cuda_stream) {
  cudaStream_t stream = (cudaStream_t)cuda_stream;
  if (h && h->cfg.C_local != h->cfg.C_total)
    return fail(h, ASM_ERR_INVALID_ARG, "asm_forward needs a shard that owns every class%s", "");
  int rc = run_forward(h, X, B, labels, label_bytes, W, lambda, logits_out_or_null, false, stream);
  if (rc != ASM_OK) return rc;
  if (!loss_out) return fail(h, ASM_ERR_INVALID_ARG, "loss_out is NULL%s", "");
  return run_backward(h, nullptr, 1, loss_out, nullptr, nullptr, false, stream);
}

namespace {
struct P2PLayout { size_t off_x, off_y, off_st, off_dx, off_fl, total; int b_max; };
P2PLayout p2p_layout(const asm_config& c) {
  P2PLayout L{};
  const size_t B = c.B_max, D = c.D;
  L.b_max = (int)((B + c.world - 1) / c.world);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  L.off_x = take(2 * (size_t)L.b_max * D * 4);
  L.off_y = take(2 * (size_t)L.b_max * 4);
  L.off_st = take(2 * 3 * B * 4);
  L.off_dx = take(2 * B * D * 4);
  L.off_fl = take(3 * kFlagStride * 4);
  L.total = off;
  return L;
}
}  // namespace

size_t asm_p2p_bytes(const asm_config* cfg) {
  if (!valid_cfg(cfg) || cfg->world < 2 || cfg->world > kMaxPeers) return 0;
  return p2p_layout(*cfg).total;
}

int asm_p2p_attach(asm_head* h, void* const* peer_bases) {
  if (!h || !peer_bases) return ASM_ERR_INVALID_ARG;
  if (h->cfg.world < 2 || h->cfg.world > kMaxPeers)
    return fail(h, ASM_ERR_INVALID_ARG, "asm_p2p_attach needs 2..8 ranks%s", "");
  const P2PLayout L = p2p_layout(h->cfg);
  P2P& p = h->p2p;
  p.rank = h->cfg.rank;
  p.world = h->cfg.world;
  p.b_max = L.b_max;
  p.B_max = h->cfg.B_max;
  p.D = h->cfg.D;
  p.off_x = L.off_x; p.off_y = L.off_y; p.off_st = L.off_st; p.off_dx = L.off_dx; p.off_fl = L.off_fl;
  for (int r = 0; r < p.world; ++r) {
    if (!peer_bases[r]) return fail(h, ASM_ERR_INVALID_ARG, "peer base is NULL%s", "");
    p.base[r] = (char*)peer_bases[r];
  }
  // per-wait limit: ASM_P2P_TIMEOUT_MS (default 60 s; 0 = wait for ever), see asm_p2p_set_timeout
  const char* e = getenv("ASM_P2P_TIMEOUT_MS");
  p.timeout_ns = (unsigned long long)(e ? atoll(e) : 60000ll) * 1000000ull;
  e = getenv("ASM_P2P_WAITERS");        // several ranks on one GPU (tests): keep the spinning blocks few
  p.waiters = e ? atoi(e) : 1 << 20;
  if (p.waiters < 1) p.waiters = 1;
  p2p_preload_kernels();
  h->p2p_ready = true;
  return ASM_OK;
}

int asm_step_p2p(asm_head* h, const float* X_local, int32_t b_local, const void* labels_local,
                 int32_t label_bytes, const float* W, float lambda, float* loss_out,
                 float* dX_local, float* dW, void* cuda_stream) {
  if (!h) return ASM_ERR_INVALID_ARG;
  if (!h->p2p_ready) return fail(h, ASM_ERR_INVALID_ARG, "asm_step_p2p before asm_p2p_attach%s", "");
  if (!X_local || !labels_local || !W || !loss_out || !dX_local || (!dW && h->st.opt.kind == 0))
    return fail(h, ASM_ERR_INVALID_ARG, "null pointer%s", "");
  if (label_bytes != 4 && label_bytes != 8)
    return fail(h, ASM_ERR_INVALID_ARG, "label_bytes must be 4 or 8%s", "");
  P2P& p = h->p2p;
  if (b_local <= 0 || b_local > p.b_max || (long long)b_local * p.world > h->cfg.B_max)
    return fail(h, ASM_ERR_INVALID_ARG, "b_local out of range%s", "");
  cudaStream_t stream = (cudaStream_t)cuda_stream;
  p.b_local = b_local;
  p.x_local = X_local;
  p.y_local = labels_local;
  p.y_bytes = label_bytes;
  p.dx_local = dX_local;
  p.Xg = h->Xg;
  const int B = b_local * p.world;
  // 7 launches, none of them transport-only: prep publishes this rank's rows and gathers
  // everybody's, the statistics and dX exchanges ride in the combine and dx_finish kernels
  int rc = run_forward(h, h->Xg, B, labels_local, label_bytes, W, lambda, nullptr, false, stream, &p);
  if (rc == ASM_OK) rc = run_backward(h, nullptr, p.world, loss_out, nullptr, dW, true, stream, &p);
  return rc;
}

int asm_p2p_set_timeout(asm_head* h, int32_t milliseconds) {
  if (!h || milliseconds < 0) return ASM_ERR_INVALID_ARG;
  h->p2p.timeout_ns = (unsigned long long)milliseconds * 1000000ull;
  return ASM_OK;
}

int asm_p2p_status(asm_head* h, void* cuda_stream) {
  if (!h) return ASM_ERR_INVALID_ARG;
  if (!h->p2p_ready) return ASM_OK;
  unsigned code = 0;
  CU_TRY(h, cudaMemcpyAsync(&code, h->p2p.err_dev, sizeof(code), cudaMemcpyDeviceToHost,
                            (cudaStream_t)cuda_stream));
  CU_TRY(h, cudaStreamSynchronize((cudaStream_t)cuda_stream));
  if (code == 0) return ASM_OK;
  snprintf(h->err, sizeof(h->err), "peer %u did not publish phase %u in time (ranks must stay in lock-step)",
           code & 0xffu, (code >> 8) & 0xffu);
  return ASM_ERR_PEER_TIMEOUT;
}

int asm_set_optimizer(asm_head* h, const asm_optimizer* opt, float* state0, float* state1) {
  if (!h) return ASM_ERR_INVALID_ARG;
  Step& s = h->st;
  if (!opt || opt->kind == ASM_OPT_NONE) {
    s.opt.kind = 0;
    s.opt_s0 = s.opt_s1 = nullptr;
    return ASM_OK;
  }
  if (opt->kind != ASM_OPT_MOMENTUM && opt->kind != ASM_OPT_ADAM)
    return fail(h, ASM_ERR_INVALID_ARG, "unknown optimizer kind%s", "");
  if (!state0 || (opt->kind == ASM_OPT_ADAM && !state1))
    return fail(h, ASM_ERR_INVALID_ARG, "optimizer state buffer is NULL%s", "");
  if (opt->kind == ASM_OPT_ADAM && opt->step < 1)
    return fail(h, ASM_ERR_INVALID_ARG, "adam needs step >= 1%s", "");
  s.opt.kind = opt->kind;
  s.opt.mu = opt->momentum;
  s.opt.b1 = opt->beta1;
  s.opt.b2 = opt->beta2;
  s.opt.eps = opt->epsilon;
  s.opt.wd = opt->weight_decay;
  s.opt.lr = opt->lr;
  if (opt->kind == ASM_OPT_ADAM) {
    const double t = (double)opt->step;
    s.opt.lr = (float)((double)opt->lr * sqrt(1.0 - pow((double)opt->beta2, t)) /
                       (1.0 - pow((double)opt->beta1, t)));
  }
  s.opt_s0 = state0;
  s.opt_s1 = state1;
  return ASM_OK;
}

int asm_set_gradient_transform(asm_head* h, float grad_scale, float weight_decay, float* reg_loss_out) {
  if (!h) return ASM_ERR_INVALID_ARG;
  if (!(weight_decay >= 0.f) || !(grad_scale == grad_scale))
    return fail(h, ASM_ERR_INVALID_ARG, "bad grad_scale / weight_decay%s", "");
  Step& s = h->st;
  s.gscale = grad_scale;
  s.wd_g = grad_scale * weight_decay;
  s.reg_scale = 0.5f * weight_decay;
  s.reg_out = reg_loss_out;
  return ASM_OK;
}

int asm_set_embedding_dtype(asm_head* h, int32_t bytes_per_element) {
  if (!h) return ASM_ERR_INVALID_ARG;
  if (bytes_per_element != 4 && bytes_per_element != 2)
    return fail(h, ASM_ERR_INVALID_ARG, "embedding elements are 4 (fp32) or 2 (bf16) bytes%s", "");
  if (bytes_per_element == 2 && h->cfg.mode != ASM_MODE_BF16)
    return fail(h, ASM_ERR_INVALID_ARG, "bf16 embeddings need ASM_MODE_BF16%s", "");
  h->st.x_bf16 = bytes_per_element == 2 ? 1 : 0;
  return ASM_OK;
}

int asm_set_margin(asm_head* h, const asm_margin* margin) {
  if (!h) return ASM_ERR_INVALID_ARG;
  Margin g{};
  if (margin && margin->kind == ASM_MARGIN_ADDITIVE) {
    const float s = margin->s, m2 = margin->m2, m3 = margin->m3;
    if (!(isfinite(s) && s > 0.f) || !(m2 >= 0.f && m2 <= (float)(M_PI / 2)) || !(isfinite(m3) && m3 >= 0.f))
      return fail(h, ASM_ERR_INVALID_ARG, "additive margin needs finite s > 0, m2 in [0, pi/2], finite m3 >= 0%s", "");
    g.kind = kMarginAdditive;
    g.s = s;
    g.inv_s = (float)(1.0 / (double)s);
    g.cm = (float)cos((double)m2);
    g.sm = (float)sin((double)m2);
    g.tau = (float)cos(M_PI - (double)m2);
    g.fb = (float)((double)m2 * sin((double)m2) + (double)m3);
    g.m3 = m3;
  } else if (margin && margin->kind == ASM_MARGIN_LINEAR) {
    g.kind = kMarginLinear;                 // s, m2, m3 are ignored
  } else if (margin && margin->kind != ASM_MARGIN_ASOFTMAX) {
    return fail(h, ASM_ERR_INVALID_ARG, "unknown margin kind%s", "");
  }
  h->st.mg = g;
  // the linear kind's dW has no normalisation term: its coefficient reads zeros instead of 1/c_j
  h->st.wcorr = g.kind == kMarginLinear ? h->wzero : h->st.inv_c;
  return ASM_OK;
}

int asm_set_loss(asm_head* h, const asm_loss* loss) {
  if (!h) return ASM_ERR_INVALID_ARG;
  LossParams l{0, 1.0f, 0.0f};
  if (loss && loss->kind == ASM_LOSS_FOCAL) {
    if (!(isfinite(loss->gamma) && loss->gamma > 0.f) || !(isfinite(loss->alpha) && loss->alpha >= 0.f))
      return fail(h, ASM_ERR_INVALID_ARG, "focal loss needs finite gamma > 0 and finite alpha >= 0%s", "");
    l = LossParams{1, loss->gamma, loss->alpha};
  } else if (loss && loss->kind != ASM_LOSS_SOFTMAX_CE) {
    return fail(h, ASM_ERR_INVALID_ARG, "unknown loss kind%s", "");
  }
  h->st.ls = l;
  return ASM_OK;
}

int asm_set_lambda_device(asm_head* h, const float* lambda_dev) {
  if (!h) return ASM_ERR_INVALID_ARG;
  h->st.lambda_dev = lambda_dev;
  return ASM_OK;
}

int asm_set_profiling(asm_head* h, int enable) {
  if (!h) return ASM_ERR_INVALID_ARG;
  if (enable && !h->ev[0]) {
    for (int i = 0; i <= asm_head::kMaxMarks; ++i) CU_TRY(h, cudaEventCreate(&h->ev[i]));
  }
  h->profiling = enable != 0;
  h->phase_profiling = enable == 2;
  h->n_marks = 0;
  return ASM_OK;
}

int asm_get_profile(asm_head* h, int32_t max_n, float* ms_out, char* names_out) {
  if (!h || !ms_out || !names_out || max_n < 0) return ASM_ERR_INVALID_ARG;
  if (!h->profiling || h->n_marks == 0) return 0;
  CU_TRY(h, cudaEventSynchronize(h->ev[h->n_marks]));
  const int n = h->n_marks < max_n ? h->n_marks : max_n;
  // marks of the forward half end at the event recorded by mark_end of run_forward; when a
  // backward half followed, its first event was recorded right after, so consecutive
  // differences are per-kernel durations either way.
  for (int i = 0; i < n; ++i) {
    float ms = 0.f;
    CU_TRY(h, cudaEventElapsedTime(&ms, h->ev[i], h->ev[i + 1]));
    ms_out[i] = ms;
    strncpy(names_out + (size_t)i * 32, h->mark_name[i], 31);
    names_out[(size_t)i * 32 + 31] = 0;
  }
  return n;
}

int asm_check_labels(asm_head* h, void* cuda_stream) {
  if (!h) return ASM_ERR_INVALID_ARG;
  // the norm kernel marks out-of-range labels in its label -> local-class table
  const int B = h->st.B;
  if (B <= 0) return ASM_OK;
  std::vector<int> yl((size_t)B);
  CU_TRY(h, cudaMemcpyAsync(yl.data(), h->st.ylocal, (size_t)B * 4, cudaMemcpyDeviceToHost,
                            (cudaStream_t)cuda_stream));
  CU_TRY(h, cudaStreamSynchronize((cudaStream_t)cuda_stream));
  for (int i = 0; i < B; ++i)
    if (yl[i] == -2) return fail(h, ASM_ERR_LABEL_RANGE, "label outside [0, C_total)%s", "");
  return ASM_OK;
}

}  // extern "C"
