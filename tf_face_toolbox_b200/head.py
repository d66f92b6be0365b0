"""Python host side of the A-softmax head: the call surface the reference's towers use.

Reference contract mirrored here (file:line in /root/reference):
  * data_parallel.py:220   logits = model.forward(images, labels, num_classes=..., is_training=True)
  * data_parallel.py:223   losses, losses_name, others = model.loss_function(scope, labels, **logits)
  * data_parallel.py:32-38 tf.gradients(total_loss, params) scaled by mult_lr * 1/num_gpus
  * nets/sphere.py:84-90   classifier/fc_classifier weights [D, C], N(0, 0.001) init, no bias, L2 reg
  * nets/sphere.py:103-118 losses = [cross_entropy, reg_loss]
  * train.py:157 + data_parallel.py:252-253  global_step, the lambda-annealing clock

`asoftmax_head(...)` is the functional entry point named by BASELINE.json's north_star:
(embeddings, labels, num_classes, m, lambda state) -> (loss, logits | None, dX, dW).
`ASoftmaxHead` wraps it in the forward / loss_function / param_list shape of
nets/net_base.py:80-101, and `ASoftmaxLoss` exposes it to torch autograd so a torch
backbone can be trained through it.  Everything executes in libasoftmax_b200.so
(hand-written sm_100a CUDA) through ctypes; torch only owns the device buffers and the
stream.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os
from collections import OrderedDict
from dataclasses import dataclass
from typing import Dict, Optional, Tuple

import torch

from . import _lib


# --------------------------------------------------------------------------------------
# lambda annealing state (host scalar; kernels are stateless)
# --------------------------------------------------------------------------------------
@dataclass
class LambdaState:
    """SphereFace schedule lambda(it) = max(lambda_min, base * (1 + gamma*it)^(-power)).

    `iteration` plays the role of global_step (train.py:157): `step()` is the analogue of
    `global_step.assign_add(1)` (data_parallel.py:252-253) and the first training step uses
    it = 1.  `explicit` overrides the schedule with a fixed lambda.
    """
    iteration: int = 0
    base: float = 1000.0
    gamma: float = 0.12
    power: float = 1.0
    lambda_min: float = 5.0
    explicit: Optional[float] = None

    def value(self) -> float:
        if self.explicit is not None:
            return float(self.explicit)
        return max(self.lambda_min, self.base * (1.0 + self.gamma * self.iteration) ** (-self.power))

    def step(self) -> float:
        self.iteration += 1
        return self.value()


# --------------------------------------------------------------------------------------
# additive-margin heads (ArcFace / CosFace) on L2-normalised embeddings
# --------------------------------------------------------------------------------------
@dataclass(frozen=True)
class AdditiveMargin:
    """Target logit s * phi(cos theta) on normalised embeddings and weights, every other logit
    s * cos(theta_j), with phi(t) = cos(theta + m2) - m3 for t >= cos(pi - m2) and
    t - m2 sin(m2) - m3 below that (InsightFace's combined margin without m1; no "easy margin").
    m2 = 0 is CosFace, m3 = 0 is ArcFace.  Pass it as `margin=` to the head's entry points;
    `m` and lambda are then ignored.  s > 0, 0 <= m2 <= pi/2 and m3 >= 0 are checked by the library."""
    s: float = 64.0
    m2: float = 0.5
    m3: float = 0.0

    @classmethod
    def arcface(cls, s: float = 64.0, m: float = 0.5) -> "AdditiveMargin":
        """s * cos(theta + m)."""
        return cls(float(s), float(m), 0.0)

    @classmethod
    def cosface(cls, s: float = 64.0, m: float = 0.35) -> "AdditiveMargin":
        """s * (cos(theta) - m)."""
        return cls(float(s), 0.0, float(m))

    def _struct(self) -> "_lib.AsmMargin":
        return _lib.AsmMargin(_lib.MARGIN_ADDITIVE, self.s, self.m2, self.m3)


# --------------------------------------------------------------------------------------
# focal loss (loss.py:18-27 of the reference) in place of the softmax cross-entropy
# --------------------------------------------------------------------------------------
@dataclass(frozen=True)
class FocalLoss:
    """The reference's focal_loss on the head's (margin) logits f:
    L = mean_i gamma * (1 - p_iy)^alpha * (lse_i - f_iy), p_iy = softmax(f_i)[y_i].
    The names follow the reference, not Lin et al.: gamma is the multiplier and alpha the
    exponent (the paper calls them the other way round).  The gradient goes through the
    modulating factor (1 - p)^alpha; it is not a stop-gradient.  gamma=1, alpha=0 is the plain
    cross-entropy.  Pass it as `loss=` to the head's entry points (None: cross-entropy).
    gamma > 0 and alpha >= 0, both finite, are checked by the library."""
    gamma: float = 1.0
    alpha: float = 2.0

    def _struct(self) -> "_lib.AsmLoss":
        return _lib.AsmLoss(_lib.LOSS_FOCAL, self.gamma, self.alpha)


def _as_lambda(lambda_state) -> float:
    if lambda_state is None:
        return 0.0
    if isinstance(lambda_state, LambdaState):
        return lambda_state.value()
    return float(lambda_state)


# --------------------------------------------------------------------------------------
# handle cache: one asm_head per (device, shard geometry, B_max, m, mode, margin, loss)
# --------------------------------------------------------------------------------------
class _Handle:
    def __init__(self, device: torch.device, D: int, C_total: int, C_local: int, class_offset: int,
                 B_max: int, m: int, mode: str, rank: int = 0, world: int = 1,
                 margin: Optional[AdditiveMargin] = None, loss: Optional[FocalLoss] = None):
        self.lib = _lib.load()
        if device.type != "cuda":
            raise RuntimeError("the A-softmax head runs on a CUDA (B200) device only; no CPU fallback")
        self.device = device
        self.cfg = _lib.AsmConfig(D, C_total, C_local, class_offset, B_max, m, _lib.MODES[mode],
                                  rank, world, None)
        self.ptr = C.c_void_p()
        with torch.cuda.device(device):
            rc = self.lib.asm_create(C.byref(self.ptr), C.byref(self.cfg))
        if rc != _lib.ASM_OK:
            raise _lib.AsmError(rc, (self.lib.asm_last_error(None) or b"").decode())
        if margin is not None:
            # set once: the margin is part of the handle-cache key, never switched per call
            rc = self.lib.asm_set_margin(self.ptr, C.byref(margin._struct()))
            if rc != _lib.ASM_OK:
                err = _lib.AsmError(rc, (self.lib.asm_last_error(self.ptr) or b"").decode())
                self.close()
                raise err
        if loss is not None:
            # likewise part of the key
            rc = self.lib.asm_set_loss(self.ptr, C.byref(loss._struct()))
            if rc != _lib.ASM_OK:
                err = _lib.AsmError(rc, (self.lib.asm_last_error(self.ptr) or b"").decode())
                self.close()
                raise err

    def close(self):
        if self.ptr:
            self.lib.asm_destroy(self.ptr)
            self.ptr = C.c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass


# Handles hold a device workspace (>= 200 MB at BASELINE config 3), so the cache is bounded:
# untagged handles (plain asoftmax_head calls) are evicted least-recently-used beyond
# ASM_MAX_HANDLES; tagged handles belong to the object that made them (a CUDA-graph step, a
# sharded head) and are dropped with it (drop_handle).
_HANDLES: "OrderedDict[tuple, _Handle]" = OrderedDict()
_MAX_HANDLES = int(os.environ.get("ASM_MAX_HANDLES", "8"))


def _round_batch(B: int) -> int:
    return max(128, (B + 127) // 128 * 128)


def get_handle(device, D, C_total, C_local, class_offset, B, m, mode, rank=0, world=1, tag=None,
               margin: Optional[AdditiveMargin] = None, loss: Optional[FocalLoss] = None) -> _Handle:
    """`tag` separates handles with different per-handle state (e.g. a CUDA-graph step that
    reads lambda from device memory) from the plain eager ones."""
    device = torch.device(device)
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    if margin is not None and not isinstance(margin, AdditiveMargin):
        raise TypeError("margin must be None (A-softmax) or an AdditiveMargin")
    if loss is not None and not isinstance(loss, FocalLoss):
        raise TypeError("loss must be None (softmax cross-entropy) or a FocalLoss")
    key = (device.index, D, C_total, C_local, class_offset, _round_batch(B), m, mode, rank, world, margin, loss, tag)
    h = _HANDLES.get(key)
    if h is None:
        h = _Handle(device, D, C_total, C_local, class_offset, _round_batch(B), m, mode, rank, world, margin, loss)
        h.key = key
        _HANDLES[key] = h
        untagged = [k for k in _HANDLES if k[-1] is None]
        for k in untagged[:max(0, len(untagged) - _MAX_HANDLES)]:
            # stream-ordered frees: work already enqueued on the evicted handle still completes
            _HANDLES.pop(k).close()
    else:
        _HANDLES.move_to_end(key)
    return h


def drop_handle(h: Optional[_Handle]) -> None:
    """Release a tagged handle together with the object that owned it."""
    if h is None:
        return
    _HANDLES.pop(getattr(h, "key", None), None)
    h.close()


def release_handles() -> None:
    for h in _HANDLES.values():
        h.close()
    _HANDLES.clear()


# --------------------------------------------------------------------------------------
# fused classifier optimizer (the head's share of data_parallel.py:186-196)
# --------------------------------------------------------------------------------------
class FusedOptimizer:
    """Momentum(0.9) / Adam(beta1=0.5, beta2=0.999) update of the classifier weights, with the
    L2 weight-decay gradient (nets/sphere.py:88, train.py:82 wd=5e-4), executed inside the dW
    kernel's epilogue: W is updated in place and dW is never written to HBM.

        opt = FusedOptimizer("Momentum", lr=0.1)           # or "Adam"
        loss, _, dX, _ = asoftmax_head(X, y, C, 4, lam, weights=W, optimizer=opt)   # W updated
    """

    def __init__(self, kind: str = "Momentum", lr: float = 0.1, momentum: float = 0.9, beta1: float = 0.5,
                 beta2: float = 0.999, epsilon: float = 1e-8, weight_decay: float = 5e-4):
        self.kind = {"momentum": _lib.OPT_MOMENTUM, "adam": _lib.OPT_ADAM}[kind.lower()]
        self.lr, self.momentum, self.beta1, self.beta2 = lr, momentum, beta1, beta2
        self.epsilon, self.weight_decay = epsilon, weight_decay
        self.step = 0
        self.state0 = None
        self.state1 = None

    def _arm(self, h, weights: torch.Tensor):
        if self.state0 is None or self.state0.shape != weights.shape:
            self.state0 = torch.zeros_like(weights)
            self.state1 = torch.zeros_like(weights) if self.kind == _lib.OPT_ADAM else None
        self.step += 1
        o = _lib.AsmOptimizer(self.kind, self.lr, self.momentum, self.beta1, self.beta2, self.epsilon,
                              self.weight_decay, self.step)
        _lib.check(h.lib.asm_set_optimizer(h.ptr, C.byref(o), self.state0.data_ptr(),
                                           self.state1.data_ptr() if self.state1 is not None else None), h.ptr)

    @staticmethod
    def _disarm(h):
        h.lib.asm_set_optimizer(h.ptr, None, None, None)


def _check_inputs(embeddings, labels, weights, num_classes):
    if not (embeddings.is_cuda and labels.is_cuda and weights.is_cuda):
        raise RuntimeError("embeddings, labels and weights must be CUDA tensors (no CPU fallback)")
    if weights.dtype != torch.float32:
        raise TypeError("weights must be float32 (the master copy; bf16 rounding happens inside the library)")
    if embeddings.dtype not in (torch.float32, torch.bfloat16):
        raise TypeError("embeddings must be float32, or bfloat16 in bf16 mode")
    if labels.dtype not in (torch.int32, torch.int64):
        raise TypeError("labels must be int32 (reference dtype, data.py:259) or int64")
    if embeddings.dim() != 2 or weights.dim() != 2 or labels.dim() != 1:
        raise ValueError("expected embeddings [B,D], weights [D,C], labels [B]")
    if embeddings.shape[1] != weights.shape[0] or labels.shape[0] != embeddings.shape[0]:
        raise ValueError("shape mismatch between embeddings / weights / labels")
    if num_classes is not None and weights.shape[1] != num_classes:
        raise ValueError(f"weights has {weights.shape[1]} classes, num_classes={num_classes}")


def asoftmax_head(embeddings: torch.Tensor, labels: torch.Tensor, num_classes: int, m: int = 4,
                  lambda_state=None, *, weights: torch.Tensor, mode: str = "bf16",
                  return_logits: bool = False, compute_grads: bool = True,
                  check_labels: bool = False, optimizer: Optional["FusedOptimizer"] = None,
                  grad_scale: float = 1.0, weight_decay: float = 0.0,
                  reg_loss_out: Optional[torch.Tensor] = None, margin: Optional[AdditiveMargin] = None,
                  loss: Optional[FocalLoss] = None, _handle_tag=None
                  ) -> Tuple[torch.Tensor, Optional[torch.Tensor], Optional[torch.Tensor], Optional[torch.Tensor]]:
    """A-softmax head forward + backward on one GPU that owns every class.

    embeddings [B, D] fp32, labels [B] int32/int64, weights [D, num_classes] fp32 (the
    `classifier/fc_classifier/weights` variable, nets/sphere.py:86), margin m in 1..4,
    lambda_state a LambdaState or a float.  Returns (loss, logits | None, dX, dW): loss is the
    batch-mean softmax cross-entropy over the margin logits (nets/sphere.py:109), logits are
    the margin-modified f (only when return_logits: the benchmark path never writes the
    [B, C] matrix to HBM), dX / dW are d(loss)/d(embeddings, weights).
    With `optimizer` (a FusedOptimizer) the classifier update is fused into the dW kernel:
    `weights` is updated IN PLACE and the returned dW is None.
    `grad_scale`, `weight_decay`, `reg_loss_out` reproduce what the reference's towers do to the
    gradients without a single extra pass over [D, C]: dX, dW come back multiplied by grad_scale
    (mult_lr / num_gpus, data_parallel.py:37), dW includes weight_decay * W (the gradient of
    reg_loss, nets/sphere.py:88) and reg_loss_out (a 1-element CUDA float tensor) receives
    weight_decay/2 * |W|^2 (nets/net_base.py:103-107).  The returned loss is the unscaled loss
    without reg_loss.
    `margin` (an AdditiveMargin) selects the ArcFace / CosFace head on normalised embeddings
    instead of A-softmax; `m` and lambda_state are then ignored.  None: A-softmax.
    `loss` (a FocalLoss) replaces the softmax cross-entropy by the reference's focal loss on the
    same logits; loss, dX and dW are then those of the focal loss.  None: cross-entropy.
    Asynchronous on the current CUDA stream.
    """
    _check_inputs(embeddings, labels, weights, num_classes)
    if embeddings.dtype == torch.bfloat16 and mode != "bf16":
        raise TypeError("bfloat16 embeddings need mode='bf16'")
    X = embeddings.contiguous()
    if optimizer is not None and not weights.is_contiguous():
        raise ValueError("a fused optimizer updates `weights` in place: it must be contiguous")
    W = weights.contiguous()
    y = labels.contiguous()
    B, D = X.shape
    Cn = W.shape[1]
    h = get_handle(X.device, D, Cn, Cn, 0, B, m, mode, tag=_handle_tag, margin=margin, loss=loss)
    lam = _as_lambda(lambda_state)
    loss_out = torch.empty(1, device=X.device, dtype=torch.float32)
    logits = torch.empty(B, Cn, device=X.device, dtype=torch.float32) if return_logits else None
    stream = C.c_void_p(torch.cuda.current_stream(X.device).cuda_stream)
    transform = grad_scale != 1.0 or weight_decay != 0.0 or reg_loss_out is not None
    if reg_loss_out is not None and not (reg_loss_out.is_cuda and reg_loss_out.dtype == torch.float32
                                         and reg_loss_out.numel() == 1):
        raise TypeError("reg_loss_out must be a 1-element CUDA float32 tensor")
    x16 = X.dtype == torch.bfloat16
    with torch.cuda.device(X.device):
        if x16:
            _lib.check(h.lib.asm_set_embedding_dtype(h.ptr, 2), h.ptr)
        if transform:
            _lib.check(h.lib.asm_set_gradient_transform(
                h.ptr, grad_scale, weight_decay, reg_loss_out.data_ptr() if reg_loss_out is not None else None), h.ptr)
        if compute_grads:
            dX = torch.empty(X.shape, device=X.device, dtype=torch.float32)
            dW = torch.empty_like(W) if optimizer is None else None
            if optimizer is not None:
                optimizer._arm(h, W)
            try:
                rc = h.lib.asm_forward_backward(
                    h.ptr, X.data_ptr(), B, y.data_ptr(), y.element_size(), W.data_ptr(), lam,
                    loss_out.data_ptr(), logits.data_ptr() if logits is not None else None,
                    dX.data_ptr(), dW.data_ptr() if dW is not None else None, stream)
            finally:
                if optimizer is not None:
                    optimizer._disarm(h)
        else:
            dX = dW = None
            rc = h.lib.asm_forward(
                h.ptr, X.data_ptr(), B, y.data_ptr(), y.element_size(), W.data_ptr(), lam,
                loss_out.data_ptr(), logits.data_ptr() if logits is not None else None, stream)
        if transform:
            h.lib.asm_set_gradient_transform(h.ptr, 1.0, 0.0, None)     # the handle is shared: back to defaults
        if x16:
            h.lib.asm_set_embedding_dtype(h.ptr, 4)
        _lib.check(rc, h.ptr)
        if check_labels:
            _lib.check(h.lib.asm_check_labels(h.ptr, stream), h.ptr)
    return loss_out[0], logits, dX, dW


def last_launch_count(device, D, C_total, B, m, mode) -> int:
    h = get_handle(device, D, C_total, C_total, 0, B, m, mode)
    return int(h.lib.asm_last_launch_count(h.ptr))


# --------------------------------------------------------------------------------------
# CUDA-graph step: the whole head (7 launches, fork/join included) replayed as one graph
# --------------------------------------------------------------------------------------
class GraphedASoftmaxStep:
    """One fixed-shape A-softmax step captured into a CUDA graph.

        step = GraphedASoftmaxStep(weights, batch_size=512, m=4, mode="bf16")
        loss, dX, dW = step(embeddings, labels, lambda_state)     # copies inputs, replays

    Inputs are copied into static device buffers (so host tensors in pinned memory are fine);
    lambda lives in a device scalar the kernels read (asm_set_lambda_device), because kernel
    arguments are frozen at capture.  `weights` is used in place: update it in place
    (optimizer step), never rebind it.  Outputs are static tensors overwritten by each replay.
    """

    def __init__(self, weights: torch.Tensor, batch_size: int, m: int = 4, mode: str = "bf16",
                 labels_dtype=torch.int32, margin: Optional[AdditiveMargin] = None,
                 loss: Optional[FocalLoss] = None):
        assert weights.is_cuda and weights.dtype == torch.float32 and weights.is_contiguous()
        dev = weights.device
        self.W = weights
        D, Cn = weights.shape
        self.X = torch.zeros(batch_size, D, device=dev, dtype=torch.float32)
        self.y = torch.zeros(batch_size, device=dev, dtype=labels_dtype)
        self.lam = torch.zeros(1, device=dev, dtype=torch.float32)
        self._lam_host = torch.zeros(1, dtype=torch.float32).pin_memory()
        self.m, self.mode, self.Cn, self.margin, self.loss_kind = m, mode, Cn, margin, loss
        self._tag = ("graph", id(self))
        h = get_handle(dev, D, Cn, Cn, 0, batch_size, m, mode, tag=self._tag, margin=margin, loss=loss)
        self._key = h.key
        _lib.check(h.lib.asm_set_lambda_device(h.ptr, self.lam.data_ptr()), h.ptr)
        cur = torch.cuda.current_stream(dev)
        side = torch.cuda.Stream(dev)
        side.wait_stream(cur)
        with torch.cuda.stream(side):          # warm-up outside capture (builds the TMA maps)
            for _ in range(2):
                self._run()
        cur.wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss, self.dX, self.dW = self._run()

    def _run(self):
        loss, _, dX, dW = asoftmax_head(self.X, self.y, self.Cn, self.m, 0.0, weights=self.W,
                                        mode=self.mode, margin=self.margin, loss=self.loss_kind,
                                        _handle_tag=self._tag)
        return loss, dX, dW

    def close(self):
        """Drop the captured graph and this step's private handle (its device workspace)."""
        self.graph = None
        h = _HANDLES.get(getattr(self, "_key", None))
        if h is not None:
            drop_handle(h)
        self._key = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def __call__(self, embeddings: torch.Tensor, labels: torch.Tensor, lambda_state=None):
        self._lam_host[0] = _as_lambda(lambda_state)
        self.lam.copy_(self._lam_host, non_blocking=True)
        self.X.copy_(embeddings, non_blocking=True)
        self.y.copy_(labels, non_blocking=True)
        self.graph.replay()
        return self.loss, self.dX, self.dW


# --------------------------------------------------------------------------------------
# torch autograd bridge: lets a torch backbone train through the fused head
# --------------------------------------------------------------------------------------
class ASoftmaxLoss(torch.autograd.Function):
    """loss = ASoftmaxLoss.apply(embeddings, weights, labels, m, lam, mode[, upstream[, margin[, loss]]]).  The fused
    call already produced dX and dW, so backward only hands them on.  `upstream` (a float) is the
    gradient the caller promises to send into this loss (1.0 for a plain `loss.backward()`, the loss
    scale otherwise): it is applied inside the kernels and backward returns the stored gradients
    untouched -- no pass over [D, C].  Without it backward multiplies by the incoming gradient.
    `margin` (an AdditiveMargin, or None for A-softmax) and `loss` (a FocalLoss, or None for the
    cross-entropy) as in asoftmax_head."""

    @staticmethod
    def forward(ctx, embeddings, weights, labels, m, lam, mode, upstream=None, margin=None, loss=None):
        value, _, dX, dW = asoftmax_head(embeddings, labels, weights.shape[1], m, lam, weights=weights, mode=mode,
                                         grad_scale=1.0 if upstream is None else float(upstream), margin=margin,
                                         loss=loss)
        ctx.save_for_backward(dX, dW)
        ctx.upstream = upstream
        return value

    @staticmethod
    def backward(ctx, grad_out):
        dX, dW = ctx.saved_tensors
        if ctx.upstream is not None:
            return dX, dW, None, None, None, None, None, None, None
        return grad_out * dX, grad_out * dW, None, None, None, None, None, None, None


# --------------------------------------------------------------------------------------
# Network-shaped wrapper: forward / loss_function / param_list of nets/net_base.py:80-101
# --------------------------------------------------------------------------------------
class ASoftmaxHead:
    """The `classifier` scope of a margin network, as DataParallel_margin drives it.

        logits = head.forward(features, labels, num_classes=C, is_training=True)   # data_parallel.py:220
        losses, names, others = head.loss_function(scope, labels, **logits)        # data_parallel.py:223
        dX, dW = head.gradients()                                                   # data_parallel.py:32-38

    `features` are the backbone's embeddings (the reference passes images to the full
    network; the head is the part after `features = self.backbone(images)`, nets/sphere.py:82).
    """
    name = "classifier"

    def __init__(self, num_features: int, num_classes: int, m: int = 4, weight_decay: float = 5e-4,
                 mode: str = "bf16", device="cuda", lambda_state: Optional[LambdaState] = None,
                 return_logits: bool = False, seed: Optional[int] = None, num_gpus: int = 1,
                 mult_lr: float = 1.0, margin: Optional[AdditiveMargin] = None,
                 loss: Optional[FocalLoss] = None):
        gen = None
        if seed is not None:
            gen = torch.Generator(device="cpu").manual_seed(seed)
        # weights_initializer=tf.random_normal_initializer(stddev=0.001)  (nets/sphere.py:87)
        w = torch.randn(num_features, num_classes, generator=gen, dtype=torch.float32) * 0.001
        self.weights = w.to(device)                  # classifier/fc_classifier/weights [D, C]
        self.num_classes = num_classes
        self.m = m
        self.margin = margin                         # None: A-softmax; AdditiveMargin: ArcFace / CosFace
        self.loss = loss                             # None: cross-entropy; FocalLoss: loss.py's focal_loss
        self.weight_decay = weight_decay
        self.mode = mode
        self.lambda_state = lambda_state if lambda_state is not None else LambdaState()
        self.return_logits = return_logits
        # _grad_var scales every gradient by mult_lr * 1/num_gpus (data_parallel.py:37): known when
        # the tower is built, so the kernels apply it and gradients() costs nothing
        self.num_gpus, self.mult_lr = num_gpus, mult_lr
        self._reg = torch.zeros(1, device=self.weights.device, dtype=torch.float32)
        self._last = None

    # nets/net_base.py:84-86, margin form data_parallel.py:220
    def forward(self, features, labels=None, num_classes=None, is_training=True):
        if not is_training:
            return features                           # nets/sphere.py:96-101: bare features
        assert num_classes is not None, "num_classes must be given when is_training=True"
        assert labels is not None, "a margin head needs labels in forward (data_parallel.py:220)"
        lam = self.lambda_state.step()                # global_step += 1, first step uses it = 1
        scale = self.mult_lr / self.num_gpus
        loss, logits, dX, dW = asoftmax_head(features, labels, num_classes, self.m, lam,
                                             weights=self.weights, mode=self.mode,
                                             return_logits=self.return_logits, grad_scale=scale,
                                             weight_decay=self.weight_decay, reg_loss_out=self._reg,
                                             margin=self.margin, loss=self.loss)
        self._last = dict(loss=loss, dX=dX, dW=dW, lam=lam, scale=scale, reg=self._reg[0].clone())
        out = {"logits": logits, "features": features}
        return out

    # nets/net_base.py:88-90; nets/sphere.py:103-118
    def loss_function(self, scope, labels, **logits):
        assert self._last is not None, "forward(...) must run first"
        losses = [self._last["loss"]]
        losses_name = ["focal_loss" if self.loss is not None else "cross_entropy"]
        # _regularize (nets/net_base.py:103-107): contrib l2_regularizer = wd * sum(w^2)/2, a
        # by-product of the norm kernel's column sums (no pass over W here)
        losses.append(self._last["reg"])
        losses_name.append("reg_loss")
        others = OrderedDict()
        if self.margin is None:                       # lambda means nothing to the additive margins
            others["lambda"] = self._last["lam"]
        return losses, losses_name, others

    def gradients(self, num_gpus: Optional[int] = None, mult_lr: Optional[float] = None):
        """(dX, dW) of total_loss = cross_entropy (or focal_loss) + reg_loss, scaled like _grad_var
        (data_parallel.py:37): both came out of the kernels in that form (dW includes wd * W).
        Asking for a scale other than the configured one rescales them (one eager pass)."""
        want = (self.mult_lr if mult_lr is None else mult_lr) / (self.num_gpus if num_gpus is None else num_gpus)
        dX, dW = self._last["dX"], self._last["dW"]
        if want != self._last["scale"]:
            r = want / self._last["scale"]
            return dX * r, dW * r
        return dX, dW

    def param_list(self, is_training=True, trainable=True, scope=None):
        return [[self.weights]] if is_training else []

    def mult_lr_list(self, scope=None):
        return [self.mult_lr]
