"""Class-sharded A-softmax head: one process per GPU, W partitioned by class.

Replaces the reference's replicated classifier + per-variable gradient all-reduce
(`nccl.all_sum(grads)`, data_parallel.py:175-181: a full [D, C] fp32 message per tower per
step) with a class partition in which dW never leaves its shard.  Per step (SURVEY.md 8e):

  1. all-gather the embeddings X [B/G, D] -> [B, D] and the labels      (torch.distributed)
  2. asm_forward_partial on the local shard -> per-row (max, sumexp, target logit | 0)
  3. ONE all-gather of the [3, B] statistics                             (torch.distributed)
  4. asm_backward_partial: global logsumexp / loss, G'', dW_local, dX partial
  5. reduce-scatter dX partial [B, D] -> the owner's [B/G, D]            (torch.distributed)

Semantics equal the reference's towers: per-tower mean over B/G, grads x 1/G, all_sum
== gradient of the global-batch mean (data_parallel.py:37,179,248).  The collectives run
through torch.distributed (NCCL over NVLink on the GPU box; gloo in the CPU tests, where
the per-shard compute is injected by the test).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import torch
import torch.distributed as dist

from . import _lib
from .head import FocalLoss, LambdaState, _as_lambda, get_handle


def shard_bounds(num_classes: int, world: int, rank: int) -> Tuple[int, int]:
    """Rank g owns classes [g*ceil(C/G), min(C, (g+1)*ceil(C/G)))."""
    per = -(-num_classes // world)
    return min(num_classes, rank * per), min(num_classes, (rank + 1) * per)


class _CudaShard:
    """Per-shard compute through the C ABI (asm_forward_partial / asm_backward_partial)."""

    def __init__(self, D, C_total, lo, hi, m, mode, rank, world, device, margin=None, loss=None):
        self.args = (D, C_total, hi - lo, lo, m, mode, rank, world)
        self.margin, self.loss = margin, loss
        self.device = torch.device(device)
        # a handle carries per-step state (the pointers of the step in flight, an armed optimizer):
        # every shard object gets its own instead of sharing one with same-shaped callers
        self.tag = ("shard", id(self))
        self.lambda_dev = None      # device scalar read by the kernels (CUDA-graph replay)

    def _handle(self, B):
        D, C_total, C_local, lo, m, mode, rank, world = self.args
        h = get_handle(self.device, D, C_total, C_local, lo, B, m, mode, rank, world, tag=self.tag,
                       margin=self.margin, loss=self.loss)
        if self.lambda_dev is not None:
            _lib.check(h.lib.asm_set_lambda_device(h.ptr, self.lambda_dev.data_ptr()), h.ptr)
        return h

    def forward_partial(self, X, y, W, lam):
        B = X.shape[0]
        h = self._handle(B)
        _lib.check(h.lib.asm_set_embedding_dtype(h.ptr, X.element_size()), h.ptr)    # fp32, or bf16 in bf16 mode
        stats = torch.empty(3, B, device=X.device, dtype=torch.float32)
        stream = C.c_void_p(torch.cuda.current_stream(X.device).cuda_stream)
        with torch.cuda.device(X.device):
            _lib.check(h.lib.asm_forward_partial(h.ptr, X.data_ptr(), B, y.data_ptr(), y.element_size(),
                                                 W.data_ptr(), lam, stats.data_ptr(), None, stream), h.ptr)
        self._keep = (X, y, W)          # borrowed until backward_partial has been enqueued
        return stats

    def backward_partial(self, stats_all, X, W, optimizer=None):
        B = X.shape[0]
        h = self._handle(B)
        loss = torch.empty(1, device=X.device, dtype=torch.float32)
        dXp = torch.empty(X.shape, device=X.device, dtype=torch.float32)
        dW = torch.empty_like(W) if optimizer is None else None     # fused update: dW never exists
        stream = C.c_void_p(torch.cuda.current_stream(X.device).cuda_stream)
        with torch.cuda.device(X.device):
            if optimizer is not None:
                optimizer._arm(h, W)
            try:
                rc = h.lib.asm_backward_partial(h.ptr, stats_all.data_ptr(), stats_all.shape[0],
                                                loss.data_ptr(), dXp.data_ptr(),
                                                dW.data_ptr() if dW is not None else None, stream)
            finally:
                if optimizer is not None:
                    optimizer._disarm(h)
            _lib.check(rc, h.ptr)
        return loss[0], dXp, dW


class ShardedASoftmaxHead:
    """Class-parallel head over a torch.distributed process group (one rank per GPU)."""

    def __init__(self, num_features: int, num_classes: int, m: int = 4, mode: str = "bf16",
                 device="cuda", group=None, lambda_state: Optional[LambdaState] = None,
                 weights_full: Optional[torch.Tensor] = None, seed: int = 0, shard_compute=None,
                 transport: str = "nccl", batch_global: Optional[int] = None,
                 weights_shard: Optional[torch.Tensor] = None, margin=None,
                 loss: Optional[FocalLoss] = None):
        """`margin` (an AdditiveMargin) selects the ArcFace / CosFace head, LinearSoftmax() the plain
        classifier x_i . w_j; None: A-softmax.
        `loss` (a FocalLoss) replaces the cross-entropy by the focal loss on both transports;
        None: cross-entropy.  An injected `shard_compute` is given the margin and the loss
        through its own constructor."""
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.D, self.C, self.m, self.mode, self.margin = num_features, num_classes, m, mode, margin
        self.loss = loss
        self.lo, self.hi = shard_bounds(num_classes, self.world, self.rank)
        if self.hi <= self.lo:
            raise ValueError("more ranks than classes: empty shard")
        self.device = torch.device(device)
        if weights_shard is not None:              # this rank's [D, C_local] slice, e.g. scattered on the device
            if tuple(weights_shard.shape) != (num_features, self.hi - self.lo):
                raise ValueError(f"weights_shard must be [{num_features}, {self.hi - self.lo}]")
            w = weights_shard.to(torch.float32)
        elif weights_full is not None:
            w = weights_full[:, self.lo:self.hi].to(torch.float32)
        else:   # N(0, 0.001) like nets/sphere.py:87, generated shard-locally but rank-independent
            g = torch.Generator().manual_seed(seed)
            w = (torch.randn(num_features, num_classes, generator=g) * 0.001)[:, self.lo:self.hi]
        self.weights = w.contiguous().to(self.device)            # [D, C_local]
        self.lambda_state = lambda_state if lambda_state is not None else LambdaState()
        self.compute = shard_compute if shard_compute is not None else _CudaShard(
            num_features, num_classes, self.lo, self.hi, m, mode, self.rank, self.world, self.device, margin, loss)
        # transport "nvlink": no NCCL in the step -- the library's kernels read the peers'
        # symmetric buffers over NVLink (asm_step_p2p).  Needs the global batch up front.
        self.transport = transport
        self._p2p = None
        if transport == "nvlink" and self.world > 1:
            if batch_global is None:
                raise ValueError("transport='nvlink' needs batch_global (rows of the gathered batch)")
            self._p2p = self._attach_p2p(batch_global)
        elif transport not in ("nccl", "nvlink"):
            raise ValueError("transport must be 'nccl' or 'nvlink'")

    # ---- collectives (torch.distributed plumbing) ------------------------------------
    def _all_gather(self, t: torch.Tensor) -> torch.Tensor:
        if self.world == 1:
            return t
        t = t.contiguous()
        out = torch.empty((self.world * t.shape[0],) + tuple(t.shape[1:]), device=t.device, dtype=t.dtype)
        dist.all_gather_into_tensor(out, t, group=self.group)      # concatenated along dim 0
        return out.view((self.world,) + tuple(t.shape))

    def _reduce_scatter_rows(self, full: torch.Tensor, rows_local: int) -> torch.Tensor:
        if self.world == 1:
            return full
        out = torch.empty(rows_local, full.shape[1], device=full.device, dtype=full.dtype)
        if dist.get_backend(self.group) == "gloo":      # gloo has no reduce_scatter
            dist.all_reduce(full, group=self.group)
            out.copy_(full[self.rank * rows_local:(self.rank + 1) * rows_local])
        else:
            dist.reduce_scatter_tensor(out, full, group=self.group)
        return out

    # ---- NVLink peer-memory transport ------------------------------------------------------
    def _attach_p2p(self, batch_global: int, tag="p2p"):
        import torch.distributed._symmetric_memory as symm_mem
        D, C_total, C_local, lo, m, mode, rank, world = self.compute.args
        h = get_handle(self.device, D, C_total, C_local, lo, batch_global, m, mode, rank, world,
                       tag=(tag, id(self)), margin=self.margin, loss=self.loss)
        nbytes = int(h.lib.asm_p2p_bytes(C.byref(h.cfg)))
        if nbytes == 0:
            raise RuntimeError("asm_p2p_bytes: unsupported configuration (2..8 ranks)")
        buf = symm_mem.empty(nbytes, dtype=torch.uint8, device=self.device)
        buf.zero_()
        hdl = symm_mem.rendezvous(buf, self.group if self.group is not None else dist.group.WORLD)
        torch.cuda.synchronize(self.device)
        dist.barrier(group=self.group)            # every block is zero before anyone signals
        ptrs = (C.c_void_p * world)(*[int(p) for p in hdl.buffer_ptrs])
        _lib.check(h.lib.asm_p2p_attach(h.ptr, ptrs), h.ptr)
        return dict(handle=h, buf=buf, hdl=hdl, batch=batch_global)

    def _step_p2p(self, embeddings_local, labels_local, lam, p2p=None, optimizer=None):
        p2p = p2p or self._p2p
        h = p2p["handle"]
        X = embeddings_local.contiguous()
        y = labels_local.contiguous()
        b = X.shape[0]
        loss = torch.empty(1, device=X.device, dtype=torch.float32)
        dX = torch.empty(X.shape, device=X.device, dtype=torch.float32)
        dW = torch.empty_like(self.weights) if optimizer is None else None
        stream = C.c_void_p(torch.cuda.current_stream(X.device).cuda_stream)
        with torch.cuda.device(X.device):
            _lib.check(h.lib.asm_set_embedding_dtype(h.ptr, X.element_size()), h.ptr)   # bf16 rows: half the NVLink bytes
            if optimizer is not None:
                optimizer._arm(h, self.weights)
            try:
                rc = h.lib.asm_step_p2p(h.ptr, X.data_ptr(), b, y.data_ptr(), y.element_size(),
                                        self.weights.data_ptr(), lam, loss.data_ptr(), dX.data_ptr(),
                                        dW.data_ptr() if dW is not None else None, stream)
            finally:
                if optimizer is not None:
                    optimizer._disarm(h)
            _lib.check(rc, h.ptr)
        return loss[0], dX, dW

    # ---- one training step of the head -------------------------------------------------
    def step(self, embeddings_local: torch.Tensor, labels_local: torch.Tensor, lambda_state=None,
             optimizer=None, center: Optional[dict] = None):
        """embeddings_local [B/G, D], labels_local [B/G] (this rank's data-parallel slice,
        data_parallel.py:206-207).  Returns (loss, dX_local [B/G, D], dW_local [D, C_local]);
        loss is the global-batch mean and identical on every rank.
        With `optimizer` (a FusedOptimizer owned by this rank) the shard's weights and optimizer
        state are updated in place inside the dW kernel and dW_local is None: this is the
        per-tower `apply_gradients` of data_parallel.py:186-196 without the G-fold redundancy --
        each class column is updated exactly once, on the rank that owns it.
        `center` = dict(centers=[C_local, D] shard, alpha=.., weight=..) adds the class-sharded
        center loss (loss.py:29-45) on the same gathered batch: the shard's centers are updated in
        place, its gradient joins the dX contribution before the reduce-scatter, and the returned
        loss becomes (cross_entropy or focal loss, center_loss summed over the shards).  Host-collective
        transport only."""
        lam = _as_lambda(lambda_state) if lambda_state is not None else self.lambda_state.step()
        if self._p2p is not None:
            if center is not None:
                raise ValueError("the center loss runs with transport='nccl' (it needs the gathered batch on the host side)")
            return self._step_p2p(embeddings_local, labels_local, lam, optimizer=optimizer)
        b = embeddings_local.shape[0]
        X = self._all_gather(embeddings_local).reshape(-1, self.D)
        y = self._all_gather(labels_local).reshape(-1)
        stats = self.compute.forward_partial(X, y, self.weights, lam)             # [3, B]
        stats_all = self._all_gather(stats).reshape(self.world, 3, X.shape[0])    # [G, 3, B]
        if optimizer is not None:
            loss, dX_partial, dW = self.compute.backward_partial(stats_all, X, self.weights, optimizer=optimizer)
        else:
            loss, dX_partial, dW = self.compute.backward_partial(stats_all, X, self.weights)
        if center is not None:
            from .center import center_loss
            closs, _ = center_loss(X, y, center["centers"], center.get("alpha", 0.99), center.get("weight", 1.0),
                                   class_offset=self.lo, grad_accum=dX_partial)
            if self.world > 1:
                closs = closs.clone()
                dist.all_reduce(closs, group=self.group)
            loss = (loss, closs)
        dX_local = self._reduce_scatter_rows(dX_partial, b)
        return loss, dX_local, dW

    # ---- CUDA-graph replay of the whole sharded step (collectives included) --------------
    def capture(self, batch_local: int, labels_dtype=torch.int32):
        """Capture step() for a fixed local batch into a CUDA graph.  Afterwards
        `step_graphed(X_local, y_local, lam)` copies the inputs into static buffers and
        replays: one graph launch instead of 3 collectives + 11 kernel launches."""
        dev = self.device
        self._gX = torch.zeros(batch_local, self.D, device=dev, dtype=torch.float32)
        self._gy = torch.zeros(batch_local, device=dev, dtype=labels_dtype)
        self._glam = torch.zeros(1, device=dev, dtype=torch.float32)
        self._glam_host = torch.zeros(1, dtype=torch.float32).pin_memory()
        if self._p2p is not None:
            # NVLink transport: a second symmetric block + handle whose kernels read lambda from
            # the device scalar; the captured graph contains no NCCL node at all
            p2pg = self._attach_p2p(batch_local * self.world, tag="p2pgraph")
            hg = p2pg["handle"]
            _lib.check(hg.lib.asm_set_lambda_device(hg.ptr, self._glam.data_ptr()), hg.ptr)
            self._p2pg = p2pg
            cur = torch.cuda.current_stream(dev)
            side = torch.cuda.Stream(dev)
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                for _ in range(3):
                    self._step_p2p(self._gX, self._gy, 0.0, p2p=p2pg)
            cur.wait_stream(side)
            torch.cuda.synchronize(dev)
            dist.barrier(group=self.group)
            self._graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self._graph):
                self._gout = self._step_p2p(self._gX, self._gy, 0.0, p2p=p2pg)
            return self
        # a dedicated shard-compute object (own handle / workspace) whose kernels read lambda
        # from the device scalar; the eager step() keeps its own by-value handle
        eager_compute = self.compute
        gcompute = _CudaShard(self.D, self.C, self.lo, self.hi, self.m, self.mode, self.rank,
                              self.world, self.device, self.margin, self.loss)
        gcompute.tag = ("graph", id(self))
        gcompute.lambda_dev = self._glam
        self.compute = gcompute
        try:
            cur = torch.cuda.current_stream(dev)
            side = torch.cuda.Stream(dev)
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                for _ in range(3):
                    self.step(self._gX, self._gy, 0.0)
            cur.wait_stream(side)
            torch.cuda.synchronize(dev)
            self._graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self._graph):
                self._gout = self.step(self._gX, self._gy, 0.0)
        finally:
            self.compute = eager_compute
        return self

    def step_graphed(self, embeddings_local, labels_local, lambda_state=None):
        lam = _as_lambda(lambda_state) if lambda_state is not None else self.lambda_state.step()
        self._glam_host[0] = lam
        self._glam.copy_(self._glam_host, non_blocking=True)
        self._gX.copy_(embeddings_local, non_blocking=True)
        self._gy.copy_(labels_local, non_blocking=True)
        self._graph.replay()
        return self._gout

    def gather_shard(self, shard: torch.Tensor) -> torch.Tensor:
        """Any class-sharded [D, C_local] tensor (the weights, an optimizer slot) -> [D, C] on every rank."""
        if self.world == 1:
            return shard.clone()
        per = -(-self.C // self.world)
        pad = torch.zeros(self.D, per, device=shard.device, dtype=torch.float32)
        pad[:, : self.hi - self.lo] = shard
        allw = self._all_gather(pad)                                     # [G, D, per]
        return allw.permute(1, 0, 2).reshape(self.D, -1)[:, : self.C].contiguous()

    def gather_weights(self) -> torch.Tensor:
        """All shards -> one [D, C] fp32 tensor (`classifier/fc_classifier/weights`, the
        layout saver.py:36-40 writes), for checkpoint compatibility."""
        return self.gather_shard(self.weights)

    # ---- checkpoint layout (saver.py:30-80) ------------------------------------------------
    VARIABLE_NAME = "classifier/fc_classifier/weights"      # nets/sphere.py:84-90

    def state_dict(self) -> dict:
        """What DataParallelSaverBuilder.save_op writes for the classifier: ONE [D, C] fp32
        tensor under the variable name with the tower prefix (`replicated_<k>/`) stripped
        (saver.py:36-40).  Collective: every rank must call it; every rank gets the full tensor."""
        return {self.VARIABLE_NAME: self.gather_weights()}

    def load_weights(self, weights_full: torch.Tensor) -> None:
        """Inverse of gather_weights(): keep this rank's class slice of a [D, C] tensor.  The
        shard is overwritten in place, so captured CUDA graphs keep pointing at it."""
        if tuple(weights_full.shape) != (self.D, self.C):
            raise ValueError(f"expected weights [{self.D}, {self.C}], got {tuple(weights_full.shape)}")
        self.weights.copy_(weights_full[:, self.lo:self.hi].to(torch.float32))

    def load_state_dict(self, state: dict) -> None:
        """Restore from a reference-format checkpoint dict.  Accepts the stripped name or any
        `replicated_<k>/...` spelling of it (restore_op strips the first path component for
        tower variables, saver.py:62-72); tower 0 wins if several are present."""
        found = None
        for name in sorted(state.keys()):
            base = "/".join(name.split("/")[1:]) if name.startswith("replicated_") else name
            if base == self.VARIABLE_NAME:
                found = state[name]
                break
        if found is None:
            raise KeyError(f"no '{self.VARIABLE_NAME}' (or replicated_<k>/ variant) in checkpoint")
        self.load_weights(torch.as_tensor(found))
