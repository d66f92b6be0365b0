"""The focal loss (asm_set_loss, FocalLoss) on the B200 against the float64 oracle
(oracle/focal_ref.py), with the bounds of tests/head_checks.py, on every path the head runs:
bf16 and fp32 tensor cores, the CUDA-core fp32 kernels (D % 64 != 0, and ASM_FP32_SIMT=1),
A-softmax / ArcFace / CosFace, the features the loss combines with and the class-sharded paths.
Also: FocalLoss(1, 0) keeps the cross-entropy's bits, a row whose focal weight is zero stays
finite, invalid parameters are refused, and the CUDA-core recompute applies grad_scale."""
import ctypes as C
import functools
import os

import numpy as np
import pytest
import torch

from head_checks import LOSS_TOL, assert_within_oracle_bounds, cosine
from oracle import asoftmax_ref as ref
from oracle import focal_ref as fr
from test_oracle_margins_cpu import spread_inputs
from test_p2p_gpu import FakeRanks
from tf_face_toolbox_b200 import (AdditiveMargin, FocalLoss, FusedOptimizer, GraphedASoftmaxStep,
                                  ShardedASoftmaxHead, _lib, asoftmax_head)
from tf_face_toolbox_b200.head import _HANDLES, drop_handle, get_handle
from tf_face_toolbox_b200.synthetic import make_inputs

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
# head -> (m, lambda, AdditiveMargin or None)
HEADS = {"asoftmax": (4, 5.0, None), "arcface": (4, 0.0, AdditiveMargin.arcface(64.0, 0.5)),
         "cosface": (4, 0.0, AdditiveMargin.cosface(64.0, 0.35))}
# path -> (mode, D of the "edge" shape, D of the "wide" shape, ASM_FP32_SIMT)
PATHS = {"bf16": ("bf16", 128, 512, False), "fp32": ("fp32", 128, 512, False),
         "d80": ("fp32", 80, 80, False), "simt": ("fp32", 128, 512, True)}
# B not a multiple of 128 with C % 4 == 2, and a BASELINE-like shape
SHAPES = {"edge": (130, 1002), "wide": (256, 4000)}


@functools.lru_cache(maxsize=None)
def inputs(head, B, D, Cn, seed=21):
    mg = HEADS[head][2]
    if mg is None:
        return make_inputs(B, D, Cn, seed=seed)
    return spread_inputs(B, D, Cn, seed=seed, m2=mg.m2)


def _mg_tuple(mg):
    return None if mg is None else (mg.s, mg.m2, mg.m3)


def oracle_of(head, X, W, y, gamma, alpha):
    m, lam, mg = HEADS[head]
    return fr.focal_head(X, W, y, gamma, alpha, m, lam, _mg_tuple(mg))


@functools.lru_cache(maxsize=None)
def oracle(head, B, D, Cn, gamma, alpha):
    inp = inputs(head, B, D, Cn)
    return oracle_of(head, inp.X.numpy(), inp.W.numpy(), inp.y.numpy(), gamma, alpha)


def make_handle(head, path, B, D, Cn, loss, tag):
    """The handle `tag` names, created with the path's environment (ASM_FP32_SIMT is read at creation)."""
    mode, _, _, simt = PATHS[path]
    old = os.environ.get("ASM_FP32_SIMT")
    if simt:
        os.environ["ASM_FP32_SIMT"] = "1"
    try:
        return get_handle(DEV, D, Cn, Cn, 0, B, HEADS[head][0], mode, tag=tag, margin=HEADS[head][2], loss=loss)
    finally:
        if simt:
            if old is None:
                os.environ.pop("ASM_FP32_SIMT")
            else:
                os.environ["ASM_FP32_SIMT"] = old


def run(inp, head, path, loss, tag=None, grads=True, X=None, W=None, **kw):
    m, lam, mg = HEADS[head]
    mode = PATHS[path][0]
    X = inp.X.to(DEV) if X is None else X
    W = inp.W.to(DEV) if W is None else W
    tag = ("focal", path, tag)
    make_handle(head, path, X.shape[0], X.shape[1], W.shape[1], loss, tag)
    out, _, dX, dW = asoftmax_head(X, inp.y.to(DEV), W.shape[1], m, lam, weights=W, mode=mode, compute_grads=grads,
                                   margin=mg, loss=loss, _handle_tag=tag, **kw)
    torch.cuda.synchronize()
    cpu = lambda t: None if t is None else t.cpu().numpy()      # noqa: E731
    return float(out), cpu(dX), cpu(dW)


def check(inp, r, mode, out):
    loss, dX, dW = out
    assert_within_oracle_bounds(inp, r, mode, loss, None, dX, dW)


def bitwise(a, b):
    assert a[0] == b[0] or (np.isnan(a[0]) and np.isnan(b[0])), (a[0], b[0])
    for x, y in zip(a[1:], b[1:]):
        assert (x is None) == (y is None)
        if x is not None:
            assert np.array_equal(x, y)


def shape(path, name):
    B, Cn = SHAPES[name]
    return B, PATHS[path][1 if name == "edge" else 2], Cn


@pytest.fixture(autouse=True)
def _drop_handles():
    yield
    for k in [k for k in _HANDLES if isinstance(k[-1], tuple) and k[-1][:1] == ("focal",)]:
        drop_handle(_HANDLES[k])


# ----------------------------------------------------------------------------- coverage matrix
@pytest.mark.parametrize("name", sorted(SHAPES))
@pytest.mark.parametrize("alpha", [0.5, 2.0])
@pytest.mark.parametrize("path", sorted(PATHS))
@pytest.mark.parametrize("head", sorted(HEADS))
def test_matrix(head, path, alpha, name):
    B, D, Cn = shape(path, name)
    inp = inputs(head, B, D, Cn)
    fl = FocalLoss(0.75, alpha)
    r = oracle(head, B, D, Cn, 0.75, alpha)
    mode = PATHS[path][0]
    loss, dX, dW = run(inp, head, path, fl)
    assert_within_oracle_bounds(inp, r, mode, loss, None, dX, dW)
    # asm_forward: the focal loss alone, the same value as the step's
    loss_only, none, _ = run(inp, head, path, fl, grads=False)
    assert none is None
    assert abs(loss_only - r.loss) <= LOSS_TOL[mode] * abs(r.loss), (loss_only, r.loss)
    assert loss_only == loss


@pytest.mark.parametrize("path", sorted(PATHS))
@pytest.mark.parametrize("head", sorted(HEADS))
def test_gamma1_alpha0_keeps_cross_entropy_bits(head, path):
    """w_i = 1 exactly: the focal branch adds log2(1) = 0 and multiplies by 1."""
    B, D, Cn = shape(path, "edge")
    inp = inputs(head, B, D, Cn)
    ce = run(inp, head, path, None)
    bitwise(ce, run(inp, head, path, FocalLoss(1.0, 0.0)))
    bitwise(run(inp, head, path, None, grads=False), run(inp, head, path, FocalLoss(1.0, 0.0), grads=False))


# ----------------------------------------------------------------------------- other features
@pytest.mark.parametrize("path", ["bf16", "fp32", "d80", "simt"])
def test_gradient_transform(path):
    """dX, dW = grad_scale * d(focal)/d. (+ grad_scale * wd * W on dW); the loss stays unscaled."""
    head = "arcface" if path != "simt" else "asoftmax"
    B, D, Cn = shape(path, "wide")
    inp = inputs(head, B, D, Cn)
    r = oracle(head, B, D, Cn, 0.75, 2.0)
    reg = torch.zeros(1, device=DEV)
    loss, dX, dW = run(inp, head, path, FocalLoss(0.75, 2.0), grad_scale=0.25, weight_decay=5e-4, reg_loss_out=reg)
    W = inp.W.double().numpy()
    want = fr.FocalResult(r.loss, r.logits, 0.25 * r.dX, 0.25 * (r.dW + 5e-4 * W), r.c, r.ce, r.w)
    assert_within_oracle_bounds(inp, want, PATHS[path][0], loss, None, dX, dW)
    assert float(reg) == pytest.approx(2.5e-4 * (W * W).sum(), rel=1e-4)


@pytest.mark.parametrize("path", ["d80", "simt"])
def test_cuda_core_recompute_applies_grad_scale(path):
    """Cross-entropy on the CUDA-core kernels with grad_scale = 0.125: every part of dX and dW is
    scaled, the non-target softmax gradient of the recompute kernel included."""
    head = "asoftmax"
    B, D, Cn = shape(path, "edge")
    inp = inputs(head, B, D, Cn)
    r = ref.asoftmax_head(inp.X.numpy(), inp.W.numpy(), inp.y.numpy(), 4, 5.0)
    loss, dX, dW = run(inp, head, path, None, grad_scale=0.125)
    want = ref.HeadResult(r.loss, r.logits, 0.125 * r.dX, 0.125 * r.dW, r.n, r.c, r.t, r.psi, r.row_max, r.row_logz)
    assert_within_oracle_bounds(inp, want, "fp32", loss, None, dX, dW)


@pytest.mark.parametrize("kind", ["Momentum", "Adam"])
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_fused_optimizer_three_steps(kind, mode):
    head = "asoftmax" if kind == "Momentum" else "cosface"
    m, lam, mg = HEADS[head]
    fl = FocalLoss(0.75, 2.0)
    B, D, Cn = 128, 128, 3000
    inp = inputs(head, B, D, Cn)
    lr = 0.05 if kind == "Momentum" else 1e-3
    opt = FusedOptimizer(kind, lr=lr, weight_decay=5e-4)
    W_f = inp.W.to(DEV).clone()
    Wr = inp.W.double().numpy().copy()
    s0, s1 = np.zeros_like(Wr), np.zeros_like(Wr)
    X = inp.X.to(DEV)
    for step in range(1, 4):
        Wcur = torch.from_numpy(Wr).float().to(DEV)
        _, _, dW = run(inp, head, mode, fl, tag="opt-ref", W=Wcur)
        Wr, s0, s1n = ref.optimizer_step(Wcur.double().cpu().numpy(), dW, s0, s1, kind.lower(), lr=lr, step=step)
        s1 = s1n if s1n is not None else s1
        loss, _, _, none = asoftmax_head(X, inp.y.to(DEV), Cn, m, lam, weights=W_f, mode=mode, optimizer=opt,
                                         margin=mg, loss=fl, _handle_tag=("focal", "opt"))
        assert none is None and np.isfinite(float(loss))
        torch.cuda.synchronize()
        upd_f = W_f.double().cpu().numpy() - inp.W.double().numpy()
        upd_r = Wr - inp.W.double().numpy()
        assert cosine(upd_f, upd_r) >= (0.999 if (kind, mode) == ("Adam", "bf16") else 0.9999), step


def test_bf16_embeddings():
    head = "arcface"
    B, D, Cn = 256, 512, 4000
    inp = inputs(head, B, D, Cn)
    inp = type(inp)(inp.X.to(torch.bfloat16).float(), inp.W, inp.y)     # exactly representable
    fl = FocalLoss(0.75, 2.0)
    a = run(inp, head, "bf16", fl)
    b = run(inp, head, "bf16", fl, X=inp.X.to(DEV).to(torch.bfloat16))
    r = oracle_of(head, inp.X.numpy(), inp.W.numpy(), inp.y.numpy(), 0.75, 2.0)
    check(inp, r, "bf16", b)
    np.testing.assert_allclose(b[1], a[1], rtol=1e-4, atol=1e-6 * np.abs(a[1]).max())


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
@pytest.mark.parametrize("head", ["asoftmax", "arcface"])
def test_graph_replay_and_determinism(head, mode):
    m, lam, mg = HEADS[head]
    fl = FocalLoss(0.75, 2.0)
    B, D, Cn = 256, 512, 4000
    inp = inputs(head, B, D, Cn)
    W = inp.W.to(DEV)
    step = GraphedASoftmaxStep(W, B, m=m, mode=mode, margin=mg, loss=fl)
    try:
        loss, dX, dW = step(inp.X.to(DEV), inp.y.to(DEV), lam)
        torch.cuda.synchronize()
        got = (float(loss), dX.cpu().numpy(), dW.cpu().numpy())
        eager = run(inp, head, mode, fl)
        bitwise(eager, run(inp, head, mode, fl))                 # two runs, same bits
        bitwise(eager, got)
        check(inp, oracle(head, B, D, Cn, 0.75, 2.0), mode, got)
    finally:
        step.close()


# ----------------------------------------------------------------------------- edge rows, argument checks
@pytest.mark.parametrize("alpha", [0.5, 20.0])
@pytest.mark.parametrize("path", ["bf16", "fp32", "d80"])
def test_zero_weight_row_stays_finite(path, alpha):
    """Row 0 lies so far along w_{y_0} that every other class's exp underflows: Z_0 = 1 and ce_0 = 0
    on the CUDA-core path, so w_0 = 0 and negoff_0 = -inf.  (The tensor-core forward sums the target's
    own exp2 with a rounding residual, so there ce_0 is tiny instead; alpha = 20 then underflows w_0
    to 0 on every path.)  Row 1 has a tiny but non-zero ce."""
    head = "asoftmax"
    B, D, Cn = shape(path, "edge")
    inp = inputs(head, B, D, Cn)
    X = inp.X.clone()
    for i, n in ((0, 1000.0), (1, 20.0)):
        w = inp.W[:, inp.y[i].long()]
        X[i] = n * w / w.norm()
    inp = type(inp)(X, inp.W, inp.y)
    r = oracle_of(head, X.numpy(), inp.W.numpy(), inp.y.numpy(), 0.75, alpha)
    assert r.ce[0] < 1e-12 and r.w[0] < 1e-30 and 0 < r.ce[1] < 1e-2, (r.ce[:2], r.w[:2])
    loss, dX, dW = run(inp, head, path, FocalLoss(0.75, alpha))
    assert np.isfinite(loss) and np.isfinite(dX).all() and np.isfinite(dW).all()
    if path == "d80" or alpha == 20.0:
        assert not dX[0].any()                                   # the row contributes nothing
    assert_within_oracle_bounds(inp, r, PATHS[path][0], loss, None, dX, dW)


def test_invalid_parameters_and_switching_back():
    """Refused parameters leave the previous loss in effect; NULL restores the cross-entropy bit for bit."""
    head, path = "asoftmax", "bf16"
    B, D, Cn = shape(path, "wide")
    inp = inputs(head, B, D, Cn)
    fresh = run(inp, head, path, None, tag="fresh")
    h = make_handle(head, path, B, D, Cn, None, ("focal", path, "switch"))
    _lib.check(h.lib.asm_set_loss(h.ptr, C.byref(_lib.AsmLoss(_lib.LOSS_FOCAL, 0.75, 2.0))), h.ptr)
    focal = run(inp, head, path, None, tag="switch")
    check(inp, oracle(head, B, D, Cn, 0.75, 2.0), "bf16", focal)
    for bad in ((1, 0.0, 2.0), (1, -1.0, 2.0), (1, float("nan"), 2.0), (1, 1.0, -0.5), (1, 1.0, float("inf")),
                (1, float("inf"), 2.0), (1, 1.0, float("nan")), (2, 1.0, 2.0)):
        assert h.lib.asm_set_loss(h.ptr, C.byref(_lib.AsmLoss(*bad))) == _lib.ASM_ERR_INVALID_ARG, bad
    bitwise(focal, run(inp, head, path, None, tag="switch"))     # the refused calls changed nothing
    _lib.check(h.lib.asm_set_loss(h.ptr, None), h.ptr)
    bitwise(fresh, run(inp, head, path, None, tag="switch"))
    _lib.check(h.lib.asm_set_loss(h.ptr, C.byref(_lib.AsmLoss(_lib.LOSS_SOFTMAX_CE, 0.0, 0.0))), h.ptr)
    bitwise(fresh, run(inp, head, path, None, tag="switch"))
    with pytest.raises(_lib.AsmError):
        run(inp, head, path, FocalLoss(-1.0, 2.0))
    with pytest.raises(TypeError):
        run(inp, head, path, (1.0, 2.0))


# ----------------------------------------------------------------------------- class-sharded
@pytest.mark.parametrize("G", [2, 3])
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
@pytest.mark.parametrize("head", sorted(HEADS))
def test_partial_calls_host_combine(head, mode, G):
    m, lam, mg = HEADS[head]
    fl = FocalLoss(0.75, 2.0)
    B, D, Cn = 256, 512, 4000
    inp = inputs(head, B, D, Cn)
    r = oracle(head, B, D, Cn, 0.75, 2.0)
    X, y = inp.X.to(DEV), inp.y.to(DEV)
    bounds = fr.shard_bounds(Cn, G)
    hs, Ws, stats = [], [], torch.zeros(G, 3, B, device=DEV)
    for g, (lo, hi) in enumerate(bounds):
        h = get_handle(DEV, D, Cn, hi - lo, lo, B, m, mode, g, G, tag=("focal", "part", g), margin=mg, loss=fl)
        Ws.append(inp.W[:, lo:hi].contiguous().to(DEV))
        _lib.check(h.lib.asm_forward_partial(h.ptr, X.data_ptr(), B, y.data_ptr(), 4, Ws[g].data_ptr(), lam,
                                             stats[g].data_ptr(), None, None), h.ptr)
        hs.append(h)
    dX = torch.zeros(B, D, device=DEV)
    losses = []
    for g, h in enumerate(hs):
        loss = torch.zeros(1, device=DEV)
        dXp = torch.empty(B, D, device=DEV)
        dW = torch.empty_like(Ws[g])
        _lib.check(h.lib.asm_backward_partial(h.ptr, stats.data_ptr(), G, loss.data_ptr(), dXp.data_ptr(),
                                              dW.data_ptr(), None), h.ptr)
        dX += dXp
        lo, hi = bounds[g]
        torch.cuda.synchronize()
        losses.append(float(loss))
        sub = fr.FocalResult(r.loss, None, r.dX, r.dW[:, lo:hi], r.c[lo:hi], r.ce, r.w)
        assert_within_oracle_bounds(inp, sub, mode, float(loss), None, r.dX, dW.cpu().numpy())
    assert len(set(losses)) == 1, losses                          # every shard, the same loss bits
    torch.cuda.synchronize()
    assert_within_oracle_bounds(inp, r, mode, losses[0], None, dX.cpu().numpy(), r.dW)


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_sharded_head_host_collective(mode):
    """ShardedASoftmaxHead(loss=...) on one GPU: the host-collective step, eager and graph-captured."""
    head = "cosface"
    m, lam, mg = HEADS[head]
    fl = FocalLoss(0.75, 2.0)
    B, D, Cn = 256, 512, 4000
    inp = inputs(head, B, D, Cn)
    sh = ShardedASoftmaxHead(D, Cn, m=m, mode=mode, device=DEV, weights_full=inp.W, margin=mg, loss=fl)
    loss, dX, dW = sh.step(inp.X.to(DEV), inp.y.to(DEV), lam)
    torch.cuda.synchronize()
    eager = (float(loss), dX.cpu().numpy(), dW.cpu().numpy())
    check(inp, oracle(head, B, D, Cn, 0.75, 2.0), mode, eager)
    sh.capture(B)
    loss, dX, dW = sh.step_graphed(inp.X.to(DEV), inp.y.to(DEV), lam)
    torch.cuda.synchronize()
    bitwise(eager, (float(loss), dX.cpu().numpy(), dW.cpu().numpy()))


class FocalRanks(FakeRanks):
    """test_p2p_gpu's in-process ranks, with the margin and the loss set once on every rank's handle."""

    def __init__(self, inp, G, mode, tag, mg, fl):
        super().__init__(inp, G, mode, tag)
        for h in self.handles:
            if mg is not None:
                _lib.check(h.lib.asm_set_margin(h.ptr, C.byref(mg._struct())), h.ptr)
            _lib.check(h.lib.asm_set_loss(h.ptr, C.byref(fl._struct())), h.ptr)


@pytest.mark.parametrize("G", [2, 4])
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_nvlink_transport_eager_and_graph(mode, G):
    head = "arcface" if G == 2 else "asoftmax"
    m, lam, mg = HEADS[head]
    fl = FocalLoss(0.75, 0.5 if G == 2 else 2.0)
    B, D, Cn = 128, 128, 5000
    inp = inputs(head, B, D, Cn)
    r = oracle(head, B, D, Cn, fl.gamma, fl.alpha)
    ranks = FocalRanks(inp, G, mode, ("focal", "p2p", mode, G), mg, fl)
    try:
        for _ in range(3):
            ranks.step(lam)
            ranks.check(r)                                        # same loss bits on every rank
            for g, (lo, hi) in enumerate(ranks.bounds):           # every element, not only cosines
                rows = slice(g * ranks.b, (g + 1) * ranks.b)
                sub = fr.FocalResult(r.loss, None, r.dX[rows], r.dW[:, lo:hi], r.c, r.ce, r.w)
                assert_within_oracle_bounds(inp, sub, mode, float(ranks.loss[g]), None,
                                            ranks.dX[g].cpu().numpy(), ranks.dW[g].cpu().numpy())
        eager = [float(l) for l in ranks.loss]
        graphs = []
        for g in range(G):
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr, stream=ranks.streams[g]):
                ranks.enqueue(g, lam)
            graphs.append(gr)
        for _ in range(3):
            torch.cuda.synchronize()
            for g in range(G):
                with torch.cuda.stream(ranks.streams[g]):
                    graphs[g].replay()
            ranks.check(r)
            assert [float(l) for l in ranks.loss] == eager
    finally:
        for h in ranks.handles:
            drop_handle(h)
