"""The plain softmax classifier (asm_set_margin(ASM_MARGIN_LINEAR), LinearSoftmax) on the B200 against
the float64 oracle (oracle/linear_softmax_ref.py), with the bounds of tests/head_checks.py, on every
path the head runs: bf16 and fp32 tensor cores, the CUDA-core fp32 kernels, every tensor-core kernel
variant of test_kernel_variants_gpu, the features the head combines with and both class-sharded
transports.  Outputs are written into NaN-filled buffers, so an element a kernel skips fails."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from head_checks import LOSS_TOL, assert_within_oracle_bounds, cosine
from oracle import asoftmax_ref as ref
from oracle import linear_softmax_ref as lr
from test_kernel_variants_gpu import OPT_VARIANTS, TESTED_KNOBS, VARIANTS
from test_p2p_gpu import FakeRanks
from tf_face_toolbox_b200 import (ASoftmaxHead, FocalLoss, FusedOptimizer, GraphedASoftmaxStep, LinearSoftmax, _lib,
                                  asoftmax_head)
from tf_face_toolbox_b200.head import _HANDLES, drop_handle, get_handle
from tf_face_toolbox_b200.synthetic import make_inputs

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
LIN = LinearSoftmax()
TAG = "linear"


def inputs(B, D, Cn, regime="trained", seed=17):
    """'init': the reference's N(0, 0.001) weights, loss about log C.  'trained': |w_j| about
    8/sqrt(D), so that the target logits of make_inputs' mixture reach +-12 whatever D: the regime of
    a trained classifier.  (Much larger margins make 1 - p_iy smaller than the fp32 resolution of
    the sum-exp, where no fp32 softmax, the reference's included, resolves the target gradient.)"""
    return make_inputs(B, D, Cn, seed=seed + B + Cn, w_std=0.001 if regime == "init" else 8.0 / D)


def oracle(inp):
    return lr.linear_head(inp.X.numpy(), inp.W.numpy(), inp.y.numpy())


def handle(D, Cn, B, mode, name, simt=False, loss=None):
    old = os.environ.get("ASM_FP32_SIMT")
    if simt:
        os.environ["ASM_FP32_SIMT"] = "1"                  # read by asm_create
    try:
        return get_handle(DEV, D, Cn, Cn, 0, B, 4, mode, tag=(TAG, name, simt), margin=LIN, loss=loss)
    finally:
        if simt:
            if old is None:
                os.environ.pop("ASM_FP32_SIMT")
            else:
                os.environ["ASM_FP32_SIMT"] = old


def run_h(h, inp, logits=False, grads=True, W=None):
    """One asm_forward_backward (or asm_forward) on `h` into NaN-filled output buffers."""
    B, D = inp.X.shape
    X, y = inp.X.to(DEV), inp.y.to(DEV)
    W = inp.W.to(DEV) if W is None else W
    Cn = W.shape[1]
    nan = float("nan")
    loss = torch.full((1,), nan, device=DEV)
    f = torch.full((B, Cn), nan, device=DEV) if logits else None
    dX = torch.full((B, D), nan, device=DEV) if grads else None
    dW = torch.full((D, Cn), nan, device=DEV) if grads else None
    stream = torch.cuda.current_stream().cuda_stream
    fp = f.data_ptr() if logits else None
    with torch.cuda.device(DEV):
        if grads:
            rc = h.lib.asm_forward_backward(h.ptr, X.data_ptr(), B, y.data_ptr(), 4, W.data_ptr(), 5.0, loss.data_ptr(),
                                            fp, dX.data_ptr(), dW.data_ptr(), stream)
        else:
            rc = h.lib.asm_forward(h.ptr, X.data_ptr(), B, y.data_ptr(), 4, W.data_ptr(), 5.0, loss.data_ptr(), fp, stream)
        _lib.check(rc, h.ptr)
    torch.cuda.synchronize()
    cpu = lambda t: None if t is None else t.cpu().numpy()      # noqa: E731
    return float(loss.item()), cpu(f), cpu(dX), cpu(dW)


def run(inp, mode, name="main", simt=False, **kw):
    B, D = inp.X.shape
    return run_h(handle(D, inp.W.shape[1], B, mode, name, simt), inp, **kw)


def assert_linear_logits(inp, mode, f):
    """Every logit against x_i . w_j in float64, bounded by the rounding of the operands:
    |f_ij - x_i.w_j| <= tol |x_i| |w_j| (Cauchy-Schwarz scale of the products)."""
    X, W = inp.X.double().numpy(), inp.W.double().numpy()
    exact = X @ W
    scale = np.linalg.norm(X, axis=1)[:, None] * np.linalg.norm(W, axis=0)[None, :]
    tol = 1e-5 if mode == "fp32" else 2.0 ** -7
    err = np.abs(f - exact)
    assert (err <= tol * scale + 1e-6).all(), float((err / scale).max())


def check(inp, mode, out, r=None, grads=True, loss_floor=None):
    loss, f, dX, dW = out
    r = oracle(inp) if r is None else r
    floor = (1.0 if inp.X.shape[0] > 1 else 10.0) if loss_floor is None else loss_floor
    assert np.isfinite(loss)
    if grads:
        assert_within_oracle_bounds(inp, r, mode, loss, None, dX, dW, loss_floor=floor)
        if mode == "bf16":
            ew = np.abs(dW - r.dW).max() / np.abs(r.dW).max()
            assert ew <= 2e-2, ew                                   # every element of dW within 2 %
    else:
        assert abs(loss - r.loss) <= LOSS_TOL[mode] * max(abs(r.loss), floor), (loss, r.loss)
    if f is not None:
        assert_linear_logits(inp, mode, f)


def bitwise(a, b):
    assert a[0] == b[0] or (np.isnan(a[0]) and np.isnan(b[0])), (a[0], b[0])
    for x, y in zip(a[1:], b[1:]):
        assert (x is None) == (y is None)
        if x is not None:
            assert np.array_equal(x, y)


@pytest.fixture(autouse=True)
def _drop_handles(monkeypatch):
    for k in TESTED_KNOBS:
        monkeypatch.delenv(k, raising=False)
    yield monkeypatch
    for k in [k for k in _HANDLES if isinstance(k[-1], tuple) and k[-1][:1] == (TAG,)]:
        drop_handle(_HANDLES[k])


# ----------------------------------------------------------------------------- coverage matrix
@pytest.mark.parametrize("D", [128, 512])
@pytest.mark.parametrize("Cn", [200, 3002, 10572])
@pytest.mark.parametrize("B", [1, 129, 512])
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_matrix(mode, B, Cn, D):
    inp = inputs(B, D, Cn)
    logits = Cn <= 3002
    check(inp, mode, run(inp, mode, logits=logits))
    if B == 129:
        check(inp, mode, run(inp, mode, grads=False, logits=logits), grads=False)


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
@pytest.mark.parametrize("B,Cn,D", [(129, 3002, 128), (512, 10572, 512)])
def test_reference_init_regime(mode, B, Cn, D):
    """N(0, 0.001) weights (nets/sphere.py:87): loss about log C, logits near zero."""
    inp = inputs(B, D, Cn, "init")
    r = oracle(inp)
    assert abs(r.loss - np.log(Cn)) < 0.1
    out = run(inp, mode, logits=Cn <= 3002)
    check(inp, mode, out, r)


@pytest.mark.parametrize("B", [1, 129, 512])
@pytest.mark.parametrize("Cn", [200, 3002, 10572])
@pytest.mark.parametrize("path", ["d80", "simt"])
def test_cuda_core_path(path, Cn, B):
    """D % 64 != 0, and ASM_FP32_SIMT=1 at D = 128: fp32 on the CUDA cores."""
    D = 80 if path == "d80" else 128
    inp = inputs(B, D, Cn)
    check(inp, "fp32", run(inp, "fp32", simt=path == "simt", logits=Cn <= 3002))
    if B == 129:
        check(inp, "fp32", run(inp, "fp32", simt=path == "simt", grads=False), grads=False)


# ----------------------------------------------------------------------------- kernel variants
VARIANT_SHAPES = [(129, 192, 1001), (256, 512, 4000), (512, 512, 3002)]


@pytest.mark.parametrize("B,D,Cn", VARIANT_SHAPES)
@pytest.mark.parametrize("variant,mode", [(v, m) for v, (_, modes, _) in VARIANTS.items() for m in modes])
def test_kernel_variant(variant, mode, B, D, Cn, _drop_handles):
    env, _, _ = VARIANTS[variant]
    for k, v in env.items():
        _drop_handles.setenv(k, v)
    inp = inputs(B, D, Cn)
    h = get_handle(DEV, D, Cn, Cn, 0, B, 4, mode, tag=(TAG, "variant", variant), margin=LIN)
    a = run_h(h, inp, logits=Cn == 1001)
    check(inp, mode, a)
    bitwise(a, run_h(h, inp, logits=Cn == 1001))


def fused_optimizer_three_steps(kind, mode, name):
    inp = inputs(128, 128, 3000)
    lrate = 0.05 if kind == "Momentum" else 1e-3
    opt = FusedOptimizer(kind, lr=lrate, weight_decay=5e-4)
    W_f = inp.W.to(DEV).clone()
    Wr = inp.W.double().numpy().copy()
    s0, s1 = np.zeros_like(Wr), np.zeros_like(Wr)
    X, y = inp.X.to(DEV), inp.y.to(DEV)
    for step in range(1, 4):
        Wcur = torch.from_numpy(Wr).float().to(DEV)
        _, _, _, dW = asoftmax_head(X, y, 3000, 4, 0.0, weights=Wcur, mode=mode, margin=LIN,
                                    _handle_tag=(TAG, "opt-ref", name))
        Wr, s0, s1n = ref.optimizer_step(Wcur.double().cpu().numpy(), dW.double().cpu().numpy(), s0, s1, kind.lower(),
                                         lr=lrate, step=step)
        s1 = s1n if s1n is not None else s1
        loss, _, _, none = asoftmax_head(X, y, 3000, 4, 0.0, weights=W_f, mode=mode, optimizer=opt, margin=LIN,
                                         _handle_tag=(TAG, "opt", name))
        assert none is None and np.isfinite(float(loss))
        torch.cuda.synchronize()
        upd_f = W_f.double().cpu().numpy() - inp.W.double().numpy()
        upd_r = Wr - inp.W.double().numpy()
        assert cosine(upd_f, upd_r) >= (0.999 if (kind, mode) == ("Adam", "bf16") else 0.9999), step
        if kind == "Momentum":
            np.testing.assert_allclose(upd_f, upd_r, rtol=0, atol=(2e-3 if mode == "fp32" else 3e-2) * np.abs(upd_r).max())


@pytest.mark.parametrize("kind", ["Momentum", "Adam"])
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
@pytest.mark.parametrize("variant", ["default"] + list(OPT_VARIANTS))
def test_fused_optimizer_three_steps(variant, mode, kind, _drop_handles):
    """The update fused into the dW kernel (and the streaming update) equals grad-then-update."""
    for k, v in OPT_VARIANTS.get(variant, {}).items():
        _drop_handles.setenv(k, v)
    fused_optimizer_three_steps(kind, mode, variant)


# ----------------------------------------------------------------------------- semantics
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_zero_column_and_bad_label(mode):
    """A zero column of W is an ordinary class with logit 0 (not a masked one), and its dW column is
    X^T g; a label outside [0, C) gives a NaN loss."""
    inp = inputs(129, 128, 3002)
    W = inp.W.clone()
    W[:, 7] = 0.0
    y = inp.y.clone()
    y[y == 7] = 8
    inp = type(inp)(inp.X, W, y)
    out = run(inp, mode, logits=True)
    check(inp, mode, out)
    assert np.all(out[1][:, 7] == 0.0)
    assert np.abs(out[3][:, 7]).max() > 0.0
    bad = y.clone()
    bad[5] = 3002
    loss = run(type(inp)(inp.X, W, bad), mode)[0]
    assert np.isnan(loss)


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_gradient_transform(mode):
    inp = inputs(256, 512, 4000)
    reg = torch.zeros(1, device=DEV)
    loss, _, dX, dW = asoftmax_head(inp.X.to(DEV), inp.y.to(DEV), 4000, 4, 0.0, weights=inp.W.to(DEV), mode=mode,
                                    margin=LIN, grad_scale=0.25, weight_decay=5e-4, reg_loss_out=reg,
                                    _handle_tag=(TAG, "transform"))
    torch.cuda.synchronize()
    r = oracle(inp)
    W = inp.W.double().numpy()
    want = type(r)(r.loss, r.logits, 0.25 * r.dX, 0.25 * (r.dW + 5e-4 * W), r.ce, r.w)
    check(inp, mode, (float(loss), None, dX.cpu().numpy(), dW.cpu().numpy()), want)
    assert float(reg) == pytest.approx(2.5e-4 * (W * W).sum(), rel=1e-4)


def test_bf16_embeddings():
    inp = inputs(256, 512, 4000)
    inp = type(inp)(inp.X.to(torch.bfloat16).float(), inp.W, inp.y)     # exactly representable
    tag = (TAG, "x16")
    a = asoftmax_head(inp.X.to(DEV), inp.y.to(DEV), 4000, weights=inp.W.to(DEV), mode="bf16", margin=LIN,
                      _handle_tag=tag)
    b = asoftmax_head(inp.X.to(DEV).to(torch.bfloat16), inp.y.to(DEV), 4000, weights=inp.W.to(DEV), mode="bf16",
                      margin=LIN, _handle_tag=tag)
    torch.cuda.synchronize()
    out = (float(b[0]), None, b[2].cpu().numpy(), b[3].cpu().numpy())
    check(inp, "bf16", out)
    np.testing.assert_array_equal(out[2], a[2].cpu().numpy())
    np.testing.assert_array_equal(out[3], a[3].cpu().numpy())


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_graph_replay_and_profiling_same_bits(mode):
    inp = inputs(256, 512, 4000)
    eager = run(inp, mode, name="graph")
    bitwise(eager, run(inp, mode, name="graph"))
    step = GraphedASoftmaxStep(inp.W.to(DEV), 256, mode=mode, margin=LIN)
    try:
        for _ in range(2):
            loss, dX, dW = step(inp.X.to(DEV), inp.y.to(DEV))
            torch.cuda.synchronize()
            bitwise(eager, (float(loss), None, dX.cpu().numpy(), dW.cpu().numpy()))
    finally:
        step.close()
    h = handle(512, 4000, 256, mode, "prof")
    base = run_h(h, inp)
    names = (C.c_char * (32 * 16))()
    ms = (C.c_float * 16)()
    for level in (1, 2, 0):
        _lib.check(h.lib.asm_set_profiling(h.ptr, level), h.ptr)
        out = run_h(h, inp)
        if level == 1:
            # every SM to the dX kernel: another split-K count, so only dX is summed in another order
            n = h.lib.asm_get_profile(h.ptr, 16, ms, names)
            got = [bytes(names[i * 32:(i + 1) * 32]).split(b"\0")[0].decode() for i in range(n)]
            assert "dx_finish" in got and "dx_finish_margin" not in got, got
            check(inp, mode, out)
            bitwise(base[:2] + (None, base[3]), out[:2] + (None, out[3]))
        else:
            bitwise(base, out)


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_focal_composition(mode):
    inp = inputs(256, 512, 4000)
    r = lr.focal_head(inp.X.numpy(), inp.W.numpy(), inp.y.numpy(), 0.7, 2.0)
    h = handle(512, 4000, 256, mode, "focal", loss=FocalLoss(0.7, 2.0))
    check(inp, mode, run_h(h, inp), r)
    # FocalLoss(1, 0) keeps the cross-entropy's bits
    h1 = handle(512, 4000, 256, mode, "focal10", loss=FocalLoss(1.0, 0.0))
    bitwise(run_h(h1, inp), run(inp, mode, name="ce"))


def test_no_state_leak_and_kind_switch():
    """A-softmax -> linear -> A-softmax on one handle: the A-softmax outputs equal a fresh handle's bit
    for bit, and the linear step in between equals a fresh linear handle's."""
    inp = inputs(256, 512, 4000)
    tag = (TAG, "leak")
    h = get_handle(DEV, 512, 4000, 4000, 0, 256, 4, "bf16", tag=tag)
    fresh = get_handle(DEV, 512, 4000, 4000, 0, 256, 4, "bf16", tag=(TAG, "fresh"))
    want = run_h(fresh, inp)
    bitwise(run_h(h, inp), want)
    _lib.check(h.lib.asm_set_margin(h.ptr, C.byref(_lib.AsmMargin(_lib.MARGIN_LINEAR, 0.0, 0.0, 0.0))), h.ptr)
    lin = run_h(h, inp)
    check(inp, "bf16", lin)
    bitwise(lin, run(inp, "bf16", name="leak-fresh-linear"))
    _lib.check(h.lib.asm_set_margin(h.ptr, None), h.ptr)
    bitwise(run_h(h, inp), want)
    assert h.lib.asm_set_margin(h.ptr, C.byref(_lib.AsmMargin(2, 0.0, 0.0, 0.0))) == _lib.ASM_ERR_INVALID_ARG


# ----------------------------------------------------------------------------- class-sharded
@pytest.mark.parametrize("G", [2, 4])
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_partial_calls_host_combine(mode, G):
    B, D, Cn = 256, 512, 6000
    inp = inputs(B, D, Cn)
    r = oracle(inp)
    X, y = inp.X.to(DEV), inp.y.to(DEV)
    per = -(-Cn // G)
    bounds = [(g * per, min(Cn, (g + 1) * per)) for g in range(G)]
    hs, Ws, stats = [], [], torch.zeros(G, 3, B, device=DEV)
    for g, (lo, hi) in enumerate(bounds):
        h = get_handle(DEV, D, Cn, hi - lo, lo, B, 4, mode, g, G, tag=(TAG, "part", g), margin=LIN)
        Ws.append(inp.W[:, lo:hi].contiguous().to(DEV))
        _lib.check(h.lib.asm_forward_partial(h.ptr, X.data_ptr(), B, y.data_ptr(), 4, Ws[g].data_ptr(), 0.0,
                                             stats[g].data_ptr(), None, None), h.ptr)
        hs.append(h)
    dX = torch.zeros(B, D, device=DEV)
    dWs = []
    loss = torch.full((1,), float("nan"), device=DEV)
    for g, h in enumerate(hs):
        dXp = torch.full((B, D), float("nan"), device=DEV)
        dW = torch.full_like(Ws[g], float("nan"))
        _lib.check(h.lib.asm_backward_partial(h.ptr, stats.data_ptr(), G, loss.data_ptr(), dXp.data_ptr(),
                                              dW.data_ptr(), None), h.ptr)
        dX += dXp
        dWs.append(dW)
    torch.cuda.synchronize()
    check(inp, mode, (float(loss), None, dX.cpu().numpy(), torch.cat(dWs, dim=1).cpu().numpy()), r)


class LinearRanks(FakeRanks):
    """test_p2p_gpu's in-process ranks, with the linear kind set once on every rank's handle."""

    def __init__(self, inp, G, mode, tag):
        super().__init__(inp, G, mode, tag)
        st = _lib.AsmMargin(_lib.MARGIN_LINEAR, 0.0, 0.0, 0.0)
        for h in self.handles:
            _lib.check(h.lib.asm_set_margin(h.ptr, C.byref(st)), h.ptr)


@pytest.mark.parametrize("G", [2, 4])
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_nvlink_transport_eager_and_graph(mode, G):
    inp = inputs(128, 128, 5000)
    r = oracle(inp)
    ranks = LinearRanks(inp, G, mode, (TAG, "p2p", mode, G))

    def every_element():
        dX = np.concatenate([ranks.dX[g].cpu().numpy() for g in range(G)])
        dW = np.concatenate([ranks.dW[g].cpu().numpy() for g in range(G)], axis=1)
        check(inp, mode, (float(ranks.loss[0]), None, dX, dW), r)

    try:
        for _ in range(3):
            ranks.step(0.0)
            ranks.check(r)
            every_element()
        graphs = []
        for g in range(G):
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr, stream=ranks.streams[g]):
                ranks.enqueue(g, 0.0)
            graphs.append(gr)
        for _ in range(3):
            torch.cuda.synchronize()
            for g in range(G):
                with torch.cuda.stream(ranks.streams[g]):
                    graphs[g].replay()
            ranks.check(r)
            every_element()
    finally:
        for h in ranks.handles:
            drop_handle(h)


# ----------------------------------------------------------------------------- tower orders
@pytest.mark.parametrize("order", ["margin", "plain"])
def test_head_call_orders(order):
    """Both orders the reference's towers use: forward(features, labels) then loss_function (margin
    networks, data_parallel.py:220-223), and forward(features) then loss_function(scope, labels)
    (Singular / DataParallel, data_parallel.py:51, :133).  Same step, same bits."""
    inp = inputs(256, 512, 4000)
    head = ASoftmaxHead(512, 4000, mode="bf16", device=DEV, margin=LIN, seed=3)
    head.weights = inp.W.to(DEV)
    X, y = inp.X.to(DEV), inp.y.to(DEV)
    if order == "margin":
        out = head.forward(X, y, num_classes=4000)
    else:
        out = head.forward(X, num_classes=4000)
        assert out["logits"] is None and out["features"] is X
    losses, names, others = head.loss_function("tower_0", y, **out)
    assert names == ["cross_entropy", "reg_loss"] and "lambda" not in others
    dX, dW = head.gradients()
    torch.cuda.synchronize()
    r = oracle(inp)
    W = inp.W.double().numpy()
    want = type(r)(r.loss, r.logits, r.dX, r.dW + 5e-4 * W, r.ce, r.w)
    check(inp, "bf16", (float(losses[0]), None, dX.cpu().numpy(), dW.cpu().numpy()), want)
    assert float(losses[1]) == pytest.approx(2.5e-4 * (W * W).sum(), rel=1e-4)
    # the other kinds still need labels in forward
    with pytest.raises(AssertionError):
        ASoftmaxHead(512, 4000, mode="bf16", device=DEV, seed=3).forward(X, num_classes=4000)
