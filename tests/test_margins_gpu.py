"""The additive-margin heads (ArcFace, CosFace and the combined margin) on the B200 against the
float64 oracle (oracle/additive_margin_ref.py): every element of the outputs with the BASELINE
bounds of tests/head_checks.py, over kinds x modes x shapes, the features the margin combines
with, the class-sharded paths and the schedule knobs that touch the new code."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from head_checks import LOSS_TOL, assert_within_oracle_bounds, cosine
from oracle import additive_margin_ref as am
from oracle import asoftmax_ref as ref
from test_oracle_margins_cpu import spread_inputs
from test_p2p_gpu import FakeRanks
from tf_face_toolbox_b200 import AdditiveMargin, FusedOptimizer, GraphedASoftmaxStep, _lib, asoftmax_head
from tf_face_toolbox_b200.head import _HANDLES, drop_handle, get_handle

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TESTS = os.path.dirname(os.path.abspath(__file__))
KINDS = {"arcface": AdditiveMargin.arcface(64.0, 0.5), "cosface": AdditiveMargin.cosface(64.0, 0.35),
         "combined": AdditiveMargin(30.0, 0.3, 0.2)}


def inputs(B, D, Cn, kind, seed=11):
    return spread_inputs(B, D, Cn, seed=seed, m2=KINDS[kind].m2)


def oracle(inp, mg):
    return am.additive_head(inp.X.numpy(), inp.W.numpy(), inp.y.numpy(), mg.s, mg.m2, mg.m3)


def run(inp, mode, mg, logits=False, grads=True, tag=None, **kw):
    X = kw.pop("X", None)
    X = inp.X.to(DEV) if X is None else X
    W = kw.pop("W", None)
    W = inp.W.to(DEV) if W is None else W
    loss, f, dX, dW = asoftmax_head(X, inp.y.to(DEV), W.shape[1], 4, 0.0, weights=W, mode=mode,
                                    return_logits=logits, compute_grads=grads, margin=mg, _handle_tag=tag, **kw)
    torch.cuda.synchronize()
    cpu = lambda t: None if t is None else t.cpu().numpy()      # noqa: E731
    return float(loss), cpu(f), cpu(dX), cpu(dW)


def assert_margin_logits(inp, r, mg, mode, f):
    """Every logit against the oracle (the scale s multiplies the bf16 rounding of a cosine), the
    margin entry at exactly column y_i, and argmax agreement wherever the top-2 gap is clear."""
    tol = (1e-5 if mode == "fp32" else 6e-3) * mg.s
    np.testing.assert_allclose(f, r.logits, rtol=0, atol=tol)
    rows = np.arange(f.shape[0])
    y = inp.y.numpy().astype(np.int64)
    raw = mg.s * (inp.X.double().numpy() / r.n[:, None]) @ (inp.W.double().numpy() / r.c)
    moved = np.abs(f - raw) > 4 * tol                      # entries the margin changed, on the device
    want = np.abs(r.logits - raw) > 8 * tol                # entries it must have changed
    off = moved.copy()
    off[rows, y] = False
    assert not off.any(), np.argwhere(off)[:5]
    assert moved[rows, y][want[rows, y]].all()
    top2 = np.sort(r.logits, axis=1)[:, -2:]
    clear = (top2[:, 1] - top2[:, 0]) > 4 * tol
    assert np.array_equal(f.argmax(axis=1)[clear], r.logits.argmax(axis=1)[clear])


def check(inp, mg, mode, out, grads=True):
    loss, f, dX, dW = out
    r = oracle(inp, mg)
    assert np.isfinite(loss)
    if grads:
        assert_within_oracle_bounds(inp, r, mode, loss, None, dX, dW)
    else:
        assert abs(loss - r.loss) <= LOSS_TOL[mode] * abs(r.loss), (loss, r.loss)
    if f is not None:
        assert_margin_logits(inp, r, mg, mode, f)


def bitwise(a, b):
    assert a[0] == b[0] or (np.isnan(a[0]) and np.isnan(b[0]))
    for x, y in zip(a[1:], b[1:]):
        assert (x is None) == (y is None)
        if x is not None:
            assert np.array_equal(x, y)


@pytest.fixture(autouse=True)
def _drop_handles():
    yield
    for k in [k for k in _HANDLES if isinstance(k[-1], tuple) and k[-1][:1] == ("margins",)]:
        drop_handle(_HANDLES[k])


# ----------------------------------------------------------------------------- coverage matrix
@pytest.mark.parametrize("D", [128, 512])
@pytest.mark.parametrize("Cn", [200, 3002, 10572])
@pytest.mark.parametrize("B", [1, 129, 512])
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
@pytest.mark.parametrize("kind", sorted(KINDS))
def test_matrix(kind, mode, B, Cn, D):
    mg = KINDS[kind]
    inp = inputs(B, D, Cn, kind)
    logits = Cn <= 3002
    check(inp, mg, mode, run(inp, mode, mg, logits=logits))
    if B == 129:
        check(inp, mg, mode, run(inp, mode, mg, grads=False, logits=logits), grads=False)


@pytest.mark.parametrize("B", [1, 129, 512])
@pytest.mark.parametrize("Cn", [200, 3002, 10572])
@pytest.mark.parametrize("kind", sorted(KINDS))
def test_cuda_core_path_d80(kind, Cn, B):
    """D % 64 != 0: fp32 on the CUDA cores, which read the scaled, normalised fp32 copy."""
    mg = KINDS[kind]
    inp = inputs(B, 80, Cn, kind)
    check(inp, mg, "fp32", run(inp, "fp32", mg, logits=Cn <= 3002))
    if B == 129:
        check(inp, mg, "fp32", run(inp, "fp32", mg, grads=False), grads=False)


@pytest.mark.parametrize("kind", sorted(KINDS))
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_target_parallel_to_class_weight(kind, mode):
    """x_i proportional to w_{y_i} (t = 1 up to rounding, where phi' has its 1e-12 floor): finite
    loss and gradients, and the other rows still meet the bounds."""
    mg = KINDS[kind]
    inp = inputs(128, 128, 3002, kind)
    X = inp.X.clone()
    w = inp.W[:, inp.y[0].long()]
    X[0] = 10.0 * w / w.norm()
    inp = type(inp)(X, inp.W, inp.y)
    loss, _, dX, dW = run(inp, mode, mg)
    assert np.isfinite(loss) and np.isfinite(dX).all() and np.isfinite(dW).all()
    r = oracle(inp, mg)
    assert abs(loss - r.loss) <= LOSS_TOL[mode] * abs(r.loss)
    assert cosine(dX[1:], r.dX[1:]) >= 0.9999 and cosine(dW, r.dW) >= 0.9999


# ----------------------------------------------------------------------------- other features
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_gradient_transform(mode):
    mg = KINDS["arcface"]
    inp = inputs(256, 512, 4000, "arcface")
    reg = torch.zeros(1, device=DEV)
    loss, _, dX, dW = run(inp, mode, mg, grad_scale=0.25, weight_decay=5e-4, reg_loss_out=reg)
    r = oracle(inp, mg)
    W = inp.W.double().numpy()
    want = type(r)(r.loss, r.logits, 0.25 * r.dX, 0.25 * (r.dW + 5e-4 * W), r.n, r.c, r.t, r.first)
    assert_within_oracle_bounds(inp, want, mode, loss, None, dX, dW)
    assert float(reg) == pytest.approx(2.5e-4 * (W * W).sum(), rel=1e-4)


@pytest.mark.parametrize("kind", ["Momentum", "Adam"])
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_fused_optimizer_three_steps(kind, mode):
    mg = KINDS["combined"]
    inp = inputs(128, 128, 3000, "combined")
    lr = 0.05 if kind == "Momentum" else 1e-3
    opt = FusedOptimizer(kind, lr=lr, weight_decay=5e-4)
    W_f = inp.W.to(DEV).clone()
    Wr = inp.W.double().numpy().copy()
    s0, s1 = np.zeros_like(Wr), np.zeros_like(Wr)
    X = inp.X.to(DEV)
    for step in range(1, 4):
        Wcur = torch.from_numpy(Wr).float().to(DEV)
        _, _, _, dW = run(inp, mode, mg, W=Wcur, tag=("margins", "opt-ref"))
        Wr, s0, s1n = ref.optimizer_step(Wcur.double().cpu().numpy(), dW, s0, s1, kind.lower(), lr=lr, step=step)
        s1 = s1n if s1n is not None else s1
        loss, _, _, none = asoftmax_head(X, inp.y.to(DEV), 3000, 4, 0.0, weights=W_f, mode=mode, optimizer=opt,
                                         margin=mg, _handle_tag=("margins", "opt"))
        assert none is None and np.isfinite(float(loss))
        torch.cuda.synchronize()
        upd_f = W_f.double().cpu().numpy() - inp.W.double().numpy()
        upd_r = Wr - inp.W.double().numpy()
        assert cosine(upd_f, upd_r) >= (0.999 if (kind, mode) == ("Adam", "bf16") else 0.9999), step


def test_bf16_embeddings():
    mg = KINDS["arcface"]
    inp = inputs(256, 512, 4000, "arcface")
    inp = type(inp)(inp.X.to(torch.bfloat16).float(), inp.W, inp.y)     # exactly representable
    a = run(inp, "bf16", mg)
    b = run(inp, "bf16", mg, X=inp.X.to(DEV).to(torch.bfloat16))
    check(inp, mg, "bf16", b)
    np.testing.assert_allclose(b[2], a[2], rtol=1e-4, atol=1e-6 * np.abs(a[2]).max())


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_graph_replay_and_determinism(mode):
    mg = KINDS["cosface"]
    inp = inputs(256, 512, 4000, "cosface")
    eager = run(inp, mode, mg)
    bitwise(eager, run(inp, mode, mg))                      # two runs, same bits
    W = inp.W.to(DEV)
    step = GraphedASoftmaxStep(W, 256, mode=mode, margin=mg)
    try:
        loss, dX, dW = step(inp.X.to(DEV), inp.y.to(DEV))
        torch.cuda.synchronize()
        bitwise(eager, (float(loss), None, dX.cpu().numpy(), dW.cpu().numpy()))
    finally:
        step.close()


@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_profiling_modes_same_bits(mode):
    """Mode 2 keeps the schedule and its arithmetic: same bits.  Mode 1 gives the dX kernel every
    SM, which raises its split-K count, so only dX is summed in another order there (as for
    A-softmax, test_kernel_variants_gpu.py); the loss and dW keep their bits and dX meets the bounds."""
    mg = KINDS["arcface"]
    inp = inputs(256, 512, 4000, "arcface")
    tag = ("margins", "prof", mode)
    base = run(inp, mode, mg, tag=tag)
    h = get_handle(DEV, 512, 4000, 4000, 0, 256, 4, mode, tag=tag, margin=mg)
    names = (C.c_char * (32 * 16))()
    ms = (C.c_float * 16)()
    for level in (1, 2, 0):
        _lib.check(h.lib.asm_set_profiling(h.ptr, level), h.ptr)
        out = run(inp, mode, mg, tag=tag)
        if level == 1:
            n = h.lib.asm_get_profile(h.ptr, 16, ms, names)
            got = [bytes(names[i * 32:(i + 1) * 32]).split(b"\0")[0].decode() for i in range(n)]
            assert "dx_finish_margin" in got, got
            check(inp, mg, mode, out)
            bitwise(base[:2] + (None, base[3]), out[:2] + (None, out[3]))
        else:
            bitwise(base, out)


def test_no_state_leak_and_argument_checks():
    """A handle switched to the additive kind and back to A-softmax equals a fresh handle bit for
    bit; an invalid margin is refused and changes nothing."""
    inp = inputs(256, 512, 4000, "arcface")
    tag = ("margins", "leak")
    h = get_handle(DEV, 512, 4000, 4000, 0, 256, 4, "bf16", tag=tag)
    fresh = run(inp, "bf16", None, tag=("margins", "fresh"))
    mg = _lib.AsmMargin(_lib.MARGIN_ADDITIVE, 64.0, 0.5, 0.0)
    _lib.check(h.lib.asm_set_margin(h.ptr, C.byref(mg)), h.ptr)
    add = run(inp, "bf16", None, tag=tag)
    check(inp, KINDS["arcface"], "bf16", add)
    for bad in ((2, 64.0, 0.5, 0.0), (1, 0.0, 0.5, 0.0), (1, float("nan"), 0.5, 0.0), (1, 64.0, 1.6, 0.0),
                (1, 64.0, -0.1, 0.0), (1, 64.0, 0.5, -1.0), (1, 64.0, 0.5, float("inf"))):
        assert h.lib.asm_set_margin(h.ptr, C.byref(_lib.AsmMargin(*bad))) == _lib.ASM_ERR_INVALID_ARG
    bitwise(add, run(inp, "bf16", None, tag=tag))           # the refused calls changed nothing
    _lib.check(h.lib.asm_set_margin(h.ptr, None), h.ptr)
    bitwise(fresh, run(inp, "bf16", None, tag=tag))
    with pytest.raises(_lib.AsmError):
        run(inp, "bf16", AdditiveMargin(-1.0, 0.5, 0.0))


# ----------------------------------------------------------------------------- class-sharded
@pytest.mark.parametrize("G", [2, 4])
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
@pytest.mark.parametrize("kind", sorted(KINDS))
def test_partial_calls_host_combine(kind, mode, G):
    mg = KINDS[kind]
    B, D, Cn = 256, 512, 6000
    inp = inputs(B, D, Cn, kind)
    r = oracle(inp, mg)
    X, y = inp.X.to(DEV), inp.y.to(DEV)
    per = -(-Cn // G)
    bounds = [(g * per, min(Cn, (g + 1) * per)) for g in range(G)]
    hs, Ws, stats = [], [], torch.zeros(G, 3, B, device=DEV)
    for g, (lo, hi) in enumerate(bounds):
        h = get_handle(DEV, D, Cn, hi - lo, lo, B, 4, mode, g, G, tag=("margins", "part", g), margin=mg)
        Ws.append(inp.W[:, lo:hi].contiguous().to(DEV))
        _lib.check(h.lib.asm_forward_partial(h.ptr, X.data_ptr(), B, y.data_ptr(), 4, Ws[g].data_ptr(), 0.0,
                                             stats[g].data_ptr(), None, None), h.ptr)
        hs.append(h)
    dX = torch.zeros(B, D, device=DEV)
    loss = torch.zeros(1, device=DEV)
    for g, h in enumerate(hs):
        dXp = torch.empty(B, D, device=DEV)
        dW = torch.empty_like(Ws[g])
        _lib.check(h.lib.asm_backward_partial(h.ptr, stats.data_ptr(), G, loss.data_ptr(), dXp.data_ptr(),
                                              dW.data_ptr(), None), h.ptr)
        dX += dXp
        lo, hi = bounds[g]
        torch.cuda.synchronize()
        sub = type(r)(r.loss, None, r.dX, r.dW[:, lo:hi], r.n, r.c[lo:hi], r.t, r.first)
        assert_within_oracle_bounds(inp, sub, mode, float(loss), None, r.dX, dW.cpu().numpy())
    torch.cuda.synchronize()
    assert_within_oracle_bounds(inp, r, mode, float(loss), None, dX.cpu().numpy(), r.dW)


class MarginRanks(FakeRanks):
    """test_p2p_gpu's in-process ranks, with the margin set once on every rank's handle."""

    def __init__(self, inp, G, mode, tag, mg):
        super().__init__(inp, G, mode, tag)
        st = _lib.AsmMargin(_lib.MARGIN_ADDITIVE, mg.s, mg.m2, mg.m3)
        for h in self.handles:
            _lib.check(h.lib.asm_set_margin(h.ptr, C.byref(st)), h.ptr)


@pytest.mark.parametrize("G", [2, 4])
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_nvlink_transport_eager_and_graph(mode, G):
    mg = KINDS["arcface"] if G == 2 else KINDS["combined"]
    inp = inputs(128, 128, 5000, "arcface" if G == 2 else "combined")
    r = am.additive_head(inp.X.numpy(), inp.W.numpy(), inp.y.numpy(), mg.s, mg.m2, mg.m3)
    ranks = MarginRanks(inp, G, mode, ("margins", "p2p", mode, G), mg)
    try:
        for _ in range(3):
            ranks.step(0.0)
            ranks.check(r)
            for g, (lo, hi) in enumerate(ranks.bounds):          # every element, not only cosines
                rows = slice(g * ranks.b, (g + 1) * ranks.b)
                sub = type(r)(r.loss, None, r.dX[rows], r.dW[:, lo:hi], r.n, r.c, r.t, r.first)
                assert_within_oracle_bounds(inp, sub, mode, float(ranks.loss[g]), None,
                                            ranks.dX[g].cpu().numpy(), ranks.dW[g].cpu().numpy())
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
    finally:
        for h in ranks.handles:
            drop_handle(h)


# ----------------------------------------------------------------------------- process-wide knobs
KNOBS = {"prep1": {"ASM_PREP_SHAPE": "1"}, "prep2": {"ASM_PREP_SHAPE": "2"}, "prep3": {"ASM_PREP_SHAPE": "3"},
         "defer0": {"ASM_DEFER_LOSS": "0"}, "nooverlap": {"ASM_NO_OVERLAP": "1"}, "pdl0": {"ASM_PDL": "0"},
         "x3segs3": {"ASM_X3_SEGS": "3"}, "simt": {"ASM_FP32_SIMT": "1"}}
KNOB_SHAPES = [(129, 512, 3002), (256, 128, 10572)]
_CHILD = ("import sys; sys.path[:0] = sys.argv[1:3]; import test_margins_gpu as t; "
          "t.child_main(sys.argv[3])")


def child_main(outdir):
    for kind in sorted(KINDS):
        for mode in ("bf16", "fp32"):
            for B, D, Cn in KNOB_SHAPES:
                inp = inputs(B, D, Cn, kind)
                a = run(inp, mode, KINDS[kind], logits=True)
                bitwise(a, run(inp, mode, KINDS[kind], logits=True))
                np.savez(os.path.join(outdir, f"{kind}-{mode}-{B}-{D}-{Cn}.npz"), loss=a[0], f=a[1], dX=a[2], dW=a[3])


@pytest.mark.parametrize("knob", sorted(KNOBS))
def test_knobs_in_child_process(knob, tmp_path):
    env = dict(os.environ, **KNOBS[knob])
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", _CHILD, ROOT, TESTS, str(tmp_path)]
    p = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    for kind in sorted(KINDS):
        for mode in ("bf16", "fp32"):
            for B, D, Cn in KNOB_SHAPES:
                z = np.load(tmp_path / f"{kind}-{mode}-{B}-{D}-{Cn}.npz")
                inp = inputs(B, D, Cn, kind)
                if knob == "x3segs3" and mode == "fp32":
                    # three plane-pair segments: the bf16 bound scaled by 2^-14 / 2^-8 (see test_kernel_variants_gpu)
                    r = oracle(inp, KINDS[kind])
                    assert_within_oracle_bounds(inp, r, "bf16", float(z["loss"]), None, z["dX"], z["dW"],
                                                bf16_scale=2.0 ** -6)
                else:
                    check(inp, KINDS[kind], mode, (float(z["loss"]), z["f"], z["dX"], z["dW"]))
