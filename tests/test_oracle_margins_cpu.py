"""The float64 oracle of the additive-margin heads (oracle/additive_margin_ref.py) checked against
finite differences, an independent torch autograd restatement, known values of phi, invariances
and its own class-sharded form; plus the C ABI's argument checks of asm_set_margin, which need
no GPU."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from oracle import additive_margin_ref as am
from oracle import asoftmax_ref as ref
from tf_face_toolbox_b200 import AdditiveMargin, _lib
from tf_face_toolbox_b200.synthetic import make_inputs

KINDS = {"arcface": (64.0, 0.5, 0.0), "cosface": (64.0, 0.0, 0.35), "combined": (30.0, 0.3, 0.2)}


def spread_inputs(B, D, C, seed, m2=0.5, t_max=0.97):
    """Rows with target cosines spread over [-t_max, t_max], kept 0.02 away from tau(m2), and
    random norms: rows sit on both sides of tau."""
    inp = make_inputs(B, D, C, seed=seed, w_std=0.05)
    g = torch.Generator().manual_seed(seed + 7)
    W = inp.W.double()
    y = inp.y.long()
    wy = W[:, y].t()
    wy = wy / wy.norm(dim=1, keepdim=True)
    t = torch.linspace(-t_max, t_max, B, dtype=torch.float64)[torch.randperm(B, generator=g)]
    if B == 1:
        t[0] = 0.3                   # one row: a typical cosine, not the extreme end of the range
    tau = am.tau(m2)
    near = (t - tau).abs() < 0.02
    t[near] = tau - 0.03
    u = torch.randn(B, D, generator=g, dtype=torch.float64)
    u = u - (u * wy).sum(1, keepdim=True) * wy
    u = u / u.norm(dim=1, keepdim=True)
    n = 5.0 + 25.0 * torch.rand(B, 1, generator=g, dtype=torch.float64)
    X = n * (t[:, None] * wy + torch.sqrt(1 - t[:, None] ** 2) * u)
    return type(inp)(X.float().contiguous(), inp.W, inp.y)


def _np(inp):
    return inp.X.double().numpy(), inp.W.double().numpy(), inp.y.numpy()


def test_inputs_straddle_tau():
    X, W, y = _np(spread_inputs(64, 32, 50, seed=1, m2=0.5))
    r = am.additive_head(X, W, y, 64.0, 0.5, 0.0)
    assert r.first.any() and (~r.first).any()
    assert np.abs(r.t - am.tau(0.5)).min() > 0.01


@pytest.mark.parametrize("kind", sorted(KINDS))
def test_finite_differences(kind):
    s, m2, m3 = KINDS[kind]
    X, W, y = _np(spread_inputs(12, 8, 7, seed=3, m2=m2))
    r = am.additive_head(X, W, y, s, m2, m3)
    if m2 > 0:
        assert r.first.any() and (~r.first).any()          # both branches of phi are differentiated
    h = 1e-6
    for M, G, name in ((X, r.dX, "X"), (W, r.dW, "W")):
        num = np.zeros_like(M)
        for idx in np.ndindex(M.shape):
            old = M[idx]
            M[idx] = old + h
            lp = am.additive_loss_only(X, W, y, s, m2, m3)
            M[idx] = old - h
            lm = am.additive_loss_only(X, W, y, s, m2, m3)
            M[idx] = old
            num[idx] = (lp - lm) / (2 * h)
        np.testing.assert_allclose(G, num, rtol=1e-6, atol=1e-6 * np.abs(G).max(), err_msg=name)


@pytest.mark.parametrize("kind", sorted(KINDS))
def test_torch_autograd_restatement(kind):
    """acos / cos(theta + m2) instead of the sqrt identity, differentiated by autograd."""
    s, m2, m3 = KINDS[kind]
    X, W, y = _np(spread_inputs(16, 12, 9, seed=4, m2=m2))
    r = am.additive_head(X, W, y, s, m2, m3)
    Xt = torch.tensor(X, requires_grad=True)
    Wt = torch.tensor(W, requires_grad=True)
    yt = torch.tensor(y, dtype=torch.long)
    cosm = (Xt / Xt.norm(dim=1, keepdim=True)) @ (Wt / Wt.norm(dim=0, keepdim=True))
    rows = torch.arange(X.shape[0])
    t = cosm[rows, yt].clamp(-1, 1)
    theta = torch.acos(t)
    tau = math.cos(math.pi - m2)
    phi = torch.where(t >= tau, torch.cos(theta + m2) - m3, t - m2 * math.sin(m2) - m3)
    f = s * cosm
    f = f.index_put((rows, yt), s * phi)
    loss = torch.nn.functional.cross_entropy(f, yt)
    loss.backward()
    assert abs(float(loss.detach()) - r.loss) <= 1e-10 * abs(r.loss)
    np.testing.assert_allclose(Xt.grad.numpy(), r.dX, rtol=1e-10, atol=1e-10 * np.abs(r.dX).max())
    np.testing.assert_allclose(Wt.grad.numpy(), r.dW, rtol=1e-10, atol=1e-10 * np.abs(r.dW).max())
    np.testing.assert_allclose(f.detach().numpy(), r.logits, rtol=1e-12, atol=1e-12 * s)


@pytest.mark.parametrize("m2,m3", [(0.5, 0.0), (0.0, 0.35), (0.3, 0.2), (1.2, 0.1)])
def test_phi_known_values(m2, m3):
    ph, dph, _ = am.phi(np.array([1.0, 0.0]), m2, m3)
    assert ph[0] == pytest.approx(math.cos(m2) - m3, abs=1e-6 * math.sin(m2) + 1e-15)   # sin(theta) floored at 1e-6
    assert ph[1] == pytest.approx(-math.sin(m2) - m3, abs=1e-15)
    assert dph[1] == pytest.approx(math.cos(m2), abs=1e-15)
    tau = am.tau(m2)
    if tau > -1.0:
        # the fallback's jump at tau: cos(pi) - m3 from above, tau - m2 sin m2 - m3 from below
        above, _, fa = am.phi(np.array([tau]), m2, m3)
        below, _, fb = am.phi(np.array([np.nextafter(tau, -2.0)]), m2, m3)
        assert fa[0] and not fb[0]
        assert above[0] == pytest.approx(-1.0 - m3, abs=1e-12)
        assert below[0] == pytest.approx(tau - m2 * math.sin(m2) - m3, abs=1e-12)


def test_zero_margin_is_scaled_normalised_softmax():
    """m2 = m3 = 0: the loss and dW of A-softmax with m = 1, lambda = 0 on s X / |X|."""
    s = 30.0
    X, W, y = _np(spread_inputs(20, 16, 11, seed=5))
    r = am.additive_head(X, W, y, s, 0.0, 0.0)
    Xs = s * X / np.linalg.norm(X, axis=1, keepdims=True)
    a = ref.asoftmax_head(Xs, W, y, 1, 0.0)
    assert r.loss == pytest.approx(a.loss, rel=1e-12)
    np.testing.assert_allclose(r.dW, a.dW, rtol=1e-10, atol=1e-12 * np.abs(a.dW).max())
    np.testing.assert_allclose(r.logits, a.logits, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("kind", sorted(KINDS))
def test_invariances(kind):
    s, m2, m3 = KINDS[kind]
    X, W, y = _np(spread_inputs(16, 12, 9, seed=6, m2=m2))
    r = am.additive_head(X, W, y, s, m2, m3)
    alpha = np.linspace(0.25, 4.0, X.shape[0])[:, None]
    r2 = am.additive_head(X * alpha, W, y, s, m2, m3)
    assert r2.loss == pytest.approx(r.loss, rel=1e-12)
    np.testing.assert_allclose(r2.dW, r.dW, rtol=1e-9, atol=1e-12 * np.abs(r.dW).max())
    np.testing.assert_allclose(r2.dX, r.dX / alpha, rtol=1e-9, atol=1e-12 * np.abs(r.dX).max())
    # the gradients are orthogonal to the vectors that are normalised
    dx_dot = np.abs((r.dX * X).sum(1)) / (np.linalg.norm(r.dX, axis=1) * np.linalg.norm(X, axis=1))
    dw_dot = np.abs((r.dW * W).sum(0)) / (np.linalg.norm(r.dW, axis=0) * np.linalg.norm(W, axis=0))
    assert dx_dot.max() <= 1e-12 and dw_dot.max() <= 1e-12, (dx_dot.max(), dw_dot.max())


@pytest.mark.parametrize("G", [2, 3, 8])
@pytest.mark.parametrize("kind", sorted(KINDS))
def test_sharded_equals_unsharded(G, kind):
    s, m2, m3 = KINDS[kind]
    X, W, y = _np(spread_inputs(24, 16, 41, seed=7, m2=m2))
    r = am.additive_head(X, W, y, s, m2, m3)
    bounds = am.shard_bounds(W.shape[1], G)
    stats = [am.sharded_partial_stats(X, W[:, lo:hi], y, lo, s, m2, m3)[:3] for lo, hi in bounds]
    M, logZ, loss = am.sharded_combine(stats)
    assert loss == pytest.approx(r.loss, rel=1e-12)
    dX = np.zeros_like(X)
    for lo, hi in bounds:
        dXp, dW = am.sharded_backward(X, W[:, lo:hi], y, lo, M, logZ, s, m2, m3)
        dX += dXp
        np.testing.assert_allclose(dW, r.dW[:, lo:hi], rtol=1e-9, atol=1e-12 * np.abs(r.dW).max())
    np.testing.assert_allclose(dX, r.dX, rtol=1e-9, atol=1e-12 * np.abs(r.dX).max())


def test_constructors():
    assert AdditiveMargin.arcface(64, 0.5) == AdditiveMargin(64.0, 0.5, 0.0)
    assert AdditiveMargin.cosface(30, 0.35) == AdditiveMargin(30.0, 0.0, 0.35)
    assert AdditiveMargin() == AdditiveMargin(64.0, 0.5, 0.0)
    assert hash(AdditiveMargin.arcface()) == hash(AdditiveMargin(64.0, 0.5, 0.0))   # a handle-cache key


INVALID = [(2, 64.0, 0.5, 0.0), (-1, 64.0, 0.5, 0.0), (1, 0.0, 0.5, 0.0), (1, -1.0, 0.5, 0.0),
           (1, math.inf, 0.5, 0.0), (1, math.nan, 0.5, 0.0), (1, 64.0, -0.1, 0.0), (1, 64.0, 1.6, 0.0),
           (1, 64.0, math.nan, 0.0), (1, 64.0, 0.5, -0.1), (1, 64.0, 0.5, math.inf), (1, 64.0, 0.5, math.nan)]


@pytest.mark.parametrize("kind,s,m2,m3", INVALID + [(1, 64.0, 0.5, 0.0), (0, 0.0, 0.0, 0.0)])
def test_cabi_set_margin_without_handle(kind, s, m2, m3):
    lib = _lib.load()
    mg = _lib.AsmMargin(kind, s, m2, m3)
    assert lib.asm_set_margin(None, C.byref(mg)) == _lib.ASM_ERR_INVALID_ARG
    assert lib.asm_set_margin(None, None) == _lib.ASM_ERR_INVALID_ARG
