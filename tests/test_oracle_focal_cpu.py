"""The float64 focal-loss oracle (oracle/focal_ref.py) checked against finite differences, an
independent torch autograd restatement from materialised logits, its reductions to the
cross-entropy, its numerics at p -> 1 and its own class-sharded form; plus the C ABI's loss
struct, constants and argument checks, which need no GPU."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest
import torch

from oracle import additive_margin_ref as am
from oracle import asoftmax_ref as ref
from oracle import focal_ref as fr
from test_oracle_margins_cpu import spread_inputs
from tf_face_toolbox_b200 import FocalLoss, _lib
from tf_face_toolbox_b200.synthetic import make_inputs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# margin -> (m, lambda, additive margin tuple or None)
HEADS = {"asoftmax-l0": (4, 0.0, None), "asoftmax-l5": (4, 5.0, None),
         "arcface": (4, 0.0, (64.0, 0.5, 0.0)), "cosface": (4, 0.0, (64.0, 0.0, 0.35))}
ALPHAS = [0.0, 0.5, 2.0, 5.0]


def inputs(head, B, D, Cn, seed):
    m, lam, mg = HEADS[head]
    if mg is None:
        inp = make_inputs(B, D, Cn, seed=seed, w_std=0.05)
    else:
        inp = spread_inputs(B, D, Cn, seed=seed, m2=mg[1])
    return inp.X.double().numpy(), inp.W.double().numpy(), inp.y.numpy()


def oracle(head, X, W, y, gamma, alpha):
    m, lam, mg = HEADS[head]
    return fr.focal_head(X, W, y, gamma, alpha, m, lam, mg)


def ce_oracle(head, X, W, y):
    m, lam, mg = HEADS[head]
    if mg is None:
        return ref.asoftmax_head(X, W, y, m, lam)
    return am.additive_head(X, W, y, *mg)


@pytest.mark.parametrize("alpha", ALPHAS)
@pytest.mark.parametrize("head", sorted(HEADS))
def test_finite_differences(head, alpha):
    m, lam, mg = HEADS[head]
    gamma = 0.75
    X, W, y = inputs(head, 8, 8, 7, seed=3)
    r = oracle(head, X, W, y, gamma, alpha)
    h = 1e-6
    for M, G, name in ((X, r.dX, "X"), (W, r.dW, "W")):
        num = np.zeros_like(M)
        for idx in np.ndindex(M.shape):
            old = M[idx]
            M[idx] = old + h
            lp = fr.focal_loss_only(X, W, y, gamma, alpha, m, lam, mg)
            M[idx] = old - h
            lm = fr.focal_loss_only(X, W, y, gamma, alpha, m, lam, mg)
            M[idx] = old
            num[idx] = (lp - lm) / (2 * h)
        np.testing.assert_allclose(G, num, rtol=1e-6, atol=1e-6 * np.abs(G).max(), err_msg=name)
    assert r.loss == pytest.approx(fr.focal_loss_only(X, W, y, gamma, alpha, m, lam, mg), rel=1e-12)


def _torch_logits(head, Xt, Wt, yt):
    """The margin logits restated in torch: Chebyshev psi with its branch k held constant, or
    acos / cos(theta + m2) for the additive heads."""
    m, lam, mg = HEADS[head]
    rows = torch.arange(Xt.shape[0])
    n = Xt.norm(dim=1)
    What = Wt / Wt.norm(dim=0, keepdim=True)
    if mg is None:
        S = Xt @ What
        s_y = S[rows, yt]
        t = (s_y / n).clamp(-1, 1)
        k = torch.clamp(torch.floor(m * torch.acos(t.detach()) / math.pi), max=m - 1)
        psi = (-1.0) ** k * torch.cos(m * torch.acos(t)) - 2.0 * k
        return S.index_put((rows, yt), (lam * s_y + n * psi) / (1.0 + lam))
    s, m2, m3 = mg
    cosm = (Xt / n[:, None]) @ What
    t = cosm[rows, yt].clamp(-1, 1)
    phi = torch.where(t >= math.cos(math.pi - m2), torch.cos(torch.acos(t) + m2) - m3, t - m2 * math.sin(m2) - m3)
    return (s * cosm).index_put((rows, yt), s * phi)


@pytest.mark.parametrize("alpha", ALPHAS)
@pytest.mark.parametrize("head", sorted(HEADS))
def test_torch_autograd_restatement(head, alpha):
    """gamma (1 - p)^alpha CE on materialised logits, differentiated by autograd through the factor."""
    gamma = 1.5
    X, W, y = inputs(head, 16, 12, 9, seed=4)
    r = oracle(head, X, W, y, gamma, alpha)
    Xt = torch.tensor(X, requires_grad=True)
    Wt = torch.tensor(W, requires_grad=True)
    yt = torch.tensor(y, dtype=torch.long)
    f = _torch_logits(head, Xt, Wt, yt)
    ce = torch.nn.functional.cross_entropy(f, yt, reduction="none")
    p = torch.softmax(f, dim=1)[torch.arange(len(y)), yt]
    loss = (gamma * (1.0 - p) ** alpha * ce).mean()
    loss.backward()
    assert abs(float(loss.detach()) - r.loss) <= 1e-10 * abs(r.loss)
    np.testing.assert_allclose(Xt.grad.numpy(), r.dX, rtol=1e-10, atol=1e-10 * np.abs(r.dX).max())
    np.testing.assert_allclose(Wt.grad.numpy(), r.dW, rtol=1e-10, atol=1e-10 * np.abs(r.dW).max())
    np.testing.assert_allclose(f.detach().numpy(), r.logits, rtol=1e-12, atol=1e-12 * np.abs(r.logits).max())


@pytest.mark.parametrize("head", sorted(HEADS))
def test_alpha_zero_is_scaled_cross_entropy(head):
    X, W, y = inputs(head, 20, 16, 11, seed=5)
    ce = ce_oracle(head, X, W, y)
    for gamma in (1.0, 0.3, 2.5):
        r = oracle(head, X, W, y, gamma, 0.0)
        assert np.all(r.w == gamma)                              # exactly: powf(u, 0) = 1
        assert r.loss == pytest.approx(gamma * ce.loss, rel=1e-12)
        np.testing.assert_allclose(r.dX, gamma * ce.dX, rtol=1e-10, atol=1e-13 * np.abs(ce.dX).max())
        np.testing.assert_allclose(r.dW, gamma * ce.dW, rtol=1e-10, atol=1e-13 * np.abs(ce.dW).max())
        np.testing.assert_allclose(r.logits, ce.logits, rtol=1e-12, atol=1e-12 * np.abs(ce.logits).max())


def test_weight_finite_at_p_one():
    """w_i >= 0 and finite as p -> 1 and at p = 1 exactly (ce = 0), also for alpha < 1, where
    the textbook form alpha p u^(alpha - 1) ce is 0 * inf at ce = 0."""
    ce = np.array([0.0, 1e-300, 1e-30, 1e-12, 1e-6, 1e-2, 1.0, 30.0, 800.0])
    for alpha in (0.0, 0.25, 0.5, 0.9, 1.0, 2.0, 5.0):
        loss, w = fr.focal_weight(ce, 2.0, alpha)
        assert np.isfinite(w).all() and np.isfinite(loss).all() and (w >= 0).all() and (loss >= 0).all(), alpha
        if alpha > 0:
            assert w[0] == 0.0 and loss[0] == 0.0
        # against the textbook form wherever it is defined
        p, u = np.exp(-ce[1:]), -np.expm1(-ce[1:])
        want = 2.0 * (u ** alpha + alpha * p * u ** (alpha - 1.0) * ce[1:])
        np.testing.assert_allclose(w[1:], want, rtol=1e-12)
    # ce / u -> 1 as ce -> 0: alpha < 1 gives w ~ gamma (1 + alpha) u^alpha
    _, w = fr.focal_weight(np.array([1e-20]), 1.0, 0.5)
    assert w[0] == pytest.approx(1.5 * 1e-10, rel=1e-9)


@pytest.mark.parametrize("G", [2, 3, 5])
@pytest.mark.parametrize("head", sorted(HEADS))
def test_sharded_equals_unsharded(head, G):
    m, lam, mg = HEADS[head]
    gamma, alpha = 0.8, 2.0
    X, W, y = inputs(head, 24, 16, 41, seed=7)
    r = oracle(head, X, W, y, gamma, alpha)
    bounds = fr.shard_bounds(W.shape[1], G)
    stats = [fr.sharded_partial_stats(X, W[:, lo:hi], y, lo, m, lam, mg)[:3] for lo, hi in bounds]
    M, logZ, w, loss = fr.sharded_combine(stats, gamma, alpha)
    assert loss == pytest.approx(r.loss, rel=1e-12)
    np.testing.assert_allclose(w, r.w, rtol=1e-12)
    dX = np.zeros_like(X)
    for lo, hi in bounds:
        dXp, dW = fr.sharded_backward(X, W[:, lo:hi], y, lo, M, logZ, w, m, lam, mg)
        dX += dXp
        np.testing.assert_allclose(dW, r.dW[:, lo:hi], rtol=1e-9, atol=1e-12 * np.abs(r.dW).max())
    np.testing.assert_allclose(dX, r.dX, rtol=1e-9, atol=1e-12 * np.abs(r.dX).max())


# ----------------------------------------------------------------------------- Python and C ABI
def test_focal_loss_dataclass():
    assert FocalLoss() == FocalLoss(1.0, 2.0)
    assert hash(FocalLoss(0.5, 1.0)) == hash(FocalLoss(0.5, 1.0))     # a handle-cache key
    st = FocalLoss(0.5, 1.5)._struct()
    assert (st.kind, st.gamma, st.alpha) == (_lib.LOSS_FOCAL, 0.5, 1.5)
    with pytest.raises(Exception):
        FocalLoss().gamma = 2.0                                      # frozen


def test_cabi_loss_struct_and_constants():
    hdr = open(os.path.join(ROOT, "include", "asoftmax_b200.h")).read()
    enum = re.search(r"enum\s*\{\s*ASM_LOSS_SOFTMAX_CE\s*=\s*(\d+)\s*,\s*ASM_LOSS_FOCAL\s*=\s*(\d+)\s*\}", hdr)
    assert enum and (int(enum[1]), int(enum[2])) == (_lib.LOSS_SOFTMAX_CE, _lib.LOSS_FOCAL) == (0, 1)
    body = re.search(r"typedef struct \{([^}]*)\} asm_loss;", hdr)
    assert body and re.sub(r"\s+", " ", body[1]).strip() == "int32_t kind; float gamma, alpha;"
    assert C.sizeof(_lib.AsmLoss) == 12
    assert [(n, getattr(_lib.AsmLoss, n).offset) for n, _ in _lib.AsmLoss._fields_] == \
        [("kind", 0), ("gamma", 4), ("alpha", 8)]
    assert "asm_set_loss" in _lib.SYMBOLS


INVALID = [(2, 1.0, 2.0), (-1, 1.0, 2.0), (1, 0.0, 2.0), (1, -1.0, 2.0), (1, math.nan, 2.0), (1, math.inf, 2.0),
           (1, 1.0, -0.5), (1, 1.0, math.inf), (1, 1.0, math.nan)]


@pytest.mark.parametrize("kind,gamma,alpha", INVALID + [(1, 1.0, 2.0), (0, 0.0, 0.0)])
def test_cabi_set_loss_without_handle(kind, gamma, alpha):
    lib = _lib.load()
    assert lib.asm_set_loss(None, C.byref(_lib.AsmLoss(kind, gamma, alpha))) == _lib.ASM_ERR_INVALID_ARG
    assert lib.asm_set_loss(None, None) == _lib.ASM_ERR_INVALID_ARG
