"""CPU checks of the plain softmax classifier's float64 oracle (oracle/linear_softmax_ref.py): finite
differences, the one-piece / class-streamed / class-sharded forms against each other, the torch
autograd restatement of the reference's graph, the focal loss on these logits, and the one
structural difference from A-softmax: dW keeps its component along w_j."""
import numpy as np
import pytest
import torch

from oracle import asoftmax_ref as ref
from oracle import focal_ref as fr
from oracle import linear_softmax_ref as lr
from tf_face_toolbox_b200.synthetic import make_inputs


def linear_inputs(B, D, C, regime="trained", seed=3):
    """'init': the reference's N(0, 0.001) weights (loss about log C); 'trained': weights scaled so
    that target logits reach +-12."""
    w_std = 0.001 if regime == "init" else 8.0 / D
    return make_inputs(B, D, C, seed=seed, w_std=w_std)


def _np(inp):
    return inp.X.double().numpy(), inp.W.double().numpy(), inp.y.numpy().astype(np.int64)


def test_regimes():
    X, W, y = _np(linear_inputs(64, 128, 500, "init"))
    r = lr.linear_head(X, W, y)
    assert abs(r.loss - np.log(500)) < 0.05
    X, W, y = _np(linear_inputs(64, 128, 500, "trained"))
    r = lr.linear_head(X, W, y)
    assert np.abs(r.logits).max() > 10.0


@pytest.mark.parametrize("regime", ["init", "trained"])
def test_finite_differences(regime):
    X, W, y = _np(linear_inputs(6, 8, 11, regime, seed=7))
    r = lr.linear_head(X, W, y)
    eps = 1e-6
    for i, k in [(0, 0), (3, 5), (5, 7)]:
        Xp, Xm = X.copy(), X.copy()
        Xp[i, k] += eps
        Xm[i, k] -= eps
        num = (lr.linear_loss_only(Xp, W, y) - lr.linear_loss_only(Xm, W, y)) / (2 * eps)
        assert num == pytest.approx(r.dX[i, k], rel=1e-6, abs=1e-9)
    for k, j in [(0, 0), (2, y[1]), (7, 10)]:
        Wp, Wm = W.copy(), W.copy()
        Wp[k, j] += eps
        Wm[k, j] -= eps
        num = (lr.linear_loss_only(X, Wp, y) - lr.linear_loss_only(X, Wm, y)) / (2 * eps)
        assert num == pytest.approx(r.dW[k, j], rel=1e-6, abs=1e-9)


def test_closed_form_is_softmax_minus_onehot():
    X, W, y = _np(linear_inputs(9, 16, 30))
    r = lr.linear_head(X, W, y)
    f = X @ W
    p = np.exp(f - f.max(axis=1, keepdims=True))
    p /= p.sum(axis=1, keepdims=True)
    p[np.arange(9), y] -= 1.0
    np.testing.assert_allclose(r.dX, p @ W.T / 9, rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(r.dW, X.T @ p / 9, rtol=1e-12, atol=1e-15)
    np.testing.assert_array_equal(r.logits, f)


@pytest.mark.parametrize("regime", ["init", "trained"])
def test_streamed_equals_one_piece(regime):
    X, W, y = _np(linear_inputs(20, 32, 1003, regime))
    a = lr.linear_head(X, W, y)
    b = lr.linear_head_streamed(X, W, y, chunk=128)
    assert b.loss == pytest.approx(a.loss, rel=1e-12)
    np.testing.assert_allclose(b.dX, a.dX, rtol=1e-10, atol=1e-15)
    np.testing.assert_allclose(b.dW, a.dW, rtol=1e-10, atol=1e-15)


def test_streamed_at_cfg3_class_count():
    """C = 85,742 (BASELINE config 3) in the streamed form, against the one piece."""
    X, W, y = _np(linear_inputs(8, 32, 85742, "init"))
    a = lr.linear_head(X, W, y)
    b = lr.linear_head_streamed(X, W, y)
    assert a.loss == pytest.approx(np.log(85742), rel=1e-3)
    assert b.loss == pytest.approx(a.loss, rel=1e-12)
    np.testing.assert_allclose(b.dW, a.dW, rtol=1e-9, atol=1e-18)
    np.testing.assert_allclose(b.dX, a.dX, rtol=1e-9, atol=1e-18)


@pytest.mark.parametrize("G", [2, 3, 5])
@pytest.mark.parametrize("regime", ["init", "trained"])
def test_sharded_combine_equals_one_piece(G, regime):
    X, W, y = _np(linear_inputs(17, 24, 101, regime))
    a = lr.linear_head(X, W, y)
    bounds = lr.shard_bounds(101, G)
    stats = [lr.sharded_partial_stats(X, W[:, lo:hi], y, lo)[:3] for lo, hi in bounds]
    M, logZ, loss = lr.sharded_combine(stats)
    assert loss == pytest.approx(a.loss, rel=1e-12)
    dX = np.zeros_like(X)
    dW = np.empty_like(W)
    for lo, hi in bounds:
        dXp, dW[:, lo:hi] = lr.sharded_backward(X, W[:, lo:hi], y, lo, M, logZ)
        dX += dXp
    np.testing.assert_allclose(dX, a.dX, rtol=1e-10, atol=1e-15)
    np.testing.assert_allclose(dW, a.dW, rtol=1e-10, atol=1e-15)


@pytest.mark.parametrize("regime", ["init", "trained"])
def test_equals_torch_graph_port(regime):
    inp = linear_inputs(33, 64, 257, regime)
    X, W, y = _np(inp)
    a = lr.linear_head(X, W, y)
    loss, dX, dW = lr.step(torch.from_numpy(X), torch.from_numpy(W), torch.from_numpy(y))
    assert abs(float(loss) - a.loss) <= 1e-12 * abs(a.loss)
    np.testing.assert_allclose(dX.numpy(), a.dX, rtol=1e-12, atol=1e-12 * np.abs(a.dX).max())
    np.testing.assert_allclose(dW.numpy(), a.dW, rtol=1e-12, atol=1e-12 * np.abs(a.dW).max())


@pytest.mark.parametrize("gamma,alpha", [(1.0, 2.0), (0.7, 0.5), (2.0, 0.0)])
def test_focal_on_linear_logits(gamma, alpha):
    X, W, y = _np(linear_inputs(10, 16, 40, seed=9))
    r = lr.focal_head(X, W, y, gamma, alpha)
    # against the focal oracle's row-weight construction on the linear one-row heads
    rows = [lr.linear_head(X[i:i + 1], W, y[i:i + 1]) for i in range(10)]
    ce = np.array([q.loss for q in rows])
    loss, w = fr.focal_weight(ce, gamma, alpha)
    assert r.loss == pytest.approx(float(np.mean(loss)), rel=1e-12)
    np.testing.assert_allclose(r.dX, np.concatenate([w[i] / 10 * q.dX for i, q in enumerate(rows)]), rtol=1e-10,
                               atol=1e-16)
    np.testing.assert_allclose(r.dW, sum(w[i] / 10 * q.dW for i, q in enumerate(rows)), rtol=1e-10, atol=1e-16)
    # finite differences through the modulating factor
    eps = 1e-6
    Xp, Xm = X.copy(), X.copy()
    Xp[2, 3] += eps
    Xm[2, 3] -= eps
    num = (lr.focal_loss_only(Xp, W, y, gamma, alpha) - lr.focal_loss_only(Xm, W, y, gamma, alpha)) / (2 * eps)
    assert num == pytest.approx(r.dX[2, 3], rel=1e-6, abs=1e-10)


def test_focal_1_0_is_cross_entropy():
    X, W, y = _np(linear_inputs(10, 16, 40))
    a, b = lr.linear_head(X, W, y), lr.focal_head(X, W, y, 1.0, 0.0)
    assert b.loss == pytest.approx(a.loss, rel=1e-14)
    np.testing.assert_allclose(b.dX, a.dX, rtol=1e-12, atol=1e-15 * np.abs(a.dX).max())
    np.testing.assert_allclose(b.dW, a.dW, rtol=1e-12, atol=1e-15 * np.abs(a.dW).max())


def test_focal_sharded_weights():
    """The focal weights follow from the combined statistics: sharded backward with w equals the one piece."""
    X, W, y = _np(linear_inputs(12, 16, 37))
    full = lr.focal_head(X, W, y, 0.7, 2.0)
    bounds = lr.shard_bounds(37, 3)
    stats = [lr.sharded_partial_stats(X, W[:, lo:hi], y, lo)[:3] for lo, hi in bounds]
    M, logZ, w, loss = fr.sharded_combine(stats, 0.7, 2.0)
    assert loss == pytest.approx(full.loss, rel=1e-12)
    dX = sum(lr.sharded_backward(X, W[:, lo:hi], y, lo, M, logZ, w)[0] for lo, hi in bounds)
    np.testing.assert_allclose(dX, full.dX, rtol=1e-10, atol=1e-16)


def test_dw_keeps_component_along_w():
    """A-softmax's dW_j is orthogonal to w_j (the logits depend on w_j / |w_j| only); the linear
    head's is not: it is exactly X^T g."""
    X, W, y = _np(linear_inputs(16, 32, 50))
    a = ref.asoftmax_head(X, W, y, 4, 0.0)
    along_a = np.abs((a.dW * W).sum(axis=0)) / (np.linalg.norm(a.dW, axis=0) * np.linalg.norm(W, axis=0))
    assert along_a.max() < 1e-10
    r = lr.linear_head(X, W, y)
    along = np.abs((r.dW * W).sum(axis=0)) / (np.linalg.norm(r.dW, axis=0) * np.linalg.norm(W, axis=0))
    assert along.max() > 0.1
    g = np.exp(r.logits - r.logits.max(axis=1, keepdims=True))
    g /= g.sum(axis=1, keepdims=True)
    g[np.arange(16), y] -= 1.0
    np.testing.assert_allclose(r.dW, X.T @ (g / 16), rtol=1e-12, atol=1e-14 * np.abs(r.dW).max())


def test_zero_column_gives_zero_logit():
    X, W, y = _np(linear_inputs(8, 16, 20))
    W[:, 5] = 0.0
    y[y == 5] = 6
    r = lr.linear_head(X, W, y)
    assert np.all(r.logits[:, 5] == 0.0)
    assert np.all(r.dW[:, 5] != 0.0)          # a zero class still receives the softmax gradient
