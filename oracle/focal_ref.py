"""CPU oracle for the focal loss on the head's margin logits (the reference's loss.py:18-27).

TEST INFRASTRUCTURE ONLY, like asoftmax_ref.py: nothing in the product path imports it.

The loss sits on top of whichever margin produces the logits f (A-softmax psi with lambda, or
the additive phi), in float64 NumPy:

  ce_i = lse_i - f_iy,   p_i = e^{-ce_i},   u_i = 1 - p_i
  L    = mean_i gamma u_i^alpha ce_i
  dL_i / df_ij = w_i (softmax(f_i)_j - delta_{j,y_i}),
  w_i  = gamma (u_i^alpha + alpha p_i u_i^(alpha - 1) ce_i)

Names follow the reference, not Lin et al.: gamma is the multiplier and alpha the exponent.
The gradient goes through the modulating factor (no stop-gradient).  So every row's gradient
is the cross-entropy gradient of that row times w_i.  The one-piece form therefore adds no
margin math of its own: it runs each row through the existing oracles as a one-row batch
(whose loss is ce_i and whose gradients are those of ce_i) and sums the rows with the weights
w_i / B.  The class-sharded form combines the same (max, sum-exp, f_y) statistics as the
cross-entropy; w_i follows from the combined row, so every shard scales its rows by the same
w_i.  Its per-shard backward is the cross-entropy closed form of the margin head (as in
additive_margin_ref.sharded_backward; asoftmax_ref.py shards only up to the combine) on the
existing oracles' psi_kform / phi, with each row of G' scaled by w_i.  Being vectorised, it is
also the fast form for large shapes (one shard holding every class).

`margin` is None for A-softmax (with m, lam) or a tuple (s, m2, m3) for the additive heads.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from . import additive_margin_ref as am
from . import asoftmax_ref as ref
from .asoftmax_ref import shard_bounds  # noqa: F401  (the same class partition)


def focal_weight(ce, gamma: float, alpha: float):
    """(loss_i, w_i) from the rows' cross-entropies, evaluated without cancellation:
    u = -expm1(-ce); the second term of w as alpha p (ce/u) u^alpha with ce/u := 1 at u == 0, so
    alpha < 1 stays finite as p -> 1; alpha = 0 gives w = gamma exactly."""
    ce = np.asarray(ce, dtype=np.float64)
    c = np.maximum(ce, 0.0)
    p = np.exp(-c)
    u = -np.expm1(-c)
    ua = np.power(u, alpha)
    with np.errstate(divide="ignore", invalid="ignore"):
        cu = np.where(u > 0.0, c / np.where(u > 0.0, u, 1.0), 1.0)
    w = gamma * (ua + alpha * p * cu * ua)
    return gamma * ua * ce, w


@dataclass
class FocalResult:
    loss: float
    logits: np.ndarray      # f [B, C], the margin logits
    dX: np.ndarray          # [B, D]
    dW: np.ndarray          # [D, C]
    c: np.ndarray           # [C] class-weight column norms
    ce: np.ndarray          # [B] per-row cross-entropy
    w: np.ndarray           # [B] per-row gradient weight


def _row_head(Xi, W, yi, m, lam, margin):
    if margin is None:
        return ref.asoftmax_head(Xi, W, yi, m, lam)
    s, m2, m3 = margin
    return am.additive_head(Xi, W, yi, s, m2, m3)


def focal_head(X, W, y, gamma: float = 1.0, alpha: float = 2.0, m: int = 4, lam: float = 0.0,
               margin=None) -> FocalResult:
    """Forward + backward of the focal loss on the margin head, in one piece."""
    X = np.asarray(X, dtype=np.float64)
    W = np.asarray(W, dtype=np.float64)
    y = np.asarray(y).astype(np.int64)
    B = X.shape[0]
    rows = [_row_head(X[i:i + 1], W, y[i:i + 1], m, lam, margin) for i in range(B)]
    ce = np.array([r.loss for r in rows])
    loss, w = focal_weight(ce, gamma, alpha)
    k = w / B
    dX = np.concatenate([k[i] * r.dX for i, r in enumerate(rows)])
    dW = np.zeros_like(W)
    for i, r in enumerate(rows):
        dW += k[i] * r.dW
    logits = np.concatenate([r.logits for r in rows])
    return FocalResult(float(np.mean(loss)), logits, dX, dW, rows[0].c, ce, w)


def focal_loss_only(X, W, y, gamma: float = 1.0, alpha: float = 2.0, m: int = 4, lam: float = 0.0,
                    margin=None) -> float:
    """Loss without gradients (for finite differences)."""
    X = np.asarray(X, dtype=np.float64)
    W = np.asarray(W, dtype=np.float64)
    y = np.asarray(y).astype(np.int64)
    if margin is None:
        ce = [ref.asoftmax_loss_only(X[i:i + 1], W, y[i:i + 1], m, lam) for i in range(X.shape[0])]
    else:
        s, m2, m3 = margin
        ce = [am.additive_loss_only(X[i:i + 1], W, y[i:i + 1], s, m2, m3) for i in range(X.shape[0])]
    return float(np.mean(focal_weight(np.array(ce), gamma, alpha)[0]))


# --------------------------------------------------------------------------------------
# class-sharded evaluation: what each of G shards computes and exchanges
# --------------------------------------------------------------------------------------
def sharded_partial_stats(X, W_shard, y, class_offset, m=4, lam=0.0, margin=None):
    """Per-shard forward of the margin head (unchanged by the loss): (local max [B], local
    sum-exp [B], target logit or 0 [B], owned [B])."""
    if margin is None:
        return ref.sharded_partial_stats(X, W_shard, y, class_offset, m, lam)
    s, m2, m3 = margin
    return am.sharded_partial_stats(X, W_shard, y, class_offset, s, m2, m3)


def sharded_combine(stats, gamma: float, alpha: float):
    """Combine per-shard (max, sum-exp, target-or-0) exactly as the cross-entropy does, then the
    focal quantities of every row: returns (M, log Z, w [B], loss)."""
    M, logZ, _ = ref.sharded_combine(stats)
    fy = np.sum(np.stack([s[2] for s in stats]), axis=0)
    loss, w = focal_weight(M + logZ - fy, gamma, alpha)
    return M, logZ, w, float(np.mean(loss))


def sharded_backward(X, W_shard, y, class_offset, M, logZ, w, m=4, lam=0.0, margin=None):
    """Per-shard backward of the focal loss from the combined (M, log Z) and the rows' w: the
    cross-entropy closed form of the margin head with every row's G' (and the A-softmax r_i)
    scaled by w_i.  The target column and r_i go to the shard that owns y_i.  Returns (this
    shard's dX contribution [B, D], the shard's dW)."""
    X = np.asarray(X, dtype=np.float64)
    W_shard = np.asarray(W_shard, dtype=np.float64)
    y = np.asarray(y).astype(np.int64)
    w = np.asarray(w, dtype=np.float64)
    B = X.shape[0]
    lse = np.asarray(M) + np.asarray(logZ)
    yl = y - class_offset
    own = np.nonzero((yl >= 0) & (yl < W_shard.shape[1]))[0]
    if margin is not None:
        s, m2, m3 = margin
        n, c, Xh, What, S = am._logits(X, W_shard, s)
        t = np.clip(S[own, yl[own]] / s, -1.0, 1.0)
        ph, dph, _ = am.phi(t, m2, m3)
        f = S.copy()
        f[own, yl[own]] = s * ph
        Gp = np.exp(f - lse[:, None]) / B
        Gp[own, yl[own]] = (Gp[own, yl[own]] - 1.0 / B) * dph
        Gp *= w[:, None]
        v = Gp @ What.T
        dXp = (s / n)[:, None] * (v - (Xh * v).sum(axis=1)[:, None] * Xh)
        q = (Gp * S).sum(axis=0)
        return dXp, (s * (Xh.T @ Gp) - What * q) / c
    n = np.sqrt((X * X).sum(axis=1))
    c = np.sqrt((W_shard * W_shard).sum(axis=0))
    What = W_shard / c
    S = X @ What
    Gp = np.exp(S - lse[:, None]) / B
    r = np.zeros(B)
    if len(own):
        s_y = S[own, yl[own]]
        t = np.clip(s_y / n[own], -1.0, 1.0)
        psi, dpsi, _ = ref.psi_kform(t, m)
        f_y = (lam * s_y + n[own] * psi) / (1.0 + lam)
        g_y = (np.exp(f_y - lse[own]) - 1.0) / B
        Gp[own, yl[own]] = g_y * (lam + dpsi) / (1.0 + lam)
        r[own] = g_y * (psi - t * dpsi) / ((1.0 + lam) * n[own])
    Gp *= w[:, None]
    r *= w
    dXp = Gp @ What.T + r[:, None] * X
    q = (Gp * S).sum(axis=0)
    return dXp, (X.T @ Gp - What * q) / c
