"""CPU oracle for the additive-margin heads (ArcFace / CosFace) on L2-normalised embeddings.

TEST INFRASTRUCTURE ONLY, like asoftmax_ref.py: nothing in the product path imports it.

No reference pins these heads; the conventions are the ones DESIGN.md section 2.1 fixes
(InsightFace's combined margin without m1), in float64 NumPy:

  n_i = |x_i|,  x^_i = x_i / n_i,  c_j = |w_j|,  s_ij = s x^_i . w_j / c_j,  t_i = clip(s_iy / s, -1, 1)
  tau = cos(pi - m2)
  phi(t) = t cos m2 - sin(theta) sin m2 - m3   (= cos(theta + m2) - m3)   if t >= tau,
           sin(theta) = sqrt(max(1 - t^2, 1e-12))
         = t - m2 sin m2 - m3                                             otherwise
  (the usual non-"easy-margin" fallback; phi is discontinuous at tau)
  f_iy = s phi(t_i),  f_ij = s_ij otherwise,  L = mean_i [logsumexp_j f_ij - f_iy]

Backward (phi' and the branch are piecewise constants, as k is for psi):
  g = (softmax(f) - onehot) / B,  G' = g except G'_iy = g_iy phi'(t_i)
  dW = (s X^T G' - W^ diag(q)) diag(1/c),  q_j = sum_i G'_ij s_ij
  dX_i = (s / n_i) (v_i - (x^_i . v_i) x^_i),  v_i = sum_j G'_ij w^_j
m2 = 0 is CosFace, m3 = 0 ArcFace, both zero the normalised-feature softmax with scale s.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np

from .asoftmax_ref import shard_bounds, sharded_combine  # noqa: F401  (same combine for every margin)


def tau(m2: float) -> float:
    """Threshold of the first branch: cos(pi - m2)."""
    return math.cos(math.pi - m2)


def phi(t, m2: float, m3: float):
    """(phi(t), phi'(t), first-branch mask) for t already clipped to [-1, 1]."""
    t = np.asarray(t, dtype=np.float64)
    st = np.sqrt(np.maximum(1.0 - t * t, 1e-12))
    first = t >= tau(m2)
    cm, sm = math.cos(m2), math.sin(m2)
    ph = np.where(first, t * cm - st * sm - m3, t - m2 * sm - m3)
    dph = np.where(first, cm + t * sm / st, 1.0)
    return ph, dph, first


@dataclass
class MarginResult:
    loss: float
    logits: np.ndarray      # f [B, C]
    dX: np.ndarray          # [B, D]
    dW: np.ndarray          # [D, C]
    n: np.ndarray           # [B]
    c: np.ndarray           # [C]
    t: np.ndarray           # [B] target cosine
    first: np.ndarray       # [B] bool: t >= tau


def _logits(X, W, s):
    n = np.sqrt((X * X).sum(axis=1))
    c = np.sqrt((W * W).sum(axis=0))
    Xh = X / n[:, None]
    What = W / c
    return n, c, Xh, What, s * (Xh @ What)


def additive_head(X, W, y, s: float = 64.0, m2: float = 0.5, m3: float = 0.0) -> MarginResult:
    """Forward + closed-form backward of the additive-margin head, in one piece."""
    X = np.asarray(X, dtype=np.float64)
    W = np.asarray(W, dtype=np.float64)
    y = np.asarray(y).astype(np.int64)
    B = X.shape[0]
    rows = np.arange(B)
    n, c, Xh, What, S = _logits(X, W, s)
    t = np.clip(S[rows, y] / s, -1.0, 1.0)
    ph, dph, first = phi(t, m2, m3)
    f = S.copy()
    f[rows, y] = s * ph
    mx = f.max(axis=1)
    E = np.exp(f - mx[:, None])
    Z = E.sum(axis=1)
    loss = float(np.mean(np.log(Z) + mx - f[rows, y]))
    Gp = E / Z[:, None]
    Gp[rows, y] -= 1.0
    Gp /= B
    Gp[rows, y] *= dph
    v = Gp @ What.T
    dX = (s / n)[:, None] * (v - (Xh * v).sum(axis=1)[:, None] * Xh)
    q = (Gp * S).sum(axis=0)
    dW = (s * (Xh.T @ Gp) - What * q) / c
    return MarginResult(loss, f, dX, dW, n, c, t, first)


def additive_loss_only(X, W, y, s: float = 64.0, m2: float = 0.5, m3: float = 0.0) -> float:
    """Loss without gradients (for finite differences)."""
    X = np.asarray(X, dtype=np.float64)
    W = np.asarray(W, dtype=np.float64)
    y = np.asarray(y).astype(np.int64)
    rows = np.arange(X.shape[0])
    _, _, _, _, f = _logits(X, W, s)
    t = np.clip(f[rows, y] / s, -1.0, 1.0)
    f[rows, y] = s * phi(t, m2, m3)[0]
    mx = f.max(axis=1)
    return float(np.mean(np.log(np.exp(f - mx[:, None]).sum(axis=1)) + mx - f[rows, y]))


# --------------------------------------------------------------------------------------
# class-sharded evaluation: what each of G shards computes and exchanges
# --------------------------------------------------------------------------------------
def sharded_partial_stats(X, W_shard, y, class_offset, s=64.0, m2=0.5, m3=0.0):
    """Per-shard forward: (local max [B], local sum-exp [B], target logit or 0 [B], owned [B])."""
    X = np.asarray(X, dtype=np.float64)
    W_shard = np.asarray(W_shard, dtype=np.float64)
    y = np.asarray(y).astype(np.int64)
    B, Cl = X.shape[0], W_shard.shape[1]
    _, _, _, _, f = _logits(X, W_shard, s)
    yl = y - class_offset
    owned = (yl >= 0) & (yl < Cl)
    ro = np.nonzero(owned)[0]
    t = np.clip(f[ro, yl[ro]] / s, -1.0, 1.0)
    f[ro, yl[ro]] = s * phi(t, m2, m3)[0]
    mloc = f.max(axis=1) if Cl > 0 else np.full(B, -np.inf)
    zloc = np.exp(f - mloc[:, None]).sum(axis=1) if Cl > 0 else np.zeros(B)
    fy = np.zeros(B)
    fy[ro] = f[ro, yl[ro]]
    return mloc, zloc, fy, owned


def sharded_backward(X, W_shard, y, class_offset, M, logZ, s=64.0, m2=0.5, m3=0.0):
    """Per-shard backward from the combined (M, log Z): (this shard's dX contribution [B, D],
    already projected -- the projection is linear in v --, and the shard's complete dW)."""
    X = np.asarray(X, dtype=np.float64)
    W_shard = np.asarray(W_shard, dtype=np.float64)
    y = np.asarray(y).astype(np.int64)
    B = X.shape[0]
    n, c, Xh, What, S = _logits(X, W_shard, s)
    lse = np.asarray(M) + np.asarray(logZ)
    yl = y - class_offset
    own = np.nonzero((yl >= 0) & (yl < W_shard.shape[1]))[0]
    f = S.copy()
    t = np.clip(S[own, yl[own]] / s, -1.0, 1.0)
    ph, dph, _ = phi(t, m2, m3)
    f[own, yl[own]] = s * ph
    Gp = np.exp(f - lse[:, None]) / B
    Gp[own, yl[own]] = (Gp[own, yl[own]] - 1.0 / B) * dph
    v = Gp @ What.T
    dXp = (s / n)[:, None] * (v - (Xh * v).sum(axis=1)[:, None] * Xh)
    q = (Gp * S).sum(axis=0)
    dW = (s * (Xh.T @ Gp) - What * q) / c
    return dXp, dW
