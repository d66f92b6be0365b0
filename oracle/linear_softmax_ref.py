"""CPU oracle for the plain softmax classifier: unnormalised logits x_i . w_j, no margin.

TEST INFRASTRUCTURE ONLY, like asoftmax_ref.py: nothing in the product path imports it.

This is the head every network of the reference ships in the classifier slot: a bias-free
`fully_connected(features, num_classes)` followed by `sparse_softmax_cross_entropy`
(nets/sphere.py:84-111, nets/resnet.py:151-177, nets/shufflenet_v2.py:179-208).  Its
arithmetic is fixed by those two standard ops (DESIGN.md section 2.3), in float64 NumPy:

  f_ij = x_i . w_j  for every j, the target column included
  L    = mean_i (lse_i - f_iy)
  g    = (softmax(f) - onehot) / B,   dX = g W^T,   dW = X^T g

No norms enter anywhere, so dW has no component removed along w_j (the A-softmax dW does).
The file also holds the focal loss on these logits (focal_head / focal_loss_only, with the
weights of focal_ref.focal_weight) and the reference's graph restated in torch autograd
(linear_graph / step), which tests compare the closed forms against.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch

from .asoftmax_ref import shard_bounds, sharded_combine  # noqa: F401  (same partition and combine)
from .focal_ref import focal_weight


@dataclass
class LinearResult:
    loss: float
    logits: np.ndarray      # f [B, C]
    dX: np.ndarray          # [B, D]
    dW: np.ndarray          # [D, C]
    ce: np.ndarray          # [B] per-row cross-entropy
    w: np.ndarray           # [B] per-row gradient weight (1 for the cross-entropy)


def _f64(X, W, y):
    return (np.asarray(X, dtype=np.float64), np.asarray(W, dtype=np.float64),
            np.asarray(y).astype(np.int64))


def _lse(f):
    M = f.max(axis=1)
    return M + np.log(np.exp(f - M[:, None]).sum(axis=1))


def linear_head(X, W, y) -> LinearResult:
    """Forward + backward of mean softmax cross-entropy on f = X W, in one piece."""
    X, W, y = _f64(X, W, y)
    B = X.shape[0]
    rows = np.arange(B)
    f = X @ W
    lse = _lse(f)
    ce = lse - f[rows, y]
    g = np.exp(f - lse[:, None])
    g[rows, y] -= 1.0
    g /= B
    return LinearResult(float(ce.mean()), f, g @ W.T, X.T @ g, ce, np.ones(B))


def linear_loss_only(X, W, y) -> float:
    X, W, y = _f64(X, W, y)
    f = X @ W
    return float(np.mean(_lse(f) - f[np.arange(X.shape[0]), y]))


def linear_head_streamed(X, W, y, chunk: int = 16384) -> LinearResult:
    """The same head with the classes streamed in chunks: an online (max, sum-exp) pass, then the
    gradients chunk by chunk.  Never holds [B, C]; the fast form for C = 85,742 (logits is None)."""
    X, W, y = _f64(X, W, y)
    B, C = X.shape[0], W.shape[1]
    rows = np.arange(B)
    M = np.full(B, -np.inf)
    Z = np.zeros(B)
    for lo in range(0, C, chunk):
        f = X @ W[:, lo:lo + chunk]
        m = np.maximum(M, f.max(axis=1))
        Z = Z * np.exp(M - m) + np.exp(f - m[:, None]).sum(axis=1)
        M = m
    lse = M + np.log(Z)
    fy = np.einsum("bd,db->b", X, W[:, y])
    ce = lse - fy
    dX = np.zeros_like(X)
    dW = np.empty_like(W)
    for lo in range(0, C, chunk):
        hi = min(C, lo + chunk)
        g = np.exp(X @ W[:, lo:hi] - lse[:, None])
        own = (y >= lo) & (y < hi)
        g[rows[own], y[own] - lo] -= 1.0
        g /= B
        dX += g @ W[:, lo:hi].T
        dW[:, lo:hi] = X.T @ g
    return LinearResult(float(ce.mean()), None, dX, dW, ce, np.ones(B))


# --------------------------------------------------------------------------------------
# class-sharded evaluation: what each of G shards computes and exchanges
# --------------------------------------------------------------------------------------
def sharded_partial_stats(X, W_shard, y, class_offset):
    """Per-shard forward: (local max [B], local sum-exp [B], target logit or 0 [B], owned [B])."""
    X, W_shard, y = _f64(X, W_shard, y)
    f = X @ W_shard
    m = f.max(axis=1)
    z = np.exp(f - m[:, None]).sum(axis=1)
    yl = y - class_offset
    own = (yl >= 0) & (yl < W_shard.shape[1])
    fy = np.zeros(X.shape[0])
    fy[own] = f[np.nonzero(own)[0], yl[own]]
    return m, z, fy, own


def sharded_backward(X, W_shard, y, class_offset, M, logZ, w=None):
    """Per-shard backward from the combined (M, log Z) and, for the focal loss, the rows' weights
    w (None: cross-entropy).  The -1 of the target column goes to the shard that owns y_i.
    Returns (this shard's dX contribution [B, D], the shard's dW)."""
    X, W_shard, y = _f64(X, W_shard, y)
    B = X.shape[0]
    lse = np.asarray(M) + np.asarray(logZ)
    g = np.exp(X @ W_shard - lse[:, None])
    yl = y - class_offset
    own = np.nonzero((yl >= 0) & (yl < W_shard.shape[1]))[0]
    g[own, yl[own]] -= 1.0
    g /= B
    if w is not None:
        g *= np.asarray(w, dtype=np.float64)[:, None]
    return g @ W_shard.T, X.T @ g


# --------------------------------------------------------------------------------------
# the reference's focal loss (loss.py:18-27) on the linear logits
# --------------------------------------------------------------------------------------
def focal_head(X, W, y, gamma: float = 1.0, alpha: float = 2.0) -> LinearResult:
    """L = mean_i gamma (1 - p_iy)^alpha ce_i on f = X W: every row's cross-entropy gradient
    times w_i (focal_ref.focal_weight)."""
    r = linear_head(X, W, y)
    loss, w = focal_weight(r.ce, gamma, alpha)
    X, W, y = _f64(X, W, y)
    B = X.shape[0]
    g = np.exp(r.logits - _lse(r.logits)[:, None])
    g[np.arange(B), y] -= 1.0
    g *= (w / B)[:, None]
    return LinearResult(float(np.mean(loss)), r.logits, g @ W.T, X.T @ g, r.ce, w)


def focal_loss_only(X, W, y, gamma: float = 1.0, alpha: float = 2.0) -> float:
    X, W, y = _f64(X, W, y)
    f = X @ W
    ce = _lse(f) - f[np.arange(X.shape[0]), y]
    return float(np.mean(focal_weight(ce, gamma, alpha)[0]))


# --------------------------------------------------------------------------------------
# the reference's shipped graph in torch autograd: tf.matmul, sparse softmax CE, tf.gradients
# --------------------------------------------------------------------------------------
def linear_graph(X: torch.Tensor, W: torch.Tensor, y: torch.Tensor):
    """Forward graph of fully_connected(features, C, biases=None) + mean sparse softmax CE;
    returns (loss, logits).  Differentiable w.r.t. X and W."""
    f = X @ W
    return torch.nn.functional.cross_entropy(f, y.long()), f


def step(X: torch.Tensor, W: torch.Tensor, y: torch.Tensor):
    """One fwd+bwd pass: (loss, dX, dW) like tf.gradients(cross_entropy, [features, weights])."""
    Xr = X.detach().clone().requires_grad_(True)
    Wr = W.detach().clone().requires_grad_(True)
    loss, _ = linear_graph(Xr, Wr, y)
    loss.backward()
    return loss.detach(), Xr.grad, Wr.grad
