"""Bounds of the head's outputs against the float64 oracle, shared by the GPU test modules.

Tolerances are BASELINE.json's: exact label / argmax indexing, loss within 1e-5 relative
(fp32 mode) / 2e-3 relative (bf16 mode), gradient cosine similarity >= 0.9999, and every
element of dX and dW within a bound of its matrix scale.
"""
import numpy as np
import torch

from oracle import asoftmax_ref as ref
from tf_face_toolbox_b200 import FusedOptimizer, asoftmax_head
from tf_face_toolbox_b200.synthetic import make_inputs

LOSS_TOL = {"fp32": 1e-5, "bf16": 2e-3}


def cosine(a, b):
    a = np.asarray(a, dtype=np.float64).ravel()
    b = np.asarray(b, dtype=np.float64).ravel()
    return float(a @ b / np.sqrt((a @ a) * (b @ b)))


def assert_within_oracle_bounds(inp, r, mode, loss, f, dX, dW, cos_min=0.9999, loss_floor=0.0, bf16_scale=1.0,
                                fp32_dx_atol=4e-6):
    """`r` is the oracle's result for `inp`; `f` the logits, or None to skip them.  `mode` selects
    the set of bounds; `bf16_scale` multiplies the tolerances of the bf16 set (for arithmetic
    whose products are that much more accurate than one bf16 rounding of each operand);
    `fp32_dx_atol` is the fp32 set's bound on every element of dX, relative to max |dX|."""
    assert np.isfinite(loss)
    # loss_floor: a single well-classified row has a loss near 0, where a relative bound on
    # the loss is a bound on the (bf16) logit error itself
    loss_tol = LOSS_TOL[mode] * (bf16_scale if mode == "bf16" else 1.0)
    assert abs(loss - r.loss) <= loss_tol * max(abs(r.loss), loss_floor), (loss, r.loss)
    assert cosine(dX, r.dX) >= cos_min, cosine(dX, r.dX)
    assert cosine(dW, r.dW) >= cos_min, cosine(dW, r.dW)
    if mode == "fp32":
        # fp32 mode runs on the tensor cores with G'' carried as two bf16 planes (2^-16):
        # element errors stay below a few 1e-6 of the matrix scale
        np.testing.assert_allclose(dX, r.dX, rtol=2e-3, atol=fp32_dx_atol * np.abs(r.dX).max() + 1e-12)
        np.testing.assert_allclose(dW, r.dW, rtol=2e-3, atol=1e-5 * np.abs(r.dW).max() + 1e-12)
    else:
        # bf16 mode: every element within 3 % of the matrix scale (a cosine over the whole matrix
        # does not notice one wrong column)
        ex, ew = np.abs(dX - r.dX).max() / np.abs(r.dX).max(), np.abs(dW - r.dW).max() / np.abs(r.dW).max()
        el = 3e-2 * bf16_scale
        assert ex <= el and ew <= el, (ex, ew, int(np.abs(dW - r.dW).max(axis=0).argmax()))
    if f is not None:
        tol = 1e-4 if mode == "fp32" else 0.35 * bf16_scale
        np.testing.assert_allclose(f, r.logits, atol=tol, rtol=1e-4 if mode == "fp32" else 2e-2 * bf16_scale)
        # exact label indexing: the margin-modified entry sits exactly at column y_i
        rows = np.arange(f.shape[0])
        y = inp.y.numpy()
        S = (inp.X.double().numpy() @ (inp.W.double().numpy() / r.c))
        moved = np.abs(S - r.logits) > 1e-9
        assert np.array_equal(np.nonzero(moved.any(axis=1))[0], rows[moved[rows, y]])
        # argmax equal wherever the oracle's top-2 gap exceeds the mode tolerance
        top2 = np.sort(r.logits, axis=1)[:, -2:]
        clear = (top2[:, 1] - top2[:, 0]) > (1e-3 if mode == "fp32" else 0.7 * bf16_scale)
        assert np.array_equal(f.argmax(axis=1)[clear], r.logits.argmax(axis=1)[clear])


def check_fused_optimizer_against_unfused(kind, mode, tag=None):
    """The optimizer fused into the dW kernel equals grad-then-update over 3 steps (TF Momentum /
    Adam semantics on cross_entropy + L2 reg_loss, data_parallel.py:186-196).  `tag` selects the
    handle, so that both calls run the kernels of the handle's environment."""
    dev = torch.device("cuda:0")
    B, D, Cn = 128, 128, 3000
    inp = make_inputs(B, D, Cn, seed=41)
    lr = 0.05 if kind == "Momentum" else 1e-3
    W_f = inp.W.to(dev).clone()
    opt = FusedOptimizer(kind, lr=lr, weight_decay=5e-4)
    Wr = inp.W.double().numpy().copy()
    s0 = np.zeros_like(Wr)
    s1 = np.zeros_like(Wr)
    X, y = inp.X.to(dev), inp.y.to(dev)
    for step in range(1, 4):
        # reference: gradient from the (already parity-tested) unfused call on the same weights
        Wcur = torch.from_numpy(Wr).float().to(dev)
        _, _, _, dW = asoftmax_head(X, y, Cn, 4, 5.0, weights=Wcur, mode=mode, _handle_tag=tag)
        Wr32 = Wcur.double().cpu().numpy()
        Wr, s0, s1n = ref.optimizer_step(Wr32, dW.double().cpu().numpy(), s0, s1, kind.lower(), lr=lr, step=step)
        s1 = s1n if s1n is not None else s1
        loss, _, dX, dW_none = asoftmax_head(X, y, Cn, 4, 5.0, weights=W_f, mode=mode, optimizer=opt,
                                             _handle_tag=tag)
        assert dW_none is None and np.isfinite(float(loss))
        torch.cuda.synchronize()
        upd_f = (W_f.double().cpu().numpy() - inp.W.double().numpy())
        upd_r = (Wr - inp.W.double().numpy())
        # Adam's m/sqrt(v) is sign-like on its first steps, which amplifies the bf16-vs-fp32
        # projection difference on near-zero gradient entries
        cos_min = 0.999 if (kind == "Adam" and mode == "bf16") else 0.9999
        assert cosine(upd_f, upd_r) >= cos_min, (step, cosine(upd_f, upd_r))
        # fp32: same arithmetic up to rounding.  bf16: the fused epilogue projects with the fp32
        # master weight, the unfused one with its bf16 copy (2^-9 relative on that term)
        if not (kind == "Adam" and mode == "bf16"):
            tol = 2e-3 if mode == "fp32" else 3e-2
            np.testing.assert_allclose(upd_f, upd_r, rtol=0, atol=tol * np.abs(upd_r).max())
        else:
            # Adam's first steps are sign-like (m / sqrt(v) = +-1), so an element whose gradient is
            # near zero may flip between the two projections and move by 2 lr; everywhere else the
            # updates agree.  Bound the flips instead of waving every element through: at most
            # 2 % of the elements may differ by more than 10 % of the step, none by more than 2 lr.
            diff = np.abs(upd_f - upd_r)
            step_sz = np.abs(upd_r).max()
            assert diff.max() <= 2.05 * step_sz
            assert (diff > 0.1 * step_sz).mean() <= 0.02, (diff > 0.1 * step_sz).mean()
    # the plain path is unaffected afterwards (optimizer disarmed): dW is returned again
    _, _, _, dW2 = asoftmax_head(X, y, Cn, 4, 5.0, weights=W_f, mode=mode, _handle_tag=tag)
    assert dW2 is not None
