"""Every tensor-core kernel instantiation and every schedule knob against the float64 oracle.

The library picks among 17 `umma_kernel<KIND, CG, BNT>` instantiations (single CTA, 256-wide CTA
pair, 128-wide CTA pair) and several schedules; the default settings reach only some of them at
any given shape.  Each variant below is selected through the environment variables asm_create
reads, on a handle of its own (a tag), at shapes chosen for the edges where tiles go wrong, and
is checked on every element against the oracle, for determinism, and -- where the knob changes
only the schedule -- bit for bit against the default.

Outputs are written into NaN-filled buffers, so an element no kernel writes cannot pass.
"""
import collections
import functools
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from head_checks import assert_within_oracle_bounds, check_fused_optimizer_against_unfused
from oracle import asoftmax_ref as ref
from tf_face_toolbox_b200 import _lib, head
from tf_face_toolbox_b200.head import drop_handle, get_handle
from tf_face_toolbox_b200.synthetic import make_inputs

pytestmark = pytest.mark.gpu
TESTS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(TESTS)
DEV = "cuda:0"
TAG = "kernel-variants"          # first element of the tag of every handle this module creates
LAM = 5.0
MODES = ("fp32", "bf16")

# (B, D, C) and the edge each shape targets
SHAPES = [
    (1, 64, 300),          # one row, one K block, maximal KS
    (128, 128, 1000),      # exactly one row tile: the pair FWD / DX fall back to single CTAs
    (129, 192, 1001),      # second 128-row half nearly empty; odd C (no dW TMA); partial 256-wide d tile
    (384, 320, 2050),      # three row tiles (half-empty pair); C % 4 == 2 shifted odd-row boxes
    (257, 512, 4099),      # C % 4 == 3
    (1000, 64, 40),        # C below one 64-class box; every class labelled many times; B % 64 != 0
    (64, 2048, 700),       # many K blocks
    (512, 512, 20000),     # several tiles per CTA pair with a ragged last round, at both widths
]
# (B, D, C, m): m = 4 everywhere, m = 1 and m = 3 on two shapes
CASES = [s + (4,) for s in SHAPES] + [(129, 192, 1001, 1), (129, 192, 1001, 3),
                                      (384, 320, 2050, 1), (384, 320, 2050, 3)]
LOGITS_CASE = (129, 192, 1001, 4)    # the logits are checked on this case of every variant
OUTPUTS = ("loss", "logits", "dX", "dW")


def case_id(case):
    return "B{}-D{}-C{}-m{}".format(*case)


# name -> (environment, modes, outputs that equal the default's bit for bit)
VARIANTS = {
    "default": ({}, MODES, OUTPUTS),
    # every single-CTA instantiation: FWD / BWDG / DW / DWF / DX <1>
    "cg0": ({"ASM_UMMA_CG": "0"}, MODES, ()),
    # mixed pairing; the dW / dX side-by-side split needs bits 2 and 3, so it is off
    "cg5": ({"ASM_UMMA_CG": "5"}, MODES, ()),
    "cg10": ({"ASM_UMMA_CG": "10"}, MODES, ()),
    # each pair kernel at a forced width
    "bn128": ({"ASM_UMMA_BN": "128"}, MODES, ()),
    "bn256": ({"ASM_UMMA_BN": "256"}, MODES, ()),
    # The dX split-K count follows the SMs the dX kernel gets, which changes its sums; dW tiles are
    # computed whole by one CTA (pair) whatever the grid, and the loss and logits come before.
    "dw_pairs0": ({"ASM_DW_PAIRS": "0"}, MODES, ("loss", "logits", "dW")),
    "dw_pairs10": ({"ASM_DW_PAIRS": "10"}, MODES, ("loss", "logits", "dW")),
    "dw_pairs70": ({"ASM_DW_PAIRS": "70"}, MODES, ("loss", "logits", "dW")),
    "no_overlap": ({"ASM_NO_OVERLAP": "1"}, MODES, ("loss", "logits", "dW")),
    # contiguous split-K ranges instead of interleaved ones: other dX sums; BWDG's sweep direction
    # only reorders whole tiles
    "l2_order0": ({"ASM_L2_ORDER": "0"}, MODES, ("loss", "logits", "dW")),
    # store paths, cache policies and launch chaining do not touch the arithmetic
    "dw_tma0": ({"ASM_DW_TMA": "0"}, MODES, OUTPUTS),
    "l2_hints0": ({"ASM_L2_HINTS": "0"}, MODES, OUTPUTS),
    "l2_hints1": ({"ASM_L2_HINTS": "1"}, MODES, OUTPUTS),
    "l2_hints2": ({"ASM_L2_HINTS": "2"}, MODES, OUTPUTS),
    "pdl0": ({"ASM_PDL": "0"}, MODES, OUTPUTS),
    # the dX kernel's deferred loss reproduces combine's fixed-order reduction, so the loss is
    # compared too
    "defer_loss0": ({"ASM_DEFER_LOSS": "0"}, MODES, OUTPUTS),
    "fp32_simt": ({"ASM_FP32_SIMT": "1"}, ("fp32",), ()),
}

# Knobs cached in function-static variables (x3_segments(), launch_prep): one child process per
# setting.  name -> (environment, modes, bf16_scale of the oracle bounds, or None for the mode's own)
STATIC_VARIANTS = {
    # ASM_X3_SEGS=3 keeps the plane pairs (0,0), (0,1), (1,0).  test_x3_split_cpu pins the error of
    # that chain below 2^-14 of sum_k |a_k||b_k|; one bf16 rounding of each operand (bf16 mode, whose
    # bounds hold) errs by up to 2^-8 of the same scale.  Loss, logits, dX and dW move linearly with
    # the product error to first order, so the bf16 bounds scaled by 2^-14 / 2^-8 = 1/64 hold.  (The
    # backward chains against the two-plane G'' drop (1,1) and (0,2): 2 * 2^-16, inside 2^-14 too.)
    "x3_segs3": ({"ASM_X3_SEGS": "3"}, ("fp32",), 2.0 ** -6),
    # the other block shapes of the norm kernel sum the column norms in another order
    "prep_shape1": ({"ASM_PREP_SHAPE": "1"}, MODES, None),
    "prep_shape2": ({"ASM_PREP_SHAPE": "2"}, MODES, None),
    "prep_shape3": ({"ASM_PREP_SHAPE": "3"}, MODES, None),
    "prep_auto": ({"ASM_PREP_AUTO": "1"}, MODES, None),
}

# the fused optimizer (DWOPT) at all three geometries, and the streaming update instead of it;
# the default settings are covered by test_head_gpu's test_fused_optimizer_matches_unfused_update
OPT_VARIANTS = {
    "cg0": {"ASM_UMMA_CG": "0"},
    "bn128": {"ASM_UMMA_BN": "128"},
    "bn256": {"ASM_UMMA_BN": "256"},
    "opt_stream": {"ASM_OPT_STREAM": "1"},
}

# knobs read by the library that this module does not vary, and why
EXCLUDED = {
    "ASM_P2P_TIMEOUT_MS": "NVLink transport, covered by test_p2p_gpu.py",
    "ASM_P2P_WAITERS": "NVLink transport, covered by test_p2p_gpu.py",
    "ASM_MAX_HANDLES": "size of the Python handle cache, no kernel path",
    "ASM_B200_LIB": "selects another build of the library, no kernel path",
}

TESTED_KNOBS = sorted({k for env, *_ in VARIANTS.values() for k in env}
                      | {k for env, *_ in STATIC_VARIANTS.values() for k in env}
                      | {k for env in OPT_VARIANTS.values() for k in env})

Out = collections.namedtuple("Out", OUTPUTS)


@functools.lru_cache(maxsize=None)
def case_inputs(B, D, C):
    """make_inputs' mixture around labels that include the first and the last class (the
    classes next to the padded columns)."""
    g = torch.Generator().manual_seed(B * 131 + D * 7 + C)
    y = torch.randint(0, C, (B,), generator=g)
    if B >= 2:
        y[1::7] = 0
        y[3::7] = C - 1
        y[-2], y[-1] = 0, C - 1
    return make_inputs(B, D, C, seed=B + D + C, labels=y)


@functools.lru_cache(maxsize=None)
def oracle(case):
    B, D, C, m = case
    inp = case_inputs(B, D, C)
    return ref.asoftmax_head(inp.X.numpy(), inp.W.numpy(), inp.y.numpy(), m, LAM)


def handle(case, mode, name):
    B, D, C, m = case
    return get_handle(DEV, D, C, C, 0, B, m, mode, tag=(TAG, name))


def run(h, case, logits=False):
    """One asm_forward_backward on `h` into NaN-filled output buffers."""
    B, D, C, _ = case
    inp = case_inputs(B, D, C)
    X, y, W = inp.X.to(DEV), inp.y.to(DEV), inp.W.to(DEV)
    nan = float("nan")
    loss = torch.full((1,), nan, device=DEV)
    f = torch.full((B, C), nan, device=DEV) if logits else None
    dX = torch.full((B, D), nan, device=DEV)
    dW = torch.full((D, C), nan, device=DEV)
    with torch.cuda.device(DEV):
        rc = h.lib.asm_forward_backward(h.ptr, X.data_ptr(), B, y.data_ptr(), 4, W.data_ptr(), LAM, loss.data_ptr(),
                                        f.data_ptr() if logits else None, dX.data_ptr(), dW.data_ptr(),
                                        torch.cuda.current_stream().cuda_stream)
        _lib.check(rc, h.ptr)
    torch.cuda.synchronize()
    return Out(float(loss.item()), f.cpu().numpy() if logits else None, dX.cpu().numpy(), dW.cpu().numpy())


def assert_bitwise(a, b, names=OUTPUTS):
    for name in names:
        x, z = getattr(a, name), getattr(b, name)
        if x is None and z is None:
            continue
        assert np.array_equal(np.asarray(x), np.asarray(z)), (name, float(np.nanmax(np.abs(np.asarray(x) - z))))


# fp32 mode, every element of dX relative to max |dX|: 4e-6 (test_head_gpu's bound) holds up to
# C ~ 4k.  At C = 20000 the B200 measured 5.1e-6 (default) and 1.1e-5 (ASM_DW_PAIRS=70, where the dX
# kernel gets 4 CTA pairs and KS = 1: one fp32 accumulator chain over 20224 classes x 5 plane pairs),
# and logits near 24 resolve f_y - lse only to ~2e-6, which a confident row's 1 - p_y of ~1e-5
# turns into a percent-level error of that row.  There the bound is the project's fp32
# every-element parity bound (bench.py ELEM_TOL, BASELINE.md).
FP32_DX_ATOL = {(512, 512, 20000, 4): 5e-5}


def assert_oracle(case, mode, out, bf16_scale=1.0):
    B, D, C, _ = case
    assert_within_oracle_bounds(case_inputs(B, D, C), oracle(case), mode, out.loss, out.logits, out.dX, out.dW,
                                loss_floor=10.0 if B == 1 else 0.0, bf16_scale=bf16_scale,
                                fp32_dx_atol=FP32_DX_ATOL.get(case, 4e-6))


@pytest.fixture
def knobs(monkeypatch):
    """No tested knob from the caller's environment; every handle this module made is released
    afterwards (tagged handles are never evicted, and each holds a device workspace)."""
    for k in TESTED_KNOBS:
        monkeypatch.delenv(k, raising=False)
    yield monkeypatch
    for key in [k for k in head._HANDLES if isinstance(k[-1], tuple) and k[-1][:1] == (TAG,)]:
        drop_handle(head._HANDLES[key])


_DEFAULTS = {}


def default_outputs(case, mode):
    """The production path's outputs (computed once, before any knob is set)."""
    key = (case, mode)
    if key not in _DEFAULTS:
        h = handle(case, mode, "default-reference")
        _DEFAULTS[key] = run(h, case, logits=case == LOGITS_CASE)
        drop_handle(h)
    return _DEFAULTS[key]


# ------------------------------------------------------------------------- handle state
@pytest.mark.parametrize("mode", MODES)
def test_profiling_round_trip_keeps_results(mode, knobs):
    """asm_set_profiling(h, 1) gives the dX kernel every SM (no dW / dX split), which raises the dX
    split-K count at the same B: the dX partials' TMA map has to follow it, or the stores of the
    extra splits fall outside the map and dx_finish adds stale workspace.  Mode 2 keeps the split."""
    case = (256, 512, 4000, 4)
    def profiling(h, level):
        _lib.check(h.lib.asm_set_profiling(h.ptr, level), h.ptr)

    h = handle(case, mode, "profiling")
    A = run(h, case)
    profiling(h, 1)
    P1 = run(h, case)
    profiling(h, 2)
    P2 = run(h, case)
    profiling(h, 0)
    A2 = run(h, case)
    fresh = handle(case, mode, "profiling-fresh")
    profiling(fresh, 1)
    F1 = run(fresh, case)
    assert_oracle(case, mode, P1)
    assert_oracle(case, mode, P2)
    assert_bitwise(A2, A)
    # dW tiles are computed whole on one CTA pair whatever the grid; the deferred loss is reduced
    # by block 0 of the dX kernel alone, in an order fixed by B, so it does not depend on KS either
    assert_bitwise(P1, A, ("loss", "dW"))
    assert_bitwise(P2, A)          # per-phase events keep the schedule and its arithmetic
    assert_bitwise(F1, P1)


@pytest.mark.parametrize("mode", MODES)
def test_batch_sizes_within_one_handle_bucket(mode, knobs):
    """Handles are keyed by B rounded up to 128: one handle runs B = 256, 130, 256, 200, 129 and
    each result equals a fresh handle's at that B (no state of an earlier, larger batch leaks)."""
    shared = handle((256, 512, 4000, 4), mode, "bucket")
    for B in (256, 130, 256, 200, 129):
        case = (B, 512, 4000, 4)
        got = run(shared, case)
        fresh = handle(case, mode, ("fresh", B))
        want = run(fresh, case)
        drop_handle(fresh)
        assert_bitwise(got, want)


# ------------------------------------------------------------------------- variant matrix
@pytest.mark.parametrize("case", CASES, ids=case_id)
@pytest.mark.parametrize("variant,mode", [(v, m) for v, (_, modes, _) in VARIANTS.items() for m in modes])
def test_variant_against_oracle(variant, mode, case, knobs):
    env, _, same_as_default = VARIANTS[variant]
    base = default_outputs(case, mode)
    for k, v in env.items():
        knobs.setenv(k, v)
    h = handle(case, mode, variant)           # asm_create reads the knobs
    a = run(h, case, logits=case == LOGITS_CASE)
    b = run(h, case, logits=case == LOGITS_CASE)
    assert_oracle(case, mode, a)
    assert_bitwise(a, b)                      # deterministic
    assert_bitwise(a, base, same_as_default)


_CHILD = ("import sys; sys.path[:0] = sys.argv[1:3]; import test_kernel_variants_gpu as kv; "
          "kv.child_main(sys.argv[3], sys.argv[4:])")


def child_main(outdir, modes):
    """Runs every case twice in this process's environment, checks the two runs are equal bit for
    bit, and saves the outputs for the parent to check against the oracle."""
    for mode in modes:
        for case in CASES:
            h = handle(case, mode, "child")
            a = run(h, case, logits=case == LOGITS_CASE)
            assert_bitwise(a, run(h, case, logits=case == LOGITS_CASE))
            drop_handle(h)
            np.savez(os.path.join(outdir, f"{mode}-{case_id(case)}.npz"),
                     **{k: v for k, v in a._asdict().items() if v is not None})


@pytest.mark.parametrize("variant", list(STATIC_VARIANTS))
def test_process_wide_variant_against_oracle(variant, knobs, tmp_path):
    env, modes, scale = STATIC_VARIANTS[variant]
    child_env = dict(os.environ, **env)
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", _CHILD, ROOT, TESTS, str(tmp_path), *modes]
    p = subprocess.run(cmd, env=child_env, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    for mode in modes:
        for case in CASES:
            z = np.load(tmp_path / f"{mode}-{case_id(case)}.npz")
            out = Out(float(z["loss"]), z["logits"] if "logits" in z.files else None, z["dX"], z["dW"])
            if scale is None:
                assert_oracle(case, mode, out)
            else:
                assert_oracle(case, "bf16", out, bf16_scale=scale)


# ------------------------------------------------------------------------- fused optimizer
@pytest.mark.parametrize("kind", ["Momentum", "Adam"])
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("variant", list(OPT_VARIANTS))
def test_fused_optimizer_variant(variant, mode, kind, knobs):
    for k, v in OPT_VARIANTS[variant].items():
        knobs.setenv(k, v)
    check_fused_optimizer_against_unfused(kind, mode, tag=(TAG, "opt", variant))
