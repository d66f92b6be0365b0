"""Cost of the additive-margin heads next to A-softmax, on one B200, in one process.

The GEMMs of the three kinds are the same kernels; the additive kind adds a second pass over
each embedding row in the norm kernel and runs the row-wise dX finish.  Workloads:
  cfg3      B = 512, C = 85,742, D = 512, bf16           (asm_forward_backward)
  cfg1      B = 256, C = 10,572, D = 512, fp32           (asm_forward_backward)
  cfg3_g2   cfg3 over G = 2 class shards with the NVLink transport, both ranks in this process on
            one GPU (tests/test_p2p_gpu.py's FakeRanks); a step is both ranks' asm_step_p2p
Every workload is first checked against the float64 oracles (loss, cosine and largest element
error of dX / dW).  Then A-softmax, ArcFace and CosFace steps are timed alternately: CUDA events
around a graph replay of the step on one GPU, a host clock around both ranks' eager step and a
device synchronise for cfg3_g2.  A per-kernel (asm_set_profiling 1) and per-phase (2) breakdown
of the eager step is averaged over separate runs.  The card's name, power limit and SM clock are
read in the same process.  Writes one JSON file.

    python scripts/bench_margins.py --out profiles/margins_b200.json [--steps 200] [--warmup 20]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from oracle import additive_margin_ref as am  # noqa: E402
from oracle import asoftmax_ref as ref  # noqa: E402
from tf_face_toolbox_b200 import AdditiveMargin, GraphedASoftmaxStep, _lib, asoftmax_head  # noqa: E402
from tf_face_toolbox_b200.head import get_handle  # noqa: E402
from tf_face_toolbox_b200.synthetic import make_inputs  # noqa: E402

DEV = torch.device("cuda:0")
KINDS = {"asoftmax": None, "arcface": AdditiveMargin.arcface(64.0, 0.5), "cosface": AdditiveMargin.cosface(64.0, 0.35)}
LAM = 5.0
TOL = {"fp32": (1e-5, 5e-5), "bf16": (2e-3, 3e-2)}      # loss relative, largest element error / matrix scale


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(zip(q.split(","), [v.strip() for v in r.stdout.strip().splitlines()[0].split(",")])) if r.returncode == 0 else {}


def oracle(inp, mg):
    X, W, y = inp.X.numpy(), inp.W.numpy(), inp.y.numpy()
    if mg is None:
        return ref.asoftmax_head(X, W, y, 4, LAM)
    return am.additive_head(X, W, y, mg.s, mg.m2, mg.m3)


def parity(r, mode, loss, dX, dW):
    def cos(a, b):
        a, b = a.astype(np.float64).ravel(), b.astype(np.float64).ravel()
        return float(a @ b / np.sqrt((a @ a) * (b @ b)))
    out = dict(loss_rel=abs(loss - r.loss) / abs(r.loss), cos_dX=cos(dX, r.dX), cos_dW=cos(dW, r.dW),
               max_err_dX=float(np.abs(dX - r.dX).max() / np.abs(r.dX).max()),
               max_err_dW=float(np.abs(dW - r.dW).max() / np.abs(r.dW).max()))
    lt, et = TOL[mode]
    ok = out["loss_rel"] <= lt and out["cos_dX"] >= 0.9999 and out["cos_dW"] >= 0.9999 and \
        out["max_err_dX"] <= et and out["max_err_dW"] <= et
    if not ok:
        raise SystemExit(f"parity with the oracle failed ({mode}): {out}")
    return out


def stats(ms):
    a = np.asarray(ms)
    return dict(median_ms=float(np.median(a)), p10_ms=float(np.percentile(a, 10)), p90_ms=float(np.percentile(a, 90)),
                steps=len(a))


def profile(h, step, level, n):
    names = (C.c_char * (32 * 16))()
    ms = (C.c_float * 16)()
    acc = {}
    _lib.check(h.lib.asm_set_profiling(h.ptr, level), h.ptr)
    for _ in range(n):
        step()
        k = h.lib.asm_get_profile(h.ptr, 16, ms, names)
        for i in range(k):
            nm = bytes(names[i * 32:(i + 1) * 32]).split(b"\0")[0].decode()
            acc[nm] = acc.get(nm, 0.0) + ms[i] / n * 1e3
    _lib.check(h.lib.asm_set_profiling(h.ptr, 0), h.ptr)
    return {k: round(v, 2) for k, v in acc.items()}        # microseconds


def single_gpu(name, B, D, Cn, mode, steps, warmup):
    inp = make_inputs(B, D, Cn)
    X, y, W = inp.X.to(DEV), inp.y.to(DEV), inp.W.to(DEV)
    res = {"shape": dict(B=B, D=D, C=Cn, mode=mode), "kinds": {}}
    fns = {}
    for kind, mg in KINDS.items():
        def step(mg=mg):
            return asoftmax_head(X, y, Cn, 4, LAM, weights=W, mode=mode, margin=mg)
        loss, _, dX, dW = step()
        torch.cuda.synchronize()
        res["kinds"][kind] = {"parity": parity(oracle(inp, mg), mode, float(loss), dX.cpu().numpy(), dW.cpu().numpy())}
        fns[kind] = step
    # timed: CUDA-graph replays of each kind's step (GraphedASoftmaxStep), so that host overhead of
    # the eager Python call does not hide the device time; inputs are loaded once, then replayed
    graphs = {}
    for kind, mg in KINDS.items():
        g = GraphedASoftmaxStep(W, B, m=4, mode=mode, margin=mg)
        g(X, y, LAM)
        graphs[kind] = g
    for _ in range(warmup):
        for g in graphs.values():
            g.graph.replay()
    ev = {k: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
          for k in graphs}
    for i in range(steps):                                  # alternate the kinds step by step
        for k, g in graphs.items():
            ev[k][i][0].record()
            g.graph.replay()
            ev[k][i][1].record()
    torch.cuda.synchronize()
    for k, g in graphs.items():
        res["kinds"][k]["step"] = stats([a.elapsed_time(b) for a, b in ev[k]])
        res["kinds"][k]["step"]["clock"] = "CUDA events around one graph replay of the step"
        g.close()
    for k in fns:
        h = get_handle(DEV, D, Cn, Cn, 0, B, 4, mode, margin=KINDS[k])
        res["kinds"][k]["per_kernel_us"] = profile(h, fns[k], 1, 20)
        res["kinds"][k]["per_phase_us"] = profile(h, fns[k], 2, 20)
    return res


def nvlink_g2(steps, warmup):
    from test_p2p_gpu import FakeRanks
    B, D, Cn, G = 512, 512, 85742, 2
    inp = make_inputs(B, D, Cn)
    res = {"shape": dict(B=B, D=D, C=Cn, mode="bf16", G=G), "kinds": {}}
    ranks = {}
    for kind, mg in KINDS.items():
        rk = FakeRanks(inp, G, "bf16", ("bench-margins", kind))
        if mg is not None:
            st = _lib.AsmMargin(_lib.MARGIN_ADDITIVE, mg.s, mg.m2, mg.m3)
            for h in rk.handles:
                _lib.check(h.lib.asm_set_margin(h.ptr, C.byref(st)), h.ptr)
        rk.step(LAM)
        torch.cuda.synchronize()
        r = oracle(inp, mg)
        dX = torch.cat([d for d in rk.dX]).cpu().numpy()
        dW = torch.cat([d for d in rk.dW], dim=1).cpu().numpy()
        res["kinds"][kind] = {"parity": parity(r, "bf16", float(rk.loss[0]), dX, dW)}
        ranks[kind] = rk
    for _ in range(warmup):
        for rk in ranks.values():
            rk.step(LAM)
    times = {k: [] for k in ranks}
    torch.cuda.synchronize()
    for _ in range(steps):
        for k, rk in ranks.items():
            t0 = time.perf_counter()
            rk.step(LAM)
            torch.cuda.synchronize()
            times[k].append((time.perf_counter() - t0) * 1e3)
    for k in ranks:
        res["kinds"][k]["step"] = stats(times[k])
        res["kinds"][k]["step"]["clock"] = "host clock around both ranks' step and a device synchronise"
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a B200"
    out = {"card": card(), "torch": torch.__version__, "lambda": LAM,
           "margins": {k: (None if v is None else vars(v)) for k, v in KINDS.items()},
           "workloads": {}}
    out["workloads"]["cfg3"] = single_gpu("cfg3", 512, 512, 85742, "bf16", args.steps, args.warmup)
    out["workloads"]["cfg1"] = single_gpu("cfg1", 256, 512, 10572, "fp32", args.steps, args.warmup)
    out["workloads"]["cfg3_g2"] = nvlink_g2(args.steps, args.warmup)
    out["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    for w, r in out["workloads"].items():
        print(w, {k: round(v["step"]["median_ms"], 4) for k, v in r["kinds"].items()})


if __name__ == "__main__":
    main()
