"""Cost of the focal loss next to the softmax cross-entropy, on one B200, in one process.

The focal loss changes only the per-row epilogue of the combine kernel (one scalar w_i per row
folded into the backward's exp2 offset and target coefficients); every GEMM is the same kernel.
Workloads:
  cfg3      B = 512, C = 85,742, D = 512, bf16           (asm_forward_backward)
  cfg1      B = 256, C = 10,572, D = 512, fp32           (asm_forward_backward)
each under A-softmax (m = 4, lambda = 5) and ArcFace (s = 64, m = 0.5), with the cross-entropy
and with FocalLoss(gamma = 1, alpha = 2).  Every line is first checked against the float64
oracles (loss, cosine and largest element error of dX / dW).  Then the four steps are timed
alternately: CUDA events around a graph replay of the step.  A per-phase (asm_set_profiling 2)
breakdown of the eager step is averaged over separate runs.  The card's name, power limit and SM
clock are read in the same process.  Writes one JSON file.

    python scripts/bench_focal.py --out profiles/focal_b200.json [--steps 200] [--warmup 20]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "scripts")]
from bench_margins import card, parity, profile, stats  # noqa: E402
from oracle import additive_margin_ref as am  # noqa: E402
from oracle import asoftmax_ref as ref  # noqa: E402
from oracle import focal_ref as fr  # noqa: E402
from tf_face_toolbox_b200 import AdditiveMargin, FocalLoss, GraphedASoftmaxStep, asoftmax_head  # noqa: E402
from tf_face_toolbox_b200.head import get_handle  # noqa: E402
from tf_face_toolbox_b200.synthetic import make_inputs  # noqa: E402

DEV = torch.device("cuda:0")
MARGINS = {"asoftmax": None, "arcface": AdditiveMargin.arcface(64.0, 0.5)}
LOSSES = {"ce": None, "focal": FocalLoss(1.0, 2.0)}
LAM = 5.0


def oracle(inp, mg, fl):
    X, W, y = inp.X.numpy(), inp.W.numpy(), inp.y.numpy()
    if fl is None:
        return ref.asoftmax_head(X, W, y, 4, LAM) if mg is None else am.additive_head(X, W, y, mg.s, mg.m2, mg.m3)
    # the class-sharded focal oracle with one shard holding every class: vectorised, so it is
    # affordable at C = 85,742 (tests/test_oracle_focal_cpu.py checks it against the one-piece form)
    mt = None if mg is None else (mg.s, mg.m2, mg.m3)
    st = fr.sharded_partial_stats(X, W, y, 0, 4, LAM, mt)[:3]
    M, logZ, w, loss = fr.sharded_combine([st], fl.gamma, fl.alpha)
    dX, dW = fr.sharded_backward(X, W, y, 0, M, logZ, w, 4, LAM, mt)
    return fr.FocalResult(loss, None, dX, dW, None, None, w)


def single_gpu(B, D, Cn, mode, steps, warmup):
    inp = make_inputs(B, D, Cn)
    X, y, W = inp.X.to(DEV), inp.y.to(DEV), inp.W.to(DEV)
    res = {"shape": dict(B=B, D=D, C=Cn, mode=mode), "lines": {}}
    lines = {f"{mk}-{lk}": (mg, fl) for mk, mg in MARGINS.items() for lk, fl in LOSSES.items()}
    fns = {}
    for name, (mg, fl) in lines.items():
        def step(mg=mg, fl=fl):
            return asoftmax_head(X, y, Cn, 4, LAM, weights=W, mode=mode, margin=mg, loss=fl)
        loss, _, dX, dW = step()
        torch.cuda.synchronize()
        res["lines"][name] = {"parity": parity(oracle(inp, mg, fl), mode, float(loss), dX.cpu().numpy(),
                                               dW.cpu().numpy())}
        fns[name] = step
    graphs = {}
    for name, (mg, fl) in lines.items():
        g = GraphedASoftmaxStep(W, B, m=4, mode=mode, margin=mg, loss=fl)
        g(X, y, LAM)
        graphs[name] = g
    for _ in range(warmup):
        for g in graphs.values():
            g.graph.replay()
    ev = {k: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
          for k in graphs}
    for i in range(steps):                                  # alternate the lines step by step
        for k, g in graphs.items():
            ev[k][i][0].record()
            g.graph.replay()
            ev[k][i][1].record()
    torch.cuda.synchronize()
    for k, g in graphs.items():
        res["lines"][k]["step"] = stats([a.elapsed_time(b) for a, b in ev[k]])
        res["lines"][k]["step"]["clock"] = "CUDA events around one graph replay of the step"
        g.close()
    for name, (mg, fl) in lines.items():
        h = get_handle(DEV, D, Cn, Cn, 0, B, 4, mode, margin=mg, loss=fl)
        res["lines"][name]["per_phase_us"] = profile(h, fns[name], 2, 20)
    for mk in MARGINS:
        ce, fo = res["lines"][f"{mk}-ce"]["step"], res["lines"][f"{mk}-focal"]["step"]
        res[f"{mk}_focal_over_ce_median"] = fo["median_ms"] / ce["median_ms"] - 1.0
        res[f"{mk}_ce_spread_p10_p90_ms"] = ce["p90_ms"] - ce["p10_ms"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a B200"
    out = {"card": card(), "torch": torch.__version__, "lambda": LAM,
           "margins": {k: (None if v is None else vars(v)) for k, v in MARGINS.items()},
           "losses": {k: (None if v is None else vars(v)) for k, v in LOSSES.items()},
           "workloads": {}}
    out["workloads"]["cfg3"] = single_gpu(512, 512, 85742, "bf16", args.steps, args.warmup)
    out["workloads"]["cfg1"] = single_gpu(256, 512, 10572, "fp32", args.steps, args.warmup)
    out["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    for w, r in out["workloads"].items():
        print(w, {k: round(v["step"]["median_ms"], 4) for k, v in r["lines"].items()})
        print(w, {k: {p: us for p, us in v["per_phase_us"].items()} for k, v in r["lines"].items()})


if __name__ == "__main__":
    main()
