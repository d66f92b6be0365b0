"""Cost of the plain softmax classifier (LinearSoftmax) next to A-softmax, on one B200, in one process.

The linear kind runs the same four GEMMs as A-softmax; only the norm kernel's 1/c_j (set to 1),
the forward's target patch, the combine's target coefficients and the dW correction (zero) differ.
Workloads:
  cfg3      B = 512, C = 85,742, D = 512, bf16           (asm_forward_backward)
  cfg1      B = 256, C = 10,572, D = 512, fp32 on the tensor cores
each under A-softmax (m = 4, lambda = 5) and the linear kind, on the same inputs.  Every line is
first checked against the float64 oracles (loss, cosine and largest element error of dX / dW).
Then the two steps are timed alternately: CUDA events around a graph replay of the step.  A
per-phase (asm_set_profiling 2) breakdown of the eager step is averaged over separate runs.  The
card's name, power limit and SM clock are read in the same process.  Writes one JSON file.

    python scripts/bench_linear.py --out profiles/linear_b200.json [--steps 200] [--warmup 20]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "scripts")]
from bench_margins import card, parity, profile, stats  # noqa: E402
from oracle import asoftmax_ref as ref  # noqa: E402
from oracle import linear_softmax_ref as lr  # noqa: E402
from tf_face_toolbox_b200 import GraphedASoftmaxStep, LinearSoftmax, asoftmax_head  # noqa: E402
from tf_face_toolbox_b200.head import get_handle  # noqa: E402
from tf_face_toolbox_b200.synthetic import make_inputs  # noqa: E402

DEV = torch.device("cuda:0")
MARGINS = {"asoftmax": None, "linear": LinearSoftmax()}
LAM = 5.0


def oracle(inp, mg):
    X, W, y = inp.X.numpy(), inp.W.numpy(), inp.y.numpy()
    if mg is None:
        return ref.asoftmax_head(X, W, y, 4, LAM)
    return lr.linear_head_streamed(X, W, y)


def single_gpu(B, D, Cn, mode, steps, warmup):
    inp = make_inputs(B, D, Cn)
    X, y, W = inp.X.to(DEV), inp.y.to(DEV), inp.W.to(DEV)
    res = {"shape": dict(B=B, D=D, C=Cn, mode=mode), "lines": {}}
    fns = {}
    for name, mg in MARGINS.items():
        def step(mg=mg):
            return asoftmax_head(X, y, Cn, 4, LAM, weights=W, mode=mode, margin=mg)
        loss, _, dX, dW = step()
        torch.cuda.synchronize()
        res["lines"][name] = {"parity": parity(oracle(inp, mg), mode, float(loss), dX.cpu().numpy(),
                                               dW.cpu().numpy())}
        fns[name] = step
    graphs = {}
    for name, mg in MARGINS.items():
        g = GraphedASoftmaxStep(W, B, m=4, mode=mode, margin=mg)
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
    for name, mg in MARGINS.items():
        h = get_handle(DEV, D, Cn, Cn, 0, B, 4, mode, margin=mg)
        res["lines"][name]["per_phase_us"] = profile(h, fns[name], 2, 20)
    a, b = res["lines"]["asoftmax"]["step"], res["lines"]["linear"]["step"]
    res["linear_over_asoftmax_median"] = b["median_ms"] / a["median_ms"] - 1.0
    res["asoftmax_spread_p10_p90_ms"] = a["p90_ms"] - a["p10_ms"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a B200"
    out = {"card": card(), "torch": torch.__version__, "lambda": LAM, "margins": list(MARGINS), "workloads": {}}
    out["workloads"]["cfg3"] = single_gpu(512, 512, 85742, "bf16", args.steps, args.warmup)
    out["workloads"]["cfg1"] = single_gpu(256, 512, 10572, "fp32", args.steps, args.warmup)
    out["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    for w, r in out["workloads"].items():
        print(w, {k: round(v["step"]["median_ms"], 4) for k, v in r["lines"].items()},
              "linear/asoftmax - 1 =", round(r["linear_over_asoftmax_median"], 4))
        print(w, {k: v["per_phase_us"] for k, v in r["lines"].items()})


if __name__ == "__main__":
    main()
