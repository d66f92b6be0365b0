#!/usr/bin/env python
"""Benchmark of the A-softmax head hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload cfg3|cfg1|cfg2_head|cfg4|cfg5_head|cfg5] [--mode bf16|fp32]
                    [--dump-outputs DIR]

One "step" = one forward+backward pass of the head over one batch of synthetic input
(everything behind asm_forward_backward: norms, contractions, epilogues; excluding the
optimizer).  At N=1 the workload is BASELINE config 3 (C=85,742, D=512, batch 512, bf16), the
configuration the metric is quoted on.  For N>1 (launched by torchrun, one rank per GPU) the
same global batch is class-sharded over the ranks (strong scaling): the embeddings gather, the
statistics exchange and the dX reduce-scatter ride inside the head's own kernels over NVLink
peer memory (transport "nvlink") or go through three NCCL collectives (transport "nccl") -- no
collective on dW either way.

Every launch path is run ONCE on the bench inputs and compared with the float64 oracle before
anything is timed (`parity` in the JSON line); a failed gate exits non-zero without a number.

Prints ONE JSON line on rank 0 (see the keys in main()).  `--impl reference` times the CPU
stand-in for the reference's TensorFlow path (oracle/tf_graph_port.py; the TF code itself
cannot run, see DESIGN.md) on the host cores for the same metric and config.

`--dump-outputs DIR` writes, on rank 0, what the headline path returned from its last timed
step as DIR/<name>.npy (see step_arrays), so that two builds run with the same arguments (hence
the same seeded inputs) can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "A-softmax head fwd+bwd samples/sec at C=85,742 D=512, 1/2/4/8 B200"
UNIT = "samples/s"
M_MARGIN = 4
LAMBDA = 5.0      # lambda_min of the SphereFace schedule (SURVEY.md 8d: timing uses lambda=5)
LOSS_TOL = {"fp32": 1e-5, "bf16": 2e-3}      # BASELINE.json north_star
COS_MIN = 0.9999
ELEM_TOL = {"fp32": 5e-5, "bf16": 2e-2}      # max |dW - oracle| / max |oracle|, every element of the checked shard
DUMP_DW_BYTES = 32 << 20     # --dump-outputs: dW beyond this is cut to a seeded choice of class columns
DUMP_SEED = 0


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=float(d["hbm_gbs"]), tf_burst=float(d["bf16_tflops"]),
                    tf_sustained=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


# ----------------------------------------------------------------------------------------
# clocks: sample nvidia-smi while the GPU is under the benchmark load
# ----------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,utilization.gpu,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons, allsm = [], None, set(), []
        for ts, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                clk, mx = float(f[1]), float(f[2])
            except ValueError:
                continue
            smax = mx
            allsm.append(clk)
            if t0 - 0.05 <= ts <= t1 + 0.15:
                sm.append(clk)
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        use = sm if sm else allsm
        return {"sm_mhz": statistics.median(use) if use else None, "sm_max_mhz": smax,
                "reasons": sorted(reasons), "samples": len(use)}


# ----------------------------------------------------------------------------------------
# CPU stand-in for the reference (oracle/tf_graph_port.py): used ONLY as a timed baseline
# ----------------------------------------------------------------------------------------
def time_cpu_port(cfg, steps: int, warmup: int, budget_s: float):
    import torch
    from oracle import tf_graph_port as port
    from tf_face_toolbox_b200.synthetic import make_inputs
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    inp = make_inputs(cfg["B"], cfg["D"], cfg["C"])
    Bs = cfg["B"]
    t = time.perf_counter()
    port.step(inp.X, inp.W, inp.y, M_MARGIN, LAMBDA)
    est = time.perf_counter() - t
    # bound the run: shrink the per-step sample (rows of the batch) if K steps would not fit
    while Bs > 64 and est * (Bs / cfg["B"]) * (steps + warmup) > budget_s:
        Bs //= 2
    X, y = inp.X[:Bs].contiguous(), inp.y[:Bs].contiguous()
    for _ in range(warmup):
        port.step(X, inp.W, y, M_MARGIN, LAMBDA)
    times = []
    for _ in range(steps):
        t = time.perf_counter()
        last = port.step(X, inp.W, y, M_MARGIN, LAMBDA)
        times.append(time.perf_counter() - t)
    total = sum(times)
    sample = (f"full workload: {steps} steps of B={Bs} rows x C={cfg['C']} classes x D={cfg['D']}, fp32, torch-CPU"
              if Bs == cfg["B"] else
              f"{steps} steps over the first {Bs} of {cfg['B']} batch rows x all C={cfg['C']} classes, fp32, torch-CPU")
    return dict(value=Bs * steps / total, ms_per_step=1e3 * total / steps, cores=cores, sample=sample, B_sample=Bs,
                last=last)


def run_reference(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = time_cpu_port(cfg, args.steps, args.warmup, budget_s=150.0)
    if args.dump_outputs:
        write_arrays(args.dump_outputs, step_arrays(r["last"]))
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": workload_config(args, cfg, 1),
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "reference TensorFlow path cannot run (no TF, py2 code, missing module); timed the op-by-op torch-CPU port",
    }
    print(json.dumps(line), flush=True)


def workload_config(args, cfg, world):
    extra = " + center loss (loss.py:29-45)" if cfg.get("center") else ""
    return {"workload": f"{args.workload}: A-softmax head fwd+bwd{extra}, C={cfg['C']} D={cfg['D']} batch={cfg['B']} "
                        f"m={M_MARGIN} lambda={LAMBDA} {args.mode}",
            "global_batch": cfg["B"], "num_classes": cfg["C"], "embedding_dim": cfg["D"],
            "parallelism": f"class-sharded x{world}" if world > 1 else "single shard",
            "l2": "inputs larger than L2 (W fp32 %.1f MB + bf16 operand copies; no explicit flush)" % (cfg["C"] * cfg["D"] * 4 / 1e6)
                  if cfg["C"] * cfg["D"] * 4 > 126e6 else "L2 flushed between timed iterations (256 MB write)"}


def _cos(a, b):
    import numpy as np
    a = np.asarray(a, dtype=np.float64).ravel()
    b = np.asarray(b, dtype=np.float64).ravel()
    return float(a @ b / max(np.sqrt((a @ a) * (b @ b)), 1e-300))


def step_arrays(res):
    """What a caller of a launch path receives from one step, (loss, dX, dW) with loss a tensor
    or (cross-entropy, center loss), as float32 NumPy arrays: loss [1], center_loss [1], dX
    [B_local, D], dW [D, C_local].  A dW larger than DUMP_DW_BYTES keeps only a fixed, seeded
    choice of class columns (in increasing order), the same for every run of one workload."""
    import numpy as np
    import torch
    loss, dX, dW = res[0], res[1], res[2]
    out = {}
    if isinstance(loss, tuple):
        loss, out["center_loss"] = loss[0], loss[1].detach().float().reshape(1).cpu().numpy()
    out["loss"] = loss.detach().float().reshape(1).cpu().numpy()
    out["dX"] = dX.detach().float().cpu().numpy()
    if dW is not None:
        D, Cl = dW.shape
        keep = DUMP_DW_BYTES // (4 * D)
        if Cl > keep:
            cols = np.sort(np.random.default_rng(DUMP_SEED).choice(Cl, keep, replace=False))
            dW = dW.index_select(1, torch.from_numpy(cols).to(dW.device))
        out["dW"] = dW.detach().float().cpu().numpy()
    return out


def write_arrays(directory, arrays):
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


# ----------------------------------------------------------------------------------------
# one workload on this process group: parity gate, then the timed loops
# ----------------------------------------------------------------------------------------
class Workload:
    def __init__(self, args, cfg, mode, rank, world, dev, center=False):
        import torch
        import torch.distributed as dist
        from tf_face_toolbox_b200 import ShardedASoftmaxHead
        from tf_face_toolbox_b200.synthetic import make_inputs
        self.args, self.cfg, self.mode, self.rank, self.world, self.dev = args, cfg, mode, rank, world, dev
        self.torch, self.dist = torch, dist
        B, D, Cn = cfg["B"], cfg["D"], cfg["C"]
        self.B, self.D, self.Cn = B, D, Cn
        if B % world:
            raise SystemExit("global batch must divide by the number of ranks")
        self.b_local = B // world
        # Inputs: generated once, on rank 0 (identical bits to what the oracle sees), then the
        # embeddings / labels are broadcast and the class shards scattered on the device -- for
        # C = 1,000,000 every rank generating 2 GB of weights itself would dominate the run.
        self.inp = make_inputs(B, D, Cn) if rank == 0 else None
        if world == 1:
            self.Xfull, self.yfull = self.inp.X, self.inp.y
            self.Xd, self.yd, self.Wd = self.inp.X.to(dev), self.inp.y.to(dev), self.inp.W.to(dev)
            self.head = self.head_nv = None
            self.lo, self.hi = 0, Cn
        else:
            from tf_face_toolbox_b200.sharded import shard_bounds
            Xg = self.inp.X.to(dev) if rank == 0 else torch.empty(B, D, device=dev)
            yg = self.inp.y.to(dev) if rank == 0 else torch.empty(B, dtype=torch.int32, device=dev)
            dist.broadcast(Xg, 0)
            dist.broadcast(yg, 0)
            self.lo, self.hi = shard_bounds(Cn, world, rank)
            per = -(-Cn // world)
            mine = torch.zeros(D, per, device=dev)
            if rank == 0:
                Wg = self.inp.W.to(dev)
                parts = []
                for r in range(world):
                    a, b = shard_bounds(Cn, world, r)
                    t = torch.zeros(D, per, device=dev)
                    t[:, :b - a] = Wg[:, a:b]
                    parts.append(t)
                dist.scatter(mine, parts, src=0)
                del parts, Wg
            else:
                dist.scatter(mine, None, src=0)
            Wshard = mine[:, :self.hi - self.lo].contiguous()
            del mine
            self.Xfull, self.yfull = Xg.cpu(), yg.cpu()
            self.Xd = Xg[rank * self.b_local:(rank + 1) * self.b_local].contiguous()
            self.yd = yg[rank * self.b_local:(rank + 1) * self.b_local].contiguous()
            self.head = ShardedASoftmaxHead(D, Cn, m=M_MARGIN, mode=mode, device=dev, weights_shard=Wshard)
            self.head_nv = None
            if not args.no_nvlink:
                try:
                    self.head_nv = ShardedASoftmaxHead(D, Cn, m=M_MARGIN, mode=mode, device=dev, weights_shard=Wshard,
                                                       transport="nvlink", batch_global=B)
                    self.head_nv.step(self.Xd, self.yd, LAMBDA)
                    torch.cuda.synchronize()
                except Exception as e:      # pragma: no cover
                    print(f"bench: nvlink transport unavailable ({type(e).__name__}: {e})", file=sys.stderr)
                    self.head_nv = None
                okt = torch.tensor([1 if self.head_nv is not None else 0], device=dev)
                dist.all_reduce(okt, op=dist.ReduceOp.MIN)
                if int(okt.item()) == 0:
                    self.head_nv = None
            torch.cuda.empty_cache()
        # config 5: the center loss (loss.py:29-45) on the same gathered batch, class-sharded like W
        self.center = None
        if center:
            g = torch.Generator().manual_seed(4321)
            full = torch.randn(Cn, D, generator=g) * 0.1        # same bits on every rank
            cen = full[self.lo:self.hi].contiguous()
            self.center = dict(centers=cen.to(dev), init=cen, init_full=full, alpha=0.95, weight=0.008)
        self.need_flush = Cn * D * 4 <= 126e6
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if self.need_flush else None
        self.paths, self.host_paths = {}, {}
        self.outputs = {}
        self._build_paths()

    # ---- launch paths --------------------------------------------------------------------
    def _center_step(self, X, y, dX):
        """Center loss of this shard's classes on the batch rows this rank holds the gradient of."""
        from tf_face_toolbox_b200.center import center_loss
        c = self.center
        return center_loss(X, y, c["centers"], c["alpha"], c["weight"], class_offset=self.lo, grad_accum=dX)[0]

    def _build_paths(self):
        torch, dist = self.torch, self.dist
        from tf_face_toolbox_b200 import GraphedASoftmaxStep, asoftmax_head
        args, B, Cn, mode, world = self.args, self.B, self.Cn, self.mode, self.world
        if world == 1:
            def step():
                loss, _, dX, dW = asoftmax_head(self.Xd, self.yd, Cn, M_MARGIN, LAMBDA, weights=self.Wd, mode=mode)
                if self.center is not None:
                    loss = (loss, self._center_step(self.Xd, self.yd, dX))
                return loss, dX, dW
        else:
            def step():
                if self.center is not None:
                    return self.head.step(self.Xd, self.yd, LAMBDA, center=self.center)
                return self.head.step(self.Xd, self.yd, LAMBDA)
        self.paths["eager"] = step
        if self.center is not None:
            return                                   # config 5 is timed through the eager calls only

        def try_capture(make):
            g = None
            if not args.no_graph:
                try:
                    g = make()
                    g(self.Xd, self.yd)
                    torch.cuda.synchronize()
                except Exception as e:      # pragma: no cover
                    print(f"bench: CUDA-graph capture unavailable ({type(e).__name__}: {e})", file=sys.stderr)
                    g = None
            if world > 1:
                ok = torch.tensor([1 if g is not None else 0], device=self.dev)
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)
                if int(ok.item()) == 0:
                    g = None
            return g

        def make_graph_main():
            if world == 1:
                self.gstep = GraphedASoftmaxStep(self.Wd, batch_size=B, m=M_MARGIN, mode=mode)
                return lambda X, y: self.gstep(X, y, LAMBDA)
            self.head.capture(self.b_local)
            return lambda X, y: self.head.step_graphed(X, y, LAMBDA)

        def make_graph_nv():
            self.head_nv.capture(self.b_local)
            return lambda X, y: self.head_nv.step_graphed(X, y, LAMBDA)
        graphed = try_capture(make_graph_main)
        if graphed is not None:
            self.paths["graph"] = lambda: graphed(self.Xd, self.yd)
            self.host_paths["graph"] = graphed
        if world > 1 and self.head_nv is not None:
            self.paths["nvlink"] = lambda: self.head_nv.step(self.Xd, self.yd, LAMBDA)
            graphed_nv = try_capture(make_graph_nv)
            if graphed_nv is not None:
                self.paths["nvlink_graph"] = lambda: graphed_nv(self.Xd, self.yd)
                self.host_paths["nvlink_graph"] = graphed_nv

    # ---- parity gate -----------------------------------------------------------------------
    def parity(self):
        """Every launch path, run once on the bench inputs, against the float64 oracle: loss on
        every rank (identical bits across ranks), this rank's dX rows on every rank, dW on rank
        0's class shard.  BASELINE.md: parity gates must pass before any number is reported."""
        import numpy as np
        torch, dist = self.torch, self.dist
        from oracle import asoftmax_ref as ref
        rank, world, B, D, Cn = self.rank, self.world, self.B, self.D, self.Cn
        t0 = time.time()
        ref_loss = torch.zeros(1, dtype=torch.float64)
        ref_dX = torch.zeros(B, D, dtype=torch.float64)
        ref_dW = None
        ref_center = None
        if rank == 0:
            big = Cn >= 500000           # config 4: float32 matmuls inside the float64 streaming oracle
            r = ref.asoftmax_head_streamed(self.inp.X.numpy(), self.inp.W.numpy(), self.inp.y.numpy(), M_MARGIN, LAMBDA,
                                           chunk=16384, dw_ranges=[(self.lo, self.hi)],
                                           dtype=np.float32 if big else np.float64)
            ref_loss[0] = r.loss
            ref_dX = torch.from_numpy(r.dX)
            ref_dW = r.dW[(self.lo, self.hi)]
        if world > 1:
            rl, rx = ref_loss.to(self.dev), ref_dX.to(self.dev)
            dist.broadcast(rl, 0)
            dist.broadcast(rx, 0)
            ref_loss, ref_dX = rl.cpu(), rx.cpu()
        rows = slice(rank * self.b_local, (rank + 1) * self.b_local)
        want_dX = ref_dX[rows].numpy()
        if self.center is not None:
            # oracle of the center loss on the whole batch (loss.py:29-45): total loss, the gradient
            # it sends to every row, and the updated centers -- this rank checks its slice of each
            closs_ref, cen_new, cgrad = ref.center_loss(self.Xfull.numpy(), self.yfull.numpy(),
                                                        self.center["init_full"].numpy(),
                                                        alpha=self.center["alpha"], weight=self.center["weight"])
            ref_center = dict(loss=closs_ref, grad=cgrad, centers=cen_new[self.lo:self.hi])
        out = {}
        ok_all = True
        for name, fn in self.paths.items():
            if self.center is not None:
                self.center["centers"].copy_(self.center["init"])
            res = fn()
            torch.cuda.synchronize()
            loss, dX, dW = res[0], res[1], res[2]
            closs = None
            if isinstance(loss, tuple):
                loss, closs = loss
            loss = float(loss)
            rec = {"loss_rel": abs(loss - float(ref_loss[0])) / abs(float(ref_loss[0]))}
            dXn = dX.double().cpu().numpy()
            if ref_center is not None:
                # dX also carries the center-loss gradient of this rank's rows
                rec["center_loss_rel"] = abs(float(closs) - ref_center["loss"]) / max(ref_center["loss"], 1e-30)
                rec["center_update_max_abs"] = float(np.abs(self.center["centers"].double().cpu().numpy()
                                                            - ref_center["centers"]).max())
                rec["cos_dX"] = _cos(dXn, want_dX + ref_center["grad"][rows])
            else:
                rec["cos_dX"] = _cos(dXn, want_dX)
            if rank == 0 and dW is not None:
                dWn = dW.double().cpu().numpy()
                rec["cos_dW"] = _cos(dWn, ref_dW)
                # every element (a cosine over 44 M elements does not see one wrong column)
                rec["max_err_dW"] = float(np.abs(dWn - ref_dW).max() / np.abs(ref_dW).max())
            ok = rec["loss_rel"] <= LOSS_TOL[self.mode] and rec["cos_dX"] >= COS_MIN and rec.get("cos_dW", 1.0) >= COS_MIN
            ok = ok and rec.get("max_err_dW", 0.0) <= ELEM_TOL[self.mode]
            if ref_center is not None:
                ok = ok and rec["center_loss_rel"] <= 1e-4 and rec["center_update_max_abs"] <= 1e-5
            if world > 1:
                # same loss bits on every rank, and every rank's rows pass
                t = torch.tensor([loss, -loss, rec["cos_dX"], 1.0 if ok else 0.0], device=self.dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MIN)
                rec["loss_identical_across_ranks"] = bool(float(t[0]) == -float(t[1]))
                rec["cos_dX"] = float(t[2])                      # worst rank
                ok = bool(float(t[3]) == 1.0) and rec["loss_identical_across_ranks"]
            rec["ok"] = bool(ok)
            ok_all = ok_all and rec["ok"]
            out[name] = rec
        return {"ok": bool(ok_all), "tolerance": {"loss_rel": LOSS_TOL[self.mode], "cos_min": COS_MIN,
                                                  "max_err_dW_over_max_abs": ELEM_TOL[self.mode]},
                "oracle": "oracle/asoftmax_ref.py::asoftmax_head_streamed (float64 statistics, "
                          + ("float32" if Cn >= 500000 else "float64") + " matmuls)",
                "checked": "loss and dX rows on every rank (worst rank reported), dW on rank 0's class shard",
                "seconds": round(time.time() - t0, 2), "paths": out}

    # ---- timing ----------------------------------------------------------------------------
    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, fn, n, keep=None):
        """n calls of fn between CUDA events on the current stream; returns ms (max over ranks).
        With `keep`, what the last call returned goes to self.outputs[keep] (step_arrays)."""
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n - 1):
            if self.flush is not None:
                self.flush.zero_()
            fn()
        if self.flush is not None:
            self.flush.zero_()
        last = fn()
        e1.record()
        self.barrier()
        if keep is not None:
            self.outputs[keep] = step_arrays(last)
        ms = e0.elapsed_time(e1)
        if self.world > 1:
            t = torch.tensor([ms], device=self.dev)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def flush_cost(self):
        torch = self.torch
        if self.flush is None:
            return 0.0
        for _ in range(3):
            self.flush.zero_()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            self.flush.zero_()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 20

    def time_value(self, K, Wm, keep_outputs=False):
        """Device-resident timing of every launch path; the fastest is the headline.  With
        keep_outputs, self.outputs[path] holds what each path returned from its last timed step."""
        self.flush_ms = self.flush_cost()
        value_ms = {}
        for name, fn in self.paths.items():
            for _ in range(max(Wm, 3)):
                fn()
            value_ms[name] = self.timed(fn, K, keep=name if keep_outputs else None) / K - self.flush_ms
        best = min(value_ms, key=value_ms.get)
        return best, value_ms

    def close(self):
        for hd in (self.head, self.head_nv):
            for attr in ("_graph", "_gout"):
                if hd is not None and hasattr(hd, attr):
                    setattr(hd, attr, None)
        if getattr(self, "gstep", None) is not None:
            self.gstep.close()
        self.paths.clear()
        self.host_paths.clear()
        self.head = self.head_nv = None
        from tf_face_toolbox_b200.head import release_handles
        release_handles()
        self.Xd = self.yd = self.Wd = self.flush = None
        self.torch.cuda.empty_cache()


# ----------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------
def run_ours(args, cfg):
    import torch
    import torch.distributed as dist
    from tf_face_toolbox_b200 import _lib
    from tf_face_toolbox_b200.head import get_handle
    from tf_face_toolbox_b200.synthetic import CONFIGS

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the A-softmax head has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # a stuck collective must not hang the caller: dump every thread's stack and exit
    import faulthandler
    faulthandler.dump_traceback_later(float(os.environ.get("BENCH_WATCHDOG_S", "900")), exit=True)
    if world > 1:
        # communicator lines (ranks, transports) go to stderr so that the driver can check them
        os.environ.setdefault("NCCL_DEBUG", os.environ.get("BENCH_NCCL_DEBUG", "INFO"))
        os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)
    mode = args.mode
    K, Wm = args.steps, args.warmup
    peaks = load_peaks()
    t_start = time.time()
    # anything that changes what the library does is part of the record
    knobs = {k: v for k, v in sorted(os.environ.items()) if k.startswith("ASM_")}
    bringup = "ASM_B200_LIB" in knobs or "ASM_UMMA_DEBUG" in knobs

    def note(msg):
        if rank == 0 and os.environ.get("BENCH_VERBOSE"):
            print(f"[bench {time.time() - t_start:6.1f}s] {msg}", file=sys.stderr, flush=True)

    def fail_parity(par, what):
        if rank == 0:
            print(json.dumps({"metric": METRIC, "value": None, "unit": UNIT, "n_gpus": world, "parity": par,
                              "error": f"parity gate failed for {what}: no number is reported"}), flush=True)
        sys.stdout.flush()
        os._exit(3)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()

    wl = Workload(args, cfg, mode, rank, world, dev, center=bool(cfg.get("center")))
    B, D, Cn, b_local = wl.B, wl.D, wl.Cn, wl.b_local
    note("setup done, paths=%s" % list(wl.paths))
    parity = wl.parity()
    note("parity gate: %s (%.1fs)" % (parity["ok"], parity["seconds"]))
    if not parity["ok"]:
        fail_parity(parity, args.workload)

    # ---- (1) device-resident timing: the headline `value`
    t_load0 = time.time()
    value_path, value_ms = wl.time_value(K, Wm, keep_outputs=bool(args.dump_outputs) and rank == 0)
    if wl.outputs:
        write_arrays(args.dump_outputs, wl.outputs[value_path])
        wl.outputs.clear()
    run_step = wl.paths[value_path]
    ms_step = value_ms[value_path]
    flush_ms = wl.flush_ms
    value = B / (ms_step * 1e-3)

    # distribution of the chosen path (SURVEY 8d asks for median and p10/p90): events between
    # GROUPS of 5 steps (a timing event after every step costs ~20 us of stream serialisation,
    # which would measure the events), K steps in all; the headline stays the K-step mean above
    grp = 5 if K >= 10 else 1
    sizes = [grp] * (K // grp) + ([K % grp] if K % grp else [])
    ngrp = len(sizes)
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(ngrp + 1)]
    wl.barrier()
    for gi, size in enumerate(sizes):
        evs[gi].record()
        for _ in range(size):
            if wl.flush is not None:
                wl.flush.zero_()
            run_step()
    evs[ngrp].record()
    wl.barrier()
    per = sorted(evs[i].elapsed_time(evs[i + 1]) / sizes[i] - flush_ms for i in range(ngrp))
    step_dist = {"p10": per[int(0.1 * (ngrp - 1))], "p50": per[(ngrp - 1) // 2],
                 "p90": per[int(round(0.9 * (ngrp - 1)))], "group": grp, "groups": ngrp,
                 "note": "rank-0 CUDA-event time per step over groups of `group` steps, same loop as value"}
    note("value loop done: %.4f ms/step (%s)" % (ms_step, value_path))

    # ---- (2) per-kernel durations (CUDA events on the launching stream, inside the library)
    # of the transport the headline uses: the NVLink-transport handle when it won, else the plain one
    kernels = {}
    if world == 1:
        h = get_handle(dev, D, Cn, Cn, 0, B, M_MARGIN, mode)
        prof_step = wl.paths["eager"]
    elif value_path.startswith("nvlink") and wl.head_nv is not None:
        h = wl.head_nv._p2p["handle"]
        prof_step = wl.paths["nvlink"]
    else:
        h = wl.head.compute._handle(B)
        prof_step = wl.paths["eager"]
    prof_step()
    launches_per_step = int(h.lib.asm_last_launch_count(h.ptr))
    if wl.center is not None:
        launches_per_step += 2                      # center_loss_kernel + center_update_kernel
    h.lib.asm_set_profiling(h.ptr, 1)
    ms_buf = (C.c_float * 16)()
    names = C.create_string_buffer(16 * 32)
    for _ in range(K):
        if wl.flush is not None:
            wl.flush.zero_()
        prof_step()
        n = h.lib.asm_get_profile(h.ptr, 16, ms_buf, names)
        for i in range(max(n, 0)):
            nm = names.raw[i * 32:(i + 1) * 32].split(b"\0")[0].decode()
            kernels.setdefault(nm, []).append(ms_buf[i])
    h.lib.asm_set_profiling(h.ptr, 0)
    kavg = {k: sum(v) / len(v) for k, v in kernels.items()}
    # the same with events only between PHASES, which leaves the real schedule in place (the dW
    # kernel next to the dX branch on disjoint CTA pairs counts as one phase)
    phases = {}
    h.lib.asm_set_profiling(h.ptr, 2)
    for _ in range(K):
        if wl.flush is not None:
            wl.flush.zero_()
        prof_step()
        n = h.lib.asm_get_profile(h.ptr, 16, ms_buf, names)
        for i in range(max(n, 0)):
            nm = names.raw[i * 32:(i + 1) * 32].split(b"\0")[0].decode()
            phases.setdefault(nm, []).append(ms_buf[i])
    h.lib.asm_set_profiling(h.ptr, 0)
    pavg = {k: sum(v) / len(v) for k, v in phases.items()}
    note("profile loops done")

    # ---- (3) end to end with HOST buffers: H2D of the step's inputs and D2H of its results (the
    # loss AND dX, the gradient the backbone consumes) inside the timed region, every step
    Xh = wl.Xfull[rank * b_local:(rank + 1) * b_local].contiguous().pin_memory()
    yh = wl.yfull[rank * b_local:(rank + 1) * b_local].contiguous().pin_memory()
    loss_h = torch.empty(1, dtype=torch.float32).pin_memory()
    dX_h = torch.empty(b_local, D, dtype=torch.float32).pin_memory()

    def first_loss(out):
        l0 = out[0][0] if isinstance(out[0], tuple) else out[0]
        return l0.reshape(1)

    def make_e2e(name):
        if name in wl.host_paths:                # graph steps copy their (host) inputs themselves
            g = wl.host_paths[name]

            def fn():
                out = g(Xh, yh)
                dX_h.copy_(out[1], non_blocking=True)
                loss_h.copy_(first_loss(out), non_blocking=False)     # D2H read of the results (syncs)
                return out
        else:
            dev_step = wl.paths[name]

            def fn():
                wl.Xd.copy_(Xh, non_blocking=True)
                wl.yd.copy_(yh, non_blocking=True)
                out = dev_step()
                dX_h.copy_(out[1], non_blocking=True)
                loss_h.copy_(first_loss(out), non_blocking=False)
                return out
        return fn
    e2e_ms = {}
    for name in wl.paths:
        fn = make_e2e(name)
        for _ in range(3):
            fn()
        e2e_ms[name] = wl.timed(fn, K) / K - flush_ms
    # the same through the package's host input pipeline (HostPipelinedStep): every step still
    # copies its inputs H2D and has its loss and dX read D2H, but the copies overlap the
    # neighbouring steps' kernels and the results are read one step late
    from tf_face_toolbox_b200.pipeline import HostPipelinedStep
    from tf_face_toolbox_b200 import asoftmax_head
    for name in list(wl.paths):
        if name in wl.host_paths or wl.center is not None:
            continue                          # graph steps own their static input buffers
        src = wl.head_nv if name == "nvlink" else (wl.head if world > 1 else None)
        # results read back on the compute stream (between two steps) or on a stream of their own
        for suffix, own_stream in (("_pipelined", False), ("_pipelined_d2h_stream", True)):
            if src is not None:
                runner = HostPipelinedStep(lambda X, y, _h=src: _h.step(X, y, LAMBDA), b_local, D, dev,
                                           read_dx=True, loss_stream=own_stream)
            else:
                runner = HostPipelinedStep(lambda X, y: (lambda o: (o[0], o[2], o[3]))(
                    asoftmax_head(X, y, Cn, M_MARGIN, LAMBDA, weights=wl.Wd, mode=mode)), b_local, D, dev,
                    read_dx=True, loss_stream=own_stream)

            def fn(_r=runner):
                return _r.submit(Xh, yh)
            for _ in range(3):
                fn()
            runner.flush()
            e2e_ms[name + suffix] = wl.timed(lambda: (fn()), K) / K - flush_ms
            runner.flush()
    # ... and through the reference-shaped drop-in surface: forward / loss_function / gradients of
    # the Network-shaped wrapper (nets/net_base.py:84-107, data_parallel.py:220-236)
    if world == 1 and wl.center is None:
        from tf_face_toolbox_b200 import ASoftmaxHead, LambdaState
        net = ASoftmaxHead(D, Cn, m=M_MARGIN, mode=mode, device=dev, lambda_state=LambdaState(explicit=LAMBDA))
        net.weights = wl.Wd

        def fn_net():
            wl.Xd.copy_(Xh, non_blocking=True)
            wl.yd.copy_(yh, non_blocking=True)
            out = net.forward(wl.Xd, wl.yd, num_classes=Cn, is_training=True)
            losses, _names, _others = net.loss_function("TOWER_0", wl.yd, **out)
            dXn, _dWn = net.gradients()
            dX_h.copy_(dXn, non_blocking=True)
            loss_h.copy_((losses[0] + losses[1]).reshape(1), non_blocking=False)
        for _ in range(3):
            fn_net()
        e2e_ms["network_api"] = wl.timed(fn_net, K) / K - flush_ms
    note("e2e loops done")
    e2e_path = min(e2e_ms, key=e2e_ms.get)
    ms_e2e = e2e_ms[e2e_path]
    e2e_value = B / (ms_e2e * 1e-3)

    # keep the GPU under the same load long enough for nvidia-smi to sample clocks; the
    # number of extra (untimed) steps is derived from the all-reduced step time so that every
    # rank issues the same collectives
    n_extra = min(20000, int(1200.0 / max(ms_step, 1e-3)))
    done = 0
    while done < n_extra:
        for _ in range(min(50, n_extra - done)):
            run_step()
        done += 50
        torch.cuda.synchronize()
    t_load1 = time.time()
    clocks = sampler.stop(t_load0, t_load1) if rank == 0 else None
    if world > 1:
        dist.barrier()
    note("main workload done")

    line = None
    if rank == 0:
        line = build_line(args, cfg, world, mode, peaks, kavg, pavg, value, ms_step, value_path, value_ms, step_dist,
                          e2e_value, ms_e2e, e2e_path, e2e_ms, b_local, launches_per_step, K, Wm, clocks, parity,
                          knobs, bringup, _lib.load().asm_version().decode(), "graph" in wl.paths or "nvlink_graph" in wl.paths)
    wl.close()
    del wl

    # ---- (4) config 4 in the same process (C = 1,000,000, batch 1024): the configuration the
    # north star's ">= 6x at 8 GPUs" is stated on, same version, same box, parity-gated
    if args.workload == "cfg3" and not args.no_cfg4:
        cfg4 = dict(CONFIGS["cfg4"])
        note("config 4 ...")
        w4 = Workload(args, cfg4, cfg4["mode"], rank, world, dev)
        par4 = w4.parity()
        note("config 4 parity: %s (%.1fs)" % (par4["ok"], par4["seconds"]))
        if not par4["ok"]:
            fail_parity(par4, "cfg4")
        p4, ms4 = w4.time_value(K, 3)
        if rank == 0:
            line["cfg4"] = {"workload": "cfg4: A-softmax head fwd+bwd, C=1000000 D=512 batch=1024 m=4 lambda=5.0 bf16",
                            "value": cfg4["B"] / (ms4[p4] * 1e-3), "unit": UNIT, "ms_per_step": ms4[p4], "steps": K,
                            "value_path": p4, "ms_per_step_by_path": ms4, "n_gpus": world, "scaling": "strong",
                            "parity": par4,
                            "step_algorithmic_tflops": 6.0 * cfg4["B"] * cfg4["D"] * cfg4["C"] / (ms4[p4] * 1e-3) / 1e12}
        w4.close()
        del w4

    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            r = time_cpu_port(cfg, 8, 1, budget_s=25.0)
            line["cpu_baseline"] = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                                    "sample": r["sample"]}
        print(json.dumps(line), flush=True)
    # teardown must never turn a finished measurement into a hang
    sys.stdout.flush()
    faulthandler.cancel_dump_traceback_later()
    if world > 1:
        bail = threading.Timer(20.0, lambda: os._exit(0))
        bail.daemon = True
        bail.start()
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()
        bail.cancel()


def build_line(args, cfg, world, mode, peaks, kavg, pavg, value, ms_step, value_path, value_ms, step_dist, e2e_value,
               ms_e2e, e2e_path, e2e_ms, b_local, launches_per_step, K, Wm, clocks, parity, knobs, bringup, version,
               has_graph):
    B, D, Cn = cfg["B"], cfg["D"], cfg["C"]
    C_local = Cn if world == 1 else -(-Cn // world)
    Cp_l = (C_local + 255) // 256 * 256
    gemm_flops = 2.0 * B * D * C_local
    roof_kernels = []
    for nm, ms in kavg.items():
        t = ms * 1e-3
        if nm == "dw_gemm":
            # SURVEY 8(d) algorithmic work of the dW contraction: 2 B D C flop and ONE fp32 write of
            # dW (4 D C bytes).  What the kernel's plan additionally reads (G'' and the bf16 weights
            # for the normalisation-Jacobian term) is reported separately, not credited.
            alg = 4.0 * D * C_local
            plan = alg + (2.0 * B * Cp_l + 2.0 * D * Cp_l if mode == "bf16" else 0.0)
            roof_kernels.append({"kernel": nm, "ms": ms, "bound": "hbm", "achieved": alg / t / 1e9, "unit": "GB/s",
                                 "frac": alg / t / 1e9 / peaks["hbm"], "algorithmic_bytes": alg,
                                 "plan_bytes": plan, "plan_gbs": plan / t / 1e9,
                                 "tensor_tflops": gemm_flops / t / 1e12,
                                 "tensor_frac": gemm_flops / t / 1e12 / peaks["tf_burst"]})
        elif nm in ("fwd_logits_stats", "bwd_recompute_g", "dx_gemm"):
            ach = gemm_flops / t / 1e12
            roof_kernels.append({"kernel": nm, "ms": ms, "bound": "tensor", "achieved": ach, "unit": "TFLOP/s",
                                 "frac": ach / peaks["tf_burst"]})
        elif nm == "prep_norms":
            by = 4.0 * D * C_local + (2.0 * D * Cp_l if mode == "bf16" else 0) + 4.0 * B * D
            ach = by / t / 1e9
            roof_kernels.append({"kernel": nm, "ms": ms, "bound": "hbm", "achieved": ach, "unit": "GB/s",
                                 "frac": ach / peaks["hbm"], "algorithmic_bytes": by})
        else:
            roof_kernels.append({"kernel": nm, "ms": ms})
    # phases as they really run (events only where the main stream serialises anyway)
    phase_list = []
    for nm, ms in pavg.items():
        rec = {"phase": nm, "ms": ms}
        if nm.startswith("dw+dx"):
            # two contractions (4 B D C flop) and the one fp32 write of dW (4 D C bytes), side by side
            rec.update({"algorithmic_flops": 2 * gemm_flops, "tensor_tflops": 2 * gemm_flops / (ms * 1e-3) / 1e12,
                        "tensor_frac": 2 * gemm_flops / (ms * 1e-3) / 1e12 / peaks["tf_burst"],
                        "algorithmic_bytes": 4.0 * D * C_local, "hbm_gbs": 4.0 * D * C_local / (ms * 1e-3) / 1e9,
                        "hbm_frac": 4.0 * D * C_local / (ms * 1e-3) / 1e9 / peaks["hbm"]})
        phase_list.append(rec)
    dom = max((k for k in roof_kernels if "bound" in k), key=lambda k: k["ms"], default=None)
    # DRAM traffic per launch comes from an ncu capture (profiles/), never from this run; it is only
    # quoted when that capture was taken from the same library version and workload
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic_cfg3.json")
    traffic_note = None
    if world == 1 and args.workload == "cfg3" and mode == "bf16" and os.path.exists(tpath):
        tj = json.load(open(tpath))
        if tj.get("library_version") == version:
            traffic = tj.get("kernels", {})
        else:
            traffic_note = f"profiles/traffic_cfg3.json is for '{tj.get('library_version')}', this library is '{version}'"
    roofline = None
    if dom is not None:
        roofline = {"kernel": dom["kernel"], "bound": dom["bound"], "achieved": dom["achieved"],
                    "peak": peaks["tf_burst"] if dom["bound"] == "tensor" else peaks["hbm"],
                    "unit": dom["unit"], "frac": dom["frac"],
                    "traffic": (traffic or {}).get(dom["kernel"]),
                    "traffic_source": "profiles/traffic_cfg3.json (ncu, same library version)" if traffic else traffic_note,
                    "peak_source": peaks["src"] + (" burst bf16" if dom["bound"] == "tensor" else " copy"),
                    "ms": dom["ms"]}
        for k in ("algorithmic_bytes", "plan_bytes", "plan_gbs", "tensor_frac"):
            if k in dom:
                roofline[k] = dom[k]
    step_flops = 6.0 * B * D * Cn
    transport = ("nvlink-p2p (the head's own kernels over peer memory, no collective launch)"
                 if value_path.startswith("nvlink") else ("nccl (3 collectives per step)" if world > 1 else "none"))
    return {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": max(Wm, 3),
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": mode, "data": "synthetic", "config": workload_config(args, cfg, world),
        "parity": parity, "transport": transport,
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e, "path": e2e_path,
                "ms_per_step_by_path": e2e_ms,
                "h2d_bytes_per_step": int(b_local * D * 4 + b_local * 4),
                "d2h_bytes_per_step": int(b_local * D * 4 + 4)},
        "gpu_launches": launches_per_step * K, "launches_per_step": launches_per_step,
        "cuda_graph": has_graph, "value_path": value_path, "ms_per_step_by_path": value_ms,
        "ms_per_step_dist": step_dist,
        "roofline": roofline,
        "step_tensor_frac": step_flops / (ms_step * 1e-3) / 1e12 / peaks["tf_burst"],
        "step_algorithmic_tflops": step_flops / (ms_step * 1e-3) / 1e12,
        "kernels": roof_kernels,
        "kernels_note": "per-kernel CUDA-event times with every kernel on ONE stream, one after the other "
                        "(no programmatic launch overlap, dW and dX each on the whole chip)",
        "phases": phase_list,
        "phases_note": "events only between phases: the real schedule, dW next to the dX branch on disjoint CTA pairs",
        "library": version, "env": knobs, "bringup_build": bringup,
    }


def main():
    from tf_face_toolbox_b200.synthetic import CONFIGS
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(CONFIGS))
    ap.add_argument("--mode", default=None, choices=["bf16", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time the eager per-kernel launches")
    ap.add_argument("--graph", action="store_true", help="(default) also time the CUDA-graph replay of the step")
    ap.add_argument("--no-nvlink", action="store_true", help="N>1: skip the NVLink peer-memory transport")
    ap.add_argument("--no-cfg4", action="store_true", help="skip the config-4 (C = 1M) sub-record of the cfg3 line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss, dX and dW (at most %d MB of dW class columns, a seeded choice) of the "
                         "headline path's last timed step as DIR/<name>.npy, float32" % (DUMP_DW_BYTES >> 20))
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    cfg = dict(CONFIGS[args.workload])
    if args.mode is None:
        args.mode = cfg["mode"]
    if args.impl == "reference":
        run_reference(args, cfg)
    else:
        run_ours(args, cfg)


if __name__ == "__main__":
    main()
