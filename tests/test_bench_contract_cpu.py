"""The driver-facing bench.py contract, as far as it can be checked without a GPU: the
reference arm (`--impl reference`, the CPU restatement of the reference's graph timed on the
host cores) prints one JSON line with the agreed keys, and the product arm refuses to run
without a CUDA device instead of falling back to the CPU."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT,
                          capture_output=True, text=True, timeout=600)


def test_reference_arm_json_line():
    p = run("--impl", "reference", "--workload", "cfg1", "--steps", "2", "--warmup", "1")
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference"
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["unit"] == "samples/s" and line["higher_is_better"] is True
    assert line["steps"] == 2 and line["warmup"] == 1 and line["n_gpus"] == 1
    assert line["value"] > 0 and line["ms_per_step"] > 0
    assert line["value"] == line["config"]["global_batch"] / (line["ms_per_step"] * 1e-3) or \
        abs(line["value"] - line["config"]["global_batch"] / (line["ms_per_step"] * 1e-3)) < 1e-6 * line["value"]
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    e2e = line["e2e"]
    assert e2e["value"] == line["value"] and e2e["unit"] == line["unit"]
    assert e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"] and "model" not in line["config"]


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    argv, sys.argv = sys.argv, ["bench.py"]
    try:
        spec.loader.exec_module(b)
    finally:
        sys.argv = argv
    return b


def test_reference_arm_dumps_its_last_step(tmp_path):
    """--dump-outputs: the loss, dX and dW the timed path returned from its last step, float32,
    on the seeded bench inputs (config 1 is small enough for the whole dW)."""
    import numpy as np
    from oracle import asoftmax_ref as ref
    from tf_face_toolbox_b200.synthetic import CONFIGS, make_inputs
    out = tmp_path / "dump"
    p = run("--impl", "reference", "--workload", "cfg1", "--steps", "2", "--warmup", "0", "--dump-outputs", str(out))
    assert p.returncode == 0, p.stderr[-2000:]
    got = {f.stem: np.load(f) for f in out.iterdir()}
    assert sorted(got) == ["dW", "dX", "loss"] and all(a.dtype == np.float32 for a in got.values())
    assert sum(f.stat().st_size for f in out.iterdir()) <= 64 << 20
    c = CONFIGS["cfg1"]
    inp = make_inputs(c["B"], c["D"], c["C"])
    rows = got["dX"].shape[0]                     # the reference arm may time the first rows of the batch only
    assert got["dW"].shape == (c["D"], c["C"]) and got["dX"].shape == (rows, c["D"]) and 64 <= rows <= c["B"]
    r = ref.asoftmax_head(inp.X[:rows].numpy(), inp.W.numpy(), inp.y[:rows].numpy(), 4, 5.0)
    assert abs(float(got["loss"][0]) - r.loss) <= 1e-5 * r.loss
    np.testing.assert_allclose(got["dX"], r.dX, rtol=0, atol=1e-5 * np.abs(r.dX).max())
    np.testing.assert_allclose(got["dW"], r.dW, rtol=0, atol=1e-5 * np.abs(r.dW).max())


def test_dumped_dw_is_a_fixed_choice_of_class_columns():
    import numpy as np
    import torch
    b = _bench_module()
    D, Cn = 512, 20000
    dW = torch.randn(D, Cn, generator=torch.Generator().manual_seed(0))
    res = ((torch.tensor(1.5), torch.tensor(0.25)), torch.ones(8, D), dW)
    a, a2 = b.step_arrays(res), b.step_arrays(res)
    assert sorted(a) == ["center_loss", "dW", "dX", "loss"]
    assert a["loss"].tolist() == [1.5] and a["center_loss"].tolist() == [0.25]
    keep = b.DUMP_DW_BYTES // (4 * D)
    assert a["dW"].shape == (D, keep) and a["dW"].nbytes <= b.DUMP_DW_BYTES
    np.testing.assert_array_equal(a["dW"], a2["dW"])
    # the columns are whole dW columns, in increasing class order
    cols = [int(np.nonzero((dW.numpy() == a["dW"][:, [j]]).all(axis=0))[0][0]) for j in range(0, keep, 997)]
    assert cols == sorted(cols) and len(set(cols)) == len(cols)


def test_steps_must_be_positive():
    p = run("--impl", "reference", "--workload", "cfg1", "--steps", "0")
    assert p.returncode != 0 and "--steps" in p.stderr


def test_product_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present: the product arm would run")
    p = run("--steps", "2", "--warmup", "1")
    out = p.stdout.strip().splitlines()
    line = json.loads(out[-1]) if out and out[-1].startswith("{") else None
    # no measurement may come out of a box without a CUDA device
    assert line is None or line.get("gpu_launches", 0) == 0 and not line.get("value")
    assert "no CUDA device" in (p.stderr + p.stdout)


def test_committed_evidence_is_self_consistent():
    """profiles/: the N = 1 bench line of the final run carries the agreed extra objects, its parity
    record bounds every element of dW, and the DRAM-traffic file bench.py quotes was captured from
    the same library version (bench.py refuses it otherwise)."""
    prof = os.path.join(ROOT, "profiles")
    line = json.loads(open(os.path.join(prof, "r2_bench_n1.json")).read().strip().splitlines()[-1])
    for key in ("roofline", "cpu_baseline", "e2e", "clocks", "gpu_launches", "parity", "kernels", "phases", "cfg4",
                "library", "env"):
        assert key in line, key
    assert line["parity"]["ok"] and line["cfg4"]["parity"]["ok"]
    for rec in line["parity"]["paths"].values():
        assert rec["max_err_dW"] <= line["parity"]["tolerance"]["max_err_dW_over_max_abs"]
    roof = line["roofline"]
    assert roof["bound"] in ("hbm", "tensor") and 0 < roof["frac"] <= 1 and roof["peak"] > 0
    assert abs(roof["frac"] - roof["achieved"] / roof["peak"]) < 1e-9
    assert line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["d2h_bytes_per_step"] > 0
    assert line["gpu_launches"] == line["steps"] * line["launches_per_step"]
    traffic = json.load(open(os.path.join(prof, "traffic_cfg3.json")))
    assert traffic["library_version"] == line["library"]
    assert abs(sum(traffic["kernels"].values()) - traffic["step_total"]) <= len(traffic["kernels"])
    # the multi-GPU lines passed their parity gate on every launch path, with identical loss bits
    for n in (2, 4, 8):
        ln = json.loads(open(os.path.join(prof, f"r2_bench_n{n}.json")).read().strip().splitlines()[-1])
        assert ln["n_gpus"] == n and ln["parity"]["ok"]
        assert all(r["ok"] and r["loss_identical_across_ranks"] for r in ln["parity"]["paths"].values())


def test_build_line_quotes_the_traffic_capture_of_the_same_library():
    """bench.py's line builder, fed with the recorded N = 1 measurements: the dominant kernel's
    roofline carries the per-launch DRAM traffic of the ncu capture -- and drops it for any other
    library version."""
    import types
    b = _bench_module()
    line = json.loads(open(os.path.join(ROOT, "profiles", "r2_bench_n1.json")).read().strip().splitlines()[-1])
    args = types.SimpleNamespace(workload="cfg3", gpus=1, steps=100, warmup=10, mode="bf16", impl="b200")
    cfg = {"B": 512, "D": 512, "C": 85742}

    def build(version):
        return b.build_line(args, cfg, 1, "bf16", b.load_peaks(), {k["kernel"]: k["ms"] for k in line["kernels"]},
                            {p["phase"]: p["ms"] for p in line["phases"]}, line["value"], line["ms_per_step"], "eager",
                            line["ms_per_step_by_path"], line["ms_per_step_dist"], line["e2e"]["value"],
                            line["e2e"]["ms_per_step"], line["e2e"]["path"], line["e2e"]["ms_per_step_by_path"], 512, 7,
                            100, 10, line["clocks"], line["parity"], {}, False, version, True)

    roof = build(line["library"])["roofline"]
    traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic_cfg3.json")))
    assert roof["kernel"] == "dw_gemm" and roof["traffic"] == traffic["kernels"]["dw_gemm"]
    assert roof["traffic"] > roof["algorithmic_bytes"]          # what the kernel really moves vs what it is credited
    other = build("some other build")["roofline"]
    assert other["traffic"] is None and "some other build" in other["traffic_source"]
