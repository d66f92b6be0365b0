"""The knob list stays complete: every ASM_* variable the library reads, and every one the README
documents, is either varied by test_kernel_variants_gpu.py or excluded there with a reason, and
the README documents no variable that nothing reads."""
import glob
import importlib.util
import os
import re

TESTS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(TESTS)


def _variants_module():
    spec = importlib.util.spec_from_file_location("kernel_variants", os.path.join(TESTS, "test_kernel_variants_gpu.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _found(pattern, paths):
    names = set()
    for p in paths:
        with open(p) as f:
            names |= set(re.findall(pattern, f.read()))
    return names


def test_every_knob_is_tested_or_excluded():
    kv = _variants_module()
    pkg = os.path.join(ROOT, "tf_face_toolbox_b200")
    native = _found(r'getenv\("(ASM_[A-Z0-9_]+)"\)', glob.glob(os.path.join(pkg, "csrc", "*.cu*")))
    python = _found(r'environ(?:\.get\(|\[)"(ASM_[A-Z0-9_]+)"', glob.glob(os.path.join(pkg, "*.py")))
    with open(os.path.join(ROOT, "README.md")) as f:
        rows = [line for line in f if line.startswith("| `ASM_")]
    readme = set(re.findall(r"`(ASM_[A-Z0-9_]+)", "".join(rows)))
    covered = set(kv.TESTED_KNOBS) | set(kv.EXCLUDED)
    assert native, "no getenv(\"ASM_...\") found in the library sources"
    assert not native - covered, sorted(native - covered)
    assert not readme - covered, sorted(readme - covered)
    assert not readme - (native | python), ("documented but read nowhere", sorted(readme - (native | python)))
    assert not covered - (native | python), ("listed but read nowhere", sorted(covered - (native | python)))
    assert set(kv.TESTED_KNOBS).isdisjoint(kv.EXCLUDED)
    assert all(reason.strip() for reason in kv.EXCLUDED.values())
