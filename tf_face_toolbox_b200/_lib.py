"""ctypes binding of libasoftmax_b200.so (include/asoftmax_b200.h).

The shared library is built in-tree by `__graft_entry__.build()` (nvcc, sm_100a) into
tf_face_toolbox_b200/lib/.  There is no CPU fallback and no alternative backend: if the
library is missing or no B200 is present, the product path raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
# ASM_B200_LIB selects another build of the same library (the `make TIMING=1` one under lib/timing/,
# or a build of another commit for an A/B run; bench.py reports any ASM_* variable in its JSON line)
LIB_PATH = os.environ.get("ASM_B200_LIB") or os.path.join(_HERE, "lib", "libasoftmax_b200.so")
CSRC = os.path.join(_HERE, "csrc")

ASM_OK = 0
ASM_ERR_INVALID_ARG = -1
ASM_ERR_CUDA = -2
ASM_ERR_NO_DEVICE = -3
ASM_ERR_LABEL_RANGE = -4
ASM_ERR_ALLOC = -5
ASM_ERR_PEER_TIMEOUT = -6
MODE_FP32, MODE_BF16 = 0, 1
MODES = {"fp32": MODE_FP32, "bf16": MODE_BF16}


class AsmConfig(C.Structure):
    _fields_ = [
        ("D", C.c_int32), ("C_total", C.c_int32), ("C_local", C.c_int32),
        ("class_offset", C.c_int32), ("B_max", C.c_int32), ("m", C.c_int32),
        ("mode", C.c_int32), ("rank", C.c_int32), ("world", C.c_int32),
        ("nccl_comm", C.c_void_p),
    ]


class AsmOptimizer(C.Structure):
    _fields_ = [("kind", C.c_int32), ("lr", C.c_float), ("momentum", C.c_float), ("beta1", C.c_float),
                ("beta2", C.c_float), ("epsilon", C.c_float), ("weight_decay", C.c_float),
                ("step", C.c_int64)]


OPT_NONE, OPT_MOMENTUM, OPT_ADAM = 0, 1, 2


class AsmMargin(C.Structure):
    _fields_ = [("kind", C.c_int32), ("s", C.c_float), ("m2", C.c_float), ("m3", C.c_float)]


MARGIN_ASOFTMAX, MARGIN_ADDITIVE, MARGIN_LINEAR = 0, 1, 3


class AsmLoss(C.Structure):
    _fields_ = [("kind", C.c_int32), ("gamma", C.c_float), ("alpha", C.c_float)]


LOSS_SOFTMAX_CE, LOSS_FOCAL = 0, 1


class AsmError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"asoftmax_b200 error {code}: {msg}")
        self.code = code


# every symbol include/asoftmax_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "asm_workspace_bytes": (C.c_size_t, [C.POINTER(AsmConfig)]),
    "asm_create": (C.c_int, [C.POINTER(_P), C.POINTER(AsmConfig)]),
    "asm_destroy": (C.c_int, [_P]),
    "asm_last_error": (C.c_char_p, [_P]),
    "asm_lambda": (C.c_float, [C.c_int64, C.c_float, C.c_float, C.c_float, C.c_float]),
    "asm_forward_backward": (C.c_int, [_P, _P, C.c_int32, _P, C.c_int32, _P, C.c_float, _P, _P, _P, _P, _P]),
    "asm_forward": (C.c_int, [_P, _P, C.c_int32, _P, C.c_int32, _P, C.c_float, _P, _P, _P]),
    "asm_forward_partial": (C.c_int, [_P, _P, C.c_int32, _P, C.c_int32, _P, C.c_float, _P, _P, _P]),
    "asm_backward_partial": (C.c_int, [_P, _P, C.c_int32, _P, _P, _P, _P]),
    "asm_check_labels": (C.c_int, [_P, _P]),
    "asm_last_launch_count": (C.c_int, [_P]),
    "asm_set_optimizer": (C.c_int, [_P, C.POINTER(AsmOptimizer), _P, _P]),
    "asm_center_scratch_bytes": (C.c_size_t, [C.c_int32]),
    "asm_center_loss": (C.c_int, [_P, C.c_int32, C.c_int32, _P, C.c_int32, _P, C.c_int32, C.c_int32,
                                  C.c_float, C.c_float, _P, _P, _P, _P]),
    "asm_p2p_bytes": (C.c_size_t, [C.POINTER(AsmConfig)]),
    "asm_p2p_attach": (C.c_int, [_P, C.POINTER(C.c_void_p)]),
    "asm_step_p2p": (C.c_int, [_P, _P, C.c_int32, _P, C.c_int32, _P, C.c_float, _P, _P, _P, _P]),
    "asm_p2p_set_timeout": (C.c_int, [_P, C.c_int32]),
    "asm_p2p_status": (C.c_int, [_P, _P]),
    "asm_set_gradient_transform": (C.c_int, [_P, C.c_float, C.c_float, _P]),
    "asm_set_embedding_dtype": (C.c_int, [_P, C.c_int32]),
    "asm_set_margin": (C.c_int, [_P, C.POINTER(AsmMargin)]),
    "asm_set_loss": (C.c_int, [_P, C.POINTER(AsmLoss)]),
    "asm_set_lambda_device": (C.c_int, [_P, _P]),
    "asm_set_profiling": (C.c_int, [_P, C.c_int]),
    "asm_get_profile": (C.c_int, [_P, C.c_int32, _P, _P]),
    "asm_version": (C.c_char_p, []),
}

_lib = None


def build(verbose: bool = False) -> str:
    """Compile the CUDA sources for sm_100a (nvcc cross-compiles without a GPU)."""
    r = subprocess.run(["make", "-C", CSRC, "-j8"], capture_output=True, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout[-4000:])
        print(r.stderr[-4000:])
    if r.returncode != 0:
        raise RuntimeError("building libasoftmax_b200.so failed")
    return LIB_PATH


def load() -> C.CDLL:
    """Load the C-ABI library and bind every declared symbol (fails loudly if absent)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU / PyTorch fallback for the A-softmax head)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, handle=None) -> None:
    if rc != ASM_OK:
        msg = load().asm_last_error(handle)
        raise AsmError(rc, msg.decode() if msg else "")
