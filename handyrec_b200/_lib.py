"""ctypes binding of libhrb200.so (the C ABI declared in include/hrb200.h).

The prototypes are parsed from the header itself, so the binding cannot drift from
the ABI.  There is NO fallback: if the shared library is missing this module raises
at first use, and every compute entry point raises on a non-zero status.
"""
from __future__ import annotations

import ctypes
import os
import re
from typing import Dict, List, Tuple

HERE = os.path.dirname(os.path.abspath(__file__))
HEADER = os.path.join(HERE, "..", "include", "hrb200.h")
LIB_PATH = os.path.join(HERE, "libhrb200.so")

# status codes (include/hrb200.h: hrb_status)
HRB_OK, HRB_BAD_ARG, HRB_UNSUPPORTED, HRB_CUDA_ERROR, HRB_WORKSPACE = 0, 1, 2, 3, 4
# enums
POOL = {"none": 0, None: 0, "mean": 1, "sum": 2, "max": 3}
ACT = {None: 0, "linear": 0, "relu": 1, "sigmoid": 2, "tanh": 3, "dice": 4}
OPT_SGD, OPT_ADAM_LAZY, OPT_ADAGRAD, OPT_FTRL = 0, 1, 2, 3
GEMM_AUTO, GEMM_FP32, GEMM_3XTF32 = 0, 1, 2
BWD_AUTO, BWD_UNITS, BWD_SORT = 0, 1, 2


class HrbError(RuntimeError):
    def __init__(self, status: int, fn: str, detail: str):
        self.status = status
        super().__init__(f"{fn} failed with status {status}: {detail}")


class TableDesc(ctypes.Structure):
    _fields_ = [
        ("weight", ctypes.c_void_p),
        ("adam_m", ctypes.c_void_p),
        ("adam_v", ctypes.c_void_p),
        ("rows", ctypes.c_int64),
        ("dim", ctypes.c_int32),
        ("pad_", ctypes.c_int32),
    ]


class FieldDesc(ctypes.Structure):
    _fields_ = [
        ("table", ctypes.c_int32),
        ("seq_len", ctypes.c_int32),
        ("pool", ctypes.c_int32),
        ("ids_col", ctypes.c_int32),
        ("out_col", ctypes.c_int32),
        ("pad_", ctypes.c_int32),
    ]


class OptParams(ctypes.Structure):
    _fields_ = [
        ("opt", ctypes.c_int32),
        ("lr", ctypes.c_float),
        ("beta1", ctypes.c_float),
        ("beta2", ctypes.c_float),
        ("eps", ctypes.c_float),
        ("l2_scale", ctypes.c_float),
        ("bias_corr1", ctypes.c_float),
        ("bias_corr2", ctypes.c_float),
        ("l1", ctypes.c_float),  # Ftrl only (l2: with beta / (2*lr) added)
        ("l2", ctypes.c_float),
        ("lr_power", ctypes.c_float),
        ("l2_shrinkage", ctypes.c_float),
    ]


_SCALARS = {
    "int": ctypes.c_int,
    "int32_t": ctypes.c_int32,
    "uint32_t": ctypes.c_uint32,
    "int64_t": ctypes.c_int64,
    "size_t": ctypes.c_size_t,
    "float": ctypes.c_float,
}


def parse_header(path: str = HEADER) -> Dict[str, Tuple[object, List[object]]]:
    """Return {function name: (restype, [argtypes])} for every prototype in the header."""
    text = open(path).read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    text = re.sub(r"//[^\n]*", " ", text)
    protos: Dict[str, Tuple[object, List[object]]] = {}
    for m in re.finditer(r"\b(int|const char\s*\*)\s+(hrb_\w+)\s*\(([^;{}]*?)\)\s*;", text, flags=re.S):
        ret, name, args = m.group(1), m.group(2), m.group(3)
        restype = ctypes.c_char_p if "char" in ret else ctypes.c_int
        argtypes: List[object] = []
        args = " ".join(args.split())
        if args and args != "void":
            for a in args.split(","):
                a = a.strip()
                if "*" in a:
                    argtypes.append(ctypes.c_void_p)
                else:
                    ty = a.replace("const ", "").split()[0]
                    argtypes.append(_SCALARS[ty])
        protos[name] = (restype, argtypes)
    return protos


_lib = None


def lib() -> ctypes.CDLL:
    """Load libhrb200.so once; raise loudly when it is absent (no CPU fallback exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: build it with `python -m handyrec_b200.build` "
                "(handyrec_b200 has no CPU fallback)"
            )
        L = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in parse_header().items():
            fn = getattr(L, name)  # AttributeError if the .so does not export a declared symbol
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = L
    return _lib


def call(name: str, *args) -> None:
    """Call a status-returning entry point and raise HrbError on failure."""
    L = lib()
    rc = getattr(L, name)(*args)
    if rc != HRB_OK:
        raise HrbError(rc, name, L.hrb_last_error().decode("utf-8", "replace"))
