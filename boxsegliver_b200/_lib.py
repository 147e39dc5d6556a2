"""ctypes binding of libbsl_b200.so -- the only way host code reaches the sm_100a kernels.

There is deliberately no fallback: if the shared library is missing or a symbol is absent, importing
the product path raises. (The CPU oracle lives under oracle/ and is test infrastructure only.)
"""
from __future__ import annotations

import ctypes as C
import os
import re
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "libbsl_b200.so"
HEADER = PKG_DIR.parent / "include" / "bsl_b200.h"


class BslError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"bsl error {code}: {msg}")
        self.code = code


class Conv2dDesc(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("n", "h", "w", "cin", "cout", "kh", "kw", "x_ld", "y_ld")]


class ConvT2dDesc(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("n", "h", "w", "cin", "cout", "x_ld", "y_ld", "relu")]


class Conv3dDesc(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("n", "d", "h", "w", "cin", "cout", "kd", "kh", "kw", "sd", "sh", "sw", "x_ld",
                                       "y_ld")]


class ConvT3dDesc(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("n", "d", "h", "w", "cin", "cout", "sd", "x_ld", "y_ld", "relu")]


class NormDesc(C.Structure):
    _fields_ = [
        ("mode", C.c_int), ("n", C.c_int), ("hw", C.c_int), ("c", C.c_int),
        ("x_ld", C.c_int), ("y_ld", C.c_int),
        ("eps", C.c_float), ("decay", C.c_float),
        ("relu", C.c_int), ("center", C.c_int), ("scale", C.c_int),
    ]


class InputDesc(C.Structure):
    _fields_ = [("n", C.c_int), ("channels", C.c_int), ("src_h", C.c_int), ("src_w", C.c_int), ("out_h", C.c_int),
                ("out_w", C.c_int), ("max_centers", C.c_int), ("noise_scale", C.c_float), ("min_std", C.c_float),
                ("seed", C.c_ulonglong), ("offset", C.c_ulonglong)]


class InputParams(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("bbox", "clip", "lab_scale", "present", "flips", "centers", "stddevs",
                                          "n_centers")]


class Guide(C.Structure):
    _fields_ = [("map", C.c_void_p), ("channels", C.c_int), ("w", C.c_void_p), ("w_ld", C.c_int)]


class DropoutDesc(C.Structure):
    _fields_ = [("keep_prob", C.c_float), ("seed", C.c_ulonglong), ("offset", C.c_ulonglong)]


class FcDesc(C.Structure):
    _fields_ = [("n", C.c_int), ("cin", C.c_int), ("cout", C.c_int), ("relu", C.c_int), ("use_dropout", C.c_int),
                ("dropout", DropoutDesc)]


class SmallConvDesc(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("n", "h", "w", "cin", "cout", "kh", "kw", "x_ld", "y_ld")]


class LossDesc(C.Structure):
    _fields_ = [
        ("n", C.c_int), ("hw", C.c_int), ("classes", C.c_int), ("weight_type", C.c_int),
        ("numeric_w", C.c_float * 8), ("proportion_decay", C.c_float), ("loss_scale", C.c_float),
    ]


class AdamDesc(C.Structure):
    _fields_ = [
        ("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float),
        ("l2_rate", C.c_float), ("grad_scale", C.c_float), ("step", C.c_int), ("decoupled_decay", C.c_float),
    ]


def exported_symbols_in_header() -> list[str]:
    """Every function name declared in include/bsl_b200.h (used by the CPU-side ABI test)."""
    text = HEADER.read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(bsl_[a-zA-Z0-9_]+)\s*\(", text)))


_lib = None


def load() -> C.CDLL:
    """Load libbsl_b200.so (built in-tree by boxsegliver_b200.build). Raises if it is not there."""
    global _lib
    if _lib is not None:
        return _lib
    global LIB_PATH
    if os.environ.get("BSL_LIB"):       # tuning aid: A/B of two builds of the library in one process launch each
        LIB_PATH = Path(os.environ["BSL_LIB"]).resolve()
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU or PyTorch fallback for the hot path)")
    lib = C.CDLL(str(LIB_PATH))
    lib.bsl_last_error.restype = C.c_char_p
    lib.bsl_version.restype = C.c_char_p
    for name in exported_symbols_in_header():
        fn = getattr(lib, name)  # AttributeError here == header/library mismatch
        if name.endswith("_workspace"):
            fn.restype = C.c_size_t
        elif name == "bsl_crc32c":
            fn.restype, fn.argtypes = C.c_uint32, (C.c_uint32, C.c_void_p, C.c_size_t)
        elif name not in ("bsl_last_error", "bsl_version", "bsl_destroy"):
            fn.restype = C.c_int
    lib.bsl_destroy.restype = None
    _lib = lib
    return lib
