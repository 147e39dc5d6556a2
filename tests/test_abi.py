"""The C-ABI library loads on a CPU-only box and exports every symbol include/bsl_b200.h declares."""
import ctypes as C

import pytest

from boxsegliver_b200 import _lib, build


def test_library_builds_and_exports_header_symbols():
    path = build.build_library()
    assert path.exists()
    lib = C.CDLL(str(path))
    names = _lib.exported_symbols_in_header()
    assert len(names) >= 60
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/bsl_b200.h but not exported"


def test_struct_layouts_match_header():
    # sizes follow from the C declarations (ints / floats only, no padding surprises)
    assert C.sizeof(_lib.Conv2dDesc) == 9 * 4
    assert C.sizeof(_lib.ConvT2dDesc) == 8 * 4
    assert C.sizeof(_lib.NormDesc) == 11 * 4
    assert C.sizeof(_lib.LossDesc) == 4 * 4 + 8 * 4 + 2 * 4
    assert C.sizeof(_lib.AdamDesc) == 8 * 4
    assert C.sizeof(_lib.InputDesc) == 7 * 4 + 2 * 4 + 4 + 2 * 8      # bsl_input_desc (4 bytes of padding before seed)
    assert C.sizeof(_lib.InputParams) == 8 * 8                        # bsl_input_params


def test_product_path_has_no_cpu_fallback():
    """bsl_init must refuse to run without an sm_100 device instead of degrading to a CPU path."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is visible; the refusal path is exercised on CPU boxes")
    lib = _lib.load()
    h = C.c_void_p()
    rc = lib.bsl_init(C.c_int(0), C.byref(h))
    assert rc != 0 and not h.value


def test_version_string():
    assert b"sm_100a" in _lib.load().bsl_version()
