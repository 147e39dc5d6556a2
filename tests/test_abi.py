"""The C-ABI library loads on a CPU-only box and exports every symbol include/bsl_b200.h declares."""
import ctypes as C
import re
from pathlib import Path

import pytest

from boxsegliver_b200 import _lib, build

# Entry points of include/bsl_b200.h that no tests/test_gpu_*.py names, each with the reason it needs no op-level test.
NOT_NAMED_BY_GPU_TESTS = {
    "bsl_init": "context lifecycle: every GPU test runs through device.Context",
    "bsl_destroy": "context lifecycle: device.Context.close",
    "bsl_last_error": "host-side error text, read by device.Context.call on every failure",
    "bsl_version": "host-side string, checked by test_version_string",
    "bsl_crc32c": "host-only checksum of the checkpoint format, tested by tests/test_checkpoint.py",
    "bsl_device_status": "host read-back of the watchdog word: device.Context.check_device",
    "bsl_launch_count": "host-side launch counter (bench.py)",
    "bsl_debug_set": "tuning probe of the UMMA descriptors (tools/gpu_conv_probe.py)",
    "bsl_debug_read_waits": "tuning probe of the conv issue loop (tools/gpu_conv_bench.py)",
    "bsl_mem_info": "cudaMemGetInfo wrapper",
    "bsl_malloc": "allocator wrapper: device.DeviceBuffer",
    "bsl_free": "allocator wrapper: device.DeviceBuffer.free",
    "bsl_memcpy_h2d": "copy wrapper: device.DeviceBuffer.upload",
    "bsl_memcpy_d2h": "copy wrapper: device.DeviceBuffer.download",
    "bsl_memcpy_d2d": "copy wrapper",
    "bsl_host_alloc": "pinned-memory wrapper",
    "bsl_host_free": "pinned-memory wrapper",
    "bsl_stream_create": "stream wrapper: device.Context",
    "bsl_stream_destroy": "stream wrapper",
    "bsl_stream_sync": "stream wrapper: device.Context.sync",
    "bsl_stream_wait_event": "event wrapper",
    "bsl_event_create": "event wrapper",
    "bsl_event_destroy": "event wrapper",
    "bsl_event_record": "event wrapper",
    "bsl_event_sync": "event wrapper",
    "bsl_event_elapsed_ms": "event wrapper",
    "bsl_graph_begin": "CUDA-graph capture wrapper",
    "bsl_graph_end": "CUDA-graph capture wrapper",
    "bsl_graph_launch": "CUDA-graph capture wrapper",
    "bsl_graph_destroy": "CUDA-graph capture wrapper",
    "bsl_comm_unique_id": "NCCL set-up: needs one process per GPU (tools/dp_check.py)",
    "bsl_comm_init": "NCCL set-up: needs one process per GPU (tools/dp_check.py)",
    "bsl_comm_destroy": "NCCL set-up: needs one process per GPU (tools/dp_check.py)",
    "bsl_allreduce_sum_f32": "NCCL all-reduce: needs one process per GPU (tools/dp_check.py)",
    "bsl_input_stage": "reached through input_pipeline.DeviceInputStage in tests/test_gpu_input.py",
}


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


def test_every_entry_point_is_named_by_a_gpu_test():
    """Every function include/bsl_b200.h declares is called by name in some tests/test_gpu_*.py, apart from the
    host-side API listed in NOT_NAMED_BY_GPU_TESTS: a new kernel cannot ship without a GPU test that calls it."""
    names = set(_lib.exported_symbols_in_header())
    stale = sorted(set(NOT_NAMED_BY_GPU_TESTS) - names)
    assert not stale, f"listed in NOT_NAMED_BY_GPU_TESTS but not declared in include/bsl_b200.h: {stale}"
    text = "\n".join(p.read_text() for p in sorted(Path(__file__).resolve().parent.glob("test_gpu_*.py")))
    named = set(re.findall(r"\bbsl_[A-Za-z0-9_]+\b", text))
    missing = sorted(names - named - set(NOT_NAMED_BY_GPU_TESTS))
    assert not missing, f"declared in include/bsl_b200.h but named by no tests/test_gpu_*.py: {missing}"
