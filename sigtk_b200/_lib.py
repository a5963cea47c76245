"""ctypes binding of the C-ABI declared in include/sigtk_b200.h.

The shared library is the product; this module only loads it.  There is no
Python or CPU fallback: if ``libsigtk_b200.so`` is missing the import of the
compute entry points fails loudly, and every compute call returns an error
code (raised as :class:`SgpuError`) when no CUDA device is usable.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsigtk_b200.so")

WANT_EVENTS, WANT_PA, WANT_STAT, WANT_ENT, WANT_JNN, WANT_PREFIX = 1, 2, 4, 8, 16, 32
F_DEFAULT, F_FORCE_GENERIC, F_NO_HOST_SLOTS, F_STAGE_TIMERS = 0, 1, 2, 4
ALIGN = 8

E_FULL, E_TOOBIG = -4, -5
LIVE_START, LIVE_END, LIVE_RNA = 1, 2, 4  # flags of a live entry (sgpu_slot_add_live, sgpu_slot_add_live_pa)

# every symbol include/sigtk_b200.h declares
EXPORTS = (
    "sgpu_abi_version", "sgpu_device_count", "sgpu_create", "sgpu_destroy", "sgpu_strerror",
    "sgpu_last_error", "sgpu_slot_batch", "sgpu_slot_reset", "sgpu_slot_add_read", "sgpu_submit",
    "sgpu_wait", "sgpu_run_device", "sgpu_counters", "sgpu_memcpy_d2h", "sgpu_stage_times",
    "sgpu_slot_add_read_svbzd", "sgpu_decode_svbzd_device", "sgpu_set_param", "sgpu_slot_add_read_pa",
    "sgpu_run_device_pa", "sgpu_live_open", "sgpu_slot_add_live", "sgpu_wait_live", "sgpu_run_device_live",
    "sgpu_slot_add_live_pa", "sgpu_run_device_live_pa", "sgpu_set_detector",
)
PARAM_CHUNK_LEN, PARAM_WARMUP, PARAM_THR_LONG, PARAM_PORE, PARAM_STAT_CTA_MIN = 1, 2, 3, 4, 5  # sgpu_set_param keys (development / test parameters)


class SgpuError(RuntimeError):
    def __init__(self, code: int, detail: str = ""):
        self.code = code
        super().__init__(f"sigtk_b200 error {code}: {detail}")


class Batch(C.Structure):  # sgpu_batch_t
    _fields_ = [
        ("samples", C.POINTER(C.c_int16)), ("read_off", C.POINTER(C.c_uint64)),
        ("read_len", C.POINTER(C.c_uint32)), ("offset_f", C.POINTER(C.c_float)),
        ("raw_unit_f", C.POINTER(C.c_float)), ("n_reads", C.c_uint32), ("rna", C.c_uint32),
    ]


class Result(C.Structure):  # sgpu_result_t
    _fields_ = [
        ("ev_off", C.c_void_p), ("ev_start", C.c_void_p), ("ev_mean", C.c_void_p), ("ev_stdv", C.c_void_p),
        ("pa", C.c_void_p), ("stat", C.c_void_p), ("seq_order", C.c_void_p), ("fixups", C.c_void_p),
        ("n_events", C.c_uint64), ("ent", C.c_void_p), ("jnn_cnt", C.c_void_p), ("jnn_seg", C.c_void_p),
        ("prefix_pos", C.c_void_p), ("prefix_stat", C.c_void_p),
    ]


class DevBatch(C.Structure):  # sgpu_dev_batch_t
    _fields_ = [
        ("samples", C.c_void_p), ("read_off", C.c_void_p), ("read_len", C.c_void_p), ("offset_f", C.c_void_p),
        ("raw_unit_f", C.c_void_p), ("n_reads", C.c_uint32), ("rna", C.c_uint32), ("span", C.c_uint64),
    ]


class DevPaBatch(C.Structure):  # sgpu_dev_pa_batch_t
    _fields_ = [
        ("pa", C.c_void_p), ("read_off", C.c_void_p), ("read_len", C.c_void_p), ("n_reads", C.c_uint32),
        ("rna", C.c_uint32), ("span", C.c_uint64),
    ]


class SvbDevBatch(C.Structure):  # sgpu_svb_dev_batch_t
    _fields_ = [
        ("bytes", C.c_void_p), ("n_bytes", C.c_uint64), ("comp_off", C.c_void_p), ("comp_len", C.c_void_p),
        ("read_off", C.c_void_p), ("read_len", C.c_void_p), ("n_reads", C.c_uint32), ("n_blocks", C.c_uint64),
    ]


class LiveResult(C.Structure):  # sgpu_live_result_t
    _fields_ = [
        ("ev_off", C.c_void_p), ("ev_start", C.c_void_p), ("ev_len", C.c_void_p), ("ev_mean", C.c_void_p),
        ("ev_stdv", C.c_void_p), ("n_events", C.c_uint64),
    ]


class DevLiveBatch(C.Structure):  # sgpu_dev_live_batch_t
    _fields_ = [
        ("samples", C.c_void_p), ("read_off", C.c_void_p), ("read_len", C.c_void_p), ("channel", C.c_void_p),
        ("flags", C.c_void_p), ("offset_f", C.c_void_p), ("raw_unit_f", C.c_void_p), ("n_entries", C.c_uint32),
        ("span", C.c_uint64),
    ]


class DevLivePaBatch(C.Structure):  # sgpu_dev_live_pa_batch_t
    _fields_ = [
        ("pa", C.c_void_p), ("read_off", C.c_void_p), ("read_len", C.c_void_p), ("channel", C.c_void_p),
        ("flags", C.c_void_p), ("n_entries", C.c_uint32), ("span", C.c_uint64),
    ]


class Counters(C.Structure):  # sgpu_counters_t
    _fields_ = [
        ("n_events", C.c_uint64), ("n_seq_order_reads", C.c_uint64), ("n_fixups", C.c_uint64),
        ("n_kernel_launches", C.c_uint64), ("status", C.c_int32), ("n_long_jobs", C.c_uint64),
    ]


class DetectorParams(C.Structure):  # sgpu_detector_t (detector_param, events.c:35-41)
    _fields_ = [("w_short", C.c_uint32), ("w_long", C.c_uint32), ("thr_short", C.c_float), ("thr_long", C.c_float),
                ("peak_height", C.c_float)]


class StageTime(C.Structure):  # sgpu_stage_time_t
    _fields_ = [("name", C.c_char_p), ("ms", C.c_float), ("launches", C.c_uint32)]


_lib = None


def load() -> C.CDLL:
    """Load the CUDA library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C sigtk_b200/csrc`. sigtk_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, u32, u64, i32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int
    lib.sgpu_abi_version.restype = i32
    lib.sgpu_device_count.restype = i32
    lib.sgpu_create.argtypes = [C.POINTER(vp), i32, u64, u32, u32, u32]
    lib.sgpu_create.restype = i32
    lib.sgpu_destroy.argtypes = [vp]
    lib.sgpu_destroy.restype = None
    lib.sgpu_strerror.argtypes = [i32]
    lib.sgpu_strerror.restype = C.c_char_p
    lib.sgpu_last_error.argtypes = [vp]
    lib.sgpu_last_error.restype = C.c_char_p
    lib.sgpu_slot_batch.argtypes = [vp, u32, C.POINTER(C.POINTER(Batch))]
    lib.sgpu_slot_batch.restype = i32
    lib.sgpu_slot_reset.argtypes = [vp, u32, u32]
    lib.sgpu_slot_reset.restype = i32
    lib.sgpu_slot_add_read.argtypes = [vp, u32, vp, u64, C.c_double, C.c_double, C.c_double]
    lib.sgpu_slot_add_read.restype = C.c_int64
    lib.sgpu_slot_add_read_svbzd.argtypes = [vp, u32, vp, u64, C.c_double, C.c_double, C.c_double]
    lib.sgpu_slot_add_read_svbzd.restype = C.c_int64
    lib.sgpu_slot_add_read_pa.argtypes = [vp, u32, vp, u64]
    lib.sgpu_slot_add_read_pa.restype = C.c_int64
    lib.sgpu_run_device_pa.argtypes = [vp, C.POINTER(DevPaBatch), u32, vp, C.POINTER(Result)]
    lib.sgpu_run_device_pa.restype = i32
    lib.sgpu_decode_svbzd_device.argtypes = [vp, C.POINTER(SvbDevBatch), vp, vp]
    lib.sgpu_decode_svbzd_device.restype = i32
    lib.sgpu_submit.argtypes = [vp, u32, u32]
    lib.sgpu_submit.restype = i32
    lib.sgpu_wait.argtypes = [vp, u32, C.POINTER(Result)]
    lib.sgpu_wait.restype = i32
    lib.sgpu_run_device.argtypes = [vp, C.POINTER(DevBatch), u32, vp, C.POINTER(Result)]
    lib.sgpu_run_device.restype = i32
    lib.sgpu_counters.argtypes = [vp, C.POINTER(Counters)]
    lib.sgpu_counters.restype = i32
    lib.sgpu_stage_times.argtypes = [vp, C.POINTER(StageTime), u32]
    lib.sgpu_stage_times.restype = i32
    lib.sgpu_memcpy_d2h.argtypes = [vp, vp, vp, u64]
    lib.sgpu_memcpy_d2h.restype = i32
    lib.sgpu_live_open.argtypes = [vp, u32]
    lib.sgpu_live_open.restype = i32
    lib.sgpu_slot_add_live.argtypes = [vp, u32, u32, u32, vp, u64, C.c_double, C.c_double, C.c_double]
    lib.sgpu_slot_add_live.restype = C.c_int64
    lib.sgpu_wait_live.argtypes = [vp, u32, C.POINTER(LiveResult)]
    lib.sgpu_wait_live.restype = i32
    lib.sgpu_run_device_live.argtypes = [vp, C.POINTER(DevLiveBatch), vp, C.POINTER(LiveResult)]
    lib.sgpu_run_device_live.restype = i32
    lib.sgpu_slot_add_live_pa.argtypes = [vp, u32, u32, u32, vp, u64]
    lib.sgpu_slot_add_live_pa.restype = C.c_int64
    lib.sgpu_run_device_live_pa.argtypes = [vp, C.POINTER(DevLivePaBatch), vp, C.POINTER(LiveResult)]
    lib.sgpu_run_device_live_pa.restype = i32
    lib.sgpu_set_param.argtypes = [vp, i32, C.c_double]
    lib.sgpu_set_param.restype = i32
    lib.sgpu_set_detector.argtypes = [vp, C.POINTER(DetectorParams)]
    lib.sgpu_set_detector.restype = i32
    _lib = lib
    return lib
