"""ctypes view of include/amsweep.h (the C-ABI a cgo shim would bind).

Loading fails loudly when libamsweep.so has not been built: there is no Python
or CPU fallback for the sweep.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

PKG = os.path.dirname(os.path.abspath(__file__))
# AMSWEEP_LIB: developer override to load an experimental build of the same ABI
LIB_PATH = os.environ.get("AMSWEEP_LIB") or os.path.join(PKG, "lib", "libamsweep.so")

u64, i64, u32, i32, u8 = C.c_uint64, C.c_int64, C.c_uint32, C.c_int32, C.c_uint8

# error codes
AM_OK, AM_E_INVAL, AM_E_RANGE, AM_E_NOSPACE, AM_E_DEVICE = 0, -1, -2, -3, -4
AM_E_NOMEM, AM_E_PARSE, AM_E_UNSUPPORTED, AM_E_BUSY = -5, -6, -7, -8
AM_CRON_ERROR, AM_CRON_SPEC, AM_CRON_EVERY = 0, 1, 2
STAR_BIT = 1 << 63

KIND_MASK = 0x7
KIND_NO_RESOURCE, KIND_STOPPED, KIND_INTERVAL, KIND_CRON_SPEC = 0, 1, 2, 3
KIND_CRON_EVERY, KIND_PARSE_ERROR, KIND_HOST_FALLBACK = 4, 5, 6
F_HAS_REMEDY, F_PENDING_OK, F_PENDING_FAIL = 1 << 3, 1 << 4, 1 << 5
F_REMEDY_PENDING, F_REMEDY_OUTCOME_OK = 1 << 6, 1 << 7
F_TOMBSTONE, F_STOPPED_REPORTED, F_TIMER_ARMED = 1 << 8, 1 << 9, 1 << 10
F_CARRY_MASK = 0x1F << 11  # library-internal (drain -> same tick's sweep), never visible
F_FAILP_SHIFT = 16
F_TZ_SHIFT = 24

ACT_SUBMIT_HC, ACT_RUN_REMEDY, ACT_STOPPED, ACT_PARSE_ERROR = 0x01, 0x02, 0x04, 0x08
ACT_REMEDY_SKIP, ACT_RESET_ON_PASS, ACT_RESET_ON_INTERVAL, ACT_ANOMALY = 0x10, 0x20, 0x40, 0x80

SWEEP_CLOSED_LOOP, SWEEP_FULL_SCAN, SWEEP_BLOCKED = 0x1, 0x2, 0x4
PHASE_NONE, PHASE_SUCCEEDED, PHASE_FAILED = 0, 1, 2
IPC_HANDLE_BYTES = 64


class AmCron(C.Structure):
    _fields_ = [("minute", u64), ("hour", u64), ("dom", u64), ("month", u64), ("dow", u64),
                ("delay_sec", i64), ("kind", i32), ("tz_id", i32)]


class AmHealthCheck(C.Structure):
    _fields_ = [("repeat_after_sec", i64), ("cron", C.c_char_p), ("cron_len", C.c_size_t),
                ("has_resource", i32), ("has_remedy", i32),
                ("remedy_runs_limit", i64), ("remedy_reset_interval", i64),
                ("finished_at", i64), ("remedy_finished_at", i64),
                ("finished_at_set", i32), ("remedy_finished_at_set", i32),
                ("success_count", i64), ("failed_count", i64),
                ("remedy_success_count", i64), ("remedy_failed_count", i64),
                ("remedy_total_runs", i64), ("fail_p8", u32), ("timer_armed", u32)]


class AmRecord(C.Structure):
    _fields_ = [("minute", u64), ("hour", u64), ("dom", u64), ("month", u64), ("dow", u64),
                ("finished_at", i64), ("remedy_finished_at", i64), ("ras", i32), ("flags", u32),
                ("runs_limit", i32), ("reset_interval", i32), ("success", i32), ("failed", i32),
                ("remedy_success", i32), ("remedy_failed", i32), ("remedy_total", i32),
                ("reserved", i32)]


RECORD_DTYPE = np.dtype([
    ("minute", "<u8"), ("hour", "<u8"), ("dom", "<u8"), ("month", "<u8"), ("dow", "<u8"),
    ("finished_at", "<i8"), ("remedy_finished_at", "<i8"), ("ras", "<i4"), ("flags", "<u4"),
    ("runs_limit", "<i4"), ("reset_interval", "<i4"), ("success", "<i4"), ("failed", "<i4"),
    ("remedy_success", "<i4"), ("remedy_failed", "<i4"), ("remedy_total", "<i4"),
    ("reserved", "<i4")])
assert RECORD_DTYPE.itemsize == C.sizeof(AmRecord) == 96

# column order == am_record_cols_t member order == am_sweep_column_ptr ids
COLUMNS = [("minute", np.uint64), ("hour", np.uint64), ("dom", np.uint64), ("month", np.uint64),
           ("dow", np.uint64), ("ras", np.int32), ("flags", np.uint32), ("finished_at", np.int64),
           ("runs_limit", np.int32), ("reset_interval", np.int32), ("success", np.int32),
           ("failed", np.int32), ("remedy_success", np.int32), ("remedy_failed", np.int32),
           ("remedy_total", np.int32), ("remedy_finished_at", np.int64)]
COLUMN_NAMES = [n for n, _ in COLUMNS]
SCHEDULE_COLUMNS = COLUMN_NAMES[:8]  # the 56 B/record a schedule-only tick reads


class AmRecordCols(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in COLUMN_NAMES]


STAT_FIELDS = ["n_records", "n_emitted", "n_submit_hc", "n_run_remedy", "n_stopped",
               "n_parse_error", "n_remedy_skip", "n_reset_on_pass", "n_reset_on_interval",
               "n_anomaly", "n_result_ok", "n_result_fail", "n_remedy_ok", "n_remedy_fail",
               "idx_xor", "idx_sum"]


class AmWorkItem(C.Structure):
    _fields_ = [("idx", u64), ("unix_sec", i64), ("action", u32), ("reserved", u32)]


WORK_ITEM_DTYPE = np.dtype([("idx", "<u8"), ("unix_sec", "<i8"), ("action", "<u4"), ("reserved", "<u4")])
assert WORK_ITEM_DTYPE.itemsize == C.sizeof(AmWorkItem) == 24


class AmTickView(C.Structure):
    _fields_ = [("idx_local", C.c_void_p), ("action", C.c_void_p), ("n", u64), ("shard_base", u64)]


class AmTickStats(C.Structure):
    _fields_ = [(n, u64) for n in STAT_FIELDS]

    def as_dict(self) -> dict:
        return {n: int(getattr(self, n)) for n in STAT_FIELDS}


STATS_DTYPE = np.dtype([(n, "<u8") for n in STAT_FIELDS])
assert STATS_DTYPE.itemsize == C.sizeof(AmTickStats) == 128

# every symbol include/amsweep.h declares: name -> (restype, argtypes)
P = C.POINTER
SYMBOLS = {
    "am_cron_parse": (C.c_int, [C.c_char_p, C.c_size_t, P(AmCron), C.c_char_p, C.c_size_t]),
    "am_tz_lookup": (C.c_int, [C.c_char_p, C.c_size_t, P(i32)]),
    "am_tz_offset": (C.c_int, [i32, i64, P(i32)]),
    "am_cron_matches": (C.c_int, [P(AmCron), i64]),
    "am_cron_next": (i64, [P(AmCron), i64]),
    "am_cron_repeat_after_sec": (i64, [P(AmCron), i64]),
    "am_healthcheck_classify": (C.c_int, [P(AmHealthCheck), P(AmRecord)]),
    "am_healthcheck_classify_batch": (C.c_int, [C.c_void_p, u64, C.c_void_p, C.c_void_p, C.c_int, P(u64)]),
    "am_healthcheck_ingest_json": (C.c_int, [C.c_char_p, C.c_size_t, u32, C.c_void_p, C.c_void_p, u64, P(u64), C.c_int]),
    "am_remedy_is_empty": (C.c_int, [C.c_size_t, C.c_int, i64, C.c_int]),
    "am_sweep_create": (C.c_int, [P(C.c_void_p), C.c_int, u64, u64]),
    "am_sweep_destroy": (None, [C.c_void_p]),
    "am_sweep_load_range": (C.c_int, [C.c_void_p, u64, u64, P(AmRecordCols)]),
    "am_sweep_upsert": (C.c_int, [C.c_void_p, u64, C.c_void_p, C.c_void_p]),
    "am_sweep_remove": (C.c_int, [C.c_void_p, u64, C.c_void_p]),
    "am_sweep_post_result": (C.c_int, [C.c_void_p, u64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "am_sweep_tick": (C.c_int, [C.c_void_p, i64, u32, C.c_void_p, C.c_void_p, u64, P(u64),
                                P(AmTickStats)]),
    "am_sweep_tick_view": (C.c_int, [C.c_void_p, i64, u32, P(AmTickView), P(AmTickStats)]),
    "am_sweep_last_list": (C.c_int, [C.c_void_p, u64, C.c_void_p, C.c_void_p, u64, P(u64)]),
    "am_sweep_tick_shard": (C.c_int, [C.c_void_p, i64, u32, C.c_void_p]),
    "am_sweep_tick_device": (C.c_int, [C.c_void_p, i64, u32, C.c_void_p, C.c_void_p, u64,
                                       C.c_void_p, C.c_void_p, C.c_void_p]),
    "am_sweep_run_ticks": (C.c_int, [C.c_void_p, i64, u64, u32, u64, C.c_void_p]),
    "am_sweep_run_ticks_view": (C.c_int, [C.c_void_p, i64, u64, u32, u64, C.c_void_p, C.c_void_p]),
    "am_sweep_repeat_after_sec": (C.c_int, [C.c_void_p, i64, u64, u64, C.c_void_p]),
    "am_sweep_next_due": (C.c_int, [C.c_void_p, i64, P(i64)]),
    "am_sweep_read": (C.c_int, [C.c_void_p, u64, u64, C.c_void_p, P(AmRecordCols)]),
    "am_sweep_size": (u64, [C.c_void_p]),
    "am_sweep_capacity": (u64, [C.c_void_p]),
    "am_sweep_device": (C.c_int, [C.c_void_p]),
    "am_sweep_last_kernel_ms": (C.c_double, [C.c_void_p]),
    "am_sweep_set_profiling": (C.c_int, [C.c_void_p, C.c_int]),
    "am_sweep_last_profile": (C.c_int, [C.c_void_p, P(C.c_double), P(C.c_double)]),
    "am_sweep_launch_count": (u64, [C.c_void_p]),
    "am_sweep_column_ptr": (C.c_void_p, [C.c_void_p, C.c_int]),
    "am_sweep_set_seed": (C.c_int, [C.c_void_p, u64]),
    "am_sweep_stream": (C.c_void_p, [C.c_void_p]),
    "am_gather_create": (C.c_int, [P(C.c_void_p), C.c_int, C.c_int, C.c_int, u64, C.c_int]),
    "am_gather_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "am_gather_connect": (C.c_int, [C.c_void_p, C.c_void_p]),
    "am_gather_set_layout": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "am_gather_exchange": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "am_gather_bind": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "am_gather_tick_view": (C.c_int, [C.c_void_p, i64, u32, P(AmTickView), P(AmTickStats)]),
    "am_gather_push": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, u64, C.c_void_p]),
    "am_gather_out_idx": (C.c_void_p, [C.c_void_p]),
    "am_gather_out_act": (C.c_void_p, [C.c_void_p]),
    "am_gather_out_counts": (C.c_void_p, [C.c_void_p]),
    "am_gather_set_profiling": (C.c_int, [C.c_void_p, C.c_int]),
    "am_gather_last_profile": (C.c_int, [C.c_void_p, P(C.c_double), P(C.c_double), P(C.c_double)]),
    "am_gather_last_error": (C.c_char_p, [C.c_void_p]),
    "am_gather_destroy": (None, [C.c_void_p]),
    "am_handoff_create": (C.c_int, [P(C.c_void_p), u64]),
    "am_handoff_destroy": (None, [C.c_void_p]),
    "am_handoff_publish": (C.c_int, [C.c_void_p, i64, u64, C.c_void_p, C.c_void_p, u32, P(u64)]),
    "am_handoff_pop": (C.c_int, [C.c_void_p, u64, C.c_void_p, P(u64)]),
    "am_handoff_stats": (C.c_int, [C.c_void_p, P(u64), P(u64), P(u64), P(u64)]),
    "am_civil_from_unix": (None, [i64, P(i32 * 6)]),
    "am_strerror": (C.c_char_p, [C.c_int]),
    "am_last_error_detail": (C.c_char_p, [C.c_void_p]),
    "am_abi_version": (C.c_int, []),
}

_lib = None


def load() -> C.CDLL:
    """dlopen libamsweep.so and type every entry point; raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python active-monitor_b200/build.py` "
            "(__graft_entry__.build()).  The sweep has no CPU or Python fallback.")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
