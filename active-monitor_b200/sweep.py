"""Python face of the C-ABI (include/amsweep.h) — plumbing for tests and bench.

The reference controller is Go; a Go shim would bind the same entry points with
cgo (INTEGRATION.md).  This module mirrors them one to one:

    cron_parse()            cron.ParseStandard            hcc.go:253
    classify()              processHealthCheck ladder     hcc.go:227/238/251/264
    Sweep.upsert()/remove() Reconcile create/update/delete hcc.go:170-188
    Sweep.post_result()     watch loops' terminal phases  hcc.go:635/662/821/836
    Sweep.tick()            every per-CR decision at once  hcc.go:238-267, 649-721, 751

Nothing here computes: every call goes through libamsweep.so.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _lib as L


class AmError(RuntimeError):
    def __init__(self, code: int, where: str, detail: str = ""):
        self.code = code
        msg = L.load().am_strerror(code).decode()
        super().__init__(f"{where}: {msg} ({code})" + (f": {detail}" if detail else ""))


class CronParseError(ValueError):
    """cron.ParseStandard would return an error (hcc.go:254-257)."""


class CronUnsupported(ValueError):
    """Valid for robfig, not evaluated on the device path (named time zone)."""


@dataclass(frozen=True)
class Cron:
    kind: int
    minute: int = 0
    hour: int = 0
    dom: int = 0
    month: int = 0
    dow: int = 0
    delay_sec: int = 0
    tz_id: int = 0  # SpecSchedule.Location: 0 = UTC, else an am_tz_lookup id

    def _c(self) -> L.AmCron:
        return L.AmCron(self.minute, self.hour, self.dom, self.month, self.dow, self.delay_sec,
                        self.kind, self.tz_id)

    def matches(self, unix_sec: int) -> bool:
        return bool(L.load().am_cron_matches(C.byref(self._c()), unix_sec))

    def next(self, unix_sec: int):
        v = L.load().am_cron_next(C.byref(self._c()), unix_sec)
        return None if v == -(1 << 63) else v

    def repeat_after_sec(self, unix_sec: int) -> int:
        return L.load().am_cron_repeat_after_sec(C.byref(self._c()), unix_sec)


def _as_bytes(spec) -> bytes:
    return spec if isinstance(spec, (bytes, bytearray)) else spec.encode("utf-8", "surrogateescape")


def cron_parse(spec) -> Cron:
    lib = L.load()
    raw = bytes(_as_bytes(spec))
    out = L.AmCron()
    err = C.create_string_buffer(256)
    rc = lib.am_cron_parse(raw, len(raw), C.byref(out), err, len(err))
    if rc == L.AM_E_PARSE:
        raise CronParseError(err.value.decode("utf-8", "replace"))
    if rc == L.AM_E_UNSUPPORTED:
        raise CronUnsupported(err.value.decode("utf-8", "replace"))
    if rc != L.AM_OK:
        raise AmError(rc, "am_cron_parse")
    return Cron(out.kind, out.minute, out.hour, out.dom, out.month, out.dow, out.delay_sec, out.tz_id)


def tz_lookup(name: str) -> int:
    """time.LoadLocation: the id of a named time zone (0 = UTC); raises CronParseError when unknown"""
    raw = name.encode()
    i = L.i32(0)
    rc = L.load().am_tz_lookup(raw, len(raw), C.byref(i))
    if rc == L.AM_E_PARSE:
        raise CronParseError(f"provided bad location {name}")
    if rc != L.AM_OK:
        raise AmError(rc, "am_tz_lookup")
    return i.value


def tz_offset(tz_id: int, unix_sec: int) -> int:
    off = L.i32(0)
    rc = L.load().am_tz_offset(tz_id, unix_sec, C.byref(off))
    if rc != L.AM_OK:
        raise AmError(rc, "am_tz_offset")
    return off.value


def civil_from_unix(unix_sec: int):
    out = (L.i32 * 6)()
    L.load().am_civil_from_unix(unix_sec, C.byref(out))
    return tuple(out)


def remedy_is_empty(generate_name: str, resource_is_nil: bool, timeout: int,
                    rbac_rules_is_nil: bool) -> bool:
    return bool(L.load().am_remedy_is_empty(len(generate_name.encode()), int(resource_is_nil),
                                            timeout, int(rbac_rules_is_nil)))


def classify(*, repeat_after_sec=0, cron="", has_resource=True, has_remedy=False,
             remedy_runs_limit=0, remedy_reset_interval=0, finished_at=None,
             remedy_finished_at=None, success_count=0, failed_count=0, remedy_success_count=0,
             remedy_failed_count=0, remedy_total_runs=0, fail_p8=0, timer_armed=True):
    """am_healthcheck_classify -> (rc, record as a 1-element RECORD_DTYPE array)."""
    raw = bytes(_as_bytes(cron))
    hc = L.AmHealthCheck(repeat_after_sec, raw, len(raw), int(has_resource), int(has_remedy),
                         remedy_runs_limit, remedy_reset_interval,
                         finished_at or 0, remedy_finished_at or 0,
                         int(finished_at is not None), int(remedy_finished_at is not None),
                         success_count, failed_count, remedy_success_count, remedy_failed_count,
                         remedy_total_runs, fail_p8, int(bool(timer_armed)))
    rec = L.AmRecord()
    rc = L.load().am_healthcheck_classify(C.byref(hc), C.byref(rec))
    arr = np.frombuffer(bytes(rec), dtype=L.RECORD_DTYPE).copy()
    return rc, arr


# ---- SoA helpers -------------------------------------------------------------
def alloc_columns(n: int) -> dict:
    return {name: np.zeros(n, dtype=dt) for name, dt in L.COLUMNS}


def cols_struct(cols: dict, names=None) -> L.AmRecordCols:
    """am_record_cols_t pointing at the given numpy arrays (missing -> NULL)."""
    s = L.AmRecordCols()
    for name, dt in L.COLUMNS:
        a = cols.get(name) if (names is None or name in names) else None
        if a is None:
            setattr(s, name, None)
            continue
        if a.dtype != np.dtype(dt) or not a.flags["C_CONTIGUOUS"]:
            raise TypeError(f"column {name}: need contiguous {np.dtype(dt)}, got {a.dtype}")
        setattr(s, name, a.ctypes.data)
    return s


def records_to_columns(recs: np.ndarray) -> dict:
    return {name: np.ascontiguousarray(recs[name]) for name in L.COLUMN_NAMES}


def columns_to_records(cols: dict) -> np.ndarray:
    n = len(cols["flags"])
    out = np.zeros(n, dtype=L.RECORD_DTYPE)
    for name in L.COLUMN_NAMES:
        out[name] = cols[name]
    return out


class Sweep:
    """One shard of the HealthCheck record array on one CUDA device."""

    def __init__(self, capacity: int, device: int = 0, shard_base: int = 0, lib=None):
        self._lib = lib or L.load()  # `lib`: another build of the same ABI (tests/emu)
        h = C.c_void_p()
        rc = self._lib.am_sweep_create(C.byref(h), device, capacity, shard_base)
        if rc != L.AM_OK:
            detail = self._lib.am_last_error_detail(None)
            raise AmError(rc, "am_sweep_create", detail.decode() if detail else "")
        self._h = h
        self.capacity = capacity
        self.shard_base = shard_base
        self.device = device

    # -- lifetime
    def close(self):
        if getattr(self, "_h", None):
            self._lib.am_sweep_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int, where: str):
        if rc != L.AM_OK:
            d = self._lib.am_last_error_detail(self._h)
            raise AmError(rc, where, d.decode() if d else "")

    # -- state in
    def load_range(self, first: int, cols: dict, names=None):
        n = len(cols["flags"])
        cs = cols_struct(cols, names)
        self._check(self._lib.am_sweep_load_range(self._h, first, n, C.byref(cs)), "am_sweep_load_range")

    def upsert(self, idx, recs: np.ndarray):
        idx = np.ascontiguousarray(idx, dtype=np.uint64)
        recs = np.ascontiguousarray(recs, dtype=L.RECORD_DTYPE)
        assert len(idx) == len(recs)
        self._check(self._lib.am_sweep_upsert(self._h, len(idx), idx.ctypes.data, recs.ctypes.data),
                    "am_sweep_upsert")

    def remove(self, idx):
        idx = np.ascontiguousarray(idx, dtype=np.uint64)
        self._check(self._lib.am_sweep_remove(self._h, len(idx), idx.ctypes.data), "am_sweep_remove")

    def post_result(self, idx, phase, remedy_phase=None):
        idx = np.ascontiguousarray(idx, dtype=np.uint64)
        phase = np.ascontiguousarray(phase, dtype=np.uint8)
        rp = None if remedy_phase is None else np.ascontiguousarray(remedy_phase, dtype=np.uint8)
        self._check(self._lib.am_sweep_post_result(self._h, len(idx), idx.ctypes.data,
                                                   phase.ctypes.data,
                                                   None if rp is None else rp.ctypes.data),
                    "am_sweep_post_result")

    # -- the tick
    def tick(self, unix_sec: int, mode: int = 0, cap: int | None = None, buffers=None):
        """Host-buffer tick.  Returns (global idx u64[n], action u32[n], stats dict).
        Raises AmError(AM_E_NOSPACE) with .needed set when cap is too small."""
        if buffers is not None:
            idx, act = buffers
            cap = len(idx)
        else:
            cap = self.capacity if cap is None else cap
            idx = np.empty(cap, dtype=np.uint64)
            act = np.empty(cap, dtype=np.uint32)
        n = L.u64(0)
        st = L.AmTickStats()
        rc = self._lib.am_sweep_tick(self._h, unix_sec, mode, idx.ctypes.data if cap else None,
                                     act.ctypes.data if cap else None, cap, C.byref(n), C.byref(st))
        if rc == L.AM_E_NOSPACE:
            e = AmError(rc, "am_sweep_tick")
            e.needed = n.value
            e.partial = (idx[:cap], act[:cap], st.as_dict())
            raise e
        self._check(rc, "am_sweep_tick")
        return idx[:n.value], act[:n.value], st.as_dict()

    def tick_view(self, unix_sec: int, mode: int = 0):
        """Host tick without the per-entry pass: (u32 LOCAL idx view, u8 action view, stats).
        The arrays alias the library's pinned buffer: valid until the next tick on the handle."""
        v = L.AmTickView()
        st = L.AmTickStats()
        self._check(self._lib.am_sweep_tick_view(self._h, unix_sec, mode, C.byref(v), C.byref(st)),
                    "am_sweep_tick_view")
        n = int(v.n)
        if n == 0:
            return np.empty(0, np.uint32), np.empty(0, np.uint8), st.as_dict()
        idx = np.ctypeslib.as_array(C.cast(v.idx_local, C.POINTER(C.c_uint32)), shape=(n,))
        act = np.ctypeslib.as_array(C.cast(v.action, C.POINTER(C.c_uint8)), shape=(n,))
        return idx, act, st.as_dict()

    def last_list(self, offset: int, cap: int):
        """Entries [offset, offset+cap) of the last host tick's list, widened; (idx, act, left)."""
        idx = np.empty(cap, dtype=np.uint64)
        act = np.empty(cap, dtype=np.uint32)
        n = L.u64(0)
        rc = self._lib.am_sweep_last_list(self._h, offset, idx.ctypes.data if cap else None,
                                          act.ctypes.data if cap else None, cap, C.byref(n))
        if rc not in (L.AM_OK, L.AM_E_NOSPACE):
            self._check(rc, "am_sweep_last_list")
        k = min(int(n.value), cap)
        return idx[:k], act[:k], int(n.value)

    def tick_shard(self, unix_sec: int, mode: int = 0, stream: int = 0):
        """Multi-GPU tick, first half (sweep + group scan); PeerGather.exchange does the rest."""
        self._check(self._lib.am_sweep_tick_shard(self._h, unix_sec, mode, stream or None), "am_sweep_tick_shard")

    def tick_device(self, unix_sec: int, mode: int, d_idx: int, d_act: int, cap: int,
                    d_count: int, d_stats: int = 0, stream: int = 0):
        """Device-resident tick on a caller stream (0 = CUDA default stream); raw
        device pointers (ints).  Does not synchronise."""
        self._check(self._lib.am_sweep_tick_device(self._h, unix_sec, mode, d_idx, d_act, cap,
                                                   d_count, d_stats or None, stream or None),
                    "am_sweep_tick_device")

    def run_ticks(self, unix_sec0: int, n_ticks: int, mode: int = 0, seed: int = 0) -> np.ndarray:
        out = np.zeros(n_ticks, dtype=L.STATS_DTYPE)
        self._check(self._lib.am_sweep_run_ticks(self._h, unix_sec0, n_ticks, mode, seed,
                                                 out.ctypes.data), "am_sweep_run_ticks")
        return out

    def run_ticks_view(self, unix_sec0: int, n_ticks: int, mode: int = 0, seed: int = 0):
        """run_ticks with every tick's list: (stats, [(u32 LOCAL idx view, u8 action view), ...]).
        The arrays alias the library's pinned buffer: valid until the next tick or run on the handle."""
        out = np.zeros(n_ticks, dtype=L.STATS_DTYPE)
        views = (L.AmTickView * max(n_ticks, 1))()
        self._check(self._lib.am_sweep_run_ticks_view(self._h, unix_sec0, n_ticks, mode, seed,
                                                      out.ctypes.data, views), "am_sweep_run_ticks_view")
        lists = []
        for v in views[:n_ticks]:
            n = int(v.n)
            if n == 0:
                lists.append((np.empty(0, np.uint32), np.empty(0, np.uint8)))
                continue
            idx = np.ctypeslib.as_array(C.cast(v.idx_local, C.POINTER(C.c_uint32)), shape=(n,))
            act = np.ctypeslib.as_array(C.cast(v.action, C.POINTER(C.c_uint8)), shape=(n,))
            lists.append((idx, act))
        return out, lists

    def repeat_after_sec(self, unix_sec: int, first: int, n: int) -> np.ndarray:
        """hcc.go:262 for every record of [first, first+n): Next() evaluated on the device."""
        out = np.zeros(n, dtype=np.int64)
        self._check(self._lib.am_sweep_repeat_after_sec(self._h, unix_sec, first, n, out.ctypes.data),
                    "am_sweep_repeat_after_sec")
        return out

    def next_due(self, unix_sec: int):
        """earliest second after unix_sec at which a tick would emit anything (None: never)"""
        v = L.i64(0)
        self._check(self._lib.am_sweep_next_due(self._h, unix_sec, C.byref(v)), "am_sweep_next_due")
        return None if v.value == (1 << 63) - 1 else v.value

    # -- state out
    def read_range(self, first: int, n: int, names=None) -> dict:
        cols = {name: np.zeros(n, dtype=dt) for name, dt in L.COLUMNS
                if names is None or name in names}
        cs = cols_struct(cols)
        self._check(self._lib.am_sweep_read(self._h, first, n, None, C.byref(cs)), "am_sweep_read")
        return cols

    def read(self, idx) -> dict:
        idx = np.ascontiguousarray(idx, dtype=np.uint64)
        cols = alloc_columns(len(idx))
        cs = cols_struct(cols)
        self._check(self._lib.am_sweep_read(self._h, 0, len(idx), idx.ctypes.data, C.byref(cs)),
                    "am_sweep_read")
        return cols

    # -- introspection
    def set_seed(self, seed: int):
        self._check(self._lib.am_sweep_set_seed(self._h, seed), "am_sweep_set_seed")

    def set_profiling(self, on: bool):
        self._check(self._lib.am_sweep_set_profiling(self._h, int(on)), "am_sweep_set_profiling")

    def last_profile(self):
        """(sweep_tick_kernel ms, rest of the tick ms) of the last tick; waits for it."""
        a, b = C.c_double(), C.c_double()
        self._check(self._lib.am_sweep_last_profile(self._h, C.byref(a), C.byref(b)), "am_sweep_last_profile")
        return a.value, b.value

    @property
    def stream(self) -> int:
        """the handle's own cudaStream_t"""
        return self._lib.am_sweep_stream(self._h) or 0

    @property
    def size(self) -> int:
        return self._lib.am_sweep_size(self._h)

    @property
    def last_kernel_ms(self) -> float:
        return self._lib.am_sweep_last_kernel_ms(self._h)

    @property
    def launch_count(self) -> int:
        return self._lib.am_sweep_launch_count(self._h)

    def column_ptr(self, name: str) -> int:
        return self._lib.am_sweep_column_ptr(self._h, L.COLUMN_NAMES.index(name)) or 0
