"""am_sweep_run_ticks_view: a run of consecutive ticks that returns every tick's (index, action) list,
with and without temporal blocking (AM_SWEEP_BLOCKED, sweep_block.cuh).  Every tick's list, action
bytes and statistics, and every column afterwards, must equal the CPU oracle evaluated tick by tick —
so the blocked and the unblocked run are also equal to each other.

The last test runs this file's GPU cases against the CPU-emulated build of the library.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

T0 = 1789982100  # 2026-09-21 09:15:00 UTC Monday


def _gen_pair(gen, am, orc, config, seed, n, T, first=0):
    prod = gen.fill(config, seed, first, n, T, am.load().am_healthcheck_classify)
    orac = gen.fill(config, seed, first, n, T, orc.load().orc_classify)
    return prod, orac


def _copy(cols):
    return {k: v.copy() for k, v in cols.items()}


def _check_run(am, orc, got, orac, t0, nt, mode, seed=0, base=0, what=""):
    """`got` = Sweep.run_ticks_view(t0, nt, mode, seed); advances `orac` through the same ticks."""
    stats, lists = got
    assert len(stats) == nt and len(lists) == nt
    emitted = 0
    for k in range(nt):
        wi, wa, ws = orc.sweep(orac, t0 + k, mode=mode & am.SWEEP_CLOSED_LOOP, seed=seed, shard_base=base)
        gs = {f: int(stats[f][k]) for f in am.abi.STAT_FIELDS}
        assert gs == ws, f"{what} tick {k}: stats\n got={gs}\n want={ws}"
        gi, ga = lists[k]
        assert gi.dtype == np.uint32 and ga.dtype == np.uint8
        np.testing.assert_array_equal(gi.astype(np.uint64) + np.uint64(base), wi, err_msg=f"{what} tick {k}: indices")
        np.testing.assert_array_equal(ga.astype(np.uint32), wa, err_msg=f"{what} tick {k}: actions")
        emitted += len(wi)
    return emitted


def _check_columns(am, s, orac, n, what="", skip=None):
    dev = s.read_range(0, n)
    keep = np.ones(n, bool)
    if skip is not None:
        keep[skip] = False
    for name in am.COLUMN_NAMES:
        np.testing.assert_array_equal(dev[name][keep], orac[name][keep], err_msg=f"{what}: column {name}")


def _run(am, s, t0, nt, mode, seed):
    """Sweep.run_ticks_view, checking from the handle's launch count that the form asked for ran: a blocked run
    launches, per block of ticks, the block kernel, one ring scan and one expand per 16 ticks (plus at most a
    drain's four kernels and two extra blocks where a zone changes its offset); an unblocked run at least the
    sweep, scan, expand and publish of every tick."""
    l0 = s.launch_count
    got = s.run_ticks_view(t0, nt, mode, seed)
    launches = s.launch_count - l0
    if s.size and nt:
        if mode & am.SWEEP_BLOCKED:
            b = min(int(os.environ.get("AMSWEEP_BLOCK_TICKS", "96")), nt)
            blocks = -(-nt // b) + 2
            assert launches <= blocks * (2 + -(-b // 16)) + 4, f"blocked run of {nt} ticks: {launches} launches"
        else:
            assert launches >= 4 * nt, f"unblocked run of {nt} ticks: {launches} launches"
    return got


def _both_modes(am, orc, setup, n, t0, nt, mode, seed=0, base=0, capacity=None, skip=None):
    """setup(sweep) -> oracle columns; runs the blocked and the unblocked form on fresh handles"""
    total = 0
    for blocked in (True, False):
        with am.Sweep(capacity=capacity or n, shard_base=base) as s:
            orac = setup(s)
            m = mode | (am.SWEEP_BLOCKED if blocked else 0)
            what = "blocked" if blocked else "unblocked"
            total = _check_run(am, orc, _run(am, s, t0, nt, m, seed), orac, t0, nt, m, seed, base, what)
            _check_columns(am, s, orac, n, what, skip)
    return total


@pytest.mark.gpu
@pytest.mark.parametrize("config,closed,start,nt,block", [
    (5, True, -30, 200, 0),      # cron + intervals, closed loop, three minute boundaries
    (22, False, -70, 150, 0),    # open loop, zone-bound schedules among the crons
    (55, True, -75, 160, 7),     # remedy mix, closed loop, short blocks
    (3, False, -10, 90, 0),      # open loop: posted results and remedy gates at the first tick, unarmed checks every tick
    (2, False, 45, 70, 64),      # open loop config 2
    (5, True, -100, 300, 128),   # the longest blocks
    (5, True, -20, 200, 96),     # the default block length, explicitly
    (5, True, 0, 1, 0),          # a single tick
])
def test_run_ticks_view_equals_the_oracle_tick_by_tick(am, orc, gen, monkeypatch, config, closed, start, nt, block):
    n, seed = 30_000, 9
    if block:
        monkeypatch.setenv("AMSWEEP_BLOCK_TICKS", str(block))
    prod, orac0 = _gen_pair(gen, am, orc, config, seed, n, T0)
    mode = am.SWEEP_CLOSED_LOOP if closed else 0

    def setup(s):
        s.load_range(0, prod)
        return _copy(orac0)
    emitted = _both_modes(am, orc, setup, n, T0 + start, nt, mode, seed)
    assert emitted > nt


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 511, 513, 1025, 8191, 8193, 20_001])
def test_sizes_that_are_not_whole_ctas_tiles_or_groups(am, orc, gen, monkeypatch, n):
    monkeypatch.setenv("AMSWEEP_BLOCK_TICKS", "16")
    prod, orac0 = _gen_pair(gen, am, orc, 2, 4, n, T0)

    def setup(s):
        s.load_range(0, prod)
        return _copy(orac0)
    _both_modes(am, orc, setup, n, T0 - 5, 40, 0)


@pytest.mark.gpu
def test_shard_base(am, orc, gen):
    n, base = 3000, 12_500_000
    prod = gen.fill(2, 4, base, n, T0, am.load().am_healthcheck_classify)
    orac0 = gen.fill(2, 4, base, n, T0, orc.load().orc_classify)

    def setup(s):
        s.load_range(0, prod)
        return _copy(orac0)
    assert _both_modes(am, orc, setup, n, T0 - 3, 70, 0, base=base) > 0


def _posted(am, n, every, seed):
    rng = np.random.default_rng(seed)
    idx = np.arange(0, n, every, dtype=np.uint64)
    phase = rng.integers(1, 3, len(idx)).astype(np.uint8)
    return idx, phase


@pytest.mark.gpu
@pytest.mark.parametrize("every", [11, 2])  # sparse (< 1 record in 8: applied at once by a tick) and dense
@pytest.mark.parametrize("closed", [False, True])
def test_posted_results_are_applied_and_counted_at_the_first_tick(am, orc, gen, every, closed):
    n, seed = 20_000, 3
    prod, orac0 = _gen_pair(gen, am, orc, 3, seed, n, T0)
    idx, phase = _posted(am, n, every, seed)
    mode = am.SWEEP_CLOSED_LOOP if closed else 0

    def setup(s):
        s.load_range(0, prod)
        s.post_result(idx, phase)
        o = _copy(orac0)
        bits = np.where(phase == am.PHASE_FAILED, am.F_PENDING_FAIL, am.F_PENDING_OK).astype(np.uint32)
        i = idx.astype(np.int64)
        o["flags"][i] = (o["flags"][i] & ~np.uint32(am.F_PENDING_OK | am.F_PENDING_FAIL)) | bits  # the latest result wins
        return o
    for blocked in (True, False):
        with am.Sweep(capacity=n) as s:
            orac = setup(s)
            m = mode | (am.SWEEP_BLOCKED if blocked else 0)
            got = _run(am, s, T0 + 1, 130, m, seed)
            _check_run(am, orc, got, orac, T0 + 1, 130, m, seed, what=f"blocked={blocked}")
            first = got[0][0]
            assert int(first["n_result_ok"]) + int(first["n_result_fail"]) > 0  # (the block kernel's own counts)
            _check_columns(am, s, orac, n)


@pytest.mark.gpu
def test_staged_upserts_and_removes_before_the_run(am, orc, gen):
    n = 5000
    prod, orac0 = _gen_pair(gen, am, orc, 55, 11, n, T0)
    recs = am.columns_to_records(prod)
    gone = np.array([3, 77, 1024, n - 1], dtype=np.uint64)

    def setup(s):
        perm = np.random.default_rng(0).permutation(n)
        s.upsert(perm[: n // 2], recs[perm[: n // 2]])
        s.upsert(perm[n // 2:], recs[perm[n // 2:]])
        s.remove(gone)
        o = _copy(orac0)
        o["flags"][gone.astype(np.int64)] = am.F_TOMBSTONE
        return o
    _both_modes(am, orc, setup, n, T0 - 40, 100, am.SWEEP_CLOSED_LOOP, seed=5, capacity=n + 100,
                skip=gone.astype(np.int64))


@pytest.mark.gpu
def test_a_block_across_a_daylight_saving_transition(am, orc):
    e = 1793512800  # 2026-11-01 06:00 UTC: New York, EDT -> EST
    zones = ["America/New_York", "Europe/Paris", "Australia/Lord_Howe", "Asia/Kathmandu"]
    specs = [f"CRON_TZ={z} * * * * *" for z in zones] + [f"CRON_TZ={z} {m} {h} * * *" for z in zones for h in (1, 2) for m in (0, 30)]
    specs += ["* * * * *", "0 6 * * *"]
    recs = [am.classify(cron=sp, finished_at=T0 - 5)[1] for sp in specs]
    cols = am.records_to_columns(np.concatenate(recs))
    ocols = _copy(cols)
    for k, sp in enumerate(specs):
        rc, oc, _ = orc.cron_parse(sp)
        assert rc == 0
        ocols["flags"][k] = (int(ocols["flags"][k]) & 0x00FFFFFF) | (oc.tz_id << 24)

    def setup(s):
        s.load_range(0, cols)
        return _copy(ocols)
    assert _both_modes(am, orc, setup, len(specs), e - 130, 260, 0) > 20


@pytest.mark.gpu
def test_empty_shard_zero_ticks_and_ticks_that_emit_nothing(am, orc):
    for mode in (0, am.SWEEP_BLOCKED):
        with am.Sweep(capacity=100) as s:
            stats, lists = s.run_ticks_view(T0, 5, mode)
            assert [len(i) for i, _ in lists] == [0] * 5
            assert (stats["n_emitted"] == 0).all() and (stats["n_records"] == 0).all()
            stats, lists = s.run_ticks_view(T0, 0, mode)
            assert len(stats) == 0 and lists == []
    # one daily schedule, a run far from 06:00: every tick emits nothing
    rc, rec = am.classify(cron="0 6 * * *", finished_at=T0 - 5)
    assert rc == 0
    cols = am.records_to_columns(rec)

    def setup(s):
        s.load_range(0, cols)
        return _copy(cols)
    assert _both_modes(am, orc, setup, 1, T0, 50, am.SWEEP_CLOSED_LOOP) == 0


@pytest.mark.gpu
def test_argument_errors(am, gen):
    lib = am.load()
    n = 1000
    prod = gen.fill(2, 1, 0, n, T0, lib.am_healthcheck_classify)
    with am.Sweep(capacity=n) as s:
        s.load_range(0, prod)
        st = np.zeros(4, dtype=am.abi.STATS_DTYPE)
        views = (am.abi.AmTickView * 4)()
        h = s._h
        for mode in (0, am.SWEEP_BLOCKED):
            assert lib.am_sweep_run_ticks_view(None, T0, 4, mode, 0, st.ctypes.data, views) == am.AM_E_INVAL
            assert lib.am_sweep_run_ticks_view(h, T0, 4, mode, 0, None, views) == am.AM_E_INVAL
            assert lib.am_sweep_run_ticks_view(h, T0, 4, mode, 0, st.ctypes.data, None) == am.AM_E_INVAL
            assert lib.am_sweep_run_ticks_view(h, T0, (1 << 24) + 1, mode, 0, st.ctypes.data, views) == am.AM_E_INVAL
            assert lib.am_sweep_run_ticks_view(h, 1 << 55, 4, mode, 0, st.ctypes.data, views) == am.AM_E_RANGE
            assert lib.am_sweep_run_ticks_view(h, -(1 << 55), 4, mode, 0, st.ctypes.data, views) == am.AM_E_RANGE
            assert lib.am_sweep_run_ticks_view(h, T0, 0, mode, 0, st.ctypes.data, views) == am.AM_OK
        # nothing ran: the columns are untouched
        dev = s.read_range(0, n)
        for name in am.COLUMN_NAMES:
            np.testing.assert_array_equal(dev[name], prod[name], err_msg=name)


@pytest.mark.gpu
def test_views_stay_valid_until_the_next_call_and_the_ring_grows(am, orc, gen, monkeypatch):
    n, seed = 30_000, 9
    prod, orac = _gen_pair(gen, am, orc, 5, seed, n, T0)
    mode = am.SWEEP_CLOSED_LOOP | am.SWEEP_BLOCKED
    with am.Sweep(capacity=n) as s:
        s.load_range(0, prod)
        monkeypatch.setenv("AMSWEEP_BLOCK_TICKS", "7")
        first = _run(am, s, T0, 40, mode, seed)
        kept = [(i.copy(), a.copy()) for i, a in first[1]]
        # read back and the statistics of an unrelated call in between do not touch the views
        s.read_range(0, 10)
        for (i, a), (ki, ka) in zip(first[1], kept):
            np.testing.assert_array_equal(i, ki)
            np.testing.assert_array_equal(a, ka)
        _check_run(am, orc, first, orac, T0, 40, mode, seed, what="first run")
        # a longer block: the ring grows; the second run's views replace the first's
        monkeypatch.setenv("AMSWEEP_BLOCK_TICKS", "96")
        second = _run(am, s, T0 + 40, 200, mode, seed)
        _check_run(am, orc, second, orac, T0 + 40, 200, mode, seed, what="second run")
        _check_columns(am, s, orac, n)
        # the buffer now holds a run, not a single tick's list
        _, _, left = s.last_list(0, 10)
        assert left == 0
        # and a plain tick afterwards is unaffected
        gi, ga, gs = s.tick(T0 + 240, mode=am.SWEEP_CLOSED_LOOP)
        wi, wa, ws = orc.sweep(orac, T0 + 240, mode=1, seed=seed)
        assert gs == ws
        np.testing.assert_array_equal(gi, wi)
        np.testing.assert_array_equal(ga, wa)


def test_gpu_cases_on_the_emulated_library():
    """This file's GPU cases through the C-ABI of the CPU-emulated build (tests/emu)."""
    from conftest import ROOT
    emu = os.path.join(ROOT, "tests", "emu")
    sys.path.insert(0, emu)
    import emu_sweep
    env = dict(os.environ, AMSWEEP_LIB=emu_sweep.build())
    out = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-m", "gpu", "-q", "-x",
                          "-p", "no:cacheprovider"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    tail = out.stdout[-3000:] + out.stderr[-2000:]
    assert out.returncode == 0, tail
    last = out.stdout.strip().splitlines()[-1]
    assert " passed" in last and "failed" not in last and "error" not in last, tail
