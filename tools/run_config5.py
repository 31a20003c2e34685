"""BASELINE configs[4]: 10 M HealthChecks x 86 400 consecutive one-second ticks
(one simulated day), streaming on one GPU, closed loop (SURVEY.md 8d).

Verification (the oracle is the checker, never the thing timed):
  * the first `--sub` records for the WHOLE day: per-tick statistics (counts and
    index checksums) of a GPU run over that sub-population == the CPU oracle's;
  * the full population for the first `--full-ticks` ticks: per-tick statistics
    of the timed run == the oracle's.
Prints one JSON object.
"""
import argparse
import importlib
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools", "amgen"), os.path.join(ROOT, "oracle")):
    sys.path.insert(0, p)
import numpy as np  # noqa: E402
import amgen  # noqa: E402
import oracle_c  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=10_000_000)
ap.add_argument("--ticks", type=int, default=86_400)
ap.add_argument("--sub", type=int, default=10_000)
ap.add_argument("--full-ticks", type=int, default=60)
ap.add_argument("--config", type=int, default=5)
ap.add_argument("--full-scan", action="store_true")
ap.add_argument("--blocked", action="store_true", help="AM_SWEEP_BLOCKED: temporal blocking (csrc/sweep_block.cuh)")
ap.add_argument("--compare-unblocked", action="store_true", help="with --blocked: also run the whole day tick by tick "
                "on a second handle and compare every tick's statistics and every column afterwards")
ap.add_argument("--per-tick", type=int, default=0,
                help="also time this many ticks one by one (CUDA events around the three kernels of "
                     "each tick) and report p50 / p99 / max per-tick device time")
ap.add_argument("--lists", action="store_true", help="time am_sweep_run_ticks_view (every tick's list to host memory), "
                "blocked and unblocked, against am_sweep_run_ticks(BLOCKED) without lists, over --windows windows of "
                "--window ticks; compare the lists of the two forms and, on the first --sub records, with the oracle")
ap.add_argument("--window", type=int, default=960, help="with --lists: ticks per call")
ap.add_argument("--windows", type=int, default=2, help="with --lists: consecutive calls (the first one allocates; "
                "86400 / 960 = 90 is the whole day)")
ap.add_argument("--profile-dir", default="", help="with --lists: write the torch.profiler kernel table here")
a = ap.parse_args()

am = importlib.import_module("active-monitor_b200")
lib = am.load()
T0, seed = amgen.T0_DAY_START, 5
mode = am.SWEEP_CLOSED_LOOP | (am.SWEEP_FULL_SCAN if a.full_scan else 0) | (am.SWEEP_BLOCKED if a.blocked else 0)
fields = am.abi.STAT_FIELDS

cols = amgen.fill(a.config, seed, 0, a.n, T0, lib.am_healthcheck_classify)


def gpu_name_and_power_limit():
    import subprocess
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # (reported, never guessed)
        return f"unknown ({e})"


def lists_run():
    """--lists: what the per-tick lists cost, and that both forms return the same lists."""
    W, nw = a.window, a.windows
    blocked, plain = mode | am.SWEEP_BLOCKED, mode & ~am.SWEEP_BLOCKED
    with am.Sweep(capacity=1000) as w:  # load the modules of every kernel once
        w.load_range(0, {k: np.ascontiguousarray(v[:1000]) for k, v in cols.items()})
        for m in (blocked, plain):
            w.run_ticks_view(T0, 4, m, seed)
        w.run_ticks(T0, 4, blocked, seed)
    out = {"gpu": gpu_name_and_power_limit(), "window_ticks": W, "windows": nw, "per_window": []}
    hb, hu, hn = am.Sweep(capacity=a.n), am.Sweep(capacity=a.n), am.Sweep(capacity=a.n)
    identical = True
    for h in (hb, hu, hn):
        h.load_range(0, cols)
    for k in range(nw):
        t = T0 + k * W
        row = {"first_tick": t}
        t0 = time.perf_counter()
        sb, lb = hb.run_ticks_view(t, W, blocked, seed)
        row["blocked_lists_us_per_tick"] = (time.perf_counter() - t0) * 1e6 / W
        t0 = time.perf_counter()
        su, lu = hu.run_ticks_view(t, W, plain, seed)
        row["unblocked_lists_us_per_tick"] = (time.perf_counter() - t0) * 1e6 / W
        t0 = time.perf_counter()
        sn = hn.run_ticks(t, W, blocked, seed)
        row["blocked_no_lists_us_per_tick"] = (time.perf_counter() - t0) * 1e6 / W
        row["blocked_no_lists_device_us_per_tick"] = hn.last_kernel_ms * 1e3 / W
        same = all(np.array_equal(sb[f], su[f]) and np.array_equal(sb[f], sn[f]) for f in fields)
        same &= all(np.array_equal(bi, ui) and np.array_equal(ba, ua) for (bi, ba), (ui, ua) in zip(lb, lu))
        identical &= bool(same)
        n_ent = np.array([len(i) for i, _ in lb], dtype=np.float64)
        row["entries_per_tick_mean"] = float(n_ent.mean())
        row["entries_per_tick_max"] = int(n_ent.max())
        row["host_bytes_per_tick_mean"] = float(n_ent.mean() * 5)
        out["per_window"].append(row)
    out["lists_identical"] = identical
    out["columns_identical"] = bool(all(np.array_equal(x, y) and np.array_equal(x, z) for x, y, z in
                                        ((hb.read_range(0, a.n)[c], hu.read_range(0, a.n)[c], hn.read_range(0, a.n)[c])
                                         for c in am.COLUMN_NAMES)))
    for h in (hb, hu, hn):
        h.close()
    # the split of one steady-state window: kernel time by kernel from torch.profiler (CUPTI), in a run of its own
    if a.profile_dir:
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.init()
        with am.Sweep(capacity=a.n) as hp:
            hp.load_range(0, cols)
            hp.run_ticks_view(T0, W, blocked, seed)  # allocations
            with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
                t0 = time.perf_counter()
                hp.run_ticks_view(T0 + W, W, blocked, seed)
                wall = time.perf_counter() - t0
        split = {}
        for ev in prof.key_averages():
            us = getattr(ev, "device_time_total", 0) or getattr(ev, "cuda_time_total", 0)
            for key in ("sweep_block_kernel", "ring_scan_kernel", "expand_kernel", "Memset"):
                if key in ev.key and us:
                    split[key] = split.get(key, 0.0) + us / W
        busy = sum(split.values())
        out["split_us_per_tick"] = dict(split, wall=wall * 1e6 / W, host_and_synchronisation=wall * 1e6 / W - busy)
        os.makedirs(a.profile_dir, exist_ok=True)
        with open(os.path.join(a.profile_dir, "run_ticks_view_kernels.txt"), "w") as f:
            f.write(prof.key_averages().table(sort_by="self_device_time_total" if hasattr(prof.key_averages()[0], "self_device_time_total") else "self_cuda_time_total", row_limit=30))
    # the oracle's lists on the first --sub records, both forms
    if a.sub:
        sub = {k: np.ascontiguousarray(v[: a.sub]) for k, v in cols.items()}
        osub = amgen.fill(a.config, seed, 0, a.sub, T0, oracle_c.load().orc_classify)
        got = {}
        for m in (blocked, plain):
            with am.Sweep(capacity=a.sub) as h:
                h.load_range(0, sub)
                st, li = h.run_ticks_view(T0, W, m, seed)
                got[m] = (st, [(i.copy(), x.copy()) for i, x in li])
        ok = True
        for k in range(W):
            wi, wa, ws = oracle_c.sweep(osub, T0 + k, mode=1, seed=seed)
            for m in (blocked, plain):
                st, li = got[m]
                ok &= all(int(st[f][k]) == ws[f] for f in fields)
                ok &= np.array_equal(li[k][0].astype(np.uint64), wi) and np.array_equal(li[k][1].astype(np.uint32), wa)
        out["oracle_lists_equal"] = {"records": a.sub, "ticks": W, "ok": bool(ok)}
    out["workload"] = (f"config {a.config}: {a.n} records, closed loop, seed 5, {nw} x {W} one-second ticks from "
                       "2026-09-21T00:00:00Z; times are host clocks around each call (every call ends synchronised)")
    return out


if a.lists:
    print(json.dumps(lists_run()))
    sys.exit(0)
with am.Sweep(capacity=a.n) as s:
    s.load_range(0, cols)
    t0 = time.perf_counter()
    stats = s.run_ticks(T0, a.ticks, mode=mode, seed=seed)
    wall = time.perf_counter() - t0
    dev_ms = s.last_kernel_ms
    launches = s.launch_count
    final = s.read_range(0, a.n) if a.compare_unblocked else None

same_as_unblocked = None
if a.blocked and a.compare_unblocked:
    with am.Sweep(capacity=a.n) as s4:
        s4.load_range(0, cols)
        plain = s4.run_ticks(T0, a.ticks, mode=mode & ~am.SWEEP_BLOCKED, seed=seed)
        plain_ms = s4.last_kernel_ms
        plain_final = s4.read_range(0, a.n)
    same_as_unblocked = {"per_tick_statistics": bool(all(np.array_equal(stats[f], plain[f]) for f in fields)),
                         "columns_afterwards": bool(all(np.array_equal(final[c], plain_final[c]) for c in am.COLUMN_NAMES)),
                         "unblocked_device_ms_total": plain_ms, "speed_up": plain_ms / dev_ms}
    del plain_final, final

# per-tick latency distribution: the streaming run above only has a total
per_tick = None
if a.per_tick:
    with am.Sweep(capacity=a.n) as s3:
        s3.load_range(0, cols)
        s3.set_seed(seed)
        bufs = (np.empty(a.n, dtype=np.uint64), np.empty(a.n, dtype=np.uint32))
        ms = np.empty(a.per_tick)
        same = True
        for k in range(a.per_tick):
            _, _, st = s3.tick(T0 + k, mode=mode, buffers=bufs)
            ms[k] = s3.last_kernel_ms
            if k < a.ticks:  # same ticks as the streaming run: statistics must agree
                same &= all(int(stats[f][k]) == st[f] for f in fields)
        on = np.arange(a.per_tick) % 60 == 0
        per_tick = {"ticks": a.per_tick, "equals_streaming_run": bool(same),
                    "us_p50": float(np.percentile(ms, 50) * 1e3), "us_p99": float(np.percentile(ms, 99) * 1e3),
                    "us_max": float(ms.max() * 1e3), "us_on_minute_p50": float(np.percentile(ms[on], 50) * 1e3),
                    "us_off_minute_p50": float(np.percentile(ms[~on], 50) * 1e3) if (~on).any() else None}

# full population, first ticks, against the oracle
ocols = amgen.fill(a.config, seed, 0, a.n, T0, oracle_c.load().orc_classify)
threads = os.cpu_count() or 1
full_ok = True
for k in range(min(a.full_ticks, a.ticks)):
    _, _, ws = oracle_c.sweep(ocols, T0 + k, mode=1, seed=seed, threads=threads)
    gs = {f: int(stats[f][k]) for f in fields}
    if gs != ws:
        full_ok = False
        print("MISMATCH full tick", k, gs, ws, file=sys.stderr)
        break

# sub-population, whole day
sub_ok = None
if a.sub:
    sub = {k: np.ascontiguousarray(v[: a.sub]) for k, v in amgen.fill(a.config, seed, 0, a.sub, T0, lib.am_healthcheck_classify).items()}
    with am.Sweep(capacity=a.sub) as s2:
        s2.load_range(0, sub)
        sub_stats = s2.run_ticks(T0, a.ticks, mode=mode, seed=seed)
        sub_final = s2.read_range(0, a.sub)
    osub = amgen.fill(a.config, seed, 0, a.sub, T0, oracle_c.load().orc_classify)
    sub_ok = True
    for k in range(a.ticks):
        _, _, ws = oracle_c.sweep(osub, T0 + k, mode=1, seed=seed)
        if any(int(sub_stats[f][k]) != ws[f] for f in fields):
            sub_ok = False
            print("MISMATCH sub tick", k, file=sys.stderr)
            break
    if sub_ok:
        sub_ok = all(np.array_equal(sub_final[name], osub[name]) for name in am.COLUMN_NAMES)

due = stats["n_submit_hc"].astype(np.float64)
on_min = np.arange(a.ticks) % 60 == 0
print(json.dumps({
    "workload": f"config {a.config}: {a.n} records x {a.ticks} one-second ticks from 2026-09-21T00:00:00Z, closed loop, seed 5",
    "mode": ("full-scan" if a.full_scan else "default (masks read only on the minute)") +
            (", AM_SWEEP_BLOCKED (96 ticks per pass over the columns, per-tick statistics only)" if a.blocked else ""),
    "identical_to_tick_by_tick": same_as_unblocked,
    "device_ms_total": dev_ms, "wall_s": wall, "evals_per_sec": a.n * a.ticks / (dev_ms * 1e-3),
    "us_per_tick_mean": dev_ms * 1e3 / a.ticks, "kernel_launches": int(launches),
    "due_per_tick_mean": float(due.mean()), "due_per_tick_on_minute_mean": float(due[on_min].mean()),
    "due_per_tick_off_minute_mean": float(due[~on_min].mean()) if (~on_min).any() else None,
    "total_submits": int(due.sum()), "total_remedies": int(stats["n_run_remedy"].sum()),
    "checksum_xor_of_idx_xor": int(np.bitwise_xor.reduce(stats["idx_xor"])),
    "verified_full_population_ticks": min(a.full_ticks, a.ticks), "full_ok": full_ok,
    "verified_subsample": f"{a.sub} records x {a.ticks} ticks", "sub_ok": sub_ok,
    "per_tick": per_tick,
    "algorithmic_bytes": int(a.n * (16 * a.ticks + 40 * (a.ticks if a.full_scan else int(on_min.sum())))),
}))
