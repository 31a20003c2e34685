#!/usr/bin/env python
"""bench.py — HealthCheck schedule evaluations/sec of the B200 sweep.

One "step" = one tick of the hot path (schedule ladder + remedy state machine,
SURVEY.md Appendix B.3) over the whole resident record array.

  --config 2 (default; BASELINE.json configs[1], the configuration `metric` is quoted on)
      10 M HealthChecks per GPU, mixed 5-field cron + repeatAfterSec, the single tick T0.
      At N>1 every rank owns an index-range shard of the same size (weak scaling; N=8 with
      --n 12500000 is BASELINE configs[3] at its literal 100 M) and the step ends with the
      global due list rebuilt on every GPU (NVLink tick exchange, csrc/gather.cu).
  --config 3 (BASELINE configs[2])  10 M HealthChecks, 50 % pending Failed / 25 % Succeeded
      through the remedy gate; state restored and L2 flushed between steps, outside the timing.
  --config 5 (BASELINE configs[4])  consecutive one-second ticks, closed loop, streaming.

  value     device-resident: state and outputs stay in HBM, CUDA events on the launching
            stream, max over ranks.
  e2e       through the host C-ABI calls a cgo shim makes (am_sweep_post_result +
            am_sweep_tick_view [+ am_gather_exchange at N>1]): results posted from host
            memory, the due list read in host memory, every step.
  roofline  algorithmic bytes of the sweep kernel / its measured duration, against
            MEASURED_PEAKS.json's HBM copy bandwidth.
  cpu_baseline / --impl reference
            the CPU oracle (our restatement of hcc.go + robfig/cron v3.0.1; the Go reference
            cannot be executed here) on the box's host cores.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tools", "amgen")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "healthcheck_schedule_evals_per_sec"
UNIT = "evals/s"
N_PER_GPU = 10_000_000
B_READ = 56          # algorithmic bytes read per evaluation, schedule-only (SURVEY §8d)
B_READ_REMEDY = 36   # + remedy/counter state of a record with a posted result (92 B in all)
B_BITMAP = 1.0 / 8   # emitted set: one bit per record (this layout; SURVEY assumed 4 B per due record)
B_EXC = 4            # per record whose action is not the bare SUBMIT_HC: (offset << 8 | action)
B_STOP = 12          # flags + finishedAt written when "Stopped" is first reported
CONFIG_SEED = {2: 2, 3: 3, 5: 5}
DUMP_BYTES = 64 << 20  # --dump-outputs writes at most this much in all
WORKLOAD = {
    2: "BASELINE configs[1]: {n} HealthChecks per GPU, mixed 5-field cron + repeatAfterSec (tools/amgen config 2, "
       "seed 2); step = the single tick T0=2026-09-21T09:15:00Z",
    3: "BASELINE configs[2]: {n} HealthChecks, 50 % pending Failed / 25 % pending Succeeded through RemedyRunsLimit / "
       "RemedyResetInterval (tools/amgen config 3, seed 3); step = the tick T0 that applies them; mutable columns "
       "restored and L2 flushed (256 MB read) between steps, outside the per-step CUDA-event interval",
    5: "BASELINE configs[4]: {n} HealthChecks x consecutive one-second ticks from 2026-09-21T00:00:00Z, closed loop "
       "(a due check completes in its tick), streaming on the device (tools/amgen config 5, seed 5); step = one tick",
}


def gpu_numa_cpus(torch, device_index: int):
    """CPUs of the NUMA node the GPU hangs off (its PCIe root), within the process's affinity; None when
    the topology cannot be read.  The timed GPU arm runs on them, as any GPU host process is normally bound
    (numactl): pinned buffers are then allocated on that node and the threads that fill and read them are
    next to them — without it a whole e2e run moved by up to 1.8x with where the scheduler put the threads."""
    try:
        p = torch.cuda.get_device_properties(device_index)
        bus = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        return (node, cpus) if len(cpus) >= 2 else None
    except Exception:
        return None


def host_threads() -> int:
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return os.cpu_count() or 1


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(config: int, n: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of one sweep_tick_kernel launch, from the
    `ncu --set full` capture of THIS round's kernel (profiles/r02_traffic.json, written by
    tools/ncu_traffic.py from the capture it names); null when no capture matches."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            for e in json.load(f)["captures"]:
                if e["config"] == config and e["n"] == n:
                    return int(e["dram_bytes"]), e["source"]
    except Exception:
        pass
    return None, None


class ClockSampler:
    """nvidia-smi clocks/throttle reasons while the GPU is under the bench load."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for t, line in self.rows:
            if t < t0 or t > t1:
                continue
            p = [x.strip() for x in line.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_sweep_times(cols, T0, reps, threads, oracle_c, seconds=None):
    """Per-tick wall times (s) of the oracle sweep — the same step as the GPU arm: the single
    tick T0 over the whole population — `reps` times (or for about `seconds`)."""
    import numpy as np
    n = len(cols["flags"])
    work = {k: v.copy() for k, v in cols.items()}
    # output lists preallocated once, as the GPU e2e arm's host buffers are
    bufs = (np.zeros(n, dtype=np.uint64), np.zeros(n, dtype=np.uint32))
    oracle_c.sweep(work, T0, threads=threads, buffers=bufs)  # warm caches / page in / first "Stopped" reports
    times, t_start = [], time.perf_counter()
    while True:
        t0 = time.perf_counter()
        oracle_c.sweep(work, T0, threads=threads, buffers=bufs)
        times.append(time.perf_counter() - t0)
        if seconds is None:
            if len(times) >= reps:
                break
        elif time.perf_counter() - t_start >= seconds or len(times) >= 2000:
            break
    return times


def write_outputs(out_dir, stats, idx=None, act=None):
    """--dump-outputs: the last timed step's outputs as out_dir/<name>.npy.  stats.npy holds the tick's
    statistics in STAT_FIELDS order (float64); due_index.npy / due_action.npy its due list (float64 /
    float32, exact for these values).  A list too long for DUMP_BYTES is cut to a fixed, seeded sample of
    its entries, kept in list order, so that two runs with the same arguments write the same files."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "stats.npy"), np.asarray(stats, dtype=np.float64))
    if idx is None:
        return
    room = (DUMP_BYTES - 4096) // 12  # 8 B index + 4 B action per entry; 4 KB for stats.npy and the headers
    if len(idx) > room:
        keep = np.sort(np.random.default_rng(0).choice(len(idx), room, replace=False))
        idx, act = idx[keep], act[keep]
    np.save(os.path.join(out_dir, "due_index.npy"), np.asarray(idx, dtype=np.float64))
    np.save(os.path.join(out_dir, "due_action.npy"), np.asarray(act, dtype=np.float32))


def run_reference(args, rank, world):
    """--impl reference: the CPU path on this box's host cores.  The reference is Go
    (robfig/cron un-vendored, no Go toolchain): this times oracle/ — our C restatement of the
    same decisions — on every host thread the process may use, pinned, on the SAME workload
    as the repo arm at this N (n records per GPU x N GPUs, one tick per step)."""
    if rank != 0:
        return
    import amgen
    import oracle_c
    import numpy as np
    threads = host_threads()
    config = args.config
    if config != 2:
        print(json.dumps({"impl": "reference", "unavailable": f"the reference arm times config 2 only (asked: {config})"}))
        return
    n = args.n * world
    T0 = amgen.T0_MON_0915
    cols = amgen.fill(config, CONFIG_SEED[config], 0, n, T0, oracle_c.load().orc_classify, threads=min(threads, 64))
    work = {k: v.copy() for k, v in cols.items()}
    bufs = (np.zeros(n, dtype=np.uint64), np.zeros(n, dtype=np.uint32))
    for w in range(args.warmup):
        oracle_c.sweep(work, T0, threads=threads, buffers=bufs)
    times = []
    t0 = time.perf_counter()
    for k in range(args.steps):
        t1 = time.perf_counter()
        last = oracle_c.sweep(work, T0, threads=threads, buffers=bufs)
        times.append(time.perf_counter() - t1)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        idx, act, st = last
        write_outputs(args.dump_outputs, [st[f] for f in oracle_c.STAT_FIELDS], idx, act)
    value = n * args.steps / dt
    sample = f"{n} records x {args.steps} ticks (whole config-2 population of the N={world} run each step)"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
        "data": "synthetic",
        "config": {"workload": WORKLOAD[2].format(n=args.n), "records_per_gpu": args.n, "records_total": n,
                   "note": "CPU oracle port of hcc.go + robfig/cron v3.0.1; Go reference not runnable here"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "ms_per_tick_min": min(times) * 1e3, "ms_per_tick_median": statistics.median(times) * 1e3,
                         "note": "threads = sched_getaffinity, workers pinned one per core; chunk per thread, two "
                                 "passes (evaluate + count, then write at the prefix), parked worker threads, "
                                 "preallocated output lists"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 5])
    ap.add_argument("--n", "--records-per-gpu", dest="n", type=int, default=N_PER_GPU, help="records per GPU "
                    "(spell it --records-per-gpu under torchrun: its parser rejects the abbreviation-like --n)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--e2e-workers", type=int, default=10, help="consumer threads of the e2e loop (walk the tick's "
                    "list and post results back: the reference's reconcile workers, hcc.go:170-188); default = the "
                    "reference's default --max-workers (cmd/main.go:144).  Bound to the GPU's NUMA node the step is "
                    "0.34 / 0.32 / 0.32 / 0.32 ms with 4 / 6 / 10 / 16 workers (profiles/r02_e2e_breakdown.json)")
    ap.add_argument("--e2e-python-loop", action="store_true", help="N>1: the round-2 python e2e loop (tick_shard, exchange, "
                    "read-back with torch copies) instead of the compiled loop over am_gather_tick_view")
    ap.add_argument("--no-verify", action="store_true", help="N>1: skip the oracle check of the gathered list")
    ap.add_argument("--gather", default="exchange", choices=["exchange", "plain", "nccl"],
                    help="N>1: NVLink tick exchange (bitmap + exceptions, list rebuilt on every GPU), the round-1 "
                         "plain list push, or the padded NCCL all-gather")
    ap.add_argument("--settle-ms", type=float, default=400.0,
                    help="untimed load before the warm-up steps so SM clocks settle (reported as settle_steps)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (at most 64 MB): "
                         "stats.npy (the tick's statistics) and, except for --config 5, whose step returns statistics "
                         "only, due_index.npy / due_action.npy (the tick's due list).  Inputs are seeded, so two "
                         "builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and args.impl == "ours" and world > 1:
        raise SystemExit("--dump-outputs writes the outputs of one GPU: run it with --gpus 1")
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import amgen
    am = importlib.import_module("active-monitor_b200")
    gather = importlib.import_module("active-monitor_b200.gather")
    lib = am.load()  # no fallback: raises if the CUDA library is missing

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the sweep has no CPU fallback")
    if args.config != 2 and world > 1:
        raise SystemExit("--config 3 / 5 are single-GPU lines; the multi-GPU step is config 2 (BASELINE configs[3])")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    all_cpus = os.sched_getaffinity(0)
    numa = gpu_numa_cpus(torch, local_rank)
    if numa is not None:
        os.sched_setaffinity(0, numa[1])  # (the CPU baseline below widens it again for its own run)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    config, seed = args.config, CONFIG_SEED[args.config]
    T0 = amgen.T0_MON_0915 if config != 5 else amgen.T0_DAY_START  # config 5: 2026-09-21 00:00:00 UTC
    n = args.n
    base = rank * n
    cols = amgen.fill(config, seed, base, n, T0, lib.am_healthcheck_classify, threads=min(host_threads(), 32))
    sweep = am.Sweep(capacity=n, device=local_rank, shard_base=base)
    sweep.load_range(0, cols)

    d_idx = torch.empty(n, dtype=torch.int32, device=dev)
    d_act = torch.empty(n, dtype=torch.uint8, device=dev)
    d_cnt = torch.zeros(1, dtype=torch.int32, device=dev)
    d_st = torch.zeros(16, dtype=torch.int64, device=dev)
    stream = torch.cuda.Stream(device=dev)  # explicit stream: kernels and events all on it
    torch.cuda.set_stream(stream)
    peer = gstream = None
    mode_gather = args.gather if world > 1 else None
    if world > 1 and args.gather != "nccl":
        ok = 1
        try:
            peer = gather.PeerGather(local_rank, cap_total=n * world, idx_bytes=4 if n * world < (1 << 32) else 8,
                                     shard=(base, n))
        except Exception as e:  # noqa: BLE001
            print(f"[bench] rank {rank}: peer gather unavailable ({e}); using NCCL", file=sys.stderr)
            ok = 0
        flag = torch.tensor([ok], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            if peer is not None:
                peer.close()
            peer, mode_gather = None, "nccl"
    if peer is not None:
        gstream = torch.cuda.Stream(device=dev, priority=-1)  # exchange CTAs are placed ahead of pending sweep CTAs
        ev_sweep = [torch.cuda.Event() for _ in range(2)]
        ev_gather = [torch.cuda.Event() for _ in range(2)]
        d_idx2 = [d_idx, torch.empty(n, dtype=torch.int32, device=dev)]
        d_act2 = [d_act, torch.empty(n, dtype=torch.uint8, device=dev)]
        d_cnt2 = [d_cnt, torch.zeros(1, dtype=torch.int32, device=dev)]
    step_no = [0]
    gather_launches = [0]

    # ---- config 3: the step consumes its inputs (pending results): snapshot / restore ----
    snap = flush = flush_sink = None
    if config == 3:
        MUT = ["flags", "finished_at", "success", "failed", "remedy_success", "remedy_failed", "remedy_total",
               "remedy_finished_at"]

        def col_view(name):
            dt = {"flags": torch.int32, "finished_at": torch.int64, "remedy_finished_at": torch.int64}.get(name, torch.int32)
            return peer_wrap(sweep.column_ptr(name), n, dt)

        def peer_wrap(ptr, count, dtype):
            class _A:
                pass
            a = _A()
            a.__cuda_array_interface__ = {"shape": (count,), "typestr": {torch.int32: "<i4", torch.int64: "<i8"}[dtype],
                                          "data": (ptr, False), "version": 3,
                                          "strides": (torch.empty(0, dtype=dtype).element_size(),)}
            return torch.as_tensor(a, device=dev)

        live = {m: col_view(m) for m in MUT}
        torch.cuda.synchronize()
        snap = {m: v.clone() for m, v in live.items()}
        flush = torch.zeros(64 << 20, dtype=torch.int32, device=dev)  # 256 MB
        flush_sink = torch.zeros((), dtype=torch.int64, device=dev)

    def restore():
        for m, v in snap.items():
            live[m].copy_(v)
        # READ 256 MB (> the 126 MB L2): the tick starts with none of its inputs cached and with no
        # dirty lines of the flush itself left to write back during the timed interval
        flush_sink.copy_(flush.sum())

    def step(_k):
        """one tick of the configured workload, device resident, asynchronous"""
        if config == 2 and peer is not None and mode_gather == "exchange":
            # tick k's exchange (NVLink + list rebuild) overlaps tick k+1's sweep (two streams; the
            # library alternates two buffer sets and makes tick k+2 wait for exchange k)
            sweep.tick_shard(T0, 0, stream.cuda_stream)
            peer.exchange(sweep, d_st.data_ptr(), gstream.cuda_stream)
            gather_launches[0] += 2
            step_no[0] += 1
            return
        if config == 2 and peer is not None:  # round-1 plain list push, overlapped the same way
            b = step_no[0] % 2
            if step_no[0] >= 2:
                stream.wait_event(ev_gather[b])
            sweep.tick_device(T0, 0, d_idx2[b].data_ptr(), d_act2[b].data_ptr(), n, d_cnt2[b].data_ptr(),
                              d_st.data_ptr(), stream.cuda_stream)
            ev_sweep[b].record(stream)
            gstream.wait_event(ev_sweep[b])
            peer.push(d_idx2[b].data_ptr(), d_act2[b].data_ptr(), d_cnt2[b].data_ptr(), base, gstream.cuda_stream)
            ev_gather[b].record(gstream)
            gather_launches[0] += 1
            step_no[0] += 1
            return
        sweep.tick_device(T0, 0, d_idx.data_ptr(), d_act.data_ptr(), n, d_cnt.data_ptr(), d_st.data_ptr(),
                          stream.cuda_stream)
        step_no[0] += 1
        if world > 1:
            gather.allgather_due(d_idx, d_act, d_cnt, base)

    def drain():
        """make `stream` wait for every exchange still in flight on the gather stream"""
        if peer is not None:
            e = torch.cuda.Event()
            e.record(gstream)
            stream.wait_event(e)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def last_list():
        """host copies of what the last tick_device step left on the device: (stats, due list, actions)"""
        cnt = int(d_cnt.item())
        return d_st.cpu().numpy(), d_idx[:cnt].cpu().numpy(), d_act[:cnt].cpu().numpy()

    # ---- N>1: is the gathered list right?  checked before and after the timed loop ----
    verify = None

    def verify_gathered(tag):
        """Every rank: checksum of the gathered global list == all-reduced per-shard statistics of
        an independent LOCAL tick of each shard; rank 0 (once): the whole list == the oracle's
        sweep of the unsharded population."""
        nonlocal verify
        if world == 1 or peer is None or mode_gather != "exchange" or args.no_verify:
            return
        # independent per-shard figures: a plain local tick (list rebuilt from this shard's bitmap only)
        sweep.tick_device(T0, 0, d_idx.data_ptr(), d_act.data_ptr(), n, d_cnt.data_ptr(), d_st.data_ptr(),
                          stream.cuda_stream)
        stream.synchronize()
        st = dict(zip(am.abi.STAT_FIELDS, [int(v) & ((1 << 64) - 1) for v in d_st.cpu().tolist()]))
        mine = torch.tensor([st["n_emitted"], st["idx_sum"] & 0x7FFFFFFFFFFFFFFF, st["idx_xor"] & 0x7FFFFFFFFFFFFFFF,
                             st["n_submit_hc"], st["n_stopped"], st["n_parse_error"]], dtype=torch.int64, device=dev)
        allst = torch.empty(world * 6, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(allst, mine)
        allst = allst.cpu().numpy().reshape(world, 6)
        # the exchanged tick
        sweep.tick_shard(T0, 0, stream.cuda_stream)
        peer.exchange(sweep, d_st.data_ptr(), stream.cuda_stream)
        stream.synchronize()
        gi, ga, counts = peer.result()
        gi = gi.cpu().numpy()
        gi = (gi.astype(np.int64) & 0xFFFFFFFF).astype(np.uint64) if gi.dtype == np.int32 else gi.astype(np.uint64)
        ga = ga.cpu().numpy()
        ok = counts == [int(c) for c in allst[:, 0]]
        ok &= len(gi) == int(allst[:, 0].sum())
        ok &= bool((np.diff(gi.astype(np.int64)) > 0).all())
        ok &= int(gi.sum(dtype=np.uint64)) & 0x7FFFFFFFFFFFFFFF == int(np.bitwise_and(allst[:, 1].astype(np.uint64).sum(dtype=np.uint64), np.uint64(0x7FFFFFFFFFFFFFFF)))
        ok &= int(np.bitwise_xor.reduce(gi)) & 0x7FFFFFFFFFFFFFFF == int(np.bitwise_xor.reduce(allst[:, 2].astype(np.uint64)))
        ok &= int((ga & 1 != 0).sum()) == int(allst[:, 3].sum())
        ok &= int((ga & 4 != 0).sum()) == int(allst[:, 4].sum())
        ok &= int((ga & 8 != 0).sum()) == int(allst[:, 5].sum())
        oracle_ok = None
        if rank == 0 and tag == "before":
            import oracle_c
            threads = host_threads()
            whole = amgen.fill(config, seed, 0, n * world, T0, oracle_c.load().orc_classify, threads=min(threads, 64))
            oracle_c.sweep(whole, T0, threads=threads)  # the tick the warm-up applied first ("Stopped" is reported once)
            wi, wa, _ = oracle_c.sweep(whole, T0, threads=threads)
            oracle_ok = bool(np.array_equal(gi, wi) and np.array_equal(ga.astype(np.uint32), wa))
            del whole
        flag = torch.tensor([1 if ok else 0, 1 if oracle_ok in (None, True) else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        verify = verify or {"gather_verified": True, "checks": []}
        verify["gather_verified"] &= bool(flag[0].item()) and bool(flag[1].item())
        verify["checks"].append({"when": tag, "entries": int(len(gi)), "checksums_all_ranks": bool(flag[0].item()),
                                 "rank0_list_equals_unsharded_oracle": None if tag != "before" else bool(flag[1].item())})

    sampler = ClockSampler(local_rank) if rank == 0 else None
    torch.cuda.synchronize()

    if config == 5:
        # streaming: K consecutive ticks back to back inside the library (CUDA events around them)
        sweep.set_seed(seed)
        t_load0 = time.perf_counter()
        settle = max(args.warmup, int(args.settle_ms / 0.1))
        sweep.run_ticks(T0, settle, am.SWEEP_CLOSED_LOOP, seed)
        launches0 = sweep.launch_count
        w0 = time.perf_counter()
        stats_k = sweep.run_ticks(T0 + settle, args.steps, am.SWEEP_CLOSED_LOOP, seed)
        wall = time.perf_counter() - w0
        last = ([stats_k[f][-1] for f in am.abi.STAT_FIELDS],)
        ms = sweep.last_kernel_ms
        launches = sweep.launch_count - launches0
        sweep.run_ticks(T0 + settle + args.steps, max(64, int(800 / 0.1)), am.SWEEP_CLOSED_LOOP, seed)
        t_load1 = time.perf_counter()
        clocks = sampler.stop(t_load0, t_load1) if sampler else None
        stats = {f: int(stats_k[f].mean()) for f in am.abi.STAT_FIELDS}
        e2e = {"value": n * args.steps / wall, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 128,
               "ms_per_step": wall / args.steps * 1e3, "steps": args.steps,
               "api": "am_sweep_run_ticks (state resident, per-tick statistics copied to host memory)"}
        settle_steps, per_step_ms = settle, None
        # the same run with temporal blocking (AM_SWEEP_BLOCKED, csrc/sweep_block.cuh: 96 ticks per pass over
        # the columns, records stepped from event to event), on a second handle from the same initial state;
        # reported separately from the K = 1 number (SURVEY 7 step 9), and checked against it tick by tick
        blocking = None
        if rank == 0 or world == 1:
            with am.Sweep(capacity=n, device=local_rank, shard_base=base) as s2:
                s2.load_range(0, cols)
                s2.set_seed(seed)
                b_stats = s2.run_ticks(T0, settle + args.steps, am.SWEEP_CLOSED_LOOP | am.SWEEP_BLOCKED, seed)
                b_ms = s2.last_kernel_ms
                same = all(np.array_equal(b_stats[f][settle:], stats_k[f]) for f in am.abi.STAT_FIELDS)
                blocking = {"ticks_per_pass": int(os.environ.get("AMSWEEP_BLOCK_TICKS", 96)),
                            "ticks": settle + args.steps, "ms_per_tick": b_ms / (settle + args.steps),
                            "value": n / (b_ms / (settle + args.steps) * 1e-3), "unit": UNIT,
                            "identical_to_tick_by_tick": bool(same),
                            "what": "am_sweep_run_ticks with AM_SWEEP_BLOCKED: per-tick statistics only (no per-tick lists); "
                                    "not the roofline number"}
    elif config == 3:
        t_load0 = time.perf_counter()
        settle_steps = 0
        for i in range(args.warmup):
            restore()
            step(i)
        torch.cuda.synchronize()
        launches0 = sweep.launch_count
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for k in range(args.steps):
            restore()
            evs[k][0].record(stream)
            step(k)
            evs[k][1].record(stream)
        torch.cuda.synchronize()
        last = last_list() if args.dump_outputs else None
        per_step_ms = [a.elapsed_time(b) for a, b in evs]
        ms = sum(per_step_ms)
        launches = sweep.launch_count - launches0
        stats = dict(zip(am.abi.STAT_FIELDS, [int(v) for v in d_st.cpu().tolist()]))
        t_load1 = time.perf_counter()
        clocks = sampler.stop(t_load0, t_load1) if sampler else None
        e2e = None
    else:
        # settle (untimed, reported), then exactly W warm-up and K timed steps; every rank runs the
        # SAME number of steps (each ends in a cross-GPU exchange at N>1)
        probe0, probe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        probe0.record(stream)
        for i in range(8):
            step(-1)
        drain()
        probe1.record(stream)
        barrier()
        est_ms = max(probe0.elapsed_time(probe1) / 8, 1e-3)
        settle_steps = int(args.settle_ms / est_ms)
        if world > 1:
            t = torch.tensor([settle_steps], dtype=torch.int64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            settle_steps = int(t.item())
        t_load0 = time.perf_counter()
        for i in range(settle_steps):
            step(-1)
            if i % 256 == 255:
                torch.cuda.synchronize()
        drain()
        barrier()
        verify_gathered("before")
        for i in range(args.warmup):
            step(-1)
        drain()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        # host time to ISSUE a step: a short burst into an empty queue (a long loop blocks on the full launch queue and
        # shows the device time instead); when this is close to ms_per_step the loop is launch-bound, not GPU-bound
        torch.cuda.synchronize()
        h0 = time.perf_counter()
        for i in range(16):
            step(-1)
        host_issue_ms = (time.perf_counter() - h0) * 1e3 / 16
        drain()
        barrier()
        launches0, gl0 = sweep.launch_count, gather_launches[0]
        ev0.record(stream)
        for k in range(args.steps):
            step(k)
        drain()
        ev1.record(stream)
        barrier()
        last = last_list() if args.dump_outputs else None
        ms = ev0.elapsed_time(ev1)
        launches = sweep.launch_count - launches0 + gather_launches[0] - gl0
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        # keep the identical load running ~0.8 s more (same count on every rank) so the
        # 100 ms nvidia-smi sampler sees the GPU under exactly this load
        extra = min(20000, max(64, int(0.8 / max(ms / args.steps * 1e-3, 1e-6))))
        for k in range(extra):
            step(k)
            if k % 256 == 255:
                torch.cuda.synchronize()
        drain()
        barrier()
        t_load1 = time.perf_counter()
        clocks = sampler.stop(t_load0, t_load1) if sampler else None
        verify_gathered("after")
        sweep.tick_device(T0, 0, d_idx.data_ptr(), d_act.data_ptr(), n, d_cnt.data_ptr(), d_st.data_ptr(),
                          stream.cuda_stream)
        stream.synchronize()
        stats = dict(zip(am.abi.STAT_FIELDS, [int(v) for v in d_st.cpu().tolist()]))
        per_step_ms = None

    # ---- per-kernel durations for the roofline (CUDA events on the launching stream
    #      around the sweep kernel and around the rest of the tick, inside the library) ----
    ks, kc = [], []
    kreps = max(20, min(args.steps, 200))
    if config != 5:
        sweep.set_profiling(True)
        for k in range(kreps):
            if config == 3:
                restore()
            sweep.tick_device(T0, 0, d_idx.data_ptr(), d_act.data_ptr(), n, d_cnt.data_ptr(), d_st.data_ptr(),
                              stream.cuda_stream)
            a_ms, b_ms = sweep.last_profile()
            ks.append(a_ms); kc.append(b_ms)
        sweep.set_profiling(False)
        k_ms, c_ms = statistics.mean(ks), statistics.mean(kc)
    else:
        k_ms = c_ms = None
    # exceptions = emitted entries whose action is not the bare SUBMIT_HC, counted from the list itself
    n_exc = int((d_act[: min(int(d_cnt.item()), n)] > 1).sum().item()) if config != 5 else 0
    if config == 3:
        n_res = stats["n_result_ok"] + stats["n_result_fail"]
        changed = n_res * 16 + (stats["n_remedy_ok"] + stats["n_remedy_fail"]) * 16  # flags+fa+S|F, RS|RF+RT+rfa
        alg_bytes = int(n * B_READ + n_res * B_READ_REMEDY + changed + n * B_BITMAP + n_exc * B_EXC)
        model = "N*56 + results*36 + results*16 + remedy_results*16 + N/8 (bitmap) + exceptions*4"
        # SURVEY 8(d) literal: every record of config 3 reads 92 B, up to 36 B written per transitioned record
        survey_bytes = int(n * (B_READ + B_READ_REMEDY) + n_res * B_READ_REMEDY + n * B_BITMAP + n_exc * B_EXC)
    else:
        alg_bytes = int(n * B_READ + n * B_BITMAP + n_exc * B_EXC + stats["n_stopped"] * B_STOP)
        model = f"N*{B_READ} + N/8 (bitmap) + exceptions*{B_EXC} + stopped*{B_STOP}"
    peak, peak_src = measured_peaks()
    traffic, traffic_src = ncu_traffic(config, n)

    # ---- e2e: the calls a cgo shim makes, host buffers both ways, real cadence ----
    # consecutive one-second ticks; the host closes the loop: every check the previous tick
    # submitted is posted back as Succeeded (H2D), then the tick runs and its due list is read in
    # host memory (D2H).  AM_SWEEP_FULL_SCAN keeps the device work per step identical to the
    # `value` step (all 56 B/record read on every tick).  At N>1 the step includes the NVLink
    # exchange and the read-back of this rank's part of the global list.
    if config == 2:
        ok_phase = np.full(n, am.PHASE_SUCCEEDED, dtype=np.uint8)
        sel = np.empty(n, dtype=np.uint64)
        prev = None
        reps = max(10, min(args.steps, 120))
        tick_no = 0
        h2d = d2h = 0
        h_part = torch.empty(n * 9 + 64, dtype=torch.uint8).pin_memory() if peer is not None and mode_gather == "exchange" else None
        c_loop = None
        if h_part is not None and not args.e2e_python_loop:
            # N>1: the same compiled loop; its tick is am_gather_tick_view — am_sweep_tick_shard + the NVLink exchange +
            # this rank's own part of the global list into pinned host memory, one synchronisation.  The ranks run their
            # loops side by side and meet in every exchange.
            workers = max(1, min(args.e2e_workers, len(os.sched_getaffinity(0)) - 1))
            peer.bind(sweep, stream.cuda_stream, gstream.cuda_stream)
            barrier()
            runs = []
            for r in range(3):
                runs.append(amgen.e2e_closed_loop(lib, sweep._h, T0 + r * (reps + 8), am.SWEEP_FULL_SCAN, 8, reps, n,
                                                  workers=workers, gather_handle=peer._h))
            c_loop = sorted(runs, key=lambda c: c["seconds"])[1]
            c_loop["runs_ms_per_step"] = [round(c["seconds"] / reps * 1e3, 4) for c in runs]
            dt, h2d, d2h = c_loop["seconds"], c_loop["h2d_bytes"], c_loop["d2h_bytes"]
            torch.cuda.synchronize()
            barrier()
        elif h_part is None:
            # N=1: the loop itself is compiled code calling the C-ABI, as the cgo shim is — ctypes and
            # numpy plumbing per call would otherwise be a tenth of the step
            workers = max(1, min(args.e2e_workers, len(os.sched_getaffinity(0)) - 1))
            # five runs of the loop, the median reported (all five are in the line): where the scheduler puts the
            # consumer threads relative to the pinned buffers moves a whole run by up to 1.7x (0.42 vs 0.73 ms seen)
            runs = []
            for r in range(5):
                runs.append(amgen.e2e_closed_loop(lib, sweep._h, T0 + r * (reps + 8), am.SWEEP_FULL_SCAN, 8, reps, n, workers=workers))
            c_loop = sorted(runs, key=lambda c: c["seconds"])[2]
            c_loop["runs_ms_per_step"] = [round(c["seconds"] / reps * 1e3, 4) for c in runs]
            dt, h2d, d2h = c_loop["seconds"], c_loop["h2d_bytes"], c_loop["d2h_bytes"]
        for phase_name in (() if c_loop else ("warm", "timed")):
            if phase_name == "timed":
                barrier()
                t0 = time.perf_counter()
                h2d = d2h = 0
            for k in range(5 if phase_name == "warm" else reps):
                if prev is not None and len(prev):
                    sweep.post_result(prev, ok_phase[: len(prev)])
                    h2d += len(prev) * 8 if phase_name == "timed" else 0
                if h_part is None:
                    vi, va, st = sweep.tick_view(T0 + tick_no, mode=am.SWEEP_FULL_SCAN)
                    # the checks just submitted, as local slots (compiled loop standing in for the
                    # Go shim's walk over the tick's result, hcc.go:269-288)
                    prev = amgen.select_submitted_view(vi, va, sel)
                    if phase_name == "timed":
                        d2h += len(vi) * 5 + 128
                else:
                    sweep.tick_shard(T0 + tick_no, am.SWEEP_FULL_SCAN, stream.cuda_stream)
                    peer.exchange(sweep, d_st.data_ptr(), stream.cuda_stream)
                    cnts = peer.counts().cpu()  # stream-ordered D2H of world+1 counts (synchronises)
                    off, mine_n = int(cnts[:rank].sum()), int(cnts[rank])
                    gi_d, ga_d = peer.buffers()
                    ib = gi_d.element_size()
                    h_idx = h_part[: mine_n * ib].view(gi_d.dtype)
                    h_act = h_part[n * 8: n * 8 + mine_n]
                    h_idx.copy_(gi_d[off: off + mine_n], non_blocking=True)
                    h_act.copy_(ga_d[off: off + mine_n], non_blocking=True)
                    stream.synchronize()
                    loc = (h_idx.numpy().astype(np.int64) & 0xFFFFFFFF).astype(np.uint32) - np.uint32(base & 0xFFFFFFFF) \
                        if ib == 4 else (h_idx.numpy() - base).astype(np.uint32)
                    prev = amgen.select_submitted_view(np.ascontiguousarray(loc), h_act.numpy(), sel)
                    if phase_name == "timed":
                        d2h += mine_n * (ib + 1) + (world + 1) * 4
                tick_no += 1
            if phase_name == "timed":
                barrier()
                dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        e2e = {"value": n * world * reps / dt, "unit": UNIT, "h2d_bytes_per_step": h2d // reps,
               "d2h_bytes_per_step": d2h // reps, "ms_per_step": dt / reps * 1e3, "steps": reps,
               "split_ms_per_step": None if not c_loop else {
                   "tick_view": c_loop["tick_s"] / reps * 1e3,
                   "consumer_wall": c_loop["consumer_s"] / reps * 1e3,
                   "post_result_per_worker": c_loop["post_s"] / reps * 1e3,
                   "walk_list_per_worker": c_loop["walk_s"] / reps * 1e3},
               "consumer_workers": c_loop["workers"] if c_loop else 1,
               "runs_ms_per_step": c_loop["runs_ms_per_step"] if c_loop else None,
               "host_cpus": (f"NUMA node {numa[0]} of the GPU ({len(numa[1])} CPUs)" if numa is not None else "unbound"),
               "driver": ("compiled loop calling the C-ABI (tools/amgen/amgen.c amgen_e2e_closed_loop): tick on one thread, "
                          "then the list walked in pieces and posted back by the consumer workers (the controller's "
                          "reconcile workers, hcc.go:170-188)") if c_loop
                         else "python loop (ctypes + torch)",
               "api": ("am_sweep_post_result + am_sweep_tick_view (the GPU writes the list into the library's pinned "
                       "host buffer)" if h_part is None else
                       ("am_sweep_post_result + am_gather_tick_view (am_sweep_tick_shard + the NVLink exchange + this rank's "
                        "own part of the global list extracted into pinned host memory, one synchronisation)" if c_loop else
                        "am_sweep_post_result + am_sweep_tick_shard + am_gather_exchange + read-back of this rank's "
                        "part of the global list")) + ", consecutive 1 s ticks, host-closed loop, AM_SWEEP_FULL_SCAN"}
    elif config == 3:
        # the host path of this step: post the 7.5 M pending results, tick, read the list
        fl = cols["flags"]
        pend = np.flatnonzero(fl & (am.F_PENDING_OK | am.F_PENDING_FAIL | am.F_REMEDY_PENDING)).astype(np.uint64)
        ph = np.where(fl[pend] & am.F_PENDING_OK, 1, np.where(fl[pend] & am.F_PENDING_FAIL, 2, 0)).astype(np.uint8)
        rp = np.where(fl[pend] & am.F_REMEDY_PENDING, np.where(fl[pend] & am.F_REMEDY_OUTCOME_OK, 1, 2), 0).astype(np.uint8)
        clear = ~np.uint32(am.F_PENDING_OK | am.F_PENDING_FAIL | am.F_REMEDY_PENDING | am.F_REMEDY_OUTCOME_OK)
        snap["flags"].copy_(torch.from_numpy((fl & clear).view(np.int32)).to(dev))
        reps, dt = max(5, min(args.steps, 20)), 0.0
        for k in range(reps + 2):
            restore()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            sweep.post_result(pend, ph, rp)
            vi, va, st = sweep.tick_view(T0)
            if k >= 2:
                dt += time.perf_counter() - t0
        assert st["n_emitted"] == stats["n_emitted"] and st["n_run_remedy"] == stats["n_run_remedy"], (st, stats)
        e2e = {"value": n * reps / dt, "unit": UNIT, "h2d_bytes_per_step": int(len(pend) * 8),
               "d2h_bytes_per_step": int(st["n_emitted"] * 5 + 128), "ms_per_step": dt / reps * 1e3, "steps": reps,
               "api": "am_sweep_post_result (every pending result of the step) + am_sweep_tick_view"}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu and config == 2:
        import oracle_c
        os.sched_setaffinity(0, all_cpus)  # the CPU arm gets every core the process was given
        threads = host_threads()
        host_cols = amgen.fill(config, seed, 0, n, T0, oracle_c.load().orc_classify, threads=min(threads, 64))
        t_mt = cpu_sweep_times(host_cols, T0, 0, threads, oracle_c, seconds=args.cpu_seconds)
        t_1t = cpu_sweep_times(host_cols, T0, 0, 1, oracle_c, seconds=min(4.0, args.cpu_seconds))
        # B1 "faithful shape": re-parse + Next() per evaluation, 100k-record subsample
        hcs, _, _ = amgen.healthchecks(config, seed, 0, 100_000, T0)
        import ctypes as C
        t0 = time.perf_counter()
        reps_b1 = 0
        while time.perf_counter() - t0 < 2.0:
            oracle_c.load().orc_faithful_eval(C.byref(hcs), 100_000, T0)
            reps_b1 += 1
        v_b1 = 100_000 * reps_b1 / (time.perf_counter() - t0)
        cpu = {"value": n / statistics.median(t_mt), "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"{len(t_mt)} ticks x {n} records (whole config-2 population), oracle sweep on {threads} "
                         "pinned threads; value = records / median tick",
               "best_tick_value": n / min(t_mt), "ms_per_tick_min": min(t_mt) * 1e3,
               "ms_per_tick_median": statistics.median(t_mt) * 1e3,
               "single_thread_value": n / statistics.median(t_1t),
               "faithful_shape_value": v_b1,
               "faithful_shape_note": "1 thread, re-parse cron + Next() per evaluation as hcc.go:253-262 does, 100k-record subsample"}

    if rank == 0:
        value = n * world * args.steps / (ms * 1e-3)
        par = f"index-range shards x{world}"
        if world > 1:
            par += {"exchange": ", global list on every GPU by the NVLink tick exchange (1 bit per record + non-default "
                                "actions on the wire, list rebuilt locally; overlapped with the next sweep)",
                    "plain": ", due lists concatenated by the round-1 plain peer-write push (5 B per entry on the wire; "
                             "overlapped with the next sweep)",
                    "nccl": ", padded NCCL all-gather of due lists"}[mode_gather]
        roof = None
        if k_ms is not None:
            achieved = alg_bytes / (k_ms * 1e-3) / 1e9
            roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                    "kernel": "sweep_tick_kernel<false,true>", "kernel_ms": k_ms, "algorithmic_bytes": alg_bytes,
                    "bytes_model": model,
                    **({"survey_bytes": survey_bytes, "survey_model": "SURVEY 8(d) literal: N*92 + transitioned*36 "
                        "+ N/8 + exceptions*4", "survey_frac": survey_bytes / (k_ms * 1e-3) / 1e9 / peak}
                       if config == 3 else {}),
                    "rest_of_tick": {"kernels": "scan_groups_kernel + expand_kernel + publish_kernel", "ms": c_ms,
                                     "bytes": int(n * B_BITMAP + stats["n_emitted"] * 5)},
                    "kernel_share_of_step": k_ms / (ms / args.steps),
                    "step_level": {"bytes": int(alg_bytes + n * B_BITMAP + stats["n_emitted"] * 5),
                                   "frac": (alg_bytes + n * B_BITMAP + stats["n_emitted"] * 5) / (ms / args.steps * 1e-3) / 1e9 / peak}}
        else:  # config 5: the step is the streaming tick; off-minute ticks read 16 B/record, not 56
            roof = {"bound": "hbm", "achieved": None, "peak": peak, "unit": "GB/s", "frac": None, "traffic": None,
                    "peak_source": peak_src, "kernel": "sweep_tick_kernel<true,*>",
                    "note": "59 of 60 ticks skip the 40 B/record of cron masks (no 5-field schedule can fire off the "
                            "minute) and are instruction-bound; see profiles/ for the per-variant captures"}
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "settle_steps": settle_steps, "ms_per_step": ms / args.steps,
            "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": WORKLOAD[config].format(n=n), "records_per_gpu": n, "records_total": n * world,
                       "l2": ("inputs (560 MB/GPU) larger than L2 (126 MB); no flush needed" if config != 3 else
                              "L2 flushed by a 256 MB read before every step"),
                       "parallelism": par,
                       "due_per_tick": stats["n_submit_hc"], "emitted_per_tick": stats["n_emitted"]},
            "roofline": roof,
            "cpu_baseline": cpu,
            "e2e": e2e,
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        if per_step_ms is not None:
            out["per_step_ms"] = {"min": min(per_step_ms), "median": statistics.median(per_step_ms), "max": max(per_step_ms)}
        if config == 2:
            out["host_issue_ms_per_step"] = host_issue_ms
        if verify is not None:
            out.update(verify)
        if config == 5 and blocking is not None:
            out["temporal_blocking"] = blocking
        if args.dump_outputs:
            write_outputs(args.dump_outputs, *last)
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        if peer is not None:
            peer.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
