"""bench.py's JSON line and its --dump-outputs files.  The reference arm runs on CPU: pin the JSON line's
contract here (the GPU arm's line has the same keys plus roofline / clocks).  The files either arm dumps
must be the last timed step's outputs: the oracle's tick of the same seeded population."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from conftest import ROOT
from oracle_c import STAT_FIELDS


def _run(*args, env=None):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         timeout=300, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    return out.stdout.strip().splitlines()


def _oracle_last_tick(orc, gen, config, n, ticks):
    """the oracle's list and statistics of the last of `ticks` ticks, as bench.py steps that config"""
    T0 = gen.T0_DAY_START if config == 5 else gen.T0_MON_0915
    seed = bench.CONFIG_SEED[config]
    cols = gen.fill(config, seed, 0, n, T0, orc.load().orc_classify)
    for k in range(ticks):  # config 5 steps through consecutive seconds, closed loop; 2 and 3 repeat T0
        idx, act, st = orc.sweep(cols, T0 + k if config == 5 else T0, mode=1 if config == 5 else 0, seed=seed)
    return idx, act, st


def _check_dump(d, idx, act, st, with_list=True):
    files = sorted(os.listdir(d))
    assert files == (["due_action.npy", "due_index.npy", "stats.npy"] if with_list else ["stats.npy"])
    assert sum(os.path.getsize(os.path.join(d, f)) for f in files) <= bench.DUMP_BYTES
    got = {f[:-4]: np.load(os.path.join(d, f)) for f in files}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert got["stats"].tolist() == [float(st[f]) for f in STAT_FIELDS]
    if with_list:
        np.testing.assert_array_equal(got["due_index"], idx.astype(np.float64))
        np.testing.assert_array_equal(got["due_action"], act.astype(np.float32))


def test_reference_arm_json_line():
    lines = _run("--impl", "reference", "--steps", "3", "--warmup", "1", "--n", "200000")
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "healthcheck_schedule_evals_per_sec"
    assert d["unit"] == "evals/s" and d["higher_is_better"] is True and d["steps"] == 3
    assert d["value"] > 1e5 and abs(d["ms_per_step"] * 1e-3 * d["value"] - 200000) < 1
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and d["dtype"] == "u64"
    assert set(d["cpu_baseline"]) >= {"value", "unit", "cores", "kind", "sample"}
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0))
    assert d["e2e"] == {"value": d["value"], "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_print_nothing():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    assert _run("--impl", "reference", "--gpus", "2", "--steps", "2", "--warmup", "1", "--n", "50000", env=env) == []


def test_reference_arm_dumps_its_last_step(orc, gen, tmp_path):
    n = 200_000
    _run("--impl", "reference", "--steps", "2", "--warmup", "1", "--n", str(n), "--dump-outputs", str(tmp_path))
    _check_dump(tmp_path, *_oracle_last_tick(orc, gen, 2, n, 2))


def test_a_long_list_is_dumped_as_the_same_seeded_sample(tmp_path):
    n = bench.DUMP_BYTES // 12 + 12345
    idx = np.arange(n, dtype=np.uint32) * 3
    act = (np.arange(n) % 7 + 1).astype(np.uint8)
    for run in ("a", "b"):
        bench.write_outputs(str(tmp_path / run), np.arange(16), idx, act)
        assert sum(os.path.getsize(tmp_path / run / f) for f in os.listdir(tmp_path / run)) <= bench.DUMP_BYTES
    a, b = (np.load(tmp_path / run / "due_index.npy") for run in ("a", "b"))
    assert len(a) < n and np.array_equal(a, b) and (np.diff(a) > 0).all()
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "due_action.npy"), (a / 3) % 7 + 1)


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=60)
    assert out.returncode == 2 and "--steps" in out.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("config", [2, 3, 5])
def test_gpu_arm_dumps_its_last_step(orc, gen, tmp_path, config):
    n, steps = 200_000, 3
    lines = _run("--config", str(config), "--steps", str(steps), "--warmup", "1", "--n", str(n), "--no-cpu",
                 "--settle-ms", "0", "--dump-outputs", str(tmp_path))
    d = json.loads(lines[-1])
    assert d["steps"] == steps
    # config 2 repeats T0 ("Stopped" is reported on the first tick only); config 3 restores its state before
    # every step; config 5 runs the warm-up ticks (at least 3) and the timed ones as consecutive seconds
    idx, act, st = _oracle_last_tick(orc, gen, config, n, {2: 2, 3: 1, 5: 3 + steps}[config])
    _check_dump(tmp_path, idx, act, st, with_list=config != 5)
