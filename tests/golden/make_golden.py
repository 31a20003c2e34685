"""Generate the committed golden fixtures (tests/golden/*.json).

There is no executable reference here (Go, no toolchain), so these vectors are
NOT outputs of the reference: they are outputs of the C oracle, accepted only
when the independent Python oracle reproduces them, frozen so that later edits
to either oracle or to the kernel are checked against a fixed point.
Re-run:  python tests/golden/make_golden.py

examples/healthchecks.json holds the HealthCheck manifests of active-monitor's
examples/ directory (Apache-2.0), converted from YAML to JSON and keyed by their
path there, so that the ingest tests need no checkout of that project.
Re-run:  python tests/golden/make_golden.py --examples <active-monitor>/examples
"""
import hashlib
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tools", "amgen")):
    sys.path.insert(0, p)
import numpy as np  # noqa: E402
import amgen  # noqa: E402
import oracle_c  # noqa: E402
import oracle_py  # noqa: E402

for _z in amgen.ZONES:  # zone ids in the generator's order in every implementation
    oracle_py.tz_lookup(_z)
T0, T_OCT1 = 1789982100, 1790812800
CASES = [  # name, config, seed, n, ticks [(T, mode)]
    ("config1_ras60", 1, 1, 1000, [(T0, 0)]),
    ("config1_every1m", 11, 1, 1000, [(T0, 0)]),
    ("config2_mixed", 2, 2, 4000, [(T0, 0), (T0 + 1, 0), (T_OCT1, 0)]),
    ("config22_zones", 22, 2, 4000, [(T0, 0), (1790013600, 0), (1793512800, 0)]),  # + 2026-09-21T18:00Z, 2026-11-01T06:00Z (New York falls back)
    ("config3_remedy", 3, 3, 4000, [(T0, 0), (T0 + 60, 0)]),
    ("config5_closed_loop", 55, 5, 1500, [(T0 - 2 + k, 1) for k in range(64)]),
]


def columns_digest(cols):
    h = hashlib.sha256()
    for name, _ in oracle_c.COLUMNS:
        h.update(np.ascontiguousarray(cols[name]).tobytes())
    return h.hexdigest()


def main():
    for name, config, seed, n, ticks in CASES:
        cols = amgen.fill(config, seed, 0, n, T0, oracle_c.load().orc_classify)
        recs = [oracle_py.Record(**{c: int(cols[c][i]) for c, _ in oracle_c.COLUMNS}) for i in range(n)]
        out = {"config": config, "seed": seed, "n": n, "T0": T0,
               "initial_columns_sha256": columns_digest(cols), "ticks": []}
        for T, mode in ticks:
            idx, act, st = oracle_c.sweep(cols, T, mode=mode, seed=seed)
            due_py, st_py = oracle_py.sweep(recs, T, mode=mode, seed=seed)
            assert [(int(a), int(b)) for a, b in zip(idx, act)] == due_py, (name, T)
            for k, v in st.items():
                assert getattr(st_py, k) == v, (name, T, k)
            entry = {"T": T, "mode": mode, "stats": st, "columns_sha256": columns_digest(cols)}
            if len(idx) <= 2500:
                entry["idx"] = [int(v) for v in idx]
                entry["act"] = [int(v) for v in act]
            else:
                entry["idx_act_sha256"] = hashlib.sha256(idx.tobytes() + act.tobytes()).hexdigest()
            out["ticks"].append(entry)
        for i in range(n):
            for c, _ in oracle_c.COLUMNS:
                assert int(cols[c][i]) == getattr(recs[i], c), (name, i, c)
        with open(os.path.join(HERE, name + ".json"), "w") as f:
            json.dump(out, f, separators=(",", ":"))
        print(name, "ok", [t["stats"]["n_emitted"] for t in out["ticks"]][:6])


def examples(src):
    import glob
    import yaml
    docs = {}
    for path in sorted(glob.glob(os.path.join(src, "**", "*.yaml"), recursive=True)):
        for doc in yaml.safe_load_all(open(path)):
            if isinstance(doc, dict) and doc.get("kind") == "HealthCheck":
                docs[os.path.relpath(path, src)] = doc
    os.makedirs(os.path.join(HERE, "examples"), exist_ok=True)
    with open(os.path.join(HERE, "examples", "healthchecks.json"), "w") as f:
        json.dump(docs, f, indent=1, ensure_ascii=False)
        f.write("\n")
    print("examples ok", len(docs))


if __name__ == "__main__":
    if sys.argv[1:2] == ["--examples"]:
        examples(sys.argv[2])
    else:
        main()
