"""Native manifest ingest (am_healthcheck_ingest_json, SURVEY 8f-2): JSON as the API server serves it ->
packed records, against (a) the ORACLE's ladder fed by an independent Python reading of the same documents
(json.loads + the field names of healthcheck_types.go) and (b) the reference's example / BDD manifests."""
import importlib
import json
import os
import random

import numpy as np
import pytest

from conftest import ROOT

ingest = importlib.import_module("active-monitor_b200.ingest")
am = importlib.import_module("active-monitor_b200")


def _oracle_record(orc, opy_unused, doc):
    """the oracle's classify on an independent reading of the document"""
    import ctypes as C
    kw = ingest.healthcheck_kwargs(doc)
    raw = kw["cron"].encode("utf-8", "surrogateescape")
    # orc_healthcheck_t / orc_record_t are layout-identical to the product's structs (sizes asserted in
    # the oracle): the ctypes declarations of active-monitor_b200._lib serve for both
    hc = am.abi.AmHealthCheck(kw["repeat_after_sec"], raw, len(raw), int(kw["has_resource"]), int(kw["has_remedy"]),
                              kw["remedy_runs_limit"], kw["remedy_reset_interval"], kw["finished_at"] or 0,
                              kw["remedy_finished_at"] or 0, int(kw["finished_at"] is not None),
                              int(kw["remedy_finished_at"] is not None), kw["success_count"], kw["failed_count"],
                              kw["remedy_success_count"], kw["remedy_failed_count"], kw["remedy_total_runs"], 0, 1)
    rec = am.abi.AmRecord()
    rc = orc.load().orc_classify(C.byref(hc), C.byref(rec))
    return rc, bytes(rec)


def _population(n, seed):
    rng = random.Random(seed)
    crons = ["", "@every 5s", "*/5 * * * *", "0 9 * * MON-FRI", "NOT_A_VALID_CRON", "@daily", "CRON_TZ=Europe/Paris 30 8 * * *",
             "0 0 1 1 *", "@every 1h30m", "*/15 9-17 * * 1-5", "\t5  4 * * *", "tab\there", "quote\"inside", "unié中\U0001F600"]
    docs = []
    for i in range(n):
        spec = {"workflow": {"generateName": f"wf-{i}-", "resource": None if rng.random() < 0.03 else {"namespace": "health", "source": {"inline": "x: {y: [1, 2, \"}\"]}"}}}}
        k = rng.random()
        if k < 0.4:
            spec["repeatAfterSec"] = rng.choice([5, 60, 300, 3600, 0, -1])
        if k > 0.3:
            spec["schedule"] = {"cron": rng.choice(crons)}
        if rng.random() < 0.5:
            rw = {}
            if rng.random() < 0.8:
                rw["generateName"] = "remedy-"
            if rng.random() < 0.8:
                rw["resource"] = {"namespace": "health"}
            if rng.random() < 0.3:
                rw["workflowtimeout"] = rng.choice([0, 30])
            if rng.random() < 0.2:
                rw["rbacRules"] = [] if rng.random() < 0.5 else None
            spec["remedyworkflow"] = rw
            spec["remedyRunsLimit"] = rng.choice([0, 1, 2, 5])
            spec["remedyResetInterval"] = rng.choice([0, 60, 300])
        doc = {"apiVersion": "activemonitor.keikoproj.io/v1alpha1", "kind": "HealthCheck",
               "metadata": {"name": f"hc-{i}", "namespace": "health", "annotations": {"note": "a \"quoted\" {brace} [bracket] \\ backslash"}},
               "spec": spec}
        if rng.random() < 0.7:
            st = {"successCount": rng.randrange(0, 1000), "failedCount": rng.randrange(0, 1000), "status": "Succeeded"}
            if rng.random() < 0.9:
                st["finishedAt"] = rng.choice(["2026-09-21T09:14:00Z", "2026-09-21T11:14:30+02:00", "2026-09-20T23:59:59.5Z", "2026-09-21T03:44:00-05:30"])
            if rng.random() < 0.4:
                rs, rf = rng.randrange(0, 4), rng.randrange(0, 4)
                st.update(remedySuccessCount=rs, remedyFailedCount=rf, remedyTotalRuns=rs + rf)
                if rs + rf:
                    st["remedyFinishedAt"] = "2026-09-21T09:10:00Z"
            doc["status"] = st
        docs.append(doc)
    return docs


@pytest.mark.parametrize("shape", ["list", "array", "single"])
def test_native_ingest_equals_the_oracle_ladder_on_an_independent_reading(orc, opy, shape):
    docs = _population(3000 if shape != "single" else 1, seed=5)
    text = {"list": json.dumps({"apiVersion": "v1", "kind": "List", "metadata": {"resourceVersion": ""}, "items": docs}, ensure_ascii=False, indent=1),
            "array": json.dumps(docs),  # ASCII-escaped: \\uXXXX incl. surrogate pairs
            "single": json.dumps(docs[0])}[shape]
    for threads in (1, 3):
        rcs, recs = ingest.ingest_json(text, n_threads=threads)
        assert len(recs) == len(docs)
        for i, doc in enumerate(docs):
            want_rc, want = _oracle_record(orc, opy, doc)
            assert int(rcs[i]) == want_rc, (i, doc)
            if want_rc in (0, am.AM_E_UNSUPPORTED):
                assert recs[i:i + 1].tobytes() == want, (i, doc)
    kinds = set(int(f) & 7 for f in recs["flags"])
    if shape != "single":
        assert {am.KIND_NO_RESOURCE, am.KIND_STOPPED, am.KIND_INTERVAL, am.KIND_CRON_SPEC, am.KIND_CRON_EVERY,
                am.KIND_PARSE_ERROR} <= kinds


def test_restart_semantics_and_errors():
    doc = {"kind": "HealthCheck", "spec": {"repeatAfterSec": 60, "workflow": {"resource": {}}}, "status": {"finishedAt": "2026-09-21T09:14:00Z"}}
    _, armed = ingest.ingest_json(json.dumps(doc), timer_armed=True)
    _, cold = ingest.ingest_json(json.dumps(doc), timer_armed=False)  # after a controller restart, hcc.go:161
    assert armed["flags"][0] & am.F_TIMER_ARMED and not cold["flags"][0] & am.F_TIMER_ARMED
    assert armed["finished_at"][0] == 1789982040
    rcs, _ = ingest.ingest_json(json.dumps([doc, {"spec": {"repeatAfterSec": "sixty"}}, {"status": {"finishedAt": "yesterday"}}]))
    assert rcs.tolist() == [0, am.AM_E_PARSE, am.AM_E_PARSE]
    for bad in ("", "nonsense", "[1, 2", '{"items": [}'):
        with pytest.raises(am.AmError):
            ingest.ingest_json(bad)
    rcs, recs = ingest.ingest_json("[]")
    assert len(recs) == 0


def test_reference_examples_through_the_native_ingest():
    with open(os.path.join(ROOT, "tests", "golden", "examples", "healthchecks.json"), encoding="utf-8") as f:
        docs = list(json.load(f).values())
    assert len(docs) >= 12
    rcs, recs = ingest.ingest_json(json.dumps({"kind": "List", "items": docs}))
    for i, doc in enumerate(docs):
        rc, rec = ingest.record_from_manifest(doc)
        assert int(rcs[i]) == rc and recs[i:i + 1].tobytes() == rec.tobytes(), doc["metadata"]["name"]
