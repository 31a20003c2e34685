"""The reference's own example / BDD manifests through the product's ladder
(SURVEY.md section 8f-2).  The manifests are stored as JSON in
tests/golden/examples/healthchecks.json, keyed by their path under the reference's examples/."""
import importlib
import json
import os

from conftest import ROOT

EXAMPLES = os.path.join(ROOT, "tests", "golden", "examples", "healthchecks.json")


def _docs():
    with open(EXAMPLES, encoding="utf-8") as f:
        return json.load(f)


def test_every_example_classifies(am):
    ingest = importlib.import_module("active-monitor_b200.ingest")
    docs = _docs()
    assert len(docs) >= 12
    kinds = {}
    for name, doc in docs.items():
        rc, rec = ingest.record_from_manifest(doc)
        assert rc == 0, name
        kinds[name] = (int(rec["flags"][0]) & 7, int(rec["ras"][0]), bool(rec["flags"][0] & am.F_HAS_REMEDY))
    # examples/inlineHello.yaml:8-10 ships `cron: "@every 1m"` with repeatAfterSec commented out
    assert kinds["inlineHello.yaml"] == (am.KIND_CRON_EVERY, 60, False)
    assert kinds["inlineHello_cluster.yaml"] == (am.KIND_INTERVAL, 60, False)
    # despite its name this manifest carries neither repeatAfterSec nor schedule: the
    # reference's pause rule (hcc.go:238) stops it, and so does the product's ladder
    assert kinds["inlineHello_cluster_cron_repeat.yaml"][0] == am.KIND_STOPPED
    assert kinds["inlineHello_cluster_cron.yaml"] == (am.KIND_CRON_EVERY, 60, False)
    # envtest fixtures (healthcheck_controller_test.go)
    assert kinds["bdd/inlineHelloTest.yaml"][0] == am.KIND_STOPPED          # repeatAfterSec: 0 -> "Stopped"
    assert kinds["bdd/inlineCustomBackoffTest.yaml"] == (am.KIND_CRON_EVERY, 3, False)
    assert kinds["bdd/inlineMemoryRemedyUnitTest_Namespace.yaml"][:2] == (am.KIND_CRON_EVERY, 5)
    rem = docs["bdd/inlineMemoryRemedyUnitTest.yaml"]
    rc, rec = ingest.record_from_manifest(rem)
    assert kinds["bdd/inlineMemoryRemedyUnitTest.yaml"] == (am.KIND_INTERVAL, 5, True)
    assert (int(rec["runs_limit"][0]), int(rec["reset_interval"][0])) == (2, 300)
    # every manifest with a remedyworkflow block is non-empty, the others are empty
    for name, doc in docs.items():
        assert kinds[name][2] == bool((doc.get("spec") or {}).get("remedyworkflow")), name


def test_batch_classifier_equals_per_record_calls_on_the_examples(am):
    ingest = importlib.import_module("active-monitor_b200.ingest")
    docs = list(_docs().values())
    rcs, recs = ingest.classify_batch(docs, n_threads=3)
    assert len(recs) == len(docs)
    for i, doc in enumerate(docs):
        rc, rec = ingest.record_from_manifest(doc)
        assert rc == int(rcs[i])
        assert rec.tobytes() == recs[i:i + 1].tobytes()
