"""CPU tests that PIN THE HNSW ORACLE: the plain-C restatement (oracle/hnsw_oracle.c) must reproduce, bit for bit, the
reference-recorded golden search results (ids, order, distance bits) of

* tests/golden/hnsw_toy  -- the reference's own 90-point, d = 2 fixture index (+ two indices trained by the reference), and
* tests/golden/hnsw_mid  -- reference-built indices with d in {768, 128, 70, 20}, both metrics, a six-fold duplicated index
  (exact ties), efS up to 600 (tests/golden/make_golden_hnsw.py).

The goldens were produced by the avx512f clone of the reference's distance kernels (provenance.json), restated as isa=0.
"""
import json
import os

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.mark.parametrize("suite", ["hnsw_toy", "hnsw_mid"])
def test_hnsw_restatement_reproduces_reference_goldens(built, suite):
    from oracle import restatement

    gold = os.path.join(HERE, "golden", suite)
    assert json.load(open(os.path.join(gold, "provenance.json")))["distance_isa_clone"] == "avx512f"
    E = np.load(os.path.join(gold, "expected.npz"))
    index = json.load(open(os.path.join(gold, "expected_index.json")))
    models, n = {}, 0
    for it in index:
        folder = os.path.join(gold, it["model"])
        m = models.get(it["model"]) or models.setdefault(it["model"], restatement.OracleHNSW(folder, isa=0))
        Q = np.load(os.path.join(folder, "Q.npy")) if suite == "hnsw_mid" else np.load(os.path.join(gold, "X.tst.npy"))
        idx, dist = m.predict(Q, it["efS"], it["topk"])
        assert np.array_equal(idx, E[it["key"] + "|idx"]), it["key"]
        assert np.array_equal(dist.view(np.uint32), E[it["key"] + "|dist"].view(np.uint32)), it["key"]
        n += 1
    assert n >= 20


def test_hnsw_mid_goldens_cover_the_simd_paths():
    """The fixture set must keep exercising: full 16-lane blocks (d >= 16), the 4-wide remainder and the scalar tail
    (d = 70 = 64 + 4 + 2), a large d (768), both metrics, and exact ties."""
    prov = json.load(open(os.path.join(HERE, "golden", "hnsw_mid", "provenance.json")))
    dims = {c["d"] for c in prov["cases"]}
    assert {768, 128, 70} <= dims
    assert {c["metric"] for c in prov["cases"]} == {"ip", "l2"}
    assert any(c["dup"] > 1 for c in prov["cases"])
    assert max(e for e, _ in prov["grid"]) >= 600


SPARSE = os.path.join(HERE, "golden", "hnsw_sparse")


def test_sparse_hnsw_restatement_reproduces_reference_goldens(built):
    """Sparse (csr) indices, tests/golden/make_golden_hnsw_sparse.py: the reference's own prebuilt sparse fixture index and three
    reference-built ones (ip / l2 -- the reference's sparse "l2" is -2<x,y> --, rows shorter than the 4-wide intersection blocks,
    empty rows, a query row longer than every stored row): ids, order and distance bits."""
    import scipy.sparse as smat

    from oracle import restatement

    E = np.load(os.path.join(SPARSE, "expected.npz"))
    index = json.load(open(os.path.join(SPARSE, "expected_index.json")))
    models, n = {}, 0
    for it in index:
        folder = os.path.join(SPARSE, it["model"])
        m = models.get(it["model"]) or models.setdefault(it["model"], restatement.OracleHNSW(folder, isa=0))
        assert m.sparse
        Q = smat.load_npz(os.path.join(folder, "Q.npz"))
        idx, dist = m.predict(Q, it["efS"], it["topk"])
        assert np.array_equal(idx, E[it["key"] + "|idx"]), it["key"]
        assert np.array_equal(dist.view(np.uint32), E[it["key"] + "|dist"].view(np.uint32)), it["key"]
        n += 1
    assert n >= 20 and {it["model"] for it in index} >= {"fixture_ip", "ip_tfidf", "l2_tfidf", "ip_short"}


def test_sparse_hnsw_restatement_equals_the_reference_library_on_random_indices(built):
    """Diff against oracle/_ref on sparse indices it trained from seeded random rows (both metrics; indices and search results
    recorded under tests/golden/ref_results/), incl. recall of the reference's own test (test/pecos/ann/test_hnsw.py:86-124: recall
    vs brute force >= 0.99 on the prebuilt sparse fixture)."""
    import scipy.sparse as smat

    from oracle import ref, restatement

    from .util import RecordedReference

    rec = RecordedReference("hnsw_sparse_random")
    # the restatement follows the distance kernels of the host the reference ran on
    isa = int(rec.arrays("isa", lambda: (np.int64(restatement.host_isa()),))[0])

    sys_path_golden = os.path.join(HERE, "golden")
    import importlib.util

    spec = importlib.util.spec_from_file_location("mgs", os.path.join(sys_path_golden, "make_golden_hnsw_sparse.py"))
    mgs = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mgs)
    for metric, (N, D, nnz) in (("ip", (1200, 3000, 30)), ("l2", (900, 200, 12))):
        X = mgs.make_rows(7, N, D, nnz, 50)
        Q = mgs.make_rows(8, 40, D, nnz, 9)
        r = ref.RefHNSW.train(X, M=8, efC=40, metric=metric, threads=1) if rec.recording else None

        def write(folder):
            r.save(os.path.join(folder, "c_model"))
            json.dump({"data_type": "csr", "metric_type": metric}, open(os.path.join(folder, "param.json"), "w"))

        o = restatement.OracleHNSW(rec.folder(metric, write), isa=isa)
        assert abs(o.vectors() - X).max() == 0
        for efS, topk in ((30, 10), (120, 20)):
            a, b = o.predict(Q, efS, topk), rec.arrays(f"{metric} {efS} {topk}", lambda: r.predict(Q, efS, topk))
            assert np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32))
    rec.save()
    # recall on the reference's fixture
    fx = os.path.join(SPARSE, "fixture_ip")
    o = restatement.OracleHNSW(fx, isa=0)
    Xtrn = o.vectors()
    Q = smat.load_npz(os.path.join(fx, "Q.npz"))
    exact = np.argsort(1.0 - (Q @ Xtrn.T).toarray(), axis=1, kind="stable")[:, :10]
    for efS in (50, 75, 100):
        idx, _ = o.predict(Q, efS, 10)
        recall = np.mean([len(set(idx[i]) & set(exact[i])) / 10.0 for i in range(Q.shape[0])])
        assert recall >= 0.99
