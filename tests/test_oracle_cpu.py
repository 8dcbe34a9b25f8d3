"""CPU tests that PIN THE ORACLE: our plain-C restatement vs (a) the committed golden vectors produced by the reference
(tests/golden/make_golden.py) and (b) what the reference library itself (oracle/_ref) returned on seeded random models, recorded
under tests/golden/ref_results/ (tests/util.py RecordedReference).

These are the tests behind the "parity pinned" statement in oracle/xlinear_oracle.c and DESIGN.md.
"""
import json
import os

import numpy as np
import pytest
import scipy.sparse as smat

from pecos_b200 import synth

from .util import RecordedReference, assert_csr_parity, random_tree

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "xlinear_toy")


def _expected(E, key):
    return E[key + "|indptr"], E[key + "|indices"], E[key + "|data"]


@pytest.fixture(scope="module")
def golden(built):
    E = np.load(os.path.join(GOLD, "expected.npz"))
    index = json.load(open(os.path.join(GOLD, "expected_index.json")))
    Xt = smat.load_npz(os.path.join(GOLD, "Xt.npz")).tocsr().astype(np.float32)
    Xt.sort_indices()
    return E, index, Xt


def test_restatement_reproduces_reference_golden_vectors(golden):
    """Every (model, post-processor, beam, topk, csr|drm) entry recorded from the reference: ids, ranks AND score bits."""
    from oracle import restatement

    E, index, Xt = golden
    models = {}
    n = 0
    for item in index:
        name = item["model"]
        if name not in models:
            models[name] = restatement.OracleXLinear(os.path.join(GOLD, name, "ranker"))
        Xq = Xt if item["kind"] == "csr" else np.ascontiguousarray(Xt.toarray())
        got = models[name].predict(Xq, item["beam_size"] or 0, item["post_processor"], item["only_topk"] or 0)
        indptr, indices, data = _expected(E, item["key"])
        want = smat.csr_matrix((data, indices, indptr), shape=tuple(item["shape"]))
        exact = assert_csr_parity(got, want, rtol=0.0, what=item["key"])
        assert exact == 1.0
        n += 1
    assert n == len(index) and n >= 80


def test_default_prediction_matches_the_reference_repo_golden_file(golden):
    """tests/golden/xlinear_toy/Yt_pred_reference_golden.npy is the reference's own test/tst-data/xmc/xlinear/Yt_pred.npz
    (test_xlinear.py:366-370 compares with abs=1e-6)."""
    from oracle import restatement

    E, index, Xt = golden
    gold = np.load(os.path.join(GOLD, "Yt_pred_reference_golden.npy"))
    got = restatement.OracleXLinear(os.path.join(GOLD, "model", "ranker")).predict(Xt).toarray()
    assert np.abs(got - gold).max() <= 1e-6


@pytest.mark.parametrize("permute,prune,bias", [(False, 0.0, 1.0), (True, 0.0, 1.0), (True, 0.25, 1.0), (False, 0.0, -1.0)])
def test_restatement_equals_reference_library_on_random_trees(tmp_path, built, permute, prune, bias):
    from oracle import ref, restatement

    rec = RecordedReference(f"random_trees_{int(permute)}_{prune}_{bias}")
    folder = str(tmp_path / "m")
    layers = random_tree(5, [3, 18, 160], 220, 18, bias=bias, permute=permute, prune=prune)
    synth.save_xlinear_model(folder, layers, bias=bias, only_topk=6)
    X = synth.make_queries(6, 40, 220, 25)
    r = ref.RefXLinear(os.path.join(folder, "ranker")) if rec.recording else None
    o = restatement.OracleXLinear(os.path.join(folder, "ranker"))
    for pp in [None, "noop", "sigmoid", "log-sigmoid", "l2-hinge", "log-l3-hinge"]:
        for beam, topk in [(0, 0), (2, 3), (8, 8), (30, 200)]:
            a = rec.csr(f"csr {pp} {beam} {topk}", lambda: r.predict(X, beam, pp, topk))
            b = o.predict(X, beam, pp, topk)
            assert assert_csr_parity(b, a, rtol=0.0, what=f"csr {pp} {beam} {topk}") == 1.0
        a, b = rec.csr(f"drm {pp}", lambda: r.predict(X.toarray(), 4, pp, 5)), o.predict(X.toarray(), 4, pp, 5)
        assert assert_csr_parity(b, a, rtol=0.0, what=f"drm {pp}") == 1.0
    rec.save()


def test_reference_library_layer_types_agree(tmp_path, built):
    """BINARY_SEARCH_CHUNKED / HASH_CHUNKED / CSC return the same ids (reference test_xlinear.py:179-187); this is why
    the GPU engine serves all three requests from one layout.  The restatement returns them too."""
    from oracle import ref, restatement

    rec = RecordedReference("layer_types")
    folder = str(tmp_path / "m")
    synth.save_xlinear_model(folder, random_tree(9, [4, 30, 250], 300, 20), bias=1.0, only_topk=5)
    X = synth.make_queries(10, 30, 300, 30)
    base = rec.csr("BINARY_SEARCH_CHUNKED", lambda: ref.RefXLinear(os.path.join(folder, "ranker"), "BINARY_SEARCH_CHUNKED").predict(X, 5, None, 5))
    for t in ("HASH_CHUNKED", "CSC"):
        other = rec.csr(t, lambda: ref.RefXLinear(os.path.join(folder, "ranker"), t).predict(X, 5, None, 5))
        assert np.array_equal(base.indices, other.indices)
        assert np.allclose(base.data, other.data, atol=1e-6)
    rec.save()
    assert assert_csr_parity(restatement.OracleXLinear(os.path.join(folder, "ranker")).predict(X, 5, None, 5), base, rtol=0.0) == 1.0


@pytest.mark.parametrize("permute,prune", [(False, 0.0), (True, 0.25)])
def test_single_layer_restatement_equals_reference_library(built, permute, prune):
    """Next scope row (SURVEY 8f-2): c_xlinear_single_layer_predict_{csr,drm}_f32, the per-layer entry point of the python
    prediction chain (pecos/core/libpecos.cpp:201-235, pecos/xmc/base.py:890-949).  Pins the restatement
    (xlo_predict_from) bit-for-bit against oracle/_ref: with and without csr_codes, csr and dense queries, every kind of
    post-processor, previous-layer entries in NON-sorted stored order, empty code rows; and checks that chaining the
    single-layer calls reproduces the predict-only model (same arithmetic: bias + dot == dot + bias)."""
    from oracle import ref, restatement

    rec = RecordedReference(f"single_layer_{int(permute)}_{prune}")
    layers = random_tree(91, [5, 30, 240], 150, 20, bias=1.0, permute=permute, prune=prune)
    X = synth.make_queries(92, 40, 150, 25)
    rng = np.random.default_rng(93)
    prev = None
    for d, (W, C) in enumerate(layers):
        for pp in ["l3-hinge", "noop", "sigmoid", "log-sigmoid", "log-l2-hinge"]:
            for Xq in (X, X[:7].toarray()):
                codes = prev if (prev is None or isinstance(Xq, smat.csr_matrix)) else prev[:7]
                kind = "csr" if Xq is X else "drm"
                want = rec.csr(f"layer {d} {pp} {kind}", lambda: ref.single_layer_predict(Xq, codes, W, C, pp, 6, 1.0))
                got = restatement.single_layer_predict(Xq, codes, W, C, pp, 6, 1.0)
                assert_csr_parity(got, want, rtol=0.0, what=f"layer {d} {pp} {kind}")
        prev = rec.csr(f"beam {d}", lambda: ref.single_layer_predict(X, prev, W, C, "l3-hinge", 4, 1.0))
        # the beam is consumed in stored order: shuffle the entries inside every row and empty two rows
        lil = prev.tolil()
        lil.rows[3], lil.data[3] = [], []
        lil.rows[11], lil.data[11] = [], []
        shuffled = lil.tocsr().astype(np.float32)
        for r in range(shuffled.shape[0]):
            s, e = shuffled.indptr[r], shuffled.indptr[r + 1]
            perm = rng.permutation(e - s)
            shuffled.indices[s:e] = shuffled.indices[s:e][perm]
            shuffled.data[s:e] = shuffled.data[s:e][perm]
        shuffled.has_sorted_indices = False
        if d + 1 < len(layers):
            Wn, Cn = layers[d + 1]
            want = rec.csr(f"layer {d + 1} shuffled", lambda: ref.single_layer_predict(X, shuffled, Wn, Cn, "l3-hinge", 6, 1.0))
            got = restatement.single_layer_predict(X, shuffled, Wn, Cn, "l3-hinge", 6, 1.0)
            assert_csr_parity(got, want, rtol=0.0, what=f"layer {d + 1}, shuffled codes")
    # chain of single-layer calls == one predict-only call (beam 4, top-6 at the leaf)
    chain = None
    for d, (W, C) in enumerate(layers):
        chain = rec.csr(f"chain {d}", lambda: ref.single_layer_predict(X, chain, W, C, "l3-hinge", 6 if d == len(layers) - 1 else 4, 1.0))
    import tempfile

    with tempfile.TemporaryDirectory() as folder:
        synth.save_xlinear_model(folder, layers, bias=1.0, only_topk=6)
        full = rec.csr("predict-only", lambda: ref.RefXLinear(os.path.join(folder, "ranker")).predict(X, 4, "l3-hinge", 6))
    rec.save()
    assert_csr_parity(chain, full, rtol=0.0, what="python chain vs predict-only")


@pytest.mark.parametrize("permute", [False, True])
def test_selected_outputs_restatement_equals_reference_library(tmp_path, built, permute):
    """Next scope row (SURVEY 8f-2): c_xlinear_predict_on_selected_outputs_{csr,drm}_f32 (pecos/core/libpecos.cpp:179-198):
    scores of exactly the given (query, label) pairs through the hierarchy, no top-k, CSC layers only.  Pins the restatement
    (xlo_predict_selected) bit-for-bit: entry order (parents in the previous layer's order, children in C's column order),
    every kind of post-processor, csr and dense queries, empty rows."""
    from oracle import ref, restatement

    rec = RecordedReference(f"selected_outputs_{int(permute)}")
    folder = str(tmp_path / "m")
    layers = random_tree(95, [6, 40, 300], 200, 25, bias=1.0, permute=permute)
    synth.save_xlinear_model(folder, layers, bias=1.0, only_topk=6)
    X = synth.make_queries(96, 50, 200, 30)
    rng = np.random.default_rng(97)
    rows, cols = [], []
    for q in range(50):
        c = rng.choice(300, size=int(rng.integers(0, 12)), replace=False)  # some rows select nothing
        rows += [q] * len(c)
        cols += list(c)
    S = smat.csr_matrix((np.ones(len(rows), dtype=np.float32), (rows, cols)), shape=(50, 300))
    m = ref.RefXLinear(os.path.join(folder, "ranker"), weight_matrix_type="CSC") if rec.recording else None
    o = restatement.OracleXLinear(os.path.join(folder, "ranker"))
    for pp in [None, "noop", "sigmoid", "log-sigmoid", "l2-hinge", "log-l3-hinge"]:
        for Xq, Sq in ((X, S), (X.toarray()[:9], S[:9])):
            kind = "csr" if Xq is X else "drm"
            want = rec.csr(f"selected {pp} {kind}", lambda: ref.predict_on_selected_outputs(m, Xq, Sq, pp))
            got = o.predict_on_selected_outputs(Xq, Sq, pp)
            assert want.nnz == Sq.nnz
            assert_csr_parity(got, want, rtol=0.0, what=f"selected outputs {pp} {kind}")
    # consistency with beam search: a label returned by predict has the same score when selected explicitly
    full = rec.csr("beam 40", lambda: ref.RefXLinear(os.path.join(folder, "ranker")).predict(X, 40, None, 5))  # beam 40 = exhaustive at the middle layer
    sel_scores = rec.csr("selected beam 40", lambda: ref.predict_on_selected_outputs(m, X, smat.csr_matrix(full, dtype=np.float32), None))
    rec.save()
    a = smat.csr_matrix(full).toarray()
    b = sel_scores.toarray()
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
