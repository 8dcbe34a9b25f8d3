"""CPU tests of the host-side logic: C-ABI surface, model ingest (npz / mmap readers, chunk layout), Python mirror."""
import os
import re
import subprocess

import numpy as np
import pytest
import scipy.sparse as smat

from pecos_b200 import synth

from .util import random_tree

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "xlinear_toy")


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "pecos_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b((?:c_xlinear|c_ann_hnsw|pb200)_[A-Za-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(clib):
    names = _declared_symbols()
    assert len(names) >= 30
    out = subprocess.run(["nm", "-D", "--defined-only", clib.path], stdout=subprocess.PIPE, text=True, check=True).stdout
    exported = set(line.split()[-1] for line in out.splitlines() if line.strip())
    missing = [n for n in names if n not in exported]
    assert not missing, f"declared in include/pecos_b200.h but not exported: {missing}"
    for n in names:
        assert hasattr(clib.clib_float32, n)


def test_no_gpu_means_loud_failure_not_fallback(clib, tmp_path):
    if clib.device_count() > 0:
        pytest.skip("a GPU is visible here")
    from pecos_b200.xlinear import XLinearModel

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        XLinearModel.load(os.path.join(GOLD, "model"), is_predict_only=True)
    # the python chain keeps W / C on the host like the reference (loading needs no GPU), predicting raises loudly
    chain = XLinearModel.load(os.path.join(GOLD, "model"), is_predict_only=False)
    assert not chain.is_predict_only and chain.depth >= 1
    X = np.zeros((1, chain.nr_features), dtype=np.float32)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        chain.predict(X)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "pecos_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".h", ".cpp", ".cuh")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f"{f} imports the oracle"
                assert "liboracle" not in text and "oracle/_ref" not in text, f"{f} references the oracle"


def _check_layout(layers, Ws, Cs, bias):
    """Structural properties of the HBM chunk layout + exact content vs the source CSC matrices."""
    for d, L in enumerate(layers):
        W, C = smat.csc_matrix(Ws[d]), smat.csc_matrix(Cs[d])
        chunks, meta, ent = L["chunks"], L["meta"], L["entries"]
        assert L["n_chunks"] == C.shape[1]
        assert L["n_cols"] == C.nnz
        assert L["out_cols"] == C.shape[0]
        contiguous = C.nnz >= C.shape[0] and np.array_equal(C.indices, np.arange(C.nnz))
        assert (len(L["label_of_col"]) == 0) == contiguous
        col_cursor = 0
        dense_W = W.toarray()
        for p in range(L["n_chunks"]):
            h = chunks[p]
            R, nc = int(h["nnz_rows"]), int(h["n_cols"])
            assert int(h["col_begin"]) == col_cursor
            col_cursor += nc
            assert int(h["meta_off"]) % 4 == 0  # 16-byte aligned row-index list for 128-bit loads
            rows = meta[int(h["meta_off"]): int(h["meta_off"]) + R].astype(np.int64)
            R4 = (R + 3) // 4 * 4
            assert (meta[int(h["meta_off"]) + R: int(h["meta_off"]) + R4] == 0xFFFFFFFF).all()
            rp = meta[int(h["meta_off"]) + R4: int(h["meta_off"]) + R4 + R + 1].astype(np.int64)
            assert (np.diff(rows) > 0).all()           # sorted, distinct
            assert rp[0] == 0 and (np.diff(rp) > 0).all()
            cols = (np.arange(nc) + int(h["col_begin"]))
            labels = L["label_of_col"][cols] if len(L["label_of_col"]) else cols
            sub = dense_W[:, labels]                    # (w_rows, nc) block of the source matrix
            want_rows = np.nonzero((sub != 0).any(axis=1))[0]
            assert np.array_equal(rows, want_rows)
            e = ent[int(h["ent_off"]): int(h["ent_off"]) + rp[-1]]
            rebuilt = np.zeros_like(sub)
            for i, r in enumerate(rows):
                seg = e[rp[i]: rp[i + 1]]
                assert (np.diff(seg["col_offset"].astype(np.int64)) > 0).all()
                rebuilt[r, seg["col_offset"]] = seg["val"]
            assert np.array_equal(rebuilt, sub)
            has_bias = bias > 0 and R > 0 and rows[-1] == W.shape[0] - 1
            assert bool(h["has_bias"]) == bool(has_bias)
        assert col_cursor == L["n_cols"]


@pytest.mark.parametrize("permute,prune,bias", [(False, 0.0, 1.0), (True, 0.0, 1.0), (True, 0.3, 1.0), (False, 0.0, -1.0)])
def test_chunk_layout_from_npz(clib, tmp_path, permute, prune, bias):
    folder = str(tmp_path / "m")
    layers = random_tree(3, [3, 14, 90], 120, 12, bias=bias, permute=permute, prune=prune)
    synth.save_xlinear_model(folder, layers, bias=bias, only_topk=4)
    got = clib.host_model_layout(os.path.join(folder, "ranker"), is_mmap=False)
    _check_layout(got, [w for w, _ in layers], [c for _, c in layers], bias)


def test_root_layer_without_C_file(clib, tmp_path):
    folder = str(tmp_path / "m")
    layers = random_tree(4, [5, 40], 64, 8, bias=1.0)
    synth.save_xlinear_model(folder, layers, bias=1.0, only_topk=4, skip_root_C=True)
    assert not os.path.exists(os.path.join(folder, "ranker", "0.model", "C.npz"))
    got = clib.host_model_layout(os.path.join(folder, "ranker"))
    assert got[0]["n_chunks"] == 1 and got[0]["n_cols"] == 5


def test_mmap_reader_repacks_to_the_same_layout_as_the_npz_builder(clib):
    """tests/golden/xlinear_toy/model_mmap was written by the reference's c_xlinear_compile_mmap_model."""
    a = clib.host_model_layout(os.path.join(GOLD, "model", "ranker"), is_mmap=False)
    b = clib.host_model_layout(os.path.join(GOLD, "model_mmap", "ranker"), is_mmap=True)
    assert len(a) == len(b) >= 2
    for la, lb in zip(a, b):
        for k in ("w_rows", "n_cols", "out_cols", "n_chunks", "c_max"):
            assert la[k] == lb[k]
        for k in ("chunks", "meta", "entries", "label_of_col"):
            assert np.array_equal(la[k], lb[k]), k


def test_npz_reader_dtype_conversion_and_compressed_rejection(clib, tmp_path):
    # int64 indices / float64 data are converted (scipy_loader.hpp:153-184); compressed archives are rejected (:247-249)
    folder = str(tmp_path / "m")
    layers = random_tree(8, [4, 30], 50, 6, bias=1.0)
    synth.save_xlinear_model(folder, layers, bias=1.0, only_topk=4)
    base = clib.host_model_layout(os.path.join(folder, "ranker"))
    wpath = os.path.join(folder, "ranker", "1.model", "W.npz")
    W = smat.load_npz(wpath).tocsc()
    W64 = smat.csc_matrix((W.data.astype(np.float64), W.indices.astype(np.int64), W.indptr.astype(np.int64)), shape=W.shape)
    with open(wpath, "wb") as f:
        smat.save_npz(f, W64, compressed=False)
    again = clib.host_model_layout(os.path.join(folder, "ranker"))
    assert np.array_equal(base[1]["entries"], again[1]["entries"]) and np.array_equal(base[1]["meta"], again[1]["meta"])
    # a compressed archive must be refused loudly: run in a child process because the C ABI aborts
    with open(wpath, "wb") as f:
        smat.save_npz(f, W, compressed=True)
    code = ("import sys; sys.path.insert(0, %r); from pecos_b200 import core; "
            "core.get_clib().host_model_layout(%r)" % (ROOT, os.path.join(folder, "ranker")))
    r = subprocess.run(["python", "-c", code], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode != 0 and "compressed" in r.stderr


def test_pred_params_override_semantics():
    """beam_size -> only_topk of all non-final layers, only_topk -> final layer (pecos/xmc/base.py:1158-1166)."""
    from pecos_b200.xlinear import HierarchicalPredParams, MLModelPredParams

    p = HierarchicalPredParams(model_chain=[MLModelPredParams(20, "l3-hinge") for _ in range(3)])
    p.override_with_kwargs({"beam_size": 7, "only_topk": 3, "post_processor": "sigmoid"})
    assert [m.only_topk for m in p.model_chain] == [7, 7, 3]
    assert all(m.post_processor == "sigmoid" for m in p.model_chain)
    with pytest.raises(TypeError):
        p.override_with_kwargs([1, 2])


def test_ctypes_views_keep_reference_struct_layout():
    import ctypes

    from pecos_b200.core import ScipyCsrF32, ScipyDrmF32

    assert ctypes.sizeof(ScipyCsrF32) == 32 and ctypes.sizeof(ScipyDrmF32) == 16  # matrix.hpp:49-71
    X = synth.make_queries(1, 5, 20, 4)
    v = ScipyCsrF32.init_from(X)
    assert (v.rows, v.cols) == (5, 20) and v.indptr[5] == X.nnz
    with pytest.raises(ValueError):
        ScipyCsrF32.init_from(X.astype(np.float64))


@pytest.mark.parametrize("permute,prune,bias", [(False, 0.0, 1.0), (True, 0.3, 1.0), (False, 0.0, -1.0)])
def test_single_layer_model_from_in_memory_csc_equals_the_folder_loader(clib, tmp_path, permute, prune, bias):
    """c_xlinear_single_layer_predict_* receives W and C as in-memory CSC matrices (pecos/core/libpecos.cpp:201-235); the
    one-layer host model built from them must be the layer the npz loader builds."""
    folder = str(tmp_path / "m")
    layers = random_tree(13, [4, 18, 120], 90, 10, bias=bias, permute=permute, prune=prune)
    synth.save_xlinear_model(folder, layers, bias=bias, only_topk=4)
    from_folder = clib.host_model_layout(os.path.join(folder, "ranker"))
    for d, (W, C) in enumerate(layers):
        got = clib.host_layer_layout_from_csc(W, C, bias)
        assert len(got) == 1
        for k in ("w_rows", "n_cols", "out_cols", "n_chunks", "c_max"):
            assert got[0][k] == from_folder[d][k], k
        for k in ("chunks", "meta", "entries", "label_of_col"):
            assert np.array_equal(got[0][k], from_folder[d][k]), k
    _check_layout([clib.host_layer_layout_from_csc(*layers[-1], bias)[0]], [layers[-1][0]], [layers[-1][1]], bias)


@pytest.mark.parametrize("permute,prune,bias", [(False, 0.0, 1.0), (True, 0.25, 1.0), (False, 0.0, -1.0)])
def test_mmap_writer_output_loads_in_the_reference_library(tmp_path, clib, have_ref, permute, prune, bias):
    """c_xlinear_compile_mmap_model of THIS library (host-only writer, pecos_b200/csrc/xlinear_host.h write_xlinear_mmap_model):
    our own mmap loader must read the folder it writes back to the same chunked layout as the npz model and as the folder the
    REFERENCE's own writer makes from it (recorded under tests/golden/ref_results/), and -- where oracle/_ref is built -- the
    reference library must load it and predict exactly what it predicts from the npz model."""
    from .util import RecordedReference, assert_csr_parity, random_tree

    rec = RecordedReference(f"mmap_writer_{int(permute)}_{prune}_{bias}")

    folder = str(tmp_path / "m")
    layers = random_tree(77, [5, 30, 400], 300, 20, bias=bias, permute=permute, prune=prune)
    synth.save_xlinear_model(folder, layers, bias=bias, only_topk=7, post_processor="l2-hinge")
    ours = str(tmp_path / "ours")
    clib.clib_float32.c_xlinear_compile_mmap_model(os.path.join(folder, "ranker").encode(), os.path.join(ours, "ranker").encode())
    a = clib.host_model_layout(os.path.join(folder, "ranker"))
    b = clib.host_model_layout(os.path.join(ours, "ranker"), is_mmap=True)
    assert len(a) == len(b)
    for la, lb in zip(a, b):
        for key in la:
            assert np.array_equal(np.asarray(la[key]), np.asarray(lb[key])), key
    from oracle import ref

    if have_ref:
        X = synth.make_queries(78, 60, 300, 25)
        want = ref.RefXLinear(os.path.join(folder, "ranker")).predict(X, 6, None, 5)
        got = ref.RefXLinear(os.path.join(ours, "ranker"), is_mmap=True).predict(X, 6, None, 5)
        assert_csr_parity(got, want, rtol=0.0, what="reference library on the folder written by pecos_b200")

    def write(path):
        os.makedirs(path)
        ref.compile_mmap_model(os.path.join(folder, "ranker"), os.path.join(path, "ranker"))

    theirs = rec.folder("theirs", write)
    rec.save()
    c = clib.host_model_layout(os.path.join(theirs, "ranker"), is_mmap=True)
    assert len(c) == len(b)
    for lb, lc in zip(b, c):
        for key in lb:
            assert np.array_equal(np.asarray(lb[key]), np.asarray(lc[key])), key


def test_hnsw_host_ingest_of_dense_and_sparse_indices(clib):
    """The C++ loader (pecos_b200/csrc/hnsw_host.h) on the committed reference-built indices, without a GPU: header fields, record
    walk and totals agree with the independent numpy parse of the oracle; a folder of the wrong index type is rejected."""
    from ctypes import c_uint64

    from oracle import restatement

    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    c = clib.clib_float32
    cases = [("hnsw_toy/model_ip", 0, 0), ("hnsw_mid/l2_d128", 1, 0), ("hnsw_mid/ip_d70", 0, 0), ("hnsw_sparse/fixture_ip", 0, 1),
             ("hnsw_sparse/ip_tfidf", 0, 1), ("hnsw_sparse/l2_tfidf", 1, 1), ("hnsw_sparse/ip_short", 0, 1)]
    for rel, metric, sparse in cases:
        folder = os.path.join(gold, rel)
        out = (c_uint64 * 8)()
        assert c.pb200_hnsw_host_info(os.path.join(folder, "c_model").encode(), metric, sparse, out) == 0, rel
        o = restatement.OracleHNSW(folder, isa=0)
        assert [int(x) for x in out[:6]] == [o.num_node, o.feat_dim, o.maxM, o.maxM0, o.max_level, o.init_node], rel
        V = o.vectors()
        assert int(out[6]) == (V.nnz if sparse else V.size), rel
        # wrong metric / wrong data type: the hnsw_t string of config.json does not match (hnsw.hpp:541-546)
        assert c.pb200_hnsw_host_info(os.path.join(folder, "c_model").encode(), 1 - metric, sparse, out) == 1
        assert c.pb200_hnsw_host_info(os.path.join(folder, "c_model").encode(), metric, 1 - sparse, out) == 1


@pytest.mark.parametrize("permute,prune", [(False, 0.0), (True, 0.25)])
def test_mlmodel_mmap_writer_is_interchangeable_with_the_reference(tmp_path, clib, have_ref, permute, prune):
    """c_mlmodel_compile_mmap_model of THIS library (host-only; pecos_b200/csrc/xlinear_host.h compile_mlmodel_mmap): every layer
    folder it writes holds the same blocks (W.mmap_store, C.mmap_store) as the reference's output (recorded under
    tests/golden/ref_results/) and -- where oracle/_ref is built -- loads in the reference library and predicts what the reference
    predicts from its own copy; incl. the root layer, whose C.npz may be absent."""
    from oracle import ref, restatement

    from .util import RecordedReference, assert_csr_parity, random_tree

    rec = RecordedReference(f"mlmodel_writer_{int(permute)}_{prune}")

    folder = str(tmp_path / "m")
    layers = random_tree(91, [4, 24, 300], 200, 18, bias=1.0, permute=permute, prune=prune)
    synth.save_xlinear_model(folder, layers, bias=1.0, only_topk=6, post_processor="l3-hinge")
    X = synth.make_queries(92, 40, 200, 20)
    for d in range(3):
        src = os.path.join(folder, "ranker", f"{d}.model")
        if d == 0 and os.path.exists(os.path.join(src, "C.npz")):
            os.remove(os.path.join(src, "C.npz"))  # the root layer's C is optional (inference.hpp:1580-1583)
        ours = str(tmp_path / f"ours{d}")
        ref.compile_mlmodel_mmap(src, ours, clib=clib.clib_float32)
        theirs = rec.folder(f"layer{d}", lambda path: ref.compile_mlmodel_mmap(src, path))
        for f in ("W.mmap_store", "C.mmap_store"):  # block by block (the padding between blocks is not initialised by the reference)
            ba, bb = restatement.read_mmap_store(os.path.join(ours, f)), restatement.read_mmap_store(os.path.join(theirs, f))
            assert len(ba) == len(bb) == 6 and all(np.array_equal(x, y) for x, y in zip(ba, bb)), (d, f)
        if not have_ref:
            continue
        a, b = ref.MLModelHandle(ours), ref.MLModelHandle(theirs)
        assert [a.attr(k) for k in ("nr_labels", "nr_codes", "nr_features")] == [b.attr(k) for k in ("nr_labels", "nr_codes", "nr_features")]
        assert_csr_parity(a.predict(X, None, None, 0), b.predict(X, None, None, 0), rtol=0.0, what=f"layer {d}: reference on our folder")
        assert_csr_parity(a.predict(X, None, "sigmoid", 3), b.predict(X, None, "sigmoid", 3), rtol=0.0, what=f"layer {d}: overrides")
    rec.save()
