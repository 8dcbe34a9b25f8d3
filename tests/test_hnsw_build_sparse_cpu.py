"""CPU tests of the sparse (csr) HNSW writer and the builder's argument checks (pecos_b200/hnsw_build.py).  The writer is checked
against the four reference-built golden sparse indices: their levels, adjacency and rows, read back with the restatement's
reader and written again, must give the same blocks (live neighbour slots; slots beyond a degree are zero in ours), and the
restatement / reference library must search both folders identically.  The GPU build itself: tests/test_hnsw_build_sparse_gpu.py."""
import json
import os

import numpy as np
import pytest
import scipy.sparse as smat

HERE = os.path.dirname(os.path.abspath(__file__))
SPARSE = os.path.join(HERE, "golden", "hnsw_sparse")
CASES = ["fixture_ip", "ip_tfidf", "l2_tfidf", "ip_short"]


def _graph(o):
    """(level_lists, per-level adjacency) of an index read by the restatement: every node listed on every level."""
    N = o.num_node
    l0 = o.l0
    head_w = 1 + o.maxM0
    heads = np.stack([l0[int(s): int(s) + 4 * head_w].view(np.uint32) for s in o.mem_start[:-1]])
    deg0 = heads[:, 0].astype(np.int64)
    lists0 = np.where(np.arange(o.maxM0)[None, :] < deg0[:, None], heads[:, 1:].astype(np.int64), -1)
    levels = [(np.arange(N), lists0, deg0)]
    if o.max_level:
        l1 = o.l1.view(np.uint32)[: N * o.l1_node_mem].reshape(N, o.l1_node_mem)
        for l in range(1, o.max_level + 1):
            slot = l1[:, (l - 1) * o.l1_level_mem: l * o.l1_level_mem]
            deg = slot[:, 0].astype(np.int64)
            lists = np.where(np.arange(o.maxM)[None, :] < deg[:, None], slot[:, 1:].astype(np.int64), -1)
            levels.append((np.arange(N), lists, deg))
    return levels


@pytest.mark.parametrize("case", CASES)
def test_writer_reproduces_the_reference_files(tmp_path, built, have_ref, case):
    from oracle import restatement
    from oracle.restatement import read_mmap_store
    from pecos_b200.hnsw_build import write_sparse_index

    theirs = os.path.join(SPARSE, case)
    param = json.load(open(os.path.join(theirs, "param.json")))
    cfg = json.load(open(os.path.join(theirs, "c_model", "config.json")))
    o = restatement.OracleHNSW(theirs, isa=0)
    X = o.vectors()
    levels = _graph(o)
    ours = str(tmp_path / case)
    write_sparse_index(ours, X, levels, o.maxM, o.maxM0, o.efC, o.init_node, param["metric_type"],
                       pred_kwargs=param.get("pred_kwargs"))

    a = read_mmap_store(os.path.join(theirs, "c_model", "index.mmap_store"))
    b = read_mmap_store(os.path.join(ours, "c_model", "index.mmap_store"))
    assert len(a) == len(b) == 21
    for i in list(range(0, 13)) + list(range(14, 20)):  # header scalars, mem_start_of_node, sizes
        assert np.array_equal(a[i], b[i]), f"block {i}"
    assert int(b[9].view(np.uint32)[0]) == 0  # node_mem_size
    # level-0 records: degree, live ids, len, value and index bytes; zeros beyond the degree in ours
    ms = a[11].view(np.uint64)
    head_w = 1 + o.maxM0
    for i in range(o.num_node):
        s, e = int(ms[i]), int(ms[i + 1])
        ra, rb = a[13][s:e].view(np.uint32), b[13][s:e].view(np.uint32)
        deg = int(ra[0])
        assert rb[0] == deg and np.array_equal(ra[1:1 + deg], rb[1:1 + deg]), f"node {i}"
        assert not rb[1 + deg:head_w].any()
        assert np.array_equal(ra[head_w:], rb[head_w:]), f"node {i} row"
    # GraphL1: live slots equal, the rest zero
    l1a = a[20].view(np.uint32).reshape(o.num_node, -1) if o.max_level else None
    l1b = b[20].view(np.uint32).reshape(o.num_node, -1) if o.max_level else None
    for l in range(o.max_level):
        sa = l1a[:, l * o.l1_level_mem:(l + 1) * o.l1_level_mem]
        sb = l1b[:, l * o.l1_level_mem:(l + 1) * o.l1_level_mem]
        assert np.array_equal(sa[:, 0], sb[:, 0])
        live = np.arange(o.maxM)[None, :] < sa[:, :1]
        assert np.array_equal(np.where(live, sa[:, 1:], 0), sb[:, 1:])
    mine = json.load(open(os.path.join(ours, "c_model", "config.json")))
    assert mine["hnsw_t"] == cfg["hnsw_t"] and mine["train_params"] == cfg["train_params"]
    mp = json.load(open(os.path.join(ours, "param.json")))
    assert mp["data_type"] == "csr" and mp["metric_type"] == param["metric_type"] and mp["feat_dim"] == X.shape[1]

    # both folders search identically (restatement), and the reference library loads ours
    Q = smat.load_npz(os.path.join(theirs, "Q.npz")).astype(np.float32)
    ob = restatement.OracleHNSW(ours, isa=0)
    for efS, topk in [(10, 10), (50, 10), (200, 20)]:
        ia, da = o.predict(Q, efS, topk)
        ib, db = ob.predict(Q, efS, topk)
        assert np.array_equal(ia, ib) and np.array_equal(da.view(np.uint32), db.view(np.uint32)), (efS, topk)
        if have_ref:
            from oracle import ref

            r = ref.RefHNSW.load(os.path.join(ours, "c_model"), param["metric_type"], data_type="csr")
            ri, rd = r.predict(Q, efS, topk, threads=1)
            assert np.array_equal(ri, ib) and np.array_equal(rd.view(np.uint32), db.view(np.uint32)), (efS, topk)


@pytest.mark.parametrize("case", CASES)
def test_host_loader_accepts_the_written_folders(tmp_path, clib, case):
    from ctypes import c_uint64

    from oracle import restatement
    from pecos_b200.hnsw_build import write_sparse_index

    theirs = os.path.join(SPARSE, case)
    metric = json.load(open(os.path.join(theirs, "param.json")))["metric_type"]
    o = restatement.OracleHNSW(theirs, isa=0)
    X = o.vectors()
    ours = str(tmp_path / case)
    write_sparse_index(ours, X, _graph(o), o.maxM, o.maxM0, o.efC, o.init_node, metric)
    m = 0 if metric == "ip" else 1
    out = (c_uint64 * 8)()
    assert clib.clib_float32.pb200_hnsw_host_info(os.path.join(ours, "c_model").encode(), m, 1, out) == 0
    assert [int(v) for v in out[:6]] == [o.num_node, X.shape[1], o.maxM, o.maxM0, o.max_level, o.init_node]
    assert int(out[6]) == X.nnz
    assert clib.clib_float32.pb200_hnsw_host_info(os.path.join(ours, "c_model").encode(), m, 0, out) == 1  # not a drm index


def test_sparse_build_has_no_cpu_path_and_checks_the_metric(tmp_path):
    from pecos_b200.hnsw_build import build_hnsw_index

    X = smat.random(50, 30, density=0.2, format="csr", dtype=np.float32, random_state=0)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        build_hnsw_index(X, str(tmp_path / "a"), M=4, efC=10, device="cpu")
    with pytest.raises(ValueError):
        build_hnsw_index(X, str(tmp_path / "b"), M=4, efC=10, metric="cosine")
    assert not os.path.exists(str(tmp_path / "a")) and not os.path.exists(str(tmp_path / "b"))


def test_canonical_csr_keeps_explicit_zeros_and_empty_rows():
    from pecos_b200.hnsw_build import canonical_csr

    # row 0: unsorted with a duplicate (3 appears twice) and an explicit zero; row 1 empty
    X = smat.csr_matrix((np.array([1.0, 0.0, 2.0, 0.5], dtype=np.float64), np.array([3, 1, 3, 0]), np.array([0, 4, 4])), shape=(2, 5))
    Xc = canonical_csr(X)
    assert Xc.dtype == np.float32 and Xc.has_sorted_indices
    assert Xc.indices.tolist() == [0, 1, 3] and Xc.data.tolist() == [0.5, 0.0, 3.0] and Xc.indptr.tolist() == [0, 3, 3]
    assert X.indices.tolist() == [3, 1, 3, 0]  # the caller's matrix is untouched
