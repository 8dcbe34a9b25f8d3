"""GPU construction of SPARSE (csr) HNSW indices (pecos_b200/hnsw_build.py + csrc/hnsw_build_sparse.cu): the exact prefix kNN
against a brute force by the restatement's hno_sparse_distance (ids and distance bits), bit-level search parity of the CUDA
engine, the restatement and the reference library on the GPU-built file, recall against the reference's own build, the
structural invariants of the records, determinism and edge sizes."""
import importlib.util
import os
from ctypes import POINTER, c_float, c_uint32

import numpy as np
import pytest
import scipy.sparse as smat

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


def _make_rows():
    spec = importlib.util.spec_from_file_location("mgs", os.path.join(HERE, "golden", "make_golden_hnsw_sparse.py"))
    mgs = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mgs)
    return mgs.make_rows


def _awkward_rows(seed, n, D, nnz):
    """Random rows plus empty rows, duplicated rows, an explicit zero and one row far longer than the rest."""
    rng = np.random.default_rng(seed)
    X = smat.random(n, D, density=nnz / D, format="lil", dtype=np.float32, random_state=seed)
    X = smat.csr_matrix(X)
    X.data = np.abs(X.data) + 0.05
    X = smat.lil_matrix(X)
    for i in range(0, n, 97):
        X[i, :] = 0  # empty rows
    for i in range(5, n, 211):
        X[i, :] = X[i - 3, :]  # duplicate rows
    long_cols = rng.choice(D, size=min(D, 40 * nnz), replace=False)
    X[n // 2, long_cols] = rng.random(long_cols.size).astype(np.float32) + 0.01
    X = smat.csr_matrix(X, dtype=np.float32)
    X.sort_indices()
    j = X.indptr[7]
    if X.indptr[8] > j:
        X.data[j] = 0.0  # explicit zero, stored as given
    return X


def _brute_prefix(X, ids, k, metric):
    """(positions, distance bits) of the k nearest earlier rows by (distance, id), distances by hno_sparse_distance."""
    from oracle import restatement

    L = restatement._hnsw_lib()
    m = 0 if metric == "ip" else 1
    rows = []
    for i in ids:
        s, e = X.indptr[i], X.indptr[i + 1]
        v = np.ascontiguousarray(X.data[s:e], dtype=np.float32)
        c = np.ascontiguousarray(X.indices[s:e], dtype=np.uint32)
        rows.append((e - s, v, c, v.ctypes.data_as(POINTER(c_float)), c.ctypes.data_as(POINTER(c_uint32))))
    n = len(ids)
    pos = np.full((n, k), -1, dtype=np.int64)
    bits = np.full((n, k), np.float32(np.inf).view(np.uint32), dtype=np.uint32)
    for q in range(1, n):
        a = rows[q]
        d = np.array([L.hno_sparse_distance(a[0], a[3], a[4], rows[c][0], rows[c][3], rows[c][4], m, 0) for c in range(q)],
                     dtype=np.float32)
        d[d == 0] = 0.0  # -0.0 ties +0.0
        order = np.lexsort((np.arange(q), d))[:k]
        pos[q, :order.size] = order
        bits[q, :order.size] = d[order].view(np.uint32)
    return pos, bits


@pytest.mark.parametrize("metric,n,subset", [("ip", 2300, False), ("l2", 1200, False), ("ip", 1500, True), ("l2", 1500, True)])
def test_prefix_knn_is_exact(gpu_clib, metric, n, subset):
    """n > 2048 crosses the kernel's shared-memory candidate block; `subset` = the node set of an upper level."""
    from pecos_b200.hnsw_build import canonical_csr, sparse_prefix_knn

    X = canonical_csr(_awkward_rows(n, n, 400, 12))
    ids = np.arange(n)
    if subset:
        ids = np.sort(np.random.default_rng(1).choice(n, size=n // 3, replace=False))
    k = 40
    pos, dist = sparse_prefix_knn(X, k, metric, ids=ids, device="cuda:0")
    bp, bb = _brute_prefix(X, ids, k, metric)
    assert np.array_equal(pos, bp)
    assert np.array_equal(dist.view(np.uint32), bb)


def _recall(idx, exact):
    return float(np.mean([len(set(idx[i]) & set(exact[i])) / exact.shape[1] for i in range(idx.shape[0])]))


@pytest.mark.parametrize("N,D,nnz,M,metric", [(5000, 30000, 80, 12, "ip"), (3000, 2000, 25, 8, "l2"), (2000, 40, 4, 6, "ip")])
def test_gpu_built_sparse_index_search_parity_and_recall(tmp_path, gpu_clib, have_ref, N, D, nnz, M, metric):
    if not have_ref:
        pytest.fail("oracle/_ref/libpecos_float32.so did not travel to this box; the reference library is the yardstick here")
    from oracle import ref, restatement
    from pecos_b200.hnsw import HNSW
    from pecos_b200.hnsw_build import build_hnsw_index

    make_rows = _make_rows()
    X = make_rows(N + D, N, D, nnz, 61)
    Q = make_rows(N + D + 1, 300, D, nnz, 17, long_row=(11, min(D, 5000)))
    folder = str(tmp_path / "idx")
    stats = build_hnsw_index(X, folder, M=M, efC=60, metric=metric, seed=7, device="cuda:0")
    assert stats["knn_products"] > 0 and stats["num_node"] == N
    m = HNSW.load(folder)
    assert m.data_type == "csr"
    o = restatement.OracleHNSW(folder, isa=0)
    r = ref.RefHNSW.load(os.path.join(folder, "c_model"), metric, data_type="csr")
    for efS, topk in [(10, 10), (64, 10), (200, 10), (5, 40), (600, 100)]:
        gi, gd = m.predict(Q, pred_params=HNSW.PredParams(efS=efS, topk=topk, threads=1), ret_csr=False)
        oi, od = o.predict(Q, efS, topk)
        assert np.array_equal(gi, oi) and np.array_equal(gd.view(np.uint32), od.view(np.uint32)), (efS, topk)
        ri, rd = r.predict(Q, efS, topk, threads=8)
        assert np.array_equal(gi, ri) and np.array_equal(gd.view(np.uint32), rd.view(np.uint32)), (efS, topk)
    Xs = smat.csr_matrix(X, dtype=np.float32)
    S = (Q @ Xs.T).toarray()
    exact = np.argsort((1.0 - S) if metric == "ip" else -2.0 * S, axis=1, kind="stable")[:, :10]
    gi, _ = m.predict(Q, pred_params=HNSW.PredParams(efS=100, topk=10, threads=1), ret_csr=False)
    trained = ref.RefHNSW.train(X, M=M, efC=60, metric=metric, threads=8)
    ti, _ = trained.predict(Q, 100, 10, threads=8)
    assert _recall(gi, exact) >= _recall(ti, exact) - 0.02


def _records(folder):
    from oracle import restatement

    o = restatement.OracleHNSW(folder, isa=0)
    heads = np.stack([o.l0[int(s): int(s) + 4 * (1 + o.maxM0)].view(np.uint32) for s in o.mem_start[:-1]])
    return o, heads


@pytest.mark.parametrize("metric", ["ip", "l2"])
def test_structure_rows_and_input_canonicalisation(tmp_path, gpu_clib, metric):
    from oracle import restatement
    from pecos_b200.hnsw_build import build_hnsw_index, canonical_csr

    X = _awkward_rows(3, 1800, 300, 10)
    M = 6
    folder = str(tmp_path / "a")
    build_hnsw_index(X, folder, M=M, efC=30, metric=metric, seed=2, device="cuda:0")
    o, heads = _records(folder)
    N = X.shape[0]
    Xc = canonical_csr(X)
    got = o.vectors()
    assert np.array_equal(got.indptr, Xc.indptr) and np.array_equal(got.indices, Xc.indices)
    assert np.array_equal(got.data.view(np.uint32), Xc.data.view(np.uint32))  # explicit zeros, empty rows included
    deg = heads[:, 0]
    assert deg.max() <= 2 * M and deg.min() >= 1
    L = restatement._hnsw_lib()
    m = 0 if metric == "ip" else 1

    def dist(u, v):
        a, b = slice(Xc.indptr[u], Xc.indptr[u + 1]), slice(Xc.indptr[v], Xc.indptr[v + 1])
        va, ia = np.ascontiguousarray(Xc.data[a]), np.ascontiguousarray(Xc.indices[a], dtype=np.uint32)
        vb, ib = np.ascontiguousarray(Xc.data[b]), np.ascontiguousarray(Xc.indices[b], dtype=np.uint32)
        d = L.hno_sparse_distance(va.size, va.ctypes.data_as(POINTER(c_float)), ia.ctypes.data_as(POINTER(c_uint32)), vb.size,
                                  vb.ctypes.data_as(POINTER(c_float)), ib.ctypes.data_as(POINTER(c_uint32)), m, 0)
        return 0.0 if d == 0 else d

    for u in range(N):
        nb = heads[u, 1:1 + deg[u]]
        assert u not in nb and len(set(nb.tolist())) == nb.size
        assert not heads[u, 1 + deg[u]:].any()
        keys = [(dist(u, int(v)), int(v)) for v in nb]
        assert keys == sorted(keys), u
    # unsorted / duplicated input indices: the same file as the canonical input
    Xu = Xc.copy()
    for i in range(0, N, 3):
        s, e = Xu.indptr[i], Xu.indptr[i + 1]
        Xu.indices[s:e] = Xu.indices[s:e][::-1].copy()
        Xu.data[s:e] = Xu.data[s:e][::-1].copy()
    Xu.has_sorted_indices = False
    f2 = str(tmp_path / "unsorted")
    build_hnsw_index(Xu, f2, M=M, efC=30, metric=metric, seed=2, device="cuda:0")
    assert _bytes(folder) == _bytes(f2)
    # a duplicated entry (v split into v/2 + v/2, which sum back exactly) is summed as the reference's create_pymat does
    r = 10
    while Xc.indptr[r + 1] == Xc.indptr[r]:
        r += 1
    s, e = Xc.indptr[r], Xc.indptr[r + 1]
    data = Xc.data.copy()
    half = data[s] / np.float32(2)
    data[s] = half
    Xd = smat.csr_matrix((np.insert(data, e, half), np.insert(Xc.indices, e, Xc.indices[s]),
                          np.concatenate([Xc.indptr[:r + 1], Xc.indptr[r + 1:] + 1])), shape=Xc.shape)
    Xd.has_canonical_format = False
    f3 = str(tmp_path / "dup")
    build_hnsw_index(Xd, f3, M=M, efC=30, metric=metric, seed=2, device="cuda:0")
    assert _bytes(folder) == _bytes(f3)


def _bytes(folder):
    with open(os.path.join(folder, "c_model", "index.mmap_store"), "rb") as f:
        return f.read()


def test_build_is_deterministic(tmp_path, gpu_clib):
    from pecos_b200.hnsw_build import build_hnsw_index

    X = _make_rows()(99, 6000, 20000, 60, 61)
    for f in ("a", "b"):
        build_hnsw_index(X, str(tmp_path / f), M=12, efC=80, metric="ip", seed=4, device="cuda:0")
    assert _bytes(str(tmp_path / "a")) == _bytes(str(tmp_path / "b"))


@pytest.mark.parametrize("N,empty", [(1, False), (2, False), (7, False), (50, True)])
def test_edge_sizes(tmp_path, gpu_clib, N, empty):
    """N = 1, N = 2, N < efC and all rows empty: every node gets neighbours (degree >= 1 when N > 1), searches agree."""
    from oracle import restatement
    from pecos_b200.hnsw import HNSW
    from pecos_b200.hnsw_build import build_hnsw_index

    D = 30
    X = smat.csr_matrix((N, D), dtype=np.float32) if empty else \
        smat.random(N, D, density=0.3, format="csr", dtype=np.float32, random_state=N)
    folder = str(tmp_path / "idx")
    build_hnsw_index(X, folder, M=4, efC=20, metric="ip", seed=1, device="cuda:0")
    o, heads = _records(folder)
    deg = heads[:, 0]
    assert deg.min() >= (1 if N > 1 else 0) and deg.max() <= 8
    if empty:  # all distances tie: node u > 0 links to the smallest ids
        assert list(heads[N - 1, 1:1 + deg[N - 1]]) == sorted(heads[N - 1, 1:1 + deg[N - 1]])
    Q = smat.random(5, D, density=0.3, format="csr", dtype=np.float32, random_state=3)
    m = HNSW.load(folder)
    gi, gd = m.predict(Q, pred_params=HNSW.PredParams(efS=10, topk=min(N, 5), threads=1), ret_csr=False)
    oi, od = o.predict(Q, 10, min(N, 5))
    assert np.array_equal(gi, oi) and np.array_equal(gd.view(np.uint32), od.view(np.uint32))
