"""Shared helpers for the parity tests (test infrastructure)."""
import os
import shutil

import numpy as np
import scipy.sparse as smat

from pecos_b200 import synth

REF_RESULTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_results")


class RecordedReference(object):
    """What the reference library (oracle/_ref) returned for one test's seeded inputs, stored under tests/golden/ref_results/<name>
    so that the test compares with the reference without needing it at test time.

    With PB200_RECORD_REFERENCE=1 (and oracle/_ref built) every call runs the reference, stores its result and returns it; `save()`
    then writes the recording.  Otherwise the stored result is returned and the reference is never called."""

    def __init__(self, name):
        self.dir = os.path.join(REF_RESULTS, name)
        self.recording = os.environ.get("PB200_RECORD_REFERENCE") == "1"
        self.store = {}
        if self.recording:
            shutil.rmtree(self.dir, ignore_errors=True)
            os.makedirs(self.dir)
        else:
            with np.load(os.path.join(self.dir, "results.npz")) as f:
                self.store = dict(f)

    def csr(self, key, compute):
        """A csr result (ids, stored order and score bits are kept)."""
        if self.recording:
            Y = smat.csr_matrix(compute())
            self.store.update({key + "|indptr": Y.indptr.astype(np.int32), key + "|indices": Y.indices.astype(np.int32),
                               key + "|data": Y.data.astype(np.float32), key + "|shape": np.asarray(Y.shape, dtype=np.int64)})
            return Y
        s = self.store
        return smat.csr_matrix((s[key + "|data"], s[key + "|indices"], s[key + "|indptr"]), shape=tuple(s[key + "|shape"]))

    def arrays(self, key, compute):
        """A tuple of dense arrays, returned with the dtypes they were recorded with."""
        if self.recording:
            out = tuple(np.asarray(a) for a in compute())
            self.store.update({f"{key}|{i}": a for i, a in enumerate(out)})
            return out
        n = sum(1 for k in self.store if k.startswith(key + "|"))
        return tuple(self.store[f"{key}|{i}"] for i in range(n))

    def folder(self, key, write):
        """A folder the reference writes (an index, a compiled model): `write(path)` when recording, the stored copy otherwise."""
        path = os.path.join(self.dir, key)
        if self.recording:
            write(path)
        assert os.path.isdir(path), path
        return path

    def save(self):
        if self.recording:
            np.savez_compressed(os.path.join(self.dir, "results.npz"), **self.store)


def assert_csr_parity(got, want, rtol=1e-5, what=""):
    """Bit-exact label ids and ranks (stored order), scores within `rtol` relative (BASELINE.json north_star)."""
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    assert np.array_equal(np.asarray(got.indptr, dtype=np.int64), np.asarray(want.indptr, dtype=np.int64)), f"{what}: row sizes differ"
    gi, wi = np.asarray(got.indices, dtype=np.int64), np.asarray(want.indices, dtype=np.int64)
    if not np.array_equal(gi, wi):
        bad = np.nonzero(gi != wi)[0]
        row = np.searchsorted(got.indptr, bad[0], side="right") - 1
        raise AssertionError(
            f"{what}: {bad.size} label ids / ranks differ; first at row {row}: got {gi[got.indptr[row]:got.indptr[row+1]]} "
            f"want {wi[want.indptr[row]:want.indptr[row+1]]}; scores got {got.data[got.indptr[row]:got.indptr[row+1]]} "
            f"want {want.data[want.indptr[row]:want.indptr[row+1]]}"
        )
    gd, wd = np.asarray(got.data, dtype=np.float32), np.asarray(want.data, dtype=np.float32)
    denom = np.maximum(np.abs(wd), np.finfo(np.float32).tiny)
    rel = np.abs(gd.astype(np.float64) - wd.astype(np.float64)) / denom
    assert rel.size == 0 or rel.max() <= rtol, f"{what}: max relative score error {rel.max():.3e} > {rtol}"
    exact = float(np.mean(gd.view(np.uint32) == wd.view(np.uint32))) if gd.size else 1.0
    return exact


def random_tree(seed, layer_sizes, D, nnz_per_col, bias=1.0, permute=False, prune=0.0, saturate=False):
    """Random label tree; `permute` shuffles child->parent assignment (non-contiguous C), `prune` drops that fraction of
    rows from every non-root C (pruned tree, pecos set_output_constraint style), `saturate` scales weights up so that the
    hinge post-processors saturate and ties decide the ranking."""
    rng = np.random.default_rng(seed)
    layers = synth.make_tree_model(seed, layer_sizes, D, nnz_per_col, bias=bias)
    out = []
    for d, (W, C) in enumerate(layers):
        if saturate:
            W = W * np.float32(8.0)
        C = smat.csc_matrix(C)
        if permute and d > 0 and C.shape[0] > 1:
            perm = rng.permutation(C.shape[0])
            C = smat.csc_matrix(C.tocsr()[perm, :])
        if prune > 0 and d > 0 and C.shape[0] > 4:
            keep = rng.random(C.shape[0]) >= prune
            keep[:2] = True
            Cr = C.tocsr().tolil()
            for r in np.nonzero(~keep)[0]:
                Cr.rows[r] = []
                Cr.data[r] = []
            C = smat.csc_matrix(Cr.tocsr())
        out.append((smat.csc_matrix(W, dtype=np.float32), smat.csc_matrix(C, dtype=np.float32)))
    return out


def csr_with_empty_rows(X, rows):
    X = X.tolil()
    for r in rows:
        X.rows[r] = []
        X.data[r] = []
    X = X.tocsr().astype(np.float32)
    X.sort_indices()
    return X


def merge_topk_numpy(g_keys, g_ids, g_vals, g_cnt, k):
    """Reference semantics of the index-sharding merge kernel (test-only): per query keep the k largest 64-bit keys
    among the valid entries of all ranks.  g_* have shape [world, rows, stride], g_cnt [world, rows]."""
    world, rows, stride = g_keys.shape
    out_ids = np.zeros((rows, k), dtype=np.uint32)
    out_vals = np.zeros((rows, k), dtype=np.float32)
    out_cnt = np.zeros(rows, dtype=np.uint32)
    for q in range(rows):
        cand = [(int(np.uint64(g_keys[g, q, r])), int(g_ids[g, q, r]), float(g_vals[g, q, r]))
                for g in range(world) for r in range(int(g_cnt[g, q]))]
        cand.sort(key=lambda t: -t[0])
        kk = min(k, len(cand))
        out_cnt[q] = kk
        for r in range(kk):
            out_ids[q, r], out_vals[q, r] = cand[r][1], cand[r][2]
    return out_ids, out_vals, out_cnt


def reachable_labels(layers):
    """Labels of the last layer with a complete path to the root (pruned trees drop rows of C at every layer).  The reference's
    predict_on_selected_outputs leaves the entry of an unreachable selected label UNINITIALISED and then indexes with it
    (pecos/core/xmc/inference.hpp:1302-1358), so in-contract selections only contain reachable labels."""
    reach = np.ones(1, dtype=bool)
    for _, C in layers:
        C = smat.csr_matrix(C)
        reach = np.asarray((C.astype(np.float32) @ reach.astype(np.float32)) > 0).ravel()
    return np.nonzero(reach)[0]
