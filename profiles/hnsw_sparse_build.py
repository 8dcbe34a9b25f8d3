"""GPU build of a sparse (csr) HNSW index on bench.py's sparse workloads (hnsw-rcv1, hnsw-sparse-100k), measured end to end.

For each workload: total build seconds, device ms per phase (CUDA events: posting lists, kNN, forward selection, reverse links;
the writer is host time), the kNN kernel's product count and achieved rate, recall@10 at efS = 100 against a brute force on
the first 256 queries, and the CUDA engine's resident search rate on the GPU-built index.  --with-reference repeats the build
with the reference's HNSW.train (all host threads) on the same rows and measures the same numbers on its index.  The card's
name and power limit are read in the same run.  Without a GPU it fails.

    python profiles/hnsw_sparse_build.py --workloads hnsw-sparse-100k hnsw-rcv1 --with-reference --out hnsw_sparse_build.json
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         stdout=subprocess.PIPE, text=True, check=True).stdout.strip().splitlines()
    return out[0]


def evaluate(folder, X, Q, cfg, n_recall=256):
    from ctypes import byref

    from pecos_b200 import core
    from pecos_b200.hnsw import HNSW

    m = HNSW.load(folder)
    Qr = Q[:n_recall]
    gi, _ = m.predict(Qr, pred_params=HNSW.PredParams(efS=100, topk=10, threads=1), ret_csr=False)
    S = (Qr @ X.T).toarray()
    exact = np.argsort((1.0 - S) if cfg["metric"] == "ip" else -2.0 * S, axis=1, kind="stable")[:, :10]
    recall = float(np.mean([len(set(gi[i]) & set(exact[i])) / 10.0 for i in range(Qr.shape[0])]))
    c = core.get_clib().clib_float32
    px = core.ScipyCsrF32.init_from(Q)
    c.pb200_hnsw_resident_upload_csr(m.model_ptr, byref(px))
    c.pb200_hnsw_resident_predict(m.model_ptr, cfg["efS"], cfg["topk"])  # warm-up
    ms = [c.pb200_hnsw_resident_predict(m.model_ptr, cfg["efS"], cfg["topk"]) for _ in range(3)]
    return {"recall_at_10_efS100": recall, "recall_queries": int(Qr.shape[0]),
            "search_qps_resident": Q.shape[0] / (min(ms) / 1000.0), "search_ms": min(ms), "search_queries": int(Q.shape[0])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["hnsw-sparse-100k", "hnsw-rcv1"])
    ap.add_argument("--with-reference", action="store_true")
    ap.add_argument("--out", required=True)
    args = ap.parse_args()

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device visible: this measurement runs on the GPU only")
    import __graft_entry__ as g

    g.build()
    from bench import HNSW_WORKLOADS, make_sparse_rows
    from pecos_b200.hnsw_build import build_hnsw_index

    result = {"card": card(), "torch": torch.__version__, "workloads": {}}
    print(result["card"], flush=True)
    tmp = tempfile.mkdtemp(prefix="hnsw_sparse_build_")
    for name in args.workloads:
        cfg = dict(HNSW_WORKLOADS[name])
        X = make_sparse_rows(30, cfg["N"], cfg["d"], cfg["nnz"])
        Q = make_sparse_rows(31, cfg["Q"], cfg["d"], cfg["nnz"])
        folder = os.path.join(tmp, name + "_gpu")
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        stats = build_hnsw_index(X, folder, M=cfg["M"], efC=cfg["efC"], metric=cfg["metric"], seed=30, device="cuda:0",
                                 pred_kwargs={"efS": cfg["efS"], "topk": cfg["topk"], "threads": 1})
        torch.cuda.synchronize()
        build_s = time.perf_counter() - t0
        knn_s = stats["phase_ms"]["knn"] / 1000.0
        entry = {"config": {k: cfg[k] for k in ("N", "d", "nnz", "M", "efC", "efS", "topk", "metric", "Q")},
                 "stored_entries": stats["nnz"],
                 "gpu_build": {"build_seconds": build_s, "phase_ms": stats["phase_ms"], "knn_products": stats["knn_products"],
                               "knn_products_per_s": stats["knn_products"] / knn_s if knn_s > 0 else None,
                               "knn_posting_bytes_per_s": 8 * stats["knn_products"] / knn_s if knn_s > 0 else None,
                               "nodes_per_level": stats["nodes_per_level"], "mean_degree_l0": stats["mean_degree_l0"]}}
        entry["gpu_build"].update(evaluate(folder, X, Q, cfg))
        print(name, json.dumps(entry["gpu_build"]), flush=True)
        if args.with_reference:
            import oracle
            from oracle import ref

            oracle.build()
            rf = os.path.join(tmp, name + "_ref")
            t0 = time.perf_counter()
            r = ref.RefHNSW.train(X, M=cfg["M"], efC=cfg["efC"], metric=cfg["metric"], threads=-1)
            ref_s = time.perf_counter() - t0
            r.save(os.path.join(rf, "c_model"))
            del r
            with open(os.path.join(rf, "param.json"), "w") as f:
                json.dump({"model": "HNSW", "data_type": "csr", "metric_type": cfg["metric"], "num_item": cfg["N"],
                           "feat_dim": cfg["d"], "pred_kwargs": {"efS": cfg["efS"], "topk": cfg["topk"], "threads": 1}}, f)
            entry["reference_build"] = {"build_seconds": ref_s, "host_threads": os.cpu_count(), **evaluate(rf, X, Q, cfg)}
            entry["speedup_vs_reference"] = ref_s / build_s
            print(name, "reference", json.dumps(entry["reference_build"]), flush=True)
        result["workloads"][name] = entry
        shutil.rmtree(folder, ignore_errors=True)
        if args.with_reference:
            shutil.rmtree(rf, ignore_errors=True)
    shutil.rmtree(tmp, ignore_errors=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
