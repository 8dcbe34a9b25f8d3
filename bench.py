#!/usr/bin/env python
"""bench.py -- XR-Linear beam-search prediction throughput on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload eurlex-4k|synthetic-small|synthetic-3m]

A "step" is one pass of the hot path (all tree layers: chunk-score kernel + top-k kernel per layer) over one batch of
synthetic queries.  At N=1 the workload is BASELINE.json configs[1] ("eurlex-4k": N=15,449 queries, D=5,000,
L=3,956, beam 10, top-10).  For N>1 (launched by torchrun, one rank per GPU) every rank holds a replica of the model
and processes its own batch of the same shape: query-sharded, no data-path collective, weak scaling.

Printed JSON line (rank 0): `value` = queries/s with the batch already resident in HBM (CUDA-event time of the K
steps, max over ranks); `e2e` = queries/s through the reference-facing C-ABI call `c_xlinear_predict_csr_f32` with
pinned HOST buffers (H2D + kernels + D2H + result marshalling inside the timed region); `roofline` = achieved
algorithmic HBM GB/s of the dominant kernel vs the measured peak; `cpu_baseline` = the reference's own OpenMP C++
library (oracle/_ref) timed on this box's host cores.  `--impl reference` times that reference library alone.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "XR-Linear top-10 queries/sec"
UNIT = "queries/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="eurlex-4k")
    ap.add_argument("--cache-dir", default=os.environ.get("PB200_BENCH_CACHE", os.path.join(tempfile.gettempdir(), "pecos_b200_bench")))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true",
                    help="skip the other target configurations (synthetic-3m; at N > 1 also the index-sharded run) that the default "
                         "eurlex-4k run reports under `secondary`")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline workload returned as DIR/<name>.npy (rank 0), so that two "
                         "builds can be compared output for output on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Saves `arrays` ({name: float32 or float64 array}) as out_dir/<name>.npy; refuses to write more than DUMP_LIMIT_BYTES."""
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def csr_result_arrays(Y, max_bytes=DUMP_LIMIT_BYTES, seed=0):
    """The CSR result of an XR-Linear prediction as float arrays (row pointers and label ids exactly representable in float64).
    A result larger than `max_bytes` is cut to a fixed, seeded sample of its rows (row ids saved beside it)."""
    import scipy.sparse as smat

    Y = smat.csr_matrix(Y)
    rows = np.arange(Y.shape[0])
    per_row = 12.0 * Y.nnz / max(Y.shape[0], 1) + 16.0
    if per_row * Y.shape[0] > max_bytes:
        rows = np.sort(np.random.default_rng(seed).choice(Y.shape[0], size=int(max_bytes // per_row), replace=False))
        Y = Y[rows]
    return {"rows": rows.astype(np.float64), "indptr": Y.indptr.astype(np.float64), "labels": Y.indices.astype(np.float64),
            "scores": Y.data.astype(np.float32)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


class ClockSampler(object):
    """Samples SM clocks / throttle reasons while the timed region runs (B200_PROFILING.md recipe).

    Primary source: NVML polled every ~2 ms from a thread (the timed region of the default run is only tens of
    milliseconds, far below nvidia-smi's sampling period); fallback: `nvidia-smi -lms 100`.  Every NVML call is guarded:
    a sampling failure must never fail the bench."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NVML_REASONS = (("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40), ("sw_power_cap", 0x4))

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []
        self.nvml_samples = []   # (sm_mhz, reasons bitmask)
        self.nvml_max = None
        self.nvml_thread = None
        self.stop_flag = False
        self.active = True       # NVML samples are only kept while a timed region runs (pause / resume)
        self.mark_at = 0
        self.nvml_mark_at = 0

    def _nvml_index(self):
        # CUDA_VISIBLE_DEVICES may renumber the devices; NVML counts physical ones
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        try:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if ids and all(v.isdigit() for v in ids) and self.gpu_index < len(ids):
                return int(ids[self.gpu_index])
        except Exception:
            pass
        return self.gpu_index

    def _nvml_loop(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self._nvml_index())
            try:
                self.nvml_max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            except Exception:
                self.nvml_max = None
            while not self.stop_flag:
                try:
                    mhz = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                    try:
                        bits = int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))
                    except Exception:
                        bits = int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                    if self.active:
                        self.nvml_samples.append((mhz, bits))
                except Exception:
                    break
                time.sleep(0.001)
        except Exception:
            pass

    def start(self):
        try:
            self.nvml_thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.nvml_thread.start()
        except Exception:
            self.nvml_thread = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        try:
            for line in self.proc.stdout:
                self.lines.append(line.strip())
        except Exception:
            pass

    def mark(self):
        """Samples taken before this call (warm-up) are dropped if enough samples follow."""
        self.mark_at = len(self.lines)
        self.nvml_mark_at = len(self.nvml_samples)

    def pause(self):
        self.active = False

    def resume(self):
        self.active = True

    def stop(self):
        self.stop_flag = True
        if self.nvml_thread is not None:
            try:
                self.nvml_thread.join(timeout=1.0)
            except Exception:
                pass
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        timed = self.nvml_samples[self.nvml_mark_at:]
        if len(timed) >= 3:
            sm = [m for m, _ in timed]
            reasons = sorted({name for _, bits in timed for name, mask in self.NVML_REASONS if bits & mask})
            return {"sm_mhz": statistics.median(sm), "sm_max_mhz": self.nvml_max if self.nvml_max else max(sm),
                    "reasons": reasons, "samples": len(sm), "source": "nvml, ~1 ms period, both timed regions (resident steps + end-to-end calls)"}
        if self.proc is None and not self.nvml_samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi and NVML unavailable"], "samples": 0}
        lines = self.lines[self.mark_at:]
        if len(lines) < 3:
            lines = self.lines
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm and self.nvml_samples:  # NVML gave something, but not enough inside the timed region
            sm = [m for m, _ in self.nvml_samples]
            smax = [self.nvml_max] if self.nvml_max else [max(sm)]
            reasons = {name for _, bits in self.nvml_samples for name, mask in self.NVML_REASONS if bits & mask}
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 100 (incl. warm-up if the timed region was too short)"}


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def prepare_workload(args, rank, world, barrier, same_batch=False):
    """Rank 0 writes the synthetic model folder once; every rank generates its own query batch from a seed (same_batch: the
    SAME batch on every rank, for strong scaling)."""
    from pecos_b200 import synth

    folder = os.path.join(args.cache_dir, args.workload)
    if rank == 0:
        os.makedirs(args.cache_dir, exist_ok=True)
        synth.build_workload(args.workload, folder, scale_queries=8)  # writes the model if absent
    barrier()
    cfg = dict(synth.WORKLOADS[args.workload])
    cdf = synth.zipf_cdf(cfg["D"]) if cfg["zipf"] else None
    X = synth.make_queries(cfg["query_seed"] + (0 if same_batch else 1000 * rank), cfg["Q"], cfg["D"], cfg["nnz_per_row"], cdf)
    return folder, X, cfg


class ReferenceUnavailable(RuntimeError):
    pass


def _require_ref():
    """The reference arm is the UNMODIFIED reference library (oracle/_ref), never the scalar restatement."""
    import oracle

    if not oracle.have_ref():
        raise ReferenceUnavailable(
            "oracle/_ref/libpecos_float32.so is missing: build it where /root/reference exists (`make -C oracle`, "
            "done by __graft_entry__.build()); it is git-ignored but travels to the GPU box with the snapshot")


def _thread_grid(n_cores):
    """Thread counts the reference is tried with (pecos/core/utils/parallel.hpp:27-34: -1 = omp_get_num_procs())."""
    g = sorted({t for t in (1, 8, 32, n_cores) if 1 <= t <= n_cores})
    return g


def time_reference(folder, X, cfg, steps, warmup, budget_s=120.0, layouts=None):
    """Times the reference's own OpenMP C++ library (oracle/_ref) on this box's host cores.

    The headline is the reference's BEST configuration on this box: a short sweep over its two chunked weight layouts
    (BINARY_SEARCH_CHUNKED = its default, HASH_CHUNKED; pecos/core/xmc/inference.hpp:43) and over thread counts
    {1, 8, 32, all} picks the fastest (layout, threads); the K timed steps then run that configuration on a bounded
    sample of the workload.  The whole sweep is reported next to it."""
    _require_ref()
    from oracle import ref

    n_cores = os.cpu_count() or 1
    if layouts is None:
        layouts = ["BINARY_SEARCH_CHUNKED", "HASH_CHUNKED"]
        if cfg["layer_sizes"][-1] > 1_000_000:
            layouts = ["BINARY_SEARCH_CHUNKED"]  # the reference builds a layout single-threaded at load: minutes each on S
    beam, topk = cfg["beam_size"], cfg["only_topk"]
    probe = X[: min(X.shape[0], 4096)]
    sweep, best = [], None
    models = {}
    t_sweep0 = time.perf_counter()
    for lay in layouts:
        t0 = time.perf_counter()
        models[lay] = ref.RefXLinear(os.path.join(folder, "ranker"), weight_matrix_type=lay)
        load_s = time.perf_counter() - t0
        for th in _thread_grid(n_cores):
            rows = probe if th > 1 else probe[: min(probe.shape[0], 512)]
            models[lay].predict(rows[:64], beam, None, topk, th)
            t0 = time.perf_counter()
            models[lay].predict(rows, beam, None, topk, th)
            dt = time.perf_counter() - t0
            qps = rows.shape[0] / dt
            sweep.append({"layout": lay, "threads": th, "queries": int(rows.shape[0]), "qps": qps, "load_s": round(load_s, 3)})
            if best is None or qps > best[2]:
                best = (lay, th, qps)
            if time.perf_counter() - t_sweep0 > budget_s * 0.4:
                break
    lay, th, qps_est = best
    model = models[lay]
    # bound the sample so that warmup + steps stays within the remaining budget
    remaining = max(5.0, budget_s - (time.perf_counter() - t_sweep0))
    rows = int(min(X.shape[0], max(256, qps_est * remaining / max(1, steps + warmup))))
    sample = X[:rows]

    def run():
        return model.predict(sample, beam, None, topk, th)

    for _ in range(max(1, warmup)):
        run()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        run()
        times.append(time.perf_counter() - t0)
    mean_t = sum(times) / len(times)
    return {
        "value": sample.shape[0] / mean_t,
        "best": sample.shape[0] / min(times),
        "ms_per_step": 1e3 * mean_t,
        "kind": "reference",
        "cores": n_cores,
        "threads": th,
        "layout": lay,
        "sweep": sweep,
        "sample": (f"{sample.shape[0]} of {X.shape[0]} queries of the workload per step, {steps} steps; reference library "
                   f"oracle/_ref (unmodified libpecos.cpp, -fopenmp -O3), best of the sweep over layouts x threads "
                   f"{_thread_grid(n_cores)}: {lay}, threads={th} on a {n_cores}-thread host"),
    }


def run_reference_arm(args):
    rank, world, local = dist_env()
    if rank != 0:
        return 0
    try:
        _require_ref()
    except ReferenceUnavailable as e:
        print(f"bench.py --impl reference: {e}", file=sys.stderr)
        return 3  # never silently time something else
    folder, X, cfg = prepare_workload(args, 0, 1, lambda: None)
    r = time_reference(folder, X, cfg, args.steps, args.warmup)
    line = {
        "impl": "reference",
        "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, cfg, X),
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"],
                         "threads": r["threads"], "layout": r["layout"], "sweep": r["sweep"]},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def workload_config(name, cfg, X, extra=None):
    c = {
        "workload": name,
        "queries_per_step_per_gpu": int(X.shape[0]),
        "nnz_per_query": int(X.nnz // max(1, X.shape[0])),
        "features": int(cfg["D"]),
        "labels": int(cfg["layer_sizes"][-1]),
        "tree_layers": list(cfg["layer_sizes"]),
        "nnz_per_weight_col": int(cfg["nnz_per_col"]) + 1,
        "beam_size": int(cfg["beam_size"]),
        "only_topk": int(cfg["only_topk"]),
        "post_processor": "l3-hinge",
        "parallelism": "query-sharded replicas (no collective)",
    }
    if extra:
        c.update(extra)
    return c


SCORE_KERNELS = ["xl_chunk_scores_kernel<stream>", "xl_chunk_scores_kernel", "xl_chunk_scores_kernel<dense>", "xl_query_warp_scores_kernel",
                 "xl_cm_scores_kernel", "xl_cmg_scores_kernel"]
TOPK_KERNELS = ["xl_topk_kernel", "xl_topk_warp_kernel", "xl_topk_filter_kernel"]

HNSW_WORKLOADS = {
    # BASELINE.json configs[3] shape (dense d=768, ip, M=32, efS=200, top-10) at sizes the reference trainer can build
    # inside a GPU lease; the index is built once per box by the reference's own HNSW.train (oracle/_ref), all host threads
    "hnsw-100k": dict(N=100_000, d=768, M=32, efC=100, Q=10_000, efS=200, topk=10, metric="ip"),
    "hnsw-1m": dict(N=1_000_000, d=768, M=32, efC=100, Q=50_000, efS=200, topk=10, metric="ip"),
    "hnsw-10m": dict(N=10_000_000, d=768, M=32, efC=200, Q=100_000, efS=200, topk=10, metric="ip"),
    # SPARSE (csr) indices, SURVEY 8(f)-4.  hnsw-rcv1 has the shape of the one HNSW result the reference publishes (BASELINE.md:
    # RCV1, 781,265 x 47,236 sparse ip, 23,149 queries, M=32, efC=100, efS=100, top-10) on synthetic tf-idf-like rows (topic
    # mixture over a Zipf vocabulary, ~76 stored entries per row); the index is built by the reference's HNSW.train on the host.
    "hnsw-rcv1": dict(N=781_265, d=47_236, nnz=76, M=32, efC=100, Q=23_149, efS=100, topk=10, metric="ip", sparse=True),
    "hnsw-sparse-100k": dict(N=100_000, d=47_236, nnz=76, M=32, efC=100, Q=10_000, efS=100, topk=10, metric="ip", sparse=True),
}


def make_sparse_rows(seed, n, D, nnz, topics=2000):
    """tf-idf-like csr rows: every row draws half of its features from its topic's own popularity ranking of the vocabulary and
    half from a global Zipf law (duplicates dropped: ~nnz distinct per row), values |N(0,1)| row-L2-normalised, indices ascending."""
    import scipy.sparse as smat

    rng = np.random.default_rng(seed)
    draws = int(nnz * 1.04)
    cdf = np.cumsum(1.0 / (np.arange(D) + 10.0))
    cdf /= cdf[-1]
    z = np.searchsorted(cdf, rng.random((n, draws))).astype(np.int64)
    topic = rng.integers(0, topics, size=n)
    trng = np.random.default_rng(12345)  # the topics are the same for the base rows and the queries
    mult = (2 * trng.integers(1000, D, size=topics) + 1).astype(np.int64)
    while True:
        bad = np.gcd(mult, D) != 1
        if not bad.any():
            break
        mult[bad] += 2
    shift = trng.integers(0, D, size=topics).astype(np.int64)
    half = draws // 2
    z[:, :half] = (z[:, :half] * mult[topic][:, None] + shift[topic][:, None]) % D
    z.sort(axis=1)
    keep = np.ones(z.shape, dtype=bool)
    keep[:, 1:] = z[:, 1:] != z[:, :-1]
    vals = (np.abs(rng.standard_normal(z.shape)) + 0.05).astype(np.float32) * keep
    vals /= np.maximum(np.linalg.norm(vals, axis=1, keepdims=True), 1e-12)
    indptr = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(keep.sum(axis=1), out=indptr[1:])
    X = smat.csr_matrix((vals[keep].astype(np.float32), z[keep].astype(np.int32), indptr), shape=(n, D), dtype=np.float32)
    X.has_sorted_indices = True
    return X


def hnsw_prepare(args, rank, barrier, local=0):
    """Rank 0 builds the index once per box ON THE GPU (pecos_b200.hnsw_build: exact kNN by tiled GEMMs + the reference's
    neighbour-selection heuristic) and writes it in the reference's index.mmap_store format -- the same file is then searched by
    the CUDA engine and by the reference library (cpu_baseline / parity gate).  PB200_BENCH_HNSW_BUILDER=reference uses the
    reference's own (CPU, minutes to hours) HNSW.train instead."""
    cfg = dict(HNSW_WORKLOADS[args.workload])
    folder = os.path.join(args.cache_dir, args.workload)
    if cfg.get("sparse"):
        import scipy.sparse as smat

        if rank == 0 and not os.path.exists(os.path.join(folder, "c_model", "index.mmap_store")):
            import oracle
            from oracle import ref

            os.makedirs(folder, exist_ok=True)
            oracle.build()
            X = make_sparse_rows(30, cfg["N"], cfg["d"], cfg["nnz"])
            t0 = time.perf_counter()
            r = ref.RefHNSW.train(X, M=cfg["M"], efC=cfg["efC"], metric=cfg["metric"], threads=-1)
            build_s = time.perf_counter() - t0
            r.save(os.path.join(folder, "c_model"))
            del r
            smat.save_npz(os.path.join(folder, "X.npz"), X, compressed=False)
            with open(os.path.join(folder, "param.json"), "w") as f:
                json.dump({"model": "HNSW", "data_type": "csr", "metric_type": cfg["metric"], "num_item": cfg["N"],
                           "feat_dim": cfg["d"], "pred_kwargs": {"efS": cfg["efS"], "topk": cfg["topk"], "threads": 1}}, f)
            with open(os.path.join(folder, "build.json"), "w") as f:
                json.dump({"builder": "reference HNSW.train (csr, all host threads)", "build_seconds": build_s,
                           "stored_entries_per_row": X.nnz / X.shape[0]}, f)
            del X
        barrier()
        Q = make_sparse_rows(31 + 1000 * rank, cfg["Q"], cfg["d"], cfg["nnz"])
        try:
            cfg["index_build"] = json.load(open(os.path.join(folder, "build.json")))
        except Exception:
            cfg["index_build"] = None
        return folder, Q, cfg
    if rank == 0 and not os.path.exists(os.path.join(folder, "c_model", "index.mmap_store")):
        os.makedirs(folder, exist_ok=True)
        rng = np.random.default_rng(30)
        X = rng.standard_normal((cfg["N"], cfg["d"]), dtype=np.float32)
        X /= np.linalg.norm(X, axis=1, keepdims=True)
        t0 = time.perf_counter()
        if os.environ.get("PB200_BENCH_HNSW_BUILDER", "gpu") == "reference":
            import oracle
            from oracle import ref

            oracle.build()
            r = ref.RefHNSW.train(X, M=cfg["M"], efC=cfg["efC"], metric=cfg["metric"], threads=-1)
            r.save(os.path.join(folder, "c_model"))
            del r
            builder = "reference HNSW.train (all host threads)"
            with open(os.path.join(folder, "param.json"), "w") as f:
                json.dump({"model": "HNSW", "data_type": "drm", "metric_type": cfg["metric"], "num_item": cfg["N"],
                           "feat_dim": cfg["d"], "pred_kwargs": {"efS": cfg["efS"], "topk": cfg["topk"], "threads": 1}}, f)
        else:
            from pecos_b200.hnsw_build import build_hnsw_index

            build_hnsw_index(X, folder, M=cfg["M"], efC=cfg["efC"], metric=cfg["metric"], seed=30, device=f"cuda:{local}",
                             pred_kwargs={"efS": cfg["efS"], "topk": cfg["topk"], "threads": 1}, allow_tf32=cfg["N"] > 2_000_000)
            builder = "pecos_b200.hnsw_build on the GPU"
        with open(os.path.join(folder, "build.json"), "w") as f:
            json.dump({"builder": builder, "build_seconds": time.perf_counter() - t0}, f)
        del X
    barrier()
    rng = np.random.default_rng(31 + 1000 * rank)
    Q = rng.standard_normal((cfg["Q"], cfg["d"]), dtype=np.float32)
    Q /= np.linalg.norm(Q, axis=1, keepdims=True)
    try:
        cfg["index_build"] = json.load(open(os.path.join(folder, "build.json")))
    except Exception:
        cfg["index_build"] = None
    return folder, np.ascontiguousarray(Q), cfg


def hnsw_config(name, cfg, extra=None):
    c = {"workload": name, "base_vectors": cfg["N"], "dim": cfg["d"], "M": cfg["M"], "efC": cfg["efC"], "efS": cfg["efS"],
         "topk": cfg["topk"], "metric": cfg["metric"], "queries_per_step_per_gpu": cfg["Q"],
         "rows": ("csr, ~%d stored entries per row" % cfg["nnz"]) if cfg.get("sparse") else "dense",
         "parallelism": "query-sharded replicas (no collective)", "index_build": cfg.get("index_build")}
    if name == "hnsw-rcv1":
        # informational only: `vs_baseline` stays null because the published number is for the REAL RCV1 vectors, one searcher thread
        c["published_by_the_reference"] = {"value": 1478.6, "unit": "queries/s", "recall_at_10": 0.9020,
                                           "setup": "RCV1-47236 sparse ip, N=781,265, 23,149 queries, M=32, efC=100, efS=100, top-10, 1 searcher thread, "
                                                    "AWS r5dn.24xlarge", "source": "BASELINE.md (tutorials/kdd22 Session 3 notebook)"}
    if extra:
        c.update(extra)
    return c


def hnsw_time_reference(folder, Q, cfg, steps, warmup, budget_s=60.0):
    from oracle import ref

    n_cores = os.cpu_count() or 1
    m = ref.RefHNSW.load(os.path.join(folder, "c_model"), cfg["metric"], data_type="csr" if cfg.get("sparse") else "drm")
    sample = Q
    t0 = time.perf_counter()
    m.predict(sample[:2048], cfg["efS"], cfg["topk"], threads=n_cores)
    first = (time.perf_counter() - t0) * sample.shape[0] / 2048.0
    if first * (steps + warmup) > budget_s:
        sample = sample[: max(2048, int(sample.shape[0] * budget_s / (first * (steps + warmup))))]
    for _ in range(max(0, warmup - 1)):
        m.predict(sample, cfg["efS"], cfg["topk"], threads=n_cores)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        m.predict(sample, cfg["efS"], cfg["topk"], threads=n_cores)
        times.append(time.perf_counter() - t0)
    mean_t = sum(times) / len(times)
    return {"value": sample.shape[0] / mean_t, "ms_per_step": 1e3 * mean_t, "kind": "reference", "cores": n_cores,
            "sample": f"{sample.shape[0]} of {Q.shape[0]} queries per step, {steps} steps, {n_cores} searchers (all host threads)"}


def measure_hnsw(args, workload, rank, n_gpus, local, dist, barrier, steps, warmup, with_cpu=True, dump_dir=None):
    """One HNSW workload on this rank's GPU (replicas: every rank its own query batch, same index file); returns the JSON line as
    a dict on rank 0 (None elsewhere)."""
    from ctypes import POINTER, byref, c_float, c_uint32, c_uint64

    from pecos_b200 import core
    from pecos_b200.core import ScipyCsrF32, ScipyDrmF32
    from pecos_b200.hnsw import HNSW

    wargs = argparse.Namespace(**vars(args))
    wargs.workload, wargs.steps, wargs.warmup = workload, steps, warmup
    wargs.no_cpu_baseline = args.no_cpu_baseline or not with_cpu
    args = wargs
    metric_name, unit = "HNSW top-10 queries/sec (efS=%d)" % HNSW_WORKLOADS[args.workload]["efS"], UNIT
    barrier()
    lib = core.get_clib()
    lib.require_gpu()
    lib.set_device(local)
    c = lib.clib_float32
    folder, Q, cfg = hnsw_prepare(args, rank, barrier, local)
    model = HNSW.load(folder)
    h = model.model_ptr
    nq, d, efS, topk = Q.shape[0], Q.shape[1], cfg["efS"], cfg["topk"]
    sparse = bool(cfg.get("sparse"))
    if sparse:
        qv = ScipyCsrF32.init_from(Q)
        c.pb200_hnsw_resident_upload_csr(h, byref(qv))
    else:
        qv = ScipyDrmF32.init_from(Q)
        c.pb200_hnsw_resident_upload(h, byref(qv))

    def one_step():
        c.pb200_l2_flush()
        return c.pb200_hnsw_resident_predict(h, efS, topk)

    for _ in range(max(3, args.warmup)):
        one_step()
    cnt = (c_uint64 * 4)()
    c.pb200_hnsw_get_counters(h, cnt)
    n_dist, n_expand, n_hops, _ = [int(x) for x in cnt]
    info = (c_uint64 * 8)()
    c.pb200_hnsw_get_info(h, info)
    maxM, maxM0 = int(info[2]), int(info[3])
    # SURVEY.md 8(d): n_dist * 4d + n_expand * 4(1+maxM0) + hops * 4(1+maxM) + 4d + 8k per query
    bytes_per_step = n_dist * 4.0 * d + n_expand * 4.0 * (1 + maxM0) + n_hops * 4.0 * (1 + maxM) + nq * (4.0 * d + 8.0 * topk)
    n_entries = 0
    if sparse:  # a distance reads the row's two offsets + its stored {index, value} entries; the query row is read once
        n_entries = int(c.pb200_hnsw_sparse_entries(h))
        bytes_per_step = (n_entries * 8.0 + n_dist * 16.0 + n_expand * 4.0 * (1 + maxM0) + n_hops * 4.0 * (1 + maxM) +
                          Q.nnz * 8.0 + nq * (16.0 + 8.0 * topk))

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = int(info[7])
    barrier()
    step_ms = [one_step() for _ in range(args.steps)]
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    c.pb200_hnsw_get_info(h, info)
    launches = int(info[7]) - launches0
    total_ms = float(sum(step_ms))
    if dist is not None:
        import torch

        t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    value = n_gpus * nq / (ms_per_step * 1e-3)
    peak, peak_src = measured_peak_gbs()
    achieved = bytes_per_step / (ms_per_step * 1e-3) / 1e9
    ncu_traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            ncu_traffic = json.load(f).get(args.workload, {}).get("hnsw_search_kernel")
            if isinstance(ncu_traffic, dict):
                ncu_traffic = ncu_traffic.get("dram_bytes_per_launch")
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": ncu_traffic,
                "kernel": "hnsw_search_kernel", "kernel_ms": ms_per_step, "algorithmic_bytes_per_launch": bytes_per_step,
                "peak_source": peak_src, "per_query": {"distance_evals": n_dist / nq, "expansions": n_expand / nq,
                                                       "upper_level_reads": n_hops / nq, "bytes": bytes_per_step / nq}}
    if sparse:
        roofline["per_query"]["stored_entries_read"] = n_entries / nq

    # parity gate: the first queries of the timed batch, searched by the reference library ON THE SAME index file
    gi = np.zeros((nq, topk), dtype=np.uint32)
    gd = np.zeros((nq, topk), dtype=np.float32)
    c.pb200_hnsw_resident_fetch(h, gi.ctypes.data_as(POINTER(c_uint32)), gd.ctypes.data_as(POINTER(c_float)))
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, {"neighbours": gi.astype(np.float64), "distances": gd})
    parity = {"checked_queries": 0, "checker": "unavailable (oracle/_ref absent)"}
    import oracle

    if oracle.have_ref():
        from oracle import ref, restatement

        n_chk = min(512, nq)
        ri, rd = ref.RefHNSW.load(os.path.join(folder, "c_model"), cfg["metric"], data_type="csr" if sparse else "drm").predict(
            Q[:n_chk], efS, topk, threads=os.cpu_count() or 1)
        if not np.array_equal(ri, gi[:n_chk]):
            raise RuntimeError("parity gate (hnsw): neighbour ids / ranks differ from the reference library on the same index file")
        bits = bool(np.array_equal(rd.view(np.uint32), gd[:n_chk].view(np.uint32)))
        if not bits and (sparse or restatement.host_isa() == 0 or not np.allclose(rd, gd[:n_chk], rtol=1e-5, atol=1e-7)):
            raise RuntimeError("parity gate (hnsw): distances differ from the reference library")
        parity = {"checked_queries": n_chk, "checker": "reference library (oracle/_ref), same index file", "ids_bit_equal": True,
                  "distance_bits_equal": bits}

    # recall@topk of the timed results against brute force (a sample of the batch; exact distances by a GEMM on the GPU)
    recall = None
    try:
        import torch

        from oracle import restatement as _rs

        n_rc = min(256, nq)
        if sparse:
            import scipy.sparse as smat

            n_rc = min(128, nq)
            Xb = smat.load_npz(os.path.join(folder, "X.npz"))
            sc = np.asarray((Q[:n_rc] @ Xb.T).todense(), dtype=np.float32)
            dist_np = (1.0 - sc) if cfg["metric"] == "ip" else (-2.0 * sc)  # the reference's sparse "l2" (feat_vectors.hpp:186-192)
            exact = np.argpartition(dist_np, topk, axis=1)[:, :topk]
            recall = float(np.mean([len(set(gi[i].tolist()) & set(exact[i].tolist())) / topk for i in range(n_rc)]))
            del Xb, sc, dist_np
            raise StopIteration
        base = torch.from_numpy(_rs.OracleHNSW(folder, isa=0).vectors()).to(f"cuda:{local}")
        qs = torch.from_numpy(Q[:n_rc]).to(base.device)
        sc = qs @ base.T
        dist_all = (1.0 - sc) if cfg["metric"] == "ip" else ((base * base).sum(1)[None, :] - 2.0 * sc)
        exact = torch.topk(dist_all, topk, dim=1, largest=False).indices.cpu().numpy()
        recall = float(np.mean([len(set(gi[i].tolist()) & set(exact[i].tolist())) / topk for i in range(n_rc)]))
        del base, sc, dist_all
        torch.cuda.empty_cache()
    except StopIteration:
        pass
    except Exception as e:  # noqa: BLE001
        print(f"bench.py: recall check skipped: {e}", file=sys.stderr)
    parity["recall_at_topk_vs_brute_force"] = recall

    # end to end through the C ABI with pinned host buffers
    ip = lib.pinned_empty(nq * topk, np.uint32)
    dp = lib.pinned_empty(nq * topk, np.float32)
    if sparse:
        p_ptr, p_idx, p_val = lib.pinned_empty(nq + 1, np.uint64), lib.pinned_empty(max(Q.nnz, 1), np.uint32), lib.pinned_empty(max(Q.nnz, 1), np.float32)
        p_ptr.array[:] = Q.indptr
        p_idx.array[:Q.nnz] = Q.indices
        p_val.array[:Q.nnz] = Q.data
        qv_p = ScipyCsrF32.init_from_arrays(nq, d, p_ptr.array, p_idx.array, p_val.array)
        h2d_bytes = int(8 * (nq + 1) + 8 * Q.nnz)
    else:
        qp = lib.pinned_empty(Q.size, np.float32)
        qp.array[:] = Q.ravel()
        qpin = qp.array.reshape(Q.shape)
        qv_p = ScipyDrmF32.init_from(qpin)
        h2d_bytes = int(Q.nbytes)
    predict = model.fn_dict["predict"]

    def e2e_step():
        ip.array[:] = 0
        dp.array[:] = 0
        predict(h, byref(qv_p), ip.array.ctypes.data_as(POINTER(c_uint32)), dp.array.ctypes.data_as(POINTER(c_float)), efS, topk, 1, None)

    for _ in range(2):
        e2e_step()
    barrier()
    e2e_times = []
    for _ in range(args.steps):
        c.pb200_l2_flush()
        t0 = time.perf_counter()
        e2e_step()
        e2e_times.append(time.perf_counter() - t0)
    barrier()
    e2e_total = float(sum(e2e_times))
    if dist is not None:
        import torch

        t = torch.tensor([e2e_total], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_total = float(t.item())
    cpu = None
    if rank == 0 and n_gpus == 1 and not args.no_cpu_baseline:
        import oracle

        if oracle.have_ref():
            r = hnsw_time_reference(folder, Q, cfg, steps=3, warmup=1, budget_s=30.0)
            cpu = {"value": r["value"], "unit": unit, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]}
    line = None
    if rank == 0:
        line = {
            "metric": metric_name, "value": value, "unit": unit, "n_gpus": n_gpus, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": hnsw_config(args.workload, cfg),
            "l2": "flushed between timed iterations; index (%.1f GB) >> L2" % (int(info[6]) / 1e9),
            "timing": "CUDA events around the search kernel per step, summed, max over ranks",
            "parity": parity,
            "clocks": clocks,
            "e2e": {"value": n_gpus * nq * args.steps / e2e_total, "unit": unit, "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": int(nq * topk * 8), "ms_per_step": 1e3 * e2e_total / args.steps,
                    "api": "c_ann_hnsw_predict_%s_%s_f32 (pinned host queries in, host id/distance arrays out)" % ("csr" if sparse else "drm", cfg["metric"])},
            "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu}
    return line


def main_hnsw(args):
    rank, world, local = dist_env()
    n_gpus = max(world, 1)
    metric_name, unit = "HNSW top-10 queries/sec (efS=%d)" % HNSW_WORKLOADS[args.workload]["efS"], UNIT
    if args.impl == "reference":
        if rank != 0:
            return 0
        folder, Q, cfg = hnsw_prepare(args, 0, lambda: None)
        r = hnsw_time_reference(folder, Q, cfg, args.steps, args.warmup)
        print(json.dumps({"impl": "reference", "metric": metric_name, "value": r["value"], "unit": unit, "n_gpus": args.gpus,
                          "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "config": hnsw_config(args.workload, cfg),
                          "cpu_baseline": {"value": r["value"], "unit": unit, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
                          "e2e": {"value": r["value"], "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "gpu_launches": 0}))
        return 0

    from ctypes import POINTER, byref, c_float, c_uint32, c_uint64

    from pecos_b200 import core
    from pecos_b200.core import ScipyCsrF32, ScipyDrmF32
    from pecos_b200.hnsw import HNSW

    dist = None
    if n_gpus > 1:
        import torch
        import torch.distributed as dist_mod

        torch.cuda.set_device(local)
        dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist = dist_mod

    def barrier():
        if dist is not None:
            dist.barrier()

    barrier()
    line = measure_hnsw(args, args.workload, rank, n_gpus, local, dist, barrier, args.steps, args.warmup, dump_dir=args.dump_outputs)
    if rank == 0:
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0




def parity_gate_xlinear(got, folder, X, cfg, rows=1024, what="resident batch"):
    """BASELINE.md section 2: no timing counts before parity.  The first `rows` queries of the timed batch are predicted by the
    reference library (oracle/_ref; the pinned restatement only if the library is absent) and compared with the GPU result:
    label ids and ranks bit-equal, scores within 1e-5 relative.  Raises on any difference."""
    import oracle

    rows = int(min(rows, X.shape[0]))
    beam, topk = cfg["beam_size"], cfg["only_topk"]
    if oracle.have_ref():
        from oracle import ref

        want = ref.RefXLinear(os.path.join(folder, "ranker")).predict(X[:rows], beam, None, topk, -1)
        checker = "reference library (oracle/_ref)"
    else:
        from oracle import restatement

        want = restatement.OracleXLinear(os.path.join(folder, "ranker")).predict(X[:rows], beam, None, topk)
        checker = "C restatement (oracle/liboracle.so; oracle/_ref absent)"
    g = got[:rows]
    if not np.array_equal(np.asarray(g.indptr, dtype=np.int64), np.asarray(want.indptr, dtype=np.int64)):
        raise RuntimeError(f"parity gate ({what}): row sizes differ from the {checker}")
    if not np.array_equal(np.asarray(g.indices, dtype=np.int64), np.asarray(want.indices, dtype=np.int64)):
        bad = int(np.count_nonzero(np.asarray(g.indices, dtype=np.int64) != np.asarray(want.indices, dtype=np.int64)))
        raise RuntimeError(f"parity gate ({what}): {bad} label ids / ranks differ from the {checker}")
    gd, wd = np.asarray(g.data, dtype=np.float64), np.asarray(want.data, dtype=np.float64)
    rel = float(np.max(np.abs(gd - wd) / np.maximum(np.abs(wd), 1e-30))) if gd.size else 0.0
    if rel > 1e-5:
        raise RuntimeError(f"parity gate ({what}): max relative score error {rel:.3e} > 1e-5 vs the {checker}")
    bits = float(np.mean(np.asarray(g.data, dtype=np.float32).view(np.uint32) == np.asarray(want.data, dtype=np.float32).view(np.uint32))) if gd.size else 1.0
    return {"checked_queries": rows, "checker": checker, "ids_bit_equal": True, "max_rel_score_err": rel,
            "scores_bit_equal_frac": bits}


def _max_over_ranks(dist, x):
    if dist is None:
        return float(x)
    import torch

    t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def _ncu_notes(workload, kernel):
    """What the committed ncu captures (profiles/ncu_traffic.json, written from `ncu --set full` runs) say about a kernel."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return json.load(f).get(workload, {}).get(kernel)
    except Exception:
        return None


def measure_xlinear(args, workload, rank, n_gpus, local, dist, barrier, lib, steps, warmup, strong=False, with_cpu=True,
                    with_clocks=True, dump_dir=None):
    """One XR-Linear workload on this rank's GPU.  strong=False: every rank its own batch of the workload's shape (weak
    scaling, replicas); strong=True: ONE batch of the workload's size, rows split over the ranks by nnz (strong scaling).
    Returns the JSON-able record (rank 0) -- parity-gated: raises if the GPU result differs from the reference."""
    from ctypes import byref, c_double, c_int, c_uint64

    from pecos_b200.core import ScipyCompressedSparseAllocator, ScipyCsrF32
    from pecos_b200.distributed import split_rows_by_nnz
    from pecos_b200.xlinear import XLinearModel

    c = lib.clib_float32
    wargs = argparse.Namespace(**vars(args))
    wargs.workload = workload
    folder, X, cfg = prepare_workload(wargs, rank, n_gpus, barrier, same_batch=strong)
    Q_total = X.shape[0] * (1 if strong else n_gpus)
    if strong and n_gpus > 1:
        cut = split_rows_by_nnz(X.indptr, n_gpus)
        X = X[cut[rank]:cut[rank + 1]]
        X.has_sorted_indices = True
    model = XLinearModel.load(folder, is_predict_only=True)
    h = model.model.model_chain
    depth = model.depth
    beam, topk = cfg["beam_size"], cfg["only_topk"]
    Q = X.shape[0]

    # ------------------------------------------------------------ resident batch + algorithmic-byte counters
    cx = ScipyCsrF32.init_from(X)
    c.pb200_xlinear_resident_upload_csr(h, byref(cx))
    c.pb200_xlinear_resident_predict(h, beam, None, topk, 1)
    stats = (c_uint64 * (7 * depth))()
    c.pb200_xlinear_get_stats(h, stats)
    st = np.array(list(stats), dtype=np.float64).reshape(depth, 7)  # chunks, sum R, sum m, sum e, sum c, sum nnz, beam out
    # SURVEY.md 8(d) yardstick: per (query, chunk) 32 + 4R + 16m + 8e + 4c ; per query and layer 8 nnz(x) + 8 min(k, sum c)
    survey_scores = 32 * st[:, 0] + 4 * st[:, 1] + 16 * st[:, 2] + 8 * st[:, 3] + 4 * st[:, 4] + 8 * st[:, 5]
    # Bytes the IMPLEMENTED kernels must move: no 4R row-list term (they look features up instead of streaming the row
    # list): one 32-byte sector per lookup (query-major kernels; the chunk-major kernel reads the query once per pair,
    # 8 B x nnz, and its chunk images once per CTA and chunk), 8 B per matched row extent, 8 B per entry, 4 B per output.
    topk_bytes = 4 * st[:, 4] + 8 * st[:, 6]

    def one_step():
        c.pb200_l2_flush()  # outside the event-timed region: every step starts with a cold L2
        return c.pb200_xlinear_resident_predict(h, beam, None, topk, 0)

    sampler = ClockSampler(local)
    if rank == 0 and with_clocks:
        sampler.start()  # started before the warm-up: nvidia-smi needs ~0.3 s before its first sample
    for _ in range(max(3, warmup)):
        one_step()
    if rank == 0 and with_clocks:
        sampler.mark()

    # ------------------------------------------------------------ timed region: K steps, device time, max over ranks
    c.pb200_xlinear_reset_profile(h)
    barrier()
    wall0 = time.perf_counter()
    step_ms = [one_step() for _ in range(steps)]
    wall1 = time.perf_counter()
    launches = int(c.pb200_xlinear_launches(h))
    sampler.pause()
    barrier()
    total_ms = _max_over_ranks(dist, sum(step_ms))
    ms_per_step = total_ms / steps
    value = Q_total / (ms_per_step * 1e-3)

    # ------------------------------------------------------------ parity gate on the result of the LAST timed step
    fetch = ScipyCompressedSparseAllocator()
    c.pb200_xlinear_resident_fetch(h, fetch.cfunc)
    got_resident = fetch.get()
    parity = parity_gate_xlinear(got_resident, folder, X, cfg, rows=(1024 if rank == 0 else 128), what=f"{workload} resident batch")
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, csr_result_arrays(got_resident))

    # ------------------------------------------------------------ per-kernel timing (CUDA events on the launch stream)
    c.pb200_xlinear_set_profile(h, 1)
    c.pb200_xlinear_reset_profile(h)
    prof_steps = max(3, min(steps, 10))
    for _ in range(prof_steps):
        one_step()
    prof = (c_double * (2 * depth))()
    c.pb200_xlinear_get_profile(h, prof)
    kid = (c_int * (2 * depth))()
    c.pb200_xlinear_get_kernel_ids(h, kid)
    c.pb200_xlinear_set_profile(h, 0)
    pm = np.array(list(prof), dtype=np.float64).reshape(depth, 2) / prof_steps
    peak, peak_src = measured_peak_gbs()
    # per feature of a (query, chunk) pair: the chunk-major kernel (id 4) reads the query once per pair (8 B); the query-major
    # lookup kernels read one 32-byte sector of the chunk's feature map per feature on top of the query (8 B, once per query)
    probe = np.array([{4: 8.0, 5: 40.0}.get(kid[2 * d], 32.0) for d in range(depth)])  # 5: query once per pair + one map sector per lookup
    pairs_per_query = st[:, 0] / np.maximum(st[:, 5] / np.maximum(X.nnz / max(Q, 1), 1e-9), 1.0)  # st5 = sum nnz over queries with a beam
    impl_scores = (32 * st[:, 0] + probe * st[:, 5] * np.maximum(pairs_per_query, 1.0) + 8 * st[:, 2] + 8 * st[:, 3] + 4 * st[:, 4]
                   + np.where(probe == 32.0, 8 * st[:, 5], 0.0))
    kernels = []
    for d in range(depth):
        kernels.append({"kernel": f"{SCORE_KERNELS[kid[2 * d]]}[layer {d}]", "ms": pm[d, 0], "algorithmic_bytes": float(impl_scores[d]),
                        "survey_formula_bytes": float(survey_scores[d]), "pairs": float(st[d, 0]), "matched_rows": float(st[d, 2]),
                        "entries": float(st[d, 3])})
        kernels.append({"kernel": f"{TOPK_KERNELS[kid[2 * d + 1]]}[layer {d}]", "ms": pm[d, 1], "algorithmic_bytes": float(topk_bytes[d])})
    dom = max(kernels, key=lambda k: k["ms"])
    achieved = dom["algorithmic_bytes"] / (dom["ms"] * 1e-3) / 1e9 if dom["ms"] > 0 else 0.0
    notes = _ncu_notes(workload, dom["kernel"].split("[")[0]) or {}
    step_bytes = float(impl_scores.sum() + topk_bytes.sum())
    roofline = {
        "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
        "traffic": notes.get("dram_bytes_per_launch") if isinstance(notes, dict) else notes,
        "kernel": dom["kernel"], "kernel_ms": dom["ms"], "algorithmic_bytes_per_launch": dom["algorithmic_bytes"],
        "algorithmic_bytes_definition": "bytes the implemented kernel must move per launch: per (query, chunk) pair 32 B chunk header + "
                                        "nnz(query) x 8 B (chunk-major kernel: the query is read once per pair, lookups hit the staged "
                                        "image) or x 32 B (query-major kernels: one feature-map sector per lookup) + 8 B per matched "
                                        "row + 8 B per entry + 4 B per output column; NOT the 4R row list the SURVEY 8d yardstick "
                                        "charges (kept per kernel as survey_formula_bytes)",
        "peak_source": peak_src,
        "ncu": notes if isinstance(notes, dict) else None,
        "whole_step": {"algorithmic_bytes": step_bytes, "achieved": step_bytes / (ms_per_step * 1e-3) / 1e9,
                       "bytes_per_query": step_bytes / max(Q, 1), "survey_formula_bytes": float(survey_scores.sum() + 8 * st[:, 6].sum())},
        "kernels": kernels,
    }

    # ------------------------------------------------------------ end to end through the C ABI with pinned host buffers
    ip = lib.pinned_empty(Q + 1, np.uint64)
    ix = lib.pinned_empty(max(X.nnz, 1), np.uint32)
    dv = lib.pinned_empty(max(X.nnz, 1), np.float32)
    ip.array[:] = X.indptr
    ix.array[: X.nnz] = X.indices
    dv.array[: X.nnz] = X.data
    cx_pinned = ScipyCsrF32.init_from_arrays(X.shape[0], X.shape[1], ip.array, ix.array, dv.array)

    def e2e_step():
        alloc = ScipyCompressedSparseAllocator()
        c.c_xlinear_predict_csr_f32(h, byref(cx_pinned), beam, None, topk, -1, alloc.cfunc)
        return alloc

    for _ in range(max(3, warmup)):
        e2e_step()
    barrier()
    sampler.resume()
    e2e_times = []
    for _ in range(steps):
        c.pb200_l2_flush()
        t0 = time.perf_counter()
        out = e2e_step()
        e2e_times.append(time.perf_counter() - t0)
    sampler.pause()
    barrier()
    # clocks / throttle reasons were sampled over BOTH timed regions (device-resident steps and end-to-end calls)
    clocks = sampler.stop() if (rank == 0 and with_clocks) else None
    e2e_total = _max_over_ranks(dist, sum(e2e_times))
    e2e_value = Q_total * steps / e2e_total
    h2d = int(ip.array.nbytes + X.nnz * 8)
    d2h = int(out.indices.nbytes + out.data.nbytes + 4 * Q)
    got_e2e = out.get()
    if not (np.array_equal(got_e2e.indptr, got_resident.indptr) and np.array_equal(got_e2e.indices, got_resident.indices)
            and np.array_equal(got_e2e.data.view(np.uint32), got_resident.data.view(np.uint32))):
        raise RuntimeError("parity gate (e2e): the C-ABI result of the host-buffer call differs from the resident-batch result")
    parity["e2e_equals_resident_bits"] = True
    # the same call with PAGEABLE host memory (what scipy hands the reference's ctypes shim)
    cx_pageable = ScipyCsrF32.init_from(X)
    pg_times = []
    for i in range(2 + min(steps, 10)):
        c.pb200_l2_flush()
        t0 = time.perf_counter()
        alloc = ScipyCompressedSparseAllocator()
        c.c_xlinear_predict_csr_f32(h, byref(cx_pageable), beam, None, topk, -1, alloc.cfunc)
        if i >= 2:
            pg_times.append(time.perf_counter() - t0)
    e2e_pageable = Q / (sum(pg_times) / len(pg_times))

    # ------------------------------------------------------------ CPU baseline beside it (rank 0, N=1 only)
    cpu = None
    if rank == 0 and n_gpus == 1 and with_cpu and not args.no_cpu_baseline:
        try:
            r = time_reference(folder, X, cfg, steps=5, warmup=2, budget_s=30.0)
            cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"],
                   "best": r["best"], "threads": r["threads"], "layout": r["layout"], "sweep": r["sweep"]}
        except ReferenceUnavailable as e:  # never substitute the scalar port for the reference
            print(f"bench.py: cpu_baseline unavailable: {e}", file=sys.stderr)
            cpu = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "unavailable", "sample": str(e)}

    cfgd = workload_config(workload, cfg, X)
    if strong:
        cfgd["queries_total"] = int(Q_total)
        cfgd["parallelism"] = "one batch, rows split over the ranks by nnz (strong scaling, no collective)"
    return {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": steps, "warmup": max(3, warmup),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": cfgd,
        "l2": "flushed between timed iterations (512 MiB memset outside the event-timed region)",
        "timing": "CUDA events on the engine stream per step, summed over steps, max over ranks",
        "parity": parity,
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": 1e3 * e2e_total / steps, "api": "c_xlinear_predict_csr_f32 (pinned host CSR in, scipy CSR out)",
                "pageable_value_per_gpu": e2e_pageable},
        "gpu_launches": launches,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "wall_s_timed_region": wall1 - wall0,
    }, (model, folder, X, cfg)


def measure_index_sharded(args, rank, n_gpus, local, dist, barrier, lib, whole, folder, X, cfg, rows=20000, calls=3):
    """BASELINE.json configs[4]: the leaf layer of the 3M-label tree split over the ranks' GPUs (contiguous chunk ranges),
    every rank scores the SAME queries on its shard, ONE NCCL all-gather of the packed per-rank top-k, merge.  The merged
    result must be bit-identical to the unsharded model's (`whole`, loaded on every rank for the query-sharded line)."""
    import torch

    from pecos_b200.distributed import ShardedXLinearModel

    Xs = X[: min(rows, X.shape[0])]
    Xs.has_sorted_indices = True
    beam, topk = cfg["beam_size"], cfg["only_topk"]
    sharded = ShardedXLinearModel.load(folder, device=local)
    got = sharded.predict(Xs, beam_size=beam, only_topk=topk)
    want = whole.predict(Xs, beam_size=beam, only_topk=topk)
    ok = bool(np.array_equal(got.indptr, want.indptr) and np.array_equal(got.indices, want.indices)
              and np.array_equal(got.data.view(np.uint32), want.data.view(np.uint32)))
    if not ok:
        raise RuntimeError("parity gate (index sharding): merged result differs from the unsharded prediction")
    barrier()
    times = []
    for _ in range(calls):
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        sharded.predict(Xs, beam_size=beam, only_topk=topk)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    dt = _max_over_ranks(dist, sum(times) / len(times))
    return {"workload": "synthetic-3m-sharded", "value": Xs.shape[0] / dt, "unit": UNIT, "n_gpus": n_gpus,
            "queries": int(Xs.shape[0]), "ms_per_call": 1e3 * dt, "bit_identical_to_unsharded": ok,
            "exchange": "ONE ncclAllGather of %d bytes per rank (16-byte {key, id, value} records)" % sharded.last_exchange_bytes,
            "shard_of_rank0": list(sharded.shard),
            "timing": "wall clock around ShardedXLinearModel.predict (host CSR in, H2D + kernels + all-gather + merge + D2H), max over ranks"}


def main():
    args = parse_args()
    if args.workload.startswith("hnsw"):
        return main_hnsw(args)
    if args.impl == "reference":
        return run_reference_arm(args)

    rank, world, local = dist_env()
    if world != args.gpus and world > 1:
        print(f"warning: WORLD_SIZE={world} != --gpus {args.gpus}", file=sys.stderr)
    n_gpus = max(world, 1)

    import __graft_entry__ as entry

    from pecos_b200 import core

    if rank == 0 and not os.path.exists(core.LIB_PATH):
        entry.build()

    dist = None
    if n_gpus > 1:
        import torch
        import torch.distributed as dist_mod

        torch.cuda.set_device(local)
        dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist = dist_mod

    def barrier():
        if dist is not None:
            dist.barrier()

    barrier()
    lib = core.get_clib()
    lib.require_gpu()
    lib.set_device(local)

    line, keep = measure_xlinear(args, args.workload, rank, n_gpus, local, dist, barrier, lib, args.steps, args.warmup,
                                 dump_dir=args.dump_outputs)
    del keep

    # ------------------------------------------------------------ the other target configurations, in the same run
    # (BASELINE.json configs[2..4]; each parity-gated like the headline; a failure is recorded, not fatal for the headline)
    secondary = {}
    if not args.no_secondary and args.workload == "eurlex-4k":
        t_sec = time.perf_counter()
        try:
            s_line, (whole, s_folder, s_X, s_cfg) = measure_xlinear(args, "synthetic-3m", rank, n_gpus, local, dist, barrier, lib,
                                                                    steps=5, warmup=3, strong=(n_gpus > 1), with_cpu=False, with_clocks=False)
            secondary["synthetic-3m"] = {k: s_line[k] for k in ("value", "unit", "n_gpus", "steps", "ms_per_step", "scaling", "config",
                                                                "parity", "e2e", "gpu_launches", "roofline")}
            if n_gpus > 1:
                # the batch of the strong-scaled line is per-rank; the index-sharded line needs the SAME queries on every rank
                from pecos_b200 import synth

                wcfg = dict(synth.WORKLOADS["synthetic-3m"])
                Xall = synth.make_queries(wcfg["query_seed"] + 77, 20000, wcfg["D"], wcfg["nnz_per_row"], synth.zipf_cdf(wcfg["D"]))
                secondary["synthetic-3m-sharded"] = measure_index_sharded(args, rank, n_gpus, local, dist, barrier, lib, whole, s_folder,
                                                                          Xall, s_cfg)
            del whole
        except Exception as e:  # noqa: BLE001
            secondary["error"] = f"{type(e).__name__}: {e}"
            print(f"bench.py: secondary workloads failed: {e}", file=sys.stderr)
        if n_gpus == 1:
            # the HNSW path (BASELINE configs[3] shape at a size whose index builds in seconds, dense + sparse), same gates
            for w in ("hnsw-100k", "hnsw-sparse-100k"):
                try:
                    h_line = measure_hnsw(args, w, rank, n_gpus, local, dist, barrier, steps=3, warmup=3, with_cpu=False)
                    secondary[w] = {k: h_line[k] for k in ("metric", "value", "unit", "n_gpus", "steps", "ms_per_step", "config", "parity",
                                                           "e2e", "gpu_launches", "roofline")}
                except Exception as e:  # noqa: BLE001
                    secondary[w] = {"error": f"{type(e).__name__}: {e}"}
                    print(f"bench.py: secondary workload {w} failed: {e}", file=sys.stderr)
        secondary["wall_s"] = time.perf_counter() - t_sec
    if rank == 0:
        if secondary:
            line["secondary"] = secondary
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    # Exactly ONE line goes to stdout (the JSON record): libraries that write banners to fd 1 (e.g. "NCCL version ...")
    # are diverted to stderr for the whole run; print() is re-pointed at the saved descriptor.
    sys.stdout.flush()
    _real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = _real_stdout
    rc = main()
    sys.stdout.flush()
    sys.exit(rc)
