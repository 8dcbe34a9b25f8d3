"""CPU tests of bench.py's contract: the reference arm (`--impl reference`) times the UNMODIFIED reference library and prints
one JSON line with the agreed keys; without oracle/_ref it must fail instead of timing a substitute; the product arm has no CPU
fallback."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
        "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"}


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                          env=e, cwd=ROOT)


def test_reference_arm_contract_xlinear(built, have_ref, tmp_path):
    if not have_ref:
        pytest.skip("oracle/_ref not built")
    r = _run(["--impl", "reference", "--workload", "synthetic-small", "--steps", "2", "--warmup", "1", "--cache-dir", str(tmp_path)])
    assert r.returncode == 0, r.stderr[-1500:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, "exactly one JSON line on stdout"
    d = json.loads(lines[0])
    assert KEYS <= set(d), KEYS - set(d)
    assert d["impl"] == "reference" and d["cpu_baseline"]["kind"] == "reference" and d["gpu_launches"] == 0
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["config"]["workload"] == "synthetic-small" and "model" not in d["config"]
    assert "sweep" in json.dumps(d["cpu_baseline"]) or "best of the sweep" in d["cpu_baseline"]["sample"]


def test_reference_arm_contract_sparse_hnsw(built, have_ref, tmp_path, monkeypatch):
    """The HNSW reference arm on a tiny sparse workload: index built by the reference's HNSW.train, searched by its predict."""
    if not have_ref:
        pytest.skip("oracle/_ref not built")
    code = ("import sys, json; sys.argv = ['bench.py', '--impl', 'reference', '--workload', 'hnsw-tiny', '--steps', '2', '--warmup', '1', "
            "'--cache-dir', %r]\n"
            "import importlib.util\n"
            "spec = importlib.util.spec_from_file_location('bench', %r); b = importlib.util.module_from_spec(spec); spec.loader.exec_module(b)\n"
            "b.HNSW_WORKLOADS['hnsw-tiny'] = dict(N=3000, d=2000, nnz=20, M=8, efC=40, Q=200, efS=50, topk=10, metric='ip', sparse=True)\n"
            "sys.exit(b.main())\n" % (str(tmp_path), os.path.join(ROOT, "bench.py")))
    r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-1500:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.strip()][-1])
    assert KEYS <= set(d)
    assert d["impl"] == "reference" and d["cpu_baseline"]["kind"] == "reference" and d["value"] > 0
    assert d["config"]["rows"].startswith("csr") and d["metric"].endswith("(efS=50)")


def test_reference_arm_fails_without_the_reference_library(built, tmp_path):
    """No oracle/_ref -> exit code != 0 and no number (round 1 silently timed the scalar port instead)."""
    code = ("import sys; sys.argv = ['bench.py', '--impl', 'reference', '--workload', 'synthetic-small', '--steps', '1', '--warmup', '1', "
            "'--cache-dir', %r]\n"
            "import oracle; oracle.have_ref = lambda: False; oracle.REF_LIB = '/nonexistent/libpecos_float32.so'\n"
            "import oracle.ref as r; r.REF_LIB = oracle.REF_LIB; r._lib = None\n"
            "import importlib.util\n"
            "spec = importlib.util.spec_from_file_location('bench', %r); b = importlib.util.module_from_spec(spec); spec.loader.exec_module(b)\n"
            "sys.exit(b.main())\n" % (str(tmp_path), os.path.join(ROOT, "bench.py")))
    r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, cwd=ROOT)
    assert r.returncode != 0
    assert not [ln for ln in r.stdout.splitlines() if ln.strip().startswith("{") and '"value"' in ln]


def test_product_arm_needs_a_gpu(built, tmp_path):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is visible")
    r = _run(["--workload", "synthetic-small", "--steps", "1", "--warmup", "1", "--no-cpu-baseline", "--no-secondary", "--cache-dir", str(tmp_path)])
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)


def test_sparse_row_generator_is_deterministic_and_canonical():
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    argv, sys.argv = sys.argv, ["bench.py"]
    try:
        spec.loader.exec_module(b)
    finally:
        sys.argv = argv
    A, B = b.make_sparse_rows(5, 500, 3000, 40), b.make_sparse_rows(5, 500, 3000, 40)
    assert (A != B).nnz == 0 and A.has_canonical_format and A.dtype == np.float32
    assert 30 < A.nnz / A.shape[0] < 45
    assert np.allclose(np.sqrt(np.asarray(A.multiply(A).sum(axis=1)).ravel()), 1.0, atol=1e-5)


def test_dump_outputs_writes_float_arrays_within_the_limit(tmp_path):
    """--dump-outputs: the csr result of the timed step round-trips through float arrays; a result over the byte limit is cut to
    the same seeded sample of rows every time; nothing over the limit is written."""
    import importlib.util

    import scipy.sparse as smat

    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    argv, sys.argv = sys.argv, ["bench.py"]
    try:
        spec.loader.exec_module(b)
    finally:
        sys.argv = argv
    Y = smat.random(300, 5000, density=0.002, format="csr", dtype=np.float32, random_state=3)
    full = b.csr_result_arrays(Y)
    b.dump_outputs(str(tmp_path / "full"), full)
    got = {k: np.load(str(tmp_path / "full" / (k + ".npy"))) for k in full}
    assert all(got[k].dtype in (np.float32, np.float64) for k in got)
    back = smat.csr_matrix((got["scores"], got["labels"].astype(np.int64), got["indptr"].astype(np.int64)), shape=Y.shape)
    assert (back != Y).nnz == 0 and np.array_equal(got["rows"], np.arange(300))
    small, again = b.csr_result_arrays(Y, max_bytes=4096), b.csr_result_arrays(Y, max_bytes=4096)
    assert 0 < small["rows"].size < 300 and sum(a.nbytes for a in small.values()) <= 4096
    assert all(np.array_equal(small[k], again[k]) for k in small)
    rows = small["rows"].astype(np.int64)
    assert (smat.csr_matrix((small["scores"], small["labels"].astype(np.int64), small["indptr"].astype(np.int64)),
                            shape=(rows.size, Y.shape[1])) != Y[rows]).nnz == 0
    with pytest.raises(RuntimeError):
        b.dump_outputs(str(tmp_path / "big"), {"x": np.zeros(b.DUMP_LIMIT_BYTES // 8 + 1)})
    assert not os.path.exists(str(tmp_path / "big"))
    r = _run(["--steps", "0"])
    assert r.returncode != 0 and "--steps" in r.stderr
