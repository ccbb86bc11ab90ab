"""CPU: the bench.py contract that can be checked without a GPU — the reference arm prints exactly one JSON line with the
agreed keys, and the product arm refuses to run (non-zero exit, nothing on stdout) when there is no CUDA device."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, timeout=600):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=timeout, cwd=ROOT)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    p = _run("--impl", "reference", "--steps", "1", "--warmup", "0")
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0
    for k in ("metric", "value", "unit", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline"):
        assert k in d, k
    assert d["unit"] == "steps/s" and d["vs_baseline"] is None and "workload" in d["config"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    staged = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "MANIFEST.json"))
    assert cb["kind"] == ("reference" if staged else "port") and cb["value"] == d["value"] and cb["cores"] >= 1 and cb["sample"]
    assert d["extrapolated"] is False and d["same_config"] is True and d["measured_blocks"] == 28      # whole 28-block steps, not a depth sample
    assert abs(d["value"] * d["ms_per_step"] - 1000.0) < 1e-6 * 1000.0        # steps/s and ms/step describe the same run


def test_product_arm_has_no_cpu_path():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present: the product arm would run")
    p = _run("--steps", "1", "--warmup", "0", "--no-cpu", "--no-vae", timeout=300)
    assert p.returncode != 0
    assert p.stdout.strip() == ""


def test_bad_arguments_are_refused_before_any_work():
    for args in (("--steps", "0"), ("--impl", "reference", "--dump-outputs", "out")):
        p = _run(*args, timeout=120)
        assert p.returncode == 2 and p.stdout.strip() == "", args


def test_dump_outputs_writes_float32_and_samples_past_the_limit(tmp_path):
    import importlib.util

    import numpy as np
    import torch
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    flag = sys.dont_write_bytecode
    try:
        spec.loader.exec_module(bench)
    finally:
        sys.dont_write_bytecode = flag
    small = {"sample": torch.randn(1, 2048, 68), "model_output": torch.randn(1, 2048, 136).half()}
    bench.dump_outputs(str(tmp_path / "small"), small)
    for k, v in small.items():
        a = np.load(tmp_path / "small" / f"{k}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, v.float().numpy())
    big = {"recon_param": torch.randn(4, 2048, 3076), "sample": torch.randn(4, 2048, 68)}      # --config 5: 103 MB
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), big)
    written = sum(os.path.getsize(tmp_path / "a" / f"{k}.npy") for k in big)
    assert 0.99 * bench.DUMP_BYTES < written <= bench.DUMP_BYTES
    for k in big:
        a, b = (np.load(tmp_path / d / f"{k}.npy") for d in ("a", "b"))
        assert a.dtype == np.float32 and np.array_equal(a, b)                                    # the same sample every run
    assert np.isin(a, big["sample"].numpy()).all()


def test_reference_arm_under_torchrun_prints_once():
    """N > 1: rank 0 alone measures and prints; the other rank exits 0 without work."""
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2
