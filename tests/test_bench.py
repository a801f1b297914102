"""bench.py's driver contract: the reference arm runs anywhere (oracle/ only, never the product package), the GPU arm
refuses to run without a GPU, and (GPU) the default arm prints ONE JSON line with the keys the driver reads."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "cpu_baseline"}


def _run(args, timeout=600, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, BENCH, *args], capture_output=True, text=True, timeout=timeout, cwd=ROOT, env=e)


def test_reference_arm_prints_the_contract_line_and_stays_off_the_product_package(tmp_path):
    # a probe appended through PYTHONSTARTUP-free means: sitecustomize is not ours to touch, so ask the child itself
    code = ("import runpy, sys; sys.argv = ['bench.py', '--impl', 'reference', '--steps', '2', '--warmup', '0', "
            "'--ref-batch', '4', '--dump-outputs', %r]; runpy.run_path(%r, run_name='__main__'); "
            "print('LOADED_PRODUCT', any(m == 'honk2_b200' or m.startswith('honk2_b200.') for m in sys.modules), file=sys.stderr)"
            % (str(tmp_path), BENCH))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert BASE_KEYS <= set(d), BASE_KEYS - set(d)
    assert d["impl"] == "reference" and d["gpu_launches"] == 0 and d["higher_is_better"] is True
    assert d["metric"].startswith("res15 utterances/sec") and d["unit"] == "utterances/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["model_config"] == "res15" and d["config"]["batch_per_gpu"] == 8192
    assert "LOADED_PRODUCT False" in r.stderr, "the reference arm must not import honk2_b200"
    y = np.load(tmp_path / "logits.npy")
    assert y.shape == (4, 12) and y.dtype == np.float32
    # the dump is the LAST timed step's logits: step i of the arm runs the clips of seed 1000 + warmup + i
    from oracle import bench_ref
    bench, threads = load_bench(), torch.get_num_threads()
    try:
        ref = bench_ref.CpuReference("res15")
        last, first = (ref.step(bench.pcm_round(bench_ref.broadband(4, N=16000, seed=s)))[2].numpy() for s in (1001, 1000))
    finally:
        torch.set_num_threads(threads)
    assert np.allclose(y, last, rtol=0, atol=1e-5) and not np.allclose(y, first, rtol=0, atol=1e-3)


def load_bench():
    spec = importlib.util.spec_from_file_location("bench_under_test", BENCH)
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_dump_outputs_keeps_a_fixed_sample_under_the_limit(tmp_path):
    bench = load_bench()
    big = torch.arange(1000 * 12, dtype=torch.float64).view(1000, 12)
    small = torch.ones(10, 12)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"big": big, "small": small}, limit=2 * 100 * 12 * 4)
    a, b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert a.dtype == np.float32 and a.shape == (100, 12) and np.array_equal(a, b)
    rows = a[:, 0].astype(np.int64) // 12
    assert np.all(np.diff(rows) > 0) and np.array_equal(a, big.numpy()[rows])
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), small.numpy())


def test_steps_must_be_positive():
    r = _run(["--impl", "reference", "--steps", "0"])
    assert r.returncode != 0 and "--steps must be at least 1" in r.stderr


def test_reference_arm_on_other_ranks_is_silent():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "0"], env={"RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_gpu_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = _run(["--steps", "1"])
    assert r.returncode != 0
    assert "no CPU path" in (r.stderr + r.stdout)


@pytest.mark.gpu
def test_gpu_arm_prints_the_contract_line(tmp_path):
    r = _run(["--steps", "2", "--warmup", "3", "--batch", "592", "--no-cpu-baseline", "--no-other-configs",
              "--dump-outputs", str(tmp_path)], timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert (BASE_KEYS | {"clocks", "roofline", "e2e_pcm16", "parity", "parity_mode"}) <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 3 and d["dtype"] == "bf16" and d["gpu_launches"] >= 2 * 3
    assert d["value"] > 0 and d["e2e"]["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] == 592 * 16000 * 4
    assert d["e2e_pcm16"]["h2d_bytes_per_step"] == 592 * 16000 * 2 and d["e2e_pcm16"]["logits_bit_identical_to_f32_path"] is True
    ro = d["roofline"]
    assert ro["bound"] == "tensor" and ro["unit"] == "TFLOP/s" and 0 < ro["frac"] < 1 and abs(ro["frac"] - ro["achieved"] / ro["peak"]) < 1e-9
    assert d["parity_mode"]["precision"] == "bf16x3" and d["parity_mode"]["parity"]["argmax_agree"] == 1.0
    assert d["parity_mode"]["parity"]["max_logit_err"] <= 1e-3
    # the last timed step of each path: the same clips, and every mode is bit-reproducible and batch-order invariant
    y = np.load(tmp_path / "logits.npy")
    assert y.shape == (592, 12) and y.dtype == np.float32 and np.isfinite(y).all()
    assert np.array_equal(np.load(tmp_path / "e2e_logits.npy"), y)
    assert np.array_equal(np.load(tmp_path / "e2e_pcm16_logits.npy"), y)
