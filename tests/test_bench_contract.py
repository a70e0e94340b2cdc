"""Tests of bench.py's contract: the reference arm prints one JSON line with the agreed keys, our arm refuses to run
without a GPU instead of falling back to anything, and (on the GPU) --dump-outputs writes the last timed step's outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and d["unit"] == "images/sec" and d["higher_is_better"] is True
    assert d["metric"].startswith("64x64 images/sec IAN encode->decode")
    assert d["value"] > 0 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]


@pytest.mark.skipif(torch.cuda.is_available(), reason="CPU-only behaviour")
def test_our_arm_has_no_cpu_fallback():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "3"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0
    assert "no CPU fallback" in (out.stderr + out.stdout)


def test_bad_step_count_and_dump_request_are_refused(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                             timeout=600, cwd=ROOT)
        assert out.returncode == 2 and "error:" in out.stderr, (extra, out.stderr[-2000:])
    assert os.listdir(tmp_path) == []


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(npe, tmp_path):
    """--steps sets the timed steps; --dump-outputs writes what the library returns for bench.py's input (batch 256 drawn
    from default_rng(1234), synthetic weights of seed 0), bit for bit: the path has no atomics."""
    from oracle import weights as ow
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-cpu-baseline",
                          "--no-edit", "--no-full", "--no-config5", "--dump-outputs", str(tmp_path / "dump")],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 2 and d["gpu_launches"] == 14 * 2
    dump = tmp_path / "dump"
    assert sorted(os.listdir(dump)) == ["xhat.npy", "z.npy"]
    assert sum(os.path.getsize(dump / f) for f in os.listdir(dump)) <= 64 << 20
    z, xh = np.load(dump / "z.npy"), np.load(dump / "xhat.npy")
    assert z.dtype == xh.dtype == np.float32 and z.shape == (256, 100) and xh.shape == (256, 3, 64, 64)
    x = np.random.default_rng(1234).uniform(-1, 1, (256, 3, 64, 64)).astype(np.float32)
    m = npe.IAN("IAN_simple.py", dnn=True, weights=ow.make_simple_weights(0), device=0)
    try:
        want_xh, want_z = m.reconstruct(x, return_z=True)
    finally:
        m.close()
    assert np.array_equal(z, want_z) and np.array_equal(xh, want_xh)


def test_reference_arm_nonzero_ranks_do_no_work():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert out.returncode == 0 and not [l for l in out.stdout.splitlines() if l.startswith("{")]


def test_roofline_traffic_resolves_from_the_committed_ncu_summary():
    """`roofline.traffic` is read at run time from profiles/r2_ncu_tc_kernels_full_summary.csv (the ncu --set full capture of
    the same command), not a constant in the source: the 9 tap-GEMM launches of one batch-256 step must all be there, their
    DRAM bytes between the algorithmic 0.94 GB and 2x that, and the bench line committed beside it must carry that figure."""
    sys.path.insert(0, ROOT)
    import importlib
    bench = importlib.import_module("bench")
    t = bench.ncu_traffic("tapgemm_tc", 9)
    assert t is not None and 0.94e9 <= t <= 1.9e9, t
    assert bench.ncu_traffic("tapgemm_tc", 10) is None           # a step has exactly nine of them: more cannot be resolved
    line = [l for l in open(os.path.join(ROOT, "profiles", "r2_bench_n1.json")) if l.startswith("{")][-1]
    d = json.loads(line)
    assert abs(d["roofline"]["traffic"] - t) <= 0.1 * t          # (that line was printed just before the capture was refreshed in the same call)
    assert d["roofline"]["traffic_src"].endswith("r2_ncu_tc_kernels_full_summary.csv")
    assert d["roofline"]["frac"] == d["roofline"]["frac_burst"] and 0.5 < d["roofline"]["frac_burst"] <= 1.0
    assert d["gpu_launches"] == 14 * d["steps"]                  # conv1, 3 convs, fc1 + finalize, head + finalize, sample, fc2, 3 deconvs, dec_out
