"""CPU tests of bench.py's contract pieces that need no GPU: the reference arm's JSON line (run as the
driver runs it, on the tiny config) and the launch-list lookup behind `roofline.traffic`."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--model", "tiny",
                          "--size", "16", "--steps", "2", "--warmup", "1"], capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1
    assert d["higher_is_better"] is True and d["value"] > 0 and d["data"] == "synthetic"
    for key in ("metric", "unit", "ms_per_step", "dtype", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 == d["e2e"]["d2h_bytes_per_step"]
    assert "workload" in d["config"] and "model" not in d["config"]


def _bench_module():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    argv, sys.argv = sys.argv, ["bench.py"]
    try:
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
    finally:
        sys.argv = argv
    return m


def test_reference_arm_dumps_the_output_of_its_last_step(tmp_path):
    """Same arguments, same inputs: two runs write the same float32 array of the UNet's output shape."""
    got = []
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--model", "tiny",
                              "--size", "16", "--steps", "2", "--warmup", "1", "--dump-outputs", str(tmp_path / run)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        assert sorted(os.listdir(tmp_path / run)) == ["sample.npy"]
        a = np.load(tmp_path / run / "sample.npy")
        assert a.dtype == np.float32 and a.shape == (2, 4, 16, 16) and np.isfinite(a).all() and a.any()
        got.append(a)
    assert np.array_equal(*got)


def test_reference_arm_runs_exactly_the_requested_steps_however_slow_the_host(monkeypatch):
    """A host clock that makes every forward look 1000 s long must not cut --steps or --warmup, so the
    last timed step (the one --dump-outputs writes) depends on the arguments only."""
    import argparse
    import itertools

    from oracle import unet_oracle as uo
    m = _bench_module()
    timesteps, build = [], uo.build_unet

    def counting_build(*a, **k):
        net = build(*a, **k)

        def forward(s, t, e, **kw):
            timesteps.append(float(t))
            return net(s, t, e, **kw)
        return forward

    monkeypatch.setattr(uo, "build_unet", counting_build)
    clock = itertools.count(0.0, 1000.0)
    monkeypatch.setattr(m.time, "perf_counter", lambda: next(clock))
    r = m.cpu_reference_run(argparse.Namespace(model="tiny", batch=2, size=16), steps=3, warmup=2)
    assert r["steps"] == 3 and r["warmup"] == 2
    assert timesteps == [999.0, 999.0, 999.0, 949.0, 899.0]
    assert tuple(r["sample_out"].shape) == (2, 4, 16, 16)


def test_dump_outputs_samples_what_exceeds_the_budget(tmp_path):
    m = _bench_module()
    small, big = torch.randn(2, 3), torch.arange(10000.0).reshape(100, 100)
    m.dump_outputs(str(tmp_path), {"small": small, "big": big}, budget=2 * (4096 + 12 * 500))
    assert np.array_equal(np.load(tmp_path / "small.npy"), small.numpy())
    assert not (tmp_path / "small_index.npy").exists()
    idx, vals = np.load(tmp_path / "big_index.npy"), np.load(tmp_path / "big.npy")
    assert idx.dtype == np.float64 and vals.dtype == np.float32 and idx.shape == vals.shape == (500,)
    assert np.all(np.diff(idx) > 0) and np.array_equal(vals, idx.astype(np.float32))
    assert sum(f.stat().st_size for f in tmp_path.iterdir()) <= 2 * (4096 + 12 * 500)


def test_ncu_traffic_picks_the_launch_list_of_its_workload():
    m = _bench_module()
    a = m.ncu_traffic("gemm_tc_kernel", "sd15-b2-s64")
    b = m.ncu_traffic("gemm_tc_kernel", "sd15-b8-s64")
    assert a["traffic"] and a["traffic_source"].endswith("_ncu_launch_summary.json")
    assert b["traffic"] and b["traffic_source"].endswith("_ncu_launch_summary_b8.json") and b["traffic"] > a["traffic"]
    none = m.ncu_traffic("gemm_tc_kernel", "no-such-workload")
    assert none["traffic"] is None and "no-such-workload" in none["traffic_note"]
