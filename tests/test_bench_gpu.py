"""GPU test of bench.py's B200 arm: `--dump-outputs` writes what the last timed step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZE = 32


def _bench_dump(steps, out_dir):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--model", "tiny",
                          "--size", str(SIZE), "--steps", str(steps), "--warmup", "1", "--no-cpu-baseline",
                          "--no-roofline", "--no-extras", "--dump-outputs", str(out_dir)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == steps
    assert sorted(os.listdir(out_dir)) == ["sample.npy"]
    a = np.load(out_dir / "sample.npy")
    assert a.dtype == np.float32 and a.shape == (2, 4, SIZE, SIZE)
    return a


def _oracle_step(i):
    """The fp32 oracle on bench.py's weights and on the inputs of its timed step i (one GPU)."""
    from oracle import unet_oracle as uo
    from sfast_b200.synthetic import CONFIGS
    from sfast_b200.unet_spec import random_state_dict, spec_from_config
    sd = random_state_dict(spec_from_config(CONFIGS["tiny"]), seed=0, dtype=torch.float16)
    m = uo.UNet2DConditionModel(uo.tiny_config())
    m.load_state_dict({k: v.float() for k, v in sd.items()})
    m = m.eval().cuda()
    g = torch.Generator().manual_seed(1234)
    s = [torch.randn(2, 4, SIZE, SIZE, generator=g).half() for _ in range(4)]
    e = [torch.randn(2, 77, 128, generator=g).half() for _ in range(4)]
    with torch.no_grad():
        ref = m(s[i % 4].float().cuda(), torch.tensor(999.0 - 50 * (i % 20), device="cuda"),
                e[i % 4].float().cuda()).sample
    return ref.cpu()


@pytest.mark.gpu
def test_b200_arm_dumps_the_output_of_its_last_timed_step(tmp_path):
    a, b, c = _bench_dump(2, tmp_path / "a"), _bench_dump(2, tmp_path / "b"), _bench_dump(3, tmp_path / "c")
    assert np.array_equal(a, b)          # same arguments, same inputs, same output
    assert not np.array_equal(a, c)      # the last step of 3 has other inputs than the last step of 2
    for got, last in ((a, 1), (c, 2)):
        ref = _oracle_step(last)
        d = (torch.from_numpy(got) - ref).abs()
        err = max((d.max() / ref.abs().max()).item(), (d / (ref.abs() + ref.pow(2).mean().sqrt())).max().item())
        assert err < 1e-2, (last, err)
