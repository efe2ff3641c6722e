"""GPU: `bench.py --dump-outputs` writes what the last timed step of the headline workload computed — the loss and the
gradients of both student logit tensors for the input set that step read."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_is_the_last_timed_step(tmp_path):
    K, W = 4, 3
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(K), "--warmup", str(W),
                        "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(out)],
                       capture_output=True, text=True, cwd=tmp_path, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["steps"] == K
    assert sorted(os.listdir(out)) == ["grad_outputs.npy", "grad_outputs_kd.npy", "loss.npy"]

    sys.path.insert(0, ROOT)
    import bench
    dev = torch.device("cuda", 0)
    w = bench.LogitKD(dev, 0)
    w.setup()
    ds = w.to_device(w.host_sets(1 + (W + K - 1) % w.nsets())[-1])
    loss = w.step(ds)
    want = {"loss.npy": loss.detach(), "grad_outputs.npy": ds[0].grad, "grad_outputs_kd.npy": ds[1].grad}
    for f, t in want.items():
        got = np.load(out / f)
        assert got.dtype == np.float32 and got.shape == tuple(t.shape), f
        torch.testing.assert_close(torch.from_numpy(got), t.float().cpu(), rtol=1e-2, atol=1e-6, msg=f)
    assert float(np.load(out / "loss.npy")) == pytest.approx(d["config"]["loss"], rel=1e-6)
