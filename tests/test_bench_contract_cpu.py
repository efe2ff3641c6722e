"""CPU: the reference arm of bench.py (`--impl reference`: the oracle port timed on the host cores) prints ONE JSON line
with the keys the driver reads, and the non-zero ranks of a torchrun launch exit 0 without work."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra=None, *flags):
    env = dict(os.environ)
    env.pop("RANK", None)
    env.update(env_extra or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                           *flags], capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)


def test_reference_arm_prints_the_contract_line():
    r = _run()
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "distill-loss fwd+bwd samples/s" and d["unit"] == "samples/s"
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["config"]["workload"] == "soft_kd_logits_b256_c1000_bf16"          # BASELINE.json configs[1]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "256" in cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_reference_arm_other_ranks_do_nothing():
    r = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_caps_size_and_repeats_its_sample(tmp_path):
    """--dump-outputs: float64 stays float64, other dtypes become float32, small outputs keep their shape, and an output
    above its share of the 64 MB budget is written as a sample that is the same in every run."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    g = torch.Generator().manual_seed(3)
    outs = {"loss": torch.tensor(2.5), "grad_a": torch.randn(256, 1000, generator=g).bfloat16(),
            "grad_b": torch.randn(512, 197, 192, generator=g), "grad_c": torch.randn(7, generator=g).double()}
    for d in ("a", "b"):
        bench.dump_outputs(outs, str(tmp_path / d))
    arrays = {f: np.load(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")}
    assert sorted(arrays) == ["grad_a.npy", "grad_b.npy", "grad_c.npy", "loss.npy"]
    assert sum(a.nbytes for a in arrays.values()) <= bench.DUMP_BYTES
    assert arrays["loss.npy"].dtype == np.float32 and float(arrays["loss.npy"]) == 2.5
    assert arrays["grad_a.npy"].shape == (256, 1000) and arrays["grad_a.npy"].dtype == np.float32
    assert np.array_equal(arrays["grad_a.npy"], outs["grad_a"].float().numpy())
    assert arrays["grad_c.npy"].dtype == np.float64 and np.array_equal(arrays["grad_c.npy"], outs["grad_c"].numpy())
    b = arrays["grad_b.npy"]
    assert b.ndim == 1 and 0 < b.size < outs["grad_b"].numel()
    assert np.isin(b, outs["grad_b"].numpy()).all()
    for f, a in arrays.items():
        assert np.array_equal(a, np.load(tmp_path / "b" / f)), f


def test_workload_registry_covers_the_baseline_configs():
    sys.path.insert(0, ROOT)
    import bench
    names = set(bench.WORKLOADS)
    assert bench.HEADLINE.name == "soft_kd_logits_b256_c1000_bf16"
    for must in ("curkd_early_3layers_b512_f32", "curkd_mid_4layers_b512_f32", "mgd_b512_f32", "saliency_mgd_m1_b512_f32",
                 "lrkd_r64_b512_f32", "wasskd_l1_b512_f32", "wasskd_sinkhorn_b512_f32", "deit_tiny_kd_step_soft_b256_bf16"):
        assert must in names, must
