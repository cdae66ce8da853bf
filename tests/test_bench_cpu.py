"""CPU: the reference arm of bench.py (`--impl reference`, the oracle port on the host cores) prints ONE JSON line with
the contract's keys; non-zero ranks of a multi-rank launch exit without work."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra, *args):
    env = dict(os.environ, **env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", *args], env=env,
                          capture_output=True, text=True, timeout=600, cwd=ROOT)


def test_reference_arm_prints_the_contract_line():
    r = _run({}, "--steps", "1", "--warmup", "1", "--cpu-batch", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"].startswith("utterances/sec") and d["unit"] == "utterances/s"
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "sample" in d["cpu_baseline"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert abs(d["e2e"]["value"] - d["value"]) < 1e-9 and "workload" in d["config"]


def test_reference_arm_other_ranks_exit_without_work():
    r = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, "--gpus", "2", "--steps", "1", "--warmup", "0")
    assert r.returncode == 0 and not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]


def test_dump_outputs_writes_float32_arrays_and_a_fixed_parameter_sample(tmp_path):
    """--dump-outputs: what train_step returned plus a seeded sample of the updated parameters, float32, identical for
    identical parameters (two builds are compared array by array)."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    from types import SimpleNamespace
    model = torch.nn.Sequential(torch.nn.Linear(300, 200), torch.nn.Linear(200, 4))
    trainer = SimpleNamespace(model=model, consolidate=lambda: None)
    out = (torch.tensor([1.5], dtype=torch.float64), torch.arange(6.0).reshape(1, 6))
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), trainer, out)
    bench.dump_outputs(str(tmp_path / "rank1"), trainer, out, rank=1)
    assert not (tmp_path / "rank1").exists()  # (only rank 0 writes)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["losses.npy", "params_sample.npy", "stats.npy"] == sorted(os.listdir(tmp_path / "b"))
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype == np.float32 and np.array_equal(a, b), n
    assert np.load(tmp_path / "a" / "losses.npy").tolist() == [1.5]
    flat = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
    sample = np.load(tmp_path / "a" / "params_sample.npy")
    assert sample.shape == (min(bench.DUMP_PARAM_SAMPLE, flat.numel()),)
    assert np.isin(sample, flat.numpy()).all()


def test_dump_outputs_is_refused_where_it_is_not_implemented(tmp_path):
    r = _run({}, "--steps", "1", "--dump-outputs", str(tmp_path / "out"))
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and not (tmp_path / "out").exists()
