"""-m gpu: bench.py --dump-outputs on the device writes what the last timed update computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_hold_the_last_timed_update(cuda, tmp_path):
    """The dumped loss is the one the JSON line reports for the last timed update, and the parameter sample holds
    updated weights, not the initial ones (bench.py builds the model from torch.manual_seed(1337))."""
    sys.path.insert(0, ROOT)
    import bench
    from speecht5_b200.models import make_args
    from speecht5_b200.tasks import SpeechT5Task
    d = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--batch", "4",
                        "--no-parity", "--no-cpu-baseline", "--dump-outputs", str(d)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["steps"] == 2
    losses, stats, sample = (np.load(d / f"{n}.npy") for n in ("losses", "stats", "params_sample"))
    assert losses.dtype == stats.dtype == sample.dtype == np.float32
    assert losses.shape == (1,) and losses[0] == np.float32(line["config"]["loss"])
    assert stats.shape[0] == 1 and np.isfinite(stats).all() and np.isfinite(sample).all()
    torch.manual_seed(1337)
    margs = make_args(bench.WORKLOAD["arch"], encoder_layerdrop=0.0, decoder_layerdrop=0.0, bert_init=True,
                      decoder_layers=bench.WORKLOAD["decoder_layers"], share_input_output_embed=True,
                      max_text_positions=600, max_speech_positions=1876)
    before = torch.cat([p.detach().reshape(-1).float() for p in SpeechT5Task(margs).build_model(margs).parameters()])
    idx = bench.dump_sample_index(before.numel())
    assert sample.shape == tuple(idx.shape)
    assert (torch.from_numpy(sample) != before[idx]).float().mean().item() > 0.8
