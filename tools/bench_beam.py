"""Beam search with joint CTC/attention scoring on one GPU: Base 12 + 6 ASR model, 8 x 10 s waveforms (T = 499 encoder
frames), V = 81, beam 5 and 10, ctc_weight 0 and 0.5, min_len = max_len so that every run takes the same number of
decoder steps. Reports, CUDA-event timed after a warm-up run of the same shape:
  ms_per_step         whole decode (encoder included) / decoder steps, prefix recomputation and key/value cache;
  ctc_ms_per_step     the CTC prefix kernel per step (events around st5_ctc_prefix_score, cached path);
  host_ms_per_step    the oracle's numpy scorer (the reference's method: one call per hypothesis) for the same shapes.
usage (GPU box): python tools/bench_beam.py [--steps 40] [--out profiles/r03_bench_beam.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        return q.splitlines()[0] if q else "unknown"
    except Exception:  # noqa: BLE001
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=40, help="decoder steps per decode (min_len = max_len)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    import beam_oracle as BO
    from speecht5_b200.beam import beam_search
    from speecht5_b200.models import T5TransformerModel, make_args
    from speecht5_b200.ops import RT
    assert torch.cuda.is_available(), "bench_beam.py measures on the GPU"
    dev = torch.device("cuda", 0)
    RT.dtype = torch.bfloat16
    torch.manual_seed(0)
    margs = make_args("t5_transformer_base_asr", build_speech_encoder=True, build_text_decoder=True, bert_init=True,
                      encoder_layerdrop=0.0, decoder_layerdrop=0.0, max_text_positions=600)
    model = T5TransformerModel.build_model(margs).to(dev).eval()
    wav = torch.randn(8, 160000, device=dev) * 0.1
    wpm = torch.zeros(8, 160000, dtype=torch.bool, device=dev)
    n = args.steps
    out = {"gpu": _gpu_info(), "dtype": "bf16", "batch": 8, "wave_s": 10.0, "decoder_steps": n + 1, "runs": []}
    for beam in (5, 10):
        for w in (0.0, 0.5):
            row = {"beam": beam, "ctc_weight": w}
            for name, uc in (("prefix", False), ("kv_cache", True)):
                def run(stats=None):
                    return beam_search(model, wav, wpm, beam_size=beam, ctc_weight=w, max_len_b=n, min_len=n,
                                       blank=80, mask_idx=79, use_cache=uc, stats=stats)
                run()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                stats = {}
                e0.record()
                run(stats if w > 0 and uc else None)
                e1.record()
                torch.cuda.synchronize()
                row[f"{name}_ms_per_step"] = e0.elapsed_time(e1) / (n + 1)
                if stats:
                    ev = stats["ctc_events"]
                    row["ctc_ms_per_step"] = sum(a.elapsed_time(b) for a, b in ev) / len(ev)
                    row["ctc_share_of_cached_step"] = row["ctc_ms_per_step"] / row["kv_cache_ms_per_step"]
            if w > 0:  # the reference's method: numpy, one scorer call per hypothesis per step (K = int(7 beam))
                enc = model.forward_encoder(wav, padding_mask=wpm)
                x = model.get_normalized_probs_for_ctc(enc, log_probs=True)[:, 0].cpu().numpy()  # [T, V]
                T = x.shape[0]
                r = BO.ctc_initial_state(x, 80)
                Kc = min(81, int(7 * beam))
                cs = np.arange(Kc)
                reps = 3
                t0 = time.perf_counter()
                for _ in range(reps):
                    for _h in range(8 * beam):
                        BO.ctc_prefix_score(x, r, 5, 10, cs, 80, 2)
                host = (time.perf_counter() - t0) * 1e3 / reps
                row["host_ms_per_step"] = host
                row["encoder_frames"] = T
                row["gpu_vs_host_speedup"] = host / row["ctc_ms_per_step"]
            out["runs"].append(row)
            print(json.dumps(row), file=sys.stderr)
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
