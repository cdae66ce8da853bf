#!/usr/bin/env python
"""Benchmark of the SpeechT5 hot path on B200: BASELINE.json metric "utterances/sec (TTS fine-tune step, 10s@16kHz)".

  python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU under torchrun for N>1)
  python bench.py --impl reference --gpus N --steps K ...  # the reference math (CPU oracle port) on the host cores

A step = one full update of SpeechT5-Base (12 enc + 6 dec, d=768) on a batch of 32 synthetic 10 s utterances per GPU
(160 text tokens -> 626 mel frames -> 313 decoder steps at r=2): forward, TTS criterion (L1 + BCE + guided attention),
backward, gradient exchange (N>1), grad-norm clip 25, Adam -- dropout active, nothing cached or skipped.
Prints ONE JSON line (see the task contract); `value` has inputs resident in HBM, `e2e` goes through
B200Trainer.train_step with pinned host batches (H2D inside the timed region, loss statistics read back every step).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = dict(arch="t5_transformer_base_asr", batch_per_gpu=32, text_len=160, mel_frames=626, decoder_steps=313,
                encoder_layers=12, decoder_layers=6)
# SURVEY.md 8(d): forward 67.4 GFLOP/utt, training step = 3x forward (GEMM-shaped work)
ALGO_GFLOP_PER_UTT_STEP = 202.0


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed updates of the tts / tts_ragged / asr / pretrain workloads (both the resident and the "
                         "end-to-end pass). Bounded legs use their own counts, each reported in its JSON entry: the "
                         "tts parity leg times max(3, min(K, 6)) updates, the CPU baselines a fixed 3 (asr) or 8 (tts) "
                         "updates (--impl reference: max(1, min(K, 10))), and hifigan max(1, K // 10) passes over its "
                         "512 spectrograms")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=WORKLOAD["batch_per_gpu"])
    ap.add_argument("--decoder-layers", type=int, default=WORKLOAD["decoder_layers"])
    ap.add_argument("--workload", default="tts", choices=["tts", "tts_ragged", "asr", "hifigan", "pretrain"],
                    help="tts = the BASELINE.json metric (config 2, default); tts_ragged = the same model on a stream of "
                         "distinct batch shapes through the shape-bucket graph cache; asr = config 3 (speech -> text "
                         "fine-tune step); hifigan = config 5 (vocoder inference, waveform samples/s); pretrain = config "
                         "4 (t5_transformer_large joint pre-training update: one speech + one text micro-batch)")
    ap.add_argument("--pretrain-arch", default="t5_transformer_large", choices=["t5_transformer_large", "t5_transformer_base"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-parity", action="store_true",
                    help="skip the parity-mode (fp32 activations, 3-pass split-bf16 GEMMs) leg and the mel-L2 measurement")
    ap.add_argument("--exchange", default=None, choices=["shard", "allreduce"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-batch", type=int, default=2)
    ap.add_argument("--profile-step", action="store_true",
                    help="run 2 eager warm-up updates, then ONE eager update between cudaProfilerStart/Stop and exit "
                         "(for `ncu --profile-from-start off`); prints no bench line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="tts workload: after the timed steps, write what the last timed update returned and a seeded "
                         "sample of the parameters it updated as DIR/<name>.npy (float32), to compare two builds")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.workload != "tts" or args.profile_step):
        ap.error("--dump-outputs is implemented for the timed tts workload of --impl b200")
    return args


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def window(self, t0, t1):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.rows:
            if ts < t0 or ts > t1 + 0.2:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0])); mx = max(mx, float(f[1]))
            except Exception:  # noqa: BLE001
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()


# ------------------------------------------------------------------------------------------------ reference arm
def run_reference(args, emit=True):
    """The reference's own CPU path for this metric: the oracle port of the fairseq modules (the reference cannot be
    installed here: fairseq pins omegaconf<2.1 / numpy<1.24, espnet absent -- DESIGN.md), fp32, all host threads."""
    import torch
    from oracle.speecht5_oracle import T5TransformerModelOracle, base_args, synthetic_tts_batch, tts_loss
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    cores = min(os.cpu_count() or 1, 32)  # beyond ~32 threads the small CPU ops of this model only contend
    torch.set_num_threads(cores)
    torch.manual_seed(1337)
    B = args.cpu_batch
    model = T5TransformerModelOracle(base_args(encoder_layerdrop=0.0, decoder_layerdrop=0.0,
                                               decoder_layers=args.decoder_layers, bert_init=True)).train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-4, betas=(0.9, 0.98), eps=1e-8)
    sample = synthetic_tts_batch(B, WORKLOAD["text_len"], WORKLOAD["mel_frames"], seed=1)

    def step():
        opt.zero_grad(set_to_none=False)
        loss = tts_loss(model(**sample["net_input"]), sample)[0]
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 25.0)
        opt.step()
        return loss.item()

    warm = 1
    steps = max(1, min(args.steps, 10)) if emit else 8  # ~10-15 s of CPU work: a bounded sample of the same workload
    for _ in range(warm):
        step()
    t0 = time.time()
    for _ in range(steps):
        step()
    dt = (time.time() - t0) / steps
    val = B / dt
    cb = {"value": val, "unit": "utterances/s", "cores": cores, "kind": "port",
          "sample": f"{steps} full update steps of SpeechT5-Base on {B} x 10 s utterances (same shapes as one "
                    f"GPU batch row), fp32 PyTorch CPU, {cores} threads, {dt:.2f} s/step"}
    if emit:
        line = {"impl": "reference", "metric": "utterances/sec (TTS fine-tune step, 10s@16kHz)", "value": val,
                "unit": "utterances/s", "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": dt * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": "SpeechT5-Base TTS fine-tune step, 10 s utterances (160 tokens -> 626 mel "
                                       f"frames), CPU batch {B}", **{k: WORKLOAD[k] for k in ("text_len", "mel_frames")}},
                "cpu_baseline": cb,
                "e2e": {"value": val, "unit": "utterances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), flush=True)
    return cb



# ------------------------------------------------------------------------------------------------ shared pieces
def _init_dist():
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)
    return world, rank, local, dev


def _timed_steps(trainer, batches, steps, warmup, world, dev, read_back):
    """W untimed + exactly K timed updates, barrier + synchronize on both sides, CUDA events, max over ranks."""
    import torch
    import torch.distributed as dist
    from speecht5_b200 import kernels as K

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    out = None
    micro = lambda b: b if isinstance(b, list) else [b]  # noqa: E731  (an element may already be a list of micro-batches)
    # end-to-end runs (host batches): the input pipeline of B200Trainer -- the NEXT step's pinned batch is copied to the
    # device on a copy stream while the current update executes (every timed step still issues one full host->device
    # copy inside the timed region: the one for its successor)
    pipelined = read_back and hasattr(trainer, "prefetch")
    for i in range(warmup):
        out = trainer.train_step(micro(batches[i % len(batches)]))
        if pipelined:
            trainer.prefetch(micro(batches[(i + 1) % len(batches)]))
        if read_back and out[1] is not None:
            out[1].cpu()
    barrier()
    K.LAUNCHES = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.time()
    e0.record()
    last = None
    for i in range(steps):
        out = trainer.train_step(micro(batches[(warmup + i) % len(batches)] if pipelined else batches[i % len(batches)]))
        if pipelined:
            trainer.prefetch(micro(batches[(warmup + i + 1) % len(batches)]))
        if read_back:
            last = (out[1] if out[1] is not None else out[0]).cpu()  # device->host read of the step's loss statistics
    e1.record()
    barrier()
    w1 = time.time()
    ms = e0.elapsed_time(e1) / steps
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    return ms, (w0, w1), last, out


DUMP_PARAM_SAMPLE = 1 << 22  # 16 MB of fp32 out of the 144.5 M parameters of the TTS model


def dump_sample_index(numel):
    """The fixed, seeded flat indices of the parameter sample (sorted; drawn with replacement)."""
    import torch
    idx = torch.randint(0, numel, (min(DUMP_PARAM_SAMPLE, numel),), generator=torch.Generator().manual_seed(0))
    return idx.sort().values


def dump_outputs(path, trainer, out, rank=0):
    """What one update computed, for comparing two builds output for output: the per-micro-batch losses and logging
    statistics train_step returns, and a fixed seeded sample of the updated parameters, drawn from model.named_parameters()
    concatenated in order (so that it does not depend on the trainer's flat buffer layout). Every rank calls it: under the
    sharded exchange a rank updates only its own shard of the fp32 masters, so they are gathered first (collective);
    rank 0 writes."""
    import numpy as np
    import torch
    trainer.consolidate()
    if rank != 0:
        return
    losses, stats = out
    arrays = {"losses": losses}
    if stats is not None:
        arrays["stats"] = stats
    flat = torch.cat([p.detach().reshape(-1).float() for _, p in trainer.model.named_parameters()])
    arrays["params_sample"] = flat[dump_sample_index(flat.numel()).to(flat.device)]
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.detach().float().cpu().numpy())


def _peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        return {}


def _fresh_runtime(dtype, seed):
    import torch  # noqa: F401
    from speecht5_b200.ops import RT
    RT.dtype = dtype
    RT.clear_static()
    RT.invalidate_shadows()
    RT.manual_seed(seed)
    RT.stage_callback = None
    RT.layer_keep = RT.layer_keep_host = None


def mel_l2_full_depth(dev, dtypes):
    """BASELINE config 1 at full depth (SpeechT5-Base 12 + 6, one 4 s utterance: 64 tokens -> 250 mel frames, eval,
    teacher forced, prenet dropout 0): relative L2 of `after` (the mel) of the CUDA path against the fp32 CPU oracle on
    the same weights -- the number each mode's throughput is quoted next to (tests/test_ref_pin_gpu.py J1 asserts it)."""
    import torch
    from oracle.speecht5_oracle import T5TransformerModelOracle, base_args, synthetic_tts_batch as oracle_batch
    from speecht5_b200.models import make_args
    from speecht5_b200.tasks import SpeechT5Task
    from speecht5_b200.trainer import _to_device
    over = dict(dropout=0.0, attention_dropout=0.0, activation_dropout=0.0, encoder_layerdrop=0.0, decoder_layerdrop=0.0,
                postnet_dropout_rate=0.0, dprenet_dropout_rate=0.0, transformer_enc_positional_dropout_rate=0.0,
                transformer_dec_positional_dropout_rate=0.0, bert_init=True)
    torch.manual_seed(1337)
    oracle = T5TransformerModelOracle(base_args(**over)).eval()
    sample = oracle_batch(1, 64, 250, seed=1, ragged=False)
    with torch.no_grad():
        ref = oracle(**sample["net_input"])[1]
    out = {}
    for name, dtype in dtypes:
        _fresh_runtime(dtype, 1)
        margs = make_args("t5_transformer_base_asr", **over)
        model = SpeechT5Task(margs).build_model(margs).to(dev).eval()
        model.load_state_dict(oracle.state_dict())
        with torch.no_grad():
            after = model(**_to_device(sample, dev)["net_input"])[1]
        out[name] = ((after.float().cpu() - ref).norm() / ref.norm()).item()
        del model
    return out


def parity_leg(args, dev, world):
    """The same training step in PARITY MODE (fp32 activations, every GEMM as hi*hi + hi*lo + lo*hi over bf16 splits):
    its own utterances/s, so that the mode that meets the north_star mel tolerance has a throughput number too."""
    import torch
    from speecht5_b200.criterions import SpeechT5Criterion
    from speecht5_b200.data import synthetic_tts_batch
    from speecht5_b200.models import make_args
    from speecht5_b200.tasks import SpeechT5Task
    from speecht5_b200.trainer import B200Trainer, _to_device
    _fresh_runtime(torch.float32, 1)
    torch.manual_seed(1337)
    margs = make_args(WORKLOAD["arch"], encoder_layerdrop=0.0, decoder_layerdrop=0.0, bert_init=True,
                      decoder_layers=args.decoder_layers, share_input_output_embed=True, max_text_positions=600,
                      max_speech_positions=1876)
    task = SpeechT5Task(margs)
    model = task.build_model(margs).to(dev).train()
    trainer = B200Trainer(model, SpeechT5Criterion(task, use_guided_attn_loss=True), task, lr=1e-4, betas=(0.9, 0.98),
                          eps=1e-8, clip_norm=25.0, use_cuda_graph=not args.no_graph, exchange="allreduce")
    B = args.batch
    resident = [_to_device(synthetic_tts_batch(B, WORKLOAD["text_len"], WORKLOAD["mel_frames"], seed=i), dev)
                for i in range(2)]
    steps = max(3, min(args.steps, 6))
    ms, _, _, out = _timed_steps(trainer, resident, steps, 3, 1, dev, read_back=False)
    loss = float(out[0][0].item())
    del trainer, model
    torch.cuda.empty_cache()
    return {"value": B / (ms * 1e-3), "unit": "utterances/s", "ms_per_step": ms, "steps": steps, "loss": loss,
            "dtype": "f32 activations, 3-pass split-bf16 tcgen05 GEMMs, fp32 row-kernel attention"}

# ------------------------------------------------------------------------------------------------ our arm
def _finish(world):
    """Multi-rank exit: the captured update graph holds NCCL kernels, and tearing the communicator down under it can
    block in ncclCommAbort; all timed work is done and synchronised, so leave without running the destructors."""
    sys.stdout.flush()
    sys.stderr.flush()
    if world > 1:
        os._exit(0)



# ------------------------------------------------------------------------------------------------ other workloads
ASR = dict(arch="t5_transformer_base_asr", batch_per_gpu=8, n_samples=160000, frames=499, target_len=160)
ASR_GFLOP_PER_UTT_STEP = 528.0  # SURVEY 8(d): forward 176 GFLOP/utt (conv FE 49.1 + pos-conv 4.7 + enc 96.9 + dec 24.9), x3


def _emit(line, world):
    print(json.dumps(line), flush=True)
    _finish(world)


def run_asr(args):
    """BASELINE config 3: SpeechT5-Base ASR fine-tune step, 8 x 10 s waveforms per GPU -> 499 frames, 160 target tokens,
    CE + CTC (0.5 / 0.5, label smoothing 0.1), HuBERT time + channel masks, feature_grad_mult 1.0, LayerDrop 0.1 / 0.1,
    dropout 0.1 -- the t5_transformer_base_asr recipe. Same JSON contract; `roofline` is the tcgen05 GEMM set of the
    step, `roofline_conv0` the HBM-bound first conv layer (SURVEY 8d: 33.4 MB algorithmic per utterance, forward)."""
    import torch
    import torch.distributed as dist
    world, rank, local, dev = _init_dist()
    from speecht5_b200 import kernels as K
    from speecht5_b200 import _lib, frontend
    from speecht5_b200.criterions import SpeechT5Criterion
    from speecht5_b200.data import synthetic_asr_batch
    from speecht5_b200.models import make_args
    from speecht5_b200.ops import RT
    from speecht5_b200.tasks import SpeechT5Task
    from speecht5_b200.trainer import B200Trainer, _to_device, h2d_bytes
    _lib.check(_lib.load().st5_device_ok(), "st5_device_ok")
    _fresh_runtime(torch.bfloat16, 1 + rank)
    torch.manual_seed(1337)
    import numpy as np
    np.random.seed(17 + rank)
    margs = make_args(ASR["arch"], build_speech_encoder=True, build_text_decoder=True, bert_init=True,
                      feature_grad_mult=1.0, max_text_positions=600)
    task = SpeechT5Task(margs)
    model = task.build_model(margs).to(dev).train()
    crit = SpeechT5Criterion(task, label_smoothing=0.1, ce_weight=0.5, ctc_weight=0.5, zero_infinity=True)
    trainer = B200Trainer(model, crit, task, lr=1e-4, betas=(0.9, 0.98), eps=1e-8, clip_norm=25.0,
                          use_cuda_graph=not args.no_graph, exchange=args.exchange)
    B = args.batch if args.batch != WORKLOAD["batch_per_gpu"] else ASR["batch_per_gpu"]
    host = [synthetic_asr_batch(B, ASR["n_samples"], ASR["target_len"], seed=100 * rank + i, pin=True) for i in range(4)]
    resident = [_to_device(s, dev) for s in host]
    if args.profile_step:  # one eager update between cudaProfilerStart/Stop (ncu --profile-from-start off)
        trainer.use_cuda_graph = False
        for i in range(2):
            trainer.train_step([resident[i]])
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        trainer.train_step([resident[2]])
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return
    sampler = ClockSampler(local) if rank == 0 else None
    ms_dev, win_dev, _, out = _timed_steps(trainer, resident, args.steps, args.warmup, world, dev, read_back=False)
    ms_e2e, _, last, out = _timed_steps(trainer, host, args.steps, args.warmup, world, dev, read_back=True)
    loss_val = float(out[0][0].item())
    K.LAUNCHES = 0
    eager = B200Trainer.__new__(B200Trainer)
    eager.__dict__.update(trainer.__dict__)
    eager.use_cuda_graph = False
    K.GEMM_RECORD = []
    eager.train_step([resident[0]])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    launches_step = K.LAUNCHES
    records, K.GEMM_RECORD = K.GEMM_RECORD, None
    gemm_flops = sum(2.0 * g.M * g.N * g.K * g.nb1 * g.nb2 for g in records)
    K.gemm_replay(records)
    torch.cuda.synchronize()
    rg = torch.cuda.CUDAGraph()
    with torch.cuda.graph(rg):
        K.gemm_replay(records)
    rg.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        rg.replay()
    e1.record()
    torch.cuda.synchronize()
    gemm_ms = e0.elapsed_time(e1) / 5
    # first conv layer alone (forward: statistics pass + normalise/GELU/store pass), warm, CUDA events on this stream
    fe = model.speech_encoder_prenet.feature_extractor
    blk0 = fe.conv_layers[0]
    wave = resident[0]["net_input"]["source"]

    def conv0():
        with torch.no_grad():
            return frontend.Conv0GroupNormGeluFn.apply(wave, blk0[0].weight, blk0[2].weight, blk0[2].bias, fe.specs[0][2],
                                                       blk0[2].eps, torch.bfloat16)
    y0 = conv0()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(20):
        conv0()
    e1.record()
    torch.cuda.synchronize()
    conv0_ms = e0.elapsed_time(e1) / 20
    conv0_bytes = B * (2 * ASR["n_samples"] * 4 + y0.shape[1] * y0.shape[2] * 2)  # waveform read by both passes + bf16 store
    peaks = _peaks()
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_bw = peaks.get("hbm_gbs", 6500.0)
    clocks = sampler.window(*win_dev) if sampler else None
    if sampler:
        sampler.stop()
    if rank != 0:
        _finish(world)
        return
    utt = B * world
    value, e2e = utt / (ms_dev * 1e-3), utt / (ms_e2e * 1e-3)
    achieved_tf = gemm_flops / (gemm_ms * 1e-3) / 1e12
    line = {
        "metric": "utterances/sec (ASR fine-tune step, 10s@16kHz)", "value": value, "unit": "utterances/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"SpeechT5-Base ASR fine-tune step (BASELINE config 3): {B} x 10 s waveforms per GPU "
                               "(160000 samples -> 499 frames), 160 target tokens, CE + CTC 0.5/0.5, label smoothing "
                               "0.1, time mask 0.75/10 + channel mask 0.5/64, feature_grad_mult 1.0, LayerDrop 0.1/0.1 "
                               "(device keep mask under the captured graph), clip 25, Adam",
                   "global_batch": utt, "parallelism": f"dp{world}", "exchange": trainer.exchange,
                   "cuda_graph": not args.no_graph, "loss": loss_val, "graphs_captured": trainer.graph_misses,
                   "l2": "4 distinct input batches are cycled; the step's activations exceed the 126 MB L2"},
        "e2e": {"value": e2e, "unit": "utterances/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d_bytes(host[0]),
                "d2h_bytes_per_step": int(last.numel() * 4)},
        "gpu_launches": launches_step * args.steps, "gpu_launches_per_step": launches_step, "clocks": clocks,
        "step_tflops": ASR_GFLOP_PER_UTT_STEP * value / 1e3,
        "roofline": {"bound": "tensor", "kernel": "gemm_bf16_tcgen05 (all GEMM launches of one step)",
                     "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
                     "traffic": None, "launches": len(records), "gemm_ms_per_step": gemm_ms,
                     "gemm_share_of_step": gemm_ms / ms_dev},
        "roofline_conv0": {"bound": "hbm", "kernel": "conv0_stats + conv0_finalize + conv0_apply (layer 0 forward)",
                           "achieved": conv0_bytes / (conv0_ms * 1e-3) / 1e9, "peak": peak_bw, "unit": "GB/s",
                           "frac": conv0_bytes / (conv0_ms * 1e-3) / 1e9 / peak_bw, "ms": conv0_ms,
                           "algorithmic_bytes": conv0_bytes, "traffic": None,
                           "note": "the 10-tap convolution is recomputed in both passes instead of stored: the kernel "
                                   "is bound by its fp32 FMA + GELU work, not by HBM (DESIGN.md section 4)"},
    }
    if not args.no_cpu_baseline:
        del trainer, model, eager
        torch.cuda.empty_cache()
        line["cpu_baseline"] = asr_cpu_baseline()
    _emit(line, world)


PRETRAIN = dict(speech_batch=5, n_samples=250000, text_batch=23, text_len=512, vocab=10000, km_classes=500)
# SURVEY 8(d) config 4: forward GFLOP per speech utterance (conv FE 76.7 + encoder 544 + 6-layer decoder 121) and per
# 512-token text sample (encoder 343 + decoder 116); an update is 3x the forward of one micro-batch of each
PRETRAIN_GFLOP_PER_UPDATE = 3.0 * (5 * (76.7 + 544.0 + 121.0) + 23 * (343.0 + 116.0))


def run_pretrain(args):
    """BASELINE config 4: t5_transformer_large (24 + 6 layers, d = 1024, layer_norm waveform extractor, pre-LN) joint
    pre-training update -- one speech micro-batch (5 x 250 000 samples -> 781 frames, HuBERT k-means labels at 50 Hz,
    mask p = 0.8, mel reconstruction through the speech decoder) and one text micro-batch (23 x 512 tokens, V = 10 000,
    BART denoising), `--update-freq 2`, shared Gumbel quantizer (codebook-prob 0.1, loss weights [10, 0.1]), clip 5, Adam
    (0.9, 0.98) eps 1e-6 wd 0.01 -- the README's pre-training recipe. The pre-training criteria gather the masked
    frames (a different count every draw) and read their statistics back inside forward, so these updates run eagerly:
    the step includes the host's launch overhead. Same JSON contract; `value` counts speech utterances + text samples."""
    import torch
    import torch.distributed as dist
    world, rank, local, dev = _init_dist()
    from speecht5_b200 import kernels as K
    from speecht5_b200 import _lib
    from speecht5_b200.criterions import SpeechT5Criterion
    from speecht5_b200.data import synthetic_speech_pretrain_batch, synthetic_text_pretrain_batch
    from speecht5_b200.models import make_args
    from speecht5_b200.tasks import SpeechT5Task
    from speecht5_b200.trainer import B200Trainer, _to_device, h2d_bytes
    _lib.check(_lib.load().st5_device_ok(), "st5_device_ok")
    _fresh_runtime(torch.bfloat16, 1 + rank)
    torch.manual_seed(1337)
    import numpy as np
    np.random.seed(17 + rank)
    P = PRETRAIN
    V = P["vocab"]
    margs = make_args(args.pretrain_arch, build_speech_encoder=True, build_text_decoder=True, bert_init=True,
                      share_input_output_embed=True, use_codebook=True, codebook_prob=0.1, vocab_size=V,
                      hubert_num_classes=[P["km_classes"] + 4], max_text_positions=600)
    task = SpeechT5Task(margs)
    model = task.build_model(margs).to(dev).train()
    n_params = sum(p.numel() for p in model.parameters())
    crit = SpeechT5Criterion(task, loss_weights=[10.0, 0.1], dec_weight=0.5, bart_weight=1.0, hubert_weight=1.0)
    trainer = B200Trainer(model, crit, task, lr=2e-4, betas=(0.9, 0.98), eps=1e-6, weight_decay=0.01, clip_norm=5.0,
                          use_cuda_graph=False, exchange=args.exchange)
    host = [[synthetic_speech_pretrain_batch(P["speech_batch"], P["n_samples"], n_classes=P["km_classes"],
                                             seed=100 * rank + i, pin=True),
             synthetic_text_pretrain_batch(P["text_batch"], P["text_len"], V, mask_idx=V - 2, seed=200 * rank + i, pin=True)]
            for i in range(2)]
    resident = [[_to_device(s, dev) for s in pair] for pair in host]
    mem_log = []
    if os.environ.get("ST5_MEMLOG", "0") == "1":  # per micro-batch: live / peak bytes on the device (to stderr)
        inner = task.train_step

        def logged(sample, *a, **kw):
            torch.cuda.reset_peak_memory_stats()
            r = inner(sample, *a, **kw)
            mem_log.append((sample["task_name"], torch.cuda.memory_allocated() / 2**30, torch.cuda.max_memory_allocated() / 2**30))
            print("mem", mem_log[-1], file=sys.stderr, flush=True)
            return r
        task.train_step = logged
        for name in ("speech_encoder_prenet", "speech_encoder_prenet.feature_extractor", "text_encoder_prenet", "encoder",
                     "hubert_layer", "quantizer", "decoder", "speech_decoder_postnet", "text_decoder_postnet"):
            mod = model.get_submodule(name)
            mod.register_forward_hook(lambda m, i, o, name=name: print(
                "  after", name, round(torch.cuda.memory_allocated() / 2**30, 2), "GiB, peak",
                round(torch.cuda.max_memory_allocated() / 2**30, 2), file=sys.stderr, flush=True))
    sampler = ClockSampler(local) if rank == 0 else None
    try:
        ms_dev, win_dev, _, out = _timed_steps(trainer, resident, args.steps, args.warmup, world, dev, read_back=False)
    except torch.OutOfMemoryError:
        import gc
        seen = {}
        for o in gc.get_objects():
            try:
                if torch.is_tensor(o) and o.is_cuda:
                    st = o.untyped_storage()
                    seen[st.data_ptr()] = (st.nbytes() / 2**30, tuple(o.shape), str(o.dtype))
            except Exception:  # noqa: BLE001
                pass
        print("OOM: live python-visible GiB", sum(v[0] for v in seen.values()), "allocated GiB",
              torch.cuda.memory_allocated() / 2**30, file=sys.stderr)
        for v in sorted(seen.values(), reverse=True)[:25]:
            print("   ", v, file=sys.stderr)
        raise
    ms_e2e, _, last, out = _timed_steps(trainer, host, args.steps, args.warmup, world, dev, read_back=True)
    losses = [float(v) for v in out[0].tolist()]
    K.LAUNCHES = 0
    K.GEMM_RECORD = []
    trainer.train_step(resident[0])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    launches_step = K.LAUNCHES
    records, K.GEMM_RECORD = K.GEMM_RECORD, None
    gemm_flops = sum(2.0 * g.M * g.N * g.K * g.nb1 * g.nb2 for g in records)
    K.gemm_replay(records)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        K.gemm_replay(records)
    e1.record()
    torch.cuda.synchronize()
    gemm_ms = e0.elapsed_time(e1) / 3
    peak_tf = _peaks().get("bf16_tflops_sustained", 1400.0)
    clocks = sampler.window(*win_dev) if sampler else None
    if sampler:
        sampler.stop()
    if rank != 0:
        _finish(world)
        return
    per_update = (P["speech_batch"] + P["text_batch"]) * world
    value, e2e = per_update / (ms_dev * 1e-3), per_update / (ms_e2e * 1e-3)
    achieved_tf = gemm_flops / (gemm_ms * 1e-3) / 1e12
    line = {
        "metric": "samples/sec (joint pre-training update: speech utterances + text samples)", "value": value,
        "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"{args.pretrain_arch} joint pre-training update (BASELINE config 4): speech micro-batch "
                               f"{P['speech_batch']} x {P['n_samples']} samples (781 frames, k-means labels @ 50 Hz, mask "
                               f"0.8 / 10, mel reconstruction 977 -> 488 decoder steps) + text micro-batch "
                               f"{P['text_batch']} x {P['text_len']} tokens (V = {V}), update-freq 2, Gumbel quantizer "
                               "(codebook-prob 0.1, loss weights [10, 0.1]), clip 5, Adam wd 0.01; eager (the masked-frame "
                               "gather has a data-dependent size)",
                   "global_batch": per_update, "parallelism": f"dp{world}", "exchange": trainer.exchange,
                   "cuda_graph": False, "parameters": n_params, "losses_speech_text": losses,
                   "extractor_mode": margs.extractor_mode, "peak_memory_gib": torch.cuda.max_memory_allocated() / 2**30,
                   "l2": "2 distinct input pairs are cycled; the update's activations exceed the 126 MB L2"},
        "e2e": {"value": e2e, "unit": "samples/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": sum(h2d_bytes(s) for s in host[0]), "d2h_bytes_per_step": int(last.numel() * 4)},
        "gpu_launches": launches_step * args.steps, "gpu_launches_per_step": launches_step, "clocks": clocks,
        "step_tflops": PRETRAIN_GFLOP_PER_UPDATE * world / 1e3 / (ms_dev * 1e-3),
        "roofline": {"bound": "tensor", "kernel": "gemm_bf16_tcgen05 (all GEMM launches of one update)",
                     "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
                     "traffic": None, "launches": len(records), "gemm_ms_per_step": gemm_ms,
                     "gemm_share_of_step": gemm_ms / ms_dev},
        "cpu_baseline": None,
    }
    _emit(line, world)


def asr_cpu_baseline(B=2, steps=3):
    """The reference math of the same step on the host cores: oracle port (pinned to the reference by
    tests/test_ref_pin_cpu.py), fp32, no masks / LayerDrop (they only remove work), a bounded sample."""
    import torch
    from oracle.speecht5_oracle_asr import T5TransformerModelASROracle, asr_loss, base_asr_args, synthetic_asr_batch
    cores = min(os.cpu_count() or 1, 32)
    torch.set_num_threads(cores)
    torch.manual_seed(1337)
    model = T5TransformerModelASROracle(base_asr_args(bert_init=True, feature_grad_mult=1.0)).train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-4, betas=(0.9, 0.98), eps=1e-8)
    sample = synthetic_asr_batch(B, ASR["n_samples"], ASR["target_len"], seed=1)

    def step():
        opt.zero_grad(set_to_none=False)
        loss = asr_loss(model, sample, ce_weight=0.5, ctc_weight=0.5, label_smoothing=0.1)[0] / B
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 25.0)
        opt.step()
    step()
    t0 = time.time()
    for _ in range(steps):
        step()
    dt = (time.time() - t0) / steps
    return {"value": B / dt, "unit": "utterances/s", "cores": cores, "kind": "port",
            "sample": f"{steps} full ASR update steps on {B} x 10 s waveforms, fp32 PyTorch CPU, {cores} threads, "
                      f"{dt:.2f} s/step"}


def run_hifigan(args):
    """BASELINE config 5: HiFi-GAN vocoder inference, 512 mel spectrograms [800, 80] -> 512 x 204800 samples, one GPU
    (N > 1: independent replicas, 512 / N each -- no collective, SURVEY 8e)."""
    import torch
    world, rank, local, dev = _init_dist()
    from speecht5_b200 import kernels as K
    from speecht5_b200 import vocoder
    from oracle.audio_oracle import HifiGanGenerator as Ref
    _fresh_runtime(torch.bfloat16, 1)
    ref = Ref(std=0.01, seed=7).eval()
    gen = vocoder.HifiGanGenerator(ref.state_dict(), device=dev)
    total, chunk = 512 // world, 16
    g = torch.Generator().manual_seed(3 + rank)
    host = torch.randn(total, 800, 80, generator=g).pin_memory()
    mel = host.to(dev)
    out_host = torch.empty(chunk, 204800, dtype=torch.float32).pin_memory()

    def run(resident):
        n = 0
        for i in range(0, total, chunk):
            x = mel[i:i + chunk] if resident else host[i:i + chunk].to(dev, non_blocking=True)
            y = gen(x, normalize_before=False)
            if not resident:
                out_host[: y.shape[0]].copy_(y.float(), non_blocking=True)
            n += y.numel()
        return n
    for _ in range(max(1, args.warmup // 2)):
        run(True)
    torch.cuda.synchronize()
    K.LAUNCHES = 0
    reps = max(1, args.steps // 10)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local) if rank == 0 else None
    w0 = time.time()
    e0.record()
    for _ in range(reps):
        n = run(True)
    e1.record()
    torch.cuda.synchronize()
    w1 = time.time()
    ms = e0.elapsed_time(e1) / reps
    launches = K.LAUNCHES // reps
    e0.record()
    for _ in range(reps):
        run(False)
    e1.record()
    torch.cuda.synchronize()
    ms_e2e = e0.elapsed_time(e1) / reps
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms, ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = t.tolist()
    clocks = sampler.window(w0, w1) if sampler else None
    if sampler:
        sampler.stop()
    if rank != 0:
        _finish(world)
        return
    samples = 512 * 204800
    peaks = _peaks()
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    tf = 512 * 218.65e9 / (ms * 1e-3) / 1e12
    line = {"metric": "waveform samples/sec (HiFi-GAN vocoder inference)", "value": samples / (ms * 1e-3),
            "unit": "samples/s", "n_gpus": world, "steps": reps, "warmup": max(1, args.warmup // 2), "ms_per_step": ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "HiFi-GAN generator (BASELINE config 5): 512 x [800, 80] mels -> 512 x 204800 samples, "
                                   f"chunks of {chunk}; rates 4.4.4.4, 512 initial channels, resblock kernels 3/7/11",
                       "parallelism": f"replicas{world}", "realtime_factor": samples / 16000.0 / (ms * 1e-3)},
            "e2e": {"value": samples / (ms_e2e * 1e-3), "unit": "samples/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": 512 * 800 * 80 * 4, "d2h_bytes_per_step": samples * 4},
            "gpu_launches": launches * reps, "gpu_launches_per_step": launches, "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": "gemm_bf16_tcgen05 window GEMMs (every convolution of the generator)",
                         "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": tf / peak_tf, "traffic": None,
                         "note": "whole-generator figure: 218.65 GFLOP per utterance (SURVEY 8d) / wall time of the pass; "
                                 "layer-by-layer execution moves 0.94 GB of bf16 activations per utterance"}}
    if not args.no_cpu_baseline:
        cores = min(os.cpu_count() or 1, 32)
        torch.set_num_threads(cores)
        x = torch.randn(1, 800, 80)
        with torch.no_grad():
            ref(x, normalize_before=False)
            t0 = time.time()
            for _ in range(2):
                ref(x, normalize_before=False)
            dt = (time.time() - t0) / 2
        line["cpu_baseline"] = {"value": 204800 / dt, "unit": "samples/s", "cores": cores, "kind": "port",
                                "sample": f"2 utterances of 800 frames, fp32 PyTorch CPU conv1d, {cores} threads, {dt:.2f} s each"}
    _emit(line, world)


def run_ragged(args):
    """Variable-shape training (fairseq batches by --max-tokens, so (T_text, T_mel) changes nearly every step): a
    stream of >= 16 distinct batch shapes through the trainer's shape buckets (text to multiples of 32, frames to 64) and
    its LRU cache of captured graphs; reports utterances/s over the stream incl. every capture, the steady-state step
    time once the buckets are captured, and the cache hit rate."""
    import torch
    world, rank, local, dev = _init_dist()
    from speecht5_b200.criterions import SpeechT5Criterion
    from speecht5_b200.data import synthetic_tts_batch
    from speecht5_b200.models import make_args
    from speecht5_b200.tasks import SpeechT5Task
    from speecht5_b200.trainer import B200Trainer
    _fresh_runtime(torch.bfloat16, 1 + rank)
    torch.manual_seed(1337)
    margs = make_args(WORKLOAD["arch"], encoder_layerdrop=0.0, decoder_layerdrop=0.0, bert_init=True,
                      share_input_output_embed=True, max_text_positions=600, max_speech_positions=1876)
    task = SpeechT5Task(margs)
    model = task.build_model(margs).to(dev).train()
    trainer = B200Trainer(model, SpeechT5Criterion(task, use_guided_attn_loss=True), task, lr=1e-4, betas=(0.9, 0.98),
                          eps=1e-8, clip_norm=25.0, graph_cache=16, shape_buckets={"text": 32, "frames": 64},
                          exchange=args.exchange)
    g = torch.Generator().manual_seed(5)
    B = args.batch
    shapes = sorted({(int(torch.randint(97, 161, (1,), generator=g)), 2 * int(torch.randint(200, 314, (1,), generator=g)))
                     for _ in range(40)})[:24]
    stream = [synthetic_tts_batch(B, t, m, seed=i, pin=True) for i, (t, m) in enumerate(shapes)]
    order = [int(i) for i in torch.randint(0, len(stream), (max(args.steps * 3, 60),), generator=g)]
    torch.cuda.synchronize()
    t0 = time.time()
    for i in order:
        trainer.train_step([stream[i]])
    torch.cuda.synchronize()
    total_s = time.time() - t0
    hits, misses = trainer.graph_hits, trainer.graph_misses
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    # steady state through the input pipeline: bucket padding (host) and the host->device copy of the NEXT batch run
    # under the current update (B200Trainer.prefetch), like the end-to-end leg of the fixed-shape bench
    timed = order[:args.steps]
    trainer.prefetch([stream[timed[0]]])
    for k, i in enumerate(timed):
        out = trainer.train_step([stream[i]])
        trainer.prefetch([stream[timed[(k + 1) % len(timed)]]])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    if rank != 0:
        _finish(world)
        return
    line = {"metric": "utterances/sec (TTS fine-tune step, ragged batch shapes)", "value": B * world / (ms * 1e-3),
            "unit": "utterances/s", "n_gpus": world, "steps": args.steps, "warmup": len(order), "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"SpeechT5-Base TTS fine-tune step on {len(shapes)} distinct (T_text, T_mel) batch "
                                   f"shapes, {B} utterances each, padded to buckets (text 32, frames 64)",
                       "distinct_shapes": len(shapes), "graphs_captured": misses, "cache_hit_rate": hits / max(1, hits + misses),
                       "stream_steps": len(order), "stream_seconds_incl_captures": total_s,
                       "stream_utt_per_s_incl_captures": B * len(order) / total_s,
                       "hit_rate_second_pass": (trainer.graph_hits - hits) / max(1, args.steps),
                       "loss": float(out[0][0].item())}}
    _emit(line, world)


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    if args.workload == "asr":
        return run_asr(args)
    if args.workload == "hifigan":
        return run_hifigan(args)
    if args.workload == "tts_ragged":
        return run_ragged(args)
    if args.workload == "pretrain":
        return run_pretrain(args)
    import torch
    import torch.distributed as dist
    world, rank, local, dev = _init_dist()
    from speecht5_b200 import kernels as K
    from speecht5_b200 import _lib
    from speecht5_b200.criterions import SpeechT5Criterion
    from speecht5_b200.data import synthetic_tts_batch
    from speecht5_b200.models import make_args
    from speecht5_b200.ops import RT
    from speecht5_b200.tasks import SpeechT5Task
    from speecht5_b200.trainer import B200Trainer, _to_device, h2d_bytes
    lib = _lib.load()
    _lib.check(lib.st5_device_ok(), "st5_device_ok")
    RT.dtype = torch.bfloat16
    RT.manual_seed(1 + rank)
    torch.manual_seed(1337)  # identical initial weights on every rank (what DDP's broadcast would give)
    margs = make_args(WORKLOAD["arch"], encoder_layerdrop=0.0, decoder_layerdrop=0.0, bert_init=True,
                      decoder_layers=args.decoder_layers, share_input_output_embed=True, max_text_positions=600,
                      max_speech_positions=1876)
    task = SpeechT5Task(margs)
    model = task.build_model(margs).to(dev).train()
    crit = SpeechT5Criterion(task, use_guided_attn_loss=True)
    trainer = B200Trainer(model, crit, task, lr=1e-4, betas=(0.9, 0.98), eps=1e-8, clip_norm=25.0,
                          use_cuda_graph=not args.no_graph, exchange=args.exchange)
    nparams = sum(p.numel() for p in model.parameters())
    B = args.batch
    host = [synthetic_tts_batch(B, WORKLOAD["text_len"], WORKLOAD["mel_frames"], seed=100 * rank + i, pin=True)
            for i in range(4)]
    resident = [_to_device(s, dev) for s in host]
    torch.cuda.synchronize()
    if args.profile_step:
        trainer.use_cuda_graph = False
        for i in range(2):
            trainer.train_step([resident[i]])
        torch.cuda.synchronize()
        K.GEMM_RECORD = []
        torch.cuda.profiler.start()
        trainer.train_step([resident[2]])
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
        with open(os.path.join(ROOT, "gpurun_out", "gemm_shapes.json"), "w") as fh:  # launch-ordered, joins the ncu list
            json.dump([dict(M=g.M, N=g.N, K=g.K, nb=g.nb1 * g.nb2, a_mn=g.a_mn, b_mn=g.b_mn, c_fp32=g.c_fp32,
                            acc=g.accumulate, act=g.act, drop=g.drop_p > 0, pre=bool(g.c_pre), ag=bool(g.actgrad_pre))
                       for g in K.GEMM_RECORD], fh)
        return
    sampler = ClockSampler(local) if rank == 0 else None

    def timed(batches, read_back):
        return _timed_steps(trainer, batches, args.steps, args.warmup, world, dev, read_back)

    ms_dev, win_dev, _, out = timed(resident, read_back=False)
    launches_step = None
    ms_e2e, win_e2e, last, out = timed(host, read_back=True)
    if args.dump_outputs:  # the last timed update of the run (end-to-end pass), before anything else runs
        dump_outputs(args.dump_outputs, trainer, out, rank)
    loss_val = float(out[0][0].item())
    # kernels launched per step: counted once while the step was traced (graph mode replays the same launches)
    K.LAUNCHES = 0
    eager = B200Trainer.__new__(B200Trainer)
    eager.__dict__.update(trainer.__dict__)
    eager.use_cuda_graph = False
    K.GEMM_RECORD = []
    eager.train_step([resident[0]])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    launches_step = K.LAUNCHES
    records, K.GEMM_RECORD = K.GEMM_RECORD, None
    # ---- roofline of the dominant kernel (the tcgen05 GEMM): replay exactly this step's GEMM launches back to back
    gemm_flops = sum(2.0 * g.M * g.N * g.K * g.nb1 * g.nb2 for g in records)
    K.gemm_replay(records)
    torch.cuda.synchronize()
    rg = torch.cuda.CUDAGraph()  # one graph of the step's GEMM launches: no host launch gaps in the measurement
    with torch.cuda.graph(rg):
        K.gemm_replay(records)
    rg.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 5
    e0.record()
    for _ in range(reps):
        rg.replay()
    e1.record()
    torch.cuda.synchronize()
    gemm_ms = e0.elapsed_time(e1) / reps
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (measured)" if peaks else "fallback 1.4 PF sustained"
    achieved_tf = gemm_flops / (gemm_ms * 1e-3) / 1e12
    # DRAM traffic of the same kernel from the committed ncu pass (profiles/, per launch like `achieved`): measured
    # under ncu (cold L2 per launch), so it is an upper bound of what the warm step moves
    traffic, traffic_note = None, "no ncu traffic file committed"
    try:
        tpath = os.path.join(ROOT, "profiles", "r02_gemm_traffic.json")
        tj = json.load(open(tpath if os.path.exists(tpath) else os.path.join(ROOT, "profiles", "r01_gemm_traffic.json")))
        traffic = tj["dram_bytes_per_launch"]
        traffic_note = tj.get("note", "")
    except Exception:  # noqa: BLE001
        pass
    clocks = sampler.window(*win_dev) if sampler else None
    if sampler:
        sampler.stop()
    if rank != 0:
        _finish(world)
        return
    utt_per_step = B * world
    value = utt_per_step / (ms_dev * 1e-3)
    e2e = utt_per_step / (ms_e2e * 1e-3)
    line = {
        "metric": "utterances/sec (TTS fine-tune step, 10s@16kHz)", "value": value, "unit": "utterances/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"SpeechT5-Base (12+{args.decoder_layers}, d=768, RPE encoder) TTS fine-tune step: "
                               f"{B} x 10 s utterances per GPU (160 text tokens, 626 mel frames, 313 decoder steps), "
                               "criterion L1+BCE+guided-attention, clip 25, Adam; dropout 0.1 / prenet+postnet 0.5 on",
                   "global_batch": utt_per_step, "params": nparams, "parallelism": f"dp{world}",
                   "exchange": trainer.exchange, "cuda_graph": not args.no_graph, "loss": loss_val,
                   "l2": "per-step working set (>3 GB activations + 0.9 GB parameter/optimizer state) exceeds the "
                         "126 MB L2; 4 distinct input batches are cycled"},
        "e2e": {"value": e2e, "unit": "utterances/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": h2d_bytes(host[0]), "d2h_bytes_per_step": int(last.numel() * 4),
                "input_pipeline": "B200Trainer.prefetch: the next step's pinned batch is copied host->device on a copy "
                                  "stream while the current update runs (one full copy per timed step, inside the timed "
                                  "region); the step's loss statistics are read back every step"},
        "gpu_launches": launches_step * args.steps, "gpu_launches_per_step": launches_step,
        "clocks": clocks,
        # SURVEY 8(d): fwd/utt = text-encoder 29.07 + decoder 6.00/layer + pre/post-nets 2.36 GFLOP; step = 3x forward
        "step_tflops": 3.0 * (29.07 + 6.0 * args.decoder_layers + 2.36) * value / 1e3,
        "roofline": {"bound": "tensor", "kernel": "gemm_bf16_tcgen05 (all GEMM launches of one step)",
                     "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
                     "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_src,
                     "launches": len(records),
                     "avg_launch_us": gemm_ms * 1e3 / max(1, len(records)), "gemm_ms_per_step": gemm_ms,
                     "gemm_share_of_step": gemm_ms / ms_dev,
                     "how": "algorithmic 2*M*N*K of every st5_gemm_bf16 launch of one update (recorded from the live "
                            "step) / CUDA-event time of those launches re-issued back to back on the launch stream"},
    }
    del trainer, model, eager
    torch.cuda.empty_cache()
    if world == 1 and not args.no_parity:
        # each numeric mode's throughput next to ITS OWN mel error (full-depth model, BASELINE config 1, vs the CPU path)
        mel = mel_l2_full_depth(dev, (("bf16", torch.bfloat16), ("parity", torch.float32)))
        par = parity_leg(args, dev, world)
        line["modes"] = {
            "bf16": {"value": value, "unit": "utterances/s", "mel_rel_l2_vs_cpu_path": mel["bf16"],
                     "note": "the mode of `value` / `e2e`; bf16 operand rounding alone costs 5.5e-3 at this depth"},
            "parity": dict(par, mel_rel_l2_vs_cpu_path=mel["parity"],
                           note="meets the north_star mel tolerance (1e-3); resident inputs, same step"),
            "mel_config": "SpeechT5-Base 12+6, 1 x 4 s utterance (64 tokens -> 250 mel frames), eval, teacher forced"}
        _fresh_runtime(torch.bfloat16, 1)
    if not args.no_cpu_baseline:
        line["cpu_baseline"] = run_reference(args, emit=False)
    print(json.dumps(line), flush=True)
    _finish(world)


if __name__ == "__main__":
    main()
