"""B200Trainer host logic on the CPU (kernel entry points emulated by tests/gemm_emulator.py, gloo for world > 1):
stage-ordered flat buffers, per-stage exchange launched from the backward hooks, reduce-scatter + sharded Adam +
all-gather against plain all-reduce against a single process with two micro-batches (fairseq --update-freq 2 computes
the same mean gradient), optimizer state round trip, non-finite guard, shadows after load_state_dict, shape buckets."""
import os
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def _build(dtype, patch):
    """`patch`: pytest's monkeypatch in the test process (undone after the test, so later tests see the real kernels),
    gemm_emulator.Patcher() in a spawned worker."""
    import gemm_emulator
    from helpers import NO_DROPOUT, TINY
    from speecht5_b200.criterions import SpeechT5Criterion
    from speecht5_b200.models import make_args
    from speecht5_b200.ops import RT
    from speecht5_b200.tasks import SpeechT5Task
    gemm_emulator.install_trainer(patch)
    patch.setattr(RT, "dtype", dtype)
    RT.disable_device_seed()
    RT.clear_static()
    RT.invalidate_shadows()
    torch.manual_seed(11)
    args = make_args("t5_transformer_base_asr", **TINY, **NO_DROPOUT, bert_init=True)
    task = SpeechT5Task(args)
    model = task.build_model(args).train()
    crit = SpeechT5Criterion(task, use_guided_attn_loss=True)
    return task, model, crit


def _batches():
    from speecht5_b200.data import synthetic_tts_batch
    return [[synthetic_tts_batch(2, 13, 20, seed=10 * step + r) for r in range(2)] for step in range(2)]


def _run_single(dtype, patch):
    from speecht5_b200.trainer import B200Trainer
    task, model, crit = _build(dtype, patch)
    tr = B200Trainer(model, crit, task, lr=1e-2, use_cuda_graph=False)
    for step in _batches():
        tr.train_step(step)  # two micro-batches per update == two ranks with one each
    return {n: p.detach().clone() for n, p in model.named_parameters()}, tr


def _worker(rank, world, port, mode, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import gemm_emulator
    from speecht5_b200.trainer import B200Trainer
    task, model, crit = _build(torch.bfloat16, gemm_emulator.Patcher())
    tr = B200Trainer(model, crit, task, lr=1e-2, use_cuda_graph=False, exchange=mode)
    for step in _batches():
        tr.train_step([step[rank]])
    fired = tr.overlapped_stages
    stale = None
    if mode == "shard":  # before consolidation the fp32 master of a foreign shard is stale, the bf16 shadow is not
        sk = next(iter(tr.fp.stages))
        lo, hi = tr.fp.shard(sk, rank=1 - rank)
        stale = float((tr.fp.flat[lo:hi].to(torch.bfloat16).float() - tr.fp.shadow[lo:hi].float()).abs().max())
    tr.consolidate()
    out = {n: p.detach().numpy().copy() for n, p in model.named_parameters()}  # numpy: no fd passing through the queue
    shadow_err = float((tr.fp.flat.to(torch.bfloat16).float() - tr.fp.shadow.float()).abs().max())
    q.put((rank, out, fired, len(tr.fp.stages), stale, shadow_err, tr.grad_norm()))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("mode", ["shard", "allreduce"])
def test_two_rank_exchange_equals_two_micro_batches_on_one_rank(mode, monkeypatch):
    """legacy_distributed_data_parallel.py:76-165 + trainer.py:776-826: the mean over ranks of per-rank normalised
    gradients. Both exchanges (reduce-scatter + sharded Adam + all-gather; per-stage all-reduce) give the parameters a
    single process reaches with the two batches as micro-batches; every stage's exchange is launched from its backward
    hook (ADVICE r1: the old hook never fired)."""
    ref, tr1 = _run_single(torch.bfloat16, monkeypatch)
    gn1 = tr1.grad_norm()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29611 + (os.getpid() * 3 + (mode == "shard")) % 300
    procs = [ctx.Process(target=_worker, args=(r, 2, port, mode, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=300) for _ in range(2)], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
    for rank, out, fired, n_stages, stale, shadow_err, gn in res:
        assert fired == 2 * n_stages, (fired, n_stages)  # 2 updates x every stage, all from the hooks
        assert shadow_err == 0.0  # after consolidate(): shadow == bf16(master) everywhere
        assert abs(gn - gn1) < 1e-3 * gn1, (gn, gn1)
        if mode == "shard":
            assert stale is not None and stale > 0.0
        for n, v in out.items():
            v = torch.from_numpy(v)
            err = ((v - ref[n]).norm() / (ref[n].norm() + 1e-12)).item()
            assert err < 2e-3, (n, err)
    for n in res[0][1]:
        assert (res[0][1][n] == res[1][1][n]).all(), n  # ranks agree bit for bit


def test_optimizer_state_round_trip_and_overflow_guard(monkeypatch):
    from speecht5_b200.trainer import B200Trainer
    ref, tr = _run_single(torch.float32, monkeypatch)
    sd = tr.state_dict()
    assert set(sd) >= {"state", "param_groups"} and sd["state"][0]["step"] == 2
    assert sd["param_groups"][0]["betas"] == (0.9, 0.98)
    # a non-finite gradient norm: the update is skipped, the counter raises at the next check
    flat0, m0, step0 = tr.fp.flat.clone(), tr.fp.exp_avg.clone(), tr.step_dev.clone()
    batch = _batches()[0][0]
    batch["net_input"]["spkembs"] = batch["net_input"]["spkembs"].clone()
    batch["net_input"]["spkembs"][0, 0] = float("nan")  # NaN activations -> NaN gradients everywhere
    tr.train_step([batch])
    assert not bool(torch.isfinite(tr.gnorm_sq).all())
    assert torch.equal(tr.fp.flat, flat0) and torch.equal(tr.fp.exp_avg, m0) and torch.equal(tr.step_dev, step0)
    with pytest.raises(FloatingPointError):
        tr.check_overflow()
    tr.check_overflow()  # counter was reset
    # round trip into a fresh trainer: same next update
    task, model, crit = _build(torch.float32, monkeypatch)
    model.load_state_dict({n: p for n, p in ref.items()})
    tr2 = B200Trainer(model, crit, task, lr=1e-2, use_cuda_graph=False)
    tr2.load_state_dict(sd)
    nxt = _batches()[1][1]
    tr.train_step([nxt])
    tr2.train_step([nxt])
    a = dict(tr.model.named_parameters())
    for n, p in tr2.model.named_parameters():
        assert torch.allclose(p, a[n], atol=1e-7), n


def test_static_shadows_follow_load_state_dict(monkeypatch):
    """ADVICE r1: fairseq builds the trainer first and loads the checkpoint second; the flat bf16 shadow the GEMMs read
    must follow."""
    from speecht5_b200.ops import RT
    from speecht5_b200.trainer import B200Trainer
    task, model, crit = _build(torch.bfloat16, monkeypatch)
    tr = B200Trainer(model, crit, task, use_cuda_graph=False)
    w = model.encoder.layers[0].fc1.weight
    new = {k: v.clone() for k, v in model.state_dict().items()}
    new["encoder.layers.0.fc1.weight"] = torch.randn_like(w)
    model.load_state_dict(new)
    hi, _ = RT.shadow(("lin", id(w)), lambda: w)
    assert torch.equal(hi, new["encoder.layers.0.fc1.weight"].to(torch.bfloat16))
    assert hi.data_ptr() == tr.fp.shadow[tr.fp.offsets[id(w)]:].data_ptr()  # still the static view, refreshed


def test_stage_layout_is_world_divisible_and_ordered(monkeypatch):
    from speecht5_b200.trainer import FlatParams
    task, model, crit = _build(torch.bfloat16, monkeypatch)
    fp = FlatParams(model, world=8, rank=3)
    keys = list(fp.stages)
    assert keys == sorted(keys, key=lambda k: (k[0] != "enc", k[1])) and len(keys) == 4
    prev = 0
    for sk, (lo, hi) in fp.stages.items():
        assert lo == prev and (hi - lo) % 64 == 0
        slo, shi = fp.shard(sk)
        assert (shi - slo) * 8 == hi - lo and slo == lo + 3 * (shi - slo)
        prev = hi
    assert fp.tail == prev
    names = dict(model.named_parameters())
    for n, p in names.items():
        o = fp.offsets[id(p)]
        in_stage = any(lo <= o < hi for lo, hi in fp.stages.values())
        assert in_stage == (p.dim() == 2 and n.startswith(("encoder.layers.", "decoder.layers."))), n


def test_pad_to_buckets_keeps_the_valid_region():
    from speecht5_b200.data import synthetic_tts_batch
    from speecht5_b200.trainer import pad_to_buckets
    s = synthetic_tts_batch(3, 37, 150, seed=2)
    p = pad_to_buckets(s, {"text": 32, "frames": 64})
    assert p["net_input"]["src_tokens"].shape == (3, 64) and (p["net_input"]["src_tokens"][:, 37:] == 1).all()
    assert p["dec_target"].shape == (3, 192, 80) and p["labels"].shape == (3, 192)
    assert p["net_input"]["prev_output_tokens"].shape == (3, 96, 80)
    assert torch.equal(p["dec_target"][:, :150], s["dec_target"]) and torch.equal(p["dec_target_lengths"], s["dec_target_lengths"])
    # every tensor whose shape follows the raw lengths is padded: batches of 12 raw shapes fall into 2 x 2 signatures
    # (the collater's `target` features were once left at their raw length -- every raw shape then captured its own graph)
    from speecht5_b200.trainer import _flatten
    sigs = set()
    for i, (t, m) in enumerate([(t, m) for t in (40, 50, 60, 70) for m in (130, 150, 200)]):
        q = pad_to_buckets(synthetic_tts_batch(3, t, m, seed=i), {"text": 32, "frames": 64})
        sigs.add(tuple((k, tuple(v.shape)) for k, v in _flatten(q).items()))
    assert len(sigs) == 4, len(sigs)


def test_packed_device_copies_keep_structure_and_share_one_buffer():
    """trainer._to_device_packed (the graph's static inputs and the prefetch staging set): same nested structure and
    values as the samples, every tensor a 256-byte aligned view of ONE byte buffer, so two sets built from batches of the
    same shapes can be moved over each other with a single copy."""
    from speecht5_b200.trainer import _flatten, _to_device_packed
    torch.manual_seed(0)
    mk = lambda seed: {"id": torch.arange(3) + seed, "task_name": "t2s",  # noqa: E731
                       "net_input": {"src_tokens": torch.randint(0, 50, (3, 7)) + seed, "spkembs": torch.randn(3, 5),
                                     "pad": torch.tensor([[True, False, True]])},
                       "labels": torch.randn(3, 9).to(torch.bfloat16)}
    a, b = [mk(0), mk(1)], [mk(7), mk(8)]
    va, fa = _to_device_packed(a, torch.device("cpu"))
    vb, fb = _to_device_packed(b, torch.device("cpu"))
    assert fa.numel() == fb.numel() and fa.dtype == torch.uint8
    for s, v in zip(a, va):
        assert v["task_name"] == "t2s"
        for (k, x), (k2, y) in zip(_flatten(s).items(), _flatten(v).items()):
            assert k == k2 and x.dtype == y.dtype and x.shape == y.shape and torch.equal(x, y)
            off = y.data_ptr() - fa.data_ptr()
            assert 0 <= off < fa.numel() and off % 256 == 0
    fa.copy_(fb)  # ONE copy moves the second set of batches over the first
    for s, v in zip(b, va):
        for x, y in zip(_flatten(s).values(), _flatten(v).values()):
            assert torch.equal(x, y)


# ------------------------------------------------------------------------- joint pre-training update on two ranks
def _pretrain_build(patch):
    """`patch` as in _build."""
    import gemm_emulator
    from helpers import NO_DROPOUT, TINY
    from speecht5_b200 import frontend
    from speecht5_b200.criterions import SpeechT5Criterion
    from speecht5_b200.models import make_args
    from speecht5_b200.ops import RT
    from speecht5_b200.tasks import SpeechT5Task
    gemm_emulator.install_autograd(patch)
    gemm_emulator.install_trainer(patch)
    patch.setattr(frontend.ConvFeatureExtractor, "forward", lambda self, wave: self._layers(wave))  # (no CUDA guard)
    patch.setattr(RT, "dtype", torch.bfloat16)
    RT.disable_device_seed()
    RT.clear_static()
    RT.invalidate_shadows()
    torch.manual_seed(7)
    args = make_args("t5_transformer_large", **dict(TINY, **NO_DROPOUT), bert_init=True, build_speech_encoder=True,
                     build_text_decoder=True, share_input_output_embed=True, hubert_num_classes=[23], final_dim=16,
                     vocab_size=40, conv_feature_layers="[(32, 10, 5)] + [(32, 3, 2)] * 4 + [(32, 2, 2)] * 2",
                     conv_pos=16, conv_pos_groups=4, mask_prob=0.5, hubert_mask_length=3, max_text_positions=600)
    task = SpeechT5Task(args)
    model = task.build_model(args).train()
    crit = SpeechT5Criterion(task, loss_weights=[10.0], dec_weight=0.5, bart_weight=1.0, hubert_weight=1.0)
    return task, model, crit


def _pretrain_batches(r):
    """(speech, text) micro-batches of rank r; the HuBERT mask is part of the batch (the in-model numpy draw would differ
    between a one-process and a two-process run)."""
    from speecht5_b200.data import synthetic_speech_pretrain_batch, synthetic_text_pretrain_batch
    speech = synthetic_speech_pretrain_batch(2, 6400, n_classes=23, seed=11 + r)
    g = torch.Generator().manual_seed(5 + r)
    speech["net_input"]["mask_indices"] = torch.rand(2, 19, generator=g) < 0.5
    return [speech, synthetic_text_pretrain_batch(3, 12, 40, mask_idx=38, seed=21 + r)]


def _pretrain_worker(rank, world, port, mode, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import gemm_emulator
    from speecht5_b200.trainer import B200Trainer
    task, model, crit = _pretrain_build(gemm_emulator.Patcher())
    tr = B200Trainer(model, crit, task, lr=1e-2, use_cuda_graph=False, exchange=mode)
    for _ in range(2):
        tr.train_step(_pretrain_batches(rank))
    tr.consolidate()
    q.put((rank, {n: p.detach().numpy().copy() for n, p in model.named_parameters()}, tr.grad_norm()))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("mode", ["shard", "allreduce"])
def test_two_rank_joint_pretraining_update_equals_four_micro_batches_on_one_rank(mode, monkeypatch):
    """The pre-training recipe trains with `--find-unused-parameters` (README): the text micro-batch -- the LAST one of an
    update -- never touches the waveform front end, the masked-prediction head or the speech decoder pre/post-net, and
    the speech one never touches the text pre/post-nets. Stages whose backward hook does not fire on the last
    micro-batch are exchanged at the end of the update: two ranks with (speech_r, text_r) each reach the parameters one
    process reaches with the four micro-batches."""
    from speecht5_b200.trainer import B200Trainer
    task, model, crit = _pretrain_build(monkeypatch)
    tr = B200Trainer(model, crit, task, lr=1e-2, use_cuda_graph=False)
    for _ in range(2):
        tr.train_step(_pretrain_batches(0) + _pretrain_batches(1))
    ref = {n: p.detach().clone() for n, p in model.named_parameters()}
    gn1 = tr.grad_norm()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29911 + (os.getpid() * 3 + (mode == "shard")) % 300
    procs = [ctx.Process(target=_pretrain_worker, args=(r, 2, port, mode, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=120) for _ in range(2)], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
    for rank, out, gn in res:
        assert abs(gn - gn1) < 1e-3 * gn1, (gn, gn1)
        for n, v in out.items():
            if n.endswith("norm_k.bias"):
                continue  # shifts every logit of a row alike: analytically zero gradient, Adam normalises its rounding noise
            err = ((torch.from_numpy(v) - ref[n]).norm() / (ref[n].norm() + 1e-12)).item()
            assert err < 2e-3, (n, err)
    for n in res[0][1]:
        assert (res[0][1][n] == res[1][1][n]).all(), n
    moved = [n for n in ("speech_encoder_prenet.feature_extractor.conv_layers.0.0.weight", "hubert_layer.label_embs_concat",
                         "text_encoder_prenet.encoder_prenet.0.weight", "speech_decoder_postnet.feat_out.weight")
             if not torch.equal(ref[n], dict(_pretrain_build(monkeypatch)[1].named_parameters())[n].detach())]
    assert len(moved) == 4, moved


# ------------------------------------------------------------------------- bench.py --dump-outputs on two ranks
def _dump_worker(rank, world, port, path, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import bench
    import gemm_emulator
    from speecht5_b200.trainer import B200Trainer
    task, model, crit = _build(torch.bfloat16, gemm_emulator.Patcher())
    tr = B200Trainer(model, crit, task, lr=1e-2, use_cuda_graph=False, exchange="shard")
    for step in _batches():
        out = tr.train_step([step[rank]])
    bench.dump_outputs(path, tr, out, rank)
    q.put(rank)
    dist.barrier()
    dist.destroy_process_group()


def test_bench_dump_of_a_sharded_update_holds_the_updated_parameters(monkeypatch, tmp_path):
    """bench.py --dump-outputs under --gpus 2 with the sharded exchange, where each rank runs Adam only on its own shard
    of the fp32 masters: the parameter sample rank 0 writes is the model one process reaches with both batches as
    micro-batches, not rank 0's stale copy of the other rank's shards."""
    import numpy as np
    import bench
    ref, _ = _run_single(torch.bfloat16, monkeypatch)
    init = _build(torch.bfloat16, monkeypatch)[1]
    want = torch.cat([p.reshape(-1).float() for p in ref.values()])
    before = torch.cat([p.detach().reshape(-1).float() for p in init.parameters()])
    idx = bench.dump_sample_index(want.numel())
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29311 + os.getpid() % 300
    path = str(tmp_path / "dump")
    procs = [ctx.Process(target=_dump_worker, args=(r, 2, port, path, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=300) for _ in range(2)])
    for p in procs:
        p.join(timeout=60)
    assert res == [0, 1]
    assert sorted(os.listdir(path)) == ["losses.npy", "params_sample.npy", "stats.npy"]
    got = torch.from_numpy(np.load(os.path.join(path, "params_sample.npy")))
    assert got.shape == idx.shape
    assert (got != before[idx]).float().mean().item() > 0.9
    assert ((got - want[idx]).norm() / want[idx].norm()).item() < 2e-3
