"""Pins the oracle restatements and the plugin's host code against the REFERENCE'S OWN CODE.

Everything the reference computed is stored under tests/golden/, so these tests run without the reference tree:
* fixtures `tests/golden/ref_*.npz` (generator `tests/golden/make_golden_from_ref.py`, which runs the reference's
  `speecht5/**` unmodified through `oracle/ref_loader.py`): weights, inputs, outputs, the reference criterions' loss
  terms, gradients, its SequenceGenerator's token ids, its compute_mask_indices draws. The oracle is replayed on the
  stored weights + inputs and must agree to fp32 round-off (tolerances in each test).
* `tests/golden/ref_pins.{npz,json}` (generator `tests/golden/make_golden_ref_pins.py`): the reference at real width /
  long sequences on seeded weights (outputs stored as a seeded sample of elements), its pre-training criteria on fixed
  model outputs, and what its arch functions, add_args, criterion dataclass, reduce_metrics and Dictionary return.
When the reference tree is available, the fixtures are also regenerated in memory and must equal the committed ones
(stale-fixture guard).
"""
import json
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, GOLD)
import make_golden_from_ref as mg  # noqa: E402  (constants + case builders; touches the reference only inside cases)
import make_golden_ref_pins as gp  # noqa: E402  (seeded inputs / weights shared with the generator)
from oracle import ref_loader as rl  # noqa: E402

needs_ref = pytest.mark.skipif(not rl.available(), reason="reference tree not mounted (GPU box): fixtures only")
FP32 = 2e-5   # relative L2, fp32 forward of a 2+2-layer model: different summation orders only
GRAD = 2e-4   # relative L2 of fp32 gradients


def rel(a, b):
    a, b = torch.as_tensor(a).double(), torch.as_tensor(b).double()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def load(name):
    return dict(np.load(os.path.join(GOLD, name + ".npz")))


def pins_json():
    with open(os.path.join(GOLD, "ref_pins.json"), encoding="utf-8") as fh:
        return json.load(fh)


def state_of(blob, prefix="state/"):
    return {k[len(prefix):]: torch.from_numpy(v) for k, v in blob.items() if k.startswith(prefix)}


def conv_layers():
    return eval(mg.TINY_CONV)


# ------------------------------------------------------------------------------------------------------------------ t2s
@pytest.mark.parametrize("name,pre_ln", [("ref_tts_tiny", False), ("ref_tts_preln_tiny", True)])
def test_tts_oracle_matches_reference_outputs_loss_and_gradients(name, pre_ln):
    from oracle.speecht5_oracle import T5TransformerModelOracle, base_args, tts_loss
    blob = load(name)
    over = dict(mg.TINY)
    if pre_ln:
        over.update(layer_norm_first=True, decoder_normalize_before=True)
    model = T5TransformerModelOracle(base_args(**over)).train()
    missing = model.load_state_dict(state_of(blob), strict=False)
    assert not missing.unexpected_keys and all("num_batches_tracked" in k for k in missing.missing_keys), missing
    ni = {k[3:]: torch.from_numpy(v) for k, v in blob.items() if k.startswith("in/")}
    out = model(**ni, task_name="t2s")
    assert rel(out[0], blob["out/before"]) < FP32
    assert rel(out[1], blob["out/after"]) < FP32
    assert rel(out[2], blob["out/logits"]) < FP32
    assert rel(torch.stack(out[3]), blob["out/attn"]) < FP32
    sample = {k[7:]: torch.from_numpy(v) for k, v in blob.items() if k.startswith("sample/")}
    loss, l1, l2, bce, ga = tts_loss(out, sample)
    got = np.array([loss.item(), l1.item(), l2.item(), bce.item(), ga.item()])
    np.testing.assert_allclose(got, blob["loss"], rtol=2e-5)
    loss.backward()
    named = dict(model.named_parameters())
    for k, v in blob.items():
        if k.startswith("grad/"):
            assert rel(named[k[5:]].grad, v) < GRAD, (k, rel(named[k[5:]].grad, v))


# ------------------------------------------------------------------------------------------------------------------ s2t
def _asr_oracle(blob, ln_mode):
    from oracle.speecht5_oracle_asr import T5TransformerModelASROracle, base_asr_args, reference_to_oracle_keys
    over = dict(mg.TINY, conv_feature_layers=conv_layers(), feature_grad_mult=1.0, conv_pos=16, conv_pos_groups=4,
                dropout=0.0, attention_dropout=0.0, activation_dropout=0.0)
    if ln_mode:
        over.update(extractor_mode="layer_norm", layer_norm_first=True, decoder_normalize_before=True,
                    conv_bias=ln_mode != "no_conv_bias", share_input_output_embed=True)
    model = T5TransformerModelASROracle(base_asr_args(**over), vocab_size=mg.VOCAB).train()
    missing = model.load_state_dict(reference_to_oracle_keys(state_of(blob)), strict=False)
    assert not missing.unexpected_keys, missing.unexpected_keys
    assert all(k.endswith("num_batches_tracked") for k in missing.missing_keys), missing.missing_keys
    return model


@pytest.mark.parametrize("name,ln_mode", [("ref_asr_tiny", False), ("ref_asr_ln_tiny", True),
                                          ("ref_asr_large_style_tiny", "no_conv_bias")])
def test_asr_oracle_matches_reference_outputs_loss_and_gradients(name, ln_mode):
    """Conv feature extractor (GroupNorm / LayerNorm modes), speech prenet with the reference's OWN mask draws, encoder +
    CTC head, text decoder pre/post-net; SpeechtoTextLoss CE + CTC; gradients down to conv layer 0."""
    from oracle.speecht5_oracle_asr import asr_loss, reference_to_oracle_keys
    blob = load(name)
    model = _asr_oracle(blob, ln_mode)
    ni = dict(source=torch.from_numpy(blob["in/source"]), padding_mask=torch.from_numpy(blob["in/padding_mask"]),
              prev_output_tokens=torch.from_numpy(blob["in/prev_output_tokens"]),
              mask_indices=torch.from_numpy(blob["in/mask_indices"]),
              mask_channel_indices=torch.from_numpy(blob["in/mask_channel_indices"]))
    sample = {"net_input": ni, "target": torch.from_numpy(blob["sample/target"]),
              "target_lengths": torch.from_numpy(blob["sample/target_lengths"])}
    (logits, _), enc = model(**ni)
    assert rel(enc["encoder_out"][0], blob["out/encoder_out"]) < FP32
    assert rel(enc["encoder_out_for_ctc"][0], blob["out/encoder_out_for_ctc"]) < FP32
    assert torch.equal(enc["encoder_padding_mask"][0], torch.from_numpy(blob["out/encoder_padding_mask"]))
    assert rel(logits, blob["out/logits"]) < FP32
    loss, ce, ctc, _ = asr_loss(model, sample, ce_weight=0.5, ctc_weight=0.5, label_smoothing=0.1, blank_idx=mg.VOCAB - 1)
    np.testing.assert_allclose([loss.item(), ce.item(), ctc.item()], blob["loss"][:3], rtol=2e-5)
    loss.backward()
    named = dict(model.named_parameters())
    n = 0
    for k, v in reference_to_oracle_keys({k[5:]: v for k, v in blob.items() if k.startswith("grad/")}).items():
        assert rel(named[k].grad, v) < GRAD, (k, rel(named[k].grad, v))
        n += 1
    assert n >= 8


@pytest.mark.parametrize("name,ln_mode", [("ref_asr_tiny", False), ("ref_asr_ln_tiny", True)])
def test_oracle_greedy_token_ids_equal_the_reference_sequence_generator(name, ln_mode):
    """north_star: bit-exact token ids for ASR greedy decode. The reference side is speecht5/sequence_generator.py itself
    (beam 1, max_len_b 12), stored in the fixture."""
    from oracle.speecht5_oracle_asr import greedy_decode
    blob = load(name)
    model = _asr_oracle(blob, ln_mode).eval()
    hyp = greedy_decode(model, torch.from_numpy(blob["in/source"]), torch.from_numpy(blob["in/padding_mask"]),
                        max_len_b=12, blank=mg.VOCAB - 1, mask_idx=mg.VOCAB - 2)
    for b, t in enumerate(hyp):
        n = int(blob["out/greedy_lengths"][b])
        assert t.tolist() == blob["out/greedy_tokens"][b, :n].tolist(), (b, t.tolist())


def test_t2t_oracle_matches_reference():
    from oracle.speecht5_oracle_asr import T5TransformerModelT2TOracle, base_asr_args
    blob = load("ref_t2t_tiny")
    over = dict(mg.TINY, share_input_output_embed=True, dropout=0.0, attention_dropout=0.0, activation_dropout=0.0)
    model = T5TransformerModelT2TOracle(base_asr_args(**over), vocab_size=mg.VOCAB).train()
    missing = model.load_state_dict(state_of(blob), strict=False)
    assert not missing.missing_keys, missing.missing_keys
    out = model(src_tokens=torch.from_numpy(blob["in/src_tokens"]),
                prev_output_tokens=torch.from_numpy(blob["in/prev_output_tokens"]))
    assert rel(out[0][0], blob["out/logits"]) < FP32
    assert rel(out[2]["encoder_out"][0], blob["out/encoder_out"]) < FP32


# ------------------------------------------------------------------------------------------------------------ audio ends
def test_hifigan_oracle_matches_the_reference_generator():
    """SpeechUT/fairseq/.../hifigan.py Generator -> oracle.audio_oracle.HifiGanGenerator on the same weights."""
    from oracle.audio_oracle import HifiGanGenerator
    blob = load("ref_hifigan_tiny")
    cfg = dict(model_in_dim=80, upsample_initial_channel=64, upsample_rates=[4, 4, 4],
               upsample_kernel_sizes=[8, 8, 8], resblock_kernel_sizes=[3, 7, 11],
               resblock_dilation_sizes=[[1, 3, 5]] * 3)
    gen = HifiGanGenerator(cfg).eval()
    from oracle.audio_oracle import load_reference_hifigan_state
    load_reference_hifigan_state(gen, state_of(blob))
    with torch.no_grad():
        y = gen(torch.from_numpy(blob["in/mel"]).transpose(1, 2), normalize_before=False)
    ref = torch.from_numpy(blob["out/wav"]).squeeze(1)
    assert rel(y, ref) < 5e-5, rel(y, ref)


def test_pretrain_oracles_match_reference_quantizer_and_hubert_head():
    from oracle.pretrain_oracle import GumbelVectorQuantizer, SpeechEncoderPostnet
    blob = load("ref_pretrain_tiny")
    vq = GumbelVectorQuantizer(dim=64, num_vars=10, groups=2, vq_dim=64).eval()
    sd = state_of(blob, "vq/state/")
    vq.load_state_dict({"vars": sd["vars"], "weight_proj.weight": sd["weight_proj.weight"],
                        "weight_proj.bias": sd["weight_proj.bias"]})
    with torch.no_grad():
        r = vq(torch.from_numpy(blob["vq/in"]))
    assert rel(r["x"], blob["vq/x"]) < 1e-6
    assert abs(r["code_perplexity"].item() - float(blob["vq/code_perplexity"])) < 1e-4
    assert abs(r["prob_perplexity"].item() - float(blob["vq/prob_perplexity"])) < 1e-4
    head = SpeechEncoderPostnet([20], encoder_embed_dim=64, final_dim=16, untie_final_proj=True).train()
    head.load_state_dict(state_of(blob, "head/state/"))
    out = head(torch.from_numpy(blob["head/in/x"]), torch.from_numpy(blob["head/in/padding_mask"]),
               torch.from_numpy(blob["head/in/mask_indices"]), [torch.from_numpy(blob["head/in/target"])])
    for got, want in ((out["logit_m_list"][0], blob["head/logit_m"]), (out["logit_u_list"][0], blob["head/logit_u"])):
        want = torch.from_numpy(want)
        assert torch.equal(torch.isinf(got), torch.isinf(want))  # a negative equal to the positive is -inf (:61-74)
        fin = ~torch.isinf(want)
        assert rel(got[fin], want[fin]) < 1e-5


def test_host_mask_sampler_reproduces_the_reference_draws():
    """speecht5_b200/data.py compute_mask_indices (host logic of the product) == fairseq/data/data_utils.py:393-520 under
    the same numpy seed: the draw ORDER matters, so this is bit-exact."""
    from speecht5_b200.data import compute_mask_indices
    blob = load("ref_masks")
    pad = torch.from_numpy(blob["padding_mask"])
    for i in range(4):
        seed, prob, length = blob[f"cfg/{i}"]
        np.random.seed(int(seed))
        m = compute_mask_indices((4, 120), pad, float(prob), int(length), "static", 0.0, min_masks=2)
        c = compute_mask_indices((4, 64), None, 0.5, 16, "static", 0.0)
        assert np.array_equal(np.asarray(m), blob[f"time/{i}"]), i
        assert np.array_equal(np.asarray(c), blob[f"chan/{i}"]), i


# ------------------------------------------------------------------------------------------- live reference (container)
@needs_ref
@pytest.mark.parametrize("name", sorted(mg.CASES))
def test_committed_fixture_is_what_the_reference_produces_now(name):
    fresh = mg.CASES[name]()
    stored = load(name)
    assert set(fresh) == set(stored)
    for k in fresh:
        a, b = np.asarray(fresh[k]), stored[k]
        if a.dtype.kind in "biu":
            assert np.array_equal(a, b), k
        else:
            np.testing.assert_allclose(a, b, rtol=1e-5, atol=1e-6, err_msg=k)


@needs_ref
def test_committed_ref_pins_are_what_the_reference_produces_now():
    """The same stale-data guard for tests/golden/ref_pins.{json,npz}."""
    assert json.loads(json.dumps(gp.json_pins())) == pins_json()
    fresh, stored = gp.array_pins(), load("ref_pins")
    assert set(fresh) == set(stored)
    for k in fresh:
        a, b = np.asarray(fresh[k]), stored[k]
        if a.dtype.kind in "biu":
            assert np.array_equal(a, b), k
        else:
            np.testing.assert_allclose(a, b, rtol=1e-5, atol=1e-6, err_msg=k)


@pytest.mark.parametrize("T", gp.ENCODER_T)
def test_reference_encoder_at_asr_lengths_matches_oracle(T):
    """VERDICT r1 item 2: `TransformerEncoder.forward` of the reference at T = 199 / 499 (relative positions clipped at
    +-160, key padding) against the oracle encoder on the same seeded weights, Base width, 2 layers."""
    from oracle.speecht5_oracle import TransformerEncoder, base_args
    pins = load("ref_pins")
    enc = gp.seeded_fill(TransformerEncoder(base_args(**gp.encoder_over()), mg.VOCAB, None), 3).eval()
    x, pad = gp.encoder_input(T)
    with torch.no_grad():
        b = enc(x, pad)
    assert rel(gp.sampled(b["encoder_out"][0], T), pins[f"encoder/{T}/encoder_out"]) < 1e-5
    assert rel(gp.sampled(b["encoder_out_for_ctc"][0], T + 1), pins[f"encoder/{T}/encoder_out_for_ctc"]) < 1e-5


def test_reference_conv_feature_extractor_real_width_matches_oracle():
    """ConvFeatureExtractionModel (speech_encoder_prenet.py:277-374) at the real 512 channels, both modes, 1 s of audio,
    on the same seeded weights."""
    from oracle.speecht5_oracle_asr import CONV_FEATURE_LAYERS, ConvFeatureExtractionModel
    pins = load("ref_pins")
    x = gp.conv_input()
    for mode in ("default", "layer_norm"):
        orc = gp.seeded_fill(ConvFeatureExtractionModel(CONV_FEATURE_LAYERS, mode, False), 5).eval()
        with torch.no_grad():
            y = orc(x)
        assert list(y.shape) == pins[f"conv/{mode}/shape"].tolist(), mode
        assert rel(gp.sampled(y, 5), pins[f"conv/{mode}/out"]) < 1e-5, mode


def test_reference_generate_speech_matches_oracle_autoregressive_synthesis():
    """`T5TransformerModel.generate_speech` (models/speecht5.py:1188-1249; its always-on prenet dropout disabled with
    dprenet_dropout_rate 0) against the oracle's synthesis loop on the same seeded weights: same number of frames, same
    mel."""
    from oracle.speecht5_oracle import T5TransformerModelOracle, base_args
    want = load("ref_pins")["generate_speech/mel"]
    orc = gp.seeded_fill(T5TransformerModelOracle(base_args(**mg.TINY)), 21).eval()
    toks, spk = gp.speech_input()
    with torch.no_grad():
        b = orc.generate_speech(src_tokens=toks, spkembs=spk, threshold=0.5, minlenratio=0.0, maxlenratio=2.0)
    assert tuple(b[0].shape) == want.shape
    assert rel(b[0], want) < 1e-4


def test_reduce_metrics_logs_the_reference_keys_and_values():
    """SpeechT5Criterion.reduce_metrics (criterions/speecht5_criterion.py:123-436) run by the reference itself and by the
    plugin on the same logging outputs: same meter names, same values."""
    from speecht5_b200.criterions import SpeechT5Criterion
    from speecht5_b200.fairseq_shim import metrics as ours
    want = pins_json()["reduce_metrics"]
    ours.reset()
    SpeechT5Criterion.reduce_metrics(gp.metric_logs())
    assert set(ours.scalars) == set(want["logged"]), set(ours.scalars) ^ set(want["logged"])
    for k, v in want["logged"].items():
        assert abs(float(ours.scalars[k]) - v) < 1e-9, k
    assert set(ours.derived) == set(want["derived"])


def test_train_step_returns_the_reference_logging_shape():
    """tasks/speecht5.py:519-556: (loss, 1.0, {task_name: log, 'sample_size': 1, 'loss': ..})."""
    import inspect
    from speecht5_b200.tasks import SpeechT5Task
    src = inspect.getsource(SpeechT5Task.train_step)
    assert 'agg[sample["task_name"]] = logging_output' in src and '"sample_size": 1' in src


class _PretrainStub(torch.nn.Module):
    """A model-shaped object that returns canned tensors: what the pre-training criteria read from a model
    (models/speecht5.py:731-784 helpers, shared by the reference's criterion and ours, so that the comparison isolates the
    criterion arithmetic). The forward outputs carry gradients back to `self.leaf` tensors."""

    reduction_factor = 2

    def __init__(self, seed, text=False):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        B, T, r, odim, V = 3, 11, 2, 80, 37
        self.text = text
        if text:
            self.logits = torch.nn.Parameter(torch.randn(B, 9, V, generator=g))
            self.pp = torch.nn.Parameter(torch.tensor(12.5))
        else:
            self.lm = torch.nn.Parameter(torch.randn(17, 101, generator=g))
            self.lu = torch.nn.Parameter(torch.randn(40, 101, generator=g))
            self.pen = torch.nn.Parameter(torch.tensor(0.37))
            self.pp = torch.nn.Parameter(torch.tensor(55.0))
            self.before = torch.nn.Parameter(torch.randn(B, T * r, odim, generator=g))
            self.after = torch.nn.Parameter(torch.randn(B, T * r, odim, generator=g))
            self.stop = torch.nn.Parameter(torch.randn(B, T * r, generator=g))
        self.calls = []

    def forward(self, target_list=None, **net_input):
        self.calls.append(dict(net_input, has_targets=target_list is not None))
        if self.text:
            return (self.logits, None), {"prob_perplexity": self.pp, "code_perplexity": torch.tensor(7.0), "num_vars": 200,
                                         "temp": 2.0}, {"encoder_out": [None]}
        out = {"logit_m_list": [self.lm], "logit_u_list": [self.lu], "features_pen": self.pen, "prob_perplexity": self.pp,
               "code_perplexity": torch.tensor(31.0), "num_vars": 200, "temp": torch.tensor(2.0)}
        if net_input.get("only_hubert"):
            return out, None
        attn = torch.softmax(torch.zeros(3, 12, 11, 6), -1)
        return out, (self.before, self.after, self.stop, [attn, attn])

    from speecht5_b200.models.speecht5 import T5TransformerModel as _M
    get_logits, get_targets, get_extra_losses = _M.get_logits, _M.get_targets, _M.get_extra_losses
    get_normalized_probs = _M.get_normalized_probs


def _speech_pretrain_sample():
    g = torch.Generator().manual_seed(9)
    B, L, odim = 3, 22, 80
    lens = torch.tensor([22, 18, 13])
    labels = torch.zeros(B, L)
    for b, n in enumerate(lens):
        labels[b, n - 1:] = 1.0
    return {"id": torch.arange(B), "target_list": [torch.zeros(B, 30, dtype=torch.long)], "net_input": {"source": None},
            "labels": labels, "dec_target": torch.randn(B, L, odim, generator=g), "dec_target_lengths": lens,
            "src_lengths": torch.tensor([6, 5, 4]), "task_name": "speech_pretrain"}


def text_pretrain_sample(pad):
    tgt = torch.randint(4, 37, (3, 9), generator=torch.Generator().manual_seed(2))
    tgt[1, 6:] = pad
    tgt[2, 3:] = pad
    return {"net_input": {"src_tokens": None}, "target": tgt, "ntokens": int(tgt.ne(pad).sum()), "task_name": "text_pretrain"}


def speech_pretrain_kwargs(dec_weight, nomask, weights):
    return dict(pred_masked_weight=1.0, pred_nomask_weight=nomask, loss_weights=None if weights is None else list(weights),
                log_keys=["temp"], hubert_weight=0.7, dec_weight=dec_weight)


def _close(a, b, tol=1e-5):
    a, b = float(a), float(b)
    return abs(a - b) <= tol * max(1.0, abs(b))


def _assert_criterion_matches(pins, key, stub, got, n_got, log_got):
    """Loss, sample size, every logging key and the gradients on the stub's outputs against the reference's (stored)."""
    assert n_got == pins[key + "/sample_size"] and _close(got, pins[key + "/loss"])
    prefix = key + "/log/"
    log_want = {k[len(prefix):]: v for k, v in pins.items() if k.startswith(prefix)}
    assert set(log_got) == set(log_want), (sorted(log_got), sorted(log_want))
    for k, v in log_want.items():
        assert _close(log_got[k], v), (k, log_got[k], v)
    got.backward()
    for n, q in stub.named_parameters():
        want = pins.get(f"{key}/grad/{n}")
        if want is None:
            assert q.grad is None, n
        else:
            assert torch.allclose(gp.sampled(q.grad, 7), torch.from_numpy(want), rtol=1e-5, atol=1e-7), n


@pytest.mark.parametrize("dec_weight,nomask,weights", gp.SPEECH_PRETRAIN_CASES)
def test_speech_pretrain_criterion_equals_the_reference_criterion(dec_weight, nomask, weights):
    """speecht5_b200/criterions/speech_pretrain_criterion.py against the reference's own SpeechPretrainCriterion
    (speech_pretrain_criterion.py:50-190, loaded unmodified): loss, sample size, every logging key and the gradients on
    the model outputs, with / without the decoder branch, the unmasked term and 1 / 2 / 3 configured extra weights."""
    from speecht5_b200.criterions import SpeechPretrainCriterion
    pins = load("ref_pins")
    key = f"speech_pretrain/{gp.SPEECH_PRETRAIN_CASES.index((dec_weight, nomask, weights))}"
    our_crit = SpeechPretrainCriterion(rl.RefTask(mg.VOCAB, "pretrain"), True,
                                       **speech_pretrain_kwargs(dec_weight, nomask, weights))
    ms_our = _PretrainStub(4)
    got, n_got, log_got = our_crit(ms_our, _speech_pretrain_sample())
    assert ms_our.calls[0].get("only_hubert", False) == bool(pins[key + "/only_hubert"]) == (dec_weight == 0)
    _assert_criterion_matches(pins, key, ms_our, got, n_got, log_got)


@pytest.mark.parametrize("sentence_avg,weights", gp.TEXT_PRETRAIN_CASES)
def test_text_pretrain_criterion_equals_the_reference_criterion(sentence_avg, weights):
    """speecht5_b200/criterions/text_pretrain_criterion.py against the reference's TextPretrainCriterion
    (text_pretrain_criterion.py:36-105): padded targets, both sample-size modes, and the reference's weight-list rule
    when more weights than extra terms are configured (it keeps the tail, :74-75)."""
    from speecht5_b200.criterions import TextPretrainCriterion
    pins = load("ref_pins")
    key = f"text_pretrain/{gp.TEXT_PRETRAIN_CASES.index((sentence_avg, weights))}"
    task = rl.RefTask(mg.VOCAB, "pretrain")
    ms_our = _PretrainStub(6, text=True)
    got, n_got, log_got = TextPretrainCriterion(task, sentence_avg, 0.9, list(weights))(
        ms_our, text_pretrain_sample(task.target_dictionary.pad()))
    _assert_criterion_matches(pins, key, ms_our, got, n_got, log_got)


def test_vocabulary_files_load_like_the_reference_dictionary(tmp_path):
    """speecht5_b200/dictionary.py (what SpeechT5Task.setup_task loads `dict.txt` / `dict.<label>.txt` with when fairseq
    is not importable) against the reference's own fairseq Dictionary: same indices, length, lookups, appended task
    symbols and id -> text conversion; then the task built from a data directory (tasks/speecht5.py:272-318)."""
    from speecht5_b200.dictionary import Vocabulary
    from speecht5_b200.tasks import SpeechT5Task
    from speecht5_b200.models import make_args
    ref = pins_json()["dictionary"]
    words = gp.VOCAB_WORDS
    (tmp_path / "dict.txt").write_text("".join(f"{w} {100 - i}\n" for i, w in enumerate(words)), encoding="utf-8")
    (tmp_path / "dict.km.txt").write_text("".join(f"{i} 1\n" for i in range(25)), encoding="utf-8")
    got = Vocabulary.load(str(tmp_path / "dict.txt"))
    assert len(got) == ref["len"] == 4 + len(words) and got.symbols == ref["symbols"] and got.indices == ref["indices"]
    assert [got.bos(), got.pad(), got.eos(), got.unk()] == ref["specials"] == [0, 1, 2, 3]
    for w in words + ["missing", "<pad>"]:
        assert got.index(w) == ref["index"][w]
    assert [got.add_symbol("<mask>"), got.add_symbol("e")] == ref["add_symbol"]
    assert list(got.count) == ref["count"] and got[999] == ref["item_999"]
    ids = torch.tensor(gp.VOCAB_IDS)
    assert got.string(ids, extra_symbols_to_ignore={1}) == ref["string_ignore_pad"]
    assert got.string(ids[0], include_eos=True, unk_string="?") == ref["string_eos_unk"]
    (tmp_path / "dup.txt").write_text("a 1\na 2\n")
    with pytest.raises(RuntimeError):
        Vocabulary.load(str(tmp_path / "dup.txt"))
    # the task: vocabulary from <data>/dict.txt, <mask> and <ctc_blank> appended, HuBERT label sets for pre-training
    args = make_args("t5_transformer_base_asr", data=str(tmp_path), t5_task="pretrain", hubert_labels=["km"],
                     hubert_label_dir=str(tmp_path), build_speech_encoder=True, use_conv_pos=True, use_sinc_pos=True,
                     encoder_layers=1, decoder_layers=1)
    task = SpeechT5Task.setup_task(args)
    n = 4 + len(words)
    assert (task.mask_idx, task.blank_symbol_idx) == (n, n + 1) and len(task.target_dictionary) == n + 2
    assert len(task.dicts["hubert"]) == 1 and len(task.dicts["hubert"][0]) == 4 + 25
    model = task.build_model(args)
    assert model.text_encoder_prenet.encoder_prenet[0].weight.shape[0] == n + 2
    assert model.hubert_layer is not None


@pytest.mark.parametrize("arch", gp.ARCHS)
def test_arch_presets_equal_the_reference_arch_functions(arch):
    """models/speecht5.py:1252-1447: every option both sides know gets the value the reference's OWN arch function
    assigns (run unmodified through oracle/ref_loader.py) -- layer counts, widths, dropouts, extractor mode, final_dim,
    codebook sizes, positional options: what decides whether a reference checkpoint loads and trains the same."""
    from speecht5_b200.models import make_args
    ref = pins_json()["arch_presets"][arch]
    ours = gp.plain(vars(make_args(arch)))
    shared = [k for k in ours if k in ref]
    assert len(shared) >= 80
    for k in ("final_dim", "latent_vars", "latent_groups", "latent_temp", "codebook_prob", "logit_temp", "extractor_mode",
              "use_conv_pos", "use_sinc_pos", "untie_final_proj", "label_rates"):
        assert k in shared, k
    diff = {k: (ours[k], ref[k]) for k in shared if ours[k] != ref[k]}
    assert not diff, diff


def test_criterion_config_defaults_equal_the_reference_dataclass():
    """speecht5_criterion.py:23-30: fairseq builds the criterion from this dataclass, so its defaults decide what a
    recipe that omits a flag trains with. Every field both sides define has the reference's default (sentence_avg is an
    interpolation of optimization.sentence_avg there)."""
    from speecht5_b200.criterions.speecht5_criterion import SpeechT5CriterionConfig
    ref, ours = pins_json()["criterion_config_defaults"], gp.plain(gp.dataclass_defaults(SpeechT5CriterionConfig))
    shared = [k for k in ours if k in ref and k != "sentence_avg"]
    assert len(shared) >= 20
    diff = {k: (ours[k], ref[k]) for k in shared
            if (list(ours[k]) != list(ref[k]) if isinstance(ours[k], (list, tuple)) else ours[k] != ref[k])}
    assert not diff, diff


def test_model_command_line_options_cover_the_reference_add_args():
    """models/speecht5.py:117-560 (T5TransformerModel.add_args of the reference, run unmodified): every option it
    defines is defined here with the same value type and choices, so a recipe's command line -- README fine-tuning
    commands pass --freeze-encoder-updates, --mask-prob, --mask-channel-prob, --feature-grad-mult -- parses under this
    plugin; ours adds only the two opt-in builders."""
    from speecht5_b200.models import T5TransformerModel
    ref = pins_json()["model_options"]
    parser, ours = gp.model_options(T5TransformerModel)
    ours = gp.plain(ours)
    assert sorted(k for k in ref if k not in ours) == []
    assert sorted(k for k in ours if k not in ref) == ["build_speech_encoder", "build_text_decoder"]
    loose = {"latent_temp", "mask_selection", "mask_channel_selection"}  # (str vs literal_eval / untyped: same strings accepted)
    diff = {k: (ours[k], ref[k]) for k in ref if k not in loose and ours[k] != ref[k]}
    assert not diff, diff
    got = parser.parse_args("--share-input-output-embed --bert-init --relative-position-embedding --freeze-encoder-updates "
                            "13000 --mask-prob 0.5 --mask-channel-prob 0.5 --feature-grad-mult 1.0 --dropout 0.1 "
                            "--use-codebook --codebook-prob 0.1 --sid-no-pooling-bn --sid-no-embed-postnet".split())
    assert got.freeze_encoder_updates == 13000 and got.mask_prob == 0.5 and got.feature_grad_mult == 1.0
    assert not hasattr(got, "encoder_layers")  # unset options fall through to the arch function


def test_task_command_line_options_equal_the_reference_add_args():
    """tasks/speecht5.py:44-213 (SpeechT5Task.add_args; the module itself needs fairseq's data package, so its
    add_argument calls are read from the source text): same flags, value types, defaults, choices and actions here."""
    from speecht5_b200.tasks.speecht5 import SpeechT5Task
    ref = pins_json()["task_options"]
    ours = {}
    for flag, kw in SpeechT5Task._OPTIONS:
        kw = {k: (getattr(v, "__name__", v) if k == "type" else v) for k, v in kw.items() if k not in ("help", "metavar")}
        ours[flag] = gp.plain(kw)
    assert sorted(k for k in ref if k not in ours) == ["data"]  # (the positional argument, added in add_args itself)
    assert sorted(k for k in ours if k not in ref) == []
    ref["--t5-task"]["choices"] = gp.plain(SpeechT5Task.TASK_NAME)  # (the reference names its list the same way, :40)
    diff = {k: (ours[k], ref[k]) for k in ours if ours[k] != ref[k]}
    assert not diff, diff
    assert len(ours) >= 35
