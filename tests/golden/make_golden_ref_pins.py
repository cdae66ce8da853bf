"""Golden data for the reference pins of tests/test_ref_pin_cpu.py and tests/test_docs_cpu.py that used to need the
reference tree at test time. Run where the reference is available (ST5_REFERENCE_ROOT, see oracle/ref_loader.py):

    python tests/golden/make_golden_ref_pins.py   -> tests/golden/ref_pins.json, tests/golden/ref_pins.npz

ref_pins.json holds what the reference's own code returns for the configuration pins (arch functions, add_args,
criterion dataclass, reduce_metrics, fairseq Dictionary) and the line count of every reference file the sources cite.
ref_pins.npz holds reference outputs on seeded weights (`seeded_fill`): the encoder at ASR lengths, the conv feature
extractor at real width, generate_speech, and the two pre-training criteria on fixed stub outputs. Large outputs are
stored as a seeded sample of elements (`sample_index`), so every file stays small.
"""
import argparse
import ast
import dataclasses
import glob
import importlib
import json
import os
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (ROOT, HERE, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
import make_golden_from_ref as mg  # noqa: E402
from oracle import ref_loader as rl  # noqa: E402

JSON_PATH = os.path.join(HERE, "ref_pins.json")
NPZ_PATH = os.path.join(HERE, "ref_pins.npz")
SAMPLE = 2048  # elements kept of an output larger than that
ENCODER_T = (199, 499)
ARCHS = ("t5_transformer", "t5_transformer_base", "t5_transformer_large", "t5_transformer_base_asr")
SPEECH_PRETRAIN_CASES = ((1.0, 0.0, [10.0]), (0.0, 0.5, [10.0, 0.1]), (0.5, 1.0, [10.0, 0.1, 3.0]), (1.0, 0.0, None))
TEXT_PRETRAIN_CASES = ((False, [0.1]), (True, [0.1]), (False, [0.1, 2.0]))
VOCAB_WORDS = ["▁", "e", "t", "a", "o", "n", "'", "<weird token>", "zz"]
VOCAB_IDS = [[0, 5, 6, 3, 2, 1], [7, 8, 4, 2, 1, 1]]


# ----------------------------------------------------------------------------------------- shared with the tests
def seeded_fill(module, seed):
    """Deterministic weights independent of how a module initialises itself: parameters in name order, matrices
    N(0, 1/fan_in), 1-D weights / scales 1 + N(0, 0.1^2), other 1-D parameters N(0, 0.1^2). Buffers are left as built."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in sorted(module.named_parameters()):
            z = torch.randn(p.shape, generator=g, dtype=torch.float64)
            if p.dim() >= 2:
                p.copy_(z * p[0].numel() ** -0.5)
            elif name.endswith(("weight", "alpha", "weight_g")):
                p.copy_(1.0 + 0.1 * z)
            else:
                p.copy_(0.1 * z)
    return module


def sample_index(numel, seed, n=SAMPLE):
    """Fixed flat indices of an output of `numel` elements (all of them when it is small)."""
    if numel <= n:
        return torch.arange(numel)
    return torch.randperm(numel, generator=torch.Generator().manual_seed(seed))[:n].sort().values


def sampled(t, seed):
    t = t.detach().reshape(-1)
    return t[sample_index(t.numel(), seed)]


def encoder_input(T):
    x = torch.randn(2, T, 768, generator=torch.Generator().manual_seed(1))
    pad = torch.zeros(2, T, dtype=torch.bool)
    pad[1, T - 37:] = True
    return x, pad


def encoder_over():
    return dict(encoder_layers=2, dropout=0.0, attention_dropout=0.0, activation_dropout=0.0, encoder_layerdrop=0.0)


def conv_input():
    return torch.randn(2, 16000, generator=torch.Generator().manual_seed(1)) * 0.1


def speech_input():
    g = torch.Generator().manual_seed(2)
    return torch.randint(4, 70, (1, 12), generator=g), torch.randn(1, 512, generator=g)


def task_options_from_source(src):
    """The add_argument calls of a task module's source text: flag -> keyword values (help / metavar dropped)."""
    ref = {}
    for node in ast.walk(ast.parse(src)):
        if isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute) and node.func.attr == "add_argument":
            flags = [a.value for a in node.args if isinstance(a, ast.Constant)]
            kw = {}
            for k in node.keywords:
                if k.arg in ("help", "metavar"):
                    continue
                try:
                    kw[k.arg] = ast.literal_eval(k.value)
                except ValueError:
                    kw[k.arg] = getattr(k.value, "id", None) or ast.unparse(k.value)
            ref[flags[-1]] = kw
    return ref


def model_options(cls):
    """dest -> (option strings, action class, value type, choices) of a model's add_args."""
    p = argparse.ArgumentParser(allow_abbrev=False)
    cls.add_args(p)
    return p, {a.dest: (tuple(a.option_strings), type(a).__name__, getattr(a.type, "__name__", a.type),
                        tuple(a.choices) if a.choices else None) for a in p._actions if a.dest != "help"}


def dataclass_defaults(cls):
    out = {}
    for f in dataclasses.fields(cls):
        if f.default is not dataclasses.MISSING:
            out[f.name] = f.default
        elif f.default_factory is not dataclasses.MISSING:
            out[f.name] = f.default_factory()
    return out


def metric_logs():
    """Logging outputs of one update per task, as SpeechT5Criterion.reduce_metrics receives them."""
    t2s = {"loss": 1.5, "l1_loss": 1.0, "l2_loss": 2.0, "bce_loss": 0.5, "sample_size": 1, "ntokens": 100,
           "nsentences": 4, "enc_dec_attn_loss": 0.01, "encoder_alpha": 1.0, "decoder_alpha": 1.1}
    s2t = {"loss": 80.0, "ce_loss": 60.0, "ctc_loss": 100.0, "nll_loss": 55.0, "ntokens": 37, "nsentences": 3,
           "sample_size": 3, "n_correct": 11, "total": 37, "c_errors": 5, "c_total": 30, "w_errors": 2, "wv_errors": 3,
           "w_total": 9}
    text = {"loss": 12.0, "bart_loss": 12.0, "ntokens": 50, "sample_size": 50, "loss_prob_perplexity": 0.3,
            "code_perplexity": 17.0}
    hub = {"loss": 9.0, "ntokens": 20, "sample_size": 20, "dec_loss": 1.0, "l1_loss": 0.5, "l2_loss": 0.6, "bce_loss": 0.1,
           "ngpu": 1, "count_m_0": 12, "correct_m_0": 5, "loss_m_0": 7.0, "enc_dec_attn_loss": 0.02}
    return [{"t2s": t2s, "sample_size": 1, "loss": 1.5}, {"t2s": dict(t2s, loss=2.5), "sample_size": 1, "loss": 2.5},
            {"s2t": s2t, "sample_size": 1, "loss": 80.0 / 3}, {"text_pretrain": text, "sample_size": 1, "loss": 0.24},
            {"speech_pretrain": hub, "sample_size": 1, "loss": 0.45}]


def cited_reference_paths(root=ROOT):
    """Every `<file>.py:<line>[-<line>]` citation in the sources and docs that does not name a file of this repository
    (tools/check_citations.py)."""
    sys.path.insert(0, os.path.join(root, "tools"))
    import check_citations as cc
    return cc.citations(root)


def plain(v):
    """JSON form of an option value (tuples as lists, callables by name)."""
    if isinstance(v, (list, tuple)):
        return [plain(x) for x in v]
    if isinstance(v, dict):
        return {k: plain(x) for k, x in v.items()}
    if v is None or isinstance(v, (bool, int, float, str)):
        return v
    return getattr(v, "__name__", repr(v))


# ------------------------------------------------------------------------------------------------- generation
def json_pins():
    ns = rl.load()
    out = {}
    out["arch_presets"] = {a: plain(vars(rl.reference_args(arch=a))) for a in ARCHS}
    crit = importlib.import_module("speecht5.criterions.speecht5_criterion")
    out["criterion_config_defaults"] = plain(dataclass_defaults(crit.SpeechT5CriterionConfig))
    out["model_options"] = plain(model_options(ns.T5TransformerModel)[1])
    with open(os.path.join(rl.ST5, "speecht5", "tasks", "speecht5.py")) as fh:
        out["task_options"] = plain(task_options_from_source(fh.read()))
    ns.metrics.logged.clear()
    ns.metrics.derived.clear()
    crit.SpeechT5Criterion.reduce_metrics(metric_logs())
    out["reduce_metrics"] = {"logged": {k: float(v) for k, v in ns.metrics.logged.items()},
                             "derived": sorted(ns.metrics.derived)}
    out["dictionary"] = _dictionary_pins()
    out["reference_line_counts"] = _line_counts()
    return out


def _reference_dictionary_class():
    """fairseq/data/dictionary.py of the reference, executed unmodified with its five package imports stubbed (utils,
    binarizer.safe_readline, data.data_utils, file_io.PathManager, tokenizer.tokenize_line: none of them is reached by
    load / add_symbol / index / string on an in-memory id list)."""
    import types
    path = os.path.join(rl.FAIRSEQ, "data", "dictionary.py")
    names = ["fairseq", "fairseq.utils", "fairseq.binarizer", "fairseq.data", "fairseq.data.data_utils", "fairseq.file_io",
             "fairseq.tokenizer"]
    saved = {n: sys.modules.get(n) for n in names}
    try:
        mods = {n: types.ModuleType(n) for n in names}
        mods["fairseq"].utils = mods["fairseq.utils"]
        mods["fairseq.utils"].item = lambda t: t.item() if hasattr(t, "item") else t
        mods["fairseq.binarizer"].safe_readline = lambda f: f.readline()
        mods["fairseq.data"].data_utils = mods["fairseq.data.data_utils"]
        mods["fairseq.data.data_utils"].post_process = lambda s, sym: s
        mods["fairseq.file_io"].PathManager = type("PathManager", (), {"get_local_path": staticmethod(lambda p: p)})
        mods["fairseq.tokenizer"].tokenize_line = lambda line: line.split()
        sys.modules.update(mods)
        ns = {"__name__": "fairseq_dictionary_under_test"}
        exec(compile(open(path).read(), path, "exec"), ns)
        return ns["Dictionary"]
    finally:
        for n, m in saved.items():
            if m is None:
                sys.modules.pop(n, None)
            else:
                sys.modules[n] = m


def _dictionary_pins():
    Ref = _reference_dictionary_class()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "dict.txt")
        with open(path, "w", encoding="utf-8") as fh:
            fh.write("".join(f"{w} {100 - i}\n" for i, w in enumerate(VOCAB_WORDS)))
        ref = Ref.load(path)
    out = {"len": len(ref), "symbols": list(ref.symbols), "indices": dict(ref.indices),
           "specials": [ref.bos(), ref.pad(), ref.eos(), ref.unk()],
           "index": {w: ref.index(w) for w in VOCAB_WORDS + ["missing", "<pad>"]}}
    out["add_symbol"] = [ref.add_symbol("<mask>"), ref.add_symbol("e")]
    out["count"] = list(ref.count)
    out["item_999"] = ref[999]
    ids = torch.tensor(VOCAB_IDS)
    out["string_ignore_pad"] = ref.string(ids, extra_symbols_to_ignore={1})
    out["string_eos_unk"] = ref.string(ids[0], include_eos=True, unk_string="?")
    return out


def _line_counts():
    """Line count of every reference .py file a citation can resolve to (all files sharing a cited path's tail)."""
    ref_root = rl.REF_ROOT
    files = [p[len(ref_root) + 1:] for p in glob.glob(ref_root + "/**/*.py", recursive=True)]
    tails = {c[0] for c in cited_reference_paths()}
    keep = sorted(f for f in files if any(f == t or f.endswith("/" + t) for t in tails))
    out = {}
    for f in keep:
        with open(os.path.join(ref_root, f), errors="ignore") as fh:
            out[f] = sum(1 for _ in fh)
    return out


def array_pins():
    import test_ref_pin_cpu as t
    from oracle.speecht5_oracle import T5TransformerModelOracle, TransformerEncoder, base_args
    from oracle.speecht5_oracle_asr import CONV_FEATURE_LAYERS, ConvFeatureExtractionModel, reference_to_oracle_keys
    ns = rl.load()
    blob = {}
    # encoder at ASR lengths (Base width, 2 layers, relative positions clipped at +-160, key padding)
    over = encoder_over()
    enc_ref = ns.encoder.TransformerEncoder(rl.reference_args(**over), rl.RefDictionary(mg.VOCAB), None).eval()
    enc = seeded_fill(TransformerEncoder(base_args(**over), mg.VOCAB, None), 3)
    enc_ref.load_state_dict(enc.state_dict())
    for T in ENCODER_T:
        x, pad = encoder_input(T)
        with torch.no_grad():
            a = enc_ref(x, pad)
        blob[f"encoder/{T}/encoder_out"] = sampled(a["encoder_out"][0], T).numpy()
        blob[f"encoder/{T}/encoder_out_for_ctc"] = sampled(a["encoder_out_for_ctc"][0], T + 1).numpy()
    # conv feature extractor at the real 512 channels, both modes
    for mode in ("default", "layer_norm"):
        ref = ns.speech_encoder_prenet.ConvFeatureExtractionModel(CONV_FEATURE_LAYERS, 0.0, mode, False).eval()
        orc = seeded_fill(ConvFeatureExtractionModel(CONV_FEATURE_LAYERS, mode, False), 5)
        names = reference_to_oracle_keys({k: k for k in ref.state_dict()})
        osd = orc.state_dict()
        ref.load_state_dict({rk: osd[ok] for ok, rk in names.items()})
        with torch.no_grad():
            y = ref(conv_input())
        blob[f"conv/{mode}/shape"] = np.array(y.shape)
        blob[f"conv/{mode}/out"] = sampled(y, 5).numpy()
    # generate_speech of the full reference model on the oracle's seeded weights
    over = dict(mg.TINY, conv_feature_layers=mg.TINY_CONV, conv_pos=16, conv_pos_groups=4)
    ref = rl.build_reference_model(rl.reference_args(**over), rl.RefTask(mg.VOCAB, "t2s")).eval()
    orc = seeded_fill(T5TransformerModelOracle(base_args(**mg.TINY)), 21).eval()
    rsd, osd = ref.state_dict(), orc.state_dict()
    assert set(osd) <= set(rsd), set(osd) - set(rsd)
    with torch.no_grad():  # (in place: the reference model's load_state_dict expects a full checkpoint)
        for k, v in osd.items():
            rsd[k].copy_(v)
    toks, spk = speech_input()
    with torch.no_grad():
        mel = ref.generate_speech(source=None, src_tokens=toks, spkembs=spk, threshold=0.5, minlenratio=0.0,
                                  maxlenratio=2.0)[0]
    blob["generate_speech/mel"] = mel.numpy()
    # pre-training criteria on fixed stub outputs
    from_ref = importlib.import_module("speecht5.criterions.speech_pretrain_criterion")
    for i, (dec_weight, nomask, weights) in enumerate(SPEECH_PRETRAIN_CASES):
        crit = from_ref.SpeechPretrainCriterion(rl.RefTask(mg.VOCAB, "pretrain"), True,
                                                **t.speech_pretrain_kwargs(dec_weight, nomask, weights))
        stub = t._PretrainStub(4)
        loss, n, log = crit(stub, t._speech_pretrain_sample())
        loss.backward()
        _store_criterion(blob, f"speech_pretrain/{i}", stub, loss, n, log)
        blob[f"speech_pretrain/{i}/only_hubert"] = np.array(bool(stub.calls[0].get("only_hubert", False)))
    from_ref = importlib.import_module("speecht5.criterions.text_pretrain_criterion")
    for i, (sentence_avg, weights) in enumerate(TEXT_PRETRAIN_CASES):
        task = rl.RefTask(mg.VOCAB, "pretrain")
        stub = t._PretrainStub(6, text=True)
        loss, n, log = from_ref.TextPretrainCriterion(task, sentence_avg, 0.9, list(weights))(
            stub, t.text_pretrain_sample(task.target_dictionary.pad()))
        loss.backward()
        _store_criterion(blob, f"text_pretrain/{i}", stub, loss, n, log)
    return blob


def _store_criterion(blob, key, stub, loss, n, log):
    blob[key + "/loss"] = np.array(loss.item(), dtype=np.float64)
    blob[key + "/sample_size"] = np.array(float(n), dtype=np.float64)
    for k, v in log.items():
        blob[f"{key}/log/{k}"] = np.array(float(v), dtype=np.float64)
    for name, p in stub.named_parameters():
        if p.grad is not None:
            blob[f"{key}/grad/{name}"] = sampled(p.grad, 7).numpy()


def main():
    assert rl.available(), f"reference tree not found under {rl.REF_ROOT}"
    pins = json_pins()
    with open(JSON_PATH, "w", encoding="utf-8") as fh:
        json.dump(pins, fh, indent=0, sort_keys=True, ensure_ascii=False)
        fh.write("\n")
    np.savez_compressed(NPZ_PATH, **array_pins())
    print(JSON_PATH, os.path.getsize(JSON_PATH), NPZ_PATH, os.path.getsize(NPZ_PATH))


if __name__ == "__main__":
    main()
