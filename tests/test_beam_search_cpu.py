"""CPU: beam search with joint CTC/attention scoring (speecht5_b200/beam.py, csrc/ctc_prefix.cu). The oracle scorer
(tests/beam_oracle.py) against brute-force enumeration of CTC alignments and against the reference's own scorer; the
oracle search and the product's BeamSearchGenerator (kernels restated on the CPU) against the reference
SequenceGenerator's n-best lists (tests/golden/ref_asr_beam_tiny.npz, tests/golden/make_golden_beam.py)."""
import itertools
import math
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import beam_oracle as BO
import gemm_emulator

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden", "ref_asr_beam_tiny.npz")
V_TINY = 81
BLANK, MASK = V_TINY - 1, V_TINY - 2
CASES = {"a": dict(beam=4, ctc_weight=0.0, alone=False), "b": dict(beam=4, ctc_weight=0.5, alone=True),
         "c": dict(beam=3, ctc_weight=0.3, alone=True, len_penalty=0.5, min_len=3)}


def _reference_tree():
    from oracle import ref_loader as rl
    return rl.REF_ROOT if rl.available() else None


# ---------------------------------------------------------------------------------------------- brute force
def _collapse(path, blank):
    out, prev = [], None
    for s in path:
        if s != blank and s != prev:
            out.append(s)
        prev = s
    return out


def _brute_states(p, g, blank):
    """r_n[t], r_b[t] of prefix g: probability that frames 0..t collapse to g, ending in a label / in blank."""
    T, V = p.shape
    rn, rb = np.zeros(T), np.zeros(T)
    for t in range(T):
        for path in itertools.product(range(V), repeat=t + 1):
            if _collapse(path, blank) == list(g):
                pr = np.prod([p[i, s] for i, s in enumerate(path)])
                if path[-1] == blank:
                    rb[t] += pr
                else:
                    rn[t] += pr
    return rn, rb


def _brute_psi(p, g, c, blank, eos):
    T, V = p.shape
    total = 0.0
    for path in itertools.product(range(V), repeat=T):
        out = _collapse(path, blank)
        pr = np.prod([p[i, s] for i, s in enumerate(path)])
        if c == eos:
            total += pr if out == list(g) else 0.0
        elif out[: len(g) + 1] == list(g) + [c]:
            total += pr
    return total


def _log(v):
    return np.where(v > 0, np.log(np.maximum(v, 1e-300)), BO.LOGZERO)


@pytest.mark.parametrize("T,g", [(5, []), (5, [1]), (5, [1, 1]), (5, [2, 1]), (4, [1, 2, 1]), (3, [1, 2, 1]),
                                 (3, [1, 2, 1, 2]), (6, [2])])
def test_oracle_scorer_equals_brute_force_enumeration(T, g):
    """psi = sum over every alignment whose collapse starts with g + c (eos: equals g); states r_n / r_b of g + c;
    blank (0), eos (3), the repeated last label and out_len >= T included."""
    rng = np.random.default_rng(T * 7 + len(g))
    V, blank, eos = 4, 0, 3
    p = rng.dirichlet(np.ones(V), size=T)
    x = np.log(p)
    rn, rb = _brute_states(p, g, blank)
    if len(g) == 0:
        r_prev = BO.ctc_initial_state(x, blank, dtype=np.float64)
        assert np.allclose(np.exp(r_prev[:, 1]), rb, atol=1e-12)
    else:
        r_prev = np.stack([_log(rn), _log(rb)], -1)
    cs = np.arange(V)
    psi, r = BO.ctc_prefix_score(x, r_prev, g[-1] if g else eos, len(g), cs, blank, eos, dtype=np.float64)
    for k, c in enumerate(cs):
        if c == blank:
            assert psi[k] == BO.LOGZERO
            continue
        want = _brute_psi(p, g, c, blank, eos)
        assert abs(math.exp(psi[k]) - want) < 1e-10, (c, math.exp(psi[k]), want)
        if c != eos:
            wn, wb = _brute_states(p, list(g) + [c], blank)
            assert np.allclose(np.exp(r[k, :, 0]), wn, atol=1e-10) and np.allclose(np.exp(r[k, :, 1]), wb, atol=1e-10)


def test_oracle_scorer_equals_the_reference_scorer():
    """The reference tree's own CTCPrefixScore (the vendored espnet file) on random inputs, float32 as it runs."""
    root = _reference_tree()
    if root is None:
        pytest.skip("reference tree not present")
    import importlib.util
    spec = importlib.util.spec_from_file_location("_cps", os.path.join(root, "SpeechUT", "speechut", "modules",
                                                                       "ctc_prefix_score.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    rng = np.random.default_rng(0)
    T, V, blank, eos = 23, 12, 11, 2
    x = torch.log_softmax(torch.from_numpy(rng.normal(size=(T, V)) * 3), -1).float().numpy()
    ref = mod.CTCPrefixScore(x, blank, eos, np)
    r_ref, r_mine = ref.initial_state(), BO.ctc_initial_state(x, blank)
    assert np.array_equal(r_ref, r_mine)
    y = [eos]
    for step in range(T + 1):
        cs = rng.permutation(V)[:8]
        cs[0] = eos if step % 3 == 0 else cs[0]
        if step > 0:
            cs[1] = y[-1]
        psi_ref, st_ref = ref(np.array(y), cs, r_ref)
        psi, st = BO.ctc_prefix_score(x, r_mine, y[-1], len(y) - 1, cs, blank, eos)
        assert np.allclose(psi, psi_ref, rtol=1e-6, atol=1e-4), (step, psi, psi_ref)
        j = 1 if step > 0 and cs[1] != eos else 2
        lo = max(len(y) - 2, 0)  # (rows below out_len - 1 are uninitialised in the reference)
        assert np.allclose(st[j][lo:], st_ref[j][lo:], rtol=1e-6, atol=1e-4)
        if len(y) - 1 >= T:
            break
        y.append(int(cs[j]))
        r_ref, r_mine = st_ref[j], st[j]


# ---------------------------------------------------------------------------------------------- kernel program
CHUNK = 32


def kernel_ctc_prefix_init(x, t_valid, r, blank):
    """st5_ctc_prefix_init restated: thread per utterance, sequential fp32 running sum over the valid frames."""
    B, T, _ = x.shape
    for b in range(B):
        Tb = min(T, int(t_valid[b]))
        acc = torch.zeros((), dtype=torch.float32)
        for t in range(T):
            if t < Tb:
                acc = x[b, 0, blank].clone() if t == 0 else acc + x[b, t, blank]
            r[b, t, 0] = BO.LOGZERO
            r[b, t, 1] = acc if t < Tb else BO.LOGZERO


def _lae(a, b):
    a64, b64 = a.double(), b.double()
    return torch.where(a64 == b64, a64 + math.log(2), torch.logaddexp(a64, b64)).float()


def kernel_ctc_prefix_score(x, t_valid, utt, r_prev, last, out_len, cs, log_psi, r, blank, eos):
    """st5_ctc_prefix_score restated: a CTA per hypothesis h, thread k per candidate (vectorised here), frames staged
    CHUNK at a time, output layout [H, T, 2, K], rows outside [start, T_b) logzero, the reference's start row."""
    H, Kc = cs.shape
    T = x.shape[1]
    for h in range(H):
        u = int(utt[h])
        Tb = min(T, int(t_valid[u]))
        L = int(out_len[h])
        c = cs[h]
        rep = (c == last[h]) & (L > 0)
        start = max(min(L, T + 1), 1)
        r[h].fill_(BO.LOGZERO)
        rn = torch.full((Kc,), BO.LOGZERO)
        rb = torch.full((Kc,), BO.LOGZERO)
        psi = torch.full((Kc,), BO.LOGZERO)
        if L == 0 and Tb > 0:
            rn = x[u, 0, c].clone()
            psi = rn.clone()
            r[h, 0, 0] = rn
        for t0 in range(start, Tb, CHUNK):
            n = min(CHUNK, Tb - t0)
            xs = x[u, t0: t0 + n][:, c]                       # staged candidate columns
            xb = x[u, t0: t0 + n, blank]                      # staged blank column
            rp = r_prev[h, t0 - 1: t0 - 1 + n]
            phi_all, rpb = _lae(rp[:, 0], rp[:, 1]), rp[:, 1]
            for i in range(n):
                phi = torch.where(rep, rpb[i], phi_all[i])
                rn_new = _lae(rn, phi) + xs[i]
                rb_new = _lae(rn, rb) + xb[i]
                psi = _lae(psi, phi + xs[i])
                rn, rb = rn_new, rb_new
                r[h, t0 + i, 0] = rn
                r[h, t0 + i, 1] = rb
        if Tb > 0:
            psi = torch.where(c == eos, _lae(r_prev[h, Tb - 1, 0], r_prev[h, Tb - 1, 1]), psi)
        psi = torch.where(c == blank, torch.tensor(BO.LOGZERO), psi)
        log_psi[h] = psi


def kernel_beam_gather_rows(src, dst, parent, n_rows):
    for s, d in zip(src, dst):
        d[:, :n_rows] = s.index_select(0, parent)[:, :n_rows]


def install_kernels(monkeypatch):
    from speecht5_b200 import kernels as K
    monkeypatch.setattr(K, "ctc_prefix_init", kernel_ctc_prefix_init)
    monkeypatch.setattr(K, "ctc_prefix_score", kernel_ctc_prefix_score)
    monkeypatch.setattr(K, "beam_gather_rows", kernel_beam_gather_rows)


def test_kernel_program_equals_the_oracle():
    """Ownership, layout [H, T, 2, K], start row, sentinel and T_b clipping of the restated kernel program against the
    oracle, on two utterances of different valid lengths and mixed prefix lengths (out_len >= T_b included)."""
    rng = np.random.default_rng(5)
    B, T, V, blank, eos = 2, 45, 9, 8, 2
    x = torch.log_softmax(torch.from_numpy(rng.normal(size=(B, T, V)) * 2).float(), -1)
    t_valid = torch.tensor([45, 37])
    r0 = torch.empty(B, T, 2)
    kernel_ctc_prefix_init(x, t_valid, r0, blank)
    for b in range(B):
        want = BO.ctc_initial_state(x[b, : int(t_valid[b])].numpy(), blank)
        assert np.array_equal(r0[b, : int(t_valid[b])].numpy(), want)
    H, Kc = 6, 5
    utt = torch.tensor([0, 0, 1, 1, 1, 0])
    out_len = torch.tensor([0, 3, 1, 36, 40, 44])
    last = torch.tensor([eos, 4, 4, 1, 3, 0])
    cs = torch.stack([torch.from_numpy(rng.permutation(V)[:Kc]) for _ in range(H)])
    cs[1, 0], cs[2, 1], cs[3, 2], cs[4, 0] = 4, eos, blank, eos
    r_prev = torch.stack([r0[int(u)] for u in utt]) + torch.from_numpy(rng.normal(size=(H, T, 2))).float() * 0.1
    psi, r = torch.empty(H, Kc), torch.empty(H, T, 2, Kc)
    kernel_ctc_prefix_score(x, t_valid, utt, r_prev, last, out_len, cs, psi, r, blank, eos)
    for h in range(H):
        u, Tb = int(utt[h]), int(t_valid[int(utt[h])])
        want_psi, want_r = BO.ctc_prefix_score(x[u, :Tb].numpy(), r_prev[h, :Tb].numpy(), int(last[h]), int(out_len[h]),
                                               cs[h].numpy(), blank, eos)
        assert np.allclose(psi[h].numpy(), want_psi, rtol=1e-6, atol=1e-4), h
        assert np.allclose(r[h, :Tb].permute(2, 0, 1).numpy(), want_r, rtol=1e-6, atol=1e-4), h
        assert bool((r[h, Tb:] == BO.LOGZERO).all())


# ---------------------------------------------------------------------------------------------- search
def _blob():
    return dict(np.load(GOLD))


def _emulated_model(monkeypatch, blob):
    from helpers import NO_DROPOUT, TINY
    from test_frontend_cpu import _cpu_extractor_forward
    from speecht5_b200 import frontend
    from speecht5_b200.models import T5TransformerModel, make_args
    from speecht5_b200.ops import RT
    gemm_emulator.install(monkeypatch)
    install_kernels(monkeypatch)
    monkeypatch.setattr(RT, "dtype", torch.float32)
    monkeypatch.setattr(frontend.ConvFeatureExtractor, "forward", _cpu_extractor_forward)
    RT.invalidate_shadows()
    over = dict(TINY, **NO_DROPOUT, bert_init=True, build_speech_encoder=True, build_text_decoder=True,
                conv_feature_layers="[(32, 10, 5)] + [(32, 3, 2)] * 4 + [(32, 2, 2)] * 2", feature_grad_mult=1.0,
                conv_pos=16, conv_pos_groups=4, use_conv_pos=True, use_sinc_pos=True, mask_prob=0.5,
                hubert_mask_length=4, mask_channel_prob=0.25, mask_channel_length=8, max_text_positions=600)
    model = T5TransformerModel.build_model(make_args("t5_transformer_base_asr", **over)).eval()
    model.load_state_dict({k[6:]: torch.from_numpy(v) for k, v in blob.items() if k.startswith("state/")}, strict=False)
    return model


def _inputs(blob, alone):
    src, pm = torch.from_numpy(blob["in/source"]), torch.from_numpy(blob["in/padding_mask"])
    if not alone:
        return [(src, pm)]
    return [(src[i: i + 1, :n], pm[i: i + 1, :n]) for i, n in enumerate((~pm).sum(1).tolist())]


def _expect(blob, name, b, j):
    t = blob[f"{name}/tokens"][b, j]
    n = int((t >= 0).sum())
    return t[:n].tolist(), float(blob[f"{name}/scores"][b, j]), blob[f"{name}/pos_scores"][b, j, :n]


def test_fixture_selections_are_decided_by_clear_margins():
    blob = _blob()
    for name in CASES:
        assert float(blob[f"gap/{name}"]) > 1e-5, name


@pytest.mark.parametrize("name", list(CASES))
def test_oracle_search_reproduces_the_reference_n_best_lists(monkeypatch, name):
    """tests/beam_oracle.py (decoder log-probabilities from the product model on emulated kernels, CTC posteriors the
    reference's own) gives the reference SequenceGenerator's n-best lists: tokens exactly, scores within 1e-5."""
    blob = _blob()
    model = _emulated_model(monkeypatch, blob)
    c = CASES[name]
    b = 0
    for src, pm in _inputs(blob, c["alone"]):
        enc = model.forward_encoder(src, padding_mask=pm)
        for i in range(src.size(0)):
            e_i = model.encoder.reorder_encoder_out(enc, torch.tensor([i]))

            def step_fn(prefixes, e_i=e_i):
                e = model.encoder.reorder_encoder_out(e_i, torch.zeros(prefixes.size(0), dtype=torch.long))
                logits, _ = model.forward_decoder(prefixes, e, incremental_state={})
                return torch.log_softmax(logits[:, -1, :].float(), -1)
            got = BO.beam_search_one(step_fn, c["beam"], V_TINY, 12, ctc_x=blob.get(f"ctc_lprobs/{b}"),
                                     ctc_weight=c["ctc_weight"], min_len=c.get("min_len", 1),
                                     len_penalty=c.get("len_penalty", 1.0), blank=BLANK, mask_idx=MASK)
            assert len(got) == blob[f"{name}/tokens"].shape[1]
            for j, (tok, score, pos) in enumerate(got):
                w_tok, w_score, w_pos = _expect(blob, name, b, j)
                assert tok == w_tok, (name, b, j, tok, w_tok)
                assert abs(score - w_score) < 1e-5, (name, b, j, score, w_score)
                assert np.allclose(pos, w_pos, atol=1e-5)
            b += 1


@pytest.mark.parametrize("use_cache", [False, True])
def test_beam_search_generator_on_emulated_kernels_reproduces_the_fixture(monkeypatch, use_cache):
    """BeamSearchGenerator (the product search, kernels restated on the CPU) on the reference's weights: the reference's
    tokens for every case, on the prefix-recomputing and the key/value-cached path."""
    from speecht5_b200.generator import BeamSearchGenerator
    blob = _blob()
    model = _emulated_model(monkeypatch, blob)
    vocab = SimpleNamespace(pad=lambda: 1, eos=lambda: 2, unk=lambda: 3)
    for name, c in CASES.items():
        gen = BeamSearchGenerator([model], vocab, beam_size=c["beam"], max_len_b=12, min_len=c.get("min_len", 1),
                                  len_penalty=c.get("len_penalty", 1.0), ctc_weight=c["ctc_weight"], blank=BLANK,
                                  mask_idx=MASK, use_cache=use_cache)
        b = 0
        for src, pm in _inputs(blob, c["alone"]):
            for hs in gen.generate([model], {"net_input": {"source": src, "padding_mask": pm}}):
                assert len(hs) == c["beam"]
                for j, h in enumerate(hs):
                    w_tok, w_score, w_pos = _expect(blob, name, b, j)
                    assert h["tokens"].tolist() == w_tok, (name, use_cache, b, j)
                    assert abs(float(h["score"]) - w_score) < 1e-4, (name, b, j)
                    assert h["attention"] is None and h["positional_scores"].shape == (len(w_tok),)
                b += 1


class _TableModel(torch.nn.Module):
    """A decoder that returns a fixed log-probability table per prefix length and fixed CTC posteriors."""

    def __init__(self, lp, ctc):
        super().__init__()
        self.lp, self.ctc = lp, ctc
        self.args = SimpleNamespace(max_text_positions=64)
        self.encoder = SimpleNamespace(reorder_encoder_out=lambda e, order: {**e, "n": order.numel()})

    def forward_encoder(self, source, padding_mask=None):
        return {"encoder_out_for_ctc": [self.ctc[:, None].expand(-1, source.size(0), -1)],
                "encoder_padding_mask": [], "n": source.size(0)}

    def get_normalized_probs_for_ctc(self, enc, log_probs=True):
        return torch.log_softmax(enc["encoder_out_for_ctc"][0], -1)

    def forward_decoder(self, tokens, enc, incremental_state=None):
        return self.lp[min(tokens.size(1) - 1, self.lp.size(0) - 1)][None, None].expand(tokens.size(0), 1, -1), None


def test_a_non_candidate_reaching_the_beam_gets_a_state(monkeypatch):
    """Beam 2, V 20: the CTC term goes to the top ctc_beam = 14 tokens of the decoder's distribution only. The CTC
    posteriors put almost all mass on blank, so every candidate's joint score collapses while the tokens outside the
    candidates keep their attention score and win. The reference would raise KeyError at the next step; here each such
    token is scored with K = 1 and decoding completes, equal to the oracle, which follows the same rule."""
    install_kernels(monkeypatch)
    from speecht5_b200.beam import beam_search
    V, blank, eos = 20, 19, 2
    g = torch.Generator().manual_seed(3)
    lp = torch.log_softmax(torch.randn(6, V, generator=g) * 0.3, -1)
    logits = torch.full((8, V), -12.0)
    logits[:, blank] = 0.0
    model = _TableModel(lp, logits)
    src = torch.zeros(1, 10)
    hyps = beam_search(model, src, None, beam_size=2, ctc_weight=0.9, max_len_b=5, eos=eos, blank=blank, mask_idx=None,
                       vocab_size=V)[0]
    c_lp = lp[0].clone()
    c_lp[blank] = -math.inf
    candidates = set(torch.topk(c_lp, 14).indices.tolist())
    assert all(h["tokens"][0].item() not in candidates for h in hyps)
    x = torch.log_softmax(logits, -1).numpy()
    want = BO.beam_search_one(lambda p: lp[min(p.size(1) - 1, 5)][None].expand(p.size(0), -1), 2, V, 5, ctc_x=x,
                              ctc_weight=0.9, eos=eos, blank=blank)
    assert [h["tokens"].tolist() for h in hyps] == [w[0] for w in want]
    assert np.allclose([float(h["score"]) for h in hyps], [w[1] for w in want], atol=1e-5)


def test_beam_one_equals_greedy(monkeypatch):
    from speecht5_b200.generator import BeamSearchGenerator
    blob = _blob()
    model = _emulated_model(monkeypatch, blob)
    src, pm = _inputs(blob, False)[0]
    greedy = model.generate_text_greedy(src, pm, max_len_b=12, blank=BLANK, mask_idx=MASK)
    vocab = SimpleNamespace(pad=lambda: 1, eos=lambda: 2, unk=lambda: 3)
    gen = BeamSearchGenerator([model], vocab, beam_size=1, max_len_b=12, blank=BLANK, mask_idx=MASK, use_cache=False)
    got = gen.generate([model], {"net_input": {"source": src, "padding_mask": pm}})
    assert [h[0]["tokens"].tolist() for h in got] == [t.tolist() for t in greedy]


def test_build_generator_honours_seq_gen_cls():
    """fairseq's seq_gen_cls selects the beam search, with the task's ctc_weight; without it the default stays."""
    from speecht5_b200.dictionary import Vocabulary
    from speecht5_b200.generator import BeamSearchGenerator, GreedyGenerator
    from speecht5_b200.tasks.speecht5 import SpeechT5Task
    vocab = Vocabulary()
    vocab.add_symbol("<mask>"), vocab.add_symbol("<ctc_blank>")
    task = SpeechT5Task.__new__(SpeechT5Task)
    task.args, task.dicts = SimpleNamespace(ctc_weight=0.5), {"text": vocab}
    task.blank_symbol_idx, task.mask_idx = vocab.index("<ctc_blank>"), vocab.index("<mask>")
    model = SimpleNamespace()
    gen = task.build_generator([model], SimpleNamespace(beam=5), seq_gen_cls=BeamSearchGenerator)
    assert isinstance(gen, BeamSearchGenerator) and gen.beam_size == 5 and gen.ctc_weight == 0.5
    assert gen.blank == vocab.index("<ctc_blank>") and gen.mask_idx == vocab.index("<mask>") and gen.mask_idxs == []
    task.args.ctc_weight = 0.0
    assert isinstance(task.build_generator([model], SimpleNamespace(beam=1)), GreedyGenerator)


def test_regenerating_the_fixture_gives_the_committed_file(tmp_path):
    if _reference_tree() is None:
        pytest.skip("reference tree not present")
    out = tmp_path / "beam.npz"
    r = subprocess.run([sys.executable, os.path.join(HERE, "golden", "make_golden_beam.py"), str(out)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    new, old = dict(np.load(out)), _blob()
    assert sorted(new) == sorted(old)
    for k in old:
        assert np.array_equal(new[k], old[k]), k
