"""-m gpu: the beam-search kernels (csrc/ctc_prefix.cu) against the fp64 oracle (tests/beam_oracle.py), the key/value
row gather against index_select, and BeamSearchGenerator in parity mode against the reference SequenceGenerator's n-best
lists (tests/golden/ref_asr_beam_tiny.npz)."""
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import beam_oracle as BO
from test_ref_pin_gpu import _asr_model

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "ref_asr_beam_tiny.npz")
VOCAB = 81
BLANK, MASK = VOCAB - 1, VOCAB - 2
CASES = {"a": dict(beam=4, ctc_weight=0.0, alone=False), "b": dict(beam=4, ctc_weight=0.5, alone=True),
         "c": dict(beam=3, ctc_weight=0.3, alone=True, len_penalty=0.5, min_len=3)}


@pytest.mark.parametrize("T,H,Kc", [(37, 80, 70), (499, 80, 70), (1500, 24, 64)])
def test_ctc_prefix_kernels_equal_the_fp64_oracle(cuda, T, H, Kc):
    from speecht5_b200 import kernels as K
    rng = np.random.default_rng(T)
    B, V, blank, eos = 4, 81, 80, 2
    x64 = torch.log_softmax(torch.from_numpy(rng.normal(size=(B, T, V)) * 2.5), -1)
    x = x64.float().to(cuda)
    t_valid = torch.tensor([T, T - 5, max(T // 2, 3), T - 1], dtype=torch.long)
    r0 = torch.empty(B, T, 2, device=cuda)
    K.ctc_prefix_init(x, t_valid.to(cuda), r0, blank)
    for b in range(B):
        Tb = int(t_valid[b])
        want = BO.ctc_initial_state(x64[b, :Tb].numpy(), blank, dtype=np.float64)
        got = r0[b, :Tb].double().cpu().numpy()
        assert np.abs(got[:, 1] - want[:, 1]).max() <= 1e-4 * max(1.0, np.abs(want[:, 1]).max())
        assert bool((r0[b, Tb:] == BO.LOGZERO).all()) and bool((r0[b, :, 0] == BO.LOGZERO).all())
    utt = torch.from_numpy(rng.integers(0, B, H))
    out_len = torch.from_numpy(rng.integers(0, T + 3, H))
    out_len[:4] = torch.tensor([0, 1, T, T + 2])  # empty prefix, first label, out_len >= T_b
    out_len[4] = int(t_valid[utt[4]]) - 1
    last = torch.from_numpy(rng.integers(0, V - 1, H))
    last[out_len == 0] = eos
    cs = torch.stack([torch.from_numpy(rng.permutation(V)[:Kc]) for _ in range(H)])
    cs[:, 0] = last  # a repeated last label in every row
    cs[::3, 1] = eos
    cs[::5, 2] = blank
    # previous states: a CTC prefix state of a random prefix (the init state pushed through a few random labels)
    r_prev = torch.stack([r0[int(u)] for u in utt]).double().cpu()
    r_prev[:, :, 0] = torch.where(torch.arange(T)[None] >= 2, r_prev[:, :, 1] - 3.0, torch.tensor(BO.LOGZERO).double())
    r_prev_d = r_prev.float().to(cuda)
    psi = torch.empty(H, Kc, device=cuda)
    r = torch.empty(H, T, 2, Kc, device=cuda)
    K.ctc_prefix_score(x, t_valid.to(cuda), utt.to(cuda), r_prev_d, last.to(cuda), out_len.to(cuda), cs.to(cuda), psi, r,
                       blank, eos)
    psi, r = psi.double().cpu().numpy(), r.double().cpu()
    for h in range(H):
        u = int(utt[h])
        Tb = int(t_valid[u])
        want_psi, want_r = BO.ctc_prefix_score(x64[u, :Tb].numpy(), r_prev_d[h, :Tb].double().cpu().numpy(),
                                               int(last[h]), int(out_len[h]), cs[h].numpy(), blank, eos,
                                               dtype=np.float64)
        bound = 1e-4 * np.maximum(1.0, np.abs(want_psi))
        assert (np.abs(psi[h] - want_psi) <= bound).all(), (h, int(out_len[h]), psi[h][:4], want_psi[:4])
        if h % 7 == 0:  # selected states
            got = r[h, :Tb].permute(2, 0, 1).numpy()
            assert (np.abs(got - want_r) <= 1e-4 * np.maximum(1.0, np.abs(want_r))).all(), h
            assert bool((r[h, Tb:] == BO.LOGZERO).all())


def test_ctc_prefix_limits_are_errors(cuda):
    from speecht5_b200 import kernels as K
    x = torch.zeros(1, 1501, 8, device=cuda)
    with pytest.raises(RuntimeError, match="st5_ctc_prefix_init"):
        K.ctc_prefix_init(x, torch.ones(1, dtype=torch.long, device=cuda), torch.empty(1, 1501, 2, device=cuda), 7)
    x = torch.zeros(1, 10, 300, device=cuda)
    z = torch.zeros(1, dtype=torch.long, device=cuda)
    with pytest.raises(RuntimeError, match="st5_ctc_prefix_score"):
        K.ctc_prefix_score(x, z + 10, z, torch.zeros(1, 10, 2, device=cuda), z, z, torch.zeros(1, 257, dtype=torch.long,
                           device=cuda), torch.empty(1, 257, device=cuda), torch.empty(1, 10, 2, 257, device=cuda), 0, 2)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_beam_gather_rows_equals_index_select(cuda, dtype):
    from speecht5_b200 import kernels as K
    H, L, W, n = 40, 7, 1536, 33
    src = [torch.randn(H, L * 9, W, device=cuda).to(dtype) for _ in range(6)]
    dst = [torch.full_like(s, 7.0) for s in src]
    parent = torch.randint(0, H, (30,), device=cuda)
    K.beam_gather_rows(src, [d[:30] for d in dst], parent, n)
    torch.cuda.synchronize()
    for s, d in zip(src, dst):
        assert torch.equal(d[:30, :n], s.index_select(0, parent)[:, :n])
        assert bool((d[:30, n:] == 7.0).all()) and bool((d[30:] == 7.0).all())


def _blob():
    return dict(np.load(GOLD))


def _inputs(blob, alone, dev):
    src, pm = torch.from_numpy(blob["in/source"]), torch.from_numpy(blob["in/padding_mask"])
    if not alone:
        return [(src.to(dev), pm.to(dev))]
    return [(src[i: i + 1, :n].to(dev), pm[i: i + 1, :n].to(dev)) for i, n in enumerate((~pm).sum(1).tolist())]


def _gen(model, c, use_cache):
    from speecht5_b200.generator import BeamSearchGenerator
    vocab = SimpleNamespace(pad=lambda: 1, eos=lambda: 2, unk=lambda: 3)
    return BeamSearchGenerator([model], vocab, beam_size=c["beam"], max_len_b=12, min_len=c.get("min_len", 1),
                               len_penalty=c.get("len_penalty", 1.0), ctc_weight=c["ctc_weight"], blank=BLANK,
                               mask_idx=MASK, use_cache=use_cache)


@pytest.mark.parametrize("use_cache", [False, True])
def test_beam_search_parity_mode_equals_the_reference_n_best_lists(cuda, use_cache):
    """Parity mode (fp32): every fixture case -- tokens bit-exact, scores and positional scores within 1e-4."""
    blob = _blob()
    model = _asr_model(cuda, torch.float32, blob).eval()
    for name, c in CASES.items():
        gen = _gen(model, c, use_cache)
        b = 0
        for src, pm in _inputs(blob, c["alone"], cuda):
            for hs in gen.generate([model], {"net_input": {"source": src, "padding_mask": pm}}):
                assert len(hs) == c["beam"]
                for j, h in enumerate(hs):
                    t = blob[f"{name}/tokens"][b, j]
                    n = int((t >= 0).sum())
                    assert h["tokens"].tolist() == t[:n].tolist(), (name, use_cache, b, j)
                    w = float(blob[f"{name}/scores"][b, j])
                    assert abs(float(h["score"]) - w) <= 1e-4 * max(1.0, abs(w)), (name, b, j)
                    wp = torch.from_numpy(blob[f"{name}/pos_scores"][b, j, :n])
                    assert (h["positional_scores"].cpu() - wp).abs().max() <= 1e-4 * max(1.0, float(wp.abs().max()))
                b += 1


def test_a_batch_equals_each_utterance_alone(cuda):
    """Equal-length utterances decoded together (joint CTC scoring, both cache paths) give what each gives alone."""
    blob = _blob()
    model = _asr_model(cuda, torch.float32, blob).eval()
    n = int((~torch.from_numpy(blob["in/padding_mask"])).sum(1).min())
    src = torch.from_numpy(blob["in/source"])[:, :n].to(cuda)
    pm = torch.zeros_like(src, dtype=torch.bool)
    c = dict(beam=4, ctc_weight=0.5)
    for use_cache in (False, True):
        gen = _gen(model, c, use_cache)
        together = gen.generate([model], {"net_input": {"source": src, "padding_mask": pm}})
        for i in range(src.size(0)):
            alone = gen.generate([model], {"net_input": {"source": src[i: i + 1], "padding_mask": pm[i: i + 1]}})[0]
            assert [h["tokens"].tolist() for h in together[i]] == [h["tokens"].tolist() for h in alone]
            assert np.allclose([float(h["score"]) for h in together[i]], [float(h["score"]) for h in alone], atol=1e-5)


def test_bf16_mode_returns_well_formed_n_best_lists(cuda):
    """Throughput mode: the score gaps of this tiny model are below bf16 resolution, so no token equality is asserted;
    the lists are complete, sorted, end in eos and carry finite scores."""
    blob = _blob()
    model = _asr_model(cuda, torch.bfloat16, blob).eval()
    for use_cache in (False, True):
        gen = _gen(model, CASES["b"], use_cache)
        for src, pm in _inputs(blob, False, cuda):
            for hs in gen.generate([model], {"net_input": {"source": src, "padding_mask": pm}}):
                assert len(hs) == 4
                scores = [float(h["score"]) for h in hs]
                assert scores == sorted(scores, reverse=True) and all(np.isfinite(scores))
                for h in hs:
                    assert h["tokens"][-1].item() == 2 and h["positional_scores"].shape == h["tokens"].shape
