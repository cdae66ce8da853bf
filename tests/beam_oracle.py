"""CPU restatement of joint CTC/attention beam search, written from the algorithm (Watanabe et al., "Hybrid
CTC/attention architecture for end-to-end speech recognition", Algorithm 2, extended to score many next labels at once)
and from the search loop of speecht5/sequence_generator.py:346-654, with the per-utterance semantics of
speecht5_b200/beam.py: every sentence is decoded on its own, against its own CTC posteriors.

The numbers follow the reference's conventions: the finite sentinel LOGZERO = -1e10, numpy's logaddexp, and (by
default) float32 arithmetic, so that even the scores of CTC-infeasible candidates come out as the reference's do. The
kernel checks use dtype=np.float64."""
import math

import numpy as np
import torch

LOGZERO = -1e10
CTC_SCORING_RATIO = 7.0


def ctc_initial_state(x, blank, dtype=np.float32):
    """x [T_b, V] log-probabilities of ONE utterance's valid frames -> r [T_b, 2]: r_n = LOGZERO, r_b[t] = the
    log-probability of blanks on frames 0..t (a running sum)."""
    x = np.asarray(x, dtype=dtype)
    T = x.shape[0]
    r = np.full((T, 2), LOGZERO, dtype=dtype)
    acc = dtype(0)
    for t in range(T):
        acc = x[0, blank] if t == 0 else dtype(acc + x[t, blank])
        r[t, 1] = acc
    return r


def ctc_prefix_score(x, r_prev, last, out_len, cs, blank, eos, dtype=np.float32):
    """Scores of appending each label of cs [K] to a prefix of out_len labels (leading eos excluded) whose last label is
    `last` and whose state is r_prev [T_b, 2]. Returns (psi [K], r [K, T_b, 2]).

    gamma_n(t) / gamma_b(t): probability of the extended prefix over frames 0..t ending in its new label / in blank.
    The new label may start at frame t only if the old prefix had ended by t - 1 (phi(t - 1)); a repeated label must be
    separated by a blank, so phi is then the old prefix's blank-ending part alone. psi sums, over the frame where the new
    label starts, the probability of every path that starts it there. An eos candidate scores the whole old prefix at
    the last frame; a blank candidate is never a label."""
    x = np.asarray(x, dtype=dtype)
    r_prev = np.asarray(r_prev, dtype=dtype)
    cs = np.asarray(cs, dtype=np.int64)
    T, Kc = x.shape[0], len(cs)
    lae = np.logaddexp
    gn = np.full((T, Kc), LOGZERO, dtype=dtype)
    gb = np.full((T, Kc), LOGZERO, dtype=dtype)
    xs = x[:, cs]
    whole = lae(r_prev[:, 0], r_prev[:, 1])
    phi = np.repeat(whole[:, None], Kc, axis=1)
    if out_len > 0:
        phi[:, cs == last] = r_prev[:, 1:2]
    if out_len == 0:
        start = 1
        psi = xs[0].copy() if T > 0 else np.full(Kc, LOGZERO, dtype=dtype)
        if T > 0:
            gn[0] = xs[0]
    else:
        start = out_len
        psi = np.full(Kc, LOGZERO, dtype=dtype)
    for t in range(start, T):
        gn[t] = lae(gn[t - 1], phi[t - 1]) + xs[t]
        gb[t] = lae(gn[t - 1], gb[t - 1]) + x[t, blank]
        psi = lae(psi, phi[t - 1] + xs[t])
    psi = np.array(psi, dtype=dtype)
    psi[cs == eos] = whole[T - 1] if T > 0 else LOGZERO
    psi[cs == blank] = LOGZERO
    return psi, np.stack([gn, gb], -1).transpose(1, 0, 2)


def beam_search_one(step_fn, beam, V, max_len, ctc_x=None, ctc_weight=0.0, min_len=1, normalize_scores=True,
                    len_penalty=1.0, unk_penalty=0.0, pad=1, eos=2, unk=3, blank=0, mask_idx=None, mask_idxs=(),
                    gaps=None):
    """One sentence. step_fn(prefixes [n, step + 1] LongTensor) -> decoder log-probabilities [n, V] float32 (torch).
    ctc_x: [T_b, V] CTC log-probabilities of the utterance's valid frames (numpy float32). Returns the n-best list
    [(tokens list, score float, positional scores list)] sorted by score. `gaps` (a list) receives, per step, the
    smallest difference between neighbouring candidate scores among the top 2 beam + 1 finite ones."""
    beam = min(beam, V - 1)
    masked = [blank] + ([mask_idx] if mask_idx is not None and mask_idx != unk else []) + list(mask_idxs)
    ctc_beam = min(V - len(mask_idxs), int(beam * CTC_SCORING_RATIO))
    hyps = [[eos] for _ in range(beam)]
    cum = [[] for _ in range(beam)]          # cumulative score after each token
    ignore = [False] * beam
    state = None
    if ctc_weight > 0:
        r0 = ctc_initial_state(ctc_x, blank)
        state = [(r0, np.float32(0.0)) for _ in range(beam)]
    finalized = []
    cand_size = 2 * beam
    for step in range(max_len + 1):
        lp = step_fn(torch.tensor(hyps, dtype=torch.long)).float().clone()
        new_states = {}
        if ctc_weight > 0:
            c_lp = lp.clone()
            c_lp[:, masked] = -math.inf
            ids = torch.topk(c_lp, ctc_beam, dim=-1).indices
            for b in range(beam):
                cs = ids[b].numpy()
                psi, r = ctc_prefix_score(ctc_x, state[b][0], hyps[b][-1], step, cs, blank, eos)
                d = torch.from_numpy(psi - state[b][1])
                lp[b, ids[b]] = (1 - ctc_weight) * lp[b, ids[b]] + ctc_weight * d
                for j, c in enumerate(cs.tolist()):
                    new_states[(b, c)] = (r[j], psi[j])
        if step < min_len:
            lp[:, eos] = -math.inf
        lp[lp != lp] = -math.inf
        lp[:, pad] = -math.inf
        lp[:, unk] -= unk_penalty
        lp[:, masked] = -math.inf
        if step >= max_len:
            lp[:, :eos] = -math.inf
            lp[:, eos + 1:] = -math.inf
        if step == 0:
            flat = lp[0]
        else:
            flat = (lp + torch.tensor([c[-1] for c in cum], dtype=torch.float32)[:, None]).view(-1)
        vals, idx = torch.topk(flat, k=min(cand_size, flat.numel() - 1))
        if gaps is not None:
            top = torch.topk(flat, k=min(cand_size + 1, flat.numel())).values
            top = top[torch.isfinite(top)]
            if top.numel() > 1:
                gaps.append(float((top[:-1] - top[1:]).min()))
        cands = [(float(v), int(i) % V, int(i) // V) for v, i in zip(vals, idx)]
        # finalisation: eos among the first `beam` candidate columns, columns of ignored slots excluded
        is_eos = [c[1] == eos and c[0] != -math.inf for c in cands]
        for j in range(beam):
            if ignore[j]:
                is_eos[j] = False
        for j in range(beam):
            if is_eos[j] and len(finalized) < beam:
                v, tok, b = cands[j]
                seq = hyps[b][1:] + [eos]
                cumv = cum[b] + [v]
                pos = [cumv[0]] + [np.float32(cumv[i]) - np.float32(cumv[i - 1]) for i in range(1, len(cumv))]
                score = np.float32(v)
                if normalize_scores:
                    score = np.float32(torch.tensor(v, dtype=torch.float32) / (step + 1) ** len_penalty)
                finalized.append((seq, float(score), [float(p) for p in pos]))
        if any(is_eos[:beam]) and (len(finalized) == beam or step == max_len):
            break
        assert step < max_len
        excluded = [is_eos[j] or (j < beam and ignore[j]) for j in range(len(cands))]
        order = sorted(range(len(cands)), key=lambda j: (excluded[j], j))[:beam]
        ignore = [excluded[j] for j in order]
        new_hyps, new_cum, new_state = [], [], []
        for j in order:
            v, tok, b = cands[j]
            new_hyps.append(hyps[b] + [tok])
            new_cum.append(cum[b] + [np.float32(v)])
            if ctc_weight > 0:
                if (b, tok) not in new_states:  # not a CTC candidate of its parent: score it alone
                    psi, r = ctc_prefix_score(ctc_x, state[b][0], hyps[b][-1], step, [tok], blank, eos)
                    new_states[(b, tok)] = (r[0], psi[0])
                new_state.append(new_states[(b, tok)])
        hyps, cum, state = new_hyps, new_cum, new_state
    finalized.sort(key=lambda h: -h[1])
    return finalized
