"""Beam search with joint CTC/attention scoring for speech-to-text decoding: the search of
speecht5/sequence_generator.py:207-655 (fairseq's BeamSearch candidate step, eos finalisation :690-816, removal of
finished sentences, the final sort) on device tensors, with the CTC prefix scorer of :273-284 / :370-418 on the
project's own kernels (st5_ctc_prefix_init / st5_ctc_prefix_score) instead of one numpy call per hypothesis per step.

Per step, on the device: the decoder (prefix recomputation, or the key/value cache reordered by st5_beam_gather_rows),
log_softmax, the CTC term for the top ctc_beam = min(V - len(mask_idxs), int(7 * beam)) tokens of the decoder's own
distribution (blank and mask symbols excluded, pad kept: lprobs <- (1 - w) lprobs + w (psi - psi_prev) for those tokens,
every other token keeps its attention score), the masking order of :437-454, and the candidate top-k. ONE small
device->host copy per step brings the 2 x beam candidates of every sentence (score, token, beam, position in the CTC
candidate list) to the host, where the finalisation bookkeeping runs on the same few numbers as in the reference.

Two reference behaviours need a rule here:
- Batch > 1. The reference scores every sentence against the FIRST utterance's CTC posteriors (ctc_lprobs[0], :280) and
  keys its states by the token prefix alone (:380-391), so states are shared across sentences: it is only right at
  batch 1. Here every hypothesis carries its own state and is scored against its own utterance's posteriors over that
  utterance's valid frames: decoding a batch gives what decoding each utterance alone gives.
- A token outside the CTC candidates reaches the beam (it kept its attention score and won). The reference has no
  state for that prefix and raises KeyError at the next step (:381). The scoring is the reference's; afterwards every
  selected non-candidate is scored by the same kernel with K = 1, so its state and psi_prev are defined. Results equal
  the reference's wherever the reference completes."""
import math

import torch
import torch.nn.functional as F

from . import kernels as K

CTC_SCORING_RATIO = 7.0    # sequence_generator.py:24


class BeamSearch:
    """fairseq search.BeamSearch.step: step 0 expands beam 0 only; later steps add each hypothesis's cumulative score,
    then the top min(2 beam, beam V - 1) of every sentence (the last term keeps pad out)."""

    def step(self, step, lprobs, scores):
        """lprobs [bsz, beam, V]; scores [bsz, beam] cumulative score of each hypothesis (ignored at step 0).
        Returns (cand_scores, cand_indices, cand_beams), each [bsz, k]."""
        bsz, beam, V = lprobs.shape
        if step == 0:
            lprobs = lprobs[:, ::beam, :].contiguous()
        else:
            lprobs = lprobs + scores.unsqueeze(-1)
        flat = lprobs.view(bsz, -1)
        vals, idx = torch.topk(flat, k=min(2 * beam, flat.size(1) - 1))
        return vals, idx.fmod(V), torch.div(idx, V, rounding_mode="floor")


class CTCPrefixScorer:
    """The CTC prefix state of every hypothesis, on the device: r_prev [H, T, 2] and psi_prev [H], the utterance each
    hypothesis decodes (utt [H]) and its last label. x [B, T, V] fp32 CTC log-probabilities, t_valid [B] valid frames."""

    def __init__(self, x, t_valid, blank, eos, beam):
        self.x, self.t_valid = x.contiguous(), t_valid.contiguous()
        self.blank, self.eos = blank, eos
        B, T, _ = x.shape
        r0 = torch.empty((B, T, 2), dtype=torch.float32, device=x.device)
        K.ctc_prefix_init(self.x, self.t_valid, r0, blank)
        self.utt = torch.arange(B, device=x.device).repeat_interleave(beam)
        self.r_prev = r0.repeat_interleave(beam, 0)
        self.psi_prev = torch.zeros(B * beam, dtype=torch.float32, device=x.device)
        self.last = None

    def _score(self, utt, r_prev, last, out_len, cs):
        H, Kc = cs.shape
        T = self.x.shape[1]
        psi = torch.empty((H, Kc), dtype=torch.float32, device=cs.device)
        r = torch.empty((H, T, 2, Kc), dtype=torch.float32, device=cs.device)
        K.ctc_prefix_score(self.x, self.t_valid, utt.contiguous(), r_prev.contiguous(), last.contiguous(),
                           torch.full((H,), int(out_len), dtype=torch.long, device=cs.device), cs.contiguous(), psi, r,
                           self.blank, self.eos)
        return psi, r

    def score(self, last, out_len, cs):
        """Scores of the candidates cs [H, K] of every hypothesis; remembers the candidate states for select()."""
        self.last, self.out_len = last, out_len
        self.psi, self.r = self._score(self.utt, self.r_prev, last, out_len, cs)
        return self.psi - self.psi_prev[:, None]

    def select(self, parent, kpos, tokens, fresh):
        """Hypothesis j continues parent[j] with tokens[j], which is candidate kpos[j] of its parent (-1: not a
        candidate; `fresh` lists those j on the host, scored here with K = 1). parent / kpos / tokens on the device."""
        old_r, old_utt = self.r_prev, self.utt
        k = kpos.clamp(min=0)
        self.r_prev = self.r[parent, :, :, k].contiguous()
        self.psi_prev = self.psi[parent, k].contiguous()
        if fresh:
            j = torch.tensor(fresh, dtype=torch.long, device=parent.device)
            p = parent.index_select(0, j)
            psi, r = self._score(old_utt.index_select(0, p), old_r.index_select(0, p), self.last.index_select(0, p),
                                 self.out_len, tokens.index_select(0, j)[:, None])
            self.r_prev.index_copy_(0, j, r[..., 0])
            self.psi_prev.index_copy_(0, j, psi[:, 0])
        self.utt = old_utt.index_select(0, parent)


def _mask_symbols(lprobs, blank, mask_idx, unk, mask_idxs):
    lprobs[:, blank] = -math.inf
    if mask_idx is not None and mask_idx != unk:
        lprobs[:, mask_idx] = -math.inf
    if mask_idxs is not None and mask_idxs.numel() > 0:
        lprobs[:, mask_idxs] = -math.inf


@torch.no_grad()
def beam_search(model, source, padding_mask=None, beam_size=5, ctc_weight=0.0, max_len_a=0.0, max_len_b=200,
                min_len=1, normalize_scores=True, len_penalty=1.0, unk_penalty=0.0, temperature=1.0, pad=1, eos=2,
                unk=3, blank=0, mask_idx=None, mask_idxs=None, use_cache=False, vocab_size=None, stats=None):
    """The n-best lists of every utterance: a list over sentences of `beam` dicts {"tokens", "score",
    "positional_scores", "alignment", "attention"} sorted by score (see the module docstring). use_cache=False
    recomputes the prefix every step (the reference's shape), True keeps the key/value cache. `stats` (a dict) receives
    per-step CUDA events around the CTC kernels when given (tools/bench_beam.py)."""
    dev = source.device
    bsz, src_len = source.size(0), source.size(1)
    V = vocab_size or model.text_decoder_postnet.output_projection.weight.shape[0]
    beam = min(beam_size, V - 1)
    max_len = min(int(max_len_a * src_len + max_len_b), model.args.max_text_positions - 1)
    assert min_len <= max_len, "min_len cannot be larger than max_len, please adjust these!"
    if mask_idxs is not None and not torch.is_tensor(mask_idxs):
        mask_idxs = torch.tensor(list(mask_idxs), dtype=torch.long)
    n_mask = 0 if mask_idxs is None else int(mask_idxs.numel())
    if mask_idxs is not None:
        mask_idxs = mask_idxs.to(dev)
    enc = model.forward_encoder(source, padding_mask=padding_mask)
    scorer = None
    if ctc_weight > 0:
        x = model.get_normalized_probs_for_ctc(enc, log_probs=True).transpose(0, 1).contiguous()  # [B, T, V]
        pm = enc["encoder_padding_mask"]
        T = x.shape[1]
        if len(pm) > 0 and pm[0] is not None:
            t_valid = (~pm[0].bool()).sum(1).to(torch.long)
        else:
            t_valid = torch.full((bsz,), T, dtype=torch.long, device=dev)
        scorer = CTCPrefixScorer(x, t_valid, blank, eos, beam)
        ctc_beam = min(V - n_mask, int(beam * CTC_SCORING_RATIO))
    rows = torch.arange(bsz, device=dev).repeat_interleave(beam)
    enc = model.encoder.reorder_encoder_out(enc, rows)  # once: a hypothesis never changes utterance
    cache = None
    if use_cache:
        from .incremental import DecoderCache, decoder_step
        cache = DecoderCache(model.decoder, enc, max_len + 1)
    search = BeamSearch()

    # host bookkeeping, as in the reference (:294-345)
    scores = torch.zeros(bsz * beam, max_len + 1, dtype=torch.float32)
    tokens = torch.full((bsz * beam, max_len + 2), pad, dtype=torch.long)
    tokens[:, 0] = eos
    cands_to_ignore = torch.zeros(bsz, beam, dtype=torch.bool)
    finalized = [[] for _ in range(bsz)]
    finished = [False] * bsz
    num_remaining = bsz
    cand_size = 2 * beam
    bbsz_offsets = (torch.arange(bsz) * beam).unsqueeze(1)
    cand_offsets = torch.arange(cand_size)
    cum_dev = torch.zeros(bsz * beam, dtype=torch.float32, device=dev)
    tokens_dev = tokens.to(dev)

    for step in range(max_len + 1):
        if cache is not None:
            dec_in, _, _ = model.text_decoder_prenet(tokens_dev[:, : step + 1])
            z, _ = decoder_step(model.decoder, dec_in[:, -1:], cache)
            logits = model.text_decoder_postnet(z)
        else:
            logits, _ = model.forward_decoder(tokens_dev[:, : step + 1], enc, incremental_state={})
        lprobs = F.log_softmax(logits[:, -1, :].float() / temperature, dim=-1)
        kpos_map = None
        if scorer is not None:  # (:370-418)
            ctc_lprobs = lprobs.clone()
            _mask_symbols(ctc_lprobs, blank, mask_idx, unk, mask_idxs)
            ids = torch.topk(ctc_lprobs, ctc_beam, dim=-1).indices
            if stats is not None:
                e0 = torch.cuda.Event(enable_timing=True)
                e0.record()
            dpsi = scorer.score(tokens_dev[:, step].contiguous(), step, ids)
            if stats is not None:
                e1 = torch.cuda.Event(enable_timing=True)
                e1.record()
                stats.setdefault("ctc_events", []).append((e0, e1))
            lprobs.scatter_(1, ids, (1 - ctc_weight) * lprobs.gather(1, ids) + ctc_weight * dpsi)
            kpos_map = torch.full_like(lprobs, -1, dtype=torch.long).scatter_(
                1, ids, torch.arange(ctc_beam, device=dev).expand_as(ids).contiguous())
        if step < min_len:  # (:437-454)
            lprobs[:, eos] = -math.inf
        lprobs[lprobs != lprobs] = -math.inf
        lprobs[:, pad] = -math.inf
        lprobs[:, unk] -= unk_penalty
        _mask_symbols(lprobs, blank, mask_idx, unk, mask_idxs)
        if step >= max_len:
            lprobs[:, :eos] = -math.inf
            lprobs[:, eos + 1:] = -math.inf

        cs_d, ci_d, cb_d = search.step(step, lprobs.view(bsz, -1, V), cum_dev.view(bsz, beam))
        kp_d = kpos_map[(cb_d + bbsz_offsets.to(dev)).view(-1), ci_d.view(-1)].view_as(ci_d) if kpos_map is not None \
            else torch.full_like(ci_d, -1)
        packed = torch.stack([cs_d.double(), ci_d.double(), cb_d.double(), kp_d.double()], -1).cpu()  # the one D2H copy
        cand_scores = packed[..., 0].float()
        cand_indices, cand_beams, cand_kpos = packed[..., 1].long(), packed[..., 2].long(), packed[..., 3].long()

        cand_bbsz_idx = cand_beams + bbsz_offsets
        eos_mask = cand_indices.eq(eos) & cand_scores.ne(-math.inf)
        eos_mask[:, :beam][cands_to_ignore] = False
        eos_bbsz_idx = torch.masked_select(cand_bbsz_idx[:, :beam], mask=eos_mask[:, :beam])
        finalized_sents = []
        if eos_bbsz_idx.numel() > 0:
            eos_scores = torch.masked_select(cand_scores[:, :beam], mask=eos_mask[:, :beam])
            finalized_sents = _finalize(step, eos_bbsz_idx, eos_scores, tokens, scores, finalized, finished, beam,
                                        max_len, eos, normalize_scores, len_penalty)
            num_remaining -= len(finalized_sents)
        if num_remaining == 0:
            break
        assert step < max_len, f"{step} < {max_len}"

        keep = None
        corr = None
        if finalized_sents:
            new_bsz = bsz - len(finalized_sents)
            batch_mask = torch.ones(bsz, dtype=torch.bool)
            batch_mask[finalized_sents] = False
            batch_idxs = torch.arange(bsz).masked_select(batch_mask)
            eos_mask = eos_mask[batch_idxs]
            cand_beams = cand_beams[batch_idxs]
            bbsz_offsets = bbsz_offsets[:new_bsz]
            cand_bbsz_idx = cand_beams + bbsz_offsets
            cand_scores = cand_scores[batch_idxs]
            cand_indices = cand_indices[batch_idxs]
            cand_kpos = cand_kpos[batch_idxs]
            cands_to_ignore = cands_to_ignore[batch_idxs]
            scores = scores.view(bsz, -1)[batch_idxs].view(new_bsz * beam, -1)
            tokens = tokens.view(bsz, -1)[batch_idxs].view(new_bsz * beam, -1)
            keep = (batch_idxs[:, None] * beam + torch.arange(beam)).view(-1)
            corr = batch_idxs - torch.arange(new_bsz)
            bsz = new_bsz

        eos_mask[:, :beam] = ~((~cands_to_ignore) & (~eos_mask[:, :beam]))
        active_mask = eos_mask.long() * cand_size + cand_offsets[: eos_mask.size(1)]
        new_cands_to_ignore, active_hypos = torch.topk(active_mask, k=beam, dim=1, largest=False)
        cands_to_ignore = new_cands_to_ignore.ge(cand_size)[:, :beam]
        assert (~cands_to_ignore).any(dim=1).all()
        active_bbsz_idx = torch.gather(cand_bbsz_idx, 1, active_hypos).view(-1)
        active_scores = torch.gather(cand_scores, 1, active_hypos)
        tokens[:, : step + 1] = torch.index_select(tokens[:, : step + 1], 0, active_bbsz_idx)
        new_tok = torch.gather(cand_indices, 1, active_hypos)
        tokens.view(bsz, beam, -1)[:, :, step + 1] = new_tok
        if step > 0:
            scores[:, :step] = torch.index_select(scores[:, :step], 0, active_bbsz_idx)
        scores.view(bsz, beam, -1)[:, :, step] = active_scores

        # the device side follows: parent rows in the numbering of this step's hypotheses (:349-361)
        parent = active_bbsz_idx.view(bsz, beam)
        if corr is not None:
            parent = parent + corr[:, None] * beam
        parent_dev = parent.view(-1).to(dev)
        if cache is not None:
            cache.gather_rows(parent_dev, keep=keep.to(dev) if keep is not None else None)
        elif keep is not None:
            enc = model.encoder.reorder_encoder_out(enc, keep.to(dev))
        if scorer is not None:
            sel_kpos = torch.gather(cand_kpos, 1, active_hypos).view(-1)
            fresh = torch.nonzero(sel_kpos < 0).view(-1).tolist()
            scorer.select(parent_dev, sel_kpos.to(dev), new_tok.view(-1).to(dev), fresh)
        cum_dev = active_scores.view(-1).to(dev)
        tokens_dev = tokens.to(dev)

    for sent in range(len(finalized)):  # sort by score, descending (:644-653)
        order = torch.sort(torch.tensor([float(h["score"]) for h in finalized[sent]]), descending=True)[1]
        finalized[sent] = [finalized[sent][i] for i in order]
        for h in finalized[sent]:
            for k in ("tokens", "score", "positional_scores"):
                h[k] = h[k].to(dev)
    return finalized


def _finalize(step, bbsz_idx, eos_scores, tokens, scores, finalized, finished, beam, max_len, eos, normalize_scores,
              len_penalty):
    """finalize_hypos + is_finished (:690-816) on the host copies; returns the newly finished sentences' indices in
    the current (reduced) batch."""
    tokens_clone = tokens.index_select(0, bbsz_idx)[:, 1: step + 2]
    tokens_clone[:, step] = eos
    pos_scores = scores.index_select(0, bbsz_idx)[:, : step + 1]
    pos_scores[:, step] = eos_scores
    pos_scores[:, 1:] = pos_scores[:, 1:] - pos_scores[:, :-1]
    if normalize_scores:
        eos_scores = eos_scores / (step + 1) ** len_penalty
    cum_unfin = []
    prev = 0
    for f in finished:
        if f:
            prev += 1
        else:
            cum_unfin.append(prev)
    cum_fin = torch.tensor(cum_unfin, dtype=torch.long)
    unfin_idx = torch.div(bbsz_idx, beam, rounding_mode="floor")
    sent = unfin_idx + torch.index_select(cum_fin, 0, unfin_idx)
    seen = torch.unique((sent << 32) + unfin_idx).tolist()
    sent_list = sent.tolist()
    for i in range(bbsz_idx.size(0)):
        if len(finalized[sent_list[i]]) < beam:
            finalized[sent_list[i]].append({"tokens": tokens_clone[i], "score": eos_scores[i], "attention": None,
                                            "alignment": torch.empty(0), "positional_scores": pos_scores[i]})
    newly = []
    for s in seen:
        us = s >> 32
        ui = s - (us << 32)
        if not finished[us] and (len(finalized[us]) == beam or step == max_len):
            finished[us] = True
            newly.append(ui)
    return newly
