"""The generator objects fairseq's `generate.py` drives (`task.build_generator(models, args)` ->
`task.inference_step(generator, models, sample)` -> `generator.generate(models, sample)`), with the SequenceGenerator
call / return shape (speecht5/sequence_generator.py:191-205, :596-655: a list over sentences of a list over beams of
{"tokens", "score", "attention", "alignment", "positional_scores"}, score = sum of the token log-probabilities divided by
length ** len_penalty when normalize_scores is on).

- GreedyGenerator: beam size 1 without CTC scoring (`T5TransformerModel.generate_text_greedy`; the task's default).
- BeamSearchGenerator: beam search with optional joint CTC/attention scoring (`T5TransformerModel.generate_text_beam`,
  speecht5_b200/beam.py); `task.build_generator(models, args, seq_gen_cls=BeamSearchGenerator)` builds it.
LM shallow fusion, prefix tokens, constraints and n-gram blocking are not built and raise."""
import torch


class GreedyGenerator:
    def __init__(self, models, tgt_dict, beam_size=1, max_len_a=0, max_len_b=200, min_len=1, normalize_scores=True,
                 len_penalty=1.0, unk_penalty=0.0, temperature=1.0, ctc_weight=0.0, lm_model=None, use_cache=True,
                 blank=None, mask_idx=None, **unused):
        if beam_size != 1:
            raise NotImplementedError("beam search > 1 is not built in the B200 path (SURVEY section 2): use --beam 1")
        if ctc_weight and ctc_weight > 0 or lm_model is not None:
            raise NotImplementedError("CTC rescoring / LM fusion are not built in the B200 path")
        self.model = models[0] if isinstance(models, (list, tuple)) else models
        self.tgt_dict = tgt_dict
        self.pad, self.eos, self.unk = tgt_dict.pad(), tgt_dict.eos(), tgt_dict.unk()
        self.max_len_a, self.max_len_b, self.min_len = max_len_a, max_len_b, min_len
        self.normalize_scores, self.len_penalty = normalize_scores, len_penalty
        self.unk_penalty, self.temperature, self.use_cache = unk_penalty, temperature, use_cache
        index = getattr(tgt_dict, "index", None)
        self.blank = blank if blank is not None else (index("<ctc_blank>") if index else 0)
        self.mask_idx = mask_idx if mask_idx is not None else (index("<mask>") if index else None)

    @torch.no_grad()
    def generate(self, models, sample, prefix_tokens=None, constraints=None, bos_token=None):
        if prefix_tokens is not None or constraints is not None:
            raise NotImplementedError("prefix tokens / constraints are not built for the greedy path")
        ni = sample["net_input"]
        hyp, scores = self.model.generate_text_greedy(
            ni["source"], ni.get("padding_mask"), max_len_a=self.max_len_a, max_len_b=self.max_len_b, min_len=self.min_len,
            unk_penalty=self.unk_penalty, temperature=self.temperature, pad=self.pad, eos=self.eos, unk=self.unk,
            blank=self.blank, mask_idx=self.mask_idx, use_cache=self.use_cache, return_scores=True)
        out = []
        for tok, pos in zip(hyp, scores):
            total = pos.sum()
            if self.normalize_scores:
                total = total / (len(tok) ** self.len_penalty)
            out.append([{"tokens": tok, "score": total, "attention": None, "alignment": torch.empty(0),
                         "positional_scores": pos}])
        return out


class BeamSearchGenerator:
    """The reference SequenceGenerator's beam search (sequence_generator.py:207-655) with its CTC prefix scoring
    (:273-284, :370-418, weight `ctc_weight`), on the project's kernels. Same constructor keywords and generate() call as
    the reference; `beam_size` hypotheses per sentence, sorted by score, "attention" None as in GreedyGenerator.
    use_cache: False recomputes the prefix every step, True keeps the key/value cache."""

    def __init__(self, models, tgt_dict, beam_size=1, max_len_a=0, max_len_b=200, min_len=1, normalize_scores=True,
                 len_penalty=1.0, unk_penalty=0.0, temperature=1.0, ctc_weight=0.0, lm_model=None, use_cache=True,
                 no_repeat_ngram_size=0, blank=None, mask_idx=None, mask_idxs=None, **unused):
        if lm_model is not None:
            raise NotImplementedError("LM shallow fusion is not built in the B200 path")
        if no_repeat_ngram_size and no_repeat_ngram_size > 0:
            raise NotImplementedError("n-gram blocking (--no-repeat-ngram-size) is not built in the B200 path")
        assert temperature > 0, "--temperature must be greater than 0"
        self.model = models[0] if isinstance(models, (list, tuple)) else models
        self.tgt_dict = tgt_dict
        self.pad, self.eos, self.unk = tgt_dict.pad(), tgt_dict.eos(), tgt_dict.unk()
        self.beam_size, self.ctc_weight = beam_size, float(ctc_weight or 0.0)
        self.max_len_a, self.max_len_b, self.min_len = max_len_a, max_len_b, min_len
        self.normalize_scores, self.len_penalty = normalize_scores, len_penalty
        self.unk_penalty, self.temperature, self.use_cache = unk_penalty, temperature, use_cache
        index = getattr(tgt_dict, "index", None)
        self.blank = blank if blank is not None else (index("<ctc_blank>") if index else 0)
        self.mask_idx = mask_idx if mask_idx is not None else (index("<mask>") if index else None)
        if mask_idxs is None:  # (:84-90) <mask>0, <mask>1, ... while the dictionary knows them
            mask_idxs = []
            if index is not None:
                while index("<mask>" + str(len(mask_idxs))) != self.unk:
                    mask_idxs.append(index("<mask>" + str(len(mask_idxs))))
        self.mask_idxs = list(mask_idxs)

    @torch.no_grad()
    def generate(self, models, sample, prefix_tokens=None, constraints=None, bos_token=None):
        if prefix_tokens is not None or constraints is not None:
            raise NotImplementedError("prefix tokens / constraints are not built for the beam search")
        ni = sample["net_input"]
        return self.model.generate_text_beam(
            ni["source"], ni.get("padding_mask"), beam_size=self.beam_size, ctc_weight=self.ctc_weight,
            max_len_a=self.max_len_a, max_len_b=self.max_len_b, min_len=self.min_len,
            normalize_scores=self.normalize_scores, len_penalty=self.len_penalty, unk_penalty=self.unk_penalty,
            temperature=self.temperature, pad=self.pad, eos=self.eos, unk=self.unk, blank=self.blank,
            mask_idx=self.mask_idx, mask_idxs=self.mask_idxs, use_cache=self.use_cache)
