"""Incremental decoding with a key/value cache (SURVEY section 8a row 21 / 8f-2; the reference keeps fairseq
incremental state: speecht5/models/modules/multihead_attention.py:255-330, transformer_layer.py:262-404,
decoder.py:171-269). Opt-in: `use_cache=True` on generate_speech / generate_text_greedy runs the step eagerly,
`use_cache="graph"` on generate_speech replays ONE captured CUDA graph per decoder step (SynthesisGraph below). Checked
on the CPU against the prefix-recomputing path through the kernel emulation (tests/test_frontend_cpu.py) and on the
device (tests/test_frontend_gpu.py); nothing on the training path imports this module.

Per utterance batch the cross-attention keys / values of every decoder layer are projected ONCE; every step projects
q | k | v of the single new row, appends k | v to the layer's [B, T_max, 2C] cache and attends over the cache with a
one-row query -- O(L) work per step instead of the O(L^2) prefix recomputation. All contractions run on the existing
GEMM, the one-row attention on the exact row kernels (st5_attn_fwd), which take strided key / value views."""
import torch

from . import ops
from .ops import RT


def _act_dtype(x):
    return x if x.dtype == RT.dtype else x.to(RT.dtype)


def _attend(*a, **kw):
    """One-row queries: the row kernels (the fused tcgen05 path works on 128-query tiles)."""
    prev = RT.attn_tensor_core
    RT.attn_tensor_core = False
    try:
        return ops.attention(*a, **kw)
    finally:
        RT.attn_tensor_core = prev


class DecoderCache:
    def __init__(self, decoder, encoder_out, max_len):
        enc = encoder_out.get("_encoder_out_btc")
        if enc is None:
            enc = encoder_out["encoder_out"][0].transpose(0, 1).contiguous()
        enc = _act_dtype(enc)
        pm = encoder_out["encoder_padding_mask"]
        self.enc_pad = pm[0] if len(pm) > 0 else None
        B, _, C = enc.shape
        self.t = 0
        self.max_len = max_len
        self.cross, self.self_kv = [], []
        for layer in decoder.layers:
            ca = layer.encoder_attn
            self.cross.append(ops.linear(enc, (ca.k_proj.weight, ca.v_proj.weight), (ca.k_proj.bias, ca.v_proj.bias)))
            self.self_kv.append(torch.zeros((B, max_len, 2 * C), dtype=RT.dtype, device=enc.device))

    def reorder(self, new_order):
        """decoder.reorder_incremental_state_scripting (beam reordering): select utterances along the batch axis."""
        self.cross = [c.index_select(0, new_order) for c in self.cross]
        self.self_kv = [c.index_select(0, new_order) for c in self.self_kv]
        if self.enc_pad is not None:
            self.enc_pad = self.enc_pad.index_select(0, new_order)

    def gather_rows(self, parent, keep=None):
        """Beam reorder of the self-attention keys / values: hypothesis h continues parent[h] (int64 [H'] on the device).
        One st5_beam_gather_rows launch copies the rows written so far (the first `t`) of every layer into a second
        buffer set, which then becomes the cache (ping-pong: the previous one is reused by the next reorder). `keep`
        (rows of the hypotheses still decoding, when sentences finished) compacts the cross-attention keys / values and
        the padding mask; otherwise they stay as they are -- a hypothesis never changes utterance."""
        from . import kernels as K
        spare = getattr(self, "_spare", None)
        if spare is None or spare[0].shape[0] < parent.numel():
            spare = [torch.empty_like(c) for c in self.self_kv]
        dst = [s[: parent.numel()] for s in spare]
        K.beam_gather_rows(self.self_kv, dst, parent, self.t)
        self._spare = [c if c._base is None else c._base for c in self.self_kv]
        self.self_kv = dst
        if keep is not None:
            self.cross = [c.index_select(0, keep) for c in self.cross]
            if self.enc_pad is not None:
                self.enc_pad = self.enc_pad.index_select(0, keep)


@torch.no_grad()
def decoder_step(decoder, x_new, cache, need_head_weights=False, t_dev=None, span=None, self_pad=None):
    """x_new [B, 1, C] = decoder-prenet output of the newest position. Returns (x [B, 1, C], [attn [B, H, 1, S]] per
    layer or None). Evaluation semantics (no dropout, no LayerDrop) -- generation only.

    Device-side step index (the form a captured graph replays): `t_dev` int64 [1] holds the position, the new key / value
    row is written with index_copy_, and self-attention runs over the first `span` cache rows with `self_pad` (uint8
    [B, span], 1 = position > t) masking what has not been written yet -- no host scalar depends on the step."""
    assert not decoder.training
    x = _act_dtype(x_new).contiguous()
    t = cache.t
    assert t_dev is not None or t < cache.max_len
    attns = []
    for li, layer in enumerate(decoder.layers):
        sa, ca = layer.self_attn, layer.encoder_attn
        C = sa.embed_dim
        residual = x
        h = ops.residual_layer_norm(x, None, layer.self_attn_layer_norm) if layer.normalize_before else x
        qkv = ops.linear(h, (sa.q_proj.weight, sa.k_proj.weight, sa.v_proj.weight),
                         (sa.q_proj.bias, sa.k_proj.bias, sa.v_proj.bias))  # [B, 1, 3C]
        if t_dev is None:
            cache.self_kv[li][:, t] = qkv[:, 0, C:]
            a, _ = _attend(qkv, cache.self_kv[li][:, : t + 1], H=sa.num_heads, d=C, q_col=0, k_col=0, v_col=1,
                           scale=sa.scaling)
        else:
            cache.self_kv[li].index_copy_(1, t_dev, qkv[:, :, C:])
            a, _ = _attend(qkv, cache.self_kv[li][:, :span], H=sa.num_heads, d=C, q_col=0, k_col=0, v_col=1,
                           scale=sa.scaling, key_pad=self_pad)
        if layer.normalize_before:
            x = ops.linear(a, sa.out_proj.weight, sa.out_proj.bias, residual=residual)
        else:
            x = ops.residual_layer_norm(ops.linear(a, sa.out_proj.weight, sa.out_proj.bias), residual,
                                        layer.self_attn_layer_norm)
        residual = x
        h = ops.residual_layer_norm(x, None, layer.encoder_attn_layer_norm) if layer.normalize_before else x
        q = ops.linear(h, ca.q_proj.weight, ca.q_proj.bias)
        a, probs = _attend(q, cache.cross[li], H=ca.num_heads, d=C, q_col=0, k_col=0, v_col=1, scale=ca.scaling,
                           key_pad=cache.enc_pad, return_probs=need_head_weights)
        if need_head_weights:
            attns.append(probs.float())
        if layer.normalize_before:
            x = ops.linear(a, ca.out_proj.weight, ca.out_proj.bias, residual=residual)
            x = ops.ffn(ops.residual_layer_norm(x, None, layer.final_layer_norm), layer.fc1, layer.fc2,
                        layer.activation_fn, residual=x)
        else:
            x = ops.residual_layer_norm(ops.linear(a, ca.out_proj.weight, ca.out_proj.bias), residual,
                                        layer.encoder_attn_layer_norm)
            x = ops.residual_layer_norm(ops.ffn(x, layer.fc1, layer.fc2, layer.activation_fn), x,
                                        layer.final_layer_norm)
    if decoder.layer_norm is not None:
        x = ops.residual_layer_norm(x, None, decoder.layer_norm)
    if t_dev is None:
        cache.t = t + 1
    return x, (attns if need_head_weights else None)


class _StaticCache:
    """DecoderCache with caller-owned, fixed-size buffers (a captured graph bakes their addresses)."""

    def __init__(self, cross, self_kv, enc_pad, max_len):
        self.cross, self.self_kv, self.enc_pad, self.max_len, self.t = cross, self_kv, enc_pad, max_len, 0


class SynthesisGraph:
    """Greedy speech synthesis (models/speecht5.py:1188-1249) with every decoder step = ONE CUDA-graph replay: prenet on
    the newest frame (always-on dropout drawn from the device-resident seed, advanced inside the graph), positional row
    gathered by the device step counter, the key/value-cached decoder, feat_out | prob_out, and the step's outputs
    written into preallocated result buffers at the step index.

    The object is utterance-independent and is kept on the model (`synthesis_graph`): every buffer a graph reads has a
    fixed size -- the cross-attention keys / values of an utterance are copied into [1, S_bucket, 2C] buffers with the
    tail masked, the frame budget is a bucket too -- so the graphs captured for one utterance serve every later one of
    the same buckets (serving: no capture on the request path after the first). Self-attention spans are bucketed (128,
    256, ...): one graph per span, so a step attends over at most 2x the keys it needs. The host replays `chunk` steps,
    then reads their stop flags in one copy (the reference's `int(sum(probs[-1] >= threshold)) > 0`, :1235); steps
    replayed past the stopping one are discarded."""

    CHUNK = 8

    def __init__(self, model, S_bucket, maxlen_bucket, device, capture=True):
        self.m = model
        self.capture = capture  # False: the same step body runs eagerly (CPU checks of the device-counter form)
        dec, post = model.decoder, model.speech_decoder_postnet
        dev = torch.device(device)
        self.dev, self.r, self.odim = dev, model.reduction_factor, post.odim
        self.S, self.maxlen = int(S_bucket), int(maxlen_bucket)
        rows = self.maxlen + self.CHUNK
        L, H = len(dec.layers), dec.layers[0].encoder_attn.num_heads
        C = dec.layers[0].self_attn.embed_dim
        self.cache = _StaticCache([torch.zeros((1, self.S, 2 * C), dtype=RT.dtype, device=dev) for _ in dec.layers],
                                  [torch.zeros((1, rows, 2 * C), dtype=RT.dtype, device=dev) for _ in dec.layers],
                                  torch.zeros((1, self.S), dtype=torch.uint8, device=dev), rows)
        self.t = torch.zeros(1, dtype=torch.int64, device=dev)
        self.ys_last = torch.zeros(1, 1, self.odim, dtype=torch.float32, device=dev)
        self.outs = torch.zeros(rows, self.r, self.odim, dtype=torch.float32, device=dev)
        self.probs = torch.zeros(rows, self.r, dtype=torch.float32, device=dev)
        self.attn = torch.zeros(rows, L, H, self.S, dtype=torch.float32, device=dev)
        self.stop = torch.zeros(rows, dtype=torch.int32, device=dev)
        self.threshold = torch.full((1,), 0.5, dtype=torch.float32, device=dev)
        self.pos = torch.arange(rows, device=dev)
        pre = model.speech_decoder_prenet
        self.pe = pre.decoder_prenet[1].table(rows, dev)
        self.spk_bias = torch.zeros((1, pre.embed_dim), dtype=torch.float32, device=dev)
        self.with_spk = False
        self.graphs = {}
        self.stream = torch.cuda.Stream(device=dev) if capture else None
        self.dtype = RT.dtype
        # the graphs bake the address of the dropout seed they dereference and advance: it must be THIS object's tensor,
        # installed as the runtime's device seed for the duration of a synthesis (generate_speech restores the caller's)
        self.seed_t = torch.zeros(1, dtype=torch.int64, device=dev)

    @torch.no_grad()
    def begin(self, encoder_out, spkembs, threshold):
        """Load one utterance: project its cross-attention keys / values into the static buffers, reset the counters."""
        enc = encoder_out.get("_encoder_out_btc")
        if enc is None:
            enc = encoder_out["encoder_out"][0].transpose(0, 1).contiguous()
        enc = _act_dtype(enc)
        S = enc.shape[1]
        assert enc.shape[0] == 1 and S <= self.S and RT.dtype == self.dtype
        pm = encoder_out["encoder_padding_mask"]
        self.cache.enc_pad.fill_(1)
        self.cache.enc_pad[:, :S] = pm[0].to(torch.uint8) if len(pm) > 0 and pm[0] is not None else 0
        for li, layer in enumerate(self.m.decoder.layers):
            ca = layer.encoder_attn
            self.cache.cross[li][:, :S] = ops.linear(enc, (ca.k_proj.weight, ca.v_proj.weight),
                                                     (ca.k_proj.bias, ca.v_proj.bias))
        pre = self.m.speech_decoder_prenet
        with_spk = spkembs is not None
        if self.graphs and with_spk != self.with_spk:
            self.graphs = {}  # (the merge layer is part of the captured body)
        self.with_spk = with_spk
        if with_spk:  # (speech_decoder_prenet.py:76-89) the speaker half of the merge layer: once per utterance
            W, d = pre.spkembs_layer[0].weight, pre.embed_dim
            spk = torch.nn.functional.normalize(spkembs.float()).to(RT.dtype)
            self.spk_bias.copy_(ops.linear(spk, W[:, d:], (), out_dtype=torch.float32, key=("spk_w", id(W)), need_dx=False))
        self.threshold.fill_(float(threshold))
        self.t.zero_()
        self.ys_last.zero_()
        if self.capture:
            self.seed_t.fill_(RT._seed + (RT._draws << 20))  # a fresh stream of prenet masks per utterance
            RT._draws += 1
            RT._seed_t = self.seed_t
        return S

    def _body(self, span):
        m, pre, post = self.m, self.m.speech_decoder_prenet, self.m.speech_decoder_postnet
        taco, lin, pos = pre.decoder_prenet[0][0], pre.decoder_prenet[0][1], pre.decoder_prenet[1]
        x = self.ys_last.to(RT.dtype)
        for layer in taco.prenet:  # dropout in eval too (espnet Prenet semantics)
            x = ops.linear(x, layer[0].weight, layer[0].bias, act="relu", drop_p=taco.dropout_rate)
        x = ops.linear(x, lin.weight, lin.bias)
        x = ops.scaled_posenc(self.pe.index_select(0, self.t), pos.alpha, 0.0, x=x)
        if self.with_spk:
            W, b, d = pre.spkembs_layer[0].weight, pre.spkembs_layer[0].bias, pre.embed_dim
            x = ops.linear(x, W[:, :d], b, act="relu", bias2=self.spk_bias, bias2_rows=1, key=("spk_h", id(W)))
        self_pad = (self.pos[:span] > self.t).to(torch.uint8)[None].contiguous()
        z, layer_attn = decoder_step(m.decoder, x, self.cache, need_head_weights=True, t_dev=self.t, span=span,
                                     self_pad=self_pad)
        before, logits = post.project(z.contiguous())  # [1, r, odim], [1, r]
        p = torch.sigmoid(logits)
        self.outs.index_copy_(0, self.t, before)
        self.probs.index_copy_(0, self.t, p)
        self.attn.index_copy_(0, self.t, torch.stack([a[0, :, 0, :] for a in layer_attn], 0)[None])
        self.ys_last.copy_(before[:, -1:, :])
        self.stop.index_copy_(0, self.t, (p >= self.threshold).any().to(torch.int32).reshape(1))
        self.t += 1
        RT.advance_seed()

    def _span(self, t):
        span = 128
        while span < t + 1:
            span *= 2
        return min(span, self.cache.max_len)

    def _snapshot(self):
        """State the step body overwrites that a replay of the same step does not rewrite first (capture warm-up)."""
        keep = self.ys_last.clone()

        def undo():
            self.seed_t -= 1  # (the pass drew from the seed the replay of this step must see)
            self.ys_last.copy_(keep)
        return undo

    @torch.no_grad()
    def run(self, t0, n):
        """Decoder steps t0 .. t0+n-1 (the device counter holds t0). Returns their stop flags (one device->host copy)."""
        for t in range(t0, t0 + n):
            span = self._span(t)
            if not self.capture:
                self._body(span)
                continue
            g = self.graphs.get(span)
            if g is None:
                # one eager pass builds every weight shadow and scratch outside the capture, then its effects are
                # undone: the cache row / result rows it wrote are rewritten by the replay of the same step
                self.stream.wait_stream(torch.cuda.current_stream(self.dev))
                with torch.cuda.stream(self.stream):
                    undo = self._snapshot()
                    self._body(span)
                    self.t -= 1
                    undo()
                    self.stream.synchronize()
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=self.stream):
                        self._body(span)
                torch.cuda.current_stream(self.dev).wait_stream(self.stream)
                self.graphs[span] = g
            g.replay()
        return self.stop[t0:t0 + n].tolist()

    @torch.no_grad()
    def synthesize(self, encoder_out, spkembs, threshold, minlen, maxlen):
        """The reference's loop (:1222-1249): returns (before frames [1, L, odim], stop probabilities [L], attention
        [layers, H, L/r, S])."""
        assert maxlen <= self.maxlen
        minlen = min(minlen, max(maxlen, 1))  # (the reference's loop has no exit past maxlen frames otherwise)
        S = self.begin(encoder_out, spkembs, threshold)
        idx = 0
        while True:
            n = max(1, min(self.CHUNK, max(maxlen, 1) - idx))
            flags = self.run(idx, n)
            done = None
            for k, f in enumerate(flags):
                i = idx + k + 1  # the reference's idx after this step
                if (f or i >= maxlen) and i >= minlen:
                    done = i
                    break
            if done is not None:
                idx = done
                break
            idx += n
        return (self.outs[:idx].reshape(1, idx * self.r, self.odim).clone(), self.probs[:idx].reshape(-1).clone(),
                self.attn[:idx, :, :, :S].permute(1, 2, 0, 3).contiguous())


def synthesis_graph(model, S, maxlen, device, capture=True):
    """The model's SynthesisGraph for text length S and a frame budget of maxlen decoder steps (buckets: S to multiples of
    64, maxlen to powers of two >= 256); rebuilt when the numeric mode or the weights' owner changed."""
    S_b = max(64, (S + 63) // 64 * 64)
    M_b = 256
    while M_b < maxlen:
        M_b *= 2
    store = model.__dict__.setdefault("_synthesis_graphs", {})
    key = (S_b, M_b, RT.dtype, str(device), bool(capture), RT.param_epoch)
    sg = store.get(key)
    if sg is None:
        for k in [k for k in store if k[:5] == key[:5]]:  # same buckets, stale weights
            del store[k]
        sg = store[key] = SynthesisGraph(model, S_b, M_b, device, capture=capture)
    return sg


class GreedyGraph:
    """Beam-1 text decoding (speecht5/sequence_generator.py:207-655 with ctc_weight 0 and no LM, as
    T5TransformerModel.generate_text_greedy states it) with every step = ONE CUDA-graph replay: embedding + position row
    of the newest token (gathered by the device step counter), the key/value-cached decoder, the vocabulary projection,
    log-softmax, the reference's score masking (:430-446) as one additive mask plus two step-dependent terms, arg-max,
    and the bookkeeping (token written at t+1, finished flags, lengths) -- all on the device. Utterance-independent like
    SynthesisGraph: encoder length and step budget are buckets, cross keys / values are copied into fixed buffers."""

    CHUNK = 8

    def __init__(self, model, B, S_bucket, maxlen_bucket, device, capture=True):
        self.m, self.capture = model, capture
        dec = model.decoder
        dev = torch.device(device)
        self.dev, self.B, self.S, self.maxlen = dev, int(B), int(S_bucket), int(maxlen_bucket)
        rows = self.maxlen + 1 + self.CHUNK
        C = dec.layers[0].self_attn.embed_dim
        self.cache = _StaticCache([torch.zeros((B, self.S, 2 * C), dtype=RT.dtype, device=dev) for _ in dec.layers],
                                  [torch.zeros((B, rows, 2 * C), dtype=RT.dtype, device=dev) for _ in dec.layers],
                                  torch.zeros((B, self.S), dtype=torch.uint8, device=dev), rows)
        self.t = torch.zeros(1, dtype=torch.int64, device=dev)
        self.tokens = torch.zeros((B, rows + 1), dtype=torch.long, device=dev)
        self.done = torch.zeros(B, dtype=torch.bool, device=dev)
        self.lengths = torch.zeros(B, dtype=torch.long, device=dev)
        self.stop = torch.zeros(rows, dtype=torch.int32, device=dev)
        self.pos_scores = torch.zeros((B, rows), dtype=torch.float32, device=dev)  # log-probability of the token emitted at t
        self.pos = torch.arange(rows, device=dev)
        pre = model.text_decoder_prenet
        self.pe = pre._table(rows, dev)
        V = model.text_decoder_postnet.output_projection.weight.shape[0]
        self.base_mask = torch.zeros(V, dtype=torch.float32, device=dev)   # pad / blank / mask symbol never, unk penalty
        self.only_eos = torch.zeros(V, dtype=torch.float32, device=dev)    # added once the step budget is reached
        self.eos_early = torch.zeros(V, dtype=torch.float32, device=dev)   # added while step < min_len
        self.min_len = torch.zeros(1, dtype=torch.int64, device=dev)
        self.max_len = torch.zeros(1, dtype=torch.int64, device=dev)
        self.inv_temp = torch.ones(1, dtype=torch.float32, device=dev)
        self.eos = 2
        self.graphs = {}
        self.stream = torch.cuda.Stream(device=dev) if capture else None
        self.dtype = RT.dtype

    @torch.no_grad()
    def begin(self, encoder_out, max_len, min_len, unk_penalty, temperature, pad, eos, unk, blank, mask_idx):
        import math
        enc = encoder_out.get("_encoder_out_btc")
        if enc is None:
            enc = encoder_out["encoder_out"][0].transpose(0, 1).contiguous()
        enc = _act_dtype(enc)
        B, S = enc.shape[0], enc.shape[1]
        assert B == self.B and S <= self.S and max_len <= self.maxlen and RT.dtype == self.dtype
        pm = encoder_out["encoder_padding_mask"]
        self.cache.enc_pad.fill_(1)
        self.cache.enc_pad[:, :S] = pm[0].to(torch.uint8) if len(pm) > 0 and pm[0] is not None else 0
        for li, layer in enumerate(self.m.decoder.layers):
            ca = layer.encoder_attn
            self.cache.cross[li][:, :S] = ops.linear(enc, (ca.k_proj.weight, ca.v_proj.weight),
                                                     (ca.k_proj.bias, ca.v_proj.bias))
        self.base_mask.zero_()
        self.base_mask[pad] = -math.inf
        self.base_mask[unk] -= unk_penalty
        self.base_mask[blank] = -math.inf
        if mask_idx is not None and mask_idx != unk:
            self.base_mask[mask_idx] = -math.inf
        self.only_eos.fill_(-math.inf)
        self.only_eos[eos] = 0.0
        self.eos_early.zero_()
        self.eos_early[eos] = -math.inf
        self.min_len.fill_(int(min_len))
        self.max_len.fill_(int(max_len))
        self.inv_temp.fill_(1.0 / float(temperature))
        if self.graphs and eos != self.eos:
            self.graphs = {}
        self.eos = int(eos)
        self.tokens.fill_(pad)
        self.tokens[:, 0] = eos
        self.done.zero_()
        self.lengths.zero_()
        self.t.zero_()

    def _body(self, span):
        m, pre = self.m, self.m.text_decoder_prenet
        tok = self.tokens.index_select(1, self.t).contiguous()  # [B, 1]
        x = ops.scaled_posenc(self.pe.index_select(0, self.t), pre._unit, 0.0, tokens=tok, emb=pre.embed_tokens.weight,
                              padding_idx=pre.padding_idx)
        self_pad = (self.pos[:span] > self.t).to(torch.uint8)[None].expand(self.B, span).contiguous()
        z, _ = decoder_step(m.decoder, x, self.cache, t_dev=self.t, span=span, self_pad=self_pad)
        logits = m.text_decoder_postnet(z)
        lp = torch.log_softmax(logits[:, -1, :].float() * self.inv_temp, dim=-1)
        lp = torch.where(lp != lp, torch.full_like(lp, float("-inf")), lp)
        zero = torch.zeros_like(self.base_mask)
        lp = lp + self.base_mask + torch.where(self.t < self.min_len, self.eos_early, zero) \
            + torch.where(self.t >= self.max_len, self.only_eos, zero)
        nxt = lp.argmax(dim=-1)
        self.tokens.index_copy_(1, self.t + 1, nxt[:, None])
        self.pos_scores.index_copy_(1, self.t, lp.gather(1, nxt[:, None]))
        newly = (~self.done) & nxt.eq(self.eos)
        self.lengths.copy_(torch.where(newly, (self.t + 1).expand(self.B), self.lengths))
        self.done |= newly
        self.stop.index_copy_(0, self.t, self.done.all().to(torch.int32).reshape(1))
        self.t += 1

    _span = SynthesisGraph._span
    run = SynthesisGraph.run

    def _snapshot(self):
        done, lengths = self.done.clone(), self.lengths.clone()

        def undo():  # (tokens[t+1] and stop[t] are rewritten by the replay; the finished flags are read-modify-write)
            self.done.copy_(done)
            self.lengths.copy_(lengths)
        return undo

    @torch.no_grad()
    def decode(self, encoder_out, max_len, **kw):
        """Returns a list of 1-D LongTensors ending in eos (generate_text_greedy's contract)."""
        self.begin(encoder_out, max_len, **kw)
        idx = 0
        while idx <= max_len:
            n = min(self.CHUNK, max_len + 1 - idx)
            flags = self.run(idx, n)
            idx += n
            if any(flags):
                break
        lengths = self.lengths.tolist()
        return [self.tokens[b, 1: lengths[b] + 1].clone() for b in range(self.B)]


def greedy_graph(model, B, S, max_len, device, capture=True):
    """The model's GreedyGraph for batch B, encoder length S and max_len steps (buckets: S to multiples of 64, max_len to
    powers of two >= 64); rebuilt when the numeric mode or the weights changed."""
    S_b = max(64, (S + 63) // 64 * 64)
    M_b = 64
    while M_b < max_len:
        M_b *= 2
    store = model.__dict__.setdefault("_greedy_graphs", {})
    key = (B, S_b, M_b, RT.dtype, str(device), bool(capture), RT.param_epoch)
    gg = store.get(key)
    if gg is None:
        for k in [k for k in store if k[:6] == key[:6]]:
            del store[k]
        gg = store[key] = GreedyGraph(model, B, S_b, M_b, device, capture=capture)
    return gg
