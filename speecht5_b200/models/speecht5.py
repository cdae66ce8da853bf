"""`t5_transformer` model and its architecture presets on the B200 kernel library -- drop-in for
speecht5/models/speecht5.py (reference): same registry names (@register_model "t5_transformer"; archs t5_transformer,
t5_transformer_base, t5_transformer_large, t5_transformer_base_asr :1252,1385,1402,1427), same forward signature
(:786) and return tuples, same parameter names (checkpoints load with load_state_dict).

Coverage of forward(): text -> speech (t2s, the BASELINE.json metric path), speech -> text (s2t: waveform front end,
CE + CTC), text -> text (t2t / text pre-training), speech pre-training (HuBERT targets, masked-prediction head, shared
Gumbel quantizer, reconstruction through the speech decoder; only_hubert / feature_only returns), greedy generation of
speech and text. The branches SURVEY.md section 2 leaves out (speaker identification s2c, voice conversion /
enhancement s2s inputs) raise NotImplementedError rather than silently falling back to PyTorch."""
import argparse
import logging
from argparse import Namespace

import torch
import torch.nn as nn
import torch.nn.functional as F

from ..fairseq_shim import FairseqEncoderDecoderModel, register_model, register_model_architecture
from ..ops import RT
from .modules.nets import (SpeechDecoderPostnet, SpeechDecoderPrenet, TextDecoderPostnet, TextDecoderPrenet,
                           TextEncoderPrenet)
from .modules.transformer import MultiheadAttention, TransformerDecoder, TransformerEncoder

logger = logging.getLogger(__name__)

DEFAULT_MAX_TEXT_POSITIONS = 450
DEFAULT_MAX_SPEECH_POSITIONS = 4000


def Embedding(num_embeddings, embedding_dim, padding_idx):  # fairseq/models/transformer.py:1054
    m = nn.Embedding(num_embeddings, embedding_dim, padding_idx=padding_idx)
    nn.init.normal_(m.weight, mean=0, std=embedding_dim ** -0.5)
    nn.init.constant_(m.weight[padding_idx], 0)
    return m


def init_bert_params(module):  # fairseq/modules/transformer_sentence_encoder.py:21-53
    def normal_(data):
        data.copy_(data.cpu().normal_(mean=0.0, std=0.02).to(data.device))
    if isinstance(module, nn.Linear):
        normal_(module.weight.data)
        if module.bias is not None:
            module.bias.data.zero_()
    if isinstance(module, nn.Embedding):
        normal_(module.weight.data)
        if module.padding_idx is not None:
            module.weight.data[module.padding_idx].zero_()
    if isinstance(module, MultiheadAttention):
        normal_(module.q_proj.weight.data)
        normal_(module.k_proj.weight.data)
        normal_(module.v_proj.weight.data)


class _Dict:
    """Tiny stand-in for fairseq Dictionary when building without a task (len/pad only)."""

    def __init__(self, n, pad=1):
        self.n, self._pad = n, pad

    def __len__(self):
        return self.n

    def pad(self):
        return self._pad

    def eos(self):
        return 2

    def unk(self):
        return 3


@register_model("t5_transformer")
class T5TransformerModel(FairseqEncoderDecoderModel):
    def __init__(self, args, encoder, decoder, text_encoder_prenet, speech_encoder_prenet, text_decoder_prenet,
                 speech_decoder_prenet, text_decoder_postnet, speech_decoder_postnet, speaker_decoder_postnet,
                 speech_encoder_postnet):
        super().__init__(encoder, decoder)
        self.encoder, self.decoder = encoder, decoder
        self.text_encoder_prenet = text_encoder_prenet
        self.speech_encoder_prenet = speech_encoder_prenet
        self.text_decoder_prenet = text_decoder_prenet
        self.speech_decoder_prenet = speech_decoder_prenet
        self.text_decoder_postnet = text_decoder_postnet
        self.speech_decoder_postnet = speech_decoder_postnet
        self.speaker_decoder_postnet = speaker_decoder_postnet
        self.hubert_layer = speech_encoder_postnet
        self.reduction_factor = args.reduction_factor
        self.spk_embed_dim = args.spk_embed_dim
        self.spk_embed_integration_type = args.spk_embed_integration_type
        assert self.spk_embed_integration_type == "pre" or self.spk_embed_dim is None, \
            "only spk_embed_integration_type='pre' (the reference default) is implemented"
        self.use_codebook = args.use_codebook
        self.codebook_prob = getattr(args, "codebook_prob", 0.5)
        if self.use_codebook:  # (:93-106) Gumbel vector quantizer of the pre-training recipes
            from ..pretrain import GumbelVectorQuantizer
            if getattr(args, "quantizer_depth", 1) != 1:
                raise NotImplementedError("quantizer_depth > 1 (no SpeechT5 recipe uses it)")
            temp = getattr(args, "latent_temp", (2.0, 0.5, 0.999995))
            temp = eval(temp) if isinstance(temp, str) else temp
            vq_dim = args.latent_dim if getattr(args, "latent_dim", 0) > 0 else args.encoder_embed_dim
            self.quantizer = GumbelVectorQuantizer(dim=args.encoder_embed_dim, num_vars=getattr(args, "latent_vars", 100),
                                                   temp=tuple(temp), groups=getattr(args, "latent_groups", 2), vq_dim=vq_dim)
        self.num_updates = 0
        if args.bert_init:
            self.apply(init_bert_params)
        self.args = args

    # ------------------------------------------------------------------ command-line surface (models/speecht5.py:118-700)
    # Same option names and types as the reference, so a recipe's command line parses unchanged. Options of branches
    # that are not built are accepted and rejected at build time if they are switched on.
    _OPTIONS = (
        ("--activation-fn", dict(type=str, choices=["relu", "gelu", "gelu_fast", "gelu_accurate", "tanh", "linear"])),
        ("--dropout", dict(type=float, metavar="D")),
        ("--attention-dropout", dict(type=float, metavar="D")),
        (("--activation-dropout", "--relu-dropout"), dict(type=float, metavar="D")),
        ("--encoder-embed-dim", dict(type=int, metavar="N")),
        ("--encoder-ffn-embed-dim", dict(type=int, metavar="N")),
        ("--encoder-layers", dict(type=int, metavar="N")),
        ("--encoder-attention-heads", dict(type=int, metavar="N")),
        ("--encoder-normalize-before", dict(action="store_true")),
        ("--decoder-normalize-before", dict(action="store_true")),
        ("--decoder-embed-dim", dict(type=int, metavar="N")),
        ("--decoder-ffn-embed-dim", dict(type=int, metavar="N")),
        ("--decoder-layers", dict(type=int, metavar="N")),
        ("--decoder-attention-heads", dict(type=int, metavar="N")),
        ("--reduction-factor", dict(type=int)),
        ("--spk-embed-dim", dict(type=int)),
        ("--layernorm-embedding", dict(action="store_true")),
        ("--load-pretrained-encoder-from", dict(type=str, metavar="STR")),
        ("--share-input-output-embed", dict(action="store_true")),
        ("--share-ctc-embed", dict(action="store_true")),
        ("--encoder-speech-prenet", dict(default="conv", type=str, choices=["conv", "linear"])),
        ("--spk-embed-integration-type", dict(type=str, choices=["pre", "add"])),
        ("--dprenet-dropout-rate", dict(default=0.5, type=float)),
        ("--modules-filter", dict(default=None, type=str)),
        ("--encoder-layerdrop", dict(type=float, metavar="D")),
        ("--decoder-layerdrop", dict(type=float, metavar="D")),
        ("--mask-selection", dict(type=str, choices=["static", "uniform", "normal", "poisson"])),
        ("--mask-channel-selection", dict(type=str, choices=["static", "uniform", "normal", "poisson"])),
        ("--use-codebook", dict(action="store_true")),
        ("--codebook-prob", dict(type=float)),
        ("--latent-vars", dict(type=int)),
        ("--latent-groups", dict(type=int)),
        ("--latent-dim", dict(type=int)),
        ("--latent-temp", dict(type=str)),
        ("--quantizer-depth", dict(type=int)),
        ("--quantizer-factor", dict(type=int)),
        ("--relative-position-embedding", dict(action="store_true")),
        ("--num-buckets", dict(type=int)),
        ("--max-distance", dict(type=int)),
        ("--encoder-max-relative-position", dict(type=int)),
        ("--decoder-max-relative-position", dict(type=int)),
        ("--conv-feature-layers", dict(type=str, metavar="EXPR")),
        ("--conv-bias", dict(action="store_true")),
        ("--extractor-mode", dict(choices=["default", "layer_norm"])),
        ("--bert-init", dict(action="store_true")),
        ("--unb-enc-layer", dict(type=int, default=-1)),
        # waveform front end, HuBERT masking and head, freezing (add_args :217-232, :418-520): read by the speech-input branch
        ("--freeze-encoder-updates", dict(type=int)),
        ("--freeze-decoder-updates", dict(type=int)),
        ("--no-freeze-encoder-layer", dict(type=str)),
        ("--feature-grad-mult", dict(type=float)),
        ("--logit-temp", dict(type=float)),
        ("--final-dim", dict(type=int)),
        ("--hubert-mask-length", dict(type=int)),
        ("--mask-prob", dict(type=float)),
        ("--mask-other", dict(type=float)),
        ("--mask-min-space", dict(type=int)),
        ("--mask-channel-length", dict(type=int)),
        ("--mask-channel-prob", dict(type=float)),
        ("--mask-channel-other", dict(type=float)),
        ("--mask-channel-min-space", dict(type=int)),
        ("--conv-pos", dict(type=int)),
        ("--conv-pos-groups", dict(type=int)),
        ("--get-code-distribution", dict(action="store_true")),
        # options of branches this implementation does not build (speaker identification, enhancement, the
        # convolutional subsampler, sliding-window / branched encoders): accepted so that every recipe's command line
        # parses; they only matter once such a branch is called, and those raise NotImplementedError
        ("--encoder-sliding-window-attn", dict(type=int, default=None)),
        ("--conv-kernel-sizes", dict(type=str, default="5,5")),
        ("--conv-channels", dict(type=int, default=1024)),
        ("--subsample-stride", dict(type=str, default="2,2")),
        ("--se-predict", dict(default=None, choices=["masking", "target", "delta"])),
        ("--se-decoder-input", dict(type=str, default="previous_target", choices=["previous_target", "source"])),
        ("--encoder-attn-branch", dict(type=str, default="identity,full")),
        ("--encoder-block-branch", dict(type=str, default=None)),
        ("--sid-pad-prenet", dict(action="store_true")),
        ("--sid-encoder-cls", dict(default=None, choices=["encoder"])),
        ("--sid-shuffle-encoder-input", dict(action="store_true")),
        ("--sid-decoder-speaker", dict(action="store_true")),
        ("--sid-decoder-attn-dim", dict(type=int, default=128)),
        ("--sid-t5-postnet", dict(action="store_true")),
        ("--sid-embed-dim", dict(type=int, default=128)),
        ("--sid-pooling-layer", dict(type=str, default="decoder",
                                     choices=["decoder-las", "decoder", "encoder", "encoder-cls", "encoder-speaker"])),
        ("--sid-no-pooling-bn", dict(action="store_true")),
        ("--sid-no-embed-postnet", dict(action="store_true")),
        ("--sid-normalize-postnet", dict(action="store_true")),
        ("--sid-softmax-type", dict(default="softmax", choices=["softmax", "amsoftmax", "aamsoftmax"])),
        ("--softmax-scale", dict(type=float, default=1.0)),
        ("--softmax-margin", dict(type=float, default=0.0)),
        ("--softmax-easy-margin", dict(action="store_true")),
        # this implementation only: construct the text decoder pre/post-net (the reference always does)
        ("--build-text-decoder", dict(action="store_true")),
        ("--build-speech-encoder", dict(action="store_true")),
    )

    @classmethod
    def add_args(cls, parser):
        for flags, kw in cls._OPTIONS:
            flags = flags if isinstance(flags, tuple) else (flags,)
            kw = dict(kw)
            if kw.get("action") != "store_true" and "default" not in kw:
                kw["default"] = argparse.SUPPRESS  # unset options fall through to the arch function, like fairseq's
            elif kw.get("action") == "store_true":
                kw["default"] = argparse.SUPPRESS
            parser.add_argument(*flags, **kw)

    # ------------------------------------------------------------------ construction
    @classmethod
    def build_model(cls, args, task=None):
        base_architecture(args)
        text_dict = task.dicts["text"] if task is not None else _Dict(getattr(args, "vocab_size", 81))

        def build_embedding(dictionary, embed_dim):
            return Embedding(len(dictionary), embed_dim, dictionary.pad())

        text_decoder_embed_tokens = build_embedding(text_dict, args.decoder_embed_dim)
        text_encoder_embed_tokens = (text_decoder_embed_tokens if args.share_input_output_embed
                                     else build_embedding(text_dict, args.encoder_embed_dim))
        speech_odim = getattr(args, "speech_odim", 80)
        encoder = TransformerEncoder(args, text_dict, text_encoder_embed_tokens)
        decoder = TransformerDecoder(args)
        text_encoder_prenet = TextEncoderPrenet(text_encoder_embed_tokens, args)
        speech_decoder_prenet = SpeechDecoderPrenet(speech_odim, args)
        speech_decoder_postnet = SpeechDecoderPostnet(speech_odim, args)
        # text decoder pre/post-net (SURVEY 8a rows 9, 14): opt-in (--build-text-decoder) until the rest of the
        # text-output path (ASR front-end, incremental decoding) is built; the reference always constructs them
        text_decoder_prenet = text_decoder_postnet = None
        if getattr(args, "build_text_decoder", False):
            text_decoder_prenet = TextDecoderPrenet(text_decoder_embed_tokens, args)
            text_decoder_postnet = TextDecoderPostnet(text_decoder_embed_tokens, len(text_dict), args)
        # waveform front end (SURVEY 8a rows 2, 3): opt-in (--build-speech-encoder), see frontend.py
        speech_encoder_prenet = None
        if getattr(args, "build_speech_encoder", False):
            from ..frontend import SpeechEncoderPrenet
            speech_encoder_prenet = SpeechEncoderPrenet(args)
        # masked-prediction head of speech pre-training (:717-720): built when the task carries HuBERT label dictionaries
        speech_encoder_postnet = None
        hub = task.dicts.get("hubert") if (task is not None and hasattr(task, "dicts")) else None
        classes = [len(dct) for dct in hub] if hub else getattr(args, "hubert_num_classes", None)
        if classes:
            from ..pretrain import SpeechEncoderPostnet
            fd = getattr(args, "final_dim", 0)
            speech_encoder_postnet = SpeechEncoderPostnet(
                classes, args.encoder_embed_dim, fd if fd > 0 else args.encoder_embed_dim,
                logit_temp=getattr(args, "logit_temp", 0.1), untie_final_proj=getattr(args, "untie_final_proj", True),
                skip_masked=getattr(args, "skip_masked", False), skip_nomask=getattr(args, "skip_nomask", False),
                target_glu=getattr(args, "target_glu", False))
        return cls(args, encoder, decoder, text_encoder_prenet, speech_encoder_prenet, text_decoder_prenet,
                   speech_decoder_prenet, text_decoder_postnet, speech_decoder_postnet, None, speech_encoder_postnet)

    # ------------------------------------------------------------------ forward (models/speecht5.py:786-963)
    def forward(self, source=None, src_tokens=None, src_lengths=None, prev_output_tokens=None, tgt_lengths=None,
                spkembs=None, target_list=None, task_name=None, padding_mask=None, only_hubert=False, only_ctc=False,
                feature_only=False, tgt_enc_layer=None, mask=True, mask_indices=None, mask_channel_indices=None):
        """Reference signature (:786) + two optional extras: `mask_indices` / `mask_channel_indices`, a HuBERT-style mask
        draw made by the caller (the trainer draws on the host before replaying a captured step)."""
        assert source is not None or src_tokens is not None
        input_type = "text" if (source is None and padding_mask is None and not feature_only) else "speech"
        output_type = "text" if (prev_output_tokens is not None and prev_output_tokens.dim() == 2) else "speech"
        text_out = output_type == "text" and self.text_decoder_prenet is not None
        t2t = input_type == "text" and text_out
        speech_in = input_type == "speech" and self.speech_encoder_prenet is not None and not feature_only
        built = (input_type == "text" and output_type == "speech") or t2t or (
            speech_in and (text_out or output_type == "speech" or prev_output_tokens is None))
        if target_list is not None and (self.hubert_layer is None or not speech_in):
            raise NotImplementedError("pre-training targets need speech input and the masked-prediction head "
                                      "(task with HuBERT label dictionaries, or --hubert-num-classes)")
        if not built:
            raise NotImplementedError(
                f"T5TransformerModel.forward: {input_type}->{output_type} (task {task_name}) is not built in the B200 "
                "path (speaker identification / voice conversion / enhancement branches)")
        features_pen = frame_mask_indices = None
        if speech_in and target_list is not None:  # (:813-815) speech pre-training: frames aligned with the labels
            enc_in, encoder_padding_mask = self.speech_encoder_prenet(
                source, require_feat_pen=True, target_list=target_list, padding_mask=padding_mask, mask=mask,
                mask_indices=mask_indices, mask_channel_indices=mask_channel_indices)
            encoder_input, features_pen, frame_mask_indices, target_list = enc_in
        elif speech_in:  # (:815-820) waveform -> frames; the HuBERT-style mask is drawn only in training
            encoder_input, encoder_padding_mask = self.speech_encoder_prenet(
                source, padding_mask=padding_mask, mask=self.training and mask, mask_indices=mask_indices,
                mask_channel_indices=mask_channel_indices)
        else:
            encoder_input, encoder_padding_mask = self.text_encoder_prenet(src_tokens)
        encoder_output = self.encoder(encoder_input, encoder_padding_mask, tgt_layer=tgt_enc_layer)
        if task_name == "speech_pretrain" and feature_only:  # (:832-833)
            return encoder_output["encoder_out"][0].transpose(0, 1)
        hubert_results = None
        if target_list is not None:  # (:844-852) masked / unmasked frame logits against the label embeddings
            pm = encoder_padding_mask if encoder_padding_mask is not None else torch.zeros(
                encoder_input.shape[:2], dtype=torch.bool, device=encoder_input.device)
            mi = frame_mask_indices if frame_mask_indices is not None else torch.zeros_like(pm)
            hubert_results = self.hubert_layer(encoder_output["_encoder_out_btc"], pm, mi, target_list)
            hubert_results["features_pen"] = features_pen
        if "decoder_input" in encoder_output and encoder_output["decoder_input"][0] is not None:
            encoder_output["encoder_out"] = encoder_output["decoder_input"]
            encoder_output["_encoder_out_btc"] = encoder_output["decoder_input"][0].transpose(0, 1)
        codebook_out = {}
        if self.use_codebook:  # (:858-882) a random share of the time steps is replaced by its quantized code
            from ..pretrain import mix_codes
            x_btc = encoder_output["_encoder_out_btc"]
            q = self.quantizer(x_btc, gumbel_noise=getattr(self, "_gumbel_noise", None))
            mixed = mix_codes(x_btc, q["x"], self.codebook_prob, perm=getattr(self, "_codebook_perm", None))
            encoder_output["_encoder_out_btc"] = mixed
            encoder_output["encoder_out"] = [mixed.transpose(0, 1)]
            stats = {k: q[k] for k in ("prob_perplexity", "code_perplexity", "num_vars", "temp")}
            if output_type == "speech" and hubert_results is not None:
                hubert_results.update(stats)
            elif output_type == "text":
                codebook_out.update(stats)
        if only_hubert and target_list is not None:  # (:884-885)
            return hubert_results, None
        if speech_in and task_name == "s2t":  # (:885-888)
            if only_ctc:
                return None, encoder_output
            if not self.training and prev_output_tokens is None:
                return encoder_output
        if text_out:  # (:901-903, 955-957): decoder on token embeddings, vocabulary logits
            dec_in, tgt_mask, _ = self.text_decoder_prenet(prev_output_tokens)
            decoder_output, extra = self.decoder(
                dec_in, tgt_mask, encoder_output,
                full_context_alignment=getattr(self.args, "decoder_full_context_alignment", False),
                alignment_layer=None)
            logits = self.text_decoder_postnet(decoder_output)
            if task_name == "s2t":  # (:955-956)
                return (logits, None), encoder_output
            return (logits, None), codebook_out, encoder_output
        prev_output_tokens, tgt_mask = self.speech_decoder_prenet(prev_output_tokens, tgt_lengths, spkembs)
        decoder_output, extra = self.decoder(
            prev_output_tokens, tgt_mask, encoder_output,
            full_context_alignment=getattr(self.args, "decoder_full_context_alignment", False),
            alignment_layer=-1 if target_list is None else None)  # (:921-923)
        if target_list is not None:  # (:960-961) speech pre-training: head results + the reconstruction branch
            return hubert_results, (self.speech_decoder_postnet(decoder_output) + (extra["attn"][0],))
        return self.speech_decoder_postnet(decoder_output) + (extra["attn"][0],)

    # ------------------------------------------------------------------ fairseq model API used by callers
    def set_num_updates(self, num_updates):
        for m in self.modules():
            if m is not self and hasattr(m, "set_num_updates"):
                m.set_num_updates(num_updates)
        self.num_updates = num_updates
        RT.invalidate_shadows()  # fairseq calls this once per optimizer update: refresh bf16 weight shadows

    def load_state_dict(self, state_dict, strict=True, model_cfg=None, args=None):
        """Non-strict per-submodule loading like the reference (:1022-1058): missing sub-modules are skipped."""
        own = self.state_dict()
        filtered = {k: v for k, v in state_dict.items() if k in own and own[k].shape == v.shape}
        dropped = [k for k in state_dict if k not in filtered]
        if dropped:
            logger.info("load_state_dict: ignoring %d keys absent/mismatched in the B200 t2s model", len(dropped))
        out = super().load_state_dict(filtered, strict=False)
        RT.params_written_externally()  # incl. the trainer's flat bf16 shadow, if one exists (fairseq: build, then load)
        return out

    def max_positions(self):
        return (self.args.max_speech_positions, self.args.max_text_positions)

    # ---- criterion-facing helpers of the reference model (models/speecht5.py:731-784). They post-process tensors the
    # device path produced (vocabulary-sized softmax of the text heads); the text-output heads themselves are "next" rows.
    def get_normalized_probs(self, net_output, log_probs, sample=None):
        logits = net_output[0]
        out = F.log_softmax(logits.float(), dim=-1) if log_probs else F.softmax(logits.float(), dim=-1)
        out.batch_first = True  # :739
        return out

    def get_normalized_probs_for_ctc(self, net_output, log_probs):
        logits = net_output["encoder_out_for_ctc"][0]
        return F.log_softmax(logits.float(), dim=-1) if log_probs else F.softmax(logits.float(), dim=-1)

    def get_logits(self, net_output, is_masked=True):
        logits_list = net_output["logit_m_list"] if is_masked else net_output["logit_u_list"]
        return [x.float() for x in logits_list if x is not None]

    def get_targets(self, sample, net_output, is_masked=True):
        if "logit_m_list" in net_output:
            return [x.new_zeros(x.size(0), dtype=torch.long) for x in self.get_logits(net_output, is_masked)]
        return sample["target"]

    def get_extra_losses(self, net_output):
        extra_losses, names = [], []
        if "features_pen" in net_output:
            extra_losses.append(net_output["features_pen"])
            names.append("features_pen")
        if "prob_perplexity" in net_output:
            extra_losses.append((net_output["num_vars"] - net_output["prob_perplexity"]) / net_output["num_vars"])
            names.append("prob_perplexity")
        return extra_losses, names

    def forward_encoder(self, source, padding_mask=None):
        if getattr(self, "speech_encoder_prenet", None) is not None:  # (:1133-1140)
            encoder_input, encoder_padding_mask = self.speech_encoder_prenet(source, padding_mask=padding_mask,
                                                                             mask=False)
            return self.encoder(encoder_input, encoder_padding_mask)
        raise NotImplementedError("forward_encoder takes a waveform: build the model with --build-speech-encoder "
                                  "(use forward_text_encoder for text input)")

    def forward_encoder_torchscript(self, net_input):
        """(:1112-1124) what fairseq's generator calls; TorchScript export is not a target of this implementation."""
        return self.forward_encoder_non_torchscript(net_input)

    def forward_encoder_non_torchscript(self, net_input):  # (:1126-1131)
        return self.forward_encoder(**{k: v for k, v in net_input.items() if k not in ("prev_output_tokens", "task_name")})

    def forward_decoder(self, tokens, encoder_out, incremental_state):
        """(:1151-1164) vocabulary logits of the text decoder. With an incremental state the reference feeds only the
        last token and returns [B, 1, V]; this entry point re-runs the decoder on the whole prefix (causal
        self-attention makes the last row identical) and returns the last position. The cached forms -- key/value cache
        and one captured CUDA graph per step -- live in speecht5_b200/incremental.py (generate_text_greedy use_cache)."""
        if getattr(self, "text_decoder_prenet", None) is None:
            raise NotImplementedError("text decoding needs the opt-in text decoder (--build-text-decoder): "
                                      "SURVEY.md section 8a rows 9, 14, 21")
        dec_in, tgt_mask, _ = self.text_decoder_prenet(tokens)
        decoder_output, extra = self.decoder(dec_in, tgt_mask, encoder_out, alignment_layer=None)
        if incremental_state is not None:
            decoder_output = decoder_output[:, -1:, :]
        return self.text_decoder_postnet(decoder_output), extra

    @torch.no_grad()
    def generate_text_greedy(self, source, padding_mask=None, max_len_a=0.0, max_len_b=200, min_len=1, unk_penalty=0.0,
                             temperature=1.0, pad=1, eos=2, unk=3, blank=0, mask_idx=None, use_cache=False,
                             return_scores=False):
        """Beam-1 decoding as `generate.py --beam 1` runs it (speecht5/sequence_generator.py:207-655 with ctc_weight 0
        and no LM): encoder once, then per step log_softmax(logits / T) of the last position with the reference's
        masking order (:430-446: eos forbidden before min_len, NaN -> -inf, pad never, unk penalty, CTC blank and mask
        symbol never, only eos once max_len is reached) and argmax. The prefix starts with eos; max_len counts PADDED
        source samples (:249,262-265). Returns a list of 1-D LongTensors ending in eos.
        use_cache: False (prefix recomputation), True (key/value cache), "graph" (one captured CUDA graph per step)."""
        import math
        B, src_len = source.size(0), source.size(1)
        max_len = min(int(max_len_a * src_len + max_len_b), self.args.max_text_positions - 1)
        assert min_len <= max_len
        enc = self.forward_encoder(source, padding_mask=padding_mask)
        if use_cache in ("graph", "graph_body_eager"):  # one captured CUDA graph per step (incremental.GreedyGraph)
            from ..incremental import greedy_graph
            S = enc["encoder_out"][0].size(0)
            gg = greedy_graph(self, B, S, max_len, source.device, capture=use_cache == "graph")
            hyp = gg.decode(enc, max_len, min_len=min_len, unk_penalty=unk_penalty, temperature=temperature, pad=pad,
                            eos=eos, unk=unk, blank=blank, mask_idx=mask_idx)
            if return_scores:  # (log-probability of every emitted token, eos included)
                return hyp, [gg.pos_scores[b, : len(h)].clone() for b, h in enumerate(hyp)]
            return hyp
        tokens = torch.full((B, max_len + 2), pad, dtype=torch.long, device=source.device)
        tokens[:, 0] = eos
        done = torch.zeros(B, dtype=torch.bool, device=source.device)
        lengths = torch.zeros(B, dtype=torch.long, device=source.device)
        pos_scores = torch.zeros((B, max_len + 1), dtype=torch.float32, device=source.device)
        cache = None
        if use_cache:  # key/value cache (speecht5_b200/incremental.py): one new row per step
            from ..incremental import DecoderCache, decoder_step
            cache = DecoderCache(self.decoder, enc, max_len + 1)
        for step in range(max_len + 1):
            if cache is not None:
                dec_in, _, _ = self.text_decoder_prenet(tokens[:, : step + 1])
                z, _ = decoder_step(self.decoder, dec_in[:, -1:], cache)
                logits = self.text_decoder_postnet(z)
            else:
                logits, _ = self.forward_decoder(tokens[:, : step + 1], enc, incremental_state={})
            lprobs = F.log_softmax(logits[:, -1, :].float() / temperature, dim=-1)
            if step < min_len:
                lprobs[:, eos] = -math.inf
            lprobs[lprobs != lprobs] = -math.inf
            lprobs[:, pad] = -math.inf
            lprobs[:, unk] -= unk_penalty
            lprobs[:, blank] = -math.inf
            if mask_idx is not None and mask_idx != unk:
                lprobs[:, mask_idx] = -math.inf
            if step >= max_len:
                lprobs[:, :eos] = -math.inf
                lprobs[:, eos + 1:] = -math.inf
            nxt = lprobs.argmax(dim=-1)
            tokens[:, step + 1] = nxt
            pos_scores[:, step] = lprobs.gather(1, nxt[:, None])[:, 0]
            newly = (~done) & nxt.eq(eos)
            lengths = torch.where(newly, torch.full_like(lengths, step + 1), lengths)
            done |= newly
            if bool(done.all()):
                break
        hyp = [tokens[b, 1: int(lengths[b]) + 1].clone() for b in range(B)]
        if return_scores:
            return hyp, [pos_scores[b, : len(h)].clone() for b, h in enumerate(hyp)]
        return hyp

    @torch.no_grad()
    def generate_text_beam(self, source, padding_mask=None, beam_size=5, ctc_weight=0.0, max_len_a=0.0, max_len_b=200,
                           min_len=1, normalize_scores=True, len_penalty=1.0, unk_penalty=0.0, temperature=1.0, pad=1,
                           eos=2, unk=3, blank=0, mask_idx=None, mask_idxs=None, use_cache=False):
        """Beam search with optional joint CTC/attention scoring, as `generate.py --beam N --ctc-weight W` runs it
        (speecht5/sequence_generator.py:207-655; speecht5_b200/beam.py states the two deliberate deviations: per-utterance
        CTC posteriors at batch > 1, and a defined state for a selected token outside the CTC candidates). Returns, per
        sentence, min(beam_size, V - 1) hypotheses {"tokens", "score", "positional_scores", "alignment", "attention"}
        sorted by score. use_cache: False (prefix recomputation), True (key/value cache, rows reordered by
        st5_beam_gather_rows)."""
        from ..beam import beam_search
        return beam_search(self, source, padding_mask, beam_size=beam_size, ctc_weight=ctc_weight, max_len_a=max_len_a,
                           max_len_b=max_len_b, min_len=min_len, normalize_scores=normalize_scores,
                           len_penalty=len_penalty, unk_penalty=unk_penalty, temperature=temperature, pad=pad, eos=eos,
                           unk=unk, blank=blank, mask_idx=mask_idx, mask_idxs=mask_idxs, use_cache=bool(use_cache))

    def forward_text_encoder(self, src_tokens):
        encoder_input, encoder_padding_mask = self.text_encoder_prenet(src_tokens)
        return self.encoder(encoder_input, encoder_padding_mask)

    @torch.no_grad()
    def generate_speech(self, source=None, src_tokens=None, spkembs=None, **kwargs):
        """models/speecht5.py:1188-1249, text input: greedy frame-by-frame synthesis until a stop probability of the
        current r-frame group reaches the threshold (or maxlen). Same knobs and quirk as the reference, which reads
        kwargs["threshold"] for the threshold, minlenratio AND maxlenratio (:1190-1199); defaults 0.5 / 0.0 / 20.0.
        Returns (mel [L, odim] fp32, stop probabilities [L], cross-attention [layers, H, L/r, T_text]).

        use_cache=False re-runs the decoder on the whole prefix every step (causal self-attention makes that equal to
        the reference's incremental state, and every step reuses the training kernels; the always-on prenet dropout then
        draws one mask per step for the whole prefix, where the reference keeps the cached keys/values of earlier draws
        -- identical in distribution for the newest frame); use_cache=True keeps a key/value cache, "graph" replays one
        captured CUDA graph per decoder step (speecht5_b200/incremental.py)."""
        assert source is not None or src_tokens is not None
        if source is not None:
            raise NotImplementedError("generate_speech from speech input (voice conversion, out of scope: SURVEY.md section 2)")
        assert src_tokens.size(0) == 1
        threshold = kwargs.get("threshold", 0.5)
        minlenratio = kwargs.get("threshold", 0.0)
        maxlenratio = kwargs.get("threshold", 20.0)
        if spkembs is not None and getattr(self.args, "spk_embed_integration_type", "pre") != "pre":
            raise NotImplementedError("spk_embed_integration_type != 'pre'")
        encoder_out = self.forward_text_encoder(src_tokens)
        post = self.speech_decoder_postnet
        r, odim = self.reduction_factor, post.odim
        T_enc = encoder_out["encoder_out"][0].size(0)
        maxlen, minlen = int(T_enc * maxlenratio / r), int(T_enc * minlenratio / r)
        ys = torch.zeros(1, 1, odim, dtype=torch.float32, device=src_tokens.device)
        outs, probs, attns, idx = [], [], [], 0
        cache = None
        if kwargs.get("use_cache", False) in ("graph", "graph_body_eager"):
            # key/value cache + ONE captured CUDA graph per decoder step (speecht5_b200/incremental.py SynthesisGraph):
            # the host replays steps and reads their stop flags, nothing else; graphs are kept on the model
            from ..incremental import synthesis_graph
            seed_t = RT._seed_t
            try:
                sg = synthesis_graph(self, T_enc, max(maxlen, 1), src_tokens.device,
                                     capture=kwargs["use_cache"] == "graph")
                before, stop_probs, attn = sg.synthesize(encoder_out, spkembs, threshold, minlen, maxlen)
                return post.refine(before)[0], stop_probs, attn
            finally:
                RT._seed_t = seed_t
        if kwargs.get("use_cache", False):  # key/value cache, eager step (speecht5_b200/incremental.py)
            from ..incremental import DecoderCache, decoder_step
            cache = DecoderCache(self.decoder, encoder_out, max(maxlen, 1) + 1)
        while True:
            idx += 1
            decoder_in, _ = self.speech_decoder_prenet(ys, spkembs=spkembs)
            if cache is not None:
                z, layer_attn = decoder_step(self.decoder, decoder_in[:, -1:], cache, need_head_weights=True)
            else:
                z, extra = self.decoder(decoder_in, None, encoder_out, alignment_layer=-1)
                layer_attn = extra["attn"][0]
            before, logits = post.project(z[:, -1:].contiguous())  # [1, r, odim], [1, r]
            outs.append(before[0])
            probs.append(torch.sigmoid(logits[0]))
            ys = torch.cat((ys, before[:, -1:, :]), dim=1)
            layer_attn = layer_attn if isinstance(layer_attn, (list, tuple)) else [layer_attn]
            attns.append(torch.stack([a[0, :, -1:, :].float() for a in layer_attn], dim=0))  # [layers, H, 1, T]
            if bool((probs[-1] >= threshold).any()) or idx >= maxlen:
                if idx < minlen:
                    continue
                mel = post.refine(torch.cat(outs, dim=0).unsqueeze(0))[0]
                return mel, torch.cat(probs, dim=0), torch.cat(attns, dim=2)


# ---------------------------------------------------------------------------------------------- architectures
@register_model_architecture(model_name="t5_transformer", arch_name="t5_transformer")
def base_architecture(args):  # models/speecht5.py:1252-1383 (fields used by the built path)
    g = lambda k, v: setattr(args, k, getattr(args, k, v))  # noqa: E731
    g("bert_init", False)
    g("encoder_embed_dim", 768)
    g("encoder_ffn_embed_dim", 768 * 4)
    g("encoder_layers", 12)
    g("encoder_attention_heads", 12)
    g("encoder_normalize_before", False)
    g("decoder_embed_dim", args.encoder_embed_dim)
    g("decoder_ffn_embed_dim", args.encoder_ffn_embed_dim)
    g("decoder_layers", 6)
    g("decoder_attention_heads", 12)
    g("decoder_normalize_before", False)
    g("dropout", 0.1)
    g("attention_dropout", args.dropout)
    g("activation_dropout", args.dropout)
    g("activation_fn", "gelu")
    g("decoder_layerdrop", 0.0)
    g("encoder_layerdrop", 0)
    g("max_text_positions", DEFAULT_MAX_TEXT_POSITIONS)
    g("max_speech_positions", DEFAULT_MAX_SPEECH_POSITIONS)
    g("use_batch_norm", True)
    g("enc_use_scaled_pos_enc", True)
    g("dec_use_scaled_pos_enc", True)
    g("postnet_layers", 5)
    g("postnet_chans", 256)
    g("postnet_filts", 5)
    g("postnet_dropout_rate", 0.5)
    g("dprenet_dropout_rate", 0.5)
    g("dprenet_layers", 2)
    g("dprenet_units", 256)
    g("initial_encoder_alpha", 1.0)
    g("initial_decoder_alpha", 1.0)
    g("spk_embed_integration_type", "pre")
    g("spk_embed_dim", 512)
    g("encoder_reduction_factor", 1)
    g("reduction_factor", 2)
    g("transformer_enc_positional_dropout_rate", 0.1)
    g("transformer_dec_positional_dropout_rate", 0.1)
    g("layer_norm_eps", 1e-5)
    g("no_scale_embedding", True)
    g("share_input_output_embed", False)
    g("share_ctc_embed", False)
    g("freeze_encoder_updates", 0)
    g("freeze_decoder_updates", 0)
    g("no_freeze_encoder_layer", None)
    g("layer_norm_first", False)
    g("use_sent_enc_layer", True)
    g("use_codebook", False)
    # pre-training options (:1338-1339, :1370-1376 of the reference's base_architecture): the Base checkpoints carry
    # 256-d label embeddings and a 100 x 2 codebook
    g("final_dim", 256)
    g("untie_final_proj", True)
    g("logit_temp", 0.1)
    g("target_glu", False)
    g("skip_masked", False)
    g("skip_nomask", False)
    g("label_rates", 50)
    g("sample_rate", 16000)
    g("latent_vars", 100)
    g("latent_groups", 2)
    g("latent_dim", 0)
    g("latent_temp", (2, 0.5, 0.999995))
    g("codebook_prob", 0.5)
    g("relative_position_embedding", False)
    g("encoder_max_relative_position", 160)
    g("decoder_max_relative_position", 160)
    g("feature_grad_mult", 0.1)
    g("mask_prob", 0.0)
    # waveform front end (:1337-1368), read only by the opt-in speech encoder prenet
    g("conv_pos", 128)
    g("conv_pos_groups", 16)
    g("extractor_mode", "default")
    g("conv_feature_layers", "[(512,10,5)] + [(512,3,2)] * 4 + [(512,2,2)] * 2")
    g("conv_bias", False)
    g("hubert_mask_length", 10)
    g("mask_selection", "static")
    g("mask_other", 0)
    g("no_mask_overlap", False)
    g("mask_min_space", 1)
    g("mask_channel_prob", 0.0)
    g("mask_channel_length", 10)
    g("mask_channel_selection", "static")
    g("mask_channel_other", 0)
    g("no_mask_channel_overlap", False)
    g("mask_channel_min_space", 1)
    g("use_conv_pos", False)
    g("use_sinc_pos", False)
    g("encoder_speech_prenet", "conv")


@register_model_architecture("t5_transformer", "t5_transformer_base")
def t5_transformer_base(args):  # :1385-1400
    g = lambda k, v: setattr(args, k, getattr(args, k, v))  # noqa: E731
    g("use_conv_pos", True)
    g("use_sinc_pos", True)
    g("layer_norm_first", False)
    g("relative_position_embedding", True)
    g("dropout", 0.1)
    g("activation_dropout", 0.0)
    g("attention_dropout", 0.1)
    g("encoder_layerdrop", 0.05)
    g("decoder_layerdrop", 0.05)
    g("mask_prob", 0.80)
    base_architecture(args)


@register_model_architecture("t5_transformer", "t5_transformer_large")
def t5_transformer_large(args):  # :1402-1425
    g = lambda k, v: setattr(args, k, getattr(args, k, v))  # noqa: E731
    g("decoder_normalize_before", True)
    g("layer_norm_first", True)
    g("relative_position_embedding", True)
    g("dropout", 0.0)
    g("activation_dropout", 0.0)
    g("attention_dropout", 0.0)
    g("encoder_layerdrop", 0.0)
    g("decoder_layerdrop", 0.0)
    g("encoder_embed_dim", 1024)
    g("encoder_layers", 24)
    g("decoder_layers", 6)
    g("encoder_ffn_embed_dim", 4096)
    g("encoder_attention_heads", 16)
    g("decoder_attention_heads", 16)
    g("feature_grad_mult", 1.0)
    g("extractor_mode", "layer_norm")
    g("final_dim", 768)
    g("use_conv_pos", True)
    g("use_sinc_pos", True)
    g("mask_prob", 0.80)
    base_architecture(args)


@register_model_architecture("t5_transformer", "t5_transformer_base_asr")
def t5_transformer_base_asr(args):  # :1427-1447
    g = lambda k, v: setattr(args, k, getattr(args, k, v))  # noqa: E731
    g("layer_norm_first", False)
    g("relative_position_embedding", True)
    g("dropout", 0.1)
    g("activation_dropout", 0.1)
    g("attention_dropout", 0.1)
    g("feature_grad_mult", 0.0)
    g("encoder_layerdrop", 0.1)
    g("decoder_layerdrop", 0.1)
    g("mask_prob", 0.75)
    g("mask_selection", "static")
    g("mask_channel_length", 64)
    g("mask_channel_prob", 0.5)
    g("mask_channel_selection", "static")
    g("use_conv_pos", True)
    g("use_sinc_pos", True)
    g("max_text_positions", 600)
    base_architecture(args)


def make_args(arch="t5_transformer_base_asr", **overrides):
    """Namespace with an arch preset applied (what fairseq's option parser would hand to build_model)."""
    args = Namespace(**overrides)
    {"t5_transformer": base_architecture, "t5_transformer_base": t5_transformer_base,
     "t5_transformer_large": t5_transformer_large, "t5_transformer_base_asr": t5_transformer_base_asr}[arch](args)
    return args
