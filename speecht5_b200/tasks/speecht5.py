"""@register_task("speecht5"): the train_step / valid_step contract of speecht5/tasks/speecht5.py:519-571 (loss is
normalised locally by its own sample_size and the task reports sample_size 1, so data-parallel averaging is a plain
mean over ranks). Dataset loading (tasks/speecht5.py:324-517) is host I/O outside the hot path: synthetic batches with
the collater's key contract (data/text_to_speech_dataset.py:262-281) come from speecht5_b200.data."""
import torch

from ..fairseq_shim import LegacyFairseqTask, register_task
from ..models.speecht5 import T5TransformerModel, _Dict


@register_task("speecht5")
class SpeechT5Task(LegacyFairseqTask):
    def __init__(self, args, dicts=None, config=None):
        super().__init__(args)
        self.dicts = dicts if dicts is not None else {"text": _Dict(getattr(args, "vocab_size", 81))}
        self.config = config
        self.t5_task = getattr(args, "t5_task", "t2s")

    # tasks/speecht5.py:44-213: the task's command-line surface (same option names, types and defaults), so that a
    # recipe's command line parses unchanged; the dataset-side options are consumed by the host data pipeline only.
    TASK_NAME = ["s2t", "t2s", "s2s", "s2c", "pretrain"]
    _OPTIONS = (
        ("--config-yaml", dict(type=str, default="config.yaml")),
        ("--max-speech-sample-size", dict(default=None, type=int, metavar="N")),
        ("--min-speech-sample-size", dict(default=None, type=int, metavar="N")),
        ("--max-speech-positions", dict(default=4000, type=int, metavar="N")),
        ("--max-text-positions", dict(default=450, type=int, metavar="N")),
        ("--t5-task", dict(choices=TASK_NAME)),
        ("--bpe-tokenizer", dict(type=str, default=None)),
        ("--finetune-from-modules", dict(default=None)),
        ("--finetune-out-of-modules", dict(default=None)),
        ("--shorten-method", dict(default="none", choices=["none", "truncate", "random_crop"])),
        ("--shorten-data-split-list", dict(default="")),
        ("--tokens-per-sample", dict(default=512, type=int)),
        ("--sample-break-mode", dict(default="eos", type=str)),
        ("--mask", dict(default=0.3, type=float)),
        ("--mask-random", dict(default=0.1, type=float)),
        ("--insert", dict(default=0.0, type=float)),
        ("--permute", dict(default=0.0, type=float)),
        ("--rotate", dict(default=0.0, type=float)),
        ("--poisson-lambda", dict(default=3.5, type=float)),
        ("--permute-sentences", dict(default=0.0, type=float)),
        ("--mask-length", dict(default="span-poisson", type=str, choices=["subword", "word", "span-poisson"])),
        ("--replace-length", dict(default=1, type=int)),
        ("--iid-noise-target", dict(action="store_true")),
        ("--hubert-labels", dict(nargs="*", type=str, default=["km"])),
        ("--hubert-label-dir", dict(type=str, default=None)),
        ("--sample-rate", dict(default=100, type=float)),
        ("--label-rates", dict(default=-1, type=float)),
        ("--normalize", dict(action="store_true")),
        ("--enable-padding", dict(action="store_true")),
        ("--pad-audio", dict(action="store_true")),
        ("--random-crop", dict(action="store_true")),
        ("--single-target", dict(action="store_true")),
        ("--batch-ratio", dict(default=None, type=str)),
        ("--sample-ratios", dict(default=None, type=str)),
        ("--ctc-weight", dict(type=float, default=0.0)),
    )

    @classmethod
    def add_args(cls, parser):
        parser.add_argument("data", help="manifest root path")
        for flag, kw in cls._OPTIONS:
            parser.add_argument(flag, **kw)

    @classmethod
    def setup_task(cls, args, **kwargs):
        """tasks/speecht5.py:298-318: the text vocabulary is `<data>/dict.txt`, pre-training adds one HuBERT label
        vocabulary per `--hubert-labels` entry from `<hubert-label-dir>/dict.<label>.txt`; `<mask>` and `<ctc_blank>` are
        appended to the text vocabulary like the reference's constructor does (:282-286). Without a data directory (unit
        tests, synthetic benches) the length-only stand-in of `__init__` is used."""
        import os
        from ..dictionary import load_dictionary
        data = getattr(args, "data", None)
        path = os.path.join(data, "dict.txt") if data else None
        if path is None or not os.path.exists(path):
            return cls(args)
        dicts = {"text": load_dictionary(path)}
        if getattr(args, "t5_task", "t2s") == "pretrain":
            if not hasattr(args, "shuffle_instance"):
                args.shuffle_instance = False
            label_dir = getattr(args, "hubert_label_dir", None) or data
            dicts["hubert"] = [load_dictionary(os.path.join(label_dir, f"dict.{label}.txt"))
                               for label in (getattr(args, "hubert_labels", None) or ["km"])]
        task = cls(args, dicts=dicts)
        task.mask_idx = dicts["text"].add_symbol("<mask>")
        task.blank_symbol_idx = dicts["text"].add_symbol("<ctc_blank>")
        task.blank_symbol = "<ctc_blank>"
        if getattr(args, "iid_noise_target", False):  # (:289-293)
            task.uni_mask_idxs = torch.tensor([dicts["text"].add_symbol("<mask>" + str(i)) for i in range(600)])
        return task

    @property
    def target_dictionary(self):  # tasks/speecht5.py:573-579
        return self.dicts["text"]

    @property
    def source_dictionary(self):
        return None

    def build_generator(self, models, args, seq_gen_cls=None, extra_gen_cls_kwargs=None):
        """tasks/speecht5.py:599-613 (the reference hands its SequenceGenerator the task's ctc_weight). Without
        `seq_gen_cls` the generator is GreedyGenerator (beam 1 without CTC scoring; anything else raises); fairseq's
        `seq_gen_cls` is honoured: seq_gen_cls=BeamSearchGenerator builds the beam search with the same keywords."""
        from ..generator import GreedyGenerator
        kw = dict(beam_size=getattr(args, "beam", 1), max_len_a=getattr(args, "max_len_a", 0),
                  max_len_b=getattr(args, "max_len_b", 200), min_len=getattr(args, "min_len", 1),
                  normalize_scores=not getattr(args, "unnormalized", False), len_penalty=getattr(args, "lenpen", 1.0),
                  unk_penalty=getattr(args, "unkpen", 0.0), temperature=getattr(args, "temperature", 1.0),
                  ctc_weight=getattr(self.args, "ctc_weight", 0.0), blank=getattr(self, "blank_symbol_idx", None),
                  mask_idx=getattr(self, "mask_idx", None))
        kw.update(extra_gen_cls_kwargs or {})
        return (seq_gen_cls or GreedyGenerator)(models, self.target_dictionary, **kw)

    def inference_step(self, generator, models, sample, prefix_tokens=None, constraints=None):
        with torch.no_grad():  # fairseq/tasks/fairseq_task.py inference_step
            return generator.generate(models, sample, prefix_tokens=prefix_tokens, constraints=constraints)

    def generate_speech(self, models, net_input, **kwargs):
        """tasks/speecht5.py:640-646 (what scripts/generate_speech.py calls)."""
        with torch.no_grad():
            encoder_input = {k: v for k, v in net_input.items() if k not in ("prev_output_tokens", "task_name")}
            encoder_input.update(kwargs)
            return models[0].generate_speech(**encoder_input)

    def build_model(self, args):
        args.speech_odim = 80  # tasks/speecht5.py:581-597
        return T5TransformerModel.build_model(args, self)

    def train_step(self, sample, model, criterion, optimizer, update_num, ignore_grad=False):
        """tasks/speecht5.py:519-556: the loss is normalised by the criterion's own sample_size, the task reports
        sample_size 1.0 and a logging dict {task_name: criterion log, "sample_size": 1, "ntokens", "nsentences",
        "loss"} -- the shape SpeechT5Criterion.reduce_metrics consumes. Under B200Trainer (CUDA graph) the criterion
        defers its scalars (`_stats` device tensor) and the loss stays a device tensor: no host sync inside the step."""
        model.train()
        model.set_num_updates(update_num)
        loss, sample_size, logging_output = criterion(model, sample)
        if ignore_grad:
            loss = loss * 0
        loss = loss / sample_size
        if optimizer is not None:
            optimizer.backward(loss)
        else:
            loss.backward()
        agg = {"sample_size": 1}
        for k in ("ntokens", "nsentences"):
            if k in logging_output:
                agg[k] = logging_output[k]
        agg[sample["task_name"]] = logging_output
        deferred = "_stats" in logging_output
        agg["loss"] = loss.detach() if deferred else loss.detach().item()
        return agg["loss"], 1.0, agg

    def valid_step(self, sample, model, criterion):  # tasks/speecht5.py:558-571
        model.eval()
        with torch.no_grad():
            loss, sample_size, logging_output = criterion(model, sample)
            loss = loss / sample_size
            agg_loss = loss.item() if torch.is_tensor(loss) else loss
        return agg_loss, 1.0, {"sample_size": 1, sample["task_name"]: logging_output, "loss": agg_loss}
