"""Test infrastructure only: load the UNMODIFIED reference (the upstream model.py / util.py, from
SAT_REFERENCE_DIR or oracle/_ref/) so golden vectors can be generated from it.

The reference imports `pytorch_lightning` and `nltk` at module import time
(model.py:1-4, util.py:7-8); neither is installed in this image, so tiny stand-in
modules are injected into sys.modules first.  Nothing here is used by the product
path; `oracle/make_golden.py` (run by hand), bench.py's reference arm and the CPU tests import
this file (the tests for its shared inputs; only the `reference`-marked ones load the reference).
"""
import inspect
import os
import sys
import types

import torch
from torch import nn

_HERE = os.path.dirname(os.path.abspath(__file__))
# The repository does not contain the reference.  SAT_REFERENCE_DIR names a checkout of it; __graft_entry__.build() copies
# that checkout's model.py / util.py UNMODIFIED into the git-ignored oracle/_ref/, which travels with the built tree, so that
# bench.py's `--impl reference` arm can time the real reference there.  Nothing under oracle/_ref is ever committed.
_CANDIDATES = [os.environ.get("SAT_REFERENCE_DIR", ""), os.path.join(_HERE, "_ref")]
REFERENCE_DIR = next((d for d in _CANDIDATES if d and os.path.isfile(os.path.join(d, "model.py"))), os.path.join(_HERE, "_ref"))


class _HParams(dict):
    """attribute-style dict; get_encoder assigns args.encoder_dim (model.py:56)."""

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:
            raise AttributeError(k) from e

    def __setattr__(self, k, v):
        self[k] = v


class _NullExperiment:
    def add_scalar(self, *a, **k):
        pass


class _NullLogger:
    experiment = _NullExperiment()


class _NullTrainer:
    global_step = 0


class _LightningModule(nn.Module):
    """what the reference's SAT needs from pl.LightningModule (SURVEY.md §8c): hparams capture, device, and -- for
    training_step / the epoch hooks -- logger, trainer, optimizers(), log(), current_epoch, global_step."""
    current_epoch = 0
    global_step = 0
    logger = _NullLogger()
    trainer = _NullTrainer()

    def save_hyperparameters(self):
        frame = inspect.currentframe().f_back
        kwargs = frame.f_locals.get("kwargs", {})
        object.__setattr__(self, "_hparams", _HParams(kwargs))

    def optimizers(self):
        return getattr(self, "_optimizer", None)

    def log(self, *a, **k):
        pass

    @property
    def hparams(self):
        return self._hparams

    @property
    def device(self):
        try:
            return next(self.parameters()).device
        except StopIteration:
            return torch.device("cpu")


def available():
    return os.path.isfile(os.path.join(REFERENCE_DIR, "model.py"))


def load_reference():
    """Returns (model_module, util_module) of the unmodified reference."""
    if not available():
        raise RuntimeError("reference tree not present at %s" % REFERENCE_DIR)
    if "pytorch_lightning" not in sys.modules:
        pl = types.ModuleType("pytorch_lightning")
        pl.LightningModule = _LightningModule
        pl.Trainer = type("Trainer", (), {})
        cb = types.ModuleType("pytorch_lightning.callbacks")
        cb.ModelCheckpoint = type("ModelCheckpoint", (), {"__init__": lambda self, *a, **k: None})
        pl.callbacks = cb
        sys.modules["pytorch_lightning"] = pl
        sys.modules["pytorch_lightning.callbacks"] = cb
    if "nltk" not in sys.modules:
        nltk = types.ModuleType("nltk")
        tr = types.ModuleType("nltk.translate")
        bl = types.ModuleType("nltk.translate.bleu_score")
        gl = types.ModuleType("nltk.translate.gleu_score")
        bl.corpus_bleu = lambda *a, **k: 0.0
        gl.corpus_gleu = lambda *a, **k: 0.0
        nltk.translate = tr
        tr.bleu_score = bl
        tr.gleu_score = gl
        for name, m in (("nltk", nltk), ("nltk.translate", tr),
                        ("nltk.translate.bleu_score", bl), ("nltk.translate.gleu_score", gl)):
            sys.modules[name] = m
    # the reference's files are named model.py / util.py; import them under private
    # names so they never shadow anything of ours.
    import importlib.util
    saved = {k: sys.modules.get(k) for k in ("model", "util")}
    sys.path.insert(0, REFERENCE_DIR)
    try:
        for k in ("model", "util"):
            sys.modules.pop(k, None)
        spec_u = importlib.util.spec_from_file_location("util", os.path.join(REFERENCE_DIR, "util.py"))
        util = importlib.util.module_from_spec(spec_u)
        sys.modules["util"] = util
        spec_u.loader.exec_module(util)
        spec_m = importlib.util.spec_from_file_location("model", os.path.join(REFERENCE_DIR, "model.py"))
        model = importlib.util.module_from_spec(spec_m)
        sys.modules["model"] = model
        spec_m.loader.exec_module(model)
    finally:
        sys.path.remove(REFERENCE_DIR)
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return model, util


def make_vocab(vocab_size):
    """<PAD>=0, words 1..V-4, <UNK>=V-3, <START>=V-2, <END>=V-1 (preprocess.ipynb cell 15 ordering)."""
    stoi = {"<PAD>": 0}
    for i in range(1, vocab_size - 3):
        stoi["w%d" % i] = i
    stoi["<UNK>"] = vocab_size - 3
    stoi["<START>"] = vocab_size - 2
    stoi["<END>"] = vocab_size - 1
    itos = {v: k for k, v in stoi.items()}
    return stoi, itos


def default_hparams(**over):
    hp = dict(encoder_arch="resnet18", pretrained=False, input_size=224, encoder_dim=512,
              mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225], embed_dim=256, embed_norm=None,
              attention_dim=128, decoder_dim=512, decoder_layers=1, dropout=0.0, embedding_dropout=0.0,
              label_smoothing=0.0, weight_tying=False, deep_output=True, vocab_size=6400,
              pretrained_embedding=None, att_gamma=1.0, decoder_tf="always",
              # read by training_step / configure_optimizers (model.py:608-617,720-817)
              lr_warmup_steps=0, scheduler=None, opt="adam", adam_b1=0.9, adam_b2=0.999, decoder_lr=4e-4, embedding_lr=4e-4,
              encoder_lr=1e-4, weight_decay=0.0, encoder_finetune_after=-1)
    hp.update(over)
    stoi, itos = make_vocab(hp["vocab_size"])
    hp.setdefault("vocab_stoi", stoi)
    hp.setdefault("vocab_itos", itos)
    return hp


# inputs shared by oracle/make_golden.py api_case and the tests that read its golden file (tests/test_callers_cpu.py)
LR_SCHEDULERS = ["step", "exp", "cosine", "one_cycle", "plateau"]
LR_EXTRA = dict(epochs=3, train_loader_len=6, lr_warmup_steps=4, cosine_iterations=5, cosine_multi=2, min_lr=1e-6, accumulate=1,
                milestones=[1, 2], lr_gamma=0.5, plateau_patience=0, one_cycle_pct=0.3, one_cycle_div=10.0, one_cycle_fdiv=100.0,
                encoder_finetune_after=1, momentum=0.9, nesterov=False)


def small_hparams(**over):
    hp = default_hparams(encoder_arch="resnet18", encoder_dim=64, attention_dim=32, embed_dim=32, decoder_dim=64, vocab_size=128,
                         input_size=64)
    hp.update(over)
    return hp


def score_inputs():
    """(captions, encoded captions, lengths, perplexities) arguments of SAT.score_captions"""
    g = torch.Generator().manual_seed(4)
    enc = torch.randint(1, 124, (5, 3, 9), generator=g)
    enc[:, :, 0] = 126
    lens = torch.randint(2, 8, (5, 3), generator=g)
    caps = [torch.randint(1, 124, (int(n),), generator=g).tolist() for n in (3, 7, 1, 5, 4)]
    return caps, enc, lens, [1.0, 2.0, 3.0, 4.0, 5.0]
