"""CPU: the callers / data formats on either side of the hot path (SURVEY.md §8 f4): BLEU / GLEU without nltk (known answers
from nltk's own docstrings), score_captions' embedding similarity against the unmodified reference, the learning-rate
schedule and warm-up of training_step / configure_optimizers against the reference, PL-format checkpoints, the caption JSON
dataset and the bucket sampler."""
import json
import os
import warnings

import numpy as np
import pytest
import torch

from oracle import ref_harness as rh

warnings.filterwarnings("ignore")

HYP1 = ['It', 'is', 'a', 'guide', 'to', 'action', 'which', 'ensures', 'that', 'the', 'military', 'always', 'obeys', 'the', 'commands', 'of',
        'the', 'party']
REF1A = ['It', 'is', 'a', 'guide', 'to', 'action', 'that', 'ensures', 'that', 'the', 'military', 'will', 'forever', 'heed', 'Party', 'commands']
REF1B = ['It', 'is', 'the', 'guiding', 'principle', 'which', 'guarantees', 'the', 'military', 'forces', 'always', 'being', 'under', 'the',
         'command', 'of', 'the', 'Party']
REF1C = ['It', 'is', 'the', 'practical', 'guide', 'for', 'the', 'army', 'always', 'to', 'heed', 'the', 'directions', 'of', 'the', 'party']
HYP2 = ['he', 'read', 'the', 'book', 'because', 'he', 'was', 'interested', 'in', 'world', 'history']
REF2A = ['he', 'was', 'interested', 'in', 'world', 'history', 'because', 'he', 'read', 'the', 'book']


def small_hparams(**over):
    hp = rh.default_hparams(encoder_arch="resnet18", encoder_dim=64, attention_dim=32, embed_dim=32, decoder_dim=64, vocab_size=128,
                            input_size=64)
    hp.update(over)
    return hp


def test_bleu_gleu_known_answers():
    """the values nltk 3.6's docstrings give for these examples (bleu_score.corpus_bleu / sentence_bleu / modified_precision,
    gleu_score.corpus_gleu)"""
    import sat_b200  # noqa: F401
    from sat_b200 import metrics as M
    assert abs(M.corpus_bleu([[REF1A, REF1B, REF1C], [REF2A]], [HYP1, HYP2]) - 0.5920778868801042) < 1e-12
    assert abs(M.sentence_bleu([REF1A, REF1B, REF1C], HYP1) - 0.5045666840058485) < 1e-12
    assert abs(M.sentence_bleu([REF2A], HYP2) - 0.7400828044922853) < 1e-12
    assert abs(M.corpus_gleu([[REF1A, REF1B, REF1C], [REF2A]], [HYP1, HYP2]) - 0.5673076923076923) < 1e-12
    assert M.modified_precision([['the', 'cat', 'is', 'on', 'the', 'mat'], ['there', 'is', 'a', 'cat', 'on', 'the', 'mat']], ['the'] * 7, 1) == (2, 7)
    assert M.corpus_bleu([[REF2A]], [[]]) == 0 and M.corpus_gleu([[[]]], [[]]) == 0.0
    assert M.closest_ref_length([[0] * 13, [0] * 11], 12) == 11                 # tie on distance: the shorter reference
    assert M.brevity_penalty(12, 13) == 1.0 and abs(M.brevity_penalty(12, 6) - np.exp(-1.0)) < 1e-15


@pytest.mark.reference
def test_score_captions_cosine_similarity_matches_reference():
    import sat_b200  # noqa: F401
    from sat_b200.model import SAT
    model_mod, _ = rh.load_reference()
    torch.manual_seed(3)
    ref = model_mod.SAT(**small_hparams())
    torch.manual_seed(3)
    m = SAT(**small_hparams())
    g = torch.Generator().manual_seed(4)
    enc = torch.randint(1, 124, (5, 3, 9), generator=g)
    enc[:, :, 0] = 126
    lens = torch.randint(2, 8, (5, 3), generator=g)
    caps = [torch.randint(1, 124, (int(n),), generator=g).tolist() for n in (3, 7, 1, 5, 4)]
    a = ref.score_captions(caps, enc, lens, [1.0, 2.0, 3.0, 4.0, 5.0])
    b = m.score_captions(caps, enc, lens, [1.0, 2.0, 3.0, 4.0, 5.0])
    assert abs(a["cosine_similarity"] - b["cosine_similarity"]) < 1e-6
    assert b["perplexity"] == 3.0 and set(a.keys()) == set(b.keys())
    assert 0 <= b["bleu4"] <= b["bleu1"] <= 1 and 0 <= b["gleu"] <= 1


def test_score_captions_cosine_similarity_matches_reference_golden():
    """the same check against the reference's result in tests/golden/reference_api.npz (oracle/make_golden.py api)"""
    import sat_b200  # noqa: F401
    from conftest import golden_arrays
    from sat_b200.model import SAT
    z = golden_arrays("reference_api")
    torch.manual_seed(3)
    m = SAT(**small_hparams())
    b = m.score_captions(*rh.score_inputs())
    assert abs(float(z["score/cosine_similarity"]) - b["cosine_similarity"]) < 1e-6
    assert sorted(b.keys()) == z["score/keys"].tolist()
    assert b["perplexity"] == 3.0
    assert 0 <= b["bleu4"] <= b["bleu1"] <= 1 and 0 <= b["gleu"] <= 1


@pytest.mark.reference
@pytest.mark.parametrize("sched", ["step", "exp", "cosine", "one_cycle", "plateau"])
def test_lr_schedule_and_warmup_match_reference(sched):
    """configure_optimizers builds the reference's scheduler; training_step's warm-up / per-batch stepping (model.py:608-617)
    and the epoch hooks (model.py:633-635) move the learning rates exactly like the reference's"""
    import sat_b200  # noqa: F401
    from sat_b200.model import SAT
    model_mod, _ = rh.load_reference()
    extra = dict(scheduler=sched, epochs=3, train_loader_len=6, lr_warmup_steps=4, cosine_iterations=5, cosine_multi=2, min_lr=1e-6,
                 accumulate=1, milestones=[1, 2], lr_gamma=0.5, plateau_patience=0, one_cycle_pct=0.3, one_cycle_div=10.0,
                 one_cycle_fdiv=100.0, encoder_finetune_after=1, momentum=0.9, nesterov=False)
    hp = small_hparams(**extra)
    ref = model_mod.SAT(**dict(hp))
    mine = SAT(**dict(hp))
    ro, mo = ref.configure_optimizers(), mine.configure_optimizers()
    ref._optimizer = ro
    assert type(ref.scheduler) is type(mine.scheduler)
    assert [pg["lr"] for pg in ro.param_groups] == [pg["lr"] for pg in mo.param_groups]
    tr = type("T", (), {"global_step": 0})()
    ref.trainer, mine.trainer = tr, tr
    lrs_r, lrs_m = [], []
    for epoch in range(3):
        for it in range(6):
            # the part of training_step after the forward (the forward itself needs the GPU library)
            if tr.global_step < ref.hparams.lr_warmup_steps:
                lr_scale = min(1, float(tr.global_step + 1) / ref.hparams.lr_warmup_steps)
                for pg, init_lr in zip(ro.param_groups, ref.opt_init_lr):
                    pg["lr"] = lr_scale * init_lr
            elif tr.global_step > 0 and type(ref.scheduler) in (torch.optim.lr_scheduler.CosineAnnealingWarmRestarts, torch.optim.lr_scheduler.OneCycleLR):
                ref.scheduler.step()
            mine._step_lr_schedule()
            ro.step(); mo.step()
            lrs_r.append([pg["lr"] for pg in ro.param_groups]); lrs_m.append([pg["lr"] for pg in mo.param_groups])
            tr.global_step += 1
        ref.current_epoch = mine.current_epoch = epoch
        ref.training_epoch_end([{"loss": 1.0}])
        mine.training_epoch_end([{"loss": 1.0}])
        if sched == "plateau":
            ref.hparams.plateau_monitor = mine.hparams.plateau_monitor = "bleu4"
            ref.hparams.save_monitor = mine.hparams.save_monitor = "bleu4"
            ref.hparams.early_stop_monitor = mine.hparams.early_stop_monitor = "bleu4"
            ref.validation_epoch_end([{"bleu4": 0.1}])
            mine.validation_epoch_end([{"bleu4": 0.1}])
    assert np.allclose(np.array(lrs_r), np.array(lrs_m), rtol=1e-12, atol=0)


@pytest.mark.parametrize("sched", ["step", "exp", "cosine", "one_cycle", "plateau"])
def test_lr_schedule_and_warmup_match_reference_golden(sched):
    """the same learning-rate trajectory check against the reference's rates in tests/golden/reference_api.npz
    (oracle/make_golden.py api: the reference's optimizer and scheduler driven like its training loop)"""
    import sat_b200  # noqa: F401
    from conftest import golden_arrays
    from sat_b200.model import SAT
    z = golden_arrays("reference_api")
    mine = SAT(**dict(small_hparams(scheduler=sched, **rh.LR_EXTRA)))
    mo = mine.configure_optimizers()
    assert type(mine.scheduler).__name__ == str(z["lr/%s/scheduler" % sched])
    assert [pg["lr"] for pg in mo.param_groups] == z["lr/%s/init" % sched].tolist()
    tr = type("T", (), {"global_step": 0})()
    mine.trainer = tr
    lrs_m = []
    for epoch in range(3):
        for it in range(6):
            mine._step_lr_schedule()
            mo.step()
            lrs_m.append([pg["lr"] for pg in mo.param_groups])
            tr.global_step += 1
        mine.current_epoch = epoch
        mine.training_epoch_end([{"loss": 1.0}])
        if sched == "plateau":
            mine.hparams.plateau_monitor = mine.hparams.save_monitor = mine.hparams.early_stop_monitor = "bleu4"
            mine.validation_epoch_end([{"bleu4": 0.1}])
    assert np.allclose(np.array(lrs_m), z["lr/%s/lrs" % sched], rtol=1e-12, atol=0)


def test_load_from_checkpoint_pl_format(tmp_path):
    import sat_b200  # noqa: F401
    from sat_b200.model import SAT
    torch.manual_seed(5)
    m = SAT(**small_hparams())
    ckpt = {"epoch": 7, "global_step": 123, "pytorch-lightning_version": "1.4.0", "state_dict": m.state_dict(),
            "hyper_parameters": dict(m.hparams)}
    path = os.path.join(tmp_path, "last.ckpt")
    torch.save(ckpt, path)
    m2 = SAT.load_from_checkpoint(path, map_location="cpu")
    assert m2.current_epoch == 7 and m2.global_step == 123
    for (k1, v1), (k2, v2) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert k1 == k2 and torch.equal(v1, v2)
    m2.freeze()
    assert not m2.training and all(not p.requires_grad for p in m2.parameters())


def test_dataset_json_and_bucket_sampler(tmp_path):
    import sat_b200  # noqa: F401
    from sat_b200.util import BucketSampler, CocoCaptionDataset
    from PIL import Image
    paths = []
    for i in range(6):
        p = os.path.join(tmp_path, "img%d.png" % i)
        Image.fromarray(np.full((8, 8, 3), 40 * i, dtype=np.uint8)).save(p)
        paths.append(p)
    stoi = {"<PAD>": 0, "a": 1, "cat": 2, "<UNK>": 3, "<START>": 4, "<END>": 5}
    caps = [[[4, 1, 2, 5, 0], [4, 2, 5, 0, 0]]] * 6
    lens = [[3, 2], [3, 3], [1, 1], [3, 2], [2, 2], [1, 1]]
    js = {"vocab_stoi": stoi, "vocab_size": 6, "train": {"samples": 6, "img_paths": paths, "encoded_captions": caps, "lengths": lens}}
    jp = os.path.join(tmp_path, "d.json")
    json.dump(js, open(jp, "w"))
    ds = CocoCaptionDataset(jp, split="train")
    img, enc, ln = ds[2]
    assert img.shape == (3, 8, 8) and abs(float(img.max()) - 80 / 255) < 1e-6 and enc.shape == (2, 5) and ln.tolist() == [1, 1]
    assert ds.stoi("dog") == 3 and ds.itos(2) == "cat" and len(ds) == 6
    np.random.seed(0)
    order = list(BucketSampler(lens, batch_size=2))
    assert sorted(order) == list(range(6))
    totals = [sum(lens[i]) for i in order]
    assert totals == sorted(totals, reverse=True)                    # longest target counts first, groups shuffled inside
    assert len(BucketSampler(lens, 2)) == 6
