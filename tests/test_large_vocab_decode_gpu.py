"""GPU: beam search and sampling at vocabulary sizes the shared-memory row kernels cannot hold (bf16 tensor-core decode).  There the
vocabulary GEMM's epilogue keeps per 128-column tile the soft-max statistics and the tile's best kcap candidates
(VOCAB_TOPK / VOCAB_SAMPLE, csrc/sat_vocab_ce.cuh) and a finalize kernel merges the tiles of each row; no [R, V] logits.

* exact selection: with a zero output weight the logits are the fp32 output bias, so planted biases fix every candidate and
  a float64 host computation gives the expected words and scores (tile boundaries, the last partial tile, exact ties, the
  special words carrying the largest biases);
* where both paths run (V = 10,000), SAT_VOCAB_TOPK=1 must reproduce the row kernels' captions;
* against the fp32 oracle at V0 = 70,001, the multinomial distribution at V0 = 40,003, the module API at V = 100,003, and
  guard bands around every buffer of the fused path."""
import json
import os
import subprocess
import sys
import warnings

import numpy as np
import pytest
import torch
from torch import nn

from oracle import ref_harness as rh
from oracle import sat_oracle as O

warnings.filterwarnings("ignore")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VOC = lambda V: dict(PAD=0, UNK=V - 3, START=V - 2, END=V - 1)


def _decode(W, ann, k, max_len, temperature=1.0, rescore=None, return_all=False, **kw):
    from sat_b200 import decode, decoder
    V = W["embedding.weight"].shape[0]
    dw = decode.DecodeWeights(W, torch.bfloat16, torch.device("cuda"), False, True)
    bld = decoder.annotations_as_bld(ann.cuda(), torch.bfloat16)
    t = decode.decode_annotations(dw, bld, k, max_len, temperature, rescore, 0.5, VOC(V), **kw)
    out = decode.assemble(t, tuple(ann.shape[2:]), return_all=return_all)
    torch.cuda.synchronize()
    return out, t


def _planted_weights(V0, bias, seed=3):
    D, A, E, H = 64, 32, 32, 64
    W = O.random_weights(D, A, E, H, V0, seed=seed)
    W["output.output.weight"].zero_()                    # logits = the fp32 output bias at every step
    W["output.output.bias"] = torch.from_numpy(bias.astype(np.float32))
    return W, torch.randn(1, D, 3, 3, generator=torch.Generator().manual_seed(seed + 1))


def _plant(V0, k, placement, seed):
    """output bias: background in [-4, 0]; <END> largest (every hypothesis ends at step 1); <START>, <PAD>, <UNK> next (masked at
    step 0, but in the log-sum-exp); k + 8 planted winners in [5, 8] placed as `placement` says"""
    rng = np.random.default_rng(seed)
    bias = rng.uniform(-4.0, 0.0, V0).astype(np.float32)
    v = VOC(V0)
    bias[v["END"]], bias[v["START"]], bias[v["PAD"]], bias[v["UNK"]] = 30.0, 28.0, 28.0, 20.0
    n = k + 8
    last0 = (V0 - 1) // 128 * 128                         # first column of the last (partial) tile
    last_words = [c for c in range(last0, V0) if c not in v.values()]
    if placement == "one_tile":
        idx = 7 * 128 + 3 + rng.choice(120, n, replace=False)
        vals = rng.uniform(5.0, 8.0, n)
    elif placement == "boundaries":
        tiles = rng.choice(np.arange(2, (V0 - 1) // 128), n, replace=False)
        idx = np.unique(np.concatenate([[1, 127, 128], last_words[:2], tiles * 128 - 1, tiles * 128]))
        vals = rng.uniform(5.0, 8.0, len(idx))
        vals[np.isin(idx, [1, 127, 128] + last_words[:2])] = 8.0 + np.arange(5) * 0.25   # these must win
    else:                                                 # "ties": a few values, each shared within and across tiles
        idx = np.concatenate([300 + rng.choice(100, n // 2, replace=False), rng.choice(np.arange(1, V0 - 3), n - n // 2, replace=False)])
        idx = np.unique(idx)
        vals = rng.choice([7.0, 6.5, 6.0], len(idx))
    bias[idx] = vals.astype(np.float32)
    bias[v["END"]], bias[v["START"]], bias[v["PAD"]], bias[v["UNK"]] = 30.0, 28.0, 28.0, 20.0
    return bias


def _expected(bias, k, T):
    """float64: the k step-0 winners (ties -> lower word) and their scores lp0(w) + lp1(<END>) (no rescoring)"""
    V0 = len(bias)
    v = VOC(V0)
    x = bias.astype(np.float32) * np.float32(1.0 / T)     # the kernel's x, exactly
    x64 = x.astype(np.float64)
    lse = x64.max() + np.log(np.exp(x64 - x64.max()).sum())
    cand = np.ones(V0, bool)
    cand[[v["START"], v["PAD"], v["END"], v["UNK"]]] = False
    words = np.flatnonzero(cand)
    order = np.lexsort((words, -x64[words]))[:k]
    win = words[order]
    return [([int(w)], float(x64[w] - lse + x64[v["END"]] - lse)) for w in win]


@pytest.mark.parametrize("V0", [58073, 131077])
@pytest.mark.parametrize("placement", ["one_tile", "boundaries", "ties"])
def test_fused_beam_selection_is_exact_with_planted_logits(V0, placement):
    for k in (3, 5, 32):
        bias = _plant(V0, k, placement, seed=V0 + k)
        W, ann = _planted_weights(V0, bias)
        for T in (1.0, 0.7):
            (caps, scores, _, _), t = _decode(W, ann, k, 4, temperature=T, return_all=True)
            assert "logits" not in t and "tile_val" in t                  # the fused path ran
            exp = _expected(bias, k, T)
            got = sorted(zip(caps[0], scores[0]), key=lambda cs: (-cs[1], cs[0]))
            exp = sorted(exp, key=lambda cs: (-cs[1], cs[0]))
            assert [c for c, _ in got] == [c for c, _ in exp], (k, T)
            for (_, s), (_, e) in zip(got, exp):
                assert abs(s - e) <= 1e-5 * abs(e), (k, T, s, e)


_CHILD = r"""
import json, sys, torch
from oracle import sat_oracle as O
sys.path.insert(0, %r)
from test_large_vocab_decode_gpu import _decode
W = O.random_weights(512, 128, 256, 512, 10000, seed=21, sharpen=True)
ann = torch.randn(64, 512, 7, 7, generator=torch.Generator().manual_seed(22))
(bc, bs, _, _), tb = _decode(W, ann, 5, 30, rescore="LN")
(mc, ms, _, _), tm = _decode(W, ann, 5, 30, rescore="LN", sample_method="multinomial", seed=77)
print(json.dumps(dict(fused="tile_val" in tb and "tile_val" in tm, beam=[bc, bs], mult=mc)))
"""


def _child(force):
    env = dict(os.environ, PYTHONPATH=ROOT)
    env.pop("SAT_VOCAB_TOPK", None)
    if force:
        env["SAT_VOCAB_TOPK"] = "1"
    r = subprocess.run([sys.executable, "-c", _CHILD % os.path.dirname(os.path.abspath(__file__))], cwd=ROOT, env=env,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_fused_candidates_match_the_row_kernels_where_both_run():
    rows, fused = _child(False), _child(True)
    assert not rows["fused"] and fused["fused"]
    assert fused["beam"][0] == rows["beam"][0]
    for a, b in zip(fused["beam"][1], rows["beam"][1]):
        assert abs(a - b) <= 1e-5 * abs(b), (a, b)
    same = sum(a == b for a, b in zip(fused["mult"], rows["mult"]))
    print("multinomial: %d/64 images draw the same caption on both paths" % same)
    assert same >= 62


def _as_packed(W, ann):
    """the operands the bf16 kernels see: every weight matrix (not attention.f_att.weight) and the annotations rounded to bf16,
    as PackedWeights / annotations_as_bld round them; biases stay fp32"""
    Wb = {n: (p.to(torch.bfloat16).float() if p.dim() == 2 and n != "attention.f_att.weight" else p) for n, p in W.items()}
    return Wb, ann.to(torch.bfloat16).float()


@pytest.mark.parametrize("k", [3, 5])
def test_fused_beam_vs_oracle_at_70001_words(k):
    """floors of test_beam_c5_bf16_vs_oracle_on_a_subset, on its decoder dims (D=2048, L=256, A=128, E=256, H=512) at V0 = 70,001:
    >= 6 of 8 best captions identical, identical captions within 2e-2 relative, every score within 0.15 of the oracle's best.
    The oracle runs on the bf16-rounded weights and annotations, so the comparison measures the decode, not the model's
    quantization: rounding the weights alone moves the fp32 oracle's own beam result (on CPU, at these dims: 2 of 16 captions
    change, scores by up to 0.05; at D=64, E=32, where every hypothesis runs to the length limit at ~-2 nats a word, by 0.36)."""
    V0 = 70001
    W = O.random_weights(2048, 128, 256, 512, V0, seed=31, sharpen=True)
    ann = torch.randn(8, 2048, 16, 16, generator=torch.Generator().manual_seed(32))
    (caps, scores, _, _), t = _decode(W, ann, k, 30, rescore="LN")
    assert "logits" not in t
    ref = O.caption(*_as_packed(W, ann), VOC(V0), beamk=k, max_gen_length=30, rescore_method="LN")
    same = [caps[i] == ref[0][i] for i in range(8)]
    print("V0=70001 k=%d: %d/8 best captions identical; score deltas %s" % (k, sum(same), [round(scores[i] - ref[1][i], 4) for i in range(8)]))
    assert sum(same) >= 6, same
    for i in range(8):
        if same[i]:
            assert abs(scores[i] - ref[1][i]) < 2e-2 * abs(ref[1][i])
        assert abs(scores[i] - ref[1][i]) < 0.15


def test_fused_topk_sampler_stays_inside_each_beams_top_candidates():
    """every chosen word is among its beam's sample_topk best under the teacher-forced fp32 oracle (a bf16 near-tie with the
    sample_topk-th word, within 0.05 nats, also counts)"""
    V0, tk = 70001, 3
    W = O.random_weights(64, 32, 32, 64, V0, seed=33, sharpen=True)
    ann = torch.randn(4, 64, 3, 3, generator=torch.Generator().manual_seed(34))
    (caps, _, _, _), t = _decode(W, ann, 3, 6, return_all=True, sample_method="topk", sample_topk=tk, seed=5)
    assert "logits" not in t
    vocab = VOC(V0)
    for n in range(ann.shape[0]):
        for cap in caps[n]:
            h, c = O.init_lstm(W, ann[n:n + 1])
            prev = torch.tensor([vocab["START"]])
            for step, w in enumerate(cap):
                logit, _, h, c = O.decoder_step(W, ann[n:n + 1], prev, h, c)
                sc = torch.log_softmax(logit, 1)[0]
                sc[[vocab["START"], vocab["PAD"]]] = float("-inf")
                if step == 0:
                    sc[[vocab["END"], vocab["UNK"]]] = float("-inf")
                top = torch.topk(sc, 3 if step == 0 else tk)              # step 0 is the beam's plain top-k (model.py:343)
                assert w in top.indices.tolist() or float(top.values[-1] - sc[w]) < 0.05, (n, step, w)
                prev = torch.tensor([w])


def test_fused_multinomial_distribution_above_the_row_kernel_limit():
    """k = 1, step 1 at V0 = 40,003 (the row sampler holds <= 29,032 words): 2048 copies of one image, planted logits; the
    histogram of the step-1 draws must match softmax(20 * log_softmax(bias)_masked) within the bound of
    test_multinomial_sampler_distribution_matches_reference_formula"""
    V0 = 40003
    v = VOC(V0)
    rng = np.random.default_rng(41)
    bias = rng.uniform(-4.0, 0.0, V0).astype(np.float32)
    planted = [5, 127, 128, 777, 12345, 30000, 39990, 40000]
    bias[planted] = 3.0 + np.arange(len(planted)) * 0.02
    w0 = 20000
    bias[w0] = 3.3
    bias[v["END"]], bias[v["START"]], bias[v["PAD"]], bias[v["UNK"]] = 3.05, 9.0, 9.0, 2.9
    W, ann1 = _planted_weights(V0, bias, seed=42)
    n = 2048
    ann = ann1.expand(n, *ann1.shape[1:]).contiguous()
    (caps, _, _, _), t = _decode(W, ann, 1, 2, sample_method="multinomial", seed=99)
    assert "logits" not in t and "tile_key" in t
    x = bias.astype(np.float64)
    lp = x - (x.max() + np.log(np.exp(x - x.max()).sum()))
    lp[[v["START"], v["PAD"]]] = -np.inf
    y = 20.0 * lp
    p = np.exp(y - y.max())
    p /= p.sum()
    counts = np.zeros(V0)
    for cap in caps:
        assert cap[0] == w0
        counts[cap[1] if len(cap) > 1 else v["END"]] += 1
    freq = counts / n
    assert float(np.abs(freq - p).max()) < 4.0 * float(np.sqrt(p * (1 - p) / n).max()) + 2e-3
    assert int((counts > 0).sum()) >= 2


def _module(precision, V=100003):
    from sat_b200.model import SAT
    torch.manual_seed(0)
    hp = rh.default_hparams(encoder_dim=64, attention_dim=32, embed_dim=32, decoder_dim=64, vocab_size=V, input_size=64,
                            precision=precision)
    m = SAT(**hp)
    m.encoder = nn.Identity()
    return m.cuda()


def _batch(V, Bi=4, ncap=3, T=7):
    g = torch.Generator().manual_seed(51)
    ann = torch.randn(Bi, 64, 4, 3, generator=g)
    caps = torch.randint(1, V - 3, (Bi, ncap, T + 1), generator=g)
    caps[:, :, 0] = V - 2
    lens = torch.randint(2, T + 1, (Bi, ncap), generator=g)
    for i in range(Bi):
        for j in range(ncap):
            caps[i, j, int(lens[i, j])] = V - 1
            caps[i, j, int(lens[i, j]) + 1:] = 0
    return ann, caps, lens


def test_module_trains_validates_and_samples_at_100003_words():
    from sat_b200 import _lib
    V = 100003
    m = _module("bf16")
    ann, caps, lens = _batch(V)
    m.train()
    out = m.training_step((ann.cuda(), caps[:, :1].contiguous().cuda(), lens[:, :1].contiguous().cuda()), 0)
    out["loss"].backward()
    assert torch.isfinite(out["loss"]) and all(torch.isfinite(p.grad).all() for p in m.parameters() if p.grad is not None)
    m.eval()
    m.hparams["val_beamk"], m.hparams["val_max_len"] = 3, 8
    vs = m.validation_step((ann.cuda(), caps.cuda(), lens.cuda()), 0)
    assert all(np.isfinite(float(vs[key])) for key in vs)
    got, scores, _, _ = m.caption(ann.cuda(), beamk=3, max_gen_length=8, sample_method="multinomial")
    assert len(got) == 4 and all(np.isfinite(s) for s in scores)
    streamed = list(m.caption_stream([ann.pin_memory()], beamk=3, max_gen_length=8, rescore_method="LN"))
    assert len(streamed) == 1 and len(streamed[0][0]) == 4
    f32 = _module("fp32")
    with pytest.raises(_lib.SatError, match="bf16 tensor-core path"):
        f32.caption(ann.cuda(), beamk=3, max_gen_length=8)


@pytest.mark.parametrize("method", ["beam", "multinomial"])
def test_fused_decode_keeps_guard_bands(method, monkeypatch):
    from sat_b200 import _redzone
    monkeypatch.setenv("SAT_REDZONE", "1")
    _redzone.violations()
    V0 = 60001
    W = O.random_weights(64, 32, 32, 64, V0, seed=61, sharpen=True)
    ann = torch.randn(3, 64, 3, 3, generator=torch.Generator().manual_seed(62))
    _, t = _decode(W, ann, 5, 10, rescore="LN", sample_method=method, seed=7)
    assert "logits" not in t and "tile_val" in t and ("tile_key" in t) == (method == "multinomial")
    assert _redzone.violations() == []
