"""GPU: scheduled-sampling training on the fused vocabulary path (bf16 tensor cores), where a sampled step t feeds back the
arg-max of step t-1 read from the VOCAB_STATS tiles of the vocabulary GEMM's epilogue (csrc/sat_train.cu, ss_feedback_kernel)
and no [T, B, V] logits exist.  The path is taken where the cross-entropy row kernel cannot hold a logits row (V > 58,072), or
everywhere under SAT_TRAIN_FUSED_SS=1.

* a module at 100,003 words trains with decoder_tf=None and "inv_sigmoid" (fp32 raises, naming the bf16 tensor-core path);
* the feedback invariant: the word fed at a sampled step is the arg-max the accuracy counts (row_argmax of the step before);
* exact arg-max with planted logits (zero output weight: the logits are the output bias), at tile boundaries, in the last
  partial tile and in exact ties;
* where both paths run (V = 10,000), the fused path feeds the same words as the logits path;
* loss, accuracy, every parameter gradient and d_ann against float64 autograd of the oracle fed the library's words;
* determinism and guard bands.
`pytest -s` prints the measured values."""
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
HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)


def _plan(T, eps=0.0, seed=0):
    """the host-side schedule of SAT._sampling_plan: steps 0..2 teacher-forced, a later step sampled when its draw exceeds eps"""
    g = torch.Generator().manual_seed(seed)
    return [0 if t <= 2 or float(torch.rand(1, generator=g)) <= eps else 1 for t in range(T)]


def _run(W, ann, caps, lens, sampled, ls=0.0, dropout=(0.0, 0.0, 0), backward=True, keep_logits=False):
    """one bf16 tensor-core training step of the decoder API; returns (buffers, packed weights)"""
    from sat_b200 import decoder
    from sat_b200.packing import PackedWeights
    pw = PackedWeights(W, dtype=torch.bfloat16, device="cuda")
    bld = decoder.annotations_as_bld(ann.cuda(), torch.bfloat16)
    buf = decoder.train_forward(pw, bld, caps.cuda(), lens.cuda(), ls, 1.0, exact=False, use_tc=True, backward=backward,
                                keep_logits=keep_logits, sampled=sampled, dropout=dropout, fuse_ce=not keep_logits)
    return buf, pw


def _feedback_violations(tok, row_argmax, caps, lens, sampled, V0):
    """tok, row_argmax [T, B]; caps [B, T+1]; lens [B] (cpu).  Every id in [0, V0); at a sampled step t every row with t < lens[b]
    is fed row_argmax[t-1, b]; at a teacher-forced step every row is fed caps[b, t].  Returns the list of violations."""
    tok, row_argmax, caps, lens = (x.cpu().long() for x in (tok, row_argmax, caps, lens))
    T, B = tok.shape
    bad = []
    if bool(((tok < 0) | (tok >= V0)).any()):
        bad.append("ids outside [0, V0)")
    for t in range(T):
        if t > 0 and sampled[t]:
            act = lens > t
            diff = (tok[t] != row_argmax[t - 1]) & act
        else:
            diff = tok[t] != caps[:, t]
        if bool(diff.any()):
            bad.append("step %d (%s): %d rows" % (t, "sampled" if t > 0 and sampled[t] else "teacher", int(diff.sum())))
    return bad


def _caps_batch(B, T, V0, g, min_len=2):
    caps = torch.randint(1, V0 - 3, (B, T + 1), generator=g)
    caps[:, 0] = V0 - 2
    lens = torch.randint(min_len, T + 1, (B,), generator=g)
    lens[-2:] = T
    for b in range(B):
        caps[b, int(lens[b]) + 1:] = 0
        if int(lens[b]) < T + 1:
            caps[b, int(lens[b])] = V0 - 1
    return caps, lens


# ---- 1. the module at 100,003 words ------------------------------------------------------------------------------------------
def _module(precision, V, **over):
    from sat_b200.model import SAT
    torch.manual_seed(0)
    hp = rh.default_hparams(encoder_dim=64, attention_dim=32, embed_dim=32, decoder_dim=64, vocab_size=V, input_size=64,
                            precision=precision, **over)
    m = SAT(**hp)
    m.encoder = nn.Identity()
    return m.cuda()


@pytest.mark.parametrize("decoder_tf", [None, "inv_sigmoid"])
def test_module_trains_with_scheduled_sampling_at_100003_words(decoder_tf, monkeypatch):
    from sat_b200 import _lib, decoder
    V, T = 100003, 12
    m = _module("bf16", V, decoder_tf=decoder_tf, decoder_tf_min=0.1, epochs=10)
    m.current_epoch = 10                                  # inv_sigmoid at the last epoch: epsilon = 0.10
    seen = []
    real = decoder.train_forward

    def spy(*a, **k):
        buf = real(*a, **k)
        seen.append((buf, k.get("sampled")))
        return buf

    monkeypatch.setattr(decoder, "train_forward", spy)
    g = torch.Generator().manual_seed(51)
    caps, lens = _caps_batch(8, T, V, g, min_len=6)
    ann = torch.randn(8, 64, 4, 3, generator=g)
    torch.manual_seed(5)
    m.train()
    out = m.training_step((ann.cuda(), caps.reshape(8, 1, -1).cuda(), lens.reshape(8, 1).cuda()), 0)
    out["loss"].backward()
    torch.cuda.synchronize()
    assert torch.isfinite(out["loss"]) and all(torch.isfinite(p.grad).all() for p in m.parameters() if p.grad is not None)
    buf, sampled = seen[-1]
    assert sampled is not None and sum(sampled) > 0, sampled
    assert buf.fuse_ce and "logits" not in buf.t                          # the fused path ran
    assert float(buf.t["out"][6]) == 0.0
    assert _feedback_violations(buf.t["tok"], buf.t["row_argmax"], caps, lens, sampled, V) == []
    f32 = _module("fp32", V, decoder_tf=decoder_tf, decoder_tf_min=0.1, epochs=10)
    f32.current_epoch = 10
    f32.train()
    with pytest.raises(_lib.SatError, match="bf16 tensor-core path"):
        f32.training_step((ann.cuda(), caps.reshape(8, 1, -1).cuda(), lens.reshape(8, 1).cuda()), 0)


# ---- 2 / 4. both paths at 10,000 words (child processes: SAT_TRAIN_FUSED_SS is read once per process) --------------------------
_CHILD = r"""
import json, sys, torch
sys.path.insert(0, %r)
from oracle import sat_oracle as O
from test_scheduled_sampling_vocab_gpu import _run, _caps_batch, _plan
V, T, Bi = 10000, 16, 64
W = O.random_weights(512, 128, 256, 512, V, seed=71, sharpen=True)
g = torch.Generator().manual_seed(72)
ann = torch.randn(Bi, 512, 7, 7, generator=g)
caps, lens = _caps_batch(Bi, T, V, g, min_len=8)
sampled = _plan(T)
buf, _ = _run(W, ann, caps, lens, sampled, backward=False, keep_logits=%r)
torch.cuda.synchronize()
rec = dict(fused=buf.fuse_ce, tok=buf.t["tok"].tolist(), row_argmax=buf.t["row_argmax"].tolist(), loss=float(buf.t["out"][0]),
           out6=float(buf.t["out"][6]), row_loss=buf.t["row_loss"].tolist(), caps=caps.tolist(), lens=lens.tolist(), sampled=sampled)
if "logits" in buf.t:
    top = buf.t["logits"].float().topk(2, dim=2).values
    rec["tie"] = (top[..., 0] == top[..., 1]).tolist()
print(json.dumps(rec))
"""


@pytest.fixture(scope="module")
def both_paths_10k():
    out = {}
    for force in (False, True):
        env = dict(os.environ, PYTHONPATH=ROOT)
        env.pop("SAT_TRAIN_FUSED_SS", None)
        if force:
            env["SAT_TRAIN_FUSED_SS"] = "1"
        r = subprocess.run([sys.executable, "-c", _CHILD % (HERE, not force)], cwd=ROOT, env=env, capture_output=True, text=True,
                           timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        out["fused" if force else "logits"] = json.loads(r.stdout.strip().splitlines()[-1])
    return out


def test_feedback_invariant_forced_fused_at_10000_words(both_paths_10k):
    f = both_paths_10k["fused"]
    assert f["fused"] and f["out6"] == 0.0
    bad = _feedback_violations(torch.tensor(f["tok"]), torch.tensor(f["row_argmax"]), torch.tensor(f["caps"]), torch.tensor(f["lens"]),
                               f["sampled"], 10000)
    assert bad == [], bad


def test_feedback_invariant_at_100003_words():
    V, T, Bi = 100003, 10, 40
    W = O.random_weights(64, 32, 32, 64, V, seed=81, sharpen=True)
    g = torch.Generator().manual_seed(82)
    ann = torch.randn(Bi, 64, 4, 4, generator=g)
    caps, lens = _caps_batch(Bi, T, V, g)
    sampled = _plan(T)
    buf, _ = _run(W, ann, caps, lens, sampled)
    torch.cuda.synchronize()
    assert buf.fuse_ce and "logits" not in buf.t and float(buf.t["out"][6]) == 0.0
    bad = _feedback_violations(buf.t["tok"], buf.t["row_argmax"], caps, lens, sampled, V)
    assert bad == [], bad


def test_fused_feedback_matches_the_logits_path_at_10000_words(both_paths_10k):
    """Walk each row's steps: while the logits path's stored bf16 logits of the step before have a unique maximum, both paths
    must feed the same word (bf16 rounding is monotonic and both add the bias to the same fp32 accumulator); after a bf16 tie
    the row is no longer compared.  The token losses of the (row, step) pairs fed identical words agree within 1e-2 relative
    (their sum; the logits path's cross entropy reads bf16 logits), and so does the loss when no row diverged.  Measured on a
    B200: 534 sampled (row, step) pairs compared, all equal; 11 of the 64 rows meet a bf16 tie, so the two losses (15.78 vs
    15.75) differ by those rows' later steps."""
    u, f = both_paths_10k["logits"], both_paths_10k["fused"]
    assert not u["fused"] and f["fused"]
    tok_u, tok_f, tie = np.array(u["tok"]), np.array(f["tok"]), np.array(u["tie"])
    lens, sampled = np.array(u["lens"]), u["sampled"]
    T, B = tok_u.shape
    rl_u, rl_f = np.array(u["row_loss"]), np.array(f["row_loss"])
    diverged, bad, compared, same_u, same_f = 0, [], 0, 0.0, 0.0
    for b in range(B):
        upto = int(lens[b])                                  # steps < upto were fed the same words on both paths
        for t in range(1, min(T, int(lens[b]))):
            if not sampled[t]:
                assert tok_u[t, b] == tok_f[t, b]
                continue
            if tie[t - 1, b]:
                diverged += 1
                upto = t
                break
            compared += 1
            if tok_u[t, b] != tok_f[t, b]:
                bad.append((b, t, int(tok_u[t, b]), int(tok_f[t, b])))
                break
        same_u += float(rl_u[:upto, b].sum())
        same_f += float(rl_f[:upto, b].sum())
    print("\n%d sampled (row, step) pairs compared; %d of %d rows diverged after a bf16 tie; loss %.6f (logits path) vs %.6f "
          "(fused); token losses before any divergence %.4f vs %.4f" % (compared, diverged, B, u["loss"], f["loss"], same_u, same_f))
    assert bad == [], bad[:10]
    assert abs(same_u - same_f) <= 1e-2 * abs(same_u)
    if diverged == 0:
        assert abs(u["loss"] - f["loss"]) <= 1e-2 * abs(u["loss"])


# ---- 3. exact arg-max with planted logits at 100,003 words --------------------------------------------------------------------
def _planted(V0, placement, seed):
    """output bias: background in [-4, 0], winners planted as `placement` says; returns (bias, expected arg-max)"""
    rng = np.random.default_rng(seed)
    bias = rng.uniform(-4.0, 0.0, V0).astype(np.float32)
    last0 = (V0 - 1) // 128 * 128                              # first column of the last (partial) tile
    if placement == "inside":
        bias[7 * 128 + 45], bias[7 * 128 + 46] = 8.0, 7.75
    elif placement == "col127":
        bias[127], bias[128] = 8.0, 7.99
    elif placement == "col128":
        bias[127], bias[128] = 7.99, 8.0
    elif placement == "last_tile":
        bias[last0 - 1], bias[V0 - 1] = 7.9, 8.0
    elif placement == "tie_in_tile":
        bias[30 * 128 + 100], bias[30 * 128 + 5], bias[90000] = 8.0, 8.0, 8.0
    else:                                                      # "tie_tiles": equal maxima in different tiles and at 127 / 128
        bias[128], bias[127], bias[V0 - 1], bias[50001] = 8.0, 8.0, 8.0, 8.0
    x = bias.astype(np.float64)
    return bias, int(np.flatnonzero(x == x.max())[0])


@pytest.mark.parametrize("placement", ["inside", "col127", "col128", "last_tile", "tie_in_tile", "tie_tiles"])
def test_feedback_is_the_exact_argmax_with_planted_logits(placement):
    V0, T, Bi = 100003, 6, 12
    bias, want = _planted(V0, placement, seed=91)
    W = O.random_weights(64, 32, 32, 64, V0, seed=92)
    W["output.output.weight"].zero_()                          # logits = the fp32 output bias at every step
    W["output.output.bias"] = torch.from_numpy(bias)
    g = torch.Generator().manual_seed(93)
    ann = torch.randn(Bi, 64, 3, 3, generator=g)
    caps, lens = _caps_batch(Bi, T, V0, g)
    sampled = [0, 1, 1, 1, 1, 1]                               # every step after the first is fed back
    buf, _ = _run(W, ann, caps, lens, sampled)
    torch.cuda.synchronize()
    assert buf.fuse_ce and "logits" not in buf.t
    tok, ra = buf.t["tok"].cpu(), buf.t["row_argmax"].cpu()
    for t in range(1, T):
        for b in range(Bi):
            if t < int(lens[b]):
                assert int(tok[t, b]) == want, (placement, t, b, int(tok[t, b]), want)
            if t - 1 < int(lens[b]):
                assert int(ra[t - 1, b]) == want
    assert _feedback_violations(tok, ra, caps, lens, sampled, V0) == []


# ---- 5. values against float64 ------------------------------------------------------------------------------------------------
VALUE_CASES = {
    # C2 dims (BASELINE configs[1]), every step after step 2 fed back
    "C2_10k": dict(Bi=256, ncap=1, hw=(14, 14), D=512, A=128, E=256, H=512, V=10000, T=20, layers=1, eps=0.0, ls=0.0, drop=None),
    "C2_100k": dict(Bi=256, ncap=1, hw=(14, 14), D=512, A=128, E=256, H=512, V=100003, T=20, layers=1, eps=0.0, ls=0.0, drop=None),
    # odd true dims (storage padded), two LSTM layers, 3 captions per image, dropout, label smoothing, half the steps sampled
    "odd_60k": dict(Bi=24, ncap=3, hw=(5, 5), D=510, A=100, E=300, H=500, V=60001, T=14, layers=2, eps=0.5, ls=0.1,
                    drop=(0.3, 0.2, 12345)),
}
# about 3x the worst values measured on a B200 at a 1000 W power limit (the values are in the docstrings of the tests); loss
# bounds the relative error of the loss and its parts
VALUE_BOUNDS = {
    "C2_10k": dict(rel=1.9e-2, frob=1.5e-2, row=2.9e-2, loss=1e-6),
    "C2_100k": dict(rel=1.8e-2, frob=1.5e-2, row=3.5e-2, loss=1e-6),
    "odd_60k": dict(rel=1.8e-2, frob=1.8e-2, row=4.4e-2, loss=1e-4),
}


def _pad8(n):
    return (n + 7) // 8 * 8


def _drop_mask(p, seed, stream, idx):
    """numpy mirror of sat_dropout_scale (csrc/sat_common.cuh) over an int64 index array"""
    with np.errstate(over="ignore"):
        x = idx.astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15) + np.uint64(seed) + np.uint64(stream << 56)
        x ^= x >> np.uint64(30)
        x *= np.uint64(0xBF58476D1CE4E5B9)
        x ^= x >> np.uint64(27)
        x *= np.uint64(0x94D049BB133111EB)
        x ^= x >> np.uint64(31)
    u = ((x >> np.uint64(32)).astype(np.uint32) >> np.uint32(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)
    return torch.from_numpy(np.where(u < np.float32(p), np.float32(0.0), np.float32(1.0) / (np.float32(1.0) - np.float32(p))))


def _masks(c, B, T):
    """the kernels' dropout multipliers in the oracle's layout (indices over the storage dims, cropped to the true dims)"""
    p, pe, seed = c["drop"]
    Ds, Es = _pad8(c["D"]), _pad8(c["E"])
    img = torch.arange(B) // c["ncap"]
    mean = _drop_mask(p, seed, 1, (img[:, None] * Ds + torch.arange(c["D"])[None]).numpy())
    row = (torch.arange(T)[None, :] * B + torch.arange(B)[:, None])                       # [B, T]: time-major row t*B + b
    idx = (row[..., None] * Es + torch.arange(c["E"])[None, None]).numpy()
    from sat_b200 import _lib
    import ctypes as C
    for i in (0, 7, 12345):                                   # the mirror agrees with the library's own
        v = _lib.lib().sat_dropout_multiplier(C.c_float(pe), C.c_uint64(seed), C.c_uint32(2), C.c_uint64(int(idx.reshape(-1)[i])))
        assert float(_drop_mask(pe, seed, 2, idx.reshape(-1)[i:i + 1])[0]) == v
    return dict(mean=mean, emb=_drop_mask(pe, seed, 2, idx), out=_drop_mask(p, seed, 3, idx))


def _reference_fed(W, ann_img, encoded_captions, lengths, label_smoothing, att_gamma, masks, feed):
    """oracle.train_loss (model.py:474-597) teacher-forced on `feed` [B, T]: the words the library fed at every step, instead of
    the captions' words or the oracle's own arg-max, so that the values compare step by step (built from the oracle's
    per-step pieces; compaction, masks and loss exactly as oracle.train_batch / train_loss)"""
    ncap = lengths.shape[1]
    ann = ann_img.repeat_interleave(ncap, dim=0)
    caps = encoded_captions.reshape(-1, encoded_captions.shape[2])
    lens = lengths.reshape(-1)
    B, T = caps.shape[0], caps.shape[1] - 1
    L, V = ann.shape[2] * ann.shape[3], W["embedding.weight"].shape[0]
    if masks is not None:
        f1 = (ann.mean((2, 3)) * masks["mean"]) @ W["init_lstm.factorize.weight"].t() + W["init_lstm.factorize.bias"]
        h, c = O._split_init(W, f1 @ W["init_lstm.init.weight"].t() + W["init_lstm.init.bias"])
    else:
        h, c = O.init_lstm(W, ann)
    h, c = h.clone(), c.clone()
    dev = ann.device
    logits = torch.zeros(B, T, V, dtype=ann.dtype, device=dev)
    alphas = torch.zeros(B, T, L, dtype=ann.dtype, device=dev)
    for step in range(T):
        act = lens > step
        if not bool(act.any()):
            break
        idx = act.nonzero().squeeze(1)
        ed = masks["emb"][idx, step] if masks is not None else None
        od = masks["out"][idx, step] if masks is not None else None
        stacked = h.dim() == 3
        logit, alpha, h2, c2 = O.decoder_step(W, ann[idx], feed[idx, step].long(), h[:, idx] if stacked else h[idx],
                                              c[:, idx] if stacked else c[idx], True, ed, od)
        alphas = alphas.index_put((idx, torch.tensor(step, device=dev)), alpha)
        logits = logits.index_put((idx, torch.tensor(step, device=dev)), logit)
        h = h.index_copy(1, idx, h2) if stacked else h.index_put((idx,), h2)
        c = c.index_copy(1, idx, c2) if stacked else c.index_put((idx,), c2)
    lp, tp = O.pack(logits, caps, lens)
    ce = O.label_smoothing_loss(lp.data, tp.data, label_smoothing)
    reg = ((1 - alphas.sum(dim=1)) ** 2).mean()
    acc = (torch.argmax(lp.data, dim=1) == tp.data).sum() / lp.data.shape[0]
    return dict(loss=ce + att_gamma * reg, ce=ce, reg=reg, acc=acc)


def _values_case(name):
    """one library step and float64 autograd of the oracle fed the library's words; prints and checks every value"""
    from sat_b200 import decoder
    from test_full_size_grads_gpu import captions, check, to_bld
    c = VALUE_CASES[name]
    B, T, V0 = c["Bi"] * c["ncap"], c["T"], c["V"]
    W = O.random_weights(c["D"], c["A"], c["E"], c["H"], V0, seed=101, layers=c["layers"])
    W["attention.f_att.weight"] *= 10
    g = torch.Generator().manual_seed(102)
    ann = torch.randn(c["Bi"], c["D"], *c["hw"], generator=g)
    caps, lens = captions(B, T, V0, g)
    sampled = _plan(T, c["eps"], seed=103)
    print("\n%s: B=%d, T=%d, V0=%d, sampled steps %s" % (name, B, T, V0, [t for t in range(T) if sampled[t]]))
    buf, pw = _run(W, ann, caps.reshape(c["Bi"], c["ncap"], -1), lens.reshape(c["Bi"], c["ncap"]), sampled, ls=c["ls"],
                   dropout=c["drop"] or (0.0, 0.0, 0))
    assert buf.fuse_ce and "logits" not in buf.t and float(buf.t["out"][6]) == 0.0
    tok = buf.t["tok"].cpu()
    assert _feedback_violations(tok, buf.t["row_argmax"], caps, lens, sampled, V0) == []
    G, d_ann = decoder.train_backward(pw, buf)
    torch.cuda.synchronize()
    out = buf.t["out"].cpu()
    stats = dict(loss=float(out[0]), ce=float(out[1]), reg=float(out[2]), acc=float(out[3]))
    ntok = float(out[5])
    dev = torch.device("cuda")
    Wd = {}
    for k, v in W.items():
        x = v.detach().to(device=dev, dtype=torch.float32)
        if x.dim() == 2 and k != "attention.f_att.weight":
            x = x.to(torch.bfloat16)
        Wd[k] = x.double().requires_grad_(True)
    a = ann.to(device=dev, dtype=torch.bfloat16).double().requires_grad_(True)
    masks = None
    if c["drop"] is not None:
        masks = {k: v.to(dev, torch.float64) for k, v in _masks(c, B, T).items()}
    r = _reference_fed(Wd, a, caps.reshape(c["Bi"], c["ncap"], -1).to(dev), lens.reshape(c["Bi"], c["ncap"]).to(dev), c["ls"], 1.0,
                       masks, tok.t().contiguous().to(dev))
    r["loss"].backward()
    ref_stats = {k: float(r[k].detach()) for k in ("loss", "ce", "reg", "acc")}
    Gref = {k: v.grad for k, v in Wd.items()}
    print("  N_tok %d: accuracy bound 4/N_tok = %.2e" % (ntok, 4.0 / ntok))
    check(name, stats, G, d_ann, {}, ref_stats, Gref, to_bld(a.grad), {}, VALUE_BOUNDS[name],
          dict(loss=VALUE_BOUNDS[name]["loss"], acc=4.0 / ntok))
    del Gref, r
    torch.cuda.empty_cache()


def test_values_vs_float64_c2_10000_words_forced_fused():
    """C2 dims, V = 10,000, epsilon = 0, fused path forced (SAT_TRAIN_FUSED_SS=1, in a child process).

    Measured on a B200 (1000 W), worst over the gradients and d_ann, rel / frob / row: 6.2e-3 / 4.9e-3 / 9.5e-3; loss parts
    1.0e-7 relative; accuracy equal (the random targets are never the arg-max: the invariant and planted tests cover it)."""
    env = dict(os.environ, PYTHONPATH=ROOT, SAT_TRAIN_FUSED_SS="1")
    code = "import sys; sys.path.insert(0, %r); import test_scheduled_sampling_vocab_gpu as m; m._values_case('C2_10k')" % HERE
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    print(r.stdout[-6000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


def test_values_vs_float64_c2_100003_words():
    """C2 dims, V = 100,003, epsilon = 0.  Measured on a B200 (1000 W): 5.9e-3 / 4.9e-3 / 1.2e-2; loss parts 2.3e-7; accuracy
    equal."""
    _values_case("C2_100k")


def test_values_vs_float64_odd_dims_two_layers_dropout_60001_words():
    """D=510, A=100, E=300, H=500 (storage padded), two LSTM layers, 3 captions per image, dropout 0.3 / embedding dropout 0.2,
    label smoothing 0.1, V = 60,001, epsilon = 0.5.  Measured on a B200 (1000 W): 5.9e-3 / 6.0e-3 / 1.5e-2; loss parts 3.0e-5
    (the doubly-stochastic term; the cross entropy 4.3e-6); accuracy equal."""
    _values_case("odd_60k")


# ---- 6 / 7. determinism and guard bands ---------------------------------------------------------------------------------------
def _small_sampled_step(V0, seed):
    from sat_b200 import decoder
    T, Bi = 9, 20
    W = O.random_weights(64, 32, 32, 64, V0, seed=seed, sharpen=True)
    g = torch.Generator().manual_seed(seed + 1)
    ann = torch.randn(Bi, 64, 4, 4, generator=g)
    caps, lens = _caps_batch(Bi, T, V0, g)
    buf, pw = _run(W, ann, caps, lens, _plan(T, 0.3, seed), ls=0.1, dropout=(0.2, 0.1, 77))
    G, d_ann = decoder.train_backward(pw, buf)
    torch.cuda.synchronize()
    assert buf.fuse_ce and "logits" not in buf.t
    return buf.t["tok"].clone(), buf.t["out"].clone(), {k: v.clone() for k, v in G.items()}, d_ann.clone()


def test_sampled_fused_steps_are_bit_reproducible():
    a, b = _small_sampled_step(100003, 111), _small_sampled_step(100003, 111)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[3], b[3])
    for k in a[2]:
        assert torch.equal(a[2][k], b[2][k]), k


def test_sampled_fused_step_keeps_guard_bands(monkeypatch):
    from sat_b200 import _redzone
    monkeypatch.setenv("SAT_REDZONE", "1")
    _redzone.violations()
    _small_sampled_step(60001, 121)
    assert _redzone.violations() == []
