"""GPU: attention_dim from 248 to 1024 on the attention-step kernels, against float64.

The pipelined kernels are instantiated for KA = 2 / 4 / 8 column slices of 128 per lane (A <= 256 / 512 / 1024,
csrc/sat_attention_pipe.cuh); the step-by-step backward kernel for KA = 4 / 8 (csrc/sat_kernels.cuh).  Every path is run at
the dispatch boundaries (A0 = 248 .. 1024, 1021 padded to 1024 storage):
  * fp32 exact through SoftAttention (sat_attention_step_fwd, per-row kernel), L = 196 and L = 1;
  * training steps (forward + backward, the decoder API): bf16 per-row (ncap = 1) and grouped (ncap 3 / 5 / 8: the
    tensor-core box kernel at D = 512, the row-streamed one at D = 1024 / 2048, the fp32-context one at L > 256), fp32 exact;
    loss, alphas, every parameter gradient and d_ann against float64 autograd of the oracle (the checks of
    test_full_size_grads_gpu.py); ragged captions (finished rows), L = 1, ncap = 8 at L = 196 (the last 128-row box overruns
    the image), and T = 60 at A = 1024, where dP_deferred_kernel splits the columns into chunks;
  * the step-by-step backward (SAT_ATTB_MODE=0) and the plain forward (SAT_ATT_MODE=0), in child processes (both switches
    are read once per process), against float64 and against the pipelined kernels;
  * beam / greedy decode token ids against the oracle (fp32), the module API at attention_dim = 1024, the training limit
    (A0 = 1032 raises at backward, decodes) and guard bands.
`pytest -s` prints every measured value."""
import json
import os
import subprocess
import sys
import warnings

import pytest
import torch
from torch import nn

from oracle import ref_harness as rh
from oracle import sat_oracle as O
from test_decode_gpu import cuda_caption
from test_full_size_grads_gpu import captions, check, reference, run_library, to_bld

warnings.filterwarnings("ignore")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))

E, H, V = 64, 128, 500                # small trunk: the attention stage dominates the step
BOUNDS = {"bf16": dict(rel=6e-2, frob=2e-2, row=6e-2, fwd=2e-2), "fp32": dict(rel=5e-5, frob=5e-5, row=1e-4, fwd=1e-5)}
STAT_BOUNDS = {"bf16": dict(loss=5e-4, acc=2e-2), "fp32": dict(loss=1e-6, acc=1e-6)}
VOC = dict(PAD=0, UNK=V - 3, START=V - 2, END=V - 1)


def case(A, path, ncap=1, D=512, hw=(14, 14), Bi=4, T=6, seed=0):
    return dict(A=A, path=path, ncap=ncap, D=D, hw=list(hw), Bi=Bi, T=T, seed=seed)


def inputs(c):
    W = O.random_weights(c["D"], c["A"], E, H, V, seed=c["seed"])
    W["attention.f_att.weight"] *= 10          # non-uniform alpha so the softmax backward is exercised
    g = torch.Generator().manual_seed(c["seed"] + 100)
    ann = torch.randn(c["Bi"], c["D"], *c["hw"], generator=g)
    caps, lens = captions(c["Bi"] * c["ncap"], c["T"], V, g)
    return W, ann, caps.reshape(c["Bi"], c["ncap"], -1), lens.reshape(c["Bi"], c["ncap"])


def library_step(c):
    W, ann, caps, lens = inputs(c)
    stats, G, d_ann, _, alphas = run_library(W, ann, caps, lens, 0.0, c["path"])
    return stats, {k: v.cpu() for k, v in G.items()}, d_ann.cpu(), alphas.cpu()


def check_step(c, got, label=""):
    """a library step (stats, grads, d_ann, alphas) against float64 autograd of the oracle on the same inputs"""
    W, ann, caps, lens = inputs(c)
    print("\n%s%s" % (label, c))
    ref_stats, Gref, da_ref, _, alphas_ref = reference(W, ann, caps, lens, 0.0, c["path"] == "bf16", torch.device("cuda"))
    stats, G, d_ann, alphas = got
    check(label + str(c), stats, G, d_ann, dict(alphas=alphas), ref_stats, Gref, to_bld(da_ref), dict(alphas=alphas_ref),
          BOUNDS[c["path"]], STAT_BOUNDS[c["path"]])


# ---- 1. forward, fp32 exact through SoftAttention ----------------------------------------------------------------------------
ALL_A = [248, 256, 264, 384, 512, 520, 768, 1000, 1021, 1024]


@pytest.mark.parametrize("A0", ALL_A)
@pytest.mark.parametrize("hw", [(14, 14), (1, 1)])
def test_soft_attention_fp32_vs_float64(A0, hw):
    from sat_b200.model import SoftAttention
    D, Hd, B = 512, 128, 6
    args = type("Args", (), dict(encoder_dim=D, attention_dim=A0, decoder_dim=Hd))()
    torch.manual_seed(A0)
    m = SoftAttention(args)
    with torch.no_grad():
        m.f_att.weight *= 10
    g = torch.Generator().manual_seed(7)
    ann = torch.randn(B, D, *hw, generator=g)
    h = torch.randn(B, Hd, generator=g)
    W = {"attention." + k: v.double() for k, v in m.state_dict().items()}
    z_ref, a_ref = O.attention(W, ann.double(), h.double())
    z, alpha = m.cuda()(ann.cuda(), h.cuda())
    ez = float((z.double().cpu() - z_ref).abs().max() / z_ref.abs().max())
    ea = float((alpha.double().cpu().reshape(B, -1) - a_ref).abs().max() / a_ref.abs().max())
    print("A0=%d L=%d: z %.2e alpha %.2e" % (A0, hw[0] * hw[1], ez, ea))
    assert ez < 1e-5 and ea < 1e-5


# ---- 1 / 2. training steps: forward and backward of every kernel variant ----------------------------------------------------
STEP_CASES = (
    [case(A, "bf16") for A in [248, 256, 264, 384, 512, 520, 768, 1000, 1021, 1024]]                     # per-row pipe, K1b
    + [case(A, "fp32") for A in [264, 512, 520, 1024]]                                                    # exact path
    + [case(A, "bf16", ncap=n) for A in [264, 520, 1024] for n in [3, 5, 8]]                              # box tc kernel
    + [case(A, "fp32", ncap=5) for A in [520, 1024]]                                                      # grouped, fp32
    + [case(1024, "bf16", ncap=5, D=D, hw=hw) for D in [1024, 2048] for hw in [(14, 14), (16, 16)]]      # row-streamed tc
    + [case(520, "bf16", ncap=5, D=2048, hw=(16, 16)), case(1024, "bf16", ncap=5, D=512, hw=(16, 16))]
    + [case(1024, "bf16", ncap=5, hw=(18, 18))]                                                           # L > 256: fp32 context
    + [case(1024, "bf16", hw=(1, 1)), case(1024, "bf16", ncap=5, hw=(1, 1)), case(1024, "fp32", hw=(1, 1))]  # L = 1
    + [case(1024, "fp32", hw=(7, 7), T=60), case(1024, "bf16", hw=(7, 7), T=60)]                           # dP_deferred chunks
)


def _cid(c):
    return "A%d-%s-n%d-D%d-L%d-T%d" % (c["A"], c["path"], c["ncap"], c["D"], c["hw"][0] * c["hw"][1], c["T"])


@pytest.mark.parametrize("c", STEP_CASES, ids=_cid)
def test_training_step_vs_float64(c):
    check_step(c, library_step(c))


# ---- child processes: SAT_ATT_MODE / SAT_ATTB_MODE are read once per process ------------------------------------------------
_CHILD = """
import sys, json, torch
sys.path.insert(0, %r)
import test_attention_dim_gpu as M
jobs = json.loads(sys.argv[1])
torch.save([M.run_job(j) for j in jobs], sys.argv[2])
"""


def run_job(j):
    """one job of a child process: a training step ("train") or a decode ("decode": W of `case`, k, dtype)"""
    c = j["case"]
    if j["kind"] == "train":
        return library_step(c)
    W, ann, _, _ = inputs(c)
    W = O.random_weights(c["D"], c["A"], E, H, V, seed=c["seed"], sharpen=True)
    dt = torch.float32 if c["path"] == "fp32" else torch.bfloat16
    caps, scores, _, _ = cuda_caption(W, ann, j["k"], 16, 1.0, "LN", 0.5, False, dtype=dt, use_tc=dt == torch.bfloat16)
    return caps, scores


def run_child(jobs, tmp_path, tag, **env_extra):
    env = dict(os.environ, PYTHONPATH=ROOT)
    for k in ("SAT_ATT_MODE", "SAT_ATTB_MODE"):
        env.pop(k, None)
    env.update(env_extra)
    out = str(tmp_path / ("%s.pt" % tag))
    r = subprocess.run([sys.executable, "-c", _CHILD % HERE, json.dumps(jobs), out], cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=1800)
    assert r.returncode == 0, r.stderr[-4000:]
    return torch.load(out, weights_only=False)


def test_plain_backward_vs_float64(tmp_path):
    """the step-by-step backward kernel (SAT_ATTB_MODE=0), KA = 4 and 8, with the pipelined forward"""
    cs = [case(1024, "bf16"), case(1024, "fp32"), case(520, "bf16", ncap=5), case(768, "fp32", ncap=3),
          case(1024, "fp32", hw=(7, 7), T=60)]
    res = run_child([dict(kind="train", case=c) for c in cs], tmp_path, "plain_bwd", SAT_ATTB_MODE="0")
    for c, got in zip(cs, res):
        check_step(c, got, "plain backward ")


def _same_caption_rule(caps, scores, ref_caps, ref_scores, label):
    """as test_full_size_gpu.py compares bf16 against fp32: at least half the best captions identical, identical captions
    score within 2e-2 relative, every length-normalised score within 0.15 of the reference's best"""
    same = [a == b for a, b in zip(caps, ref_caps)]
    print("%s: %d/%d best captions identical" % (label, sum(same), len(same)))
    assert 2 * sum(same) >= len(same), same
    for s, r, sm in zip(scores, ref_scores, same):
        if sm:
            assert abs(s - r) < 2e-2 * abs(r)
        assert abs(s - r) < 0.15


@pytest.mark.parametrize("A0", [384, 512])
def test_pipelined_against_plain_kernels(A0, tmp_path):
    """256 < A <= 512, where the pipelined kernels replace the plain ones: the same seeded inputs in a child process with the
    pipelined kernels and in one with SAT_ATT_MODE=0 SAT_ATTB_MODE=0.  fp32 greedy and beam-5 token ids are identical;
    bf16 training steps are each within the bf16 bounds of float64; bf16 beam captions against the fp32 ones."""
    cd = case(A0, "fp32", Bi=6, seed=3)
    cb = dict(cd, path="bf16")
    jobs = [dict(kind="decode", case=cd, k=1), dict(kind="decode", case=cd, k=5), dict(kind="decode", case=cb, k=5),
            dict(kind="train", case=case(A0, "bf16")), dict(kind="train", case=case(A0, "bf16", ncap=5))]
    new = run_child(jobs, tmp_path, "pipe")
    old = run_child(jobs, tmp_path, "plain", SAT_ATT_MODE="0", SAT_ATTB_MODE="0")
    for i in (0, 1):
        assert new[i][0] == old[i][0], "fp32 k=%d token ids differ" % jobs[i]["k"]
    for r, label in ((new, "pipelined"), (old, "plain")):
        _same_caption_rule(r[2][0], r[2][1], new[1][0], new[1][1], "A0=%d bf16 beam-5 (%s) vs fp32" % (A0, label))
        for j in (3, 4):
            check_step(jobs[j]["case"], r[j], label + " ")


# ---- decode against the oracle ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("A0", [264, 520, 1024])
@pytest.mark.parametrize("k", [1, 5])
def test_decode_fp32_vs_oracle(A0, k):
    """fp32 parity mode: token ids bit-identical to the CPU oracle, scores within 1e-4"""
    c = case(A0, "fp32", Bi=5, seed=4)
    W = O.random_weights(c["D"], A0, E, H, V, seed=4, sharpen=True)
    _, ann, _, _ = inputs(c)
    ref = O.caption(W, ann, VOC, beamk=k, max_gen_length=16, rescore_method="LN")
    got = cuda_caption(W, ann, k, 16, 1.0, "LN", 0.5, False)
    assert got[0] == ref[0]
    assert max(abs(x - y) for x, y in zip(got[1], ref[1])) < 1e-4


@pytest.mark.parametrize("D,hw", [(512, (14, 14)), (2048, (16, 16))])
def test_beam_bf16_vs_fp32(D, hw):
    """bf16 beam 5 at attention_dim 1024 (grouped tensor-core kernels) against the fp32 decode of the same weights"""
    c = case(1024, "fp32", D=D, hw=hw, Bi=6, seed=5)
    W = O.random_weights(D, 1024, E, H, V, seed=5, sharpen=True)
    _, ann, _, _ = inputs(c)
    ref = cuda_caption(W, ann, 5, 16, 1.0, "LN", 0.5, False)
    got = cuda_caption(W, ann, 5, 16, 1.0, "LN", 0.5, False, dtype=torch.bfloat16, use_tc=True)
    _same_caption_rule(got[0], got[1], ref[0], ref[1], "D=%d bf16 beam-5" % D)


# ---- 4. module level ------------------------------------------------------------------------------------------------------------
def _module(A0, precision, seed=0):
    from sat_b200.model import SAT
    torch.manual_seed(seed)
    hp = rh.default_hparams(encoder_dim=256, attention_dim=A0, embed_dim=E, decoder_dim=H, vocab_size=V, input_size=64,
                            precision=precision, cudnn_batchnorm=False)
    m = SAT(**hp)
    m.encoder = nn.Identity()
    with torch.no_grad():
        m.attention.f_att.weight *= 6
    return m.cuda()


def _batch(seed, Bi=4, ncap=3, T=7, D=256, hw=(7, 7)):
    g = torch.Generator().manual_seed(seed)
    ann = torch.randn(Bi, D, *hw, generator=g)
    caps = torch.randint(1, V - 3, (Bi, ncap, T + 2), generator=g)
    caps[:, :, 0] = V - 2
    lens = torch.randint(2, T + 1, (Bi, ncap), generator=g)
    for i in range(Bi):
        for j in range(ncap):
            caps[i, j, int(lens[i, j])] = V - 1
            caps[i, j, int(lens[i, j]) + 1:] = 0
    return ann.cuda(), caps.cuda(), lens.cuda()


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_module_at_attention_dim_1024(precision):
    """SAT(attention_dim=1024): training_step + backward + Adam (finite gradients, the loss moves), validation_step, caption
    with beam / multinomial / topk, caption_stream (the same captions as caption)"""
    m = _module(1024, precision).train()
    ann, caps, lens = _batch(1)
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    losses = []
    for step in range(2):
        out = m.training_step((ann, caps, lens), step)
        opt.zero_grad()
        out["loss"].backward()
        assert all(p.grad is None or bool(torch.isfinite(p.grad).all()) for p in m.parameters())
        assert m.attention.encoder_att.weight.grad.abs().max() > 0
        opt.step()
        losses.append(float(out["loss"].detach()))
    print("%s losses %s" % (precision, losses))
    assert all(x == x for x in losses) and losses[1] != losses[0]
    m.eval()
    m.hparams["val_beamk"], m.hparams["val_max_len"] = 3, 8
    vs = m.validation_step((ann, caps, lens), 0)
    assert "bleu4" in vs
    for method in ("beam", "multinomial", "topk"):
        c, s, _, _ = m.caption(ann, beamk=3, max_gen_length=8, sample_method=method)
        assert len(c) == ann.shape[0] and all(all(0 <= w < V for w in cc) for cc in c), method
    batches = [_batch(10 + i)[0].cpu().pin_memory() for i in range(2)]
    got = list(m.caption_stream(batches, beamk=3, max_gen_length=8, rescore_method="LN"))
    for b, out in zip(batches, got):
        ref = m.caption(b.cuda(), beamk=3, max_gen_length=8, rescore_method="LN")
        assert out[0] == ref[0]


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_attention_dim_above_the_training_limit(precision):
    """A0 = 1032 (storage 1040): the forward runs, backward raises naming the 1024 limit, decoding still works"""
    from sat_b200._lib import SatError
    m = _module(1032, precision).train()
    ann, caps, lens = _batch(2)
    out = m.training_step((ann, caps, lens), 0)
    assert bool(torch.isfinite(out["loss"]))
    with pytest.raises(SatError, match="1024"):
        out["loss"].backward()
    m.eval()
    c, _, _, _ = m.caption(ann, beamk=3, max_gen_length=8)
    assert len(c) == ann.shape[0]


# ---- 5. guard bands -------------------------------------------------------------------------------------------------------------
def test_guard_bands_at_attention_dim_1024(monkeypatch):
    from sat_b200 import _redzone
    monkeypatch.setenv("SAT_REDZONE", "1")
    _redzone.violations()
    library_step(case(1024, "bf16", ncap=5))
    library_step(case(1024, "bf16"))
    c = case(1024, "bf16", Bi=3)
    W = O.random_weights(c["D"], 1024, E, H, V, seed=0, sharpen=True)
    _, ann, _, _ = inputs(c)
    cuda_caption(W, ann, 5, 8, 1.0, "LN", 0.5, False, dtype=torch.bfloat16, use_tc=True)
    torch.cuda.synchronize()
    assert _redzone.violations() == []
