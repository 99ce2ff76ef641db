"""Parity at BASELINE.json's FULL sizes (bf16 / tcgen05 product path), where the CPU oracle cannot run the whole batch:
size-independent properties of the path plus a CPU-oracle check of a few rows.

* a caption row's alpha / logits depend only on that row (image, caption, weights): the full batch must reproduce a
  run over a small subset of its rows (to bf16 rounding), and that subset is checked against the oracle (2e-2, bf16);
* every attention row of an active step sums to 1, finished steps are exactly zero;
* the backward is linear in the upstream gradient: scaling it by 2 scales every gradient by exactly 2;
* decoding is independent per image: decoding a batch equals decoding its halves, and is repeatable.
"""
import pytest
import torch

from oracle import sat_oracle as O
from test_train_forward_gpu import relerr, synth

pytestmark = pytest.mark.gpu

CONFIGS = {
    # BASELINE configs[1]: resnet50 decoder dims, batch 256
    "C2": dict(Bi=256, ncap=1, hw=(14, 14), D=512, A=128, E=256, H=512, V=6400, T=20, ragged=True),
    # BASELINE configs[2]: resnet101 dims (D=2048, H=1024), batch 512 per GPU
    "C3": dict(Bi=512, ncap=1, hw=(14, 14), D=2048, A=128, E=256, H=1024, V=6400, T=20, ragged=True),
}


def _forward(W, ann, caps, lens, backward=False, gscale=None):
    from sat_b200 import decoder
    from sat_b200.packing import PackedWeights
    pw = PackedWeights(W, dtype=torch.bfloat16, device="cuda", backward=backward)
    bld = decoder.annotations_as_bld(ann.cuda(), torch.bfloat16)
    buf = decoder.train_forward(pw, bld, caps.cuda(), lens.cuda(), 0.0, 1.0, exact=False, use_tc=True, logits_f32=False,
                                backward=backward, keep_logits=True)
    out = dict(alphas=buf.t["alphas"].clone(), logits=buf.t["logits"].permute(1, 0, 2).clone(), loss=float(buf.t["out"][0]))
    if backward:
        G, d_ann = decoder.train_backward(pw, buf, grad_loss=None if gscale is None else torch.tensor(gscale, device="cuda"))
        out["G"] = {k: v.clone() for k, v in G.items()}
        out["d_ann"] = d_ann.clone()
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("name", ["C2", "C3"])
def test_train_forward_full_size_rows_are_batch_independent(name):
    cfg = CONFIGS[name]
    W, ann, caps, lens = synth(**cfg, seed=3)
    full = _forward(W, ann, caps, lens)
    B, T = cfg["Bi"], cfg["T"]
    fl = lens.reshape(-1)
    # attention rows: sum to 1 while the caption is running, exactly zero afterwards
    s = full["alphas"].sum(-1).cpu()
    for b in range(0, B, 17):
        n = int(fl[b])
        assert float((s[b, :n] - 1).abs().max()) < 1e-5
        assert n == T or float(full["alphas"][b, n:].abs().max()) == 0.0
    # a subset of rows, run alone, reproduces its rows of the full batch (bf16 rounding only: the GEMM tile shapes, and
    # with them the accumulation order, depend on the batch size)
    idx = torch.tensor([0, 1, B // 3, B // 2, B - 2, B - 1, 5, 77])
    sub = _forward(W, ann[idx], caps[idx], lens[idx])
    assert relerr(sub["alphas"], full["alphas"][idx.cuda()]) < 2e-2          # north_star bf16 tolerance
    assert relerr(sub["logits"].float(), full["logits"][idx.cuda()].float()) < 2e-2
    # ... and that subset against the CPU oracle
    ref = O.train_loss(W, ann[idx], caps[idx], lens[idx], label_smoothing=0.0, att_gamma=1.0)
    assert relerr(sub["alphas"], ref["alphas"]) < 2e-2
    assert relerr(sub["logits"].float(), ref["logits"]) < 2e-2
    assert abs(sub["loss"] - float(ref["loss"])) < 2e-2 * abs(float(ref["loss"]))


def test_train_backward_full_size_is_linear_in_the_upstream_gradient():
    cfg = CONFIGS["C2"]
    W, ann, caps, lens = synth(**cfg, seed=4)
    one = _forward(W, ann, caps, lens, backward=True)
    two = _forward(W, ann, caps, lens, backward=True, gscale=2.0)
    assert one["loss"] == two["loss"]
    for k, g in one["G"].items():
        assert torch.isfinite(g).all(), k
        assert relerr(two["G"][k], 2.0 * g) < 1e-6, k      # power-of-two scaling: exact up to the summation order of torch reductions
    assert torch.equal(two["d_ann"].float(), 2.0 * one["d_ann"].float())


DECODE = {
    # BASELINE configs[3]: greedy, resnet50 dims, batch 1024
    "C4": dict(B=1024, hw=(14, 14), D=512, A=128, E=256, H=512, V=6400, k=1),
    # BASELINE configs[4]: beam 5, wide_resnet101_2 dims (L=256, D=2048, V=10000), batch 256
    "C5": dict(B=256, hw=(16, 16), D=2048, A=128, E=256, H=512, V=10000, k=5),
}


def _decode(W, ann, k, V, dtype=torch.bfloat16):
    from sat_b200 import decode, decoder
    fp32 = dtype == torch.float32
    dw = decode.DecodeWeights(W, dtype, torch.device("cuda"), fp32, not fp32)
    bld = decoder.annotations_as_bld(ann.cuda(), dtype)
    vocab = dict(PAD=0, UNK=V - 3, START=V - 2, END=V - 1)
    t = decode.decode_annotations(dw, bld, k, 30, 1.0, "LN", 0.5, vocab)
    return decode.assemble(t, tuple(ann.shape[2:]), return_all=False)


@pytest.mark.parametrize("name", ["C4", "C5"])
def test_decode_full_size_is_per_image_and_repeatable(name):
    c = DECODE[name]
    W = O.random_weights(c["D"], c["A"], c["E"], c["H"], c["V"], seed=5, sharpen=True)
    g = torch.Generator().manual_seed(6)
    ann = torch.randn(c["B"], c["D"], *c["hw"], generator=g)
    caps, scores, alphas, ppl = _decode(W, ann, c["k"], c["V"])
    assert len(caps) == c["B"] and all(len(x) >= 0 for x in caps)
    again = _decode(W, ann, c["k"], c["V"])
    assert again[0] == caps and again[1] == scores                       # repeatable bit for bit
    h = c["B"] // 2
    lo, hi = _decode(W, ann[:h], c["k"], c["V"]), _decode(W, ann[h:], c["k"], c["V"])
    assert lo[0] + hi[0] == caps                                         # beams of an image never see another image
    assert max(abs(a - b) for a, b in zip(lo[1] + hi[1], scores)) == 0.0
    for i in (0, h, c["B"] - 1):
        assert tuple(alphas[i].shape[1:]) == c["hw"]
        assert float((alphas[i].reshape(alphas[i].shape[0], -1).sum(-1) - 1).abs().max()) < 1e-4


def oracle_gaps(W, ann, captions, vocab, max_len=30):
    """Teacher-forces the fp32 oracle on `captions` (greedy, one per image) and returns, per image, the per-step gap in nats
    between the oracle's best admissible word and the word the caption holds (0 = the oracle would have chosen it too)."""
    out = []
    for i, toks in enumerate(captions):
        a = ann[i:i + 1]
        h, c = O.init_lstm(W, a)
        prev = torch.tensor([vocab["START"]])
        gaps = []
        seq = list(toks) + ([vocab["END"]] if len(toks) < max_len else [])     # a caption shorter than max_len ended with <END>
        for step, w in enumerate(seq):
            logit, _, h, c = O.decoder_step(W, a, prev, h, c)
            sc = torch.log_softmax(logit, dim=1)[0]
            sc[[vocab["START"], vocab["PAD"]]] = float("-inf")
            if step == 0:
                sc[[vocab["END"], vocab["UNK"]]] = float("-inf")
            gaps.append(float(sc.max() - sc[w]))
            prev = torch.tensor([w])
        out.append(gaps)
    return out


def test_beam_full_dims_fp32_tokens_match_oracle():
    """BASELINE configs[4] decoder dims (L=256, D=2048, V=10000, k=5) in fp32 on two images: token ids equal the CPU oracle."""
    c = DECODE["C5"]
    W = O.random_weights(c["D"], c["A"], c["E"], c["H"], c["V"], seed=7, sharpen=True)
    g = torch.Generator().manual_seed(8)
    ann = torch.randn(2, c["D"], *c["hw"], generator=g)
    vocab = dict(PAD=0, UNK=c["V"] - 3, START=c["V"] - 2, END=c["V"] - 1)
    ref = O.caption(W, ann, vocab, beamk=5, max_gen_length=30, rescore_method="LN")
    got = _decode(W, ann, 5, c["V"], dtype=torch.float32)
    assert got[0] == ref[0]
    assert max(abs(x - y) for x, y in zip(got[1], ref[1])) < 1e-4


def test_greedy_c4_bf16_vs_oracle_on_a_subset():
    """BASELINE configs[3] (greedy, batch 1024, bf16 tensor-core path incl. the fused vocabulary arg-max): 8 rows of the full
    batch against the fp32 CPU oracle.  bf16 token ids are not bit-exact by construction (SURVEY.md appendix D-6), so the
    stated floors are: (1) at least 6 of the 8 captions equal the oracle's token for token (measured: 7 of 8);
    (2) EVERY word the bf16 path chose is a near-tie under the oracle teacher-forced on the same prefix: its log-prob is
    within 0.05 nats of the oracle's best word (measured worst case 0.003 nats; tools/bf16_decode_agreement.py prints it);
    (3) the scores of identical captions agree to 2e-2 relative."""
    c = DECODE["C4"]
    W = O.random_weights(c["D"], c["A"], c["E"], c["H"], c["V"], seed=5, sharpen=True)
    g = torch.Generator().manual_seed(6)
    ann = torch.randn(c["B"], c["D"], *c["hw"], generator=g)
    vocab = dict(PAD=0, UNK=c["V"] - 3, START=c["V"] - 2, END=c["V"] - 1)
    caps, scores, _, _ = _decode(W, ann, 1, c["V"])
    idx = [0, 1, 2, 3, 4, 5, 511, 1023]
    sub = ann[idx]
    ref = O.caption(W, sub, vocab, beamk=1, max_gen_length=30, rescore_method="LN")
    same = [caps[i] == ref[0][j] for j, i in enumerate(idx)]
    assert sum(same) >= 6, same
    for j, i in enumerate(idx):
        if same[j]:
            assert abs(scores[i] - ref[1][j]) < 2e-2 * abs(ref[1][j])
    gaps = oracle_gaps(W, sub, [caps[i] for i in idx], vocab)
    worst = max(max(gp) for gp in gaps)
    print("greedy C4 bf16: %d/8 captions identical, worst oracle gap %.4f nats" % (sum(same), worst))
    assert worst < 0.05


def test_beam_c5_bf16_vs_oracle_on_a_subset():
    """BASELINE configs[4] (beam 5, L=256, D=2048, V=10000, batch 256, bf16): 4 images of the full batch against the fp32 CPU
    oracle.  Floor: at least 2 of the 4 best captions are identical (measured: 3 of 4), identical captions score within
    2e-2 relative, and every best caption's length-normalised score is within 0.15 of the oracle's best (a different but
    equally good hypothesis)."""
    c = DECODE["C5"]
    W = O.random_weights(c["D"], c["A"], c["E"], c["H"], c["V"], seed=5, sharpen=True)
    g = torch.Generator().manual_seed(6)
    ann = torch.randn(c["B"], c["D"], *c["hw"], generator=g)
    vocab = dict(PAD=0, UNK=c["V"] - 3, START=c["V"] - 2, END=c["V"] - 1)
    caps, scores, _, _ = _decode(W, ann, 5, c["V"])
    idx = [0, 1, 2, 255]
    ref = O.caption(W, ann[idx], vocab, beamk=5, max_gen_length=30, rescore_method="LN")
    same = [caps[i] == ref[0][j] for j, i in enumerate(idx)]
    print("beam C5 bf16: %d/4 best captions identical; score deltas %s" % (sum(same), [round(scores[i] - ref[1][j], 4) for j, i in enumerate(idx)]))
    assert sum(same) >= 2, same
    for j, i in enumerate(idx):
        if same[j]:
            assert abs(scores[i] - ref[1][j]) < 2e-2 * abs(ref[1][j])
        assert abs(scores[i] - ref[1][j]) < 0.15


def _fused_fwd_bwd(W, ann, caps, lens):
    """product path of the module: bf16, tensor cores, cross entropy fused into the vocabulary GEMM"""
    from sat_b200 import decoder
    from sat_b200.packing import PackedWeights
    pw = PackedWeights(W, dtype=torch.bfloat16, device="cuda")
    bld = decoder.annotations_as_bld(ann.cuda(), torch.bfloat16)
    buf = decoder.train_forward(pw, bld, caps.cuda(), lens.cuda(), 0.0, 1.0, exact=False, use_tc=True, backward=True, fuse_ce=True)
    assert buf.fuse_ce
    G, d_ann = decoder.train_backward(pw, buf)
    torch.cuda.synchronize()
    Bi, D, h, w = ann.shape
    return float(buf.t["out"][0]), {k: v.cpu() for k, v in G.items()}, d_ann.float().reshape(Bi, h, w, D).permute(0, 3, 1, 2).cpu()


def test_train_backward_c3_dims_vs_oracle():
    """BASELINE configs[2] decoder dims (D=2048, H=1024, L=196, V=6400, T=20) with a batch the CPU oracle can differentiate
    (12 ragged captions): loss, every parameter gradient and d_ann of the fused bf16 path against autograd of the oracle."""
    from test_train_backward_gpu import oracle_grads
    cfg = dict(CONFIGS["C3"], Bi=12)
    W, ann, caps, lens = synth(**cfg, seed=9)
    loss_ref, Gref, da_ref = oracle_grads(W, ann, caps, lens, 0.0, 1.0)
    loss, G, d_ann = _fused_fwd_bwd(W, ann, caps, lens)
    assert abs(loss - loss_ref) < 2e-2 * abs(loss_ref)
    for k, g in Gref.items():
        assert relerr(G[k], g) < 6e-2, k
    assert relerr(d_ann, da_ref) < 6e-2
