"""Pins oracle/sat_oracle.py against outputs of the unmodified reference (tests/golden/*.npz,
made by oracle/make_golden.py from the upstream model.py).  CPU only."""
import numpy as np
import pytest
import torch

from oracle import sat_oracle as O
from conftest import load_golden


def relerr(a, b):
    a = torch.as_tensor(a, dtype=torch.float64)
    b = torch.as_tensor(b, dtype=torch.float64)
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


VOC = lambda V: dict(PAD=0, UNK=V - 3, START=V - 2, END=V - 1)


@pytest.mark.parametrize("name", ["train_tiny", "train_small", "train_ragged", "train_layers2", "train_layers3"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_train_forward_loss_and_grads(name, dtype):
    z, W, G = load_golden(name)
    W = {k: v.to(dtype).requires_grad_(True) for k, v in W.items()}
    ann = torch.from_numpy(z["ann"]).to(dtype).requires_grad_(True)
    caps, lengths = torch.from_numpy(z["caps"]), torch.from_numpy(z["lengths"])
    r = O.train_loss(W, ann, caps, lengths, float(z["label_smoothing"]), float(z["att_gamma"]))
    assert relerr(r["logits"], z["logits"]) < 2e-6
    assert relerr(r["alphas"], z["alphas"]) < 2e-6
    assert relerr(r["logits_packed"].data, z["logits_packed"]) < 2e-6
    assert torch.equal(r["targets_packed"].data, torch.from_numpy(z["targets_packed"]))
    assert abs(float(r["loss"]) - float(z["loss"])) < 2e-6 * abs(float(z["loss"]))
    assert abs(float(r["acc"]) - float(z["acc"])) < 1e-7
    r["loss"].backward()
    for k, g in G.items():
        assert relerr(W[k].grad, g) < 5e-6, k
    assert relerr(ann.grad, z["d_ann"]) < 5e-6


def test_label_smoothing_zero_is_cross_entropy():
    # the reference's only implied known answer: dev/dev_label_smoothing.py:18-23
    g = torch.Generator().manual_seed(0)
    x = torch.randn(20, 10, generator=g)
    y = torch.randint(0, 10, (20,), generator=g)
    assert torch.allclose(O.label_smoothing_loss(x, y, 0.0), torch.nn.functional.cross_entropy(x, y), atol=1e-6)


@pytest.mark.parametrize("name", ["decode_tiny", "decode_small", "decode_layers2"])
@pytest.mark.parametrize("k", [1, 3, 5])
@pytest.mark.parametrize("rescore", [None, "LN", "WR", "BAR"])
@pytest.mark.parametrize("return_all", [False, True])
def test_decode_tokens_scores_alphas(name, k, rescore, return_all):
    z, W, _ = load_golden(name)
    V = int(z["dims"][4])
    max_len = int(z["dims"][5])
    ann = torch.from_numpy(z["ann"])
    caps, scores, alphas, ppl = O.caption(W, ann, VOC(V), beamk=k, max_gen_length=max_len, temperature=1.0,
                                          rescore_method=rescore, rescore_reward=0.5, return_all=return_all)
    tag = "k%d_%s_%s" % (k, rescore, "all" if return_all else "best")
    for i in range(ann.shape[0]):
        cc, ss, aa, pp = (caps[i], scores[i], alphas[i], ppl[i]) if return_all else ([caps[i]], [scores[i]], [alphas[i]], [ppl[i]])
        assert len(cc) == int(z["%s/n%d/count" % (tag, i)])
        for j in range(len(cc)):
            assert cc[j] == z["%s/n%d/h%d/tokens" % (tag, i, j)].tolist()          # bit-exact ids
            assert abs(ss[j] - float(z["%s/n%d/h%d/score" % (tag, i, j)])) < 1e-4
            assert abs(pp[j] - float(z["%s/n%d/h%d/ppl" % (tag, i, j)])) < 1e-4 * max(1.0, pp[j])
            assert relerr(aa[j], z["%s/n%d/h%d/alphas" % (tag, i, j)]) < 1e-5


def test_decode_temperature():
    z, W, _ = load_golden("decode_small")
    V = int(z["dims"][4])
    ann = torch.from_numpy(z["ann"])
    caps, scores, _, _ = O.caption(W, ann, VOC(V), beamk=3, max_gen_length=int(z["dims"][5]), temperature=0.7,
                                   rescore_method="LN")
    for i in range(ann.shape[0]):
        assert caps[i] == z["k3_LN_T0.7/n%d/tokens" % i].tolist()
        assert abs(scores[i] - float(z["k3_LN_T0.7/n%d/score" % i])) < 1e-4
