"""GPU parity at BASELINE configs[0] (C1: resnet18 trunk + readme resize -> L=196, D=512, A=128, E=256, H=512, V=6400, batch 8,
20 targets, fp32) against outputs of the UNMODIFIED reference (tests/golden/c1_resnet18*.npz, oracle/make_golden.py::c1_case).
The fixture stores seeds instead of weights / images: the module's seeded default init is bit-identical to the reference's
(tests/test_model_api.py) and the inputs come from seeded CPU generators.

* decoder on the reference's own annotations (the stored trunk output): alpha / logits / loss <= 1e-5, accuracy exact,
  gradients (digests) <= 2e-5, greedy and beam-5 token ids bit-exact incl. early <END> and shrinking beams;
* the whole SAT.training_step with the real trunk on cuDNN (TF32 off): loss within 1e-4 of the reference's CPU step
  (convolution rounding differs between cuDNN and the CPU's oneDNN; the decoder itself is checked at 1e-5 above)."""
import warnings

import pytest
import torch
from torch import nn

from conftest import golden_arrays
from oracle import ref_harness as rh
from test_train_forward_gpu import relerr

warnings.filterwarnings("ignore")
pytestmark = pytest.mark.gpu

C1 = dict(D=512, A=128, E=256, H=512, V=6400, T=20, B=8, size=14, arch="resnet18")
SHARPEN = dict(wo=8.0, emb=2.0, fatt=30.0, end_bias=9.5)


def inputs(seed=1):
    g = torch.Generator().manual_seed(seed)
    V, T, B = C1["V"], C1["T"], C1["B"]
    img = torch.rand(B, 3, 224, 224, generator=g)
    caps = torch.randint(1, V - 3, (B, 1, T + 1), generator=g)
    caps[:, :, 0] = V - 2
    caps[:, :, T] = V - 1
    lens = torch.full((B, 1), T, dtype=torch.long)
    return img, caps, lens


def digest_indices(n, k=64, seed=7):
    g = torch.Generator().manual_seed(seed + n % 1000)
    return torch.randint(0, n, (k,), generator=g)


def model(seed=0, sharpen=False):
    from sat_b200.model import SAT
    torch.manual_seed(seed)
    hp = rh.default_hparams(encoder_arch=C1["arch"], encoder_dim=C1["D"], attention_dim=C1["A"], embed_dim=C1["E"], decoder_dim=C1["H"],
                            vocab_size=C1["V"], encoder_size=C1["size"])
    m = SAT(**hp)
    if sharpen:
        V = C1["V"]
        with torch.no_grad():
            m.output.output.weight *= SHARPEN["wo"]
            m.embedding.weight *= SHARPEN["emb"]
            m.attention.f_att.weight *= SHARPEN["fatt"]
            m.output.output.bias[V - 1] = SHARPEN["end_bias"]
    return m


@pytest.fixture(scope="module")
def gold():
    return golden_arrays("c1_resnet18")


def test_c1_decoder_forward_backward_on_reference_annotations(gold):
    img, caps, lens = inputs()
    m = model()
    resize = list(m.encoder)[-1]
    m.encoder = resize                                   # annotations = resize(stored trunk output), as in the generator
    m = m.cuda().train()
    ann7 = torch.from_numpy(gold["train/ann7"]).cuda().requires_grad_(True)
    lp, tp, alphas = m.train_batch((ann7, caps.cuda(), lens.cuda()), epsilon=1)
    assert relerr(alphas, gold["train/alphas"]) < 1e-5
    assert relerr(lp.data[:, ::16], gold["train/logits_sub"]) < 1e-5
    assert relerr(torch.logsumexp(lp.data, 1), gold["train/lse"]) < 1e-5
    assert torch.equal(torch.argmax(lp.data, 1).cpu(), torch.from_numpy(gold["train/argmax"]))
    loss = m.criterion(lp.data, tp.data) + m.hparams.att_gamma * ((1 - alphas.sum(dim=1)) ** 2).mean()
    assert abs(float(loss) - float(gold["train/loss"])) < 1e-5 * abs(float(gold["train/loss"]))
    loss.backward()
    for k, p in m.named_parameters():
        if k.startswith("encoder"):
            continue
        g = p.grad.reshape(-1).cpu()
        ref_norm = float(gold["grad_norm/" + k])
        assert abs(float(g.double().norm()) - ref_norm) < 2e-5 * ref_norm, k
        samp = torch.from_numpy(gold["grad_samp/" + k])
        assert float((g[digest_indices(g.numel())] - samp).abs().max()) < 2e-5 * float(g.abs().max()), k
    ga = ann7.grad.reshape(-1).cpu()
    assert abs(float(ga.double().norm()) - float(gold["grad_norm/ann7"])) < 2e-5 * float(gold["grad_norm/ann7"])
    assert float((ga[digest_indices(ga.numel())] - torch.from_numpy(gold["grad_samp/ann7"])).abs().max()) < 2e-5 * float(ga.abs().max())
    # the fused training_step path on the same annotations
    m.zero_grad()
    out = m.training_step((ann7.detach(), caps.cuda(), lens.cuda()), 0)
    assert abs(float(out["loss"]) - float(gold["train/loss"])) < 1e-5 * abs(float(gold["train/loss"]))
    assert abs(float(out["accuracy"]) - float(gold["train/acc"])) < 1e-6


def test_c1_training_step_with_the_real_trunk(gold):
    img, caps, lens = inputs()
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        m = model().cuda().train()
        ann7 = nn.Sequential(*list(m.encoder)[:-1])(img.clone().cuda())
        assert relerr(ann7, gold["train/ann7"]) < 1e-3          # cuDNN vs oneDNN convolutions through 17 conv + batch-norm layers
        m2 = model().cuda().train()
        out = m2.training_step((img.clone().cuda(), caps.cuda(), lens.cuda()), 0)
        ref = float(gold["train/loss_training_step"])
        assert abs(float(out["loss"]) - ref) < 1e-4 * abs(ref)
        out["loss"].backward()
        assert all(p.grad is not None and bool(torch.isfinite(p.grad).all()) for p in m2.parameters())
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32


@pytest.mark.parametrize("k", [1, 5])
def test_c1_decode_tokens_bit_exact_on_reference_annotations(gold, k):
    m = model(sharpen=True)
    m.encoder = list(m.encoder)[-1]
    m = m.cuda().eval()
    ann7 = torch.from_numpy(gold["decode/ann7"]).cuda()
    caps, scores, alphas, ppl = m.caption(ann7, beamk=k, max_gen_length=30, temperature=1.0, rescore_method="LN")
    lens_seen = []
    for i in range(4):
        ref_tok = gold["decode/k%d/n%d/tokens" % (k, i)].tolist()
        assert caps[i] == ref_tok, (k, i)
        ref_s = float(gold["decode/k%d/n%d/score" % (k, i)])
        assert abs(scores[i] - ref_s) < 1e-5 * max(1.0, abs(ref_s))
        assert relerr(alphas[i].sum(0), gold["decode/k%d/n%d/alpha_sum" % (k, i)]) < 1e-5
        lens_seen.append(len(caps[i]))
    assert min(lens_seen) < 30                         # the sharpened model ends captions early: <END> handling is exercised
