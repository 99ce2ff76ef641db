"""CPU checks of the drop-in module surface (model.py:134-212): parameter names/shapes, seeded default
init identical to the reference (against its golden digests; live when the upstream files are present), vocabulary helpers."""
import warnings

import pytest
import torch

from oracle import ref_harness as rh

warnings.filterwarnings("ignore")


def small_hp(**over):
    return rh.default_hparams(vocab_size=400, **over)


@pytest.mark.reference
def test_state_dict_and_seeded_init_match_reference():
    from sat_b200.model import SAT
    rm, _ = rh.load_reference()
    torch.manual_seed(3)
    a = rm.SAT(**small_hp())
    torch.manual_seed(3)
    b = SAT(**small_hp())
    sa, sb = a.state_dict(), b.state_dict()
    assert list(sa.keys()) == list(sb.keys())
    for k in sa:
        assert sa[k].shape == sb[k].shape and torch.equal(sa[k], sb[k]), k
    b.load_state_dict(sa)          # a reference checkpoint loads into the new module


def test_state_dict_and_seeded_init_match_reference_golden():
    """the same check against tests/golden/reference_api.npz (oracle/make_golden.py api): keys in order, shapes, and per-tensor
    digests (norm + 64 sampled entries, exact) of the reference's seeded init"""
    from conftest import golden_arrays
    from sat_b200.model import SAT
    z = golden_arrays("reference_api")
    torch.manual_seed(3)
    sb = SAT(**small_hp()).state_dict()
    keys = z["init/keys"].tolist()
    assert list(sb.keys()) == keys
    for k in keys:
        flat = sb[k].reshape(-1)
        assert tuple(sb[k].shape) == tuple(z["init/shape/" + k].tolist()), k
        idx = torch.randint(0, flat.numel(), (64,), generator=torch.Generator().manual_seed(7 + flat.numel() % 1000))
        assert torch.equal(flat[idx], torch.from_numpy(z["init/samp/" + k])), k
        ref_norm = float(z["init/norm/" + k])
        assert abs(float(flat.double().norm()) - ref_norm) <= 1e-12 * ref_norm, k
    # a checkpoint with the reference's keys and shapes loads into the new module
    SAT(**small_hp()).load_state_dict({k: torch.zeros(tuple(z["init/shape/" + k].tolist()), dtype=sb[k].dtype) for k in keys})


def test_surface_and_helpers():
    from sat_b200 import model as M
    from sat_b200.model import SAT
    for name in ("get_encoder", "InitLSTM", "SoftAttention", "DeepOutput", "SAT"):
        assert hasattr(M, name)
    m = SAT(**small_hp(encoder_size=14))
    for attr in ("encoder", "embedding", "embedding_dropout", "init_lstm", "lstm", "attention", "beta", "output", "criterion",
                 "special_idxs", "scheduler", "opt_init_lr", "hparams"):
        assert hasattr(m, attr), attr
    for meth in ("stoi", "itos", "decode_seq", "caption", "forward", "train_batch", "training_step", "configure_optimizers"):
        assert callable(getattr(m, meth)), meth
    assert m.stoi("<PAD>") == 0 and m.stoi("nonsense") == m.stoi("<UNK>") == 397
    assert m.decode_seq([398, 5, 399], remove_special=True) == ["w5"]
    assert m.encoder(torch.rand(1, 3, 224, 224)).shape == (1, 512, 14, 14)
    assert m.hparams.encoder_dim == 512
    expected = {"embedding.weight": (400, 256), "lstm.weight_ih_l0": (2048, 768), "attention.f_att.weight": (1, 128),
                "beta.0.bias": (512,), "output.context.weight": (256, 512), "init_lstm.init.weight": (1024, 256)}
    sd = m.state_dict()
    for k, shp in expected.items():
        assert tuple(sd[k].shape) == shp
    assert float(sd["beta.0.bias"][0]) == pytest.approx(1 / 512)       # model.py:191-192


def test_label_smoothing_known_answer():
    from sat_b200.model import LabelSmoothing
    g = torch.Generator().manual_seed(0)
    x = torch.randn(20, 10, generator=g)
    y = torch.randint(0, 10, (20,), generator=g)
    assert torch.allclose(LabelSmoothing(0.0)(x, y), torch.nn.functional.cross_entropy(x, y), atol=1e-6)


def test_gate_interleave_roundtrip():
    from sat_b200.packing import deinterleave_gates, interleave_gates
    w = torch.arange(4 * 6 * 3, dtype=torch.float32).reshape(24, 3)
    p = interleave_gates(w)
    assert torch.equal(p[4 * 2 + 1], w[1 * 6 + 2])
    assert torch.equal(deinterleave_gates(p), w)


def test_precision_spellings_and_stacked_layers_surface():
    """PL's 16-bit spellings select the bf16 kernels (the fp16-AMP equivalent on B200); decoder_layers > 1 builds the reference's
    parameter set (lstm.*_l{l}, init_lstm.init of 2*layers*H rows)."""
    from sat_b200.model import SAT
    for prec, want in ((32, torch.float32), ("32-true", torch.float32), (16, torch.bfloat16), ("16-mixed", torch.bfloat16),
                       ("bf16", torch.bfloat16), ("bf16-mixed", torch.bfloat16)):
        m = SAT(**small_hp(precision=prec, encoder_arch="resnet18"))
        assert m._dtype() == want, prec
    m = SAT(**small_hp(decoder_layers=3, encoder_arch="resnet18"))
    sd = m.state_dict()
    assert sd["lstm.weight_ih_l2"].shape == (4 * 512, 512) and sd["init_lstm.init.weight"].shape == (2 * 3 * 512, 256)
    names = [n for n, _ in zip(__import__("sat_b200.packing", fromlist=["x"]).param_names(3), m.decoder_weights())]
    assert names[-4:] == ["lstm.weight_ih_l2", "lstm.weight_hh_l2", "lstm.bias_ih_l2", "lstm.bias_hh_l2"]
    with pytest.raises(NotImplementedError):
        SAT(**small_hp(decoder_layers=9, encoder_arch="resnet18"))


@pytest.mark.parametrize("arch", ["resnet18", "densenet121", "shufflenet_v2_x0_5"])
def test_encoder_boundary_swaps_keep_keys_and_cpu_results(arch):
    """bf16 mode swaps batch-norm / ReLU / max-pool modules of the third-party trunk for the cuDNN-routed ones (sat_b200/cudnn_bn.py);
    the state_dict keys stay the reference's and every swapped module falls back to the stock computation where cuDNN does not
    apply (here: CPU, fp32), bit for bit."""
    from sat_b200.model import SAT
    torch.manual_seed(0)
    a = SAT(**small_hp(encoder_arch=arch, precision="bf16"))
    torch.manual_seed(0)
    b = SAT(**small_hp(encoder_arch=arch, precision="bf16", cudnn_batchnorm=False))
    assert list(a.state_dict().keys()) == list(b.state_dict().keys())
    assert any(type(m).__name__ == "CudnnBatchNorm2d" for m in a.encoder.modules())
    assert not any(type(m).__name__ == "CudnnBatchNorm2d" for m in b.encoder.modules())
    x = torch.rand(2, 3, 224, 224)
    for mode in ("eval", "train"):
        getattr(a, mode)()
        getattr(b, mode)()
        with torch.no_grad():
            assert torch.equal(a.encoder(x.clone()), b.encoder(x.clone())), mode


def test_bf16_module_is_deepcopyable_and_picklable():
    """the encoder-boundary swaps use subclasses registered in sat_b200.cudnn_bn and module-level helper streams: copy.deepcopy and
    torch.save(model) (what PL's checkpoint / EMA / SWA utilities do) keep working"""
    import copy
    import io
    from sat_b200.model import SAT
    m = SAT(**small_hp(encoder_arch="resnet18", precision="bf16"))
    m2 = copy.deepcopy(m)
    buf = io.BytesIO()
    torch.save(m, buf)
    buf.seek(0)
    m3 = torch.load(buf, weights_only=False)
    for other in (m2, m3):
        assert list(other.state_dict().keys()) == list(m.state_dict().keys())
        assert type(other.encoder[5][0]).__name__ == "FusedBasicBlock"
