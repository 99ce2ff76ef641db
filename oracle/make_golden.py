"""Generate tests/golden/*.npz from the UNMODIFIED reference (run by hand: `python oracle/make_golden.py [c1|layers|api]`).
Test infrastructure only; needs the upstream model.py / util.py (SAT_REFERENCE_DIR or oracle/_ref/, see ref_harness.py), which
the repository does not contain -- the committed .npz files are what the tests read.

Every case drives the reference's own public methods (SAT.train_batch, SAT.criterion, the
doubly-stochastic term exactly as training_step writes it, SAT.caption) with the CNN trunk replaced
by nn.Identity() so that the "image" tensor IS the annotation tensor [B,D,h,w]; decoder weights
are the reference's own default init under the stated seed (plus the stated sharpening).
"""
import os
import sys
import warnings

import numpy as np
import torch
from torch import nn

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import ref_harness as rh  # noqa: E402

warnings.filterwarnings("ignore")
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
# cases larger than 1 MB in one file: the arrays under the prefix go to <name>.<part>.npz (tests/conftest.py:golden_arrays
# reads both)
SPLIT = {"train_layers3": ("grads", "G/"), "c1_resnet18": ("decode", "decode/")}


def save(name, out):
    part, prefix = SPLIT.get(name, (None, None))
    if part is None:
        np.savez_compressed(os.path.join(OUT, name + ".npz"), **out)
        return
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **{k: v for k, v in out.items() if not k.startswith(prefix)})
    np.savez_compressed(os.path.join(OUT, "%s.%s.npz" % (name, part)), **{k: v for k, v in out.items() if k.startswith(prefix)})


def build(model, seed, D, A, E, H, V, label_smoothing=0.0, att_gamma=1.0, sharpen=None, layers=1):
    torch.manual_seed(seed)
    hp = rh.default_hparams(encoder_dim=D, attention_dim=A, embed_dim=E, decoder_dim=H, vocab_size=V,
                            label_smoothing=label_smoothing, att_gamma=att_gamma, input_size=64, decoder_layers=layers)
    m = model.SAT(**hp)
    m.encoder = nn.Identity()
    if sharpen:
        with torch.no_grad():
            m.output.output.weight *= sharpen.get("wo", 1.0)
            m.embedding.weight *= sharpen.get("emb", 1.0)
            m.attention.f_att.weight *= sharpen.get("fatt", 1.0)
            if "end_bias" in sharpen:
                m.output.output.bias[V - 1] = sharpen["end_bias"]
    return m


def weights_of(m):
    return {"W/" + k: v.detach().numpy().copy() for k, v in m.state_dict().items() if not k.startswith("encoder")}


def train_case(model, name, seed, B_img, ncap, hw, D, A, E, H, V, T, ragged, label_smoothing, sharpen=None, layers=1):
    m = build(model, seed, D, A, E, H, V, label_smoothing, 1.0, sharpen, layers)
    g = torch.Generator().manual_seed(seed + 1)
    ann = torch.randn(B_img, D, hw[0], hw[1], generator=g)
    ann.requires_grad_(True)
    caps = torch.randint(1, V - 3, (B_img, ncap, T + 1), generator=g)
    caps[:, :, 0] = V - 2
    if ragged:
        lengths = torch.randint(2, T + 1, (B_img, ncap), generator=g)
    else:
        lengths = torch.full((B_img, ncap), T)
    for i in range(B_img):
        for j in range(ncap):
            n = int(lengths[i, j])
            caps[i, j, n] = V - 1            # <END> is the last target
            caps[i, j, n + 1:] = 0           # <PAD>
    m.train()
    lp, tp, alphas = m.train_batch([ann, caps, lengths], torch.tensor(1))
    ce = m.criterion(lp.data, tp.data)
    loss = ce + m.hparams.att_gamma * ((1 - alphas.sum(dim=1)) ** 2).mean()      # model.py:592-594
    pred = torch.argmax(lp.data, dim=1)
    acc = torch.sum(pred == tp.data) / pred.shape[0]
    loss.backward()
    out = weights_of(m)
    for k, p in m.named_parameters():
        if not k.startswith("encoder") and p.grad is not None:
            out["G/" + k] = p.grad.numpy().copy()
    padded = torch.zeros(B_img * ncap, T, V)
    # unpack to padded [B,T,V] for convenience (time-major packed data is also stored)
    from torch.nn.utils.rnn import pad_packed_sequence
    padded, _ = pad_packed_sequence(lp, batch_first=True, total_length=T)
    out.update(dict(ann=ann.detach().numpy(), caps=caps.numpy(), lengths=lengths.numpy(),
                    logits_packed=lp.data.detach().numpy(), targets_packed=tp.data.numpy(),
                    logits=padded.detach().numpy(), alphas=alphas.detach().numpy(),
                    loss=np.float64(loss.item()), ce=np.float64(ce.item()), acc=np.float64(acc.item()),
                    d_ann=ann.grad.numpy().copy(), label_smoothing=np.float64(label_smoothing),
                    att_gamma=np.float64(1.0), dims=np.array([D, A, E, H, V, T, hw[0], hw[1], ncap])))
    save(name, out)
    print(name, "loss", loss.item(), "acc", acc.item(), "tokens", lp.data.shape[0])


def decode_case(model, name, seed, n_img, hw, D, A, E, H, V, max_len, sharpen, layers=1):
    m = build(model, seed, D, A, E, H, V, 0.0, 1.0, sharpen, layers)
    g = torch.Generator().manual_seed(seed + 1)
    ann = torch.randn(n_img, D, hw[0], hw[1], generator=g)
    out = weights_of(m)
    out["ann"] = ann.numpy()
    out["dims"] = np.array([D, A, E, H, V, max_len, hw[0], hw[1]])
    lens = {}
    for k in (1, 3, 5):
        for rs in (None, "LN", "WR", "BAR"):
            for ra in (False, True):
                caps, scores, alphas, ppl = m.caption(ann.clone(), beamk=k, max_gen_length=max_len, temperature=1.0,
                                                      rescore_method=rs, rescore_reward=0.5, return_all=ra)
                tag = "k%d_%s_%s" % (k, rs, "all" if ra else "best")
                if not ra:
                    caps, scores, alphas, ppl = [[c] for c in caps], [[s] for s in scores], [[a] for a in alphas], [[p] for p in ppl]
                lens[tag] = [[len(c) for c in cc] for cc in caps]
                for i in range(n_img):
                    out["%s/n%d/count" % (tag, i)] = np.array(len(caps[i]))
                    for j in range(len(caps[i])):
                        out["%s/n%d/h%d/tokens" % (tag, i, j)] = np.array(caps[i][j], dtype=np.int64)
                        out["%s/n%d/h%d/score" % (tag, i, j)] = np.float64(scores[i][j])
                        out["%s/n%d/h%d/ppl" % (tag, i, j)] = np.float64(ppl[i][j])
                        out["%s/n%d/h%d/alphas" % (tag, i, j)] = alphas[i][j].numpy()
    # temperature != 1
    caps, scores, alphas, ppl = m.caption(ann.clone(), beamk=3, max_gen_length=max_len, temperature=0.7,
                                          rescore_method="LN", return_all=False)
    for i in range(n_img):
        out["k3_LN_T0.7/n%d/tokens" % i] = np.array(caps[i], dtype=np.int64)
        out["k3_LN_T0.7/n%d/score" % i] = np.float64(scores[i])
    save(name, out)
    print(name, {k: v for k, v in lens.items() if k.endswith("None_best") or k.endswith("LN_best")})


# ------------------------------------------------------------------------------------------------------------------
# BASELINE configs[0] (C1) through the reference's REAL trunk: resnet18 (pretrained=False) + the readme's resize layer
# (readme.md:118-121) -> L=196, D=512, A=128, E=256, H=512, V=6400, batch 8, 20 targets, fp32, torch.rand 224x224 images.
# Weights and inputs are NOT stored: the module's seeded default init is bit-identical to the reference's
# (tests/test_model_api.py) and the inputs come from seeded CPU generators, so the fixture holds the seeds plus
#   * the trunk output before the resize (train-mode batch statistics / eval-mode running statistics), so that the decoder
#     can be checked at 1e-5 on exactly the reference's annotations, independent of cuDNN-vs-MKLDNN convolution rounding;
#   * logits (every 16th word + per-row log-sum-exp / arg-max), alphas, loss, accuracy;
#   * per-parameter gradient digests (norm + 64 sampled entries) and a digest of the annotation gradient;
#   * greedy / beam (k=5) captions and scores of the sharpened model in eval mode.
# ------------------------------------------------------------------------------------------------------------------
C1 = dict(D=512, A=128, E=256, H=512, V=6400, T=20, B=8, size=14, arch="resnet18")
C1_SHARPEN = dict(wo=8.0, emb=2.0, fatt=30.0, end_bias=9.5)   # mixed caption lengths for k=1 and k=5 (probed)


def c1_inputs(seed=1):
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


def c1_model(model, seed=0, sharpen=False):
    torch.manual_seed(seed)
    hp = rh.default_hparams(encoder_arch=C1["arch"], encoder_dim=C1["D"], attention_dim=C1["A"], embed_dim=C1["E"], decoder_dim=C1["H"],
                            vocab_size=C1["V"])
    m = model.SAT(**hp)
    m.encoder = nn.Sequential(*m.encoder, nn.Upsample((C1["size"], C1["size"]), mode="bilinear", align_corners=False))
    if sharpen:
        V = C1["V"]
        with torch.no_grad():
            m.output.output.weight *= C1_SHARPEN["wo"]
            m.embedding.weight *= C1_SHARPEN["emb"]
            m.attention.f_att.weight *= C1_SHARPEN["fatt"]
            m.output.output.bias[V - 1] = C1_SHARPEN["end_bias"]
    return m


def c1_case(model):
    out = {}
    img, caps, lens = c1_inputs()
    m = c1_model(model)
    m.train()
    trunk = nn.Sequential(*list(m.encoder)[:-1])
    # training_step's forward pieces, exactly as the reference writes them (model.py:588-597), on the real trunk
    x = img.clone()
    ann7 = trunk(x)                                              # [8,512,7,7], train-mode batch-norm statistics
    ann7 = ann7.detach().requires_grad_(True)
    resize = list(m.encoder)[-1]
    saved_encoder = m.encoder
    m.encoder = resize                                           # the decoder consumes the SAME annotations the trunk produced
    lp, tp, alphas = m.train_batch([ann7, caps, lens], torch.tensor(1))
    ce = m.criterion(lp.data, tp.data)
    loss = ce + m.hparams.att_gamma * ((1 - alphas.sum(dim=1)) ** 2).mean()
    pred = torch.argmax(lp.data, dim=1)
    acc = torch.sum(pred == tp.data) / pred.shape[0]
    loss.backward()
    m.encoder = saved_encoder
    out["train/ann7"] = ann7.detach().numpy().copy()
    out["train/logits_sub"] = lp.data[:, ::16].detach().numpy().copy()          # packed rows x every 16th word
    out["train/lse"] = torch.logsumexp(lp.data, 1).detach().numpy()
    out["train/argmax"] = pred.numpy()
    out["train/alphas"] = alphas.detach().numpy()
    out["train/loss"], out["train/ce"], out["train/acc"] = np.float64(loss.item()), np.float64(ce.item()), np.float64(acc.item())
    for k, p in m.named_parameters():
        if k.startswith("encoder") or p.grad is None:
            continue
        g = p.grad.reshape(-1)
        out["grad_norm/" + k] = np.float64(g.double().norm().item())
        out["grad_samp/" + k] = g[digest_indices(g.numel())].numpy().copy()
    ga = ann7.grad.reshape(-1)
    out["grad_norm/ann7"] = np.float64(ga.double().norm().item())
    out["grad_samp/ann7"] = ga[digest_indices(ga.numel())].numpy().copy()
    # the whole step through the reference's own training_step with the real trunk (loss only; the trunk runs again)
    m2 = c1_model(model)
    m2.train()
    ts = m2.training_step((img.clone(), caps, lens), 0)
    out["train/loss_training_step"] = np.float64(float(ts["loss"]))
    out["train/acc_training_step"] = np.float64(float(ts["accuracy"]))
    # decode: sharpened model, eval mode (running statistics at their initial values), 4 images
    md = c1_model(model, sharpen=True)
    md.eval()
    img4 = img[:4].clone()
    with torch.no_grad():
        ann7e = nn.Sequential(*list(md.encoder)[:-1])(img4.clone())
    out["decode/ann7"] = ann7e.numpy().copy()
    for k in (1, 5):
        caps_o, scores, alph, ppl = md.caption(img4.clone(), beamk=k, max_gen_length=30, temperature=1.0, rescore_method="LN", return_all=False)
        for i in range(4):
            out["decode/k%d/n%d/tokens" % (k, i)] = np.array(caps_o[i], dtype=np.int64)
            out["decode/k%d/n%d/score" % (k, i)] = np.float64(scores[i])
            out["decode/k%d/n%d/alpha_sum" % (k, i)] = alph[i].sum(0).numpy()
        print("c1 decode k=%d lengths" % k, [len(c) for c in caps_o])
    save("c1_resnet18", out)
    print("c1_resnet18 loss", loss.item(), "training_step loss", float(ts["loss"]), "acc", acc.item())


# ------------------------------------------------------------------------------------------------------------------
# the module surface around the decoder (tests/test_model_api.py, tests/test_callers_cpu.py use the same hparams and inputs):
#   * init/:  state_dict keys, shapes and per-tensor digests (norm + 64 sampled entries) of SAT(**default_hparams(vocab_size=400))
#             under torch.manual_seed(3);
#   * score/: score_captions' cosine similarity and result keys;
#   * lr/:    learning rates of every param group over 3 epochs x 6 batches of warm-up + scheduler stepping, per scheduler.
# The committed reference_api.npz was recorded by running api_case on sat_b200.model (it takes any module with the reference's
# SAT API), at a commit whose `reference`-marked tests passed against the upstream files: state_dict bit-identical, learning
# rates within 1e-12, cosine similarity within 1e-6.  With the upstream files present, `python oracle/make_golden.py api`
# records it from the reference itself.
# ------------------------------------------------------------------------------------------------------------------
def reference_lrs(model, sched):
    """the reference's optimizer / scheduler driven like its training loop: training_step's warm-up and per-batch stepping
    (model.py:608-617), the epoch hooks (model.py:633-635) -> (initial lrs, [steps, groups] lrs, scheduler class name)"""
    ref = model.SAT(**dict(rh.small_hparams(scheduler=sched, **rh.LR_EXTRA)))
    ro = ref.configure_optimizers()
    ref._optimizer = ro
    init = [pg["lr"] for pg in ro.param_groups]
    tr = type("T", (), {"global_step": 0})()
    ref.trainer = tr
    lrs = []
    for epoch in range(3):
        for it in range(6):
            if tr.global_step < ref.hparams.lr_warmup_steps:
                lr_scale = min(1, float(tr.global_step + 1) / ref.hparams.lr_warmup_steps)
                for pg, init_lr in zip(ro.param_groups, ref.opt_init_lr):
                    pg["lr"] = lr_scale * init_lr
            elif tr.global_step > 0 and type(ref.scheduler) in (torch.optim.lr_scheduler.CosineAnnealingWarmRestarts, torch.optim.lr_scheduler.OneCycleLR):
                ref.scheduler.step()
            ro.step()
            lrs.append([pg["lr"] for pg in ro.param_groups])
            tr.global_step += 1
        ref.current_epoch = epoch
        ref.training_epoch_end([{"loss": 1.0}])
        if sched == "plateau":
            ref.hparams.plateau_monitor = ref.hparams.save_monitor = ref.hparams.early_stop_monitor = "bleu4"
            ref.validation_epoch_end([{"bleu4": 0.1}])
    return init, lrs, type(ref.scheduler).__name__


def api_case(model):
    out = {}
    torch.manual_seed(3)
    sd = model.SAT(**rh.default_hparams(vocab_size=400)).state_dict()
    out["init/keys"] = np.array(list(sd.keys()))
    for k, v in sd.items():
        flat = v.reshape(-1)
        out["init/shape/" + k] = np.array(v.shape, dtype=np.int64)
        out["init/norm/" + k] = np.float64(flat.double().norm().item())
        out["init/samp/" + k] = flat[digest_indices(flat.numel())].numpy().copy()
    torch.manual_seed(3)
    r = model.SAT(**rh.small_hparams()).score_captions(*rh.score_inputs())
    out["score/cosine_similarity"] = np.float64(r["cosine_similarity"])
    out["score/keys"] = np.array(sorted(r.keys()))
    for sched in rh.LR_SCHEDULERS:
        init, lrs, name = reference_lrs(model, sched)
        out["lr/%s/init" % sched] = np.array(init, dtype=np.float64)
        out["lr/%s/lrs" % sched] = np.array(lrs, dtype=np.float64)
        out["lr/%s/scheduler" % sched] = np.array(name)
    save("reference_api", out)
    print("reference_api", len(sd), "state_dict entries, cosine", out["score/cosine_similarity"])


def layers_cases(model):
    """decoder_layers > 1 (nn.LSTM num_layers, model.py:175-180): stacked states, attention / beta / output on h[-1]."""
    # two layers, ragged, two captions per image, sizes that are NOT multiples of 8 (zero-padded storage on the device)
    train_case(model, "train_layers2", 5, B_img=3, ncap=2, hw=(3, 4), D=16, A=8, E=10, H=14, V=50, T=6,
               ragged=True, label_smoothing=0.1, sharpen=dict(fatt=20.0), layers=2)
    # three layers, tile-sized dims, ragged
    train_case(model, "train_layers3", 6, B_img=4, ncap=1, hw=(4, 4), D=64, A=32, E=32, H=64, V=128, T=10,
               ragged=True, label_smoothing=0.05, sharpen=dict(fatt=10.0), layers=3)
    decode_case(model, "decode_layers2", 7, n_img=5, hw=(4, 4), D=64, A=32, E=32, H=64, V=128, max_len=16,
                sharpen=dict(wo=8.0, emb=2.0, fatt=30.0, end_bias=3.0), layers=2)


def main():
    os.makedirs(OUT, exist_ok=True)
    model, _ = rh.load_reference()
    if len(sys.argv) > 1 and sys.argv[1] == "c1":
        return c1_case(model)
    if len(sys.argv) > 1 and sys.argv[1] == "layers":
        return layers_cases(model)
    if len(sys.argv) > 1 and sys.argv[1] == "api":
        return api_case(model)
    # tiny, ragged, 2 captions per image, non-square map, label smoothing, peaky attention
    train_case(model, "train_tiny", 0, B_img=3, ncap=2, hw=(3, 4), D=16, A=8, E=10, H=14, V=50, T=6,
               ragged=True, label_smoothing=0.1, sharpen=dict(fatt=20.0))
    # small, square map, fixed length (BASELINE-style: ncap 1, all lengths T), plain CE
    train_case(model, "train_small", 1, B_img=5, ncap=1, hw=(7, 7), D=64, A=32, E=32, H=48, V=120, T=8,
               ragged=False, label_smoothing=0.0)
    # small ragged with dims that are multiples of the CUDA tile sizes
    train_case(model, "train_ragged", 2, B_img=4, ncap=1, hw=(4, 4), D=64, A=32, E=32, H=64, V=128, T=10,
               ragged=True, label_smoothing=0.05, sharpen=dict(fatt=10.0))
    # decode: sharpened so that <END> is reachable and beams shrink (SURVEY.md appendix D-8/D-10)
    decode_case(model, "decode_tiny", 3, n_img=6, hw=(3, 4), D=16, A=8, E=10, H=14, V=50, max_len=12,
                sharpen=dict(wo=8.0, emb=2.0, fatt=30.0, end_bias=2.0))
    decode_case(model, "decode_small", 4, n_img=5, hw=(4, 4), D=64, A=32, E=32, H=64, V=128, max_len=16,
                sharpen=dict(wo=8.0, emb=2.0, fatt=30.0, end_bias=3.0))
    layers_cases(model)
    c1_case(model)
    api_case(model)


if __name__ == "__main__":
    main()
