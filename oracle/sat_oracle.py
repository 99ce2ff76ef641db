"""CPU oracle for the Show-Attend-and-Tell decoder hot path.

TEST INFRASTRUCTURE ONLY.  This is a plain-torch (CPU, fp32 or fp64) restatement of the
algorithm in the reference's model.py / util.py.  `train_batch` / `train_loss` also run on a CUDA device when the inputs
live there (the full-batch float64 references of tests/test_full_size_grads_gpu.py).  Only `tests/`, `__graft_entry__.smoke()`
and `bench.py`'s cpu_baseline / `--impl reference` legs may import it, and only as the
checker or as the timed CPU baseline.  The product path (`sat_b200`) never imports this file
and has no CPU fallback.

Parity pinning: the reference ships no tests or golden vectors (SURVEY.md §4), so the
oracle is pinned against OUTPUTS OF THE REFERENCE ITSELF, generated in the build container
by `oracle/make_golden.py` (imports the unmodified upstream model.py through
`oracle/ref_harness.py`) and committed under `tests/golden/`.  `tests/test_oracle_golden.py`
checks every function here against those vectors (forward, loss, gradients via autograd,
greedy and beam token ids, scores, alphas, perplexities).

Weights are passed as a dict keyed by the reference's state_dict names (SURVEY.md §A.3):
  embedding.weight [V,E]; init_lstm.factorize.{weight [E,D],bias}; init_lstm.init.{weight [2H,E],bias};
  lstm.weight_ih_l0 [4H,E+D]; lstm.weight_hh_l0 [4H,H]; lstm.bias_ih_l0; lstm.bias_hh_l0;
  attention.encoder_att.weight [A,D]; attention.decoder_att.weight [A,H]; attention.f_att.weight [1,A];
  beta.0.{weight [D,H],bias [D]}; output.hidden.weight [E,H]; output.context.weight [E,D];
  output.output.{weight [V,E], bias [V]}.
decoder_layers > 1 (nn.LSTM num_layers, model.py:175-180) adds lstm.{weight_ih,weight_hh,bias_ih,bias_hh}_l{l} ([4H,H] / [4H]) per
layer l >= 1 and widens init_lstm.init to [2*layers*H, E]; the states are then [layers,B,H] and attention, the beta gate and
the output layer read the top layer's state h[-1] (model.py:299-300,327,538-547).  With one layer the states stay [B,H].
"""
import math

import torch
from torch.nn.utils.rnn import pack_padded_sequence


# --------------------------------------------------------------------------------------
# building blocks
# --------------------------------------------------------------------------------------
def init_lstm(W, ann):
    """model.py:76-81.  ann [B,D,h,w] -> (h0, c0) each [B,H] (layers == 1).

    mean over (h,w) -> factorize -> init (no nonlinearity between) -> the [B,2H] result is
    REINTERPRETED row-major as [2,B,H] (reshape, not a per-row split): SURVEY.md §A.2-1.
    """
    mean = ann.mean((2, 3))
    f1 = mean @ W["init_lstm.factorize.weight"].t() + W["init_lstm.factorize.bias"]
    out = f1 @ W["init_lstm.init.weight"].t() + W["init_lstm.init.bias"]
    return _split_init(W, out)


def num_layers(W):
    """decoder_layers of a weight dict (presence of lstm.weight_ih_l{l})."""
    n = 1
    while ("lstm.weight_ih_l%d" % n) in W:
        n += 1
    return n


def _split_init(W, out):
    """model.py:79-80: the [B, 2*layers*H] init output reinterpreted row-major as [2*layers, B, H]; first `layers` states are h."""
    nl = num_layers(W)
    B = out.shape[0]
    H = out.shape[1] // (2 * nl)
    st = out.reshape(2 * nl, B, H)
    if nl == 1:
        return st[0], st[1]
    return st[:nl], st[nl:]


def attention(W, ann, h):
    """model.py:94-109.  ann [B,D,h,w], h [B,H] -> z [B,D], alpha [B,h*w]."""
    B, D, hh, ww = ann.shape
    L = hh * ww
    a = ann.reshape(B, D, L).permute(0, 2, 1)                      # [B,L,D]
    p = a @ W["attention.encoder_att.weight"].t()                  # [B,L,A]   model.py:100
    q = (h @ W["attention.decoder_att.weight"].t()).unsqueeze(1)   # [B,1,A]   model.py:102
    e = (torch.tanh(p + q) @ W["attention.f_att.weight"].t()) * L ** -0.5   # model.py:104
    alpha = torch.softmax(e, dim=1)                                # over locations, model.py:106
    z = (a * alpha).sum(1)                                         # model.py:108
    return z, alpha.squeeze(2)


def beta_gate(W, h):
    """model.py:187-192: sigmoid(Linear(H->D))."""
    return torch.sigmoid(h @ W["beta.0.weight"].t() + W["beta.0.bias"])


def lstm_cell(W, x, h, c):
    """torch.nn.LSTM, seq_len 1 (model.py:175-180,326,544): gate order i,f,g,o.  h, c [B,H] (one layer) or [layers,B,H]:
    layer l > 0 takes the new hidden state of layer l-1 as its input (no dropout between layers: nn.LSTM(dropout=0))."""
    def cell(l, x, h, c):
        G = x @ W["lstm.weight_ih_l%d" % l].t() + W["lstm.bias_ih_l%d" % l] + h @ W["lstm.weight_hh_l%d" % l].t() + W["lstm.bias_hh_l%d" % l]
        i, f, g, o = G.chunk(4, dim=1)
        c2 = torch.sigmoid(f) * c + torch.sigmoid(i) * torch.tanh(g)
        h2 = torch.sigmoid(o) * torch.tanh(c2)
        return h2, c2

    if h.dim() == 2:
        return cell(0, x, h, c)
    hs, cs = [], []
    for l in range(h.shape[0]):
        x, c2 = cell(l, x, h[l], c[l])
        hs.append(x)
        cs.append(c2)
    return torch.stack(hs), torch.stack(cs)


def deep_output(W, x_e, h, z, deep=True, drop=None):
    """model.py:125-131; `drop` = explicit dropout multipliers (0 or 1/(1-p)) for the activations before the output layer."""
    if deep:
        x = torch.tanh(x_e + h @ W["output.hidden.weight"].t() + z @ W["output.context.weight"].t())
    else:
        x = h @ W["output.hidden.weight"].t()
    if drop is not None:
        x = x * drop
    logit = x @ W["output.output.weight"].t()
    if W.get("output.output.bias", None) is not None:
        logit = logit + W["output.output.bias"]
    return logit


def decoder_step(W, ann, words, h, c, deep=True, emb_drop=None, out_drop=None):
    """One pass of the per-timestep hot path: model.py:298-327 (decode) == 526-547 (train)."""
    x_e = W["embedding.weight"][words]
    if emb_drop is not None:
        x_e = x_e * emb_drop                      # embedding_dropout (model.py:526)
    htop = h if h.dim() == 2 else h[-1]
    z, alpha = attention(W, ann, htop)
    beta = beta_gate(W, htop)
    h2, c2 = lstm_cell(W, torch.cat([x_e, beta * z], dim=1), h, c)
    logit = deep_output(W, x_e, h2 if h2.dim() == 2 else h2[-1], z, deep, out_drop)      # ungated z, new (top) h
    return logit, alpha, h2, c2


# --------------------------------------------------------------------------------------
# teacher-forced forward (model.py:474-557) + loss (model.py:592-597, util.py:105-112)
# --------------------------------------------------------------------------------------
def train_batch(W, ann_img, encoded_captions, lengths, epsilon=1.0, deep=True, rand=None, masks=None):
    """ann_img [B_img,D,h,w]; encoded_captions [B_img,ncap,T+1] int64; lengths [B_img,ncap].

    Returns padded logits [B,T,V], alphas [B,T,L], flat captions [B,T+1], flat lengths [B].
    Rows are compacted by boolean index each step exactly like model.py:512-548;
    finished rows keep zeros in logits/alphas.
    `rand`: optional callable giving the per-step uniform draw for scheduled sampling.
    """
    ncap = lengths.shape[1]
    ann = ann_img.repeat_interleave(ncap, dim=0)                    # model.py:487
    caps = encoded_captions.reshape(-1, encoded_captions.shape[2])
    lens = lengths.reshape(-1)
    B, caplen = caps.shape
    T = caplen - 1
    L = ann.shape[2] * ann.shape[3]
    V = W["embedding.weight"].shape[0]
    # masks: optional explicit dropout multipliers dict(mean [B,D], emb [B,T,E], out [B,T,E]) so that the train-mode
    # path (model.py:78,526,130) can be checked with the masks the CUDA kernels generate
    if masks is not None and masks.get("mean") is not None:
        mean = ann.mean((2, 3)) * masks["mean"]
        f1 = mean @ W["init_lstm.factorize.weight"].t() + W["init_lstm.factorize.bias"]
        out0 = f1 @ W["init_lstm.init.weight"].t() + W["init_lstm.init.bias"]
        h, c = _split_init(W, out0)
    else:
        h, c = init_lstm(W, ann)
    h, c = h.clone(), c.clone()
    dt, dev = ann.dtype, ann.device
    logits = torch.zeros(B, T, V, dtype=dt, device=dev)
    alphas = torch.zeros(B, T, L, dtype=dt, device=dev)
    for step in range(T):
        act = lens > step
        if not bool(act.any()):
            break
        idx = act.nonzero().squeeze(1)
        teacher = step <= 2
        if not teacher:
            u = rand() if rand is not None else float(torch.rand(1))
            teacher = u <= float(epsilon)
        if teacher:
            words = caps[idx, step]
        else:
            words = torch.argmax(logits[idx, step - 1, :], dim=1)   # model.py:523 (no grad path)
        ed = masks["emb"][idx, step] if masks is not None and masks.get("emb") is not None else None
        od = masks["out"][idx, step] if masks is not None and masks.get("out") is not None else None
        stacked = h.dim() == 3
        logit, alpha, h2, c2 = decoder_step(W, ann[idx], words, h[:, idx] if stacked else h[idx], c[:, idx] if stacked else c[idx],
                                            deep, ed, od)
        alphas = alphas.index_put((idx, torch.tensor(step, device=dev)), alpha)
        logits = logits.index_put((idx, torch.tensor(step, device=dev)), logit)
        if stacked:
            h = h.index_copy(1, idx, h2)
            c = c.index_copy(1, idx, c2)
        else:
            h = h.index_put((idx,), h2)
            c = c.index_put((idx,), c2)
    return logits, alphas, caps, lens


def pack(logits, caps, lens):
    """model.py:553-554: time-major packed logits / targets."""
    lp = pack_padded_sequence(logits, lens.tolist(), batch_first=True, enforce_sorted=False)
    tp = pack_padded_sequence(caps[:, 1:], lens.tolist(), batch_first=True, enforce_sorted=False)
    return lp, tp


def label_smoothing_loss(x, target, smoothing=0.0):
    """util.py:105-112."""
    lp = torch.log_softmax(x, dim=-1)
    nll = -lp.gather(-1, target.unsqueeze(1)).squeeze(1)
    smooth = -lp.mean(-1)
    return ((1.0 - smoothing) * nll + smoothing * smooth).mean()


def train_loss(W, ann_img, encoded_captions, lengths, label_smoothing=0.0, att_gamma=1.0,
               epsilon=1.0, deep=True, rand=None, masks=None):
    """model.py:588-597: returns dict(loss, acc, ce, reg, logits, alphas)."""
    logits, alphas, caps, lens = train_batch(W, ann_img, encoded_captions, lengths, epsilon, deep, rand, masks)
    lp, tp = pack(logits, caps, lens)
    ce = label_smoothing_loss(lp.data, tp.data, label_smoothing)
    reg = ((1 - alphas.sum(dim=1)) ** 2).mean()                     # model.py:594
    loss = ce + att_gamma * reg
    pred = torch.argmax(lp.data, dim=1)
    acc = (pred == tp.data).sum() / pred.shape[0]
    return dict(loss=loss, acc=acc, ce=ce, reg=reg, logits=logits, alphas=alphas,
                logits_packed=lp, targets_packed=tp)


# --------------------------------------------------------------------------------------
# greedy (beamk=1) / beam decode: model.py:237-472 with sample_method="beam", no decoder noise
# --------------------------------------------------------------------------------------
def caption(W, ann_img, vocab, beamk=3, max_gen_length=32, temperature=1.0,
            rescore_method=None, rescore_reward=0.5, return_all=False, deep=True):
    """ann_img [B_img,D,h,w]; vocab = dict(PAD=,START=,END=,UNK=) token ids.

    One image at a time, its beam is the batch (model.py:260-269).  Returns the reference's
    four lists: captions, scores, alphas ([len,h,w] tensors), perplexities.
    """
    PAD, START, END, UNK = vocab["PAD"], vocab["START"], vocab["END"], vocab["UNK"]
    V = W["embedding.weight"].shape[0]
    temps = temperature if isinstance(temperature, list) else [temperature]
    _, D, hh, ww = ann_img.shape
    out_caps, out_scores, out_alphas, out_ppl = [], [], [], []
    for n in range(ann_img.shape[0]):
        k = beamk
        ann = ann_img[n].expand(k, D, hh, ww)
        h, c = init_lstm(W, ann)                      # rows identical -> reinterpretation quirk
        preds = torch.full((1, k), START, dtype=torch.long)
        top = torch.zeros(k, dtype=ann_img.dtype)
        alph = torch.zeros(1, k, hh, ww, dtype=ann_img.dtype)
        f_caps, f_alph, f_sc, f_ppl = [], [], [], []
        step = 0
        while True:
            temp = temps[step % len(temps)]
            logit, alpha, h, c = decoder_step(W, ann, preds[step], h, c, deep)
            alpha = alpha.reshape(-1, hh, ww)
            sc = torch.log_softmax(logit / temp, dim=1)
            sc[:, [START, PAD]] = float("-inf")                   # model.py:333
            if step == 0:
                sc[:, [END, UNK]] = float("-inf")                 # model.py:340
                top, widx = torch.topk(sc[0], k)                  # beam 0 only, model.py:343
                preds = torch.cat([preds, widx.unsqueeze(0)], 0)
                alph = torch.cat([alph, alpha.unsqueeze(0)], 0)
            else:
                seq = sc + top.unsqueeze(1)
                _, flat = torch.topk(seq.reshape(-1), k, dim=0)   # model.py:359
                top = seq.reshape(-1)[flat]
                src = torch.div(flat, V, rounding_mode="floor")
                wrd = torch.remainder(flat, V).unsqueeze(0)
                preds = torch.cat([preds[:, src], wrd], 0)
                alph = torch.cat([alph[:, src], alpha.unsqueeze(0)[:, src]], 0)
                h, c, ann = (h[:, src], c[:, src], ann[src]) if h.dim() == 3 else (h[src], c[src], ann[src])
            done = preds[step + 1] == END

            def rescore(s):
                if rescore_method == "LN":
                    return s / step
                if rescore_method == "WR":
                    return s + rescore_reward * step
                if rescore_method == "BAR":
                    return s + rescore_reward * (-torch.mean(top))
                return s

            if bool(done.any()):
                dp, da, ds = preds[:, done], alph[:, done], top[done]
                for i in range(dp.shape[1]):
                    f_caps.append(dp[:, i][1:-1].tolist())
                    f_alph.append(da[:, i][1:-1].clone())
                    f_sc.append(float(rescore(ds[i])))
                    f_ppl.append(float(torch.exp(-ds[i] / step)))
                keep = ~done
                preds, alph, top = preds[:, keep], alph[:, keep], top[keep]
                h, c, ann = (h[:, keep], c[:, keep], ann[keep]) if h.dim() == 3 else (h[keep], c[keep], ann[keep])
                k = int(keep.sum())
                if k == 0:
                    break
            if step >= max_gen_length:                              # model.py:441-446
                for i in range(preds.shape[1]):
                    f_caps.append(preds[:, i][1:-1].tolist())
                    f_alph.append(alph[:, i][1:-1].clone())
                    f_sc.append(float(rescore(top[i])))
                    f_ppl.append(float(torch.exp(-top[i] / step)))
                break
            step += 1
        if return_all:
            order = sorted([[f_sc[i], i] for i in range(len(f_sc))], reverse=True)
            order = [x[1] for x in order]
            out_caps.append([f_caps[i] for i in order])
            out_alphas.append([f_alph[i] for i in order])
            out_scores.append([f_sc[i] for i in order])
            out_ppl.append([f_ppl[i] for i in order])
        else:
            best = f_sc.index(max(f_sc))
            out_caps.append(f_caps[best])
            out_alphas.append(f_alph[best])
            out_scores.append(f_sc[best])
            out_ppl.append(f_ppl[best])
    return out_caps, out_scores, out_alphas, out_ppl


# --------------------------------------------------------------------------------------
# encoder (boundary only; third-party torchvision trunk, model.py:16-63 + readme.md:118-121)
# --------------------------------------------------------------------------------------
def build_encoder(arch="resnet18", encoder_dim=512, encoder_size=None, input_size=224,
                  mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225)):
    """CPU torchvision trunk producing [B,D,h,w] annotations, used by the cpu_baseline leg."""
    from torch import nn
    from torchvision import models
    m = models.__dict__[arch](weights=None)
    layers = list(m.children())[:-2]
    with torch.no_grad():
        final_dim = nn.Sequential(*layers)(torch.zeros(1, 3, input_size, input_size)).shape[1]
    if encoder_dim is not None and encoder_dim != final_dim:
        layers.append(nn.Conv2d(final_dim, encoder_dim, kernel_size=1, stride=1, bias=True))
    if encoder_size is not None:
        layers.append(nn.Upsample((encoder_size, encoder_size), mode="bilinear", align_corners=False))

    class _Norm(nn.Module):
        def forward(self, x):
            mu = torch.tensor(mean, dtype=x.dtype).view(1, 3, 1, 1)
            sd = torch.tensor(std, dtype=x.dtype).view(1, 3, 1, 1)
            return (x - mu) / sd

    return nn.Sequential(_Norm(), *layers)


def random_weights(D, A, E, H, V, seed=0, dtype=torch.float32, sharpen=False, layers=1):
    """Synthetic decoder weights with torch-default-like scales (for sizes where no reference run is stored)."""
    g = torch.Generator().manual_seed(seed)

    def U(shape, fan):
        b = 1.0 / math.sqrt(fan)
        return ((torch.rand(shape, generator=g, dtype=torch.float64) * 2 - 1) * b).to(dtype)

    W = {
        "embedding.weight": torch.randn(V, E, generator=g, dtype=torch.float64).to(dtype),
        "init_lstm.factorize.weight": U((E, D), D), "init_lstm.factorize.bias": U((E,), D),
        "init_lstm.init.weight": U((2 * H, E), E), "init_lstm.init.bias": U((2 * H,), E),
        "lstm.weight_ih_l0": U((4 * H, E + D), H), "lstm.weight_hh_l0": U((4 * H, H), H),
        "lstm.bias_ih_l0": U((4 * H,), H), "lstm.bias_hh_l0": U((4 * H,), H),
        "attention.encoder_att.weight": U((A, D), D), "attention.decoder_att.weight": U((A, H), H),
        "attention.f_att.weight": U((1, A), A),
        "beta.0.weight": U((D, H), H), "beta.0.bias": torch.full((D,), 1.0 / H, dtype=dtype),
        "output.hidden.weight": U((E, H), H), "output.context.weight": U((E, D), D),
        "output.output.weight": U((V, E), E), "output.output.bias": U((V,), E),
    }
    if layers > 1:                             # drawn after the one-layer parameters: the layers=1 streams stay what they were
        W["init_lstm.init.weight"], W["init_lstm.init.bias"] = U((2 * layers * H, E), E), U((2 * layers * H,), E)
        for l in range(1, layers):
            W["lstm.weight_ih_l%d" % l], W["lstm.weight_hh_l%d" % l] = U((4 * H, H), H), U((4 * H, H), H)
            W["lstm.bias_ih_l%d" % l], W["lstm.bias_hh_l%d" % l] = U((4 * H,), H), U((4 * H,), H)
    W["embedding.weight"][0].zero_()          # padding_idx row
    if sharpen:                                # SURVEY.md §8d: makes <END>/beam-shrink paths reachable
        W["output.output.weight"] *= 8
        W["embedding.weight"] *= 2
        W["attention.f_att.weight"] *= 30
        W["output.output.bias"][V - 1] = 6.6
    return W
