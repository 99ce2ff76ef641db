"""GPU: every stage of the bf16 training step against a float64 replay of its own saved inputs.

The end-to-end checks (library vs the float64 oracle after all T steps) need bounds of 2e-2 .. 6e-2, because T steps of
legitimate bf16 rounding separate the two sides.  Here each stage is recomputed in float64 from the library's own inputs to
that stage (the packed weights in pw.t, which are the exact bf16 values the kernels read, and the saved buffers of
SatTrainBuffers), so the only thing separating the two sides is that stage's own arithmetic: one fp32 accumulation, at most
one or two bf16 roundings and the documented MUFU approximations.  Every element is held to

    |got - ref| <= r |ref| + C_ACC u sqrt(K) S + m

with S = sum |a_k b_k| (+ |bias|) computed by the same replay on absolute values, u = 2^-24, r = 0 (fp32 output) or R16 per bf16
rounding, and m the MUFU terms propagated through the nonlinearity (constants below, each with its derivation).

Also checked, bit for bit: the fed words and embeddings, the initial states, dP16 = bf16(dP), the frozen rows of finished
captions, out[4..6]; the invariants (inactive rows zero, padded lanes zero, every read buffer finite); and that a step whose
work buffers start as NaN gives bit-identical results to one whose work buffers start as zero (no kernel reads an element no
kernel wrote).  The mutation tests apply the smallest defect each stage check claims to catch and assert the check fails.
`pytest -s` prints the worst error / bound per stage and configuration."""
import math
import os
import sys
import warnings
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import sat_oracle as O

warnings.filterwarnings("ignore")
pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)

# ---- error constants --------------------------------------------------------------------------------------------------------
U = 2.0 ** -24          # fp32 unit roundoff (round to nearest)
ULP = 2.0 ** -23        # one fp32 ulp relative to the value it is an ulp of (ulp(x) <= 2^-23 |x|)
R16 = 2.0 ** -8         # one round to nearest into bf16 (8 significant bits): relative error <= 2^-8
C_ACC = 4.0             # fp32 sums of K terms: each of the K roundings is at most u times a partial sum bounded by S and they
                        # do not all point the same way; their total stays within C_ACC standard deviations of that random walk
T_TANH = 2.0 ** -10.99  # tanh.approx.f32: maximum relative error 2^-10.99 (PTX ISA)
E_EX2 = 2.0 ** -22      # ex2.approx.ftz.f32: maximum relative error 2^-22 (PTX ISA), doubled for the ftz range used here
LOGF_ABS = 2.0 ** -21.41  # __logf: absolute error 2^-21.41 on [0.5, 2], otherwise 3 ulp (CUDA Programming Guide)
GSCALE = 0.75           # upstream d(loss): exact in binary, and not 1, so every place that applies it is exercised


def e_expf(x):
    """__expf(x): 2 + floor(1.173 |x|) ulp (CUDA Programming Guide), as a relative error"""
    return (2.0 + torch.floor(1.173 * x.abs())) * ULP


def e_sigmoid(x):
    """relative error of __fdividef(1, 1 + __expf(-x)): __expf's ulps (damped by e^-x / (1 + e^-x) <= 1), the add (u) and
    __fdividef (2 ulp)"""
    return e_expf(x) + U + 2.0 * ULP


def acc_err(K, S):
    return C_ACC * U * math.sqrt(max(int(K), 1)) * S


def bf16_bound(ref, delta, n_round=1):
    """n_round bf16 roundings of a value that was within `delta` of ref before rounding"""
    return n_round * R16 * ref.abs() + (1.0 + n_round * R16) * delta


def mm(a, b):
    """a [..., K] @ b [N, K]^T in float64 and the same product of absolute values"""
    a, b = a.double(), b.double()
    return a @ b.t(), a.abs() @ b.abs().t()


def word_or_pad(w, V0):
    return torch.where((w >= 0) & (w < V0), w, torch.zeros_like(w))


# ---- configurations -----------------------------------------------------------------------------------------------------------
CONFIGS = {
    # per-row pipelined attention, persistent vocabulary GEMM (K = 256), fused cross entropy
    "c2s": dict(Bi=16, ncap=1, hw=(14, 14), D=512, A=128, E=256, H=512, V=6400, T=12, ls=0.1),
    # grouped tensor-core box attention, V not a multiple of 128, ncap_sum_kernel for dW_a
    "coco": dict(Bi=4, ncap=5, hw=(7, 7), D=512, A=128, E=256, H=512, V=1000, T=12, alpha_bf16=True),
    # row-streamed grouped attention, one-tile-per-CTA vocabulary kernel (K = 512 > 256)
    "wide": dict(Bi=2, ncap=5, hw=(16, 16), D=2048, A=128, E=512, H=1024, V=1000, T=8, alpha_bf16=True),
    # padded lanes, K tails, three stacked layers
    "odd3": dict(Bi=3, ncap=2, hw=(3, 3), D=36, A=20, E=100, H=50, V=1003, T=9, layers=3, ls=0.1),
    # dropout on all three streams, DeepOutput(deep=False), weight tying without an output bias
    "drop_plain_tied": dict(Bi=4, ncap=2, hw=(5, 5), D=128, A=64, E=128, H=128, V=1200, T=10, drop=(0.3, 0.2, 4242), plain=True,
                            tied=True),
    # attention_dim 1024: KA = 8 kernels, dP_deferred_kernel column chunks
    "a1024": dict(Bi=2, ncap=2, hw=(7, 7), D=256, A=1024, E=128, H=256, V=1000, T=60),
    # bf16 on the SIMT cores: bf16 logits and ce_rows_kernel
    "simt": dict(Bi=4, ncap=1, hw=(5, 5), D=128, A=64, E=64, H=128, V=800, T=8, use_tc=False),
    # scheduled-sampling steps on the default path (the logits path at this vocabulary)
    "ss": dict(Bi=8, ncap=1, hw=(7, 7), D=256, A=64, E=128, H=256, V=1000, T=10, sampled=(0, 0, 0, 1, 0, 1, 1, 0, 1, 1)),
    # out-of-range word ids on the fused path: ids in [V0, V), ids >= V and negative ids, as inputs and as targets
    "badid": dict(Bi=8, ncap=1, hw=(7, 7), D=256, A=128, E=256, H=256, V=1003, T=8, ls=0.1, badid=True),
    # the same step with the logits kept (bf16 logits + ce_rows_kernel): the reference path for out-of-range targets
    "badid_rows": dict(Bi=8, ncap=1, hw=(7, 7), D=256, A=128, E=256, H=256, V=1003, T=8, ls=0.1, badid=True, unfused=True),
}
NAMES = list(CONFIGS)

# buffers that hold indices: filled with 0 (a valid index) instead of NaN, so that an unwritten index cannot address memory
# out of bounds.  ce_stats' fourth lane is an arg-max stored as integer bits.
INDEX_BUFS = ("tok", "row_argmax", "ce_stats")
# scratch whose unwritten part no kernel reads: excluded from the bit-identity comparison
SCRATCH = {
    "hp": "per-step scratch of the h-projection GEMM; after the loop only its first partials of sum (1-S)^2 are live",
    "dgz": "split-K partial slabs of dG * Wihz: slabs beyond the split factor are never written nor read",
    "dh": "split-K partial slabs of the h-chain GEMM (same)",
    "dxl": "split-K partial slabs of the stacked layers' input GEMM (same)",
    "dhq": "split-K partial slabs of the q / beta GEMM of stacked layers (same)",
    "gscale": "the shared device scalar 1.0 (decoder._one), never poisoned",
}
# bf16 operand copies that only the tensor-core GEMMs read: on the SIMT path no kernel writes or reads them
SIMT_UNUSED = ("dP16", "d_init_out16", "df116")


def _pad8(n):
    return (n + 7) // 8 * 8


def _inputs(name):
    from test_scheduled_sampling_vocab_gpu import _caps_batch
    c = CONFIGS[name]
    B, T, V0 = c["Bi"] * c["ncap"], c["T"], c["V"]
    W = O.random_weights(c["D"], c["A"], c["E"], c["H"], V0, seed=7, layers=c.get("layers", 1))
    W["attention.f_att.weight"] *= 10                      # non-uniform alpha
    if c.get("plain"):
        W["output.context.weight"] = None
    if c.get("tied"):
        W["output.output.weight"] = W["embedding.weight"]
        W["output.output.bias"] = None
    g = torch.Generator().manual_seed(8)
    ann = torch.randn(c["Bi"], c["D"], *c["hw"], generator=g)
    caps, lens = _caps_batch(B, T, V0, g)
    if c.get("badid"):
        Vs = _pad8(V0)
        bad = [V0, Vs - 1, Vs, Vs + 977, 1 << 20, -1, -7, -(1 << 20)]
        for i, w in enumerate(bad):                        # as fed words (column t) and as targets (column t + 1)
            b = i % B
            caps[b, 1 + i % max(1, int(lens[b]) - 1)] = w
        caps[B - 1, 1:T + 1] = torch.tensor((bad * T)[:T])
    return W, ann, caps.to(torch.int32), lens.to(torch.int32)


def _step(name, fill):
    """one forward + backward with every work buffer pre-filled: 'zero' or 'nan' (index buffers 0)"""
    from sat_b200 import decoder
    from sat_b200.packing import PackedWeights
    c = CONFIGS[name]
    W, ann, caps, lens = _inputs(name)
    use_tc = c.get("use_tc", True)
    pw = PackedWeights(W, dtype=torch.bfloat16, device="cuda")
    bld = decoder.annotations_as_bld(ann.cuda(), torch.bfloat16, pw.dims["D"])
    B, T = caps.shape[0], caps.shape[1] - 1
    sampled = list(c["sampled"]) if c.get("sampled") else None
    d = decoder.make_dims(B, c["Bi"], bld.shape[1], pw, T, torch.bfloat16, False, use_tc)
    fuse = decoder.vocab_path_fused(d, sampled, True) and not c.get("unfused")
    buf = decoder.TrainBuffers(d, torch.bfloat16, torch.device("cuda"), backward=True, keep_logits=not fuse, fuse_ce=fuse)
    for k, v in buf.t.items():
        if k == "gscale":
            continue
        if k in INDEX_BUFS or not v.is_floating_point():
            v.zero_()
        else:
            v.fill_(0.0 if fill == "zero" else float("nan"))
    buf.ws = torch.full((int(decoder._lib.lib().sat_param_grads_workspace_bytes(decoder.C.byref(d))),),
                        0 if fill == "zero" else 0xFF, dtype=torch.uint8, device="cuda")       # 0xFFFFFFFF is a NaN
    drop = c.get("drop") or (0.0, 0.0, 0)
    buf = decoder.train_forward(pw, bld, caps.cuda(), lens.cuda(), c.get("ls", 0.0), 1.0, exact=False, use_tc=use_tc, backward=True,
                                keep_logits=not fuse, buffers=buf, sampled=sampled, dropout=drop, fuse_ce=fuse)
    G, d_ann = decoder.train_backward(pw, buf, grad_loss=torch.tensor(GSCALE, device="cuda"), weight_tying=bool(c.get("tied")))
    torch.cuda.synchronize()
    return SimpleNamespace(name=name, c=c, W=W, pw=pw, t=buf.t, G=G, d_ann=d_ann, fused=fuse, caps_in=caps, lens_in=lens,
                           sampled=sampled)


_RUNS = {}


def run(name):
    if name not in _RUNS:
        r = _step(name, "zero")
        _prepare(r)
        _RUNS[name] = r
    return _RUNS[name]


def _prepare(r):
    """dims, activity mask and dropout masks of a run"""
    from test_scheduled_sampling_vocab_gpu import _drop_mask
    c, pw = r.c, r.pw
    r.D, r.A, r.E, r.H, r.V = (pw.dims[k] for k in "DAEHV")
    r.D0, r.A0, r.E0, r.H0, r.V0 = (pw.dims0[k] for k in "DAEHV")
    r.nl = pw.layers
    r.B, r.T = r.caps_in.shape[0], r.caps_in.shape[1] - 1
    r.Bi, r.ncap = c["Bi"], c["ncap"]
    r.L = c["hw"][0] * c["hw"][1]
    r.M = r.T * r.B
    dev = torch.device("cuda")
    lens = r.t["lens"].long()
    r.act = torch.arange(r.T, device=dev)[:, None] < lens[None, :]              # [T, B]
    r.img = torch.arange(r.B, device=dev) // r.ncap
    p, pe, seed = c.get("drop") or (0.0, 0.0, 0)
    i1 = (torch.arange(r.Bi)[:, None] * r.D + torch.arange(r.D)[None]).numpy()
    i23 = (torch.arange(r.M)[:, None] * r.E + torch.arange(r.E)[None]).numpy()
    r.m1 = _drop_mask(p, seed, 1, i1).double().to(dev) if p > 0 else torch.ones(r.Bi, r.D, dtype=torch.float64, device=dev)
    r.m2 = _drop_mask(pe, seed, 2, i23).double().to(dev).reshape(r.T, r.B, r.E) if pe > 0 else None
    r.m3 = _drop_mask(p, seed, 3, i23).double().to(dev).reshape(r.T, r.B, r.E) if p > 0 else None
    r.keep = 1.0 - p
    r.NH3 = r.A + r.D + 4 * r.H
    r.plain = bool(c.get("plain"))
    caps = r.t["caps"].long()
    r.target = word_or_pad(caps[:, 1:].t(), r.V0)                                # [T, B]
    r.bad_ids = bool(((caps < 0) | (caps >= r.V0))[:, :r.T].any())


# ---- comparison ---------------------------------------------------------------------------------------------------------------
class Report:
    """worst |got - ref| / bound of every named check of a stage"""

    def __init__(self):
        self.r = {}
        self.aux = {}

    def close(self, label, got, ref, bound, mask=None):
        got, ref, bound = got.double(), ref.double(), bound.double()
        got, ref, bound = torch.broadcast_tensors(got, ref, bound)
        if mask is not None:
            m = mask
            while m.dim() < got.dim():
                m = m.unsqueeze(-1)
            m = m.expand_as(got)
            got, ref, bound = got[m], ref[m], bound[m]
        same = (got == ref) | (torch.isinf(got) & torch.isinf(ref) & (torch.sign(got) == torch.sign(ref)))
        err = torch.where(same, torch.zeros_like(got), (got - ref).abs())
        ratio = torch.where(err == 0, torch.zeros_like(err), err / bound.clamp_min(1e-300))
        ratio = torch.where(torch.isfinite(got) | same, ratio, torch.full_like(ratio, float("inf")))
        w = float(ratio.max()) if ratio.numel() else 0.0
        self.r[label] = max(self.r.get(label, 0.0), w)

    def exact(self, label, got, ref, mask=None):
        got, ref = torch.broadcast_tensors(got, ref.to(got.dtype))
        if mask is not None:
            m = mask
            while m.dim() < got.dim():
                m = m.unsqueeze(-1)
            m = m.expand_as(got)
            got, ref = got[m], ref[m]
        ok = torch.equal(_bits(got), _bits(ref))
        self.r[label] = max(self.r.get(label, 0.0), 0.0 if ok else float("inf"))

    def worst(self):
        return max(self.r.values()) if self.r else 0.0


def _bits(x):
    if x.dtype in (torch.float32, torch.int32):
        return x.contiguous().view(torch.int32)
    if x.dtype in (torch.bfloat16, torch.float16, torch.int16):
        return x.contiguous().view(torch.int16)
    return x


def f64(t, k):
    return t[k].double()


# ---- forward stages -------------------------------------------------------------------------------------------------------------
def st_P(r, t):
    """P = ann Wa^T (bf16 out), K = D"""
    rep = Report()
    ref, S = mm(f64(t, "ann"), r.pw.t["Wa"])
    rep.close("P", t["P"], ref, bf16_bound(ref, acc_err(r.D, S)))
    return rep


def st_init(r, t):
    """mean over L (+ dropout 1), factorize (bf16), init (fp32)"""
    rep = Report()
    ann = f64(t, "ann")
    s = ann.sum(1)
    # fp32 sum of L terms, then * fp32(1/L) (one rounding of 1/L, one of the product) and * mask (exact: 0 or 1/(1-p) rounded,
    # the multiplier itself is taken from the mirror)
    ref = s / r.L * r.m1
    S = ann.abs().sum(1) / r.L * r.m1
    rep.close("meanv", t["meanv"], ref, bf16_bound(ref, acc_err(r.L, S) + 3 * U * ref.abs()))
    ref, S = mm(f64(t, "meanv"), r.pw.t["Wfact"])
    b = r.pw.t["bfact"].double()
    rep.close("f1", t["f1"], ref + b, bf16_bound(ref + b, acc_err(r.D + 1, S + b.abs())))
    ref, S = mm(f64(t, "f1"), r.pw.t["Winit"])
    b = r.pw.t["binit"].double()
    rep.close("init_out", t["init_out"], ref + b, acc_err(r.E + 1, S + b.abs()))
    return rep


def st_init_state(r, t):
    """init_state_kernel: the [B, 2nH0] init output read row-major as [2n, B, H0] (model.py:79-80); exact"""
    rep = Report()
    nl, H0, B = r.nl, r.H0, r.B
    io = t["init_out"][:, :2 * nl * H0].repeat_interleave(r.ncap, 0).reshape(2 * nl, B, H0)
    for l in range(nl):
        rep.exact("Hs[%d][0]" % l, t["Hs"][l, 0, :, :H0], io[l].to(torch.bfloat16))
        rep.exact("Cs[%d][0]" % l, t["Cs"][l, 0, :, :H0], io[nl + l])
        rep.exact("Hs[%d][0] pad" % l, t["Hs"][l, 0, :, H0:], torch.zeros(1, dtype=torch.bfloat16, device="cuda"))
        rep.exact("Cs[%d][0] pad" % l, t["Cs"][l, 0, :, H0:], torch.zeros(1, device="cuda"))
    return rep


def st_embed(r, t):
    """tok_init_kernel / scheduled-sampling feedback and embed_gather_kernel (+ dropout 2); exact"""
    rep = Report()
    caps = t["caps"].long()
    want = word_or_pad(caps[:, :r.T].t(), r.V0)                                  # [T, B]
    tok = t["tok"].long()
    if r.sampled:
        ra = t["row_argmax"].long()
        for s in range(1, r.T):
            if r.sampled[s]:
                fb = r.act[s - 1]                                              # rows still running at s-1 are fed its arg-max
                want[s] = torch.where(fb, word_or_pad(ra[s - 1], r.V0), want[s])
                # a row finished before s-1 is fed the logits path's arg-max of a row nothing reads; it only has to be a word
                want[s] = torch.where(fb, want[s], tok[s].clamp(0, r.V0 - 1))
    rep.exact("tok", t["tok"], want.to(torch.int32))
    x = r.pw.t["Emb"].float()[tok]
    if r.m2 is not None:
        x = x * r.m2.float()
    rep.exact("Xe", t["Xe"], x.to(torch.bfloat16))
    return rep


def st_Gx(r, t):
    rep = Report()
    ref, S = mm(f64(t, "Xe"), r.pw.t["Wihe"])
    b = r.pw.t["bg"].double()
    rep.close("Gx", t["Gx"], ref + b, acc_err(r.E + 1, S + b.abs()))
    return rep


def _top(r, t, k):
    return t[k][r.nl - 1]


def st_Q(r, t):
    """h-projection q = W_h h_t (fp32), active rows"""
    rep = Report()
    ref, S = mm(_top(r, t, "Hs")[:r.T].double(), r.pw.t["Whcat"][:r.A])
    rep.close("Q", t["Q"], ref, acc_err(r.H, S), r.act)
    return rep


def _attention_ref(r, t):
    """float64 attention of every (t, b) from the library's P, Q, ann, Hs_top; returns refs and pre-rounding bounds"""
    A, D, L = r.A, r.D, r.L
    scale = float(np.float32(1.0 / math.sqrt(L)))
    P = f64(t, "P")[r.img]                                                         # [B, L, A]
    q = f64(t, "Q")                                                                # [T, B, A]
    wf = r.pw.t["wf"].double()
    x = P[None] + q[:, :, None, :]                                                 # [T, B, L, A]
    u = torch.tanh(x)
    e = (u @ wf) * scale
    du = T_TANH * u.abs() + U * x.abs()                                            # tanh.approx + the fp32 add P + q
    de = scale * (du @ wf.abs()) + acc_err(A, scale * (u.abs() @ wf.abs())) + U * e.abs()
    alpha = torch.softmax(e, -1)
    mx = e.max(-1, keepdim=True).values
    # softmax: d alpha_l = alpha_l (de_l - sum alpha de) <= 2 alpha_l max de; plus __expf, the fp32 sum of L terms and the division
    e_sm = e_expf(e - mx).amax(-1, keepdim=True) + acc_err(L, 1.0) + U
    d_alpha = alpha * (2 * de.amax(-1, keepdim=True) + e_sm)
    ann = f64(t, "ann")[r.img]                                                     # [B, L, D]
    z = torch.einsum("tbl,bld->tbd", alpha, ann)
    sz = torch.einsum("tbl,bld->tbd", alpha, ann.abs())
    dz = torch.einsum("tbl,bld->tbd", d_alpha, ann.abs()) + acc_err(L, sz)
    if r.c.get("alpha_bf16"):
        dz = dz + R16 * sz                 # the grouped tensor-core kernels round alpha to bf16 before the context MMA
    pre, S = mm(_top(r, t, "Hs")[:r.T].double(), r.pw.t["Whcat"][A:A + D])
    pre = pre + r.pw.t["bhcat"][A:A + D].double()
    beta = torch.sigmoid(pre)
    dbeta = acc_err(r.H + 1, S + r.pw.t["bhcat"][A:A + D].double().abs()) / 4 + e_sigmoid(pre) * beta
    return SimpleNamespace(alpha=alpha, d_alpha=d_alpha, z=z, dz=dz, beta=beta, dbeta=dbeta, u=u, scale=scale)


def st_attention(r, t):
    rep = Report()
    a = _attention_ref(r, t)
    rep.close("alphas", t["alphas"].permute(1, 0, 2), a.alpha, a.d_alpha, r.act)
    rep.close("Z", t["Z"], a.z, bf16_bound(a.z, a.dz), r.act)
    rep.close("Beta", t["Beta"], a.beta, bf16_bound(a.beta, a.dbeta), r.act)
    gz = a.beta * a.z
    rep.close("GZ", t["GZ"], gz, bf16_bound(gz, a.beta * a.dz + a.z.abs() * a.dbeta + U * gz.abs()), r.act)
    return rep


def _gate_parts(pre, dpre):
    """post-activation gates i, f, g, o of gate-interleaved pre-activations and their error bounds"""
    p = [pre[..., k::4] for k in range(4)]
    dp = [dpre[..., k::4] for k in range(4)]
    g, dg = [], []
    for k in range(4):
        if k == 2:
            v = torch.tanh(p[k])
            g.append(v)
            dg.append(dp[k] + T_TANH * v.abs())
        else:
            v = torch.sigmoid(p[k])
            g.append(v)
            dg.append(dp[k] / 4 + e_sigmoid(p[k]) * v)
    return g, dg


def st_lstm(r, t):
    """gate GEMM + EpiLstm of every layer: Gates (bf16), Cs[t+1] (fp32), Hs[t+1] (bf16); finished rows frozen exactly"""
    rep = Report()
    A, D, H, T = r.A, r.D, r.H, r.T
    Hs, Cs = t["Hs"], t["Cs"]
    for l in range(r.nl):
        if l == 0:
            a, Sa = mm(f64(t, "GZ"), r.pw.t["Wihz"])
            h, Sh = mm(Hs[0, :T].double(), r.pw.t["Whcat"][A + D:A + D + 4 * H])
            gx = f64(t, "Gx")
            pre = gx + a + h
            dpre = acc_err(D + H + 1, gx.abs() + Sa + Sh) + U * pre.abs()
        else:
            Wl = r.pw.t["Wl%d" % l]
            a, Sa = mm(Hs[l - 1, 1:].double(), Wl[:, :H])
            h, Sh = mm(Hs[l, :T].double(), Wl[:, H:])
            b = r.pw.t["bgl%d" % l].double()
            pre = a + h + b
            dpre = acc_err(2 * H + 1, Sa + Sh + b.abs())
        (gi, gf, gg, go), (dgi, dgf, dgg, dgo) = _gate_parts(pre, dpre)
        G = t["Gates"][l]
        for k, (v, dv) in enumerate(((gi, dgi), (gf, dgf), (gg, dgg), (go, dgo))):
            rep.close("Gates[%d]" % l, G[..., k::4], v, bf16_bound(v, dv), r.act)
        cp = Cs[l, :T].double()
        cn = gf * cp + gi * gg
        dcn = cp.abs() * dgf + gg.abs() * dgi + gi.abs() * dgg + 2 * U * ((gf * cp).abs() + (gi * gg).abs())
        rep.close("Cs[%d]" % l, Cs[l, 1:], cn, dcn, r.act)
        rep.aux["dCs[%d]" % l] = dcn
        tc = torch.tanh(Cs[l, 1:].double())                                        # the kernel's own c_{t+1}
        hn = go * tc
        dhn = tc.abs() * dgo + go.abs() * T_TANH * tc.abs() + U * hn.abs()
        rep.close("Hs[%d]" % l, Hs[l, 1:], hn, bf16_bound(hn, dhn), r.act)
        rep.exact("Hs[%d] frozen" % l, Hs[l, 1:], Hs[l, :T], ~r.act)
        rep.exact("Cs[%d] frozen" % l, Cs[l, 1:], Cs[l, :T], ~r.act)
    return rep


def _xo_ref(r, t, h_shift=1):
    H, T = r.H, r.T
    h = _top(r, t, "Hs")[h_shift:h_shift + T].double()
    a, S = mm(h, r.pw.t["Whozo"][:, :H])
    if not r.plain:
        z, Sz = mm(f64(t, "Z"), r.pw.t["Whozo"][:, H:])
        xe = f64(t, "Xe")
        pre = xe + a + z
        dpre = acc_err(H + r.D + 1, xe.abs() + S + Sz) + U * pre.abs()
        y = torch.tanh(pre)
        dy = dpre + T_TANH * y.abs()
    else:
        y, dy = a, acc_err(H, S)
    if r.m3 is not None:
        y, dy = y * r.m3, dy * r.m3 + U * (y * r.m3).abs()
    return y, dy


def st_Xo(r, t):
    """deep output EpiTanhAdd (+ dropout 3; DeepOutput(deep=False): x = W_ho h')"""
    rep = Report()
    y, dy = _xo_ref(r, t)
    rep.close("Xo", t["Xo"], y, bf16_bound(y, dy))
    return rep


def _logits_ref(r, t):
    """float64 logits of every row from the library's Xo and Wo, [M, V]; their error bound before any rounding"""
    x, S = mm(t["Xo"].reshape(r.M, r.E), r.pw.t["Wo"])
    bo = r.pw.t["bo"]
    if bo is not None:
        b = bo.double()
        x = x + b
        S = S + torch.where(torch.isfinite(b), b.abs(), torch.zeros_like(b))
    dx = acc_err(r.E + 1, S) + U * torch.where(torch.isfinite(x), x.abs(), torch.zeros_like(x))
    return x, dx


def _lse_bound(se_terms, gaps, n):
    """log of a sum of n exponentials formed with __expf: the terms' relative errors (weighted), the fp32 sum, and __logf"""
    w = (se_terms * e_expf(gaps)).sum(-1) / se_terms.sum(-1)
    return w + acc_err(n, 1.0) + LOGF_ABS + 3 * ULP


def st_vocab(r, t):
    """fused: VOCAB_STATS tiles (max, sum exp, sum x, arg-max), row_xt, then ce_finalize_kernel (row_lse, row_loss, row_argmax)
    from the library's tiles; unfused: the bf16 logits and ce_rows_kernel from them"""
    rep = Report()
    V0, M = r.V0, r.M
    x, dx = _logits_ref(r, t)
    act = r.act.reshape(M)
    valid = torch.arange(r.V, device="cuda") < V0
    xv = torch.where(valid, x, torch.full_like(x, -math.inf))
    tgt = r.target.reshape(M)
    ls = r.c.get("ls", 0.0)
    if r.fused:
        NT = (r.V + 127) // 128
        pad = NT * 128 - r.V
        xt_ = torch.nn.functional.pad(xv, (0, pad), value=-math.inf).reshape(M, NT, 128)
        dx_ = torch.nn.functional.pad(dx, (0, pad)).reshape(M, NT, 128)
        st = t["ce_stats"].reshape(M, NT, 4)
        mx = xt_.max(-1).values
        dmx = dx_.amax(-1)
        rep.close("ce_stats max", st[..., 0], mx, dmx, act)
        # tile sum of exponentials, rescaled by the library's own maximum so that only the sum is compared
        se_ref = torch.exp(xt_ - mx[..., None]).sum(-1)
        absx = torch.where(torch.isfinite(xt_), xt_.abs(), torch.zeros_like(xt_)).amax(-1)
        # per term: the logit (2 dx, exponent and max), ex2.approx, the fma forming the exponent (u |x log2 e| and u |max log2 e|,
        # times ln 2); per tile: up to 8 rescalings / merges by ex2.approx and the fp32 sum of 128 terms
        rel = 2 * dmx + 9 * E_EX2 + 4 * U * absx + acc_err(128, 1.0)
        got_se = st[..., 1].double() * torch.exp(st[..., 0].double() - mx)
        rep.close("ce_stats sum exp", got_se, se_ref, se_ref * rel, act)
        xf = torch.where(torch.isfinite(xt_), xt_, torch.zeros_like(xt_))
        rep.close("ce_stats sum x", st[..., 2], xf.sum(-1), dx_.sum(-1) + acc_err(128, xf.abs().sum(-1)), act)
        arg = st[..., 3].contiguous().view(torch.int32).long()
        col = arg - torch.arange(NT, device="cuda")[None, :] * 128
        inside = (col >= 0) & (col < 128) & (arg < V0)
        x_at = torch.gather(xt_, 2, col.clamp(0, 127)[..., None])[..., 0]
        ok_arg = inside & (x_at >= mx - 2 * dmx)
        rep.exact("ce_stats arg-max", ok_arg | ~torch.isfinite(mx), torch.ones_like(ok_arg), act[:, None].expand_as(ok_arg))
        rep.close("row_xt", t["row_xt"], x.gather(1, tgt[:, None])[:, 0], dx.gather(1, tgt[:, None])[:, 0], act)
        # ce_finalize_kernel from the library's tiles
        gm = st[..., 0].double()
        rmx = gm.amax(-1, keepdim=True)
        terms = st[..., 1].double() * torch.exp(gm - rmx)
        lse_f = rmx[:, 0] + torch.log(terms.sum(-1))
        dl_f = _lse_bound(terms, gm - rmx, NT) + U * lse_f.abs()
        rep.close("row_lse (finalize)", t["row_lse"], lse_f, dl_f, act)
        xt = t["row_xt"].double()
        sx = st[..., 2].double().sum(-1)
        loss_f = (1 - ls) * (lse_f - xt) + ls * (lse_f - sx / V0)
        dloss_f = dl_f + 3 * U * (lse_f.abs() + xt.abs() + sx.abs() / V0) + acc_err(NT, st[..., 2].double().abs().sum(-1)) * ls / V0
        rep.close("row_loss (finalize)", t["row_loss"].reshape(M), loss_f, dloss_f, act)
        # the row's log-sum-exp against the logits: + the tiles' errors
        lse_x = torch.logsumexp(xv, -1)
        rep.close("row_lse (logits)", t["row_lse"], lse_x, dl_f + dx.amax(-1) * 2 + rel.amax(-1), act)
        lse = t["row_lse"].double()
    else:
        lg = t["logits"].reshape(M, r.V)
        rep.close("logits", lg, xv, bf16_bound(xv, dx), act[:, None] & valid[None, :])
        q = torch.where(valid, lg.double(), torch.full_like(xv, -math.inf))
        rmx = q.max(-1, keepdim=True).values
        terms = torch.exp(q - rmx)
        lse = torch.logsumexp(q, -1)
        dl = _lse_bound(terms.nan_to_num(0.0), (q - rmx).nan_to_num(0.0).clamp(-1e4, 0), r.V) + U * lse.abs()
        xt = q.gather(1, tgt[:, None])[:, 0]
        sx = torch.where(valid, lg.double(), torch.zeros_like(xv)).sum(-1)
        loss = (1 - ls) * (lse - xt) + ls * (lse - sx / V0)
        dloss = dl + 3 * U * (lse.abs() + xt.abs() + sx.abs() / V0) + acc_err(r.V, lg.double().abs().sum(-1)) * ls / V0
        rep.close("row_loss (ce_rows)", t["row_loss"].reshape(M), loss, dloss, act)
        x, dx, xv = q, torch.zeros_like(q), q                                       # the row's arg-max is over the stored logits
    # row_argmax: a maximum of the row, to within the logits' error
    ra = t["row_argmax"].reshape(M).long()
    okr = (ra >= 0) & (ra < V0)
    x_at = xv.gather(1, ra.clamp(0, r.V - 1)[:, None])[:, 0]
    okr = okr & (x_at >= xv.max(-1).values - 2 * dx.amax(-1))
    rep.exact("row_argmax", okr, torch.ones_like(okr), act)
    return rep


def st_loss(r, t):
    """alpha_sum_kernel and loss_finalize_kernel from the library's alphas, row_loss and row_argmax"""
    rep = Report()
    al = f64(t, "alphas")                                                          # [B, T, L]
    S = al.sum(1)
    rep.close("S", t["S"], S, acc_err(r.T, al.abs().sum(1)))
    out = t["out"]
    ntok = int(r.act.sum())
    rep.exact("out[5]", out[5:6], torch.tensor([float(ntok)], device="cuda"))
    rep.exact("out[4]", out[4:5], torch.tensor([1.0], device="cuda") / float(ntok))
    rep.exact("out[6]", out[6:7], torch.tensor([1.0 if r.bad_ids else 0.0], device="cuda"))
    hits = int(((t["row_argmax"].long() == t["caps"][:, 1:].t().long()) & r.act).sum())     # the raw ids, as the kernel counts
    rep.exact("out[3]", out[3:4], torch.tensor([float(hits)], device="cuda") * out[4:5])
    rl = f64(t, "row_loss")
    ce = (rl * r.act).sum() * float(out[4])
    rep.close("out[1]", out[1:2], ce.reshape(1), (acc_err(ntok, (rl.abs() * r.act).sum()) * float(out[4]) + U * ce.abs()).reshape(1))
    Sl = f64(t, "S")
    reg = ((1 - Sl) ** 2).sum() / (r.B * r.L)
    dreg = acc_err(r.B * r.L, ((1 - Sl) ** 2).sum()) / (r.B * r.L) + 4 * U * reg + 2 * U * ((1 - Sl).abs() * (1 + Sl.abs())).sum() / (r.B * r.L)
    rep.close("out[2]", out[2:3], reg.reshape(1), dreg.reshape(1))
    o0 = out[1].double() + out[2].double()                                         # att_gamma = 1
    rep.close("out[0]", out[0:1], o0.reshape(1), (2 * U * (out[1].double().abs() + out[2].double().abs())).reshape(1))
    return rep


def st_dlogits(r, t):
    """VOCAB_DLOGITS pass (fused) or ce_rows_kernel (unfused): (softmax - target distribution) / N_tok, bf16"""
    rep = Report()
    M, V0, V = r.M, r.V0, r.V
    act = r.act.reshape(M)
    valid = torch.arange(V, device="cuda") < V0
    ls = r.c.get("ls", 0.0)
    inv = float(t["out"][4])
    tgt = r.target.reshape(M)
    if r.fused:
        x, dx = _logits_ref(r, t)
        lse = f64(t, "row_lse")
        dlse = torch.zeros_like(lse)
    else:
        x = t["logits"].reshape(M, V).double()
        dx = torch.zeros_like(x)
        lse = torch.logsumexp(torch.where(valid, x, torch.full_like(x, -math.inf)), -1)
        dlse = st_vocab_lse_bound(r, t, x, valid)
    arg = (x - lse[:, None]).clamp(max=80.0)
    pe = torch.exp(arg)
    onehot = torch.zeros_like(x).scatter_(1, tgt[:, None], 1.0)
    p = pe - ls / V0 - (1 - ls) * onehot
    ref = p * inv
    # exponential: the logit and lse errors, ex2.approx / __expf, the fma forming the exponent; then the subtractions and * inv
    dpe = pe * (dx + dlse[:, None] + E_EX2 + e_expf(arg) + 2 * U * (x.abs().nan_to_num(0.0) + lse.abs()[:, None]))
    dref = (dpe + 2 * U * (pe + 1)) * inv + U * ref.abs()
    got = t["dlogits"].reshape(M, V)
    m = act[:, None] & valid[None, :]
    rep.close("dlogits", got, ref, bf16_bound(ref, dref), m)
    return rep


def st_vocab_lse_bound(r, t, q, valid):
    qv = torch.where(valid, q, torch.full_like(q, -math.inf))
    rmx = qv.max(-1, keepdim=True).values
    terms = torch.exp(qv - rmx)
    lse = torch.logsumexp(qv, -1)
    return _lse_bound(terms, (qv - rmx).clamp(-1e4, 0), r.V) + U * lse.abs()


# ---- backward stages ------------------------------------------------------------------------------------------------------------
def st_dpre(r, t):
    """EpiDpre: gscale * mask3 * (dlogits Wo) * (1 - x^2), x = Xo (1 - p); bf16.  Then dHZ = dpre [W_ho | W_zo] (fp32)"""
    rep = Report()
    dl = t["dlogits"].reshape(r.T, r.B, r.V).double()
    acc, S = mm(dl, r.pw.t["WoT"])
    xo = f64(t, "Xo")
    x = torch.zeros_like(xo) if r.plain else (xo * r.keep if r.m3 is not None else xo)
    k = r.m3 if r.m3 is not None else torch.ones_like(xo)
    f = 1 - x * x
    ref = GSCALE * k * acc * f
    dref = GSCALE * k * (f.abs() * acc_err(r.V, S) + acc.abs() * 4 * U * (x * x + 1)) + 4 * U * ref.abs()
    rep.close("dpre", t["dpre"], ref, bf16_bound(ref, dref))
    ref, S = mm(f64(t, "dpre"), r.pw.t["WhozoT"])
    rep.close("dHZ", t["dHZ"], ref, acc_err(r.E, S))
    return rep


def _dG(r, t, l):
    """pre-activation gate gradients of layer l as the library stored them, [T, B, 4H] (bf16)"""
    return t["DY"][..., r.A + r.D:] if l == 0 else t["dGl"][l - 1]


def _lstm_bwd(r, t):
    """replays lstm_bwd_step_kernel of every layer and step, with dc carried in float64; returns the per-stage report and the
    state gradients (and their bounds) left at step 0"""
    rep = Report()
    A, D, H, T, B, nl = r.A, r.D, r.H, r.T, r.B, r.nl
    zero_row = torch.zeros(1, B, 4 * H, dtype=torch.bfloat16, device="cuda")
    Whc = r.pw.t["Whcat"]
    dh_in, ddh_in = {}, {}
    for l in range(nl):
        # grad wrt the new state h_{t+1} of layer l, from the library's own saved gradients, for t = -1 .. T-1 (index t + 1)
        nxt = torch.cat([_dG(r, t, l), zero_row], 0)                                # dG_l of step t+1 (zero after the last)
        Wrec = Whc[A + D:A + D + 4 * H] if l == 0 else r.pw.t["Wl%d" % l][:, H:]
        v, S = mm(nxt.double(), Wrec.t().contiguous())                              # [T+1, B, H]: index s = own step s
        K = 4 * H
        if l == nl - 1:
            dy = torch.cat([t["DY"][..., :A + D], torch.zeros(1, B, A + D, dtype=torch.bfloat16, device="cuda")], 0)
            a2, S2 = mm(dy.double(), Whc[:A + D].t().contiguous())
            v, S, K = v + a2, S + S2, K + A + D
        # index s of v holds what step s's consumers send to h_s, the state entering step s = the state left by step s-1
        dh = torch.zeros(T + 1, B, H, dtype=torch.float64, device="cuda")
        Sdh = torch.zeros_like(dh)
        dh[:] = v
        Sdh[:] = S
        if l == nl - 1:
            hz = t["dHZ"][..., :H].double()
            dh[1:] += hz
            Sdh[1:] += hz.abs()
        if l < nl - 1:
            up, S3 = mm(_dG(r, t, l + 1).double(), r.pw.t["Wl%d" % (l + 1)][:, :H].t().contiguous())
            dh[1:] += up
            Sdh[1:] += S3
            K += 4 * H
        dh_in[l], ddh_in[l] = dh, acc_err(K + 1, Sdh)
    dc0, ddc0 = {}, {}
    for l in range(nl):
        G = t["Gates"][l].double()
        Cs = t["Cs"][l].double()
        dGl = _dG(r, t, l)
        dc = torch.zeros(B, H, dtype=torch.float64, device="cuda")
        ddc = torch.zeros_like(dc)
        for s in range(T - 1, -1, -1):
            a = r.act[s][:, None]
            gi, gf, gg, go = (G[s][..., k::4] for k in range(4))
            tc = torch.tanh(Cs[s + 1])
            dht, ddht = dh_in[l][s + 1], ddh_in[l][s + 1]
            f1 = go * (1 - tc * tc)
            dct = dc + dht * f1
            # tanh.approx of c_{t+1}: |d(1 - tc^2)| <= 2 tc^2 T_TANH
            ddct = ddc + ddht * f1.abs() + (dht * go).abs() * 2 * tc * tc * T_TANH + 3 * U * (dc.abs() + (dht * f1).abs())
            refs = (dct * gg * gi * (1 - gi), dct * Cs[s] * gf * (1 - gf), dct * gi * (1 - gg * gg), dht * tc * go * (1 - go))
            facs = ((gg * gi * (1 - gi)).abs(), (Cs[s] * gf * (1 - gf)).abs(), (gi * (1 - gg * gg)).abs(), None)
            for k in range(4):
                if k < 3:
                    d = ddct * facs[k] + 5 * U * refs[k].abs()
                else:
                    d = ddht * (tc * go * (1 - go)).abs() + dht.abs() * T_TANH * (tc * go * (1 - go)).abs() + 5 * U * refs[k].abs()
                rep.close("dG[%d]" % l, dGl[s][..., k::4], refs[k], bf16_bound(refs[k], d), a)
            dc = torch.where(a, dct * gf, dc)
            ddc = torch.where(a, ddct * gf + U * (dct * gf).abs(), ddc)
        dc0[l], ddc0[l] = dc, ddc
    return rep, SimpleNamespace(dh0={l: dh_in[l][0] for l in range(nl)}, ddh0={l: ddh_in[l][0] for l in range(nl)}, dc0=dc0, ddc0=ddc0)


def st_lstm_bwd(r, t):
    return _lstm_bwd(r, t)[0]


def st_dP(r, t):
    """dP_deferred_kernel: dP[b,l,a] = sum_t de[t,b,l] wf[a] (1 - tanh^2(P + q_t)) (fp32); dP16 = bf16(dP) exactly"""
    rep = Report()
    P = f64(t, "P")[r.img]
    q = f64(t, "Q")
    wf = r.pw.t["wf"].double()
    de = f64(t, "de")                                                              # [T, B, L]
    x = P[None] + q[:, :, None, :]
    u = torch.tanh(x)
    g = wf * (1 - u * u)
    ref = torch.einsum("tbl,tbla->bla", de, g)
    dg = wf.abs() * (2 * u * u * T_TANH + 4 * U * (u * u + 1) + 2 * U * x.abs())
    dref = torch.einsum("tbl,tbla->bla", de.abs(), dg) + acc_err(r.T, torch.einsum("tbl,tbla->bla", de.abs(), g.abs()))
    rep.close("dP", t["dP"], ref, dref)
    if r.c.get("use_tc", True):                                                    # SIMT: d_ann reads dP itself
        rep.exact("dP16", t["dP16"], t["dP"].to(torch.bfloat16))
    return rep


def st_dXe(r, t):
    """dXe = dG Wihe + dpre (deep output), then * mask 2 (fp32)"""
    rep = Report()
    acc, S = mm(_dG(r, t, 0).double(), r.pw.t["WiheT"])
    if not r.plain:
        dp = f64(t, "dpre")
        acc, S = acc + dp, S + dp.abs()
    k = r.m2 if r.m2 is not None else 1.0
    rep.close("dXe", t["dXe"], acc * k, acc_err(4 * r.H + 1, S) * k)
    return rep


def st_init_bwd(r, t):
    """init_state_bwd_kernel (inverse reinterpretation, sum over the captions of an image) and the two init GEMMs"""
    rep = Report()
    _, s = _lstm_bwd(r, t)
    nl, H0, B, Bi = r.nl, r.H0, r.B, r.Bi
    g = torch.stack([s.dh0[l][:, :H0] for l in range(nl)] + [s.dc0[l][:, :H0] for l in range(nl)])
    dg = torch.stack([s.ddh0[l][:, :H0] for l in range(nl)] + [s.ddc0[l][:, :H0] for l in range(nl)])
    g = g.reshape(B, 2 * nl * H0).reshape(Bi, r.ncap, -1).sum(1)
    dg = dg.reshape(B, 2 * nl * H0).reshape(Bi, r.ncap, -1).sum(1) + acc_err(r.ncap, g.abs())
    IO = 2 * nl * r.H
    ref = torch.zeros(Bi, IO, dtype=torch.float64, device="cuda")
    dref = torch.zeros_like(ref)
    ref[:, :g.shape[1]], dref[:, :g.shape[1]] = g, dg
    rep.close("d_init_out", t["d_init_out"], ref, dref)
    tc = r.c.get("use_tc", True)
    if tc:
        rep.exact("d_init_out16", t["d_init_out16"], t["d_init_out"].to(torch.bfloat16))
    a = t["d_init_out16"] if tc else t["d_init_out"]
    ref, S = mm(a.double(), r.pw.t["WinitT"])
    rep.close("df1", t["df1"], ref, acc_err(IO, S))
    if tc:
        rep.exact("df116", t["df116"], t["df1"].to(torch.bfloat16))
    a = t["df116"] if tc else t["df1"]
    ref, S = mm(a.double(), r.pw.t["WfactT"])
    rep.close("dmean", t["dmean"], ref * r.m1, acc_err(r.E, S) * r.m1)
    return rep


def st_d_ann(r, t):
    """dann_alpha_kernel (sum_t alpha dZ + dmean / (L ncap), bf16) + dP16 Wa added in place (second bf16 rounding); the SIMT
    path does both in one fp32 epilogue from dP"""
    rep = Report()
    al = f64(t, "alphas")                                                          # [B, T, L]
    dZ = f64(t, "dZ")                                                              # [T, B, D]
    part = torch.einsum("btl,tbd->bld", al, dZ) + (f64(t, "dmean")[r.img] / (r.L * r.ncap))[:, None, :]
    spart = torch.einsum("btl,tbd->bld", al.abs(), dZ.abs()) + (f64(t, "dmean")[r.img].abs() / (r.L * r.ncap))[:, None, :]
    tc = r.c.get("use_tc", True)
    dP = f64(t, "dP16" if tc else "dP")
    g, S = mm(dP, r.pw.t["WaT"])
    ref = part + g
    d1 = acc_err(r.T + 1, spart) + 2 * U * part.abs()
    if tc:
        dref = R16 * part.abs() * (1 + R16) + d1 + acc_err(r.A + 1, S)
        rep.close("d_ann", t["d_ann"], ref, bf16_bound(ref, dref))
    else:
        rep.close("d_ann", t["d_ann"], ref, bf16_bound(ref, d1 + acc_err(r.A, S)))
    return rep


def st_attn_bwd(r, t):
    """dgz GEMM (dG Wihz, split-K partials summed by the consumer) + the attention backward of every step, running rows:
        dz = dHZ[:, H:] + dgz beta            -> dZ (bf16)          dbeta_pre = dgz z beta (1 - beta) -> DY[:, A:A+D] (bf16)
        dalpha_l = a_l . dz + g gamma (-2)(1 - S_l) / (B L)         de_l = scale alpha_l (dalpha_l - sum alpha dalpha) (fp32)
        dq_a = sum_l de_l wf_a (1 - u_la^2) -> DY[:, :A] (bf16)     dwf_a = sum_l de_l u_la -> dwf_part (fp32)
    dz, dalpha and de are replayed as one chain from the saved forward buffers; dq and dwf from the library's de (checked here too)"""
    rep = Report()
    A, D, H, L, B = r.A, r.D, r.H, r.L, r.B
    dg, S = mm(_dG(r, t, 0).double(), r.pw.t["WihzT"])                            # [T, B, D], K = 4H
    ddg = acc_err(4 * H, S)
    beta, z = f64(t, "Beta"), f64(t, "Z")
    dz = t["dHZ"][..., H:].double() + dg * beta
    ddz = beta * ddg + 2 * U * dz.abs()
    rep.close("dZ", t["dZ"], dz, bf16_bound(dz, ddz), r.act)
    f = z * beta * (1 - beta)
    dbp = dg * f
    rep.close("DY dbeta", t["DY"][..., A:A + D], dbp, bf16_bound(dbp, f.abs() * ddg + 4 * U * dbp.abs()), r.act)
    ann = f64(t, "ann")[r.img]                                                     # [B, L, D]
    regc = float(np.float32(GSCALE * 1.0 * -2.0) / np.float32(B * L))              # g * att_gamma * (-2) / (B L) in fp32
    reg = regc * (1 - f64(t, "S"))[None]                                           # [1, B, L]
    dal = torch.einsum("tbd,bld->tbl", dz, ann) + reg
    ddal = (torch.einsum("tbd,bld->tbl", ddz, ann.abs()) + acc_err(D, torch.einsum("tbd,bld->tbl", dz.abs(), ann.abs()))
            + 3 * U * (reg.abs() + dal.abs()))
    al = t["alphas"].permute(1, 0, 2).double()                                     # [T, B, L]
    scale = float(np.float32(1.0 / math.sqrt(L)))
    dot = (al * dal).sum(-1, keepdim=True)
    de = al * (dal - dot) * scale
    dde = scale * al * (ddal + (al * ddal).sum(-1, keepdim=True) + acc_err(L, (al * dal.abs()).sum(-1, keepdim=True))
                        + 3 * U * (dal.abs() + dot.abs())) + 2 * U * de.abs()
    rep.close("de", t["de"], de, dde, r.act)
    rep.aux["de"] = dde
    x = f64(t, "P")[r.img][None] + f64(t, "Q")[:, :, None, :]                     # [T, B, L, A]
    u = torch.tanh(x)
    wf = r.pw.t["wf"].double()
    e = f64(t, "de")
    w1 = wf * (1 - u * u)
    dq = torch.einsum("tbl,tbla->tba", e, w1)
    ddq = (torch.einsum("tbl,tbla->tba", e.abs(), wf.abs() * (2 * u * u * T_TANH + 4 * U * (u * u + 1) + 2 * U * x.abs()))
           + acc_err(L, torch.einsum("tbl,tbla->tba", e.abs(), w1.abs())))
    rep.close("DY dq", t["DY"][..., :A], dq, bf16_bound(dq, ddq), r.act)
    dw = torch.einsum("tbl,tbla->tba", e, u)
    ddw = torch.einsum("tbl,tbla->tba", e.abs(), T_TANH * u.abs() + U * x.abs()) + acc_err(L, torch.einsum("tbl,tbla->tba", e.abs(), u.abs()))
    rep.close("dwf_part", t["dwf_part"], dw, ddw, r.act)
    return rep


def _deint(x, H, H0):
    """gate-interleaved rows (4j + g) -> torch order (g H0 + j), cropped to the true decoder_dim"""
    return x.reshape(H, 4, *x.shape[1:])[:H0].transpose(0, 1).reshape(4 * H0, *x.shape[1:])


def st_param_grads(r, t):
    """sat_train_param_grads: every gradient as float64 X^T dY of the library's own operand pairs (sat_param_grads.cu), with the
    ncap sum of dP rounded as ncap_sum_kernel rounds it, the column sums, the embedding segment sum (pad row zero, tying added),
    the de-interleave, the crop to the true dims and gscale (applied to dW_o / db_o only: dpre already carries it)"""
    rep = Report()
    G = t["_G"]
    A, D, H, T, nl = r.A, r.D, r.H, r.T, r.nl
    A0, D0, H0, E0, V0 = r.A0, r.D0, r.H0, r.E0, r.V0
    g = GSCALE

    def nt(X, Y):
        X = X.reshape(-1, X.shape[-1]).double()
        Y = Y.reshape(-1, Y.shape[-1]).double()
        return X.t() @ Y, X.abs().t() @ Y.abs(), X.shape[0]

    def cs(X):
        X = X.reshape(-1, X.shape[-1]).double()
        return X.sum(0), X.abs().sum(0), X.shape[0]

    def check(name, ref, S, K, scale=1.0):
        rep.close(name, G[name].reshape(ref.shape), ref * scale, acc_err(K, S) * scale + U * (ref * scale).abs())

    Hs, Htop = t["Hs"], t["Hs"][nl - 1]
    dl = t["dlogits"]
    wo, wo_s, K = nt(dl, t["Xo"])
    tied = bool(r.c.get("tied"))
    if not tied:
        check("output.output.weight", wo[:V0, :E0], wo_s[:V0, :E0], K, g)
    if "output.output.bias" in G:
        c, c_s, K = cs(dl)
        check("output.output.bias", c[:V0], c_s[:V0], K, g)
    # embedding: dXe rows summed by the word fed at that row; <PAD> (row 0) stays zero
    tok = t["tok"].reshape(-1).long()
    dxe = t["dXe"].reshape(-1, r.E).double()
    emb = torch.zeros(r.V, r.E, dtype=torch.float64, device="cuda").index_add_(0, tok, dxe)
    emb_s = torch.zeros_like(emb).index_add_(0, tok, dxe.abs())
    emb[0], emb_s[0] = 0.0, 0.0
    emb, emb_s = emb[:V0, :E0], emb_s[:V0, :E0]
    if tied:
        emb, emb_s = emb + g * wo[:V0, :E0], emb_s + g * wo_s[:V0, :E0]
    check("embedding.weight", emb, emb_s, r.M)
    a, s, K = nt(t["dpre"], Htop[1:])
    check("output.hidden.weight", a[:E0, :H0], s[:E0, :H0], K)
    if not r.plain:
        a, s, K = nt(t["dpre"], t["Z"])
        check("output.context.weight", a[:E0, :D0], s[:E0, :D0], K)
    DY = t["DY"]
    a, s, K = nt(DY[..., :A], Htop[:T])
    check("attention.decoder_att.weight", a[:A0, :H0], s[:A0, :H0], K)
    a, s, K = nt(DY[..., A:A + D], Htop[:T])
    check("beta.0.weight", a[:D0, :H0], s[:D0, :H0], K)
    c, c_s, K = cs(DY[..., A:A + D])
    check("beta.0.bias", c[:D0], c_s[:D0], K)
    dG = DY[..., A + D:]
    a, s, K = nt(dG, Hs[0, :T])
    check("lstm.weight_hh_l0", _deint(a, H, H0)[:, :H0], _deint(s, H, H0)[:, :H0], K)
    c, c_s, K = cs(dG)
    for name in ("lstm.bias_ih_l0", "lstm.bias_hh_l0"):
        check(name, _deint(c, H, H0), _deint(c_s, H, H0), K)
    a, s, K = nt(dG, t["Xe"])
    b, bs, _ = nt(dG, t["GZ"])
    wih = torch.cat([_deint(a, H, H0)[:, :E0], _deint(b, H, H0)[:, :D0]], 1)
    wih_s = torch.cat([_deint(s, H, H0)[:, :E0], _deint(bs, H, H0)[:, :D0]], 1)
    check("lstm.weight_ih_l0", wih, wih_s, K)
    for l in range(1, nl):
        dGl = t["dGl"][l - 1]
        a, s, K = nt(dGl, Hs[l - 1, 1:])
        check("lstm.weight_ih_l%d" % l, _deint(a, H, H0)[:, :H0], _deint(s, H, H0)[:, :H0], K)
        a, s, K = nt(dGl, Hs[l, :T])
        check("lstm.weight_hh_l%d" % l, _deint(a, H, H0)[:, :H0], _deint(s, H, H0)[:, :H0], K)
        c, c_s, K = cs(dGl)
        for name in ("lstm.bias_ih_l%d" % l, "lstm.bias_hh_l%d" % l):
            check(name, _deint(c, H, H0), _deint(c_s, H, H0), K)
    # dW_a = dP_img^T ann over the Bi*L image locations; dP_img = the captions' dP summed in fp32 (in caption order), rounded to the
    # operand dtype on the tensor-core path
    tc = r.c.get("use_tc", True)
    if r.ncap > 1:
        x = t["dP"].reshape(r.Bi, r.ncap, r.L, A)
        dpi = x[:, 0]
        for k in range(1, r.ncap):
            dpi = dpi + x[:, k]
        dpi = dpi.to(torch.bfloat16) if tc else dpi
    else:
        dpi = t["dP16"] if tc else t["dP"]
    a, s, K = nt(dpi, t["ann"])
    check("attention.encoder_att.weight", a[:A0, :D0], s[:A0, :D0], K + r.ncap)
    c, c_s, K = cs(t["dwf_part"])
    check("attention.f_att.weight", c[:A0], c_s[:A0], K)
    IO0 = 2 * nl * H0
    a, s, K = nt(t["d_init_out16"] if tc else t["d_init_out"], t["f1"])
    check("init_lstm.init.weight", a[:IO0, :E0], s[:IO0, :E0], K)
    c, c_s, K = cs(t["d_init_out"])
    check("init_lstm.init.bias", c[:IO0], c_s[:IO0], K)
    a, s, K = nt(t["df116"] if tc else t["df1"], t["meanv"])
    check("init_lstm.factorize.weight", a[:E0, :D0], s[:E0, :D0], K)
    c, c_s, K = cs(t["df1"])
    check("init_lstm.factorize.bias", c[:E0], c_s[:E0], K)
    missing = set(G) - set(rep.r)
    rep.r.update({"unchecked " + k: float("inf") for k in missing})
    return rep


STAGES = dict(P=st_P, init=st_init, init_state=st_init_state, embed=st_embed, Gx=st_Gx, Q=st_Q, attention=st_attention,
              lstm=st_lstm, Xo=st_Xo, vocab=st_vocab, loss=st_loss, dlogits=st_dlogits, dpre=st_dpre, lstm_bwd=st_lstm_bwd,
              attn_bwd=st_attn_bwd, dP=st_dP, dXe=st_dXe, init_bwd=st_init_bwd, d_ann=st_d_ann, param_grads=st_param_grads)


def _show(name, stage, rep):
    worst = max(rep.r.items(), key=lambda kv: kv[1]) if rep.r else ("-", 0.0)
    print("\n  %-16s %-11s worst error / bound %.3g (%s)  [%s]" % (name, stage, worst[1], worst[0],
                                                                   ", ".join("%s %.2g" % kv for kv in rep.r.items())), end="")


@pytest.mark.parametrize("stage", list(STAGES))
@pytest.mark.parametrize("name", NAMES)
def test_stage_replay(name, stage):
    r = run(name)
    rep = STAGES[stage](r, dict(r.t, _G=r.G))
    _show(name, stage, rep)
    bad = {k: v for k, v in rep.r.items() if not v <= 1.0}
    assert not bad, bad


# ---- invariants ---------------------------------------------------------------------------------------------------------------
# rows with t >= lens[b]: exactly zero.  [T, B, ...] time-major buffers unless named otherwise.  Not `de`: the attention
# backward writes de_t for running rows only, and dP_deferred_kernel reads steps t < lens[b] only (the poisoned run checks that
# nothing reads the rest).
INACTIVE_ZERO = ("DY", "dlogits", "dpre", "dZ", "dwf_part", "row_loss")
# padded lanes: exactly zero (buffer -> (dimension letter of its last axis, offset of the lane block))
# Not listed, with reason: Beta (padded lanes hold sigmoid(0) = 0.5: zero weights and bias give beta_pre = 0), Gates of active
# rows (padded units' i, f, o gates are sigmoid(0) = 0.5), Gx / dHZ / init_out (the padded lanes are zero, but by the zero weights
# of a GEMM the checks above replay anyway).


def _pad_views(r, t):
    """(label, view of padded lanes) for every buffer whose padded lanes must be zero"""
    A, A0, D, D0, H, H0, E, E0 = r.A, r.A0, r.D, r.D0, r.H, r.H0, r.E, r.E0
    v = [("P", t["P"][..., A0:]), ("Q", t["Q"][..., A0:]), ("Hs", t["Hs"][..., H0:]), ("Cs", t["Cs"][..., H0:]),
         ("Z", t["Z"][..., D0:]), ("GZ", t["GZ"][..., D0:]), ("Xo", t["Xo"][..., E0:]),
         ("DY dq", t["DY"][..., A0:A]), ("DY dbeta", t["DY"][..., A + D0:A + D]), ("dZ", t["dZ"][..., D0:]),
         ("dHZ h", t["dHZ"][..., H0:H]), ("dHZ z", t["dHZ"][..., H + D0:]), ("dXe", t["dXe"][..., E0:]), ("dP", t["dP"][..., A0:]),
         ("d_ann", t["d_ann"][..., D0:]), ("dlogits", t["dlogits"][..., r.V0:])]
    dG = t["DY"][..., A + D:].reshape(r.T, r.B, H, 4)[:, :, H0:]
    v.append(("DY dG", dG))
    if r.nl > 1:
        v.append(("dGl", t["dGl"].reshape(r.nl - 1, r.T, r.B, H, 4)[:, :, :, H0:]))
    return v


@pytest.mark.parametrize("name", NAMES)
def test_invariants(name):
    r = run(name)
    t = r.t
    bad = []
    inact = ~r.act
    for k in INACTIVE_ZERO:
        x = t[k].reshape(r.T, r.B, -1)
        if bool((x[inact] != 0).any()):
            bad.append("%s: nonzero in a finished row" % k)
    if r.nl > 1 and bool((t["dGl"][:, inact] != 0).any()):
        bad.append("dGl: nonzero in a finished row")
    if bool((t["Gates"][:, inact] != 0).any()):
        bad.append("Gates: nonzero in a finished row")
    if bool((t["alphas"].permute(1, 0, 2)[inact] != 0).any()):
        bad.append("alphas: nonzero in a finished row")
    if bool((t["row_argmax"][inact] != -1).any()):
        bad.append("row_argmax: not -1 in a finished row")
    for label, x in _pad_views(r, t):
        if x.numel() and bool((x != 0).any()):
            bad.append("%s: nonzero padded lane" % label)
    read = ["P", "meanv", "f1", "init_out", "Xe", "Gx", "Hs", "Cs", "Q", "alphas", "Z", "GZ", "Beta", "Gates", "Xo", "row_loss", "S",
            "out", "dlogits", "dpre", "dHZ", "DY", "dZ", "dP", "de", "dwf_part", "dXe", "d_init_out", "df1", "dmean", "d_ann"]
    read += ["ce_stats", "row_lse", "row_xt"] if r.fused else ["logits"]
    read += ["dGl"] if r.nl > 1 else []
    for k in read:
        x = t[k]
        if k == "ce_stats":
            x = x[..., :3].reshape(r.M, -1)[r.act.reshape(-1)]                     # finished rows' tiles are never written
        elif k in ("row_lse", "row_xt"):
            x = x[r.act.reshape(-1)]
        elif k == "logits":
            x = x[..., :r.V0]                                                      # padded words hold -inf by design
        if not bool(torch.isfinite(x.float()).all()):
            bad.append("%s: non-finite values" % k)
    for k, v in r.G.items():
        if not bool(torch.isfinite(v).all()):
            bad.append("grad %s: non-finite" % k)
    assert not bad, bad


# ---- poisoned buffers ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", NAMES)
def test_nan_filled_buffers_give_the_same_step(name):
    """every floating-point work buffer NaN-filled (index buffers 0) vs zero-filled: bit-identical results"""
    a = run(name)
    b = _step(name, "nan")
    diff = []
    for k, v in a.t.items():
        if k in SCRATCH or k in ("ann", "caps", "lens", "gscale_in"):
            continue
        if k in SIMT_UNUSED and not a.c.get("use_tc", True):
            continue
        w = b.t[k]
        if k == "ce_stats":                                  # finished rows' tiles are written by no kernel and read by none
            m = a.act.reshape(-1)
            v, w = v.reshape(a.M, -1)[m], w.reshape(a.M, -1)[m]
        elif k == "row_xt":                                  # written for running rows only, read for those only
            m = a.act.reshape(-1)
            v, w = v[m], w[m]
        elif k == "de":                                      # the same (see INACTIVE_ZERO)
            v, w = v[a.act], w[a.act]
        if not torch.equal(_bits(v), _bits(w)):
            diff.append(k)
    for k in a.G:
        if not torch.equal(_bits(a.G[k]), _bits(b.G[k])):
            diff.append("grad " + k)
    if not torch.equal(_bits(a.d_ann.float()), _bits(b.d_ann.float())):
        diff.append("d_ann (host sum)")
    del b
    torch.cuda.empty_cache()
    assert not diff, diff


# ---- out-of-range word ids on the fused path ------------------------------------------------------------------------------------
def test_bad_ids_fused_path_matches_the_unfused_path():
    """the fused path (badid) against the logits path (badid_rows) on the same out-of-range ids.  Both steps are identical up to
    Xo (same kernels, same inputs); every stage of each, the parameter gradients included, is replayed at its own bounds by
    test_stage_replay.  Here the two cross entropies are compared with each other: the logits path rounds each logit x_j to
    bf16 first, which moves it by at most R16 |x_j|, so the log-sum-exp, the target logit and the mean logit each move by at most
    R16 max|x| and every soft-max probability by a factor within exp(+-2 R16 max|x|)."""
    r, u = run("badid"), run("badid_rows")
    assert r.fused and not u.fused and r.bad_ids
    assert float(r.t["out"][6]) == 1.0 and float(u.t["out"][6]) == 1.0
    assert bool(torch.isfinite(r.t["out"]).all()) and all(bool(torch.isfinite(g).all()) for g in r.G.values())
    assert torch.equal(_bits(r.t["Xo"]), _bits(u.t["Xo"]))
    x, dx = _logits_ref(r, r.t)
    xmax = torch.where(torch.isfinite(x), x.abs(), torch.zeros_like(x)).amax(-1).reshape(r.T, r.B)
    mv = R16 * xmax * (1 + R16) + dx.amax(-1).reshape(r.T, r.B)                    # largest move of a logit between the paths
    # + the fused loss's own finalize bound (a few fp32 ulps of the loss): 8 u |loss|
    rl, ul = r.t["row_loss"].double(), u.t["row_loss"].double()
    assert bool((((rl - ul).abs() <= 3 * mv + 8 * U * rl.abs()) | ~r.act).all())
    inv = float(r.t["out"][4])
    df, du = r.t["dlogits"][..., :r.V0].double(), u.t["dlogits"][..., :r.V0].double()
    # |d p| <= (exp(2 mv) - 1) p, p <= |dlogits| / inv + 1 (the target and smoothing terms), then each path's bf16 rounding
    bound = (torch.exp(2 * mv) - 1)[..., None] * (du.abs() + inv) + R16 * (1 + R16) * (df.abs() + du.abs())
    assert bool(((df - du).abs() <= bound).all())
    # dW_o and db_o are linear in dlogits with the same Xo on both paths (times gscale)
    dd = bound.reshape(r.M, -1)
    xo = r.t["Xo"].reshape(r.M, r.E)[:, :r.E0].double()
    bw = GSCALE * (dd.t() @ xo.abs()) + acc_err(r.M, GSCALE * (df.abs() + du.abs()).reshape(r.M, -1).t() @ xo.abs())
    assert bool(((r.G["output.output.weight"].double() - u.G["output.output.weight"].double()).abs() <= bw).all())
    bb = GSCALE * dd.sum(0) + acc_err(r.M, GSCALE * (df.abs() + du.abs()).reshape(r.M, -1).sum(0))
    assert bool(((r.G["output.output.bias"].double() - u.G["output.output.bias"].double()).abs() <= bb).all())


# ---- mutations: the smallest defect each stage check claims to catch -----------------------------------------------------------
def _argmax_flat(x, mask=None):
    a = x.float().abs()
    if mask is not None:
        a = torch.where(mask, a, torch.zeros_like(a))
    return np.unravel_index(int(a.reshape(-1).argmax()), tuple(x.shape))


def _bf16_ulps(x, idx, n):
    y = x.clone()
    y.view(torch.int16)[idx] += n
    return y


def _mul(x, idx, f):
    y = x.clone()
    y[idx] = y[idx] * f
    return y


def _act_mask(r, shape_tail):
    m = r.act
    for s in shape_tail:
        m = m.unsqueeze(-1).expand(*m.shape, s)
    return m


def m_P(r, t):
    t["P"] = _bf16_ulps(t["P"], _argmax_flat(t["P"]), 2)
    return "P"


def m_meanv(r, t):
    t["meanv"] = _bf16_ulps(t["meanv"], _argmax_flat(t["meanv"]), 2)
    return "init"


def m_init_out(r, t):
    t["init_out"] = _mul(t["init_out"], _argmax_flat(t["init_out"]), 1 + 1e-4)
    return "init"


def m_h0(r, t):
    t["Hs"] = _bf16_ulps(t["Hs"], (0, 0, 0, 0), 1)
    return "init_state"


def m_Xe(r, t):
    t["Xe"] = _bf16_ulps(t["Xe"], _argmax_flat(t["Xe"]), 1)
    return "embed"


def m_Gx(r, t):
    t["Gx"] = _mul(t["Gx"], _argmax_flat(t["Gx"]), 1 + 1e-4)
    return "Gx"


def m_Q(r, t):
    t["Q"] = _mul(t["Q"], _argmax_flat(t["Q"], _act_mask(r, [r.A])), 1 + 1e-4)
    return "Q"


def m_alpha(r, t):
    al = t["alphas"].clone()
    b = int(torch.nonzero(r.act[0])[0])
    row = al[b, 0]
    i, j = int(row.argmax()), int(row.argmin())
    row[i], row[j] = row[j].clone(), row[i].clone()
    t["alphas"] = al
    return "attention"


def m_Cs(r, t):
    # ×(1 + 1e-4) on the cell state whose check is the most sensitive (largest |c| / bound): where |i g| is large, tanh.approx's
    # 2^-11 relative error in g alone allows more than 1e-4 |c| (the -s output prints the worst Cs ratio of the real kernels)
    dcn = st_lstm(r, r.t).aux["dCs[0]"]
    sens = torch.where(r.act[..., None], t["Cs"][0, 1:].double().abs() / dcn, torch.zeros_like(dcn))
    idx = np.unravel_index(int(sens.reshape(-1).argmax()), tuple(sens.shape))
    c = t["Cs"].clone()
    c[(0, idx[0] + 1) + tuple(idx[1:])] *= 1 + 1e-4
    t["Cs"] = c
    return "lstm"


def m_de(r, t):
    """one de element x (1 + 1e-3), where the de check is the most sensitive.  Not 1e-4: de_l = alpha_l (dalpha_l - sum alpha
    dalpha) cancels, and the fp32 accumulation of dalpha over D alone allows more than 1e-4 |de| (the resolution is printed)"""
    dde = st_attn_bwd(r, t).aux["de"]
    sens = torch.where(r.act[..., None], t["de"].double().abs() / dde, torch.zeros_like(dde))
    idx = np.unravel_index(int(sens.reshape(-1).argmax()), tuple(sens.shape))
    print("\n  de check: smallest relative defect it resolves %.2g" % (1.0 / float(sens.max())), end="")
    t["de"] = _mul(t["de"], idx, 1 + 1e-3)
    return "attn_bwd"


def m_dwf_without_step(r, t):
    """dwf_part of one running row without one location's contribution de_l u_l"""
    w = t["dwf_part"].clone()
    b = int(torch.nonzero(r.act[1])[0])
    x = t["P"][r.img[b]].double() + t["Q"][1, b].double()
    l = int(t["de"][1, b].abs().argmax())
    w[1, b] -= (t["de"][1, b, l].double() * torch.tanh(x[l])).float()
    t["dwf_part"] = w
    return "attn_bwd"


def m_grad_without_step(r, t):
    """output.hidden.weight without the contribution of one time step: dpre[s]^T h_{s+1}"""
    s = 1
    d = t["dpre"][s].double()[:, :r.E0]
    h = t["Hs"][r.nl - 1, s + 1].double()[:, :r.H0]
    G = t["_G"]
    G["output.hidden.weight"] = (G["output.hidden.weight"].double() - d.t() @ h).float()
    return "param_grads"


def m_grad_gscale(r, t):
    """output.output.weight scaled by 1 instead of the upstream gradient 0.75"""
    G = t["_G"]
    G["output.output.weight"] = G["output.output.weight"] / GSCALE
    return "param_grads"


def m_gates_swap(r, t):
    g = t["Gates"].clone()
    b = int(torch.nonzero(r.act[1])[0])
    gi = g[0, 1, b, 0::4]
    gf = g[0, 1, b, 1::4]
    j = int((gi.float() - gf.float()).abs().argmax())
    g[0, 1, b, 4 * j], g[0, 1, b, 4 * j + 1] = g[0, 1, b, 4 * j + 1].clone(), g[0, 1, b, 4 * j].clone()
    t["Gates"] = g
    return "lstm"


def m_Xo_stale_h(r, t):
    y, _ = _xo_ref(r, t, h_shift=0)
    xo = t["Xo"].clone()
    b = int(torch.nonzero(r.act[2])[0])
    xo[2, b] = y[2, b].to(torch.bfloat16)
    t["Xo"] = xo
    return "Xo"


def m_tile_sum(r, t):
    st = t["ce_stats"].clone()
    m = int(torch.nonzero(r.act.reshape(-1))[0])
    tile = int(st[m, :, 0].argmax())
    st[m, tile, 1] *= 1 + 1e-4
    t["ce_stats"] = st
    return "vocab"


def m_row_xt(r, t):
    x = t["row_xt"].clone()
    m = int(torch.nonzero(r.act.reshape(-1))[0])
    x[m] = x[m] + 1e-3 * max(1.0, abs(float(x[m])))
    t["row_xt"] = x
    return "vocab"


def m_dlogits(r, t):
    d = t["dlogits"]
    idx = _argmax_flat(d, _act_mask(r, [r.V]) & (torch.arange(r.V, device="cuda") < r.V0))
    t["dlogits"] = _bf16_ulps(d, idx, 2)
    return "dlogits"


def m_dpre(r, t):
    t["dpre"] = _bf16_ulps(t["dpre"], _argmax_flat(t["dpre"]), 2)
    return "dpre"


def m_dHZ(r, t):
    t["dHZ"] = _mul(t["dHZ"], _argmax_flat(t["dHZ"]), 1 + 1e-4)
    return "dpre"


def m_dG(r, t):
    dy = t["DY"].clone()
    s = r.T - 2
    idx = _argmax_flat(dy[s][..., r.A + r.D:], r.act[s][:, None].expand(r.B, 4 * r.H))
    dy[s, idx[0], r.A + r.D + idx[1]] = _bf16_ulps(dy[s, idx[0], r.A + r.D + idx[1]].reshape(1), (0,), 2)[0]
    t["DY"] = dy
    return "lstm_bwd"


def m_dP_no_step0(r, t):
    P = t["P"].double()[r.img]
    u = torch.tanh(P + t["Q"][0].double()[:, None, :])
    contrib = t["de"][0].double()[..., None] * r.pw.t["wf"].double() * (1 - u * u)
    t["dP"] = (t["dP"].double() - contrib).float()
    return "dP"


def m_dP16(r, t):
    t["dP16"] = _bf16_ulps(t["dP16"], _argmax_flat(t["dP16"]), 1)
    return "dP"


def m_dXe(r, t):
    t["dXe"] = _mul(t["dXe"], _argmax_flat(t["dXe"]), 1 + 1e-4)
    return "dXe"


def m_dmean(r, t):
    t["dmean"] = _mul(t["dmean"], _argmax_flat(t["dmean"]), 1 + 1e-4)
    return "init_bwd"


def m_d_ann(r, t):
    t["d_ann"] = _bf16_ulps(t["d_ann"], _argmax_flat(t["d_ann"]), 4)
    return "d_ann"


def m_out_acc(r, t):
    o = t["out"].clone()
    o[3] += o[4]
    t["out"] = o
    return "loss"


MUTATIONS = dict(P=m_P, meanv=m_meanv, init_out=m_init_out, h0=m_h0, Xe=m_Xe, Gx=m_Gx, Q=m_Q, alpha_swap=m_alpha, Cs=m_Cs,
                 gates_swap_i_f=m_gates_swap, Xo_stale_h=m_Xo_stale_h, tile_sum_exp=m_tile_sum, row_xt=m_row_xt, dlogits=m_dlogits,
                 dpre=m_dpre, dHZ=m_dHZ, dG=m_dG, dP_without_step0=m_dP_no_step0, dP16=m_dP16, dXe=m_dXe, dmean=m_dmean,
                 d_ann=m_d_ann, accuracy=m_out_acc, de=m_de, dwf_without_step=m_dwf_without_step,
                 grad_without_step=m_grad_without_step, grad_gscale=m_grad_gscale)


@pytest.mark.parametrize("mutation", list(MUTATIONS))
def test_stage_check_sees_mutation(mutation):
    r = run("c2s")
    t = dict(r.t, _G=dict(r.G))
    stage = MUTATIONS[mutation](r, t)
    rep = STAGES[stage](r, t)
    print("\n  mutation %-16s -> %s worst error / bound %.3g" % (mutation, stage, rep.worst()), end="")
    assert rep.worst() > 1.0


def _invariant_violations(r, t):
    bad = []
    inact = ~r.act
    if bool((t["DY"][inact] != 0).any()):
        bad.append("DY")
    for label, x in _pad_views(r, t):
        if x.numel() and bool((x != 0).any()):
            bad.append(label)
    return bad


def test_invariant_checks_see_mutations():
    r = run("odd3")
    assert _invariant_violations(r, dict(r.t)) == []
    t = dict(r.t)
    dy = t["DY"].clone()
    s, b = [int(v) for v in torch.nonzero(~r.act)[0]]
    dy[s, b, r.A + r.D + 5] = 1e-30
    t["DY"] = dy
    assert _invariant_violations(r, t) == ["DY"]
    t = dict(r.t)
    dl = t["dlogits"].clone()
    dl[0, 0, r.V0] = 1e-30
    t["dlogits"] = dl
    assert _invariant_violations(r, t) == ["dlogits"]
