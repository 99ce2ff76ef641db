"""Host side of the fused SAT decoder: buffer management and the calls into libsat_b200.so.

Reference spans replaced: SAT.train_batch (model.py:474-557) + the loss of training_step
(model.py:588-597, util.py:105-112) and, through autograd, their backward -- including the
parameter gradients (sat_train_param_grads), so no cuBLAS / ATen kernel runs on this path.
"""
import ctypes as C

import torch

from . import _lib, _redzone
from .packing import _LAYER_FIELDS, _LAYER_PARAMS, PARAM_NAMES, PackedWeights

# reference parameter name -> field of SatParamGrads (include/sat_b200.h)
_GRAD_FIELD = {
    "embedding.weight": "embedding", "init_lstm.factorize.weight": "fact_w", "init_lstm.factorize.bias": "fact_b",
    "init_lstm.init.weight": "init_w", "init_lstm.init.bias": "init_b", "lstm.weight_ih_l0": "w_ih", "lstm.weight_hh_l0": "w_hh",
    "lstm.bias_ih_l0": "b_ih", "lstm.bias_hh_l0": "b_hh", "attention.encoder_att.weight": "enc_att",
    "attention.decoder_att.weight": "dec_att", "attention.f_att.weight": "f_att", "beta.0.weight": "beta_w", "beta.0.bias": "beta_b",
    "output.hidden.weight": "out_hidden", "output.context.weight": "out_context", "output.output.weight": "out_w",
    "output.output.bias": "out_b",
}


_ONES = {}


def _one(device):
    """a persistent device scalar 1.0 (default upstream gradient of the loss)"""
    key = str(device)
    if key not in _ONES:
        _ONES[key] = torch.ones(1, dtype=torch.float32, device=device)
    return _ONES[key]


def make_dims(B, Bi, L, pw_or_dims, T, dtype, exact, use_tc, plain_output=False, dims0=None, layers=1):
    """SatDims for a PackedWeights object (storage dims + the module's true dims) or an explicit dict of storage dims."""
    d = _lib.SatDims()
    if isinstance(pw_or_dims, PackedWeights):
        dm, dm0, plain_output, layers = pw_or_dims.dims, pw_or_dims.dims0, pw_or_dims.plain_output, pw_or_dims.layers
    else:
        dm, dm0 = pw_or_dims, dims0 or pw_or_dims
    d.plain_output = 1 if plain_output else 0
    d.B, d.Bi, d.ncap = B, Bi, B // Bi
    d.L, d.D, d.A, d.E, d.H, d.V, d.T = L, dm["D"], dm["A"], dm["E"], dm["H"], dm["V"], T
    d.D0, d.A0, d.E0, d.H0, d.V0 = dm0["D"], dm0["A"], dm0["E"], dm0["H"], dm0["V"]
    d.dtype = _lib.dtype_code(dtype)
    d.exact = 1 if exact else 0
    d.use_tc = 1 if use_tc else 0
    d.layers = int(layers)
    return d


class TrainBuffers:
    """All device buffers of one training step (include/sat_b200.h: SatTrainBuffers)."""

    def __init__(self, d, dtype, device, logits_f32=False, backward=True, keep_logits=False, fuse_ce=False):
        B, Bi, L, D, A, E, H, V, T = d.B, d.Bi, d.L, d.D, d.A, d.E, d.H, d.V, d.T
        NH3 = A + D + 4 * H
        nl = max(1, d.layers)
        s, f = dtype, torch.float32
        t = self.t = {}
        mk = lambda shape, dt: _redzone.empty(shape, dt, device, "train buffer #%d" % len(t))   # torch.empty unless SAT_REDZONE=1
        t["tok"] = mk((T, B), torch.int32)
        t["P"] = mk((Bi, L, A), s)
        t["meanv"] = mk((Bi, D), s)
        t["f1"] = mk((Bi, E), s)
        t["init_out"] = mk((Bi, 2 * nl * H), f)
        t["Xe"] = mk((T, B, E), s)
        t["Gx"] = mk((T, B, 4 * H), f)
        t["Hs"] = mk((nl, T + 1, B, H), s)
        t["Cs"] = mk((nl, T + 1, B, H), f)
        t["hp"] = mk((B, NH3), f)
        t["Q"] = mk((T, B, A), f)
        t["alphas"] = mk((B, T, L), f)
        t["Z"] = mk((T, B, D), s)
        t["GZ"] = mk((T, B, D), s)
        t["Beta"] = mk((T, B, D), s)
        t["Gates"] = mk((nl, T, B, 4 * H), s)
        t["Xo"] = mk((T, B, E), s)
        # fused vocabulary projection + cross entropy (tensor-core mode): no logits buffer at all, only the per-tile statistics
        self.fuse_ce = bool(fuse_ce and d.use_tc and dtype == torch.bfloat16 and not logits_f32 and not keep_logits)
        if self.fuse_ce:
            t["ce_stats"] = mk((T * B, (V + 127) // 128, 4), f)
            t["row_lse"] = mk((T * B,), f)
            t["row_xt"] = mk((T * B,), f)
            if backward:
                t["dlogits"] = mk((T, B, V), s)
        else:
            t["logits"] = mk((T, B, V), f if logits_f32 else s)
            if backward:
                t["dlogits"] = mk((T, B, V), s) if (keep_logits or logits_f32) else t["logits"]
        t["row_loss"] = mk((T, B), f)
        t["row_argmax"] = mk((T, B), torch.int32)
        t["S"] = mk((B, L), f)
        t["out"] = mk((8,), f)                     # zeroed by sat_train_forward
        if backward:
            t["gscale"] = _one(device)
            t["dpre"] = mk((T, B, E), s)
            t["dHZ"] = mk((T, B, H + D), f)
            t["DY"] = mk((T, B, NH3), s)
            t["dgz"] = mk((16, B, D), f)        # split-K partials (SAT_MAX_SPLITK)
            t["dh"] = mk((16, B, H), f)
            t["dc"] = mk((nl, B, H), f)
            if nl > 1:
                t["dGl"] = mk((nl - 1, T, B, 4 * H), s)
                t["dxl"] = mk((nl - 1, 16, B, 2 * H), f)
                t["dhq"] = mk((16, B, H), f)
            t["dZ"] = mk((T, B, D), s)
            t["dP"] = mk((B, L, A), f)
            if dtype != torch.float32:
                t["dP16"] = mk((B, L, A), s)
            t["dwf_part"] = mk((T, B, A), f)
            t["de"] = mk((T, B, L), f)
            t["dXe"] = mk((T, B, E), f)
            t["d_init_out"] = mk((Bi, 2 * nl * H), f)
            t["df1"] = mk((Bi, E), f)
            if dtype != torch.float32:
                t["d_init_out16"] = mk((Bi, 2 * nl * H), s)
                t["df116"] = mk((Bi, E), s)
            t["dmean"] = mk((Bi, D), f)
            t["d_ann"] = mk((B, L, D), s)          # per caption row; the host sums the ncap rows of an image
        self.c = _lib.SatTrainBuffers()
        for name, typ in _lib.SatTrainBuffers._fields_:
            if typ is C.c_void_p and name in t:
                setattr(self.c, name, _lib.ptr(t[name]))
        self.c.logits_f32 = 1 if logits_f32 else 0
        self.dims = d
        self.ws = None

    def bind_inputs(self, ann, caps, lens, label_smoothing, att_gamma, sampled=None, dropout=(0.0, 0.0, 0)):
        self.t["ann"], self.t["caps"], self.t["lens"] = ann, caps, lens   # keep alive
        self.c.ann, self.c.caps, self.c.lens = _lib.ptr(ann), _lib.ptr(caps), _lib.ptr(lens)
        if sampled is not None and any(sampled):
            self._sampled = (C.c_int32 * len(sampled))(*[1 if x else 0 for x in sampled])     # host array, kept alive
            self.c.sampled = C.cast(self._sampled, C.c_void_p)
        else:
            self._sampled = None
            self.c.sampled = None
        self.c.label_smoothing = float(label_smoothing)
        self.c.att_gamma = float(att_gamma)
        self.c.dropout_p, self.c.emb_dropout_p, self.c.dropout_seed = float(dropout[0]), float(dropout[1]), int(dropout[2])


def annotations_as_bld(ann, dtype, D_storage=None):
    """[Bi,D,h,w] (any memory format) -> contiguous [Bi,L,D] of `dtype`.  Zero-copy when the encoder
    produced channels_last output in `dtype` (SURVEY.md §0.1-1).  D_storage > D zero-pads the channel dimension
    (modules whose encoder_dim is not a multiple of 8)."""
    Bi, D, h, w = ann.shape
    x = ann.permute(0, 2, 3, 1).reshape(Bi, h * w, D)
    if x.dtype != dtype:
        x = x.to(dtype)
    if D_storage is not None and D_storage != D:
        x = torch.nn.functional.pad(x, (0, D_storage - D))
    return x.contiguous()


def vocab_path_fused(d, sampled=None, fuse_ce=True):
    """Whether sat_train_forward runs the vocabulary stage fused (per-tile statistics in the GEMM epilogue, no [T,B,V] logits):
    sat_train_vocab_path decides.  Teacher-forced: fused when the caller asks for it (fuse_ce) and the library can run it.
    Scheduled sampling: the library's choice (the logits path while the cross-entropy row kernel holds a row, the fused path
    above that); a caller that wants the logits back passes fuse_ce=False and is held to the row kernel's limit.  Raises
    SatError when neither path can run these dims."""
    is_sampled = sampled is not None and any(sampled)
    path = _lib.lib().sat_train_vocab_path(C.byref(d), 1 if is_sampled else 0)
    if path < 0:
        _lib.check(path, "sat_train_vocab_path")
    return bool(fuse_ce) and path == _lib.TRAIN_PATH_FUSED


def train_forward(pw, ann_bld, caps, lens, label_smoothing=0.0, att_gamma=1.0, exact=True, use_tc=False,
                  logits_f32=False, backward=True, keep_logits=False, buffers=None, sampled=None, dropout=(0.0, 0.0, 0),
                  fuse_ce=False):
    """ann_bld [Bi,L,D] (pw.dtype, cuda); caps [Bi,ncap,T+1] or [B,T+1] int; lens [Bi,ncap] or [B].
    Runs sat_train_forward; returns the TrainBuffers (loss etc. in .t['out']).  fuse_ce=True (tensor-core mode) keeps the
    vocabulary logits on chip: .t has no 'logits' then.  With scheduled-sampling steps (sampled) the library picks the path
    (vocab_path_fused); keep_logits / logits_f32 always keep the logits."""
    L_ = _lib.lib()
    dev = ann_bld.device
    Bi, L, D = ann_bld.shape
    caps2 = caps.reshape(-1, caps.shape[-1])
    lens2 = lens.reshape(-1)
    if caps2.dtype == torch.int64 and lens2.dtype == torch.int64 and caps2.device == dev and lens2.device == dev:
        # int64 ids from the dataset: narrowed by the library (one launch) instead of two framework casts
        c64, l64 = caps2.contiguous(), lens2.contiguous()
        caps2 = torch.empty(c64.shape, dtype=torch.int32, device=dev)
        lens2 = torch.empty(l64.shape, dtype=torch.int32, device=dev)
        _lib.check(L_.sat_cast_captions(c64.data_ptr(), l64.data_ptr(), caps2.data_ptr(), lens2.data_ptr(), c64.numel(), l64.numel(),
                                        _lib.stream_ptr()), "sat_cast_captions")
    else:
        caps2 = caps2.to(device=dev, dtype=torch.int32).contiguous()
        lens2 = lens2.to(device=dev, dtype=torch.int32).contiguous()
    B, caplen = caps2.shape
    dm, dm0 = pw.dims, pw.dims0
    if D == dm0["D"] and D != dm["D"]:
        ann_bld = torch.nn.functional.pad(ann_bld, (0, dm["D"] - D)).contiguous()
        D = dm["D"]
    assert D == dm["D"], "annotation width %d != encoder_dim %d" % (D, dm0["D"])
    assert ann_bld.dtype == pw.dtype and ann_bld.is_contiguous()
    d = make_dims(B, Bi, L, pw, caplen - 1, pw.dtype, exact, use_tc)
    fuse_ce = vocab_path_fused(d, sampled, fuse_ce and not (keep_logits or logits_f32))
    if buffers is None:
        buffers = TrainBuffers(d, pw.dtype, dev, logits_f32=logits_f32, backward=backward, keep_logits=keep_logits, fuse_ce=fuse_ce)
    buffers.bind_inputs(ann_bld, caps2, lens2, label_smoothing, att_gamma, sampled, dropout)
    buffers.dims = d
    _lib.check(L_.sat_train_forward(C.byref(d), pw.ref(), C.byref(buffers.c), _lib.stream_ptr()), "sat_train_forward")
    return buffers


def train_backward(pw, buf, grad_loss=None, pad_idx=0, weight_tying=False, dalpha_ext=None):
    """Runs sat_train_backward on the buffers of a finished train_forward, then sat_train_param_grads, which reduces the saved
    per-(t,b) buffers into the parameter gradients (reference names / shapes, fp32) inside the library.
    Returns (grads dict, d_ann [Bi,L,D0])."""
    L_ = _lib.lib()
    t, d = buf.t, buf.dims
    Bi, ncap, L, D = d.Bi, d.ncap, d.L, d.D
    dm0 = pw.dims0
    dev = t["dlogits"].device
    if grad_loss is None:
        buf.c.gscale = _lib.ptr(t["gscale"])          # the ones written at allocation
    else:
        gl = grad_loss.detach().reshape(1)
        if gl.dtype != torch.float32 or gl.device != dev:
            gl = gl.to(device=dev, dtype=torch.float32)
        t["gscale_in"] = gl                            # upstream gradient read in place (kept alive with the buffers)
        buf.c.gscale = _lib.ptr(gl)
    if dalpha_ext is not None:
        t["dalpha_ext"] = dalpha_ext.to(torch.float32).contiguous()
        buf.c.dalpha_ext = _lib.ptr(t["dalpha_ext"])
    else:
        buf.c.dalpha_ext = None
    _lib.check(L_.sat_train_backward(C.byref(d), pw.ref(), C.byref(buf.c), _lib.stream_ptr()), "sat_train_backward")
    # parameter gradients: destinations with the reference's shapes
    V0, E0, H0, D0, A0 = dm0["V"], dm0["E"], dm0["H"], dm0["D"], dm0["A"]
    nl = pw.layers
    shapes = {
        "embedding.weight": (V0, E0), "init_lstm.factorize.weight": (E0, D0), "init_lstm.factorize.bias": (E0,),
        "init_lstm.init.weight": (2 * nl * H0, E0), "init_lstm.init.bias": (2 * nl * H0,), "lstm.weight_ih_l0": (4 * H0, E0 + D0),
        "lstm.weight_hh_l0": (4 * H0, H0), "lstm.bias_ih_l0": (4 * H0,), "lstm.bias_hh_l0": (4 * H0,),
        "attention.encoder_att.weight": (A0, D0), "attention.decoder_att.weight": (A0, H0), "attention.f_att.weight": (1, A0),
        "beta.0.weight": (D0, H0), "beta.0.bias": (D0,), "output.hidden.weight": (E0, H0), "output.context.weight": (E0, D0),
        "output.output.weight": (V0, E0), "output.output.bias": (V0,),
    }
    skip = set()
    if pw.plain_output:
        skip.add("output.context.weight")
    if not pw.has_out_bias:
        skip.add("output.output.bias")
    if weight_tying:
        skip.add("output.output.weight")
    G = {}
    g = _lib.SatParamGrads()
    for name in PARAM_NAMES:
        if name in skip:
            continue
        G[name] = torch.empty(shapes[name], dtype=torch.float32, device=dev)
        setattr(g, _GRAD_FIELD[name], G[name].data_ptr())
    for l in range(1, nl):
        for field, name, shp in zip(_LAYER_FIELDS, _LAYER_PARAMS, ((4 * H0, H0), (4 * H0, H0), (4 * H0,), (4 * H0,))):
            G[name % l] = torch.empty(shp, dtype=torch.float32, device=dev)
            getattr(g, field)[l - 1] = G[name % l].data_ptr()
    g.pad_idx = -1 if pad_idx is None else int(pad_idx)
    g.weight_tying = 1 if weight_tying else 0
    nbytes = int(L_.sat_param_grads_workspace_bytes(C.byref(d)))
    if buf.ws is None or buf.ws.numel() < nbytes:
        buf.ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    _lib.check(L_.sat_train_param_grads(C.byref(d), C.byref(buf.c), C.byref(g), buf.ws.data_ptr(), nbytes, _lib.stream_ptr()),
               "sat_train_param_grads")
    d_ann = t["d_ann"]
    if ncap > 1:
        d_ann = d_ann.reshape(Bi, ncap, L, D).sum(1, dtype=torch.float32)
    else:
        d_ann = d_ann.reshape(Bi, L, D)
    if D != D0:
        d_ann = d_ann[..., :D0]
    return G, d_ann
