"""Host side of batched greedy / beam decoding (SAT.forward / SAT.caption, model.py:214-472).

All images of the batch are decoded together by sat_decode (device-side beam bookkeeping, no host
sync per step); this module allocates the buffers and turns the finished-hypothesis arrays into the
reference's return format: four Python lists (captions, scores, alphas [len,h,w] CPU tensors,
perplexities), or lists of lists sorted by score when return_all=True (model.py:453-467).
"""
import ctypes as C

import numpy as np
import torch

from . import _lib, _redzone, decoder
from .packing import PackedWeights

RESCORE = {None: 0, "LN": 1, "WR": 2, "BAR": 3}
SAMPLE = {"beam": 0, "multinomial": 1, "topk": 2}


class DecodeWeights:
    """Packed inference weights + the per-vocabulary gate table GxV, cached per parameter version."""

    def __init__(self, W, dtype, device, exact, use_tc):
        self.pw = PackedWeights(W, dtype=dtype, device=device, backward=False)
        dm = self.pw.dims
        self.exact, self.use_tc = exact, use_tc
        d = decoder.make_dims(1, 1, 1, self.pw, 1, dtype, exact, use_tc)
        self.GxV = torch.empty(dm["V"], 4 * dm["H"], dtype=torch.float32, device=device)
        _lib.check(_lib.lib().sat_decode_prepare_weights(C.byref(d), self.pw.ref(), _lib.ptr(self.GxV), _lib.stream_ptr()),
                   "sat_decode_prepare_weights")
        # early-out flag (include/sat_b200.h: done_host): pinned host int the device writes when every image has used up its
        # beams; calls are told apart by a running tag
        self.done = torch.zeros(1, dtype=torch.int32).pin_memory()
        self.calls = 0


def decode_annotations(dw, ann_bld, k, max_gen_length, temperature=1.0, rescore_method=None, rescore_reward=0.5,
                       vocab=None, sample_method="beam", sample_topk=3, decoder_noise=None, seed=None, early_out=True):
    """ann_bld [n_img,L,D] (dw.pw.dtype, cuda).  Returns dict of device tensors (fin_* + alpha_all) after
    enqueueing the whole decode; nothing is synchronised here.  sample_method "multinomial" / "topk" and decoder_noise
    (model.py:322-324,360-379) draw their randomness from `seed` (default: one draw from torch's CPU generator)."""
    L_ = _lib.lib()
    dev = ann_bld.device
    n_img, L, D = ann_bld.shape
    dm = dw.pw.dims
    A, E, H, V = dm["A"], dm["E"], dm["H"], dm["V"]
    if D != dm["D"]:                      # encoder_dim that is not a multiple of 8: zero-padded channels
        assert D == dw.pw.dims0["D"], "annotation width %d != encoder_dim %d" % (D, dw.pw.dims0["D"])
        ann_bld = torch.nn.functional.pad(ann_bld, (0, dm["D"] - D)).contiguous()
        D = dm["D"]
    S = int(max_gen_length)
    R = n_img * k
    dtype = dw.pw.dtype
    d = decoder.make_dims(R, n_img, L, dw.pw, S + 1, dtype, dw.exact, dw.use_tc)
    nl = dw.pw.layers
    method = SAMPLE[sample_method]
    noise = float(decoder_noise) if decoder_noise else 0.0
    kcap = max(k, int(sample_topk)) if method == 2 else k
    if (method != 0 or noise != 0.0) and seed is None:
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    # which vocabulary stage runs (row kernels on [R,V] logits, or per-tile statistics / candidates from the GEMM epilogue)
    path = L_.sat_decode_vocab_path(C.byref(d), k, method, int(sample_topk))
    if path < 0:
        _lib.check(path, "sat_decode")
    f, s, i32 = torch.float32, dtype, torch.int32
    _n = [0]

    def mk(shape, dt):                  # torch.empty unless SAT_REDZONE=1 (guard bands, tests)
        _n[0] += 1
        return _redzone.empty(shape, dt, dev, "decode buffer #%d" % _n[0])

    t = dict(P=mk((n_img, L, A), s), meanv=mk((n_img, D), s), f1=mk((n_img, E), s), init_out=mk((n_img, 2 * nl * H), f),
             h=mk((nl, R, H), s), c=mk((nl, R, H), f), hn=mk((nl, R, H), s), cn=mk((nl, R, H), f), hp=mk((R, A + D + 4 * H), f),
             z=mk((R, D), s), gz=mk((R, D), s), xo=mk((R, E), s), alpha_all=mk((S + 1, R, L), f),
             cand_val=mk((R, kcap), f), cand_idx=mk((R, kcap), i32), tok_hist=torch.zeros((2, R, S + 1), dtype=i32, device=dev),
             asrc_hist=torch.zeros((2, R, S + 1), dtype=i32, device=dev), top_scores=mk((R,), f), cur_tok=mk((R,), i32),
             src_row=torch.zeros((R,), dtype=i32, device=dev), alive=mk((R,), i32), kcur=mk((n_img,), i32),
             fin_tokens=torch.zeros((n_img, k, S + 1), dtype=i32, device=dev),
             fin_asrc=torch.zeros((n_img, k, S + 1), dtype=i32, device=dev), fin_len=mk((n_img, k), i32),
             fin_score=torch.full((n_img, k), float("-inf"), dtype=f, device=dev), fin_ppl=mk((n_img, k), f),
             fin_count=mk((n_img,), i32))
    if method == 1:
        t["cand_key"] = mk((R, kcap), f)
    if noise != 0.0:
        t["h_noisy"] = mk((nl, R, H), s)
    NT = (V + 127) // 128
    if path == _lib.VOCAB_PATH_ROWS:
        t["logits"] = mk((R, V), f)
    else:
        t["topk_stats"] = mk((R, NT, 4), f)
    if path == _lib.VOCAB_PATH_CAND:
        t["tile_val"], t["tile_idx"] = mk((R, NT, kcap), f), mk((R, NT, kcap), i32)
        if method == 1:
            t["tile_key"], t["topk_stats2"] = mk((R, NT, kcap), f), mk((R, NT, 2), f)
    temps = temperature if isinstance(temperature, (list, tuple)) else [temperature]
    temps_arr = (C.c_float * (S + 1))(*[float(temps[i % len(temps)]) for i in range(S + 1)])
    b = _lib.SatDecodeBuffers()
    b.ann = _lib.ptr(ann_bld)
    b.GxV = _lib.ptr(dw.GxV)
    for name, tensor in t.items():
        setattr(b, name, _lib.ptr(tensor))
    b.temps = C.cast(temps_arr, C.c_void_p)
    b.k, b.max_gen_length, b.rescore, b.reward = k, S, RESCORE[rescore_method], float(rescore_reward)
    b.tokPAD, b.tokSTART, b.tokEND, b.tokUNK = vocab["PAD"], vocab["START"], vocab["END"], vocab["UNK"]
    b.sample_method, b.sample_topk, b.kcap, b.decoder_noise, b.sample_seed = method, int(sample_topk), kcap, noise, int(seed or 0)
    if early_out:
        dw.calls = dw.calls % 0x7ffffff0 + 1
        t["live_images"] = mk((1,), i32)
        b.live_images, b.done_host, b.call_id = _lib.ptr(t["live_images"]), dw.done.data_ptr(), dw.calls
    _lib.check(L_.sat_decode(C.byref(d), dw.pw.ref(), C.byref(b), _lib.stream_ptr()), "sat_decode")
    t["ann"] = ann_bld
    t["_dims"] = (n_img, k, S, L)
    return t


def assemble(t, hw, return_all=False, want_alphas=True):
    """fin_* device arrays -> the reference's four lists.  Host side is vectorised (numpy) up to the final Python lists: with many
    GPUs per host the list assembly, not the device, bounds end-to-end captioning."""
    n_img, k, S, L = t["_dims"]
    cnt = t["fin_count"].cpu().numpy()
    ln = t["fin_len"].cpu().numpy()
    sc = t["fin_score"].cpu().numpy().astype(np.float64)
    ppl = t["fin_ppl"].cpu().numpy().astype(np.float64)
    toks = t["fin_tokens"].cpu().numpy()
    # which hypotheses are returned, in which order
    if return_all:                              # sort [score, index] pairs descending (model.py:455-457)
        sel = [sorted(range(int(cnt[n])), key=lambda i: (sc[n, i], i), reverse=True) for n in range(n_img)]
    else:                                       # first index of the maximum (model.py:463)
        masked = np.where(np.arange(sc.shape[1])[None, :] < cnt[:, None], sc, -np.inf)
        sel = [[int(i)] for i in masked.argmax(1)]
    img_of = np.fromiter((n for n in range(n_img) for _ in sel[n]), dtype=np.int64)
    slot_of = np.fromiter((i for n in range(n_img) for i in sel[n]), dtype=np.int64)
    lens_sel = ln[img_of, slot_of].astype(np.int64) if len(img_of) else np.zeros(0, np.int64)
    alphas_flat = None
    if want_alphas:
        # gather alpha rows of the selected hypotheses on the device, one D2H copy
        if lens_sel.sum() > 0:
            asrc = t["fin_asrc"].cpu().numpy()
            width = asrc.shape[2]
            mask = np.arange(width)[None, :] < lens_sel[:, None]                  # [n_sel, S+1]
            rows = asrc[img_of, slot_of][mask]
            steps = np.broadcast_to(np.arange(width)[None, :], mask.shape)[mask]
            dev = t["alpha_all"].device
            st = torch.from_numpy(np.ascontiguousarray(steps)).to(dev, non_blocking=False)
            rw = torch.from_numpy(np.ascontiguousarray(rows).astype(np.int64)).to(dev, non_blocking=False)
            flat = t["alpha_all"][st, rw].cpu()
        else:
            flat = torch.zeros(0, L)
        alphas_flat = [x.reshape(x.shape[0], *hw) for x in torch.split(flat, lens_sel.tolist())] if len(lens_sel) else []
    caps, scores, ppls, alphas_out, j = [], [], [], ([] if want_alphas else None), 0
    for n in range(n_img):
        m = len(sel[n])
        caps.append([toks[n, i, :int(ln[n, i])].tolist() for i in sel[n]])
        scores.append([float(sc[n, i]) for i in sel[n]])
        ppls.append([float(ppl[n, i]) for i in sel[n]])
        if want_alphas:
            alphas_out.append(alphas_flat[j:j + m])
        j += m
    if not return_all:
        caps = [c[0] for c in caps]
        scores = [s[0] for s in scores]
        ppls = [p[0] for p in ppls]
        if alphas_out is not None:
            alphas_out = [a[0] for a in alphas_out]
    return caps, scores, alphas_out, ppls


def inference_weights(model):
    """cached DecodeWeights for a SAT module, rebuilt when any decoder parameter changed."""
    from .packing import param_names
    params = model.decoder_weights()
    PARAM_NAMES = param_names(model.hparams.decoder_layers)
    cfg = model._cfg()
    key = tuple((p.data_ptr(), p._version) if p is not None else None for p in params) + (cfg["dtype"],)
    cache = getattr(model, "_packed_infer", None)
    if cache is None or cache[0] != key:
        W = {n: p for n, p in zip(PARAM_NAMES, params) if p is not None}
        mn = model.hparams.get("embed_norm", None) if hasattr(model.hparams, "get") else None
        if mn is not None:
            # max_norm renormalisation (model.py:161): every row a decode can look up, applied to the packed copy only
            e = W["embedding.weight"].detach().clone()
            torch.embedding_renorm_(e, torch.arange(e.shape[0], device=e.device), float(mn), 2.0)
            W["embedding.weight"] = e
            if model.hparams.weight_tying and model.hparams.deep_output:
                W["output.output.weight"] = e
        dev = next(p for p in params if p is not None).device
        model._packed_infer = (key, DecodeWeights(W, cfg["dtype"], dev, cfg["exact"], cfg["use_tc"]))
    return model._packed_infer[1]


def caption_from_annotations(model, ann, beamk, max_gen_length, temperature, rescore_method, rescore_reward, return_all,
                             sample_method="beam", sample_topk=3, decoder_noise=None):
    dw = inference_weights(model)
    hw = tuple(ann.shape[2:])
    bld = decoder.annotations_as_bld(ann, dw.pw.dtype)
    vocab = dict(PAD=model.stoi("<PAD>"), START=model.stoi("<START>"), END=model.stoi("<END>"), UNK=model.stoi("<UNK>"))
    t = decode_annotations(dw, bld, int(beamk), max_gen_length, temperature, rescore_method, rescore_reward, vocab,
                           sample_method=sample_method, sample_topk=sample_topk, decoder_noise=decoder_noise)
    return assemble(t, hw, return_all=return_all)
