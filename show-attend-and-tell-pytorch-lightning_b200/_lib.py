"""ctypes binding of libsat_b200.so (include/sat_b200.h).  No CPU fallback: every op raises if the
library is missing or a call fails."""
import ctypes as C
import os
import subprocess

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsat_b200.so")
SAT_F32, SAT_BF16 = 0, 1

vp, fp, ip = C.c_void_p, C.c_void_p, C.c_void_p   # all device pointers travel as void*
SAT_MAX_LAYERS = 4
_vpl = vp * (SAT_MAX_LAYERS - 1)                   # per-layer pointers of the stacked LSTM layers l = 1 ..


class SatDims(C.Structure):
    _fields_ = [(n, C.c_int32) for n in
                ("B", "Bi", "ncap", "L", "D", "A", "E", "H", "V", "T", "dtype", "exact", "use_tc", "plain_output",
                 "D0", "A0", "E0", "H0", "V0", "layers")]


class SatWeights(C.Structure):
    _fields_ = [(n, vp) for n in
                ("Wa", "Whcat", "bhcat", "Wihz", "Wihe", "bg", "Whozo", "Wo", "bo", "wf", "Emb", "Wfact", "bfact",
                 "Winit", "binit", "WoT", "WhozoT", "WihzT", "WiheT", "WhcatT", "WaT", "WinitT", "WfactT")] + \
               [("Wl", _vpl), ("bgl", _vpl), ("WlT", _vpl)]


class SatMasterWeights(C.Structure):
    _fields_ = [(n, vp) for n in
                ("embedding", "fact_w", "fact_b", "init_w", "init_b", "w_ih", "w_hh", "b_ih", "b_hh", "enc_att", "dec_att",
                 "f_att", "beta_w", "beta_b", "out_hidden", "out_context", "out_w", "out_b")] + \
               [("w_ih_l", _vpl), ("w_hh_l", _vpl), ("b_ih_l", _vpl), ("b_hh_l", _vpl)]


class SatTrainBuffers(C.Structure):
    _fields_ = [(n, vp) for n in
                ("ann", "caps", "lens", "sampled", "tok", "P", "meanv", "f1", "init_out", "Xe", "Gx", "Hs", "Cs", "hp", "Q", "alphas",
                 "Z", "GZ", "Beta", "Gates", "Xo", "logits", "dlogits", "row_loss", "row_argmax", "S", "out",
                 "ce_stats", "row_lse", "row_xt",
                 "gscale", "dalpha_ext", "dpre", "dHZ", "DY", "dgz", "dh", "dc", "dGl", "dxl", "dhq", "dZ", "dP", "dP16", "dwf_part", "de", "dXe", "d_init_out",
                 "df1", "d_init_out16", "df116", "dmean", "d_ann")] + \
               [("label_smoothing", C.c_float), ("att_gamma", C.c_float), ("dropout_p", C.c_float),
                ("emb_dropout_p", C.c_float), ("dropout_seed", C.c_uint64), ("logits_f32", C.c_int32),
                ("reserved", C.c_int32)]


class SatDecodeBuffers(C.Structure):
    _fields_ = [(n, vp) for n in
                ("ann", "P", "meanv", "f1", "init_out", "GxV", "h", "c", "hn", "cn", "hp", "z", "gz", "xo", "logits",
                 "alpha_all", "topk_stats", "cand_val", "cand_idx", "cand_key", "h_noisy", "tok_hist", "asrc_hist", "top_scores", "cur_tok", "src_row", "alive",
                 "kcur", "fin_tokens", "fin_asrc", "fin_len", "fin_score", "fin_ppl", "fin_count", "temps", "live_images", "done_host")] + \
               [("k", C.c_int32), ("max_gen_length", C.c_int32), ("rescore", C.c_int32), ("reward", C.c_float),
                ("tokPAD", C.c_int32), ("tokSTART", C.c_int32), ("tokEND", C.c_int32), ("tokUNK", C.c_int32),
                ("sample_method", C.c_int32), ("sample_topk", C.c_int32), ("kcap", C.c_int32), ("decoder_noise", C.c_float),
                ("sample_seed", C.c_uint64), ("call_id", C.c_int32), ("reserved1", C.c_int32)] + \
               [(n, vp) for n in ("tile_val", "tile_idx", "tile_key", "topk_stats2")]


class SatParamGrads(C.Structure):
    _fields_ = [(n, vp) for n in
                ("embedding", "fact_w", "fact_b", "init_w", "init_b", "w_ih", "w_hh", "b_ih", "b_hh", "enc_att", "dec_att",
                 "f_att", "beta_w", "beta_b", "out_hidden", "out_context", "out_w", "out_b")] + \
               [("w_ih_l", _vpl), ("w_hh_l", _vpl), ("b_ih_l", _vpl), ("b_hh_l", _vpl)] + \
               [("pad_idx", C.c_int32), ("weight_tying", C.c_int32)]


EXPORTS = ["sat_version", "sat_last_error", "sat_abi_sizeof", "sat_launch_count", "sat_profile_begin", "sat_profile_end", "sat_dropout_multiplier", "sat_pack_weights",
           "sat_linear", "sat_linear_nt", "sat_prepare_images", "sat_resize_nhwc_fwd", "sat_resize_nhwc_bwd",
           "sat_attention_step_fwd", "sat_cast_captions", "sat_train_forward", "sat_train_backward", "sat_param_grads_workspace_bytes", "sat_train_param_grads",
           "sat_train_vocab_path",
           "sat_decode_prepare_weights", "sat_decode", "sat_decode_vocab_path"]
VOCAB_PATH_ROWS, VOCAB_PATH_GREEDY, VOCAB_PATH_CAND = 0, 1, 2      # sat_decode_vocab_path
TRAIN_PATH_LOGITS, TRAIN_PATH_FUSED = 0, 1                           # sat_train_vocab_path

_lib = None


class SatError(RuntimeError):
    pass


def build(verbose=False):
    """Compile libsat_b200.so for sm_100a with nvcc (works without a GPU)."""
    root = os.path.dirname(_HERE)
    r = subprocess.run(["bash", os.path.join(root, "build.sh")], capture_output=True, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout[-4000:], r.stderr[-4000:])
    if r.returncode != 0:
        raise SatError("building libsat_b200.so failed")
    return LIB_PATH


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise SatError("libsat_b200.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'` "
                       "or ./build.sh); there is no CPU fallback for the SAT decoder path")
    L = C.CDLL(LIB_PATH)
    L.sat_last_error.restype = C.c_char_p
    L.sat_launch_count.restype = C.c_ulonglong
    L.sat_abi_sizeof.argtypes = [C.c_int]
    for i, st in enumerate((SatDims, SatWeights, SatTrainBuffers, SatDecodeBuffers, SatMasterWeights, SatParamGrads)):
        if L.sat_abi_sizeof(i) != C.sizeof(st):
            raise SatError("ABI mismatch for %s: lib %d vs ctypes %d" % (st.__name__, L.sat_abi_sizeof(i), C.sizeof(st)))
    L.sat_dropout_multiplier.argtypes = [C.c_float, C.c_uint64, C.c_uint32, C.c_uint64]
    L.sat_dropout_multiplier.restype = C.c_float
    L.sat_pack_weights.argtypes = [C.POINTER(SatDims), C.POINTER(SatMasterWeights), C.POINTER(SatWeights), vp]
    L.sat_profile_begin.argtypes = [C.c_int]
    L.sat_profile_end.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_int)]
    L.sat_linear.argtypes = [vp, C.c_int64, vp, C.c_int64, vp, vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                             C.c_int32, C.c_int32, C.c_int32, vp]
    L.sat_linear_nt.argtypes = [vp, C.c_int64, vp, C.c_int64, vp, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                C.c_int32, vp]
    L.sat_prepare_images.argtypes = [C.POINTER(SatDims), C.POINTER(SatWeights), vp, vp, vp, vp, vp, vp, vp, vp]
    L.sat_attention_step_fwd.argtypes = [C.POINTER(SatDims), vp, vp, vp, vp, C.c_int64, vp, C.c_int32, vp, C.c_int64,
                                         vp, vp, vp, C.c_int64, vp]
    L.sat_resize_nhwc_fwd.argtypes = [vp, vp] + [C.c_int32] * 7 + [vp]
    L.sat_resize_nhwc_bwd.argtypes = [vp, vp] + [C.c_int32] * 7 + [vp]
    L.sat_cast_captions.argtypes = [vp, vp, vp, vp, C.c_int64, C.c_int64, vp]
    L.sat_train_forward.argtypes = [C.POINTER(SatDims), C.POINTER(SatWeights), C.POINTER(SatTrainBuffers), vp]
    L.sat_train_vocab_path.argtypes = [C.POINTER(SatDims), C.c_int32]
    L.sat_train_backward.argtypes = [C.POINTER(SatDims), C.POINTER(SatWeights), C.POINTER(SatTrainBuffers), vp]
    L.sat_param_grads_workspace_bytes.argtypes = [C.POINTER(SatDims)]
    L.sat_param_grads_workspace_bytes.restype = C.c_int64
    L.sat_train_param_grads.argtypes = [C.POINTER(SatDims), C.POINTER(SatTrainBuffers), C.POINTER(SatParamGrads), vp, C.c_int64, vp]
    L.sat_decode_prepare_weights.argtypes = [C.POINTER(SatDims), C.POINTER(SatWeights), vp, vp]
    L.sat_decode.argtypes = [C.POINTER(SatDims), C.POINTER(SatWeights), C.POINTER(SatDecodeBuffers), vp]
    L.sat_decode_vocab_path.argtypes = [C.POINTER(SatDims), C.c_int32, C.c_int32, C.c_int32]
    _lib = L
    return L


def check(rc, what):
    if rc != 0:
        msg = lib().sat_last_error().decode("utf-8", "replace")
        raise SatError("%s failed (rc=%d): %s" % (what, rc, msg))


def ptr(t):
    """device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda, "sat_b200 kernels take CUDA tensors only (no CPU fallback)"
    return t.data_ptr()


def stream_ptr():
    return torch.cuda.current_stream().cuda_stream


def dtype_code(dt):
    if dt == torch.float32:
        return SAT_F32
    if dt == torch.bfloat16:
        return SAT_BF16
    raise SatError("unsupported dtype %s" % dt)


def profile_begin(kind):
    check(lib().sat_profile_begin(kind), "sat_profile_begin")


def profile_end():
    ms, n = C.c_float(0), C.c_int(0)
    check(lib().sat_profile_end(C.byref(ms), C.byref(n)), "sat_profile_end")
    return float(ms.value), int(n.value)


def launch_count():
    return int(lib().sat_launch_count())
