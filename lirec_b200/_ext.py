"""ctypes binding of liblirec_b200.so (the C ABI in include/lirec_b200.h).

PyTorch is only the owner of device memory and streams here: every call passes raw
pointers, sizes and the current CUDA stream.  There is no fallback of any kind: if the
shared library is missing, or the device is not sm_100, the call raises.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LIREC_B200_LIB", os.path.join(_HERE, "liblirec_b200.so"))

MAX_PASSES = 4
MAX_PROBLEMS = 32

ACT_NONE, ACT_RELU, ACT_TANH = 0, 1, 2
POST_NONE, POST_DROPOUT, POST_DRELU, POST_DTANH, POST_SIGN_MASK = 0, 1, 2, 3, 4
OUT_F32, OUT_SPLIT, OUT_SPLIT_T = 0, 1, 2
LAMB_CHUNK = 8192            # LIREC_LAMB_CHUNK: lirec_lamb_flat's partials hold n // LAMB_CHUNK + n_tensors entries


class Dropout(C.Structure):
    _fields_ = [("p", C.c_float), ("seed", C.c_uint32), ("stream_id", C.c_uint32), ("col_off", C.c_int32)]


class Operand(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("rows", C.c_int64), ("cols", C.c_int64), ("ld", C.c_int64)]


class GemmPass(C.Structure):
    _fields_ = [("a", Operand), ("b", Operand),
                ("a_mn_off", C.c_int32), ("a_k_off", C.c_int32),
                ("b_mn_off", C.c_int32), ("b_k_off", C.c_int32),
                ("k_len", C.c_int32)]


class Epilogue(C.Structure):
    _fields_ = [("alpha", C.c_float), ("bias", C.c_void_p), ("row_flag", C.c_void_p),
                ("act", C.c_int32), ("post", C.c_int32), ("post_scale", C.c_float),
                ("drop", Dropout),
                ("aux", C.c_void_p), ("aux_ld", C.c_int64),
                ("aux_col_off", C.c_int32), ("aux_lo_off", C.c_int32),
                ("out_kind", C.c_int32), ("out", C.c_void_p),
                ("out_ld_m", C.c_int64), ("out_ld_n", C.c_int64),
                ("out_col_off", C.c_int32), ("out_lo_off", C.c_int32),
                ("accumulate", C.c_int32)]


class GemmProblem(C.Structure):
    _fields_ = [("M", C.c_int32), ("N", C.c_int32),
                ("a_mn_major", C.c_int32), ("b_mn_major", C.c_int32),
                ("num_passes", C.c_int32),
                ("pass_", GemmPass * MAX_PASSES),
                ("epi", Epilogue),
                ("split_k", C.c_int32), ("split_stride", C.c_int64)]


class TrackLossCfg(C.Structure):
    _fields_ = [("margin", C.c_float), ("lymbda", C.c_float), ("n_classes", C.c_int32),
                ("n_rels", C.c_int32), ("tr_correct", C.c_int32), ("max_neg", C.c_int32),
                ("max_slots", C.c_int32), ("cat_distr", C.c_int32), ("seed", C.c_uint32)]


class Linear(C.Structure):
    _fields_ = [("w_bf16", C.c_void_p), ("bias", C.c_void_p), ("grad_w", C.c_void_p),
                ("grad_b", C.c_void_p), ("out_f", C.c_int32), ("in_f", C.c_int32)]


class Encoder(C.Structure):
    _fields_ = [("l1", Linear * 4), ("l2", Linear * 4)]


class ModelParams(C.Structure):
    _fields_ = [("enc_ints", Encoder), ("enc_ctx", Encoder), ("gate", Linear),
                ("out_ints", Linear), ("out_ctx", Linear)]


class ModelCfg(C.Structure):
    _fields_ = [("text_dim", C.c_int32), ("visual_dim", C.c_int32), ("track_dim", C.c_int32),
                ("joint_dim", C.c_int32), ("gate_dim", C.c_int32),
                ("n_classes", C.c_int32), ("n_rels", C.c_int32),
                ("ctx", C.c_int32), ("gates", C.c_int32), ("guard_zero", C.c_int32),
                ("dropout_p", C.c_float), ("slot_mask", C.c_int32), ("no_ints", C.c_int32)]


class Batch(C.Structure):
    _fields_ = [("clip_bank", C.c_void_p), ("clip_ld", C.c_int64),
                ("n_clip", C.c_int32), ("n_clip_ints", C.c_int32),
                ("track_bank", C.c_void_p), ("track_ld", C.c_int64),
                ("n_track", C.c_int32), ("n_track_ints", C.c_int32),
                ("n_cand", C.c_int32), ("n_ctx_rows", C.c_int32),
                ("cand_rows", C.c_void_p), ("ctx_rows", C.c_void_p),
                ("ctx_off", C.c_void_p), ("ctx_owner", C.c_void_p),
                ("inv_cand_off", C.c_void_p * 3), ("inv_cand_idx", C.c_void_p * 3),
                ("inv_ctx_off", C.c_void_p * 3), ("inv_ctx_idx", C.c_void_p * 3),
                ("seed", C.c_uint32), ("training", C.c_int32)]


_lib = None


def lib():
    """Load the shared library (once). Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "liblirec_b200.so is missing (%s). Build it with `python -m lirec_b200.build`; "
            "lirec_b200 has no CPU or PyTorch fallback." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    L.lirec_last_error.restype = C.c_char_p
    L.lirec_abi_version.restype = C.c_int
    L.lirec_last_launch_count.restype = C.c_int
    L.lirec_device_check.argtypes = [C.c_int]
    L.lirec_dropout_keep_host.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_float]
    L.lirec_gemm_grouped.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    L.lirec_seg_reduce_f32.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                       C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
    L.lirec_seg_softmax_pool_fwd.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32,
                                             C.c_float, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
    L.lirec_seg_softmax_pool_bwd.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32,
                                             C.c_float, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                             C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    L.lirec_rows_expand_fwd.argtypes = [C.c_void_p] * 4 + [C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                                           C.c_int32, Dropout, C.c_void_p, C.c_int64,
                                                           C.c_void_p, C.c_void_p]
    L.lirec_rows_expand_bwd.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int32, C.c_int32,
                                        C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                        Dropout, C.c_void_p, C.c_int64, C.c_void_p]
    L.lirec_split_f32.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_int64,
                                  C.c_int32, C.c_void_p]
    L.lirec_roi_max_pool_f32.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                         C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                         C.c_int64, C.c_void_p]
    L.lirec_gather_rows.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int32, C.c_int32,
                                    C.c_void_p, C.c_int64, C.c_void_p]
    L.lirec_cast_bf16.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    L.lirec_loss_track_fwd_bwd.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p, TrackLossCfg,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.lirec_loss_rowmargin_fwd_bwd.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p,
                                               C.c_void_p, C.c_float, C.c_float, C.c_void_p, C.c_void_p,
                                               C.c_int64, C.c_void_p]
    L.lirec_loss_ce_fwd_bwd.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                        C.c_float, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    L.lirec_loss_bce_fwd_bwd.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    L.lirec_loss_bce_track_fwd_bwd.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, TrackLossCfg,
                                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.lirec_predict_tracks.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    L.lirec_adam_flat.argtypes = [C.c_void_p] * 5 + [C.c_int64] + [C.c_float] * 5 + [C.c_int32, C.c_float,
                                                                                  C.c_int32, C.c_void_p]
    L.lirec_lamb_flat.argtypes = [C.c_void_p] * 7 + [C.c_int32, C.c_int64, C.c_void_p, C.c_int64] + [C.c_float] * 5 + [
        C.c_int32, C.c_float, C.c_void_p, C.c_void_p]
    L.lirec_grad_clip_flat.argtypes = [C.c_void_p] * 3 + [C.c_int32, C.c_int64, C.c_void_p, C.c_int64, C.c_float,
                                                          C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]
    L.lirec_profile_sample.argtypes = [C.c_int32]
    L.lirec_dp_flag_words.argtypes = [C.c_int32]
    L.lirec_dp_flag_words.restype = C.c_int
    L.lirec_dp_reduce_adam_bcast.argtypes = [C.c_void_p] * 6 + [C.c_int64] + [C.c_float] * 5 + [
        C.c_int32, C.c_float, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]
    L.lirec_dp_reduce_adam_bcast_peer.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p,
                                                  C.c_int64] + [C.c_float] * 5 + [
        C.c_int32, C.c_float, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]
    L.lirec_dp_exchange.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                    C.c_int32, C.c_void_p]
    L.lirec_model_workspace_bytes.argtypes = [C.c_void_p, C.c_void_p]
    L.lirec_model_workspace_bytes.restype = C.c_size_t
    L.lirec_profile_end.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    L.lirec_model_workspace_layout.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    L.lirec_model_forward.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                      C.c_void_p, C.c_void_p, C.c_void_p]
    L.lirec_model_backward.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.lirec_collate_arena_bound.argtypes = [C.c_int64, C.c_int64, C.c_int64, C.c_int32]
    L.lirec_collate_arena_bound.restype = C.c_int64
    L.lirec_collate_tables.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                       C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p,
                                       C.c_void_p]
    L.lirec_collate_gather.argtypes = [C.c_void_p] * 6 + [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                                          C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    if L.lirec_abi_version() != 3:
        raise RuntimeError("liblirec_b200.so ABI version mismatch; rebuild it")
    _lib = L
    return L


EXPORTED_SYMBOLS = [
    "lirec_abi_version", "lirec_last_error", "lirec_device_check", "lirec_dropout_keep_host", "lirec_last_launch_count",
    "lirec_gemm_grouped", "lirec_profile_begin", "lirec_profile_end", "lirec_seg_reduce_f32", "lirec_seg_softmax_pool_fwd", "lirec_seg_softmax_pool_bwd", "lirec_rows_expand_fwd", "lirec_rows_expand_bwd",
    "lirec_split_f32", "lirec_cast_bf16", "lirec_gather_rows", "lirec_roi_max_pool_f32", "lirec_loss_track_fwd_bwd", "lirec_loss_rowmargin_fwd_bwd", "lirec_loss_ce_fwd_bwd",
    "lirec_loss_bce_fwd_bwd", "lirec_loss_bce_track_fwd_bwd", "lirec_predict_tracks",
    "lirec_model_workspace_bytes", "lirec_model_workspace_layout", "lirec_model_forward", "lirec_model_backward", "lirec_adam_flat", "lirec_lamb_flat", "lirec_grad_clip_flat", "lirec_profile_sample", "lirec_dp_flag_words", "lirec_dp_exchange", "lirec_dp_reduce_adam_bcast", "lirec_dp_reduce_adam_bcast_peer",
    "lirec_collate_arena_bound", "lirec_collate_tables", "lirec_collate_gather",
]

# kernels launched through this binding since import (bench.py reports it as gpu_launches)
launch_counter = 0


def check(rc):
    global launch_counter
    if rc != 0:
        raise RuntimeError("liblirec_b200: %s (code %d)" % (lib().lirec_last_error().decode(), rc))
    launch_counter += lib().lirec_last_launch_count()


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("liblirec_b200 needs CUDA tensors (got a %s tensor); there is no CPU path" % t.device)
    return t.data_ptr()


def require_device(device=None):
    L = lib()
    if not torch.cuda.is_available():
        raise RuntimeError("lirec_b200 requires a B200 (sm_100) GPU; no CUDA device is visible and "
                           "there is no CPU fallback")
    dev = torch.cuda.current_device() if device is None else torch.device(device).index or 0
    check(L.lirec_device_check(dev))


def operand(t, rows=None, cols=None, col_off=0):
    """2-D bf16 view (ptr, rows, cols, ld) of tensor `t`, optionally a column window."""
    assert t.dtype == torch.bfloat16 and t.dim() == 2 and t.stride(1) == 1
    o = Operand()
    o.ptr = t.data_ptr() + 2 * col_off
    o.rows = t.shape[0] if rows is None else rows
    o.cols = (t.shape[1] - col_off) if cols is None else cols
    o.ld = t.stride(0)
    return o


def gemm_grouped(problems):
    arr = (GemmProblem * len(problems))(*problems)
    check(lib().lirec_gemm_grouped(C.cast(arr, C.c_void_p), len(problems), stream_ptr()))


def profile_begin():
    check(lib().lirec_profile_begin())


def profile_sample(on):
    lib().lirec_profile_sample(1 if on else 0)


def profile_end(max_records=65536):
    """Returns a list of (ms, executed_flops, tiles, problems) per GEMM launch since profile_begin()."""
    ms = (C.c_float * max_records)()
    fl = (C.c_double * max_records)()
    ti = (C.c_int32 * max_records)()
    pr = (C.c_int32 * max_records)()
    n = lib().lirec_profile_end(ms, fl, ti, pr, max_records)
    if n < 0:
        check(n)
    return [(ms[i], fl[i], ti[i], pr[i]) for i in range(n)]
