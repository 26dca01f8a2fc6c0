"""Thin torch-tensor wrappers over the C ABI (one function per entry point).

These are the calls the unit parity tests exercise op by op; the model itself goes through
lirec_model_forward / lirec_model_backward (see lirec_b200/mlp/model.py).
"""
import ctypes as C

import torch

from . import _ext
from ._ext import (ACT_NONE, ACT_RELU, ACT_TANH, OUT_F32, OUT_SPLIT, OUT_SPLIT_T, POST_DRELU, POST_DROPOUT, POST_DTANH,
                   POST_NONE, POST_SIGN_MASK)

__all__ = ["gemm_problem", "gemm_grouped", "seg_reduce", "seg_softmax_pool", "seg_softmax_pool_bwd", "SegSoftmaxPool", "rows_expand_fwd", "rows_expand_bwd", "split_f32",
           "cast_bf16", "gather_rows", "roi_max_pool", "loss_track", "loss_rowmargin", "loss_ce", "loss_bce", "loss_bce_track", "predict_tracks", "adam_flat", "lamb_partials", "lamb_flat", "grad_clip_flat", "dp_exchange", "dp_reduce_adam_bcast", "dp_reduce_adam_bcast_peer", "dropout_desc"]


def dropout_desc(p=0.0, seed=0, stream_id=0, col_off=0):
    d = _ext.Dropout()
    d.p, d.seed, d.stream_id, d.col_off = float(p), int(seed) & 0xFFFFFFFF, int(stream_id), int(col_off)
    return d


def gemm_problem(M, N, passes, a_mn_major=False, b_mn_major=False, alpha=1.0, bias=None, row_flag=None,
                 act=ACT_NONE, post=POST_NONE, post_scale=1.0, drop=None, aux=None, aux_col_off=0,
                 aux_lo_off=0, out=None, out_kind=OUT_F32, out_ld_m=None, out_ld_n=1, out_col_off=0,
                 out_lo_off=0, accumulate=False, split_k=0, split_stride=0):
    """passes: list of (a_operand, a_mn_off, a_k_off, b_operand, b_mn_off, b_k_off, k_len)."""
    g = _ext.GemmProblem()
    g.M, g.N = int(M), int(N)
    g.a_mn_major, g.b_mn_major = int(a_mn_major), int(b_mn_major)
    g.num_passes = len(passes)
    assert 1 <= len(passes) <= _ext.MAX_PASSES
    for i, (a, amn, ak, b, bmn, bk, klen) in enumerate(passes):
        p = g.pass_[i]
        p.a, p.b = a, b
        p.a_mn_off, p.a_k_off, p.b_mn_off, p.b_k_off, p.k_len = int(amn), int(ak), int(bmn), int(bk), int(klen)
    e = g.epi
    e.alpha = float(alpha)
    e.bias = _ext.ptr(bias)
    e.row_flag = _ext.ptr(row_flag)
    e.act, e.post, e.post_scale = int(act), int(post), float(post_scale)
    e.drop = drop if drop is not None else dropout_desc()
    if aux is not None:
        e.aux, e.aux_ld = aux.data_ptr(), aux.stride(0)
    e.aux_col_off, e.aux_lo_off = int(aux_col_off), int(aux_lo_off)
    e.out_kind = int(out_kind)
    e.out = out.data_ptr()
    e.out_ld_m = int(out.stride(0) if out_ld_m is None else out_ld_m)
    e.out_ld_n = int(out_ld_n)
    e.out_col_off, e.out_lo_off = int(out_col_off), int(out_lo_off)
    e.accumulate = int(accumulate)
    g.split_k, g.split_stride = int(split_k), int(split_stride)
    return g


def gemm_grouped(problems):
    _ext.gemm_grouped(problems)


def seg_reduce(x, seg_off, mode="max", out_f32=None, out_bf16=None, row_idx=None):
    """Segmented max/mean of ragged fp32 rows. x [total, dim], seg_off int32 [nseg+1].  row_idx (int32):
    segment s reduces the gathered rows x[row_idx[seg_off[s]:seg_off[s+1]]] instead of a contiguous range."""
    assert x.dtype == torch.float32 and x.dim() == 2 and x.is_contiguous()
    assert seg_off.dtype == torch.int32
    nseg = seg_off.numel() - 1
    assert row_idx is None or row_idx.dtype == torch.int32
    _ext.check(_ext.lib().lirec_seg_reduce_f32(
        _ext.ptr(x), _ext.ptr(row_idx), _ext.ptr(seg_off), nseg, x.shape[1], 0 if mode == "max" else 1,
        _ext.ptr(out_f32), out_f32.stride(0) if out_f32 is not None else 0,
        _ext.ptr(out_bf16), out_bf16.stride(0) if out_bf16 is not None else 0, _ext.stream_ptr()))


def _score_mode(x, scores):
    if scores is None:
        return 0
    assert scores.dtype == torch.float32 and scores.is_contiguous()
    if scores.dim() == 1:
        assert scores.numel() == x.shape[0]
        return 2
    assert scores.shape == x.shape
    return 1


def seg_softmax_pool(x, seg_off, beta=1.0, scores=None, need_lse=True):
    """Softmax-weighted segmented reduction (lirec_seg_softmax_pool_fwd; parity unpinned — the reference has none).
    x [total, dim] fp32; scores None (score = x), [total, dim] or [total].  Returns (out [nseg, dim], lse)."""
    assert x.dtype == torch.float32 and x.dim() == 2 and x.is_contiguous() and seg_off.dtype == torch.int32
    mode = _score_mode(x, scores)
    nseg, dim = seg_off.numel() - 1, x.shape[1]
    out = torch.empty(nseg, dim, dtype=torch.float32, device=x.device)
    lse = None
    if need_lse:
        lse = torch.empty((nseg,) if mode == 2 else (nseg, dim), dtype=torch.float32, device=x.device)
    _ext.check(_ext.lib().lirec_seg_softmax_pool_fwd(
        _ext.ptr(x), _ext.ptr(scores), mode, _ext.ptr(seg_off), nseg, dim, float(beta), _ext.ptr(out), out.stride(0),
        _ext.ptr(lse), lse.stride(0) if (lse is not None and lse.dim() == 2) else 0, _ext.stream_ptr()))
    return out, lse


def seg_softmax_pool_bwd(x, seg_off, beta, scores, out, lse, d_out, need_d_scores=True):
    """Gradients of seg_softmax_pool: (d_x, d_scores | None)."""
    mode = _score_mode(x, scores)
    nseg, dim = seg_off.numel() - 1, x.shape[1]
    d_out = d_out.contiguous()
    d_x = torch.empty_like(x)                      # rows outside the segments are zero-filled by the launch itself
    d_s = torch.empty_like(scores) if (mode != 0 and need_d_scores) else None
    _ext.check(_ext.lib().lirec_seg_softmax_pool_bwd(
        _ext.ptr(x), _ext.ptr(scores), mode, _ext.ptr(seg_off), nseg, dim, float(beta), _ext.ptr(out), out.stride(0),
        _ext.ptr(lse), lse.stride(0) if lse.dim() == 2 else 0, _ext.ptr(d_out), d_out.stride(0), _ext.ptr(d_x),
        _ext.ptr(d_s), x.shape[0], _ext.stream_ptr()))
    return d_x, d_s


class SegSoftmaxPool(torch.autograd.Function):
    """Differentiable front of the two entry points (x and scores may require grad)."""

    @staticmethod
    def forward(ctx, x, seg_off, beta, scores):
        out, lse = seg_softmax_pool(x, seg_off, beta, scores)
        ctx.save_for_backward(x, seg_off, scores if scores is not None else x.new_empty(0), out, lse)
        ctx.beta, ctx.has_scores = float(beta), scores is not None
        return out

    @staticmethod
    def backward(ctx, d_out):
        x, seg_off, scores, out, lse = ctx.saved_tensors
        scores = scores if ctx.has_scores else None
        d_x, d_s = seg_softmax_pool_bwd(x, seg_off, ctx.beta, scores, out, lse, d_out)
        return d_x, None, None, d_s


def rows_expand_fwd(r1, J, rows, seg_off, n_out, guard_zero, drop, out_split, row_flag_out=None):
    L = _ext.lib()
    _ext.check(L.lirec_rows_expand_fwd(
        _ext.ptr(r1[0]), _ext.ptr(r1[1]), _ext.ptr(r1[2]), _ext.ptr(r1[3]), J, _ext.ptr(rows),
        _ext.ptr(seg_off), n_out, int(guard_zero), drop, _ext.ptr(out_split), out_split.stride(0),
        _ext.ptr(row_flag_out), _ext.stream_ptr()))


def rows_expand_bwd(d_in, d_ld, sign, J, slot, inv_off, inv_idx, n_unique, owner, seg_off, drop, out_split,
                    d_in_col_off=0):
    """sign: int32 [n_unique, >= J / 32] ReLU gate bits (LIREC_POST_SIGN_MASK layout); out_split: [2J, pitch] hi
    rows then lo rows, pitch = out_split.stride(0)."""
    L = _ext.lib()
    _ext.check(L.lirec_rows_expand_bwd(
        d_in.data_ptr() + 4 * d_in_col_off, d_ld, _ext.ptr(sign), sign.stride(0), J, slot, _ext.ptr(inv_off),
        _ext.ptr(inv_idx), n_unique, _ext.ptr(owner), _ext.ptr(seg_off), drop, _ext.ptr(out_split),
        out_split.stride(0), _ext.stream_ptr()))


def split_f32(x, out_split, pad):
    """x fp32 [rows, cols] -> out_split [2 * pad, pitch >= rows]: hi of x[r, c] at out_split[c, r], lo at
    out_split[pad + c, r], rows [cols, pad) of each half zero."""
    L = _ext.lib()
    _ext.check(L.lirec_split_f32(_ext.ptr(x), x.stride(0), x.shape[0], x.shape[1], _ext.ptr(out_split),
                                 out_split.stride(0), pad, _ext.stream_ptr()))


def cast_bf16(x, out):
    L = _ext.lib()
    _ext.check(L.lirec_cast_bf16(_ext.ptr(x), _ext.ptr(out), x.numel(), _ext.stream_ptr()))


def roi_max_pool(maps, elem, seg_off, out_f32=None, out_bf16=None, two_stage=True):
    """out[s, c] = max_{e in segment s} mean(maps[frame_e, c, y0:y1, x0:x1]) (lirec_roi_max_pool_f32).
    maps fp32 [T, C, H, W]; elem int32 [n, 5]; seg_off int32 [nseg + 1].  two_stage: give the kernel a
    scratch of per-element means (fully parallel pass + segmented max) instead of the single-pass form."""
    assert maps.dtype == torch.float32 and maps.dim() == 4 and maps.is_contiguous()
    assert elem.dtype == torch.int32 and seg_off.dtype == torch.int32 and elem.is_contiguous()
    T, Cc, H, W = maps.shape
    nseg = seg_off.numel() - 1
    if out_f32 is None and out_bf16 is None:
        out_f32 = torch.empty(nseg, Cc, dtype=torch.float32, device=maps.device)
    n_elem = elem.shape[0]
    scratch = torch.empty(n_elem, Cc, dtype=torch.float32, device=maps.device) if (two_stage and Cc % 4 == 0) else None
    _ext.check(_ext.lib().lirec_roi_max_pool_f32(
        _ext.ptr(maps), T, Cc, H, W, _ext.ptr(elem), n_elem, _ext.ptr(seg_off), nseg, _ext.ptr(scratch),
        _ext.ptr(out_f32), out_f32.stride(0) if out_f32 is not None else 0,
        _ext.ptr(out_bf16), out_bf16.stride(0) if out_bf16 is not None else 0, _ext.stream_ptr()))
    return out_f32 if out_f32 is not None else out_bf16


def gather_rows(bank, idx, out=None):
    """out[i] = bank[idx[i]] over bf16 rows on the device (lirec_gather_rows)."""
    assert bank.dtype == torch.bfloat16 and bank.dim() == 2 and bank.stride(1) == 1 and idx.dtype == torch.int32
    if out is None:
        out = torch.empty(idx.numel(), bank.shape[1], dtype=torch.bfloat16, device=bank.device)
    _ext.check(_ext.lib().lirec_gather_rows(_ext.ptr(bank), bank.stride(0), bank.shape[0], _ext.ptr(idx), idx.numel(),
                                            bank.shape[1], _ext.ptr(out), out.stride(0), _ext.stream_ptr()))
    return out


def _track_loss_cfg_and_outputs(ints, rels, cand_off, margin, lymbda, n_rels, tr_correct, max_neg, max_slots,
                                cat_distr, seed):
    """The TrackLossCfg of both track losses and their outputs (loss_per_clip, assign, d_ints, d_rels)."""
    B = cand_off.numel() - 1
    cfg = _ext.TrackLossCfg()
    cfg.margin, cfg.lymbda = float(margin), float(lymbda)
    cfg.n_classes, cfg.n_rels = int(ints.shape[1]), int(n_rels)
    cfg.tr_correct, cfg.max_neg, cfg.max_slots = int(tr_correct), int(max_neg), int(max_slots)
    cfg.cat_distr, cfg.seed = int(cat_distr), int(seed) & 0xFFFFFFFF
    loss = torch.empty(B, dtype=torch.float32, device=ints.device)
    assign = torch.empty(B, dtype=torch.int32, device=ints.device)
    d_ints = torch.empty_like(ints)
    d_rels = torch.empty_like(rels) if n_rels > 0 else None
    return cfg, (loss, assign, d_ints, d_rels)


def loss_track(ints, rels, cand_off, labels, rels_label, gt_tracks, multilab, margin, lymbda, n_rels,
               tr_correct=False, max_neg=False, max_slots=20, cat_distr=False, seed=0):
    """Fused MarginLoss / MarginTrackRelsLoss. Returns (loss_per_clip, assign, d_ints, d_rels)."""
    cfg, out = _track_loss_cfg_and_outputs(ints, rels, cand_off, margin, lymbda, n_rels, tr_correct, max_neg,
                                           max_slots, cat_distr, seed)
    loss, assign, d_ints, d_rels = out
    _ext.check(_ext.lib().lirec_loss_track_fwd_bwd(
        _ext.ptr(ints), _ext.ptr(rels) if n_rels > 0 else None, _ext.ptr(cand_off), loss.numel(), _ext.ptr(labels),
        _ext.ptr(rels_label) if n_rels > 0 else None, _ext.ptr(gt_tracks), _ext.ptr(multilab), cfg,
        _ext.ptr(loss), _ext.ptr(assign), _ext.ptr(d_ints), _ext.ptr(d_rels), _ext.stream_ptr()))
    return out


def loss_ce(logits, labels, class_weights, scale):
    """Softmax cross-entropy rows, forward + gradient (lirec_loss_ce_fwd_bwd). labels < 0 are skipped."""
    rows, Cc = logits.shape
    loss = torch.empty(rows, dtype=torch.float32, device=logits.device)
    d = torch.empty_like(logits)
    _ext.check(_ext.lib().lirec_loss_ce_fwd_bwd(_ext.ptr(logits), logits.stride(0), rows, Cc, _ext.ptr(labels),
                                                _ext.ptr(class_weights), float(scale), _ext.ptr(loss), _ext.ptr(d),
                                                d.stride(0), _ext.stream_ptr()))
    return loss, d


def loss_bce(logits, labels, neg_mask, pos_mask, scale):
    """Multi-label sigmoid BCE rows, forward + gradient (lirec_loss_bce_fwd_bwd): target 1 on the label and on
    pos_mask, non-targets with neg_mask == 0 left out (masks uint8 [rows, C] or None). labels < 0 are skipped."""
    rows, Cc = logits.shape
    loss = torch.empty(rows, dtype=torch.float32, device=logits.device)
    d = torch.empty_like(logits)
    _ext.check(_ext.lib().lirec_loss_bce_fwd_bwd(
        _ext.ptr(logits), logits.stride(0), rows, Cc, _ext.ptr(labels), _ext.ptr(neg_mask), _ext.ptr(pos_mask),
        float(scale), _ext.ptr(loss), _ext.ptr(d), d.stride(0), _ext.stream_ptr()))
    return loss, d


def loss_bce_track(ints, rels, cand_off, labels, rels_label, gt_tracks, multilab, pos_mask, lymbda, n_rels,
                   tr_correct=False, max_slots=20, cat_distr=False, seed=0):
    """Fused BCE over the weakly supervised track assignment (lirec_loss_bce_track_fwd_bwd); t* is chosen as in
    loss_track. Returns (loss_per_clip, assign, d_ints, d_rels)."""
    cfg, out = _track_loss_cfg_and_outputs(ints, rels, cand_off, 0.0, lymbda, n_rels, tr_correct, False, max_slots,
                                           cat_distr, seed)
    loss, assign, d_ints, d_rels = out
    _ext.check(_ext.lib().lirec_loss_bce_track_fwd_bwd(
        _ext.ptr(ints), _ext.ptr(rels) if n_rels > 0 else None, _ext.ptr(cand_off), loss.numel(), _ext.ptr(labels),
        _ext.ptr(rels_label) if n_rels > 0 else None, _ext.ptr(gt_tracks), _ext.ptr(multilab), _ext.ptr(pos_mask), cfg,
        _ext.ptr(loss), _ext.ptr(assign), _ext.ptr(d_ints), _ext.ptr(d_rels), _ext.stream_ptr()))
    return out


def loss_rowmargin(logits, labels, weights, margin, scale):
    rows, Cc = logits.shape
    loss = torch.empty(rows, dtype=torch.float32, device=logits.device)
    d = torch.empty_like(logits)
    L = _ext.lib()
    _ext.check(L.lirec_loss_rowmargin_fwd_bwd(
        _ext.ptr(logits), logits.stride(0), rows, Cc, _ext.ptr(labels), _ext.ptr(weights), float(margin),
        float(scale), _ext.ptr(loss), _ext.ptr(d), d.stride(0), _ext.stream_ptr()))
    return loss, d


def predict_tracks(ints, rels, cand_off, labels, rels_label, gt_tracks, n_rels):
    """Device-side prediction arg-maxes; returns int32 [B, 8] (see include/lirec_b200.h)."""
    B = cand_off.numel() - 1
    out = torch.empty(B, 8, dtype=torch.int32, device=ints.device)
    L = _ext.lib()
    _ext.check(L.lirec_predict_tracks(_ext.ptr(ints), _ext.ptr(rels) if n_rels else None, _ext.ptr(cand_off), B,
                                      _ext.ptr(labels), _ext.ptr(rels_label) if n_rels else None,
                                      _ext.ptr(gt_tracks), ints.shape[1], int(n_rels), _ext.ptr(out),
                                      _ext.stream_ptr()))
    return out


def adam_flat(param, grad, exp_avg, exp_avg_sq, param_bf16, lr, beta1, beta2, eps, weight_decay, step,
              grad_scale=1.0, offset=0, n=None, stream=None, coresident=False):
    """Fused Adam over floats [offset, offset + n) of the flat buffers (default: everything) on `stream`.
    coresident: CTAs that fit beside a resident GEMM CTA (a pass overlapped with backward on a side stream)."""
    L = _ext.lib()
    n = param.numel() - offset if n is None else n
    sp = _ext.stream_ptr() if stream is None else C.c_void_p(stream.cuda_stream)
    _ext.check(L.lirec_adam_flat(_ext.ptr(param) + 4 * offset, _ext.ptr(grad) + 4 * offset,
                                 _ext.ptr(exp_avg) + 4 * offset, _ext.ptr(exp_avg_sq) + 4 * offset,
                                 (_ext.ptr(param_bf16) + 2 * offset) if param_bf16 is not None else None, int(n),
                                 float(lr), float(beta1), float(beta2),
                                 float(eps), float(weight_decay), int(step), float(grad_scale), int(bool(coresident)),
                                 sp))


def lamb_partials(n, n_tensors, device=None):
    """Scratch of lirec_lamb_flat for flat buffers of n floats cut into n_tensors tensors (LIREC_LAMB_PARTIALS)."""
    return torch.empty(int(n) // _ext.LAMB_CHUNK + int(n_tensors), 2, dtype=torch.float64, device=device)


def lamb_flat(param, grad, exp_avg, exp_avg_sq, param_bf16, tensor_begin, tensor_len, partials, lr, beta1, beta2, eps,
              weight_decay, step, grad_scale=1.0, trust_out=None, stream=None):
    """Fused LAMB step over the flat buffers (lirec_lamb_flat).  tensor_begin / tensor_len: int64 device tensors
    [n_tensors] in floats; partials: lamb_partials(param.numel(), n_tensors); trust_out: optional float32 device
    tensor [n_tensors] that receives the trust ratios.  The entry point takes 1 - beta, formed here in double."""
    n_tensors = tensor_begin.numel()
    if any(t.numel() != param.numel() for t in (grad, exp_avg, exp_avg_sq)):
        raise ValueError("lamb_flat: param, grad, exp_avg and exp_avg_sq must have one size")
    for t in (tensor_begin, tensor_len):
        if t.dtype != torch.int64 or t.numel() != n_tensors or not t.is_contiguous():
            raise ValueError("lamb_flat: tensor_begin / tensor_len must be contiguous int64 tensors of one length")
    if partials.dtype != torch.float64 or not partials.is_contiguous():
        raise ValueError("lamb_flat: partials must be a contiguous float64 tensor (ops.lamb_partials)")
    if trust_out is not None and (trust_out.dtype != torch.float32 or trust_out.numel() < n_tensors):
        raise ValueError("lamb_flat: trust_out must be float32 with one entry per tensor")
    sp = _ext.stream_ptr() if stream is None else C.c_void_p(stream.cuda_stream)
    _ext.check(_ext.lib().lirec_lamb_flat(
        _ext.ptr(param), _ext.ptr(grad), _ext.ptr(exp_avg), _ext.ptr(exp_avg_sq), _ext.ptr(param_bf16),
        _ext.ptr(tensor_begin), _ext.ptr(tensor_len), int(n_tensors), int(param.numel()), _ext.ptr(partials),
        int(partials.numel() // 2), float(lr), 1.0 - float(beta1), 1.0 - float(beta2), float(eps), float(weight_decay),
        int(step), float(grad_scale), _ext.ptr(trust_out), sp))


def grad_clip_flat(grad, tensor_begin, tensor_len, partials, max_norm, grad_scale=1.0, norm_out=None,
                   tensor_norms_out=None, stream=None):
    """Global-norm clipping of the flat gradient buffer in place (lirec_grad_clip_flat): norm = ||grad_scale * grad||
    over the tensor table, grad *= min(max_norm / (norm + 1e-6), 1).  tensor_begin / tensor_len: int64 device tensors
    [n_tensors] in floats; partials: lamb_partials(grad.numel(), n_tensors); norm_out: optional float32 device tensor
    of one element (allocated when None); tensor_norms_out: optional float32 device tensor [n_tensors].  Returns
    norm_out, which the kernels fill on the stream without a host sync."""
    n_tensors = tensor_begin.numel()
    if grad.dtype != torch.float32 or not grad.is_contiguous():
        raise ValueError("grad_clip_flat: grad must be a contiguous float32 tensor")
    for t in (tensor_begin, tensor_len):
        if t.dtype != torch.int64 or t.numel() != n_tensors or not t.is_contiguous():
            raise ValueError("grad_clip_flat: tensor_begin / tensor_len must be contiguous int64 tensors of one length")
    if partials.dtype != torch.float64 or not partials.is_contiguous():
        raise ValueError("grad_clip_flat: partials must be a contiguous float64 tensor (ops.lamb_partials)")
    if norm_out is None:
        norm_out = torch.empty((), dtype=torch.float32, device=grad.device)
    elif norm_out.dtype != torch.float32 or norm_out.numel() != 1:
        raise ValueError("grad_clip_flat: norm_out must be a float32 tensor of one element")
    if tensor_norms_out is not None and (tensor_norms_out.dtype != torch.float32 or
                                         tensor_norms_out.numel() < n_tensors):
        raise ValueError("grad_clip_flat: tensor_norms_out must be float32 with one entry per tensor")
    sp = _ext.stream_ptr() if stream is None else C.c_void_p(stream.cuda_stream)
    _ext.check(_ext.lib().lirec_grad_clip_flat(
        _ext.ptr(grad), _ext.ptr(tensor_begin), _ext.ptr(tensor_len), int(n_tensors), int(grad.numel()),
        _ext.ptr(partials), int(partials.numel() // 2), float(max_norm), float(grad_scale), _ext.ptr(norm_out),
        _ext.ptr(tensor_norms_out), sp))
    return norm_out


def dp_reduce_adam_bcast(grad_mc, param, param_mc, bf16_mc, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay,
                         step, grad_scale, rank, world, flag_ptrs_dev, channel, stream=None, coresident=False):
    """In-switch gradient sum of this rank's shard + Adam on the shard + multicast of the new parameters and their
    bf16 shadow to every rank (lirec_dp_reduce_adam_bcast)."""
    L = _ext.lib()
    sp = _ext.stream_ptr() if stream is None else C.c_void_p(stream.cuda_stream)
    _ext.check(L.lirec_dp_reduce_adam_bcast(
        C.c_void_p(int(grad_mc)), _ext.ptr(param), C.c_void_p(int(param_mc)), C.c_void_p(int(bf16_mc)),
        _ext.ptr(exp_avg), _ext.ptr(exp_avg_sq), int(n), float(lr), float(beta1), float(beta2), float(eps),
        float(weight_decay), int(step), float(grad_scale), int(rank), int(world), C.c_void_p(int(flag_ptrs_dev)),
        int(channel), int(bool(coresident)), sp))


def dp_reduce_adam_bcast_peer(peer_bases_dev, grad_off, param_off, bf16_off, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps,
                              weight_decay, step, grad_scale, rank, world, flag_ptrs_dev, channel, stream=None,
                              coresident=False):
    """lirec_dp_reduce_adam_bcast over plain peer pointers (P2P loads / stores instead of multicast)."""
    L = _ext.lib()
    sp = _ext.stream_ptr() if stream is None else C.c_void_p(stream.cuda_stream)
    _ext.check(L.lirec_dp_reduce_adam_bcast_peer(
        C.c_void_p(int(peer_bases_dev)), int(grad_off), int(param_off), int(bf16_off), _ext.ptr(exp_avg),
        _ext.ptr(exp_avg_sq), int(n), float(lr), float(beta1), float(beta2), float(eps), float(weight_decay), int(step),
        float(grad_scale), int(rank), int(world), C.c_void_p(int(flag_ptrs_dev)), int(channel), int(bool(coresident)),
        sp))


def dp_exchange(grad_multicast_ptr, offset, n, rank, world, flag_ptrs_dev, channel, stream=None, coresident=False):
    """In-switch sum over ranks of floats [offset, offset + n) of the symmetric flat gradient buffer
    (lirec_dp_exchange: barrier, multimem reduce + broadcast of this rank's shard, barrier) on `stream`."""
    L = _ext.lib()
    sp = _ext.stream_ptr() if stream is None else C.c_void_p(stream.cuda_stream)
    _ext.check(L.lirec_dp_exchange(C.c_void_p(int(grad_multicast_ptr)), int(offset), int(n), int(rank), int(world),
                                   C.c_void_p(int(flag_ptrs_dev)), int(channel), int(bool(coresident)), sp))
