"""lirec_gemm_grouped element by element against an fp64 statement of its C ABI (include/lirec_b200.h).

`reference(spec, operands, out_before)` restates the header's semantics: the passes (exactly k_len long, at
their offsets, in each operand's layout, 0 outside a view), alpha, the bias (gated by row_flag, split-K slice 0
only), the activation, the post op (in terms of the stored aux) and the output kind, and returns the expected
value of every output element, which buffer elements the call may write and a per-element error bound:

    F32           |got - ref| <= 2^-16 P + 2^-23 (|bias| + |old value|)      P[m,n] = |alpha| sum_k |a_mk b_nk|
    hi/lo split   + 2^-17 |ref|
    tanh          + 2^-20 (tanh_fast)
    dropout / DRELU / DTANH: the bound is carried through the factor plus its fp32 rounding; a dropped or
    gated-off element must be exactly 0.

2^-16 P is far above fp32 accumulation error at these K and far below a missing or doubled k-block, tile or
pass.  Every output buffer is pre-filled with a sentinel that must survive outside the footprint.  Each GPU
launch also pins the kernel that ran by its tile count: ceil(M/256) ceil(N/bn) S (CTA-pair kernel, bn = 256 if
N > 128 else 128) or ceil(M/128) ceil(N/128) S (single-CTA kernel); a large "ballast" problem moves a launch
onto the pair kernel, a small "marker" problem makes the two counts differ on a single-CTA launch.
"""
from dataclasses import dataclass

import numpy as np
import pytest
import torch

from lirec_b200._ext import (ACT_NONE, ACT_RELU, ACT_TANH, OUT_F32, OUT_SPLIT, OUT_SPLIT_T, POST_DRELU,
                             POST_DROPOUT, POST_DTANH, POST_NONE, POST_SIGN_MASK)

BK = 64
F64 = torch.float64


# ------------------------------------------------------------------------------------------------------------
# fp64 reference of the header
# ------------------------------------------------------------------------------------------------------------
def split_k_slices(kb, split_k):
    """Slices a split-K problem writes: c = ceil(kb / min(split_k, kb)) k-blocks each, S = ceil(kb / c)."""
    split = min(split_k, kb)
    if split <= 1:
        return 1
    c = -(-kb // split)
    return -(-kb // c)


def _window(t, r0, nr, c0, nc):
    """fp64 [nr, nc] block of the 2-D view t from (r0, c0); elements outside the view are 0."""
    w = torch.zeros(nr, nc, dtype=F64, device=t.device)
    rs, re, cs, ce = max(r0, 0), min(r0 + nr, t.shape[0]), max(c0, 0), min(c0 + nc, t.shape[1])
    if rs < re and cs < ce:
        w[rs - r0:re - r0, cs - c0:ce - c0] = t[rs:re, cs:ce].double()
    return w


def _pass_matrix(t, mn_major, mn_off, k_off, mn, k_len):
    """[mn, k_len] operand of one pass: K-major view rows = MN, cols = K; MN-major view rows = K, cols = MN."""
    if mn_major:
        return _window(t, k_off, k_len, mn_off, mn).t()
    return _window(t, mn_off, mn, k_off, k_len)


@dataclass
class Expect:
    value: torch.Tensor      # [M, N] fp64: the output element (split-K: the sum of the slices; split: hi + lo)
    bound: torch.Tensor      # [M, N] fp64: allowed |got - value|
    index: torch.Tensor      # [M, N] int64: flat buffer index of the element (slice 0 / hi part)
    offsets: list            # flat offsets added to `index` for each stored part; got = sum of those elements
    written: torch.Tensor    # bool over the flat output buffer: elements the call may write
    sign: torch.Tensor = None       # SIGN_MASK: expected bit [v > 0]
    sign_free: torch.Tensor = None  # SIGN_MASK: bits whose pre-activation lies within the bound of 0


def reference(spec, operands, out_before):
    """spec: the arguments of ops.gemm_problem with tensors named (keys of `operands`) and the output given as
    an element offset `out_off` into the flat buffer `out_before`."""
    s = dict(SPEC_DEFAULTS, **spec)
    M, N = s["M"], s["N"]
    dev = out_before.device
    value = torch.zeros(M, N, dtype=F64, device=dev)
    P = torch.zeros(M, N, dtype=F64, device=dev)
    kb = 0
    for (a, amn, ak, b, bmn, bk, k_len) in s["passes"]:
        A = _pass_matrix(operands[a], s["a_mn_major"], amn, ak, M, k_len)
        B = _pass_matrix(operands[b], s["b_mn_major"], bmn, bk, N, k_len)
        value += A @ B.t()
        P += A.abs() @ B.abs().t()
        kb = max(kb, -(-k_len // BK))
    alpha = s["alpha"]
    value *= alpha
    bound = 2.0 ** -16 * abs(alpha) * P
    rows = torch.arange(M, device=dev)
    if s["bias"] is not None:
        bias = operands[s["bias"]][:N].double()
        gate = torch.ones(M, dtype=F64, device=dev)
        if s["row_flag"] is not None:
            gate = (operands[s["row_flag"]][:M] != 0).double()
        value += gate[:, None] * bias[None, :]
        bound += 2.0 ** -23 * gate[:, None] * bias.abs()[None, :]
    pre, pre_bound = value.clone(), bound.clone()
    if s["act"] == ACT_RELU:
        value = value.clamp_min(0)          # 1-Lipschitz: the bound carries over
    elif s["act"] == ACT_TANH:
        value = torch.tanh(value)
        bound = bound + 2.0 ** -20
    p, seed, stream_id, col_off = s["drop"]
    keep, ks = torch.ones(M, N, dtype=torch.bool, device=dev), 1.0
    if p > 0:
        from oracle import dropout as od
        keep = torch.from_numpy(od.keep_mask(seed, stream_id, np.arange(M), col_off + np.arange(N), p)).to(dev)
        ks = 1.0 / (1.0 - p)
    post = s["post"]
    sign = sign_free = None
    zero = torch.zeros((), dtype=F64, device=dev)
    if post == POST_DROPOUT:
        value = torch.where(keep, value * ks, zero)
        bound = torch.where(keep, bound * ks + 2.0 ** -22 * value.abs(), zero)
    elif post in (POST_DRELU, POST_DTANH):
        aux = operands[s["aux"]]
        hi = aux[:M, s["aux_col_off"]:s["aux_col_off"] + N].double()
        if post == POST_DRELU:
            on = hi > 0
            ps = s["post_scale"]
            value = torch.where(on, value * ps, zero)
            bound = torch.where(on, bound * abs(ps) + 2.0 ** -23 * value.abs(), zero)
        else:
            lo_c = s["aux_col_off"] + s["aux_lo_off"]
            t = (hi + aux[:M, lo_c:lo_c + N].double()) * (1.0 - p)
            f = 1.0 - t * t
            vin = value
            value = torch.where(keep, vin * ks * f, zero)
            bound = torch.where(keep, bound * ks * f.abs() + 2.0 ** -20 * vin.abs() * ks * (1 + t * t), zero)
    elif post == POST_SIGN_MASK:
        signed, signed_bound = (torch.tanh(pre), pre_bound + 2.0 ** -20) if s["act"] == ACT_TANH else (pre, pre_bound)
        sign, sign_free = signed > 0, signed.abs() <= signed_bound

    kind, off = s["out_kind"], s["out_off"]
    ld_m, ld_n, c_off, lo_off = s["out_ld_m"], s["out_ld_n"], s["out_col_off"], s["out_lo_off"]
    cols = torch.arange(N, device=dev)
    if kind == OUT_F32:
        index = off + rows[:, None] * ld_m + cols[None, :] * ld_n
        nsl = split_k_slices(kb, s["split_k"]) if s["split_k"] > 1 else 1
        offsets = [q * s["split_stride"] for q in range(nsl)]
        if s["accumulate"]:
            old = out_before.double()[index] if M * N else value
            value = value + old
            bound = bound + 2.0 ** -23 * old.abs()
    elif kind == OUT_SPLIT:
        index = off + rows[:, None] * ld_m + c_off + cols[None, :]
        offsets = [0, lo_off]
        bound = bound + 2.0 ** -17 * value.abs()
    else:
        index = off + (c_off + cols[None, :]) * ld_m + rows[:, None]
        offsets = [0, lo_off * ld_m]
        bound = bound + 2.0 ** -17 * value.abs()
    written = torch.zeros(out_before.numel(), dtype=torch.bool, device=dev)
    for o in offsets:
        if M * N:
            assert int((index + o).min()) >= 0 and int((index + o).max()) < out_before.numel(), "output outside buffer"
            written[(index + o).flatten()] = True
    return Expect(value, bound, index, offsets, written, sign, sign_free)


SPEC_DEFAULTS = dict(a_mn_major=False, b_mn_major=False, alpha=1.0, bias=None, row_flag=None, act=ACT_NONE,
                     post=POST_NONE, post_scale=1.0, drop=(0.0, 0, 0, 0), aux=None, aux_col_off=0, aux_lo_off=0,
                     out_kind=OUT_F32, out_off=0, out_ld_m=0, out_ld_n=1, out_col_off=0, out_lo_off=0,
                     accumulate=False, split_k=0, split_stride=0)


def gathered(exp, buf):
    """The output elements as the kernel stored them, summed over their parts in fp64."""
    flat = buf.double()
    return sum(flat[exp.index + o] for o in exp.offsets)


# ------------------------------------------------------------------------------------------------------------
# The reference itself (CPU, no GPU needed)
# ------------------------------------------------------------------------------------------------------------
def _bf(g, *shape, scale=1.0):
    return (torch.randn(*shape, generator=g) * scale).to(torch.bfloat16)


def test_reference_matches_addmm():
    g = torch.Generator().manual_seed(1)
    M, N, K = 7, 5, 130
    a, b, bias = _bf(g, M, K + 9), _bf(g, N, K), torch.randn(N, generator=g)
    buf = torch.full((M * 6,), float("nan"))
    spec = dict(M=M, N=N, passes=[("a", 0, 0, "b", 0, 0, K)], alpha=0.5, bias="bias", out_ld_m=6)
    exp = reference(spec, dict(a=a, b=b, bias=bias), buf)
    ref = torch.addmm(bias.double(), a[:, :K].double(), b.double().t(), alpha=0.5)   # the 9 extra columns excluded
    assert torch.allclose(exp.value, ref, rtol=1e-13, atol=1e-13)
    assert exp.written.view(M, 6)[:, :N].all() and not exp.written.view(M, 6)[:, N:].any()
    P = 0.5 * a[:, :K].double().abs() @ b.double().abs().t()
    assert torch.allclose(exp.bound, 2.0 ** -16 * P + 2.0 ** -23 * bias.double().abs(), rtol=1e-13)


def test_reference_mn_major_offsets_and_view_edge():
    g = torch.Generator().manual_seed(2)
    a = _bf(g, 100, 20)                        # MN-major A: rows = K, cols = M
    b = _bf(g, 4, 90)                          # K-major B
    spec = dict(M=3, N=2, a_mn_major=True, passes=[("a", 5, 10, "b", 1, 7, 85)], out_ld_m=2)
    exp = reference(spec, dict(a=a, b=b), torch.zeros(6))
    kk = torch.arange(85)
    ref = torch.zeros(3, 2, dtype=F64)
    for m in range(3):
        for n in range(2):
            bv = torch.where(7 + kk < 90, b[1 + n, (7 + kk).clamp_max(89)].double(), torch.zeros(85, dtype=F64))
            ref[m, n] = (a[10 + kk, 5 + m].double() * bv).sum()
    assert torch.allclose(exp.value, ref, rtol=1e-13)


def test_reference_split_k_footprint():
    """kb = 9, split_k = 4: three slices of three k-blocks; slice 3 is not written; the bias is counted once."""
    g = torch.Generator().manual_seed(3)
    M, N, K = 3, 2, 9 * 64 - 5
    a, b, bias = _bf(g, M, K), _bf(g, N, K), torch.randn(N, generator=g)
    flag = torch.tensor([1, 0, 1], dtype=torch.int32)
    stride = 11
    buf = torch.zeros(4 * stride)
    spec = dict(M=M, N=N, passes=[("a", 0, 0, "b", 0, 0, K)], bias="bias", row_flag="flag", out_ld_m=1, out_ld_n=3,
                split_k=4, split_stride=stride)
    exp = reference(spec, dict(a=a, b=b, bias=bias, flag=flag), buf)
    assert split_k_slices(9, 4) == 3 and split_k_slices(10, 7) == 5 and split_k_slices(2, 9) == 2
    assert exp.offsets == [0, 11, 22]
    want = torch.zeros(4 * stride, dtype=torch.bool)
    for sl in range(3):
        for m in range(M):
            for n in range(N):
                want[sl * stride + m + 3 * n] = True
    assert torch.equal(exp.written, want)
    ref = a.double() @ b.double().t() + flag.double()[:, None] * bias.double()
    assert torch.allclose(exp.value, ref, rtol=1e-13)


def test_reference_split_and_transposed_split_stores():
    g = torch.Generator().manual_seed(4)
    a, b = _bf(g, 2, 64), _bf(g, 3, 64)
    ops_ = dict(a=a, b=b)
    base = dict(M=2, N=3, passes=[("a", 0, 0, "b", 0, 0, 64)])
    # SPLIT: hi at out[off + m*ld + col_off + n], lo at + lo_off
    exp = reference(dict(base, out_kind=OUT_SPLIT, out_off=1, out_ld_m=10, out_col_off=2, out_lo_off=4),
                    ops_, torch.zeros(21, dtype=torch.bfloat16))
    assert exp.index.tolist() == [[3, 4, 5], [13, 14, 15]] and exp.offsets == [0, 4]
    # SPLIT_T: hi at out[off + (col_off + n)*ld + m], lo at + lo_off*ld
    exp = reference(dict(base, out_kind=OUT_SPLIT_T, out_ld_m=5, out_col_off=1, out_lo_off=4),
                    ops_, torch.zeros(40, dtype=torch.bfloat16))
    assert exp.index.tolist() == [[5, 10, 15], [6, 11, 16]] and exp.offsets == [0, 20]
    assert int(exp.written.sum()) == 12
    ref = a.double() @ b.double().t()
    assert torch.allclose(exp.value, ref, rtol=1e-13)
    assert torch.allclose(exp.bound, 2.0 ** -16 * (a.double().abs() @ b.double().abs().t()) + 2.0 ** -17 * ref.abs())
    # the stored parts add up through gathered()
    buf = torch.zeros(40, dtype=F64)
    buf[exp.index] = 1.5
    buf[exp.index + 20] = 0.25
    assert torch.equal(gathered(exp, buf), torch.full((2, 3), 1.75, dtype=F64))


def test_reference_post_ops():
    """DTANH / DRELU from the stored aux, as the header writes them; dropped elements are exact zeros."""
    from oracle import dropout as od
    g = torch.Generator().manual_seed(5)
    M, N, p = 4, 6, 0.4
    a, b = _bf(g, M, 64), _bf(g, N, 64)
    aux = _bf(g, M, 16, scale=0.5)
    ops_ = dict(a=a, b=b, aux=aux)
    base = dict(M=M, N=N, passes=[("a", 0, 0, "b", 0, 0, 64)], out_ld_m=N, aux="aux", aux_col_off=2,
                drop=(p, 9, 3, 4))
    acc = a.double() @ b.double().t()
    keep = torch.from_numpy(od.keep_mask(9, 3, np.arange(M), 4 + np.arange(N), p))
    exp = reference(dict(base, post=POST_DTANH, aux_lo_off=7), ops_, torch.zeros(M * N))
    t = (aux[:, 2:2 + N].double() + aux[:, 9:9 + N].double()) * (1 - p)
    assert torch.allclose(exp.value, torch.where(keep, acc / (1 - p) * (1 - t * t), torch.zeros(())), rtol=1e-13)
    assert bool((exp.bound[~keep] == 0).all())
    exp = reference(dict(base, post=POST_DRELU, post_scale=2.5), ops_, torch.zeros(M * N))
    assert torch.allclose(exp.value, torch.where(aux[:, 2:2 + N].double() > 0, 2.5 * acc, torch.zeros(())), rtol=1e-13)


# ------------------------------------------------------------------------------------------------------------
# Case builders (operands from fixed seeds; every buffer surrounds its view with nonzero data or NaN)
# ------------------------------------------------------------------------------------------------------------
def _ru(x, m):
    return -(-x // m) * m


class Builder:
    """Makes the operands, the spec and the pre-filled output buffer of one problem."""

    def __init__(self, seed, dev="cuda"):
        self.g = torch.Generator(device=dev).manual_seed(seed)
        self.dev = dev

    def randn(self, *shape, scale=1.0):
        return torch.randn(*shape, generator=self.g, device=self.dev) * scale

    def operand(self, mn, k_total, mn_major, mn_off, k_off, scale):
        assert (mn_off if mn_major else k_off) % 8 == 0, "TMA box starts along the columns are 16-byte aligned"
        """bf16 tensor holding [mn, k_total] at (mn_off, k_off) in the given layout, with nonzero data all
        around it (past the pass's k range too: a pass must read exactly k_len)."""
        if mn_major:
            t = self.randn(k_off + k_total + 37, _ru(mn_off + mn + 24, 8), scale=scale)
        else:
            t = self.randn(mn_off + mn + 3, _ru(k_off + k_total + 40, 8), scale=scale)
        return t.to(torch.bfloat16)


def _place(off, mn_major):
    """(mn_off, k_off) with the offset along the operand's columns rounded up to a multiple of 8 elements
    (k_off K-major, mn_off MN-major): the header's alignment rule; the other one is used as given."""
    mn_off, k_off = off
    return (_ru(mn_off, 8), k_off) if mn_major else (mn_off, _ru(k_off, 8))


def make_case(name, M, N, K, seed, *, a_mn=False, b_mn=False, passes="one", a_off=(0, 0), b_off=(0, 0), alpha=1.0,
              bias=None, row_flag=False, act=ACT_NONE, post=POST_NONE, post_scale=1.0, drop_p=0.0, aux_vec=True,
              out="f32", out_vec=True, accumulate=False, split_k=0, stride_pad=0, dev="cuda"):
    """One problem of the matrix.  passes: "one" | "hilo_a" (A = [hi | lo], two passes over one B) | "wgrad3"
    (x_hi dy_hi, x_lo dy_hi, x_hi dy_lo) | "two_ranges" (two passes over different k ranges and lengths).
    a_off / b_off: (mn_off, k_off) of the first pass inside its operand (see _place)."""
    bld = Builder(seed, dev)
    scale = max(K, 1) ** -0.25                       # pre-activations ~ N(0, 1): tanh not saturated
    opnds, spec = {}, dict(M=M, N=N, a_mn_major=a_mn, b_mn_major=b_mn, alpha=alpha, act=act, post=post,
                           post_scale=post_scale, accumulate=accumulate, split_k=split_k)
    Mv, Nv = max(M, 1), max(N, 1)
    (amn, ak), (bmn, bk) = _place(a_off, a_mn), _place(b_off, b_mn)
    if passes == "one":
        opnds["a"] = bld.operand(Mv, K, a_mn, amn, ak, scale)
        opnds["b"] = bld.operand(Nv, K, b_mn, bmn, bk, scale)
        spec["passes"] = [("a", amn, ak, "b", bmn, bk, K)]
    elif passes == "hilo_a":                       # hi at k_off, lo K + 5 further along K
        opnds["a"] = bld.operand(Mv, 2 * K + 5, a_mn, amn, ak, scale)
        opnds["b"] = bld.operand(Nv, K, b_mn, bmn, bk, scale)
        spec["passes"] = [("a", amn, ak, "b", bmn, bk, K), ("a", amn, ak + _ru(K, 8) + 8, "b", bmn, bk, K)]
    elif passes == "wgrad3":
        opnds["a"] = bld.operand(Mv, 2 * K + 5, a_mn, amn, ak, scale)
        opnds["b"] = bld.operand(Nv, 2 * K + 5, b_mn, bmn, bk, scale)
        ka, kb2 = ak + _ru(K, 8) + 8, bk + _ru(K, 8) + 8
        spec["passes"] = [("a", amn, ak, "b", bmn, bk, K), ("a", amn, ka, "b", bmn, bk, K),
                          ("a", amn, ak, "b", bmn, kb2, K)]
    elif passes == "two_ranges":                    # lengths K and K + 92, separate operands, odd offsets
        K2 = K + 92
        opnds["a"] = bld.operand(Mv, K, a_mn, amn, ak, scale)
        opnds["b"] = bld.operand(Nv, K, b_mn, bmn, bk, scale)
        (amn2, ak2), (bmn2, bk2) = _place((3, 67), a_mn), _place((1, 5), b_mn)
        opnds["a2"] = bld.operand(Mv, K2, a_mn, amn2, ak2, scale)
        opnds["b2"] = bld.operand(Nv, K2, b_mn, bmn2, bk2, scale)
        spec["passes"] = [("a", amn, ak, "b", bmn, bk, K), ("a2", amn2, ak2, "b2", bmn2, bk2, K2)]
    elif passes == "four_groups":                   # four k-block counts: more than MAX_GROUPS (3) groups
        for i in range(4):
            opnds["a%d" % i] = bld.operand(Mv, 64 * (i + 1), a_mn, 0, 0, scale)
            opnds["b%d" % i] = bld.operand(Nv, 64 * (i + 1), b_mn, 0, 0, scale)
        spec["passes"] = [("a%d" % i, 0, 0, "b%d" % i, 0, 0, 64 * (i + 1)) for i in range(4)]
    else:
        raise ValueError(passes)
    if bias is not None:
        bt = bld.randn(Nv + 1)
        opnds["bias"] = bt[:Nv] if bias == "aligned" else bt[1:]      # a view offset by one float
        spec["bias"] = "bias"
    if row_flag:
        opnds["flag"] = (torch.arange(Mv, device=dev) % 3 != 1).int()
        spec["row_flag"] = "flag"
    if drop_p > 0 or post == POST_DROPOUT:
        spec["drop"] = (drop_p, 1000 + seed, 3, 6)
    if post in (POST_DRELU, POST_DTANH):
        # the forward's stored output: [hi | gap | lo] bf16 with NaN past N (a partial chunk reads no further)
        col, lo = (8, _ru(Nv, 8) + 8) if aux_vec else (3, Nv + 5)
        ld = _ru(col + lo + Nv + 40, 8) if aux_vec else col + lo + Nv + 41
        auxt = torch.full((Mv, ld), float("nan"), device=dev)
        x = torch.tanh(bld.randn(Mv, Nv) * 1.5)
        x[bld.randn(Mv, Nv) > 0.8] = 0.0                             # dropped / ReLU-gated forward elements
        if drop_p > 0:
            x = x / (1 - drop_p)
        hi = x.to(torch.bfloat16)
        auxt[:, col:col + Nv] = hi.float()
        auxt[:, col + lo:col + lo + Nv] = (x - hi.float()).to(torch.bfloat16).float()
        opnds["aux"] = auxt.to(torch.bfloat16)
        spec.update(aux="aux", aux_col_off=col, aux_lo_off=lo)
    if post == POST_SIGN_MASK:
        opnds["aux"] = torch.full((Mv + 3, N // 32 + 2), -1, dtype=torch.int32, device=dev)
        spec["aux"] = "aux"
    # output buffer
    if out in ("f32", "f32_t"):
        off = 0 if out_vec else 1
        ld = (_ru(Nv, 4) + 4 if out_vec else Nv + 3) if out == "f32" else M + 5
        if out == "f32":
            spec.update(out_ld_m=ld, out_ld_n=1)
            extent = (Mv - 1) * ld + Nv
        else:
            spec.update(out_ld_m=1, out_ld_n=ld)
            extent = (Nv - 1) * ld + Mv
        nsl = max(split_k, 1)
        stride = _ru(extent + 3, 4) + stride_pad
        spec.update(out_kind=OUT_F32, out_off=off, split_stride=stride if split_k else 0)
        size = off + (nsl - 1) * stride + extent + 13
        buf = torch.full((size,), 0.75 if accumulate else float("nan"), device=dev)
    elif out == "split":
        col, lo = (8, _ru(Nv, 8) + 16) if out_vec else (3, Nv + 5)
        ld = _ru(col + lo + Nv + 8, 8) if out_vec else col + lo + Nv + 9
        spec.update(out_kind=OUT_SPLIT, out_ld_m=ld, out_col_off=col, out_lo_off=lo)
        buf = torch.full((Mv * ld + 16,), float("nan"), device=dev, dtype=torch.bfloat16)
    elif out == "split_t":
        ld = _ru(M + 3, 8) + 8 if out_vec else M + 3
        col, lo = 4, Nv + 9
        spec.update(out_kind=OUT_SPLIT_T, out_ld_m=ld, out_col_off=col, out_lo_off=lo)
        buf = torch.full(((col + lo + Nv + 2) * ld,), float("nan"), device=dev, dtype=torch.bfloat16)
    else:
        raise ValueError(out)
    return name, spec, opnds, buf


# ------------------------------------------------------------------------------------------------------------
# Launch, pin the kernel, check every element
# ------------------------------------------------------------------------------------------------------------
MARGIN = {}      # largest error / bound per output kind, reported at the end of the module


@pytest.fixture(scope="module", autouse=True)
def _report_margins(request):
    yield
    if MARGIN:
        tr = request.config.pluginmanager.get_plugin("terminalreporter")
        line = "GEMM contract: largest error / bound per output kind: " + ", ".join(
            "%s %.3g" % kv for kv in sorted(MARGIN.items()))
        if tr is not None:
            tr.write_line(line)
        print(line)


def _kb(spec):
    return max(-(-p[6] // BK) for p in spec["passes"])


def _tiles(spec, kernel, slices_rule):
    M, N = spec["M"], spec["N"]
    if M <= 0 or N <= 0:
        return 0
    sk, kb = spec.get("split_k", 0), _kb(spec)
    S = (split_k_slices(kb, sk) if sk > 1 else 1) if slices_rule == "written" else max(1, min(sk, kb))
    if kernel == "pair":
        bn = 256 if N > 128 else 128
        return -(-M // 256) * -(-N // bn) * S
    return -(-M // 128) * -(-N // 128) * S


def _fits_single(specs):
    """The header's launch rule: the single-CTA kernel when the launch fills under 60 % of the 74 pair
    clusters and fits one wave of 128 x 128 tiles on the 148 SMs (tiles counted with min(split_k, kb))."""
    pair = sum(_tiles(s, "pair", "bound") for s in specs)
    single = sum(_tiles(s, "single", "bound") for s in specs)
    return pair * 10 <= 74 * 6 and single <= 148


def _ballast(seed):
    return make_case("ballast", 2048, 1536, 64, seed)


def _marker(seed):
    return make_case("marker", 200, 200, 64, seed)


def to_problem(spec, opnds, buf):
    from lirec_b200 import _ext, ops
    s = dict(SPEC_DEFAULTS, **spec)
    passes = [(_ext.operand(opnds[a]), amn, ak, _ext.operand(opnds[b]), bmn, bk, kl)
              for (a, amn, ak, b, bmn, bk, kl) in s["passes"]]
    get = lambda k: opnds[s[k]] if s[k] is not None else None   # noqa: E731
    return ops.gemm_problem(s["M"], s["N"], passes, a_mn_major=s["a_mn_major"], b_mn_major=s["b_mn_major"],
                            alpha=s["alpha"], bias=get("bias"), row_flag=get("row_flag"), act=s["act"],
                            post=s["post"], post_scale=s["post_scale"], drop=ops.dropout_desc(*s["drop"]),
                            aux=get("aux"), aux_col_off=s["aux_col_off"], aux_lo_off=s["aux_lo_off"],
                            out=buf[s["out_off"]:], out_kind=s["out_kind"], out_ld_m=s["out_ld_m"],
                            out_ld_n=s["out_ld_n"], out_col_off=s["out_col_off"], out_lo_off=s["out_lo_off"],
                            accumulate=s["accumulate"], split_k=s["split_k"], split_stride=s["split_stride"])


def _kind(spec):
    s = dict(SPEC_DEFAULTS, **spec)
    k = {OUT_F32: "f32", OUT_SPLIT: "split", OUT_SPLIT_T: "split_t"}[s["out_kind"]]
    if s["out_kind"] == OUT_F32 and s["out_ld_n"] != 1:
        k += "_transposed"
    if s["split_k"] > 1:
        k += "_splitk"
    if s["act"] == ACT_TANH or s["post"] != POST_NONE:
        k += "_post"
    return k


def check_case(case, before, exp, aux_before=None):
    name, spec, opnds, buf = case
    M, N = spec["M"], spec["N"]
    bits = lambda t: t.view(torch.int16 if t.element_size() == 2 else torch.int32)   # noqa: E731
    untouched = ~exp.written
    assert torch.equal(bits(buf)[untouched], bits(before)[untouched]), \
        "%s: %d elements written outside the output" % (name, int((bits(buf) != bits(before))[untouched].sum()))
    if M * N == 0:
        return
    got = gathered(exp, buf)
    err = (got - exp.value).abs()
    bad = ~(err <= exp.bound)                     # NaN fails too
    if bool(bad.any()):
        m, n = [int(i) for i in torch.nonzero(bad)[0]]
        raise AssertionError("%s: %d of %d elements out of bound; first (%d, %d): got %r want %r bound %.3g" % (
            name, int(bad.sum()), M * N, m, n, float(got[m, n]), float(exp.value[m, n]), float(exp.bound[m, n])))
    pos = exp.bound > 0
    if bool(pos.any()):
        k = _kind(spec)
        MARGIN[k] = max(MARGIN.get(k, 0.0), float((err[pos] / exp.bound[pos]).max()))
    if exp.sign is not None:
        words = opnds["aux"]
        nw = N // 32
        got_bits = ((words[:M, :nw].long() & 0xFFFFFFFF)[:, :, None] >> torch.arange(32, device=words.device)) & 1
        got_bits = got_bits.reshape(M, N).bool()
        wrong = (got_bits != exp.sign) & ~exp.sign_free
        assert not bool(wrong.any()), "%s: %d sign-mask bits wrong" % (name, int(wrong.sum()))
        keep = torch.ones_like(words, dtype=torch.bool)
        keep[:M, :nw] = False
        assert bool((words[keep] == -1).all()), "%s: sign-mask words written outside [M, N/32]" % name


def run_launch(cases, kernel):
    """Run `cases` as ONE grouped launch on `kernel` ("single" | "pair"), pin the kernel by its tile count and
    check every problem against the reference."""
    from lirec_b200 import _ext, ops
    specs = [c[1] for c in cases]
    assert _fits_single(specs) == (kernel == "single"), "launch would not run on the %s kernel" % kernel
    want = {k: sum(_tiles(s, k, "written") for s in specs) for k in ("pair", "single")}
    assert want["pair"] != want["single"], "tile counts do not tell the kernels apart"
    befores = [c[3].clone() for c in cases]
    exps = [reference(c[1], c[2], c[3]) for c in cases]
    probs = [to_problem(c[1], c[2], c[3]) for c in cases]
    _ext.profile_begin()
    ops.gemm_grouped(probs)
    recs = _ext.profile_end()
    torch.cuda.synchronize()
    if want["pair"] + want["single"] > 0:
        assert len(recs) == 1 and recs[0][2] == want[kernel], (recs, want)
    for c, b, e in zip(cases, befores, exps):
        check_case(c, b, e)


def _pack(cases, kernel, seed):
    """Cases -> launches: on the pair kernel all cases plus a ballast problem; on the single-CTA kernel as many
    as keep the launch small, plus a marker problem whose tile counts differ between the kernels."""
    if kernel == "pair":
        out = []
        for i in range(0, len(cases), 31):
            out.append(cases[i:i + 31] + [_ballast(seed + i)])
        return out
    launches, cur = [], []
    for c in cases:
        trial = cur + [c]
        if cur and not _fits_single([x[1] for x in trial + [_marker(0)]]):
            launches.append(cur + [_marker(seed + len(launches))])
            trial = [c]
        cur = trial
    launches.append(cur + [_marker(seed + len(launches))])
    return launches


def run_cases(cases, kernel, seed=0):
    for launch in _pack(cases, kernel, seed):
        run_launch(launch, kernel)


# ------------------------------------------------------------------------------------------------------------
# The matrix
# ------------------------------------------------------------------------------------------------------------
# (M, N, K, a_off, b_off): M in {1, 127, 129, 255, 257, 3000}, N in {8, 31, 33, 96, 128, 129, 200, 257},
# K in {64, 100, 192, 4096}; offsets (mn_off, k_off): odd along an operand's rows, multiples of 8 but not of 64
# along its columns
SHAPES = [
    (1, 8, 64, (0, 0), (0, 0)),
    (127, 31, 100, (5, 37), (0, 0)),
    (129, 33, 192, (0, 0), (3, 70)),
    (255, 96, 100, (64, 3), (8, 1)),
    (257, 128, 64, (0, 0), (0, 0)),
    (3000, 129, 192, (7, 0), (0, 5)),
    (129, 200, 4096, (0, 64), (2, 0)),
    (257, 257, 100, (1, 1), (1, 1)),
    (255, 129, 64, (0, 0), (0, 0)),
    (127, 200, 320, (0, 9), (0, 0)),
]
KERNELS = ["single", "pair"]
MAJOR = [(False, False), (False, True), (True, False), (True, True)]


@pytest.fixture()
def gpu():
    from lirec_b200 import _ext
    _ext.require_device()


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("a_mn,b_mn", MAJOR)
def test_operand_forms_and_edge_shapes(gpu, a_mn, b_mn, kernel):
    """All four (A, B) majorness pairs over the edge shapes, one pass: even and odd k-block counts (the lone
    pass's two-k-block stages and its one-block tail group), k_len % 64 != 0 with nonzero data past it."""
    cases = [make_case("%dx%dx%d" % (M, N, K), M, N, K, 10 * i + 1, a_mn=a_mn, b_mn=b_mn, a_off=ao, b_off=bo)
             for i, (M, N, K, ao, bo) in enumerate(SHAPES)]
    run_cases(cases, kernel, seed=7)


# name -> (kwargs, (M, N, K) shapes).  Every form runs on both kernels; N <= 128 and N > 128 give the pair
# kernel's two tile widths.
FORMS = {
    "hilo_a": (dict(passes="hilo_a"), [(255, 96, 192), (129, 200, 100)]),
    "hilo_a_mn": (dict(passes="hilo_a", a_mn=True, b_off=(3, 0)), [(127, 33, 100), (300, 257, 320)]),
    "wgrad3": (dict(passes="wgrad3", a_mn=True), [(257, 96, 100), (200, 200, 192)]),
    "wgrad3_kmajor": (dict(passes="wgrad3", a_off=(1, 3)), [(129, 31, 64), (255, 129, 4096)]),
    "two_ranges": (dict(passes="two_ranges", a_off=(0, 5)), [(200, 96, 100), (129, 257, 64)]),
    "two_ranges_mn": (dict(passes="two_ranges", a_mn=True, b_mn=True), [(127, 128, 100), (257, 200, 192)]),
    "klen_inside_operand": (dict(a_off=(0, 11), b_off=(0, 29)), [(200, 96, 37), (129, 200, 100), (255, 64, 1)]),
    "klen_inside_operand_mn": (dict(a_mn=True, b_mn=True, a_off=(0, 11), b_off=(0, 29)),
                               [(200, 96, 37), (129, 200, 100)]),
    "alpha": (dict(alpha=-0.37), [(129, 33, 192), (255, 257, 100)]),
    "bias": (dict(bias="aligned"), [(200, 96, 64), (129, 200, 100)]),
    "bias_misaligned": (dict(bias="misaligned"), [(200, 96, 64), (129, 200, 100)]),
    "bias_row_flag": (dict(bias="aligned", row_flag=True, alpha=2.0), [(255, 33, 192), (257, 257, 64)]),
    "relu": (dict(bias="aligned", act=ACT_RELU), [(200, 31, 100), (129, 200, 64)]),
    "tanh": (dict(bias="aligned", act=ACT_TANH, out="split"), [(200, 33, 100), (129, 200, 192)]),
    "dropout_p0": (dict(bias="aligned", act=ACT_RELU, post=POST_DROPOUT, drop_p=0.0, out="split"),
                   [(200, 96, 64), (129, 257, 100)]),
    "dropout": (dict(bias="aligned", act=ACT_TANH, post=POST_DROPOUT, drop_p=0.3, out="split"),
                [(200, 33, 64), (129, 200, 100)]),
    "dropout_f32": (dict(act=ACT_RELU, post=POST_DROPOUT, drop_p=0.5), [(127, 96, 64), (255, 129, 192)]),
    "drelu": (dict(post=POST_DRELU, post_scale=1 / 0.7, out="split_t"), [(200, 96, 100), (129, 200, 64)]),
    "drelu_partial_nan": (dict(post=POST_DRELU, post_scale=1.5, out="split_t"), [(200, 33, 100), (129, 201, 64)]),
    "drelu_aux_scalar": (dict(post=POST_DRELU, post_scale=2.0, aux_vec=False), [(127, 96, 64), (129, 200, 100)]),
    "dtanh": (dict(post=POST_DTANH, out="split_t"), [(200, 96, 64), (129, 200, 192)]),
    "dtanh_dropout": (dict(post=POST_DTANH, drop_p=0.3, out="split_t"), [(200, 31, 100), (129, 257, 64)]),
    "dtanh_aux_scalar": (dict(post=POST_DTANH, drop_p=0.2, aux_vec=False, out="split"),
                         [(127, 64, 64), (129, 200, 100)]),
    "sign_mask": (dict(bias="aligned", act=ACT_RELU, post=POST_SIGN_MASK), [(255, 96, 100), (129, 256, 64)]),
    "f32_scalar_ptr": (dict(out_vec=False), [(200, 96, 64), (129, 200, 100)]),
    "f32_transposed": (dict(out="f32_t", bias="aligned"), [(200, 96, 100), (129, 257, 64)]),
    "f32_accumulate": (dict(accumulate=True, bias="aligned"), [(200, 96, 64), (129, 256, 192)]),
    "f32_accumulate_scalar": (dict(accumulate=True, out_vec=False), [(200, 33, 64), (129, 200, 100)]),
    "split_staged": (dict(out="split", bias="aligned"), [(200, 96, 64), (129, 256, 100)]),
    "split_direct": (dict(out="split", out_vec=False), [(200, 33, 64), (129, 200, 100)]),
    "split_t_vec": (dict(out="split_t", a_mn=True), [(200, 96, 64), (253, 200, 100)]),
    "split_t_scalar": (dict(out="split_t", out_vec=False, a_mn=True), [(200, 33, 64), (129, 257, 100)]),
}


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("form", sorted(FORMS))
def test_forms(gpu, form, kernel):
    kw, shapes = FORMS[form]
    seed = sum(map(ord, form))
    cases = [make_case("%s/%dx%dx%d" % (form, M, N, K), M, N, K, seed + i, **kw) for i, (M, N, K) in enumerate(shapes)]
    run_cases(cases, kernel, seed=seed)


# split_k cases: (M, N, K, split_k) with kb = ceil(K / 64); kb = 9, split_k = 4 and kb = 10, split_k = 7 write
# fewer slices than asked (3 and 5), split_k = 12 > kb
SPLITS = [(129, 96, 9 * 64, 4), (200, 200, 640 - 7, 7), (127, 33, 192, 2), (255, 129, 448, 3), (129, 128, 100, 12)]


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", KERNELS)
@pytest.mark.parametrize("variant", ["plain", "bias_row_flag", "transposed", "hilo_a", "wgrad3", "stride_odd"])
def test_split_k(gpu, variant, kernel):
    """Slices 0 .. S-1 hold partial sums that add up to the product (bias once, in slice 0), slices S ..
    split_k-1 keep their sentinel."""
    kw = dict(plain={}, bias_row_flag=dict(bias="aligned", row_flag=True), transposed=dict(out="f32_t", bias="aligned"),
              hilo_a=dict(passes="hilo_a"), wgrad3=dict(passes="wgrad3", a_mn=True),
              stride_odd=dict(stride_pad=1, bias="misaligned"))[variant]
    cases = [make_case("split%d/%dx%dx%d" % (sk, M, N, K), M, N, K, 50 + i, split_k=sk, **kw)
             for i, (M, N, K, sk) in enumerate(SPLITS)]
    run_cases(cases, kernel, seed=51)


@pytest.mark.gpu
def test_split_k_slice_count_documented(gpu):
    """kb = 9, split_k = 4: exactly three slices are written, the fourth keeps its sentinel."""
    case = make_case("kb9_split4", 129, 96, 9 * 64, 3, split_k=4)
    exp = reference(case[1], case[2], case[3])
    assert len(exp.offsets) == 3
    run_cases([case], "single")
    stride = case[1]["split_stride"]
    assert bool(torch.isnan(case[3][1 + 3 * stride:]).all())


@pytest.mark.gpu
def test_grouped_launch_lpt_order(gpu):
    """32 problems of mixed cost (k-blocks 1 .. 64, every epilogue cost class) in one launch: the LPT tile order.
    K is a multiple of 64 here, so every problem takes two tensor maps: 64, the launch's limit."""
    forms = [dict(), dict(out="split"), dict(out="split_t", a_mn=True), dict(act=ACT_TANH, bias="aligned"),
             dict(passes="hilo_a"), dict(passes="wgrad3", a_mn=True), dict(out="f32_t"), dict(b_mn=True)]
    shapes = [(700, 512, 64), (130, 256, 4096), (64, 101, 128), (1000, 15, 192), (257, 200, 640), (3000, 96, 128),
              (129, 33, 960), (511, 300, 320)]
    cases = [make_case("lpt%d" % i, *shapes[i % 8], 200 + i, **forms[(i + i // 8) % 8]) for i in range(32)]
    assert not _fits_single([c[1] for c in cases])
    run_launch(cases, "pair")


@pytest.mark.gpu
def test_grouped_launch_identity_order(gpu):
    """Over 5120 tiles (MAX_ORDERED_TILES) the kernel walks the tiles in identity order: split-K into 65 slices
    of 80 row tiles, next to a problem of another cost."""
    big = make_case("many_tiles", 80 * 256, 8, 65 * 64, 300, split_k=65)
    assert _tiles(big[1], "pair", "written") > 5120
    run_launch([big, make_case("other", 300, 257, 192, 301, bias="aligned")], "pair")


@pytest.mark.gpu
def test_grouped_launch_empty_problems(gpu):
    """Problems with M = 0 or N = 0 inside a launch write nothing; their neighbours are unaffected."""
    cases = [make_case("m0", 0, 96, 64, 400), make_case("n0", 129, 0, 64, 401),
             make_case("live", 200, 96, 100, 402, bias="aligned"), make_case("m0_split", 0, 33, 640, 403, split_k=4)]
    run_cases(cases, "single", seed=404)
    run_cases(cases, "pair", seed=405)


@pytest.mark.gpu
def test_determinism(gpu):
    """The same launch twice gives bit-identical outputs, split-K slices included."""
    from lirec_b200 import ops
    cases = [make_case("d0", 3000, 200, 4096, 500, passes="hilo_a", split_k=5),
             make_case("d1", 257, 96, 1000, 501, a_mn=True, split_k=3, out="f32_t"),
             make_case("d2", 255, 257, 192, 502, out="split_t", a_mn=True, act=ACT_TANH, bias="aligned")]
    outs = []
    for _ in range(2):
        for c in cases:
            c[3].fill_(float("nan"))
        ops.gemm_grouped([to_problem(*c[1:]) for c in cases])
        torch.cuda.synchronize()
        outs.append([c[3].clone() for c in cases])
    for x, y in zip(*outs):
        assert torch.equal(x.view(torch.int16 if x.element_size() == 2 else torch.int32),
                           y.view(torch.int16 if y.element_size() == 2 else torch.int32))


# ------------------------------------------------------------------------------------------------------------
# Limits and refusals: the call fails and writes nothing
# ------------------------------------------------------------------------------------------------------------
REFUSALS = {
    "four_groups": (dict(passes="four_groups"), "operand groups"),
    "split_k_split_output": (dict(split_k=2, out="split"), "split-K needs an fp32 output"),
    "split_k_act": (dict(split_k=2, act=ACT_RELU), "split-K partial sums"),
    "split_k_post": (dict(split_k=2, post=POST_DROPOUT, drop_p=0.2), "split-K partial sums"),
    "split_k_accumulate": (dict(split_k=2, accumulate=True), "split-K partial sums"),
    "accumulate_split_output": (dict(accumulate=True, out="split"), "accumulate needs an fp32 output"),
    "accumulate_split_t_output": (dict(accumulate=True, out="split_t"), "accumulate needs an fp32 output"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(REFUSALS))
def test_refused(gpu, name):
    from lirec_b200 import ops
    kw, msg = REFUSALS[name]
    case = make_case(name, 129, 96, 640, 600, **kw)
    before = case[3].clone()
    with pytest.raises(RuntimeError, match=msg):
        ops.gemm_grouped([to_problem(*case[1:])])
    torch.cuda.synchronize()
    assert torch.equal(case[3].view(torch.int16 if before.element_size() == 2 else torch.int32),
                       before.view(torch.int16 if before.element_size() == 2 else torch.int32))


@pytest.mark.gpu
def test_too_many_problems_refused(gpu):
    from lirec_b200 import _ext
    cases = [make_case("p%d" % i, 64, 64, 64, 700 + i) for i in range(33)]
    with pytest.raises(RuntimeError, match="too many GEMM problems"):
        _ext.gemm_grouped([to_problem(*c[1:]) for c in cases])


@pytest.mark.gpu
def test_too_many_tensor_maps_refused(gpu):
    """17 problems x 2 passes with their own A and B: 68 distinct operands > LIREC_GEMM_MAX_MAPS (64)."""
    from lirec_b200 import _ext
    cases = [make_case("p%d" % i, 64, 64, 64, 800 + i, passes="two_ranges") for i in range(17)]
    with pytest.raises(RuntimeError, match=r"tensor maps.*\(code -4\)"):
        _ext.gemm_grouped([to_problem(*c[1:]) for c in cases])
    for c in cases:
        assert bool(torch.isnan(c[3]).all())


@pytest.mark.gpu
@pytest.mark.parametrize("a_mn,b_mn", MAJOR)
def test_unaligned_column_offset_refused(gpu, a_mn, b_mn):
    """An offset along an operand's columns that is not a multiple of 8 elements is refused before launch."""
    from lirec_b200 import ops
    for side in (0, 1):
        name, spec, opnds, buf = make_case("unaligned", 129, 96, 128, 900, a_mn=a_mn, b_mn=b_mn)
        p = list(spec["passes"][0])
        mn_major = b_mn if side else a_mn
        p[3 * side + (1 if mn_major else 2)] += 4
        spec["passes"] = [tuple(p)]
        with pytest.raises(RuntimeError, match="multiples of 8 elements"):
            ops.gemm_grouped([to_problem(spec, opnds, buf)])
        assert bool(torch.isnan(buf).all())
