"""Ragged-row kernels (segmented pooling, expansion fwd/bwd, split, cast) vs numpy/torch restatements."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _ragged(rng, nseg, max_len, dim, empty_every=5):
    lens = rng.integers(1, max_len + 1, size=nseg)
    lens[::empty_every] = 0                                   # empty tracks / no dialog
    off = np.zeros(nseg + 1, dtype=np.int32)
    np.cumsum(lens, out=off[1:])
    x = rng.standard_normal((int(off[-1]), dim)).astype(np.float32)
    return x, off


@pytest.mark.parametrize("dim,max_len", [(2048, 64), (768, 128), (2048, 1024)])
def test_segmented_max_is_bit_exact(dim, max_len):
    """Temporal max pool (mixed_features.py:54,61,105): bit-exact, empty segment -> zeros, and the
    bf16 output equals round(max) because rounding is monotone."""
    from lirec_b200 import ops
    from oracle import pooling as op
    rng = np.random.default_rng(1)
    x, off = _ragged(rng, 37, max_len, dim)
    xd, offd = torch.from_numpy(x).cuda(), torch.from_numpy(off).cuda()
    o32 = torch.empty(37, dim, device="cuda")
    o16 = torch.empty(37, dim, device="cuda", dtype=torch.bfloat16)
    ops.seg_reduce(xd, offd, "max", out_f32=o32, out_bf16=o16)
    ref = op.segmented_max(x, off)
    assert np.array_equal(o32.cpu().numpy(), ref)
    assert torch.equal(o16.cpu(), torch.from_numpy(ref).to(torch.bfloat16))


def test_segmented_mean():
    from lirec_b200 import ops
    from oracle import pooling as op
    rng = np.random.default_rng(2)
    x, off = _ragged(rng, 20, 50, 512)
    o32 = torch.empty(20, 512, device="cuda")
    ops.seg_reduce(torch.from_numpy(x).cuda(), torch.from_numpy(off).cuda(), "mean", out_f32=o32)
    np.testing.assert_allclose(o32.cpu().numpy(), op.segmented_mean(x, off), rtol=0, atol=1e-6)


def test_max_propagates_nan_like_numpy():
    from lirec_b200 import ops
    x = np.ones((6, 8), dtype=np.float32)
    x[4, 3] = np.nan
    off = np.array([0, 3, 6], dtype=np.int32)
    o = torch.empty(2, 8, device="cuda")
    ops.seg_reduce(torch.from_numpy(x).cuda(), torch.from_numpy(off).cuda(), "max", out_f32=o)
    ref = np.stack([x[0:3].max(0), x[3:6].max(0)])
    assert np.array_equal(np.isnan(o.cpu().numpy()), np.isnan(ref))


def _expand_reference(r1, rows, seg_off, keep, J, guard):
    """numpy restatement of lirec_rows_expand_fwd (fp64)."""
    cols = [rows[:, 0], rows[:, 0], rows[:, 1], rows[:, 2]]
    per_row = np.concatenate([r1[s][cols[s]].astype(np.float64) for s in range(4)], axis=1) * keep
    if seg_off is None:
        return per_row
    out = np.zeros((len(seg_off) - 1, 4 * J))
    for c in range(len(seg_off) - 1):
        a, b = seg_off[c], seg_off[c + 1]
        if b > a:
            out[c] = per_row[a:b].sum(0) / (b - a)
        elif not guard:
            out[c] = np.nan
    return out


@pytest.mark.parametrize("p", [0.0, 0.3])
def test_expand_forward_and_transposed_backward(p):
    from lirec_b200 import ops
    from oracle import dropout as od
    rng = np.random.default_rng(3)
    J, n_clip, n_track, n_rows, n_out, seed = 512, 9, 14, 60, 17, 4242
    r1 = [np.maximum(rng.standard_normal((n, J)), 0).astype(np.float32) for n in (n_clip, n_clip, n_track, n_track)]
    rows = np.stack([rng.integers(n_clip, size=n_rows), rng.integers(n_track, size=n_rows),
                     rng.integers(n_track, size=n_rows)], 1).astype(np.int32)
    cuts = np.sort(rng.integers(0, n_rows + 1, size=n_out - 1))
    seg = np.concatenate([[0], cuts, [n_rows]]).astype(np.int32)
    seg[3] = seg[2]                                             # an empty segment
    seg = np.maximum.accumulate(seg)
    r1d = [torch.from_numpy(a).cuda() for a in r1]
    rowsd, segd = torch.from_numpy(rows).cuda(), torch.from_numpy(seg).cuda()
    keep = od.keep_mask(seed, 2, np.arange(n_rows), np.arange(4 * J), p)
    drop = ops.dropout_desc(p, seed, 2, 0)
    for seg_np, seg_t, n_o in ((None, None, n_rows), (seg, segd, n_out)):
        out = torch.zeros(n_o, 8 * J, device="cuda", dtype=torch.bfloat16)
        flag = torch.full((n_o,), -1, device="cuda", dtype=torch.int32)
        ops.rows_expand_fwd(r1d, J, rowsd, seg_t, n_o, 1, drop, out, flag if seg_t is not None else None)
        got = out.view(n_o, 4, 2, J).double().sum(2).reshape(n_o, 4 * J).cpu().numpy()
        ref = _expand_reference(r1, rows, seg_np, keep, J, guard=True)
        np.testing.assert_allclose(got, ref, rtol=0, atol=2e-5 * max(1.0, np.abs(ref).max()))
        if seg_t is not None:
            assert flag.cpu().tolist() == [int(seg[c + 1] > seg[c]) for c in range(n_out)]
    # no guard: empty segment -> NaN like the reference's 0/0 (MidFusionMultiClip, model.py:175)
    out = torch.zeros(n_out, 8 * J, device="cuda", dtype=torch.bfloat16)
    ops.rows_expand_fwd(r1d, J, rowsd, segd, n_out, 0, drop, out, None)
    empty = [c for c in range(n_out) if seg[c + 1] == seg[c]]
    assert empty and torch.isnan(out[empty].float()).all() and not torch.isnan(out[[c for c in range(n_out) if c not in empty]].float()).any()

    # backward: dZ1[u] = [r1[u] > 0] * sum_i keep_i * d[o_i] * w_i, context form (o_i = owner_i,
    # w_i = 1 / n(owner_i)) and ints form (o_i = i, w_i = 1), written transposed [2J, pitch] (hi rows, lo rows)
    from lirec_b200.packing import _csr_inverse
    owner = np.repeat(np.arange(n_out), np.diff(seg)).astype(np.int32)
    d_ctx = rng.standard_normal((n_out, 4 * J)).astype(np.float32)
    d_ints = rng.standard_normal((n_rows, 4 * J)).astype(np.float32)
    # the ReLU gate as the layer-1 GEMM writes it (LIREC_POST_SIGN_MASK): bit j & 31 of word u * J / 32 + (j >> 5)
    sign = [torch.from_numpy(np.packbits(a > 0, axis=1, bitorder="little").view("<u4").view(np.int32)).cuda()
            for a in r1]
    for d, owner_np in ((d_ctx, owner), (d_ints, None)):
        dd = torch.from_numpy(d).cuda()
        owner_t, seg_t = (torch.from_numpy(owner_np).cuda(), segd) if owner_np is not None else (None, None)
        for slot, col, n_u in ((0, 0, n_clip), (1, 0, n_clip), (2, 1, n_track), (3, 2, n_track)):
            off, idx = _csr_inverse(rows[:, col], n_u)
            pitch = (n_u + 63) // 64 * 64
            out = torch.zeros(2 * J, pitch, device="cuda", dtype=torch.bfloat16)
            ops.rows_expand_bwd(dd, 4 * J, sign[slot], J, slot, torch.from_numpy(off).cuda(),
                                torch.from_numpy(idx).cuda(), n_u, owner_t, seg_t, drop, out, d_in_col_off=slot * J)
            ref = np.zeros((n_u, J))
            for i in range(n_rows):
                o = owner_np[i] if owner_np is not None else i
                n = seg[o + 1] - seg[o] if owner_np is not None else 1
                ref[rows[i, col]] += keep[i, slot * J:(slot + 1) * J] * d[o, slot * J:(slot + 1) * J] / n
            ref *= (r1[slot] > 0)
            got = (out[:J, :n_u].double() + out[J:, :n_u].double()).t().cpu().numpy()
            np.testing.assert_allclose(got, ref, rtol=0, atol=2e-5 * np.abs(ref).max())


def test_transposed_split_and_cast():
    from lirec_b200 import ops
    x = torch.randn(37, 101, device="cuda") * 3
    out_t = torch.full((256, 40), 7.0, device="cuda", dtype=torch.bfloat16)   # transposed [2 * pad, pitch]
    ops.split_f32(x, out_t, 128)
    out = out_t[:, :37].t()                                                    # [rows, 2 * pad]: hi | lo
    assert torch.equal(out[:, :101], x.to(torch.bfloat16))
    assert (out[:, 101:128] == 0).all() and (out[:, 128 + 101:] == 0).all()
    rec = out[:, :101].double() + out[:, 128:128 + 101].double()
    assert float((rec - x.double()).abs().max() / x.abs().max()) < 2 ** -16
    y = torch.randn(100003, device="cuda")
    yb = torch.empty(100003, device="cuda", dtype=torch.bfloat16)
    ops.cast_bf16(y, yb)
    assert torch.equal(yb, y.to(torch.bfloat16))
