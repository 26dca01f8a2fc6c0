"""Fused spatial / person-box mean + temporal max on the GPU (lirec_roi_max_pool_f32) against the rows
the reference's unmodified VisualFeatures produced (tests/golden/pooling_visual.npz): the means within
2e-6 relative (a different float32 summation order than numpy's pairwise sum), the max an exact
selection of them, NaN / zero-row / empty-track quirks identical."""
import numpy as np
import pytest
import torch

from test_pooling_cpu import load_world, numpy_rows

pytestmark = pytest.mark.gpu
RTOL = 2e-6


def test_visual_pooling_matches_the_reference(opt_preset):
    from lirec_b200.utils.arg_pars import opt
    from lirec_b200.visual_utils.visual_features import VisualFeatures
    opt.sampling_fr = 0.0625
    g, meta, feats, frame2time, dims = load_world()
    v = VisualFeatures(feats, frame2time, dims, device="cuda")
    for i, tn in enumerate(meta["time_nodes"]):
        rows = v.get_features_by_time(tn).cpu().numpy()
        np.testing.assert_allclose(rows, g["time_rows_%d" % i], rtol=RTOL, atol=0)
    for i, tr in enumerate(meta["tracks"]):
        if not tr:
            continue
        rows = v.get_features_by_track(tr).cpu().numpy()
        ref = g["track_rows_%d" % i]
        assert np.array_equal(np.isnan(rows), np.isnan(ref))
        np.testing.assert_allclose(rows, ref, rtol=RTOL, atol=0)
    # one launch for every clip and track of the scene; bf16 bank rows
    pooled = v.pool(meta["time_nodes"], meta["tracks"]).cpu().numpy()
    nt = len(meta["time_nodes"])
    for i in range(nt):
        np.testing.assert_allclose(pooled[i:i + 1], g["time_max_%d" % i], rtol=RTOL, atol=0)
    for i in range(len(meta["tracks"])):
        ref = g["track_max_%d" % i]
        got = pooled[nt + i:nt + i + 1]
        assert np.array_equal(np.isnan(got), np.isnan(ref)), i
        np.testing.assert_allclose(got, ref, rtol=RTOL, atol=0)
    assert not pooled[nt + len(meta["tracks"]) - 1].any()          # the empty track
    bank = torch.empty(pooled.shape[0], pooled.shape[1], dtype=torch.bfloat16, device="cuda")
    v.pool(meta["time_nodes"], meta["tracks"], out_bf16=bank)
    ref16 = torch.from_numpy(pooled).to(torch.bfloat16)
    assert torch.equal(torch.nan_to_num(bank.cpu().float(), nan=-1.0), torch.nan_to_num(ref16.float(), nan=-1.0))


def test_roi_pool_full_size_maps_against_numpy():
    """I3D-sized maps [T, 2048, 13, 30]: random boxes, ragged segments, max is an exact selection."""
    from lirec_b200 import ops
    rng = np.random.RandomState(0)
    T, C, H, W = 6, 2048, 13, 30
    feats = np.abs(rng.standard_normal((T, C, H, W))).astype(np.float32)
    n = 40
    el = np.zeros((n, 5), dtype=np.int32)
    el[:, 0] = rng.randint(0, T, n)
    el[:, 1] = rng.randint(0, H - 1, n)
    el[:, 2] = el[:, 1] + 1 + rng.randint(0, H, n)
    el[:, 2] = np.minimum(el[:, 2], H)
    el[:, 3] = rng.randint(0, W - 1, n)
    el[:, 4] = np.minimum(el[:, 3] + 1 + rng.randint(0, W, n), W)
    el[5] = (2, 0, H, 0, W)
    el[9, 0] = -1
    seg = np.array([0, 1, 1, 7, 20, 40], dtype=np.int32)
    rows = numpy_rows(feats, el)
    ref = np.stack([rows[a:b].max(axis=0) if b > a else np.zeros(C) for a, b in zip(seg[:-1], seg[1:])])
    maps = torch.from_numpy(feats).cuda()
    out = ops.roi_max_pool(maps, torch.from_numpy(el).cuda(), torch.from_numpy(seg).cuda()).cpu().numpy()
    np.testing.assert_allclose(out, ref, rtol=RTOL, atol=0)
    one = ops.roi_max_pool(maps, torch.from_numpy(el).cuda(), torch.from_numpy(seg).cuda(), two_stage=False).cpu().numpy()
    np.testing.assert_allclose(one, ref, rtol=RTOL, atol=0)             # the single-pass form of the same pooling
    per = ops.roi_max_pool(maps, torch.from_numpy(el).cuda(),
                           torch.arange(n + 1, dtype=torch.int32).cuda()).cpu().numpy()
    sel = np.stack([per[a:b].max(axis=0) if b > a else np.zeros(C, dtype=np.float32) for a, b in zip(seg[:-1], seg[1:])])
    assert np.array_equal(out, sel)                                   # max = exact selection of the means


def test_text_pooling_matches_the_reference():
    """Gathered segmented max over dialog tokens (lirec_seg_reduce_f32 with a row index): bit-exact with np.max over
    the rows the reference's unmodified TextFeatures returned; zero row for clips without dialog."""
    from test_pooling_cpu import load_text_world
    from lirec_b200.text_utils.text_features import TextFeatures
    g, meta, feats = load_text_world()
    t = TextFeatures(feats, meta["times"], meta["ranges"], device="cuda")
    for i, tn in enumerate(meta["nodes"]):
        assert np.array_equal(t.get_features_by_time(tn).cpu().numpy(), g["rows_%d" % i])
    pooled = t.pool(meta["nodes"]).cpu().numpy()
    for i in range(len(meta["nodes"])):
        assert np.array_equal(pooled[i:i + 1], g["max_%d" % i]), i
    bank = torch.empty(len(meta["nodes"]), feats.shape[1], dtype=torch.bfloat16, device="cuda")
    t.pool(meta["nodes"], out_bf16=bank)
    assert torch.equal(bank.cpu(), torch.from_numpy(pooled).to(torch.bfloat16))
    # gathered mean against numpy on random index lists
    from lirec_b200 import ops
    rng = np.random.default_rng(0)
    x = rng.standard_normal((500, 768)).astype(np.float32)
    lists = [rng.integers(0, 500, size=int(n)) for n in rng.integers(0, 40, size=30)]
    off = np.zeros(31, dtype=np.int32)
    np.cumsum([len(l) for l in lists], out=off[1:])
    idx = np.concatenate(lists).astype(np.int32)
    out = torch.empty(30, 768, device="cuda")
    ops.seg_reduce(torch.from_numpy(x).cuda(), torch.from_numpy(off).cuda(), "mean", out_f32=out,
                   row_idx=torch.from_numpy(idx).cuda())
    ref = np.stack([x[l].mean(0) if len(l) else np.zeros(768, dtype=np.float32) for l in lists])
    np.testing.assert_allclose(out.cpu().numpy(), ref, rtol=1e-5, atol=1e-6)


# ---- softmax-weighted segmented reduction (row N1; parity unpinned by construction: the reference has none) -------
def _np_softpool(x, off, beta, scores):
    """float64 numpy statement: out, and the gradients of sum(out * dy) for a given dy."""
    x = x.astype(np.float64)
    nseg, dim = len(off) - 1, x.shape[1]
    out = np.zeros((nseg, dim))
    ws = []
    for s in range(nseg):
        a, b = off[s], off[s + 1]
        if b <= a:
            ws.append(None)
            continue
        sc = x[a:b] if scores is None else (scores[a:b].astype(np.float64) if scores.ndim == 2
                                            else np.repeat(scores[a:b, None].astype(np.float64), dim, 1))
        z = beta * sc
        w = np.exp(z - z.max(0, keepdims=True))
        w /= w.sum(0, keepdims=True)
        out[s] = (w * x[a:b]).sum(0)
        ws.append(w)
    return out, ws


def _np_softpool_bwd(x, off, beta, scores, out, ws, dy):
    x = x.astype(np.float64)
    dx = np.zeros_like(x)
    ds = None if scores is None else np.zeros(scores.shape)
    for s in range(len(off) - 1):
        a, b = off[s], off[s + 1]
        if b <= a:
            continue
        w = ws[s]
        gx = w * dy[s]
        gs = beta * gx * (x[a:b] - out[s])
        if scores is None:
            dx[a:b] = gx + gs
        else:
            dx[a:b] = gx
            ds[a:b] = gs if scores.ndim == 2 else gs.sum(1)
    return dx, ds


@pytest.mark.parametrize("many", [False, True])
@pytest.mark.parametrize("kind", ["self", "elem", "row"])
def test_softmax_pool_forward_backward_vs_numpy(kind, many):
    """The kernels' CTA shape (four row lanes of 128 columns merged in shared memory), a handful of segments and
    thousands of them, ragged lengths around the four-row batches and the row chunks of the per-row-score backward."""
    from lirec_b200 import ops
    rng = np.random.default_rng(3)
    lens = [5, 0, 1, 37, 12, 0, 64, 3]                       # ragged, with empty segments
    dim, beta = 768, 1.7
    if many:
        lens = lens + [int(v) for v in rng.integers(0, 23, size=1900)]
        dim = 1024
    off = np.concatenate(([0], np.cumsum(lens))).astype(np.int32)
    x = rng.standard_normal((off[-1], dim)).astype(np.float32)
    scores = None if kind == "self" else (rng.standard_normal((off[-1], dim)) if kind == "elem"
                                          else rng.standard_normal(off[-1])).astype(np.float32)
    dy = rng.standard_normal((len(lens), dim))
    ref, ws = _np_softpool(x, off, beta, scores)
    rdx, rds = _np_softpool_bwd(x, off, beta, scores, ref, ws, dy)
    xd = torch.from_numpy(x).cuda().requires_grad_(True)
    sd = None if scores is None else torch.from_numpy(scores).cuda().requires_grad_(True)
    offd = torch.from_numpy(off).cuda()
    out = ops.SegSoftmaxPool.apply(xd, offd, beta, sd)
    (out * torch.from_numpy(dy).float().cuda()).sum().backward()
    assert float(np.abs(out.detach().cpu().numpy() - ref).max()) < 2e-5 * max(1.0, np.abs(ref).max())
    assert (out.detach().cpu().numpy()[[1, 5]] == 0).all()    # empty segments -> zeros, like max / mean
    assert float(np.abs(xd.grad.cpu().numpy() - rdx).max()) < 3e-5 * np.abs(rdx).max()
    if scores is not None:
        assert float(np.abs(sd.grad.cpu().numpy() - rds).max()) < 3e-5 * np.abs(rds).max()


@pytest.mark.parametrize("kind", ["self", "elem", "row"])
def test_softmax_pool_backward_zero_fills_rows_no_segment_owns(kind):
    """The offsets need not tile x: rows before the first and after the last offset get zero gradients from the
    backward launch itself (the wrapper hands it uninitialised buffers, no memset)."""
    from lirec_b200 import ops
    rng = np.random.default_rng(8)
    total, dim, beta = 40, 256, 0.9
    off = torch.tensor([3, 3, 11, 30], dtype=torch.int32, device="cuda")
    x = torch.from_numpy(rng.standard_normal((total, dim)).astype(np.float32)).cuda()
    scores = None if kind == "self" else torch.from_numpy(
        (rng.standard_normal((total, dim)) if kind == "elem" else rng.standard_normal(total)).astype(np.float32)).cuda()
    out, lse = ops.seg_softmax_pool(x, off, beta, scores)
    junk = torch.full((64, total, dim), float("nan"), device="cuda")          # dirty the allocator's free blocks
    del junk
    d_x, d_s = ops.seg_softmax_pool_bwd(x, off, beta, scores, out, lse, torch.ones_like(out))
    assert bool((d_x[:3] == 0).all()) and bool((d_x[30:] == 0).all()) and bool(torch.isfinite(d_x).all())
    assert bool((d_x[3:30].abs().sum(1) > 0).all())
    if d_s is not None:
        assert bool((d_s[:3] == 0).all()) and bool((d_s[30:] == 0).all()) and bool(torch.isfinite(d_s).all())


def test_softmax_pool_limits_are_the_reference_poolings():
    """beta = 0 (uniform weights) is the masked MEAN and beta -> inf with score = x is the MAX — the two poolings
    the reference does have (mlp/model.py:301-304, mixed_features.py:54) and lirec_seg_reduce_f32 is pinned on."""
    from lirec_b200 import ops
    rng = np.random.default_rng(4)
    lens = [9, 1, 0, 128, 17]
    off = torch.from_numpy(np.concatenate(([0], np.cumsum(lens))).astype(np.int32)).cuda()
    x = torch.from_numpy(np.abs(rng.standard_normal((sum(lens), 2048))).astype(np.float32)).cuda()
    mean = torch.empty(len(lens), 2048, device="cuda")
    mx = torch.empty(len(lens), 2048, device="cuda")
    ops.seg_reduce(x, off, "mean", out_f32=mean)
    ops.seg_reduce(x, off, "max", out_f32=mx)
    soft0, _ = ops.seg_softmax_pool(x, off, beta=0.0)
    hard, _ = ops.seg_softmax_pool(x, off, beta=1e6)
    assert float((soft0 - mean).abs().max()) < 1e-6 * float(mean.abs().max())
    assert torch.equal(hard, mx)                               # an exact selection, ties included
    # all-zero scores of either kind are the mean too
    z, _ = ops.seg_softmax_pool(x, off, beta=3.0, scores=torch.zeros(x.shape[0], device="cuda"))
    assert float((z - mean).abs().max()) < 1e-6 * float(mean.abs().max())
    # temperature -> 0 on per-row scores selects the best-scored row of every segment
    sc = torch.from_numpy(rng.standard_normal(sum(lens)).astype(np.float32)).cuda()
    sel, _ = ops.seg_softmax_pool(x, off, beta=1e6, scores=sc)
    o = off.cpu().numpy()
    for s in range(len(lens)):
        if lens[s]:
            r = o[s] + int(torch.argmax(sc[o[s]:o[s + 1]]))
            assert torch.equal(sel[s], x[r])
