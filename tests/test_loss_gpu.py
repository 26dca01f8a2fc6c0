"""Fused loss kernels vs the dense oracle losses: loss value, gradient w.r.t. logits, and the
arg-max track assignment (bit-exact, lowest index on ties)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

C, R, T = 101, 15, 20


def _ragged_case(B, seed, with_rels=True, dup_ties=False):
    rng = np.random.default_rng(seed)
    counts = rng.choice([2, 6, 12, 20, 1, 7], size=B)
    off = np.zeros(B + 1, dtype=np.int32)
    np.cumsum(counts, out=off[1:])
    Ni = int(off[-1])
    ints = (rng.standard_normal((Ni, C)) * 2).astype(np.float32)
    rels = (rng.standard_normal((Ni, R)) * 2).astype(np.float32)
    if dup_ties:                      # duplicated candidates (all-zero tracks give identical rows in real data)
        for b in range(B):
            if counts[b] >= 3:
                ints[off[b] + 2] = ints[off[b] + 1]
                rels[off[b] + 2] = rels[off[b] + 1]
                ints[off[b] + 0] = ints[off[b] + 1] - 5.0     # make the tied pair the winners
    labels = rng.integers(C, size=B).astype(np.int32)
    rels_label = rng.integers(R + 1, size=Ni).astype(np.int32)   # R = None
    if dup_ties:
        for b in range(B):
            if counts[b] >= 3:
                rels_label[off[b] + 2] = rels_label[off[b] + 1]
    gt = np.zeros((B, 2), dtype=np.int32)
    gt[:, 1] = [rng.integers(c) if rng.random() < 0.4 else 0 for c in counts]
    multilab = (rng.random((B, C)) < 0.9).astype(np.uint8)
    return dict(off=off, ints=ints, rels=rels if with_rels else None, labels=labels, rels_label=rels_label, gt=gt,
                multilab=multilab, counts=counts)


def _dense(case):
    B = len(case["counts"])
    off = case["off"]
    ints = torch.zeros(B, T, C, dtype=torch.float64)
    rels = torch.zeros(B, T, R, dtype=torch.float64)
    mem = torch.zeros(B, T, dtype=torch.float64)
    rl = torch.zeros(B, T, dtype=torch.long)
    for b in range(B):
        n = case["counts"][b]
        ints[b, :n] = torch.from_numpy(case["ints"][off[b]:off[b + 1]]).double()
        if case["rels"] is not None:
            rels[b, :n] = torch.from_numpy(case["rels"][off[b]:off[b + 1]]).double()
        mem[b, :n] = 1
        rl[b, :n] = torch.from_numpy(case["rels_label"][off[b]:off[b + 1]]).long()
    # the reference computes finite logits for empty slots too before masking them: use garbage there
    g = torch.Generator().manual_seed(1)
    ints = torch.where(mem.bool().unsqueeze(-1), ints, torch.randn(B, T, C, generator=g, dtype=torch.float64))
    rels = torch.where(mem.bool().unsqueeze(-1), rels, torch.randn(B, T, R, generator=g, dtype=torch.float64))
    return ints.requires_grad_(True), rels.requires_grad_(True), mem, rl


@pytest.mark.parametrize("tr_correct,max_neg", [(False, False), (True, False), (False, True), (True, True)])
@pytest.mark.parametrize("with_rels", [True, False])
def test_track_losses(tr_correct, max_neg, with_rels):
    from lirec_b200 import ops
    from oracle import losses as ol
    case = _ragged_case(24, seed=7 + int(tr_correct) + 2 * int(max_neg), with_rels=with_rels)
    B = 24
    dev = lambda a: None if a is None else torch.from_numpy(a).cuda()
    lo, assign, d_i, d_r = ops.loss_track(dev(case["ints"]), dev(case["rels"]), dev(case["off"]), dev(case["labels"]),
                                          dev(case["rels_label"]), dev(case["gt"]), dev(case["multilab"]), 0.101,
                                          0.7 if with_rels else 1.0, R if with_rels else 0, tr_correct=tr_correct,
                                          max_neg=max_neg, max_slots=T)
    ints, rels, mem, rl = _dense(case)
    labels, gt = torch.from_numpy(case["labels"]).long(), torch.from_numpy(case["gt"]).long()
    mw = torch.from_numpy(case["multilab"]).double()
    if with_rels:
        ref, ts, _, _ = ol.margin_track_rels(ints, rels, labels, rl, mem, mw, gt, 0.101, 0.7, R, tr_correct=tr_correct,
                                             max_neg=max_neg)
    else:
        ref, ts, _ = ol.margin_loss(ints, labels, mem, mw, gt, 0.101, tr_correct=tr_correct, max_neg=max_neg)
    ref.backward()
    assert torch.equal(assign.cpu().long(), ts)                       # bit-exact assignment
    assert abs(lo.sum().item() - ref.item()) / abs(ref.item()) < 1e-5
    mm = mem.bool()
    gi = ints.grad[mm]
    assert float((d_i.cpu().double() - gi).abs().max() / gi.abs().max()) < 1e-4
    assert ints.grad[~mm].abs().max() == 0                            # empty slots get exactly zero gradient
    if with_rels:
        gr = rels.grad[mm]
        assert float((d_r.cpu().double() - gr).abs().max() / (gr.abs().max() + 1e-30)) < 1e-4


def test_assignment_ties_resolve_to_lowest_index():
    from lirec_b200 import ops
    from oracle import losses as ol
    case = _ragged_case(40, seed=3, dup_ties=True)
    dev = lambda a: torch.from_numpy(a).cuda()
    _, assign, _, _ = ops.loss_track(dev(case["ints"]), dev(case["rels"]), dev(case["off"]), dev(case["labels"]),
                                     dev(case["rels_label"]), dev(case["gt"]), dev(case["multilab"]), 0.101, 1.0, R)
    ints, rels, mem, rl = _dense(case)
    _, ts, _, _ = ol.margin_track_rels(ints.float(), rels.float(), torch.from_numpy(case["labels"]).long(), rl, mem.float(),
                                       torch.from_numpy(case["multilab"]).float(), torch.from_numpy(case["gt"]).long(),
                                       0.101, 1.0, R)
    assert torch.equal(assign.cpu().long(), ts)
    tied = [b for b in range(40) if case["counts"][b] >= 3]
    assert tied and any(int(assign[b]) == 1 for b in tied)            # slot 1 wins its tie with slot 2


def test_row_margin_loss():
    """MaxMarginCrossEntropyLoss / MultiTaskMaxMargin terms (model.py:381-441)."""
    from lirec_b200 import ops
    from oracle import losses as ol
    rng = np.random.default_rng(0)
    B = 50
    x = (rng.standard_normal((B, C)) * 2).astype(np.float32)
    y = rng.integers(C, size=B).astype(np.int32)
    w = (rng.random((B, C)) < 0.9).astype(np.uint8)
    terms, d = ops.loss_rowmargin(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), torch.from_numpy(w).cuda(),
                                  0.101, 1.0 / B)
    xt = torch.from_numpy(x).double().requires_grad_(True)
    ref = ol.max_margin_ce(xt, torch.from_numpy(y).long(), torch.from_numpy(w).double(), 0.101)
    ref.backward()
    assert abs(terms.sum().item() - ref.item()) / ref.item() < 1e-5
    assert float((d.cpu().double() - xt.grad).abs().max() / xt.grad.abs().max()) < 1e-4
    # relationship term: rows labelled None (-1 here) are skipped
    r = (rng.standard_normal((B, R)) * 2).astype(np.float32)
    lab = rng.integers(R + 1, size=B).astype(np.int32)
    sel = lab.copy()
    sel[sel == R] = -1
    n_sel = int((lab != R).sum())
    terms, d = ops.loss_rowmargin(torch.from_numpy(r).cuda(), torch.from_numpy(sel).cuda(), None, 0.101, 1.0 / n_sel)
    rt = torch.from_numpy(r).double().requires_grad_(True)
    ref = ol.multitask_max_margin(None, rt, None, torch.from_numpy(lab).long(), None, 0.101, 1.0, R, ints=0, ctx=1)
    ref.backward()
    assert abs(terms.sum().item() - ref.item()) / ref.item() < 1e-5
    assert float((d.cpu().double() - rt.grad).abs().max() / rt.grad.abs().max()) < 1e-4


def test_flat_adam_matches_torch_adam():
    from lirec_b200 import ops
    torch.manual_seed(0)
    n = 100003
    p0 = torch.randn(n, device="cuda")
    ref_p = p0.clone().requires_grad_(True)
    opt = torch.optim.Adam([ref_p], lr=3e-5, weight_decay=1e-5)
    p, m, v = p0.clone(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    pb = torch.empty(n, device="cuda", dtype=torch.bfloat16)
    for step in range(1, 4):
        g = torch.randn(n, device="cuda")
        ref_p.grad = g.clone()
        opt.step()
        ops.adam_flat(p, g, m, v, pb, 3e-5, 0.9, 0.999, 1e-8, 1e-5, step)
    assert float((p - ref_p.detach()).abs().max()) < 1e-6
    assert torch.equal(pb, p.to(torch.bfloat16))


def test_coresident_adam_launch_shape_is_bit_identical():
    """lirec_adam_flat(coresident=1) — CTAs sized to share an SM with a resident GEMM CTA, used for the pass
    overlapped with backward — is the same arithmetic on the same elements: bit-identical buffers, also on a
    sub-range and on a side stream."""
    from lirec_b200 import ops
    torch.manual_seed(1)
    n = 1 << 20
    p0, g = torch.randn(n, device="cuda"), torch.randn(n, device="cuda")
    outs = []
    for co in (False, True):
        p, m, v = p0.clone(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
        pb = torch.zeros(n, device="cuda", dtype=torch.bfloat16)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        for step in (1, 2):
            ops.adam_flat(p, g, m, v, pb, 1e-3, 0.9, 0.999, 1e-8, 1e-5, step, grad_scale=0.5, offset=4096,
                          n=n - 8192, stream=side if co else None, coresident=co)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        outs.append((p, m, v, pb))
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    assert torch.equal(outs[1][0][:4096], p0[:4096]) and torch.equal(outs[1][0][-4096:], p0[-4096:])


@pytest.mark.parametrize("with_rels", [True, False])
def test_prediction_argmaxes_are_bit_exact(with_rels):
    """Device-side evaluation arg-maxes (utils/evaluation.py:114-271) equal the numpy restatement on
    identical logits, including exact ties between duplicated candidate slots."""
    from lirec_b200 import ops
    from oracle import evaluation as oe
    case = _ragged_case(48, seed=11, with_rels=with_rels, dup_ties=True)
    dev = lambda a: None if a is None else torch.from_numpy(a).cuda()
    got = ops.predict_tracks(dev(case["ints"]), dev(case["rels"]), dev(case["off"]), dev(case["labels"]),
                             dev(case["rels_label"]), dev(case["gt"]), R if with_rels else 0).cpu().numpy()
    ints, rels, mem, rl = _dense(case)
    ref = oe.predict_tracks(ints.detach().numpy(), rels.detach().numpy() if with_rels else None, mem.numpy(),
                            case["labels"], rl.numpy(), case["gt"])
    if not with_rels:
        ref[:, 3] = -1
    assert np.array_equal(got, ref)


@pytest.mark.parametrize("with_rels", [True, False])
def test_cat_distr_sampled_assignment(with_rels):
    """opt.tr_cat_distr (model.py:468-471, 538-543): t* is drawn from the softmax scores.  The kernel's draw
    is the inverse CDF of the oracle's distribution at the mirrored counter-hash uniform; loss and gradients
    match the oracle evaluated at the same assignment; over many seeds the frequencies follow the
    distribution."""
    from lirec_b200 import ops
    from oracle import dropout as od, losses as ol
    B = 32
    case = _ragged_case(B, seed=21, with_rels=with_rels)
    dev = lambda a: None if a is None else torch.from_numpy(a).cuda()
    args = (dev(case["ints"]), dev(case["rels"]), dev(case["off"]), dev(case["labels"]), dev(case["rels_label"]),
            dev(case["gt"]), dev(case["multilab"]), 0.101, 0.7 if with_rels else 1.0, R if with_rels else 0)
    ints, rels, mem, rl = _dense(case)
    labels, gt = torch.from_numpy(case["labels"]).long(), torch.from_numpy(case["gt"]).long()
    mw = torch.from_numpy(case["multilab"]).double()
    if with_rels:
        _, _, xm, rm = ol.margin_track_rels(ints, rels, labels, rl, mem, mw, gt, 0.101, 0.7, R)
        r0 = rl[torch.arange(B), gt[:, 0]]
        probs = ol.cat_distr_probs(xm.detach(), labels, rm.detach(), r0)
    else:
        _, _, xm = ol.margin_loss(ints, labels, mem, mw, gt, 0.101)
        probs = ol.cat_distr_probs(xm.detach(), labels)
    probs = probs.numpy()
    cdf = np.cumsum(probs, axis=1)
    total = cdf[:, -1]
    seed = 12345
    lo, assign, d_i, d_r = ops.loss_track(*args, max_slots=T, cat_distr=True, seed=seed)
    u = od.cat_distr_uniform(seed, B) * total
    expect = np.array([int(np.searchsorted(cdf[b], u[b], side="right")) for b in range(B)])
    edge = np.array([np.abs(cdf[b] - u[b]).min() < 1e-5 for b in range(B)])
    got = assign.cpu().numpy()
    assert (got[~edge] == expect[~edge]).all() and (~edge).sum() >= B - 2
    assert all(got[b] < case["counts"][b] for b in range(B))
    # same draw again; a different seed moves some assignments
    _, assign2, _, _ = ops.loss_track(*args, max_slots=T, cat_distr=True, seed=seed)
    assert torch.equal(assign, assign2)
    # loss / gradients at the sampled assignment
    forced = torch.from_numpy(got).long()
    if with_rels:
        ref, _, _, _ = ol.margin_track_rels(ints, rels, labels, rl, mem, mw, gt, 0.101, 0.7, R, assign=forced)
    else:
        ref, _, _ = ol.margin_loss(ints, labels, mem, mw, gt, 0.101, assign=forced)
    ref.backward()
    assert abs(lo.sum().item() - ref.item()) / abs(ref.item()) < 1e-5
    gi = ints.grad[mem.bool()]
    assert float((d_i.cpu().double() - gi).abs().max() / gi.abs().max()) < 1e-4
    if with_rels:
        gr = rels.grad[mem.bool()]
        assert float((d_r.cpu().double() - gr).abs().max() / (gr.abs().max() + 1e-30)) < 1e-4
    # statistics: 400 seeds, clips with >= 6 candidates
    counts = np.zeros((B, T))
    n_draws = 400
    for s in range(n_draws):
        _, a, _, _ = ops.loss_track(*args, max_slots=T, cat_distr=True, seed=1000 + s)
        counts[np.arange(B), a.cpu().numpy()] += 1
    freq = counts / n_draws
    pn = probs / total[:, None]
    assert np.abs(freq - pn).max() < 0.12
    assert np.abs(freq - pn).mean() < 0.01


def test_cross_entropy_loss():
    """MultiTaskCrossEntropyLoss terms (model.py:357-378): weighted CE of the interaction logits, CE of the
    relationship logits of rows whose label is not None."""
    from lirec_b200 import ops
    from oracle import losses as ol
    rng = np.random.default_rng(5)
    B = 70
    x = (rng.standard_normal((B, C)) * 3).astype(np.float32)
    y = rng.integers(C, size=B).astype(np.int32)
    r = (rng.standard_normal((B, R)) * 3).astype(np.float32)
    lab = rng.integers(R + 1, size=B).astype(np.int32)
    for weights in (None, (rng.random(C) + 0.5).astype(np.float32)):
        xt = torch.from_numpy(x).double().requires_grad_(True)
        rt = torch.from_numpy(r).double().requires_grad_(True)
        w64 = None if weights is None else torch.from_numpy(weights).double()
        ref = ol.multitask_ce(xt, rt, torch.from_numpy(y).long(), torch.from_numpy(lab).long(), R, weights=w64)
        ref.backward()
        denom = B if weights is None else float(weights[y].sum())
        t1, d1 = ops.loss_ce(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(),
                             None if weights is None else torch.from_numpy(weights).cuda(), 1.0 / denom)
        sel = lab.copy()
        sel[sel == R] = -1
        t2, d2 = ops.loss_ce(torch.from_numpy(r).cuda(), torch.from_numpy(sel).cuda(), None, 1.0 / int((lab != R).sum()))
        total = t1.sum().item() + t2.sum().item()
        assert abs(total - ref.item()) / ref.item() < 1e-5
        assert float((d1.cpu().double() - xt.grad).abs().max() / xt.grad.abs().max()) < 1e-4
        assert float((d2.cpu().double() - rt.grad).abs().max() / rt.grad.abs().max()) < 1e-4
        assert float(d2[torch.from_numpy(lab == R).cuda()].abs().max()) == 0.0
