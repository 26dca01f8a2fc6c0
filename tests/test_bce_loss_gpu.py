"""Multi-label sigmoid BCE losses (lirec_loss_bce_fwd_bwd, lirec_loss_bce_track_fwd_bwd; --loss bce) against
torch's binary_cross_entropy_with_logits in fp64, with the target and weight masks built independently in
numpy here; the track form's assignment against the margin loss's, bit for bit; and the whole model step
(create_model --loss bce) against the dense fp64 oracle.  The reference has no BCE, so these are the pins."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import N_CLASSES, N_RELS, TOL, make_model, oracle_forward_loss, rel_err, rounded_state_dict
from test_loss_gpu import _ragged_case
from test_model_gpu import _knife_edges

pytestmark = pytest.mark.gpu

C, R, T = 101, 15, 20
KTOL = 1e-5          # kernel vs fp64: one pass of fp32 element terms, one fixed-order sum per row / clip


def _dev(a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _bce_ref(x, target, weight):
    """Per-element weighted BCE-with-logits in fp64 (x requires grad)."""
    return F.binary_cross_entropy_with_logits(x, torch.from_numpy(target).double(),
                                              weight=torch.from_numpy(weight).double(), reduction="none")


def _row_masks(labels, C, neg_mask, pos_mask):
    rows = len(labels)
    t = np.zeros((rows, C))
    sel = labels >= 0
    t[np.flatnonzero(sel), labels[sel]] = 1
    if pos_mask is not None:
        t[pos_mask != 0] = 1
    w = np.ones((rows, C))
    if neg_mask is not None:
        w[(t == 0) & (neg_mask == 0)] = 0
    w[~sel] = 0
    t[~sel] = 0
    return t, w


def _row_case(rows, C, seed, with_neg, with_pos):
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((rows, C)) * 3).astype(np.float32)
    x[rng.random((rows, C)) < 0.02] = 100.0                  # saturated logits stay finite and exact
    x[rng.random((rows, C)) < 0.02] = -100.0
    labels = rng.integers(C, size=rows).astype(np.int32)
    labels[rng.random(rows) < 0.15] = -1                     # relationship label None
    neg = (rng.random((rows, C)) < 0.85).astype(np.uint8) if with_neg else None
    pos = (rng.random((rows, C)) < 0.05).astype(np.uint8) if with_pos else None
    return x, labels, neg, pos


@pytest.mark.parametrize("with_neg,with_pos", [(False, False), (True, False), (False, True), (True, True)])
@pytest.mark.parametrize("Cc", [C, R])
def test_row_kernel_matches_fp64_bce(with_neg, with_pos, Cc):
    from lirec_b200 import ops
    x, labels, neg, pos = _row_case(700, Cc, 11 + Cc, with_neg, with_pos)
    wide = torch.zeros(700, Cc + 27, dtype=torch.float32)    # a strided logit view: ld != C
    wide[:, :Cc] = torch.from_numpy(x)
    xd = wide.cuda()[:, :Cc]
    scale = 0.37
    loss, d = ops.loss_bce(xd, _dev(labels), _dev(neg), _dev(pos), scale)
    torch.cuda.synchronize()
    xr = torch.from_numpy(x).double().requires_grad_(True)
    t, w = _row_masks(labels, Cc, neg, pos)
    ref = scale * _bce_ref(xr, t, w).sum(1)
    ref.sum().backward()
    assert bool(torch.isfinite(loss).all()) and bool(torch.isfinite(d).all())
    assert rel_err(loss, ref) < KTOL and rel_err(d, xr.grad) < KTOL
    none = torch.from_numpy(labels < 0)
    assert bool((loss.cpu()[none] == 0).all()) and bool((d.cpu()[none] == 0).all())
    assert bool((d.cpu()[torch.from_numpy(w == 0)] == 0).all())   # left-out elements: exactly zero


def _track_ref(case, ts, pos_mask, lymbda, with_rels, tr_correct):
    """fp64 BCE of the track form from assignment ts: per-clip losses and the two logit gradients."""
    off, counts, labels, gt, ml = case["off"], case["counts"], case["labels"], case["gt"], case["multilab"]
    rl = case["rels_label"]
    B, Ni = len(counts), int(off[-1])
    ti, wi = np.zeros((Ni, C)), np.zeros((Ni, C))
    tr, wr = np.zeros((Ni, R)), np.zeros((Ni, R))
    ar = np.arange(R)
    for b in range(B):
        n, y, (g0, g1) = counts[b], labels[b], gt[b]
        r0 = rl[off[b] + g0] if g0 < n else 0
        r1 = rl[off[b] + g1] if g1 < n else 0
        live = rl[off[b] + ts[b]] != R and r0 < R
        for t in range(n):
            row = off[b] + t
            neg = ml[b] != 0
            if not tr_correct or t in (g0, g1):
                neg[y] = False
            pos = np.zeros(C, dtype=bool)
            if t == ts[b]:
                pos[y] = True
                if pos_mask is not None:
                    pos |= pos_mask[b] != 0
            ti[row], wi[row] = pos, pos | (neg & ~pos)
            lab = rl[row]
            negr = np.zeros(R, dtype=bool)
            if lab != R:
                negr = (ar != lab) if tr_correct else ((ar != r0) & (ar != r1))
            posr = np.zeros(R, dtype=bool)
            if live and t == ts[b]:
                posr[r0] = True
            tr[row], wr[row] = posr, posr | (negr & ~posr)
    xi = torch.from_numpy(case["ints"]).double().requires_grad_(True)
    per = lymbda / B * _bce_ref(xi, ti, wi).sum(1)
    xr = None
    if with_rels:
        xr = torch.from_numpy(case["rels"]).double().requires_grad_(True)
        per = per + 1.0 / B * _bce_ref(xr, tr, wr).sum(1)
    owner = torch.from_numpy(np.repeat(np.arange(B), counts))
    per_clip = torch.zeros(B, dtype=torch.float64).index_add(0, owner, per)
    per_clip.sum().backward()
    return per_clip, xi.grad, (xr.grad if with_rels else None), wi, wr


def _track_call(ops, case, pos_mask, with_rels, tr_correct, cat_distr, bce=True, seed=1234):
    lymbda = 0.7 if with_rels else 1.0
    args = (_dev(case["ints"]), _dev(case["rels"]), _dev(case["off"]), _dev(case["labels"]),
            _dev(case["rels_label"]), _dev(case["gt"]), _dev(case["multilab"]))
    kw = dict(tr_correct=tr_correct, max_slots=T, cat_distr=cat_distr, seed=seed)
    if bce:
        return ops.loss_bce_track(*args, _dev(pos_mask), lymbda, R if with_rels else 0, **kw)
    return ops.loss_track(*args, 0.101, lymbda, R if with_rels else 0, **kw)


MODES = [(False, False), (True, False), (False, True)]     # (tr_correct, cat_distr)


@pytest.mark.parametrize("tr_correct,cat_distr", MODES, ids=["argmax", "tr_correct", "cat_distr"])
@pytest.mark.parametrize("with_rels", [True, False])
@pytest.mark.parametrize("dup_ties", [False, True])
def test_track_kernel_assignment_and_values(tr_correct, cat_distr, with_rels, dup_ties):
    from lirec_b200 import ops
    case = _ragged_case(40, seed=3 if dup_ties else 4, with_rels=with_rels, dup_ties=dup_ties)
    rng = np.random.default_rng(5)
    pos_mask = (rng.random((40, C)) < 0.05).astype(np.uint8)
    for pm in (None, pos_mask):
        loss, assign, d_i, d_r = _track_call(ops, case, pm, with_rels, tr_correct, cat_distr)
        _, assign_m, _, _ = _track_call(ops, case, pm, with_rels, tr_correct, cat_distr, bce=False)
        torch.cuda.synchronize()
        assert torch.equal(assign, assign_m)                 # the margin loss's t*, bit for bit
        ts = assign.cpu().numpy()
        ref, gi, gr, wi, wr = _track_ref(case, ts, pm, 0.7 if with_rels else 1.0, with_rels, tr_correct)
        assert rel_err(loss, ref) < KTOL
        assert rel_err(d_i, gi) < KTOL
        assert bool((d_i.cpu()[torch.from_numpy(wi == 0)] == 0).all())
        if with_rels:
            assert rel_err(d_r, gr) < KTOL
            assert bool((d_r.cpu()[torch.from_numpy(wr == 0)] == 0).all())
    if dup_ties and with_rels and not (tr_correct or cat_distr):    # test_loss_gpu's tie case: slot 1 beats 2
        tied = [b for b in range(40) if case["counts"][b] >= 3]
        assert tied and any(int(assign[b]) == 1 for b in tied)


def test_kernels_are_bitwise_deterministic():
    from lirec_b200 import ops
    x, labels, neg, pos = _row_case(9000, C, 2, True, True)
    a = ops.loss_bce(_dev(x), _dev(labels), _dev(neg), _dev(pos), 1.0 / 9000)
    b = ops.loss_bce(_dev(x), _dev(labels), _dev(neg), _dev(pos), 1.0 / 9000)
    assert all(torch.equal(u, v) for u, v in zip(a, b))
    case = _ragged_case(512, seed=8)
    pm = (np.random.default_rng(1).random((512, C)) < 0.05).astype(np.uint8)
    a = _track_call(ops, case, pm, True, False, False)
    b = _track_call(ops, case, pm, True, False, False)
    assert all(torch.equal(u, v) for u, v in zip(a, b))


def test_track_kernel_refuses_max_negative():
    from lirec_b200 import _ext
    case = _ragged_case(4, seed=1)
    cfg = _ext.TrackLossCfg()
    cfg.lymbda, cfg.n_classes, cfg.n_rels, cfg.max_neg, cfg.max_slots = 1.0, C, 0, 1, T
    ints, off, lab, gt, ml = (_dev(case[k]) for k in ("ints", "off", "labels", "gt", "multilab"))
    out = torch.empty(4, device="cuda")
    asg = torch.empty(4, dtype=torch.int32, device="cuda")
    d = torch.empty_like(ints)
    rc = _ext.lib().lirec_loss_bce_track_fwd_bwd(ints.data_ptr(), None, off.data_ptr(), 4, lab.data_ptr(), None,
                                                 gt.data_ptr(), ml.data_ptr(), None, cfg, out.data_ptr(),
                                                 asg.data_ptr(), d.data_ptr(), None, _ext.stream_ptr())
    assert rc != 0 and b"max_neg" in _ext.lib().lirec_last_error()


# ---- end to end: create_model(--loss bce) against the dense fp64 oracle ------------------------------------------
def _oracle_bce(pb, ragged, extra, opt, kind, soft_pos=None):
    dense = extra["dense"]
    t = pb.tables
    ml = pb.multilab.numpy()
    B = pb.B
    if kind == "maxtracks":
        case = dict(off=t["cand_off"], counts=np.diff(t["cand_off"]), labels=t["labels"], gt=t["gt_tracks"],
                    multilab=ml, rels_label=t["rels_label"] if opt.ctx else np.zeros(pb.n_cand, dtype=np.int32))
        with_rels = bool(opt.rels_multitask)
        ts = extra["assignment"].numpy()
        lymbda = opt.lymbda if with_rels else 1.0
        # the same masks as _track_ref, applied to the oracle's (graph-connected) ragged logits
        rl = case["rels_label"]
        Ni = pb.n_cand
        ti, wi, tr, wr = np.zeros((Ni, C)), np.zeros((Ni, C)), np.zeros((Ni, R)), np.zeros((Ni, R))
        case["ints"] = np.zeros((Ni, C), dtype=np.float32)
        case["rels"] = np.zeros((Ni, R), dtype=np.float32)
        _, _, _, wi, wr = _track_ref(case, ts, soft_pos, lymbda, with_rels, bool(opt.tr_correct))
        # targets: (t*, y) (+ soft positives) and (t*, r0) when live
        for b in range(B):
            row = int(t["cand_off"][b]) + int(ts[b])
            ti[row, int(t["labels"][b])] = 1
            if soft_pos is not None:
                ti[row, soft_pos[b] != 0] = 1
            if with_rels:
                g0 = int(t["gt_tracks"][b, 0])
                n = int(case["counts"][b])
                r0 = int(rl[int(t["cand_off"][b]) + g0]) if g0 < n else 0
                if rl[row] != R and r0 < R:
                    tr[row, r0] = 1
        l = lymbda / B * _bce_ref(ragged["inters"], ti, wi).sum()
        if with_rels:
            l = l + 1.0 / B * _bce_ref(ragged["rels"], tr, wr).sum()
        return l
    labels = t["labels"].astype(np.int64)
    l = 0.0
    if kind == "modalities" or opt.ints:
        ti, wi = _row_masks(labels, C, ml, soft_pos)
        w = (opt.lymbda if kind == "midfusion" else 1.0) / B
        l = l + w * _bce_ref(ragged["inters"], ti, wi).sum()
    if kind == "midfusion" and opt.ctx:
        rlab = dense["rels_label"].reshape(B).numpy().astype(np.int64)
        sel = np.where(rlab != N_RELS, rlab, -1)
        tr, wr = _row_masks(sel, R, None, None)
        l = l + 1.0 / int((sel >= 0).sum()) * _bce_ref(ragged["rels"], tr, wr).sum()
    return l


def _run_bce(preset, opt, B, seed, train, pb=None, n_classes=N_CLASSES):
    from lirec_b200.mixed_utils import synthetic
    from oracle import dropout as odrop
    kind = synthetic.PRESETS[preset]["kind"]
    model, loss_fn, _ = make_model(n_classes=n_classes)
    model.train(train)
    pb = pb if pb is not None else synthetic.make_batch(B, seed=seed, preset=preset)
    pbd = pb.to_device("cuda")
    soft = pb.soft_pos.numpy() if (opt.soft_gt and pb.soft_pos is not None) else None
    step_seed = 1000 + seed
    for _ in range(8):
        for p in model.parameters():
            p.grad = None
        out = model(pbd, seed=step_seed)
        lv = loss_fn(out, {})
        lv.backward()
        torch.cuda.synchronize()
        sd = rounded_state_dict(model)
        cw = model.out_ints.in_features if model.kind == "modalities" else None
        masks = odrop.dense_masks(pb, step_seed, opt.dropout, cat_width=cw) if train else None
        tape = {}
        ragged, _, extra = oracle_forward_loss(pb, sd, preset, opt, masks, tape=tape)
        l = _oracle_bce(pb, ragged, extra, opt, kind, soft)
        l.backward()
        bad = _knife_edges(tape)
        if not bad:
            break
        named = dict(model.named_parameters())
        with torch.no_grad():
            for pname, cols in bad.items():
                named[pname][cols] += 1e-3
    else:
        pytest.fail("could not move the oracle off its ReLU knife-edges")
    return model, loss_fn, out, lv, sd, l, extra


def _check(model, lv, sd, l):
    assert abs(lv.item() - l.item()) / abs(l.item()) < TOL
    for k, p in model.named_parameters():
        assert p.grad is not None, k
        assert rel_err(p.grad, sd[k].grad) < TOL, (k, rel_err(p.grad, sd[k].grad))


@pytest.mark.parametrize("train", [False, True])
@pytest.mark.parametrize("preset", ["modalities", "int_rels", "int_ch", "int_rel_ch"])
def test_bce_end_to_end_parity(preset, train, opt_preset):
    import lirec_b200.mlp.model as M
    opt = opt_preset(preset, loss="bce")
    for seed in (3, 4):
        model, loss_fn, out, lv, sd, l, extra = _run_bce(preset, opt, 6, seed, train)
        want = M.TrackBCELoss if opt.tr_maximize else M.MultiLabelBCELoss
        assert type(loss_fn) is want and loss_fn.n_rels == (N_RELS if opt.rels_multitask else 0)
        if "assignment" in extra:
            assert torch.equal(loss_fn.last_assignment.cpu().long(), extra["assignment"])
        _check(model, lv, sd, l)


@pytest.mark.parametrize("train", [False, True])
def test_relationship_only_model_bce(train, opt_preset):
    opt = opt_preset("int_rels", ints=0, gates=0, loss="bce")
    for seed in (3, 4):
        model, loss_fn, out, lv, sd, l, extra = _run_bce("int_rels", opt, 6, seed, train)
        assert out.ragged_inters is None
        _check(model, lv, sd, l)


def test_soft_positives_end_to_end(opt_preset):
    """--soft_gt on the annotation world: the co-occurring interactions are BCE targets of the modalities model."""
    from lirec_b200.mixed_utils import indexed_dataset as ids, synthetic_world as sw
    import lirec_b200.mlp.model as M
    opt = opt_preset("modalities", loss="bce", soft_gt=True, inter_class="all", merged=True, multilab_weights=True,
                     rels=False)
    world = sw.build_world(3, n_movies=3, n_scenes=10, n_inter_names=60, n_merged=101)
    ds = ids.IndexedMixedFeaturesDataset(sw.subset(world, "train"), world, mode="train")
    ds.cache()
    np.random.seed(0)
    records = [ds[i] for i in range(len(ds))]
    n_soft = [int((np.asarray(r["soft_labels"]) >= 0).sum()) for r in records]
    pick = [records[i] for i in np.argsort(n_soft, kind="stable")[::-1][:6]]
    pb = ids.collate_indexed(pick, ds)
    assert pb.soft_pos is not None and int(pb.soft_pos.sum()) > 6   # extra positives beyond the labels
    for train in (False, True):
        model, loss_fn, out, lv, sd, l, extra = _run_bce("modalities", opt, 6, 3, train, pb=pb,
                                                         n_classes=ds.n_classes)
        _check(model, lv, sd, l)
    # the same batch without its soft labels is refused, not trained on the hard labels
    pb.soft_pos = None
    with pytest.raises(RuntimeError, match="soft labels"):
        loss_fn(model(pb.to_device("cuda")), {})
    # and the soft positives do change the loss
    opt.soft_gt = False
    model.eval()
    hard = loss_fn(model(ids.collate_indexed(pick, ds).to_device("cuda")), {})
    opt.soft_gt = True
    soft = loss_fn(model(ids.collate_indexed(pick, ds).to_device("cuda")), {})
    assert hard.item() != soft.item()
    assert isinstance(loss_fn, M.MultiLabelBCELoss)


@pytest.mark.parametrize("preset", ["modalities", "int_rels", "int_ch", "int_rel_ch"])
def test_native_train_step_equals_autograd_path_bce(opt_preset, preset):
    from lirec_b200.mixed_utils import synthetic
    import lirec_b200.mlp.model as M
    opt_preset(preset, fused_adam=1, lr=1e-3, loss="bce")
    pb = synthetic.make_batch(12, seed=9, preset=preset).to_device("cuda")
    model, loss, optimizer = make_model(seed=5)
    model.train()
    lv = loss(model(pb, seed=77), {})
    optimizer.zero_grad()
    lv.backward()
    ref = {k: p.grad.clone() for k, p in model.named_parameters()}
    model._flat_grad.fill_(float("nan"))
    lv2 = M.train_step(model, loss, pb, seed=77)
    assert not lv2.requires_grad and torch.equal(lv.detach(), lv2)
    for k, p in model.named_parameters():
        assert p.grad is not None and torch.equal(p.grad, ref[k]), k


def test_ce_selection_end_to_end(opt_preset):
    """--loss ce on int_rels selects MultiTaskCrossEntropyLoss; one step matches the oracle."""
    import lirec_b200.mlp.model as M
    from lirec_b200.mixed_utils import synthetic
    from oracle import losses as ol, model as om
    opt_preset("int_rels", dropout=0.0, loss="ce")
    model, loss_fn, _ = make_model()
    assert type(loss_fn) is M.MultiTaskCrossEntropyLoss and loss_fn.n_rels == N_RELS and loss_fn.weights is None
    model.eval()
    pb = synthetic.make_batch(12, seed=9, preset="int_rels")
    lv = loss_fn(model(pb.to_device("cuda")), {})
    lv.backward()
    sd = rounded_state_dict(model)
    dense = pb.to_dense(np.float64)
    B, f = pb.B, dense["features"]
    o = om.midfusion_forward(sd, f.reshape(B, -1, f.shape[-1]), dense["rels_mask"].reshape(B, -1, 1),
                             om.default_cfg(ctx=1, gates=1, dropout=0.0), None)
    ref = ol.multitask_ce(o["inters"], o["rels"], dense["labels"].reshape(B), dense["rels_label"].reshape(B), N_RELS)
    ref.backward()
    assert abs(lv.item() - ref.item()) / abs(ref.item()) < TOL
    assert max(rel_err(p.grad, sd[k].grad) for k, p in model.named_parameters()) < TOL
