"""Host side of the multi-label BCE losses (--loss bce): flag parsing and loss selection, the refusals
create_model raises before any device work, the soft-label positives (--soft_gt) every batch path carries,
and the collectives an EmptyShard rank issues for MultiLabelBCELoss under data parallelism."""
import glob
import json
import os
import pickle

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
MODALITIES_GOLDEN = sorted(glob.glob(os.path.join(HERE, "golden", "dataloader_modalities_*.npz")))


# ---- flags and selection -------------------------------------------------------------------------------------
def test_loss_flag_parses_and_defaults_to_margin():
    from lirec_b200.utils.arg_pars import build_parser
    p = build_parser()
    assert p.parse_args([]).loss == "margin"
    for k in ("margin", "bce", "ce"):
        assert p.parse_args(["--loss", k]).loss == k
    with pytest.raises(SystemExit):
        p.parse_args(["--loss", "focal"])


@pytest.mark.parametrize("preset,over,match", [
    ("int_ch", dict(loss="ce"), "track-assignment"),
    ("int_rel_ch", dict(loss="ce"), "track-assignment"),
    ("int_ch", dict(loss="bce", tr_max_neg=True), "max-negative"),
    ("int_rels", dict(loss="bce", tr_max_neg=True), "max-negative"),
    ("int_rels", dict(loss="ce", ints=0, gates=0), "interaction logits"),
    ("int_rels", dict(loss="hinge"), "margin, bce or ce"),
])
def test_create_model_refuses_unsupported_loss_combinations(opt_preset, preset, over, match):
    """The refusals come before the device check and before any model is built (device='cpu' would raise a
    different error if they did not)."""
    from lirec_b200.mlp import model as M
    opt_preset(preset, device="cpu", **over)
    with pytest.raises(ValueError, match=match):
        M.create_model(101, n_rels=15)


@pytest.mark.parametrize("preset,over", [
    ("modalities", dict(loss="ce", ints=0)),          # Modalities always has its interaction head
    ("int_rels", dict(loss="bce")),
    ("int_ch", dict(loss="bce")),
    ("int_rels", dict(loss="margin", tr_max_neg=True)),
])
def test_supported_loss_combinations_reach_the_device_check(opt_preset, preset, over):
    from lirec_b200.mlp import model as M
    opt_preset(preset, device="cpu", **over)
    with pytest.raises(RuntimeError, match="B200 only"):
        M.create_model(101, n_rels=15)


# ---- soft positives on the host ------------------------------------------------------------------------------
def _dataset(opt, g, mode, soft_gt):
    from lirec_b200.mixed_utils import indexed_dataset as ids
    from lirec_b200.mixed_utils import synthetic_world as sw
    for k, v in dict(mod_check=True, tr_maximize=False, ints=1, ctx=0, gates=0, rels_multitask=False,
                     rels_multi_clip=False, tracks=True, rels=False, inter_class="all", merged=True,
                     multilab_weights=True, soft_gt=soft_gt).items():
        setattr(opt, k, v)
    opt.rels_n_clips = int(g["rels_n_clips"])
    world = sw.build_world(int(g["world_seed"]), **json.loads(str(g["world_kwargs"])))
    ds = ids.IndexedMixedFeaturesDataset(sw.subset(world, mode), world, mode=mode)
    ds.cache()
    return ds


def _records(ds, g):
    np.random.seed(int(g["numpy_seed"]))
    return [ds[i] for i in range(len(ds))]


def _expected_soft_pos(records, C):
    out = np.zeros((len(records), C), dtype=np.uint8)
    for i, r in enumerate(records):
        for v in np.asarray(r["soft_labels"]).reshape(-1):
            if v >= 0:
                out[i, int(v)] = 1
    return out


class _NoPin:
    """Pinning needs CUDA: a plain copy stands in for it on a CPU-only machine."""

    def __enter__(self):
        self.orig = torch.Tensor.pin_memory
        torch.Tensor.pin_memory = lambda t, *a, **k: t.clone()

    def __exit__(self, *exc):
        torch.Tensor.pin_memory = self.orig


def test_modalities_golden_files_present():
    assert len(MODALITIES_GOLDEN) == 2


@pytest.mark.parametrize("path", MODALITIES_GOLDEN, ids=[os.path.basename(p)[11:-4] for p in MODALITIES_GOLDEN])
def test_soft_pos_is_the_multi_hot_of_the_soft_labels(path, opt_preset):
    from lirec_b200.utils.arg_pars import opt
    from lirec_b200.mixed_utils import indexed_dataset as ids
    from lirec_b200.mixed_utils.classification_dataloader import _PinnedRing
    from lirec_b200.packing import pack_dense_batch
    g = np.load(path, allow_pickle=False)
    ds = _dataset(opt, g, "train" if "_train_" in path else "test", soft_gt=True)
    records = _records(ds, g)
    # the records' soft labels are the reference dataloader's (tests/golden: item_soft_labels)
    assert np.array_equal(np.stack([r["soft_labels"] for r in records]), g["item_soft_labels"])
    want = _expected_soft_pos(records, ds.n_classes)
    assert want.sum() > len(records)                          # some clips do have co-occurring interactions
    assert all(want[i, r["labels"]] == 1 for i, r in enumerate(records))
    for resident in (False, True):
        pn = ids.collate_indexed(records, ds, resident=resident)
        pr = ids.collate_indexed_numpy(records, ds, resident=resident)
        for pb in (pn, pr):
            assert pb.soft_pos.dtype == torch.uint8 and np.array_equal(pb.soft_pos.numpy(), want)
    # dense reference batch -> compatibility packing
    dense = {"features": torch.zeros(len(records), 1, 6912), "labels": torch.tensor([r["labels"] for r in records]),
             "multilab_weights": torch.ones(len(records), ds.n_classes),
             "soft_labels": torch.from_numpy(np.stack([r["soft_labels"] for r in records]))}
    assert np.array_equal(pack_dense_batch(dense, "modalities").soft_pos.numpy(), want)
    # across the loader-worker pipe
    back = pickle.loads(pickle.dumps(ids.collate_indexed(records, ds)))
    assert np.array_equal(back.soft_pos.numpy(), want)
    # pinned staging: one ring slot holds multilab then soft_pos, as two views
    ring, pb = _PinnedRing(slots=2), ids.collate_indexed(records, ds)
    ml = pb.multilab.clone()
    with _NoPin():
        ring.stage(pb, None)
        pb2 = ids.collate_indexed(records, ds).pin()
    assert torch.equal(pb.multilab, ml) and np.array_equal(pb.soft_pos.numpy(), want)
    k = ring._last
    assert pb.multilab.data_ptr() == ring.ml[k].data_ptr()
    assert pb.soft_pos.data_ptr() == ring.ml[k].data_ptr() + ml.numel()
    assert np.array_equal(pb2.soft_pos.numpy(), want)


@pytest.mark.parametrize("path", MODALITIES_GOLDEN, ids=[os.path.basename(p)[11:-4] for p in MODALITIES_GOLDEN])
def test_batches_without_soft_gt_are_unchanged(path, opt_preset):
    """--soft_gt off: no soft_pos, and the arena and multilab bytes are exactly those of the same records
    collated with the soft labels present (which only add soft_pos)."""
    from lirec_b200.utils.arg_pars import opt
    from lirec_b200.mixed_utils import indexed_dataset as ids
    from lirec_b200.mixed_utils.classification_dataloader import _PinnedRing
    g = np.load(path, allow_pickle=False)
    mode = "train" if "_train_" in path else "test"
    ds_soft = _dataset(opt, g, mode, soft_gt=True)
    with_soft = ids.collate_indexed(_records(ds_soft, g), ds_soft)
    ds = _dataset(opt, g, mode, soft_gt=False)
    records = _records(ds, g)
    assert "soft_labels" not in records[0]
    for pb in (ids.collate_indexed(records, ds), ids.collate_indexed_numpy(records, ds)):
        assert pb.soft_pos is None
        assert torch.equal(pb.multilab, with_soft.multilab)
    pb = ids.collate_indexed(records, ds)
    assert pb._host_arena.tobytes() == with_soft._host_arena.tobytes()
    assert pickle.loads(pickle.dumps(pb)).soft_pos is None
    ring = _PinnedRing(slots=2)
    with _NoPin():
        ring.stage(pb, None)
    assert pb.soft_pos is None and pb.multilab.numel() == with_soft.multilab.numel()
    assert bytes(pb.multilab.numpy().tobytes()) == bytes(with_soft.multilab.numpy().tobytes())


def test_bce_losses_refuse_batches_without_soft_labels(opt_preset):
    from lirec_b200.mlp import model as M
    from lirec_b200.packing import PackedBatch
    opt_preset("modalities", soft_gt=True)
    with pytest.raises(RuntimeError, match="soft labels"):
        M._soft_pos(PackedBatch())
    opt_preset("modalities", soft_gt=False)
    assert M._soft_pos(PackedBatch()) is None


# ---- empty shards ----------------------------------------------------------------------------------------------
def _empty_shard_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    import sys
    sys.argv = sys.argv[:1]
    from types import SimpleNamespace
    from lirec_b200 import dp
    from lirec_b200.mlp import model as M
    from lirec_b200.utils.arg_pars import opt
    dp.init_from_env(backend="gloo")
    opt.ctx, opt.ints = 1, 1
    loss = M.MultiLabelBCELoss(n_rels=15)
    loss._dp_world = world
    if rank == 0:          # holds clips: the relationship term's one all_reduce of the labelled-row count
        pb = SimpleNamespace(device="cpu", B=3, host=SimpleNamespace(global_clips=3))
        t, d = M._rel_term(loss, pb, 2, lambda s: (torch.ones(3) * s, torch.ones(3) * s))
        ok = t is not None and abs(float(t.sum()) - 1.5) < 1e-6    # 3 rows x (3 / 3) / (2 + 0 labelled rows)
    else:                  # an EmptyShard this step
        M.dp_empty_shard_collectives(loss, torch.device("cpu"))
        ok = True
    # if the ranks' collectives were unpaired, this marker would meet the count all_reduce instead
    marker = torch.tensor([float(10 * (rank + 1))])
    dist.all_reduce(marker)
    q.put((rank, ok, float(marker)))
    dist.destroy_process_group()


def test_empty_shard_issues_the_bce_relationship_collective():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 33500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_empty_shard_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=180) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, ok, marker in res:
        assert ok and marker == 30.0, (rank, ok, marker)


def test_empty_shard_collectives_follow_the_relationship_term(opt_preset, monkeypatch):
    """Each multi-task loss issues the relationship all_reduce exactly when its relationship term runs."""
    from lirec_b200.mlp import model as M
    calls = []
    monkeypatch.setattr(dist, "all_reduce", lambda t, *a, **k: calls.append(t.numel()))
    opt_preset("int_rels")
    for loss, n in ((M.MultiLabelBCELoss(n_rels=15), 1), (M.MultiLabelBCELoss(), 0), (M.MultiTaskMaxMargin(15), 1),
                    (M.MaxMarginCrossEntropyLoss(), 0)):
        calls.clear()
        loss._dp_world = 2
        M.dp_empty_shard_collectives(loss, torch.device("cpu"))
        assert len(calls) == n, type(loss).__name__
    ce = M.MultiTaskCrossEntropyLoss(101, n_rels=15)
    ce._dp_world = 2
    calls.clear()
    M.dp_empty_shard_collectives(ce, torch.device("cpu"))
    assert len(calls) == 1
    for preset, over in (("int_rels", dict(ctx=0)), ("modalities", {})):   # no relationship logits: no collective
        opt_preset(preset, **over)
        for loss in (M.MultiLabelBCELoss(n_rels=15), M.MultiTaskCrossEntropyLoss(101)):
            calls.clear()
            loss._dp_world = 2
            M.dp_empty_shard_collectives(loss, torch.device("cpu"))
            assert calls == [], (preset, type(loss).__name__)
