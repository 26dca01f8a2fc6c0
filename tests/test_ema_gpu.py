"""Exponential moving average of the weights on the B200 (lirec_ema_update_flat, lirec_ema_swap_flat, FlatEMA,
--ema_decay): the kernels against fp64 and against torch.lerp, determinism, refusals, the swap and its bf16 shadow,
FlatEMA against torch.optim.swa_utils.AveragedModel on real steps, training left unchanged, evaluation of the
average, checkpoints and resume, and data parallelism."""
import contextlib
import io
import os
import subprocess
import sys

import pytest
import torch

from helpers import make_model

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SENTINEL = 12345.0
SIZES = [1, 3, 4, 5, 63, 64, 65, 4 * 524_288 + 3, 4 * 1_048_577 + 3, 9_437_187]
DECAYS = [0.5, 0.9, 0.999, 0.9999]


def _ulps(a, b):
    """Elementwise distance in units in the last place between two finite float32 tensors."""
    def key(x):
        i = x.contiguous().view(torch.int32).to(torch.int64)
        return torch.where(i < 0, -(i & 0x7FFFFFFF), i)
    return (key(a) - key(b)).abs()


def _padded(n, fill, gen=None):
    """A float32 buffer of n values (randn, or `fill`) followed by 9 sentinels; returns (buffer, view of n)."""
    buf = torch.full((n + 9,), SENTINEL, device="cuda")
    buf[:n] = torch.randn(n, generator=gen, device="cuda") if fill is None else fill
    return buf, buf[:n]


@pytest.mark.parametrize("n", SIZES)
def test_update_matches_torch_lerp_and_fp64(n):
    from lirec_b200 import ops
    gen = torch.Generator(device="cuda").manual_seed(n)
    for decay in DECAYS:
        buf, ema = _padded(n, None, gen)
        ref = ema.clone()
        e64 = ema.double()
        wmax = 0.0
        for _ in range(20):
            w = torch.randn(n, generator=gen, device="cuda") * 2.0 + 0.5
            wmax = max(wmax, float(w.abs().max()))
            ops.ema_update_flat(ema, w, decay)
            torch._foreach_lerp_([ref], [w], 1 - decay)
            e64 = e64 + (1 - decay) * (w.double() - e64)
        torch.cuda.synchronize()
        assert int(_ulps(ema, ref).max()) <= 1, (n, decay)
        # fp64 statement: 20 updates, each within ~1 ulp of the operands' magnitude
        scale = float(e64.abs().max()) + wmax
        assert float((ema.double() - e64).abs().max()) <= 20 * 2.0 ** -23 * scale, (n, decay)
        assert bool((buf[n:] == SENTINEL).all()), (n, decay)


@pytest.mark.parametrize("decay", [0.9, 0.3])
def test_non_finite_values_propagate_like_torch_lerp(decay):
    from lirec_b200 import ops
    special = [float("nan"), float("inf"), float("-inf"), 0.0, 1.0, -3.0]
    e = torch.tensor([a for a in special for _ in special] * 3, device="cuda")   # every pair, bulk and tail
    w = torch.tensor([b for _ in special for b in special] * 3, device="cuda")
    e, w = e[:107], w[:107]
    want = torch.lerp(e, w, 1 - decay)
    got = e.clone()
    ops.ema_update_flat(got, w, decay)
    torch.testing.assert_close(got, want, rtol=0, atol=0, equal_nan=True)
    assert torch.equal(torch.isnan(got), torch.isnan(want))


def test_update_is_bitwise_reproducible_and_reads_param_only():
    from lirec_b200 import ops
    gen = torch.Generator(device="cuda").manual_seed(3)
    e0 = torch.randn(4 * 1_000_003 + 1, generator=gen, device="cuda")
    w = torch.randn(e0.numel(), generator=gen, device="cuda")
    w0 = w.clone()
    outs = []
    for _ in range(2):
        e = e0.clone()
        for _ in range(5):
            ops.ema_update_flat(e, w, 0.999)
        outs.append(e)
    assert torch.equal(outs[0], outs[1])
    assert torch.equal(w, w0)


def test_refusals_return_an_error_and_launch_nothing():
    from lirec_b200 import _ext, ops
    L = _ext.lib()
    buf = torch.randn(1029, device="cuda")
    w = torch.randn(1029, device="cuda")
    bf = torch.zeros(1029, dtype=torch.bfloat16, device="cuda")
    before = buf.clone()
    for bad in (0.0, 1.0, -0.5, 1.5, float("nan"), float("inf")):          # 1 - decay outside (0, 1)
        with pytest.raises(RuntimeError, match="one_minus_decay"):
            ops.ema_update_flat(buf, w, bad)
        assert L.lirec_last_launch_count() == 0
    with pytest.raises(RuntimeError, match="16-byte aligned"):
        ops.ema_update_flat(buf[1:], w[1:], 0.9)
    with pytest.raises(RuntimeError, match="16-byte aligned"):
        ops.ema_swap_flat(buf[1:], w[1:])
    with pytest.raises(RuntimeError, match="16-byte aligned"):
        ops.ema_swap_flat(buf[:1028], w[:1028], bf[1:])
    with pytest.raises(ValueError, match="float32"):
        ops.ema_update_flat(buf.double(), w, 0.9)
    with pytest.raises(ValueError, match="one size"):
        ops.ema_swap_flat(buf, w[:-4])
    with pytest.raises(ValueError, match="bfloat16"):
        ops.ema_swap_flat(buf, w, bf.float())
    p, e, s = buf.data_ptr(), w.data_ptr(), torch.cuda.current_stream().cuda_stream
    for args in ((None, e, 1029, 0.1, s), (p, None, 1029, 0.1, s), (p, e, -1, 0.1, s)):
        assert L.lirec_ema_update_flat(*args) != 0
        assert L.lirec_last_launch_count() == 0
    for args in ((None, e, None, 1029, s), (p, None, None, 1029, s), (p, e, None, -1, s)):
        assert L.lirec_ema_swap_flat(*args) != 0
        assert L.lirec_last_launch_count() == 0
    assert L.lirec_ema_update_flat(p, e, 0, 0.1, s) == 0 and L.lirec_last_launch_count() == 0
    assert L.lirec_ema_swap_flat(p, e, bf.data_ptr(), 0, s) == 0 and L.lirec_last_launch_count() == 0
    torch.cuda.synchronize()
    assert torch.equal(buf, before)


@pytest.mark.parametrize("n", [5, 4 * 262_144 + 3, 9_437_187])
def test_swap_exchanges_refreshes_the_shadow_and_undoes_itself(n):
    from lirec_b200 import ops
    gen = torch.Generator(device="cuda").manual_seed(n)
    pbuf, p = _padded(n, None, gen)
    ebuf, e = _padded(n, None, gen)
    bbuf = torch.full((n + 9,), SENTINEL, dtype=torch.bfloat16, device="cuda")
    b = bbuf[:n]
    ops.cast_bf16(p, b)
    p0, e0, b0 = pbuf.clone(), ebuf.clone(), bbuf.clone()
    ops.ema_swap_flat(p, e, b)
    want = torch.empty_like(b)
    ops.cast_bf16(e0[:n], want)
    torch.cuda.synchronize()
    assert torch.equal(p, e0[:n]) and torch.equal(e, p0[:n])
    assert torch.equal(b.view(torch.int16), want.view(torch.int16))
    ops.ema_swap_flat(p, e, b)
    torch.cuda.synchronize()
    assert torch.equal(pbuf, p0) and torch.equal(ebuf, e0)
    assert torch.equal(bbuf.view(torch.int16), b0.view(torch.int16))          # sentinels after n included
    ops.ema_swap_flat(p, e)                                                    # no shadow: only the fp32 buffers
    torch.cuda.synchronize()
    assert torch.equal(p, e0[:n]) and torch.equal(e, p0[:n])
    assert torch.equal(bbuf.view(torch.int16), b0.view(torch.int16))
    assert bool((pbuf[n:] == SENTINEL).all()) and bool((ebuf[n:] == SENTINEL).all())


# ---- FlatEMA on real training steps -----------------------------------------------------------------------------
def _setup(opt_preset, preset, kind, seed=9, **over):
    settings = dict(fused_adam=int(kind == "flat_adam"), optimizer="lamb" if kind == "flat_lamb" else "adam",
                    lr=1e-3, weight_decay=0.01 if kind == "flat_lamb" else 0.0)
    settings.update(over)
    opt_preset(preset, **settings)
    model, loss, optimizer = make_model(seed=seed)
    model.train()
    return model, loss, optimizer


def _batch(preset, s):
    from lirec_b200.mixed_utils import synthetic
    return synthetic.make_batch(16, seed=60 + s, preset=preset).to_device("cuda")


class _Holder(torch.nn.Module):
    """Detached copies of a model's parameters, for AveragedModel (which deep-copies what it averages)."""

    def __init__(self, model):
        super().__init__()
        self.ps = torch.nn.ParameterList([torch.nn.Parameter(p.detach().clone()) for p in model.parameters()])

    @torch.no_grad()
    def load(self, model):
        for q, p in zip(self.ps, model.parameters()):
            q.copy_(p)


@pytest.mark.parametrize("preset", ["int_rel_ch", "int_rels"])
@pytest.mark.parametrize("kind", ["torch_adam", "flat_adam", "flat_lamb"])
def test_flat_ema_matches_averaged_model(opt_preset, preset, kind):
    from torch.optim.swa_utils import AveragedModel, get_ema_multi_avg_fn
    import lirec_b200.mlp.model as M
    import lirec_b200.mlp.train as TR
    decay = 0.9
    model, loss, optimizer = _setup(opt_preset, preset, kind)
    ema = M.FlatEMA(model, decay)
    holder = _Holder(model)
    ref = AveragedModel(holder, multi_avg_fn=get_ema_multi_avg_fn(decay))
    for s in range(5):
        TR.train_step(model, loss, optimizer, _batch(preset, s), 1, None, 0.0, ema)
        holder.load(model)
        ref.update_parameters(holder)
    torch.cuda.synchronize()
    assert ema.n_averaged == 5 == int(ref.n_averaged)
    avg = ema.state_dict()["state_dict"]
    names = [n for n, _ in model.named_parameters()]
    assert list(avg) == list(model.state_dict())
    for name, q in zip(names, ref.module.ps):
        assert avg[name].shape == q.shape, name
        assert int(_ulps(avg[name].cuda(), q.detach()).max()) <= 1, name
    assert not torch.equal(avg[names[0]].cuda(), next(model.parameters()).detach())    # it is an average


def _run(opt_preset, kind, steps, with_ema, **over):
    """`steps` steps of mlp.train.train_step; returns per-step (loss, flat grad, launches) and the model."""
    from lirec_b200 import _ext, dp
    import lirec_b200.mlp.model as M
    import lirec_b200.mlp.train as TR
    model, loss, optimizer = _setup(opt_preset, "int_rel_ch", kind, **over)
    max_norm = float(over.get("clip_grad_norm", 0.0))
    fused = None
    if over.get("overlap_adam"):
        fused = dp.SwitchReduceAdam.attach(model, optimizer, single_gpu=True)
        assert fused is not None
    ema = M.FlatEMA(model, 0.999) if with_ema else None
    trace = []
    for s in range(steps):
        c0 = _ext.launch_counter
        lv = TR.train_step(model, loss, optimizer, _batch("int_rel_ch", s), 1, fused, max_norm, ema)
        torch.cuda.synchronize()
        trace.append((lv.detach().clone(), model._flat_grad.clone(), _ext.launch_counter - c0))
    return trace, model, ema, fused


@pytest.mark.parametrize("kind,over", [("flat_adam", dict(overlap_adam=1)), ("flat_lamb", {}),
                                       ("torch_adam", dict(clip_grad_norm=1e-3))])
def test_ema_does_not_change_training(opt_preset, kind, over):
    off, m_off, _, f_off = _run(opt_preset, kind, 4, False, **over)
    w_off = m_off._flat.clone()
    if f_off is not None:
        f_off.detach()
    on, m_on, ema, f_on = _run(opt_preset, kind, 4, True, **over)
    assert ema.n_averaged == 4
    for s, ((l0, g0, n0), (l1, g1, n1)) in enumerate(zip(off, on)):
        assert torch.equal(l0, l1) and torch.equal(g0, g1), s
        assert n1 == n0 + (1 if s else 0), (s, n0, n1)       # the first update is a copy, then one launch a step
    assert torch.equal(w_off, m_on._flat)
    if f_on is not None:
        f_on.detach()


def _val_dataset(opt_preset, monkeypatch, tmp_path, **over):
    settings = dict(synthetic=1, epochs=1, batch_size=16, num_workers=0, test=True, test_fr=1, save_model=True,
                    save_model_often=True, store_root=str(tmp_path), resume=False, resume_train=False, fused_adam=1,
                    overlap_adam=0, optimizer="adam", dp=0, lr=1e-3, tr_sum_max=False, rels_multi_clip=True,
                    ema_decay=0.0)
    settings.update(over)
    opt = opt_preset("int_rel_ch", **settings)
    from lirec_b200.mixed_utils import classification_dataloader as cd
    monkeypatch.setattr(cd.SyntheticClipsDataset, "SIZES", {"train": 48, "val": 24, "test": 24})
    return opt, cd


def test_evaluating_the_average_restores_the_model(opt_preset, monkeypatch, tmp_path):
    import lirec_b200.mlp.model as M
    import lirec_b200.mlp.test as T
    import lirec_b200.mlp.train as TR
    _, cd = _val_dataset(opt_preset, monkeypatch, tmp_path)
    val_ds = cd.MixedFeaturesDataset("val").cache().init_relships()
    n_rels = len(val_ds.rels_list) - 1

    def run(evaluate):
        torch.manual_seed(4)
        with contextlib.redirect_stdout(io.StringIO()):
            model, loss, optimizer = M.create_model(val_ds.n_classes, n_rels=n_rels)
        model.train()
        ema = M.FlatEMA(model, 0.9)
        metrics = None
        for s in range(5):
            if s == 3 and evaluate:
                w, b = model._flat.clone(), model._flat_bf16.clone()
                with contextlib.redirect_stdout(io.StringIO()), ema.applied():
                    metrics = T.testing(val_ds, model, loss, mode="val")
                assert torch.equal(model._flat, w) and torch.equal(model._flat_bf16.view(torch.int16),
                                                                   b.view(torch.int16))
                model.train()
            TR.train_step(model, loss, optimizer, _batch("int_rel_ch", s), 1, None, 0.0, ema)
        torch.cuda.synchronize()
        return model, ema, metrics

    m_eval, ema_eval, metrics = run(True)
    m_plain, ema_plain, _ = run(False)
    assert torch.equal(m_eval._flat, m_plain._flat) and torch.equal(ema_eval._ema, ema_plain._ema)

    # the metrics of the average equal those of a plain model loaded with it (after 3 steps)
    torch.manual_seed(4)
    with contextlib.redirect_stdout(io.StringIO()):
        model, loss, optimizer = M.create_model(val_ds.n_classes, n_rels=n_rels)
    ema = M.FlatEMA(model, 0.9)
    model.train()
    for s in range(3):
        TR.train_step(model, loss, optimizer, _batch("int_rel_ch", s), 1, None, 0.0, ema)
    with contextlib.redirect_stdout(io.StringIO()):
        fresh, loss2, _ = M.create_model(val_ds.n_classes, n_rels=n_rels)
        fresh.load_state_dict(ema.state_dict()["state_dict"])
        want = T.testing(val_ds, fresh, loss2, mode="val")
    assert metrics == want


def test_checkpoints_carry_the_average_and_resume_from_it(opt_preset, monkeypatch, tmp_path):
    from lirec_b200.resume import _common
    import lirec_b200.mlp.model as M
    import lirec_b200.mlp.test as T
    import lirec_b200.mlp.train as TR
    opt, cd = _val_dataset(opt_preset, monkeypatch, tmp_path, ema_decay=0.9)
    train_ds = cd.MixedFeaturesDataset("train").cache().init_relships()
    val_ds = cd.MixedFeaturesDataset("val").cache().init_relships()
    n_classes, n_rels = train_ds.n_classes, len(train_ds.rels_list) - 1
    torch.manual_seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        model, loss, optimizer = M.create_model(n_classes, n_rels=n_rels)
        TR.training(train_ds, model=model, loss=loss, optimizer=optimizer, name="t", val_dataset=val_ds)
    path = opt.resume_str
    ckpt = torch.load(path, map_location="cpu")
    assert set(ckpt) == {"epoch", "state_dict", "optimizer", "ema"}
    live = model.state_dict()
    assert all(torch.equal(ckpt["state_dict"][k], v.cpu()) for k, v in live.items())
    st = ckpt["ema"]
    assert st["decay"] == 0.9 and st["n_averaged"] >= 2
    assert list(st["state_dict"]) == list(live)
    assert all(st["state_dict"][k].shape == v.shape for k, v in live.items())
    assert any(not torch.equal(st["state_dict"][k], v.cpu()) for k, v in live.items())
    saved = [os.path.join(d, f) for d, _, fs in os.walk(str(tmp_path)) for f in fs if d != str(tmp_path)]
    assert saved and all("ema" in torch.load(f, map_location="cpu") for f in saved)

    # --resume_train: the average and n_averaged come back bit for bit
    opt.resume, opt.resume_train = False, True
    with contextlib.redirect_stdout(io.StringIO()):
        model2, loss2, _ = M.create_model(n_classes, n_rels=n_rels)
    model2.load_state_dict(ckpt["state_dict"])
    with contextlib.redirect_stdout(io.StringIO()):
        ema2 = _common.resume_ema(model2)
    back = ema2.state_dict()
    assert back["n_averaged"] == st["n_averaged"]
    assert all(torch.equal(back["state_dict"][k].cpu(), v) for k, v in st["state_dict"].items())

    # --resume: evaluates the average
    opt.resume, opt.resume_train = True, False
    with contextlib.redirect_stdout(io.StringIO()):
        got = _common.catch_inner()
        fresh, loss3, _ = M.create_model(n_classes, n_rels=n_rels)
        fresh.load_state_dict(st["state_dict"])
        want = T.testing(cd.MixedFeaturesDataset("val").cache().init_relships(), fresh, loss3, mode="val")
    assert got[0] == want

    # --resume on a checkpoint without an average refuses; with the flag off it loads as before
    old = dict(ckpt)
    del old["ema"]
    opt.resume_str = os.path.join(str(tmp_path), "old.pth.tar")
    torch.save(old, opt.resume_str)
    with pytest.raises(RuntimeError, match="has none"), contextlib.redirect_stdout(io.StringIO()):
        _common.catch_inner()
    opt.ema_decay = 0.0
    with contextlib.redirect_stdout(io.StringIO()):
        got = _common.catch_inner()
        want = T.testing(cd.MixedFeaturesDataset("val").cache().init_relships(), model, loss, mode="val")
    assert got[0] == want


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_data_parallel_averages_stay_identical_across_ranks():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29539", os.path.join(ROOT, "tools", "ema_dp_parity.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    out = res.stdout + res.stderr
    assert res.returncode == 0 and "EMA DP PARITY OK" in out, out[-3000:]
