"""Global-norm gradient clipping on the B200 (lirec_grad_clip_flat, clip_grad_norm_flat_, --clip_grad_norm): the
kernels against fp64 and against torch.nn.utils.clip_grad_norm_, determinism, refusals, real model gradients, the
optimizer steps around it, the training loop and data parallelism."""
import contextlib
import io
import math
import os
import subprocess
import sys

import pytest
import torch

from helpers import make_model, rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SENTINEL = 12345.0


def awkward_layout():
    """(begin, length) of tensors in a flat buffer: tiny, odd, empty, one over many chunks, one gate-weight sized,
    an all-zero tensor and one that starts off the 16-byte grid; padding between segments as in the model's
    256-byte-aligned layout."""
    from lirec_b200 import _ext
    lengths = [1, 3, 0, 15, 101, 3 * _ext.LAMB_CHUNK + 77, 9_437_187, 300, 777, 101]
    spans, off = [], 0
    for i, n in enumerate(lengths):
        shift = 1 if i == len(lengths) - 1 else 0                 # last tensor: begin not a multiple of 4 floats
        spans.append((off + shift, n))
        off += (n + shift + 63) // 64 * 64 if n else 64
    return spans, off, {"empty": 2, "zero": 7}


def _case(seed=0, scale=1e-2):
    spans, total, special = awkward_layout()
    gen = torch.Generator(device="cuda").manual_seed(seed)
    mask = torch.zeros(total, dtype=torch.bool, device="cuda")
    g = torch.full((total,), SENTINEL, device="cuda")
    for a, n in spans:
        mask[a:a + n] = True
        g[a:a + n] = torch.randn(n, generator=gen, device="cuda") * scale
    a, n = spans[special["zero"]]
    g[a:a + n] = 0.0
    return spans, mask, g, special


def _table(spans):
    begin = torch.tensor([a for a, _ in spans], dtype=torch.int64, device="cuda")
    length = torch.tensor([n for _, n in spans], dtype=torch.int64, device="cuda")
    return begin, length


def _clip(spans, g, max_norm, grad_scale):
    from lirec_b200 import ops
    begin, length = _table(spans)
    part = ops.lamb_partials(g.numel(), len(spans), device="cuda")
    tn = torch.full((len(spans),), float("nan"), device="cuda")
    norm = ops.grad_clip_flat(g, begin, length, part, max_norm, grad_scale, tensor_norms_out=tn)
    torch.cuda.synchronize()
    return norm, tn


def _fp64_norms(spans, g, grad_scale):
    per = [float((grad_scale * g[a:a + n].double()).norm()) for a, n in spans]
    return math.sqrt(sum(x * x for x in per)), per


def _coef(max_norm, norm):
    """torch.nn.utils.clip_grad_norm_'s factor in fp32 from the kernel's own norm (CPU: IEEE division)."""
    n = norm.detach().float().cpu()
    return torch.clamp(torch.tensor(max_norm, dtype=torch.float32) / (n + 1e-6), max=1.0)


@pytest.mark.parametrize("grad_scale", [1.0, 0.5])
def test_clipped_kernel_matches_fp64_and_scales_by_its_own_coefficient(grad_scale):
    spans, mask, g, special = _case()
    g0 = g.clone()
    ref, ref_per = _fp64_norms(spans, g0, grad_scale)
    max_norm = 0.1 * ref
    norm, tn = _clip(spans, g, max_norm, grad_scale)
    assert abs(float(norm) - ref) / ref < 1e-6
    for i, r in enumerate(ref_per):
        if r == 0.0:
            assert float(tn[i]) == 0.0, i
        else:
            assert abs(float(tn[i]) - r) / r < 1e-6, i
    assert float(tn[special["empty"]]) == 0.0 and float(tn[special["zero"]]) == 0.0
    c = _coef(max_norm, norm)
    assert 0.0 < float(c) < 1.0
    assert torch.equal(g[mask], g0[mask] * c.cuda())          # bitwise: the kernel multiplies by exactly this coef
    assert int((~mask).sum()) > 0 and bool((g[~mask] == SENTINEL).all())


def test_unclipped_kernel_leaves_the_buffer_bitwise_unchanged():
    spans, mask, g, _ = _case(seed=1)
    g0 = g.clone()
    ref, _ = _fp64_norms(spans, g0, 0.5)
    norm, _ = _clip(spans, g, 10.0 * ref, 0.5)
    assert abs(float(norm) - ref) / ref < 1e-6
    assert torch.equal(g, g0)


@pytest.mark.parametrize("bad", ["nan", "inf", "-inf"])
def test_non_finite_gradients_match_torch(bad):
    spans, mask, g, _ = _case(seed=2)
    a, n = spans[6]
    g[a + 1000] = float(bad)
    g[a + 5] = float(bad) if bad == "nan" else g[a + 5]
    params = []
    for a, n in spans:
        p = torch.nn.Parameter(torch.zeros(n, device="cuda"))
        p.grad = g[a:a + n].clone()
        params.append(p)
    max_norm = 0.05
    t_norm = torch.nn.utils.clip_grad_norm_(params, max_norm)
    norm, _ = _clip(spans, g, max_norm, 1.0)
    torch.testing.assert_close(norm.cpu(), t_norm.float().cpu(), rtol=0, atol=0, equal_nan=True)
    for (a, n), p in zip(spans, params):
        torch.testing.assert_close(g[a:a + n], p.grad, rtol=0, atol=0, equal_nan=True)
        assert torch.equal(torch.isnan(g[a:a + n]), torch.isnan(p.grad))
    if bad == "nan":
        assert bool(torch.isnan(g[mask]).all())
    else:
        assert int(torch.isnan(g[mask]).sum()) == 1 and float(g[mask].nan_to_num(0.0).abs().max()) == 0.0
    assert bool((g[~mask] == SENTINEL).all())


def test_clip_kernel_is_bitwise_reproducible():
    outs = []
    for _ in range(2):
        spans, _, g, _ = _case(seed=3)
        norm, tn = _clip(spans, g, 0.3, 0.5)
        outs.append((g, norm, tn))
    for x, y in zip(*outs):
        assert torch.equal(x, y)


def test_clip_refuses_bad_arguments():
    from lirec_b200 import _ext, ops
    spans, _, g, _ = _case()
    begin, length = _table(spans)
    part = ops.lamb_partials(g.numel(), len(spans), device="cuda")
    with pytest.raises(RuntimeError, match="partials"):
        ops.grad_clip_flat(g, begin, length, part[:-1], 1.0)
    for bad in (0.0, -1.0, float("nan"), float("inf")):
        with pytest.raises(RuntimeError, match="max_norm"):
            ops.grad_clip_flat(g, begin, length, part, bad)
    with pytest.raises(ValueError, match="float32"):
        ops.grad_clip_flat(g.double(), begin, length, part, 1.0)
    L = _ext.lib()
    norm = torch.empty((), device="cuda")

    def raw(grad, bp, lp, nt, n, pp, np_, out):
        return L.lirec_grad_clip_flat(grad, bp, lp, nt, n, pp, np_, 1.0, 1.0, out, None, None)

    args = [g.data_ptr(), begin.data_ptr(), length.data_ptr(), len(spans), g.numel(), part.data_ptr(),
            part.shape[0], norm.data_ptr()]
    for i in (0, 1, 2, 5, 7):                                  # grad, begin, len, partials, norm_out
        a = list(args)
        a[i] = None
        assert raw(*a) != 0 and b"null pointer" in L.lirec_last_error(), i
    a = list(args)
    a[3] = 0
    assert raw(*a) != 0 and b"n_tensors=0" in L.lirec_last_error()
    a = list(args)
    a[4] = 0
    assert raw(*a) != 0 and b"n=0" in L.lirec_last_error()
    before = g.clone()
    assert raw(*args) == 0                                     # the same call with every argument in range runs
    torch.cuda.synchronize()
    assert not torch.equal(g, before)


def _grads_of_a_step(opt_preset, preset, seed=5, **over):
    from lirec_b200.mixed_utils import synthetic
    import lirec_b200.mlp.model as M
    opt_preset(preset, **over)
    model, loss, optimizer = make_model(seed=seed)
    model.train()
    pb = synthetic.make_batch(16, seed=41, preset=preset).to_device("cuda")
    M.train_step(model, loss, pb, seed=201)
    return model, loss, optimizer


@pytest.mark.parametrize("preset", ["int_rel_ch", "int_rels", "modalities"])
def test_clip_grad_norm_flat_matches_torch_on_model_gradients(opt_preset, preset):
    import lirec_b200.mlp.model as M
    model, _, _ = _grads_of_a_step(opt_preset, preset)
    params = list(model.parameters())
    assert all(p.grad is not None for p in params)
    ref = []
    for p in params:
        q = torch.nn.Parameter(p.detach().clone())
        q.grad = p.grad.detach().clone()
        ref.append(q)
    per64 = [float(q.grad.double().norm()) for q in ref]
    norm64 = math.sqrt(sum(x * x for x in per64))
    max_norm = 0.3 * norm64
    t_norm = torch.nn.utils.clip_grad_norm_(ref, max_norm)
    tn = torch.empty(len(params), device="cuda")
    norm = M.clip_grad_norm_flat_(model, max_norm, tensor_norms=tn)
    assert norm.dim() == 0 and norm.is_cuda and norm.dtype == torch.float32
    assert abs(float(norm) - norm64) / norm64 < 1e-6
    assert abs(float(norm) - float(t_norm)) / float(t_norm) < 1e-6
    for i, ((name, p), q) in enumerate(zip(model.named_parameters(), ref)):
        assert abs(float(tn[i]) - per64[i]) <= 1e-6 * per64[i], name
        assert rel_err(p.grad, q.grad) < 1e-6, name


def test_clip_grad_norm_flat_refuses_a_foreign_grad(opt_preset):
    import lirec_b200.mlp.model as M
    model, _, _ = _grads_of_a_step(opt_preset, "int_rels")
    p = next(model.parameters())
    p.grad = p.grad.clone()                                    # a tensor outside the flat buffer
    with pytest.raises(RuntimeError, match="outside the flat gradient buffer"):
        M.clip_grad_norm_flat_(model, 1.0)
    with pytest.raises(ValueError, match="max_norm"):
        M.clip_grad_norm_flat_(model, 0.0)


def _train(opt_preset, kind, max_norm, steps=3):
    """`steps` steps through mlp.train.train_step from one seed; returns the model's flat weights."""
    from lirec_b200.mixed_utils import synthetic
    import lirec_b200.mlp.train as TR
    opt_preset("int_rel_ch", fused_adam=int(kind == "flat_adam"), optimizer="lamb" if kind == "flat_lamb" else "adam",
               lr=1e-3, weight_decay=0.01 if kind == "flat_lamb" else 0.0)
    model, loss, optimizer = make_model(seed=9)
    model.train()
    norms = []
    for s in range(steps):
        pb = synthetic.make_batch(16, seed=60 + s).to_device("cuda")
        TR.train_step(model, loss, optimizer, pb, 1, None, max_norm)
        if max_norm:
            norms.append(float(model._last_grad_norm))
    torch.cuda.synchronize()
    return model._flat.clone(), norms


@pytest.mark.parametrize("kind", ["torch_adam", "flat_adam", "flat_lamb"])
def test_a_max_norm_above_the_norm_changes_no_bit(opt_preset, kind):
    w_off, _ = _train(opt_preset, kind, 0.0)
    w_on, norms = _train(opt_preset, kind, 1e6)
    assert all(0.0 < n < 1e6 for n in norms)
    assert torch.equal(w_off, w_on)


def test_clipped_flat_adam_matches_fp64_clip_then_adam(opt_preset):
    from lirec_b200 import dp
    from lirec_b200.mixed_utils import synthetic
    import lirec_b200.mlp.model as M
    opt_preset("int_rel_ch", fused_adam=1, lr=1e-3, weight_decay=1e-4)
    model, loss, optimizer = make_model(seed=13)
    assert isinstance(optimizer, M.FlatAdam)
    model.train()
    spans = [(off, p.numel()) for off, p in zip(model._offsets, model._param_list)]
    grp = optimizer.param_groups[0]
    lr, eps, wd = grp["lr"], grp["eps"], grp["weight_decay"]
    # the fused Adam kernel takes its betas in fp32: 1 - fp32(0.999) is 1.3e-5 off 0.001, and v shows it
    b1, b2 = (float(torch.tensor(b, dtype=torch.float32)) for b in grp["betas"])
    w = model._flat.double().clone()
    m, v = torch.zeros_like(w), torch.zeros_like(w)
    max_norm = None
    for t in range(1, 6):
        pb = synthetic.make_batch(16, seed=80 + t).to_device("cuda")
        M.train_step(model, loss, pb, seed=400 + t)
        g = model._flat_grad.double().clone()
        norm = math.sqrt(sum(float(g[a:a + n].norm()) ** 2 for a, n in spans))
        max_norm = max_norm or 0.1 * norm
        assert norm > max_norm
        got = dp.reduce_and_step(model, optimizer, None, max_norm=max_norm)
        assert abs(float(got) - norm) / norm < 1e-6
        coef = min(max_norm / (norm + 1e-6), 1.0)
        bc1, bc2 = 1.0 - b1 ** t, 1.0 - b2 ** t
        for a, n in spans:
            gs = g[a:a + n] * coef + wd * w[a:a + n]
            m[a:a + n] = b1 * m[a:a + n] + (1 - b1) * gs
            v[a:a + n] = b2 * v[a:a + n] + (1 - b2) * gs * gs
            w[a:a + n] -= lr * (m[a:a + n] / bc1) / (v[a:a + n].sqrt() / math.sqrt(bc2) + eps)
    for (name, _), (a, n) in zip(model.named_parameters(), spans):
        assert rel_err(model._flat[a:a + n], w[a:a + n]) < 1e-5, name
        assert rel_err(optimizer._m[a:a + n], m[a:a + n]) < 1e-5, ("exp_avg", name)
        assert rel_err(optimizer._v[a:a + n], v[a:a + n]) < 1e-5, ("exp_avg_sq", name)


def test_training_loop_with_clipping_takes_the_unfused_step(tmp_path, opt_preset, monkeypatch):
    opt = opt_preset("int_rel_ch", synthetic=1, epochs=1, batch_size=16, num_workers=0, test=True, test_fr=1,
                     save_model=False, save_model_often=False, store_root=str(tmp_path), resume=False,
                     resume_train=False, fused_adam=1, overlap_adam=1, optimizer="adam", dp=0, lr=1e-3,
                     tr_sum_max=False, rels_multi_clip=True, clip_grad_norm=1e-3)
    from lirec_b200 import dp
    from lirec_b200.mixed_utils import classification_dataloader as cd
    monkeypatch.setattr(cd.SyntheticClipsDataset, "SIZES", {"train": 48, "val": 24, "test": 24})

    def no_fused_step(*args, **kwargs):
        raise AssertionError("SwitchReduceAdam.attach called while clipping")

    monkeypatch.setattr(dp.SwitchReduceAdam, "attach", no_fused_step)
    import lirec_b200.mlp.model as M
    import lirec_b200.mlp.test as T
    import lirec_b200.mlp.train as TR
    train_ds, val_ds = cd.MixedFeaturesDataset("train").cache().init_relships(), cd.MixedFeaturesDataset("val")
    torch.manual_seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        model, loss, optimizer = M.create_model(train_ds.n_classes, n_rels=len(train_ds.rels_list) - 1)
    assert isinstance(optimizer, M.FlatAdam) and opt.clip_grad_norm == 1e-3
    w0 = model._flat.clone()
    TR.training(train_ds, model=model, loss=loss, optimizer=optimizer, name="t", val_dataset=val_ds)
    assert optimizer._t >= 3
    assert not torch.equal(w0, model._flat)
    assert bool(torch.isfinite(model._flat).all())
    assert float(model._last_grad_norm) > 1e-3                 # the synthetic gradients are larger: it clipped
    after = T.testing(val_ds, model, loss, mode="val")
    assert set(after) == {"total", "ints", "rels", "tracks", "joint"}
    assert all(0.0 <= v <= 4.0 for v in after.values())


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_data_parallel_clipping_keeps_the_replicas_identical():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29537", os.path.join(ROOT, "tools", "clip_dp_parity.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    out = res.stdout + res.stderr
    assert res.returncode == 0 and "CLIP DP PARITY OK" in out, out[-3000:]
