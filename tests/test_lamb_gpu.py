"""FlatLamb / lirec_lamb_flat on the B200: the kernels against an fp64 torch statement of LAMB, determinism, the
optimizer on real model gradients, checkpoints, schedulers, the training loop and data parallelism."""
import contextlib
import copy
import io
import os
import subprocess
import sys

import pytest
import torch

from helpers import make_model, rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 1e-5
SENTINEL = 12345.0


def lamb_reference(w, m, v, g, spans, lr, betas, eps, wd, t, grad_scale):
    """One LAMB step in fp64 (You et al. 2020, decoupled weight decay, no clamp), in place on the fp64 copies.
    Returns the trust ratio of every span."""
    b1, b2 = betas
    bc1, bc2 = 1.0 - b1 ** t, 1.0 - b2 ** t
    ratios = []
    for a, n in spans:
        gs = grad_scale * g[a:a + n]
        m[a:a + n] = b1 * m[a:a + n] + (1 - b1) * gs
        v[a:a + n] = b2 * v[a:a + n] + (1 - b2) * gs * gs
        u = (m[a:a + n] / bc1) / (v[a:a + n].sqrt() / bc2 ** 0.5 + eps) + wd * w[a:a + n]
        wn, un = float(w[a:a + n].norm()), float(u.norm())
        r = wn / un if wn > 0 and un > 0 else 1.0
        w[a:a + n] -= lr * r * u
        ratios.append(r)
    return ratios


def awkward_layout():
    """(begin, length) of tensors in a flat buffer: tiny, odd, one over many chunks, one gate-weight sized, an
    all-zero weight tensor, a zero-gradient tensor and one that starts off the 16-byte grid; padding between
    segments as in the model's 256-byte-aligned layout."""
    from lirec_b200 import _ext
    lengths = [1, 3, 15, 101, 3 * _ext.LAMB_CHUNK + 77, 9_437_187, 300, 777, 101]
    spans, off = [], 0
    for i, n in enumerate(lengths):
        shift = 1 if i == len(lengths) - 1 else 0                 # last tensor: begin not a multiple of 4 floats
        spans.append((off + shift, n))
        off += (n + shift + 63) // 64 * 64
    return spans, off, {"zero_w": 6, "zero_g": 7}


def _flat_case(seed=0):
    spans, total, special = awkward_layout()
    gen = torch.Generator(device="cuda").manual_seed(seed)
    mask = torch.zeros(total, dtype=torch.bool, device="cuda")
    for a, n in spans:
        mask[a:a + n] = True
    w = torch.full((total,), SENTINEL, device="cuda")
    m, v = w.clone(), w.clone()
    for a, n in spans:
        w[a:a + n] = torch.randn(n, generator=gen, device="cuda") * 0.05
        m[a:a + n] = 0.0
        v[a:a + n] = 0.0
    a, n = spans[special["zero_w"]]
    w[a:a + n] = 0.0
    grads = []
    for _ in range(5):
        g = torch.full((total,), SENTINEL, device="cuda")
        for a, n in spans:
            g[a:a + n] = torch.randn(n, generator=gen, device="cuda") * 1e-2
        a, n = spans[special["zero_g"]]
        g[a:a + n] = 0.0
        grads.append(g)
    bf = torch.full((total,), SENTINEL, dtype=torch.bfloat16, device="cuda")
    return spans, mask, w, m, v, bf, grads, special


HP = dict(lr=2e-3, betas=(0.9, 0.999), eps=1e-6, wd=0.01, grad_scale=0.5)


def _run_kernel(spans, w, m, v, bf, grads):
    from lirec_b200 import ops
    begin = torch.tensor([a for a, _ in spans], dtype=torch.int64, device="cuda")
    length = torch.tensor([n for _, n in spans], dtype=torch.int64, device="cuda")
    part = ops.lamb_partials(w.numel(), len(spans), device="cuda")
    trust = []
    for t, g in enumerate(grads, 1):
        tr = torch.full((len(spans),), float("nan"), device="cuda")
        ops.lamb_flat(w, g, m, v, bf, begin, length, part, HP["lr"], HP["betas"][0], HP["betas"][1], HP["eps"],
                      HP["wd"], t, HP["grad_scale"], trust_out=tr)
        trust.append(tr.cpu())
    torch.cuda.synchronize()
    return trust


def test_lamb_kernel_matches_fp64_statement():
    spans, mask, w, m, v, bf, grads, special = _flat_case()
    wd, md, vd = w.double(), m.double(), v.double()
    trust = _run_kernel(spans, w, m, v, bf, grads)
    for t, g in enumerate(grads, 1):
        r_ref = lamb_reference(wd, md, vd, g.double(), spans, HP["lr"], HP["betas"], HP["eps"], HP["wd"], t,
                               HP["grad_scale"])
        assert rel_err(trust[t - 1], torch.tensor(r_ref, dtype=torch.float64)) < TOL, t
        if t == 1:
            assert float(trust[0][special["zero_w"]]) == 1.0          # ||w|| = 0
    for i, (a, n) in enumerate(spans):
        assert rel_err(w[a:a + n], wd[a:a + n]) < TOL, ("param", i)
        assert rel_err(m[a:a + n], md[a:a + n]) < TOL, ("exp_avg", i)
        assert rel_err(v[a:a + n], vd[a:a + n]) < TOL, ("exp_avg_sq", i)
    assert torch.equal(bf[mask], w[mask].to(torch.bfloat16))
    pad = ~mask
    assert int(pad.sum()) > 0
    for buf in (w, m, v):
        assert bool((buf[pad] == SENTINEL).all())
    assert bool((bf[pad] == torch.tensor(SENTINEL, dtype=torch.bfloat16)).all())


def test_lamb_kernel_is_bitwise_reproducible():
    outs = []
    for _ in range(2):
        spans, mask, w, m, v, bf, grads, _ = _flat_case(seed=3)
        trust = _run_kernel(spans, w, m, v, bf, grads)
        outs.append((w, m, v, bf, torch.stack(trust)))
    for a, b in zip(*outs):
        assert torch.equal(a, b)


def test_lamb_refuses_bad_arguments():
    from lirec_b200 import _ext, ops
    spans, mask, w, m, v, bf, grads, _ = _flat_case()
    begin = torch.tensor([a for a, _ in spans], dtype=torch.int64, device="cuda")
    length = torch.tensor([n for _, n in spans], dtype=torch.int64, device="cuda")
    part = ops.lamb_partials(w.numel(), len(spans), device="cuda")
    args = (0.1, 0.9, 0.999, 1e-6, 0.0)
    with pytest.raises(RuntimeError, match="step"):
        ops.lamb_flat(w, grads[0], m, v, bf, begin, length, part, *args, 0)
    with pytest.raises(RuntimeError, match="partials"):
        ops.lamb_flat(w, grads[0], m, v, bf, begin, length, part[:-1], *args, 1)
    with pytest.raises(RuntimeError, match="1 - beta2"):
        ops.lamb_flat(w, grads[0], m, v, bf, begin, length, part, 0.1, 0.9, 1.0, 1e-6, 0.0, 1)
    # the entry point takes 1 - beta
    rc = _ext.lib().lirec_lamb_flat(w.data_ptr(), None, m.data_ptr(), v.data_ptr(), None, begin.data_ptr(),
                                    length.data_ptr(), len(spans), w.numel(), part.data_ptr(), part.shape[0], 0.1, 0.1,
                                    0.001, 1e-6, 0.0, 1, 1.0, None, None)
    assert rc != 0 and b"null pointer" in _ext.lib().lirec_last_error()


def _lamb_model(opt_preset, preset, seed=5, **over):
    import lirec_b200.mlp.model as M
    opt_preset(preset, optimizer="lamb", lr=1e-3, weight_decay=0.01, **over)
    model, loss, optimizer = make_model(seed=seed)
    assert isinstance(optimizer, M.FlatLamb)
    return model, loss, optimizer


def _spans(model):
    return [(off, p.numel()) for off, p in zip(model._offsets, model._param_list)]


@pytest.mark.parametrize("preset", ["int_rel_ch", "int_rels", "modalities"])
def test_flat_lamb_on_model_gradients_matches_fp64_statement(opt_preset, preset):
    from lirec_b200.mixed_utils import synthetic
    import lirec_b200.mlp.model as M
    model, loss, optimizer = _lamb_model(opt_preset, preset)
    model.train()
    spans = _spans(model)
    assert len(spans) == len(list(model.parameters()))
    wd = model._flat.double().clone()
    md, vd = torch.zeros_like(wd), torch.zeros_like(wd)
    for s in range(3):
        pb = synthetic.make_batch(16, seed=40 + s, preset=preset).to_device("cuda")
        M.train_step(model, loss, pb, seed=200 + s)
        g = model._flat_grad.double().clone()
        optimizer.step()
        g_ = optimizer.param_groups[0]
        r_ref = lamb_reference(wd, md, vd, g, spans, g_["lr"], g_["betas"], g_["eps"], g_["weight_decay"], s + 1, 1.0)
        assert rel_err(optimizer.last_trust_ratios(), torch.tensor(r_ref, dtype=torch.float64)) < TOL, s
    for (name, _), (a, n) in zip(model.named_parameters(), spans):
        assert rel_err(model._flat[a:a + n], wd[a:a + n]) < TOL, name
    # the bf16 shadow the next forward reads is the rounding of the new weights
    for a, n in spans:
        assert torch.equal(model._flat_bf16[a:a + n], model._flat[a:a + n].to(torch.bfloat16))


def test_flat_lamb_state_dict_round_trip(opt_preset):
    from lirec_b200.mixed_utils import synthetic
    import lirec_b200.mlp.model as M
    pbs = [synthetic.make_batch(16, seed=70 + s).to_device("cuda") for s in range(5)]

    def steps(model, loss, optimizer, idx):
        for s in idx:
            M.train_step(model, loss, pbs[s], seed=300 + s)
            optimizer.step()

    model, loss, optimizer = _lamb_model(opt_preset, "int_rel_ch")
    model.train()
    steps(model, loss, optimizer, range(5))
    straight = {k: v.clone() for k, v in model.state_dict().items()}

    model, loss, optimizer = _lamb_model(opt_preset, "int_rel_ch")
    model.train()
    steps(model, loss, optimizer, range(3))
    sd_m, sd_o = copy.deepcopy(model.state_dict()), copy.deepcopy(optimizer.state_dict())
    assert len(sd_o["state"]) == 38
    assert all(set(st) == {"step", "exp_avg", "exp_avg_sq"} and float(st["step"]) == 3.0 for st in sd_o["state"].values())
    assert {"lr", "betas", "eps", "weight_decay"} <= set(sd_o["param_groups"][0])

    model2, loss2, optimizer2 = _lamb_model(opt_preset, "int_rel_ch", seed=11)
    model2.load_state_dict(sd_m)
    optimizer2.load_state_dict(sd_o)
    assert optimizer2._t == 3
    model2.train()
    steps(model2, loss2, optimizer2, range(3, 5))
    for k, v in model2.state_dict().items():
        assert torch.equal(v, straight[k]), k


def test_switch_reduce_adam_does_not_take_flat_lamb(opt_preset):
    from lirec_b200 import dp
    model, loss, optimizer = _lamb_model(opt_preset, "int_rel_ch")
    assert dp.SwitchReduceAdam.attach(model, optimizer, single_gpu=True) is None


def test_lr_scheduler_changes_the_applied_step(opt_preset):
    from lirec_b200.mixed_utils import synthetic
    import lirec_b200.mlp.model as M
    pb = synthetic.make_batch(16, seed=90).to_device("cuda")
    deltas = []
    for factor in (None, 0.25):
        model, loss, optimizer = _lamb_model(opt_preset, "int_rel_ch")
        model.train()
        if factor is not None:
            torch.optim.lr_scheduler.LambdaLR(optimizer, lambda epoch: factor)
            assert optimizer.param_groups[0]["lr"] == pytest.approx(0.25e-3)
        w0 = model._flat.clone()
        M.train_step(model, loss, pb, seed=7)
        optimizer.step()
        deltas.append(model._flat - w0)
    # same gradients, same moments and trust ratios at step 1: the update scales with lr (up to the fp32 rounding of
    # w - lr * r * u, ~1e-4 of an update this small)
    assert float(deltas[0].abs().max()) > 0
    assert rel_err(deltas[1], 0.25 * deltas[0]) < 1e-2


def test_training_loop_with_optimizer_lamb(tmp_path, opt_preset, monkeypatch):
    opt = opt_preset("int_rel_ch", synthetic=1, epochs=1, batch_size=16, num_workers=0, test=True, test_fr=1,
                     save_model=False, save_model_often=False, store_root=str(tmp_path), resume=False,
                     resume_train=False, fused_adam=0, optimizer="lamb", dp=0, lr=1e-3, tr_sum_max=False,
                     rels_multi_clip=True)
    from lirec_b200.mixed_utils import classification_dataloader as cd
    monkeypatch.setattr(cd.SyntheticClipsDataset, "SIZES", {"train": 48, "val": 24, "test": 24})
    import lirec_b200.mlp.model as M
    import lirec_b200.mlp.test as T
    import lirec_b200.mlp.train as TR
    train_ds, val_ds = cd.MixedFeaturesDataset("train").cache().init_relships(), cd.MixedFeaturesDataset("val")
    torch.manual_seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        model, loss, optimizer = M.create_model(train_ds.n_classes, n_rels=len(train_ds.rels_list) - 1)
    assert isinstance(optimizer, M.FlatLamb) and opt.optimizer == "lamb"
    w0 = model._flat.clone()
    TR.training(train_ds, model=model, loss=loss, optimizer=optimizer, name="t", val_dataset=val_ds)
    assert optimizer._t >= 3
    assert not torch.equal(w0, model._flat)
    assert bool(torch.isfinite(model._flat).all()) and bool(torch.isfinite(optimizer.last_trust_ratios()).all())
    after = T.testing(val_ds, model, loss, mode="val")
    assert set(after) == {"total", "ints", "rels", "tracks", "joint"}
    assert all(0.0 <= v <= 4.0 for v in after.values())


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_data_parallel_lamb_matches_single_process():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29533", os.path.join(ROOT, "tools", "lamb_dp_parity.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    out = res.stdout + res.stderr
    assert res.returncode == 0 and "LAMB DP PARITY OK" in out, out[-3000:]
