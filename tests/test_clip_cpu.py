"""--clip_grad_norm: the flag, create_model's refusal, and where dp.reduce_and_step clips (no GPU needed)."""
import pytest


def test_clip_flag_default_and_parsing():
    from lirec_b200.utils.arg_pars import build_parser
    p = build_parser()
    assert p.parse_args([]).clip_grad_norm == 0.0
    assert p.parse_args(["--clip_grad_norm", "1.0"]).clip_grad_norm == 1.0
    assert p.parse_args(["--clip_grad_norm", "0.25"]).clip_grad_norm == 0.25
    with pytest.raises(SystemExit):
        p.parse_args(["--clip_grad_norm", "big"])


@pytest.mark.parametrize("value", [-1.0, float("nan"), float("inf")])
def test_create_model_refuses_a_bad_max_norm_before_device_work(opt_preset, value):
    # device="cpu": reaching any device work would raise the "no CPU fallback" RuntimeError instead
    opt_preset("int_rel_ch", device="cpu", clip_grad_norm=value)
    import lirec_b200.mlp.model as M
    with pytest.raises(ValueError, match="--clip_grad_norm"):
        M.create_model(101, n_rels=15)


@pytest.mark.parametrize("value", [0.0, 1.0])
def test_create_model_accepts_off_and_a_positive_max_norm(opt_preset, value):
    opt_preset("int_rel_ch", device="cpu", clip_grad_norm=value)
    import lirec_b200.mlp.model as M
    with pytest.raises(RuntimeError, match="no CPU"):
        M.create_model(101, n_rels=15)


def test_clip_grad_norm_flat_is_public():
    import lirec_b200.mlp.model as M
    assert "clip_grad_norm_flat_" in M.__all__


class _Model:
    _flat_grad = "flat-grad"


def _stand_ins(monkeypatch, world, scale):
    """Record the order of clip / exchange / step calls of dp.reduce_and_step."""
    from lirec_b200 import dp
    import lirec_b200.mlp.model as M
    calls = []

    def clip(model, max_norm, grad_scale=1.0, tensor_norms=None):
        calls.append(("clip", max_norm, grad_scale))
        return "norm"

    def allreduce(flat_grad, local_clips=None, global_clips=None, average_in_place=False):
        calls.append(("allreduce", average_in_place))
        return 1.0 if average_in_place else scale

    monkeypatch.setattr(M, "clip_grad_norm_flat_", clip)
    monkeypatch.setattr(dp, "world_size", lambda: world)
    monkeypatch.setattr(dp, "allreduce_flat_grad", allreduce)

    class Flat(M._FlatOptimizer):
        def __init__(self):                      # no model, no buffers: only the step is looked at
            pass

        def step(self, closure=None, grad_scale=1.0):
            calls.append(("step", grad_scale))

        def _step_impl(self, grad_scale=1.0):
            calls.append(("step", grad_scale))

    class Plain:
        def step(self):
            calls.append(("step", None))

    return calls, Flat(), Plain()


def test_reduce_and_step_clips_before_the_flat_step_with_the_average_as_grad_scale(monkeypatch):
    from lirec_b200 import dp
    calls, flat, _ = _stand_ins(monkeypatch, world=4, scale=0.25)
    assert dp.reduce_and_step(_Model(), flat, None, 8, 32, max_norm=1.5) == "norm"
    assert calls == [("allreduce", False), ("clip", 1.5, 0.25), ("step", 0.25)]


def test_reduce_and_step_clips_the_averaged_gradient_for_torch_optimizers(monkeypatch):
    from lirec_b200 import dp
    calls, _, plain = _stand_ins(monkeypatch, world=2, scale=0.5)
    dp.reduce_and_step(_Model(), plain, None, 8, 16, max_norm=2.0)
    # torch.optim.Adam reads p.grad: the average is applied in place first, so the clip sees grad_scale 1
    assert calls == [("allreduce", True), ("clip", 2.0, 1.0), ("step", None)]


@pytest.mark.parametrize("which", ["flat", "plain"])
def test_reduce_and_step_clips_before_the_single_gpu_step(monkeypatch, which):
    from lirec_b200 import dp
    calls, flat, plain = _stand_ins(monkeypatch, world=1, scale=1.0)
    dp.reduce_and_step(_Model(), flat if which == "flat" else plain, max_norm=0.5)
    assert calls == [("clip", 0.5, 1.0), ("step", 1.0 if which == "flat" else None)]


@pytest.mark.parametrize("world", [1, 2])
def test_reduce_and_step_does_not_clip_at_zero(monkeypatch, world):
    from lirec_b200 import dp
    calls, flat, plain = _stand_ins(monkeypatch, world=world, scale=0.5)
    assert dp.reduce_and_step(_Model(), flat, None, 8, 16) is None
    assert dp.reduce_and_step(_Model(), plain, None, 8, 16, max_norm=0.0) is None
    assert not [c for c in calls if c[0] == "clip"]
    assert [c for c in calls if c[0] == "step"] == [("step", 0.5 if world == 2 else 1.0), ("step", None)]


def test_reduce_and_step_refuses_to_clip_a_fused_step(monkeypatch):
    from lirec_b200 import dp
    calls, flat, _ = _stand_ins(monkeypatch, world=2, scale=0.5)

    class Fused:
        def step(self, local_clips, global_clips):
            calls.append(("fused",))

    with pytest.raises(ValueError, match="clipping"):
        dp.reduce_and_step(_Model(), flat, Fused(), 8, 16, max_norm=1.0)
    dp.reduce_and_step(_Model(), flat, Fused(), 8, 16)
    assert calls == [("fused",)]
