"""--ema_decay: the flag, create_model's refusal, the C ABI names, and the training loop's and resume's use of
FlatEMA, with stand-ins for the device work (no GPU needed)."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMA_SYMBOLS = ("lirec_ema_update_flat", "lirec_ema_swap_flat")


def test_ema_flag_default_and_parsing():
    from lirec_b200.utils.arg_pars import build_parser
    p = build_parser()
    assert p.parse_args([]).ema_decay == 0.0
    assert p.parse_args(["--ema_decay", "0.999"]).ema_decay == 0.999
    with pytest.raises(SystemExit):
        p.parse_args(["--ema_decay", "slow"])


@pytest.mark.parametrize("value", [-0.1, 1.0, 1.5, float("nan"), float("inf")])
def test_create_model_refuses_a_bad_decay_before_device_work(opt_preset, value):
    # device="cpu": reaching any device work would raise the "no CPU fallback" RuntimeError instead
    opt_preset("int_rel_ch", device="cpu", ema_decay=value)
    import lirec_b200.mlp.model as M
    with pytest.raises(ValueError, match="--ema_decay"):
        M._check_ema_choice()
    with pytest.raises(ValueError, match="--ema_decay"):
        M.create_model(101, n_rels=15)


@pytest.mark.parametrize("value", [0.0, 0.5, 0.999, 0.9999])
def test_create_model_accepts_off_and_a_decay_in_range(opt_preset, value):
    opt_preset("int_rel_ch", device="cpu", ema_decay=value)
    import lirec_b200.mlp.model as M
    assert M._check_ema_choice() == value
    with pytest.raises(RuntimeError, match="no CPU"):
        M.create_model(101, n_rels=15)


@pytest.mark.parametrize("value", [0.0, 1.0, -0.5, float("nan")])
def test_flat_ema_refuses_a_decay_outside_the_open_interval(value):
    import lirec_b200.mlp.model as M
    with pytest.raises(ValueError, match="decay"):
        M.FlatEMA(object(), value)


def test_ema_symbols_are_bound_and_declared():
    from lirec_b200 import _ext
    import lirec_b200.mlp.model as M
    with open(os.path.join(ROOT, "include", "lirec_b200.h")) as f:
        header = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    for name in EMA_SYMBOLS:
        assert name in _ext.EXPORTED_SYMBOLS
        assert re.search(r"\bint %s\(" % name, header), name
    assert "FlatEMA" in M.__all__


class _Ema:
    def __init__(self, calls):
        self.calls = calls

    def update(self):
        self.calls.append("ema")


def test_train_step_updates_the_average_after_the_step(monkeypatch, opt_preset):
    """Both the normal path and the empty-shard path fold the new weights in, after dp.reduce_and_step."""
    opt_preset("int_rel_ch", native_step=0)
    import lirec_b200.mlp.train as TR
    calls = []
    monkeypatch.setattr(TR.dp, "reduce_and_step", lambda *a, **k: calls.append("step"))
    monkeypatch.setattr(TR, "dp_empty_shard_collectives", lambda *a, **k: calls.append("collectives"))

    class Zero:
        def zero_(self):
            return self

        def new_zeros(self, shape):
            return 0.0

    class Flat:
        device = "cpu"

    class Model:
        _flat = Flat()
        _flat_grad = Zero()

        def _sync_flat(self):
            pass

        def __call__(self, pb):
            return "out"

    class Value:
        def backward(self):
            calls.append("backward")

    class Optimizer:
        def zero_grad(self):
            pass

    class Batch:
        def __init__(self, B):
            self.B, self.global_clips, self.host = B, 2, None

    loss = lambda out, batch: Value()   # noqa: E731
    TR.train_step(Model(), loss, Optimizer(), Batch(4), 1, None, 0.0, _Ema(calls))
    assert calls == ["backward", "step", "ema"]
    del calls[:]
    TR.train_step(Model(), loss, Optimizer(), Batch(0), 2, None, 0.0, _Ema(calls))
    assert calls == ["collectives", "step", "ema"]
    del calls[:]
    TR.train_step(Model(), loss, Optimizer(), Batch(4), 1, None, 0.0)
    assert calls == ["backward", "step"]


def test_resume_refuses_to_evaluate_a_checkpoint_without_an_average(monkeypatch, opt_preset):
    opt = opt_preset("int_rel_ch", resume=True, resume_train=False, ema_decay=0.999, resume_str="old.pth.tar")
    from lirec_b200.resume import _common
    import lirec_b200.mlp.model as M
    built = []

    class Ema:
        def __init__(self, model, decay):
            built.append(decay)
            self.n_averaged = 0

        def load_state_dict(self, state):
            self.n_averaged = state["n_averaged"]

    monkeypatch.setattr(M, "FlatEMA", Ema)
    monkeypatch.setattr(_common, "load_ema", lambda: None)
    with pytest.raises(RuntimeError, match="has none"):
        _common.resume_ema("model")
    opt.resume_train = True                           # training from it: start the average from the weights
    assert _common.resume_ema("model").n_averaged == 0
    monkeypatch.setattr(_common, "load_ema", lambda: {"decay": 0.9, "n_averaged": 7, "state_dict": {}})
    assert _common.resume_ema("model").n_averaged == 7
    opt.resume_train = False
    assert _common.resume_ema("model").n_averaged == 7
    assert built == [0.999] * 4
