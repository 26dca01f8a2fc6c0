"""--optimizer: the flag, create_model's choice and its refusal, and the published LAMB chunk size (no GPU needed)."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_optimizer_flag_default_and_choices():
    from lirec_b200.utils.arg_pars import build_parser
    p = build_parser()
    assert p.parse_args([]).optimizer == "adam"
    assert p.parse_args(["--optimizer", "lamb"]).optimizer == "lamb"
    with pytest.raises(SystemExit):
        p.parse_args(["--optimizer", "sgd"])


def test_create_model_refuses_an_unknown_optimizer_before_device_work(opt_preset):
    # device="cpu": reaching any device work would raise the "no CPU fallback" RuntimeError instead
    opt_preset("int_rel_ch", device="cpu", optimizer="sgd")
    import lirec_b200.mlp.model as M
    with pytest.raises(ValueError, match="--optimizer must be adam or lamb"):
        M.create_model(101, n_rels=15)


@pytest.mark.parametrize("choice", ["adam", "lamb"])
def test_create_model_accepts_both_optimizers(opt_preset, choice):
    opt_preset("int_rel_ch", device="cpu", optimizer=choice)
    import lirec_b200.mlp.model as M
    with pytest.raises(RuntimeError, match="no CPU"):
        M.create_model(101, n_rels=15)


def test_flat_lamb_is_not_a_flat_adam():
    """The in-switch exchange and the overlapped Adam pass run Adam's arithmetic; they recognise FlatAdam by type,
    so FlatLamb must stay outside that type."""
    import lirec_b200.mlp.model as M
    assert not issubclass(M.FlatLamb, M.FlatAdam)
    assert issubclass(M.FlatLamb, M._FlatOptimizer) and issubclass(M.FlatAdam, M._FlatOptimizer)
    assert "FlatLamb" in M.__all__


def test_chunk_size_and_partials_bound_match_the_header():
    from lirec_b200 import _ext, ops
    with open(os.path.join(ROOT, "include", "lirec_b200.h")) as f:
        header = f.read()
    assert int(re.search(r"#define LIREC_LAMB_CHUNK (\d+)", header).group(1)) == _ext.LAMB_CHUNK
    assert "#define LIREC_LAMB_PARTIALS(n, n_tensors) ((n) / LIREC_LAMB_CHUNK + (n_tensors))" in header
    part = ops.lamb_partials(3 * _ext.LAMB_CHUNK + 5, 7)
    assert tuple(part.shape) == (3 + 7, 2) and part.element_size() == 8
