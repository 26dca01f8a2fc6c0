"""Host-side logic of bench.py that needs no GPU: the algorithmic FLOP figure (SURVEY.md §8d), the choice of the
tensor peak from the clocks of the timed region, and the clock sampler's bookkeeping (time-stamped samples sorted
into the timed regions after the fact)."""
import importlib.util
import os
import sys
import time

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bench():
    argv = sys.argv
    sys.argv = ["bench.py"]
    try:
        spec = importlib.util.spec_from_file_location("lirec_bench_under_test", os.path.join(ROOT, "bench.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        sys.argv = argv
    return mod


def test_algorithmic_flops_follow_the_survey_formula(bench):
    # SURVEY.md §8d: fwd MACs = (Ni + Nc) E + Ni (G + H_i + H_r), bwd = 2 fwd - (Ni + Nc) E1, FLOPs = 2 MACs
    E1, E, G, Hi, Hr = 3538944, 4325376, 9437184, 310272, 23040
    ni, nc = 8374.0, 29948.0
    fwd = (ni + nc) * E + ni * (G + Hi + Hr)
    want = 2 * (fwd + 2 * fwd - (ni + nc) * E1)
    got = bench.algorithmic_flops("int_rel_ch", ni, nc)
    assert abs(got - want) <= 1e-9 * want
    assert abs(want - 1.214e12) < 0.01e12                     # the figure VERDICT r1 recomputed
    # models without the context branch / the gate: Ni (E + 155,136)
    got = bench.algorithmic_flops("int_ch", ni, 0.0)
    fwd = ni * (E + 155136)
    assert abs(got - 2 * (3 * fwd - ni * E1)) <= 1e-9 * got


def test_peak_choice_follows_the_clocks_of_the_timed_region(bench):
    pk = {"bf16_burst": 1660.4, "bf16_sustained": 1366.2}
    full = {"sm_mhz": 1965.0, "sm_max_mhz": 1965.0, "reasons": []}
    capped = {"sm_mhz": 1740.0, "sm_max_mhz": 1965.0, "reasons": ["sw_power_cap"]}
    assert bench.pick_tensor_peak(pk, 40.0, full)[0] == 1660.4
    assert bench.pick_tensor_peak(pk, 400.0, capped)[0] == 1366.2
    assert bench.pick_tensor_peak(pk, 40.0, dict(full, reasons=["sw_power_cap"]))[0] == 1366.2
    assert bench.pick_tensor_peak(pk, 40.0, None)[0] == 1660.4 and bench.pick_tensor_peak(pk, 4000.0, None)[0] == 1366.2


def test_clock_samples_are_sorted_into_their_regions(bench):
    s = bench.ClockSampler(0)
    s.mx = 1965.0
    t = time.perf_counter()
    s.samples = [(t - 0.5, 1200.0, 90.0, []),                              # before any timed region: ignored
                 (t + 0.001, 1965.0, 400.0, []), (t + 0.02, 1950.0, 500.0, []),
                 (t + 0.5, 1700.0, 990.0, ["sw_power_cap"]), (t + 0.7, 1725.0, 995.0, ["sw_power_cap"]),
                 (t + 2.0, 1000.0, 100.0, ["hw_slowdown"])]                # after the last one: ignored
    s.spans = [("value", t, t + 0.04), ("e2e", t + 0.3, t + 0.6), ("e2e", t + 0.65, t + 0.9)]
    c = s.stop()
    assert c["samples"] == 2 and c["sm_mhz"] == 1957.5 and c["reasons"] == [] and c["sm_max_mhz"] == 1965.0
    e = c["by_region"]["e2e"]
    assert e["samples"] == 2 and e["reasons"] == ["sw_power_cap"] and e["power_w_max"] == 995.0
    # region() only records intervals
    s2 = bench.ClockSampler(0)
    s2.region(True, "value")
    s2.region(False)
    s2.region(True, "e2e")
    s2.region(False)
    assert [x[0] for x in s2.spans] == ["value", "e2e"] and all(b >= a for _, a, b in s2.spans)
    assert s2.stop()["samples"] == 0


def test_dump_outputs_writes_loss_params_and_grads(bench, tmp_path, monkeypatch):
    import numpy as np
    import torch
    model = torch.nn.Sequential(torch.nn.Linear(6, 5), torch.nn.Linear(5, 3))
    n = sum(q.numel() for q in model.parameters())
    with torch.no_grad():                     # parameter value = its position in named_parameters order
        for q, start in zip(model.parameters(), np.cumsum([0] + [q.numel() for q in model.parameters()])):
            q.copy_(torch.arange(start, start + q.numel(), dtype=torch.float32).view(q.shape))
            q.grad = 2 * q + 1
    loss = torch.tensor(0.25)

    def load(d):
        return {k: np.load(os.path.join(str(tmp_path), d, k + ".npy")) for k in ("loss", "params", "grads")}
    bench.dump_outputs(model, loss, os.path.join(str(tmp_path), "all"))
    z = load("all")
    assert all(v.dtype == np.float32 for v in z.values())
    assert z["loss"].tolist() == [0.25]
    assert np.array_equal(z["params"], np.arange(n, dtype=np.float32))
    assert np.array_equal(z["grads"], 2 * z["params"] + 1)
    # above the cap: one fixed sample of positions, the same for both arrays and from run to run
    monkeypatch.setattr(bench, "DUMP_MAX_ELEMS", 10)
    bench.dump_outputs(model, loss, os.path.join(str(tmp_path), "a"))
    bench.dump_outputs(model, loss, os.path.join(str(tmp_path), "b"))
    a, b = load("a"), load("b")
    assert a["params"].shape == (10,) and np.all(np.diff(a["params"]) > 0) and a["params"].max() < n
    assert np.array_equal(a["grads"], 2 * a["params"] + 1)
    assert all(np.array_equal(a[k], b[k]) for k in a)
