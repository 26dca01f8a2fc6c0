"""Cost of the exponential moving average of the weights (--ema_decay, lirec_ema_update_flat / lirec_ema_swap_flat),
on int_rel_ch's flat parameter buffer and on the benchmark's training steps (bench.py: synthetic MovieGraphs-shaped
batches, HBM-resident banks).

1. Kernel time, CUDA events over >= 200 back-to-back launches per window, 5 windows alternating, median (min-max), on
   the weights of int_rel_ch (18.4 M parameters, 73.7 MB with padding):
   - update: reads the average and the weights, writes the average (12 bytes per float);
   - swap with the bf16 shadow: reads and writes both fp32 buffers, writes the shadow (18 bytes per float).
   The 73.7 MB buffers fit in the 126 MB L2, so each case is timed twice: L2-warm (the same buffers every launch) and
   L2-flushed (four sets of buffers in rotation: at least 442 MB pass through L2 between two uses of one set).
   Next to them, a device-to-device copy of the same bytes (a copy moves 8 bytes per float: 1.5x the copies' time is
   what the update's 12 bytes would take at the copy rate, 2.25x for the swap's 18), warm and in rotation.
2. Training step time (forward + loss + backward + FlatAdam with its default overlap of the gate + head pass,
   bench.py's device-resident leg), alternating 30-step legs without and with --ema_decay 0.999, 5 rounds: 1024 clips
   on int_rel_ch and int_rels, 64 clips on int_rel_ch.

Prints one JSON object with the GPU name and power limit next to the numbers.  Usage:
    python tools/ema_probe.py [--launches 200] [--rounds 5] [--steps 30] [--out FILE]
"""
import argparse
import contextlib
import io
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from loss_probe import alternate, gpu_info, summary  # noqa: E402

DATASHEET_GBS = 7700.0          # HGX B200 data sheet, one GPU, at a 1000 W power limit
DECAY = 0.999
ROTATE = 4


def make_bench(preset, batch, ema):
    import bench
    import lirec_b200.mlp.model as M
    bench._ARGV = []                                         # bench.py's defaults, not this script's flags
    bargs = bench.parse_args()
    with contextlib.redirect_stdout(io.StringIO()):
        b = bench.Bench(bargs, preset, batch, 2, 0, 1, torch.device("cuda:0"))
    b.ema = None
    if ema:
        b.ema = M.FlatEMA(b.model, DECAY)
        b.step = lambda pb: b.TR.train_step(b.model, b.loss_fn, b.optimizer, pb, b.world, b.fused, 0.0, b.ema)
    return b


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ema_probe needs a B200")
    assert args.launches >= 200
    from lirec_b200 import ops
    res = {"gpu": gpu_info(), "launches_per_window": args.launches, "decay": DECAY}

    # ---- kernels on int_rel_ch's flat parameter buffer ----
    b = make_bench("int_rel_ch", 1024, False)
    m = b.model
    n = m._flat.numel()
    res["buffer"] = {"parameters": sum(p.numel() for p in m._param_list), "floats_with_padding": n}
    params = [m._flat.clone() for _ in range(ROTATE)]
    emas = [p + 1e-3 for p in params]
    shadows = [torch.empty(n, dtype=torch.bfloat16, device="cuda") for _ in range(ROTATE)]
    src = [torch.ones(2 * n, device="cuda") for _ in range(ROTATE)]   # a copy of 8 bytes per float
    dst = torch.empty(2 * n, device="cuda")
    st = {"i": 0}

    def pick(rotate):
        k = st["i"] % ROTATE if rotate else 0
        st["i"] += 1
        return k

    def update_fn(rotate):
        def fn():
            k = pick(rotate)
            ops.ema_update_flat(emas[k], params[k], DECAY)
        return fn

    def swap_fn(rotate):
        def fn():
            k = pick(rotate)
            ops.ema_swap_flat(params[k], emas[k], shadows[k])
        return fn

    def copy_fn(rotate):
        def fn():
            dst[:n].copy_(src[pick(rotate)][:n])
        return fn

    fns = {"update_warm": update_fn(False), "swap_warm": swap_fn(False), "d2d_copy_warm": copy_fn(False),
           "update_flushed": update_fn(True), "swap_flushed": swap_fn(True), "d2d_copy_flushed": copy_fn(True)}
    t = alternate(fns, args.launches, args.rounds)
    sm = {k: summary(v) for k, v in t.items()}
    nbytes = {"update": 12 * n, "swap": 18 * n, "d2d_copy": 8 * n}

    def rate(bytes_, us):
        gbs = bytes_ / us / 1e3
        return {"GB/s": round(gbs, 1), "of_datasheet": round(gbs / DATASHEET_GBS, 3)}

    res["kernels_us"] = sm
    res["bytes_per_call"] = nbytes
    res["achieved"] = {k: rate(nbytes[k.rsplit("_", 1)[0]], v["median"]) for k, v in sm.items()}
    # the copy's time scaled to the kernel's bytes, over the kernel's time: 1.0 is the copy rate
    res["fraction_of_copy_rate"] = {}
    for kind in ("update", "swap"):
        for cache in ("warm", "flushed"):
            copy_us = sm["d2d_copy_" + cache]["median"] * nbytes[kind] / nbytes["d2d_copy"]
            res["fraction_of_copy_rate"][kind + "_" + cache] = round(copy_us / sm[kind + "_" + cache]["median"], 3)
    b.close()
    del b, m, params, emas, shadows, src, dst, fns
    torch.cuda.empty_cache()

    # ---- training steps, alternating ----
    res["step_ms"] = {}
    for preset, batch in (("int_rel_ch", 1024), ("int_rels", 1024), ("int_rel_ch", 64)):
        benches = {"off": make_bench(preset, batch, False), "ema": make_bench(preset, batch, True)}
        ms = {k: [] for k in benches}
        for bb in benches.values():                          # warm-up
            bb.timed_resident(3, 3, profile=False)
        for _ in range(args.rounds):
            for k, bb in benches.items():
                total, _, _ = bb.timed_resident(args.steps, 3, profile=False)
                ms[k].append(total / args.steps)
        key = "%s@%d" % (preset, batch)
        res["step_ms"][key] = {k: summary(v) for k, v in ms.items()}
        res["step_ms"][key]["optimizer"] = "%s%s" % (type(benches["off"].optimizer).__name__,
                                                     " + overlapped gate/head pass"
                                                     if benches["off"].fused is not None else "")
        res["step_ms"][key]["ema_updates"] = benches["ema"].ema.n_averaged
        for bb in benches.values():
            bb.close()
        del benches
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
