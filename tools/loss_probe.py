"""Cost of the multi-label BCE losses next to the max-margin losses they can replace (--loss bce), on the
benchmark's inputs (bench.py: synthetic MovieGraphs-shaped batches of 1024 clips, HBM-resident banks).

1. Kernel time, CUDA events over >= 200 back-to-back launches per window, the two kernels alternating on the
   same logits: lirec_loss_track_fwd_bwd vs lirec_loss_bce_track_fwd_bwd (int_rel_ch) and
   lirec_loss_rowmargin_fwd_bwd vs lirec_loss_bce_fwd_bwd (int_rels interaction term).  Each window is queued
   behind a device-side spin, so the events time the GPU executing the launches, not the host issuing them.
2. Training step time (forward + loss + backward + Adam, bench.py's device-resident leg) with --loss margin vs
   --loss bce, alternating.

Prints one JSON object with the GPU name and power limit next to the numbers.  Usage:
    python tools/loss_probe.py [--launches 200] [--rounds 5] [--steps 30] [--out FILE]
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in q.split(",")[:2]]
    except Exception as e:                                   # the numbers are still printed, marked as such
        info["power_limit"] = "unknown (%s)" % e
    return info


def window_us(fn, launches):
    """Mean device time per launch of `fn` over `launches` back-to-back launches."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda._sleep(int(2e8))                              # the host queues the whole window meanwhile
    e0.record()
    for _ in range(launches):
        fn()
    e1.record()
    e1.synchronize()
    return 1e3 * e0.elapsed_time(e1) / launches


def alternate(fns, launches, rounds):
    """{name: [us per launch of each round]}, the kernels alternating window by window."""
    for fn in fns.values():                                  # warm-up
        window_us(fn, 20)
    out = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            out[k].append(window_us(fn, launches))
    return out


def make_bench(preset, loss, args):
    import bench
    from lirec_b200.utils.arg_pars import opt
    bench._ARGV = []                                         # bench.py's defaults, not this script's flags
    bargs = bench.parse_args()
    opt.loss = loss
    with contextlib.redirect_stdout(io.StringIO()):
        b = bench.Bench(bargs, preset, args.batch, 2, 0, 1, torch.device("cuda:0"))
    return b


def summary(v):
    v = np.asarray(v)
    return {"median": round(float(np.median(v)), 3), "min": round(float(v.min()), 3), "max": round(float(v.max()), 3),
            "rounds": [round(float(x), 3) for x in v]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("loss_probe needs a B200")
    assert args.launches >= 200
    from lirec_b200 import ops
    res = {"gpu": gpu_info(), "batch_clips": args.batch, "launches_per_window": args.launches, "kernels_us": {},
           "step_ms": {}}

    # ---- kernels on the benchmark's logits ----
    b = make_bench("int_rel_ch", "margin", args)
    pb = b.resident[0]
    with torch.no_grad():
        out = b.model(pb, seed=1)
    li, lr = out.ragged_inters.contiguous(), out.ragged_rels.contiguous()
    o = b.opt
    track = dict(
        margin=lambda: ops.loss_track(li, lr, pb["cand_off"], pb["labels"], pb["rels_label"], pb["gt_tracks"],
                                      pb.multilab, o.tr_margin, o.lymbda, 15, max_slots=pb.n_slots),
        bce=lambda: ops.loss_bce_track(li, lr, pb["cand_off"], pb["labels"], pb["rels_label"], pb["gt_tracks"],
                                       pb.multilab, None, o.lymbda, 15, max_slots=pb.n_slots))
    t = alternate(track, args.launches, args.rounds)
    res["kernels_us"]["int_rel_ch track (%d candidate rows)" % pb.n_cand] = {
        "lirec_loss_track_fwd_bwd": summary(t["margin"]), "lirec_loss_bce_track_fwd_bwd": summary(t["bce"])}
    del b, out, li, lr, track
    torch.cuda.empty_cache()

    b = make_bench("int_rels", "margin", args)
    pb = b.resident[0]
    with torch.no_grad():
        out = b.model(pb, seed=1)
    li = out.ragged_inters.contiguous()
    scale = 1.0 / li.shape[0]
    rows = dict(margin=lambda: ops.loss_rowmargin(li, pb["labels"], pb.multilab, b.opt.margin, scale),
                bce=lambda: ops.loss_bce(li, pb["labels"], pb.multilab, None, scale))
    t = alternate(rows, args.launches, args.rounds)
    res["kernels_us"]["int_rels interaction rows (%d x %d)" % tuple(li.shape)] = {
        "lirec_loss_rowmargin_fwd_bwd": summary(t["margin"]), "lirec_loss_bce_fwd_bwd": summary(t["bce"])}
    del b, out, li, rows
    torch.cuda.empty_cache()

    # ---- training steps, --loss margin vs --loss bce, alternating ----
    for preset in ("int_rel_ch", "int_rels"):
        benches = {k: make_bench(preset, k, args) for k in ("margin", "bce")}
        ms = {k: [] for k in benches}
        for k, bb in benches.items():                        # warm-up
            bb.timed_resident(3, 3, profile=False)
        for _ in range(args.rounds):
            for k, bb in benches.items():
                total, _, _ = bb.timed_resident(args.steps, 3, profile=False)
                ms[k].append(total / args.steps)
        res["step_ms"][preset] = {k: summary(v) for k, v in ms.items()}
        res["step_ms"][preset]["loss_classes"] = {k: type(bb.loss_fn).__name__ for k, bb in benches.items()}
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
