#!/usr/bin/env python
"""Where does the overlapped pass really run?  One GPU, `--overlap_adam`-style step (gate + head bucket's Adam on
a side stream behind the heads-final event of backward), with timing events on both streams:

    t_heads   heads-final event (recorded mid-backward by lirec_model_backward)
    t_a_done  end of the side-stream pass
    t_bwd     end of backward on the main stream (before the encoder bucket's Adam)
    t_end     end of the step

all in microseconds after the step's first kernel.  The pass overlaps backward iff t_a_done < t_bwd.  Also prints the
HOST time spent enqueuing a step (no synchronisation inside the loop): a step whose host time equals its device
time is launch-bound, not kernel-bound.

    python tools/overlap_probe.py [--batch 1024] [--steps 60]       (LIREC_DP_CORESIDENT=0/1 for the A/B)
"""
import argparse
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--no_overlap", action="store_true", help="plain Adam launch after backward (the baseline)")
    a = ap.parse_args()
    import bench
    bench._ARGV = ["--overlap_adam", "0" if a.no_overlap else "1", "--batch", str(a.batch)]
    args = bench.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    b = bench.Bench(args, "int_rel_ch", a.batch, 4, 0, 1, dev)
    f = b.fused
    assert a.no_overlap or f is not None, "overlap needs the fused flat Adam"
    if f is not None:
        # timing-enabled events in place of the step's own (the library re-records ev_heads by handle)
        f.ev_heads = torch.cuda.Event(enable_timing=True)
        f.ev_heads.record()
        f.ev_done = torch.cuda.Event(enable_timing=True)
    import lirec_b200.mlp.model as M
    from lirec_b200 import dp

    def one(pb, evs):
        if f is not None:
            f.arm(True)
        if evs:
            evs[0].record()
        M.train_step(b.model, b.loss_fn, pb)
        if evs:
            evs[1].record()
        dp.reduce_and_step(b.model, b.optimizer, f, None, None)
        if evs:
            evs[2].record()

    for i in range(10):
        one(b.resident[i % 4], None)
    torch.cuda.synchronize()
    rows = []
    for i in range(a.steps if f is not None else 0):
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        one(b.resident[i % 4], evs)
        torch.cuda.synchronize()
        t0 = evs[0]
        rows.append([t0.elapsed_time(f.ev_heads) * 1e3, t0.elapsed_time(f.ev_done) * 1e3,
                     t0.elapsed_time(evs[1]) * 1e3, t0.elapsed_time(evs[2]) * 1e3])
    r = np.median(np.array(rows), axis=0) if rows else np.zeros(4)
    if rows:
        print("B=%d coresident=%s  median us after step start: heads-final %.0f | side pass done %.0f | backward done "
              "%.0f | step done %.0f   -> side pass ends %+.0f us relative to backward's end"
              % (a.batch, os.environ.get("LIREC_DP_CORESIDENT", "1"), r[0], r[1], r[2], r[3], r[1] - r[2]))
    # host enqueue time vs device time of free-running steps
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 200
    e0.record()
    h0 = time.perf_counter()
    for i in range(n):
        one(b.resident[i % 4], None)
    h1 = time.perf_counter()
    e1.record()
    torch.cuda.synchronize()
    print("B=%d %s free-running: host enqueue %.1f us/step, device %.1f us/step" %
          (a.batch, "plain Adam" if f is None else "overlapped Adam", (h1 - h0) / n * 1e6, e0.elapsed_time(e1) / n * 1e3))


if __name__ == "__main__":
    main()
