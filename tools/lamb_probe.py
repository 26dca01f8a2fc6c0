"""Cost of the fused LAMB step (--optimizer lamb) next to the fused Adam step it replaces, on int_rel_ch's flat
parameter buffer and on the benchmark's training steps (bench.py: synthetic MovieGraphs-shaped batches of 1024 clips,
HBM-resident banks).

1. Kernel time, CUDA events over >= 200 back-to-back launches per window, alternating window by window:
   lirec_lamb_flat (two launches) vs lirec_adam_flat over the whole flat buffer, and a device-to-device copy for
   the bandwidth the memory system gives in the same run.  Each window is queued behind a device-side spin, so the
   events time the GPU executing the launches, not the host issuing them.  The working set (774 MB for LAMB) is six
   times the 126 MB L2, so every pass streams from HBM.
   Bytes per parameter: LAMB 42 (pass 1 reads g, w, m, v and writes m, v; pass 2 reads m, v, w and writes w and the
   bf16 shadow), Adam 30 (reads g, w, m, v; writes w, m, v and the bf16 shadow).
2. Training step time (forward + loss + backward + optimizer, bench.py's device-resident leg) with --optimizer lamb
   vs FlatAdam with its default overlap of the gate + head pass with backward, alternating.

Prints one JSON object with the GPU name and power limit next to the numbers.  Usage:
    python tools/lamb_probe.py [--launches 200] [--rounds 5] [--steps 30] [--out FILE]
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


def make_bench(preset, optimizer, args):
    import bench
    from lirec_b200.utils.arg_pars import opt
    bench._ARGV = []                                         # bench.py's defaults, not this script's flags
    bargs = bench.parse_args()
    opt.optimizer = optimizer
    with contextlib.redirect_stdout(io.StringIO()):
        b = bench.Bench(bargs, preset, args.batch, 2, 0, 1, torch.device("cuda:0"))
    return b


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("lamb_probe needs a B200")
    assert args.launches >= 200
    from lirec_b200 import ops
    res = {"gpu": gpu_info(), "batch_clips": args.batch, "launches_per_window": args.launches}

    # ---- kernels on int_rel_ch's flat buffer, with the gradients of one real step ----
    b = make_bench("int_rel_ch", "adam", args)
    b.step(b.resident[0])
    torch.cuda.synchronize()
    m = b.model
    g = b.optimizer.param_groups[0]
    n_par = sum(p.numel() for p in m._param_list)
    n_tensors = len(m._param_list)
    m2, v2 = torch.zeros_like(m._flat), torch.zeros_like(m._flat)
    begin = torch.tensor(m._offsets, dtype=torch.int64, device="cuda")
    length = torch.tensor([p.numel() for p in m._param_list], dtype=torch.int64, device="cuda")
    part = ops.lamb_partials(m._flat.numel(), n_tensors, device="cuda")
    # 1e-9: the timed windows take thousands of steps; keep the weights where they are
    fns = dict(
        lamb=lambda: ops.lamb_flat(m._flat, m._flat_grad, m2, v2, m._flat_bf16, begin, length, part, 1e-9, 0.9, 0.999,
                                   1e-6, g["weight_decay"], 10, 1.0),
        adam=lambda: ops.adam_flat(m._flat, m._flat_grad, b.optimizer._m, b.optimizer._v, m._flat_bf16, 1e-9, 0.9,
                                   0.999, 1e-8, g["weight_decay"], 10, 1.0))
    copy_bytes = 42 * n_par // 2                             # read + write = LAMB's traffic
    src = torch.empty(copy_bytes // 4, dtype=torch.float32, device="cuda").fill_(1.0)
    dst = torch.empty_like(src)
    fns["d2d_copy"] = lambda: dst.copy_(src)
    t = alternate(fns, args.launches, args.rounds)
    sm = {k: summary(v) for k, v in t.items()}
    lamb_bytes, adam_bytes = 42 * n_par, 30 * n_par
    copy_gbs = 2 * copy_bytes / sm["d2d_copy"]["median"] / 1e3

    def rate(bytes_, us):
        gbs = bytes_ / us / 1e3
        return {"GB/s": round(gbs, 1), "of_d2d_copy": round(gbs / copy_gbs, 3), "of_datasheet": round(gbs / DATASHEET_GBS, 3)}

    res["flat_buffer"] = {"parameters": n_par, "tensors": n_tensors, "floats_with_padding": int(m._flat.numel())}
    res["kernels_us"] = {"lirec_lamb_flat": sm["lamb"], "lirec_adam_flat": sm["adam"], "d2d_copy": sm["d2d_copy"]}
    res["bytes_per_step"] = {"lamb": lamb_bytes, "adam": adam_bytes, "d2d_copy": 2 * copy_bytes}
    res["achieved"] = {"lirec_lamb_flat": rate(lamb_bytes, sm["lamb"]["median"]),
                       "lirec_adam_flat": rate(adam_bytes, sm["adam"]["median"]),
                       "d2d_copy": {"GB/s": round(copy_gbs, 1), "of_datasheet": round(copy_gbs / DATASHEET_GBS, 3)}}
    b.close()
    del b, m, m2, v2, part, src, dst, fns
    torch.cuda.empty_cache()

    # ---- training steps, FlatAdam (default overlap) vs FlatLamb, alternating ----
    res["step_ms"] = {}
    for preset in ("int_rel_ch", "int_rels"):
        benches = {k: make_bench(preset, k, args) for k in ("adam", "lamb")}
        ms = {k: [] for k in benches}
        for k, bb in benches.items():                        # warm-up
            bb.timed_resident(3, 3, profile=False)
        for _ in range(args.rounds):
            for k, bb in benches.items():
                total, _, _ = bb.timed_resident(args.steps, 3, profile=False)
                ms[k].append(total / args.steps)
        res["step_ms"][preset] = {k: summary(v) for k, v in ms.items()}
        res["step_ms"][preset]["optimizers"] = {
            k: "%s%s" % (type(bb.optimizer).__name__, " + overlapped gate/head pass" if bb.fused is not None else "")
            for k, bb in benches.items()}
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
