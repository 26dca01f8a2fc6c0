"""Cost of global-norm gradient clipping (--clip_grad_norm, lirec_grad_clip_flat), on int_rel_ch's flat gradient
buffer and on the benchmark's training steps (bench.py: synthetic MovieGraphs-shaped batches, HBM-resident banks).

1. Kernel time, CUDA events over >= 200 back-to-back launches per window, 5 windows alternating, median (min-max), on
   the gradients of one real int_rel_ch step (18.4 M floats, 73.7 MB):
   - not clipped (max_norm far above the norm): the norm pass reads the buffer, the scale pass returns at once;
   - clipped (coefficient ~0.999 on every launch; grad_scale grows by 1/0.999 per launch so the norm the kernel
     sees stays put and every launch clips): the norm pass reads the buffer, the scale pass reads and writes it.
   The 73.7 MB buffer fits in the 126 MB L2, so each case is timed twice: L2-warm (the same buffer every launch)
   and L2-flushed (four copies of the buffer in rotation: 221 MB pass through L2 between two uses of one copy).
   Next to them, a device-to-device copy of the same 73.7 MB, warm and in rotation.
2. Training step time (forward + loss + backward + optimizer, bench.py's device-resident leg), alternating:
   FlatAdam with its default overlap of the gate + head pass against FlatAdam + clipping (no overlap: the pass would
   update parameters before the global norm exists), and FlatLamb against FlatLamb + clipping; max_norm 1e-3 is
   below every step's norm, so every timed step clips (the dearer case).  1024 clips on int_rel_ch and int_rels,
   and 64 clips on int_rel_ch for FlatAdam.

Prints one JSON object with the GPU name and power limit next to the numbers.  Usage:
    python tools/clip_probe.py [--launches 200] [--rounds 5] [--steps 30] [--out FILE]
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
STEP_MAX_NORM = 1e-3
ROTATE = 4


def make_bench(preset, batch, optimizer, clip):
    import bench
    from lirec_b200.utils.arg_pars import opt
    bench._ARGV = []                                         # bench.py's defaults, not this script's flags
    bargs = bench.parse_args()
    if clip:
        bargs.overlap_adam = 0                               # what training() does under --clip_grad_norm
    opt.optimizer = optimizer
    opt.clip_grad_norm = STEP_MAX_NORM if clip else 0.0
    with contextlib.redirect_stdout(io.StringIO()):
        b = bench.Bench(bargs, preset, batch, 2, 0, 1, torch.device("cuda:0"))
    opt.clip_grad_norm = 0.0
    if clip:
        assert b.fused is None
        b.step = lambda pb: b.TR.train_step(b.model, b.loss_fn, b.optimizer, pb, b.world, b.fused, STEP_MAX_NORM)
    return b


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("clip_probe needs a B200")
    assert args.launches >= 200
    from lirec_b200 import ops
    res = {"gpu": gpu_info(), "launches_per_window": args.launches}

    # ---- kernels on int_rel_ch's flat gradient buffer, from one real step ----
    b = make_bench("int_rel_ch", 1024, "adam", False)
    b.step(b.resident[0])
    torch.cuda.synchronize()
    m = b.model
    n_par = sum(p.numel() for p in m._param_list)
    begin, length = m._tensor_table()
    part = ops.lamb_partials(m._flat_grad.numel(), begin.numel(), device="cuda")
    norm_out = torch.empty((), device="cuda")
    bufs = [m._flat_grad.clone() for _ in range(ROTATE)]
    g_norm = float(ops.grad_clip_flat(bufs[0], begin, length, part, 1e30, 1.0))
    res["gradient"] = {"parameters": n_par, "tensors": int(begin.numel()), "floats_with_padding": int(bufs[0].numel()),
                       "norm": g_norm}

    def clip_fn(rotate, clipped):
        """Each clipped case owns its buffers: the grad_scale of a buffer tracks what was applied to it."""
        own = [x.clone() for x in bufs[:ROTATE if rotate else 1]] if clipped else bufs
        st = {"i": 0, "scale": [1.0] * len(own), "bufs": own}

        def fn():
            k = st["i"] % ROTATE if rotate else 0
            st["i"] += 1
            if clipped:
                ops.grad_clip_flat(own[k], begin, length, part, 0.999 * g_norm, st["scale"][k], norm_out)
                st["scale"][k] /= 0.999
            else:
                ops.grad_clip_flat(own[k], begin, length, part, 1e30, 1.0, norm_out)
        fn.state = st
        return fn

    src = [torch.ones_like(bufs[0]) for _ in range(ROTATE)]
    dst = torch.empty_like(bufs[0])
    cst = {"i": 0}

    def copy_fn(rotate):
        def fn():
            k = cst["i"] % ROTATE if rotate else 0
            cst["i"] += 1
            dst.copy_(src[k])
        return fn

    fns = {"not_clipped_warm": clip_fn(False, False), "clipped_warm": clip_fn(False, True),
           "d2d_copy_warm": copy_fn(False), "not_clipped_flushed": clip_fn(True, False),
           "clipped_flushed": clip_fn(True, True), "d2d_copy_flushed": copy_fn(True)}
    t = alternate(fns, args.launches, args.rounds)
    sm = {k: summary(v) for k, v in t.items()}
    # the clipped cases clipped to the end: the norm each buffer would show its next launch is still above max_norm
    res["clipped_to_the_end"] = {}
    for k in ("clipped_warm", "clipped_flushed"):
        st = fns[k].state
        seen = [float(ops.grad_clip_flat(bb.clone(), begin, length, part, 1e30, sc))
                for bb, sc in zip(st["bufs"], st["scale"])]
        res["clipped_to_the_end"][k] = {"launches": st["i"], "min_norm_over_max_norm": min(seen) / (0.999 * g_norm)}
    nbytes = {"not_clipped": 4 * n_par, "clipped": 12 * n_par, "d2d_copy": 8 * bufs[0].numel()}

    def rate(bytes_, us):
        gbs = bytes_ / us / 1e3
        return {"GB/s": round(gbs, 1), "of_datasheet": round(gbs / DATASHEET_GBS, 3)}

    res["kernels_us"] = sm
    res["bytes_per_call"] = nbytes
    res["achieved"] = {k: rate(nbytes[k.rsplit("_", 1)[0]], v["median"]) for k, v in sm.items()}
    b.close()
    del b, m, bufs, src, dst, fns
    torch.cuda.empty_cache()

    # ---- training steps, alternating ----
    res["step_ms"] = {}
    legs = [("int_rel_ch", 1024, ("adam", "lamb")), ("int_rels", 1024, ("adam", "lamb")), ("int_rel_ch", 64, ("adam",))]
    for preset, batch, optimizers in legs:
        benches = {}
        for o in optimizers:
            benches[o] = make_bench(preset, batch, o, False)
            benches[o + "+clip"] = make_bench(preset, batch, o, True)
        ms = {k: [] for k in benches}
        for bb in benches.values():                          # warm-up
            bb.timed_resident(3, 3, profile=False)
        for _ in range(args.rounds):
            for k, bb in benches.items():
                total, _, _ = bb.timed_resident(args.steps, 3, profile=False)
                ms[k].append(total / args.steps)
        key = "%s@%d" % (preset, batch)
        res["step_ms"][key] = {k: summary(v) for k, v in ms.items()}
        res["step_ms"][key]["optimizers"] = {
            k: "%s%s%s" % (type(bb.optimizer).__name__, " + overlapped gate/head pass" if bb.fused is not None else "",
                           " + clip" if k.endswith("+clip") else "")
            for k, bb in benches.items()}
        res["step_ms"][key]["last_norm"] = {k: float(bb.model._last_grad_norm) for k, bb in benches.items()
                                            if k.endswith("+clip")}
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
