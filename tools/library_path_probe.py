"""The "library path" on the same B200 (SURVEY.md §8d, optional row): the reference's schedule — DENSE zero-padded
batches, one ATen call per op, autograd, torch.optim.Adam — run by stock PyTorch eager ON THE GPU, next to this
package's packed / fused path on the same synthetic clips.  The reference tree is not part of this repository, so
the dense model + loss are the oracle's restatement (pinned against the unmodified reference, tests/golden,
tests/test_oracle_golden.py) with its tensors moved to cuda:0; matmuls run as TF32 tensor-core GEMMs
(cuBLAS), everything else as the usual elementwise ATen kernels.

    python tools/library_path_probe.py [--batches 64,256] [--preset int_rel_ch]

Development / measurement tool like tools/precision_study.py: it imports oracle/ and is not part of the product.
"""
import argparse
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def eager_gpu(preset, pb, steps, warmup):
    from oracle import cpu_baseline as cb
    step = cb.CpuStep(preset)                                   # parameters drawn on the CPU generator, as always
    step.sd = {k: v.detach().cuda().requires_grad_(True) for k, v in step.sd.items()}
    step.opt = torch.optim.Adam(list(step.sd.values()), lr=3e-5, weight_decay=1e-5)
    dense = {k: (v.cuda() if isinstance(v, torch.Tensor) else v) for k, v in pb.to_dense(np.float32).items()}
    torch.set_default_device("cuda")                            # the oracle's torch.arange / zeros / ones follow
    try:
        for _ in range(warmup):
            step.train_step(dense)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step.train_step(dense)
        e1.record()
        torch.cuda.synchronize()
    finally:
        torch.set_default_device(None)                          # "cpu" would leave a function mode on every torch call
    return e0.elapsed_time(e1) / steps, dense["features"].numel() * 4


def ours(preset, pb, steps, warmup):
    import bench
    bench._ARGV = ["--batch", str(pb.B), "--preset", preset, "--no_configs", "--no_cpu_baseline", "--no_traffic"]
    args = bench.parse_args()
    dev = torch.device("cuda:0")
    b = bench.Bench(args, preset, pb.B, 4, 0, 1, dev)
    for i in range(warmup):
        b.step(b.resident[i % len(b.resident)])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        b.step(b.resident[i % len(b.resident)])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="64,256")
    ap.add_argument("--preset", default="int_rel_ch")
    ap.add_argument("--steps", type=int, default=10)
    a = ap.parse_args()
    sys.argv = sys.argv[:1]
    from lirec_b200.mixed_utils import synthetic
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.allow_tf32 = True
    print("# library path (stock PyTorch eager, dense batches, TF32 matmuls, autograd, torch.optim.Adam) vs lirec_b200 "
          "on %s, preset %s, train step = fwd + loss + bwd + Adam" % (torch.cuda.get_device_name(0), a.preset))
    for B in [int(x) for x in a.batches.split(",")]:
        pb = synthetic.make_batch(B, seed=0, preset=a.preset)
        ms_o = ours(a.preset, pb, 20 * a.steps, 5)
        torch.cuda.empty_cache()
        ms_e, nbytes = eager_gpu(a.preset, pb, a.steps, 2)
        print("B=%4d  dense batch %7.1f MB  eager %9.3f ms/step %9.0f clips/s | lirec_b200 %7.3f ms/step %9.0f clips/s "
              "| x%.1f" % (B, nbytes / 1e6, ms_e, B / ms_e * 1e3, ms_o, B / ms_o * 1e3, ms_e / ms_o))
        sys.stdout.flush()
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
