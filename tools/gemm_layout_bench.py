"""Throughput of the grouped tcgen05 GEMM by operand layout (K-major / MN-major), one problem per
launch, against cuBLAS bf16 on the same shape.  Diagnostic; run on a B200:
    python tools/gemm_layout_bench.py"""
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from lirec_b200 import _ext, ops

_ext.require_device()
dev = "cuda"


def rnd(r, c):
    return torch.randn(r, c, device=dev).to(torch.bfloat16)


def timeit(fn, iters=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def run(M, N, K, a_mn, b_mn, passes=1):
    a = rnd(K, M) if a_mn else rnd(M, K)
    b = rnd(K, N) if b_mn else rnd(N, K)
    out = torch.empty(M, N, device=dev)
    ps = [(_ext.operand(a), 0, 0, _ext.operand(b), 0, 0, K)] * passes
    g = ops.gemm_problem(M, N, ps, a_mn_major=a_mn, b_mn_major=b_mn, out=out)
    ms = timeit(lambda: ops.gemm_grouped([g]))
    fl = 2.0 * M * N * K * passes
    A = a.t() if a_mn else a
    Bt = b if b_mn else b.t()
    ms_ref = timeit(lambda: torch.matmul(A, Bt))
    print("M=%-6d N=%-5d K=%-6d passes=%d A=%s B=%s : %.3f ms %7.1f TFLOP/s | cuBLAS(1 pass) %.3f ms %7.1f TFLOP/s" % (
        M, N, K, passes, "MN" if a_mn else "K ", "MN" if b_mn else "K ", ms, fl / ms / 1e9, ms_ref,
        2.0 * M * N * K / ms_ref / 1e9))
    sys.stdout.flush()


if __name__ == "__main__":
    print(torch.cuda.get_device_name(0))
    for (M, N, K) in [(8192, 3072, 6144), (8448, 3072, 3072), (3072, 1536, 8384)]:
        for a_mn, b_mn in [(False, False), (False, True), (True, False), (True, True)]:
            run(M, N, K, a_mn, b_mn)
    run(3072, 1536, 8384, True, True, passes=3)       # gate wgrad (hi.hi + hi.lo + lo.hi)
    run(8448, 1536, 3072, False, True, passes=2)      # gate dgrad
    run(512, 2048, 28032, True, True, passes=2)       # layer-1 wgrad on the unique track rows
    run(8448, 512, 512, False, False, passes=2)       # layer 2
    run(28032, 512, 2048, False, False)               # layer 1
