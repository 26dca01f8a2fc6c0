"""In-kernel timeline of the grouped GEMM launches of ONE train step (variant build with -DLIREC_GEMM_TRACE=1):

    bash tools/build_variants.sh "trace:-DLIREC_GEMM_TRACE=1"
    gpurun -- 'LIREC_B200_LIB=$PWD/variants/trace.so python tools/gemm_trace.py > gpurun_out/gemm_trace.txt'

Every persistent worker (CTA pair) stamps clock64() per tile: producer first / last TMA issue, MMA waiting for a free
accumulator / accumulator free / first operands landed / last commit issued, epilogue woken / done.  The summary
prints, per launch, the median per-tile durations of those phases in microseconds (SM clock taken as 1.9 GHz) and how
much of a worker's time the MMA thread spent waiting for operands vs for the epilogue."""
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GHZ = float(os.environ.get("LIREC_TRACE_GHZ", "1.9"))


def main():
    path = tempfile.mktemp(suffix=".trace")
    env = dict(os.environ, LIREC_GEMM_TRACE_FILE=path)
    args = sys.argv[1:] or ["--steps", "1", "--warmup", "3"]
    # warm-up steps are traced too: keep the LAST step's launches
    subprocess.run([sys.executable, os.path.join(HERE, "bench.py"), "--only_value"] + args, env=env, check=True,
                   stdout=subprocess.DEVNULL)
    launches, cur = [], None
    with open(path) as f:
        for line in f:
            if line.startswith("launch"):
                t = line.split()
                cur = dict(idx=int(t[1]), units=int(t[3]), tiles=int(t[5]), problems=int(t[7]), rows=[])
                launches.append(cur)
            else:
                cur["rows"].append([int(x) for x in line.split()])
    per_step = 8
    last = launches[-per_step:]
    us = lambda c: c / (GHZ * 1e3)
    print("# per launch: tiles, workers; median per-tile phase durations in us (SM clock %.2f GHz assumed)" % GHZ)
    print("# prod = first..last TMA issue of the tile; acc_wait = MMA waits for a free accumulator (epilogue-bound);")
    print("# op_wait = accumulator free .. first operands landed (load-bound); mma = first operands .. last commit issued;")
    print("# epi = epilogue woken .. done; tile = accumulator-free(k) .. accumulator-free(k+1) on the MMA thread")
    for L in last:
        a = np.array(L["rows"], dtype=np.float64).reshape(L["units"], 64, 8)
        valid = a[:, :, 3] > 0
        prod = (a[:, :, 1] - a[:, :, 0])[valid]
        accw = (a[:, :, 3] - a[:, :, 2])[valid]
        opw = (a[:, :, 4] - a[:, :, 3])[valid]
        mma = (a[:, :, 5] - a[:, :, 4])[valid]
        epi = (a[:, :, 7] - a[:, :, 6])[valid & (a[:, :, 6] > 0)]
        nt = valid.sum(1)
        span = []
        for u in range(L["units"]):
            k = int(nt[u])
            if k:
                span.append(a[u, k - 1, 7] - a[u, 0, 0])
        tile = []
        for u in range(L["units"]):
            k = int(nt[u])
            tile += list(np.diff(a[u, :k, 3]))
        med = lambda x: float(np.median(x)) if len(x) else 0.0
        print("tiles %4d workers %3d tiles/worker %.2f | prod %6.2f acc_wait %6.2f op_wait %6.2f mma %6.2f epi %6.2f tile %6.2f | "
              "worker span median %.1f us max %.1f us" % (
                  L["tiles"], L["units"], L["tiles"] / L["units"], us(med(prod)), us(med(accw)), us(med(opw)), us(med(mma)),
                  us(med(epi)), us(med(tile)), us(med(span)), us(max(span) if span else 0)))
    os.unlink(path)


if __name__ == "__main__":
    main()
