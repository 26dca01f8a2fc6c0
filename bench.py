#!/usr/bin/env python
"""bench.py — headline benchmark of the LIReC hot path on B200.

metric  : train clips/sec, int_rel_ch forward + loss + backward (+ gradient exchange) + Adam
workload: synthetic MovieGraphs-shaped clips (SURVEY.md §8d C4) whose pooled vectors are cached once in
          dataset-level banks (mixed_utils/cached_clips.py — the reference's cache() / __getitem__ split),
          random-init weights of the reference architecture, bf16 tensor-core operands with hi/lo-split
          activations (fp32-grade products) and fp32 accumulation.

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun)
  python bench.py --preset {modalities,int_rels,int_ch,int_rel_ch,stress} [--batch B]
  python bench.py --impl reference ...                      CPU arm: oracle port of the reference
  python bench.py ... --dump-outputs DIR                    also write the last timed step's loss, parameters and
                                                            gradients as .npy files (same arguments, same inputs)

One JSON line on stdout (rank 0).
  value   device-resident throughput (batches already staged in HBM).
  e2e     the same step driven by the product's loader: `packed_loader(dataset, num_workers=k)` — index-only
          items, native collate in worker processes, pinning, async H2D of the integer tables, device gather
          of the batch banks from the HBM-resident dataset banks, step, D2H of the loss — all inside the
          timed region.  `e2e_precollated` / `e2e_streamed` time batches collated ahead of the clock
          (index-only, and with all feature rows crossing PCIe every step).
  configs every BASELINE.json configuration (modalities, int_rels, int_ch, int_rel_ch, stress) at the
          reference batch size and at the throughput size: clips/s, ms/step, GEMM roofline, cpu_baseline.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

_ARGV = sys.argv[1:]
sys.argv = sys.argv[:1]          # utils.arg_pars parses argv at import (reference behaviour)

import numpy as np  # noqa: E402
import torch  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

# algorithmic MACs per encoder row / candidate row (SURVEY.md §8d)
E1 = 768 * 512 + 3 * 2048 * 512
E2 = 2 * 512 * 512 + 2 * 512 * 256
E = E1 + E2
G = 3072 * 3072
H_I = 3072 * 101
H_I_NOGATE = 1536 * 101
H_R = 1536 * 15

# flag presets of the reference's entry points (resume/modalties.py:79-100, int_rels.py:88-115,
# int_ch.py:77-117, int_rel_ch.py:87-124); "stress" = BASELINE config 5 (4x context rows, 4x candidate slots)
PRESETS = {
    "modalities": dict(model="modalities", flags=dict(mod_check=True, tr_maximize=False, ints=1, ctx=0, gates=0,
                                                      rels_multitask=False, rels_multi_clip=False)),
    "int_rels": dict(model="int_rels", flags=dict(mod_check=False, tr_maximize=False, ints=1, ctx=1, gates=1,
                                                  rels_multitask=True, rels_multi_clip=True, rels_n_clips=18)),
    "int_ch": dict(model="int_ch", flags=dict(mod_check=False, tr_maximize=True, ints=1, ctx=0, gates=0,
                                              rels_multitask=False, rels_multi_clip=False)),
    "int_rel_ch": dict(model="int_rel_ch", flags=dict(mod_check=False, tr_maximize=True, ints=1, ctx=1, gates=1,
                                                      rels_multitask=True, rels_multi_clip=True, rels_n_clips=18)),
    "stress": dict(model="int_rel_ch", flags=dict(mod_check=False, tr_maximize=True, ints=1, ctx=1, gates=1,
                                                  rels_multitask=True, rels_multi_clip=True, rels_n_clips=72,
                                                  max_n_tripl=80),
                   clip_kwargs=dict(n_chars_probs={k: 1.0 / 7 for k in range(2, 9)})),
}
WORKLOAD_TEXT = {
    "modalities": "modalities (Modalities + MaxMarginCrossEntropyLoss + Adam) train step",
    "int_rels": "int_rels (MidFusionMultiClip + MultiTaskMaxMargin + Adam) train step",
    "int_ch": "int_ch (MidFusionMultiClipMaxTracks + MarginLoss + Adam) train step",
    "int_rel_ch": "int_rel_ch (MidFusionMultiClipMaxTracks + MarginTrackRelsLoss + Adam) train step",
    "stress": "long-clip stress (int_rel_ch model, 72 context rows x 80 candidate slots per clip) train step",
}


def algorithmic_flops(preset, n_cand, n_ctx_rows):
    """fwd+bwd FLOPs of one step over valid rows only, no credit for dedup (SURVEY.md §8d)."""
    model = PRESETS[preset]["model"]
    if model in ("modalities", "int_ch"):
        fwd = n_cand * (E + H_I_NOGATE)
        bwd = 2 * fwd - n_cand * E1
    else:
        fwd = (n_cand + n_ctx_rows) * E + n_cand * (G + H_I + H_R)
        bwd = 2 * fwd - (n_cand + n_ctx_rows) * E1
    return 2.0 * (fwd + bwd)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="clips per GPU per step (default 1024; stress 256)")
    ap.add_argument("--preset", default="int_rel_ch", choices=sorted(PRESETS))
    ap.add_argument("--n_batches", type=int, default=4, help="distinct synthetic batches rotated per rank")
    ap.add_argument("--workers", type=int, default=-1, help="loader worker processes of the e2e leg (-1: auto)")
    ap.add_argument("--cpu_clips", type=int, default=64, help="clips per CPU-baseline step (bounded sample)")
    ap.add_argument("--no_cpu_baseline", action="store_true")
    ap.add_argument("--no_configs", action="store_true", help="skip the per-configuration table (`configs`)")
    ap.add_argument("--no_traffic", action="store_true", help="skip the live DRAM-traffic capture (ncu child process)")
    ap.add_argument("--only_value", action="store_true", help="device-resident leg only (profiling runs)")
    ap.add_argument("--dump_profile", default="", help="write the per-launch GEMM event timings to this file")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step computed to DIR/{loss,params,grads}.npy (see dump_outputs)")
    ap.add_argument("--nccl_allreduce", action="store_true",
                    help="N > 1: use ncclAllReduce + Adam instead of the in-switch reduce + Adam kernels")
    ap.add_argument("--dp_mode", default="", choices=["", "shard", "bucket"],
                    help="N > 1: 'shard' (default) = in-switch sum + sharded Adam + parameter multicast in one pass; "
                         "'bucket' = in-switch sum and full-replica Adam per bucket")
    ap.add_argument("--no_overlap", action="store_true",
                    help="N > 1, --dp_mode bucket: run the whole exchange after backward (no bucket overlapped with it)")
    ap.add_argument("--overlap_adam", type=int, default=1,
                    help="N = 1: run the gate + head bucket's Adam pass on a side stream during backward (default 1, "
                         "as lirec_b200/mlp/train.py does; 0 = one Adam launch after backward)")
    ap.add_argument("--autograd_step", action="store_true",
                    help="drive the step through model()/loss()/backward()/optimizer.step() and the autograd engine "
                         "(the drop-in surface) instead of lirec_b200.mlp.train.train_step's native sequence")
    ap.add_argument("--ncu_window", action="store_true",
                    help="bracket the device-resident timed loop with cudaProfilerStart/Stop "
                         "(run under `ncu --profile-from-start off`; numbers printed under ncu are not bench values)")
    return ap.parse_args(_ARGV)


class ClockSampler:
    """SM clock, power and throttle reasons sampled DURING the timed regions (NVML, every ~10 ms; falls back to
    an `nvidia-smi -lms` child process).  The poller runs for the whole bench and stamps every sample with its host
    time; region(True / False) only records the interval, and the samples are sorted into the regions at the end."""
    REASONS = (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown", 0x8),
               ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
               ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
               ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap", 0x4))

    def __init__(self, index):
        self.index, self.sm, self.power, self.reasons, self.mx = index, [], [], set(), None
        self.tag, self.by_tag = "value", {}          # samples per named region: tag -> ([sm], [power], {reasons})
        # the poller runs from start() to stop() at its own cadence (an idle poller needs 10-20 ms to deliver its
        # first sample: too long for a 40 ms region); every sample carries its host time and is assigned to the
        # timed region whose [begin, end] interval it falls into
        self.samples, self.spans, self._open = [], [], None
        self._stop = threading.Event()
        self.thread = self.proc = None
        self.active = False

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else self.index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nv = pynvml
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
        except Exception:
            self._start_smi()

    def _poll(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                t0 = time.perf_counter()
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                try:
                    bits = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((0.5 * (t0 + time.perf_counter()), sm, pw,
                                     [name for name, _, bit in self.REASONS if bits & bit]))
            except Exception:
                pass
            time.sleep(float(os.environ.get("LIREC_BENCH_SAMPLE_S", "0.01")))

    def _start_smi(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "10"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read_smi, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read_smi(self):
        names = [r[0] for r in self.REASONS]
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm, pw = float(f[0]), float(f[2])
                self.mx = float(f[1])
            except ValueError:
                continue
            self.samples.append((time.perf_counter(), sm, pw,
                                 [name for name, v in zip(names, f[3:7]) if v.lower().startswith("active")]))

    def _add(self, sm, pw, reasons):
        self.sm.append(sm)
        self.power.append(pw)
        self.reasons.update(reasons)
        t = self.by_tag.setdefault(self.tag, ([], [], set()))
        t[0].append(sm), t[1].append(pw), t[2].update(reasons)

    def region(self, on, tag=None):
        """Sampling on / off; `tag` names the timed region the samples belong to ("value" = the K timed steps the
        headline number comes from, "e2e" = the end-to-end legs, ...)."""
        if tag is not None:
            self.tag = tag
        now = time.perf_counter()
        if on and self._open is None:
            self._open = (self.tag, now)
        elif not on and self._open is not None:
            self.spans.append((self._open[0], self._open[1], now))
            self._open = None
        self.active = bool(on)

    def _assign(self):
        """Sort the time-stamped samples into the timed regions (idempotent)."""
        self.sm, self.power, self.reasons, self.by_tag = [], [], set(), {}
        for t, sm, pw, rs in list(self.samples):
            for tag, a, b in self.spans:
                if a <= t <= b:
                    self.tag = tag
                    self._add(sm, pw, rs)
                    break

    def summary(self, tag):
        sm, pw, rs = self.by_tag.get(tag, ([], [], set()))
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_min_mhz": float(np.min(sm)), "sm_max_mhz": self.mx,
                "power_w_max": float(np.max(pw)) if pw else None, "reasons": sorted(rs), "samples": len(sm)}

    def stop(self):
        self._stop.set()
        if self.proc is not None:
            self.proc.terminate()
        self._assign()
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.mx, "reasons": ["no samples"], "samples": 0}
        # the headline `clocks` are those of the region `value` was timed in; the other regions ride along
        main = self.summary("value") or {"sm_mhz": float(np.median(self.sm)), "sm_min_mhz": float(np.min(self.sm)),
                                         "sm_max_mhz": self.mx, "power_w_max": float(np.max(self.power)) if self.power else None,
                                         "reasons": sorted(self.reasons), "samples": len(self.sm)}
        main["how"] = ("NVML (fallback: nvidia-smi -lms) polled every ~10 ms for the whole run, every sample time-stamped; "
                       "counted here are the samples that fall INSIDE the K timed steps `value` comes from, `by_region` "
                       "has those inside the other timed legs")
        main["by_region"] = {t: self.summary(t) for t in sorted(self.by_tag) if t != "value"}
        return main


def usable_cores():
    """Host cores this process may actually use: the affinity mask, capped by a cgroup-v2 CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


def load_peaks():
    pk = {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm": 6650.0, "source": "fallback (B200_PROFILING.md)"}
    path = os.path.join(HERE, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            j = json.load(f)
        pk = {"bf16_burst": float(j.get("bf16_tflops", 1590.0)),
              "bf16_sustained": float(j.get("bf16_tflops_sustained", j.get("bf16_tflops", 1400.0))),
              "hbm": float(j.get("hbm_gbs", 6650.0)), "source": "MEASURED_PEAKS.json"}
    return pk


def pick_tensor_peak(pk, region_ms, clocks):
    """Burst peak for a region the 1 kW power cap has not caught up with (short, or SM clock still within 5 % of
    its maximum), else the sustained one (B200_PROFILING.md: burst for a kernel timed alone, sustained inside a
    long step)."""
    sm, mx = (clocks or {}).get("sm_mhz"), (clocks or {}).get("sm_max_mhz")
    capped = "sw_power_cap" in ((clocks or {}).get("reasons") or [])
    if sm and mx:
        burst = sm >= 0.95 * mx and not capped
    else:
        burst = region_ms < 1000.0
    return (pk["bf16_burst"], "bf16_tflops (burst)") if burst else (pk["bf16_sustained"], "bf16_tflops_sustained")


def apply_preset(opt, preset, **over):
    flags = dict(tracks=True, modality="m", device="cuda", fused_adam=1, tr_correct=False, tr_max_neg=False,
                 tr_cat_distr=False, tr_sum_max_flag=True, max_n_tripl=20, rels_n_clips=18, synthetic=3,
                 resident_banks=1, native_step=1)
    flags.update(PRESETS[preset]["flags"])
    flags.update(over)
    for k, v in flags.items():
        setattr(opt, k, v)


def cpu_baseline_line(preset, cpu_clips, steps, warmup):
    """The reference's CPU path (oracle port) on a bounded sample of the same workload."""
    from lirec_b200.mixed_utils import synthetic
    from oracle import cpu_baseline as cb
    torch.set_num_threads(os.cpu_count() or 1)
    model = PRESETS[preset]["model"]
    if preset == "stress":
        cpu_clips = min(cpu_clips, 2)                      # 323 MB of dense float64 per clip
        pb = synthetic.stress_batch(cpu_clips, seed=0)
    else:
        pb = synthetic.make_batch(cpu_clips, seed=0, preset=model)
    dense = pb.to_dense(np.float64)
    # the unmodified reference itself where its tree is mounted (the build container); its oracle port elsewhere
    # (the GPU box has no /root/reference: a Python reference cannot travel)
    kind = "port"
    from oracle import reference_shim as rs
    if rs.available() and preset != "stress" and os.environ.get("LIREC_BENCH_LIVE_REFERENCE", "1") != "0":
        r = cb.time_train_reference(model, dense, steps=steps, warmup=warmup)
        kind = "reference"
    else:
        r = cb.time_train(model, dense, steps=steps, warmup=warmup)
    return {"value": r["clips_per_s_mean"], "unit": "clips/s", "cores": r["threads"], "kind": kind,
            "sample": "%d-clip dense float64 batch (reference dataloader format, %s), %d timed train steps "
                      "(fwd+loss+bwd+Adam, dropout 0.3, fp32 torch CPU) after %d warm-up%s" % (
                          cpu_clips, preset, steps, warmup,
                          "; the UNMODIFIED reference model / loss / torch Adam (tree mounted)" if kind == "reference"
                          else "; oracle port of the reference (its tree is not on this box)"),
            "ms_per_step": 1e3 * cpu_clips / r["clips_per_s_mean"]}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(1, min(args.steps, 5)), max(1, min(args.warmup, 2))
    cb = cpu_baseline_line(args.preset, args.cpu_clips, steps, warmup)
    line = {"impl": "reference", "metric": "train clips/sec (%s fwd+bwd)" % args.preset, "value": cb["value"],
            "unit": "clips/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
            "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "%s, %d-clip dense batch per step on host CPU" % (WORKLOAD_TEXT[args.preset],
                                                                                     args.cpu_clips),
                       "preset": args.preset},
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


PROFILE_EVERY = 8


class Bench:
    """One (preset, clips-per-GPU) configuration: model, loss, optimizer, cached dataset, staged batches."""

    def __init__(self, args, preset, batch, n_batches, rank, world, dev, fused_ok=True):
        import contextlib
        import io
        from lirec_b200 import dp
        from lirec_b200.utils.arg_pars import opt
        from lirec_b200.mixed_utils.cached_clips import CachedClipsDataset
        from lirec_b200.mixed_utils.indexed_dataset import ResidentBanks
        import lirec_b200.mlp.model as M
        self.args, self.preset, self.batch, self.rank, self.world, self.dev = args, preset, batch, rank, world, dev
        self.opt = opt
        apply_preset(opt, preset)
        opt.native_step = 0 if args.autograd_step else 1
        opt.batch_size = batch
        torch.manual_seed(opt.seed)
        with contextlib.redirect_stdout(io.StringIO()):
            self.model, self.loss_fn, self.optimizer = M.create_model(101, n_rels=15)
        self.model.train()
        dp.broadcast_params(self.model._flat)
        if world > 1:
            self.model.set_rank(rank)
            if hasattr(self.loss_fn, "set_rank"):
                self.loss_fn.set_rank(rank)
        # gradient exchange (N > 1: in-switch, bucketed) + Adam, the gate + head bucket overlapped with backward;
        # N = 1: only the overlapped bucket-0 Adam pass
        self.fused = None
        if world > 1 and not args.nccl_allreduce and fused_ok:
            self.fused = dp.SwitchReduceAdam.attach(self.model, self.optimizer, mode=args.dp_mode or None)
            if self.fused is not None and args.no_overlap:
                self.fused.overlap = False
        elif world == 1 and args.overlap_adam:
            self.fused = dp.SwitchReduceAdam.attach(self.model, self.optimizer, single_gpu=True)
        # the rank's dataset: n_batches * batch distinct clips, cached once (the reference's dataset.cache())
        self.dataset = CachedClipsDataset("train", size=n_batches * batch, preset=PRESETS[preset]["model"],
                                          seed_base=(1000 * rank + 17) * 1000003,
                                          max_n_tripl=opt.max_n_tripl, rels_n_clips=opt.rels_n_clips,
                                          clip_kwargs=PRESETS[preset].get("clip_kwargs"))
        self.dataset.cache()
        self.banks = ResidentBanks(self.dataset, dev)
        self.dataset._resident = self.banks
        self.host = [self.dataset.collate([self.dataset[j] for j in range(i * batch, (i + 1) * batch)]).pin()
                     for i in range(n_batches)]
        self.resident = [self.banks.stage(h) for h in self.host]
        torch.cuda.synchronize()
        for pb in self.resident:                   # setup, not warm-up: the workspace covers every staged batch
            self.model.reserve_workspace(pb)
        self.n_cand = float(np.mean([h.n_cand for h in self.host]))
        self.n_ctx = float(np.mean([h.n_ctx_rows for h in self.host]))
        import lirec_b200.mlp.train as TR
        self.TR = TR

    def step(self, pb):
        return self.TR.train_step(self.model, self.loss_fn, self.optimizer, pb, self.world, self.fused)

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        if os.environ.get("LIREC_BENCH_DEBUG"):
            print("[rank %d] leg %.3f ms" % (self.rank, ms), file=sys.stderr, flush=True)
        if self.world == 1:
            return float(ms)
        import torch.distributed as dist
        t = torch.tensor([ms], dtype=torch.float64, device=self.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed_resident(self, steps, warmup, sampler=None, profile=True, ncu_window=False):
        """Device-resident leg.  Returns (ms_total max over ranks, GEMM profile records, launches)."""
        from lirec_b200 import _ext
        for i in range(max(warmup, 3)):
            self.step(self.resident[i % len(self.resident)])
        self.barrier()
        launches0 = _ext.launch_counter
        if profile:
            _ext.profile_begin()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        if ncu_window:
            torch.cuda.cudart().cudaProfilerStart()
        if sampler is not None:
            sampler.region(True, "value")
        e0.record()
        for i in range(steps):
            if profile:                       # per-launch GEMM events on every PROFILE_EVERY-th step only: an event
                _ext.profile_sample(i % PROFILE_EVERY == 0)      # pair per launch breaks the PDL chain of the step
            self.last_loss = self.step(self.resident[i % len(self.resident)])
        e1.record()
        self.barrier()
        if sampler is not None:
            sampler.region(False)
        if ncu_window:
            torch.cuda.cudart().cudaProfilerStop()
        ms = self.max_over_ranks(e0.elapsed_time(e1))
        prof = _ext.profile_end() if profile else []
        self.profiled_steps = len(range(0, steps, PROFILE_EVERY)) if profile else 0
        return ms, prof, _ext.launch_counter - launches0

    def roofline(self, prof, steps, region_ms, clocks, pk):
        steps = max(1, getattr(self, "profiled_steps", steps))      # the steps whose launches carried events
        gemm_ms = sum(p[0] for p in prof)
        exec_flops = sum(p[1] for p in prof)
        alg = algorithmic_flops(self.preset, self.n_cand, self.n_ctx)
        achieved = alg * steps / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
        executed = exec_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
        peak, src = pick_tensor_peak(pk, region_ms, clocks)
        return {"bound": "tensor", "kernel": "lirec_gemm_tcgen05_pair_kernel", "achieved": achieved, "peak": peak,
                "unit": "TFLOP/s", "frac": achieved / peak, "traffic": None, "peak_source": "%s %s" % (pk["source"], src),
                "frac_vs_burst": achieved / pk["bf16_burst"], "frac_vs_sustained": achieved / pk["bf16_sustained"],
                "launches_per_step": len(prof) / float(steps), "gemm_ms_per_step": gemm_ms / steps,
                "algorithmic_tflop_per_step": alg / 1e12, "executed_tflops": executed, "executed_frac": executed / peak}

    def close(self):
        if self.fused is not None:
            self.fused.detach()
        self.model = self.loss_fn = self.optimizer = self.fused = None
        self.dataset = self.banks = self.host = self.resident = None
        torch.cuda.empty_cache()


def measure_traffic(args):
    """DRAM bytes the GEMM launches of ONE step move, measured live: this script re-runs itself for one step
    under `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum` (the timed numbers of the parent are
    already taken; nothing printed by the child is a bench value)."""
    import shutil
    ncu = shutil.which("ncu") or "/usr/local/cuda/bin/ncu"
    if not os.path.exists(ncu):
        return None, "ncu not found"
    cmd = [ncu, "--profile-from-start", "off", "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum",
           "--clock-control", "none", "-k", "regex:lirec_gemm", "--csv", sys.executable, os.path.abspath(__file__),
           "--steps", "1", "--warmup", "3", "--ncu_window", "--only_value", "--preset", args.preset,
           "--batch", str(args.batch), "--n_batches", str(args.n_batches)]
    try:
        env = dict(os.environ)
        for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
            env.pop(k, None)
        res = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=env)
    except Exception as exc:
        return None, "ncu child failed: %r" % (exc,)
    import csv
    import io
    total, launches = 0.0, set()
    rows = [l for l in res.stdout.splitlines() if l.startswith('"')]
    if not rows:
        return None, "ncu produced no CSV (rc %d): %s" % (res.returncode, (res.stderr or res.stdout)[-200:])
    rd = csv.DictReader(io.StringIO("\n".join(rows)))
    for r in rd:
        name, unit, val = r.get("Metric Name", ""), r.get("Metric Unit", ""), r.get("Metric Value", "")
        if not name.startswith("dram__bytes"):
            continue
        v = float(val.replace(",", ""))
        mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(unit, 1.0)
        total += v * mult
        launches.add(r.get("ID"))
    if not launches:
        return None, "no GEMM launch in the ncu capture"
    return int(total), "dram__bytes_read.sum + dram__bytes_write.sum summed over the %d GEMM launches of one step, " \
                       "measured by an `ncu --metrics` child process of this run" % len(launches)


DUMP_MAX_ELEMS = 4 << 20          # per sampled array: 16 MB of float32, so the three files stay under 64 MB


def dump_outputs(model, loss, out_dir):
    """What the last timed step handed its caller, as float32 .npy files in `out_dir`: `loss` (the value
    train_step returned), `params` (every parameter after the step's Adam update) and `grads` (the step's
    gradients), both flattened in named_parameters order.  Above DUMP_MAX_ELEMS elements both keep the same
    sorted sample of positions drawn with a fixed seed, so two builds of the same model compare entry for entry."""
    os.makedirs(out_dir, exist_ok=True)
    params = list(model.parameters())
    p = torch.cat([q.detach().reshape(-1) for q in params])
    g = torch.cat([q.grad.detach().reshape(-1) for q in params])
    if p.numel() > DUMP_MAX_ELEMS:
        pick = np.sort(np.random.default_rng(0).choice(p.numel(), DUMP_MAX_ELEMS, replace=False))
        pick = torch.from_numpy(pick).to(p.device)
        p, g = p[pick], g[pick]
    for name, t in (("loss", loss.detach().reshape(1)), ("params", p), ("grads", g)):
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def dp_parity_check(b):
    """N > 1, before the line is printed: (1) every replica holds bit-identical parameters after the timed
    steps; (2) one in-switch exchange + Adam step equals one ncclAllReduce + Adam step taken from the same
    state on the same gradients."""
    import torch.distributed as dist
    from lirec_b200 import dp
    import lirec_b200.mlp.model as M
    m, o = b.model, b.optimizer
    torch.cuda.synchronize()
    flat = m._flat
    hi, lo = flat.clone(), flat.clone()
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    identical = bool(torch.equal(hi, flat) and torch.equal(lo, flat))
    out = {"replicas_bit_identical": identical}
    if b.fused is not None:
        pb = b.resident[0]
        b.fused.gather_moments()                                 # 'shard' mode: every rank sees all moments
        M.train_step(m, b.loss_fn, pb, seed=123)                 # forward + loss + backward only
        torch.cuda.synchronize()
        g_local = m._flat_grad.clone()
        state = (flat.clone(), o._m.clone(), o._v.clone(), o._t)
        b.fused.step()                                           # the in-switch step (exchange + Adam)
        torch.cuda.synchronize()
        dist.barrier()
        p_switch, g_switch = flat.clone(), m._flat_grad.clone()
        flat.copy_(state[0]), o._m.copy_(state[1]), o._v.copy_(state[2])
        o._t = state[3]
        m._flat_grad.copy_(g_local)
        torch.cuda.synchronize()
        dist.barrier()
        scale = dp.allreduce_flat_grad(m._flat_grad)
        o.step(grad_scale=scale)
        torch.cuda.synchronize()
        gmax = float(m._flat_grad.abs().max())
        out["mode"] = b.fused.mode
        if b.fused.mode != "shard":                              # 'shard' never writes the gradient sum back
            out["grad_sum_max_abs_diff_rel"] = float((g_switch - m._flat_grad).abs().max()) / max(gmax, 1e-30)
        out["param_max_abs_diff"] = float((p_switch - flat).abs().max())
        out["switch_step_equals_nccl_step"] = bool(out.get("grad_sum_max_abs_diff_rel", 0.0) < 1e-5 and
                                                   out["param_max_abs_diff"] < 1e-7)
        m.mark_bf16_fresh()
    ok = identical and out.get("switch_step_equals_nccl_step", True)
    flag = torch.tensor([1 if ok else 0], device=b.dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    out["status"] = "ok" if int(flag.item()) == 1 else "FAILED"
    return out


def run_config(args, preset, batch, steps, warmup, rank, world, dev, pk, with_cpu):
    """One row of `configs`: device-resident train throughput + GEMM roofline (+ cpu_baseline at N = 1)."""
    n_batches = 2
    b = Bench(args, preset, batch, n_batches, rank, world, dev)
    ms, prof, launches = b.timed_resident(steps, warmup)
    roof = b.roofline(prof, steps, ms, None, pk)
    row = {"preset": preset, "clips_per_gpu": batch, "value": batch * world * steps / (ms / 1e3), "unit": "clips/s",
           "ms_per_step": ms / steps, "steps": steps, "candidate_rows_per_step": b.n_cand,
           "context_rows_per_step": b.n_ctx, "gpu_launches_per_step": launches / float(steps),
           "roofline": {k: roof[k] for k in ("bound", "achieved", "peak", "unit", "frac", "frac_vs_burst",
                                             "frac_vs_sustained", "gemm_ms_per_step", "peak_source")}}
    b.close()
    if with_cpu and rank == 0:
        try:
            cb = cpu_baseline_line(preset, 64 if preset != "stress" else 2, steps=2, warmup=1)
            row["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        except Exception as exc:
            row["cpu_baseline"] = {"error": repr(exc)[:200]}
    return row


def run_ours(args):
    from lirec_b200 import dp
    import torch.distributed as dist

    rank, world, local = dp.init_from_env()
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a B200; there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pk = load_peaks()
    if not args.batch:
        args.batch = 256 if args.preset == "stress" else 1024
    if args.preset == "stress":
        args.n_batches = min(args.n_batches, 2)
    steps, warmup = args.steps, max(args.warmup, 3)

    b = Bench(args, args.preset, args.batch, args.n_batches, rank, world, dev)
    sampler = ClockSampler(local)
    if rank == 0 and not os.environ.get("LIREC_BENCH_NO_SAMPLER"):
        sampler.start()

    # ---------------- device-resident timed region ----------------
    ms_total, prof, launches = b.timed_resident(steps, warmup, sampler if rank == 0 else None,
                                                ncu_window=args.ncu_window)
    if args.dump_outputs and rank == 0:
        dump_outputs(b.model, b.last_loss, args.dump_outputs)
    clips_total = args.batch * world * steps
    value = clips_total / (ms_total / 1e3)
    profiled_steps_main = b.profiled_steps
    if args.only_value:
        if rank == 0:
            sampler.stop()
            psteps = max(1, b.profiled_steps)
            per = max(1, int(round(len(prof) / float(psteps))))
            launches_ms = [float(np.mean([r[0] for r in prof[j::per]])) for j in range(per)] if prof else []
            print(json.dumps({"value": value, "ms_per_step": ms_total / steps, "only_value": True,
                              "gemm_ms_per_step": sum(p[0] for p in prof) / psteps,
                              "gemm_launch_ms": [round(x, 4) for x in launches_ms]}))
        return

    copy_stream = torch.cuda.Stream(device=dev)
    main = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    # The end-to-end regions run max(steps, 100) steps: at the driver's --steps 20 a region is 40 ms, and one 10 ms
    # hiccup of a worker process or of the pinning thread is a quarter of it.
    e2e_steps = max(steps, 100)
    e2e_clips = args.batch * world * e2e_steps
    loss_host = torch.empty(e2e_steps, dtype=torch.float32).pin_memory()

    # ---------------- pre-collated legs (batches built before the clock starts) ----------------
    def run_prefetched(stage_fn, n_steps):
        def prefetch(i):
            with torch.cuda.stream(copy_stream):
                pb = stage_fn(i)
                ev = torch.cuda.Event()
                ev.record(copy_stream)
            return pb, ev
        copy_stream.wait_stream(main)
        for i in range(max(2 * args.n_batches, warmup)):          # every distinct batch twice: allocator pools, struct caches
            pb, ev = prefetch(i)
            main.wait_event(ev)
            pb.record_stream(main)
            b.step(pb)
        b.barrier()
        e0.record()
        nxt = prefetch(0)
        dbg = [] if os.environ.get("LIREC_BENCH_DEBUG") else None
        if dbg is not None:
            import lirec_b200.mixed_utils.indexed_dataset as _ids
            _ids.STAGE_TRACE = []
        for i in range(n_steps):
            t0 = time.perf_counter()
            pb, ev = nxt
            main.wait_event(ev)
            pb.record_stream(main)
            if i + 1 < n_steps:
                nxt = prefetch(i + 1)
            t1 = time.perf_counter()
            lv = b.step(pb)
            loss_host[i:i + 1].copy_(lv.detach().reshape(1), non_blocking=True)
            if dbg is not None:
                dbg.append((t1 - t0, time.perf_counter() - t1, i))
        e1.record()
        b.barrier()
        if dbg:
            import lirec_b200.mixed_utils.indexed_dataset as _ids
            if _ids.STAGE_TRACE:
                tr = _ids.STAGE_TRACE
                print("[rank %d] staging phases, longest (ms): table copies %.2f, bank allocations %.2f, gather launches %.2f"
                      % (rank, 1e3 * max(t[0] for t in tr), 1e3 * max(t[1] for t in tr), 1e3 * max(t[2] for t in tr)),
                      file=sys.stderr, flush=True)
                del tr[:]
            print("[rank %d] pre-staged leg: longest host times staging a batch %s, issuing a step %s (ms, step)" % (
                rank, [(round(1e3 * a, 2), i) for a, _, i in sorted(dbg, reverse=True)[:3]],
                [(round(1e3 * c, 2), i) for _, c, i in sorted(dbg, key=lambda r: -r[1])[:3]]), file=sys.stderr, flush=True)
        assert bool(torch.isfinite(loss_host[:n_steps]).all()), "pre-collated leg: non-finite loss read back"
        return args.batch * world * n_steps / (b.max_over_ranks(e0.elapsed_time(e1)) / 1e3)

    from lirec_b200.mixed_utils.indexed_dataset import ResidentBanks
    res_bytes = int(np.mean([ResidentBanks.h2d_bytes(h) for h in b.host]))
    e2e_pre = run_prefetched(lambda i: b.banks.stage(b.host[i % len(b.host)]), e2e_steps)
    # streamed: every feature row of every batch crosses PCIe every step (no resident banks)
    b.opt.resident_banks = 0
    full_host = [b.dataset.collate([b.dataset[j] for j in range(i * args.batch, (i + 1) * args.batch)]).pin()
                 for i in range(min(2, args.n_batches))]
    b.opt.resident_banks = 1
    full_bytes = int(np.mean([h.h2d_bytes() for h in full_host]))
    e2e_streamed = run_prefetched(lambda i: full_host[i % len(full_host)].to_device(dev, non_blocking=True),
                                  min(e2e_steps, 40))
    del full_host

    # ---------------- end to end through the loader (the headline e2e) ----------------
    # `packed_loader` over the cached dataset: index-only items, collate -> lirec_collate_tables in worker
    # processes, shared-memory hand-over, pinning on the DataLoader's pin thread, async H2D of the int tables on
    # a copy stream one batch ahead, device gather of the batch banks from the resident dataset banks, train step,
    # loss read-back.  The iterator is warmed (workers forked, queues primed) by `warmup` untimed steps; the
    # timed region is the next e2e_steps batches of the same iterator.
    from lirec_b200.mixed_utils.classification_dataloader import packed_loader
    cores = usable_cores()
    workers = args.workers if args.workers >= 0 else max(1, min(6, (cores - world) // max(world, 1)))
    b.opt.prefetch_factor = 2

    def loader(n_steps):
        # one DataLoader (one set of worker processes) for the whole leg: enough epochs of the rank's dataset,
        # each its own permutation, chained behind it
        rep = (n_steps + 2 * workers + 4 + args.n_batches - 1) // args.n_batches + 1
        return iter(packed_loader(b.dataset, args.batch, shuffle=True, num_workers=workers, device=dev,
                                  drop_last=True, seed=rank, repeat=rep))

    e2e_err = None
    e2e_value = e2e_host_rate = None
    e2e_legs, e2e_max_wait = [], []
    h2d_loader = 0
    import gc
    gc.collect()
    if os.environ.get("LIREC_BENCH_NO_FREEZE") != "1":
        gc.freeze()         # as lirec_b200/mlp/train.py does: the cached records never reach a full collection again
    try:
        # FIVE consecutive legs of e2e_steps batches each over the same iterator, each bracketed like the main timed
        # region (barrier + events, max over ranks); the reported e2e is their MEDIAN and all five are listed.  One
        # 100-step leg lasts 0.2 s, and during the first minutes on a freshly started box the host side shows
        # sporadic 20-120 ms stalls (any thread, any leg — the pre-staged leg too; they fade as the process's pages
        # get touched) that hit one or two legs of a run and leave the others within 3 % of each other.
        n_legs = 5
        e2e_warm = max(warmup, 30)          # loader threads up, slot ring cycled, allocator pools at their high-water marks
        it = loader(e2e_warm + n_legs * e2e_steps)
        for _ in range(e2e_warm):
            b.step(next(it))
        e2e_legs, e2e_max_wait = [], []
        for leg in range(n_legs):
            b.barrier()
            if rank == 0:
                sampler.region(True, "e2e")
            e0.record()
            t_wait = t_step = w_max = 0.0
            for i in range(e2e_steps):
                t0 = time.perf_counter()
                pb = next(it)
                t1 = time.perf_counter()
                lv = b.step(pb)
                loss_host[i:i + 1].copy_(lv.detach().reshape(1), non_blocking=True)
                t_wait, t_step, w_max = t_wait + (t1 - t0), t_step + (time.perf_counter() - t1), max(w_max, t1 - t0)
                if i == 0:
                    h2d_loader = ResidentBanks.h2d_bytes(pb.host)
            e1.record()
            b.barrier()
            if rank == 0:
                sampler.region(False)
            assert bool(torch.isfinite(loss_host[:e2e_steps]).all()), "e2e: non-finite loss read back"
            if os.environ.get("LIREC_BENCH_DEBUG"):
                print("[rank %d] e2e loader leg %d: host waited %.2f ms for batches (longest single wait %.2f ms), spent "
                      "%.2f ms issuing steps (%d steps)" % (rank, leg, 1e3 * t_wait, 1e3 * w_max, 1e3 * t_step, e2e_steps),
                      file=sys.stderr, flush=True)
            e2e_legs.append(e2e_clips / (b.max_over_ranks(e0.elapsed_time(e1)) / 1e3))
            e2e_max_wait.append(1e3 * w_max)
        e2e_value = float(np.median(e2e_legs))
        it.close()
        # the loader alone (items, collate, pin, H2D, device gather — no train step): what the host side sustains
        b.dataset.epoch = 1000
        it = loader(44)
        for _ in range(4):
            next(it)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        n_host = 0
        for _ in range(40):
            n_host += next(it).B
        torch.cuda.synchronize()
        e2e_host_rate = n_host / (time.perf_counter() - t0)
        it.close()
        del it
    except Exception as exc:                                     # never lose the headline line over this leg
        e2e_err = repr(exc)[:300]
        b.barrier()
    import gc
    gc.collect()
    b.barrier()

    # ---------------- inference: forward + device-side prediction arg-maxes (no_grad) ----------------
    from lirec_b200 import ops
    model = b.model
    model.eval()
    track_model = PRESETS[args.preset]["model"] in ("int_ch", "int_rel_ch")
    n_rels = 15 if PRESETS[args.preset]["model"] == "int_rel_ch" else 0
    with torch.no_grad():
        def infer(pb):
            out = model(pb)
            if track_model:
                return ops.predict_tracks(out.ragged_inters, out.ragged_rels, pb["cand_off"], pb["labels"],
                                          pb["rels_label"] if n_rels else None, pb["gt_tracks"], n_rels)
            return out.ragged_inters
        for i in range(3):
            infer(b.resident[i % len(b.resident)])
        b.barrier()
        e0.record()
        for i in range(steps):
            infer(b.resident[i % len(b.resident)])
        e1.record()
        b.barrier()
    infer_value = clips_total / (b.max_over_ranks(e0.elapsed_time(e1)) / 1e3)
    model.train()

    # ---------------- an HBM-bound kernel against the measured copy bandwidth: the fused Adam ----------------
    hbm_roof = None
    if world == 1:
        try:
            n_par = model._flat.numel()
            for _ in range(3):
                b.optimizer.step()
            b.barrier()
            e0.record()
            for _ in range(20):
                b.optimizer.step()
            e1.record()
            b.barrier()
            adam_ms = e0.elapsed_time(e1) / 20.0
            adam_bytes = n_par * (4 * 4 + 3 * 4 + 2)          # read p, g, m, v; write p, m, v + the bf16 shadow
            hbm_roof = {"bound": "hbm", "kernel": "adam_kernel", "achieved": adam_bytes / adam_ms / 1e6,
                        "unit": "GB/s", "bytes_per_launch": int(adam_bytes), "us_per_launch": 1e3 * adam_ms,
                        "peak": pk["hbm"], "frac": adam_bytes / adam_ms / 1e6 / pk["hbm"],
                        "peak_source": pk["source"] + " hbm_gbs"}
        except Exception as exc:                               # never lose the headline line over the extra one
            hbm_roof = {"error": repr(exc)[:200]}

    dp_parity = dp_parity_check(b) if world > 1 else None
    clocks = sampler.stop() if rank == 0 else None
    roofline = b.roofline(prof, steps, ms_total, clocks, pk) if rank == 0 else None
    exchange = "none (1 GPU)"
    if world > 1:
        exchange = ("in-switch gradient sum + sharded Adam + multicast of the new parameters in one pass "
                    "(lirec_dp_reduce_adam_bcast)" if (b.fused is not None and b.fused.mode == "shard") else
                    "in-switch multimem reduce + Adam per bucket, first bucket overlapped with backward "
                    "(lirec_dp_exchange)" if (b.fused is not None and getattr(b.fused, "overlap", False)) else
                    "in-switch multimem reduce + Adam after backward (lirec_dp_exchange)" if b.fused is not None
                    else "ncclAllReduce fp32 + Adam")
    n_cand, n_ctx, in_bytes = b.n_cand, b.n_ctx, res_bytes
    b.close()

    # ---------------- every BASELINE configuration ----------------
    configs = None
    if not args.no_configs and args.preset == "int_rel_ch":
        configs = []
        c_steps = max(5, min(steps, 20))
        plan = [("modalities", 64), ("modalities", 1024), ("int_rels", 64), ("int_rels", 1024), ("int_ch", 64),
                ("int_ch", 1024), ("int_rel_ch", 64), ("stress", 64), ("stress", 256)]
        for preset, bsz in plan:
            try:
                configs.append(run_config(args, preset, bsz, c_steps, 3, rank, world, dev, pk,
                                          with_cpu=(world == 1 and not args.no_cpu_baseline and bsz == 64)))
            except Exception as exc:
                configs.append({"preset": preset, "clips_per_gpu": bsz, "error": repr(exc)[:300]})
                if world > 1:
                    raise

    if rank != 0:
        return
    if args.dump_profile:
        psteps = max(1, profiled_steps_main)
        per = int(round(len(prof) / float(psteps)))
        with open(args.dump_profile, "w") as f:
            f.write("# GEMM launches of one step (mean over %d profiled steps of %d): idx ms executed_GFLOP TFLOP/s tiles problems\n" % (psteps, steps))
            for j in range(per):
                rows = prof[j::per]
                ms = float(np.mean([r[0] for r in rows]))
                fl = float(np.mean([r[1] for r in rows]))
                f.write("%d %.4f %.2f %.1f %d %d\n" % (j, ms, fl / 1e9, fl / ms / 1e9 if ms > 0 else 0, rows[0][2], rows[0][3]))
    if world == 1 and not args.no_traffic:
        roofline["traffic"], roofline["traffic_note"] = measure_traffic(args)
    roofline["profiled_steps"] = profiled_steps_main
    roofline["note"] = ("achieved = algorithmic fwd+bwd FLOPs of the step (SURVEY.md §8d, valid rows, no credit for "
                        "dedup) / summed CUDA-event duration of the GEMM launches, events recorded live on every "
                        "8th step of the timed region (an event pair per launch on every step breaks the "
                        "programmatic-dependent-launch chain and slows the region it measures); executed = MMA FLOPs actually "
                        "issued (layer 1 runs once per unique bank row; hi/lo split passes count 2-3x)")
    cpu = None if (args.no_cpu_baseline or world > 1) else cpu_baseline_line(args.preset, args.cpu_clips, steps=3, warmup=1)
    e2e_headline = e2e_value if e2e_value is not None else e2e_pre
    line = {"metric": "train clips/sec (%s fwd+bwd)" % args.preset, "value": value, "unit": "clips/s",
            "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms_total / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": WORKLOAD_TEXT[args.preset] + ", synthetic MovieGraphs-shaped clips cached in "
                                                               "dataset-level feature banks, packed ragged batches",
                       "preset": args.preset, "clips_per_gpu": args.batch, "global_batch": args.batch * world,
                       "candidate_rows_per_step": n_cand, "context_rows_per_step": n_ctx,
                       "parallelism": "dp%d" % world,
                       "optimizer": "fused flat Adam",
                       "step_api": ("model()/loss()/backward()/optimizer.step() (autograd)" if args.autograd_step
                                    else "lirec_b200.mlp.train.train_step (native forward+loss+backward, no autograd)"),
                       "gradient_exchange": exchange,
                       "precision": "bf16 operands, hi/lo split activations, fp32 accumulate",
                       "l2": "%d distinct batches rotate; per step the kernels stream the batch banks, the workspace and "
                             "553 MB of optimizer state (4x the 126 MB L2)" % args.n_batches},
            "clocks": clocks,
            "e2e": {"value": e2e_headline, "unit": "clips/s",
                    "h2d_bytes_per_step": int(h2d_loader or in_bytes), "d2h_bytes_per_step": 4,
                    "what": ("packed_loader(CachedClipsDataset, num_workers=%d): batch assembly from the dataset's index-only "
                             "records (native gather + lirec_collate_tables in worker threads, straight into pinned "
                             "slots), async H2D of the index tables, device gather from the HBM-resident dataset "
                             "banks, train step and loss read-back inside the timed region" % workers)
                    if e2e_value is not None else "loader leg failed (%s); pre-collated index-only batches" % e2e_err,
                    "loader_workers": workers, "host_cores": cores, "host_cores_reported": os.cpu_count(),
                    "steps": e2e_steps,
                    "legs_clips_per_s": [round(v, 1) for v in e2e_legs] if e2e_value is not None else None,
                    "legs_longest_batch_wait_ms": [round(v, 2) for v in e2e_max_wait] if e2e_value is not None else None,
                    "value_is": "median of the legs (each `steps` batches, barrier + CUDA events, max over ranks)",
                    "loader_only_clips_per_s": e2e_host_rate},
            "e2e_precollated": {"value": e2e_pre, "unit": "clips/s", "h2d_bytes_per_step": int(in_bytes),
                                "d2h_bytes_per_step": 4,
                                "note": "index-only batches collated before the clock starts; per step the pinned "
                                        "tables cross PCIe and the batch banks are gathered on the device"},
            "e2e_streamed": {"value": e2e_streamed, "unit": "clips/s", "h2d_bytes_per_step": int(full_bytes),
                             "d2h_bytes_per_step": 4,
                             "note": "no resident banks: every feature row of every batch crosses PCIe every step"},
            "inference": {"value": infer_value, "unit": "clips/s",
                          "what": "forward (eval, no_grad) + device-side track/class/relationship arg-maxes, inputs "
                                  "resident in HBM"},
            "gpu_launches": int(launches),
            "roofline": roofline}
    if hbm_roof is not None:
        line["roofline_hbm"] = hbm_roof
    if dp_parity is not None:
        line["dp_parity"] = dp_parity["status"]
        line["dp_parity_detail"] = dp_parity
    if cpu is not None:
        line["cpu_baseline"] = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
    if configs is not None:
        line["configs"] = configs
    print(json.dumps(line))
    if dp_parity is not None and dp_parity["status"] != "ok":
        raise SystemExit("dp_parity failed: %r" % (dp_parity,))


def main():
    args = parse_args()
    # stdout carries exactly ONE JSON line: library chatter written to fd 1 while the job runs (NCCL prints
    # its version banner there) is routed to stderr, and the line is written to the real stdout at the end
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
    sys.stdout.flush()
    try:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass


if __name__ == "__main__":
    main()
