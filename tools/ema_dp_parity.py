"""Two-rank check of data-parallel training with --ema_decay (run under torchrun on >= 2 B200s):
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/ema_dp_parity.py
Every rank keeps its own FlatEMA and adds no collective: the replicas' parameters are bitwise identical after every
step, so their averages must be too.  Both ranks start from the same weights and take three steps on their shards of
a global batch (the last one split unequally), once with the in-switch exchange + Adam (the model's flat buffers then
live in symmetric memory; skipped where the GPUs have no multicast) and once with NCCL all_reduce + FlatAdam
(--dp_switch_reduce 0).  Afterwards the averages, the replicas and one swap in and out of the average must agree
bitwise across ranks."""
import contextlib
import io
import os
import sys

sys.argv = sys.argv[:1]
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from lirec_b200 import dp  # noqa: E402
from lirec_b200.mixed_utils import synthetic  # noqa: E402
from lirec_b200.utils.arg_pars import opt  # noqa: E402

GLOBAL_BATCHES = (16, 16, 15)
DECAY = 0.9


def same_on_every_rank(t):
    ref = t.clone()
    dist.broadcast(ref, src=0)
    return bool(torch.equal(ref, t))


def run(rank, world, batches, switch):
    import lirec_b200.mlp.model as M
    import lirec_b200.mlp.train as TR
    torch.manual_seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        model, loss_fn, optimizer = M.create_model(101, n_rels=15)
    assert isinstance(optimizer, M.FlatAdam)
    model.eval()                                   # dropout masks are keyed by local row position
    dp.broadcast_params(model._flat)
    fused = dp.SwitchReduceAdam.attach(model, optimizer) if switch else None
    if switch and fused is None:
        return None
    ema = M.FlatEMA(model, DECAY)
    for pb in batches:
        TR.train_step(model, loss_fn, optimizer, pb, world, fused, 0.0, ema)
    torch.cuda.synchronize()
    ok = {"average": same_on_every_rank(ema._ema), "replica": same_on_every_rank(model._flat),
          "n_averaged": ema.n_averaged == len(batches)}
    w, avg = model._flat.clone(), ema._ema.clone()
    with ema.applied():
        torch.cuda.synchronize()
        ok["swapped_in"] = bool(torch.equal(model._flat, avg))
    torch.cuda.synchronize()
    ok["swapped_back"] = bool(torch.equal(model._flat, w))
    if fused is not None:
        fused.detach()
    return ok


def main():
    rank, world, local = dp.init_from_env()
    torch.cuda.set_device(local)
    for k, v in dict(tr_maximize=True, tracks=True, ints=1, ctx=1, gates=1, rels_multitask=True, rels_multi_clip=True,
                     rels_n_clips=18, mod_check=False, device="cuda", fused_adam=1, optimizer="adam", lr=1e-3,
                     weight_decay=0.0, dp=1, ema_decay=DECAY, clip_grad_norm=0.0, tr_correct=False, tr_max_neg=False,
                     tr_cat_distr=False).items():
        setattr(opt, k, v)
    batches = []
    for j, B in enumerate(GLOBAL_BATCHES):
        cl = [synthetic.make_clip(11000 * (j + 1) + i, preset="int_rel_ch") for i in range(B)]
        a, b = dp.shard_range(B, rank, world)
        mine = synthetic.pack_clips(cl[a:b])
        mine.global_clips = B
        batches.append(mine.to_device("cuda"))
    results = {"in-switch": run(rank, world, batches, True), "nccl": run(rank, world, batches, False)}
    ok = results["nccl"] is not None and all(all(r.values()) for r in results.values() if r is not None)
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        for k, r in results.items():
            print(k, "(no multicast: not run)" if r is None else r)
        print("EMA DP PARITY", "OK" if int(flag.item()) else "FAILED")
    dist.destroy_process_group()
    return 0 if int(flag.item()) else 1


if __name__ == "__main__":
    sys.exit(main())
