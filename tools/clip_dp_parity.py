"""Two-rank check of data-parallel training with --clip_grad_norm (run under torchrun on >= 2 B200s):
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/clip_dp_parity.py
Clipping takes NCCL all_reduce of the flat gradients, then clip_grad_norm_flat_ with the 1/world average as its
grad_scale, then FlatAdam.  Both ranks start from the same weights and take three clipped steps on their shards of a
global batch (the last one split unequally).  The pre-clip norms and the replicas must be bitwise identical across
ranks afterwards, and match a single-process run on the global batches within 1e-3 max-norm relative per tensor (the
exchange reorders the gradient sums)."""
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
MAX_NORM = 1e-3                 # below the synthetic gradients' norm: every step clips


def main():
    rank, world, local = dp.init_from_env()
    torch.cuda.set_device(local)
    for k, v in dict(tr_maximize=True, tracks=True, ints=1, ctx=1, gates=1, rels_multitask=True, rels_multi_clip=True,
                     rels_n_clips=18, mod_check=False, device="cuda", fused_adam=1, optimizer="adam", lr=1e-3,
                     weight_decay=0.0, dp=1, clip_grad_norm=MAX_NORM, tr_correct=False, tr_max_neg=False,
                     tr_cat_distr=False).items():
        setattr(opt, k, v)
    import lirec_b200.mlp.model as M
    import lirec_b200.mlp.train as TR
    clips, batches = [], []
    for j, B in enumerate(GLOBAL_BATCHES):
        cl = [synthetic.make_clip(9000 * (j + 1) + i, preset="int_rel_ch") for i in range(B)]
        clips.append(cl)
        a, b = dp.shard_range(B, rank, world)
        mine = synthetic.pack_clips(cl[a:b])
        mine.global_clips = B
        batches.append(mine.to_device("cuda"))

    def fresh():
        torch.manual_seed(0)
        with contextlib.redirect_stdout(io.StringIO()):
            model, loss_fn, optimizer = M.create_model(101, n_rels=15)
        assert isinstance(optimizer, M.FlatAdam)
        model.eval()                               # dropout masks are keyed by local row position
        return model, loss_fn, optimizer

    model, loss_fn, optimizer = fresh()
    dp.broadcast_params(model._flat)
    norms = []
    for pb in batches:
        TR.train_step(model, loss_fn, optimizer, pb, world, None, MAX_NORM)
        norms.append(model._last_grad_norm.clone())
    torch.cuda.synchronize()
    norms = torch.stack(norms)
    ref_norms, ref0 = norms.clone(), model._flat.clone()
    dist.broadcast(ref_norms, src=0)
    dist.broadcast(ref0, src=0)
    same = bool(torch.equal(ref0, model._flat)) and bool(torch.equal(ref_norms, norms))
    clipped = bool((norms > MAX_NORM).all())

    single, loss1, opt1 = fresh()
    for cl in clips:
        TR.train_step(single, loss1, opt1, synthetic.pack_clips(cl).to_device("cuda"), 1, None, MAX_NORM)
    torch.cuda.synchronize()
    worst = 0.0
    for off, p in zip(model._offsets, model._param_list):
        a, b = model._flat[off:off + p.numel()].double(), single._flat[off:off + p.numel()].double()
        worst = max(worst, float((a - b).abs().max() / (b.abs().max() + 1e-30)))
    ok = same and clipped and worst < 1e-3
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("pre-clip norms:", [float(x) for x in norms])
        print("norms and replicas identical across ranks:", same, "; every step clipped:", clipped)
        print("parameters vs single process on the global batch, worst max-norm relative per tensor: %.2e" % worst)
        print("CLIP DP PARITY", "OK" if int(flag.item()) else "FAILED")
    dist.destroy_process_group()
    return 0 if int(flag.item()) else 1


if __name__ == "__main__":
    sys.exit(main())
