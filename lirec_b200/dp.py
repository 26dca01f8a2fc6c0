"""Data parallelism over clips: one process per GPU, NCCL allreduce of the flat gradient buffer.

The reference is single-process (SURVEY.md §2.3); clips are independent and every loss is a
per-clip term averaged over the batch (mlp/model.py:402, 418, 439, 493, 561-573), so the only
exchange step of the hot path is the gradient sum.  Because all parameters live in ONE flat
fp32 gradient buffer (lirec_b200/mlp/model.py), that is a single `all_reduce` over NVLink /
NVSwitch per step; the 1/world_size average is folded into the fused Adam kernel's grad_scale
(or applied in place for torch.optim.Adam).

`SwitchReduceAdam` goes one step further on NVSwitch boxes: the gradient buffer lives in symmetric
memory mapped into a multicast object and is reduced inside the switch (csrc/dp.cu:lirec_dp_exchange,
multimem.ld_reduce / multimem.st) bucket by bucket, the gate + head bucket while backward is still
running — no NCCL call on the step's critical path.  torch.distributed._symmetric_memory only allocates
and rendezvous-es the buffers.
"""
import os

import torch
import torch.distributed as dist


def init_from_env(backend=None):
    """Initialise torch.distributed from torchrun's environment. Returns (rank, world, local_rank)."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        kw = {}
        if backend == "nccl":
            torch.cuda.set_device(local)
            kw["device_id"] = torch.device("cuda", local)
        dist.init_process_group(backend=backend, rank=rank, world_size=world, **kw)
    return rank, world, local


def world_size():
    return dist.get_world_size() if dist.is_initialized() else 1


def shard_range(n_items, rank, world):
    """Contiguous, near-even split of n_items over ranks: [begin, end)."""
    base, rem = divmod(n_items, world)
    begin = rank * base + min(rank, rem)
    return begin, begin + base + (1 if rank < rem else 0)


def allreduce_flat_grad(flat_grad, local_clips=None, global_clips=None, average_in_place=False):
    """Sum the flat gradient over ranks.  Per-rank losses are means over LOCAL clips; with equal
    shards the global-batch gradient is the plain average (returned scale = 1/world).  For unequal
    shards (last short batch) gradients are pre-scaled by local/global clip counts and summed
    (returned scale = 1)."""
    world = world_size()
    if world == 1:
        return 1.0
    scale = 1.0 / world
    if local_clips is not None and global_clips is not None and local_clips * world != global_clips:
        flat_grad.mul_(float(local_clips) / float(global_clips))
        scale = 1.0
    dist.all_reduce(flat_grad, op=dist.ReduceOp.SUM)
    if average_in_place and scale != 1.0:
        flat_grad.mul_(scale)
        return 1.0
    return scale


def broadcast_params(flat_param, src=0):
    if world_size() > 1:
        dist.broadcast(flat_param, src=src)


class SwitchReduceAdam:
    """Gradient exchange + Adam of one data-parallel step on NVSwitch multicast (no NCCL call on the step).

        fused = SwitchReduceAdam.attach(model, optimizer)      # collective; None if unsupported
        ...
        train_step(model, loss, optimizer, pb, world, fused)   # lirec_b200/mlp/train.py drives it

    mode 'shard' (default): lirec_dp_reduce_adam_bcast — every rank sums its 1/world shard of the gradients inside
    the switch, applies Adam to that shard (it owns the shard's moments) and multicast-stores the new fp32
    parameters and their bf16 shadow into every replica.  With `overlap` the pass is split in two: the gate +
    head parameters (53 %) run on a side stream behind the event lirec_model_backward records when their
    gradients are final, while the encoder stages of backward still go; the encoders follow after backward.  Parameters, bf16 shadow
    and gradients therefore live in ONE symmetric allocation; `optimizer.state_dict()` gathers the moments.
    Against exchange-then-Adam this removes the 553 MB full-replica optimizer pass from every rank's critical
    path and sends 6 bytes per parameter back instead of 4.

    mode 'bucket': the gradient sum (lirec_dp_exchange) and a full-replica lirec_adam_flat per bucket, the
    gate + head bucket on a side stream behind the event lirec_model_backward records when those gradients
    are final (measured: the overlap buys < 1 % — the overlapped Adam pass competes with the L2-bound encoder
    stages for the same memory system — and the exchange alone is slower than NCCL's at 2 ranks).

    world == 1 (`attach(..., single_gpu=True)`): no exchange; only 'bucket' mode's overlapped Adam (off by
    default: it measured 0.8 % slower than the plain Adam launch).
    torch.distributed._symmetric_memory only allocates and rendezvous-es the buffers."""

    overlap = True
    coresident = True        # overlapped passes in CTAs that fit beside a resident GEMM CTA (LIREC_DP_CORESIDENT=0: A/B)

    def __init__(self, model, optimizer, hdl=None, flags=None, flag_hdl=None, mode="bucket", offsets=None):
        self.model, self.optimizer = model, optimizer
        self.hdl, self.flags, self.flag_hdl, self.mode = hdl, flags, flag_hdl, mode
        self.offsets = offsets or {}
        self.rank, self.world = (hdl.rank, hdl.world_size) if hdl is not None else (0, 1)
        dev = model._flat.device
        self.side = torch.cuda.Stream(device=dev)
        self.ev_heads = torch.cuda.Event()
        self.ev_done = torch.cuda.Event()
        self.ev_heads.record()                       # creates the cudaEvent_t the library re-records
        # bucket boundary: the first parameter of the gate (models with a gate) or of the first head
        names = [n for n, _ in model.named_parameters()]
        first = next(n for n in ("gates_ints.fc_out.weight", "out_ints.weight", "out_ctx.weight") if n in names)
        self.split = int(model._offsets[names.index(first)])
        self.n = int(model._flat.numel())
        import os
        self.coresident = os.environ.get("LIREC_DP_CORESIDENT", "1") != "0"
        assert self.split % 64 == 0 and self.n % 64 == 0
        if self.world > 1 and mode == "shard":
            optimizer._shard_sync = self.gather_moments

    @staticmethod
    def supported(device):
        try:
            from torch._C._autograd import DeviceType
            from torch._C._distributed_c10d import _SymmetricMemory
            return bool(_SymmetricMemory.has_multicast_support(DeviceType.CUDA, torch.device(device).index or 0))
        except Exception:
            return False

    @classmethod
    def attach(cls, model, optimizer, single_gpu=False, mode=None):
        """Move the model's flat buffers into symmetric memory (collective over the world group).
        Returns None — and leaves everything as it was — without FlatAdam, without multicast, or on a single
        rank (unless single_gpu=True: then only the overlapped bucket-0 Adam is set up)."""
        import os
        from lirec_b200 import _ext
        from lirec_b200.mlp.model import FlatAdam
        if not isinstance(optimizer, FlatAdam):
            return None
        model._sync_flat()
        if world_size() < 2:
            return cls(model, optimizer) if single_gpu else None
        mode = mode or os.environ.get("LIREC_DP_MODE", "shard")
        dev = model._flat.device
        ok = torch.tensor([1 if cls.supported(dev) else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            return None
        import torch.distributed._symmetric_memory as symm_mem
        group = dist.group.WORLD
        n = model._flat.numel()
        words = max(64, int(_ext.lib().lirec_dp_flag_words(dist.get_world_size())))
        # one symmetric allocation: [gradients fp32 | parameters fp32 | bf16 shadow | flags], 256-byte aligned parts
        sizes = [4 * n, 4 * n if mode == "shard" else 0, 2 * n if mode == "shard" else 0, 4 * words]
        offs, total = [], 0
        for sz in sizes:
            offs.append(total)
            total += (sz + 255) // 256 * 256
        buf = symm_mem.empty(total, dtype=torch.uint8, device=dev)
        hdl = symm_mem.rendezvous(buf, group)
        if not hdl.multicast_ptr:
            return None
        buf.zero_()
        grad = buf[offs[0]:offs[0] + 4 * n].view(torch.float32)
        flags = buf[offs[3]:offs[3] + 4 * words].view(torch.int32)
        flat = bf16 = None
        if mode == "shard":
            flat = buf[offs[1]:offs[1] + 4 * n].view(torch.float32)
            bf16 = buf[offs[2]:offs[2] + 2 * n].view(torch.bfloat16)
        model.use_buffers(flat=flat, grad=grad, bf16=bf16)
        # device array of every rank's flag buffer (peer pointers of the one allocation + the flags' offset)
        ptrs = torch.tensor([int(hdl.buffer_ptrs[r]) + offs[3] for r in range(hdl.world_size)], dtype=torch.int64,
                            device=dev)
        bases = torch.tensor([int(hdl.buffer_ptrs[r]) for r in range(hdl.world_size)], dtype=torch.int64, device=dev)
        torch.cuda.synchronize(dev)
        dist.barrier()
        self = cls(model, optimizer, hdl, flags, None, mode, dict(grad=offs[0], flat=offs[1], bf16=offs[2]))
        self._buf, self._flag_ptrs, self._bases = buf, ptrs, bases
        # transport of the 'shard' pass: plain peer loads / stores at 2 ranks, the switch (multimem) from 4 on
        self.transport = os.environ.get("LIREC_DP_TRANSPORT") or ("peer" if hdl.world_size == 2 else "multimem")
        return self

    def detach(self):
        """Give the model ordinary buffers again (the symmetric allocation is released with this object)."""
        torch.cuda.synchronize()
        m = self.model
        if m is not None and self.hdl is not None:
            if self.mode == "shard":
                self.gather_moments()
            m.use_buffers(flat=torch.empty_like(m._flat) if self.mode == "shard" else None,
                          grad=torch.empty_like(m._flat_grad),
                          bf16=torch.empty_like(m._flat_bf16) if self.mode == "shard" else None)
        if m is not None:
            m._heads_event = None
        if self.optimizer is not None and getattr(self.optimizer, "_shard_sync", None) is not None:
            self.optimizer._shard_sync = None
        self.model = self.optimizer = None

    def buckets(self):
        """(offset, length) in floats of the pieces one step exchanges: with `overlap`, the gate + head parameters
        first (their pass runs on the side stream behind backward's heads-final event), then the encoders."""
        if self.overlap and 0 < self.split < self.n:
            return [(self.split, self.n - self.split), (0, self.split)]
        return [(0, self.n)]

    def shard_ranges(self, rank=None):
        """[begin, end) in floats of the shards a rank owns in 'shard' mode: 1/world of every bucket."""
        r = self.rank if rank is None else rank
        out = []
        for off, n in self.buckets():
            n4 = n // 4
            out.append((off + 4 * (n4 * r // self.world), off + 4 * (n4 * (r + 1) // self.world)))
        return out

    @torch.no_grad()
    def gather_moments(self):
        """'shard' mode: every rank receives the Adam moments of all shards (checkpoints, mode switches)."""
        if self.world < 2 or self.mode != "shard":
            return
        o = self.optimizer
        for r in range(self.world):
            for a, b in self.shard_ranges(r):
                dist.broadcast(o._m[a:b], src=r)
                dist.broadcast(o._v[a:b], src=r)

    # ---- per-step protocol --------------------------------------------------------------------------
    def arm(self, equal_shards=True):
        """Before backward: ask lirec_model_backward for the heads-final event (only when this step's exchange
        needs no host-side re-weighting)."""
        self._armed = bool(self.overlap and equal_shards and 0 < self.split < self.n)
        self.model._heads_event = self.ev_heads if self._armed else None
        return self._armed

    def _mc(self, what):
        return int(self.hdl.multicast_ptr) + self.offsets[what]

    def _bucket(self, off, n, channel, stream, scale, co=False):
        from lirec_b200 import ops
        m, o = self.model, self.optimizer
        g = o.param_groups[0]
        if self.world > 1:
            ops.dp_exchange(self._mc("grad"), off, n, self.rank, self.world, self._flag_ptrs.data_ptr(), channel, stream,
                            coresident=co)
        ops.adam_flat(m._flat, m._flat_grad, o._m, o._v, m._flat_bf16, g["lr"], g["betas"][0], g["betas"][1],
                      g["eps"], g["weight_decay"], o._t, scale, offset=off, n=n, stream=stream, coresident=co)

    def _shard_pass(self, bucket, channel, stream, scale, co=False):
        """lirec_dp_reduce_adam_bcast over floats [off, off + n) on `stream`; co: the pass runs beside backward's
        GEMMs (CTAs sized to share their SMs)."""
        from lirec_b200 import ops
        m, o = self.model, self.optimizer
        g = o.param_groups[0]
        off, n = bucket
        if self.transport == "peer" and self.world in (2, 4, 8):
            ops.dp_reduce_adam_bcast_peer(self._bases.data_ptr(), self.offsets["grad"] + 4 * off,
                                          self.offsets["flat"] + 4 * off, self.offsets["bf16"] + 2 * off, o._m[off:],
                                          o._v[off:], n, g["lr"], g["betas"][0], g["betas"][1], g["eps"],
                                          g["weight_decay"], o._t, scale, self.rank, self.world,
                                          self._flag_ptrs.data_ptr(), channel, stream, coresident=co)
        else:
            ops.dp_reduce_adam_bcast(self._mc("grad") + 4 * off, m._flat[off:], self._mc("flat") + 4 * off,
                                     self._mc("bf16") + 2 * off, o._m[off:], o._v[off:], n, g["lr"], g["betas"][0],
                                     g["betas"][1], g["eps"], g["weight_decay"], o._t, scale, self.rank, self.world,
                                     self._flag_ptrs.data_ptr(), channel, stream, coresident=co)

    @torch.no_grad()
    def step(self, local_clips=None, global_clips=None):
        """After backward: the exchange + Adam of the step."""
        from lirec_b200 import ops
        m, o = self.model, self.optimizer
        scale = 1.0 / self.world
        armed = bool(getattr(self, "_armed", False))
        self._armed = False
        m._heads_event = None
        if local_clips is not None and global_clips is not None and local_clips * self.world != global_clips:
            assert not armed, "unequal shards are re-weighted on the host: arm(equal_shards=False)"
            m._flat_grad.mul_(float(local_clips) / float(global_clips))      # unequal last shards: weighted sum
            scale = 1.0
        o._t += 1
        main = torch.cuda.current_stream()
        if self.world > 1 and self.mode == "shard":
            # one fused pass per bucket; the ownership of the moments follows buckets(), armed or not
            bk = self.buckets()
            if armed and len(bk) == 2:
                self.side.wait_event(self.ev_heads)          # recorded mid-backward on the main stream
                self._shard_pass(bk[0], 0, self.side, scale, co=self.coresident)
                self.ev_done.record(self.side)
                self._shard_pass(bk[1], 1, main, scale)
                main.wait_event(self.ev_done)
            else:
                for ch, b in enumerate(bk):
                    self._shard_pass(b, ch, main, scale)
        elif armed:
            self.side.wait_event(self.ev_heads)              # recorded mid-backward on the main stream
            self._bucket(self.split, self.n - self.split, 0, self.side, scale, co=self.coresident)
            self.ev_done.record(self.side)
            if self.split:
                self._bucket(0, self.split, 1, main, scale)
            main.wait_event(self.ev_done)
        else:
            self._bucket(0, self.n, 0, main, scale)
        m.mark_bf16_fresh()          # FlatAdam materialises the per-parameter step counters lazily


def _clip(model, max_norm, grad_scale=1.0):
    from lirec_b200.mlp import model as M
    return M.clip_grad_norm_flat_(model, max_norm, grad_scale=grad_scale)


def reduce_and_step(model, optimizer, fused=None, local_clips=None, global_clips=None, max_norm=0.0):
    """Gradient exchange + optimizer step of one data-parallel iteration: the in-switch fused kernel when
    `fused` (SwitchReduceAdam.attach) is available, else NCCL all_reduce + the optimizer's own step.
    max_norm > 0 clips the reduced gradient to that global L2 norm between the exchange and the step
    (mlp.model.clip_grad_norm_flat_; the norm of the averaged gradient, identical on every rank) and returns the
    pre-clip norm as a 0-d device tensor; otherwise returns None.  The fused step updates parameters before the
    global norm exists, so it cannot clip."""
    if fused is not None:
        if max_norm:
            raise ValueError("reduce_and_step: gradient clipping needs the unfused step (do not attach "
                             "SwitchReduceAdam with --clip_grad_norm)")
        fused.step(local_clips, global_clips)
        return None
    norm = None
    if world_size() > 1:
        from lirec_b200.mlp.model import _FlatOptimizer
        if isinstance(optimizer, _FlatOptimizer):        # FlatAdam, FlatLamb: the average rides in grad_scale
            scale = allreduce_flat_grad(model._flat_grad, local_clips, global_clips)
            if max_norm:
                norm = _clip(model, max_norm, scale)
            optimizer.step(grad_scale=scale)
        else:
            allreduce_flat_grad(model._flat_grad, local_clips, global_clips, average_in_place=True)
            if max_norm:
                norm = _clip(model, max_norm)
            optimizer.step()
    else:
        if max_norm:
            norm = _clip(model, max_norm)
        step = getattr(optimizer, "_step_impl", None)       # FlatAdam / FlatLamb: skip the Optimizer.step hook wrapper
        if step is not None:
            step()
        else:
            optimizer.step()
    return norm
