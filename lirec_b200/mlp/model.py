"""Model family, losses and factory — the reference's mlp/model.py surface on the B200 path.

Same class names, constructor signatures `(n_classes, n_rels=0)`, `forward(x: dict) ->
{'inters', 'rels'}`, loss `forward(output, batch) -> scalar`, `create_model(n_classes, n_rels)
-> (model, loss, optimizer)` and the same `state_dict` names/shapes as the reference
(mlp/model.py:19-609), so released checkpoints load and `torch.optim.Adam` / `torch.save` keep
working.  Everything numeric happens in liblirec_b200.so (hand-written sm_100a kernels behind the
C ABI of include/lirec_b200.h); the nn.Linear submodules below only OWN parameters — their
storage is re-pointed into one flat fp32 buffer (plus a flat gradient buffer and a bf16 shadow)
that the kernels read and write in place.  There is no PyTorch or CPU fallback.
"""
import ctypes as C
import math

import numpy as np
import torch
import torch.nn as nn

from lirec_b200 import _ext, ops
from lirec_b200.packing import PackedBatch, pack_dense_batch
from lirec_b200.utils.arg_pars import opt

__all__ = ["Modalities", "MidFusionMultiClip", "MidFusionMultiClipMaxTracks", "GatingUnit",
           "MultiTaskCrossEntropyLoss", "MultiTaskMaxMargin", "MaxMarginCrossEntropyLoss", "MarginLoss",
           "MarginTrackRelsLoss", "MultiLabelBCELoss", "TrackBCELoss", "create_model", "ModelOutput", "FlatAdam",
           "FlatLamb", "clip_grad_norm_flat_"]

_SLOTS = ("txt", "vis", "tracks1", "tracks2")
_SECOND = ("txt2", "vis2", "tracks12", "tracks22")


class ModelOutput(dict):
    """{'inters', 'rels'} like the reference, produced lazily from the ragged logits.

    `ragged_inters` [Ni, C] / `ragged_rels` [Ni, R] are what the kernels wrote and what the fused
    losses read.  The dense reference-shaped tensors ([B, T, C] / [B, T, R] for the track models)
    are only materialised when somebody indexes the dict (evaluation code); empty candidate slots
    hold -inf there, which is what the reference's track losses leave behind (mlp/model.py:460, 512).
    """

    def __init__(self, batch, ragged_inters, ragged_rels, dense_tracks):
        super().__init__()
        self.batch = batch
        self.ragged_inters = ragged_inters
        self.ragged_rels = ragged_rels
        self._dense_tracks = dense_tracks
        dict.__setitem__(self, "inters", None)
        dict.__setitem__(self, "rels", None)
        self._done = set()

    def _dense(self, ragged):
        if ragged is None:
            return None
        if not self._dense_tracks:
            return ragged
        pb = self.batch
        out = ragged.new_full((pb.B, pb.n_slots, ragged.shape[-1]), float("-inf"))
        return out.index_put((pb["cand_clip"].long(), pb["cand_slot"].long()), ragged)

    def __getitem__(self, key):
        if key in ("inters", "rels") and key not in self._done:
            dict.__setitem__(self, key, self._dense(self.ragged_inters if key == "inters" else self.ragged_rels))
            self._done.add(key)
        return dict.__getitem__(self, key)


class _ModelFn(torch.autograd.Function):
    """lirec_model_forward / lirec_model_backward as one autograd node.  Parameter gradients are
    written by the backward kernels straight into the flat gradient buffer that every `p.grad`
    aliases (`_publish_grads`), so the node takes ONE parameter as its differentiable input — the
    anchor that makes the outputs require grad — instead of all 38 (host time per step)."""

    @staticmethod
    def forward(ctx, module, pb, training, seed, anchor):
        batch_c, ws, inters, rels = module._run_forward(pb, training, seed)
        ctx.module, ctx.pb, ctx.batch_c, ctx.ws = module, pb, batch_c, ws
        if rels is None:
            none = inters.new_empty(0)
            ctx.mark_non_differentiable(none)
            return inters, none
        if inters is None:                       # opt.ints == 0: relationship logits only
            none = rels.new_empty(0)
            ctx.mark_non_differentiable(none)
            return none, rels
        return inters, rels

    @staticmethod
    def backward(ctx, d_inters, d_rels):
        ctx.module._run_backward(ctx.batch_c, ctx.ws, d_inters if ctx.module._ints else None, d_rels)
        ctx.ws = None
        return None, None, None, None, None


class _HotPath(nn.Module):
    """Shared machinery of the three model classes."""
    kind = None

    def _build(self, n_classes, n_rels, ints, ctx, gates):
        self.n_classes, self.n_rels = n_classes, n_rels
        self._ints, self._ctx, self._gates = bool(ints), bool(ctx), bool(gates and ctx)
        if not self._ints:
            # opt.ints == 0 (reference model.py:102, 140, 151, 208): no interaction branch, no interaction head —
            # the context branch and the relationship head alone.  The reference's GatingUnit reads both features
            # (model.py:349-352: None.view fails), so gates must be off, and there must be a context branch.
            if not self._ctx:
                raise ValueError("opt.ints == 0 needs opt.ctx == 1 (a model without either branch has no output)")
            if self._gates:
                raise ValueError("opt.ints == 0 needs opt.gates == 0 (the reference's GatingUnit fails on the "
                                 "missing interaction feature, mlp/model.py:349-352)")
        J = opt.joint_dim
        dims = {"txt": opt.text_dim, "vis": opt.visual_dim, "tracks1": opt.track_dim, "tracks2": opt.track_dim}
        # Modality slots.  Only Modalities switches on opt.modality / opt.tracks (model.py:27-46); the
        # context models always build all four (model.py:102-129, 220-246).
        txt = vis = tracks = True
        if self.kind == "modalities":
            txt, vis, tracks = opt.modality in ("m", "t"), opt.modality in ("m", "v"), bool(opt.tracks)
            if opt.modality not in ("m", "t", "v"):
                raise ValueError("opt.modality must be m, t or v")
            if opt.modality != "m" and tracks:
                # the reference sizes out_ints for J + J inputs but feeds it J (model.py:47, 83-86): it crashes
                raise ValueError("Modalities with opt.modality='%s' needs opt.tracks=False (the reference's "
                                 "forward fails on the out_ints shape otherwise)" % opt.modality)
        self._slot_mask = (1 if txt else 0) | (2 if vis else 0) | (12 if tracks else 0)
        # same construction order as the reference (mlp/model.py:29-50, 104-143, 222-259) so that the
        # same torch seed gives bit-identical initial weights
        for br in ((["ints"] if self._ints else []) + (["ctx"] if self._ctx else [])):
            if txt:
                setattr(self, "txt_%s" % br, nn.Linear(dims["txt"], J))
                setattr(self, "txt2_%s" % br, nn.Linear(J, J))
            if vis:
                setattr(self, "vis_%s" % br, nn.Linear(dims["vis"], J))
                setattr(self, "vis2_%s" % br, nn.Linear(J, J))
            if tracks:
                setattr(self, "tracks1_%s" % br, nn.Linear(dims["tracks1"], J))
                setattr(self, "tracks2_%s" % br, nn.Linear(dims["tracks2"], J))
                setattr(self, "tracks12_%s" % br, nn.Linear(J, J // 2))
                setattr(self, "tracks22_%s" % br, nn.Linear(J, J // 2))
        out_dim_ints = (J if txt else 0) + (J if vis else 0) + (J if tracks else 0)
        if self._gates:
            out_dim_ints = J * opt.mid_m_ints
            self.gates_ints = GatingUnit(in_dim1=3 * J, in_dim2=3 * J, out_dim=out_dim_ints)
        if self._ints:
            self.out_ints = nn.Linear(out_dim_ints, n_classes)
        if self._ctx:
            self.out_ctx = nn.Linear(3 * J, n_rels)
        self.dropout = nn.Dropout(p=opt.dropout)   # holder of p, as in the reference (model.py:52)
        self._gate_dim = out_dim_ints
        self._flat = self._flat_grad = self._flat_bf16 = None
        self._param_list = None
        self._table = self._clip_partials = None
        self._last_grad_norm = None              # pre-clip gradient norm of the last clip_grad_norm_flat_ (device)
        self._versions = None
        self._dirty = True
        self._step = 0

    # ---- flat parameter storage ----------------------------------------------------------------
    def _sync_flat(self):
        """(Re)build the flat fp32 / grad / bf16 buffers and point every parameter into them."""
        pl = self._param_list
        if pl is not None and not self._dirty and self._flat is not None:
            # fast path (every step, ~6 us): nn.Module._apply (.to / .cuda / .float) marks the model dirty;
            # the pointer walk over the cached list catches a parameter re-pointed by hand (p.data = ...)
            base = self._flat.data_ptr()
            for p, off in zip(pl, self._offsets):
                if p.data_ptr() != base + 4 * off:
                    break
            else:
                return
        params = [p for p in self.parameters()]
        dev = params[0].device
        if dev.type != "cuda":
            raise RuntimeError("lirec_b200 model parameters are on %s; move the model to a B200 "
                               "(model.to('cuda')) — there is no CPU path" % dev)
        ok = self._flat is not None and self._flat.device == dev and len(params) == len(self._param_list)
        if ok:
            base = self._flat.data_ptr()
            for p, off in zip(params, self._offsets):
                if p.data_ptr() != base + 4 * off:
                    ok = False
                    break
        if ok:
            self._dirty = False
            return
        _ext.require_device(dev)
        offsets, total = [], 0
        for p in params:
            offsets.append(total)
            total += (p.numel() + 63) // 64 * 64           # 256-byte aligned segments (TMA needs 16)
        flat = torch.zeros(total, dtype=torch.float32, device=dev)
        for p, off in zip(params, offsets):
            flat[off:off + p.numel()].copy_(p.data.reshape(-1).float())
            p.data = flat[off:off + p.numel()].view(p.shape)
        self._flat, self._offsets, self._param_list = flat, offsets, params
        self._flat_grad = torch.zeros_like(flat)
        self._flat_bf16 = torch.zeros(total, dtype=torch.bfloat16, device=dev)
        self._table = self._clip_partials = None
        self._versions = None
        self._dirty = False
        self._build_structs()

    def _tensor_table(self):
        """(begin, len): int64 device tensors [n_parameters], the float offset and length of every parameter in the
        flat buffers, in model.parameters() order (the tensor table of lirec_lamb_flat / lirec_grad_clip_flat).
        Built once per flat layout (_sync_flat must have run)."""
        if self._table is None:
            dev = self._flat.device
            self._table = (torch.tensor(self._offsets, dtype=torch.int64, device=dev),
                           torch.tensor([p.numel() for p in self._param_list], dtype=torch.int64, device=dev))
        return self._table

    def _apply(self, fn, *args, **kwargs):
        self._dirty = True                    # parameters may have been re-allocated (model.to(...))
        return super()._apply(fn, *args, **kwargs)

    def use_grad_buffer(self, buf):
        """Adopt `buf` (flat fp32, same size) as the gradient buffer — e.g. symmetric memory for the
        in-switch data-parallel reduction (lirec_b200/dp.py:SwitchReduceAdam)."""
        self.use_buffers(grad=buf)

    def use_buffers(self, flat=None, grad=None, bf16=None):
        """Adopt caller-owned storage (same sizes, same device) for the flat fp32 parameters, the flat gradient
        buffer and / or the bf16 shadow — symmetric memory for the in-switch data-parallel step
        (lirec_b200/dp.py:SwitchReduceAdam).  Contents are carried over; every nn.Parameter is re-pointed."""
        self._sync_flat()
        n, dev = self._flat.numel(), self._flat.device
        for buf, dt in ((flat, torch.float32), (grad, torch.float32), (bf16, torch.bfloat16)):
            assert buf is None or (buf.dtype == dt and buf.numel() == n and buf.device == dev and buf.is_contiguous())
        with torch.no_grad():
            if flat is not None:
                flat.copy_(self._flat)
                for p, off in zip(self._param_list, self._offsets):
                    p.data = flat[off:off + p.numel()].view(p.shape)
                self._flat = flat
            if bf16 is not None:
                bf16.copy_(self._flat_bf16)
                self._flat_bf16 = bf16
            if grad is not None:
                grad.copy_(self._flat_grad)
                self._flat_grad = grad
                for p in self._param_list:
                    p.grad = None
        self._build_structs()

    def _grad_view(self, i):
        p, off = self._param_list[i], self._offsets[i]
        return self._flat_grad[off:off + p.numel()].view(p.shape)

    def _publish_grads(self):
        """Expose the flat gradient buffer through p.grad (zero-copy when p.grad is None)."""
        for p, g in zip(self._param_list, self._grad_views):
            pg = p.grad
            if pg is None:
                p.grad = g
            elif pg is not g and pg.data_ptr() != g.data_ptr():
                pg.add_(g)
            # else: p.grad already aliases the flat buffer, which backward has just overwritten

    def _refresh_bf16(self):
        versions = tuple(p._version for p in self._param_list)
        if versions != self._versions:
            ops.cast_bf16(self._flat, self._flat_bf16)
            self._versions = versions

    def mark_bf16_fresh(self):
        """Called by FlatAdam after it has rewritten the bf16 shadow itself."""
        self._versions = tuple(p._version for p in self._param_list)

    def _linear_struct(self, lin):
        idx = {id(p): i for i, p in enumerate(self._param_list)}
        iw, ib = idx[id(lin.weight)], idx[id(lin.bias)]
        s = _ext.Linear()
        s.w_bf16 = self._flat_bf16.data_ptr() + 2 * self._offsets[iw]
        s.bias = self._flat.data_ptr() + 4 * self._offsets[ib]
        s.grad_w = self._flat_grad.data_ptr() + 4 * self._offsets[iw]
        s.grad_b = self._flat_grad.data_ptr() + 4 * self._offsets[ib]
        s.out_f, s.in_f = lin.out_features, lin.in_features
        return s

    def _build_structs(self):
        P = _ext.ModelParams()
        for br, enc in (("ints", P.enc_ints), ("ctx", P.enc_ctx)):
            if (br == "ctx" and not self._ctx) or (br == "ints" and not self._ints):
                continue
            for s in range(4):
                if not (self._slot_mask >> s) & 1:
                    continue
                enc.l1[s] = self._linear_struct(getattr(self, "%s_%s" % (_SLOTS[s], br)))
                enc.l2[s] = self._linear_struct(getattr(self, "%s_%s" % (_SECOND[s], br)))
        if self._gates:
            P.gate = self._linear_struct(self.gates_ints.fc_out)
        if self._ints:
            P.out_ints = self._linear_struct(self.out_ints)
        if self._ctx:
            P.out_ctx = self._linear_struct(self.out_ctx)
        cfg = _ext.ModelCfg()
        cfg.text_dim, cfg.visual_dim, cfg.track_dim = opt.text_dim, opt.visual_dim, opt.track_dim
        cfg.joint_dim, cfg.gate_dim = opt.joint_dim, self._gate_dim
        cfg.n_classes, cfg.n_rels = self.n_classes, self.n_rels
        cfg.ctx, cfg.gates = int(self._ctx), int(self._gates)
        cfg.guard_zero = int(self.kind == "maxtracks")
        cfg.dropout_p = float(self.dropout.p)
        cfg.slot_mask = int(self._slot_mask)
        cfg.no_ints = int(not self._ints)
        self._params_c, self._cfg_c = P, cfg
        self._grad_views = [self._grad_view(i) for i in range(len(self._param_list))]
        # index, not the Parameter itself: assigning a Parameter to a module attribute would register it
        self._anchor_idx = next((i for i, p in enumerate(self._param_list) if p.requires_grad), 0)

    def _batch_struct(self, pb, training, seed):
        """lirec_batch of `pb`; the pointer part is built once per (batch, branch set) and cached on the
        batch — per step only the dropout seed and the training flag change."""
        cache = pb.__dict__.setdefault("_c_batch", {})
        key = (self._ctx, pb.clip_bank.data_ptr(), pb.track_bank.data_ptr())   # banks may be swapped (resident staging)
        b = cache.get(key)
        if b is None:
            b = _ext.Batch()
            b.clip_bank, b.clip_ld = pb.clip_bank.data_ptr(), pb.clip_bank.stride(0)
            b.n_clip, b.n_clip_ints = pb.n_clip, pb.n_clip_ints
            b.track_bank, b.track_ld = pb.track_bank.data_ptr(), pb.track_bank.stride(0)
            b.n_track, b.n_track_ints = pb.n_track, pb.n_track_ints
            b.n_cand, b.n_ctx_rows = pb.n_cand, pb.n_ctx_rows if self._ctx else 0
            b.cand_rows = pb.table_ptr("cand_rows")
            if self._ctx:
                if not pb.has_ctx:
                    raise RuntimeError("the model has a context branch but the batch carries no context tables")
                b.ctx_rows, b.ctx_off = pb.table_ptr("ctx_rows"), pb.table_ptr("ctx_off")
                b.ctx_owner = pb.table_ptr("ctx_owner")
            else:  # ints-only models ignore context tables; bank prefixes still apply
                b.n_clip, b.n_track = pb.n_clip_ints, pb.n_track_ints
            for s in range(3):
                b.inv_cand_off[s] = pb.table_ptr("inv_cand_off%d" % s)
                b.inv_cand_idx[s] = pb.table_ptr("inv_cand_idx%d" % s)
                if self._ctx:
                    b.inv_ctx_off[s] = pb.table_ptr("inv_ctx_off%d" % s)
                    b.inv_ctx_idx[s] = pb.table_ptr("inv_ctx_idx%d" % s)
            cache[key] = b
        b = _ext.Batch.from_buffer_copy(b)       # backward keeps this step's copy (its dropout seed)
        b.seed, b.training = int(seed) & 0xFFFFFFFF, int(bool(training))
        return b

    def reserve_workspace(self, pb):
        """Size the step workspace for device batch `pb` ahead of its first step (setup, no kernel runs): the
        high-water capacity `_run_forward` allocates from then already covers it, and the batch's C struct is cached."""
        self._sync_flat()
        batch_c = self._batch_struct(pb, False, 0)
        nbytes = int(_ext.lib().lirec_model_workspace_bytes(C.byref(self._cfg_c), C.byref(batch_c)))
        if nbytes > getattr(self, "_ws_cap", 0):
            self._ws_cap = -(-int(nbytes * 1.05 + 256) // 4096) * 4096
        return self._ws_cap

    # ---- the two native calls ------------------------------------------------------------------
    def _run_forward(self, pb, training, seed):
        """lirec_model_forward on `pb`.  Returns (batch struct, workspace, inters [Ni,C], rels [Ni,R] | None);
        the first two are what lirec_model_backward needs."""
        batch_c = self._batch_struct(pb, training, seed)
        L = _ext.lib()
        nbytes = L.lirec_model_workspace_bytes(C.byref(self._cfg_c), C.byref(batch_c))
        # high-water capacity: the workspace follows the batch's row counts (+- 1 % from batch to batch), and a
        # request a little larger than every cached block costs a cudaMalloc behind the GPU's queue
        if int(nbytes) > getattr(self, "_ws_cap", 0):
            self._ws_cap = -(-int(int(nbytes) * 1.05 + 256) // 4096) * 4096
        ws = torch.empty(self._ws_cap, dtype=torch.uint8, device=pb.device)
        Ni = pb.n_cand
        inters = torch.empty(Ni, self.n_classes, dtype=torch.float32, device=pb.device) if self._ints else None
        rels = torch.empty(Ni, self.n_rels, dtype=torch.float32, device=pb.device) if self._ctx else None
        _ext.check(L.lirec_model_forward(
            C.byref(self._cfg_c), C.byref(self._params_c), C.byref(batch_c), ws.data_ptr(), ws.numel(),
            inters.data_ptr() if inters is not None else None, rels.data_ptr() if rels is not None else None,
            _ext.stream_ptr()))
        return batch_c, ws, inters, rels

    def _run_backward(self, batch_c, ws, d_inters, d_rels):
        """lirec_model_backward: every parameter gradient of the step into the flat gradient buffer."""
        d_inters_ptr = None
        if self._ints:
            d_inters = d_inters.contiguous()
            d_inters_ptr = d_inters.data_ptr()
        d_rels_ptr = None
        if self._ctx:
            d_rels = d_rels.contiguous()
            d_rels_ptr = d_rels.data_ptr()
        ev = getattr(self, "_heads_event", None)       # set by dp.SwitchReduceAdam.arm(): overlap bucket 0
        _ext.check(_ext.lib().lirec_model_backward(
            C.byref(self._cfg_c), C.byref(self._params_c), C.byref(batch_c), ws.data_ptr(), ws.numel(),
            d_inters_ptr, d_rels_ptr, _ext.stream_ptr(), C.c_void_p(ev.cuda_event) if ev is not None else None))
        self._publish_grads()

    # ---- batches -------------------------------------------------------------------------------
    def _packed(self, x):
        if isinstance(x, PackedBatch):
            pb = x
        elif isinstance(x, dict) and isinstance(x.get("packed"), PackedBatch):
            pb = x["packed"]
        elif isinstance(x, dict) and "features" in x:
            # reference dense batch: compatibility path (host-side packing, no deduplication)
            if self.kind == "maxtracks":
                feats = x["features"]
                if feats.dim() == 3 and self._ctx:      # already flattened by a previous call (model.py:274)
                    raise RuntimeError("dense 'features' must be [B, T, S+1, D]")
            pb = pack_dense_batch(x, self.kind, n_slots=None)
            x["packed"] = pb
        else:
            raise TypeError("model input must be a PackedBatch or a reference batch dict")
        if pb.device is None:
            dev = self._flat.device
            pb = pb.to_device(dev)
            if isinstance(x, dict):
                x["packed"] = pb
        return pb

    def set_rank(self, rank):
        """Data parallel: mix the rank into the dropout seeds, so that row i of rank 0's shard and row i of rank
        1's shard do not share their masks (the masks are keyed by local row position)."""
        self._seed_rank = int(rank)

    def next_seed(self):
        self._step += 1
        return (int(opt.seed) * 0x9E3779B1 + self._step * 0x85EBCA6B +
                getattr(self, "_seed_rank", 0) * 0xC2B2AE3D) & 0xFFFFFFFF

    def forward(self, x, seed=None):
        self._sync_flat()
        self._refresh_bf16()
        pb = self._packed(x)
        training = self.training and self.dropout.p > 0
        if seed is None:
            seed = self.next_seed() if training else 0
        anchor = self._param_list[self._anchor_idx]
        if not anchor.requires_grad:             # parameters frozen since the structs were built
            self._anchor_idx = next((i for i, p in enumerate(self._param_list) if p.requires_grad), self._anchor_idx)
            anchor = self._param_list[self._anchor_idx]
        if torch.is_grad_enabled() and anchor.requires_grad:
            inters, rels = _ModelFn.apply(self, pb, training, seed, anchor)
            if not self._ints:
                inters = None
        else:                                    # inference (mlp/test.py runs under no_grad): no autograd node
            _, _, inters, rels = self._run_forward(pb, training, seed)
        return ModelOutput(pb, inters, rels if self._ctx else None, dense_tracks=(self.kind == "maxtracks"))


class Modalities(_HotPath):
    """Reference: mlp/model.py:19-92 (interaction logits from text + visual + two tracks)."""
    kind = "modalities"

    def __init__(self, n_classes, n_rels=0):
        super().__init__()
        self._build(n_classes, n_rels, ints=1, ctx=0, gates=0)


class MidFusionMultiClip(_HotPath):
    """Reference: mlp/model.py:95-211 (clip + masked-mean context, gate, two heads)."""
    kind = "midfusion"

    def __init__(self, n_classes, n_rels=0):
        super().__init__()
        self._build(n_classes, n_rels, ints=opt.ints, ctx=opt.ctx, gates=opt.gates)


class MidFusionMultiClipMaxTracks(_HotPath):
    """Reference: mlp/model.py:214-339 (every candidate track pair is its own row)."""
    kind = "maxtracks"

    def __init__(self, n_classes, n_rels=0):
        super().__init__()
        self._build(n_classes, n_rels, ints=opt.ints, ctx=opt.ctx, gates=opt.gates)

    def forward(self, x, seed=None):
        assert opt.tr_maximize
        return super().forward(x, seed=seed)


class GatingUnit(nn.Module):
    """Parameter holder of the gate (reference: mlp/model.py:342-354); the computation
    dropout(relu(fc_out(cat(ctx, ints)))) runs inside lirec_model_forward."""

    def __init__(self, in_dim1, in_dim2, out_dim):
        super().__init__()
        self.in_dim1, self.in_dim2, self.out_dim = in_dim1, in_dim2, out_dim
        self.fc_out = nn.Linear(in_dim1 + in_dim2, out_dim)
        self.dropout = nn.Dropout(p=opt.dropout)


# =================================================================================================
# losses
# =================================================================================================
class _LossFn(torch.autograd.Function):
    """A fused loss kernel already produced d(loss)/d(logits); backward just scales them."""

    @staticmethod
    def forward(ctx, loss_terms, grads, *logits):
        ctx.grads = grads
        return loss_terms.sum()

    @staticmethod
    def backward(ctx, g):
        return (None, None) + tuple(None if d is None else d * g for d in ctx.grads)


def _batch_of(output, args):
    if isinstance(output, ModelOutput):
        return output.batch
    if isinstance(args, dict) and isinstance(args.get("packed"), PackedBatch):
        return args["packed"]
    raise TypeError("lirec_b200 losses expect the ModelOutput returned by a lirec_b200 model")


class _FusedLoss(nn.Module):
    """Base of the five losses.  `terms_and_grads(x, args)` runs the fused forward+gradient kernels and
    returns (loss terms, d loss / d inters | None, d loss / d rels | None); `forward` wraps that in one
    autograd node, `train_step` below consumes it directly."""

    def terms_and_grads(self, x, args):
        raise NotImplementedError

    def has_rel_term(self):
        """Whether terms_and_grads runs the relationship term of the multi-task losses (`_rel_term`)."""
        return False

    def forward(self, x, args):
        terms, d_i, d_r = self.terms_and_grads(x, args)
        grads, logits = [], []
        if d_i is not None:
            grads.append(d_i), logits.append(x.ragged_inters)
        if d_r is not None:
            grads.append(d_r), logits.append(x.ragged_rels)
        return _LossFn.apply(terms, tuple(grads), *logits)


def _rel_term(loss_mod, pb, n_sel, run):
    """The relationship term of the multi-task losses: the mean over the rows whose label is not None
    (reference mlp/model.py:404-418, 369-377).  `run(scale)` launches the fused kernel with the given row
    scale and returns (terms, d_rels).  Single process: scale = 1 / n_sel.  Data parallel (the training loop
    sets `loss_mod._dp_world`): the reference's mean runs over the non-None rows of the GLOBAL batch, while the
    gradient exchange weights rank r by B_r / B — so the rank's term is computed unscaled and multiplied, on
    the device, by (B / B_r) / sum_r n_sel_r (one 1-element all_reduce, no host sync); a rank without any
    labelled row still takes part in that all_reduce."""
    world = int(getattr(loss_mod, "_dp_world", 1) or 1)
    if world <= 1:
        return run(1.0 / n_sel) if n_sel else (None, None)
    import torch.distributed as dist
    dev = pb.device
    cnt = torch.full((1,), float(n_sel), dtype=torch.float32, device=dev)
    dist.all_reduce(cnt)
    b_glob = float(getattr(pb.host, "global_clips", None) or pb.B * world)
    scale = torch.where(cnt > 0, (b_glob / float(pb.B)) / cnt.clamp(min=1.0), torch.zeros_like(cnt))
    if not n_sel:
        return None, None
    t, d = run(1.0)
    return t * scale, d * scale


def _labelled_rel_term(loss_mod, pb, kernel):
    """`_rel_term` over the rows whose relationship label is not None (`loss_mod.n_rels`): `kernel(labels, scale)`
    launches the fused row kernel on the batch's labels with None mapped to -1, which it skips, and returns
    (terms, d_rels).  The count of labelled rows comes from the host copy of the batch."""
    host = pb.host if pb.device is not None else pb
    n_sel = int((host["rels_label"] != loss_mod.n_rels).sum())

    def run(scale):
        sel = pb["rels_label"].clone()
        sel[sel == loss_mod.n_rels] = -1                 # rows labelled None are skipped (model.py:369, 406)
        return kernel(sel, scale)
    return _rel_term(loss_mod, pb, n_sel, run)


def dp_empty_shard_collectives(loss_mod, device):
    """The collectives a loss would have issued on a rank that holds an EmptyShard this step: the one all_reduce of
    `_rel_term`, issued whenever the loss has a relationship term."""
    if int(getattr(loss_mod, "_dp_world", 1) or 1) > 1 and loss_mod.has_rel_term():
        import torch.distributed as dist
        dist.all_reduce(torch.zeros(1, dtype=torch.float32, device=device))


class MaxMarginCrossEntropyLoss(_FusedLoss):
    """Reference: mlp/model.py:422-441."""

    def __init__(self):
        super().__init__()
        self.m = opt.margin

    def terms_and_grads(self, x, args):
        pb = _batch_of(x, args)
        logits = x.ragged_inters
        terms, d = ops.loss_rowmargin(logits, pb["labels"], pb.multilab, self.m, 1.0 / logits.shape[0])
        return terms, d, None


class MultiTaskMaxMargin(_FusedLoss):
    """Reference: mlp/model.py:381-419."""

    def __init__(self, n_rels=0):
        super().__init__()
        self.m = opt.margin
        self.n_rels = n_rels

    def has_rel_term(self):
        return opt.ctx == 1

    def terms_and_grads(self, x, args):
        pb = _batch_of(x, args)
        terms, d_i, d_r = [], None, None
        if opt.ints == 1:
            li = x.ragged_inters
            t, d_i = ops.loss_rowmargin(li, pb["labels"], pb.multilab, self.m, opt.lymbda / li.shape[0])
            terms.append(t)
        if self.has_rel_term():
            lr = x.ragged_rels
            t, d_r = _labelled_rel_term(self, pb, lambda sel, scale: ops.loss_rowmargin(lr, sel, None, self.m, scale))
            if t is not None:
                terms.append(t)
        return torch.cat(terms), d_i, d_r


class _TrackLoss(_FusedLoss):
    n_rels = 0

    def set_rank(self, rank):
        self._seed_rank = int(rank)            # tr_cat_distr draws differ per data-parallel rank

    def _draw_seed(self):
        """Counter-hash seed of this step's tr_cat_distr draw (per loss call and data-parallel rank)."""
        self._draws = getattr(self, "_draws", 0) + 1
        return int(opt.seed) * 0x9E3779B1 + self._draws * 0xC2B2AE35 + getattr(self, "_seed_rank", 0) * 0x27D4EB2F

    def _run(self, x, args, kernel, lymbda, **kw):
        """terms_and_grads of a track loss: `kernel` is ops.loss_track or ops.loss_bce_track, `lymbda` the weight of
        the interaction term and `kw` the kernel's own arguments."""
        assert opt.tr_maximize
        assert not (opt.tr_cat_distr and opt.tr_correct)                 # model.py:469, 539
        seed = self._draw_seed()
        pb = _batch_of(x, args)
        n_rels = self.n_rels
        li, lr = x.ragged_inters, x.ragged_rels if n_rels else None
        if li is None:
            raise ValueError("the track-assignment losses need interaction logits (opt.ints == 1), as in the "
                             "reference (mlp/model.py:455, 507 dereference x['inters'])")
        terms, assign, d_i, d_r = kernel(
            li, lr, pb["cand_off"], pb["labels"], pb["rels_label"] if n_rels else None, pb["gt_tracks"],
            pb.multilab, lymbda=lymbda, n_rels=n_rels, tr_correct=opt.tr_correct, max_slots=pb.n_slots,
            cat_distr=bool(opt.tr_cat_distr), seed=seed, **kw)
        self.last_assignment = assign
        return terms, d_i, (d_r if n_rels else None)


class MarginLoss(_TrackLoss):
    """Reference: mlp/model.py:444-494 (weakly supervised track assignment, interactions only)."""

    def __init__(self):
        super().__init__()
        self.m = opt.tr_margin

    def terms_and_grads(self, x, args):
        return self._run(x, args, ops.loss_track, 1.0, margin=self.m,
                         max_neg=bool(opt.tr_max_neg and opt.tr_sum_max_flag))


class MarginTrackRelsLoss(_TrackLoss):
    """Reference: mlp/model.py:497-575 (joint interaction + relationship assignment)."""

    def __init__(self, n_rels=0):
        super().__init__()
        self.m = opt.tr_margin
        self.n_rels = n_rels

    def terms_and_grads(self, x, args):
        return self._run(x, args, ops.loss_track, opt.lymbda, margin=self.m,
                         max_neg=bool(opt.tr_max_neg and opt.tr_sum_max_flag))


class MultiTaskCrossEntropyLoss(_FusedLoss):
    """Reference: mlp/model.py:357-378 (never selected by create_model, model.py:586-597): softmax
    cross-entropy of the interaction logits (optionally class-weighted) plus that of the relationship
    logits of the rows whose label is not None, both as fused forward+gradient kernels."""

    def __init__(self, n_classes, weights=None, n_rels=0):
        super().__init__()
        self.n_classes, self.n_rels = n_classes, n_rels
        self.weights = None if weights is None else torch.tensor(weights).float()

    def has_rel_term(self):
        return not opt.mod_check and opt.ctx == 1          # the model has relationship logits (Modalities has none)

    def terms_and_grads(self, x, args):
        pb = _batch_of(x, args)
        host = pb.host if pb.device is not None else pb
        li = x.ragged_inters
        lab_i = pb["labels"]
        if li.shape[0] != lab_i.numel():
            raise RuntimeError("MultiTaskCrossEntropyLoss expects one interaction row per clip")
        w = None if self.weights is None else self.weights.to(li.device)
        denom = float(self.weights[torch.as_tensor(host["labels"]).long()].sum()) if w is not None else li.shape[0]
        t, d_i = ops.loss_ce(li, lab_i, w, 1.0 / denom)
        terms, d_r = [t], None
        if self.has_rel_term():
            lr = x.ragged_rels
            t, d_r = _labelled_rel_term(self, pb, lambda sel, scale: ops.loss_ce(lr, sel, None, scale))
            if t is not None:
                terms.append(t)
        return torch.cat(terms), d_i, d_r


def _soft_pos(pb):
    """The batch's soft-label positives (uint8 [B, C]) under --soft_gt, None otherwise."""
    if not opt.soft_gt:
        return None
    sp = getattr(pb, "soft_pos", None)
    if sp is None:
        raise RuntimeError("--soft_gt is set but the batch carries no soft labels (soft_pos): only the index-only "
                           "MovieGraphs dataset (and the synthetic annotation world) builds them; refusing to train "
                           "the BCE loss on the hard labels alone")
    return sp


class MultiLabelBCELoss(_FusedLoss):
    """Multi-label sigmoid BCE for Modalities / MidFusionMultiClip (lirec_loss_bce_fwd_bwd).  Interaction rows:
    target 1 on the label (and, under --soft_gt, on the co-occurring interactions of the batch's `soft_pos`),
    target 0 on the classes multilab_weights keeps as negatives, the rest left out.  Without a relationship
    term (n_rels == 0) the interaction term is a mean over the clips, like MaxMarginCrossEntropyLoss; with one it
    is weighted by lymbda and gated by opt.ints, and the relationship term (one-hot target, no mask) is the mean
    over the rows whose label is not None, like MultiTaskMaxMargin."""

    def __init__(self, n_rels=0):
        super().__init__()
        self.n_rels = n_rels

    def has_rel_term(self):
        return bool(self.n_rels) and opt.ctx == 1

    def terms_and_grads(self, x, args):
        pb = _batch_of(x, args)
        terms, d_i, d_r = [], None, None
        if not self.n_rels or opt.ints == 1:
            li = x.ragged_inters
            w = (opt.lymbda if self.n_rels else 1.0) / li.shape[0]
            t, d_i = ops.loss_bce(li, pb["labels"], pb.multilab, _soft_pos(pb), w)
            terms.append(t)
        if self.has_rel_term():
            lr = x.ragged_rels
            t, d_r = _labelled_rel_term(self, pb, lambda sel, scale: ops.loss_bce(lr, sel, None, None, scale))
            if t is not None:
                terms.append(t)
        return torch.cat(terms), d_i, d_r


class TrackBCELoss(_TrackLoss):
    """Sigmoid BCE over the weakly supervised track assignment of MidFusionMultiClipMaxTracks
    (lirec_loss_bce_track_fwd_bwd): t* is the margin losses' assignment (same arg-max, tr_correct slot and
    tr_cat_distr draw for the same step); (t*, label) and, under --soft_gt, (t*, soft positives) are the
    targets, the margin losses' negatives the zeros.  n_rels > 0 adds the relationship term, weighting the
    interaction term by lymbda as MarginTrackRelsLoss does."""

    def __init__(self, n_rels=0):
        super().__init__()
        self.n_rels = n_rels

    def terms_and_grads(self, x, args):
        return self._run(x, args, ops.loss_bce_track, opt.lymbda if self.n_rels else 1.0,
                         pos_mask=_soft_pos(_batch_of(x, args)))


def train_step(model, loss, x, seed=None):
    """forward + loss + backward of one iteration WITHOUT the autograd engine: the loss kernels already
    emit d loss / d logits, so `loss(model(x), x).backward()` (mlp/train.py:57-62) is three native calls
    in a row.  Gradients land in the flat buffer behind every `p.grad` exactly as after `.backward()`
    (bit-identical: the autograd path multiplies them by the incoming 1.0); the caller then runs
    `optimizer.step()`.  Returns the loss as a 0-d device tensor.  At the reference's batch size (64
    clips) the host time of the autograd round trip exceeded the device time of the whole step."""
    if not isinstance(model, _HotPath) or not isinstance(loss, _FusedLoss):
        raise TypeError("train_step needs a lirec_b200 model and a lirec_b200 loss")
    model._sync_flat()
    model._refresh_bf16()
    pb = model._packed(x)
    training = model.training and model.dropout.p > 0
    if seed is None:
        seed = model.next_seed() if training else 0
    with torch.no_grad():
        batch_c, ws, inters, rels = model._run_forward(pb, training, seed)
        out = ModelOutput(pb, inters, rels if model._ctx else None, dense_tracks=(model.kind == "maxtracks"))
        terms, d_i, d_r = loss.terms_and_grads(out, x if isinstance(x, dict) else {})
        value = terms.sum()
        if d_i is None and model._ints:
            d_i = torch.zeros_like(inters)
        if d_r is None and model._ctx:
            d_r = torch.zeros_like(rels)
        model._run_backward(batch_c, ws, d_i, d_r)
    return value


# =================================================================================================
# optimizer + factory
# =================================================================================================
class _FlatOptimizer(torch.optim.Optimizer):
    """What FlatAdam and FlatLamb share: Adam moments in two flat buffers laid out like the model's flat parameter
    buffer, per-parameter state views into them, and torch.optim.Adam's state_dict layout (per-parameter 'step',
    'exp_avg', 'exp_avg_sq').  Subclasses launch their kernel in _launch(step, grad_scale)."""

    def __init__(self, model, defaults):
        self.model = model
        model._sync_flat()
        super().__init__(model._param_list, defaults)
        self._m = torch.zeros_like(model._flat)
        self._v = torch.zeros_like(model._flat)
        self._t = 0
        for i, p in enumerate(model._param_list):
            off, n = model._offsets[i], p.numel()
            self.state[p] = {"step": torch.tensor(0.0), "exp_avg": self._m[off:off + n].view(p.shape),
                             "exp_avg_sq": self._v[off:off + n].view(p.shape)}

    def _step_impl(self, grad_scale=1.0):
        """The step itself, without torch.optim.Optimizer's per-call hook / profiler wrapper (lirec_b200's
        own loop calls this directly: ~25 us of host time per step at 64-clip batches).  grad_scale multiplies
        the gradients (the data-parallel 1/world average)."""
        self._t += 1
        self._launch(self.param_groups[0], grad_scale)
        self.model.mark_bf16_fresh()

    def step(self, closure=None, grad_scale=1.0):
        self._step_impl(grad_scale)

    def zero_grad(self, set_to_none=True):
        # backward overwrites the flat gradient buffer; p.grad keeps aliasing it
        if set_to_none:
            for p in self.model._param_list:
                p.grad = None

    # The per-parameter 'step' counters of torch.optim.Adam's state layout are all equal to the
    # number of fused steps taken; they are materialised when the state is looked at, not 38 times
    # per step.
    def _sync_steps(self):
        for st in self.state.values():
            st["step"].fill_(float(self._t))

    def state_dict(self):
        sync = getattr(self, "_shard_sync", None)        # data parallel, sharded moments: gather them first
        if sync is not None:
            sync()
        self._sync_steps()
        return super().state_dict()

    def load_state_dict(self, state_dict):
        """Accepts a torch.optim.Adam / FlatAdam / FlatLamb state (reference checkpoints: mlp/train.py:84-106):
        the moments are copied into the flat buffers, which the per-parameter state keeps aliasing."""
        super().load_state_dict(state_dict)
        m, steps = self.model, []
        with torch.no_grad():
            for i, p in enumerate(m._param_list):
                off, n = m._offsets[i], p.numel()
                st = self.state.get(p)
                mv, vv = self._m[off:off + n].view(p.shape), self._v[off:off + n].view(p.shape)
                if st is None or "exp_avg" not in st:      # fresh parameter (no step taken when saved)
                    mv.zero_(), vv.zero_()
                    step = 0.0
                else:
                    mv.copy_(st["exp_avg"]), vv.copy_(st["exp_avg_sq"])
                    step = float(st["step"])
                steps.append(step)
                self.state[p] = {"step": torch.tensor(step), "exp_avg": mv, "exp_avg_sq": vv}
        if len(set(steps)) > 1:
            raise RuntimeError("%s needs one common step count for all parameters, got %s"
                               % (type(self).__name__, sorted(set(steps))))
        self._t = int(steps[0]) if steps else 0


class FlatAdam(_FlatOptimizer):
    """torch.optim.Adam semantics (coupled L2, reference mlp/model.py:599-601) as ONE fused kernel
    over the model's flat buffers; also refreshes the bf16 weight shadow.  state_dict() has the
    layout of torch.optim.Adam (per-parameter 'step', 'exp_avg', 'exp_avg_sq')."""

    def __init__(self, model, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        super().__init__(model, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))

    def _launch(self, g, grad_scale):
        m = self.model
        ops.adam_flat(m._flat, m._flat_grad, self._m, self._v, m._flat_bf16, g["lr"], g["betas"][0],
                      g["betas"][1], g["eps"], g["weight_decay"], self._t, grad_scale)


class FlatLamb(_FlatOptimizer):
    """LAMB (You et al., "Large Batch Optimization for Deep Learning", ICLR 2020) for large global batches: Adam's
    moments, decoupled weight decay, and a trust ratio ||w|| / ||update|| per nn.Parameter, as two fused kernels
    over the model's flat buffers (lirec_lamb_flat); also refreshes the bf16 weight shadow.  lr is read from
    param_groups[0] every step, so torch LR schedulers apply.  state_dict() has torch.optim.Adam's layout."""

    def __init__(self, model, lr=1e-3, betas=(0.9, 0.999), eps=1e-6, weight_decay=0.0):
        super().__init__(model, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))
        dev = model._flat.device
        self._begin, self._len = model._tensor_table()
        self._partials = ops.lamb_partials(model._flat.numel(), len(model._param_list), device=dev)
        self._trust = torch.ones(len(model._param_list), dtype=torch.float32, device=dev)

    def _launch(self, g, grad_scale):
        m = self.model
        ops.lamb_flat(m._flat, m._flat_grad, self._m, self._v, m._flat_bf16, self._begin, self._len, self._partials,
                      g["lr"], g["betas"][0], g["betas"][1], g["eps"], g["weight_decay"], self._t, grad_scale,
                      trust_out=self._trust)

    def last_trust_ratios(self):
        """Device float32 tensor [n_parameters]: the trust ratio each parameter got in the last step (1 before the
        first), in model.parameters() order."""
        return self._trust


@torch.no_grad()
def clip_grad_norm_flat_(model, max_norm, grad_scale=1.0, tensor_norms=None):
    """torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm) with norm_type 2, over the model's flat gradient
    buffer in three fused launches (lirec_grad_clip_flat) and without a host sync: norm = ||grad_scale * g|| over
    every parameter, then g *= min(max_norm / (norm + 1e-6), 1) in place; nothing is written when the factor is 1.
    grad_scale is the factor the optimizer still applies to the gradients (the data-parallel 1/world average that
    FlatAdam and FlatLamb take in their step): the norm is the norm of the scaled gradient, the buffer is multiplied
    by the clip factor alone.  As in torch, a NaN norm turns the gradients into NaN, and an Inf norm gives a factor of
    0.  Returns the pre-clip total norm as a 0-d float32 device tensor; tensor_norms (optional float32 device tensor
    [n_parameters]) receives every parameter's pre-clip norm, in model.parameters() order."""
    max_norm = float(max_norm)
    if not (math.isfinite(max_norm) and max_norm > 0.0):
        raise ValueError("clip_grad_norm_flat_: max_norm must be finite and > 0 (got %r)" % (max_norm,))
    if model._flat_grad is None:
        raise RuntimeError("clip_grad_norm_flat_: the model has no flat gradient buffer yet (no backward ran)")
    for p, g in zip(model._param_list, model._grad_views):
        pg = p.grad
        if pg is not None and pg is not g and pg.data_ptr() != g.data_ptr():
            # _publish_grads adds into a p.grad that is not a view of the flat buffer; clipping the buffer would
            # leave that gradient, which the torch optimizer reads, unclipped
            raise RuntimeError("clip_grad_norm_flat_: a parameter's .grad lives outside the flat gradient buffer; "
                               "set it to None (optimizer.zero_grad()) before backward")
    begin, length = model._tensor_table()
    if model._clip_partials is None:
        model._clip_partials = ops.lamb_partials(model._flat_grad.numel(), begin.numel(), device=model._flat.device)
    norm = ops.grad_clip_flat(model._flat_grad, begin, length, model._clip_partials, max_norm, grad_scale,
                              tensor_norms_out=tensor_norms)
    model._last_grad_norm = norm
    return norm


def _check_loss_choice():
    """--loss against the rest of the configuration (host only, before any device work)."""
    kind = getattr(opt, "loss", "margin")
    if kind not in ("margin", "bce", "ce"):
        raise ValueError("--loss must be margin, bce or ce (got %r)" % (kind,))
    if kind == "ce" and opt.tr_maximize:
        raise ValueError("--loss ce has no track-assignment form: use margin or bce with --tr_maximize")
    if kind == "ce" and not opt.mod_check and opt.ints == 0:
        raise ValueError("--loss ce needs interaction logits (opt.ints == 1): MultiTaskCrossEntropyLoss always has an "
                         "interaction term")
    if kind == "bce" and opt.tr_max_neg:
        raise ValueError("--loss bce has no max-negative form (--tr_max_neg is a hinge variant)")
    return kind


def _check_optimizer_choice():
    """--optimizer (host only, before any device work)."""
    kind = getattr(opt, "optimizer", "adam")
    if kind not in ("adam", "lamb"):
        raise ValueError("--optimizer must be adam or lamb (got %r)" % (kind,))
    return kind


def _check_clip_choice():
    """--clip_grad_norm (host only, before any device work): 0 is off, anything else a finite maximum norm."""
    v = float(getattr(opt, "clip_grad_norm", 0.0) or 0.0)
    if not (math.isfinite(v) and v >= 0.0):
        raise ValueError("--clip_grad_norm must be 0 (off) or a finite maximum norm > 0 (got %r)" % (v,))
    return v


def create_model(n_classes, n_rels=0):
    """Reference: mlp/model.py:578-609 — same selection logic and return triple.  --loss bce / ce swap in the
    multi-label BCE or the softmax cross-entropy for the reference's max-margin losses; --optimizer lamb swaps in
    FlatLamb for Adam.  --clip_grad_norm is checked here; the training loop applies it."""
    loss_kind = _check_loss_choice()
    optimizer_kind = _check_optimizer_choice()
    _check_clip_choice()
    if opt.device != "cuda":
        raise RuntimeError("lirec_b200 runs on a B200 only (opt.device='%s'); no CPU fallback" % opt.device)
    if opt.tr_maximize:
        model = MidFusionMultiClipMaxTracks(n_classes=n_classes, n_rels=n_rels)
    else:
        model = MidFusionMultiClip(n_classes=n_classes, n_rels=n_rels)
    if opt.mod_check:
        model = Modalities(n_classes=n_classes)
    model = model.to(opt.device)

    if loss_kind == "bce":
        loss = (TrackBCELoss if opt.tr_maximize else MultiLabelBCELoss)(n_rels=n_rels if opt.rels_multitask else 0)
    elif loss_kind == "ce":
        loss = MultiTaskCrossEntropyLoss(n_classes, n_rels=n_rels if opt.rels_multitask else 0)
    elif opt.tr_maximize:
        loss = MarginTrackRelsLoss(n_rels=n_rels) if opt.rels_multitask else MarginLoss()
    else:
        loss = MultiTaskMaxMargin(n_rels=n_rels) if opt.rels_multitask else MaxMarginCrossEntropyLoss()

    if optimizer_kind == "lamb":
        optimizer = FlatLamb(model, lr=opt.lr, weight_decay=opt.weight_decay)
    elif getattr(opt, "fused_adam", 0):
        optimizer = FlatAdam(model, lr=opt.lr, weight_decay=opt.weight_decay)
    else:
        model._sync_flat()
        optimizer = torch.optim.Adam(model.parameters(), lr=opt.lr, weight_decay=opt.weight_decay)

    print(str(model))
    for name, param in model.named_parameters():
        print("%s\n%s" % (str(name), str(param.norm())))
    print(str(loss))
    print(str(optimizer))
    return model, loss, optimizer
