"""Packed ragged batches: the L2 -> L3 contract of this implementation.

The reference dataloader emits, per clip, a dense zero-padded float64 block
`features[20, 19, 6912]` (21 MB) in which every 6912-d row is the concatenation of three
cached vectors — clip text|visual (2816), track of slot-1 person (2048), track of slot-2
person (2048) — and most rows are np.tile copies or padding
(mixed_utils/classification_dataloader.py:329-334, 393-416, 474-497, 531-565;
mixed_utils/mixed_features.py:115-125).  A PackedBatch keeps each cached vector ONCE in two
banks and describes every encoder row as an index triple:

    clip_bank  [n_clip, 2816]   text|visual rows; rows [0, n_clip_ints) belong to the batch's clips
    track_bank [n_track, 2048]  person-track rows; rows [0, n_track_ints) are used by candidates;
                                all-zero rows stand for "no track" (zeros in the reference) — one
                                per clip, so no bank row is referenced by more than a few dozen rows
    cand_off   [B+1]            prefix sums of valid candidate slots per clip (reference slot order)
    cand_rows  [Ni, 3]          (clip, track1, track2) bank rows of every candidate
    ctx_off    [Ni+1]           prefix sums of valid context rows per candidate (= rels_mask sums)
    ctx_rows   [Nx, 3]          (clip, track1, track2) bank rows of every context row
    labels [B], rels_label [Ni], gt_tracks [B,2], multilab [B,C] (uint8)

plus the inverse CSR tables backward needs (bank row -> referencing table rows).  All integer
tables are int32; `to_device()` stages them through one pinned buffer and one async copy.
"""
import numpy as np
import torch

TEXT_DIM, VISUAL_DIM, TRACK_DIM = 768, 2048, 2048
CLIP_DIM = TEXT_DIM + VISUAL_DIM
ROW_DIM = CLIP_DIM + 2 * TRACK_DIM

_INT_TABLES = ["cand_off", "cand_rows", "ctx_off", "ctx_rows", "ctx_owner", "labels", "rels_label",
               "gt_tracks", "inv_cand_off0", "inv_cand_idx0", "inv_cand_off1", "inv_cand_idx1",
               "inv_cand_off2", "inv_cand_idx2", "inv_ctx_off0", "inv_ctx_idx0", "inv_ctx_off1",
               "inv_ctx_idx1", "inv_ctx_off2", "inv_ctx_idx2", "cand_clip", "cand_slot"]


def _csr_inverse(col, n_unique):
    """CSR (off [n_unique+1], idx) listing, for every unique id, the positions where it occurs."""
    col = np.asarray(col, dtype=np.int64)
    # numpy's stable sort is a radix sort for 16-bit keys (5x faster than the merge sort of wider ints)
    key = col.astype(np.uint16) if 0 < n_unique <= 65536 and col.size and col.min() >= 0 else col
    order = np.argsort(key, kind="stable").astype(np.int32)
    counts = np.bincount(col, minlength=n_unique)
    off = np.zeros(n_unique + 1, dtype=np.int32)
    np.cumsum(counts, out=off[1:])
    return off, order


class _DeviceTables(dict):
    """name -> int32 device view into the staged arena, materialised on first use: a train step reads
    a handful of the ~20 tables by tensor and the rest only by address (`PackedBatch.table_ptr`), so
    building every view on every `to_device` was pure host overhead."""

    def __init__(self, arena, layout):
        super().__init__()
        self._arena, self._layout = arena, layout

    def __missing__(self, k):
        off, n, shape = self._layout[k]
        v = self._arena[off:off + n].view(*shape)
        dict.__setitem__(self, k, v)
        return v

    def __contains__(self, k):
        return k in self._layout

    def __iter__(self):
        return iter(self._layout)

    def __len__(self):
        return len(self._layout)

    def keys(self):
        return self._layout.keys()

    def values(self):
        return [self[k] for k in self._layout]

    def items(self):
        return [(k, self[k]) for k in self._layout]

    def get(self, k, default=None):
        return self[k] if k in self._layout else default


class PackedBatch:
    """Host (numpy) or device (torch) packed batch. Build with `PackedBatch.from_tables`."""

    def __init__(self):
        self.B = 0
        self.n_slots = 20           # T: reference slot count (dense view, max-negative loss)
        self.n_ctx_slots = 18       # S: reference context rows per candidate (dense view)
        self.n_classes = 101
        self.has_ctx = True
        self.clip_bank = None       # bf16 [n_clip, 2816]
        self.track_bank = None      # bf16 [n_track, 2048]
        self.n_clip_ints = 0
        self.n_track_ints = 0
        self.multilab = None        # uint8 [B, C]
        self.soft_pos = None        # uint8 [B, C] multi-hot of the soft labels (--soft_gt), else None
        self.tables = {}            # name -> int32 array/tensor
        self.extras = {}            # pass-through keys (just_zeros, n_names, hash_rel, soft_labels ...)
        self.device = None

    # ---- sizes -----------------------------------------------------------------------------
    @property
    def n_cand(self):
        n = self.__dict__.get("_n_cand")
        return int(self.tables["cand_rows"].shape[0]) if n is None else n

    @property
    def n_ctx_rows(self):
        if not self.has_ctx:
            return 0
        n = self.__dict__.get("_n_ctx_rows")
        return int(self.tables["ctx_rows"].shape[0]) if n is None else n

    @property
    def n_clip(self):
        return int(self.clip_bank.shape[0])

    @property
    def n_track(self):
        return int(self.track_bank.shape[0])

    def __getitem__(self, k):
        return self.tables[k]

    def table_ptr(self, k):
        """Device address of integer table `k` (device batches only) without building a tensor view."""
        t = self.tables
        if isinstance(t, _DeviceTables):
            return t._arena.data_ptr() + 4 * t._layout[k][0]
        return t[k].data_ptr()

    # ---- construction ----------------------------------------------------------------------
    @staticmethod
    def from_tables(clip_bank, track_bank, n_clip_ints, n_track_ints, cand_off, cand_rows, ctx_off, ctx_rows,
                    labels, rels_label, gt_tracks, multilab, n_slots=20, n_ctx_slots=18, extras=None):
        """All arguments are host arrays. clip_bank/track_bank: float arrays (rounded to bf16 here) or
        bf16 torch tensors. ctx_off/ctx_rows may be None (no context branch)."""
        pb = PackedBatch()
        pb.B = int(len(cand_off) - 1)
        pb.n_slots, pb.n_ctx_slots = int(n_slots), int(n_ctx_slots)
        pb.clip_bank = _as_bf16(clip_bank)
        pb.track_bank = _as_bf16(track_bank)
        pb.n_clip_ints, pb.n_track_ints = int(n_clip_ints), int(n_track_ints)
        pb.multilab = torch.as_tensor(np.ascontiguousarray(np.asarray(multilab) != 0).astype(np.uint8))
        pb.n_classes = int(pb.multilab.shape[1])
        t = pb.tables
        t["cand_off"] = np.asarray(cand_off, dtype=np.int32)
        t["cand_rows"] = np.ascontiguousarray(np.asarray(cand_rows, dtype=np.int32).reshape(-1, 3))
        Ni = t["cand_rows"].shape[0]
        assert t["cand_off"][-1] == Ni and t["cand_off"][0] == 0
        counts = np.diff(t["cand_off"])
        assert (counts >= 1).all() and (counts <= n_slots).all(), "every clip needs 1..n_slots candidates"
        t["cand_clip"] = np.repeat(np.arange(pb.B, dtype=np.int32), counts)
        t["cand_slot"] = (np.arange(Ni, dtype=np.int32) - np.repeat(t["cand_off"][:-1], counts)).astype(np.int32)
        t["labels"] = np.asarray(labels, dtype=np.int32).reshape(pb.B)
        t["gt_tracks"] = np.ascontiguousarray(np.asarray(gt_tracks, dtype=np.int32).reshape(pb.B, 2))
        pb.has_ctx = ctx_off is not None
        if pb.has_ctx:
            t["ctx_off"] = np.asarray(ctx_off, dtype=np.int32)
            t["ctx_rows"] = np.ascontiguousarray(np.asarray(ctx_rows, dtype=np.int32).reshape(-1, 3))
            Nx = t["ctx_rows"].shape[0]
            assert t["ctx_off"].shape[0] == Ni + 1 and t["ctx_off"][-1] == Nx
            t["ctx_owner"] = np.repeat(np.arange(Ni, dtype=np.int32), np.diff(t["ctx_off"]))
            t["rels_label"] = np.asarray(rels_label, dtype=np.int32).reshape(Ni)
            assert Nx == 0 or (t["ctx_rows"][:, 0].max() < pb.n_clip and t["ctx_rows"][:, 1:].max() < pb.n_track)
        elif rels_label is not None:
            t["rels_label"] = np.asarray(rels_label, dtype=np.int32).reshape(Ni)
        assert t["cand_rows"][:, 0].max() < pb.n_clip_ints and t["cand_rows"][:, 1:].max() < pb.n_track_ints, \
            "candidate rows must reference the ints prefix of the banks"
        assert t["cand_rows"].min() >= 0
        # inverse CSRs for backward: slot 0 = clip column, 1 = track1, 2 = track2
        for s in range(3):
            t["inv_cand_off%d" % s], t["inv_cand_idx%d" % s] = _csr_inverse(
                t["cand_rows"][:, s], pb.n_clip_ints if s == 0 else pb.n_track_ints)
            if pb.has_ctx:
                t["inv_ctx_off%d" % s], t["inv_ctx_idx%d" % s] = _csr_inverse(
                    t["ctx_rows"][:, s], pb.n_clip if s == 0 else pb.n_track)
        pb.extras = dict(extras or {})
        return pb

    @staticmethod
    def from_arena(arena, layout, clip_bank, track_bank, n_clip_ints, n_track_ints, B, Ni, Nx, labels, rels_label,
                   gt_tracks, multilab, n_slots=20, n_ctx_slots=18, extras=None, src_layout=None):
        """A host batch whose integer tables already lie in one int32 arena in `_INT_TABLES` order
        (`lirec_collate_tables`, csrc/collate.cu): `layout[i] = (offset, length)` of table i, length -1 =
        absent.  The tables are views into the arena, so `pin()` is a single copy.  Nx is None without a
        context branch.  labels / rels_label / gt_tracks are written into their reserved slots here."""
        pb = PackedBatch()
        pb.B, pb.n_slots, pb.n_ctx_slots = int(B), int(n_slots), int(n_ctx_slots)
        pb.clip_bank, pb.track_bank = _as_bf16(clip_bank), _as_bf16(track_bank)
        pb.n_clip_ints, pb.n_track_ints = int(n_clip_ints), int(n_track_ints)
        pb.multilab = torch.as_tensor(np.ascontiguousarray(np.asarray(multilab) != 0).astype(np.uint8))
        pb.n_classes = int(pb.multilab.shape[1])
        pb.has_ctx = Nx is not None
        shapes = {"cand_rows": (Ni, 3), "ctx_rows": (Nx, 3), "gt_tracks": (B, 2)}
        end = 0
        host_layout = {}
        for k, (off, n) in zip(_INT_TABLES, np.asarray(layout).tolist()):
            if n < 0:
                continue
            assert off == end, "arena tables must be contiguous in _INT_TABLES order"
            shape = shapes.get(k, (n,))
            pb.tables[k] = arena[off:off + n].reshape(shape)
            host_layout[k] = (off, n, shape)
            end = off + n
        t = pb.tables
        t["labels"][:] = np.asarray(labels).reshape(B)
        t["gt_tracks"][:] = np.asarray(gt_tracks).reshape(B, 2)
        if pb.has_ctx:
            t["rels_label"][:] = np.asarray(rels_label).reshape(Ni)
        if src_layout is not None:                 # (clip offset, n, track offset, n): the dataset-bank row lists
            assert src_layout[0] >= end and src_layout[2] >= src_layout[0] + src_layout[1]
            end = src_layout[2] + src_layout[3]
            pb._src_layout = tuple(int(v) for v in src_layout)
        pb._host_arena, pb._host_layout = arena[:end], host_layout
        pb.extras = dict(extras or {})
        return pb

    # A natively collated batch crosses the DataLoader worker -> main process pipe as its arena alone: the
    # table views are rebuilt on arrival (pickling them would ship every table twice).
    # The arena (and the resident-bank row lists) travel as torch tensors: torch.multiprocessing moves tensor
    # storage into shared memory in the worker and the main process maps it, so the ~2 MB of a 1024-clip
    # batch are not copied through the pipe and un-pickled on the training process's critical path.
    def __getstate__(self):
        st = dict(self.__dict__)
        if st.get("_host_arena") is not None and st.get("device") is None:
            st["tables"] = None
            st.pop("_arena", None)
            st.pop("_bank_rows_pinned", None)
            st["_host_arena"] = torch.from_numpy(st["_host_arena"])
            rows = st.get("extras", {}).get("bank_rows")
            if rows is not None:
                st["extras"] = dict(st["extras"])
                if st.get("_src_layout") is not None:      # views of the arena: rebuilt on arrival
                    st["extras"]["bank_rows"] = None
                else:
                    st["extras"]["bank_rows"] = tuple(torch.from_numpy(np.ascontiguousarray(r)) for r in rows)
        return st

    def __setstate__(self, st):
        self.__dict__.update(st)
        if isinstance(self.__dict__.get("_host_arena"), torch.Tensor):
            self._host_arena = self._host_arena.numpy()
        rows = self.extras.get("bank_rows") if isinstance(self.extras, dict) else None
        if rows is not None and isinstance(rows[0], torch.Tensor):
            self.extras["bank_rows"] = tuple(r.numpy() for r in rows)
        src = self.__dict__.get("_src_layout")
        if src is not None and isinstance(self.extras, dict) and self.extras.get("bank_rows", 0) is None:
            a = self._host_arena
            self.extras["bank_rows"] = (a[src[0]:src[0] + src[1]], a[src[2]:src[2] + src[3]])
        if self.tables is None:
            self.tables = {k: self._host_arena[off:off + n].reshape(shape)
                           for k, (off, n, shape) in self._host_layout.items()}

    # ---- device staging --------------------------------------------------------------------
    def h2d_bytes(self):
        n = self.clip_bank.numel() * 2 + self.track_bank.numel() * 2 + self.multilab.numel()
        if self.soft_pos is not None:
            n += self.soft_pos.numel()
        for v in self.tables.values():
            n += v.size * 4
        return int(n)

    def pin_memory(self):
        """torch.utils.data.DataLoader(pin_memory=True) calls this on its pinning thread."""
        return self.pin()

    def _pin_bank_rows(self):
        rows = self.extras.get("bank_rows")
        if getattr(self, "_src_layout", None) is not None:
            return                                  # the row lists are part of the (pinned) arena
        if rows is not None and not hasattr(self, "_bank_rows_pinned"):
            self._bank_rows_pinned = tuple(torch.from_numpy(np.ascontiguousarray(r)).pin_memory() for r in rows)

    def pin(self):
        """Move the host copy into pinned memory (one int32 arena + the two banks + multilab)."""
        assert self.device is None
        if hasattr(self, "_arena"):
            return self
        if getattr(self, "_host_arena", None) is not None and not hasattr(self, "_arena"):
            self._arena = torch.from_numpy(self._host_arena).pin_memory()        # one copy: tables are arena views
            self._layout = self._host_layout
            self.clip_bank = self.clip_bank.pin_memory()
            self.track_bank = self.track_bank.pin_memory()
            self.multilab = self.multilab.pin_memory()
            if self.soft_pos is not None:
                self.soft_pos = self.soft_pos.pin_memory()
            self._pin_bank_rows()
            return self
        names = [k for k in _INT_TABLES if k in self.tables]
        sizes = [int(self.tables[k].size) for k in names]
        arena = torch.empty(sum(sizes), dtype=torch.int32).pin_memory()
        off = 0
        layout = {}
        for k, n in zip(names, sizes):
            arena[off:off + n] = torch.from_numpy(self.tables[k].reshape(-1))
            layout[k] = (off, n, self.tables[k].shape)
            off += n
        self._arena, self._layout = arena, layout
        self.clip_bank = self.clip_bank.pin_memory()
        self.track_bank = self.track_bank.pin_memory()
        self.multilab = self.multilab.pin_memory()
        if self.soft_pos is not None:
            self.soft_pos = self.soft_pos.pin_memory()
        self._pin_bank_rows()
        return self

    def to_device(self, device="cuda", non_blocking=True, banks=True):
        """Copy to the GPU: 4 async copies (int arena, clip bank, track bank, multilab).  With
        banks=False the two feature banks are left for the caller to provide on the device
        (mixed_utils/indexed_dataset.py:ResidentBanks gathers them from HBM-resident dataset banks)."""
        if not hasattr(self, "_arena"):
            self.pin()
        d = PackedBatch()
        for k in ("B", "n_slots", "n_ctx_slots", "n_classes", "has_ctx", "n_clip_ints", "n_track_ints", "extras"):
            setattr(d, k, getattr(self, k))
        d.device = torch.device(device)
        arena = self._arena.to(device, non_blocking=non_blocking)
        if banks:
            d.clip_bank = self.clip_bank.to(device, non_blocking=non_blocking)
            d.track_bank = self.track_bank.to(device, non_blocking=non_blocking)
        d.multilab = self.multilab.to(device, non_blocking=non_blocking)
        if self.soft_pos is not None:
            d.soft_pos = self.soft_pos.to(device, non_blocking=non_blocking)
        d.tables = _DeviceTables(arena, self._layout)
        d._n_cand = int(self._layout["cand_rows"][2][0])
        if self.has_ctx:
            d._n_ctx_rows = int(self._layout["ctx_rows"][2][0])
        d._arena_dev = arena
        d.host = self
        return d

    def without_banks(self, clip_rows, track_rows):
        """Host copy that shares the integer tables but carries no feature banks: `clip_rows` /
        `track_rows` name the rows of HBM-resident dataset banks to gather on the device instead
        (mixed_utils/indexed_dataset.py:ResidentBanks.stage)."""
        assert self.device is None
        d = PackedBatch()
        for k in ("B", "n_slots", "n_ctx_slots", "n_classes", "has_ctx", "n_clip_ints", "n_track_ints", "multilab",
                  "soft_pos", "tables"):
            setattr(d, k, getattr(self, k))
        d.extras = dict(self.extras)
        if getattr(self, "_host_arena", None) is not None:
            d._host_arena, d._host_layout = self._host_arena, self._host_layout
        d.clip_bank = torch.empty((self.n_clip, 0), dtype=torch.bfloat16)
        d.track_bank = torch.empty((self.n_track, 0), dtype=torch.bfloat16)
        d.extras["bank_rows"] = (np.ascontiguousarray(clip_rows, dtype=np.int32),
                                 np.ascontiguousarray(track_rows, dtype=np.int32))
        return d

    def record_stream(self, stream):
        """Tell the caching allocator that `stream` uses this batch's device tensors (they may have been
        allocated on a copy stream)."""
        for t in (self._arena_dev, self.clip_bank, self.track_bank, self.multilab) + tuple(getattr(self, "_bank_idx", ())):
            t.record_stream(stream)
        if self.soft_pos is not None:
            self.soft_pos.record_stream(stream)
        return self

    # ---- dense (reference-format) view -------------------------------------------------------
    def to_dense(self, dtype=np.float64):
        """The batch as the reference dataloader + default collate would emit it (host only)."""
        assert self.device is None
        t = self.tables
        B, T, S, C = self.B, self.n_slots, self.n_ctx_slots, self.n_classes
        clip = self.clip_bank.float().numpy().astype(dtype)
        track = self.track_bank.float().numpy().astype(dtype)

        def rows_of(tbl):
            return np.hstack((clip[tbl[:, 0]], track[tbl[:, 1]], track[tbl[:, 2]]))

        cand = rows_of(t["cand_rows"])
        ROW_DIM = cand.shape[1]
        b_idx, s_idx = t["cand_clip"], t["cand_slot"]
        out = {}
        mem_mask = np.zeros((B, T), dtype=np.float64)
        mem_mask[b_idx, s_idx] = 1
        if self.has_ctx:
            feats = np.zeros((B, T, S + 1, ROW_DIM), dtype=dtype)
            feats[b_idx, s_idx, 0] = cand
            rels_mask = np.zeros((B, T, S), dtype=np.int64)
            if self.n_ctx_rows:
                ctx = rows_of(t["ctx_rows"])
                owner = t["ctx_owner"]
                j = np.arange(self.n_ctx_rows) - t["ctx_off"][:-1][owner]
                feats[b_idx[owner], s_idx[owner], 1 + j] = ctx
                rels_mask[b_idx[owner], s_idx[owner], j] = 1
            rels_label = np.zeros((B, T), dtype=np.int64)      # pad label 0: dataloader :430
            rels_label[b_idx, s_idx] = t["rels_label"]
            out["rels_mask"] = torch.from_numpy(rels_mask)
            out["rels_label"] = torch.from_numpy(rels_label)
        else:
            feats = np.zeros((B, T, ROW_DIM), dtype=dtype)
            feats[b_idx, s_idx] = cand
        out["features"] = torch.from_numpy(feats)
        out["mem_mask"] = torch.from_numpy(mem_mask)
        out["labels"] = torch.from_numpy(t["labels"].astype(np.int64))
        out["gt_tracks"] = torch.from_numpy(t["gt_tracks"].astype(np.int64))
        out["multilab_weights"] = self.multilab.to(torch.float64)
        for k, v in self.extras.items():
            out[k] = v
        return out


def _as_bf16(x):
    if isinstance(x, torch.Tensor):
        return x.to(torch.bfloat16).contiguous()
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(torch.bfloat16)


def pack_dense_batch(batch, kind, n_slots=None):
    """Compatibility path: pack a reference-format DENSE batch dict (no deduplication — every valid
    row becomes its own bank rows).  kind: 'modalities' | 'midfusion' | 'maxtracks'.

    modalities: features [B,1,D], labels [B]
    midfusion : features [B,S+1,D], rels_mask [B,S,1], labels [B,S+1,1], rels_label [B]
    maxtracks : features [B,T,(S+1),D] or [B,T,D], mem_mask [B,T], rels_mask [B,T,S], rels_label [B,T]
    """
    f = batch["features"]
    f = f.numpy() if isinstance(f, torch.Tensor) else np.asarray(f)
    B = f.shape[0]

    def _np(k):
        v = batch[k]
        return v.numpy() if isinstance(v, torch.Tensor) else np.asarray(v)

    if kind == "modalities":
        rows = f[:, 0, :]
        counts = np.ones(B, dtype=np.int64)
        ctx = None
        T, S = 1, 0
        labels = _np("labels").reshape(B)
        rels_label = None
        gt_tracks = np.zeros((B, 2), dtype=np.int64)
    elif kind == "midfusion":
        rows = f[:, 0, :]
        counts = np.ones(B, dtype=np.int64)
        S = f.shape[1] - 1
        T = 1
        m = _np("rels_mask").reshape(B, S) != 0
        ctx = (f[:, 1:, :], m)
        labels = _np("labels").reshape(B, -1)[:, 0]
        rels_label = _np("rels_label").reshape(B)
        gt_tracks = np.zeros((B, 2), dtype=np.int64)
    else:
        T = f.shape[1]
        mem = _np("mem_mask").reshape(B, T) != 0
        counts = mem.sum(1)
        assert all(mem[b, :counts[b]].all() for b in range(B)), "valid candidate slots must be a prefix"
        if f.ndim == 4:
            S = f.shape[2] - 1
            rows = f[:, :, 0, :][mem]
            m = (_np("rels_mask").reshape(B, T, S) != 0)[mem]
            ctx = (f[:, :, 1:, :][mem], m)
            rels_label = _np("rels_label").reshape(B, T)[mem]
        else:
            S = 0
            rows = f[mem]
            ctx = None
            rels_label = None
        labels = _np("labels").reshape(B)
        gt_tracks = _np("gt_tracks").reshape(B, 2)
    Ni = rows.shape[0]
    cand_off = np.zeros(B + 1, dtype=np.int64)
    np.cumsum(counts, out=cand_off[1:])
    clip_rows = [rows[:, :CLIP_DIM]]
    tr_rows = [rows[:, CLIP_DIM:CLIP_DIM + TRACK_DIM], rows[:, CLIP_DIM + TRACK_DIM:]]
    ar = np.arange(Ni)
    cand_tbl = np.stack((ar, ar, Ni + ar), axis=1)
    n_clip_ints, n_track_ints = Ni, 2 * Ni
    ctx_off = ctx_tbl = None
    if ctx is not None:
        cf, cm = ctx
        assert all(cm[i, :cm[i].sum()].all() for i in range(Ni)), "valid context rows must be a prefix"
        ccounts = cm.sum(1)
        ctx_off = np.zeros(Ni + 1, dtype=np.int64)
        np.cumsum(ccounts, out=ctx_off[1:])
        cr = cf[cm]
        Nx = cr.shape[0]
        ax = np.arange(Nx)
        clip_rows.append(cr[:, :CLIP_DIM])
        tr_rows += [cr[:, CLIP_DIM:CLIP_DIM + TRACK_DIM], cr[:, CLIP_DIM + TRACK_DIM:]]
        ctx_tbl = np.stack((Ni + ax, 2 * Ni + ax, 2 * Ni + Nx + ax), axis=1)
    mw = batch.get("multilab_weights")
    if mw is None:
        mw = np.ones((B, int(batch.get("n_classes", 101))))
    mw = mw.numpy() if isinstance(mw, torch.Tensor) else np.asarray(mw)
    extras = {k: batch[k] for k in ("just_zeros", "n_names", "hash_rel", "soft_labels") if k in batch}
    pb = PackedBatch.from_tables(np.vstack(clip_rows), np.vstack(tr_rows), n_clip_ints, n_track_ints,
                                 cand_off, cand_tbl, ctx_off, ctx_tbl, labels, rels_label, gt_tracks, mw,
                                 n_slots=n_slots or T, n_ctx_slots=S, extras=extras)
    if "soft_labels" in batch:
        sl = batch["soft_labels"]
        pb.soft_pos = soft_pos_of(sl.numpy() if isinstance(sl, torch.Tensor) else sl, pb.n_classes)
    return pb


def soft_pos_of(soft_labels, n_classes):
    """uint8 [B, C] multi-hot of the soft-label class ids [B, K] (the dataset's `soft_labels`: the clip's label
    and the interactions that co-occur with it in time, padded with -1) — the extra positives of the BCE losses."""
    sl = np.asarray(soft_labels).reshape(len(soft_labels), -1).astype(np.int64)
    out = np.zeros((sl.shape[0], int(n_classes)), dtype=np.uint8)
    rows, cols = np.nonzero(sl >= 0)
    out[rows, sl[rows, cols]] = 1
    return torch.from_numpy(out)
