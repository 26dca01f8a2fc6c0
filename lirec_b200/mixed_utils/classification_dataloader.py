"""Dataset + packed dataloader (reference: mixed_utils/classification_dataloader.py).

The reference's `MixedFeaturesDataset.__getitem__` (:291-616) builds a dense zero-padded
float64 `[20, 19, 6912]` block per clip (21 MB, mostly np.tile copies) and torch's default collate
stacks them — 1.34 GB per 64-clip batch through worker IPC.  Here an item is a small clip RECORD
(its own pooled vectors plus index triples in the reference's slot order) and the collate function
packs records into one PackedBatch whose tables live in pinned memory; `packed_loader` copies batch
i+1 to the GPU on a side stream while batch i computes.

The MovieGraphs annotations / feature dump (~80 GB) are not available offline, and their parsing
(utils/util_functions.py, moviegraphs/py3loader) is outside the hot path (SURVEY.md §2 rows 12, 15):
without `opt.synthetic` the dataset refuses to construct instead of pretending.

  --synthetic 1   independent synthetic clips (mixed_utils/synthetic.py; the bench workload)
  --synthetic 3   the same independent clips with their vectors cached once in dataset-level banks and index-only
                  items (mixed_utils/cached_clips.py) — the reference's cache() + __getitem__ split; what
                  bench.py's end-to-end leg iterates
  --synthetic 2   a synthetic ANNOTATION world (mixed_utils/synthetic_world.py) run through the index-only
                  port of the reference dataset logic (mixed_utils/indexed_dataset.py: relationship
                  timelines, shared context clips, the reference's slot order and RNG use), the path real
                  MovieGraphs annotations would take; `--resident_banks 1` keeps the split's pooled feature
                  banks in HBM so a batch ships only index tables.
"""
import torch
from torch.utils.data import Dataset

from lirec_b200.mixed_utils import synthetic
from lirec_b200.utils.arg_pars import opt


def preset_from_opt():
    if opt.mod_check:
        return "modalities"
    if opt.tr_maximize:
        return "int_rel_ch" if (opt.ctx == 1 and opt.rels_multitask) else "int_ch"
    return "int_rels"


def MixedFeaturesDataset(mode="train", size=None):
    """Reference constructor signature (classification_dataloader.py:30); dispatches on opt.synthetic."""
    if int(getattr(opt, "synthetic", 0)) == 3:
        from lirec_b200.mixed_utils.cached_clips import CachedClipsDataset
        return CachedClipsDataset(mode, size)
    if int(getattr(opt, "synthetic", 0)) == 2:
        from lirec_b200.mixed_utils import indexed_dataset, synthetic_world
        world = synthetic_world.build_world(int(opt.seed), n_movies=int(getattr(opt, "world_movies", 6)),
                                            n_scenes=int(getattr(opt, "world_scenes", 40)), n_inter_names=324,
                                            n_merged=synthetic.N_CLASSES)
        return indexed_dataset.IndexedMixedFeaturesDataset(synthetic_world.subset(world, mode), world, mode=mode)
    return SyntheticClipsDataset(mode, size)


class SyntheticClipsDataset(Dataset):
    """Same constructor and attributes the loops use (`n_classes`, `n_rels`, `rels_list`, `cache()`,
    `init_relships()`, `epoch`), backed by the synthetic MovieGraphs-shaped generator."""
    SIZES = {"train": 4096, "val": 512, "test": 512}

    def __init__(self, mode="train", size=None):
        if not getattr(opt, "synthetic", 0):
            raise RuntimeError(
                "MixedFeaturesDataset needs the MovieGraphs feature dump and annotations (README.md:18-28 of "
                "the reference), which are not available offline; run with --synthetic 1 for the synthetic "
                "MovieGraphs-shaped dataset")
        self.mode = mode
        self.n_classes = synthetic.N_CLASSES
        self.rels_list = ["rel%02d" % i for i in range(synthetic.N_RELS)] + ["None"]
        self.n_rels = len(self.rels_list)
        self.interidx2mgdidx = list(range(self.n_classes))
        self._max_n_tripl = int(getattr(opt, "max_n_tripl", 20))
        self.rels_n_clips = opt.rels_n_clips if opt.rels_multi_clip else 18
        self.epoch = 0
        self._size = int(size or self.SIZES.get(mode, 512))
        self._base = {"train": 0, "val": 1, "test": 2}.get(mode, 3) * 10_000_019 + int(opt.seed) * 7919
        self.preset = preset_from_opt()

    def cache(self):
        """The reference precomputes pooled features here (:139-186); synthetic clips are generated on
        demand by the dataloader workers."""
        return self

    def init_relships(self):
        assert self.rels_list[-1] == "None"
        return self

    def __len__(self):
        return self._size

    def __getitem__(self, idx):
        return synthetic.make_clip(self._base + int(idx), preset=self.preset, max_n_tripl=self._max_n_tripl,
                                   rels_n_clips=self.rels_n_clips)

    def collate(self, records):
        return collate_packed(records)


def collate_packed(records):
    """records -> pinned host PackedBatch (runs in the dataloader worker / main process)."""
    return synthetic.pack_clips(records)


class EmptyShard:
    """A rank's share of a global batch that has fewer clips than ranks (the last batch of an epoch, e.g. 37
    clips, batch 8, 8 ranks: 5 clips left).  The rank has no rows to compute on but MUST still take part in the
    step's collectives — the loops zero its gradient and call the exchange with local_clips = 0 — otherwise
    the other ranks' gradient reduction pairs up with this rank's NEXT collective (hang or corruption)."""
    B = 0
    device = None

    def __init__(self, global_clips):
        self.global_clips = int(global_clips)
        self.host = self

    def pin(self):
        return self

    pin_memory = pin

    def record_stream(self, stream):
        return self


class _PinnedRing:
    """A fixed ring of pinned staging buffers for index-only batches: the worker's arena (shared memory) and the
    multi-label bytes are copied into the next slot and cross PCIe from there.  No pinned allocation happens per
    batch — the caching host allocator only recycles a block once the events of its last use have completed and
    falls back to cudaHostAlloc (milliseconds, under the driver lock every kernel launch needs) otherwise, which
    showed as erratic multi-millisecond stalls of the loader.  A slot is reused after its own H2D copies are done."""

    def __init__(self, slots=6):
        self.arena, self.ml, self.ev = [None] * slots, [None] * slots, [None] * slots
        self.k = 0

    def stage(self, pb, copy_stream):
        """Point `pb` (a host PackedBatch with `_host_arena`) at pinned copies of its arena / multilab (/ soft_pos)."""
        k = self.k
        self.k = (k + 1) % len(self.arena)
        if self.ev[k] is not None:
            self.ev[k].synchronize()                         # the slot's previous batch has crossed PCIe
        src = torch.from_numpy(pb._host_arena)
        sp = pb.soft_pos                                     # --soft_gt: staged behind multilab in the same buffer
        n, m = src.numel(), pb.multilab.numel()
        ms = m + (sp.numel() if sp is not None else 0)
        if self.arena[k] is None or self.arena[k].numel() < n:
            self.arena[k] = torch.empty(int(n * 1.25) + 1024, dtype=torch.int32).pin_memory()
        if self.ml[k] is None or self.ml[k].numel() < ms:
            self.ml[k] = torch.empty(int(ms * 1.25) + 1024, dtype=torch.uint8).pin_memory()
        self.arena[k][:n].copy_(src)
        self.ml[k][:m].copy_(pb.multilab.reshape(-1))
        pb._arena, pb._layout = self.arena[k][:n], pb._host_layout
        pb.multilab = self.ml[k][:m].view(pb.multilab.shape)
        if sp is not None:
            self.ml[k][m:ms].copy_(sp.reshape(-1))
            pb.soft_pos = self.ml[k][m:ms].view(sp.shape)
        self._last = k
        return pb

    def mark(self, copy_stream):
        ev = torch.cuda.Event()
        ev.record(copy_stream)
        self.ev[self._last] = ev


def plan_batches(n, batch_size, order, rank, world, drop_last=False):
    """[(this rank's clip indices, global batch size)] for one epoch.  EVERY rank gets one entry per global
    batch — an empty index list when the global batch is smaller than the world — so all ranks take the same
    number of steps and their collectives stay paired."""
    from lirec_b200 import dp
    batches = []
    for s in range(0, n, batch_size):
        idx = order[s:s + batch_size]
        if drop_last and len(idx) < batch_size:
            break
        a, b = dp.shard_range(len(idx), rank, world)
        batches.append((idx[a:b], len(idx)))
    return batches


def _threaded_batches(dataset, batches, num_threads, batch_size, slots_ahead):
    """Host batches of a dataset with a thread-safe `get_batch`, built by `num_threads` THREADS straight into a ring
    of pinned slots.  The assembly is native code that releases the GIL (lirec_collate_gather,
    lirec_collate_tables), so threads scale like the reference's DataLoader worker processes (mlp/train.py:33-37)
    do — without the per-batch shared-memory segment, pickling, pinning copy and their erratic multi-millisecond
    stalls.  Yields (host batch, release) in order; `release(cuda_event)` hands the slot back once the batch's H2D
    copies are recorded."""
    import threading
    from concurrent.futures import ThreadPoolExecutor
    n_slots = slots_ahead + 2
    cap = dataset.arena_bound(max(len(b[0]) for b in batches if b[0]) if any(b[0] for b in batches) else 1)
    ml_cap = batch_size * dataset.n_classes + 64
    arenas = [torch.empty(cap, dtype=torch.int32).pin_memory() for _ in range(n_slots)]
    mls = [torch.empty(ml_cap, dtype=torch.uint8).pin_memory() for _ in range(n_slots)]
    free = [threading.Event() for _ in range(n_slots)]
    last_ev = [None] * n_slots
    for f in free:
        f.set()

    def job(k):
        idx, global_size = batches[k]
        if not idx:
            return EmptyShard(global_size)
        s = k % n_slots
        free[s].wait()
        free[s].clear()
        if last_ev[s] is not None:
            last_ev[s].synchronize()                        # the slot's previous batch has crossed PCIe
        pb = dataset.get_batch(idx, arena_out=arenas[s], multilab_out=mls[s])
        pb.global_clips = global_size
        return pb

    def releaser(k):
        def release(ev):
            s = k % n_slots
            last_ev[s] = ev
            free[s].set()
        return release

    pool = ThreadPoolExecutor(max_workers=num_threads, thread_name_prefix="lirec-collate")
    try:
        futures = {}
        nxt = 0
        for k in range(len(batches)):
            while nxt < len(batches) and nxt < k + slots_ahead:
                futures[nxt] = pool.submit(job, nxt)
                nxt += 1
            pb = futures.pop(k).result()
            yield pb, (releaser(k) if not isinstance(pb, EmptyShard) else (lambda ev: None))
    finally:
        # the consumer stopped early (or we are done): nobody will release slots any more — let the queued jobs
        # through instead of leaving the pool's threads blocked on them
        for f in free:
            f.set()
        last_ev[:] = [None] * n_slots
        pool.shutdown(wait=True, cancel_futures=True)


def packed_loader(dataset, batch_size, shuffle, num_workers=0, device="cuda", rank=0, world=1, drop_last=False,
                  seed=0, repeat=1):
    """Iterate device-resident PackedBatches with one-batch-ahead async H2D prefetch.

    Data parallel: every rank iterates the same shuffled order and takes its contiguous share of each
    global batch (lirec_b200/dp.py:shard_range), so the global batch equals the single-GPU one.  A rank whose
    share is empty receives an `EmptyShard` for that step (see there).  `repeat` > 1 chains that many epochs
    (each its own permutation) behind ONE set of worker processes instead of re-forking them per epoch."""
    g = torch.Generator()
    g.manual_seed(int(seed) * 1000003 + int(getattr(dataset, "epoch", 0)))
    n = len(dataset)
    batches = []
    for _ in range(max(1, int(repeat))):
        order = torch.randperm(n, generator=g).tolist() if shuffle else list(range(n))
        batches += plan_batches(n, batch_size, order, rank, world, drop_last)
    if int(num_workers) > 0 and hasattr(dataset, "warm_records"):
        dataset.warm_records()              # workers fork with the record cache already built
    # worker processes build the batches (items + native collate)
    group = max(1, min(16, 512 // max(int(batch_size) // max(world, 1), 1))) if int(num_workers) > 0 else 1
    loader = torch.utils.data.DataLoader(_IndexView(dataset, batches, group), batch_size=None, shuffle=False,
                                         num_workers=int(num_workers), collate_fn=None,
                                         pin_memory=False,
                                         prefetch_factor=(int(getattr(opt, "prefetch_factor", 2)) if int(num_workers) > 0
                                                          else None),
                                         persistent_workers=False)
    copy_stream = torch.cuda.Stream(device=device)
    pending = None
    banks = None
    if int(getattr(opt, "resident_banks", 0)) and hasattr(dataset, "clip_bank"):
        from lirec_b200.mixed_utils.indexed_dataset import ResidentBanks
        banks = getattr(dataset, "_resident", None) or ResidentBanks(dataset, device)
        dataset._resident = banks
        copy_stream.wait_stream(torch.cuda.current_stream())
    ring = _PinnedRing() if banks is not None else None

    def flat(it):
        for item in it:
            if isinstance(item, list):
                for x in item:
                    yield x, None
            else:
                yield item, None

    # datasets whose batches are assembled by GIL-free native code (get_batch): worker THREADS, pinned from birth
    threaded = (int(num_workers) > 0 and banks is not None and hasattr(dataset, "get_batch") and
                hasattr(dataset, "arena_bound"))
    if threaded:
        if getattr(dataset, "records", 1) is None:
            dataset.cache()
        source = _threaded_batches(dataset, batches, int(num_workers), batch_size, slots_ahead=2 * int(num_workers) + 2)
    else:
        source = flat(loader)
    for host_pb, release in source:
        if isinstance(host_pb, EmptyShard):
            dev_pb, ev = host_pb, None
            if pending is not None:
                prev, pev = pending
                if pev is not None:
                    torch.cuda.current_stream().wait_event(pev)
                yield prev.record_stream(torch.cuda.current_stream())
            pending = (dev_pb, ev)
            continue
        with torch.cuda.stream(copy_stream):
            if ring is not None and getattr(host_pb, "_host_arena", None) is not None and not hasattr(host_pb, "_arena"):
                dev_pb = banks.stage(ring.stage(host_pb, copy_stream))
                ring.mark(copy_stream)
            else:
                dev_pb = banks.stage(host_pb) if banks is not None else host_pb.pin().to_device(device, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
            if release is not None:
                release(ev)
        if pending is not None:
            prev, pev = pending
            if pev is not None:
                torch.cuda.current_stream().wait_event(pev)
            yield prev.record_stream(torch.cuda.current_stream())
        pending = (dev_pb, ev)
    if pending is not None:
        prev, pev = pending
        if pev is not None:
            torch.cuda.current_stream().wait_event(pev)
        yield prev.record_stream(torch.cuda.current_stream())


class _IndexView(Dataset):
    """One item = `group` consecutive packed (per-rank) batches, so workers do the packing too and the
    DataLoader's per-item hand-over (queue, un-pickling, pinning thread: ~1 ms) is paid once per group —
    at the reference's 64-clip batches a device step is half of that."""

    def __init__(self, dataset, batches, group=1):
        self.dataset, self.batches, self.group = dataset, batches, max(1, int(group))

    def __len__(self):
        return (len(self.batches) + self.group - 1) // self.group

    def one(self, k):
        idx, global_size = self.batches[k]
        if not idx:
            return EmptyShard(global_size)
        fetch = getattr(self.dataset, "get_batch", None)          # items + collate fused (dataset-level tables)
        pb = fetch(idx) if fetch is not None else self.dataset.collate([self.dataset[j] for j in idx])
        pb.global_clips = global_size
        return pb

    def __getitem__(self, i):
        if self.group == 1:
            return self.one(i)
        return [self.one(k) for k in range(i * self.group, min((i + 1) * self.group, len(self.batches)))]


def f_dataloader(mode="train"):
    """Reference: classification_dataloader.py:623-630."""
    print("load mixed features. mode: %s" % mode)
    dataset = MixedFeaturesDataset(mode)
    loader = packed_loader(dataset, opt.batch_size, shuffle=(mode == "train"), num_workers=opt.num_workers)
    return loader, dataset.n_classes
