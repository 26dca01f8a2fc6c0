"""Index-only dataset: the reference's `MixedFeaturesDataset` (mixed_utils/classification_dataloader.py
:29-630) with every 6912-d row kept as an index TRIPLE into two feature banks instead of a
materialised float64 vector.

The reference keys its cached pooled vectors by interaction id (clip text|visual,
mixed_features.py:37-67) and by (interaction id, character name) (person track, :84-112); a context
matrix is `np.hstack((clipf, track1, track2))` of such cached vectors for a list of
`[inter_id, (inter_id, name1), (inter_id, name2)]` entries (:115-125, dataloader :188-262) and an
item is 20 x 19 of those rows, mostly `np.tile` copies (:291-573).  Here

    clip bank   row i                    = pooled clip vector of interaction i; the last row is all zero
    track bank  row 0                    = the all-zero "no track" vector
                row tr[(i, name)] (>= 1) = pooled track of `name` in interaction i (0 if it is all zero)

live once per split (on the host, and — `ResidentBanks` — in HBM), contexts are int32 `[L, 3]` tables
and `__getitem__` returns a few hundred bytes of indices in the reference's slot order.  The order
of every call to the GLOBAL numpy RNG (`get_relship_by_id` :234-239 of util_functions.py,
`Relationship.scene2rel` :70-74, the train-mode context subsampling :387, 405, 488) is the
reference's, so a seeded run emits bit-identical items (tests/test_dataloader_cpu.py, against
items produced by the reference's unmodified code: tests/golden/dataloader_*.npz).

Annotation parsing (load_annotated_inter & co.) is outside the hot path: the constructor takes the
objects those loaders return (`source`), e.g. from mixed_utils/synthetic_world.py.
"""
from collections import defaultdict
from itertools import permutations

import numpy as np
import torch
from torch.utils.data import Dataset

from lirec_b200.packing import PackedBatch, soft_pos_of
from lirec_b200.utils.arg_pars import opt


class _PairScenes:
    def __init__(self):
        self.scenes2inters = defaultdict(list)


def _mt_words(s0, s1, max_regen=64):
    """32-bit words the global MT19937 produced between two `np.random.get_state()` snapshots (None if that
    cannot be told): the position difference while the key is unchanged, else whole regenerations are
    stepped through on a scratch generator."""
    k0, p0, k1, p1 = s0[1], int(s0[2]), s1[1], int(s1[2])
    if s0[3] != s1[3]:                      # a gaussian was drawn / cached: not a stream we account for
        return None
    if np.array_equal(k0, k1):
        return p1 - p0 if p1 >= p0 else None
    rs, words, key = np.random.RandomState(), 624 - p0, k0
    for _ in range(max_regen):
        rs.set_state(("MT19937", key, 624, 0, 0.0))
        rs.bytes(4)                         # one word: regenerates the key, position 1
        key = rs.get_state()[1]
        if np.array_equal(key, k1):
            return words + p1
        words += 624
    return None


class _Blocks:
    """Read-only sequence of the context blocks of one record: block i = rows [off[i], off[i+1]) of `cat`."""

    def __init__(self, cat, counts, off=None):
        self._cat = cat
        self._off = np.concatenate(([0], np.cumsum(counts))) if off is None else off

    def __len__(self):
        return len(self._off) - 1

    def __getitem__(self, i):
        if i < 0:
            i += len(self)
        return self._cat[self._off[i]:self._off[i + 1]]

    def __iter__(self):
        return (self[i] for i in range(len(self)))


class IndexedMixedFeaturesDataset(Dataset):
    """source: dict with `interactions`, `rels`, `rels_list`, `rels_opp`, `clip_vec`, `track_vec`
    (see synthetic_world.subset) and `vocab`: object with `inter2idx`, `inter2mgd`, `mgd2idx`,
    `interaction_names`, `iou2_clips`."""

    def __init__(self, source, vocab, mode="train"):
        self.mode = mode
        self.inter2idx, self.inter2mgd, self.mgd2idx = vocab.inter2idx, vocab.inter2mgd, vocab.mgd2idx
        self.iou2_clips = vocab.iou2_clips
        # merged class of every interaction index (reference :116-122)
        self.interidx2mgdidx = np.zeros(len(self.inter2idx), dtype=int)
        col = 0 if opt.inter_class == "all" else -1
        for name, idx3 in self.inter2idx.items():
            self.interidx2mgdidx[idx3[col]] = self.mgd2idx[self.inter2mgd[name]]
        self.n_classes = len(self.mgd2idx) if opt.merged else len(vocab.interaction_names[opt.inter_class])
        self.tracks = opt.tracks if mode == "train" else True
        self.triplets = bool(opt.tr_maximize)
        self.test_rels_multi_clip = False
        self._max_n_tripl = 0
        self.rels_n_clips = 0
        self._plans, self._plan_sig, self._trace, self._trace_blk, self._forced = {}, None, None, 0, None
        self.interactions = source["interactions"]
        with_rels = bool(opt.rels or opt.rels_multitask)
        self.rels = source["rels"] if with_rels else {}
        self.rels_list = list(source["rels_list"]) if with_rels else []
        self.rels_opp = source["rels_opp"] if with_rels else {}
        self._clip_vec, self._track_vec = source["clip_vec"], source["track_vec"]
        self.rels2idx, self.idx2rels, self.n_rels = {}, {}, 0
        self.epoch = 0

        # sample list, scene -> interactions, pair -> scenes, and the relationship timeline fix-ups for
        # pairs that interact before their first annotated relationship (reference :61-100)
        self.idxs_with_triplets = []
        self.mv2sc2intersid = {}
        self.pair2scenes = defaultdict(_PairScenes)
        for inter in self.interactions:
            movie, scene = inter.video_descr["movie"], inter.video_descr["scene"][0]
            self.mv2sc2intersid.setdefault(movie, defaultdict(list))[scene].append(inter.id)
            if not self.tracks or len(inter.triplets) == 0:
                self.idxs_with_triplets.append((inter.id, 0))
                continue
            for t_idx in inter.triplets:
                self.idxs_with_triplets.append((inter.id, t_idx))
                tr = inter.triplets[t_idx]
                if len(tr) != 2:
                    continue
                a, b = tr[0], tr[1]
                self.pair2scenes[(movie, a, b)].scenes2inters[scene].append(inter.id)
                self.pair2scenes[(movie, b, a)].scenes2inters[scene].append(inter.id)
                if not opt.rels_multi_clip:
                    continue
                mrels = self.rels[movie]
                if (a, b) in mrels and scene not in mrels[(a, b)].scenes:
                    if len(mrels[(a, b)].rel2scenes) == 1:
                        mrels[(a, b)].append_scene(None, scene)
                        mrels[(b, a)].append_scene(None, scene)
                        inter.relships[t_idx] = [mrels[(a, b)].rels_name]
                    else:
                        # the reference never updates its running minimum (:92-97), so the relationship
                        # picked is the LAST one of the pair's timeline; kept
                        name = None
                        for r in mrels[(a, b)].rel2scenes:
                            name = r
                        mrels[(a, b)].append_scene(name, scene)
                        mrels[(b, a)].append_scene(self.rels_opp[name], scene)
                        inter.relships[t_idx] = [name]

    # ---- relationship vocabulary (reference :124-135) ---------------------------------------------
    def init_relships(self):
        self.rels_list = list(reversed(sorted(self.rels_list)))
        for i, r in enumerate(self.rels_list):
            self.rels2idx[r] = i
            self.idx2rels[i] = r
        assert self.rels2idx["None"] == len(self.rels_list) - 1
        self.n_rels = len(self.rels_list)
        return self

    # ---- banks + context tables (reference :139-262) ------------------------------------------------
    def cache(self):
        n = len(self.interactions)
        cd = next(iter(self._clip_vec.values())).shape[-1]
        td = next(iter(self._track_vec.values())).shape[-1]
        self.clip_bank = np.zeros((n + 1, cd), dtype=np.float32)      # row n: the all-zero clip vector
        self.zero_clip = n
        tracks = [np.zeros((1, td), dtype=np.float32)]
        self.track_row = {}
        for inter in self.interactions:
            self.clip_bank[inter.id] = np.asarray(self._clip_vec[inter.id]).reshape(-1)
            for name in inter.id2names.values():
                v = np.asarray(self._track_vec[(inter.id, name)], dtype=np.float32).reshape(1, -1)
                if not v.any():
                    self.track_row[(inter.id, name)] = 0
                else:
                    self.track_row[(inter.id, name)] = len(tracks)
                    tracks.append(v)
        self.track_bank = np.vstack(tracks)
        # relationship of 2-person triplets whose scene is covered by the pair's timeline (:149-156)
        for i_id, t_idx in self.idxs_with_triplets:
            inter = self.interactions[i_id]
            if not inter.triplets or len(inter.triplets[t_idx]) != 2 or t_idx in inter.relships:
                continue
            if opt.rels_multi_clip:
                a, b = inter.triplets[t_idx][0], inter.triplets[t_idx][1]
                movie, scene = inter.video_descr["movie"], inter.video_descr["scene"][0]
                if (a, b) in self.rels[movie] and scene in self.rels[movie][(a, b)].scenes:
                    inter.relships[t_idx] = self.rels[movie][(a, b)]._scene2rel[scene]
        self._max_n_tripl = int(getattr(opt, "max_n_tripl", 20))       # reference hard-codes 20 (:177)
        if opt.rels_multi_clip:
            self.rels_n_clips = opt.rels_n_clips
            self._cache_relationships()
        self._plans, self._plan_sig = {}, None      # cached records point into the tables built above
        return self

    def _triple(self, inter_id, a, b):
        return (inter_id, self.track_row[(inter_id, a)], self.track_row[(inter_id, b)])

    def _eval_subset(self, L):
        n = self.rels_n_clips
        return list(range(0, L, L // n))[:n]

    def _cache_relationships(self):
        self.movie_ch1_ch2_rel, self.movie_ch1_ch2_rel_inter = {}, {}
        self.hashidx_rels, self.hashrels_idx, self.context_idxs = {}, {}, {}
        cached_pairs = set()
        for movie in self.rels:
            for pair in self.rels[movie]:
                for rel, scenes in self.rels[movie][pair].rel2scenes.items():
                    key = (movie, pair[0], pair[1], rel)
                    cached_pairs.add(pair)
                    if key not in self.hashidx_rels:
                        h = len(self.hashidx_rels)
                        self.hashidx_rels[key] = h
                        self.hashrels_idx[h] = key
                    rows, classes = [], []
                    for scene in scenes:
                        for i_id in self.mv2sc2intersid[movie][scene]:
                            inter = self.interactions[i_id]
                            if pair[0] in inter.name2id and pair[1] in inter.name2id:
                                rows.append(self._triple(i_id, pair[0], pair[1]))
                                classes.append(self.mgd2idx[self.inter2mgd[inter.inter_node["name"]]])
                    self.movie_ch1_ch2_rel[key] = np.asarray(rows, dtype=np.int32).reshape(-1, 3)
                    self.movie_ch1_ch2_rel_inter[key] = np.asarray(classes, dtype=int)
                    if self.mode != "train" and len(rows) > self.rels_n_clips:
                        self.context_idxs[key] = self._eval_subset(len(rows))
        # pairs that interact but never get a relationship (reference :237-262)
        self.movie_ch1_ch2_none, self.movie_ch1_ch2_none_inter, self.context_idxs_none = {}, {}, {}
        for key, val in self.pair2scenes.items():
            movie, a, b = key
            if (a, b) in cached_pairs:
                continue
            rows, classes = [], []
            for scene in val.scenes2inters:
                for i_id in val.scenes2inters[scene]:
                    rows.append(self._triple(i_id, a, b))
                    classes.append(self.mgd2idx[self.inter2mgd[self.interactions[i_id].inter_node["name"]]])
            self.movie_ch1_ch2_none[key] = np.asarray(rows, dtype=np.int32).reshape(-1, 3)
            self.movie_ch1_ch2_none_inter[key] = np.asarray(classes, dtype=int)
            if self.mode != "train" and len(rows) > self.rels_n_clips:
                self.context_idxs_none[key] = self._eval_subset(len(rows))

    # ---- items ----------------------------------------------------------------------------------------
    def __len__(self):
        return len(self.idxs_with_triplets)

    def _context(self, table, classes, eval_idxs, key):
        """Context rows of `key`, subsampled to rels_n_clips like the reference (:381-391, 399-410)."""
        rows = table[key]
        L, n = len(rows), self.rels_n_clips
        if L <= n:
            return rows, (None if classes is None else classes[key])
        if self.mode == "train":
            # = np.random.choice(np.arange(L), n, replace=False) (reference :387), same global RNG stream
            if self._trace is not None:              # cached mode: a replayed prefix is forced, the rest accounted for
                if self._forced:
                    sel, words = self._forced.pop(0), 0
                else:
                    pre = np.random.get_state()
                    sel = np.random.permutation(L)[:n]
                    words = _mt_words(pre, np.random.get_state())
                self._trace.append(("p", self._trace_blk, rows, None if classes is None else classes[key], n, words))
            else:
                sel = np.random.permutation(L)[:n]
        else:
            sel = eval_idxs[key]
        return rows[sel], (None if classes is None else classes[key][sel])

    def _choose(self, names):
        """`np.random.choice(names)` of the annotation objects (`AnnotatedInter.get_relship_by_id`, reference
        utils/util_functions.py:234-236; `Relationship.scene2rel`, :70-73) = names[randint(0, len)] on the
        same global RNG stream (a single name consumes no random number), as a traced / replayable draw."""
        k = len(names)
        if k == 1:
            return names[0]
        if self._trace is None:
            return names[np.random.randint(0, k)]
        if self._forced:
            o, words = self._forced.pop(0), 0
        else:
            pre = np.random.get_state()
            o = int(np.random.randint(0, k))
            words = _mt_words(pre, np.random.get_state())
        self._trace.append(("c", k, o, words))
        return names[o]

    # ---- record cache -----------------------------------------------------------------------------------
    # An item is a deterministic function of the annotations and of the random numbers it draws: (a) the
    # train-mode context subsampling above and (b) the choice among several relationship names of a pair
    # (`_choose`).  (a) changes rows, (b) changes what is built next.  Per item the cache keeps the DECISION
    # TREE of its draws: ["c", k, {outcome: node}] for a choice among k names, ["p", block, rows, classes, n,
    # node] for a subsampling of `rows` to n, ["l", record] at the end.  An access walks the tree making the
    # same draws, in the same order, on the global numpy RNG — so the stream stays the reference's — then
    # copies the leaf's record and lays the freshly drawn context rows into it; an outcome met for the first
    # time builds the record with the draws made so far forced and hangs the new branch into the tree.
    # Whether a build drew anything the tree does not account for is decided by exact accounting of the
    # generator words it consumed; such items are rebuilt on every access.  Records are shared between
    # accesses: treat them as read-only.
    def _signature(self):
        return (self.mode, self.rels_n_clips, self._max_n_tripl, bool(self.triplets), opt.inter_class, bool(opt.merged),
                bool(opt.rels_multi_clip), bool(opt.tracks), bool(opt.rels_multitask), bool(opt.multilab_weights),
                bool(opt.soft_gt))

    def __getitem__(self, idx_pair):
        sig = self._signature()
        if sig != self._plan_sig:
            self._plans, self._plan_sig = {}, sig
        node = self._plans.get(idx_pair)
        if node is False:                            # draws random numbers the tree cannot account for
            return self._build_record(idx_pair)
        if node is None:
            if not int(getattr(opt, "cache_records", 1)):
                return self._build_record(idx_pair)
            return self._explore(idx_pair, None, None, [])
        drawn, perms = [], None
        while True:
            tag = node[0]
            if tag == "l":
                break
            if tag == "p":
                sel = np.random.permutation(len(node[2]))[:node[4]]
                if perms is None:
                    perms = []
                perms.append((node, sel))
                drawn.append(sel)
                node = node[5]
            else:
                o = int(np.random.randint(0, node[1]))
                drawn.append(o)
                nxt = node[2].get(o)
                if nxt is None:
                    return self._explore(idx_pair, node, o, drawn)
                node = nxt
        rec0 = node[1]
        rec = dict(rec0)
        if perms:
            cat, off = rec0["ctx_cat"].copy(), rec0["ctx_rows"]._off
            for (_, blk, rows_all, cls_all, n, _), sel in perms:
                cat[off[blk]:off[blk] + n] = rows_all[sel]
                if cls_all is not None:
                    rec["ctx_labels"] = np.asarray(cls_all[sel], dtype=int)
            rec["ctx_cat"], rec["ctx_rows"] = cat, _Blocks(cat, None, off)
        return rec

    def _explore(self, idx_pair, parent, outcome, drawn):
        """Build the record with the draws already made (`drawn`) forced, account for every generator word
        the rest of the build consumes, and hang the new branch under `parent[outcome]` (or as the root)."""
        s0 = np.random.get_state()
        self._trace, self._trace_blk, self._forced = [], 0, list(drawn)
        try:
            rec = self._build_record(idx_pair)
            events, leftover = self._trace, len(self._forced)
        finally:
            self._trace, self._forced = None, None
        total = _mt_words(s0, np.random.get_state())
        new = events[len(drawn):]
        words = [e[-1] for e in new]
        if leftover or len(events) < len(drawn) or total is None or None in words or total != sum(words):
            self._plans[idx_pair] = False
            return rec
        tail = ["l", rec]
        for e in reversed(new):
            tail = ["c", e[1], {e[2]: tail}] if e[0] == "c" else ["p", e[1], e[2], e[3], e[4], tail]
        if parent is None:
            self._plans[idx_pair] = tail
        else:
            parent[2][outcome] = tail
        return dict(rec)

    def warm_records(self, max_branches=32):
        """Build every item's decision tree ahead of use (global RNG state preserved): the path a first access
        takes, then the outcomes not met yet, up to `max_branches` per item.  DataLoader workers forked
        afterwards share the trees copy-on-write instead of each exploring them again."""
        if not int(getattr(opt, "cache_records", 1)):
            return self
        state = np.random.get_state()
        try:
            for i in range(len(self)):
                if self._plans.get(i) is None or self._plan_sig != self._signature():
                    self[i]
                budget = int(max_branches)
                stack = [(self._plans.get(i), [])]
                while stack and budget > 0 and self._plans.get(i):
                    node, drawn = stack.pop()
                    if node[0] == "p":                       # any subsample does: an access lays its own rows in
                        stack.append((node[5], drawn + [np.arange(node[4])]))
                    elif node[0] == "c":
                        for o in range(node[1]):
                            if o not in node[2] and budget > 0:
                                budget -= 1
                                self._explore(i, node, o, drawn + [o])
                            if self._plans.get(i) and o in node[2]:
                                stack.append((node[2][o], drawn + [o]))
        finally:
            np.random.set_state(state)
        return self

    def _build_record(self, idx_pair):
        i_id, t_idx = self.idxs_with_triplets[idx_pair]
        inter = self.interactions[i_id]
        movie, scene = inter.video_descr["movie"], inter.video_descr["scene"][0]
        name = inter.inter_node["name"]
        lab_col = 0 if opt.inter_class == "all" else 2
        label = self.inter2idx[name][lab_col]
        if opt.merged:
            label = int(self.interidx2mgdidx[label])
        rec = {"inter_id": i_id, "labels": label, "n_ctx_slots": self.rels_n_clips if opt.rels_multi_clip else 0}
        if not (opt.tracks and len(inter.triplets)):
            if opt.tracks:
                raise EnvironmentError                     # reference :585-586
            # opt.tracks off (reference :587-588): the item is the clip's pooled text|visual vector alone — one
            # candidate row whose two track slots point at the all-zero track row (the model drops those slots)
            rec["cand_rows"] = np.asarray([(i_id, 0, 0)], dtype=np.int32)
            rec["no_tracks"] = True
            return self._soft_labels(rec, movie, scene, name, label, lab_col)
        trip = inter.triplets[t_idx]
        tr = self.track_row
        T, S, NONE = self._max_n_tripl, self.rels_n_clips, "None"

        def row(a, b):          # a / b: character name or None (no track in that slot)
            return (i_id, 0 if a is None else tr[(i_id, a)], 0 if b is None else tr[(i_id, b)])

        gt_row = row(trip.get(0), trip.get(1))
        rec["just_zeros"] = bool(gt_row[1] == 0 and gt_row[2] == 0)
        cand, ctx, ctx_lab, rels_labs = [gt_row], [], None, []
        tiled = []              # per candidate: context block is an np.tile of the candidate's own row

        if opt.rels_multitask:
            rel_opts = inter.relships.get(t_idx)         # = inter.get_relship_by_id(t_idx), as a replayable draw
            gt_rel = self.rels2idx[self._choose(rel_opts) if rel_opts else NONE]
            rec["rels_label"] = gt_rel
            if opt.rels_multi_clip:
                if len(trip) == 2:
                    a, b = trip[0], trip[1]
                    rel_name = self.idx2rels[gt_rel]
                    if rel_name == NONE:
                        rec["hash_rel"] = -1
                        key = (movie, a, b)
                        if len(self.movie_ch1_ch2_none[key]) == 0:
                            rows, cls = np.asarray([gt_row], dtype=np.int32), np.asarray([label])
                        else:
                            rows, cls = self._context(self.movie_ch1_ch2_none, self.movie_ch1_ch2_none_inter,
                                                      self.context_idxs_none, key)
                    else:
                        key = (movie, a, b, rel_name)
                        rec["hash_rel"] = self.hashidx_rels[key]
                        rows, cls = self._context(self.movie_ch1_ch2_rel, self.movie_ch1_ch2_rel_inter,
                                                  self.context_idxs, key)
                else:
                    rec["hash_rel"] = -1
                    rows, cls = np.asarray([gt_row], dtype=np.int32), np.asarray([label])
                tiled.append(len(trip) != 2)
                ctx.append(np.asarray(rows, dtype=np.int32).reshape(-1, 3))
                ctx_lab = np.asarray(cls, dtype=int)
                # from here on a context block is either a table slice (ndarray [L, 3]) or ONE row, kept as
                # the tuple it is: the blocks are laid out back to back once, below
                rels_labs.append(gt_rel)

        if self.triplets:
            gt_tracks = [0, 0]
            zeros = True
            gt_name = None
            names = list(inter.id2names.values())
            for a, b in permutations(names, 2):
                if len(trip) == 2:
                    if a == trip[0] and b == trip[1]:
                        continue
                    if inter.bi and a == trip[1] and b == trip[0]:
                        gt_tracks[1] = len(cand) - 1             # the reference's off-by-one (:453), kept
                r = row(a, b)
                if r[1] or r[2]:
                    zeros = False
                if len(cand) >= T:
                    continue
                if opt.rels_multitask:
                    rel_name, rows = NONE, r
                    if (a, b) in self.rels[movie]:
                        rel_opts = self.rels[movie][(a, b)]._scene2rel.get(scene)  # = .scene2rel(scene)
                        rel_name = self._choose(rel_opts) if rel_opts else NONE
                        if rel_name != NONE:
                            self._trace_blk = len(ctx)
                            rows, _ = self._context(self.movie_ch1_ch2_rel, None, self.context_idxs,
                                                    (movie, a, b, rel_name))
                            # the reference fills rows 1.. of this candidate's block and leaves row 0 — the
                            # row its interaction branch reads — all zero (:461-476); kept
                            r = (self.zero_clip, 0, 0)
                    ctx.append(rows)
                    tiled.append(rel_name == NONE)
                    rels_labs.append(self.rels2idx[rel_name])
                cand.append(r)
            if len(trip) == 1:
                position, gt_name = list(trip.items())[0]
                r = row(None, gt_name) if position == 0 else row(gt_name, None)   # the wrong slot
                if r[1] or r[2]:
                    zeros = False
                if len(cand) < T:
                    if inter.bi:
                        gt_tracks[1] = len(cand)
                    if opt.rels_multitask:
                        ctx.append(r)
                        tiled.append(True)
                        rels_labs.append(self.rels2idx[NONE])
                    cand.append(r)
            for a in names:
                if len(trip) == 1 and a == gt_name:
                    continue
                if len(cand) < T - 1:
                    for r in (row(a, None), row(None, a)):
                        if opt.rels_multitask:
                            ctx.append(r)
                            tiled.append(True)
                            rels_labs.append(self.rels2idx[NONE])
                        cand.append(r)
            rec["just_zeros"] = zeros
            rec["gt_tracks"] = np.asarray(gt_tracks)
            rec["n_names"] = len(inter.id2names)
        rec["cand_rows"] = np.asarray(cand, dtype=np.int32).reshape(-1, 3)
        if opt.rels_multitask and opt.rels_multi_clip:
            # the blocks back to back + their lengths: what collate needs (one pass per item here instead
            # of thousands of small array ops per batch there); `ctx_rows` indexes into it block by block
            counts = np.fromiter((1 if type(x) is tuple else len(x) for x in ctx), dtype=np.int32, count=len(ctx))
            cat = np.empty((int(counts.sum()), 3), dtype=np.int32)
            pos = 0
            for x in ctx:
                if type(x) is tuple:
                    cat[pos] = x
                    pos += 1
                else:
                    cat[pos:pos + len(x)] = x
                    pos += len(x)
            rec["ctx_counts"], rec["ctx_cat"] = counts, cat
            rec["ctx_rows"] = _Blocks(cat, counts)
            rec["ctx_tiled"] = tiled
            rec["ctx_labels"] = ctx_lab
        if opt.rels_multitask and self.triplets:
            rec["rels_label"] = np.asarray(rels_labs, dtype=np.int64)

        return self._soft_labels(rec, movie, scene, name, label, lab_col)

    def _soft_labels(self, rec, movie, scene, name, label, lab_col):
        """multilab_weights / soft_labels of an item (reference :590-616)."""
        soft = self.iou2_clips[(movie, scene)][name]
        if opt.multilab_weights:
            w, w_axl = np.ones(self.n_classes), np.ones(len(self.interidx2mgdidx))
            for s_name in soft:
                if opt.inter_class != "all" and ["t", "v", "m"][self.inter2idx[s_name][1]] != opt.inter_class:
                    continue
                k = self.inter2idx[s_name][lab_col]
                w_axl[k] = 0
                w[self.interidx2mgdidx[k]] = 0
            rec["multilab_weights"], rec["multilab_weights_axl"] = w, w_axl
        if opt.soft_gt:
            sl, pos = np.ones(self.n_classes) * -1, 1
            sl[0] = label
            for s_name in soft:
                if opt.inter_class != "all" and ["t", "v", "m"][self.inter2idx[s_name][1]] != opt.inter_class:
                    continue
                sl[pos] = self.interidx2mgdidx[self.inter2idx[s_name][lab_col]]
                pos += 1
            rec["soft_labels"] = sl
        return rec

    def collate(self, records):
        return collate_indexed(records, self, resident=bool(getattr(opt, "resident_banks", 0)))

    # ---- the reference's dense item, rebuilt from a record (compat / parity tests) -----------------------
    def dense_item(self, rec):
        """Exactly what the reference `__getitem__` returns for this sample (float64 features)."""
        clip, track = self.clip_bank.astype(np.float64), self.track_bank.astype(np.float64)

        def vec(rows):
            rows = np.asarray(rows).reshape(-1, 3)
            return np.hstack((clip[rows[:, 0]], track[rows[:, 1]], track[rows[:, 2]]))

        out = {"labels": rec["labels"]}
        T, S = self._max_n_tripl, rec["n_ctx_slots"]
        cand = vec(rec["cand_rows"])
        D = cand.shape[1]
        for k in ("just_zeros", "hash_rel", "n_names", "gt_tracks", "multilab_weights", "multilab_weights_axl",
                  "soft_labels"):
            if k in rec:
                out[k] = rec[k]

        def context_block(r0, rows, tiled):
            blk = np.zeros((S + 1, D))
            mask = np.zeros(S, dtype=int)
            if tiled:
                blk[:] = r0
                mask[0] = 1
            else:
                blk[0] = r0
                blk[1:1 + len(rows)] = vec(rows)
                mask[:len(rows)] = 1
            return blk, mask

        if self.triplets:
            n = len(rec["cand_rows"])
            mem_mask = np.zeros(T)
            mem_mask[:n] = 1
            out["mem_mask"] = mem_mask
            if "ctx_rows" in rec:
                feats = np.zeros((T, S + 1, D))
                masks = np.zeros((T, S), dtype=int)
                for i in range(n):
                    feats[i], masks[i] = context_block(cand[i], rec["ctx_rows"][i], rec["ctx_tiled"][i])
                labs = np.zeros(T, dtype=int)
                labs[:n] = rec["rels_label"]
                out["features"], out["rels_mask"], out["rels_label"] = feats, masks, labs
            else:
                feats = np.zeros((T, D))
                cd = clip.shape[1]
                feats[:, :cd] = cand[0, :cd]                       # clip features are tiled into every slot (:335)
                feats[:n, cd:] = cand[:, cd:]
                out["features"] = feats
        elif "ctx_rows" in rec:
            blk, mask = context_block(cand[0], rec["ctx_rows"][0], rec["ctx_tiled"][0])
            gt = np.zeros((S + 1, 1), dtype=int)
            gt[0] = rec["labels"]
            if rec["ctx_tiled"][0]:
                gt[:] = rec["labels"]
            else:
                gt[1:1 + len(rec["ctx_labels"]), 0] = rec["ctx_labels"]
            out["features"], out["labels"], out["rels_mask"] = blk, gt, mask.reshape(-1, 1)
            out["rels_label"] = rec["rels_label"]
        else:
            out["features"] = cand[:1, :clip.shape[1]] if rec.get("no_tracks") else cand[:1]
            if "rels_label" in rec:
                out["rels_label"] = rec["rels_label"]
        return out


def _banks_bf16(dataset):
    """bf16 torch copies of the dataset's two feature banks (what a batch ships), made once per bank array:
    rounding a row before or after gathering it is the same row."""
    cached = dataset.__dict__.get("_bf16_banks")
    if cached is None or cached[0] is not dataset.clip_bank or cached[1] is not dataset.track_bank:
        cached = (dataset.clip_bank, dataset.track_bank,
                  torch.from_numpy(np.ascontiguousarray(dataset.clip_bank, dtype=np.float32)).to(torch.bfloat16),
                  torch.from_numpy(np.ascontiguousarray(dataset.track_bank, dtype=np.float32)).to(torch.bfloat16))
        dataset.__dict__["_bf16_banks"] = cached
    return cached[2], cached[3]


def collate_indexed(records, dataset, resident=False):
    """records -> host PackedBatch.  The batch banks hold every referenced bank row ONCE: rows used by
    candidates first (the ints-branch prefix), then the rows only context refers to; references to the
    shared all-zero track row are redirected to one private zero row per clip (a single row referenced by
    thousands of table rows serialises the backward scatter-reduce).  With `resident=True` the banks are
    left out and `pb.extras['bank_rows']` lists the dataset-bank rows to gather on the device.

    The integer tables are built by the native `lirec_collate_tables` (csrc/collate.cu; host code, safe in
    DataLoader workers) straight into one int32 arena; `collate_indexed_numpy` states the same tables in
    numpy, and the tests hold the native one to it."""
    from lirec_b200 import _ext
    L = _ext.lib()
    B = len(records)
    has_ctx = "ctx_rows" in records[0]
    track_models = "gt_tracks" in records[0]
    cand = np.ascontiguousarray(np.concatenate([r["cand_rows"] for r in records]), dtype=np.int32).reshape(-1, 3)
    counts = np.fromiter((len(r["cand_rows"]) for r in records), dtype=np.int32, count=B)
    Ni = int(cand.shape[0])
    ctx = ctx_counts = None
    Nx = 0
    if has_ctx:
        if "ctx_cat" in records[0]:
            ctx_counts = np.concatenate([r["ctx_counts"] for r in records])
            ctx = np.concatenate([r["ctx_cat"] for r in records])
        else:                                                   # records built by hand (tests, tools)
            per = [np.asarray(x, dtype=np.int32).reshape(-1, 3) for r in records for x in r["ctx_rows"]]
            ctx_counts = np.array([len(x) for x in per])
            ctx = np.concatenate(per) if len(per) else np.zeros((0, 3), dtype=np.int32)
        ctx_counts = np.ascontiguousarray(ctx_counts, dtype=np.int32)
        ctx = np.ascontiguousarray(ctx, dtype=np.int32).reshape(-1, 3)
        Nx = int(ctx.shape[0])
        if len(ctx_counts) != Ni or int(ctx_counts.sum()) != Nx:
            raise ValueError("collate_indexed: context blocks do not match the candidate rows")
    T = dataset._max_n_tripl if track_models else 1
    rels_label = None
    if has_ctx and track_models:
        rels_label = np.concatenate([np.asarray(r["rels_label"]).reshape(-1) for r in records])
    elif has_ctx:
        rels_label = np.array([r["rels_label"] for r in records])
    gt = np.concatenate([r["gt_tracks"] for r in records]).reshape(B, 2) if track_models else \
        np.zeros((B, 2), dtype=np.int64)
    mw = np.concatenate([r["multilab_weights"] for r in records]).reshape(B, -1) if "multilab_weights" in records[0] \
        else np.ones((B, dataset.n_classes))
    extras = {k: np.array([r[k] for r in records]) for k in ("just_zeros", "n_names", "hash_rel") if k in records[0]}
    pb = collate_arrays(dataset, cand, counts, ctx if has_ctx else None, ctx_counts if has_ctx else None,
                        [r["labels"] for r in records], rels_label, gt, mw, extras, T, records[0]["n_ctx_slots"],
                        resident)
    return _with_soft_pos(pb, records, dataset)


def _with_soft_pos(pb, records, dataset):
    """--soft_gt: attach the uint8 [B, C] multi-hot of the records' soft labels (`pb.soft_pos`), the positives of
    the BCE losses.  Without soft labels the batch is left exactly as it is."""
    if "soft_labels" in records[0]:
        pb.soft_pos = soft_pos_of(np.stack([np.asarray(r["soft_labels"]).reshape(-1) for r in records]),
                                  dataset.n_classes)
    return pb


def collate_arrays(dataset, cand, counts, ctx, ctx_counts, labels, rels_label, gt, multilab, extras, n_slots,
                   n_ctx_slots, resident, arena_out=None):
    """The batch-level half of `collate_indexed`: the concatenated index triples of B clips (int32, C-contiguous)
    -> every integer table by `lirec_collate_tables`, in one arena, -> host PackedBatch.  `ctx is None`: no
    context branch.  `arena_out`: a caller-owned int32 torch tensor (pinned memory, large enough) the tables are
    written into directly — the batch is then born pinned (`pb._arena`), no staging copy."""
    from lirec_b200 import _ext
    L = _ext.lib()
    B, Ni = int(len(counts)), int(cand.shape[0])
    has_ctx = ctx is not None
    Nx = int(ctx.shape[0]) if has_ctx else 0
    need = int(L.lirec_collate_arena_bound(B, Ni, Nx, int(has_ctx)))
    if arena_out is not None:
        if arena_out.numel() < need:
            raise ValueError("collate_arrays: arena_out holds %d ints, the batch needs %d" % (arena_out.numel(), need))
        arena = arena_out.numpy()[:need]
    else:
        arena = np.empty(need, dtype=np.int32)
    layout = np.empty((24, 2), dtype=np.int64)
    sizes = np.empty(4, dtype=np.int32)
    _ext.check(L.lirec_collate_tables(
        cand.ctypes.data, counts.ctypes.data, B, ctx.ctypes.data if has_ctx else None,
        ctx_counts.ctypes.data if has_ctx else None, int(dataset.zero_clip), len(dataset.clip_bank),
        len(dataset.track_bank), int(n_slots), arena.ctypes.data, arena.size, layout.ctypes.data, sizes.ctypes.data))
    n_clip, n_clip_ints, n_track, n_track_ints = (int(v) for v in sizes)
    src = (int(layout[22, 0]), n_clip, int(layout[23, 0]), n_track)
    clip_src = arena[src[0]:src[0] + n_clip]
    track_src = arena[src[2]:src[2] + n_track]
    if resident:                                                # banks are gathered on the device
        clip_bank = torch.empty((n_clip, 0), dtype=torch.bfloat16)
        track_bank = torch.empty((n_track, 0), dtype=torch.bfloat16)
    else:                                                       # gather the rows from the bf16 copy of the banks
        clip16, track16 = _banks_bf16(dataset)
        clip_bank = clip16.index_select(0, torch.from_numpy(clip_src).long())
        track_bank = track16.index_select(0, torch.from_numpy(track_src).long())
    pb = PackedBatch.from_arena(
        arena, layout[:22], clip_bank, track_bank, n_clip_ints, n_track_ints, B, Ni, Nx if has_ctx else None,
        labels, rels_label, gt, multilab, n_slots=n_slots, n_ctx_slots=n_ctx_slots, extras=extras, src_layout=src)
    pb.extras["bank_rows"] = (clip_src, track_src)              # views into the arena: they travel (and pin) with it
    if arena_out is not None:                                   # born pinned: to_device() copies straight from it
        pb._arena, pb._layout = arena_out[:pb._host_arena.size], pb._host_layout
    return pb


def collate_indexed_numpy(records, dataset, resident=False):
    """The numpy statement of `collate_indexed` (same tables, bit for bit)."""
    B = len(records)
    has_ctx = "ctx_rows" in records[0]
    track_models = "gt_tracks" in records[0]
    cand = np.concatenate([r["cand_rows"] for r in records]).astype(np.int64)
    counts = np.array([len(r["cand_rows"]) for r in records])
    cand_off = np.concatenate(([0], np.cumsum(counts)))
    cand_clip_of = np.repeat(np.arange(B), counts)
    ZERO = -1 - cand_clip_of                                    # private zero row of the owning clip
    zc = dataset.zero_clip
    cand_t = cand.copy()
    cand_t[:, 0] = np.where(cand[:, 0] == zc, ZERO, cand[:, 0])
    for c in (1, 2):
        cand_t[:, c] = np.where(cand[:, c] == 0, ZERO, cand[:, c])
    ctx_t = ctx_off = None
    if has_ctx:
        if "ctx_cat" in records[0]:
            ctx_counts = np.concatenate([r["ctx_counts"] for r in records])
            ctx_t = np.concatenate([r["ctx_cat"] for r in records]).astype(np.int64)     # fresh copy, edited below
        else:                                                   # records built by hand (tests, tools)
            per = [np.asarray(x, dtype=np.int64).reshape(-1, 3) for r in records for x in r["ctx_rows"]]
            ctx_counts = np.array([len(x) for x in per])
            ctx_t = np.concatenate(per) if len(per) else np.zeros((0, 3), dtype=np.int64)
        ctx_off = np.concatenate(([0], np.cumsum(ctx_counts)))
        owner_clip = np.repeat(cand_clip_of, ctx_counts)
        ctx_t[:, 0] = np.where(ctx_t[:, 0] == zc, -1 - owner_clip, ctx_t[:, 0])
        for c in (1, 2):
            ctx_t[:, c] = np.where(ctx_t[:, c] == 0, -1 - owner_clip, ctx_t[:, c])

    # Bank rows are small non-negative integers and the private zero rows are -1 - clip in [-B, -1]: the
    # unique / set-difference / lookup steps are marks and gathers over a table of n_rows + B entries
    # (same order as np.unique + np.setdiff1d: ints rows ascending, then the context-only rows ascending).
    def remap(cols_ints, cols_ctx, n_rows):
        size = n_rows + B
        seen = np.zeros(size, dtype=bool)
        seen[cols_ints + B] = True
        u_ints = np.flatnonzero(seen)
        if cols_ctx is not None:
            seen_ctx = np.zeros(size, dtype=bool)
            seen_ctx[cols_ctx + B] = True
            seen_ctx[u_ints] = False
            order = np.concatenate((u_ints, np.flatnonzero(seen_ctx)))
        else:
            order = u_ints
        lut = np.empty(size, dtype=np.int64)
        lut[order] = np.arange(len(order))
        return order - B, len(u_ints), lut

    c_order, n_clip_ints, c_lut = remap(cand_t[:, 0], ctx_t[:, 0] if has_ctx else None, len(dataset.clip_bank))
    t_order, n_track_ints, t_lut = remap(cand_t[:, 1:].reshape(-1), ctx_t[:, 1:].reshape(-1) if has_ctx else None,
                                         len(dataset.track_bank))

    def apply(tbl):
        return np.stack((c_lut[tbl[:, 0] + B], t_lut[tbl[:, 1] + B], t_lut[tbl[:, 2] + B]), axis=1)

    clip_src = np.where(c_order < 0, zc, c_order)
    track_src = np.where(t_order < 0, 0, t_order)               # private zero rows read the zero row
    if resident:                                                # banks are gathered on the device
        clip_bank = torch.empty((len(clip_src), 0), dtype=torch.bfloat16)
        track_bank = torch.empty((len(track_src), 0), dtype=torch.bfloat16)
    else:
        clip_bank = dataset.clip_bank[clip_src]
        track_bank = dataset.track_bank[track_src]
    rels_label = None
    if has_ctx and track_models:
        rels_label = np.concatenate([np.asarray(r["rels_label"]).reshape(-1) for r in records])
    elif has_ctx:
        rels_label = np.array([r["rels_label"] for r in records])
    gt = np.stack([r["gt_tracks"] for r in records]) if track_models else np.zeros((B, 2), dtype=np.int64)
    mw = np.stack([r["multilab_weights"] for r in records]) if "multilab_weights" in records[0] else \
        np.ones((B, dataset.n_classes))
    extras = {k: np.array([r[k] for r in records]) for k in ("just_zeros", "n_names", "hash_rel") if k in records[0]}
    pb = PackedBatch.from_tables(
        clip_bank, track_bank, n_clip_ints, n_track_ints, cand_off, apply(cand_t),
        ctx_off, apply(ctx_t) if has_ctx else None, [r["labels"] for r in records], rels_label, gt, mw,
        n_slots=dataset._max_n_tripl if track_models else 1,
        n_ctx_slots=records[0]["n_ctx_slots"], extras=extras)
    pb.extras["bank_rows"] = (clip_src.astype(np.int32), track_src.astype(np.int32))
    return _with_soft_pos(pb, records, dataset)


STAGE_TRACE = None      # measurement aid (bench.py, LIREC_BENCH_DEBUG): a list that ResidentBanks.stage appends its phase times to


class ResidentBanks:
    """The split's pooled feature banks resident in HBM (bf16; the whole MovieGraphs pooled table is
    < 1 GB).  A step's host->device traffic is then the packed batch's integer tables plus two row-index
    lists; the per-batch banks the kernels read are gathered on the device (`lirec_gather_rows`)."""

    def __init__(self, dataset=None, device="cuda", clip=None, track=None):
        from lirec_b200 import _ext
        _ext.require_device(torch.device(device))
        self.device = torch.device(device)
        if dataset is not None:
            clip, track = torch.from_numpy(dataset.clip_bank), torch.from_numpy(dataset.track_bank)
        self.clip = clip.to(torch.bfloat16).to(self.device)
        self.track = track.to(torch.bfloat16).to(self.device)

    def _rows(self, which, n, dim):
        """[n, dim] bf16 on the device, cut from an allocation of this bank's high-water capacity: every batch then
        asks the caching allocator for the SAME size, which it serves from its cache — batch banks whose size follows
        the batch (13.4 k +- 1 % clip rows, 28 k track rows: 75 + 115 MB) sooner or later exceed every cached block
        and fall through to cudaMalloc, a multi-millisecond call behind the GPU's queue (seen as one 14 ms wait
        for a batch per ~100 steps)."""
        caps = self.__dict__.setdefault("_caps", {})
        if n > caps.get(which, 0):
            caps[which] = -(-int(n * 1.06 + 64) // 512) * 512
        # The allocator's pools are per stream and only as deep as the number of blocks that were ever pending at
        # once: whenever the consumer falls one batch further behind than before, the pool grows by a cudaMalloc —
        # measured as sporadic 14-34 ms stalls of `stage` (bench.py, LIREC_BENCH_DEBUG) during a process's first
        # seconds.  The first request of a (bank, capacity, stream) therefore fills the pool to its working depth.
        key = (which, caps[which], torch.cuda.current_stream(self.device).cuda_stream)
        warmed = self.__dict__.setdefault("_warmed", set())
        if key not in warmed:
            warmed.add(key)
            hold = [torch.empty(caps[which], dim, dtype=torch.bfloat16, device=self.device)
                    for _ in range(6)]
            del hold
        return torch.empty(caps[which], dim, dtype=torch.bfloat16, device=self.device)[:n]

    def stage(self, pb, non_blocking=True):
        """Host PackedBatch from `collate_indexed` -> device PackedBatch whose banks were gathered on the GPU."""
        from lirec_b200 import ops
        trace = STAGE_TRACE
        if trace is not None:
            import time as _t
            t0 = _t.perf_counter()
        dev = pb.to_device(self.device, non_blocking=non_blocking, banks=False)
        if trace is not None:
            t1 = _t.perf_counter()
        src = getattr(pb, "_src_layout", None)
        if src is not None:                                     # the row lists crossed PCIe inside the arena
            idx_c = dev._arena_dev[src[0]:src[0] + src[1]]
            idx_t = dev._arena_dev[src[2]:src[2] + src[3]]
        else:
            if not hasattr(pb, "_bank_rows_pinned"):
                pb._pin_bank_rows()
            idx_c = pb._bank_rows_pinned[0].to(self.device, non_blocking=non_blocking)
            idx_t = pb._bank_rows_pinned[1].to(self.device, non_blocking=non_blocking)
        out_c = self._rows("clip", idx_c.numel(), self.clip.shape[1])
        out_t = self._rows("track", idx_t.numel(), self.track.shape[1])
        if trace is not None:
            t2 = _t.perf_counter()
        dev.clip_bank = ops.gather_rows(self.clip, idx_c, out=out_c)
        dev.track_bank = ops.gather_rows(self.track, idx_t, out=out_t)
        dev._bank_idx = (idx_c, idx_t)
        if trace is not None:                      # (table copies, bank allocations, gather launches) in seconds
            trace.append((t1 - t0, t2 - t1, _t.perf_counter() - t2))
        return dev

    @staticmethod
    def h2d_bytes(pb):
        """Bytes `stage` copies host -> device for this batch (integer tables, multilab, two row lists)."""
        c_rows, t_rows = pb.extras["bank_rows"]
        return int(pb.multilab.numel() + 4 * (sum(v.size for v in pb.tables.values()) + len(c_rows) + len(t_rows)))
