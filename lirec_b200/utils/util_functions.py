"""The few helpers of the reference's utils/util_functions.py that the loops touch: `Averaging`
(:23-38), `Relationship` (:53-75, the per-pair relationship timeline the dataloader queries),
`dir_check`, `load_model` / `load_optimizer` (:274-291).  Annotation parsing (the other ~550 lines)
is dataset plumbing outside the hot path and is not reimplemented."""
import os
from collections import defaultdict

import numpy as np
import torch

from lirec_b200.utils.arg_pars import opt


class Averaging(object):
    def __init__(self):
        self.reset()

    def reset(self):
        self.val = self.avg = self.sum = 0.0
        self.count = 0

    def update(self, val, n=1):
        self.val = val
        self.sum += val * n
        self.count += n
        self.avg = self.sum / self.count if self.count else 0.0


class Relationship:
    """Relationship of one ordered character pair over the scenes of a movie (reference:
    utils/util_functions.py:53-75).  `rels_name` is the most recent relationship; appending a scene
    with name None extends the current relationship to that scene.  `scene2rel` draws among the
    names recorded for a scene with the GLOBAL numpy RNG, like the reference, so seeded runs agree."""

    def __init__(self, rels_name, scene_idx):
        self.rels_name = rels_name
        self.scenes = {scene_idx}
        self.rel2scenes = defaultdict(list)
        self._scene2rel = defaultdict(list)
        self.rel2scenes[rels_name].append(scene_idx)
        self._scene2rel[scene_idx].append(rels_name)

    def append_scene(self, rels_name, scene_idx):
        if rels_name is not None and rels_name != self.rels_name:
            self.rels_name = rels_name
        if scene_idx in self.scenes and self.rels_name in self._scene2rel[scene_idx]:
            return
        self.scenes.add(scene_idx)
        self.rel2scenes[self.rels_name].append(scene_idx)
        self._scene2rel[scene_idx].append(self.rels_name)

    def scene2rel(self, scene_idx):
        names = self._scene2rel.get(scene_idx)
        if names:
            # np.random.choice(names) (reference :71-73) = names[randint(0, len)] on the same global RNG
            # stream (checked draw for draw), without building a string array per call; a single name
            # consumes no random number at all (numpy returns the lower bound for an empty range)
            return names[0] if len(names) == 1 else names[np.random.randint(0, len(names))]
        return "None"


def dir_check(path):
    os.makedirs(path, exist_ok=True)


def load_model(name=""):
    """state_dict of a checkpoint in the reference's format {'epoch','state_dict','optimizer'}."""
    ckpt = torch.load(opt.resume_str, map_location="cpu")
    print("loaded model %s (epoch %s)" % (opt.resume_str, ckpt.get("epoch")))
    return ckpt["state_dict"]


def load_optimizer():
    return torch.load(opt.resume_str, map_location="cpu")["optimizer"]


def load_ema():
    """The checkpoint's weight average (mlp.model.FlatEMA.state_dict(), saved under --ema_decay), or None."""
    return torch.load(opt.resume_str, map_location="cpu").get("ema")
