"""BERT token features of one scene on the GPU: the tokens of the subtitle lines that overlap a clip's
time span, max-pooled (reference: text_utils/text_features.py:140-178 followed by np.max in
mixed_utils/mixed_features.py:61).

The reference walks the subtitle lines on the host, concatenates the token-index ranges of every line
whose time span overlaps the clip (`Time.includes`, :24-31), indexes the `[n_tokens, 768]` feature array
with that list and takes np.max; a clip without dialog gets a zero row (:171-178).  Here the token
features are uploaded once, the index lists of as many clips as are queued are concatenated, and ONE
gathered segmented-max launch (`lirec_seg_reduce_f32` with a row index) writes the pooled bf16 rows.
WebVTT / token file parsing stays outside: the constructor takes the arrays.
"""
import numpy as np
import torch

from lirec_b200 import ops


class Time:
    """Time span of one subtitle line (reference :19-36)."""

    def __init__(self, start, end):
        self.start, self.end = start, end

    def includes(self, start, end):
        return (self.start <= start <= self.end) or (self.start <= end <= self.end) or \
            (start <= self.start and end >= self.end)

    def include_point(self, point):
        return self.start <= point <= self.end


class TextFeatures:
    """features: float32 [n_tokens, dim]; times: list of Time (or (start, end)); time_idx2token_range: the
    token indices of every subtitle line (reference `_tokens_range`, :91-104)."""

    def __init__(self, features, times, time_idx2token_range, device="cuda"):
        self.device = torch.device(device)
        self.features = torch.from_numpy(np.ascontiguousarray(features, dtype=np.float32)).to(self.device)
        self.dim = int(features.shape[1])
        self.times = [t if isinstance(t, Time) else Time(*t) for t in times]
        self.time_idx2token_range = [list(r) for r in time_idx2token_range]

    def tokens_range(self, time_node):
        """Token indices of a clip, in the reference's order (lines may repeat tokens; max is idempotent)."""
        out = []
        for i, t in enumerate(self.times):
            if t.includes(time_node["start"], time_node["end"]):
                out += self.time_idx2token_range[i]
        return out

    def _run(self, index_lists, out_f32=None, out_bf16=None):
        off = np.zeros(len(index_lists) + 1, dtype=np.int32)
        np.cumsum([len(x) for x in index_lists], out=off[1:])
        flat = np.concatenate([np.asarray(x, dtype=np.int32) for x in index_lists]) if off[-1] else \
            np.zeros(1, dtype=np.int32)
        idx = torch.from_numpy(flat.astype(np.int32)).to(self.device, non_blocking=True)
        offd = torch.from_numpy(off).to(self.device, non_blocking=True)
        if out_f32 is None and out_bf16 is None:
            out_f32 = torch.empty(len(index_lists), self.dim, dtype=torch.float32, device=self.device)
        ops.seg_reduce(self.features, offd, "max", out_f32=out_f32, out_bf16=out_bf16, row_idx=idx)
        return out_f32 if out_f32 is not None else out_bf16

    def get_features_by_time(self, time_node):
        """Token rows of the clip, fp32 [n, dim] — or one zero row when no subtitle line overlaps it."""
        rng = self.tokens_range(time_node)
        if not rng:
            return torch.zeros(1, self.dim, dtype=torch.float32, device=self.device)
        return self._run([[i] for i in rng])

    def pool(self, time_nodes, out_bf16=None):
        """max over the tokens of every clip in `time_nodes`: one launch, zero rows for clips without dialog."""
        return self._run([self.tokens_range(tn) for tn in time_nodes], out_bf16=out_bf16)
