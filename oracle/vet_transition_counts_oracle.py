"""CPU restatement of the tile transition matrix (Engine.transition_counts / vet_transition_counts_*), test
infrastructure only.

For tile count k, counts_k[p, c] = the number of (frame pair (f, f+1), user) combinations with the user present in
both frames (the common users of EU:271-276), nearest tile p of tile count k in frame f and c in frame f+1.  The pooled
conditional entropy is, by definition, transition_entropy_textbook (EU:321-327 normalisation) of the (p, c) pairs of
all frame pairs concatenated; no pair at all gives NaN instead of the ZeroDivisionError of the textbook mode.  Built on
decode, cell_luts / nearest_tile and transition_entropy_textbook of vet_oracle; tests/test_transition_counts_host.py
pins it to transition_analyzer(mode="textbook").
"""
from __future__ import annotations

from typing import Optional, Sequence

import numpy as np

from . import vet_oracle as orc


def transition_pairs(packed: np.ndarray, W: int, H: int, tile_counts: Sequence[int],
                     centres: Optional[Sequence[np.ndarray]] = None):
    """Per tile count the (p, c) tile pairs of every frame pair and common user, frame pairs in order, users in
    index order inside a pair: a list of (p[N], c[N]) int64 arrays."""
    packed = np.asarray(packed)
    F = packed.shape[0]
    px, py, valid = orc.decode(packed[..., 1], packed[..., 2], W, H)
    cell = py * (W + 1) + px
    if centres is not None:
        cv = orc.cell_vectors(W, H).reshape(-1, 3)
        luts = [orc.nearest_tile(cv, np.asarray(c, dtype=np.float64)) for c in centres]
    else:
        luts = orc.cell_luts(W, H, tile_counts)
    both = valid[:-1] & valid[1:] if F > 1 else np.zeros((0,) + valid.shape[1:], dtype=bool)
    prev, cur = cell[:-1][both], cell[1:][both]
    return [(lut[prev].astype(np.int64), lut[cur].astype(np.int64)) for lut in luts]


def transition_counts(packed: np.ndarray, W: int, H: int, tile_counts: Sequence[int],
                      centres: Optional[Sequence[np.ndarray]] = None):
    """packed[F,U,3] = (time, 2dmu, 2dmv), NaN 2dmu/2dmv = missing.  Returns dict(counts=[[T_k, T_k] int64],
    entropy (mean over k, SA:151-156 order), per_k[K], pairs=N)."""
    pairs = transition_pairs(packed, W, H, tile_counts, centres)
    Ts = [len(c) for c in centres] if centres is not None else [orc.lattice_size(n) for n in tile_counts]
    counts, per_k = [], []
    for (p, c), T in zip(pairs, Ts):
        counts.append(np.bincount(p * T + c, minlength=T * T).reshape(T, T).astype(np.int64))
        per_k.append(orc.transition_entropy_textbook(p, c, T) if len(p) else np.nan)
    ent = 0.0
    for e in per_k:
        ent = ent + e
    return dict(counts=counts, entropy=ent / len(per_k), per_k=np.array(per_k), pairs=len(pairs[0][0]))
