"""CPU restatement of the per-viewer transition entropy (Engine.user_transitions / vet_user_transitions), test
infrastructure only.

For user u and tile count k the pairs are the (p, c) tile pairs of the frames f with u present in f and f+1 -- the
pairs of transition_pairs restricted to u, in frame order -- and per_k[k, u] is, by definition,
transition_entropy_textbook (EU:321-327 normalisation) of them.  A user without any pair gets NaN instead of the
ZeroDivisionError of the textbook mode.  entropy[u] is the sequential mean over k (SA:151-156 order).
tests/test_user_transitions_host.py pins it to transition_analyzer(mode="textbook").
"""
from __future__ import annotations

from typing import Optional, Sequence

import numpy as np

from . import vet_oracle as orc
from .vet_transition_counts_oracle import transition_pairs


def user_transitions(packed: np.ndarray, W: int, H: int, tile_counts: Sequence[int],
                     centres: Optional[Sequence[np.ndarray]] = None):
    """packed[F,U,3] = (time, 2dmu, 2dmv), NaN 2dmu/2dmv = missing.  Returns dict(entropy[U], per_k[K,U],
    pairs[U] int64)."""
    packed = np.asarray(packed)
    F, U = packed.shape[0], packed.shape[1]
    Ts = [len(c) for c in centres] if centres is not None else [orc.lattice_size(n) for n in tile_counts]
    K = len(Ts)
    pairs = transition_pairs(packed, W, H, tile_counts, centres)
    # transition_pairs lists the pairs frame by frame, users in index order inside a frame: the user of every pair
    _, _, valid = orc.decode(packed[..., 1], packed[..., 2], W, H)
    users = np.nonzero(valid[:-1] & valid[1:])[1] if F > 1 else np.zeros(0, dtype=np.int64)
    order = np.argsort(users, kind="stable")           # per user, its pairs in frame order
    bounds = np.searchsorted(users[order], np.arange(U + 1))
    per_k = np.full((K, U), np.nan)
    for k, ((p, c), T) in enumerate(zip(pairs, Ts)):
        p, c = p[order], c[order]
        for u in range(U):
            b, e = bounds[u], bounds[u + 1]
            if e > b:
                per_k[k, u] = orc.transition_entropy_textbook(p[b:e], c[b:e], T)
    ent = np.zeros(U)
    for k in range(K):
        ent = ent + per_k[k]
    return dict(entropy=ent / K, per_k=per_k, pairs=np.diff(bounds).astype(np.int64))
