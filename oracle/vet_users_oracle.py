"""CPU restatement of the per-viewer exploration entropy (Engine.users / vet_users_*), test infrastructure only.

compute_spatial_entropy (EU:147-211) applied to the present samples of ONE user over the frames of the video instead
of one frame's samples over the users, averaged over the tile counts in the order of SA:142-156.  A user without any
present sample gets entropy NaN, frames 0 and a zero histogram row (the reference would raise "Empty vector
dictionary" for the empty dict).  Built on the vectorised functions of vet_oracle, which are pinned to the live
reference; tests/test_users_host.py pins `user_analyzer` to `compute_spatial_entropy_literal`.
"""
from __future__ import annotations

from typing import Optional, Sequence

import numpy as np

from . import vet_oracle as orc


def user_analyzer(packed: np.ndarray, W: int, H: int, tile_counts: Sequence[int], fov_angle=120.0, use_weight=True,
                  power_factor=2.0, centres: Optional[Sequence[np.ndarray]] = None):
    """packed[F,U,3] = (time, 2dmu, 2dmv), NaN 2dmu/2dmv = missing.  Returns dict(entropy[U], per_k[K,U],
    hist0[U,T0], frames[U] int64).  `centres` optionally replaces the Fibonacci lattices by arbitrary tile centres."""
    packed = np.asarray(packed)
    F, U, _ = packed.shape
    px, py, valid = orc.decode(packed[..., 1], packed[..., 2], W, H)
    cv = orc.cell_vectors(W, H)
    lats = [np.asarray(c, dtype=np.float64) for c in centres] if centres is not None else [orc.lattice(n) for n in tile_counts]
    K = len(lats)
    per_k = np.full((K, U), np.nan)
    hist0 = np.zeros((U, len(lats[0])))
    frames = valid.sum(axis=0).astype(np.int64)
    for u in range(U):
        ok = valid[:, u]
        if not ok.any():
            continue
        vecs = cv[py[ok, u], px[ok, u]]
        for k, c in enumerate(lats):
            e, hist, _ = orc.spatial_entropy(vecs, c, fov_angle, use_weight, power_factor)
            per_k[k, u] = e
            if k == 0:
                hist0[u] = hist
    ent = np.zeros(U)
    for k in range(K):  # SA:151-156: sequential sum, then / K
        ent = ent + per_k[k]
    return dict(entropy=ent / K, per_k=per_k, hist0=hist0, frames=frames)
