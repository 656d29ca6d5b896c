"""CPU tests of the per-viewer transition entropy: the restatement `user_transitions` equals
transition_entropy_textbook of each user's column of transition_analyzer(mode="textbook")["pairs0"], its NaN cases, and
TransitionEntropyAnalyzer.compute_user_transition_entropy uploads the host array in blocks of user columns -- here into
a numpy stand-in for the engine, so no GPU is needed."""
import re
from pathlib import Path

import numpy as np
import pytest

from oracle import vet_oracle as orc
from oracle.vet_user_transitions_oracle import user_transitions

torch = pytest.importorskip("torch")

ROOT = Path(__file__).resolve().parents[1]


def _walk(F, U, seed, missing):
    rng = np.random.default_rng(seed)
    mu = np.clip(rng.normal(0.5, 0.2, U), 0, 1)[None] + np.cumsum(rng.normal(0, 0.05, (F, U)), 0)
    mv = np.clip(rng.normal(0.5, 0.15, U), 0, 1)[None] + np.cumsum(rng.normal(0, 0.03, (F, U)), 0)
    for a in (mu, mv):
        np.abs(a, out=a)
        a[a > 1] = 2 - a[a > 1]
        np.clip(a, 0, 1, out=a)
    p = np.stack([np.broadcast_to(np.arange(F)[:, None] * 0.1, (F, U)), mu, mv], -1)
    p[rng.uniform(size=(F, U)) < missing, 1] = np.nan
    return p


@pytest.mark.parametrize("tcs", [[20], [20, 50, 200]])
def test_user_entropy_is_textbook_entropy_of_the_users_pairs0_column(tcs):
    W, H = 100, 200
    p = _walk(25, 12, 3, 0.15)
    ref = user_transitions(p, W, H, tcs)
    for k, n in enumerate(tcs):
        pairs0 = orc.transition_analyzer(p, W, H, [n], mode="textbook")["pairs0"]   # [F-1, U, 2]
        T = orc.lattice_size(n)
        for u in range(p.shape[1]):
            col = pairs0[:, u]
            col = col[col[:, 0] != orc.MISSING].astype(np.int64)
            assert ref["pairs"][u] == len(col)
            if len(col):
                assert ref["per_k"][k, u] == orc.transition_entropy_textbook(col[:, 0], col[:, 1], T)
            else:
                assert np.isnan(ref["per_k"][k, u])
    ent = np.zeros(p.shape[1])
    for k in range(len(tcs)):
        ent = ent + ref["per_k"][k]
    assert np.array_equal(ref["entropy"], ent / len(tcs), equal_nan=True)


def test_nan_cases():
    p = _walk(12, 5, 1, 0.0)
    p[::2, 0, 1] = np.nan                 # present in alternate frames only: N = 0
    p[:, 1, 2] = np.nan                   # never present
    p[2:, 2, 1] = np.nan                  # present in frames 0 and 1 only: N = 1, 0 / log2(1)
    r = user_transitions(p, 100, 200, [20, 200])
    assert list(r["pairs"][:3]) == [0, 0, 1]
    assert np.isnan(r["per_k"][:, :3]).all() and np.isnan(r["entropy"][:3]).all()
    assert (r["pairs"][3:] == 11).all() and np.isfinite(r["entropy"][3:]).all()
    one = user_transitions(p, 100, 200, [1, 20], centres=[np.array([[0.0, 0.0, 1.0]]), orc.lattice(20)])
    assert np.isnan(one["per_k"][0]).all()                         # T = 1: log2 T = 0
    assert np.isnan(one["entropy"]).all()                          # the NaN of k = 0 propagates into the mean
    assert np.array_equal(one["per_k"][1], r["per_k"][0], equal_nan=True)
    empty = user_transitions(p[:1], 100, 200, [20])                # one frame: no pair at all
    assert (empty["pairs"] == 0).all() and np.isnan(empty["entropy"]).all()


def test_smem_record_capacity_matches_the_header():
    from viewport_entropy_toolkit_b200 import _native
    header = (ROOT / "include" / "vet_b200.h").read_text()
    assert int(re.search(r"#define VET_UT_SMEM_RECORDS (\d+)", header).group(1)) == _native.UT_SMEM_RECORDS


class _StubEngine:
    """Computes the restatement per user block and records the blocks it is given."""

    def __init__(self, tcs):
        self.device = torch.device("cpu")
        self.tcs = tcs
        self.blocks = []

    def user_transitions(self, packed, want_per_k=True):
        from viewport_entropy_toolkit_b200 import UserTransitionResult
        p = packed.numpy()
        self.blocks.append(p.shape[:2])
        r = user_transitions(p, 100, 200, self.tcs)
        return UserTransitionResult(entropy=torch.from_numpy(r["entropy"]),
                                    per_k=torch.from_numpy(r["per_k"]) if want_per_k else None,
                                    pairs=torch.from_numpy(r["pairs"]).to(torch.int32))

    def raise_for_flags(self):
        pass


def test_compute_user_transition_entropy_uploads_user_column_blocks(tmp_path):
    import viewport_entropy_toolkit_b200 as vet
    cfg = vet.AnalyzerConfig(tile_counts=[20, 50], output_dir=tmp_path)
    ta = vet.TransitionEntropyAnalyzer(cfg)
    F, U = 10, 11
    p = _walk(F, U, 7, 0.1).astype(np.float32)
    p[::2, 4, 1] = np.nan
    ids = [f"viewer{u}" for u in range(U)]
    ta.load_packed(p, ids)
    ta._engine = stub = _StubEngine([20, 50])
    out = ta.compute_user_transition_entropy(batch_bytes=F * 3 * 4 * 4)   # 4 users per block
    assert stub.blocks == [(F, 4), (F, 4), (F, 3)]
    ref = user_transitions(p, 100, 200, [20, 50])
    assert list(out.columns) == ["identifier", "pairs", "entropy"]
    assert list(out["identifier"]) == ids
    assert np.array_equal(out["pairs"].to_numpy(), ref["pairs"])
    assert np.array_equal(out["entropy"].to_numpy(), ref["entropy"], equal_nan=True)
    assert np.isnan(out["entropy"][4])
