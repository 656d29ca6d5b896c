"""CPU tests of the tile transition matrix: the restatement `transition_counts` equals transition_entropy_textbook on
the concatenated pairs0 rows of transition_analyzer(mode="textbook"), its counts add up over batches that overlap by
one frame, and TransitionEntropyAnalyzer.compute_transition_counts batches the host array that way into the accumulator
it is given -- here a numpy stand-in for the engine, so no GPU is needed."""
import numpy as np
import pytest

from oracle import vet_oracle as orc
from oracle.vet_transition_counts_oracle import transition_counts

torch = pytest.importorskip("torch")


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
def test_pooled_entropy_is_textbook_entropy_of_concatenated_pairs(tcs):
    W, H = 100, 200
    p = _walk(15, 40, 3, 0.15)
    ref = transition_counts(p, W, H, tcs)
    ta = orc.transition_analyzer(p, W, H, tcs[:1], mode="textbook")
    pairs0 = ta["pairs0"].reshape(-1, 2)
    pairs0 = pairs0[pairs0[:, 0] != orc.MISSING].astype(np.int64)
    T0 = orc.lattice_size(tcs[0])
    assert ref["pairs"] == len(pairs0)
    assert np.array_equal(ref["counts"][0], np.bincount(pairs0[:, 0] * T0 + pairs0[:, 1], minlength=T0 * T0).reshape(T0, T0))
    assert np.array_equal(ref["counts"][0].sum(1), ta["prev_count0"].sum(0))
    assert ref["per_k"][0] == orc.transition_entropy_textbook(pairs0[:, 0], pairs0[:, 1], T0)
    for k, n in enumerate(tcs):
        assert ref["counts"][k].sum() == ref["pairs"]
        assert 0.0 <= ref["per_k"][k] <= 1.0
    np.testing.assert_allclose(ref["entropy"], np.mean(ref["per_k"]), rtol=1e-15)


def test_counts_add_up_over_overlapping_batches():
    W, H, tcs = 100, 200, [20, 200]
    p = _walk(30, 25, 5, 0.1)
    whole = transition_counts(p, W, H, tcs)
    for cuts in ([0, 1, 3, 20, 30], [0, 17, 30], [0, 29, 30]):
        acc = [np.zeros_like(c) for c in whole["counts"]]
        for b, e in zip(cuts[:-1], cuts[1:]):
            part = transition_counts(p[max(b - 1, 0):e], W, H, tcs)   # the halo frame b - 1
            for a, c in zip(acc, part["counts"]):
                a += c
        for a, c in zip(acc, whole["counts"]):
            assert np.array_equal(a, c)


def test_no_pair_gives_nan():
    p = _walk(1, 5, 1, 0.0)
    r = transition_counts(p, 100, 200, [20])
    assert r["pairs"] == 0 and not r["counts"][0].any() and np.isnan(r["entropy"])
    p = _walk(4, 3, 1, 0.0)
    p[::2, :, 1] = np.nan                # present in alternate frames only: no common user in any pair
    assert np.isnan(transition_counts(p, 100, 200, [20])["entropy"])
    one = _walk(2, 1, 1, 0.0)            # N = 1: 0 / log2(1)
    assert np.isnan(transition_counts(one, 100, 200, [20])["entropy"])


class _StubEngine:
    """Accumulates the restatement's counts in numpy and records the frame batches it is given."""

    def __init__(self, tcs):
        self.device = torch.device("cpu")
        self.tcs = tcs
        self.T = [orc.lattice_size(n) for n in tcs]
        self.batches = []

    def transition_counts_accumulator(self):
        return torch.zeros(sum(t * t for t in self.T), dtype=torch.int64)

    def transition_counts_accumulate(self, packed, acc):
        p = packed.numpy()
        self.batches.append(p.shape[0])
        acc += torch.from_numpy(np.concatenate([c.ravel() for c in transition_counts(p, 100, 200, self.tcs)["counts"]]))

    def transition_counts_finish(self, acc):
        from viewport_entropy_toolkit_b200 import TransitionCountsResult
        counts, off = [], 0
        for t in self.T:
            counts.append(acc[off:off + t * t].view(t, t))
            off += t * t
        n = int(counts[0].sum())
        per_k = [orc.transition_entropy_textbook(*np.divmod(np.repeat(np.arange(t * t), c.reshape(-1).numpy()), t), t)
                 for t, c in zip(self.T, counts)]
        return TransitionCountsResult(counts=counts, entropy=torch.tensor(np.mean(per_k), dtype=torch.float64),
                                      per_k=torch.tensor(per_k, dtype=torch.float64), pairs=n)

    def raise_for_flags(self):
        pass


def test_compute_transition_counts_batches_with_a_halo_frame(tmp_path):
    import viewport_entropy_toolkit_b200 as vet
    cfg = vet.AnalyzerConfig(tile_counts=[20, 50], output_dir=tmp_path)
    ta = vet.TransitionEntropyAnalyzer(cfg)
    p = _walk(10, 4, 7, 0.1).astype(np.float32)
    ta.load_packed(p)
    ta._engine = stub = _StubEngine([20, 50])
    out = ta.compute_transition_counts(batch_bytes=4 * 3 * 4 * 4)   # 4 frames per batch, one shared with the next
    assert stub.batches == [4, 4, 4]                                  # frames 0-3, 3-6, 6-9
    ref = transition_counts(p, 100, 200, [20, 50])
    assert out["pairs"] == ref["pairs"]
    for c, rc in zip(out["counts"], ref["counts"]):
        assert isinstance(c, np.ndarray) and c.dtype == np.int64
        assert np.array_equal(c, rc)
    np.testing.assert_allclose(out["per_k"], ref["per_k"], rtol=1e-12)
    np.testing.assert_allclose(out["entropy"], ref["entropy"], rtol=1e-12)
