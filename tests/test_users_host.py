"""CPU tests of the per-viewer exploration entropy: the vectorised restatement `user_analyzer` equals
compute_spatial_entropy_literal called on each user's {frame: vector} dict, and
SpatialEntropyAnalyzer.compute_user_entropy builds its DataFrame (identifiers, columns, lazy tile-weight dicts) from
the accumulator it is given -- here a numpy stand-in for the engine, so no GPU is needed."""
import numpy as np
import pytest

from oracle import vet_oracle as orc
from oracle.vet_users_oracle import user_analyzer

torch = pytest.importorskip("torch")


def _packed(F, U, seed, missing):
    rng = np.random.default_rng(seed)
    p = np.stack([np.broadcast_to(np.arange(F)[:, None] * 0.1, (F, U)), rng.uniform(0, 1, (F, U)),
                  rng.uniform(0.2, 0.6, (F, U))], -1)
    p[rng.uniform(size=(F, U)) < missing, 1] = np.nan
    return p


@pytest.mark.parametrize("use_w,fov", [(True, 90.0), (True, 120.0), (False, 90.0)])
def test_user_analyzer_equals_literal_per_user(use_w, fov):
    W, H, tcs = 100, 200, [20, 50]
    p = _packed(12, 6, 2, 0.2)
    p[:, 5, 1] = np.nan            # no sample
    p[1:, 4, 1] = np.nan           # one sample
    ref = user_analyzer(p, W, H, tcs, fov, use_w, 2.0)
    vecs, ok = orc.decode_vectors(p[..., 1], p[..., 2], W, H)
    for u in range(p.shape[1]):
        d = {str(f): vecs[f, u].tolist() for f in range(p.shape[0]) if ok[f, u]}
        assert ref["frames"][u] == len(d)
        if not d:
            assert np.isnan(ref["entropy"][u]) and not ref["hist0"][u].any()
            with pytest.raises(orc.OracleValidationError):
                orc.compute_spatial_entropy_literal(d, orc.lattice(tcs[0]), fov, use_w, 2.0)
            continue
        per_k = []
        for k, n in enumerate(tcs):
            e, wpt, _ = orc.compute_spatial_entropy_literal(d, orc.lattice(n), fov, use_w, 2.0)
            per_k.append(e)
            np.testing.assert_allclose(ref["per_k"][k, u], e, rtol=1e-12, atol=0, equal_nan=True)
            if k == 0:
                dense = np.zeros(len(orc.lattice(n)))
                for t, w in wpt.items():
                    dense[t] = w
                np.testing.assert_allclose(ref["hist0"][u], dense, rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(ref["entropy"][u], (0.0 + per_k[0] + per_k[1]) / 2, rtol=1e-12, atol=0, equal_nan=True)
    if not use_w:
        assert np.isnan(ref["entropy"][4])


class _StubEngine:
    """Accumulates the dense tile histograms of the restatement in numpy (exact for the unweighted counts used here)."""

    def __init__(self, tcs):
        self.device = torch.device("cpu")
        self.tcs = tcs
        self.T = [orc.lattice_size(n) for n in tcs]
        self.flags = 0
        self.batches = []

    def user_accumulator(self, U):
        return torch.zeros((U, sum(self.T) + 1), dtype=torch.int64)

    def users_accumulate(self, packed, acc, total_frames):
        p = packed.numpy()
        self.batches.append(p.shape[0])
        _, _, valid = orc.decode(p[..., 1], p[..., 2], 100, 200)
        vecs, _ = orc.decode_vectors(p[..., 1], p[..., 2], 100, 200)
        off = 0
        for n, T in zip(self.tcs, self.T):
            c = orc.lattice(n)
            for f, u in zip(*np.nonzero(valid)):
                acc[u, off + orc.nearest_tile(vecs[f, u][None], c)[0]] += 1
            off += T
        acc[:, -1] += torch.from_numpy(valid.sum(0))

    def users_finish(self, acc, total_frames, want_per_k=True, want_hist0=True):
        from viewport_entropy_toolkit_b200 import UserResult
        a = acc.numpy().astype(np.float64)
        ent = np.array([np.nan if r[-1] == 0 else np.mean([orc.entropy_from_hist(r[:self.T[0]], self.T[0], False)])
                        for r in a])
        return UserResult(entropy=torch.from_numpy(ent), per_k=None, hist0=torch.from_numpy(a[:, :self.T[0]]),
                          frames=acc[:, -1].to(torch.int32))

    def raise_for_flags(self):
        pass


def test_compute_user_entropy_dataframe_from_a_stub_accumulator(tmp_path):
    import viewport_entropy_toolkit_b200 as vet
    cfg = vet.AnalyzerConfig(tile_counts=[20], output_dir=tmp_path,
                             entropy_config=vet.EntropyConfig(use_weight_distribution=False))
    sa = vet.SpatialEntropyAnalyzer(cfg)
    p = _packed(9, 4, 7, 0.0).astype(np.float32)
    p[:, 3, 1] = np.nan
    sa.load_packed(p, ["a", "b", "c", "d"])
    sa._engine = stub = _StubEngine([20])
    df = sa.compute_user_entropy(batch_bytes=4 * 3 * 4 * 4)   # 4 frames per batch
    assert stub.batches == [4, 4, 1]
    assert list(df.columns) == ["identifier", "frames", "entropy", "tile_weights"]
    assert list(df["identifier"]) == ["a", "b", "c", "d"]
    assert list(df["frames"]) == [9, 9, 9, 0]
    ref = user_analyzer(p, 100, 200, [20], use_weight=False)
    np.testing.assert_allclose(df["entropy"].to_numpy(), ref["entropy"], rtol=1e-12, equal_nan=True)
    centres = sa._fibonacci_vectors[20]
    for u in range(3):
        tw = df["tile_weights"][u]
        assert isinstance(tw, vet.analyzers.LazyRowDict)
        assert dict(tw) == {centres[i]: float(ref["hist0"][u, i]) for i in np.flatnonzero(ref["hist0"][u])}
        assert sum(tw.values()) == 9
    assert len(df["tile_weights"][3]) == 0
