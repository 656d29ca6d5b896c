"""Tile transition matrix (Engine.transition_counts / vet_transition_counts_accumulate / vet_transition_counts_finish)
against the CPU restatement: counts exact, pooled conditional entropies 1e-9 relative; the same bits on a rerun and
over overlapping batches; the counts of tile count 0 equal those of the existing transition kernels' pairs0 output."""
import numpy as np
import pytest

from oracle.vet_transition_counts_oracle import transition_counts

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

DEFAULT5 = [20, 50, 100, 250, 1000]


@pytest.fixture(scope="module")
def vet():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import __graft_entry__ as ge
    ge.build()
    import viewport_entropy_toolkit_b200 as pkg
    return pkg


def _engine(vet, tcs, use_w=False, W=100, H=200, **kw):
    return vet.Engine(W, H, tcs, vet.EntropyConfig(fov_angle=90.0, use_weight_distribution=use_w, power_factor=2.0),
                      torch.device("cuda", 0), **kw)


def _walk(F, U, seed, missing=0.0, dtype=np.float32, step=0.03):
    rng = np.random.default_rng(seed)
    mu = np.clip(rng.normal(0.5, 0.2, U), 0, 1)[None] + np.cumsum(rng.normal(0, step, (F, U)), 0)
    mv = np.clip(rng.normal(0.5, 0.15, U), 0, 1)[None] + np.cumsum(rng.normal(0, step * 2 / 3, (F, U)), 0)
    for a in (mu, mv):
        np.abs(a, out=a)
        a[a > 1] = 2 - a[a > 1]
        np.clip(a, 0, 1, out=a)
    p = np.stack([np.broadcast_to(np.arange(F)[:, None] * 0.1, (F, U)), mu, mv], -1).astype(dtype)
    if missing:
        p[rng.uniform(size=(F, U)) < missing, 1] = np.nan
    return p


def _iid(F, U, seed, dtype=np.float32):
    rng = np.random.default_rng(seed)
    return np.stack([np.zeros((F, U)), rng.uniform(0, 1, (F, U)), rng.uniform(0, 1, (F, U))], -1).astype(dtype)


def _check(res, ref):
    assert res.pairs == ref["pairs"]
    assert len(res.counts) == len(ref["counts"])
    for c, rc in zip(res.counts, ref["counts"]):
        assert c.dtype == torch.int64 and tuple(c.shape) == rc.shape
        assert np.array_equal(c.cpu().numpy(), rc)
    np.testing.assert_allclose(res.per_k.cpu().numpy(), ref["per_k"], rtol=1e-9, atol=0, equal_nan=True)
    np.testing.assert_allclose(float(res.entropy), ref["entropy"], rtol=1e-9, atol=0, equal_nan=True)


def _appearing(F, U, seed):
    p = _walk(F, U, seed, 0.05)
    p[: F // 2, 0, 1] = np.nan        # joins halfway
    p[F // 3:, 1, 1] = np.nan         # leaves after a third
    p[::2, 2, 2] = np.nan             # present in every other frame: never in a pair
    p[:, 3, 1] = np.nan               # never present
    return p


CASES = [
    dict(id="200_f32", tcs=[200], make=lambda: _walk(97, 301, 11)),
    dict(id="default5_missing", tcs=DEFAULT5, make=lambda: _walk(41, 677, 12, 0.1)),
    dict(id="200_f64", tcs=[200], make=lambda: _walk(50, 333, 13, 0.05, np.float64)),
    dict(id="global_200x400", tcs=[20, 200], W=200, H=400, make=lambda: _walk(45, 517, 14, 0.1)),
    dict(id="tile_count_2000", tcs=[2000], make=lambda: _walk(30, 700, 15, 0.05)),
    dict(id="iid_odd_U", tcs=[20, 200], make=lambda: _iid(23, 1001, 16)),
    dict(id="appearing_users", tcs=[20, 200], make=lambda: _appearing(60, 259, 17)),
    dict(id="F2", tcs=[50, 200], make=lambda: _walk(2, 999, 18, 0.1)),
    dict(id="large_steps_500_1000", tcs=[200, 500, 1000], make=lambda: _walk(40, 2000, 19, 0.02, step=0.1)),
]


@pytest.mark.parametrize("c", CASES, ids=[c["id"] for c in CASES])
def test_transition_counts_match_reference(vet, c):
    W, H = c.get("W", 100), c.get("H", 200)
    eng = _engine(vet, c["tcs"], False, W, H)
    p = c["make"]()
    res = eng.transition_counts(torch.from_numpy(p).cuda())
    assert eng.poll_flags() == 0
    _check(res, transition_counts(p, W, H, c["tcs"]))
    eng.close()


def test_transition_counts_arbitrary_centres(vet):
    rng = np.random.default_rng(3)
    cs = [rng.normal(size=(37, 3)), rng.normal(size=(5, 3)), rng.normal(size=(1, 3))]
    eng = _engine(vet, [1, 2, 3], centres=cs)
    p = _walk(50, 611, 8, 0.1)
    res = eng.transition_counts(torch.from_numpy(p).cuda())
    assert eng.poll_flags() == 0
    ref = transition_counts(p, 100, 200, [1, 2, 3], centres=cs)
    _check(res, ref)
    assert np.isnan(float(res.per_k[2]))   # one tile: log2 T = 0


def test_single_frame_gives_zero_counts_and_nan(vet):
    eng = _engine(vet, [20, 200])
    res = eng.transition_counts(torch.from_numpy(_walk(1, 100, 2)).cuda())
    assert res.pairs == 0 and all(not c.any() for c in res.counts)
    assert np.isnan(float(res.entropy)) and np.isnan(res.per_k.cpu().numpy()).all()
    assert eng.poll_flags() == 0


def test_weighted_and_unweighted_handles_count_the_same(vet):
    p = torch.from_numpy(_walk(80, 1500, 4, 0.1)).cuda()
    a = _engine(vet, [20, 200], True).transition_counts(p)
    b = _engine(vet, [20, 200], False).transition_counts(p)
    for x, y in zip(a.counts, b.counts):
        assert torch.equal(x, y)
    assert torch.equal(a.per_k, b.per_k) and a.pairs == b.pairs


def _same(a, b):
    return (a.pairs == b.pairs and all(torch.equal(x, y) for x, y in zip(a.counts, b.counts))
            and torch.equal(a.per_k, b.per_k) and np.array_equal(a.entropy.cpu().numpy(), b.entropy.cpu().numpy()))


@pytest.mark.parametrize("tcs", [[200], DEFAULT5, [20, 200, 2000]], ids=["200", "default5", "with_global_2000"])
def test_bit_identical_on_rerun_and_over_overlapping_batches(vet, tcs):
    eng = _engine(vet, tcs)
    F, U = 301, 1001
    p = torch.from_numpy(_walk(F, U, 21, 0.1)).cuda()
    one = eng.transition_counts(p)
    assert _same(one, eng.transition_counts(p))
    acc = eng.transition_counts_accumulator()
    cuts = [0, 1, 3, 20, F]                       # batches of 1, 2, 17 and the rest of the pairs
    for b, e in zip(cuts[:-1], cuts[1:]):
        eng.transition_counts_accumulate(p[max(b - 1, 0):e], acc)
    assert _same(one, eng.transition_counts_finish(acc))
    # few users: the frame pairs are split over many CTA runs
    small = p[:, :5].contiguous()
    acc = eng.transition_counts_accumulator()
    for f in range(F - 1):
        eng.transition_counts_accumulate(small[f:f + 2], acc)
    assert _same(eng.transition_counts(small), eng.transition_counts_finish(acc))
    assert eng.poll_flags() == 0


@pytest.mark.parametrize("kind", ["walk", "iid"])
def test_counts_agree_with_the_transition_kernels_at_scale(vet, kind):
    eng = _engine(vet, [200, 1000])
    F, U = 201, 100_000
    p = _walk(F, U, 5, 0.02) if kind == "walk" else _iid(F, U, 6)
    p = torch.from_numpy(p).cuda()
    res = eng.transition_counts(p)
    tr = eng.transition(p, want_pairs0=True)
    assert eng.poll_flags() == 0
    pairs0 = tr.pairs0.reshape(-1, 2).to(torch.int64)
    present = pairs0[:, 0] != 0xFFFF
    T0 = eng.num_tiles[0]
    ref0 = torch.bincount(pairs0[present, 0] * T0 + pairs0[present, 1], minlength=T0 * T0).view(T0, T0)
    assert torch.equal(res.counts[0], ref0)
    assert torch.equal(res.counts[0].sum(1), tr.prev_count0.to(torch.int64).sum(0))
    assert res.pairs == int(present.sum())
    perm = torch.from_numpy(np.random.default_rng(1).permutation(U)).cuda()
    assert _same(res, eng.transition_counts(p[:, perm].contiguous()))


def test_transition_counts_errors(vet):
    eng = _engine(vet, [200])
    p = _walk(10, 20, 1)
    p[3, 7, 2] = 1.5
    eng.transition_counts(torch.from_numpy(p).cuda())
    with pytest.raises(vet.ValidationError):
        eng.raise_for_flags()
    ok = torch.from_numpy(_walk(10, 20, 1)).cuda()
    acc = eng.transition_counts_accumulator()
    with pytest.raises(TypeError):
        eng.transition_counts_accumulate(ok, acc.to(torch.int32))
    with pytest.raises(TypeError):
        eng.transition_counts_accumulate(ok, acc.cpu())
    with pytest.raises(ValueError):
        eng.transition_counts_accumulate(ok, acc[:-1])
    with pytest.raises(ValueError):
        eng.transition_counts_finish(acc.view(201, 201))
    with pytest.raises(ValueError):
        eng.transition_counts_finish(torch.zeros(2 * 201 * 201, dtype=torch.int64, device="cuda")[::2])
    direct = _engine(vet, [200], regime="direct")
    with pytest.raises(vet.UnsupportedConfigurationError, match="direct"):
        direct.transition_counts(ok)
    naive = vet.Engine(100, 200, [1], vet.EntropyConfig(), torch.device("cuda", 0), naive_tiles=(30, 30))
    with pytest.raises(vet.UnsupportedConfigurationError, match="grid"):
        naive.transition_counts(ok)
    huge = _engine(vet, [9600] * 3)   # 3 x 9601^2 entries > 2^28 (the accumulator alone takes 2.2 GB)
    with pytest.raises(vet.UnsupportedConfigurationError, match="2\\^28"):
        huge.transition_counts(ok)


def test_compute_transition_counts_in_batches(vet, tmp_path):
    from viewport_entropy_toolkit_b200 import AnalyzerConfig, TransitionEntropyAnalyzer
    F, U = 80, 50
    p = _walk(F, U, 9, 0.1)
    cfg = AnalyzerConfig(tile_counts=[20, 200], output_dir=tmp_path)
    ta = TransitionEntropyAnalyzer(cfg)
    ta.load_packed(p)
    out = ta.compute_transition_counts(batch_bytes=U * 12 * 7)   # 7 frames per batch
    whole = ta.engine.transition_counts(torch.from_numpy(p).cuda())
    assert out["pairs"] == whole.pairs
    for c, w in zip(out["counts"], whole.counts):
        assert np.array_equal(c, w.cpu().numpy())
    assert np.array_equal(out["per_k"], whole.per_k.cpu().numpy())
    assert out["entropy"] == float(whole.entropy)
    bad = p.copy()
    bad[5, 5, 1] = -0.5
    ta.load_packed(bad)
    with pytest.raises(vet.ValidationError):
        ta.compute_transition_counts()
