"""Per-viewer exploration entropy (Engine.users / vet_users_accumulate / vet_users_finish) against the CPU
restatement: compute_spatial_entropy (EU:147-211) over each user's frames, mean over the tile counts.

Bars: entropies 1e-9 relative; hist0 entries frames * 2^-b absolute (the fixed-point quantum of the weights) plus
1e-12 relative, which covers two fp64 roundings the quantum does not: the conversion of an integer sum above 2^53 to
double in k_user_entropy (a relative 2^-53 per entry) and the reference's own fp64 sums; frames exact.  Results must be bit-identical on a rerun, under a
permutation of the frames and when the frames arrive in several batches."""
import numpy as np
import pytest

from oracle.vet_users_oracle import user_analyzer

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def vet():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import __graft_entry__ as ge
    ge.build()
    import viewport_entropy_toolkit_b200 as pkg
    return pkg


def _engine(vet, tcs, fov=90.0, use_w=True, W=100, H=200, **kw):
    return vet.Engine(W, H, tcs, vet.EntropyConfig(fov_angle=fov, use_weight_distribution=use_w, power_factor=2.0),
                      torch.device("cuda", 0), **kw)


def _walk(F, U, seed, missing=0.0, dtype=np.float32):
    rng = np.random.default_rng(seed)
    mu = np.clip(rng.normal(0.5, 0.2, U), 0, 1)[None] + np.cumsum(rng.normal(0, 0.03, (F, U)), 0)
    mv = np.clip(rng.normal(0.5, 0.15, U), 0, 1)[None] + np.cumsum(rng.normal(0, 0.02, (F, U)), 0)
    for a in (mu, mv):
        np.abs(a, out=a)
        a[a > 1] = 2 - a[a > 1]
        np.clip(a, 0, 1, out=a)
    p = np.stack([np.broadcast_to(np.arange(F)[:, None] * 0.1, (F, U)), mu, mv], -1).astype(dtype)
    if missing:
        p[rng.uniform(size=(F, U)) < missing, 1] = np.nan
    return p


def _bits(total_frames):
    return 62 - int(np.ceil(np.log2(total_frames))) if total_frames > 1 else 62


def _check(res, ref, F, use_w):
    frames = res.frames.cpu().numpy()
    assert res.frames.dtype == torch.int32
    assert np.array_equal(frames, ref["frames"])
    np.testing.assert_allclose(res.entropy.cpu().numpy(), ref["entropy"], rtol=1e-9, atol=0, equal_nan=True)
    np.testing.assert_allclose(res.per_k.cpu().numpy(), ref["per_k"], rtol=1e-9, atol=0, equal_nan=True)
    h, rh = res.hist0.cpu().numpy(), ref["hist0"]
    q = 2.0 ** -_bits(F) if use_w else 0.0
    # quantum of the weights + the fp64 roundings of both sides (sums above 2^53 round when converted to double)
    assert np.all(np.abs(h - rh) <= frames[:, None] * q + 1e-12 * np.abs(rh)), np.abs(h - rh).max()
    assert np.array_equal(h > 0, rh > 0)  # same support


CASES = [
    dict(id="w90_200", tcs=[200], fov=90.0, use_w=True, F=97, U=301, missing=0.0),
    dict(id="w120_200", tcs=[200], fov=120.0, use_w=True, F=64, U=130, missing=0.0),
    dict(id="w90_default5", tcs=[20, 50, 100, 250, 1000], fov=90.0, use_w=True, F=41, U=67, missing=0.1),
    dict(id="unw_200_missing", tcs=[200], fov=90.0, use_w=False, F=120, U=257, missing=0.1),
    dict(id="unw_default5", tcs=[20, 50, 100, 250, 1000], fov=120.0, use_w=False, F=33, U=95, missing=0.0),
    dict(id="w90_global_200x400", tcs=[200], fov=90.0, use_w=True, F=45, U=77, missing=0.1, W=200, H=400),
    dict(id="unw_global_200x400", tcs=[20, 200], fov=90.0, use_w=False, F=45, U=77, missing=0.1, W=200, H=400),
]


@pytest.mark.parametrize("c", CASES, ids=[c["id"] for c in CASES])
def test_users_match_reference(vet, c):
    W, H = c.get("W", 100), c.get("H", 200)
    eng = _engine(vet, c["tcs"], c["fov"], c["use_w"], W, H)
    p = _walk(c["F"], c["U"], 11, c["missing"])
    p[:, 3, 1] = np.nan                 # a user with no sample: NaN / 0
    p[1:, 4, 1] = np.nan                # a user with one sample (NaN when unweighted)
    res = eng.users(torch.from_numpy(p).cuda())
    assert eng.poll_flags() == 0
    ref = user_analyzer(p, W, H, c["tcs"], c["fov"], c["use_w"], 2.0)
    _check(res, ref, c["F"], c["use_w"])
    e = res.entropy.cpu().numpy()
    assert np.isnan(e[3]) and int(res.frames[3]) == 0 and not res.hist0[3].any()
    assert int(res.frames[4]) == 1 and (np.isnan(e[4]) if not c["use_w"] else np.isfinite(e[4]))
    eng.close()


def test_users_float64_input_and_edge_cells(vet):
    """float64 input decodes with the fp64 product: 0.35*200 is 70.0 in fp64 (DESIGN 2)."""
    eng = _engine(vet, [200], 90.0, True)
    p = _walk(30, 40, 5, 0.05, np.float64)
    p[::3, :, 1] = 0.5
    p[::3, :, 2] = 0.35
    p[1::7, :5, 1:] = [1.0, 1.0]
    p[2::7, 5:9, 1:] = [0.0, 0.0]
    res = eng.users(torch.from_numpy(p).cuda())
    assert eng.poll_flags() == 0
    _check(res, user_analyzer(p, 100, 200, [200], 90.0, True, 2.0), 30, True)


def test_users_arbitrary_centres(vet):
    rng = np.random.default_rng(3)
    cs = [rng.normal(size=(37, 3)), rng.normal(size=(5, 3))]
    for use_w in (True, False):
        eng = _engine(vet, [1, 2], 100.0, use_w, centres=cs)
        p = _walk(50, 61, 8, 0.1)
        res = eng.users(torch.from_numpy(p).cuda())
        assert eng.poll_flags() == 0
        _check(res, user_analyzer(p, 100, 200, [1, 2], 100.0, use_w, 2.0, centres=cs), 50, use_w)
        eng.close()


def _host(res):
    return [None if t is None else t.cpu().numpy() for t in (res.entropy, res.per_k, res.hist0, res.frames)]


def _same(a, b):
    return all(np.array_equal(x, y, equal_nan=True) for x, y in zip(_host(a), _host(b)))


@pytest.mark.parametrize("use_w", [True, False], ids=["weighted", "unweighted"])
def test_users_bit_identical_under_rerun_permutation_and_batches(vet, use_w):
    eng = _engine(vet, [20, 200], 90.0, use_w)
    F, U = 301, 1001
    p = torch.from_numpy(_walk(F, U, 21, 0.1)).cuda()
    one = eng.users(p)
    assert _same(one, eng.users(p))
    perm = torch.from_numpy(np.random.default_rng(0).permutation(F)).cuda()
    assert _same(one, eng.users(p[perm].contiguous()))
    acc = eng.user_accumulator(U)
    for b, e in ((0, 17), (17, 200), (200, F)):
        eng.users_accumulate(p[b:e], acc, F)
    assert _same(one, eng.users_finish(acc, F))
    # few users: the frames are split over several CTAs whose rows meet through the atomics
    small = p[:, :5].contiguous()
    acc = eng.user_accumulator(5)
    for f in range(F):
        eng.users_accumulate(small[f:f + 1], acc, F)
    assert _same(eng.users(small), eng.users_finish(acc, F))
    assert eng.poll_flags() == 0


@pytest.mark.parametrize("use_w", [True, False], ids=["weighted", "unweighted"])
def test_users_agree_with_the_transposition_route(vet, use_w):
    """Engine.spatial on the transposed tensor treats each user as a frame: the same numbers, at twice the memory."""
    eng = _engine(vet, [20, 200], 90.0, use_w)
    F, U = 160, 700
    p = torch.from_numpy(_walk(F, U, 4, 0.1)).cuda()
    res = eng.users(p)
    tr = eng.spatial(p.transpose(0, 1).contiguous(), want_assign0=False)
    assert eng.poll_flags() == 0
    np.testing.assert_allclose(res.entropy.cpu().numpy(), tr.entropy.cpu().numpy(), rtol=1e-9, atol=0)
    np.testing.assert_allclose(res.per_k.cpu().numpy(), tr.per_k.cpu().numpy(), rtol=1e-9, atol=0)
    frames = res.frames.cpu().numpy()[:, None]
    h, th = res.hist0.cpu().numpy(), tr.hist0.cpu().numpy()
    # the transposed call's weighted histogram may take the tensor-core path (2^-39 per entry, DESIGN 4.3)
    assert np.all(np.abs(h - th) <= frames * (2.0 ** -39 if use_w else 0.0) + 1e-12 * np.abs(th))


def test_users_errors(vet):
    eng = _engine(vet, [200], 90.0, True)
    p = _walk(10, 20, 1)
    p[3, 7, 2] = 1.5
    eng.users(torch.from_numpy(p).cuda())
    with pytest.raises(vet.ValidationError):
        eng.raise_for_flags()
    ok = torch.from_numpy(_walk(10, 20, 1)).cuda()
    acc = eng.user_accumulator(20)
    with pytest.raises(ValueError):
        eng.users_accumulate(ok, acc, 9)                      # total_frames < F
    with pytest.raises(ValueError):
        eng.users_accumulate(ok, eng.user_accumulator(21), 10)  # wrong user count
    with pytest.raises(TypeError):
        eng.users_accumulate(ok, acc.to(torch.int32), 10)
    with pytest.raises(TypeError):
        eng.users_accumulate(ok, acc.cpu(), 10)
    direct = _engine(vet, [200], 90.0, True, regime="direct")
    with pytest.raises(vet.UnsupportedConfigurationError, match="direct"):
        direct.users(ok)
    naive = vet.Engine(100, 200, [1], vet.EntropyConfig(), torch.device("cuda", 0), naive_tiles=(30, 30))
    with pytest.raises(vet.UnsupportedConfigurationError, match="grid"):
        naive.users(ok)


def test_compute_user_entropy_in_batches(vet, tmp_path):
    from viewport_entropy_toolkit_b200 import AnalyzerConfig, EntropyConfig, SpatialEntropyAnalyzer
    F, U = 80, 50
    p = _walk(F, U, 9, 0.1)
    p[:, 2, 1] = np.nan
    cfg = AnalyzerConfig(tile_counts=[20, 200], output_dir=tmp_path, entropy_config=EntropyConfig(fov_angle=90.0))
    sa = SpatialEntropyAnalyzer(cfg)
    sa.load_packed(p, [f"viewer{u}" for u in range(U)])
    df = sa.compute_user_entropy(batch_bytes=U * 12 * 7)   # 7 frames per batch
    whole = sa.engine.users(torch.from_numpy(p).cuda())
    assert list(df.columns) == ["identifier", "frames", "entropy", "tile_weights"]
    assert list(df["identifier"]) == [f"viewer{u}" for u in range(U)]
    assert np.array_equal(df["entropy"].to_numpy(), whole.entropy.cpu().numpy(), equal_nan=True)
    assert np.array_equal(df["frames"].to_numpy(), whole.frames.cpu().numpy())
    h0 = whole.hist0.cpu().numpy()
    centres = sa._fibonacci_vectors[20]
    assert dict(df["tile_weights"][0]) == {centres[i]: float(h0[0, i]) for i in np.flatnonzero(h0[0])}
    assert len(df["tile_weights"][2]) == 0
    bad = p.copy()
    bad[5, 5, 1] = -0.5
    sa.load_packed(bad)
    with pytest.raises(vet.ValidationError):
        sa.compute_user_entropy()
