"""Per-viewer transition entropy (Engine.user_transitions / vet_user_transitions) against the CPU restatement: pairs
exact, per_k and entropy 1e-9 relative, NaN in the same places; and bit for bit the same outputs on a rerun, under a
user permutation, over user blocks, on a weighted handle and through the analyzer's user-column batching.  Users with
more pair records than the shared-memory sort holds go through global scratch; both sides of that switch are covered."""
import numpy as np
import pytest

from oracle.vet_user_transitions_oracle import user_transitions
from oracle.vet_transition_counts_oracle import transition_pairs

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

DEFAULT5 = [20, 50, 100, 250, 1000]
CAP = 3712   # VET_UT_SMEM_RECORDS (tests/test_user_transitions_host.py pins it to the header)


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


def _appearing(F, U, seed):
    p = _walk(F, U, seed, 0.05)
    p[: F // 2, 0, 1] = np.nan        # joins halfway
    p[F // 3:, 1, 1] = np.nan         # leaves after a third
    p[::2, 2, 2] = np.nan             # present in every other frame: N = 0
    p[:, 3, 1] = np.nan               # never present
    p[:, 4, 1] = np.nan
    p[7:9, 4, 1:] = 0.5               # present in frames 7 and 8 only: N = 1
    return p


def _check(res, ref):
    assert res.pairs.dtype == torch.int32
    assert np.array_equal(res.pairs.cpu().numpy(), ref["pairs"])
    np.testing.assert_allclose(res.per_k.cpu().numpy(), ref["per_k"], rtol=1e-9, atol=0, equal_nan=True)
    np.testing.assert_allclose(res.entropy.cpu().numpy(), ref["entropy"], rtol=1e-9, atol=0, equal_nan=True)


def _bits(t):
    return t.contiguous().cpu().numpy().view(np.int64 if t.dtype == torch.float64 else np.int32)


def _same(a, b):
    return (np.array_equal(_bits(a.entropy), _bits(b.entropy)) and np.array_equal(_bits(a.per_k), _bits(b.per_k))
            and torch.equal(a.pairs, b.pairs))


def _records(p, W, H, tcs):
    """Pair records per user (runs of one repeated pair) of tile count 0, for videos without missing samples."""
    (pp, cc), = transition_pairs(p, W, H, tcs[:1])
    F, U = p.shape[:2]
    T = int(max(pp.max(), cc.max())) + 1 if len(pp) else 1
    keys = (pp * T + cc).reshape(F - 1, U)
    return 1 + (keys[1:] != keys[:-1]).sum(0)


CASES = [
    dict(id="200_f32", tcs=[200], make=lambda: _walk(97, 301, 11)),
    dict(id="default5_missing", tcs=DEFAULT5, make=lambda: _walk(41, 677, 12, 0.1)),
    dict(id="200_f64", tcs=[200], make=lambda: _walk(50, 333, 13, 0.05, np.float64)),
    dict(id="global_200x400", tcs=[20, 200], W=200, H=400, make=lambda: _walk(45, 517, 14, 0.1)),
    dict(id="tile_count_2000", tcs=[2000], make=lambda: _walk(30, 700, 15, 0.05)),
    dict(id="iid_odd_U", tcs=[20, 200], make=lambda: _iid(23, 1001, 16)),
    dict(id="appearing_users", tcs=[20, 200], make=lambda: _appearing(60, 259, 17)),
    dict(id="F1", tcs=[50, 200], make=lambda: _walk(1, 99, 18)),
    dict(id="F2", tcs=[50, 200], make=lambda: _walk(2, 999, 18, 0.1)),
    dict(id="U1", tcs=[20, 200], make=lambda: _walk(300, 1, 19, 0.1)),
    dict(id="long_iid_past_smem", tcs=[200], make=lambda: _iid(20001, 37, 20)),
    dict(id="walk_long_large_steps", tcs=[200, 1000], make=lambda: _walk(6000, 45, 21, 0.01, step=0.1)),
]


@pytest.mark.parametrize("c", CASES, ids=[c["id"] for c in CASES])
def test_user_transitions_match_reference(vet, c):
    W, H = c.get("W", 100), c.get("H", 200)
    eng = _engine(vet, c["tcs"], False, W, H)
    p = c["make"]()
    res = eng.user_transitions(torch.from_numpy(p).cuda())
    assert eng.poll_flags() == 0
    _check(res, user_transitions(p, W, H, c["tcs"]))
    eng.close()


def test_records_on_both_sides_of_the_shared_memory_capacity(vet):
    # iid samples on 2001 tiles: practically every pair starts a record, so CAP + 1 frames give CAP records per user
    # (shared memory) and CAP + 2 frames CAP + 1 records (global scratch); both in one call, next to short users
    eng = _engine(vet, [2000, 20])
    for F, want in ((CAP + 1, CAP), (CAP + 2, CAP + 1)):
        p = _iid(F, 6, 30 + F)
        assert _records(p, 100, 200, [2000]).max() == want
        p[: F // 2, 1, 1] = np.nan                       # this user has about half the records
        res = eng.user_transitions(torch.from_numpy(p).cuda())
        _check(res, user_transitions(p, 100, 200, [2000, 20]))
    assert eng.poll_flags() == 0


def test_arbitrary_centres(vet):
    rng = np.random.default_rng(3)
    cs = [rng.normal(size=(37, 3)), rng.normal(size=(5, 3)), rng.normal(size=(1, 3))]
    eng = _engine(vet, [1, 2, 3], centres=cs)
    p = _walk(50, 611, 8, 0.1)
    res = eng.user_transitions(torch.from_numpy(p).cuda())
    assert eng.poll_flags() == 0
    _check(res, user_transitions(p, 100, 200, [1, 2, 3], centres=cs))
    assert np.isnan(res.per_k[2].cpu().numpy()).all()    # one tile: log2 T = 0
    assert np.isnan(res.entropy.cpu().numpy()).all()


@pytest.mark.parametrize("tcs", [[200], DEFAULT5, [20, 200, 2000]], ids=["200", "default5", "with_2000"])
def test_bit_identical_on_rerun_permutation_and_user_blocks(vet, tcs):
    eng = _engine(vet, tcs)
    F, U = 301, 1001
    p = torch.from_numpy(_appearing(F, U, 21)).cuda()
    one = eng.user_transitions(p)
    assert _same(one, eng.user_transitions(p))
    perm = torch.from_numpy(np.random.default_rng(1).permutation(U)).cuda()
    pm = eng.user_transitions(p[:, perm].contiguous())
    assert np.array_equal(_bits(pm.entropy), _bits(one.entropy[perm])) and torch.equal(pm.pairs, one.pairs[perm])
    assert np.array_equal(_bits(pm.per_k), _bits(one.per_k[:, perm]))
    parts = [eng.user_transitions(p[:, b:e]) for b, e in ((0, 1), (1, 8), (8, U))]   # blocks of 1, 7 and the rest
    cat = vet.UserTransitionResult(entropy=torch.cat([r.entropy for r in parts]),
                                   per_k=torch.cat([r.per_k for r in parts], 1), pairs=torch.cat([r.pairs for r in parts]))
    assert _same(one, cat)
    short = eng.user_transitions(p, want_per_k=False)
    assert short.per_k is None and np.array_equal(_bits(short.entropy), _bits(one.entropy))
    assert eng.poll_flags() == 0


def test_many_user_blocks_in_one_call(vet):
    # 5 tile counts x 3600 frames: the tile rows of 30k users exceed the 1 GiB scratch budget, so the call runs
    # several user blocks; every user must get the bits of a call over its own column block
    import bench
    eng = _engine(vet, DEFAULT5)
    p = bench.synth_on_device(torch, 3600, 40_000, 5, torch.device("cuda", 0), missing=0.05)
    one = eng.user_transitions(p)
    for b, e in ((0, 1000), (39_000, 40_000), (17_000, 17_500)):
        part = eng.user_transitions(p[:, b:e])
        assert np.array_equal(_bits(part.entropy), _bits(one.entropy[b:e]))
        assert np.array_equal(_bits(part.per_k), _bits(one.per_k[:, b:e])) and torch.equal(part.pairs, one.pairs[b:e])
    assert eng.poll_flags() == 0
    assert int(one.pairs.min()) > 0


def test_weighted_and_unweighted_handles_give_the_same_bits(vet):
    p = torch.from_numpy(_walk(80, 1500, 4, 0.1)).cuda()
    a = _engine(vet, [20, 200], True).user_transitions(p)
    b = _engine(vet, [20, 200], False).user_transitions(p)
    assert _same(a, b)


def test_per_user_transition_counts_agree(vet):
    eng = _engine(vet, [20, 200, 1000])
    p = torch.from_numpy(_walk(200, 500, 6, 0.05, step=0.06)).cuda()
    res = eng.user_transitions(p)
    for u in range(0, 500, 25):
        tc = eng.transition_counts(p[:, u:u + 1])
        assert tc.pairs == int(res.pairs[u])
        np.testing.assert_allclose(res.per_k[:, u].cpu().numpy(), tc.per_k.cpu().numpy(), rtol=1e-12, atol=0,
                                   equal_nan=True)


def test_user_transitions_errors(vet):
    eng = _engine(vet, [200])
    p = _walk(10, 20, 1)
    p[3, 7, 2] = 1.5
    eng.user_transitions(torch.from_numpy(p).cuda())
    with pytest.raises(vet.ValidationError):
        eng.raise_for_flags()
    ok = torch.from_numpy(_walk(10, 20, 1)).cuda()
    with pytest.raises(TypeError):
        eng.user_transitions(ok.to(torch.float16))
    with pytest.raises(TypeError):
        eng.user_transitions(ok.cpu().numpy())
    with pytest.raises(ValueError):
        eng.user_transitions(ok[:, :, :2].contiguous())
    with pytest.raises(ValueError):
        eng.user_transitions(ok[0])
    empty = eng.user_transitions(ok[:, :0])
    assert empty.entropy.shape == (0,) and empty.per_k.shape == (1, 0) and empty.pairs.shape == (0,)
    direct = _engine(vet, [200], regime="direct")
    with pytest.raises(vet.UnsupportedConfigurationError, match="direct"):
        direct.user_transitions(ok)
    naive = vet.Engine(100, 200, [1], vet.EntropyConfig(), torch.device("cuda", 0), naive_tiles=(30, 30))
    with pytest.raises(vet.UnsupportedConfigurationError, match="grid"):
        naive.user_transitions(ok)


def test_compute_user_transition_entropy_in_user_blocks(vet, tmp_path):
    from viewport_entropy_toolkit_b200 import AnalyzerConfig, TransitionEntropyAnalyzer
    F, U = 80, 50
    p = _appearing(F, U, 9)
    cfg = AnalyzerConfig(tile_counts=[20, 200], output_dir=tmp_path)
    ta = TransitionEntropyAnalyzer(cfg)
    ta.load_packed(p)
    small = ta.compute_user_transition_entropy(batch_bytes=F * 12 * 7)   # 7 users per block
    whole = ta.compute_user_transition_entropy()
    ref = ta.engine.user_transitions(torch.from_numpy(p).cuda())
    for out in (small, whole):
        assert list(out["identifier"]) == [f"user{u}" for u in range(U)]
        assert np.array_equal(out["pairs"].to_numpy(), ref.pairs.cpu().numpy())
        assert np.array_equal(out["entropy"].to_numpy().view(np.int64), _bits(ref.entropy))
    bad = p.copy()
    bad[5, 5, 1] = -0.5
    ta.load_packed(bad)
    with pytest.raises(vet.ValidationError):
        ta.compute_user_transition_entropy()
