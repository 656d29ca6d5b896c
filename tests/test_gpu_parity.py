"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on
the same seeded inputs and against the committed live-reference fixtures.

Bars: tile indices, histogram counts, transition counts and pairs BIT-EXACT;
entropies and FOV weights within 1e-9 relative (north_star), with an absolute
floor of 1e-12 for values that are analytically zero.
"""
import numpy as np
import pytest

from conftest import group_keys, load_golden
from oracle import vet_oracle as orc

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

RTOL = 1e-9
ATOL = 1e-12
TILE_COUNTS_ALL = [20, 50, 100, 200, 250, 500, 1000]
W0, H0 = 100, 200


@pytest.fixture(scope="module")
def vet():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import viewport_entropy_toolkit_b200 as pkg
    return pkg


def engine(vet, tile_counts, fov=120.0, use_w=True, pf=2.0, W=W0, H=H0, **kw):
    ec = vet.EntropyConfig(fov_angle=fov, use_weight_distribution=use_w, power_factor=pf)
    return vet.Engine(W, H, tile_counts, ec, **kw)


def cell_centres_packed(W, H, dtype=np.float32):
    """One sample per reachable cell: (mu, mv) that truncates to (px, py)."""
    px = np.arange(W + 1)
    py = np.arange(H + 1)
    mu = np.where(px < W, (px + 0.5) / W, 1.0)
    mv = np.where(py < H, (py + 0.5) / H, 1.0)
    p = np.zeros((H + 1, W + 1, 3), dtype=dtype)
    p[..., 1] = mu[None, :]
    p[..., 2] = mv[:, None]
    qx, qy, ok = orc.decode(p[..., 1], p[..., 2], W, H)
    assert ok.all() and np.array_equal(qx, np.broadcast_to(px, qx.shape)) and np.array_equal(qy.T, np.broadcast_to(py, qy.T.shape))
    return p


def synth(F, U, seed, iid=False, missing=0.0, dtype=np.float32):
    rng = np.random.default_rng(seed)
    if iid:
        mu = rng.uniform(0, 1, (F, U)); mv = rng.uniform(0, 1, (F, U))
    else:
        mu = np.clip(rng.normal(0.5, 0.15, U), 0, 1)[None] + np.cumsum(rng.normal(0, 0.01, (F, U)), 0)
        mv = np.clip(rng.normal(0.5, 0.10, U), 0, 1)[None] + np.cumsum(rng.normal(0, 0.006, (F, U)), 0)
        mu = np.abs(mu); mu = np.where(mu > 1, 2 - mu, mu); mu = np.clip(mu, 0, 1)
        mv = np.abs(mv); mv = np.where(mv > 1, 2 - mv, mv); mv = np.clip(mv, 0, 1)
    p = np.stack([np.broadcast_to(np.arange(F)[:, None] * 0.1, (F, U)), mu, mv], -1).astype(dtype)
    edge = [(0.5, 0.5), (0.0, 0.5), (1.0, 0.5), (1.0, 1.0), (0.29, 0.57), (0.999, 0.001), (0.123456, 0.654321), (0.75, 0.25)]
    for u, (a, b) in enumerate(edge[:U]):
        p[0, u, 1] = a; p[0, u, 2] = b
    if missing:
        m = rng.uniform(size=(F, U)) < missing
        m[:, 0] = False
        p[m, 1] = np.nan; p[m, 2] = np.nan
    return p


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ---------------------------------------------------------------------------------
def test_lattice_and_native_tables(vet):
    g = load_golden("lattices")
    e = engine(vet, [1, 2, 3, 7, 20, 21, 50, 100, 200, 250, 500, 1000], use_w=False)
    for k, n in enumerate(e.tile_counts):
        assert np.array_equal(e.lattice(k), g[f"n{n}"]), n
    e.close()
    # tables derived inside the library with libm (no numpy tables passed) give the same LUTs
    a = engine(vet, [20, 200, 1000], use_w=False)
    b = engine(vet, [20, 200, 1000], use_w=False, native_tables=True)
    for k in range(3):
        assert np.array_equal(a.lattice(k), b.lattice(k))
        assert np.array_equal(a.cell_lut(k), b.cell_lut(k))
    a.close(); b.close()


def test_cell_lut_exhaustive_vs_reference(vet):
    """Brute-force fp64 nearest-tile kernel over the whole reachable domain
    (20,301 cells) x seven tile counts == reference find_nearest_tile."""
    g = load_golden("nearest")
    e = engine(vet, TILE_COUNTS_ALL, use_w=False)
    for k, n in enumerate(TILE_COUNTS_ALL):
        assert np.array_equal(e.cell_lut(k).ravel(), g[f"lut_n{n}"]), n
    e.close()


@pytest.mark.parametrize("dims", [(100, 200), (200, 400)])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_decode_every_cell(vet, dims, dtype):
    W, H = dims
    g = load_golden("decode")
    try:
        e = engine(vet, [20], use_w=False, W=W, H=H)
    except vet.UnsupportedConfigurationError:
        pytest.skip("grid larger than the table regime")
    p = cell_centres_packed(W, H, dtype)
    vec, cell = e.decode(dev(p))
    ref = g[f"cellvec_{W}x{H}"]
    got = vec.cpu().numpy()
    assert np.array_equal(got, ref)
    assert np.array_equal(np.signbit(got), np.signbit(ref))
    assert np.array_equal(cell.cpu().numpy(), np.arange((W + 1) * (H + 1)).reshape(H + 1, W + 1))
    e.close()


def test_decode_quirks_missing_and_range(vet):
    e = engine(vet, [20], use_w=False)
    p = np.zeros((1, 6, 3), dtype=np.float32)
    p[0, :, 1] = [0.29, np.nan, 0.5, 1.5, -0.1, 1.0]
    p[0, :, 2] = [0.57, 0.5, np.nan, 0.5, 0.5, 1.0]
    vec, cell = e.decode(dev(p))
    cell = cell.cpu().numpy()[0]
    assert cell[0] == 113 * 101 + 28 and cell[5] == 200 * 101 + 100
    assert (cell[1:5] == -1).all()
    assert np.isnan(vec.cpu().numpy()[0, 1:5]).all()
    assert e.poll_flags() & 1  # VET_FLAG_OUT_OF_RANGE
    assert e.poll_flags() == 0  # cleared
    e.close()


def test_nearest_tile_arbitrary_vectors(vet):
    g = load_golden("nearest")
    e = engine(vet, [20, 200, 1000], use_w=False)
    v = dev(g["arb_vecs"])
    for k, n in enumerate([20, 200, 1000]):
        assert np.array_equal(e.nearest_tile(v, k).cpu().numpy(), g[f"arb_n{n}"].astype(np.int32))
    tie = dev(np.array([[-1.0, 0.0, 0.0], [-2.5, 0.0, 0.0]]))
    assert e.nearest_tile(tie, 0).cpu().tolist() == [6, 6]
    assert e.nearest_tile(tie, 1).cpu().tolist() == [83, 83]
    e.close()


def test_tile_weights_vs_reference(vet):
    g = load_golden("weights")
    cv = orc.cell_vectors(W0, H0).reshape(-1, 3)[g["sel"]]
    for key in g.files:
        if not key.startswith("w_"):
            continue
        _, n, fov, pf = key.split("_")
        n, fov, pf = int(n[1:]), float(fov[3:]), float(pf[2:])
        e = engine(vet, [n], fov=fov, pf=pf)
        w = e.tile_weights(dev(cv), 0).cpu().numpy()
        ref = g[key]
        near_edge = np.abs(ref) < 1e-12   # support may differ only within rounding of d == fov/2
        assert np.array_equal((w > 0) | near_edge, (ref > 0) | near_edge), key
        np.testing.assert_allclose(w, ref, rtol=RTOL, atol=1e-14, err_msg=key)
        e.close()
    e = engine(vet, [20], use_w=False)
    w = e.tile_weights(dev(cv), 0).cpu().numpy()
    assert np.array_equal(w.argmax(1), orc.nearest_tile(cv, orc.lattice(20))) and np.array_equal(w.sum(1), np.ones(len(cv)))
    e.close()


@pytest.mark.parametrize("case", ["c_small_w120", "c_small_unw", "c_w90_t200", "c_missing", "c_iid_unw", "c_iid_w",
                                  "c_oneuser", "c_t1000"])
def test_frames_vs_reference_fixtures(vet, case):
    c = group_keys(load_golden("frames"))[case]
    packed, tcs = c["packed"], [int(v) for v in c["tile_counts"]]
    fov, use_w, pf = float(c["cfg"][0]), bool(c["cfg"][1]), float(c["cfg"][2])
    e = engine(vet, tcs, fov, use_w, pf)
    sp = e.spatial(dev(packed))
    assert e.poll_flags() == 0
    assert np.array_equal(sp.assign0.cpu().numpy(), c["sp_assign0"])
    np.testing.assert_allclose(sp.per_k.cpu().numpy(), c["sp_per_k"], rtol=RTOL, atol=ATOL, equal_nan=True)
    np.testing.assert_allclose(sp.entropy.cpu().numpy(), c["sp_entropy"], rtol=RTOL, atol=ATOL, equal_nan=True)
    if use_w:
        np.testing.assert_allclose(sp.hist0.cpu().numpy(), c["sp_hist0"], rtol=RTOL, atol=ATOL)
    else:
        assert np.array_equal(sp.hist0.cpu().numpy(), c["sp_hist0"])
    if packed.shape[0] > 1:
        tr = e.transition(dev(packed))
        assert e.poll_flags() == 0
        assert np.array_equal(tr.pairs0.cpu().numpy(), c["tr_pairs0"])
        assert np.array_equal(tr.prev_count0.cpu().numpy(), c["tr_prev_count0"])
        np.testing.assert_allclose(tr.per_k.cpu().numpy(), c["tr_per_k"], rtol=RTOL, atol=ATOL, equal_nan=True)
        np.testing.assert_allclose(tr.entropy.cpu().numpy(), c["tr_entropy"], rtol=RTOL, atol=ATOL, equal_nan=True)
    e.close()


def _tile_to_sample(lut):
    """tile index -> (mu, mv) of one cell whose nearest tile it is."""
    H1, W1 = lut.shape
    rep = {}
    for cell, t in enumerate(lut.ravel()):
        rep.setdefault(int(t), cell)
    return {t: ((c % W1 + 0.5) / (W1 - 1) if c % W1 < W1 - 1 else 1.0,
                (c // W1 + 0.5) / (H1 - 1) if c // W1 < H1 - 1 else 1.0) for t, c in rep.items()}


def test_transition_quirks_vs_reference(vet):
    """Adversarial (prev,cur) index patterns of the reference fixtures, driven through
    packed samples chosen inside the wanted tiles."""
    cases = group_keys(load_golden("transition_quirks"))
    engines = {}
    for name, c in cases.items():
        T = int(c["T"])
        n = T - 1
        if n not in engines:
            engines[n] = engine(vet, [n], use_w=False)
        e = engines[n]
        rep = _tile_to_sample(e.cell_lut(0))
        p, cc = c["p"], c["c"]
        packed = np.zeros((2, len(p), 3), dtype=np.float64)
        packed[0, :, 1:] = [rep[int(t)] for t in p]
        packed[1, :, 1:] = [rep[int(t)] for t in cc]
        tr = e.transition(dev(packed))
        flags = e.poll_flags()
        assert np.array_equal(tr.pairs0.cpu().numpy()[0], np.stack([p, cc], 1).astype(np.uint16)), name
        assert np.array_equal(tr.prev_count0.cpu().numpy()[0], np.bincount(p, minlength=T)), name
        got, ref = float(tr.entropy.cpu()[0]), float(c["e"])
        if np.isnan(ref):
            assert np.isnan(got), name
        else:
            np.testing.assert_allclose(got, ref, rtol=RTOL, atol=ATOL, err_msg=name)
        assert flags == 0
    for e in engines.values():
        e.close()


@pytest.mark.parametrize("cfg", [
    dict(F=8, U=5000, tcs=[20, 50, 100, 200], use_w=False, fov=120.0, iid=False),
    dict(F=6, U=3000, tcs=[200], use_w=True, fov=90.0, iid=False),
    dict(F=4, U=2000, tcs=[20, 50], use_w=True, fov=120.0, iid=True, missing=0.2),
    dict(F=3, U=70000, tcs=[200, 20], use_w=False, fov=120.0, iid=True),        # several chunks per frame
    dict(F=3, U=1500, tcs=[250, 1000], use_w=True, fov=120.0, iid=False),
    dict(F=5, U=700, tcs=[50], use_w=True, fov=360.0, pf=3.0, iid=True),
    dict(F=5, U=700, tcs=[50], use_w=True, fov=10.0, pf=0.5, iid=True),         # most users outside every FOV
    dict(F=7, U=2501, tcs=[200, 50], use_w=True, fov=90.0, iid=True, missing=0.05),   # odd U: unaligned tile heads, tensor tail
    dict(F=5, U=4099, tcs=[1000], use_w=False, fov=120.0, iid=True),              # single tile count: direct tile-histogram kernel, u16 LUT
    dict(F=9, U=3001, tcs=[20, 50, 250, 1000], use_w=False, fov=120.0, iid=False, dtype=np.float64),  # mixed u8/u16 LUTs, f64 input
])
def test_spatial_vs_oracle(vet, cfg):
    p = synth(cfg["F"], cfg["U"], 900 + cfg["U"], cfg.get("iid", False), cfg.get("missing", 0.0),
              dtype=cfg.get("dtype", np.float32))
    pf = cfg.get("pf", 2.0)
    e = engine(vet, cfg["tcs"], cfg["fov"], cfg["use_w"], pf)
    sp = e.spatial(dev(p))
    assert e.poll_flags() == 0
    ref = orc.spatial_analyzer(p, W0, H0, cfg["tcs"], cfg["fov"], cfg["use_w"], pf)
    assert np.array_equal(sp.assign0.cpu().numpy(), ref["assign0"])
    if cfg["use_w"]:
        np.testing.assert_allclose(sp.hist0.cpu().numpy(), ref["hist0"], rtol=RTOL, atol=ATOL)
    else:
        assert np.array_equal(sp.hist0.cpu().numpy(), ref["hist0"])
    np.testing.assert_allclose(sp.per_k.cpu().numpy(), ref["per_k"], rtol=RTOL, atol=ATOL, equal_nan=True)
    np.testing.assert_allclose(sp.entropy.cpu().numpy(), ref["entropy"], rtol=RTOL, atol=ATOL, equal_nan=True)
    e.close()


@pytest.mark.parametrize("cfg", [
    dict(F=6, U=4000, tcs=[20, 50], iid=False),
    dict(F=4, U=3000, tcs=[200, 500, 1000], iid=False),
    dict(F=3, U=6000, tcs=[200], iid=True),                 # many distinct pairs: global pair table
    dict(F=5, U=900, tcs=[50, 20], iid=True, missing=0.3),
    dict(F=3, U=9000, tcs=[200, 500, 1000], iid=False),     # fast paths: dense table (201) + shared-memory hash (501, 1001)
    dict(F=3, U=20000, tcs=[1000, 200], iid=True, missing=0.1),  # hash overflow -> in-kernel fallback to the global table
    dict(F=4, U=5000, tcs=[1000], iid=False),               # one tile count: tile ids straight from the streaming kernel, hash table
    dict(F=3, U=20001, tcs=[500], iid=True, missing=0.1),   # the same with overflow rows (redone through the identity table), odd U
    dict(F=4, U=2500, tcs=[20], iid=False, dtype=np.float64),  # one tile count, dense table, float64 input
])
@pytest.mark.parametrize("mode", ["literal", "textbook"])
def test_transition_vs_oracle(vet, cfg, mode):
    p = synth(cfg["F"], cfg["U"], 700 + cfg["U"], cfg.get("iid", False), cfg.get("missing", 0.0),
              dtype=cfg.get("dtype", np.float32))
    e = engine(vet, cfg["tcs"], use_w=False)
    tr = e.transition(dev(p), mode=mode)
    assert e.poll_flags() == 0
    ref = orc.transition_analyzer(p, W0, H0, cfg["tcs"], mode=mode)
    assert np.array_equal(tr.pairs0.cpu().numpy(), ref["pairs0"])
    assert np.array_equal(tr.prev_count0.cpu().numpy(), ref["prev_count0"])
    np.testing.assert_allclose(tr.per_k.cpu().numpy(), ref["per_k"], rtol=RTOL, atol=ATOL, equal_nan=True)
    np.testing.assert_allclose(tr.entropy.cpu().numpy(), ref["entropy"], rtol=RTOL, atol=ATOL, equal_nan=True)
    e.close()


def test_float64_input_matches_float32_input(vet):
    p32 = synth(4, 2000, 5)
    e = engine(vet, [20, 200], fov=90.0)
    a = e.spatial(dev(p32))
    b = e.spatial(dev(p32.astype(np.float64)))
    assert torch.equal(a.assign0, b.assign0) and torch.equal(a.entropy, b.entropy) and torch.equal(a.hist0, b.hist0)
    # fp64-only values: 0.35*200 rounds up to 70.0 in fp64, float32(0.35)*200 does not
    p = np.zeros((1, 2, 3)); p[0, :, 1] = 0.5; p[0, :, 2] = [0.35, 0.35]
    _, cell = e.decode(dev(p))
    assert cell.cpu().numpy()[0, 0] == 70 * 101 + 50
    _, cell32 = e.decode(dev(p.astype(np.float32)))
    assert cell32.cpu().numpy()[0, 0] == 69 * 101 + 50
    e.close()


def test_error_flags_map_to_reference_exceptions(vet, tmp_path):
    cfg = vet.AnalyzerConfig(tile_counts=[20], output_dir=tmp_path)
    sa = vet.SpatialEntropyAnalyzer(cfg)
    ta = vet.TransitionEntropyAnalyzer(cfg)
    p = synth(3, 16, 1)
    bad = p.copy(); bad[1, 3, 1] = 1.25
    with pytest.raises(vet.ValidationError, match="between 0 and 1"):
        sa.compute_entropy_packed(dev(bad))
    empty = p.copy(); empty[2, :, 1] = np.nan
    with pytest.raises(vet.ValidationError, match="Empty vector dictionary"):
        sa.compute_entropy_packed(dev(empty))
    nocommon = p.copy(); nocommon[0, :8, 1] = np.nan; nocommon[1, 8:, 1] = np.nan
    with pytest.raises(ZeroDivisionError):
        ta.compute_entropy_packed(dev(nocommon))
    # and a clean run afterwards is clean
    sa.compute_entropy_packed(dev(p))
    with pytest.raises(vet.ValidationError):
        vet.Engine(101, 200, [20])
    with pytest.raises(vet.ValidationError):
        vet.EntropyConfig(fov_angle=0)


def test_host_buffer_path_equals_device_path(vet):
    p = synth(40, 3000, 77, missing=0.05)
    e = engine(vet, [200, 20], fov=90.0)
    d = e.spatial(dev(p))
    h = e.spatial_host(p)
    assert np.array_equal(h["assign0"], d.assign0.cpu().numpy())
    assert np.array_equal(h["entropy"], d.entropy.cpu().numpy())
    assert np.array_equal(h["hist0"], d.hist0.cpu().numpy())
    assert np.array_equal(h["per_k"], d.per_k.cpu().numpy())
    t = e.transition(dev(p))
    th = e.transition_host(p)
    assert np.array_equal(th["entropy"], t.entropy.cpu().numpy(), equal_nan=True)
    assert np.array_equal(th["pairs0"], t.pairs0.cpu().numpy())
    e.close()


def test_properties_at_scale(vet):
    """Size-independent checks on a tensor too large for the oracle: counts sum to the
    number of present users, entropies lie in [0,1], user permutation leaves the spatial
    result unchanged, and re-running is bit-identical (deterministic reductions)."""
    F, U = 48, 100_000
    g = torch.Generator(device="cuda").manual_seed(20260003)
    p = torch.rand((F, U, 3), generator=g, device="cuda", dtype=torch.float32)
    e = engine(vet, [200], use_w=False)
    a = e.spatial(p)
    assert e.poll_flags() == 0
    assert torch.equal(a.hist0.sum(1), torch.full((F,), float(U), dtype=torch.float64, device="cuda"))
    ent = a.entropy.cpu().numpy()
    assert ((ent >= 0) & (ent <= 1)).all()
    lut = torch.from_numpy(e.cell_lut(0).astype(np.int64)).cuda().ravel()
    # DU:261 in fp64 (exact for float32 inputs) with plain torch ops
    cell = (p[..., 2].double() * 200).to(torch.int64) * 101 + (p[..., 1].double() * 100).to(torch.int64)
    _, cell_k = e.decode(p)
    assert torch.equal(cell_k.long(), cell)
    assert torch.equal(a.assign0.long(), lut[cell_k.long()])
    perm = torch.randperm(U, device="cuda")
    b = e.spatial(p[:, perm].contiguous())
    assert torch.equal(a.hist0, b.hist0) and torch.equal(a.entropy, b.entropy)
    e.close()
    ew = engine(vet, [200], fov=90.0)
    w1 = ew.spatial(p)
    w2 = ew.spatial(p)
    assert torch.equal(w1.entropy, w2.entropy) and torch.equal(w1.hist0, w2.hist0)
    went = w1.entropy.cpu().numpy()
    assert ((went >= 0) & (went <= 1)).all()
    # weighted histogram against an independent evaluation from the dense weight kernel on frame 0
    vec, _ = ew.decode(p[:1, :4096])
    dense = ew.tile_weights(vec[0], 0).sum(0)
    part = ew.spatial(p[:1, :4096].contiguous())
    np.testing.assert_allclose(part.hist0[0].cpu().numpy(), dense.cpu().numpy(), rtol=RTOL, atol=ATOL)
    ew.close()


# ---------------------------------------------------------------------------------
# functional API (reference names, dicts of Vector, arbitrary tile-centre lists)
# ---------------------------------------------------------------------------------
def test_functional_api_vs_reference_fixtures(vet):
    """compute_spatial_entropy / compute_transition_entropy called like the reference's free
    functions (EU:147-332) on the frames of the live-reference fixtures."""
    fx = group_keys(load_golden("frames"))
    for case in ["c_small_w120", "c_small_unw", "c_missing", "c_iid_w"]:
        c = fx[case]
        packed, tcs = c["packed"], [int(v) for v in c["tile_counts"]]
        fov, use_w, pf = float(c["cfg"][0]), bool(c["cfg"][1]), float(c["cfg"][2])
        cfg = vet.EntropyConfig(fov_angle=fov, use_weight_distribution=use_w, power_factor=pf)
        vecs, ok = orc.decode_vectors(packed[..., 1], packed[..., 2], W0, H0)
        for k, n in enumerate(tcs[:2]):
            centres = vet.generate_fibonacci_lattice(n)
            for f in range(min(3, packed.shape[0])):
                d = {f"u{u:05d}": vet.Vector(*vecs[f, u]) for u in range(packed.shape[1]) if ok[f, u]}
                e, wts, asg = vet.compute_spatial_entropy(d, centres, cfg)
                np.testing.assert_allclose(e, c["sp_per_k"][k, f], rtol=RTOL, atol=ATOL, equal_nan=True)
                if k == 0:
                    assert [asg[key] for key in d] == [int(a) for a in c["sp_assign0"][f][ok[f]]]
                    ref_hist = c["sp_hist0"][f]
                    got = np.zeros_like(ref_hist)
                    idx = {ct: i for i, ct in enumerate(centres)}
                    for ct, w in wts.items():
                        got[idx[ct]] = w
                    np.testing.assert_allclose(got, ref_hist, rtol=RTOL, atol=ATOL)
                if f + 1 < packed.shape[0]:
                    d1 = {f"u{u:05d}": vet.Vector(*vecs[f + 1, u]) for u in range(packed.shape[1]) if ok[f + 1, u]}
                    te, tw, ta = vet.compute_transition_entropy(d, d1, centres, cfg, 120)
                    np.testing.assert_allclose(te, c["tr_per_k"][k, f], rtol=RTOL, atol=ATOL, equal_nan=True)
                    if k == 0:
                        both = ok[f] & ok[f + 1]
                        assert [list(ta[f"u{u:05d}"]) for u in np.flatnonzero(both)] == c["tr_pairs0"][f][both].tolist()


def test_functional_api_arbitrary_centres(vet):
    """Tile centres that are NOT a Fibonacci lattice (even count, non-unit vectors) and
    arbitrary user vectors, against the oracle's literal (reference-shaped) layer."""
    rng = np.random.default_rng(99)
    centres_np = rng.normal(size=(12, 3)) * rng.uniform(0.5, 2.0, size=(12, 1))
    centres = [vet.Vector(*c) for c in centres_np]
    users = rng.normal(size=(30, 3))
    d0 = {f"p{i}": vet.Vector(*users[i]) for i in range(30)}
    d1 = {f"p{i}": vet.Vector(*(users[i] + 0.4 * rng.normal(size=3))) for i in range(29, -1, -1) if i % 7}
    for cfg in (vet.EntropyConfig(fov_angle=100.0, power_factor=1.5), vet.EntropyConfig(use_weight_distribution=False)):
        e, wts, asg = vet.compute_spatial_entropy(d0, centres, cfg)
        re, rw, ra = orc.compute_spatial_entropy_literal({k: v.as_tuple() for k, v in d0.items()}, centres_np,
                                                         cfg.fov_angle, cfg.use_weight_distribution, cfg.power_factor)
        np.testing.assert_allclose(e, re, rtol=RTOL)
        assert asg == ra
        assert {centres.index(c) for c in wts} == set(rw)
        for ct, w in wts.items():
            np.testing.assert_allclose(w, rw[centres.index(ct)], rtol=RTOL, atol=1e-14)
    te, tw, ta = vet.compute_transition_entropy(d0, d1, centres, vet.EntropyConfig(), 120)
    rte, rtw, rta = orc.compute_transition_entropy_literal({k: v.as_tuple() for k, v in d0.items()},
                                                           {k: v.as_tuple() for k, v in d1.items()}, centres_np)
    np.testing.assert_allclose(te, rte, rtol=RTOL, atol=ATOL)
    assert ta == rta and {centres.index(c): n for c, n in tw.items()} == {int(k): int(v) for k, v in rtw.items()}
    assert list(ta) == list(rta)   # current-frame dict order
    v = vet.Vector(0.3, -0.2, 0.9)
    dist = vet.find_angular_distances(v, centres)
    ref = orc.find_angular_distances_literal(v.as_tuple(), centres_np)
    np.testing.assert_allclose(dist, ref, rtol=1e-12, atol=1e-15)
    assert vet.find_nearest_tile(v, centres) == orc.find_nearest_tile_literal(v.as_tuple(), centres_np)
    np.testing.assert_allclose(vet.vector_angle_distance(v, centres[3]), ref[3, 1], rtol=1e-12)
    cw = vet.calculate_tile_weights(v, centres, vet.EntropyConfig(fov_angle=140.0))
    rw = orc.calculate_tile_weights_literal(v.as_tuple(), centres_np, 140.0, True, 2.0)
    assert [centres.index(c) for c in cw] == list(rw)   # insertion order = ascending distance
    with pytest.raises(vet.ValidationError, match="Empty vector dictionary"):
        vet.compute_spatial_entropy({}, centres, vet.EntropyConfig())
    with pytest.raises(vet.ValidationError, match="No tile centers"):
        vet.compute_spatial_entropy(d0, [], vet.EntropyConfig())
    with pytest.raises(ZeroDivisionError):
        vet.compute_transition_entropy({"a": v}, {"b": v}, centres)


@pytest.mark.parametrize("dims,regime", [((200, 400), "global"), ((200, 400), "direct"), ((1920, 1080), "direct"),
                                         ((1920, 1080), "global")])   # 2M cells: global LUTs when unweighted, else direct
def test_large_video_direct_mode(vet, dims, regime):
    """Videos whose cell grid does not fit the shared-memory tables: up to 262,144 cells (the 200x400 of the
    reference's README) the per-cell tables stay in global memory (k_stream_global + the usual epilogues),
    beyond that -- or with regime="direct" (vet_config.regime) -- the direct per-sample path (decode -> vectors -> brute force)
    runs; results must match the oracle all the same."""
    W, H = dims
    p = synth(4, 300, 4242, iid=True, missing=0.1, dtype=np.float64)
    for use_w, tcs in ((True, [20, 50]), (False, [200])):
        e = engine(vet, tcs, fov=100.0, use_w=use_w, W=W, H=H, regime="direct" if regime == "direct" else "auto")
        if regime == "global":   # per-cell tables exist (also for the weighted 2.08 M-cell handle: its weight columns fit the budget)
            assert e.cell_lut(0).shape == (H + 1, W + 1)
        else:
            with pytest.raises(vet.UnsupportedConfigurationError):
                e.cell_lut(0)
        sp = e.spatial(dev(p))
        assert e.poll_flags() == 0
        ref = orc.spatial_analyzer(p, W, H, tcs, 100.0, use_w, 2.0)
        assert np.array_equal(sp.assign0.cpu().numpy(), ref["assign0"])
        np.testing.assert_allclose(sp.hist0.cpu().numpy(), ref["hist0"], rtol=RTOL, atol=ATOL)
        np.testing.assert_allclose(sp.entropy.cpu().numpy(), ref["entropy"], rtol=RTOL, atol=ATOL)
        tr = e.transition(dev(p))
        tref = orc.transition_analyzer(p, W, H, tcs)
        assert np.array_equal(tr.pairs0.cpu().numpy(), tref["pairs0"])
        assert np.array_equal(tr.prev_count0.cpu().numpy(), tref["prev_count0"])
        np.testing.assert_allclose(tr.entropy.cpu().numpy(), tref["entropy"], rtol=RTOL, atol=ATOL, equal_nan=True)
        h = e.spatial_host(p)
        assert np.array_equal(h["entropy"], sp.entropy.cpu().numpy())
        e.close()


def test_weight_table_budget_decides_the_regime(vet):
    """A weighted handle on a 1920x1080 video keeps per-cell tables while its weight columns stay under the budget
    (201 tiles at fov = 120: ~105 M entries); the reference's default five tile counts (1424 tiles in all) exceed it and
    run the direct per-sample regime."""
    small = engine(vet, [200], fov=120.0, use_w=True, W=1920, H=1080)
    assert small.cell_lut(0).shape == (1081, 1921)
    small.close()
    big = engine(vet, [20, 50, 100, 250, 1000], fov=120.0, use_w=True, W=1920, H=1080)
    with pytest.raises(vet.UnsupportedConfigurationError):
        big.cell_lut(0)
    big.close()


def test_analyzers_end_to_end_vs_reference(vet, tmp_path):
    """process_directory -> compute_entropy of both analyzers on CSV directories, against the
    rows the reference's analyzers produced (fixtures), incl. the ragged directory."""
    import pandas as pd
    a = load_golden("analyzers")
    g = group_keys(a)
    rag = tmp_path / "ragged"; rag.mkdir()
    pd.DataFrame({"time": [5.0, 5.1, 5.2, 5.3], "2dmu": [.5, .5, .6, .7], "2dmv": [.5] * 4}).to_csv(rag / "a.csv", index=False)
    pd.DataFrame({"time": [9.0, 9.1, 9.14, 9.3], "2dmu": [.1, .2, .3, .4], "2dmv": [.2] * 4}).to_csv(rag / "b.csv", index=False)
    pd.DataFrame({"time": [1.2, 1.0, 1.1], "2dmu": [.9] * 3, "2dmv": [.9] * 3}).to_csv(rag / "c.csv", index=False)
    d10 = tmp_path / "dir10"; d10.mkdir()
    names = [str(n) for n in g["dir10_default"]["order"]]
    for n in names:
        arr = a[f"dir10/{n}"]
        pd.DataFrame({"time": arr[:, 0], "2dmu": arr[:, 1], "2dmv": arr[:, 2]}).to_csv(d10 / f"{n}.csv", index=False)
    runs = [("ragged", rag, ["a", "b", "c"], [20], vet.EntropyConfig()),
            ("dir10_default", d10, names, [20, 50], vet.EntropyConfig()),
            ("dir10_unw", d10, names[::-1], [50, 20, 200], vet.EntropyConfig(fov_angle=90.0, use_weight_distribution=False))]
    for tag, directory, order, tcs, ec in runs:
        cfg = vet.AnalyzerConfig(tile_counts=tcs, output_dir=tmp_path / "out", entropy_config=ec)
        sa = vet.SpatialEntropyAnalyzer(cfg)
        sa.process_directory(directory, order=order)
        df = sa.compute_entropy()
        ref = g[tag]
        assert np.array_equal(df["time"].to_numpy(), ref["sp_time"])
        np.testing.assert_allclose(df["entropy"].to_numpy(), ref["sp_entropy"], rtol=RTOL, atol=ATOL)
        centres = sa._fibonacci_vectors[tcs[0]]
        for r in range(len(df)):
            hist = np.zeros(len(centres))
            for ct, w in df["tile_weights"][r].items():
                hist[centres.index(ct)] = w
            np.testing.assert_allclose(hist, ref["sp_hist0"][r], rtol=RTOL, atol=ATOL)
            asg = np.full(len(order), 0xFFFF)
            for k, t in df["tile_assignments"][r].items():
                asg[order.index(k)] = t
            assert np.array_equal(asg, ref["sp_assign0"][r])
        ta = vet.TransitionEntropyAnalyzer(cfg)
        ta.process_directory(directory, order=order)
        if tag == "ragged":   # the last pair has one common user -> NaN, no exception
            tdf = ta.compute_entropy()
        else:
            tdf = ta.compute_entropy()
        assert np.array_equal(tdf["time"].to_numpy(), ref["tr_time"])
        np.testing.assert_allclose(tdf["entropy"].to_numpy(), ref["tr_entropy"], rtol=RTOL, atol=ATOL, equal_nan=True)
        for r in range(len(tdf)):
            pc = np.zeros(len(centres), dtype=np.int64)
            for ct, w in tdf["tile_weights"][r].items():
                pc[centres.index(ct)] = w
            assert np.array_equal(pc, ref["tr_prev_count0"][r])
    sa.create_visualization("e2e_test")
    assert (tmp_path / "out" / "e2e_test.csv").exists()


@pytest.mark.parametrize("use_w,tcs,F,U", [(True, [200], 40, 20_000), (False, [50, 200, 1000], 12, 30_000), (True, [200, 20], 600, 3000)])
def test_cuda_graph_replay_equals_eager_calls(vet, use_w, tcs, F, U):
    """From the third identical call on a capturable stream, spatial / transition / analyze replay their launch sequence
    as one CUDA graph: same bits as the eager calls, also after the input changed in place, and a different call in
    between (other buffers -> other scratch sizes) does not corrupt the replay."""
    import bench
    e = engine(vet, tcs, fov=90.0, use_w=use_w)
    p = bench.synth_on_device(torch, F, U, 4242 + U, torch.device("cuda"))
    p[2, ::11, 1] = float("nan")
    q = bench.synth_on_device(torch, F, U, 777, torch.device("cuda"))
    eager = {}
    for name, x in (("p", p), ("q", q)):
        sp, tr = e.analyze(x)
        eager[name] = (sp, tr, e.spatial(x), e.transition(x))
    assert e.graph_replays() == 0, "calls on the legacy default stream stay eager"
    s = torch.cuda.Stream()
    buf = p.clone()
    with torch.cuda.stream(s):
        outs = []
        sp_out = e.spatial(buf)     # the same output tensors are passed to every call below: same key
        tr_out = e.transition(buf)
        for it in range(6):
            if it == 4:
                buf.copy_(q)                                  # new data in the same buffer: the graph reads it
            sp_i = e.spatial(buf, out=sp_out)
            tr_i = e.transition(buf, out=tr_out)
            if it == 2:
                e.spatial(q[: F // 2])                        # another shape in between
            outs.append((sp_i.entropy.clone(), sp_i.assign0.clone(), tr_i.entropy.clone(), tr_i.prev_count0.clone()))
        s.synchronize()
    assert e.poll_flags() == 0
    assert e.graph_replays() >= 6, e.graph_replays()
    for it, (se, sa, te, tc) in enumerate(outs):
        ref = eager["q" if it >= 4 else "p"]
        assert torch.equal(se, ref[2].entropy) and torch.equal(sa, ref[2].assign0), it
        assert torch.equal(te.nan_to_num(-1), ref[3].entropy.nan_to_num(-1)) and torch.equal(tc, ref[3].prev_count0), it
    e.set_option("cuda_graph", "off")
    with torch.cuda.stream(s):
        n0 = e.graph_replays()
        e.spatial(buf, out=sp_out)
        s.synchronize()
    assert e.graph_replays() == n0
    e.close()


def test_analyzer_results_are_lazy_at_scale(vet, tmp_path):
    """SpatialEntropyAnalyzer.compute_entropy() on a configs[2]-size video (100k users x 3600 frames, 4.3 GB on the
    host): the DataFrame comes back in seconds because the per-frame `tile_weights` / `tile_assignments` dicts
    (SA:152-163) are views that build themselves on access; a row that is read equals the eagerly built dict."""
    import time
    import bench
    F, U = 3600, 100_000
    packed = bench.synth_on_device(torch, F, U, 4711, torch.device("cuda")).cpu().numpy()
    cfg = vet.AnalyzerConfig(tile_counts=[200], output_dir=tmp_path, entropy_config=vet.EntropyConfig(fov_angle=90.0))
    sa = vet.SpatialEntropyAnalyzer(cfg)
    sa.load_packed(packed, identifiers=[f"u{u}" for u in range(U)])
    t0 = time.perf_counter()
    df = sa.compute_entropy()
    dt = time.perf_counter() - t0
    assert dt < 30.0, f"compute_entropy took {dt:.1f} s"
    assert list(df.columns) == ["time", "entropy", "tile_weights", "tile_assignments"] and len(df) == F
    assert all(row._d is None for row in df["tile_assignments"]), "no per-frame dict built before it is read"
    ref = sa.engine.spatial(dev(packed[1000:1002]))
    w = df["tile_weights"][1000]
    a = df["tile_assignments"][1001]
    assert len(a) == U and a["u5"] == int(ref.assign0[1, 5]) and "nobody" not in a
    centres = sa._fibonacci_vectors[200]
    h = ref.hist0[0].cpu().numpy()
    want = {centres[i]: float(h[i]) for i in np.flatnonzero(h)}   # two frames alone: the FP64 weighted kernel
    assert set(w) == set(want)
    np.testing.assert_allclose([w[k] for k in want], list(want.values()), rtol=RTOL)
    assert df["tile_weights"][1000] == dict(w)                    # a view compares equal to the dict it stands for
    np.testing.assert_allclose(df["entropy"][1000], float(ref.entropy[0]), rtol=RTOL)
    sa.create_visualization("lazy_case")   # the CSV writer of SA:211-219 only needs time and entropy
    assert (tmp_path / "lazy_case.csv").exists()


@pytest.mark.parametrize("use_w,tcs", [(True, [200, 20]), (False, [50, 200, 1000]), (False, [200])])
def test_analyze_equals_separate_stages(vet, use_w, tcs):
    """vet_analyze (one pass over the input) == vet_spatial + vet_transition: integer outputs bit for bit,
    entropies to 1e-12 (the unweighted stand-alone path reduces in a different order)."""
    p = synth(7, 9001, 31337, missing=0.05)
    e = engine(vet, tcs, fov=90.0, use_w=use_w)
    sp, tr = e.analyze(dev(p))
    assert e.poll_flags() == 0
    sp_ref = e.spatial(dev(p))
    tr_ref = e.transition(dev(p))
    for a, b in ((sp.assign0, sp_ref.assign0), (tr.entropy, tr_ref.entropy), (tr.per_k, tr_ref.per_k),
                 (tr.prev_count0, tr_ref.prev_count0), (tr.pairs0, tr_ref.pairs0)):
        assert np.array_equal(a.cpu().numpy(), b.cpu().numpy(), equal_nan=True)
    for a, b in ((sp.entropy, sp_ref.entropy), (sp.per_k, sp_ref.per_k), (sp.hist0, sp_ref.hist0)):
        np.testing.assert_allclose(a.cpu().numpy(), b.cpu().numpy(), rtol=1e-12, atol=0)
    ref = orc.spatial_analyzer(p, W0, H0, tcs, 90.0, use_w, 2.0)
    np.testing.assert_allclose(sp.entropy.cpu().numpy(), ref["entropy"], rtol=RTOL, atol=ATOL)
    e.close()


@pytest.mark.parametrize("use_w", [True, False])
def test_many_frames_cross_internal_batches(vet, use_w):
    """More frames than one internal scratch batch holds (the cell-histogram scratch is capped at
    1 GiB = ~13k frames): batch offsets, unaligned batch bases and the transition halo frame."""
    F, U = 27001, 5
    p = synth(F, U, 777, iid=True, missing=0.1)
    e = engine(vet, [20], fov=100.0, use_w=use_w)
    sp, tr = e.analyze(dev(p))
    sp2 = e.spatial(dev(p))
    assert e.poll_flags() == 0
    px, py, ok = orc.decode(p[..., 1], p[..., 2], W0, H0)
    lut = orc.cell_luts(W0, H0, [20])[0]
    assign = np.where(ok, lut[py * 101 + px], 0xFFFF).astype(np.uint16)
    assert np.array_equal(sp.assign0.cpu().numpy(), assign) and np.array_equal(sp2.assign0.cpu().numpy(), assign)
    sel = np.r_[0:40, 13100:13140, F - 40:F]          # around the batch boundaries and both ends
    ref = orc.spatial_analyzer(p[sel], W0, H0, [20], 100.0, use_w, 2.0)
    np.testing.assert_allclose(sp.entropy.cpu().numpy()[sel], ref["entropy"], rtol=RTOL, atol=ATOL, equal_nan=True)
    np.testing.assert_allclose(sp2.entropy.cpu().numpy()[sel], ref["entropy"], rtol=RTOL, atol=ATOL, equal_nan=True)
    np.testing.assert_allclose(sp.hist0.cpu().numpy()[sel], ref["hist0"], rtol=RTOL, atol=ATOL)
    pairs = tr.pairs0.cpu().numpy()
    both = ok[:-1] & ok[1:]
    assert np.array_equal(pairs[..., 0], np.where(both, assign[:-1], 0xFFFF))
    assert np.array_equal(pairs[..., 1], np.where(both, assign[1:], 0xFFFF))
    rows = np.r_[0:30, 13090:13140, F - 31:F - 1]
    for r in rows:
        if both[r].sum() == 0:
            continue
        e_ref, m_ref = orc.transition_entropy(assign[r][both[r]].astype(int), assign[r + 1][both[r]].astype(int), 21)
        np.testing.assert_allclose(float(tr.entropy[r]), e_ref, rtol=RTOL, atol=ATOL, equal_nan=True)
        assert np.array_equal(tr.prev_count0[r].cpu().numpy(), m_ref)
    e.poll_flags()
    e.close()


def test_full_size_properties_configs2(vet):
    """BASELINE configs[2] at FULL size (100k users x 3600 frames, 201 tiles, fov=90): checks that do
    not need the oracle -- every assignment equals the exhaustive LUT of its cell, entropies lie in
    [0,1], reruns are bit-identical, and sampled frames match an independent dense evaluation."""
    import bench
    F, U = 3600, 100_000
    p = bench.synth_on_device(torch, F, U, 20260000 + 3000, torch.device("cuda"))
    e = engine(vet, [200], fov=90.0)
    a = e.spatial(p)
    assert e.poll_flags() == 0
    b = e.spatial(p)
    assert torch.equal(a.entropy, b.entropy) and torch.equal(a.hist0, b.hist0) and torch.equal(a.assign0, b.assign0)
    del b
    ent = a.entropy.cpu().numpy()
    assert np.isfinite(ent).all() and ((ent > 0) & (ent <= 1)).all()
    lut = torch.from_numpy(e.cell_lut(0).astype(np.int16)).cuda().ravel()
    for f0 in range(0, F, 600):     # in slabs to bound the temporaries
        sl = p[f0:f0 + 600]
        cell = (sl[..., 2].double() * 200).to(torch.int64) * 101 + (sl[..., 1].double() * 100).to(torch.int64)
        assert torch.equal(a.assign0[f0:f0 + 600].to(torch.int16), lut[cell])
        del cell
    for f in (0, 1799, 3599):       # weighted histogram of whole frames vs the dense per-user weight kernel
        vec, _ = e.decode(p[f:f + 1])
        dense = torch.zeros(201, dtype=torch.float64, device="cuda")
        for u0 in range(0, U, 25_000):
            dense += e.tile_weights(vec[0, u0:u0 + 25_000], 0).sum(0)
        np.testing.assert_allclose(a.hist0[f].cpu().numpy(), dense.cpu().numpy(), rtol=RTOL, atol=ATOL)
    e.close()


# ---------------------------------------------------------------------------------
# tensor-core weighted histogram (k_whist_i8): exact integer GEMM over count byte planes and
# 39-bit fixed-point weight slices.  Stated tolerance of this path: entropies 1e-9 relative
# (north_star); weighted histogram entries |d| <= users * 2^-40 absolute (weight quantisation)
# on top of the 1e-9 relative bar.  The handle option "weighted_kernel" (vet_set_option) forces the
# kernel for frame counts below the heuristic threshold.
# ---------------------------------------------------------------------------------
I8_QUANT = 2.0 ** -40


@pytest.mark.parametrize("cfg", [
    dict(F=6, U=3000, tcs=[200], fov=90.0),
    dict(F=4, U=2000, tcs=[20, 50], fov=120.0, iid=True, missing=0.2),
    dict(F=3, U=1500, tcs=[250, 1000], fov=120.0),                      # 6 and 21 N blocks, u16 LUT
    dict(F=5, U=701, tcs=[50], fov=360.0, pf=3.0, iid=True),            # every tile sees every cell
    dict(F=5, U=700, tcs=[50], fov=10.0, pf=0.5, iid=True),             # most users outside every FOV
    dict(F=131, U=257, tcs=[200, 50], fov=90.0, iid=True, missing=0.05),  # two frame blocks, partial second one
    dict(F=3, U=70000, tcs=[200], fov=90.0, iid=True),                  # frames in several chunks: k_cnt_planes
])
def test_weighted_tensor_core_path_vs_oracle(vet, cfg):
    p = synth(cfg["F"], cfg["U"], 4100 + cfg["U"], cfg.get("iid", False), cfg.get("missing", 0.0))
    pf = cfg.get("pf", 2.0)
    e = engine(vet, cfg["tcs"], cfg["fov"], True, pf)
    e.set_option("weighted_kernel", "i8")
    sp = e.spatial(dev(p))
    assert e.poll_flags() == 0
    ref = orc.spatial_analyzer(p, W0, H0, cfg["tcs"], cfg["fov"], True, pf)
    assert np.array_equal(sp.assign0.cpu().numpy(), ref["assign0"])
    np.testing.assert_allclose(sp.hist0.cpu().numpy(), ref["hist0"], rtol=RTOL, atol=cfg["U"] * I8_QUANT)
    np.testing.assert_allclose(sp.per_k.cpu().numpy(), ref["per_k"], rtol=RTOL, atol=ATOL, equal_nan=True)
    np.testing.assert_allclose(sp.entropy.cpu().numpy(), ref["entropy"], rtol=RTOL, atol=ATOL, equal_nan=True)
    e.set_option("weighted_kernel", "fp64")
    sp64 = e.spatial(dev(p))
    np.testing.assert_allclose(sp.hist0.cpu().numpy(), sp64.hist0.cpu().numpy(), rtol=RTOL, atol=cfg["U"] * I8_QUANT)
    np.testing.assert_allclose(sp.entropy.cpu().numpy(), sp64.entropy.cpu().numpy(), rtol=RTOL, atol=ATOL, equal_nan=True)
    e.close()


def test_weighted_default_dispatch_sparse_frames(vet):
    """The DEFAULT dispatch (no kernel pinned) on 600 frames of 1-5 users each -- the tensor-core histogram from 384
    frames per call on -- against the oracle: the support of every hist0 row (tiles with d < fov/2, EU:133) is the
    oracle's, entries above the quantisation floor users * 2^-39 / 1e-9 agree to a pure relative 1e-9, all entries to
    users * 2^-39 absolute, entropies to 1e-9; and the first 300 frames on their own (FP64 kernel: fewer than 384
    frames) give the same support and the same values to 1e-9."""
    rng = np.random.default_rng(4242)
    F, U = 600, 5
    p = synth(F, U, 9191, iid=True)
    present = rng.integers(1, U + 1, F)                      # 1..5 users per frame
    for f in range(F):
        p[f, present[f]:, 1:] = np.nan
    e = engine(vet, [200, 50], fov=90.0)
    assert e.get_option("weighted_kernel") == "auto"
    e.profile(True)
    d = e.spatial(dev(p))
    assert e.poll_flags() == 0
    ref = orc.spatial_analyzer(p, W0, H0, [200, 50], 90.0, True, 2.0)
    h, rh = d.hist0.cpu().numpy(), ref["hist0"]
    assert np.array_equal(h > 0, rh > 0), "support of the weighted histogram rows"
    quantum = 2.0 ** -39
    floor = present[:, None] * quantum / 1e-9
    big = rh > floor
    assert big.sum() > 0.8 * (rh > 0).sum()   # the entries below the floor are the weights at the very edge of the FOV
    np.testing.assert_allclose(h[big], rh[big], rtol=1e-9, atol=0)
    assert np.all(np.abs(h - rh) <= present[:, None] * quantum)
    np.testing.assert_allclose(d.entropy.cpu().numpy(), ref["entropy"], rtol=RTOL, atol=ATOL)
    assert np.array_equal(d.assign0.cpu().numpy(), ref["assign0"])
    short = e.spatial(dev(p[:300]))                           # fewer than VET_I8_MIN_FRAMES = 384 frames: the FP64 kernel
    hs = short.hist0.cpu().numpy()
    assert np.array_equal(hs > 0, h[:300] > 0)
    np.testing.assert_allclose(hs[big[:300]], h[:300][big[:300]], rtol=1e-9, atol=0)
    np.testing.assert_allclose(short.entropy.cpu().numpy(), d.entropy.cpu().numpy()[:300], rtol=RTOL, atol=ATOL)
    e.close()


def test_weighted_tensor_core_count_planes(vet):
    """Counts of 256 and more (second byte plane) and of 65536 and more (third plane, second GEMM
    pass), rows of the higher planes left dirty by one call and cleaned by the next, analyze() ==
    spatial(); all against the FP64 kernel on the same input."""
    import bench
    F, U = 260, 70_000
    e = engine(vet, [200], fov=90.0)
    hot = bench.synth_on_device(torch, F, U, 4242, torch.device("cuda"))
    hot[:, :66_000, 1] = 0.25     # one cell holds 66k users of every frame
    hot[:, :66_000, 2] = 0.75
    hot[:, 66_000:67_000, 1] = 0.5  # another one 1000
    hot[:, 66_000:67_000, 2] = 0.5
    cold = bench.synth_on_device(torch, F - 60, U, 4243, torch.device("cuda"))
    res = {}
    for impl in ("fp64", "i8"):
        e.set_option("weighted_kernel", impl)
        a = e.spatial(hot)
        b = e.spatial(cold)          # same plane rows as `hot`, now without large counts
        c, _ = e.analyze(hot)
        res[impl] = (a, b, c)
    assert e.poll_flags() == 0
    for x, y in zip(res["fp64"], res["i8"]):
        assert torch.equal(x.assign0, y.assign0)
        np.testing.assert_allclose(y.hist0.cpu().numpy(), x.hist0.cpu().numpy(), rtol=RTOL, atol=U * I8_QUANT)
        np.testing.assert_allclose(y.entropy.cpu().numpy(), x.entropy.cpu().numpy(), rtol=RTOL, atol=0)
    assert torch.equal(res["i8"][0].hist0, res["i8"][2].hist0) and torch.equal(res["i8"][0].entropy, res["i8"][2].entropy)
    # exactness of the integer part: a frame whose users all sit on cell centres that coincide with
    # nothing special still sums to the same total weight in both kernels up to the quantisation
    tot64, tot8 = res["fp64"][0].hist0.sum(1), res["i8"][0].hist0.sum(1)
    np.testing.assert_allclose(tot8.cpu().numpy(), tot64.cpu().numpy(), rtol=1e-11)
    e.close()


def test_tensor_core_histogram_split_over_the_cells_equals_one_cta_per_tile(vet):
    """k_whist_i8 with few output tiles splits the cells of a tile over several CTAs (int32 partial sums in
    global memory, added and turned into the rows by k_whist_i8_finish): the rows of the first 200 / 450 frames
    computed on their own (split) carry the bits of the same frames inside an 1800-frame call (one CTA per tile), call
    after call, with large counts (second byte plane) in some frames, for two tile counts."""
    import bench
    F, U = 1800, 3000
    p = bench.synth_on_device(torch, F, U, 777, torch.device("cuda"))
    p[100:140, :400, 1] = 0.25          # 400 users in one cell: the second count plane in frame block 0
    p[100:140, :400, 2] = 0.75
    p[7, ::3, 1] = float("nan")
    e = engine(vet, [200, 50], fov=90.0)
    e.set_option("weighted_kernel", "i8")
    full = e.spatial(p)
    for n in (200, 450, 200):
        part = e.spatial(p[:n].contiguous())
        assert torch.equal(part.hist0, full.hist0[:n]), n
        assert torch.equal(part.entropy, full.entropy[:n]) and torch.equal(part.per_k, full.per_k[:, :n]), n
    sp, _ = e.analyze(p[:450].contiguous())
    assert torch.equal(sp.hist0, full.hist0[:450]) and torch.equal(sp.entropy, full.entropy[:450])
    e.set_option("weighted_kernel", "fp64")
    ref = e.spatial(p[:450].contiguous())
    np.testing.assert_allclose(sp.hist0.cpu().numpy(), ref.hist0.cpu().numpy(), rtol=RTOL, atol=U * I8_QUANT)
    np.testing.assert_allclose(sp.entropy.cpu().numpy(), ref.entropy.cpu().numpy(), rtol=RTOL, atol=0)
    assert e.poll_flags() == 0
    e.close()


@pytest.mark.parametrize("U", [100_000, 20_001])
def test_transition_two_pass_kernel_equals_three_pass_kernel(vet, U):
    """k_transition3 (two passes, one launch per tile count; dense table for 201 tiles, shared-memory
    hash for 501/1001, rows that overflow it handed to k_transition2) against k_transition2 alone on
    frames too large for the oracle: counts and pairs bit-exact, entropies to 1e-12."""
    import bench
    F = 40
    p = bench.synth_on_device(torch, F, U, 515, torch.device("cuda"))
    p[5, ::7, 1] = float("nan")                                   # missing users
    g = torch.Generator(device="cuda").manual_seed(99)
    p[20:23, :, 1:] = torch.rand((3, U, 2), generator=g, device="cuda")   # iid frames: ~U distinct pairs -> overflow rows
    e = engine(vet, [200, 500, 1000], use_w=False)
    res = {}
    for impl in ("v2", "v3"):
        e.set_option("transition_kernel", "v2" if impl == "v2" else "auto")
        res[impl] = e.transition(p)
        assert e.poll_flags() == 0
    a, b = res["v2"], res["v3"]
    assert torch.equal(a.pairs0, b.pairs0) and torch.equal(a.prev_count0, b.prev_count0)
    np.testing.assert_allclose(b.per_k.cpu().numpy(), a.per_k.cpu().numpy(), rtol=1e-12, atol=0)
    np.testing.assert_allclose(b.entropy.cpu().numpy(), a.entropy.cpu().numpy(), rtol=1e-12, atol=0)
    e.close()


@pytest.mark.parametrize("F,U,tcs", [
    (3, 66_000, [200]),          # 2 pairs, clusters of 8, tile ids straight from the streaming kernel
    (3, 40_001, [200, 20]),      # clusters of 4, odd U (scalar loads), rows relabelled to tile ids
    (152, 16_384, [200]),        # 151 pairs: one full round of k_transition4 + 3 pairs on clusters of 2
    (21, 131_072, [100, 200]),   # 20 pairs: more than the co-resident clusters of 8
])
def test_one_pass_cluster_tail_equals_single_cta(vet, F, U, tcs):
    """k_transition4<true> (the users of one frame pair split over a thread-block cluster, for the pairs left after
    the full rounds) against the one-pass kernel without it and against k_transition3 alone: every output bit for bit,
    transition() and analyze(); the small cases also against the oracle."""
    import bench
    p = bench.synth_on_device(torch, F, U, 616 + U, torch.device("cuda"))
    p[1, ::5, 1] = float("nan")                                   # missing users
    g = torch.Generator(device="cuda").manual_seed(7)
    p[F - 2:, :, 1:] = torch.rand((2, U, 2), generator=g, device="cuda")   # iid frames: every row of the table in use
    e = engine(vet, tcs, use_w=False)
    res = {}
    e.profile(True)
    # force: also below the frame size from which the host picks the clusters by itself; v3: one CTA per pair
    for name, tk, cl in (("v3", "v3", "off"), ("0", "auto", "off"), ("force", "auto", "force")):
        e.set_option("transition_kernel", tk)
        e.set_option("cluster_tail", cl)
        tr = e.transition(p)
        _, tr2 = e.analyze(p)
        assert e.poll_flags() == 0
        res[name] = (tr, tr2, e.profile_read()["transition_tail"][1])
    e.profile(False)
    # transition_tail also counts the k_transition3 pass over the pairs k_transition4 flags, once per tile count and call
    assert res["v3"][2] == 0 and res["force"][2] - res["0"][2] == 2 * len(tcs), "one cluster launch per tile count and call"
    # the same without the shortcuts of k_transition3: missing-user tests kept for complete frames, pair scratch kept
    e.set_option("transition_kernel", "v3")
    e.set_option("cluster_tail", "off")
    e.set_option("t3_assume_missing", "on")
    e.set_option("t3_pair_scratch", "on")
    plain = e.transition(p)
    e.set_option("t3_assume_missing", "off")
    e.set_option("t3_pair_scratch", "off")
    assert torch.equal(plain.pairs0, res["v3"][0].pairs0) and torch.equal(plain.prev_count0, res["v3"][0].prev_count0)
    assert np.array_equal(plain.entropy.cpu().numpy(), res["v3"][0].entropy.cpu().numpy(), equal_nan=True)
    for name in ("0", "force"):
        for a, b in ((res["v3"][0], res[name][0]), (res["v3"][0], res[name][1])):
            assert torch.equal(a.pairs0, b.pairs0) and torch.equal(a.prev_count0, b.prev_count0), name
            assert np.array_equal(a.per_k.cpu().numpy(), b.per_k.cpu().numpy(), equal_nan=True), name
            assert np.array_equal(a.entropy.cpu().numpy(), b.entropy.cpu().numpy(), equal_nan=True), name
    if F <= 3:
        ref = orc.transition_analyzer(p.cpu().numpy(), W0, H0, tcs, mode="literal")
        b = res["force"][0]
        assert np.array_equal(b.pairs0.cpu().numpy(), ref["pairs0"])
        assert np.array_equal(b.prev_count0.cpu().numpy(), ref["prev_count0"])
        np.testing.assert_allclose(b.entropy.cpu().numpy(), ref["entropy"], rtol=RTOL, atol=ATOL, equal_nan=True)
    e.close()


@pytest.mark.parametrize("n,alphabet,U,cap", [(200, 3, 2400, 0), (200, 40, 2400, 0), (20, 21, 999, 0), (200, 12, 640, 64), (100, 101, 5000, 0)])
def test_one_pass_kernel_on_random_tile_patterns_vs_oracle(vet, n, alphabet, U, cap):
    """Users that hop between a few tiles chosen at random (not lattice neighbours: ranked and unranked deltas mixed,
    many users per (prev, cur) pair, skewed tile probabilities, missing users) -- the order-dependent bookkeeping of
    EU:278-318 through k_transition4's first/second/count tables and its sorted list, against the literal oracle:
    pairs and counts bit-exact, entropies to 1e-9; and bit for bit against the two-pass kernels."""
    rng = np.random.default_rng(1000 * n + alphabet)
    e = engine(vet, [n], use_w=False)
    T = e.num_tiles[0]
    rep = _tile_to_sample(e.cell_lut(0))
    tiles = rng.choice(T, size=min(alphabet, T), replace=False)
    prob = rng.dirichlet(np.full(len(tiles), 0.4))
    F = 7
    seq = rng.choice(tiles, size=(F, U), p=prob)
    stay = rng.uniform(size=(F, U)) < 0.6                      # most users keep their tile, like real viewers
    for f in range(1, F):
        seq[f] = np.where(stay[f], seq[f - 1], seq[f])
    packed = np.zeros((F, U, 3), dtype=np.float64)
    lut_mu = np.array([rep[int(t)][0] if int(t) in rep else 0.5 for t in range(T)])
    lut_mv = np.array([rep[int(t)][1] if int(t) in rep else 0.5 for t in range(T)])
    packed[..., 1] = lut_mu[seq]
    packed[..., 2] = lut_mv[seq]
    miss = rng.uniform(size=(F, U)) < 0.03
    miss[:, 0] = False
    packed[miss, 1] = np.nan
    e.set_option("t4_list_cap", cap)
    res = {}
    for impl in ("auto", "v3"):
        e.set_option("transition_kernel", impl)
        res[impl] = e.transition(dev(packed))
        assert e.poll_flags() == 0
    a, b = res["auto"], res["v3"]
    assert torch.equal(a.pairs0, b.pairs0) and torch.equal(a.prev_count0, b.prev_count0)
    assert np.array_equal(a.entropy.cpu().numpy(), b.entropy.cpu().numpy(), equal_nan=True)
    ref = orc.transition_analyzer(packed, W0, H0, [n], mode="literal")
    assert np.array_equal(a.pairs0.cpu().numpy(), ref["pairs0"])
    assert np.array_equal(a.prev_count0.cpu().numpy(), ref["prev_count0"])
    np.testing.assert_allclose(a.entropy.cpu().numpy(), ref["entropy"], rtol=RTOL, atol=ATOL, equal_nan=True)
    e.close()


@pytest.mark.parametrize("cfg", [
    dict(F=40, U=100_000, tcs=[200], use_w=False),                                  # tile ids from the streaming kernel, 512-thread CTAs
    dict(F=24, U=100_000, tcs=[200, 500, 1000], use_w=False),                       # LUT staged / from global memory, 1024-thread CTAs for 1001 tiles
    dict(F=12, U=5000, tcs=[200], use_w=True, dtype=np.float64, missing=0.1),
    dict(F=7, U=3001, tcs=[100, 20], use_w=False, missing=0.02),                    # odd U: scalar loads
    dict(F=9, U=600, tcs=[200], use_w=False, iid=True),                             # iid: most users on the list of unranked deltas (sorted path)
    dict(F=5, U=3000, tcs=[50], use_w=True, iid=True),                              # iid: lists overflow -> pairs redone by the two-pass kernels
    dict(F=9, U=4000, tcs=[200, 500], use_w=False, cap=8),                          # tiny list: a mix of pairs kept and pairs handed on
    dict(F=2, U=9, tcs=[200], use_w=False),
    dict(F=6, U=4003, tcs=[700, 800, 900, 1000], use_w=False, missing=0.05),        # relabelling: four lookup tables in shared memory for one pass over the cell ids; odd U
    dict(F=4, U=66_000, tcs=[200], use_w=False, cluster="force"),                  # 3 pairs on clusters of 8 CTAs (tables merged through DSMEM)
    dict(F=152, U=16_384, tcs=[200, 500], use_w=False, cluster="force"),           # one full round + 3 pairs on clusters of 4
    dict(F=10, U=600_000, tcs=[200], use_w=True),                                   # 9 pairs of 600k users: clusters picked by the host itself
])
def test_one_pass_transition_kernel_equals_two_pass_kernels(vet, cfg):
    """k_transition4 (one walk over the users: [16][T] tables of ranked tile deltas with first/second user and count,
    sorted list of the unranked users, pairs with a full list handed to k_transition3) against k_transition3 alone on
    the same tensors: every output bit for bit, for transition() and analyze(); small cases also against the oracle."""
    import bench
    F, U, tcs = cfg["F"], cfg["U"], cfg["tcs"]
    if U >= 50_000:
        p = bench.synth_on_device(torch, F, U, 717 + U, torch.device("cuda"))
        p[3, ::9, 1] = float("nan")
        g = torch.Generator(device="cuda").manual_seed(5)
        p[F - 3:F - 1, :700, 1:] = torch.rand((2, 700, 2), generator=g, device="cuda")      # a burst of large jumps: list entries
        if F >= 8:
            p[F - 6:F - 4, :, 1:] = torch.rand((2, U, 2), generator=g, device="cuda")       # iid frames: lists overflow
    else:
        p = dev(synth(F, U, 818 + U, iid=cfg.get("iid", False), missing=cfg.get("missing", 0.0), dtype=cfg.get("dtype", np.float32)))
    e = engine(vet, tcs, fov=90.0, use_w=cfg["use_w"])
    e.set_option("weighted_kernel", "fp64")
    e.set_option("t4_list_cap", cfg.get("cap", 0))
    res = {}
    e.profile(True)
    for impl in ("v3", "auto"):
        e.set_option("transition_kernel", impl)
        e.set_option("cluster_tail", cfg.get("cluster", "auto") if impl == "auto" else "off")
        tr = e.transition(p)
        sp, tr2 = e.analyze(p)
        assert e.poll_flags() == 0
        res[impl] = (tr, tr2, sp)
        tail_launches = e.profile_read()["transition_tail"][1]
    e.profile(False)
    if "cluster" in cfg or U >= 500_000:
        assert tail_launches >= 2 * len(tcs), "the cluster launch of the one-pass kernel ran (besides the two-pass pass over flagged pairs)"
    for i in (0, 1):
        a, b = res["v3"][i], res["auto"][i]
        assert torch.equal(a.pairs0, b.pairs0) and torch.equal(a.prev_count0, b.prev_count0)
        assert np.array_equal(a.per_k.cpu().numpy(), b.per_k.cpu().numpy(), equal_nan=True)
        assert np.array_equal(a.entropy.cpu().numpy(), b.entropy.cpu().numpy(), equal_nan=True)
    a, b = res["v3"][2], res["auto"][2]
    assert torch.equal(a.assign0, b.assign0) and torch.equal(a.hist0, b.hist0) and torch.equal(a.entropy, b.entropy)
    if F * U <= 100_000:
        ref = orc.transition_analyzer(p.cpu().numpy(), W0, H0, tcs, mode="literal")
        b = res["auto"][0]
        assert np.array_equal(b.pairs0.cpu().numpy(), ref["pairs0"])
        assert np.array_equal(b.prev_count0.cpu().numpy(), ref["prev_count0"])
        np.testing.assert_allclose(b.entropy.cpu().numpy(), ref["entropy"], rtol=RTOL, atol=ATOL, equal_nan=True)
    e.close()


# ---------------------------------------------------------------------------------
# latitude/longitude grid tiling (NaiveSpatialEntropyAnalyzer, NA:39-241 / EU:335-453)
# ---------------------------------------------------------------------------------
def _naive_golden():
    npz = load_golden("naive")
    out = {}
    for k in npz.files:
        case, _, field = k.rpartition("/")
        out.setdefault(case, {})[field] = npz[k]
    return out


def test_naive_cell_table_every_cell_vs_reference(vet):
    """The grid code of every reachable cell (the cell -> tile table the streaming kernels use) against the
    reference's find_naive_tile_index on its own decode chain, for six tile sizes."""
    g = _naive_golden()
    for name, c in g.items():
        if not name.startswith("cells/"):
            continue
        tw, th = (int(x) for x in name.split("/")[1].split("x"))
        e = vet.Engine(W0, H0, [1], vet.EntropyConfig(), naive_tiles=(tw, th))
        nlat1 = 180 // th + 1
        assert e.num_tiles[0] == (360 // tw + 1) * nlat1
        lut = e.cell_lut(0).astype(np.int64)
        assert np.array_equal(lut // nlat1, c["lon_idx"]) and np.array_equal(lut % nlat1, c["lat_idx"]), name
        e.close()


@pytest.mark.parametrize("case", ["n_30_w", "n_30_u", "n_45x90_u", "n_10x20_w", "n_360_u", "n_3_u", "n_120x60_one"])
def test_naive_frames_vs_reference_fixtures(vet, case, tmp_path):
    """Packed path (streaming kernels with the grid table) and the functional API on RadialPoint dicts
    (k_naive_points) against compute_naive_spatial_entropy of the live reference; -inf / NaN quirks of
    a single 360x180 tile included."""
    c = _naive_golden()[f"frames/{case}"]
    tw, th = (int(x) for x in c["tile"])
    use_w = bool(c["use_w"])
    cfg = vet.NaiveAnalyzerConfig(tile_width=tw, tile_height=th, output_dir=tmp_path,
                                  entropy_config=vet.EntropyConfig(use_weight_distribution=use_w))
    na = vet.NaiveSpatialEntropyAnalyzer(cfg)
    packed = c["packed"]
    for p in (packed.astype(np.float32), packed.astype(np.float64)):
        res = na.compute_entropy_packed(dev(p))
        np.testing.assert_allclose(res.entropy.cpu().numpy(), c["entropy"], rtol=RTOL, atol=ATOL, equal_nan=True)
        nlat1 = 180 // th + 1
        code = res.assign0.cpu().numpy().astype(np.int64)
        ok = code != 0xFFFF
        assert np.array_equal(np.where(ok, code // nlat1, -1), c["keys"][..., 0])
        assert np.array_equal(np.where(ok, code % nlat1, -1), c["keys"][..., 1])
        hist = res.hist0.cpu().numpy()
        assert np.array_equal((hist > 0).sum(1), c["nkeys"]) and np.array_equal(hist.sum(1), ok.sum(1))
    ref = orc.naive_analyzer(packed, W0, H0, tw, th, use_w)
    assert np.array_equal(res.hist0.cpu().numpy(), ref["hist0"]) and np.array_equal(res.assign0.cpu().numpy(), ref["assign0"])
    # functional API, frame 0
    px, py, ok0 = orc.decode(packed[0, :, 1], packed[0, :, 2], W0, H0)
    lon_t, lat_t = orc.axis_tables(W0, H0)
    pts = {f"u{u:05d}": (vet.RadialPoint(float(lon_t[px[u]]), float(lat_t[py[u]])) if ok0[u] else None) for u in range(len(ok0))}
    e, wts, asg = vet.compute_naive_spatial_entropy(pts, th, tw, vet.EntropyConfig(use_weight_distribution=use_w))
    np.testing.assert_allclose(e, c["entropy"][0], rtol=RTOL, atol=ATOL, equal_nan=True)
    assert len(wts) == c["nkeys"][0] and sum(wts.values()) == ok0.sum()
    for u in np.flatnonzero(ok0):
        assert asg[f"u{u:05d}"] == f"{c['keys'][0, u, 0]}_{c['keys'][0, u, 1]}"
        assert asg[f"u{u:05d}"] == vet.find_naive_tile_index(pts[f"u{u:05d}"], th, tw)


def test_naive_analyzer_end_to_end_and_errors(vet, tmp_path):
    import pandas as pd
    a = load_golden("analyzers")
    g = _naive_golden()
    d10 = tmp_path / "dir10"; d10.mkdir()
    names = [f"user{u:02d}" for u in range(10)]
    for n in names:
        arr = a[f"dir10/{n}"]
        pd.DataFrame({"time": arr[:, 0], "2dmu": arr[:, 1], "2dmv": arr[:, 2]}).to_csv(d10 / f"{n}.csv", index=False)
    for tw, th, use_w in ((30, 30, True), (45, 90, False)):
        cfg = vet.NaiveAnalyzerConfig(output_dir=tmp_path / "out", tile_width=tw, tile_height=th,
                                      entropy_config=vet.EntropyConfig(use_weight_distribution=use_w))
        na = vet.NaiveSpatialEntropyAnalyzer(cfg)
        na.process_directory(d10, order=names)
        df = na.compute_entropy()
        ref = g[f"analyzer/{tw}x{th}_{int(use_w)}"]
        assert np.array_equal(df["time"].to_numpy(), ref["time"])
        np.testing.assert_allclose(df["entropy"].to_numpy(), ref["entropy"], rtol=RTOL, atol=ATOL)
        assert df["tile_weights"].isna().all() and df["tile_assignments"].isna().all()   # NA:136-150
    na.create_visualization("naive_e2e")
    assert (tmp_path / "out" / "naive_e2e.csv").exists()
    # error behaviour (CFG:112-115, EU:404-417)
    with pytest.raises(ValueError):
        vet.NaiveAnalyzerConfig(tile_width=0, tile_height=30, output_dir=tmp_path / "out")
    pt = {"a": vet.RadialPoint(0.0, 0.0)}
    with pytest.raises(vet.ValidationError):
        vet.compute_naive_spatial_entropy({}, 30, 30, vet.EntropyConfig())
    with pytest.raises(vet.ValidationError):
        vet.compute_naive_spatial_entropy(pt, 7, 30, vet.EntropyConfig())
    with pytest.raises(vet.ValidationError):
        vet.compute_naive_spatial_entropy(pt, 30, 7, vet.EntropyConfig())
    bad = vet.NaiveSpatialEntropyAnalyzer(vet.NaiveAnalyzerConfig(tile_width=7, tile_height=30, output_dir=tmp_path / "out"))
    bad.load_packed(np.zeros((2, 3, 3)) + 0.5)
    with pytest.raises(vet.ValidationError):
        bad.compute_entropy()
    empty = vet.NaiveSpatialEntropyAnalyzer(vet.NaiveAnalyzerConfig(tile_width=30, tile_height=30, output_dir=tmp_path / "out"))
    p = np.zeros((2, 3, 3)) + 0.5
    p[1, :, 1] = np.nan
    empty.load_packed(p)
    with pytest.raises(vet.ValidationError, match="Empty radial points"):
        empty.compute_entropy()


# ---------------------------------------------------------------------------------
# full-size runs of the remaining BASELINE configs: size-independent properties + oracle on sampled rows
# ---------------------------------------------------------------------------------
def _cells_of(frame):
    """DU:261 in fp64 (exact for float32 inputs) with plain torch ops: [U] packed rows -> cell ids"""
    return (frame[:, 2].double() * H0).to(torch.int64) * (W0 + 1) + (frame[:, 1].double() * W0).to(torch.int64)


def test_full_size_properties_configs3(vet):
    """BASELINE configs[3] at FULL size (100k users x 3600 frames, tile_counts=[200,500,1000], transition entropy):
    users per previous tile sum to U, pairs equal the exhaustive LUT of the two frames' cells, the entropy is the
    mean over tile counts, reruns are bit-identical, and sampled rows match the oracle's closed form for every
    tile count (dense table for 201 tiles, shared-memory hash + diagonal for 501 and 1001)."""
    import bench
    F, U, tcs = 3600, 100_000, [200, 500, 1000]
    p = bench.synth_on_device(torch, F, U, 20260000 + 4000, torch.device("cuda"))
    e = engine(vet, tcs, use_w=False)
    a = e.transition(p)
    assert e.poll_flags() == 0
    b = e.transition(p, want_pairs0=False)
    assert torch.equal(a.entropy, b.entropy) and torch.equal(a.per_k, b.per_k) and torch.equal(a.prev_count0, b.prev_count0)
    del b
    assert torch.equal(a.prev_count0.sum(1), torch.full((F - 1,), U, dtype=torch.int64, device="cuda"))
    ent = a.entropy.cpu().numpy()
    assert np.isfinite(ent).all() and (ent >= 0).all()
    np.testing.assert_allclose(ent, a.per_k.cpu().numpy().sum(0) / len(tcs), rtol=1e-15)
    luts = [torch.from_numpy(e.cell_lut(k).astype(np.int64)).cuda().ravel() for k in range(len(tcs))]
    for r in (0, 1799, F - 2):
        cp, cc = _cells_of(p[r]), _cells_of(p[r + 1])
        assert torch.equal(a.pairs0[r, :, 0].long(), luts[0][cp]) and torch.equal(a.pairs0[r, :, 1].long(), luts[0][cc])
        for k, n in enumerate(tcs):
            T = e.num_tiles[k]
            e_ref, m_ref = orc.transition_entropy(luts[k][cp].cpu().numpy(), luts[k][cc].cpu().numpy(), T)
            np.testing.assert_allclose(float(a.per_k[k, r]), e_ref, rtol=RTOL, atol=ATOL)
            if k == 0:
                assert np.array_equal(a.prev_count0[r].cpu().numpy(), m_ref)
    e.close()


def test_full_size_properties_configs4_shard(vet):
    """One rank's frames of BASELINE configs[4] at full WIDTH (1M users per frame, 201 tiles, fov=90, weighted
    spatial + transition entropy in one pass): analyze() equals the separate stages bit for bit, the weighted
    histogram of a whole frame matches the dense per-user weight kernel, transition rows match the oracle."""
    import bench
    F, U = 24, 1_000_000
    p = bench.synth_on_device(torch, F, U, 20260000 + 5000, torch.device("cuda"), chunk=8)
    p[3, ::1000, 1] = float("nan")                       # some users missing in one frame
    e = engine(vet, [200], fov=90.0)
    sp, tr = e.analyze(p)
    assert e.poll_flags() == 0
    sp2 = e.spatial(p)
    tr2 = e.transition(p)
    assert torch.equal(sp.entropy, sp2.entropy) and torch.equal(sp.hist0, sp2.hist0) and torch.equal(sp.assign0, sp2.assign0)
    assert torch.equal(tr.entropy, tr2.entropy) and torch.equal(tr.prev_count0, tr2.prev_count0) and torch.equal(tr.pairs0, tr2.pairs0)
    lut = torch.from_numpy(e.cell_lut(0).astype(np.int64)).cuda().ravel()
    vec, _ = e.decode(p[:1])
    dense = torch.zeros(201, dtype=torch.float64, device="cuda")
    for u0 in range(0, U, 100_000):
        dense += e.tile_weights(vec[0, u0:u0 + 100_000], 0).sum(0)
    np.testing.assert_allclose(sp.hist0[0].cpu().numpy(), dense.cpu().numpy(), rtol=RTOL, atol=ATOL)
    for r in (0, 3, F - 2):                               # row 3: current frame has missing users
        okp = ~(torch.isnan(p[r, :, 1]) | torch.isnan(p[r, :, 2]))
        okc = ~(torch.isnan(p[r + 1, :, 1]) | torch.isnan(p[r + 1, :, 2]))
        both = okp & okc
        cp, cc = _cells_of(torch.nan_to_num(p[r])), _cells_of(torch.nan_to_num(p[r + 1]))
        tp, tc = lut[cp][both].cpu().numpy(), lut[cc][both].cpu().numpy()
        e_ref, m_ref = orc.transition_entropy(tp, tc, 201)
        np.testing.assert_allclose(float(tr.entropy[r]), e_ref, rtol=RTOL, atol=ATOL)
        assert np.array_equal(tr.prev_count0[r].cpu().numpy(), m_ref)
    e.close()


def test_global_table_regime_at_scale(vet):
    """200x400 video (80,601 cells: global-table regime) with enough frames for the tensor-core weighted
    histogram (K = 80,640 cells) and the FP64 one: against the oracle, against each other, and the float32 /
    several-tile-count / analyze() variants against the per-sample direct regime."""
    W, H = 200, 400
    p = synth(520, 700, 5151, iid=False, missing=0.05)
    e = engine(vet, [200], fov=90.0, use_w=True, W=W, H=H)
    a = e.spatial(dev(p))                                   # 520 frames: k_cnt_planes + k_whist_i8
    assert e.poll_flags() == 0
    sel = np.r_[0:3, 255:258, 517:520]
    ref = orc.spatial_analyzer(p[sel], W, H, [200], 90.0, True, 2.0)
    assert np.array_equal(a.assign0.cpu().numpy()[sel], ref["assign0"])
    np.testing.assert_allclose(a.hist0.cpu().numpy()[sel], ref["hist0"], rtol=RTOL, atol=700 * I8_QUANT)
    np.testing.assert_allclose(a.entropy.cpu().numpy()[sel], ref["entropy"], rtol=RTOL, atol=ATOL)
    e.set_option("weighted_kernel", "fp64")
    b = e.spatial(dev(p))
    np.testing.assert_allclose(a.hist0.cpu().numpy(), b.hist0.cpu().numpy(), rtol=RTOL, atol=700 * I8_QUANT)
    np.testing.assert_allclose(a.entropy.cpu().numpy(), b.entropy.cpu().numpy(), rtol=RTOL, atol=0)
    e.close()
    q = synth(6, 2000, 5152, iid=True, missing=0.1)
    for use_w, tcs in ((False, [50, 100, 200]), (True, [50, 200])):
        g = engine(vet, tcs, fov=120.0, use_w=use_w, W=W, H=H)
        sp, tr = g.analyze(dev(q))
        assert g.poll_flags() == 0
        d = engine(vet, tcs, fov=120.0, use_w=use_w, W=W, H=H, regime="direct")
        sp2, tr2 = d.spatial(dev(q)), d.transition(dev(q))
        assert torch.equal(sp.assign0, sp2.assign0) and torch.equal(tr.pairs0, tr2.pairs0) and torch.equal(tr.prev_count0, tr2.prev_count0)
        np.testing.assert_allclose(sp.per_k.cpu().numpy(), sp2.per_k.cpu().numpy(), rtol=RTOL, atol=ATOL)
        np.testing.assert_allclose(sp.hist0.cpu().numpy(), sp2.hist0.cpu().numpy(), rtol=RTOL, atol=ATOL)
        np.testing.assert_allclose(tr.entropy.cpu().numpy(), tr2.entropy.cpu().numpy(), rtol=RTOL, atol=ATOL, equal_nan=True)
        g.close()
        d.close()


@pytest.mark.parametrize("dtype,use_w,tcs,batch", [(np.float32, True, [200], 7), (np.float64, False, [20, 50], 3), (np.float32, True, [200, 500], 0)])
def test_two_column_host_layout_equals_packed_records(vet, dtype, use_w, tcs, batch):
    """The host entry points on [F,U,2] = (2dmu, 2dmv) arrays (VET_OPT_HOST_LAYOUT: a third less to upload, records
    widened on the device) return, bit for bit, what they return for the [F,U,3] records with the time column."""
    p = synth(29, 3001, 1234, missing=0.05, dtype=dtype)
    uv = np.ascontiguousarray(p[..., 1:])
    e = engine(vet, tcs, 90.0, use_w)
    e.set_option("weighted_kernel", "fp64")
    e.set_option("host_batch_frames", batch)
    a_s, a_t = e.analyze_host(p)
    b_s, b_t = e.analyze_host(uv)
    c_s = e.spatial_host(uv)
    c_t = e.transition_host(uv)
    d_s = e.spatial_host(p)          # and back to the three-column layout on the same handle
    assert e.poll_flags() == 0
    for got in (b_s, c_s, d_s):
        for k in ("entropy", "per_k", "hist0", "assign0"):
            assert np.array_equal(got[k], a_s[k], equal_nan=True), k
    for got in (b_t, c_t):
        for k in ("entropy", "per_k", "prev_count0", "pairs0"):
            assert np.array_equal(got[k], a_t[k], equal_nan=True), k
    e.close()


def test_host_path_equals_device_path_at_scale(vet):
    """More frames than one host batch (512 for weighted handles) with a short last batch: the host-buffer path
    and the device path take the same weighted kernel for every batch of a call and return the same bits."""
    p = synth(1100, 1500, 6161, iid=False, missing=0.02)
    e = engine(vet, [200, 50], fov=90.0)
    d = e.spatial(dev(p))
    h = e.spatial_host(p)
    assert e.poll_flags() == 0
    assert np.array_equal(h["entropy"], d.entropy.cpu().numpy())
    assert np.array_equal(h["hist0"], d.hist0.cpu().numpy())
    assert np.array_equal(h["assign0"], d.assign0.cpu().numpy())
    ref = orc.spatial_analyzer(p[1090:], W0, H0, [200, 50], 90.0, True, 2.0)   # frames of the short last host batch
    np.testing.assert_allclose(h["entropy"][1090:], ref["entropy"], rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(h["hist0"][1090:], ref["hist0"], rtol=RTOL, atol=1500 * I8_QUANT)
    e.close()


# ---------------------------------------------------------------------------------
# host-buffer pipelines (vet_spatial_host / vet_transition_host / vet_analyze_host): frame batches on three streams,
# the last frame of a batch carried over on the device as the halo of the next
# ---------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg", [
    dict(F=23, U=4096, tcs=[200], use_w=True, batch=5, dtype=np.float32),          # 5 batches, the last one short (3 frames)
    dict(F=11, U=3001, tcs=[20, 50], use_w=False, batch=2, dtype=np.float64, missing=0.1),   # batches of 2 frames, odd U, f64, missing users
    dict(F=9, U=2000, tcs=[200, 500], use_w=True, batch=8, dtype=np.float32),      # last batch = 1 new frame + halo
    dict(F=6, U=1500, tcs=[100], use_w=True, batch=0, dtype=np.float32),           # auto batch size: one batch
    dict(F=1, U=700, tcs=[50], use_w=True, batch=4, dtype=np.float32),             # a single frame: no transition row
])
def test_host_pipelines_equal_device_calls(vet, cfg):
    """analyze_host / transition_host / spatial_host return, bit for bit, what the device entry points return
    for the same tensor, whatever the batching (weighted kernel pinned: its choice depends on the frames per call)."""
    p = synth(cfg["F"], cfg["U"], 7100 + cfg["U"], iid=False, missing=cfg.get("missing", 0.0), dtype=cfg["dtype"])
    e = engine(vet, cfg["tcs"], 90.0, cfg["use_w"])
    e.set_option("weighted_kernel", "fp64")
    e.set_option("host_batch_frames", cfg["batch"])
    sp, tr = e.analyze(dev(p))
    assert e.poll_flags() == 0
    hs, ht = e.analyze_host(p)
    ht2 = e.transition_host(p)
    hs2 = e.spatial_host(p)
    assert e.poll_flags() == 0
    for got in (hs, hs2):
        assert np.array_equal(got["entropy"], sp.entropy.cpu().numpy(), equal_nan=True)
        assert np.array_equal(got["per_k"], sp.per_k.cpu().numpy(), equal_nan=True)
        assert np.array_equal(got["hist0"], sp.hist0.cpu().numpy()) and np.array_equal(got["assign0"], sp.assign0.cpu().numpy())
    for got in (ht, ht2):
        assert np.array_equal(got["entropy"], tr.entropy.cpu().numpy(), equal_nan=True)
        assert np.array_equal(got["per_k"], tr.per_k.cpu().numpy(), equal_nan=True)
        assert np.array_equal(got["prev_count0"], tr.prev_count0.cpu().numpy())
        assert np.array_equal(got["pairs0"], tr.pairs0.cpu().numpy())
    if cfg["F"] <= 11 and cfg["F"] > 1:   # and the oracle itself
        ref = orc.transition_analyzer(p, W0, H0, cfg["tcs"], mode="literal")
        assert np.array_equal(ht["prev_count0"], ref["prev_count0"]) and np.array_equal(ht["pairs0"], ref["pairs0"])
        np.testing.assert_allclose(ht["entropy"], ref["entropy"], rtol=RTOL, atol=ATOL, equal_nan=True)
    # optional outputs left out
    hs3, ht3 = e.analyze_host(p, want_per_k=False, want_hist0=False, want_assign0=False, want_prev_count0=False, want_pairs0=False)
    assert np.array_equal(hs3["entropy"], hs["entropy"], equal_nan=True) and np.array_equal(ht3["entropy"], ht["entropy"], equal_nan=True)
    e.close()
