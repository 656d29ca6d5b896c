"""Every entry point at the tile-set sizes where its kernels switch code paths, on both sides of each switch.

The launchers choose kernels, LUT widths, table layouts and launch groups by the tile count T, its parity and the
number of tile counts K.  Each case below names the switch, the side it sits on and how the boundary was computed;
the constants it rests on are pinned to the sources by tests/test_thresholds_host.py, so a moved constant fails on a
machine without a GPU instead of leaving these cases in the interior.

Results are compared with the oracles (spatial_analyzer / transition_analyzer, user_analyzer, transition_counts,
user_transitions): indices, counts and pairs exact; entropies within 1e-9 relative (absolute floor 1e-12); weighted
histograms within 1e-9 relative plus users * 2^-40 after the tensor-core kernel and frames * 2^-b for `users`; kernel
against kernel bit for bit where DESIGN claims the same bits.

Before anything is compared, the cell LUT of every tile set is checked against orc.nearest_tile.  The samples are
then drawn only from cells whose two best normalised dot products differ by more than 1e-13: the cells left out are
rounding-level ties (DESIGN 2), where the first-minimum rule of the reference and of the kernels may pick either
tile, and the LUT check accepts a difference only there.
"""
import numpy as np
import pytest

from oracle import vet_oracle as orc
from oracle.vet_transition_counts_oracle import transition_counts as tc_oracle, transition_pairs
from oracle.vet_user_transitions_oracle import user_transitions as ut_oracle
from oracle.vet_users_oracle import user_analyzer
from thresholds_plan import (MAX_T, LUT8_MAX_T, T4_RANK_MAX_T, RELABEL_GROUP, TC_GROUP, MAX_TILE_COUNTS,
                             PACKED_LUT_MAX_K, ENTROPY_FRAMES_BYTES, T3_SLOTS, TC_THREADS, UT_ROWS_USERS,
                             I8_MIN_FRAMES, transition_max_t, t3_mode, t3_boundaries, pair_table_in_smem,
                             user_hist_ub, entropy_frames_bytes, t4_runs, t4_plan_smem, unit_staged_max_t)

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-9, 1e-12
TIE_GAP = 1e-13         # cells whose two best dots are closer than this are never sampled (rounding-level ties)
FOV = 90.0


@pytest.fixture(scope="module")
def vet():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import __graft_entry__ as ge
    ge.build()
    import viewport_entropy_toolkit_b200 as pkg
    return pkg


@pytest.fixture(scope="module")
def optin():
    return int(torch.cuda.get_device_properties(0).shared_memory_per_block_optin)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _bits(t):
    t = t.contiguous().cpu().numpy()
    return t.view(np.int64) if t.dtype == np.float64 else t


def sphere(T, seed):
    """T arbitrary tile centres (unit vectors, not a lattice)."""
    v = np.random.default_rng(seed).normal(size=(T, 3))
    return v / np.linalg.norm(v, axis=1, keepdims=True)


class Tiles:
    """One handle and its tile sets: `sets` lists ("lattice", n), ("centres", T, seed) (sphere) or ("array", centres)."""

    def __init__(self, vet, sets, use_w, W=100, H=200, fov=FOV):
        self.W, self.H, self.use_w, self.fov = W, H, use_w, fov
        self.centres = [orc.lattice(s[1]) if s[0] == "lattice" else sphere(s[1], s[2]) if s[0] == "centres" else s[1]
                        for s in sets]
        self.tcs = [s[1] if s[0] != "array" else len(s[1]) for s in sets]
        self.arbitrary = any(s[0] != "lattice" for s in sets)
        self.ref_centres = self.centres if self.arbitrary else None
        self.Ts = [len(c) for c in self.centres]
        self.eng = vet.Engine(W, H, self.tcs, vet.EntropyConfig(fov_angle=fov, use_weight_distribution=use_w,
                                                                power_factor=2.0),
                              torch.device("cuda", 0), centres=self.ref_centres)
        assert self.eng.num_tiles == self.Ts
        self.cells = self._check_luts()

    def _check_luts(self):
        """Handle LUTs against orc.nearest_tile; returns the cells that are not rounding-level ties in any tile set."""
        cv = orc.cell_vectors(self.W, self.H).reshape(-1, 3)
        safe = np.ones(len(cv), dtype=bool)
        for k, c in enumerate(self.centres):
            ref = orc.nearest_tile(cv, c, chunk=256)
            got = self.eng.cell_lut(k).ravel().astype(np.int32)
            gap = np.empty(len(cv))
            for s in range(0, len(cv), 256):
                d = np.sort(orc.dots(cv[s:s + 256], c), axis=1)
                gap[s:s + 256] = d[:, -1] - d[:, -2] if c.shape[0] > 1 else np.inf
            bad = got != ref
            assert (gap[bad] <= TIE_GAP).all(), (k, np.nonzero(bad & (gap > TIE_GAP))[0][:10])
            safe &= gap > TIE_GAP
        assert safe.sum() > 0
        return np.nonzero(safe)[0]

    def video(self, F, U, seed, stay=0.0, missing=0.0, dtype=np.float32, cells=None):
        """Samples at the centres of safe cells; every user keeps its cell with probability `stay`.  User 0 is
        present in every frame (no frame without a user)."""
        rng = np.random.default_rng(seed)
        pool = self.cells if cells is None else cells
        idx = pool[rng.integers(0, len(pool), (F, U))]
        if stay:
            keep = rng.uniform(size=(F, U)) < stay
            for f in range(1, F):
                idx[f] = np.where(keep[f], idx[f - 1], idx[f])
        px, py = idx % (self.W + 1), idx // (self.W + 1)
        mu = np.where(px < self.W, (px + 0.5) / self.W, 1.0)
        mv = np.where(py < self.H, (py + 0.5) / self.H, 1.0)
        p = np.stack([np.broadcast_to(np.arange(F)[:, None] * 0.1, (F, U)), mu, mv], -1).astype(dtype)
        if missing:
            m = rng.uniform(size=(F, U)) < missing
            m[:, 0] = False
            p[m, 1] = np.nan
        return p

    # -- checks against the oracles --------------------------------------------------------------------------
    def spatial(self, p, entry="spatial"):
        F, U = p.shape[:2]
        ref = orc.spatial_analyzer(p, self.W, self.H, self.tcs, self.fov, self.use_w, 2.0, centres=self.ref_centres)
        sp = self.eng.spatial(dev(p)) if entry == "spatial" else self.eng.analyze(dev(p))[0]
        assert self.eng.poll_flags() == 0
        assert np.array_equal(sp.assign0.cpu().numpy(), ref["assign0"])
        if self.use_w:
            tc = U * 2.0 ** -40 if F >= I8_MIN_FRAMES else 0.0
            np.testing.assert_allclose(sp.hist0.cpu().numpy(), ref["hist0"], rtol=RTOL, atol=ATOL + tc)
        else:
            assert np.array_equal(sp.hist0.cpu().numpy(), ref["hist0"])
        np.testing.assert_allclose(sp.per_k.cpu().numpy(), ref["per_k"], rtol=RTOL, atol=ATOL, equal_nan=True)
        np.testing.assert_allclose(sp.entropy.cpu().numpy(), ref["entropy"], rtol=RTOL, atol=ATOL, equal_nan=True)
        return sp

    def transition(self, p, mode="literal", entry="transition"):
        ref = orc.transition_analyzer(p, self.W, self.H, self.tcs, mode, centres=self.ref_centres)
        tr = self.eng.transition(dev(p), mode) if entry == "transition" else self.eng.analyze(dev(p), mode)[1]
        assert self.eng.poll_flags() == 0
        assert np.array_equal(tr.pairs0.cpu().numpy(), ref["pairs0"])
        assert np.array_equal(tr.prev_count0.cpu().numpy(), ref["prev_count0"])
        np.testing.assert_allclose(tr.per_k.cpu().numpy(), ref["per_k"], rtol=RTOL, atol=ATOL, equal_nan=True)
        np.testing.assert_allclose(tr.entropy.cpu().numpy(), ref["entropy"], rtol=RTOL, atol=ATOL, equal_nan=True)
        return tr

    def users(self, p):
        F = p.shape[0]
        ref = user_analyzer(p, self.W, self.H, self.tcs, self.fov, self.use_w, 2.0, centres=self.ref_centres)
        res = self.eng.users(dev(p))
        assert self.eng.poll_flags() == 0
        frames = res.frames.cpu().numpy()
        assert np.array_equal(frames, ref["frames"])
        np.testing.assert_allclose(res.entropy.cpu().numpy(), ref["entropy"], rtol=RTOL, atol=ATOL, equal_nan=True)
        np.testing.assert_allclose(res.per_k.cpu().numpy(), ref["per_k"], rtol=RTOL, atol=ATOL, equal_nan=True)
        h, rh = res.hist0.cpu().numpy(), ref["hist0"]
        q = 2.0 ** -(62 - int(np.ceil(np.log2(F))) if F > 1 else 62) if self.use_w else 0.0
        assert np.all(np.abs(h - rh) <= frames[:, None] * q + 1e-12 * np.abs(rh)), np.abs(h - rh).max()
        assert np.array_equal(h > 0, rh > 0)
        return res

    def transition_counts(self, p):
        res = self.eng.transition_counts(dev(p))
        assert self.eng.poll_flags() == 0
        if sum(T * T for T in self.Ts) <= 1 << 22:
            ref = tc_oracle(p, self.W, self.H, self.tcs, centres=self.ref_centres)
            for c, rc in zip(res.counts, ref["counts"]):
                assert c.dtype == torch.int64 and tuple(c.shape) == rc.shape
                assert np.array_equal(c.cpu().numpy(), rc)
        else:
            # up to 2^28 entries: the non-zero counts only (the dense oracle matrix would take 2 GB of host memory)
            ref = dict(per_k=[], entropy=0.0)
            for c, (pp, cc), T in zip(res.counts, transition_pairs(p, self.W, self.H, self.tcs, self.ref_centres), self.Ts):
                assert c.dtype == torch.int64 and tuple(c.shape) == (T, T)
                keys, cnt = np.unique(pp * T + cc, return_counts=True)
                flat = c.reshape(-1)
                nz = flat.nonzero().reshape(-1)
                assert np.array_equal(nz.cpu().numpy(), keys) and np.array_equal(flat[nz].cpu().numpy(), cnt)
                ref["pairs"] = len(pp)
                ref["per_k"].append(orc.transition_entropy_textbook(pp, cc, T) if len(pp) else np.nan)
            for e in ref["per_k"]:
                ref["entropy"] = ref["entropy"] + e
            ref["entropy"] /= len(self.Ts)
        assert res.pairs == ref["pairs"]
        np.testing.assert_allclose(res.per_k.cpu().numpy(), ref["per_k"], rtol=RTOL, atol=ATOL, equal_nan=True)
        np.testing.assert_allclose(float(res.entropy), ref["entropy"], rtol=RTOL, atol=ATOL, equal_nan=True)
        return res

    def user_transitions(self, p):
        ref = ut_oracle(p, self.W, self.H, self.tcs, centres=self.ref_centres)
        res = self.eng.user_transitions(dev(p))
        assert self.eng.poll_flags() == 0
        assert np.array_equal(res.pairs.cpu().numpy(), ref["pairs"])
        np.testing.assert_allclose(res.per_k.cpu().numpy(), ref["per_k"], rtol=RTOL, atol=ATOL, equal_nan=True)
        np.testing.assert_allclose(res.entropy.cpu().numpy(), ref["entropy"], rtol=RTOL, atol=ATOL, equal_nan=True)
        return res

    def all(self, p, per_user=400):
        """Every entry point; the per-user entry points on the first `per_user` users (their oracles loop per user)."""
        self.spatial(p)
        self.transition(p, "literal")
        self.transition(p, "textbook")
        self.spatial(p, entry="analyze")
        self.transition(p, "literal", entry="analyze")
        q = np.ascontiguousarray(p[:, :per_user])
        self.users(q)
        self.transition_counts(p)
        self.user_transitions(q)


# ---------------------------------------------------------------------------------------------------------------
# u8 <-> u16 LUT: T <= 255 keeps a u8 LUT (d_lut8 and the packed 4 x u8 LUT of k_stream_tiles), T = 256 is the first
# u16 LUT.  Lattices only reach odd T: n = 254 gives T = 255 (u8 side), n = 256 gives T = 257 (u16 side); T = 256
# exactly needs arbitrary centres.  U = 4500 > 4096 users: the literal pair table no longer fits shared memory
# (pair_table_in_smem), so the transition runs k_transition4 / k_transition3 rather than k_transition<true>.
LUT_SETS = {
    "centres_T255_u8": ("centres", 255, 1),
    "centres_T256_u16": ("centres", 256, 2),
    "lattice_n254_T255_u8": ("lattice", 254),
    "lattice_n256_T257_u16": ("lattice", 256),
}


@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("use_w", [False, True], ids=["unweighted", "weighted"])
@pytest.mark.parametrize("name", list(LUT_SETS))
def test_lut_width_boundary(vet, optin, name, use_w, dtype):
    s = LUT_SETS[name]
    t = Tiles(vet, [s], use_w)
    T = t.Ts[0]
    assert (T <= LUT8_MAX_T) == name.endswith("u8")
    assert not pair_table_in_smem(4500, T, optin)
    t.all(t.video(4, 4500, 10 + T, stay=0.6, missing=0.05, dtype=dtype))
    # the same tile set next to a small one: several tile counts (relabelled rows, k_entropy_frames)
    t2 = Tiles(vet, [s, ("lattice", 20)], use_w)
    t2.all(t2.video(3, 4500, 20 + T, stay=0.6, missing=0.05, dtype=dtype))


# ---------------------------------------------------------------------------------------------------------------
# Even T and tiny T.  k_transition3's dense table has a row pitch of T + (T & 1): even T (2, 4, 234, 256) is the
# other pitch than every lattice.  234 is the last dense T at 227 KB (t3_boundaries), 256 the first u16 LUT.  T = 1
# (lattice n = 1) beside larger tile counts: log2 T = 0 is the normaliser, so the spatial and textbook entropies of that
# tile count are 0 / 0 = NaN, while the literal mode's stale transition weight (EU:312-315) makes its numerator
# positive: -inf (x / -0.0) wherever two or more users share the frame pair.  One common user in a frame pair gives
# NaN in every tile count (total == 1).
def test_even_and_tiny_tile_counts(vet, optin):
    last_dense, _ = t3_boundaries(optin)
    assert last_dense % 2 == 0 and t3_mode(last_dense, optin) == "dense"
    # all T <= 255 and K = 4: the packed u8 LUT
    t = Tiles(vet, [("centres", 2, 3), ("centres", 4, 4), ("centres", last_dense, 5), ("lattice", 1)], False)
    p = t.video(5, 4500, 30, stay=0.5, missing=0.05)
    p[2, 1:, 1] = np.nan                               # frame 2: user 0 alone -> pairs (1, 2) and (2, 3) of one user
    t.all(p)
    sp = t.eng.spatial(dev(p))
    assert torch.isnan(sp.per_k[3]).all() and torch.isnan(sp.entropy).all()
    tr = t.eng.transition(dev(p))
    assert torch.isnan(tr.per_k[:, 1]).all() and torch.isnan(tr.per_k[:, 2]).all()
    assert torch.isneginf(tr.per_k[3, [0, 3]]).all()
    assert torch.isnan(t.eng.transition(dev(p), "textbook").per_k[3]).all()
    # T = 256 (u16) with T = 2 and the weighted tables
    t = Tiles(vet, [("centres", 256, 6), ("centres", 2, 7), ("lattice", 1)], True)
    t.all(t.video(4, 4500, 31, stay=0.5, missing=0.05))


# ---------------------------------------------------------------------------------------------------------------
# k_transition3's dense table -> hash table -> k_transition2, computed from plan_transition's formula and the device's
# opt-in shared memory (t3_boundaries; 234 | 235 and 2388 | 2389 at 227 KB).  Unweighted handles with one tile count
# of arbitrary centres; auto, v3 and v2 must give the same bits and match the literal oracle.  The iid frames of
# 20000 users hold ~16k distinct pairs on 235 tiles, more than the 12288 the hash table takes: those pairs overflow and
# k_transition2 redoes them; the sticky frames stay inside the table.
def _route_cases():
    return [("last_dense", 0, 0), ("first_hash", 0, 1), ("last_hash", 1, 0), ("first_v2", 1, 1)]


@pytest.mark.parametrize("case", _route_cases(), ids=[c[0] for c in _route_cases()])
def test_transition_table_routes(vet, optin, case):
    name, which, step = case
    T = t3_boundaries(optin)[which] + step
    want = {"last_dense": "dense", "first_hash": "hash", "last_hash": "hash", "first_v2": "v2"}[name]
    assert t3_mode(T, optin) == want
    U = 20000
    assert not pair_table_in_smem(U, T, optin)
    t = Tiles(vet, [("centres", T, 40 + T)], False)
    iid = t.video(3, U, 41)
    sticky = t.video(3, U, 42, stay=0.9, missing=0.05)
    if name == "first_hash":
        # the iid pairs do overflow the hash table (more distinct pairs than kT3Slots * 3/4)
        luts = t.eng.cell_lut(0).ravel()
        px = (iid[..., 1] * t.W).astype(np.int64)
        py = (iid[..., 2] * t.H).astype(np.int64)
        tiles = luts[py * (t.W + 1) + px]
        assert len(np.unique(tiles[0].astype(np.int64) * T + tiles[1])) > T3_SLOTS * 3 // 4
    for p in (iid, sticky):
        runs = {}
        for kern in ("auto", "v3", "v2"):
            t.eng.set_option("transition_kernel", kern)
            runs[kern] = t.transition(p) if kern == "auto" else t.eng.transition(dev(p))
        t.eng.set_option("transition_kernel", "auto")
        for kern in ("v3", "v2"):
            assert np.array_equal(_bits(runs[kern].entropy), _bits(runs["auto"].entropy)), kern
            assert np.array_equal(_bits(runs[kern].per_k), _bits(runs["auto"].per_k)), kern
            assert torch.equal(runs[kern].prev_count0, runs["auto"].prev_count0), kern
            assert torch.equal(runs[kern].pairs0, runs["auto"].pairs0), kern
    t.all(sticky[:, :6000])


# ---------------------------------------------------------------------------------------------------------------
def _t4_launched(eng, p):
    """Whether k_transition4 ran for a one-tile-count handle: with it, k_transition3 is recorded as the tail kernel."""
    eng.profile(True)
    eng.transition(dev(p))
    n = eng.profile_read()["transition_tail"][1]
    eng.profile(False)
    return n > 0


def _auto_equals_v3(t, p):
    auto = t.transition(p)
    t.eng.set_option("transition_kernel", "v3")
    v3 = t.eng.transition(dev(p))
    t.eng.set_option("transition_kernel", "auto")
    assert np.array_equal(_bits(auto.per_k), _bits(v3.per_k)) and np.array_equal(_bits(auto.entropy), _bits(v3.entropy))
    assert torch.equal(auto.prev_count0, v3.prev_count0) and torch.equal(auto.pairs0, v3.pairs0)


# k_transition4's plan limit: plan_transition4 needs three [16][T] tables, a 1024-entry list, T terms and the band
# tables of build_delta_ranks (at most 32 bands of 2^s tiles, +-160 deltas) within the opt-in shared memory
# (t4_plan_smem).  The band count drops from 32 to 17 at T = 1025, so at 227 KB the kernel runs for T <= 1002 and
# again for 1025 <= T <= 1055: three flips, each case on one side of one (computed from optin).  Arbitrary centres,
# one tile count; whether k_transition4 ran is read from the launch record (_t4_launched).  auto must equal v3 (which
# never runs k_transition4) bit for bit and match the literal oracle.
def _t4_flip_cases():
    flips = [T for T in range(3, T4_RANK_MAX_T + 1) if t4_runs(T, 227 * 1024) != t4_runs(T - 1, 227 * 1024)]
    assert flips == [1003, 1025, 1056]
    return [(f"T{T - 1}_{'runs' if t4_runs(T - 1, 227 * 1024) else 'no_t4'}", -1, i) for i, T in enumerate(flips)] + \
           [(f"T{T}_{'runs' if t4_runs(T, 227 * 1024) else 'no_t4'}", 0, i) for i, T in enumerate(flips)]


@pytest.mark.parametrize("case", _t4_flip_cases(), ids=[c[0] for c in _t4_flip_cases()])
def test_transition4_plan_limit(vet, optin, case):
    _, d, i = case
    flips = [T for T in range(3, T4_RANK_MAX_T + 1) if t4_runs(T, optin) != t4_runs(T - 1, optin)]
    T = flips[i] + d
    t = Tiles(vet, [("centres", T, 200 + T)], False)
    U = 6000
    assert not pair_table_in_smem(U, T, optin)
    p = t.video(4, U, 210 + T, stay=0.7, missing=0.05)
    assert _t4_launched(t.eng, p) == t4_runs(T, optin)
    _auto_equals_v3(t, p)
    t.all(p)


# The delta ranking: build_delta_ranks ranks deltas only while 15 * T * 4 < 0xFFFF, i.e. T <= 1092.  Lattice n = 1090
# (T 1091) and centres T = 1092 are ranked, lattice n = 1092 (T 1093) is not.  k_transition4 runs on none of them (its
# plan limit above lies lower), so the ranking decides k_tc_count's path: the ranked shared-memory counter table or
# the global counters.  transition_counts ranked and unranked, alone and in one handle, match the oracle's counts
# exactly; the transition kernels (auto = v3 here) match the literal oracle.
T4_SETS = {"lattice_n1090_T1091_ranked": ("lattice", 1090), "centres_T1092_ranked": ("centres", 1092, 8),
           "lattice_n1092_T1093_unranked": ("lattice", 1092)}


@pytest.mark.parametrize("name", list(T4_SETS))
def test_transition4_ranking_limit(vet, optin, name):
    s = T4_SETS[name]
    t = Tiles(vet, [s], False)
    both = Tiles(vet, [s, ("lattice", 1092)], False)
    T = t.Ts[0]
    assert (15 * T * 4 < 0xFFFF) == name.endswith("_ranked")
    U = 6000
    assert not pair_table_in_smem(U, T, optin)
    p = t.video(4, U, 50 + T, stay=0.7, missing=0.05, cells=np.intersect1d(t.cells, both.cells))
    assert not t4_runs(T, optin) and not _t4_launched(t.eng, p)
    _auto_equals_v3(t, p)
    t.all(p)
    # ranked and unranked tables of the same video in one handle: each tile count's counts equal the oracle's
    both.transition_counts(p)
    both.transition(p)


# ---------------------------------------------------------------------------------------------------------------
# Largest T.  kMaxT = 16384 tiles: the largest lattice is n = 16383 (T 16383; n = 16384 gives T = 16385, rejected);
# arbitrary centres reach T = 16384, whose last tile id 16383 equals k_transition3's 14-bit kNoTile (0x3FFF) -- the plan
# sends that T to k_transition2 (t3_mode), and samples are placed in tile 16383 to pin it.  A 40 x 20 video (861 cells)
# keeps the tables and the oracle small.  transition_counts at [16384] holds sum T^2 = 2^28 entries exactly (accepted);
# one more tile count is rejected.  user_transitions sorts keys of ceil(log2 T^2) = 28 bits: 7 radix passes of 4 bits.
# The literal / textbook transition entry points keep 24 B per tile in shared memory (transition_max_t: 9640 tiles at
# 227 KB): at these T they return VET_ERR_UNSUPPORTED before any launch (they used to fail inside k_transition2's launch).
def _max_t_entry_points(t, p, per_user=300):
    from viewport_entropy_toolkit_b200 import UnsupportedConfigurationError as UnsupportedError
    t.spatial(p)
    for call in (lambda: t.eng.transition(dev(p)), lambda: t.eng.transition(dev(p), "textbook"),
                 lambda: t.eng.analyze(dev(p)), lambda: t.eng.transition_host(p)):
        with pytest.raises(UnsupportedError, match="transition kernels hold at most"):
            call()
    q = np.ascontiguousarray(p[:, :per_user])
    t.users(q)
    res = t.transition_counts(p)
    t.user_transitions(q)
    return res

def _max_t_centres():
    c = sphere(MAX_T, 60)
    cv = orc.cell_vectors(40, 20).reshape(-1, 3)
    c[-1] = cv[700] / np.linalg.norm(cv[700])   # tile 16383 sits on cell 700: that cell's nearest tile
    return c


def test_max_tile_count(vet, optin):
    assert t3_mode(MAX_T, optin) == "v2" and transition_max_t(optin) < MAX_T - 1
    ec = vet.EntropyConfig(fov_angle=FOV, use_weight_distribution=False)
    for n in (MAX_T, MAX_T + 1):                      # lattices of 16385 tiles
        with pytest.raises(vet.UnsupportedConfigurationError):
            vet.Engine(40, 20, [n], ec, torch.device("cuda", 0))
    with pytest.raises(vet.UnsupportedConfigurationError):
        vet.Engine(40, 20, [1], ec, torch.device("cuda", 0), centres=[sphere(MAX_T + 1, 61)])

    c = _max_t_centres()
    for use_w in (False, True):
        t = Tiles(vet, [("array", c)], use_w, W=40, H=20)
        lut = t.eng.cell_lut(0).ravel()
        assert lut[700] == MAX_T - 1 and 700 in t.cells
        # half the samples on cell 700 (tile 16383 = 0x3FFF), F < 384 (weighted: FP64 histogram, no i8 slices)
        p = t.video(6, 300, 62, stay=0.5, missing=0.05)
        hot = np.random.default_rng(63).uniform(size=p.shape[:2]) < 0.5
        p[hot, 1], p[hot, 2] = (700 % 41 + 0.5) / 40, (700 // 41 + 0.5) / 20
        res = _max_t_entry_points(t, p)
        assert int(res.counts[0][MAX_T - 1].sum()) > 0 and int(res.counts[0][:, MAX_T - 1].sum()) > 0
    # transition_counts: sum T^2 = 2^28 accepted (checked above through t.all), 2^28 + 1 rejected
    assert MAX_T * MAX_T == 1 << 28
    big = vet.Engine(40, 20, [MAX_T, 1], ec, torch.device("cuda", 0), centres=[c, c[:1]])
    with pytest.raises(vet.UnsupportedConfigurationError, match="2\\^28"):
        big.transition_counts(dev(p))
    big.close()


def test_max_lattice(vet):
    # lattice n = 16383: T = 16383, the largest lattice; unweighted, every entry point
    t = Tiles(vet, [("lattice", MAX_T - 1)], False, W=40, H=20)
    assert t.Ts == [MAX_T - 1]
    _max_t_entry_points(t, t.video(6, 300, 64, stay=0.5, missing=0.05))


# The transition entry points' own limit (transition_tiles_supported): the largest accepted T is where k_transition2's
# per-tile arrays end exactly at the opt-in budget (9640 at 227 KB: its dynamic shared memory equals the budget), the
# next T is refused before any launch.  Arbitrary centres on a 40 x 20 video; calls without a frame pair stay valid.
@pytest.mark.parametrize("d", [0, 1], ids=["largest_accepted", "first_refused"])
def test_transition_tile_limit(vet, optin, d):
    from viewport_entropy_toolkit_b200 import UnsupportedConfigurationError
    T = transition_max_t(optin) + d
    t = Tiles(vet, [("centres", T, 300 + d)], False, W=40, H=20)
    p = t.video(5, 300, 310 + d, stay=0.5, missing=0.05)
    assert t.eng.transition(dev(p[:1])).entropy.numel() == 0
    if d == 0:
        t.all(p, per_user=300)    # literal: k_transition2; textbook: k_transition<false>, both at the budget exactly
        return
    for call in (lambda: t.eng.transition(dev(p)), lambda: t.eng.analyze(dev(p)), lambda: t.eng.transition_host(p),
                 lambda: t.eng.analyze_host(p)):
        with pytest.raises(UnsupportedConfigurationError, match="transition kernels hold at most"):
            call()
    assert t.eng.poll_flags() == 0
    t.spatial(p)
    t.transition_counts(p)


# k_nearest / k_tile_weights stage the unit centres in shared memory up to unit_staged_max_t (9642 at 227 KB) and read
# them from global memory beyond (unit_smem): the cell LUT, vet_nearest_tile and vet_tile_weights (weighted and
# unweighted) on both sides, against the oracle.
@pytest.mark.parametrize("d", [0, 1], ids=["staged", "global"])
def test_unit_centre_staging(vet, optin, d):
    T = unit_staged_max_t(optin) + d
    c = sphere(T, 320 + d)
    # a seed unlike the centres': a vector ON a centre has dot 1 within an ulp, and arccos there turns one ulp into ~1e-8
    v = np.random.default_rng(9001).normal(size=(500, 3))
    dd = np.sort(orc.dots(v, c), axis=1)
    v = v[dd[:, -1] - dd[:, -2] > TIE_GAP]
    for use_w in (False, True):
        t = Tiles(vet, [("array", c)], use_w, W=40, H=20)      # the LUT check runs k_nearest<uint16_t>
        assert np.array_equal(t.eng.nearest_tile(dev(v)).cpu().numpy(), orc.nearest_tile(v, c, chunk=256))
        w = t.eng.tile_weights(dev(v)).cpu().numpy()
        ref = orc.tile_weights(v, c, FOV, use_w, 2.0)
        if use_w:
            edge = np.abs(ref) < 1e-12            # support may differ only within rounding of d == fov/2
            assert np.array_equal((w > 0) | edge, (ref > 0) | edge)
            np.testing.assert_allclose(w, ref, rtol=RTOL, atol=1e-14)
        else:
            assert np.array_equal(w, ref)


# ---------------------------------------------------------------------------------------------------------------
# Users whose accumulator row exceeds 96 KB: vet_users_accumulate then runs Ub = 1 user per CTA (one warp weighted),
# as long as the row and its staged samples fit the opt-in shared memory; beyond that it returns VET_ERR_UNSUPPORTED.
#   weighted [16383]: row (16383 + 1) x 8 B = 128 KB > 96 KB -> Ub = 1, supported: matches the oracle;
#   unweighted [16383, 9000] (T 16383 + 9001 = 25384 > 24575): row 99 KB -> Ub = 1, supported: matches the oracle;
#   weighted [16383, 16383]: row 256 KB > the opt-in limit -> UnsupportedConfigurationError.
def test_users_rows_above_96k(vet, optin):
    t = Tiles(vet, [("lattice", MAX_T - 1)], True, W=40, H=20)
    assert user_hist_ub(sum(t.Ts), True) == 1
    p = t.video(20, 70, 70, stay=0.3, missing=0.1)
    t.users(p)
    t = Tiles(vet, [("lattice", MAX_T - 1), ("lattice", 9000)], False, W=40, H=20)
    assert sum(t.Ts) > 24575 and user_hist_ub(sum(t.Ts), False) == 1
    t.users(t.video(20, 70, 71, stay=0.3, missing=0.1))
    eng = vet.Engine(40, 20, [MAX_T - 1, MAX_T - 1], vet.EntropyConfig(fov_angle=FOV, use_weight_distribution=True),
                     torch.device("cuda", 0))
    assert (2 * (MAX_T - 1) + 1) * 8 > optin
    with pytest.raises(vet.UnsupportedConfigurationError, match="shared memory"):
        eng.users(dev(p))
    eng.close()


# ---------------------------------------------------------------------------------------------------------------
# Number of tile counts K.
#   K = 4 with every T <= 255: the packed 4 x u8 LUT of k_stream_tiles and one relabel pass (kRelabelGroup = 4);
#   K = 5, all T <= 255: no packed LUT, a second relabel pass for the fifth tile count;
#   K = 4 with one T = 257: no packed LUT (u16 LUT in the set).
K_SETS = {
    "K4_u8_packed": [20, 50, 100, 254],
    "K5_u8_two_relabel_passes": [20, 50, 100, 200, 254],
    "K4_with_T257": [20, 50, 100, 256],
}


@pytest.mark.parametrize("use_w", [False, True], ids=["unweighted", "weighted"])
@pytest.mark.parametrize("name", list(K_SETS))
def test_tile_count_groups(vet, optin, name, use_w):
    tcs = K_SETS[name]
    t = Tiles(vet, [("lattice", n) for n in tcs], use_w)
    packed = len(tcs) <= PACKED_LUT_MAX_K and max(t.Ts) <= LUT8_MAX_T
    assert packed == (name == "K4_u8_packed")
    assert (len(tcs) > RELABEL_GROUP) == name.startswith("K5")
    assert not pair_table_in_smem(4500, max(t.Ts), optin)
    t.all(t.video(4, 4500, 80 + len(tcs), stay=0.6, missing=0.05))


# kTcGroup = 6 tile counts per k_tc_count launch: K = 6 is one launch, K = 7 two.  Small tile sets keep each group
# within the L1 budget of the launcher (2 x 16 T x 4 B + C B per tile count), so the group size is the only split.
@pytest.mark.parametrize("K", [TC_GROUP, TC_GROUP + 1])
def test_transition_counts_group(vet, K):
    tcs = [20 + 2 * i for i in range(K)]
    C = 101 * 201
    assert TC_GROUP * (2 * 16 * max(orc.lattice_size(n) for n in tcs) * 4 + C) <= 160 * 1024
    t = Tiles(vet, [("lattice", n) for n in tcs], False)
    p = t.video(30, 700, 90 + K, stay=0.6, missing=0.1)
    t.transition_counts(p)
    t.user_transitions(p)
    t.users(p)


# K = 16 (kMaxTileCounts) mixed sizes: T = 1 and 3, u8 and u16 LUTs, ranked and unranked tile sets, dense and hash
# tables, several relabel passes and k_tc_count groups; K = 17 is rejected at handle creation.
def test_sixteen_tile_counts(vet, optin):
    tcs = [1, 2, 3, 7, 20, 21, 50, 100, 200, 254, 256, 500, 1000, 1090, 1092, 2000]
    assert len(tcs) == MAX_TILE_COUNTS
    t = Tiles(vet, [("lattice", n) for n in tcs], False)
    assert not pair_table_in_smem(4500, max(t.Ts), optin)
    t.all(t.video(3, 4500, 100, stay=0.6, missing=0.05), per_user=150)
    with pytest.raises(vet.UnsupportedConfigurationError, match="tile counts"):
        vet.Engine(100, 200, tcs + [20], vet.EntropyConfig(), torch.device("cuda", 0))


# k_entropy_frames takes several tile counts while their rows fit 40 KB (sum ceil(T/32) * 32 * 16 B):
# [200, 2000] (T 201 + 2001: 35 KB) runs k_entropy_frames, [200, 2500] (T 201 + 2501: 43 KB) k_entropy_rows.  The
# rows of the shared tile count 200 must be bit-identical whichever kernel ran (DESIGN 4.2), and hist0 too.
@pytest.mark.parametrize("use_w", [False, True], ids=["unweighted", "weighted"])
def test_entropy_kernel_switch(vet, use_w):
    a = Tiles(vet, [("lattice", 200), ("lattice", 2000)], use_w)
    b = Tiles(vet, [("lattice", 200), ("lattice", 2500)], use_w)
    assert entropy_frames_bytes(a.Ts) <= ENTROPY_FRAMES_BYTES < entropy_frames_bytes(b.Ts)
    cells = np.intersect1d(a.cells, b.cells)
    p = a.video(12, 2000, 110, stay=0.5, missing=0.05, cells=cells)
    sa, sb = a.spatial(p), b.spatial(p)
    assert np.array_equal(_bits(sa.per_k[0]), _bits(sb.per_k[0]))
    assert np.array_equal(_bits(sa.hist0), _bits(sb.hist0)) and torch.equal(sa.assign0, sb.assign0)
    a.all(p, per_user=200)
    b.all(p, per_user=200)


# ---------------------------------------------------------------------------------------------------------------
# Users per CTA, small F with missing samples:
#   U = 511 / 512 / 513 around kTcThreads = 512 (k_tc_count: one user per thread);
#   U = 31 / 32 / 33 around kUtRowsUsers = 32 (k_ut_rows);
#   U = Ub - 1 / Ub / Ub + 1 around k_user_hist's users per CTA (user_hist_ub; weighted and unweighted).
def _ub(use_w):
    return user_hist_ub(orc.lattice_size(20) + orc.lattice_size(200), use_w)


@pytest.mark.parametrize("d", [-1, 0, 1], ids=["below", "at", "above"])
def test_users_per_cta(vet, d):
    t = Tiles(vet, [("lattice", 20), ("lattice", 200)], False)
    for U in (TC_THREADS + d, UT_ROWS_USERS + d):
        p = t.video(7, U, 120 + U, stay=0.5, missing=0.2)
        t.transition_counts(p)
        t.user_transitions(p)
    for use_w in (False, True):
        tw = Tiles(vet, [("lattice", 20), ("lattice", 200)], use_w)
        U = _ub(use_w) + d
        tw.users(tw.video(7, U, 130 + U, stay=0.5, missing=0.2))
