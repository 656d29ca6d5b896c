"""CPU-only tests: the C-ABI library loads and exports every declared symbol, the
host-side mirror of the reference API (configs, data types, ingest, tables) behaves
like the reference.  No compute call is made (no GPU here)."""
import ctypes
import re
from pathlib import Path

import numpy as np
import pandas as pd
import pytest

from conftest import ROOT, group_keys, load_golden
from oracle import vet_oracle as orc


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as ge
    ge.build()
    import viewport_entropy_toolkit_b200 as p
    return p


def test_library_exports_every_declared_symbol(pkg):
    from viewport_entropy_toolkit_b200 import _native
    header = (ROOT / "include" / "vet_b200.h").read_text()
    declared = set(re.findall(r"\b(vet_[a-z0-9_]+)\s*\(", header))
    declared -= {"vet_handle", "vet_config", "vet_status"}
    assert declared == set(_native.SYMBOLS), declared ^ set(_native.SYMBOLS)
    lib = _native.load_library()
    for name in declared:
        assert getattr(lib, name) is not None
    assert b"sm_100a" in lib.vet_version()
    # the profile slots of vet_profile_read: same order and count as the header's VET_KERNEL_* enum
    slots = re.findall(r"\bVET_KERNEL_([A-Z_]+)\s*=\s*(\d+)", header)
    assert [n.lower() for n, _ in slots if n != "COUNT"] == list(_native.KERNEL_NAMES)
    assert dict(slots)["COUNT"] == str(len(_native.KERNEL_NAMES))
    # argument validation happens before any CUDA call
    h = ctypes.c_void_p()
    assert lib.vet_create(ctypes.byref(h), None) == _native.VET_ERR_INVALID_ARG
    cfg = _native.VetConfig(device=0, video_width=101, video_height=200, num_tile_counts=1,
                            tile_counts=(ctypes.c_int32 * 1)(20), fov_angle=120.0, power_factor=2.0,
                            use_weight_distribution=1)
    assert lib.vet_create(ctypes.byref(h), ctypes.byref(cfg)) == _native.VET_ERR_INVALID_ARG
    assert b"even" in lib.vet_last_error()
    cfg.video_width = 100; cfg.fov_angle = 0.0
    assert lib.vet_create(ctypes.byref(h), ctypes.byref(cfg)) == _native.VET_ERR_INVALID_ARG
    assert b"FOV" in lib.vet_last_error()


def test_no_cpu_fallback(pkg, tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="CUDA device"):
        pkg.Engine(100, 200, [20])
    with pytest.raises(RuntimeError, match="CUDA device"):
        pkg.SpatialEntropyAnalyzer(pkg.AnalyzerConfig(output_dir=tmp_path)).engine


def test_product_does_not_import_oracle():
    for f in (ROOT / "viewport_entropy_toolkit_b200").rglob("*.py"):
        src = f.read_text()
        assert "oracle" not in src.replace("# oracle", ""), f
    for f in (ROOT / "viewport_entropy_toolkit_b200" / "csrc").rglob("*"):
        if f.is_file():
            assert "oracle" not in f.read_text(), f


def test_reference_smoke_tests(pkg, tmp_path):
    """The reference's own tests/test_core.py:10-44, against this package."""
    p = pkg.Point(pixel_x=100, pixel_y=200)
    assert (p.pixel_x, p.pixel_y) == (100, 200)
    r = pkg.RadialPoint(lon=45.0, lat=30.0)
    assert (r.lon, r.lat) == (45.0, 30.0)
    v = pkg.Vector(x=1.0, y=2.0, z=3.0)
    assert (v.x, v.y, v.z) == (1.0, 2.0, 3.0)
    for cls in (pkg.SpatialEntropyAnalyzer, pkg.TransitionEntropyAnalyzer):
        a = cls(config=pkg.AnalyzerConfig(video_width=100, video_height=200, output_dir=tmp_path))
        assert a.config.video_width == 100 and a.config.video_height == 200


def test_config_and_type_validation(pkg, tmp_path):
    with pytest.raises(pkg.ValidationError):
        pkg.EntropyConfig(fov_angle=361)
    with pytest.raises(pkg.ValidationError):
        pkg.EntropyConfig(power_factor=0)
    with pytest.raises(ValueError):
        pkg.AnalyzerConfig(video_width=0, output_dir=tmp_path)
    with pytest.raises(ValueError):
        pkg.AnalyzerConfig(tile_counts=[], output_dir=tmp_path)
    with pytest.raises(ValueError):
        pkg.AnalyzerConfig(tile_counts=[20, -1], output_dir=tmp_path)
    with pytest.raises(TypeError):
        pkg.AnalyzerConfig(use_weight_distribution=True)  # documented by the reference but not a field (SURVEY 5)
    out = tmp_path / "made" / "here"
    cfg = pkg.AnalyzerConfig(output_dir=out)
    assert out.is_dir() and cfg.tile_counts == [20, 50, 100, 250, 1000]
    assert cfg.get_output_path("a", ".csv") == out / "a.csv"
    with pytest.raises(pkg.ValidationError):
        pkg.Point(-1, 0)
    with pytest.raises(pkg.ValidationError):
        pkg.RadialPoint(181, 0)
    with pytest.raises(pkg.ValidationError):
        pkg.Vector(0, 0, 0)
    assert pkg.Vector.from_spherical(-79.2, -11.7) == pkg.Vector(0.183488, -0.961878, -0.202787)
    assert pkg.RadialPoint(190 - 360, 0).normalize_coordinates().lon == -170
    assert issubclass(pkg.ValidationError, pkg.SpatialError)
    # NaiveAnalyzerConfig (CFG:84-126): -1 placeholders accepted at construction, zero rejected
    ncfg = pkg.NaiveAnalyzerConfig(output_dir=tmp_path / "naive")
    assert (ncfg.tile_width, ncfg.tile_height) == (-1, -1) and (tmp_path / "naive").is_dir()
    with pytest.raises(ValueError):
        pkg.NaiveAnalyzerConfig(tile_width=30, tile_height=0, output_dir=tmp_path)
    with pytest.raises(ValueError):
        pkg.NaiveAnalyzerConfig(video_height=-2, tile_width=30, tile_height=30, output_dir=tmp_path)
    # find_naive_tile_index / calculate_naive_tile_weights are host arithmetic (EU:335-381)
    pt = pkg.RadialPoint(-79.2, -11.7)
    assert pkg.find_naive_tile_index(pt, 30, 30) == "3_2"
    assert pkg.find_naive_tile_index(pkg.RadialPoint(180.0, 90.0), 30, 45) == "8_6"   # (point, tile_height, tile_width)
    assert pkg.calculate_naive_tile_weights(pt, 30, 30, pkg.EntropyConfig()) == {"3_2": 1.0}


def test_host_tables_equal_oracle_and_reference(pkg):
    from viewport_entropy_toolkit_b200 import _tables
    g = load_golden("lattices")
    for key in g.files:
        assert np.array_equal(_tables.fibonacci_lattice(int(key[1:])), g[key])
    d = load_golden("decode")
    for (W, H) in [(100, 200), (200, 400), (1920, 1080), (3840, 1920)]:
        lon, lat = _tables.axis_tables(W, H)
        assert np.array_equal(lon, d[f"lon_{W}x{H}"]) and np.array_equal(lat, d[f"lat_{W}x{H}"])
    lon, lat = _tables.axis_tables(100, 200)
    assert np.array_equal(_tables.spherical_to_vector(lon[None, :], lat[:, None]), d["cellvec_100x200"])


def _write_dir(tmp_path, files):
    for name, (t, mu, mv) in files.items():
        pd.DataFrame({"time": t, "2dmu": mu, "2dmv": mv}).to_csv(tmp_path / f"{name}.csv", index=False)


def test_ingest_ragged_directory(pkg, tmp_path):
    """SURVEY Appendix B ragged directory: 0.1 s bins, first-appearance frame order,
    last sample of a bin wins, absent samples are NaN."""
    from viewport_entropy_toolkit_b200 import ingest
    _write_dir(tmp_path, {
        "a": ([5.0, 5.1, 5.2, 5.3], [.5, .5, .6, .7], [.5] * 4),
        "b": ([9.0, 9.1, 9.14, 9.3], [.1, .2, .3, .4], [.2] * 4),
        "c": ([1.2, 1.0, 1.1], [.9] * 3, [.9] * 3),
    })
    packed, times, ids = ingest.load_directory(tmp_path, order=["a", "b", "c"])
    g = group_keys(load_golden("analyzers"))["ragged"]
    assert ids == ["a", "b", "c"]
    assert np.array_equal(times, g["sp_time"])
    assert packed.shape == (4, 3, 3)
    assert np.array_equal(packed[:, 1, 1], [.1, .3, np.nan, .4], equal_nan=True)   # 9.14 overwrote bin 0.1; bin 0.2 absent
    assert np.array_equal(packed[:, 2, 1], [.9, .9, .9, np.nan], equal_nan=True)   # unsorted times binned, 0.3 absent
    # the oracle on this packed tensor reproduces the reference analyzers' rows
    sp = orc.spatial_analyzer(packed, 100, 200, [20])
    np.testing.assert_allclose(sp["entropy"], g["sp_entropy"], rtol=1e-12)
    assert np.array_equal(sp["assign0"], g["sp_assign0"])


def test_ingest_matches_reference_on_synthetic_directory(pkg, tmp_path):
    from viewport_entropy_toolkit_b200 import ingest
    a = load_golden("analyzers")
    g = group_keys(a)
    names = [str(n) for n in g["dir10_default"]["order"]]
    for n in names:
        arr = a[f"dir10/{n}"]
        pd.DataFrame({"extra": 0, "time": arr[:, 0], "2dmu": arr[:, 1], "2dmv": arr[:, 2]}).to_csv(tmp_path / f"{n}.csv", index=False)
    packed, times, ids = ingest.load_directory(tmp_path, order=names)
    assert np.array_equal(times, g["dir10_default"]["sp_time"])
    sp = orc.spatial_analyzer(packed, 100, 200, [20, 50])
    np.testing.assert_allclose(sp["entropy"], g["dir10_default"]["sp_entropy"], rtol=1e-12)
    assert np.array_equal(sp["assign0"], g["dir10_default"]["sp_assign0"])
    np.testing.assert_allclose(sp["hist0"], g["dir10_default"]["sp_hist0"], rtol=1e-12)
    tr = orc.transition_analyzer(packed, 100, 200, [20, 50])
    np.testing.assert_allclose(tr["entropy"], g["dir10_default"]["tr_entropy"], rtol=1e-12, atol=1e-15, equal_nan=True)
    assert np.array_equal(tr["prev_count0"], g["dir10_default"]["tr_prev_count0"])
    # reversed user order + unweighted + three tile counts
    names_r = [str(n) for n in g["dir10_unw"]["order"]]
    packed_r, _, _ = ingest.load_directory(tmp_path, order=names_r)
    sp = orc.spatial_analyzer(packed_r, 100, 200, [50, 20, 200], 90.0, False, 2.0)
    np.testing.assert_allclose(sp["entropy"], g["dir10_unw"]["sp_entropy"], rtol=1e-12)
    tr = orc.transition_analyzer(packed_r, 100, 200, [50, 20, 200])
    np.testing.assert_allclose(tr["entropy"], g["dir10_unw"]["tr_entropy"], rtol=1e-12, atol=1e-15, equal_nan=True)


def test_ingest_errors(pkg, tmp_path):
    from viewport_entropy_toolkit_b200 import ingest
    _write_dir(tmp_path, {"bad": ([0.0, 0.1], [0.5, 1.5], [0.5, 0.5])})
    with pytest.raises(pkg.ValidationError, match="between 0 and 1"):
        ingest.load_directory(tmp_path)
    with pytest.raises(pkg.ValidationError, match="File not found"):
        ingest.read_viewport_csv(tmp_path / "nope.csv")
    a = pkg.SpatialEntropyAnalyzer(pkg.AnalyzerConfig(output_dir=tmp_path / "o"))
    with pytest.raises(FileNotFoundError):
        a.process_directory(tmp_path / "missing_dir")
    with pytest.raises(pkg.ValidationError, match="Failed to process directory"):
        a.process_directory(tmp_path)
    with pytest.raises(pkg.ValidationError, match="No data available"):
        a.compute_entropy()
    with pytest.raises(pkg.ValidationError, match="No entropy results"):
        a.create_visualization("x")
    empty = tmp_path / "empty"
    empty.mkdir()
    with pytest.raises(pkg.ValidationError, match="No trajectory data"):
        a.process_directory(empty)


def _dir10(tmp_path):
    a = load_golden("analyzers")
    names = [f"user{u:02d}" for u in range(10)]
    for n in names:
        arr = a[f"dir10/{n}"]
        pd.DataFrame({"time": arr[:, 0], "2dmu": arr[:, 1], "2dmv": arr[:, 2]}).to_csv(tmp_path / f"{n}.csv", index=False)
    pd.DataFrame({"time": [1.2, 1.0, 1.1, 1.14], "2dmu": [.9, .0, 1.0, .29], "2dmv": [.9, 1.0, 0.0, .57]}).to_csv(tmp_path / "zz.csv", index=False)
    return names + ["zz"]


def test_reference_named_ingest_functions(pkg, tmp_path):
    """process_viewport_data / format_trajectory_data (DU:289-410) under the reference's own names: consistent with
    the packed ingest + oracle decode everywhere, and identical to the LIVE reference when it is present."""
    from viewport_entropy_toolkit_b200 import ingest
    names = _dir10(tmp_path)
    ours = [pkg.process_viewport_data(tmp_path / f"{n}.csv", 100, 200)[::-1] for n in names]
    assert [i for i, _ in ours] == names
    assert list(ours[0][1].columns) == ["time", "2dmu", "2dmv", "pixel_x", "pixel_y", "lon", "lat"]
    points_df, vectors_df = pkg.format_trajectory_data(ours)
    packed, times, ids = ingest.load_directory(tmp_path, order=names)
    assert np.array_equal(points_df["time"].to_numpy(), times) and list(points_df.columns) == ["time"] + names
    vec, valid = orc.decode_vectors(packed[..., 1], packed[..., 2], 100, 200)
    for u, n in enumerate(names):
        for f in range(len(times)):
            v, p = vectors_df[n][f], points_df[n][f]
            if not valid[f, u]:
                assert v is None and p is None
            else:
                assert (v.x, v.y, v.z) == tuple(vec[f, u]) and isinstance(p, pkg.RadialPoint)
    # every point and vector against the reference's own decode chain, stored per pixel in the decode fixtures
    # (lon / lat after the rounding and wrap of DU:390-397, Vector.from_spherical of every cell)
    d = load_golden("decode")
    px, py, _ = orc.decode(packed[..., 1], packed[..., 2], 100, 200)
    checked = 0
    for u, n in enumerate(names):
        for f in np.flatnonzero(valid[:, u]):
            v, p = vectors_df[n][f], points_df[n][f]
            assert (p.lon, p.lat) == (d["lon_100x200"][px[f, u]], d["lat_100x200"][py[f, u]]), (n, f)
            assert (v.x, v.y, v.z) == tuple(d["cellvec_100x200"][py[f, u], px[f, u]]), (n, f)
            checked += 1
    assert checked == int(valid.sum()) > 0
    with pytest.raises(pkg.ValidationError, match="Error processing viewport data"):
        pkg.process_viewport_data(tmp_path / "missing.csv", 100, 200)
    with pytest.raises(pkg.ValidationError, match="even numbers"):
        pkg.process_viewport_data(tmp_path / "zz.csv", 101, 200)
    with pytest.raises(pkg.ValidationError, match="No trajectory data"):
        pkg.format_trajectory_data([])
    from oracle import _refshim
    if not _refshim.reference_available():
        return
    _refshim.load_reference()
    from viewport_entropy_toolkit import utilities as RU
    ref = []
    for (ident, do), n in zip([pkg.process_viewport_data(tmp_path / f"{n}.csv", 100, 200)[::-1] for n in names], names):
        dr, ir = RU.process_viewport_data(tmp_path / f"{n}.csv", 100, 200)
        assert ir == ident and list(dr.columns) == list(do.columns) and (dr.dtypes == do.dtypes).all()
        for c in dr.columns:
            assert np.array_equal(dr[c].to_numpy(), do[c].to_numpy())
        ref.append((ir, dr))
    pr, vr = RU.format_trajectory_data(ref)
    assert np.array_equal(pr["time"].to_numpy(), points_df["time"].to_numpy())
    for n in names:
        for x, y in zip(pr[n], points_df[n]):
            assert (x is None and y is None) or (x.lon, x.lat) == (y.lon, y.lat)
        for x, y in zip(vr[n], vectors_df[n]):
            assert (x is None and y is None) or (x.x, x.y, x.z) == (y.x, y.y, y.z)


def test_integration_stub_matches_the_abi(pkg):
    """The ctypes stub shown in INTEGRATION.md declares struct vet_config exactly like the product's binding
    (a shorter struct would make vet_create read past it)."""
    import ctypes as C
    from pathlib import Path
    from viewport_entropy_toolkit_b200 import _native
    src = (Path(__file__).resolve().parents[1] / "INTEGRATION.md").read_text()
    code = src[src.index("class VetConfig(C.Structure):"):src.index("_lib.vet_last_error.restype")]
    ns = {"C": C}
    exec(code, ns)
    stub = ns["VetConfig"]
    assert [f[0] for f in stub._fields_] == [f[0] for f in _native.VetConfig._fields_]
    assert C.sizeof(stub) == C.sizeof(_native.VetConfig)
    header = (Path(__file__).resolve().parents[1] / "include" / "vet_b200.h").read_text()
    body = header[header.index("typedef struct {"):header.index("} vet_config;")]
    for name, _ in _native.VetConfig._fields_:
        assert name in body, name


def test_committed_bench_lines_carry_the_contract_keys():
    """The bench lines kept under profiles/ (one per GPU count) have every key of the bench contract, the roofline /
    cpu_baseline / e2e objects included, and the strong-scaling block of configs[4]."""
    import json
    from pathlib import Path
    prof = Path(__file__).resolve().parents[1] / "profiles"
    for n in (1, 2, 4, 8):
        d = json.loads((prof / f"bench_r02_n{n}.json").read_text())
        for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                  "vs_baseline", "dtype", "data", "config", "roofline", "e2e", "clocks", "gpu_launches"):
            assert k in d, (n, k)
        assert d["n_gpus"] == n and d["gpu_launches"] > 0 and "workload" in d["config"]
        for k in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
            assert k in d["roofline"], (n, k)
        for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
            assert k in d["e2e"], (n, k)
        c5 = d["extra"]["c5_sharded"]
        assert c5["n_gpus"] == n and c5["scaling"] == "strong" and c5["checks_ok"] is True
        if n == 1:
            for k in ("value", "unit", "cores", "kind", "sample"):
                assert k in d["cpu_baseline"], k


def test_tensor_core_dispatch_threshold_matches_the_header():
    """distributed.py pins the weighted-histogram kernel per job with the library's own threshold."""
    import re
    from pathlib import Path
    from viewport_entropy_toolkit_b200 import _native
    header = (Path(__file__).resolve().parents[1] / "include" / "vet_b200.h").read_text()
    assert int(re.search(r"#define VET_I8_MIN_FRAMES (\d+)", header).group(1)) == _native.I8_MIN_FRAMES


def test_tile_geometry_vs_reference_fixtures(pkg):
    """Tile geometry for renders (DU:58-225, 412-743): boundary segments of the Fibonacci tiles, latitude/longitude
    tile boxes and tile areas, bit for bit against the live-reference fixtures."""
    from viewport_entropy_toolkit_b200 import geometry as G
    g = group_keys(load_golden("geometry"))
    for n in (3, 20, 50, 200):
        b = G.get_fb_tile_boundaries(n)
        assert len(b) == int(g[f"fb{n}"]["tiles"][0])
        rows = [(i, e, p1.x, p1.y, p1.z, p2.x, p2.y, p2.z) for i, edges in b.items() for e, (p1, p2) in enumerate(edges)]
        assert np.array_equal(np.array(rows, dtype=np.float64).reshape(-1, 8), g[f"fb{n}"]["edges"]), n
    for n in (20, 50):
        area, frac = G.compute_fb_tile_areas(n)
        assert np.array_equal(np.array([area[i] for i in range(len(area))]), g[f"fb{n}"]["area"])
        assert np.array_equal(np.array([frac[i] for i in range(len(frac))]), g[f"fb{n}"]["fraction"])
        assert abs(sum(frac.values()) - 1.0) < 1e-12           # the tiles cover the sphere
    for nh, nv in ((4, 2), (12, 6)):
        t = G.get_lat_lon_tiles(nh, nv)
        keys = sorted(t)
        assert keys == [str(k) for k in g[f"ll{nh}x{nv}"]["keys"]]
        rows = [(ki, e, p1.x, p1.y, p1.z, p2.x, p2.y, p2.z) for ki, k in enumerate(keys) for e, (p1, p2) in enumerate(t[k])]
        assert np.array_equal(np.array(rows, dtype=np.float64), g[f"ll{nh}x{nv}"]["edges"])
        area, frac = G.compute_lat_lon_tile_areas(nh, nv)
        assert np.array_equal(np.array([area[k] for k in keys]), g[f"ll{nh}x{nv}"]["area"])
    with pytest.raises(pkg.ValidationError):
        G.get_fb_tile_boundaries(0)
    with pytest.raises(pkg.ValidationError):
        G.compute_lat_lon_tile_areas(0, 4)
    with pytest.raises(ValueError):
        G.triangulate_spherical_polygon([pkg.Vector(1, 0, 0), pkg.Vector(0, 1, 0)])
    # convert_vectors_to_coordinates (DT:219-276)
    lons, lats = pkg.convert_vectors_to_coordinates([pkg.Vector(1, 0, 0), pkg.Vector(0, 1, 0), pkg.Vector(-1, 0, 0), pkg.Vector(0, 0, 2)])
    assert np.array_equal(lons, [0.0, 90.0, 180.0, 0.0]) and np.array_equal(lats, [0.0, 0.0, 0.0, 90.0])
    with pytest.raises(pkg.ValidationError):
        pkg.convert_vectors_to_coordinates([])
    # exported under the reference's names
    for name in ("get_fb_tile_boundaries", "get_lat_lon_tiles", "normalize", "great_circle_intersection", "get_tile_corners",
                 "compute_spherical_polygon_area", "spherical_interpolation", "find_nearest_point", "angle_at_vertex"):
        assert getattr(pkg.utilities, name) is getattr(G, name)


def test_lazy_row_dict_is_a_read_only_dict_view():
    """LazyRowDict (the per-frame `tile_weights` / `tile_assignments` cells of the analyzers' DataFrames, SA:152-163):
    built on first access, equal to the dict it stands for, usable like one."""
    import pandas as pd
    from viewport_entropy_toolkit_b200.analyzers import LazyRowDict
    calls = []

    def make():
        calls.append(1)
        return {"a": 1, "b": 2}

    d = LazyRowDict(make)
    df = pd.DataFrame({"time": [0.0], "tile_assignments": [d]})     # stays one object cell, not expanded
    assert not calls and df["tile_assignments"][0] is d
    assert d == {"a": 1, "b": 2} and {"a": 1, "b": 2} == d and len(calls) == 1
    assert len(d) == 2 and "a" in d and d.get("c", 7) == 7 and sorted(d.items()) == [("a", 1), ("b", 2)] and dict(d) == {"a": 1, "b": 2}
    assert len(calls) == 1 and repr(d) == repr({"a": 1, "b": 2})
    with pytest.raises(TypeError):
        d["c"] = 3


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm: the reference's own functions from /root/reference or baseline/_ref, else
    the oracle port) prints ONE JSON line with the contract's keys; needs no GPU."""
    import json
    import subprocess
    import sys
    root = Path(__file__).resolve().parents[1]
    out = subprocess.run([sys.executable, str(root / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=str(root))
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "samples/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("configs[2]") and d["gpu_launches"] == 0
