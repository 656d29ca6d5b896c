"""CPU oracle for the SpatialEntropyAnalyzer / TransitionEntropyAnalyzer hot path.

TEST INFRASTRUCTURE ONLY.  This module is a CPU restatement (numpy, fp64) of the
reference's algorithm for the hot path named in BASELINE.json.  Only `tests/`,
`__graft_entry__.smoke()` and `bench.py`'s CPU-baseline legs may import it; the
product (`viewport_entropy_toolkit_b200`) never does and has no CPU fallback.

Parity status: the reference's own test-suite holds NO golden vectors for this
path (tests/test_core.py:10-44 only checks constructors), so parity is pinned
by us instead: `tests/golden/make_golden.py` imports the LIVE reference in the
build container (through `oracle/_refshim.py`) and writes its outputs to
`tests/golden/*.npz`; `tests/test_oracle_golden.py` checks every function below
against those fixtures (and against the live reference when it is present).

Paths are relative to /root/reference/src/viewport_entropy_toolkit/:
  EU = utilities/entropy_utils.py   DU = utilities/data_utils.py
  DT = data_types.py                SA = analyzers/spatial_entropy.py
  TA = analyzers/transition_entropy.py

Two layers:
  * `*_literal` functions keep the reference's scalar call structure (one
    numpy-scalar distance evaluation per (vector, tile), Python dict
    bookkeeping).  They are bit-identical to the reference on the same host and
    have its performance character; the CPU baseline in bench.py times these.
  * the un-suffixed functions are numpy-vectorised restatements, used where the
    literal layer is too slow (exhaustive-domain and large-sample checks).
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

MISSING = 0xFFFF  # sentinel tile index for a missing sample (None in SA:131-135)


class OracleValidationError(Exception):
    """Stands in for the reference's ValidationError (DT:25-27)."""


# ---------------------------------------------------------------------------
# Vector.from_spherical  (DT:183-216)
# ---------------------------------------------------------------------------
def from_spherical(lon, lat) -> np.ndarray:
    """DT:204-216: theta=radians(lon), phi=radians(90-lat); components rounded
    to 6 decimals with numpy's round (== rint(v*1e6)/1e6).  Vectorised; returns
    [...,3] float64."""
    lon = np.asarray(lon, dtype=np.float64)
    lat = np.asarray(lat, dtype=np.float64)
    theta = np.radians(lon)              # DT:204
    phi = np.radians(90 - lat)           # DT:205
    x = np.sin(phi) * np.cos(theta)      # DT:208
    y = np.sin(phi) * np.sin(theta)      # DT:209
    z = np.cos(phi) + 0.0 * theta        # DT:210 (broadcast to common shape)
    out = np.stack([x, y, z], axis=-1)
    return np.round(out, 6)              # DT:212-216


# ---------------------------------------------------------------------------
# generate_fibonacci_lattice  (DU:25-56)
# ---------------------------------------------------------------------------
def lattice_size(n: int) -> int:
    """DU:43-45: the lattice has 2*int(n/2)+1 points, not n."""
    return 2 * int(n / 2) + 1


def lattice(n: int) -> np.ndarray:
    """DU:37-56.  Returns centres [T,3] float64 (6-dp rounded, not unit length)."""
    if n <= 0:
        raise OracleValidationError("Number of points must be positive")  # DU:37-38
    phi = (1 + np.sqrt(5)) / 2           # DU:40
    N = int(n / 2)                       # DU:43
    out = np.empty((2 * N + 1, 3), dtype=np.float64)
    for k, i in enumerate(range(-N, N + 1)):
        lat = np.arcsin(2 * i / (2 * N + 1)) * 180 / np.pi   # DU:46
        lon = (i % phi) * 360 / phi                          # DU:47 (python int % np.float64)
        lon = ((lon + 180) % 360) - 180                      # DU:50
        out[k] = from_spherical(lon, lat)                    # DU:53
    return out


# ---------------------------------------------------------------------------
# decode: normalize_to_pixel (DU:243-261), pixel_to_spherical (DU:264-286),
# rounding / wrap quirk (DU:390-397), Vector.from_spherical (DU:403)
# ---------------------------------------------------------------------------
def validate_video_dimensions(W: int, H: int) -> None:
    """DU:227-240."""
    if W <= 0 or H <= 0:
        raise OracleValidationError("Video dimensions must be positive")
    if W % 2 != 0 or H % 2 != 0:
        raise OracleValidationError("Video dimensions must be even numbers")


def normalize_to_pixel(normalized: np.ndarray, dimension: int) -> np.ndarray:
    """DU:256-261: reject values outside [0,1]; trunc(normalized*dimension)."""
    normalized = np.asarray(normalized, dtype=np.float64)
    if np.any((normalized < 0) | (normalized > 1)):
        raise OracleValidationError("Normalized coordinates must be between 0 and 1")
    if dimension <= 0:
        raise OracleValidationError("Dimension must be positive")
    return (normalized * dimension).astype(np.int64)


def axis_tables(W: int, H: int) -> Tuple[np.ndarray, np.ndarray]:
    """lon for every pixel column px in [0,W] and lat for every row py in [0,H]
    AFTER the 0.1-degree rounding and the wrap quirk.

    DU:283-284  lon=(px/W)*360-180, lat=90-(py/H)*180 (each op rounded, fp64)
    DU:390-391  python round(.,1)  (correctly-rounded decimal, NOT rint(x*10)/10)
    DU:394-397  lon<=-180 -> (lon+360)%360-180 (=0.0), lat<=-90 -> (lat+180)%180-90 (=0.0)
    """
    validate_video_dimensions(W, H)
    lon = np.empty(W + 1, dtype=np.float64)
    lat = np.empty(H + 1, dtype=np.float64)
    for px in range(W + 1):
        v = float((np.float64(px) / W) * 360 - 180)
        v = round(v, 1)
        if v <= -180:
            v = (v + 360) % 360 - 180
        lon[px] = v
    for py in range(H + 1):
        v = float(90 - (np.float64(py) / H) * 180)
        v = round(v, 1)
        if v <= -90:
            v = (v + 180) % 180 - 90
        lat[py] = v
    return lon, lat


def cell_vectors(W: int, H: int) -> np.ndarray:
    """Direction vector of every reachable cell: [(H+1),(W+1),3] float64.
    The decode map is a pure function of (px,py) (SURVEY A.2)."""
    lon, lat = axis_tables(W, H)
    return from_spherical(lon[None, :], lat[:, None])


def decode(mu, mv, W: int, H: int) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """(mu, mv) -> (px, py, valid).  NaN in either coordinate marks a missing
    sample (dropna at DU:314 / None at SA:131-135); a non-missing value outside
    [0,1] raises like DU:256-257."""
    mu = np.asarray(mu, dtype=np.float64)
    mv = np.asarray(mv, dtype=np.float64)
    valid = ~(np.isnan(mu) | np.isnan(mv))
    mu0 = np.where(valid, mu, 0.0)
    mv0 = np.where(valid, mv, 0.0)
    px = normalize_to_pixel(mu0, W)
    py = normalize_to_pixel(mv0, H)
    return px, py, valid


def decode_vectors(mu, mv, W: int, H: int) -> Tuple[np.ndarray, np.ndarray]:
    """(mu, mv) -> (vectors[...,3], valid)."""
    px, py, valid = decode(mu, mv, W, H)
    cv = cell_vectors(W, H)
    vec = cv[py, px]
    vec = np.where(valid[..., None], vec, np.nan)
    return vec, valid


# ---------------------------------------------------------------------------
# vector_angle_distance (EU:41-67) and friends
# ---------------------------------------------------------------------------
def vector_angle_distance_literal(v1: Sequence[float], v2: Sequence[float]) -> np.float64:
    """EU:54-64, call for call."""
    v1_np = np.array([v1[0], v1[1], v1[2]])
    v2_np = np.array([v2[0], v2[1], v2[2]])
    v1_normalized = v1_np / np.linalg.norm(v1_np)
    v2_normalized = v2_np / np.linalg.norm(v2_np)
    dot_product = np.dot(v1_normalized, v2_normalized)
    dot_product = np.clip(dot_product, -1.0, 1.0)
    return np.arccos(dot_product)


def find_angular_distances_literal(vector, centres) -> np.ndarray:
    """EU:83-87."""
    return np.array([[i, vector_angle_distance_literal(vector, c)] for i, c in enumerate(centres)])


def find_nearest_tile_literal(vector, centres) -> int:
    """EU:103-106: first minimum wins."""
    d = find_angular_distances_literal(vector, centres)
    return int(d[np.argmin(d[:, 1])][0])


def calculate_tile_weights_literal(vector, centres, fov_angle, use_weight, power_factor) -> Dict[int, float]:
    """EU:123-144 (dict keyed by tile INDEX instead of Vector; lattices hold no
    duplicate centres, checked in tests, so the keys are in 1:1 correspondence)."""
    weights: Dict[int, float] = {}
    max_d = np.radians(fov_angle / 2.0)
    d = find_angular_distances_literal(vector, centres)
    d = sorted(d, key=lambda x: x[1])
    if use_weight:
        for tile_idx, dist in d:
            if dist < max_d:
                weights[int(tile_idx)] = ((max_d - dist) / max_d) ** power_factor
            else:
                break
    else:
        weights[int(d[0][0])] = 1.0
    return weights


def _unit(v: np.ndarray) -> np.ndarray:
    """EU:58-59: v / ||v|| in fp64 (np.linalg.norm == sqrt(sum of squares))."""
    return v / np.sqrt((v * v).sum(axis=-1, keepdims=True))


def dots(vecs: np.ndarray, centres: np.ndarray) -> np.ndarray:
    """Normalised dot products [n,T] (EU:58-62).  Evaluation order differs from
    OpenBLAS ddot by <= 2 ulp; SURVEY 0.4 shows only the ordering matters and
    the smallest non-tie gap over the reachable domain is 7e-10."""
    a = _unit(np.asarray(vecs, dtype=np.float64))
    b = _unit(np.asarray(centres, dtype=np.float64))
    d = a[:, None, 0] * b[None, :, 0]
    d = d + a[:, None, 1] * b[None, :, 1]
    d = d + a[:, None, 2] * b[None, :, 2]
    return np.clip(d, -1.0, 1.0)


def angular_distances(vecs: np.ndarray, centres: np.ndarray) -> np.ndarray:
    """EU:62-64 vectorised: arccos(clip(dot)) -> [n,T]."""
    return np.arccos(dots(vecs, centres))


def nearest_tile(vecs: np.ndarray, centres: np.ndarray, chunk: int = 8192) -> np.ndarray:
    """EU:103-104 vectorised: argmin over arccos, first minimum wins -> [n] int32."""
    vecs = np.asarray(vecs, dtype=np.float64).reshape(-1, 3)
    out = np.empty(len(vecs), dtype=np.int32)
    for s in range(0, len(vecs), chunk):
        out[s:s + chunk] = np.argmin(angular_distances(vecs[s:s + chunk], centres), axis=1)
    return out


def tile_weights(vecs: np.ndarray, centres: np.ndarray, fov_angle: float,
                 use_weight: bool, power_factor: float) -> np.ndarray:
    """EU:123-144 vectorised -> dense [n,T] (0 where a tile gets no weight)."""
    d = angular_distances(vecs, centres)
    if use_weight:
        max_d = np.radians(fov_angle / 2.0)
        with np.errstate(invalid="ignore"):
            w = ((max_d - d) / max_d) ** power_factor
        return np.where(d < max_d, w, 0.0)
    w = np.zeros_like(d)
    w[np.arange(len(d)), np.argmin(d, axis=1)] = 1.0
    return w


# ---------------------------------------------------------------------------
# compute_spatial_entropy (EU:147-211)
# ---------------------------------------------------------------------------
def compute_spatial_entropy_literal(vector_dict: Dict[str, Optional[Sequence[float]]], centres,
                                    fov_angle=120.0, use_weight=True, power_factor=2.0):
    """EU:168-211, statement for statement.  Returns (entropy, {tile: weight},
    {identifier: tile})."""
    if not vector_dict:
        raise OracleValidationError("Empty vector dictionary")
    if len(centres) == 0:
        raise OracleValidationError("No tile centers provided")
    num_tiles = len(centres)
    weight_per_tile: Dict[int, float] = {}
    total_weight = 0.0
    tile_assignments: Dict[str, int] = {}
    for identifier, vector in vector_dict.items():
        if vector is None:
            continue
        weights = calculate_tile_weights_literal(vector, centres, fov_angle, use_weight, power_factor)
        tile_assignments[identifier] = find_nearest_tile_literal(vector, centres)
        for tile, weight in weights.items():
            weight_per_tile[tile] = weight_per_tile.get(tile, 0.0) + weight
            total_weight += weight
    spatial_entropy = 0.0
    with np.errstate(divide="ignore", invalid="ignore"):
        for weight in weight_per_tile.values():
            proportion = weight / total_weight
            spatial_entropy -= proportion * np.log2(proportion)
        if use_weight or total_weight > num_tiles:
            max_proportion = 1.0 / num_tiles
            max_entropy = -num_tiles * max_proportion * np.log2(max_proportion)
        else:
            max_proportion = 1.0 / total_weight
            max_entropy = -total_weight * max_proportion * np.log2(max_proportion)
        normalized = np.float64(spatial_entropy) / np.float64(max_entropy)
    return normalized, weight_per_tile, tile_assignments


def entropy_from_hist(hist: np.ndarray, num_tiles: int, use_weight: bool) -> float:
    """EU:195-209 on a dense histogram row: H=-sum p log2 p over touched tiles,
    normalised by log2(T) if weighted or total>T else log2(total)."""
    hist = np.asarray(hist, dtype=np.float64)
    total = hist.sum()
    nz = hist[hist > 0]
    with np.errstate(divide="ignore", invalid="ignore"):
        p = nz / total
        H = -(p * np.log2(p)).sum() if nz.size else 0.0
        n = np.float64(num_tiles) if (use_weight or total > num_tiles) else np.float64(total)
        max_proportion = 1.0 / n                                  # EU:202 / EU:205
        mx = -n * max_proportion * np.log2(max_proportion)        # EU:203 / EU:206
        return float(np.float64(H) / np.float64(mx))


def spatial_entropy(vecs: np.ndarray, centres: np.ndarray, fov_angle=120.0,
                    use_weight=True, power_factor=2.0):
    """EU:173-211 vectorised for one frame; `vecs` holds only present users.
    Returns (entropy, hist[T], assign[n])."""
    w = tile_weights(vecs, centres, fov_angle, use_weight, power_factor)
    hist = w.sum(axis=0)
    assign = nearest_tile(vecs, centres)
    return entropy_from_hist(hist, len(centres), use_weight), hist, assign


# ---------------------------------------------------------------------------
# compute_transition_entropy (EU:213-332) -- literal, bugs included
# ---------------------------------------------------------------------------
def compute_transition_entropy_literal(prior: Dict[str, Sequence[float]], current: Dict[str, Sequence[float]],
                                       centres):
    """EU:239-332 statement for statement.  The reference keys its inner dict
    by `int` for the first user of a prev-tile and by `Vector` for later users
    (EU:280-287); here ("i", c) / ("v", c) keep that distinction.  The stale
    `transition_weight` reuse at EU:312-315 is reproduced.  Returns (entropy,
    {prev_tile: count}, {identifier: (prev, cur)})."""
    if not prior or not current:
        raise OracleValidationError("Empty vector dictionary")
    if len(centres) == 0:
        raise OracleValidationError("No tile centers provided")
    num_tiles = len(centres)
    weight_per_tile: Dict[int, int] = {}
    transition_weight_per_tile: Dict[int, Dict[Tuple[str, int], int]] = {}
    total_weight = 0
    tile_assignments: Dict[str, Tuple[int, int]] = {}
    transition_entropy = 0
    for identifier, vector in current.items():
        if identifier not in prior or identifier not in current:
            continue
        p = find_nearest_tile_literal(prior[identifier], centres)     # EU:271
        c = find_nearest_tile_literal(current[identifier], centres)   # EU:273
        tile_assignments[identifier] = (p, c)                         # EU:276
        weight = 1
        if p not in weight_per_tile:                                  # EU:280-282
            transition_weight_per_tile[p] = {}
            transition_weight_per_tile[p][("i", c)] = weight
        else:                                                         # EU:283-287
            if ("v", c) not in transition_weight_per_tile[p]:
                transition_weight_per_tile[p][("v", c)] = weight
            else:
                transition_weight_per_tile[p][("v", c)] += weight
        if p not in weight_per_tile:                                  # EU:289-292
            weight_per_tile[p] = weight
        else:
            weight_per_tile[p] += weight
        total_weight += weight
    for p in weight_per_tile:                                         # EU:297-318
        tile_proportion = float(weight_per_tile[p]) / float(total_weight)
        total_transition_weight = 0
        total_cell = 0
        for key in transition_weight_per_tile[p]:
            transition_weight = transition_weight_per_tile[p][key]
            total_transition_weight += transition_weight
        for key in transition_weight_per_tile[p]:
            tp = float(transition_weight) / float(total_transition_weight)   # stale variable
            total_cell += tp * np.log2(tp)
        transition_entropy += -tile_proportion * total_cell
    with np.errstate(divide="ignore", invalid="ignore"):
        if total_weight > num_tiles:                                  # EU:321-327
            q = 1 / num_tiles
            mx = num_tiles * -q * np.log2(q)
        else:
            q = 1 / total_weight          # ZeroDivisionError when no common user
            mx = total_weight * -q * np.log2(q)
        result = np.float64(transition_entropy) / np.float64(mx)
    return result, weight_per_tile, tile_assignments


def transition_stats(prev_idx: np.ndarray, cur_idx: np.ndarray, T: int):
    """Closed form of the literal bookkeeping (SURVEY A.6), users in order.
    Returns m[T] (users per prev tile), K[T] (1 + #distinct cur among the
    non-first users) and w[T] (count, among non-first users, of the cur whose
    first appearance among them is latest; 1 when m==1)."""
    prev_idx = np.asarray(prev_idx, dtype=np.int64)
    cur_idx = np.asarray(cur_idx, dtype=np.int64)
    m = np.zeros(T, dtype=np.int64)
    K = np.zeros(T, dtype=np.int64)
    w = np.zeros(T, dtype=np.int64)
    seen_first = np.zeros(T, dtype=bool)
    counts: Dict[Tuple[int, int], int] = {}
    latest: Dict[int, int] = {}
    for p, c in zip(prev_idx.tolist(), cur_idx.tolist()):
        m[p] += 1
        if not seen_first[p]:
            seen_first[p] = True
            K[p] = 1
            continue
        key = (p, c)
        if key not in counts:
            counts[key] = 1
            K[p] += 1
            latest[p] = c
        else:
            counts[key] += 1
    for p in range(T):
        if m[p] == 1:
            w[p] = 1
        elif m[p] > 1:
            w[p] = counts[(p, latest[p])]
    return m, K, w


def transition_entropy_from_stats(m: np.ndarray, K: np.ndarray, w: np.ndarray, T: int) -> float:
    """H = sum_p (m_p/total) * (-K_p q_p log2 q_p), q_p = w_p/m_p; normalised by
    log2(T) if total>T else log2(total) (EU:297-330).  total==1 -> NaN.
    total==0 raises like the reference's ZeroDivisionError (EU:326)."""
    total = int(m.sum())
    if total == 0:
        raise ZeroDivisionError("division by zero")
    act = m > 0
    q = w[act] / m[act]
    with np.errstate(divide="ignore", invalid="ignore"):
        H = ((m[act] / total) * (-(K[act] * (q * np.log2(q))))).sum()
        n = np.float64(T) if total > T else np.float64(total)
        q_max = 1 / n                                             # EU:322 / EU:326
        mx = n * -q_max * np.log2(q_max)                          # EU:323 / EU:327
        return float(np.float64(H) / np.float64(mx))


def transition_entropy(prev_idx: np.ndarray, cur_idx: np.ndarray, T: int):
    """Literal transition entropy from tile indices of the common users (in
    current-frame order).  Returns (entropy, m[T])."""
    m, K, w = transition_stats(prev_idx, cur_idx, T)
    return transition_entropy_from_stats(m, K, w, T), m


def transition_entropy_textbook(prev_idx: np.ndarray, cur_idx: np.ndarray, T: int) -> float:
    """Opt-in 'textbook' mode (NOT the reference's behaviour):
    -sum_p P(p) sum_c P(c|p) log2 P(c|p), same normalisation rule."""
    prev_idx = np.asarray(prev_idx, dtype=np.int64)
    cur_idx = np.asarray(cur_idx, dtype=np.int64)
    total = len(prev_idx)
    if total == 0:
        raise ZeroDivisionError("division by zero")
    pair, cnt = np.unique(prev_idx * T + cur_idx, return_counts=True)
    m = np.bincount(prev_idx, minlength=T)
    mp = m[pair // T]
    with np.errstate(divide="ignore", invalid="ignore"):
        H = -((cnt / total) * np.log2(cnt / mp)).sum()
        mx = np.log2(np.float64(T)) if total > T else np.log2(np.float64(total))
        return float(np.float64(H) / np.float64(mx))


# ---------------------------------------------------------------------------
# analyzer frame loops (SA:129-161, TA:129-172) on packed [F,U,3] input
# ---------------------------------------------------------------------------
def cell_luts(W: int, H: int, tile_counts: Sequence[int]) -> List[np.ndarray]:
    """Nearest tile of every reachable cell, per tile count: [(H+1)*(W+1)] int32."""
    cv = cell_vectors(W, H).reshape(-1, 3)
    return [nearest_tile(cv, lattice(n)) for n in tile_counts]


def spatial_analyzer(packed: np.ndarray, W: int, H: int, tile_counts: Sequence[int],
                     fov_angle=120.0, use_weight=True, power_factor=2.0,
                     centres: Optional[Sequence[np.ndarray]] = None):
    """SA:129-161 on packed[F,U,3]=(time,2dmu,2dmv); NaN 2dmu/2dmv = missing.
    Returns dict(entropy[F] (mean over tile counts), per_k[K,F], hist0[F,T0],
    assign0[F,U] uint16 (MISSING for absent users)).  A frame without users
    raises like EU:168-169.  `centres` optionally replaces the Fibonacci
    lattices by arbitrary tile centres (the reference's free functions take any
    list of vectors)."""
    packed = np.asarray(packed)
    F, U, _ = packed.shape
    px, py, valid = decode(packed[..., 1], packed[..., 2], W, H)
    cv = cell_vectors(W, H)
    lats = [np.asarray(c, dtype=np.float64) for c in centres] if centres is not None else [lattice(n) for n in tile_counts]
    K = len(lats)
    T0 = len(lats[0])
    per_k = np.empty((K, F), dtype=np.float64)
    hist0 = np.zeros((F, T0), dtype=np.float64)
    assign0 = np.full((F, U), MISSING, dtype=np.uint16)
    for f in range(F):
        ok = valid[f]
        if not ok.any():
            raise OracleValidationError("Empty vector dictionary")
        vecs = cv[py[f][ok], px[f][ok]]
        for k, centres in enumerate(lats):
            e, hist, assign = spatial_entropy(vecs, centres, fov_angle, use_weight, power_factor)
            per_k[k, f] = e
            if k == 0:
                hist0[f] = hist
                assign0[f, ok] = assign
    ent = np.zeros(F, dtype=np.float64)
    for k in range(K):                       # SA:141-156: sequential sum, then / K
        ent = ent + per_k[k]
    return dict(entropy=ent / K, per_k=per_k, hist0=hist0, assign0=assign0)


def transition_analyzer(packed: np.ndarray, W: int, H: int, tile_counts: Sequence[int],
                        mode: str = "literal", centres: Optional[Sequence[np.ndarray]] = None):
    """TA:129-172 on packed[F,U,3].  Row r describes frames (r, r+1); users must
    be present in both.  Returns dict(entropy[F-1], per_k[K,F-1],
    prev_count0[F-1,T0] int32, pairs0[F-1,U,2] uint16).  `centres` as in
    spatial_analyzer."""
    packed = np.asarray(packed)
    F, U, _ = packed.shape
    px, py, valid = decode(packed[..., 1], packed[..., 2], W, H)
    cell = py * (W + 1) + px
    if centres is not None:
        cvf = cell_vectors(W, H).reshape(-1, 3)
        luts = [nearest_tile(cvf, np.asarray(c, dtype=np.float64), chunk=512) for c in centres]
        Ts = [len(c) for c in centres]
    else:
        luts = cell_luts(W, H, tile_counts)
        Ts = [lattice_size(n) for n in tile_counts]
    K = len(Ts)
    per_k = np.empty((K, max(F - 1, 0)), dtype=np.float64)
    prev_count0 = np.zeros((max(F - 1, 0), Ts[0]), dtype=np.int32)
    pairs0 = np.full((max(F - 1, 0), U, 2), MISSING, dtype=np.uint16)
    for r in range(F - 1):
        if not valid[r].any() or not valid[r + 1].any():
            raise OracleValidationError("Empty vector dictionary")   # EU:239-240
        both = valid[r] & valid[r + 1]
        for k in range(K):
            p = luts[k][cell[r][both]]
            c = luts[k][cell[r + 1][both]]
            if mode == "literal":
                e, m = transition_entropy(p, c, Ts[k])
            else:
                e = transition_entropy_textbook(p, c, Ts[k])
                m = np.bincount(p, minlength=Ts[k])
            per_k[k, r] = e
            if k == 0:
                prev_count0[r] = m
                pairs0[r, both, 0] = p
                pairs0[r, both, 1] = c
    ent = np.zeros(max(F - 1, 0), dtype=np.float64)
    for k in range(K):                       # TA:139-160
        ent = ent + per_k[k]
    return dict(entropy=ent / K, per_k=per_k, prev_count0=prev_count0, pairs0=pairs0)


# ---------------------------------------------------------------------------
# Latitude/longitude grid tiling (NaiveSpatialEntropyAnalyzer; EU:335-453, NA:102-152)
# ---------------------------------------------------------------------------
def naive_tile_index(lon, lat, tile_width: int, tile_height: int) -> Tuple[np.ndarray, np.ndarray]:
    """find_naive_tile_index (EU:378-379), vectorised: int((lon+180)/tile_width), int((lat+90)/tile_height)
    (true division, truncation; both operands non-negative for valid RadialPoints)."""
    li = np.trunc((np.asarray(lon, dtype=np.float64) + 180) / tile_width).astype(np.int64)
    la = np.trunc((np.asarray(lat, dtype=np.float64) + 90) / tile_height).astype(np.int64)
    return li, la


def compute_naive_spatial_entropy_literal(points: Dict[str, Optional[Tuple[float, float]]], tile_height: int,
                                          tile_width: int, use_weight: bool):
    """compute_naive_spatial_entropy (EU:404-453) with its dict bookkeeping; points maps an identifier
    to (lon, lat) or None.  Returns (entropy, {key: weight}, {identifier: key})."""
    if not points:
        raise OracleValidationError("Empty radial points dictionary")
    if not tile_height or not tile_width:
        raise OracleValidationError("No tile dimensions provided")
    if 180 % tile_height != 0:
        raise OracleValidationError("Tile height must divide 180!")
    if 360 % tile_width != 0:
        raise OracleValidationError("Tile width must divide 360!")
    num_tiles = int(180.0 / tile_height) * int(360.0 / tile_width)      # EU:409
    weight_per_tile: Dict[str, float] = {}
    total_weight = 0.0
    assignments: Dict[str, str] = {}
    for identifier, point in points.items():
        if point is None:                                                # EU:426-427
            continue
        key = f"{int((point[0] + 180) / tile_width)}_{int((point[1] + 90) / tile_height)}"   # EU:378-381
        assignments[identifier] = key
        weight_per_tile[key] = weight_per_tile.get(key, 0.0) + 1.0      # EU:357, 433-435
        total_weight += 1.0
    spatial_entropy = 0.0
    for weight in weight_per_tile.values():                              # EU:437-440
        proportion = weight / total_weight
        spatial_entropy -= proportion * np.log2(proportion)
    with np.errstate(divide="ignore", invalid="ignore"):
        if use_weight or total_weight > num_tiles:                       # EU:443-448
            max_proportion = 1.0 / num_tiles
            max_entropy = -num_tiles * max_proportion * np.log2(max_proportion)
        else:
            max_proportion = 1.0 / total_weight
            max_entropy = -total_weight * max_proportion * np.log2(max_proportion)
        return np.float64(spatial_entropy) / max_entropy, weight_per_tile, assignments


def naive_analyzer(packed: np.ndarray, W: int, H: int, tile_width: int, tile_height: int, use_weight: bool):
    """NA:125-150 on packed[F,U,3].  Returns dict(entropy[F], hist0[F,codes] (users per grid code
    lon_idx*(180/tile_height+1)+lat_idx), assign0[F,U] uint16 codes, lon_idx/lat_idx[F,U] (-1 = absent))."""
    packed = np.asarray(packed)
    F, U, _ = packed.shape
    px, py, valid = decode(packed[..., 1], packed[..., 2], W, H)
    lon_t, lat_t = axis_tables(W, H)
    li, la = naive_tile_index(lon_t[px], lat_t[py], tile_width, tile_height)
    nlat1 = 180 // tile_height + 1
    codes = (360 // tile_width + 1) * nlat1
    num_tiles = int(180.0 / tile_height) * int(360.0 / tile_width)
    ent = np.empty(F, dtype=np.float64)
    hist0 = np.zeros((F, codes), dtype=np.float64)
    assign0 = np.full((F, U), MISSING, dtype=np.uint16)
    for f in range(F):
        ok = valid[f]
        if not ok.any():
            raise OracleValidationError("Empty radial points dictionary")
        code = li[f][ok] * nlat1 + la[f][ok]
        hist = np.bincount(code, minlength=codes).astype(np.float64)
        total = float(ok.sum())
        p = hist[hist > 0] / total
        Hs = -(p * np.log2(p)).sum()
        n = float(num_tiles) if (use_weight or total > num_tiles) else total
        with np.errstate(divide="ignore", invalid="ignore"):
            ent[f] = np.float64(Hs) / (-n * (1.0 / n) * np.log2(1.0 / n))
        hist0[f] = hist
        assign0[f, ok] = code
    return dict(entropy=ent, hist0=hist0, assign0=assign0, lon_idx=np.where(valid, li, -1), lat_idx=np.where(valid, la, -1))
