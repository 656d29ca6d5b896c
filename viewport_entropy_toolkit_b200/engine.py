"""Device engine: owns one native handle per (device, configuration) and exposes
the tensor-level API of the hot path.

    packed[F, U, 3] = (time, 2dmu, 2dmv)  ->  entropy[F], hist0[F, T0], assign0[F, U]

PyTorch is used for device memory and streams only; all compute happens in
libvet_b200.so through the C ABI (include/vet_b200.h).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _native as N
from . import _tables
from .config import EntropyConfig
from .data_types import SpatialError, ValidationError


class UnsupportedConfigurationError(SpatialError):
    """The configuration is valid for the reference but outside what the device
    tables of this build can hold."""


@dataclass
class SpatialResult:
    """Outputs of SpatialEntropyAnalyzer.compute_entropy (SA:107-164) as tensors."""
    entropy: torch.Tensor            # [F] float64, mean over tile counts
    per_k: Optional[torch.Tensor]    # [K, F] float64
    hist0: Optional[torch.Tensor]    # [F, T0] float64 tile weights of tile_counts[0]
    assign0: Optional[torch.Tensor]  # [F, U] uint16 nearest tile of tile_counts[0] (0xFFFF = missing)


@dataclass
class TransitionResult:
    """Outputs of TransitionEntropyAnalyzer.compute_entropy (TA:107-175) as tensors."""
    entropy: torch.Tensor                # [F-1] float64
    per_k: Optional[torch.Tensor]        # [K, F-1]
    prev_count0: Optional[torch.Tensor]  # [F-1, T0] int32
    pairs0: Optional[torch.Tensor]       # [F-1, U, 2] uint16


@dataclass
class UserResult:
    """Per-viewer exploration entropy: compute_spatial_entropy (EU:147-211) over one user's frames (vet_users_*)."""
    entropy: torch.Tensor            # [U] float64, mean over tile counts; NaN for a user without any sample
    per_k: Optional[torch.Tensor]    # [K, U] float64
    hist0: Optional[torch.Tensor]    # [U, T0] float64 tile weights of tile_counts[0] summed over the user's frames
    frames: torch.Tensor             # [U] int32 frames in which the user's sample is present


@dataclass
class TransitionCountsResult:
    """Tile transition matrix of a video (vet_transition_counts_*): counts[k][p, c] = (frame pair, user) combinations
    moving from tile p to tile c of tile count k, and their pooled conditional entropy."""
    counts: List[torch.Tensor]       # per tile count a [T_k, T_k] int64 view of the accumulator (row = previous tile)
    entropy: torch.Tensor            # 0-d float64, mean over tile counts; NaN without any pair
    per_k: torch.Tensor              # [K] float64
    pairs: int                       # N: (frame pair, user) combinations with the user present in both frames


@dataclass
class UserTransitionResult:
    """Per-viewer transition entropy (vet_user_transitions): the textbook conditional entropy (EU:321-327) of every
    user's own (current tile, next tile) pairs over the frames, averaged over the tile counts."""
    entropy: torch.Tensor            # [U] float64, mean over tile counts; NaN for a user without any pair
    per_k: Optional[torch.Tensor]    # [K, U] float64
    pairs: torch.Tensor              # [U] int32 N_u: frames f with the user present in f and f+1


def _check(rc: int) -> None:
    if rc == N.VET_OK:
        return
    msg = N.last_error()
    if rc == N.VET_ERR_INVALID_ARG:
        raise ValidationError(msg)
    if rc == N.VET_ERR_UNSUPPORTED:
        raise UnsupportedConfigurationError(msg)
    if rc == N.VET_ERR_NOMEM:
        raise MemoryError(msg)
    raise RuntimeError(msg)


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _mode(mode: str) -> int:
    """VET_TRANSITION_* code of a transition mode name."""
    if mode not in ("literal", "textbook"):
        raise ValueError("mode must be 'literal' or 'textbook'")
    return N.VET_TRANSITION_LITERAL if mode == "literal" else N.VET_TRANSITION_TEXTBOOK


class Engine:
    """One native handle.  Not thread-safe per instance; use one per thread/stream."""

    def __init__(self, video_width: int, video_height: int, tile_counts: Sequence[int],
                 entropy_config: Optional[EntropyConfig] = None, device: Optional[torch.device] = None,
                 native_tables: bool = False, centres: Optional[Sequence[np.ndarray]] = None,
                 naive_tiles: Optional[Tuple[int, int]] = None, regime: str = "auto"):
        """native_tables=True lets the library derive the lattice and axis tables itself
        (libm) instead of receiving the numpy-made ones; used by tests to show both agree.
        centres: optional list of [T_k,3] arrays of ARBITRARY tile centres (the reference's
        free functions take any List[Vector]); tile_counts is then only a label.
        naive_tiles=(tile_width, tile_height) in degrees selects the latitude/longitude grid tiling
        of NaiveSpatialEntropyAnalyzer (NA:39-241) instead of the lattice: one tile set whose tile
        ids are grid codes lon_idx * (180/tile_height + 1) + lat_idx; tile_counts is ignored.
        regime="direct" pins the per-sample evaluation without cell tables (vet_config.regime)."""
        self._h = None
        if regime not in ("auto", "direct"):
            raise ValueError("regime must be 'auto' or 'direct'")
        lib = N.load_library()
        if not torch.cuda.is_available():
            raise RuntimeError("viewport_entropy_toolkit_b200 needs a CUDA device; there is no CPU path")
        ec = entropy_config or EntropyConfig()
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("viewport_entropy_toolkit_b200 needs a CUDA device; there is no CPU path")
        self.device = torch.device("cuda", dev.index if dev.index is not None else torch.cuda.current_device())
        self.video_width, self.video_height = int(video_width), int(video_height)
        self.naive_tiles = None if naive_tiles is None else (int(naive_tiles[0]), int(naive_tiles[1]))
        self.tile_counts = [int(c) for c in tile_counts] if naive_tiles is None else [1]
        self.entropy_config = ec
        # DU:236-240 (the reference validates dims when the first sample is converted)
        if self.video_width <= 0 or self.video_height <= 0:
            raise ValidationError("Video dimensions must be positive")
        if self.video_width % 2 or self.video_height % 2:
            raise ValidationError("Video dimensions must be even numbers")
        if not self.tile_counts or any(c <= 0 for c in self.tile_counts):
            raise ValidationError("Tile counts must be positive")
        K = len(self.tile_counts)
        if centres is not None:
            if len(centres) != K or any(len(c) == 0 for c in centres):
                raise ValidationError("No tile centers provided")  # EU:170-171
            self._centres = [np.ascontiguousarray(np.asarray(c, dtype=np.float64).reshape(-1, 3)) for c in centres]
        else:
            self._centres = [np.ascontiguousarray(_tables.fibonacci_lattice(c)) for c in self.tile_counts]
        ntiles = (C.c_int32 * K)(*[len(c) for c in self._centres]) if centres is not None else None
        lon, lat = _tables.axis_tables(self.video_width, self.video_height)
        tc = (C.c_int32 * K)(*self.tile_counts)
        cptrs = (C.POINTER(C.c_double) * K)(*[c.ctypes.data_as(C.POINTER(C.c_double)) for c in self._centres])
        cfg = N.VetConfig(
            device=self.device.index, video_width=self.video_width, video_height=self.video_height,
            num_tile_counts=K, tile_counts=tc, fov_angle=float(ec.fov_angle), power_factor=float(ec.power_factor),
            use_weight_distribution=int(bool(ec.use_weight_distribution)),
            centres=None if native_tables else cptrs,
            lon_by_px=None if native_tables else lon.ctypes.data_as(C.POINTER(C.c_double)),
            lat_by_py=None if native_tables else lat.ctypes.data_as(C.POINTER(C.c_double)),
            num_tiles=ntiles,
            naive_tile_width=self.naive_tiles[0] if self.naive_tiles else 0,
            naive_tile_height=self.naive_tiles[1] if self.naive_tiles else 0,
            regime=N.VET_REGIME_DIRECT if regime == "direct" else N.VET_REGIME_AUTO)
        h = C.c_void_p()
        _check(lib.vet_create(C.byref(h), C.byref(cfg)))
        self._h = h
        self._lib = lib
        self.num_tiles = [lib.vet_num_tiles(h, k) for k in range(K)]
        self.num_cells = int(lib.vet_num_cells(h))
        self._host_out: Dict[tuple, tuple] = {}

    # -- lifetime ---------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.vet_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- helpers ------------------------------------------------------------------
    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _packed(self, packed: torch.Tensor) -> Tuple[torch.Tensor, int]:
        if not isinstance(packed, torch.Tensor):
            raise TypeError("packed must be a torch.Tensor on the engine's device")
        if packed.device != self.device:
            raise ValueError(f"packed is on {packed.device}, engine on {self.device}")
        if packed.dtype not in (torch.float32, torch.float64):
            raise TypeError("packed must be float32 or float64")
        if packed.shape[-1] != 3:
            raise ValueError("packed must have shape [..., 3] = (time, 2dmu, 2dmv)")
        return packed.contiguous(), (N.VET_F32 if packed.dtype == torch.float32 else N.VET_F64)

    def _frames(self, packed: torch.Tensor) -> Tuple[torch.Tensor, int, int, int]:
        """_packed for the [F, U, 3] inputs of the frame-level calls -> (packed, dtype code, F, U)."""
        p, dt = self._packed(packed)
        if p.dim() != 3:
            raise ValueError("packed must be [F, U, 3]")
        return p, dt, int(p.shape[0]), int(p.shape[1])

    def _spatial_result(self, F: int, U: int, want_per_k: bool, want_hist0: bool, want_assign0: bool) -> SpatialResult:
        K, T0, dev = len(self.tile_counts), self.num_tiles[0], self.device
        return SpatialResult(
            entropy=torch.empty(F, dtype=torch.float64, device=dev),
            per_k=torch.empty((K, F), dtype=torch.float64, device=dev) if want_per_k else None,
            hist0=torch.empty((F, T0), dtype=torch.float64, device=dev) if want_hist0 else None,
            assign0=torch.empty((F, U), dtype=torch.uint16, device=dev) if want_assign0 else None)

    def _transition_result(self, F: int, U: int, want_per_k: bool, want_prev_count0: bool,
                           want_pairs0: bool) -> TransitionResult:
        R = max(F - 1, 0)
        K, T0, dev = len(self.tile_counts), self.num_tiles[0], self.device
        return TransitionResult(
            entropy=torch.empty(R, dtype=torch.float64, device=dev),
            per_k=torch.empty((K, R), dtype=torch.float64, device=dev) if want_per_k else None,
            prev_count0=torch.empty((R, T0), dtype=torch.int32, device=dev) if want_prev_count0 else None,
            pairs0=torch.empty((R, U, 2), dtype=torch.uint16, device=dev) if want_pairs0 else None)

    def set_option(self, name: str, value) -> None:
        """vet_set_option: pins a kernel choice of this handle, e.g. set_option("weighted_kernel", "i8")
        (names and values: _native.OPTIONS).  Production leaves the defaults."""
        opt, values = N.OPTIONS[name]
        _check(self._lib.vet_set_option(self._h, opt, values[value] if isinstance(value, str) else int(value)))

    def get_option(self, name: str) -> str:
        opt, values = N.OPTIONS[name]
        v = C.c_int(0)
        _check(self._lib.vet_get_option(self._h, opt, C.byref(v)))
        return next((k for k, x in values.items() if x == v.value), v.value)

    def launch_count(self) -> int:
        return int(self._lib.vet_launch_count(self._h))

    def graph_replays(self) -> int:
        """API calls that ran as one CUDA graph launch (third identical call on, on a capturable stream)."""
        return int(self._lib.vet_graph_replays(self._h))

    def profile(self, on: bool = True) -> None:
        """Starts (or stops) recording a CUDA-event pair around every kernel launch."""
        _check(self._lib.vet_profile_enable(self._h, int(on)))

    def profile_read(self) -> Dict[str, Tuple[float, int]]:
        """{kernel: (summed device milliseconds, launches)} since profile(True)."""
        ms = (C.c_double * len(N.KERNEL_NAMES))()
        cnt = (C.c_int64 * len(N.KERNEL_NAMES))()
        _check(self._lib.vet_profile_read(self._h, ms, cnt))
        return {name: (float(ms[i]), int(cnt[i])) for i, name in enumerate(N.KERNEL_NAMES)}

    def poll_flags(self) -> int:
        """Synchronises the current stream and returns (and clears) the sticky
        device flag word."""
        flags = C.c_uint32(0)
        _check(self._lib.vet_poll_flags(self._h, self._stream(), C.byref(flags)))
        return int(flags.value)

    def raise_for_flags(self) -> None:
        """Raises what the reference would have raised for the data it was given."""
        flags = self.poll_flags()
        if flags & N.VET_FLAG_OUT_OF_RANGE:
            raise ValidationError("Normalized coordinates must be between 0 and 1")  # DU:256-257
        if flags & N.VET_FLAG_EMPTY_FRAME:
            raise ValidationError("Empty vector dictionary")  # EU:168-169
        if flags & N.VET_FLAG_NO_COMMON_USER:
            raise ZeroDivisionError("division by zero")  # EU:326

    # -- tables -------------------------------------------------------------------
    def lattice(self, k: int = 0) -> np.ndarray:
        """generate_fibonacci_lattice(tile_counts[k]) as [T,3] float64 (DU:25-56)."""
        out = np.empty((self.num_tiles[k], 3), dtype=np.float64)
        _check(self._lib.vet_lattice(self._h, k, out.ctypes.data))
        return out

    def cell_lut(self, k: int = 0) -> np.ndarray:
        """Nearest tile of every reachable cell, [(H+1), (W+1)] uint16."""
        out = np.empty(self.num_cells, dtype=np.uint16)
        _check(self._lib.vet_cell_lut(self._h, k, out.ctypes.data))
        return out.reshape(self.video_height + 1, self.video_width + 1)

    # -- stage 1 / 2 ------------------------------------------------------------------
    def decode(self, packed: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """packed[..., 3] -> (vectors[..., 3] float64, cell[...] int32).  Missing or
        out-of-range samples give NaN vectors and cell -1."""
        p, dt = self._packed(packed)
        n = p.numel() // 3
        vec = torch.empty(p.shape, dtype=torch.float64, device=self.device)
        cell = torch.empty(p.shape[:-1], dtype=torch.int32, device=self.device)
        _check(self._lib.vet_decode(self._h, p.data_ptr(), dt, n, vec.data_ptr(), cell.data_ptr(), self._stream()))
        return vec, cell

    def nearest_tile(self, vectors: torch.Tensor, k: int = 0) -> torch.Tensor:
        """find_nearest_tile (EU:89-106) for vectors[..., 3] float64 -> int32[...]."""
        v = vectors.to(device=self.device, dtype=torch.float64).contiguous()
        n = v.numel() // 3
        idx = torch.empty(v.shape[:-1], dtype=torch.int32, device=self.device)
        _check(self._lib.vet_nearest_tile(self._h, k, v.data_ptr(), n, idx.data_ptr(), self._stream()))
        return idx

    def tile_weights(self, vectors: torch.Tensor, k: int = 0) -> torch.Tensor:
        """calculate_tile_weights (EU:108-144) as dense rows [..., T_k] float64."""
        v = vectors.to(device=self.device, dtype=torch.float64).contiguous()
        n = v.numel() // 3
        w = torch.empty(v.shape[:-1] + (self.num_tiles[k],), dtype=torch.float64, device=self.device)
        _check(self._lib.vet_tile_weights(self._h, k, v.data_ptr(), n, w.data_ptr(), self._stream()))
        return w

    def angular_distances(self, vectors: torch.Tensor, k: int = 0) -> torch.Tensor:
        """find_angular_distances (EU:70-87) as [..., T_k] float64 radians."""
        v = vectors.to(device=self.device, dtype=torch.float64).contiguous()
        n = v.numel() // 3
        d = torch.empty(v.shape[:-1] + (self.num_tiles[k],), dtype=torch.float64, device=self.device)
        _check(self._lib.vet_angular_distances(self._h, k, v.data_ptr(), n, d.data_ptr(), self._stream()))
        return d

    def vector_angles(self, a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
        """vector_angle_distance (EU:41-67) for pairs a[..., 3], b[..., 3] -> float64[...] radians."""
        a = a.to(device=self.device, dtype=torch.float64).contiguous()
        b = b.to(device=self.device, dtype=torch.float64).contiguous()
        if a.shape != b.shape or a.shape[-1] != 3:
            raise ValueError("a and b must both be [..., 3]")
        d = torch.empty(a.shape[:-1], dtype=torch.float64, device=self.device)
        _check(self._lib.vet_vector_angles(self._h, a.data_ptr(), b.data_ptr(), a.numel() // 3, d.data_ptr(), self._stream()))
        return d

    def spatial_vectors(self, vectors: torch.Tensor, want_per_k: bool = True, want_hist0: bool = True,
                        want_assign0: bool = True) -> SpatialResult:
        """compute_spatial_entropy (EU:147-211) on vectors[F,U,3] float64 (NaN = absent user)."""
        v = vectors.to(device=self.device, dtype=torch.float64).contiguous()
        if v.dim() != 3 or v.shape[-1] != 3:
            raise ValueError("vectors must be [F, U, 3]")
        F, U = int(v.shape[0]), int(v.shape[1])
        out = self._spatial_result(F, U, want_per_k, want_hist0, want_assign0)
        _check(self._lib.vet_spatial_vectors(self._h, v.data_ptr(), F, U, out.entropy.data_ptr(), _ptr(out.per_k),
                                             _ptr(out.hist0), _ptr(out.assign0), self._stream()))
        return out

    def transition_vectors(self, vectors: torch.Tensor, mode: str = "literal", want_per_k: bool = True,
                           want_prev_count0: bool = True, want_pairs0: bool = True) -> TransitionResult:
        """compute_transition_entropy (EU:213-332) on vectors[F,U,3]; row r pairs frames (r, r+1)."""
        v = vectors.to(device=self.device, dtype=torch.float64).contiguous()
        if v.dim() != 3 or v.shape[-1] != 3:
            raise ValueError("vectors must be [F, U, 3]")
        m = _mode(mode)
        F, U = int(v.shape[0]), int(v.shape[1])
        out = self._transition_result(F, U, want_per_k, want_prev_count0, want_pairs0)
        _check(self._lib.vet_transition_vectors(self._h, v.data_ptr(), F, U, out.entropy.data_ptr(), _ptr(out.per_k),
                                                _ptr(out.prev_count0), _ptr(out.pairs0), m, self._stream()))
        return out

    def naive_points(self, lonlat: torch.Tensor, tile_width: int, tile_height: int, use_weight_distribution: bool,
                     want_indices: bool = True):
        """compute_naive_spatial_entropy (EU:362-453) on lonlat[F,U,2] float64 degrees (NaN = absent):
        -> (entropy[F], lon_idx[F,U] int32, lat_idx[F,U] int32); the reference's tile key of a point is
        f"{lon_idx}_{lat_idx}" (EU:381)."""
        v = lonlat.to(device=self.device, dtype=torch.float64).contiguous()
        if v.dim() != 3 or v.shape[-1] != 2:
            raise ValueError("lonlat must be [F, U, 2]")
        F, U = int(v.shape[0]), int(v.shape[1])
        ent = torch.empty(F, dtype=torch.float64, device=self.device)
        li = torch.empty((F, U), dtype=torch.int32, device=self.device) if want_indices else None
        la = torch.empty((F, U), dtype=torch.int32, device=self.device) if want_indices else None
        _check(self._lib.vet_naive_points(self._h, v.data_ptr(), F, U, int(tile_width), int(tile_height),
                                          int(bool(use_weight_distribution)), ent.data_ptr(), _ptr(li), _ptr(la),
                                          self._stream()))
        return ent, li, la

    # -- stages 1-3 fused -----------------------------------------------------------
    def spatial(self, packed: torch.Tensor, want_per_k: bool = True, want_hist0: bool = True,
                want_assign0: bool = True, out: Optional[SpatialResult] = None) -> SpatialResult:
        p, dt, F, U = self._frames(packed)
        if out is None:
            out = self._spatial_result(F, U, want_per_k, want_hist0, want_assign0)
        _check(self._lib.vet_spatial(self._h, p.data_ptr(), dt, F, U, out.entropy.data_ptr(), _ptr(out.per_k),
                                     _ptr(out.hist0), _ptr(out.assign0), self._stream()))
        return out

    # -- stage 4 ---------------------------------------------------------------------
    def transition(self, packed: torch.Tensor, mode: str = "literal", want_per_k: bool = True,
                   want_prev_count0: bool = True, want_pairs0: bool = True,
                   out: Optional[TransitionResult] = None) -> TransitionResult:
        p, dt, F, U = self._frames(packed)
        m = _mode(mode)
        if out is None:
            out = self._transition_result(F, U, want_per_k, want_prev_count0, want_pairs0)
        _check(self._lib.vet_transition(self._h, p.data_ptr(), dt, F, U, out.entropy.data_ptr(), _ptr(out.per_k),
                                        _ptr(out.prev_count0), _ptr(out.pairs0), m, self._stream()))
        return out

    # -- both analyzers in one pass ----------------------------------------------------------
    def analyze(self, packed: torch.Tensor, mode: str = "literal", want_per_k: bool = True, want_hist0: bool = True,
                want_assign0: bool = True, want_prev_count0: bool = True,
                want_pairs0: bool = True) -> Tuple[SpatialResult, TransitionResult]:
        """SpatialEntropyAnalyzer.compute_entropy and TransitionEntropyAnalyzer.compute_entropy on
        the same packed tensor with a single read of the input (vet_analyze)."""
        p, dt, F, U = self._frames(packed)
        m = _mode(mode)
        sp = self._spatial_result(F, U, want_per_k, want_hist0, want_assign0)
        tr = self._transition_result(F, U, want_per_k, want_prev_count0, want_pairs0)
        _check(self._lib.vet_analyze(self._h, p.data_ptr(), dt, F, U, sp.entropy.data_ptr(), _ptr(sp.per_k), _ptr(sp.hist0),
                                     _ptr(sp.assign0), tr.entropy.data_ptr(), _ptr(tr.per_k), _ptr(tr.prev_count0),
                                     _ptr(tr.pairs0), m, self._stream()))
        return sp, tr

    # -- per-viewer exploration entropy ------------------------------------------------------
    def user_accumulator(self, U: int) -> torch.Tensor:
        """Zeroed int64 accumulator [U, sum(T_k) + 1] of users_accumulate (tile counts concatenated in k order, the last
        column counts present samples)."""
        return torch.zeros((int(U), sum(self.num_tiles) + 1), dtype=torch.int64, device=self.device)

    def _check_acc(self, acc: torch.Tensor, U: Optional[int] = None) -> int:
        if not isinstance(acc, torch.Tensor) or acc.device != self.device or acc.dtype != torch.int64:
            raise TypeError("acc must be an int64 tensor on the engine's device (Engine.user_accumulator)")
        if acc.dim() != 2 or acc.shape[1] != sum(self.num_tiles) + 1 or not acc.is_contiguous():
            raise ValueError(f"acc must be a contiguous [U, {sum(self.num_tiles) + 1}] tensor")
        if U is not None and acc.shape[0] != U:
            raise ValueError(f"acc has {acc.shape[0]} user rows, packed has {U} users")
        return int(acc.shape[0])

    def users_accumulate(self, packed: torch.Tensor, acc: torch.Tensor, total_frames: int) -> None:
        """Adds the frames of packed[F,U,3] into acc (vet_users_accumulate).  total_frames is the frame count of the
        whole video: every batch (and every rank) of one video must pass the same value, which fixes the fixed-point
        scale of the weights -- then any batching or frame order gives the same bits."""
        p, dt, F, U = self._frames(packed)
        self._check_acc(acc, U)
        if int(total_frames) < max(F, 1):
            raise ValueError(f"total_frames ({total_frames}) must be >= 1 and >= the frames of packed ({F})")
        _check(self._lib.vet_users_accumulate(self._h, p.data_ptr(), dt, F, U, int(total_frames), acc.data_ptr(),
                                              self._stream()))

    def users_finish(self, acc: torch.Tensor, total_frames: int, want_per_k: bool = True,
                     want_hist0: bool = True) -> UserResult:
        """Entropies of finished accumulator rows (vet_users_finish); total_frames as in users_accumulate."""
        U = self._check_acc(acc)
        if int(total_frames) < 1:
            raise ValueError("total_frames must be >= 1")
        K, T0, dev = len(self.tile_counts), self.num_tiles[0], self.device
        out = UserResult(
            entropy=torch.empty(U, dtype=torch.float64, device=dev),
            per_k=torch.empty((K, U), dtype=torch.float64, device=dev) if want_per_k else None,
            hist0=torch.empty((U, T0), dtype=torch.float64, device=dev) if want_hist0 else None,
            frames=acc[:, -1].to(torch.int32))
        _check(self._lib.vet_users_finish(self._h, acc.data_ptr(), U, int(total_frames), out.entropy.data_ptr(),
                                          _ptr(out.per_k), _ptr(out.hist0), self._stream()))
        return out

    def users(self, packed: torch.Tensor, want_per_k: bool = True, want_hist0: bool = True) -> UserResult:
        """Per-viewer exploration entropy of packed[F,U,3]: compute_spatial_entropy (EU:147-211) of every user's
        present samples over the frames, averaged over the tile counts (SA:142-156).  A user without any sample
        gets NaN and a zero histogram row.  Call raise_for_flags() to raise for out-of-range coordinates."""
        p, _, F, U = self._frames(packed)
        acc = self.user_accumulator(U)
        self.users_accumulate(p, acc, max(F, 1))
        return self.users_finish(acc, max(F, 1), want_per_k, want_hist0)

    # -- tile transition matrix ----------------------------------------------------------------
    def transition_counts_accumulator(self) -> torch.Tensor:
        """Zeroed int64 accumulator of transition_counts_accumulate: the [T_k, T_k] matrices of all tile counts,
        flattened and concatenated in k order."""
        return torch.zeros(sum(t * t for t in self.num_tiles), dtype=torch.int64, device=self.device)

    def _check_tc_acc(self, acc: torch.Tensor) -> None:
        n = sum(t * t for t in self.num_tiles)
        if not isinstance(acc, torch.Tensor) or acc.device != self.device or acc.dtype != torch.int64:
            raise TypeError("acc must be an int64 tensor on the engine's device (Engine.transition_counts_accumulator)")
        if acc.dim() != 1 or acc.shape[0] != n or not acc.is_contiguous():
            raise ValueError(f"acc must be a contiguous [{n}] tensor")

    def transition_counts_accumulate(self, packed: torch.Tensor, acc: torch.Tensor) -> None:
        """Adds the (f, f+1) frame pairs of packed[F,U,3] into acc (vet_transition_counts_accumulate).  Batches that
        overlap by one frame add up to the whole video, in any batching and order, with the same bits."""
        p, dt, F, U = self._frames(packed)
        self._check_tc_acc(acc)
        _check(self._lib.vet_transition_counts_accumulate(self._h, p.data_ptr(), dt, F, U, acc.data_ptr(), self._stream()))

    def transition_counts_finish(self, acc: torch.Tensor) -> TransitionCountsResult:
        """Pooled conditional entropy of the finished counts (vet_transition_counts_finish); `counts` are views of acc.
        Synchronises the current stream to read the pair count."""
        self._check_tc_acc(acc)
        K, dev = len(self.tile_counts), self.device
        entropy = torch.empty((), dtype=torch.float64, device=dev)
        per_k = torch.empty(K, dtype=torch.float64, device=dev)
        pairs = torch.empty(1, dtype=torch.int64, device=dev)
        _check(self._lib.vet_transition_counts_finish(self._h, acc.data_ptr(), entropy.data_ptr(), per_k.data_ptr(),
                                                      pairs.data_ptr(), self._stream()))
        counts, off = [], 0
        for t in self.num_tiles:
            counts.append(acc[off:off + t * t].view(t, t))
            off += t * t
        return TransitionCountsResult(counts=counts, entropy=entropy, per_k=per_k, pairs=int(pairs.item()))

    def transition_counts(self, packed: torch.Tensor) -> TransitionCountsResult:
        """Tile transition matrix of packed[F,U,3]: per tile count the users moving from tile p in frame f to tile c in
        frame f+1, summed over all frame pairs, and the pooled conditional entropy -sum (n_pc/N) log2(n_pc/n_p)
        normalised like the textbook mode.  Call raise_for_flags() to raise for out-of-range coordinates."""
        acc = self.transition_counts_accumulator()
        self.transition_counts_accumulate(packed, acc)
        return self.transition_counts_finish(acc)

    # -- per-viewer transition entropy ---------------------------------------------------------
    def user_transitions(self, packed: torch.Tensor, want_per_k: bool = True) -> UserTransitionResult:
        """Per-viewer transition entropy of packed[F,U,3] (vet_user_transitions): per user and tile count the
        conditional entropy -sum (n_pc/N_u) log2(n_pc/n_p) of the user's moves from tile p in frame f to tile c in frame
        f+1, normalised like the textbook mode, and its mean over the tile counts.  One call sees every frame of its
        users; a user's outputs do not depend on the other users of the call, so user blocks (columns of the video)
        can be computed separately.  A user without any pair gets NaN.  Call raise_for_flags() to raise for
        out-of-range coordinates."""
        p, dt, F, U = self._frames(packed)
        K, dev = len(self.tile_counts), self.device
        out = UserTransitionResult(
            entropy=torch.empty(U, dtype=torch.float64, device=dev),
            per_k=torch.empty((K, U), dtype=torch.float64, device=dev) if want_per_k else None,
            pairs=torch.empty(U, dtype=torch.int32, device=dev))
        _check(self._lib.vet_user_transitions(self._h, p.data_ptr(), dt, F, U, out.entropy.data_ptr(), _ptr(out.per_k),
                                              out.pairs.data_ptr(), self._stream()))
        return out

    # -- host-buffer (numpy) variants -----------------------------------------------------
    def spatial_host(self, packed: np.ndarray, want_per_k: bool = True, want_hist0: bool = True,
                     want_assign0: bool = True, reuse_buffers: bool = False) -> Dict[str, Optional[np.ndarray]]:
        """numpy (or pinned torch CPU tensor) in, numpy out; the H2D/D2H copies are
        pipelined inside the library (vet_spatial_host).  Results land in page-locked
        memory so that the device-to-host copies run at PCIe speed; with
        reuse_buffers=True the same engine-owned arrays are returned by every call of
        the same shape (page-locking 0.7 GB costs more than copying it)."""
        arr, dt, F, U = _host_packed(packed)
        self._host_layout(arr)
        K, T0 = len(self.tile_counts), self.num_tiles[0]
        ent, per_k, hist0, assign0 = self._host_buffers(
            ("sp", F, U, want_per_k, want_hist0, want_assign0),
            lambda: (_pinned((F,), np.float64), _pinned((K, F), np.float64) if want_per_k else None,
                     _pinned((F, T0), np.float64) if want_hist0 else None,
                     _pinned((F, U), np.uint16) if want_assign0 else None), reuse_buffers)
        _check(self._lib.vet_spatial_host(self._h, _host_ptr(arr), dt, F, U, ent.ctypes.data, _np_ptr(per_k),
                                          _np_ptr(hist0), _np_ptr(assign0)))
        return dict(entropy=ent, per_k=per_k, hist0=hist0, assign0=assign0)

    def _host_layout(self, arr) -> None:
        """[F,U,2] host arrays hold (2dmu, 2dmv) only: a third less to upload (the kernels never read the time column;
        VET_OPT_HOST_LAYOUT).  The frame times stay with the caller."""
        want = "uv" if int(arr.shape[-1]) == 2 else "tuv"
        if self.get_option("host_layout") != want:
            self.set_option("host_layout", want)

    def _host_buffers(self, key: tuple, make, reuse: bool) -> tuple:
        bufs = self._host_out.get(key) if reuse else None
        if bufs is None:
            bufs = make()
            if reuse:
                self._host_out = {key: bufs}
        return bufs

    def transition_host(self, packed: np.ndarray, mode: str = "literal", want_per_k: bool = True,
                        want_prev_count0: bool = True, want_pairs0: bool = True,
                        reuse_buffers: bool = False) -> Dict[str, Optional[np.ndarray]]:
        """TransitionEntropyAnalyzer.compute_entropy on host memory (vet_transition_host): frame batches with a
        one-frame halo, upload | kernels | download on three streams; results in page-locked memory."""
        arr, dt, F, U = _host_packed(packed)
        self._host_layout(arr)
        m = _mode(mode)
        R = max(F - 1, 0)
        K, T0 = len(self.tile_counts), self.num_tiles[0]
        ent, per_k, pc, pairs = self._host_buffers(
            ("tr", F, U, want_per_k, want_prev_count0, want_pairs0),
            lambda: (_pinned((R,), np.float64), _pinned((K, R), np.float64) if want_per_k else None,
                     _pinned((R, T0), np.int32) if want_prev_count0 else None,
                     _pinned((R, U, 2), np.uint16) if want_pairs0 else None), reuse_buffers)
        _check(self._lib.vet_transition_host(self._h, _host_ptr(arr), dt, F, U, ent.ctypes.data, _np_ptr(per_k),
                                             _np_ptr(pc), _np_ptr(pairs), m))
        return dict(entropy=ent, per_k=per_k, prev_count0=pc, pairs0=pairs)

    def analyze_host(self, packed: np.ndarray, mode: str = "literal", want_per_k: bool = True, want_hist0: bool = True,
                     want_assign0: bool = True, want_prev_count0: bool = True, want_pairs0: bool = True,
                     reuse_buffers: bool = False) -> Tuple[Dict[str, Optional[np.ndarray]], Dict[str, Optional[np.ndarray]]]:
        """Both analyzers on host memory with ONE upload of the input (vet_analyze_host) -> (spatial, transition)
        dicts of numpy arrays like spatial_host / transition_host."""
        arr, dt, F, U = _host_packed(packed)
        self._host_layout(arr)
        m = _mode(mode)
        R = max(F - 1, 0)
        K, T0 = len(self.tile_counts), self.num_tiles[0]
        bufs = self._host_buffers(
            ("an", F, U, want_per_k, want_hist0, want_assign0, want_prev_count0, want_pairs0),
            lambda: (_pinned((F,), np.float64), _pinned((K, F), np.float64) if want_per_k else None,
                     _pinned((F, T0), np.float64) if want_hist0 else None,
                     _pinned((F, U), np.uint16) if want_assign0 else None,
                     _pinned((R,), np.float64), _pinned((K, R), np.float64) if want_per_k else None,
                     _pinned((R, T0), np.int32) if want_prev_count0 else None,
                     _pinned((R, U, 2), np.uint16) if want_pairs0 else None), reuse_buffers)
        ent, per_k, hist0, assign0, tent, tper_k, pc, pairs = bufs
        _check(self._lib.vet_analyze_host(self._h, _host_ptr(arr), dt, F, U, ent.ctypes.data, _np_ptr(per_k), _np_ptr(hist0),
                                          _np_ptr(assign0), tent.ctypes.data, _np_ptr(tper_k), _np_ptr(pc), _np_ptr(pairs), m))
        return (dict(entropy=ent, per_k=per_k, hist0=hist0, assign0=assign0),
                dict(entropy=tent, per_k=tper_k, prev_count0=pc, pairs0=pairs))


_TORCH_OF = {np.float64: torch.float64, np.uint16: torch.uint16, np.int32: torch.int32}


def _pinned(shape, dtype) -> np.ndarray:
    """numpy view of a page-locked torch buffer (the tensor stays alive through .base)."""
    return torch.empty(shape, dtype=_TORCH_OF[dtype], pin_memory=True).numpy()


def _np_ptr(a: Optional[np.ndarray]) -> Optional[int]:
    return None if a is None else a.ctypes.data


def _host_packed(packed):
    if isinstance(packed, torch.Tensor):
        if packed.device.type != "cpu":
            raise ValueError("spatial_host/transition_host take host memory; use spatial()/transition() for device tensors")
        arr = packed.contiguous()
        dtype = {torch.float32: N.VET_F32, torch.float64: N.VET_F64}.get(arr.dtype)
    else:
        arr = np.ascontiguousarray(packed)
        dtype = {np.dtype(np.float32): N.VET_F32, np.dtype(np.float64): N.VET_F64}.get(arr.dtype)
    if dtype is None:
        raise TypeError("packed must be float32 or float64")
    if arr.ndim != 3 or arr.shape[-1] not in (2, 3):
        raise ValueError("packed must be [F, U, 3] = (time, 2dmu, 2dmv) or [F, U, 2] = (2dmu, 2dmv)")
    return arr, dtype, int(arr.shape[0]), int(arr.shape[1])


def _host_ptr(arr) -> int:
    return arr.data_ptr() if isinstance(arr, torch.Tensor) else arr.ctypes.data


_ENGINES: Dict[tuple, Engine] = {}        # lattice / grid configurations (analyzers, bench): kept until clear_engines()
_ADHOC_ENGINES: Dict[tuple, Engine] = {}  # arbitrary centre lists of the functional API: small LRU
_ADHOC_LIMIT = 16


def get_engine(video_width: int, video_height: int, tile_counts: Sequence[int],
               entropy_config: Optional[EntropyConfig] = None, device: Optional[torch.device] = None,
               centres: Optional[Sequence[np.ndarray]] = None,
               naive_tiles: Optional[Tuple[int, int]] = None) -> Engine:
    """Engine cache keyed by (device, configuration): building the tables costs a
    few milliseconds, analyzers and the functional API share them."""
    ec = entropy_config or EntropyConfig()
    if not torch.cuda.is_available():
        raise RuntimeError("viewport_entropy_toolkit_b200 needs a CUDA device; there is no CPU path")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    ckey = None if centres is None else tuple(np.ascontiguousarray(c, dtype=np.float64).tobytes() for c in centres)
    key = (idx, int(video_width), int(video_height), tuple(int(c) for c in tile_counts), float(ec.fov_angle),
           bool(ec.use_weight_distribution), float(ec.power_factor), ckey,
           None if naive_tiles is None else (int(naive_tiles[0]), int(naive_tiles[1])))
    cache = _ENGINES if centres is None else _ADHOC_ENGINES
    eng = cache.get(key)
    if eng is None:
        # An evicted engine is only dropped from the cache, never closed: whoever still holds it keeps a live
        # handle, and Engine.__del__ frees it with the last reference.
        while cache is _ADHOC_ENGINES and len(cache) >= _ADHOC_LIMIT:
            cache.pop(next(iter(cache)))
        eng = Engine(video_width, video_height, tile_counts, ec, torch.device("cuda", idx), centres=centres,
                     naive_tiles=naive_tiles)
    elif cache is _ADHOC_ENGINES:
        cache.pop(key)  # re-inserted below: most recently used last
    cache[key] = eng
    return eng


def clear_engines() -> None:
    """Empties the caches.  Engines still referenced elsewhere stay usable; the others free their handle."""
    _ENGINES.clear()
    _ADHOC_ENGINES.clear()
