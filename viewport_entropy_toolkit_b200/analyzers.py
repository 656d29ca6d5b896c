"""Analyzer facades with the reference's class API, backed by the device engine.

SpatialEntropyAnalyzer      <-> analyzers/spatial_entropy.py       (SA:40-253)
TransitionEntropyAnalyzer   <-> analyzers/transition_entropy.py    (TA:40-264)
NaiveSpatialEntropyAnalyzer <-> analyzers/naive_spatial_entropy.py (NA:39-241)

`process_directory` / `compute_entropy` / `create_visualization` / `run_analysis`
keep their names, arguments, return types and error behaviour; the frame loops of
SA:129-161 and TA:129-172 run as CUDA kernels over the packed tensor.  The tensor
level entry points (`compute_entropy_packed`) are the ones to use at scale: they
return tensors instead of per-frame Python dicts.
"""
from __future__ import annotations

import logging
from collections.abc import Mapping
from datetime import datetime
from pathlib import Path
from typing import Dict, List, Optional, Sequence

import numpy as np
import pandas as pd
import torch

from . import _tables
from . import _native as N
from .config import AnalyzerConfig, NaiveAnalyzerConfig, DEFAULT_OUTPUT_FORMATS
from .data_types import ValidationError, Vector
from .engine import Engine, SpatialResult, TransitionResult, get_engine
from .ingest import load_directory

logger = logging.getLogger(__name__)


class LazyRowDict(Mapping):
    """Read-only dict view of one result row (`tile_weights` / `tile_assignments` of SA:152-163, TA:163-170): the
    dict the reference stores per frame is built from the row of the result array on first access, so a
    100k-user x 3600-frame video does not allocate 3.6e8 Python objects up front.  Compares equal to the dict it
    stands for; `create_visualization`-style consumers (`.items()`, `len`, `in`, iteration) work unchanged."""
    __slots__ = ("_make", "_d")

    def __init__(self, make):
        self._make = make
        self._d = None

    def _dict(self) -> dict:
        if self._d is None:
            self._d = self._make()
            self._make = None
        return self._d

    def __getitem__(self, key):
        return self._dict()[key]

    def __iter__(self):
        return iter(self._dict())

    def __len__(self):
        return len(self._dict())

    def __repr__(self):
        return repr(self._dict())


def _lattice_vectors(tile_count: int) -> List[Vector]:
    return [Vector(float(x), float(y), float(z)) for x, y, z in _tables.fibonacci_lattice(tile_count)]


class _AnalyzerBase:
    def __init__(self, config: Optional[AnalyzerConfig] = None, device: Optional[torch.device] = None):
        self.config = config or AnalyzerConfig()
        self._device = device
        self._data_cache: Dict = {}
        self._entropy_results: Optional[pd.DataFrame] = None
        self._fibonacci_vectors = {count: _lattice_vectors(count) for count in getattr(self.config, "tile_counts", [])}
        self._engine: Optional[Engine] = None

    @property
    def engine(self) -> Engine:
        if self._engine is None:
            c = self.config
            self._engine = get_engine(c.video_width, c.video_height, c.tile_counts, c.entropy_config, self._device)
        return self._engine

    def process_directory(self, directory: Path, order: Optional[Sequence[str]] = None) -> None:
        """Reads every *.csv of `directory` into the packed tensor.  `order`
        optionally pins the user order (file stems); the default is glob order."""
        directory = Path(directory)
        if not directory.exists():
            raise FileNotFoundError(f"Directory not found: {directory}")
        try:
            packed, times, identifiers = load_directory(directory, order)
            self._data_cache = {"packed": packed, "times": times, "identifiers": identifiers}
        except Exception as e:
            logger.error(f"Error processing directory {directory}: {str(e)}")
            raise ValidationError(f"Failed to process directory: {str(e)}")

    def load_packed(self, packed: np.ndarray, identifiers: Optional[Sequence[str]] = None) -> None:
        """Uses an in-memory packed[F,U,3] array instead of a directory."""
        packed = np.asarray(packed)
        if packed.ndim != 3 or packed.shape[-1] != 3:
            raise ValidationError("packed must be [F, U, 3]")
        ids = list(identifiers) if identifiers is not None else [f"user{u}" for u in range(packed.shape[1])]
        self._data_cache = {"packed": packed, "times": packed[:, 0, 0].astype(np.float64), "identifiers": ids}

    def _device_packed(self) -> torch.Tensor:
        if not self._data_cache:
            raise ValidationError("No data available. Call process_directory first.")
        return torch.from_numpy(np.ascontiguousarray(self._data_cache["packed"])).to(self.engine.device)

    def _host_packed(self) -> np.ndarray:
        if not self._data_cache:
            raise ValidationError("No data available. Call process_directory first.")
        return np.ascontiguousarray(self._data_cache["packed"])

    def _save_csv(self, base_name: str) -> Path:
        path = self.config.get_output_path(base_name, DEFAULT_OUTPUT_FORMATS["data"])
        self._entropy_results[["time", "entropy"]].to_csv(path, index=False)
        return path

    def create_visualization(self, base_name: str) -> None:
        """Writes the [time, entropy] CSV (SA:211-219).  The matplotlib graph and the
        ffmpeg animation of the reference are outside the accelerated path; the graph
        is drawn when matplotlib is importable and skipped (with a log line) otherwise."""
        if self._entropy_results is None:
            raise ValidationError("No entropy results. Call compute_entropy first.")
        try:
            self._save_csv(base_name)
            try:
                import matplotlib
                matplotlib.use("Agg")
                import matplotlib.pyplot as plt
            except Exception:
                logger.info("matplotlib not available: skipping the entropy graph")
                return
            vc = self.config.visualization_config
            fig, ax = plt.subplots(figsize=vc.figure_size)
            ax.plot(self._entropy_results["time"], self._entropy_results["entropy"])
            ax.set_xlabel("Time (s)")
            ax.set_ylabel("Entropy")
            fig.savefig(self.config.get_output_path(f"{base_name}_graph", DEFAULT_OUTPUT_FORMATS["plot"]), dpi=vc.dpi)
            plt.close(fig)
        except Exception as e:
            logger.error(f"Error creating visualization: {str(e)}")
            raise RuntimeError(f"Failed to create visualization: {str(e)}")

    def run_analysis(self, directory: Path, output_prefix: str = "") -> None:
        """process_directory -> compute_entropy -> create_visualization (SA:225-253)."""
        try:
            directory = Path(directory)
            self.process_directory(directory)
            self.compute_entropy()
            timestamp = datetime.now().strftime("%Y%m%d_%H%M%S")
            base_name = f"{directory.stem}_{output_prefix}_{timestamp}"
            self.create_visualization(base_name)
            logger.info(f"Analysis completed successfully: {base_name}")
        except Exception as e:
            logger.error(f"Analysis failed: {str(e)}")
            raise


class SpatialEntropyAnalyzer(_AnalyzerBase):
    """Per-frame normalised Shannon entropy of the (FOV-weighted) tile histogram,
    averaged over `config.tile_counts` (SA:107-164)."""

    def compute_entropy_packed(self, packed: torch.Tensor, **kw) -> SpatialResult:
        """Tensor-level entry point: packed[F,U,3] on the device -> SpatialResult.
        Raises what the reference raises for bad data (out-of-range coordinate,
        frame without users)."""
        res = self.engine.spatial(packed, **kw)
        self.engine.raise_for_flags()
        return res

    def compute_entropy(self) -> pd.DataFrame:
        if not self._data_cache:
            raise ValidationError("No data available. Call process_directory first.")
        # host-buffer pipeline of the library (frame batches, upload | kernels | download on three streams): the
        # video need not fit the GPU, the results arrive in page-locked host arrays
        res = self.engine.spatial_host(self._host_packed())
        self.engine.raise_for_flags()
        ent, hist0, assign0 = res["entropy"], res["hist0"], res["assign0"]
        centres = self._fibonacci_vectors[self.config.tile_counts[0]]
        ids = self._data_cache["identifiers"]

        def weights(f):
            return lambda: {centres[i]: float(hist0[f, i]) for i in np.flatnonzero(hist0[f])}

        def assignments(f):
            return lambda: {ids[u]: int(assign0[f, u]) for u in np.flatnonzero(assign0[f] != 0xFFFF)}

        F = len(ent)
        self._entropy_results = pd.DataFrame({
            "time": list(self._data_cache["times"]), "entropy": list(ent),
            "tile_weights": [LazyRowDict(weights(f)) for f in range(F)],
            "tile_assignments": [LazyRowDict(assignments(f)) for f in range(F)]})
        return self._entropy_results

    def compute_user_entropy(self, batch_bytes: int = 256 << 20) -> pd.DataFrame:
        """Per-viewer exploration entropy: compute_spatial_entropy (EU:147-211) of each user's samples over the frames,
        averaged over `config.tile_counts` -- how much of the sphere one viewer covered.  One row per user:
        `identifier`, `frames` (frames with a sample), `entropy` (NaN for a user without any sample) and
        `tile_weights`, a lazy {Vector: weight} dict of the user's summed tile weights of tile_counts[0].

        The host array goes to the device in frame batches of about `batch_bytes` into one exact accumulator, so a
        video larger than the GPU's memory works and the result does not depend on the batching."""
        if not self._data_cache:
            raise ValidationError("No data available. Call process_directory first.")
        host = self._host_packed()
        F, U = int(host.shape[0]), int(host.shape[1])
        eng = self.engine
        acc = eng.user_accumulator(U)
        fb = max(1, int(batch_bytes) // max(1, U * 3 * host.itemsize))
        for f0 in range(0, F, fb):
            eng.users_accumulate(torch.from_numpy(host[f0:f0 + fb]).to(eng.device, non_blocking=True), acc, max(F, 1))
        res = eng.users_finish(acc, max(F, 1), want_per_k=False)
        eng.raise_for_flags()
        ent, frames, hist0 = res.entropy.cpu().numpy(), res.frames.cpu().numpy(), res.hist0.cpu().numpy()
        centres = self._fibonacci_vectors[self.config.tile_counts[0]]

        def weights(u):
            return lambda: {centres[i]: float(hist0[u, i]) for i in np.flatnonzero(hist0[u])}

        return pd.DataFrame({"identifier": list(self._data_cache["identifiers"]), "frames": frames.astype(np.int64),
                             "entropy": ent, "tile_weights": [LazyRowDict(weights(u)) for u in range(U)]})


class TransitionEntropyAnalyzer(_AnalyzerBase):
    """Per-frame-pair transition entropy with the reference's literal bookkeeping
    (TA:107-175, EU:213-332).  The first frame yields no row; row time is the
    CURRENT frame's time (TA:130,162)."""

    def __init__(self, config: Optional[AnalyzerConfig] = None, device: Optional[torch.device] = None,
                 mode: str = "literal"):
        super().__init__(config, device)
        self.mode = mode

    def compute_entropy_packed(self, packed: torch.Tensor, **kw) -> TransitionResult:
        res = self.engine.transition(packed, mode=self.mode, **kw)
        self.engine.raise_for_flags()
        return res

    def compute_entropy(self) -> pd.DataFrame:
        if not self._data_cache:
            raise ValidationError("No data available. Call process_directory first.")
        res = self.engine.transition_host(self._host_packed(), mode=self.mode)
        self.engine.raise_for_flags()
        ent, counts, pairs = res["entropy"], res["prev_count0"], res["pairs0"]
        centres = self._fibonacci_vectors[self.config.tile_counts[0]]
        ids = self._data_cache["identifiers"]
        times = self._data_cache["times"]

        def weights(r):
            return lambda: {centres[i]: int(counts[r, i]) for i in np.flatnonzero(counts[r])}

        def assignments(r):
            return lambda: {ids[u]: (int(pairs[r, u, 0]), int(pairs[r, u, 1])) for u in np.flatnonzero(pairs[r, :, 0] != 0xFFFF)}

        R = len(ent)
        self._entropy_results = pd.DataFrame({
            "time": [times[r + 1] for r in range(R)], "entropy": list(ent),
            "tile_weights": [LazyRowDict(weights(r)) for r in range(R)],
            "tile_assignments": [LazyRowDict(assignments(r)) for r in range(R)]})
        return self._entropy_results

    def compute_transition_counts(self, batch_bytes: int = 256 << 20) -> Dict:
        """Tile transition matrix of the video: per tile count of `config.tile_counts` the [T, T] int64 numpy array
        of users moving from tile p in one frame to tile c in the next, summed over all frame pairs, and the pooled
        conditional entropy.  Returns dict(counts=[...], entropy=float, per_k=[K] float64, pairs=int).

        The host array goes to the device in frame batches of about `batch_bytes` that overlap by one frame, into one
        exact accumulator: a video larger than the GPU's memory works and the result does not depend on the batching."""
        host = self._host_packed()
        F, U = int(host.shape[0]), int(host.shape[1])
        eng = self.engine
        acc = eng.transition_counts_accumulator()
        fb = max(2, int(batch_bytes) // max(1, U * 3 * host.itemsize))
        for f0 in range(0, max(F - 1, 1), fb - 1):
            eng.transition_counts_accumulate(torch.from_numpy(host[f0:f0 + fb]).to(eng.device, non_blocking=True), acc)
        res = eng.transition_counts_finish(acc)
        eng.raise_for_flags()
        return dict(counts=[c.cpu().numpy() for c in res.counts], entropy=float(res.entropy),
                    per_k=res.per_k.cpu().numpy(), pairs=res.pairs)

    def compute_user_transition_entropy(self, batch_bytes: int = 256 << 20) -> pd.DataFrame:
        """Per-viewer transition entropy: the textbook conditional entropy (EU:321-327) of each user's own moves from
        tile p in one frame to tile c in the next, averaged over `config.tile_counts` -- how predictable one viewer's
        movement is.  One row per user: `identifier`, `pairs` (frames f with the user present in f and f+1) and
        `entropy` (NaN for a user without any pair).

        A user's result depends on that user's samples only, so the host array goes to the device in blocks of user
        columns (all frames of about `batch_bytes` worth of users): a video larger than the GPU's memory works and the
        result does not depend on the batching."""
        host = self._host_packed()
        F, U = int(host.shape[0]), int(host.shape[1])
        eng = self.engine
        ub = max(1, int(batch_bytes) // max(1, F * 3 * host.itemsize))
        ent, pairs = np.empty(U, dtype=np.float64), np.empty(U, dtype=np.int64)
        for u0 in range(0, U, ub):
            block = torch.from_numpy(np.ascontiguousarray(host[:, u0:u0 + ub])).to(eng.device, non_blocking=True)
            res = eng.user_transitions(block, want_per_k=False)
            ent[u0:u0 + ub] = res.entropy.cpu().numpy()
            pairs[u0:u0 + ub] = res.pairs.cpu().numpy()
        eng.raise_for_flags()
        return pd.DataFrame({"identifier": list(self._data_cache["identifiers"]), "pairs": pairs, "entropy": ent})


class NaiveSpatialEntropyAnalyzer(_AnalyzerBase):
    """Per-frame normalised Shannon entropy over a latitude/longitude grid of tile_width x
    tile_height degree tiles (NA:39-241, compute_naive_spatial_entropy EU:362-453): a sample counts
    1.0 on the tile "{int((lon+180)/tile_width)}_{int((lat+90)/tile_height)}" (EU:378-381) of its
    rounded direction; entropy_config.use_weight_distribution only selects the normalisation
    (EU:443-448).  The frame loop of NA:125-150 runs in the same streaming kernels as the lattice
    analyzers, the grid being one more cell -> tile table."""

    def __init__(self, config: Optional[NaiveAnalyzerConfig] = None, device: Optional[torch.device] = None):
        super().__init__(config or NaiveAnalyzerConfig(), device)

    @property
    def engine(self) -> Engine:
        if self._engine is None:
            c = self.config
            if c.tile_width <= 0 or c.tile_height <= 0:
                # the reference's -1 placeholders (CFG:104-105) would produce meaningless negative keys
                raise ValidationError("No tile dimensions provided")
            self._engine = get_engine(c.video_width, c.video_height, [1], c.entropy_config, self._device,
                                      naive_tiles=(c.tile_width, c.tile_height))
        return self._engine

    def tile_key(self, code: int) -> str:
        """The reference's string key of a grid code (EU:381)."""
        nlat1 = 180 // self.config.tile_height + 1
        return f"{code // nlat1}_{code % nlat1}"

    def compute_entropy_packed(self, packed: torch.Tensor, **kw) -> SpatialResult:
        """packed[F,U,3] on the device -> SpatialResult; hist0[F, codes] holds the users per grid code,
        assign0[F,U] the grid code of every user (`tile_key` turns a code into the reference's key)."""
        res = self.engine.spatial(packed, **kw)
        flags = self.engine.poll_flags()
        if flags & N.VET_FLAG_OUT_OF_RANGE:
            raise ValidationError("Normalized coordinates must be between 0 and 1")  # DU:256-257
        if flags & N.VET_FLAG_EMPTY_FRAME:
            raise ValidationError("Empty radial points dictionary")  # EU:404-405
        return res

    def compute_entropy(self) -> pd.DataFrame:
        if not self._data_cache:
            raise ValidationError("No data available. Call process_directory first.")
        res = self.compute_entropy_packed(self._device_packed(), want_hist0=False, want_assign0=False)
        ent = res.entropy.cpu().numpy()
        n = len(ent)
        # NA:136-150 stores None for the weights and assignments of every frame
        self._entropy_results = pd.DataFrame({"time": list(self._data_cache["times"]), "entropy": list(ent),
                                              "tile_weights": [None] * n, "tile_assignments": [None] * n})
        return self._entropy_results
