"""Frame sharding across ranks (one process per GPU) and the single all-gather of
per-frame result rows.

The hot path shards by frames: the spatial entropy of frame f depends on frame f
only (SA:129-161); transition row r depends on frames r and r+1 (TA:143-172), so a
rank also reads ONE halo frame that it loads itself -- no sample ever crosses NVLink.
Users are never split (the literal transition bookkeeping depends on global user
order, EU:259-294).  The only collective is one all-gather of the packed per-frame
rows [entropy | transition entropy | prev_count0]; tile assignments and the hist0
rows stay sharded on the owning rank.

`users_sharded` is the per-viewer counterpart: each rank adds its frames into an exact int64 per-user accumulator,
one all_reduce(SUM) makes the rows complete on every rank.  `transition_counts_sharded` does the same for the tile
transition matrix, each rank reading its frames plus the halo frame.  `user_transitions_sharded` shards by users
instead: a viewer's transition entropy needs all of that viewer's frames and nothing of the other viewers, so each rank
reads the columns of its users and one all-gather of the per-user rows completes the result.

`analyze_sharded` is the product entry point (both analyzers, one pass over the
rank's frames through Engine.analyze / vet_analyze); `run_sharded` is the generic
wrapper around any per-rank compute function.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Callable, List, Optional, Tuple, Union

import torch
import torch.distributed as dist

from . import _native
from .engine import UserTransitionResult


def frame_range(num_frames: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous frame range [begin, end) of `rank`; the first F % world ranks get one extra frame."""
    base, extra = divmod(num_frames, world)
    begin = rank * base + min(rank, extra)
    return begin, begin + base + (1 if rank < extra else 0)


def transition_range(num_frames: int, rank: int, world: int) -> Tuple[int, int, int]:
    """Transition rows [r0, r1) owned by `rank` (row r pairs frames r and r+1) and the
    frame range [r0, r1 + 1) it must read: its own rows plus one halo frame."""
    r0, r1 = frame_range(max(num_frames - 1, 0), rank, world)
    return r0, r1, (r1 + 1 if r1 > r0 else r1)


def analyze_read_range(num_frames: int, rank: int, world: int) -> Tuple[int, int, int]:
    """(read_begin, begin, end) for the combined analysis: the rank owns frames [begin, end) -- their spatial
    rows and the transition rows that END in them, i.e. rows [begin - 1, end - 1) -- and reads
    [read_begin, end) with read_begin = begin - 1 (the halo frame; none for the rank that owns frame 0 and
    none for an empty shard)."""
    begin, end = frame_range(num_frames, rank, world)
    return (begin - 1 if (begin > 0 and end > begin) else begin), begin, end


def _world(group=None, rank: Optional[int] = None, world: Optional[int] = None) -> Tuple[int, int]:
    if world is None:
        world = dist.get_world_size(group) if dist.is_initialized() else 1
    if rank is None:
        rank = dist.get_rank(group) if dist.is_initialized() else 0
    return rank, world


def all_gather_rows(local: torch.Tensor, counts: List[int], group=None, async_op: bool = False):
    """Concatenates per-rank row blocks [n_rank, D] in rank order with ONE collective.
    Equal shards use all_gather_into_tensor directly; ragged shards are padded to the
    largest block and trimmed afterwards.  With the gloo backend (CPU collectives; two ranks
    sharing one GPU in tests) device tensors are staged through host memory.

    async_op=True returns (work, finish): `finish()` waits and returns the gathered rows."""
    world = len(counts)
    if world == 1:
        return (None, lambda: local) if async_op else local
    n_max = max(counts)
    width = tuple(local.shape[1:])
    device = local.device
    if local.shape[0] != n_max:
        pad = torch.zeros((n_max - local.shape[0],) + width, dtype=local.dtype, device=device)
        local = torch.cat([local, pad], 0)
    staged = device.type == "cuda" and dist.get_backend(group) == "gloo"
    src = local.contiguous().cpu() if staged else local.contiguous()
    out = torch.empty((world * n_max,) + width, dtype=local.dtype, device=src.device)
    work = dist.all_gather_into_tensor(out, src, group=group, async_op=async_op)

    def finish() -> torch.Tensor:
        if work is not None:
            work.wait()
        full = out.to(device) if staged else out
        if all(c == n_max for c in counts):
            return full
        return torch.cat([full[r * n_max: r * n_max + c] for r, c in enumerate(counts)], 0)

    return (work, finish) if async_op else finish()


@dataclass
class ShardedResult:
    entropy: torch.Tensor            # [F] (or [F-1]) full, on every rank
    rows: torch.Tensor               # [F, D] the gathered per-frame payload (hist0 / prev_count0 as float64)
    local_begin: int                 # first row owned by this rank
    local_end: int


def run_sharded(num_frames: int, compute_local: Callable[[int, int], Tuple[torch.Tensor, torch.Tensor]],
                transition: bool = False, group=None, rank: Optional[int] = None,
                world: Optional[int] = None) -> ShardedResult:
    """Runs `compute_local(frame_begin, frame_end)` on this rank's share and gathers.

    compute_local returns (entropy[n_rows], payload[n_rows, D]) for the rows of the given
    frame range: n_rows = frames for the spatial stage, frames - 1 for the transition stage
    (whose frame range already includes the halo frame)."""
    rank, world = _world(group, rank, world)
    if transition:
        r0, r1, fend = transition_range(num_frames, rank, world)
        counts = [transition_range(num_frames, r, world)[1] - transition_range(num_frames, r, world)[0] for r in range(world)]
        ent, payload = compute_local(r0, fend)
    else:
        r0, r1 = frame_range(num_frames, rank, world)
        counts = [frame_range(num_frames, r, world)[1] - frame_range(num_frames, r, world)[0] for r in range(world)]
        ent, payload = compute_local(r0, r1)
    if payload.dim() == 1:
        payload = payload[:, None]
    packed = torch.cat([ent.to(torch.float64)[:, None], payload.to(torch.float64)], 1)
    full = all_gather_rows(packed, counts, group)
    return ShardedResult(entropy=full[:, 0].contiguous(), rows=full[:, 1:], local_begin=r0, local_end=r1)


@dataclass
class ShardedAnalysis:
    """Both analyzers over a frame-sharded video.  The per-frame rows are complete on every rank; the bulky
    per-user outputs stay with the rank that owns the frames."""
    sp_entropy: torch.Tensor            # [F] float64, SpatialEntropyAnalyzer rows (SA:156)
    tr_entropy: torch.Tensor            # [F-1] float64, TransitionEntropyAnalyzer rows (TA:160); row r pairs frames r, r+1
    prev_count0: torch.Tensor           # [F-1, T0] int32 users per previous tile (EU:289-292)
    local_begin: int                    # this rank owns frames [local_begin, local_end)
    local_end: int
    hist0: Optional[torch.Tensor]       # [n_local, T0] float64 tile weights of the owned frames (SA:152-154)
    assign0: Optional[torch.Tensor]     # [n_local, U] uint16 tile of every user in the owned frames


class ShardedAnalyzer:
    """Runs Engine.analyze on this rank's frames (own range + the halo frame) and all-gathers the per-frame rows.

    `start(packed_local)` enqueues the kernels and the (asynchronous) collective and returns at once, so the next
    call's kernels can overlap this call's all-gather; `finish()` waits for the collective and returns the
    ShardedAnalysis.  `__call__` does both.

    packed_local holds the frames [read_begin, end) of analyze_read_range(num_frames, rank, world).

    The FOV-weighted histogram has two precision modes chosen by frame count (include/vet_b200.h,
    VET_OPT_WEIGHTED_KERNEL); the mode is pinned here from the GLOBAL frame count, so a sharded run returns the
    same bits as one rank analysing the whole video."""

    def __init__(self, engine, num_frames: int, group=None, rank: Optional[int] = None, world: Optional[int] = None,
                 mode: str = "literal", want_hist0: bool = True, want_assign0: bool = True):
        self.engine, self.num_frames, self.group, self.mode = engine, int(num_frames), group, mode
        self.rank, self.world = _world(group, rank, world)
        self.want_hist0, self.want_assign0 = want_hist0, want_assign0
        self.read_begin, self.begin, self.end = analyze_read_range(self.num_frames, self.rank, self.world)
        self.counts = [frame_range(self.num_frames, r, self.world)[1] - frame_range(self.num_frames, r, self.world)[0]
                       for r in range(self.world)]
        self.T0 = engine.num_tiles[0]
        self._pending = None

    def start(self, packed_local: torch.Tensor) -> None:
        if self._pending is not None:
            raise RuntimeError("finish() the previous call first")
        eng, T0 = self.engine, self.T0
        n_read, n_own = self.end - self.read_begin, self.end - self.begin
        if packed_local.shape[0] != n_read:
            raise ValueError(f"rank {self.rank} must be given frames [{self.read_begin}, {self.end}): "
                             f"{n_read} frames, got {packed_local.shape[0]}")
        dev = eng.device
        rows = torch.empty((n_own, 2 + T0), dtype=torch.float64, device=dev)
        hist0 = assign0 = None
        if n_own:
            pinned = eng.get_option("weighted_kernel") == "auto"
            if pinned:
                eng.set_option("weighted_kernel", "i8" if self.num_frames >= _native.I8_MIN_FRAMES else "fp64")
            try:
                sp, tr = eng.analyze(packed_local, mode=self.mode, want_per_k=False, want_hist0=self.want_hist0,
                                     want_assign0=self.want_assign0, want_pairs0=False)
            finally:
                if pinned:
                    eng.set_option("weighted_kernel", "auto")
            halo = self.begin - self.read_begin          # 1 when the first frame read is the halo frame
            rows[:, 0] = sp.entropy[halo:]
            if halo:                                       # row of frame f: the transition (f-1, f)
                rows[:, 1] = tr.entropy
                rows[:, 2:] = tr.prev_count0
            else:                                          # frame 0 ends no transition
                rows[0, 1:] = 0
                rows[1:, 1] = tr.entropy
                rows[1:, 2:] = tr.prev_count0
            hist0 = sp.hist0[halo:] if sp.hist0 is not None else None
            assign0 = sp.assign0[halo:] if sp.assign0 is not None else None
        work, finish = all_gather_rows(rows, self.counts, self.group, async_op=True)
        self._pending = (finish, hist0, assign0)

    def finish(self) -> ShardedAnalysis:
        finish, hist0, assign0 = self._pending
        self._pending = None
        full = finish()
        return ShardedAnalysis(sp_entropy=full[:, 0].contiguous(), tr_entropy=full[1:, 1].contiguous(),
                               prev_count0=full[1:, 2:].to(torch.int32), local_begin=self.begin, local_end=self.end,
                               hist0=hist0, assign0=assign0)

    def __call__(self, packed_local: torch.Tensor) -> ShardedAnalysis:
        self.start(packed_local)
        return self.finish()


def analyze_sharded(engine, packed: Union[torch.Tensor, Callable[[int, int], torch.Tensor]], num_frames: int,
                    group=None, rank: Optional[int] = None, world: Optional[int] = None, mode: str = "literal",
                    want_hist0: bool = True, want_assign0: bool = True) -> ShardedAnalysis:
    """SpatialEntropyAnalyzer.compute_entropy + TransitionEntropyAnalyzer.compute_entropy (SA:107-164,
    TA:107-175) of a video of `num_frames` frames sharded by frames over the ranks of `group`.

    `packed` is either this rank's frames [read_begin, end) (analyze_read_range) as a device tensor, or a
    callable load(frame_begin, frame_end) -> packed[frame_end - frame_begin, U, 3] that produces them."""
    sa = ShardedAnalyzer(engine, num_frames, group, rank, world, mode, want_hist0, want_assign0)
    local = packed(sa.read_begin, sa.end) if callable(packed) else packed
    return sa(local)


def users_sharded(engine, packed: Union[torch.Tensor, Callable[[int, int], torch.Tensor]], num_frames: int,
                  group=None, rank: Optional[int] = None, world: Optional[int] = None, want_per_k: bool = True,
                  want_hist0: bool = True):
    """Per-viewer exploration entropy (Engine.users) of a video of `num_frames` frames sharded by frames over the
    ranks of `group`.  Every rank adds its own frame_range (no halo frame) into an int64 accumulator with the
    fixed-point scale of the GLOBAL frame count, one all_reduce(SUM) adds the accumulators (integers: the order of
    the ranks does not matter), and every rank finishes the complete rows: the UserResult is the same on every rank
    and bit-identical to one GPU reading the whole video.  The collective moves U * (sum T_k + 1) * 8 bytes.

    `packed` is this rank's frames [begin, end) of frame_range(num_frames, rank, world) as a device tensor, or a
    callable load(frame_begin, frame_end) -> packed[frame_end - frame_begin, U, 3]."""
    rank, world = _world(group, rank, world)
    begin, end = frame_range(int(num_frames), rank, world)
    local = packed(begin, end) if callable(packed) else packed
    if local.dim() != 3 or local.shape[0] != end - begin:
        raise ValueError(f"rank {rank} must be given frames [{begin}, {end}): {end - begin} frames, got {tuple(local.shape)}")
    total = max(int(num_frames), 1)
    acc = engine.user_accumulator(int(local.shape[1]))
    if end > begin:
        engine.users_accumulate(local, acc, total)
    if world > 1:
        all_reduce_accumulator(acc, group)
    return engine.users_finish(acc, total, want_per_k, want_hist0)


def transition_counts_sharded(engine, packed: Union[torch.Tensor, Callable[[int, int], torch.Tensor]], num_frames: int,
                              group=None, rank: Optional[int] = None, world: Optional[int] = None):
    """Tile transition matrix (Engine.transition_counts) of a video of `num_frames` frames sharded by frames over the
    ranks of `group`.  Every rank reads [read_begin, end) of analyze_read_range -- its own frames plus the halo frame --
    and counts the frame pairs inside it, so each pair is counted by exactly one rank; one all_reduce(SUM) of the
    sum_k T_k^2 int64 counts adds the ranks (integers: order-free), and every rank finishes locally: the
    TransitionCountsResult is the same on every rank and bit-identical to one GPU reading the whole video.

    `packed` is this rank's frames [read_begin, end) as a device tensor, or a callable
    load(frame_begin, frame_end) -> packed[frame_end - frame_begin, U, 3]."""
    rank, world = _world(group, rank, world)
    read_begin, _, end = analyze_read_range(int(num_frames), rank, world)
    local = packed(read_begin, end) if callable(packed) else packed
    if local.dim() != 3 or local.shape[0] != end - read_begin:
        raise ValueError(f"rank {rank} must be given frames [{read_begin}, {end}): {end - read_begin} frames, "
                         f"got {tuple(local.shape)}")
    acc = engine.transition_counts_accumulator()
    if end > read_begin:
        engine.transition_counts_accumulate(local, acc)
    if world > 1:
        all_reduce_accumulator(acc, group)
    return engine.transition_counts_finish(acc)


def user_transitions_sharded(engine, packed: Union[torch.Tensor, Callable[[int, int], torch.Tensor]], num_users: int,
                             group=None, rank: Optional[int] = None, world: Optional[int] = None,
                             want_per_k: bool = True):
    """Per-viewer transition entropy (Engine.user_transitions) of a video of `num_users` users sharded by USERS over
    the ranks of `group`: a user's result depends on that user's samples only, over all frames, so rank r owns the
    users frame_range(num_users, r, world) and computes them from their columns alone.  One all_gather_rows of the
    per-user rows [entropy | pairs | per_k] makes the UserTransitionResult complete on every rank, bit-identical to one
    GPU reading the whole video.

    `packed` is this rank's user columns [F, u1 - u0, 3] as a device tensor, or a callable
    load(user_begin, user_end) -> packed[F, user_end - user_begin, 3]."""
    rank, world = _world(group, rank, world)
    u0, u1 = frame_range(int(num_users), rank, world)
    local = packed(u0, u1) if callable(packed) else packed
    if local.dim() != 3 or local.shape[1] != u1 - u0:
        raise ValueError(f"rank {rank} must be given users [{u0}, {u1}): {u1 - u0} users, got {tuple(local.shape)}")
    res = engine.user_transitions(local, want_per_k)
    cols = [res.entropy[:, None], res.pairs.to(torch.float64)[:, None]] + ([res.per_k.t()] if want_per_k else [])
    counts = [frame_range(int(num_users), r, world)[1] - frame_range(int(num_users), r, world)[0] for r in range(world)]
    full = all_gather_rows(torch.cat(cols, 1), counts, group)
    return UserTransitionResult(entropy=full[:, 0].contiguous(), per_k=full[:, 2:].t().contiguous() if want_per_k else None,
                                pairs=full[:, 1].to(torch.int32))


def all_reduce_accumulator(acc: torch.Tensor, group=None) -> None:
    """Sums the int64 accumulators (per-user rows, transition counts) of all ranks in place (one all_reduce); with the gloo backend a device
    tensor is staged through host memory, as in all_gather_rows."""
    if dist.get_backend(group) == "gloo" and acc.device.type == "cuda":
        host = acc.cpu()
        dist.all_reduce(host, op=dist.ReduceOp.SUM, group=group)
        acc.copy_(host)
    else:
        dist.all_reduce(acc, op=dist.ReduceOp.SUM, group=group)
