#!/usr/bin/env python
"""Benchmark of the viewport-entropy hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c2|c5shard|...]
    python bench.py --impl reference ...     # CPU arm: the oracle port on host cores

A "step" is one pass of the hot path (decode -> cell histogram -> FOV-weighted tile
histogram -> per-frame entropy, + tile assignment output) over one synthetic batch.
Rank 0 prints ONE JSON line.  See DESIGN.md "Measurement".
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "user-frame samples/sec (bin+weighted entropy, 200 tiles)"
UNIT = "samples/s"
ALG_BYTES_PER_SAMPLE = 14  # 12 B packed (time,2dmu,2dmv) read + 2 B uint16 tile assignment written (SURVEY 8d)

WORKLOADS = {
    # BASELINE.json configs[2]: the configuration the metric is quoted on (fits one GPU)
    "c3": dict(F=3600, U=100_000, tile_counts=[200], fov=90.0, pf=2.0, use_w=True,
               desc="configs[2]: synthetic 100k users x 3600 frames, 200 tiles, FOV-weighted (fov=90, pf=2)"),
    "c2": dict(F=1800, U=10_000, tile_counts=[20, 50, 100, 200], fov=120.0, pf=2.0, use_w=False,
               desc="configs[1]: synthetic 10k users x 1800 frames, tile_counts=[20,50,100,200], unweighted"),
    # one rank's share of configs[4] (1M users x 3600 frames over 8 GPUs)
    "c5shard": dict(F=450, U=1_000_000, tile_counts=[200], fov=90.0, pf=2.0, use_w=True,
                    desc="configs[4] shard: 1M users x 450 frames per GPU, 200 tiles, FOV-weighted"),
    "tiny": dict(F=64, U=20_000, tile_counts=[200], fov=90.0, pf=2.0, use_w=True, desc="debug size"),
}


def synth_on_device(torch, F, U, seed, device, chunk=256, keep=None, kind="walk", missing=0.0):
    """Seeded 'realistic' trajectories (SURVEY 8d): gaussian start, per-frame random-walk
    steps N(0,0.010)/N(0,0.006), reflected into [0,1]; generated on the device in frame
    chunks.  Returns packed[F,U,3] float32 = (time, 2dmu, 2dmv).

    keep=(f0, f1): the whole F-frame trajectory is generated (same seed -> same video on every rank)
    but only frames [f0, f1) are stored: a rank's shard of a frame-sharded video.
    kind="iid": the adversarial variant of SURVEY 8d, every sample iid U[0,1)^2.
    missing=p: a fraction p of the samples is absent (NaN in 2dmu; user 0 is always present)."""
    g = torch.Generator(device=device).manual_seed(seed)
    k0, k1 = (0, F) if keep is None else keep
    packed = torch.empty((max(k1 - k0, 0), U, 3), dtype=torch.float32, device=device)
    if kind == "iid":
        for f0 in range(k0, k1, chunk):
            n = min(chunk, k1 - f0)
            packed[f0 - k0:f0 - k0 + n, :, 0] = (torch.arange(f0, f0 + n, device=device, dtype=torch.float32) * 0.1)[:, None]
            packed[f0 - k0:f0 - k0 + n, :, 1:] = torch.rand((n, U, 2), generator=g, device=device)
        return _punch_missing(torch, packed, missing, g)
    mu = (torch.randn(U, generator=g, device=device) * 0.15 + 0.5).clamp_(0, 1)
    mv = (torch.randn(U, generator=g, device=device) * 0.10 + 0.5).clamp_(0, 1)

    def reflect(x):
        x = x.abs()
        x = torch.where(x > 1, 2 - x, x)
        return x.clamp_(0, 1)

    for f0 in range(0, F, chunk):
        n = min(chunk, F - f0)
        su = torch.randn((n, U), generator=g, device=device) * 0.010
        sv = torch.randn((n, U), generator=g, device=device) * 0.006
        if f0 == 0:
            su[0] = 0
            sv[0] = 0
        pu = reflect(mu[None] + torch.cumsum(su, 0))
        pv = reflect(mv[None] + torch.cumsum(sv, 0))
        mu, mv = pu[-1].clone(), pv[-1].clone()
        a0, a1 = max(f0, k0), min(f0 + n, k1)   # the part of this chunk that is kept
        if a0 < a1:
            packed[a0 - k0:a1 - k0, :, 0] = (torch.arange(a0, a1, device=device, dtype=torch.float32) * 0.1)[:, None]
            packed[a0 - k0:a1 - k0, :, 1] = pu[a0 - f0:a1 - f0]
            packed[a0 - k0:a1 - k0, :, 2] = pv[a0 - f0:a1 - f0]
        if f0 + n >= k1:
            break
    edge = [(0.5, 0.5), (0.0, 0.5), (1.0, 0.5), (1.0, 1.0), (0.29, 0.57), (0.999, 0.001), (0.123456, 0.654321), (0.75, 0.25)]
    if k0 == 0 and k1 > 0:
        for u, (a, b) in enumerate(edge[:U]):
            packed[0, u, 1] = a
            packed[0, u, 2] = b
    return _punch_missing(torch, packed, missing, g)


def _punch_missing(torch, packed, missing, g):
    if missing > 0:
        for f0 in range(0, packed.shape[0], 64):
            m = torch.rand(packed[f0:f0 + 64, :, 1].shape, generator=g, device=packed.device) < missing
            m[:, 0] = False
            packed[f0:f0 + 64, :, 1][m] = float("nan")
    return packed


def synth_numpy(F, U, seed):
    """Same distribution, numpy, for the bounded CPU samples."""
    rng = np.random.default_rng(seed)
    mu = np.clip(rng.normal(0.5, 0.15, U), 0, 1)[None] + np.cumsum(rng.normal(0, 0.010, (F, U)), 0)
    mv = np.clip(rng.normal(0.5, 0.10, U), 0, 1)[None] + np.cumsum(rng.normal(0, 0.006, (F, U)), 0)
    for a in (mu, mv):
        np.abs(a, out=a)
        a[a > 1] = 2 - a[a > 1]
        np.clip(a, 0, 1, out=a)
    t = np.broadcast_to((np.arange(F) * 0.1)[:, None], (F, U))
    return np.stack([t, mu, mv], -1).astype(np.float32)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index
        self.t_from = 0.0

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "50"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t >= self.t_from and len(r) >= 9]
        sm = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in rows if r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm),
                "window": "timed region + 0.6 s of the same steps right after it (the timed region alone is shorter than nvidia-smi's sampling period)"}


# ------------------------------------------------------------------------------------
# CPU arm: the reference's own functions when they can be imported on this box (the build container's
# /root/reference, or the offline install under baseline/_ref), else the oracle's literal (reference-shaped) port
# ------------------------------------------------------------------------------------
def cpu_kind():
    try:
        from oracle import ref_driver
        return "reference" if ref_driver.reference_available() else "port"
    except Exception:
        return "port"


def ref_where():
    from oracle import _refshim
    try:
        return str(Path(_refshim.REFERENCE_SRC).resolve().relative_to(ROOT))
    except ValueError:
        return _refshim.REFERENCE_SRC


def _cpu_frame(args):
    frame, W, H, tile_counts, fov, use_w, pf, kind = args
    if kind == "reference":  # unmodified reference code per frame, like SA:129-161
        from oracle import ref_driver
        return ref_driver.spatial_frame(frame, W, H, tile_counts, fov, use_w, pf)
    from oracle import vet_oracle as orc
    vecs, ok = orc.decode_vectors(frame[:, 1], frame[:, 2], W, H)
    d = {f"u{u}": tuple(vecs[u]) for u in range(len(vecs)) if ok[u]}
    tot = 0
    for n in tile_counts:
        e, _, _ = orc.compute_spatial_entropy_literal(d, orc.lattice(n), fov, use_w, pf)
        tot += e
    return tot / len(tile_counts)


def cpu_rate(wl, sample, cores, kind, pool=None):
    """samples/s of the CPU implementation on sample[frames, users, 3]; cores > 1: a process pool over frames
    (the only parallelism the reference documents, README.md:104-120)."""
    import multiprocessing as mp
    frames, users = sample.shape[:2]
    jobs = [(sample[f], 100, 200, wl["tile_counts"], wl["fov"], wl["use_w"], wl["pf"], kind) for f in range(frames)]
    t0 = time.perf_counter()
    if cores == 1:
        for j in jobs:
            _cpu_frame(j)
    else:
        own = pool is None
        pool = pool or mp.get_context("fork").Pool(min(cores, frames))
        pool.map(_cpu_frame, jobs, chunksize=1)
        if own:
            pool.close()
    dt = time.perf_counter() - t0
    return frames * users / dt, dt


def run_reference_arm(args, wl, rank):
    """`--impl reference`: the reference's CPU implementation of the path on every host core.  When the reference
    package is importable on this box (baseline/_ref) its own compute_spatial_entropy runs, per frame, in a process
    pool over frames; else the oracle's literal layer (same scalar call structure: one numpy-scalar arccos per
    (user, tile), twice per user, EU:147-211).  Each step is a bounded sample of the workload."""
    if rank != 0:
        return
    import multiprocessing as mp
    kind = cpu_kind()
    cores = os.cpu_count() or 1
    # one frame per core and step: ~0.6 s (reference, ~100 samples/s/core at 201 tiles) or ~0.4 s (port) of work per core
    users, frames = (64, cores) if kind == "reference" else (128, cores)
    pool = mp.get_context("fork").Pool(cores)
    for w in range(args.warmup):
        cpu_rate(wl, synth_numpy(frames, users, 20261000 + w), cores, kind, pool=pool)
    t0 = time.perf_counter()
    for s in range(args.steps):
        cpu_rate(wl, synth_numpy(frames, users, 20262000 + s), cores, kind, pool=pool)
    dt = time.perf_counter() - t0
    pool.close()
    value = args.steps * frames * users / dt
    what = f"the reference's own compute_spatial_entropy (unmodified, imported from {ref_where()})" if kind == "reference" else "literal oracle port"
    sample = f"{frames} frames x {users} users per step of the {args.workload} workload, {what}, {cores} processes over frames"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / max(args.steps, 1) * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl["desc"], "tile_counts": wl["tile_counts"], "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ------------------------------------------------------------------------------------
DUMP_USERS = 1024   # assign0 is dumped for a fixed, seeded sample of this many users (all frames)


def dump_outputs(torch, out_dir, sp, tr=None):
    """Writes the outputs of one step as out_dir/<name>.npy so that two builds can be compared output for output:
    the per-frame rows whole, assign0 [F,U] for DUMP_USERS users drawn with a fixed seed (their indices in
    assign0_users.npy).  Integer outputs are written as float32 (uint16 tile ids) or float64 (int32 counts), exactly."""
    out_dir.mkdir(parents=True, exist_ok=True)
    U = sp.assign0.shape[1]
    users = np.sort(np.random.default_rng(0).choice(U, size=min(U, DUMP_USERS), replace=False))
    idx = torch.from_numpy(users).to(sp.assign0.device)
    arrays = {"entropy": sp.entropy.double(), "hist0": sp.hist0.double(),
              "assign0": sp.assign0.index_select(1, idx).float(), "assign0_users": torch.from_numpy(users).double()}
    if tr is not None:
        arrays.update(tr_entropy=tr.entropy.double(), tr_prev_count0=tr.prev_count0.double())
    for name, t in arrays.items():
        np.save(out_dir / f"{name}.npy", t.cpu().numpy())


def time_steps(torch, fn, steps, warmup):
    """ms per call of fn: CUDA events on the current stream, synchronised on both sides."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def c5_sharded(torch, dist, device, rank, world, local_rank, peak_gbs, steps, warmup):
    """BASELINE configs[4], the north_star target: 1M users x 3600 frames x 201 tiles, FOV-weighted spatial +
    transition entropy, frame-sharded.  Rank r owns frame_range(3600, r, N) and reads one halo frame; one pass of
    vet_analyze over its frames; ONE all-gather of the [entropy | transition entropy | prev_count0] rows, waited
    for inside the timed region (ShardedAnalyzer).  Strong scaling: the video is fixed, N divides it."""
    from viewport_entropy_toolkit_b200 import EntropyConfig, get_engine
    from viewport_entropy_toolkit_b200.distributed import ShardedAnalyzer
    F, U = 3600, 1_000_000
    eng = get_engine(100, 200, [200], EntropyConfig(fov_angle=90.0, use_weight_distribution=True, power_factor=2.0), device)
    sa = ShardedAnalyzer(eng, F, want_hist0=True, want_assign0=True)
    local = synth_on_device(torch, F, U, 20260000 + 5000, device, chunk=32, keep=(sa.read_begin, sa.end))
    state = {}

    def step():
        sa.start(local)
        state["res"] = sa.finish()

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    assert eng.poll_flags() == 0
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    a.record()
    for _ in range(steps):
        step()
    b.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    eng.profile(True)   # kernel times: two more steps with an event pair around every launch
    for _ in range(2):
        step()
    torch.cuda.synchronize()
    prof = eng.profile_read()
    eng.profile(False)
    prof = {k: (v[0] * steps / 2, v[1]) for k, v in prof.items()}
    t = torch.tensor([a.elapsed_time(b) / steps], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    res = state["res"]
    ok = bool(res.sp_entropy.shape[0] == F and res.tr_entropy.shape[0] == F - 1 and
              torch.isfinite(res.sp_entropy).all() and torch.isfinite(res.tr_entropy).all() and
              int(res.prev_count0.sum()) == (F - 1) * U)   # every user of every frame pair counted once, on every rank
    own = sa.end - sa.begin
    out = {"workload": "configs[4]: synthetic 1M users x 3600 frames, 200 tiles, FOV-weighted spatial + transition entropy, "
                       "frame-sharded (frame_range + 1 halo frame per rank), one vet_analyze pass per rank, one all-gather "
                       "of [entropy | tr_entropy | prev_count0] rows waited inside the timed region",
           "n_gpus": world, "scaling": "strong", "frames_rank0": own, "frames_read_rank0": sa.end - sa.read_begin,
           "steps": steps, "warmup": warmup, "ms_per_step": ms, "value": F * U / (ms * 1e-3), "unit": UNIT,
           "gathered_bytes": int(F * (2 + eng.num_tiles[0]) * 8),
           "whole_step_frac_per_gpu": ALG_BYTES_PER_SAMPLE * (F / world) * U / (ms * 1e-3) / 1e9 / peak_gbs,
           "kernel_ms_rank0": {k: v[0] / steps for k, v in prof.items() if v[1]},
           "checks_ok": ok}
    try:  # strong-scaling efficiency against the committed N=1 figure of the same code (the driver computes its own)
        n1 = json.loads((ROOT / "profiles" / "c5_sharded_n1.json").read_text())["ms_per_step"]
        out["n1_ms_ref"] = n1
        out["efficiency_vs_n1_ref"] = n1 / (world * ms)
    except Exception:
        pass
    del local, state, res
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--transition", action="store_true", help="also run the transition stage inside the step")
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary workloads reported under 'extra'")
    ap.add_argument("--no-c5", action="store_true", help="skip extra.c5_sharded (configs[4], frame-sharded over the ranks)")
    ap.add_argument("--sustained-seconds", type=float, default=2.0)
    ap.add_argument("--gather-hist0", action="store_true",
                    help="N > 1: also all-gather the hist0[F,T0] rows (5.8 MB per rank), not only entropy[F]")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path,
                    help="write what the last timed step computed (rank 0) as DIR/<name>.npy, float32/float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, wl, rank)
        return

    # Contract: ONE JSON line on stdout.  Native libraries (NCCL's version banner, ...) write to file
    # descriptor 1 behind Python's back, so stdout is pointed at stderr for the duration of the run and the
    # JSON line goes to the saved descriptor at the end.
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist
    import __graft_entry__ as ge
    ge.build()
    from viewport_entropy_toolkit_b200 import EntropyConfig, get_engine
    from viewport_entropy_toolkit_b200.engine import SpatialResult

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    # everything below runs on one non-default stream: the library replays a repeated call as a CUDA graph, and the
    # legacy default stream cannot be captured (events, copies and collectives follow torch's current stream)
    torch.cuda.set_stream(torch.cuda.Stream(device))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # keep NCCL's version banner and warnings out of stdout (one JSON line only): the banner is what
        # NCCL_DEBUG=VERSION (set on some boxes) and WARN print; other levels are redirected to stderr
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
            os.environ.pop("NCCL_DEBUG")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=device)

    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:
        pass
    peak_gbs, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks else (6650.0, "fallback")

    F, U = wl["F"], wl["U"]
    # weak scaling of the headline: the video grows with N (N x F frames of U users), frame-sharded; rank r
    # owns frames [r F, (r+1) F), which it generates itself (own seed)
    packed = synth_on_device(torch, F, U, 20260000 + 3000 + rank, device)
    ec = EntropyConfig(fov_angle=wl["fov"], use_weight_distribution=wl["use_w"], power_factor=wl["pf"])
    eng = get_engine(100, 200, wl["tile_counts"], ec, device)
    K, T0 = len(wl["tile_counts"]), eng.num_tiles[0]

    def new_out():
        return SpatialResult(entropy=torch.empty(F, dtype=torch.float64, device=device), per_k=None,
                             hist0=torch.empty((F, T0), dtype=torch.float64, device=device),
                             assign0=torch.empty((F, U), dtype=torch.uint16, device=device))

    # N > 1: the per-frame results of step i are all-gathered asynchronously while step i+1 computes, so the
    # result buffers are double-buffered; every collective is waited for before the timed region ends.
    outs = [new_out(), new_out()] if world > 1 else [new_out()]
    gathered = [(torch.empty(world * F, dtype=torch.float64, device=device),
                 torch.empty((world * F, T0), dtype=torch.float64, device=device)) for _ in outs] if world > 1 else None
    pending = [[] for _ in outs]
    out = outs[0]
    counter = [0]
    last = [None]   # what the most recent step returned

    def drain(slot):
        for w in pending[slot]:
            w.wait()
        pending[slot] = []

    def step():
        slot = counter[0] % len(outs)
        counter[0] += 1
        drain(slot)  # the all-gather that last read this slot's buffers
        o = outs[slot]
        last[0] = None  # released before the call, so that its memory is reused as before
        if args.transition:  # both analyzers in one pass over the input (configs[4])
            last[0] = eng.analyze(packed, want_per_k=False, want_pairs0=False)
        else:
            last[0] = (eng.spatial(packed, out=o), None)
        if world > 1:  # the path's only exchange: the all-gather of the per-frame results
            pending[slot] = [dist.all_gather_into_tensor(gathered[slot][0], o.entropy, async_op=True)]
            if args.gather_hist0:  # hist0 / assign0 normally stay on the rank that owns the frames
                pending[slot].append(dist.all_gather_into_tensor(gathered[slot][1], o.hist0, async_op=True))

    def drain_all():
        for s_ in range(len(outs)):
            drain(s_)

    for _ in range(3 * len(outs)):   # set-up, not warm-up: the library captures a repeated call as a CUDA graph on its third
        # occurrence (per set of output buffers)
        step()
    for _ in range(args.warmup):
        step()
    drain_all()
    torch.cuda.synchronize()
    flags = eng.poll_flags()
    assert flags == 0, f"device flags {flags}"

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.2)
    launches0 = eng.launch_count()
    replays0 = eng.graph_replays()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.t_from = time.time()
    ev0.record()
    for _ in range(args.steps):
        step()
    drain_all()
    ev1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = ev0.elapsed_time(ev1)
    launches = eng.launch_count() - launches0
    replays = eng.graph_replays() - replays0
    if args.dump_outputs is not None and rank == 0:
        dump_outputs(torch, args.dump_outputs, *last[0])
    # per-kernel device times: the SAME steps once more with an event pair around every launch (the library then
    # launches kernel by kernel instead of replaying its graph), right after the timed region
    eng.profile(True)
    pv0, pv1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pv0.record()
    for _ in range(args.steps):
        step()
    drain_all()
    pv1.record()
    torch.cuda.synchronize()
    prof_ms = pv0.elapsed_time(pv1)
    prof = eng.profile_read()
    eng.profile(False)
    clocks = None
    if rank == 0:  # keep the same load running long enough for nvidia-smi to see it
        t_end = time.time() + 0.6
        while time.time() < t_end:
            eng.spatial(packed, out=out)
            torch.cuda.synchronize()
        clocks = sampler.stop()
    t_ms = torch.tensor([ms], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_max = float(t_ms.item())
    ms_per_step = ms_max / args.steps
    samples_per_step = F * U * world
    value = samples_per_step / (ms_per_step * 1e-3)

    # roofline of the dominant kernel (device time of its own launches inside the timed region)
    dom = max(("stream", "epilogue"), key=lambda k: prof[k][0])
    k_ms, k_n = prof["stream"]
    stream_ms = k_ms / max(k_n, 1)
    launch_bytes = ALG_BYTES_PER_SAMPLE * F * U  # one launch of the streaming kernel covers the whole batch
    achieved = launch_bytes / (stream_ms * 1e-3) / 1e9
    # DRAM bytes of one launch from the committed ncu --set full capture (profiles/)
    traffic = None
    try:
        tr_rec = json.loads((ROOT / "profiles" / "traffic.json").read_text())[args.workload]
        traffic = tr_rec["dram_bytes_read"] + tr_rec["dram_bytes_write"]
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": "k_stream_tma", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
                "frac": achieved / peak_gbs, "traffic": traffic, "peak_source": peak_src,
                "ms_per_launch": stream_ms, "launches": k_n,
                "step_share": {k: prof[k][0] / prof_ms for k in prof if prof[k][1]},
                "profiled_pass": {"steps": args.steps, "ms_per_step": prof_ms / args.steps,
                                  "note": "kernel times come from a second pass of the same steps with an event pair around "
                                          "every launch; the timed region itself runs unprofiled (CUDA graph replays)"},
                "whole_step_frac": (ALG_BYTES_PER_SAMPLE * F * U / (ms / args.steps * 1e-3) / 1e9) / peak_gbs,
                "dominant_by_time": dom}

    # sustained: the same step back to back for >= 2 s inside ONE event pair, clocks sampled over exactly that window
    sustained = None
    if args.sustained_seconds > 0 and not args.transition:
        n_sus = max(args.steps, int(args.sustained_seconds * 1e3 / ms_per_step) + 1)
        s2 = ClockSampler(local_rank)
        if rank == 0:
            s2.start()
            time.sleep(0.1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        s2.t_from = time.time()
        e0.record()
        for _ in range(n_sus):
            step()
        drain_all()
        e1.record()
        torch.cuda.synchronize()
        sc = s2.stop() if rank == 0 else None
        t_s = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t_s, op=dist.ReduceOp.MAX)
        sus_ms = float(t_s.item())
        if sc:
            sc["window"] = "the sustained run itself"
        sustained = {"steps": n_sus, "seconds": sus_ms * 1e-3, "ms_per_step": sus_ms / n_sus,
                     "value": samples_per_step * n_sus / (sus_ms * 1e-3), "unit": UNIT,
                     "whole_step_frac": ALG_BYTES_PER_SAMPLE * F * U * n_sus / (sus_ms * 1e-3) / 1e9 / peak_gbs, "clocks": sc}

    # CPU baseline (rank 0, N = 1): the first 256 users x 8 frames of the SAME tensor (BASELINE.md section 4) through the
    # reference's own functions when importable here, else the port; one core, then a process pool over the frames
    cpu_sample = packed[:8, :256].float().cpu().numpy() if (rank == 0 and world == 1 and not args.no_cpu) else None

    # end to end: host buffers in, host results out, copies inside the timed region
    e2e = None
    if not args.no_e2e:
        # the host tensor a caller hands over: (2dmu, 2dmv) per user and frame -- the frame times (time = 0.1 f, identical
        # for all users of a frame) stay with the caller, the kernels never read them (VET_OPT_HOST_LAYOUT)
        host3 = torch.empty((F, U, 3), dtype=torch.float32, pin_memory=True)
        host3.copy_(packed)
        host = torch.empty((F, U, 2), dtype=torch.float32, pin_memory=True)
        host.copy_(packed[..., 1:])
        torch.cuda.synchronize()
        eng.spatial_host(host, want_per_k=False, reuse_buffers=True)  # warm-up (allocates the staging buffers)
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            res = eng.spatial_host(host, want_per_k=False, reuse_buffers=True)
        dt = time.perf_counter() - t0
        t_e = torch.tensor([dt], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
        dt = float(t_e.item())
        e2e = {"value": samples_per_step * args.e2e_steps / dt, "unit": UNIT,
               "h2d_bytes_per_step": int(host.numel() * 4),
               "d2h_bytes_per_step": int(res["entropy"].nbytes + res["hist0"].nbytes + res["assign0"].nbytes),
               "steps": args.e2e_steps, "api": "Engine.spatial_host (vet_spatial_host), pinned host input [F,U,2] = (2dmu, 2dmv)"}
        # the same with the time column uploaded as well ([F,U,3] records, 12 B per sample)
        eng.spatial_host(host3, want_per_k=False, reuse_buffers=True)
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            eng.spatial_host(host3, want_per_k=False, reuse_buffers=True)
        dt3 = time.perf_counter() - t0
        t_e = torch.tensor([dt3], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
        e2e["packed3"] = {"value": samples_per_step * args.e2e_steps / float(t_e.item()), "unit": UNIT,
                          "h2d_bytes_per_step": int(host3.numel() * 4), "api": "the same with [F,U,3] = (time, 2dmu, 2dmv) records"}
        del host3
        # the same through vet_analyze_host: both analyzers, one upload (transition rows come back as well)
        eng.analyze_host(host, want_per_k=False, want_pairs0=False, reuse_buffers=True)
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            rs, rt = eng.analyze_host(host, want_per_k=False, want_pairs0=False, reuse_buffers=True)
        dt = time.perf_counter() - t0
        t_e = torch.tensor([dt], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
        dt = float(t_e.item())
        e2e["analyze"] = {"value": samples_per_step * args.e2e_steps / dt, "unit": UNIT,
                          "h2d_bytes_per_step": int(host.numel() * 4),
                          "d2h_bytes_per_step": int(rs["entropy"].nbytes + rs["hist0"].nbytes + rs["assign0"].nbytes +
                                                    rt["entropy"].nbytes + rt["prev_count0"].nbytes),
                          "steps": args.e2e_steps,
                          "api": "Engine.analyze_host (vet_analyze_host): spatial + transition entropy, pinned host input"}
        del host, res, rs, rt

    del packed, outs, out, gathered
    torch.cuda.empty_cache()

    # secondary workloads (not the headline), device-resident
    extra = {}
    if rank == 0 and world == 1 and not args.no_extra and args.workload == "c3":
        def timed_spatial(e2, p2, o2):
            return time_steps(torch, lambda: e2.spatial(p2, out=o2), args.steps, 3)

        def outs_for(e2, F2, U2):
            return SpatialResult(entropy=torch.empty(F2, dtype=torch.float64, device=device), per_k=None,
                                 hist0=torch.empty((F2, e2.num_tiles[0]), dtype=torch.float64, device=device),
                                 assign0=torch.empty((F2, U2), dtype=torch.uint16, device=device))

        for name in ("c5shard", "c2"):
            w2 = WORKLOADS[name]
            p2 = synth_on_device(torch, w2["F"], w2["U"], 20260000 + 5000, device, chunk=32 if w2["U"] > 200_000 else 256)
            e2 = get_engine(100, 200, w2["tile_counts"], EntropyConfig(fov_angle=w2["fov"], use_weight_distribution=w2["use_w"],
                                                                     power_factor=w2["pf"]), device)
            o2 = outs_for(e2, w2["F"], w2["U"])
            ms2 = timed_spatial(e2, p2, o2)
            rate = w2["F"] * w2["U"] / (ms2 * 1e-3)
            extra[name] = {"workload": w2["desc"], "ms_per_step": ms2, "value": rate, "unit": UNIT,
                           "whole_step_frac": ALG_BYTES_PER_SAMPLE * rate / 1e9 / peak_gbs}
            if name == "c5shard":
                # configs[4] asks for weighted spatial AND transition entropy: both analyzers in one pass (vet_analyze)
                ms3 = time_steps(torch, lambda: e2.analyze(p2, want_per_k=False, want_assign0=True, want_pairs0=False), args.steps, 4)
                extra["c5shard_analyze"] = {"workload": w2["desc"] + " + transition entropy, one pass over the input",
                                            "ms_per_step": ms3, "value": w2["F"] * w2["U"] / (ms3 * 1e-3), "unit": UNIT,
                                            "whole_step_frac": ALG_BYTES_PER_SAMPLE * w2["F"] * w2["U"] / (ms3 * 1e-3) / 1e9 / peak_gbs}
            del p2, o2
            torch.cuda.empty_cache()
        # the adversarial inputs of SURVEY 8d on the headline shape: iid U[0,1)^2 samples, and 20 % of the samples missing
        o3 = outs_for(eng, F, U)
        for name, kw in (("c3_iid", dict(kind="iid")), ("c3_missing20", dict(missing=0.2))):
            p3 = synth_on_device(torch, F, U, 20260000 + 3500, device, **kw)
            ms5 = timed_spatial(eng, p3, o3)
            assert eng.poll_flags() == 0
            extra[name] = {"workload": wl["desc"] + (", iid uniform samples" if name == "c3_iid" else ", 20 % of the samples missing (NaN)"),
                           "ms_per_step": ms5, "value": F * U / (ms5 * 1e-3), "unit": UNIT,
                           "whole_step_frac": ALG_BYTES_PER_SAMPLE * F * U / (ms5 * 1e-3) / 1e9 / peak_gbs}
            del p3
        del o3
        torch.cuda.empty_cache()
        # configs[3]: transition-entropy matrices for tile_counts=[200,500,1000] on the headline tensor shape
        p4 = synth_on_device(torch, 3600, 100_000, 20260000 + 4000, device)
        e4 = get_engine(100, 200, [200, 500, 1000], EntropyConfig(use_weight_distribution=False), device)
        ms4 = time_steps(torch, lambda: e4.transition(p4, want_pairs0=False, want_per_k=False), args.steps, 4)
        extra["c4"] = {"workload": "configs[3]: synthetic 100k users x 3600 frames, tile_counts=[200,500,1000], transition entropy",
                       "ms_per_step": ms4, "value": 3599 * 100_000 / (ms4 * 1e-3), "unit": "user frame pairs/s (each under 3 tile counts)",
                       "roofline_ms": ALG_BYTES_PER_SAMPLE * 3600 * 100_000 / (peak_gbs * 1e9) * 1e3}
        del p4
        torch.cuda.empty_cache()

    # configs[4], frame-sharded over the ranks of this run: at EVERY N, all ranks
    if not args.no_c5 and args.workload == "c3":
        extra["c5_sharded"] = c5_sharded(torch, dist, device, rank, world, local_rank, peak_gbs,
                                         steps=args.steps, warmup=3)

    cpu = None
    if cpu_sample is not None:
        kind = cpu_kind()
        rate1, dt1 = cpu_rate(wl, cpu_sample, 1, kind)
        cores = os.cpu_count() or 1
        rate_n, dt_n = cpu_rate(wl, cpu_sample, cores, kind)
        what = ("the reference's own normalize_to_pixel / pixel_to_spherical / Vector.from_spherical / compute_spatial_entropy "
                f"(unmodified, imported from {ref_where()})") if kind == "reference" else "the oracle's literal layer (port)"
        cpu = {"value": rate1, "unit": UNIT, "cores": 1, "kind": kind,
               "sample": f"the first 8 frames x 256 users of the tensor the GPU consumed, through {what}, one core ({dt1:.1f} s)",
               "all_cores": {"value": rate_n, "cores": min(cores, 8), "host_cores": cores,
                             "how": f"process pool over the 8 frames (README.md:104-120), {dt_n:.1f} s"},
               "full_config_cpu_days_one_core": F * U / rate1 / 86400.0}

    if rank == 0:
        sys.stdout.flush()
        os.write(json_fd, (json.dumps({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl["desc"], "frames_per_gpu": F, "users": U, "tile_counts": wl["tile_counts"],
                       "tiles": eng.num_tiles, "fov": wl["fov"], "power_factor": wl["pf"], "weighted": wl["use_w"],
                       "video": "100x200", "input": "float32[F,U,3] resident in HBM", "outputs": "entropy[F], hist0[F,T0], assign0[F,U] u16",
                       "l2": "input 4.32 GB per step >> 126 MB L2 (no flush needed)" if F * U * 12 > 2e9 else "input larger than L2" if F * U * 12 > 1.3e8 else "input smaller than L2",
                       "transition": bool(args.transition), "sharding": "frames: the video has N x frames_per_gpu frames, rank r owns frames [r F, (r+1) F) (weak scaling); per-frame entropy all-gathered every step" + (" together with the hist0 rows" if args.gather_hist0 else " (hist0 and assign0 stay on the owning rank)") + ", asynchronously (overlapping the next step), all waited for inside the timed region.  The strong-scaling run of configs[4] (fixed video, frame_range + halo per rank, spatial + transition) is extra.c5_sharded"},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches,
            "graph_replays": replays, "clocks": clocks,
            "sustained": sustained, "extra": extra or None,
        }) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
