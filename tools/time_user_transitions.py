"""Timing of the per-viewer transition entropy (Engine.user_transitions: k_ut_rows + k_ut_entropy) against the route
that existed before it (Engine.transition_counts on one user's column, once per user), in one process:

    python tools/time_user_transitions.py [frames] [users] [--reps N] [--loop-users N] [--out DIR]

Shapes on 3600 frames x 100k users (float32, 4.3 GB: larger than L2, so every call reads it from HBM), unweighted
handles on the 100x200 cell grid: random walks (bench.synth_on_device) and iid samples, each at [200], [200, 500,
1000] and the five default tile counts.  Reports CUDA-event milliseconds per call after warm-up, the split between
k_ut_rows and k_ut_entropy from a profiled run of its own (Engine.profile), G samples/s, the share of the 12 B/sample
HBM read bound at the measured 6535.7 GB/s (DESIGN 4.1), the scratch traffic of the tile rows (2 K U F 2 bytes: written
once, read once), the per-user loop timed on --loop-users users and scaled to all users (its per_k asserted equal
within 1e-12 relative), and the card name and power limit read in the same run.  One JSON line per shape;
--out writes them to DIR/time_user_transitions.jsonl."""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import numpy as np
import torch

import bench
from viewport_entropy_toolkit_b200 import Engine, EntropyConfig

HBM_BYTES_PER_S = 6535.7e9   # measured read bandwidth of the B200 (DESIGN 4.1)
DEFAULT5 = [20, 50, 100, 250, 1000]


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def timed(fn, n):
    """Mean CUDA-event milliseconds of fn over n calls after two warm-up calls."""
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    total = 0.0
    for _ in range(n):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        total += a.elapsed_time(b)
    return total / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("frames", type=int, nargs="?", default=3600)
    ap.add_argument("users", type=int, nargs="?", default=100_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--loop-users", type=int, default=1000)
    ap.add_argument("--out", type=Path, default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    F, U, dev = args.frames, args.users, torch.device("cuda", 0)
    info = card()
    print(json.dumps({"card": info}), flush=True)
    lines = []
    inputs = {"walk": bench.synth_on_device(torch, F, U, 7, dev), "iid": bench.synth_on_device(torch, F, U, 8, dev, kind="iid")}
    for kind in ("walk", "iid"):
        p = inputs[kind]
        for name, tcs in (("200", [200]), ("200_500_1000", [200, 500, 1000]), ("default5", DEFAULT5)):
            eng = Engine(100, 200, tcs, EntropyConfig(use_weight_distribution=False), dev)
            K = len(tcs)
            ms = timed(lambda: eng.user_transitions(p), args.reps)
            res = eng.user_transitions(p)
            eng.profile(True)
            for _ in range(args.reps):
                eng.user_transitions(p)
            torch.cuda.synchronize()
            prof = eng.profile_read()
            eng.profile(False)
            assert eng.poll_flags() == 0
            n = min(args.loop_users, U)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            loop = [eng.transition_counts(p[:, u:u + 1]).per_k for u in range(n)]
            torch.cuda.synchronize()
            loop_s = time.perf_counter() - t0
            ref = torch.stack(loop, 1).cpu().numpy()
            np.testing.assert_allclose(res.per_k[:, :n].cpu().numpy(), ref, rtol=1e-12, atol=0, equal_nan=True)
            bound_ms = F * U * 12 / HBM_BYTES_PER_S * 1e3
            line = dict(shape=f"{kind}_{name}", frames=F, users=U, tile_counts=tcs, ms=round(ms, 3),
                        k_ut_rows_ms=round(prof["user_rows"][0] / args.reps, 3),
                        k_ut_entropy_ms=round(prof["user_entropy"][0] / args.reps, 3),
                        launches_per_call=(prof["user_rows"][1] + prof["user_entropy"][1]) // args.reps,
                        gsamples_per_s=round(F * U / ms / 1e6, 1), hbm_bound_ms=round(bound_ms, 4),
                        share_of_hbm_bound=round(bound_ms / ms, 4), scratch_bytes=2 * K * U * F * 2,
                        loop_users=n, loop_s=round(loop_s, 3), loop_scaled_s=round(loop_s * U / n, 1),
                        mean_pairs=float(res.pairs.double().mean()), mean_entropy=float(np.nanmean(res.entropy.cpu().numpy())),
                        card=info)
            print(json.dumps(line), flush=True)
            lines.append(line)
            eng.close()
            del res
            torch.cuda.empty_cache()
    if args.out:
        args.out.mkdir(parents=True, exist_ok=True)
        (args.out / "time_user_transitions.jsonl").write_text("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
