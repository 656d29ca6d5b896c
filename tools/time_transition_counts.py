"""Timing of the tile transition matrix (Engine.transition_counts_accumulate: k_tc_count; transition_counts_finish:
k_tc_rows + k_tc_entropy) against the route that existed before it (Engine.transition(want_pairs0=True) + bincount of
p * T + c over the present pairs, tile count 0 only), in one process:

    python tools/time_transition_counts.py [frames] [users] [--reps N] [--out DIR]

Shapes on 3600 frames x 100k users (float32, 4.3 GB: larger than L2, so every call reads it from HBM), unweighted
handles on the 100x200 cell grid: random walks (bench.synth_on_device) at [200], [200, 500, 1000] and the five default
tile counts; iid samples at [200] (every transition unranked: 64-bit global atomics); and the global variant once
([2000]: T > 1092 has no ranked deltas).  Reports CUDA-event milliseconds per accumulate after warm-up, G samples/s,
the share of the 12 B/sample HBM read bound at the measured 6535.7 GB/s (DESIGN 4.1), the same accumulate on the
input with every sample missing (the floor of the kernel: the input read, the decode and the loop, no lookup or count),
the finish time, the old route's time with its counts asserted equal, and the card name and power limit read in the
same run.  One JSON line per shape;
--out writes them to DIR/time_transition_counts.jsonl."""
import argparse
import json
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
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


def timed(fn, n, before=None):
    """Mean CUDA-event milliseconds of fn over n calls after two warm-up calls; `before` runs untimed ahead of each."""
    for _ in range(2):
        if before:
            before()
        fn()
    torch.cuda.synchronize()
    total = 0.0
    for _ in range(n):
        if before:
            before()
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
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", type=Path, default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    F, U, dev = args.frames, args.users, torch.device("cuda", 0)
    info = card()
    print(json.dumps({"card": info}), flush=True)
    lines = []
    walk = bench.synth_on_device(torch, F, U, 7, dev)
    for name, kind, tcs in (("walk_200", "walk", [200]), ("walk_200_500_1000", "walk", [200, 500, 1000]),
                            ("walk_default5", "walk", DEFAULT5), ("iid_200", "iid", [200]),
                            ("walk_2000_global", "walk", [2000])):
        p = walk if kind == "walk" else bench.synth_on_device(torch, F, U, 8, dev, kind="iid")
        missing = p.clone()
        missing[..., 1] = float("nan")
        eng = Engine(100, 200, tcs, EntropyConfig(use_weight_distribution=False), dev)
        acc = eng.transition_counts_accumulator()
        ms = timed(lambda: eng.transition_counts_accumulate(p, acc), args.reps, before=acc.zero_)
        fin = timed(lambda: eng.transition_counts_finish(acc), args.reps)
        res = eng.transition_counts_finish(acc)
        counts = [c.clone() for c in res.counts]
        floor = timed(lambda: eng.transition_counts_accumulate(missing, acc), args.reps, before=acc.zero_)
        assert eng.poll_flags() == 0
        T0 = eng.num_tiles[0]

        def old_route():
            tr = eng.transition(p, want_per_k=False, want_prev_count0=False, want_pairs0=True)
            pr = tr.pairs0.view(-1, 2).to(torch.int64)
            ok = pr[:, 0] != 0xFFFF
            return torch.bincount(pr[ok, 0] * T0 + pr[ok, 1], minlength=T0 * T0).view(T0, T0)

        old = old_route()
        assert torch.equal(old, counts[0]), name
        del old
        old_ms = timed(old_route, max(2, args.reps // 3))
        bound_ms = F * U * 12 / HBM_BYTES_PER_S * 1e3
        line = dict(shape=name, frames=F, users=U, tile_counts=tcs, accumulate_ms=round(ms, 4),
                    gsamples_per_s=round(F * U / ms / 1e6, 1), all_missing_ms=round(floor, 4),
                    hbm_bound_ms=round(bound_ms, 4), share_of_hbm_bound=round(bound_ms / ms, 4), finish_ms=round(fin, 4),
                    old_route_tile_count0_ms=round(old_ms, 3), pairs=res.pairs, entropy=float(res.entropy),
                    card=info)
        print(json.dumps(line), flush=True)
        lines.append(line)
        eng.close()
        del acc, res, counts, missing
        torch.cuda.empty_cache()
    if args.out:
        args.out.mkdir(parents=True, exist_ok=True)
        (args.out / "time_transition_counts.jsonl").write_text("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
