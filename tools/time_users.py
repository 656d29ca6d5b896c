"""Timing of the per-viewer exploration entropy (Engine.users: k_user_hist + k_user_entropy) against the
transposition route (Engine.spatial on packed.transpose(0, 1).contiguous(), copy included), in one process:

    python tools/time_users.py [frames] [users] [--out DIR]

Shapes: configs[2] (3600 frames x 100k users, 201 tiles, fov 90, pf 2) weighted and unweighted, and the default five
tile counts [20, 50, 100, 250, 1000] weighted and unweighted.  Reports CUDA-event milliseconds per call after warm-up,
samples/s, the share of the 12 B/sample HBM read bound (7.7 TB/s), k_user_hist on the same tensor with every sample
missing (the staging floor: read, decode, barriers, no adds), the same for the transposition route (launched
without CUDA graphs), the max difference between the two, and the card name and power limit read in the same run.
The input (4.3 GB at configs[2]) is larger than L2, so every call reads it from HBM.  One JSON line per shape; --out writes them to DIR/time_users.jsonl."""
import json
import subprocess
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import torch

import bench
from viewport_entropy_toolkit_b200 import Engine, EntropyConfig

HBM_BYTES_PER_S = 7.7e12


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        out = f"unknown ({e})"
    return out


def timed(fn, n):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    out_dir = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    if out_dir in args:
        args.remove(out_dir)
    F = int(args[0]) if args else 3600
    U = int(args[1]) if len(args) > 1 else 100_000
    if not torch.cuda.is_available():
        raise SystemExit("time_users.py measures on a CUDA device; there is none")
    dev = torch.device("cuda")
    torch.cuda.set_stream(torch.cuda.Stream(dev))
    p = bench.synth_on_device(torch, F, U, 20265000, dev)
    p_missing = p.clone()
    p_missing[..., 1] = float("nan")
    lines = []
    gpu = card()
    for tcs in ([200], [20, 50, 100, 250, 1000]):
        for use_w in (True, False):
            eng = Engine(100, 200, tcs, EntropyConfig(fov_angle=90.0, power_factor=2.0, use_weight_distribution=use_w), dev)
            res = eng.users(p)
            n = 5
            t_new = timed(lambda: eng.users(p), n)
            # breakdown: accumulate alone, and accumulate on the same tensor with every sample missing (the staging
            # floor: the input read, the decode and the barriers of k_user_hist, without a single add)
            acc = eng.user_accumulator(U)
            t_acc = timed(lambda: (acc.zero_(), eng.users_accumulate(p, acc, F)), n)
            t_floor = timed(lambda: (acc.zero_(), eng.users_accumulate(p_missing, acc, F)), n)
            # transposition route: copy + spatial over U "frames" of F "users", launched kernel by kernel.  With CUDA
            # graphs on, the third identical call of the five-tile-count weighted shape fails (DESIGN 4.6): that handle
            # runs the FP64 weighted kernel, whose batches of different frame counts rebuild its schedule with a
            # cudaStreamSynchronize, which is not allowed inside the capture, and run_graphed returns that error.
            eng.set_option("cuda_graph", "off")

            def route():
                return eng.spatial(p.transpose(0, 1).contiguous(), want_assign0=False)
            tr = route()
            t_tr = timed(route, 3)
            assert eng.poll_flags() == 0
            ok = ~torch.isnan(res.entropy)
            d_ent = float((res.entropy[ok] - tr.entropy[ok]).abs().max() / tr.entropy[ok].abs().max())
            d_h0 = float((res.hist0 - tr.hist0).abs().max())
            samples = F * U
            line = dict(shape=f"{F}x{U}", tile_counts=tcs, weighted=use_w, gpu=gpu,
                        users_ms=round(t_new, 3), accumulate_ms=round(t_acc, 3), accumulate_all_missing_ms=round(t_floor, 3),
                        users_samples_per_s=samples / (t_new * 1e-3),
                        users_hbm_share=(samples * 12 / HBM_BYTES_PER_S) / (t_new * 1e-3),
                        transpose_route_ms=round(t_tr, 3), transpose_route_samples_per_s=samples / (t_tr * 1e-3),
                        speedup_vs_transpose=round(t_tr / t_new, 2),
                        max_rel_entropy_diff=d_ent, max_abs_hist0_diff=d_h0)
            print(json.dumps(line), flush=True)
            lines.append(line)
            del tr, acc
            eng.close()
            torch.cuda.empty_cache()
    if out_dir:
        Path(out_dir).mkdir(parents=True, exist_ok=True)
        (Path(out_dir) / "time_users.jsonl").write_text("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
