"""Cost of the one collective of distributed.users_sharded: all_reduce(SUM) of the int64 per-user accumulator
[U, sum T + 1] (all_reduce_accumulator), for `world` ranks in separate processes:

    python tools/time_users_allreduce.py [--out DIR]

NCCL with one GPU per rank when the box has `world` GPUs, else gloo with the ranks sharing GPUs (the accumulator staged
through host memory).  Shapes: 100k users x 201 tiles (configs[2], 162 MB) and 1M users x 201 tiles (configs[4],
1.6 GB).  Host wall time around the collective, after one warm-up, device synchronised; the card name and power limit
are read in the same run.  One JSON line per (world, users)."""
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import torch
import torch.multiprocessing as mp

TILES = 201


def _worker(rank, world, port, users, out):
    import torch.distributed as dist
    from viewport_entropy_toolkit_b200.distributed import all_reduce_accumulator
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    ndev = torch.cuda.device_count()
    device = torch.device("cuda", rank % ndev)
    torch.cuda.set_device(device)
    backend = "nccl" if ndev >= world else "gloo"
    if backend == "nccl":
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=device)
    else:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    acc = torch.full((users, TILES + 1), rank + 1, dtype=torch.int64, device=device)
    all_reduce_accumulator(acc)
    torch.cuda.synchronize()
    times = []
    for _ in range(3):
        acc.fill_(rank + 1)
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        all_reduce_accumulator(acc)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    assert int(acc[0, 0]) == world * (world + 1) // 2
    if rank == 0:
        Path(out).write_text(json.dumps(dict(world=world, backend=backend, users=users, bytes=acc.numel() * 8,
                                             ms_min=round(min(times) * 1e3, 2), ms_median=round(sorted(times)[1] * 1e3, 2))))
    dist.destroy_process_group()


def main():
    out_dir = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    if not torch.cuda.is_available():
        raise SystemExit("time_users_allreduce.py measures on a CUDA device; there is none")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()[0]
    lines = []
    for world in (2, 4):
        for users in (100_000, 1_000_000):
            with tempfile.TemporaryDirectory() as d:
                out = Path(d) / "r0.json"
                mp.spawn(_worker, args=(world, 29800 + world * 10 + users // 100_000, users, str(out)), nprocs=world, join=True)
                line = dict(json.loads(out.read_text()), gpu=gpu, gpus_on_box=torch.cuda.device_count())
            print(json.dumps(line), flush=True)
            lines.append(line)
    if out_dir:
        Path(out_dir).mkdir(parents=True, exist_ok=True)
        (Path(out_dir) / "time_users_allreduce.jsonl").write_text("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
