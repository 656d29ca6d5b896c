"""Multi-rank GPU test of `user_transitions_sharded`: every rank reads the columns of its users (frame_range over the
users) over all frames, computes them, and one all-gather of the per-user rows completes the result -- which must
equal ONE GPU's Engine.user_transitions on the whole video bit for bit, on every rank (ragged user shards, a rank
without users, missing samples, users past the shared-memory record capacity).

Ranks run as separate processes: NCCL with one GPU per rank when the box has `world` GPUs, gloo on a shared GPU
otherwise (the rows are then staged through host memory)."""
import os
import sys
from pathlib import Path

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))


def _video(F, U, seed, missing, iid=False):
    rng = np.random.default_rng(seed)
    if iid:
        mu, mv = rng.uniform(0, 1, (F, U)), rng.uniform(0, 1, (F, U))
    else:
        mu = np.clip(rng.normal(0.5, 0.15, U), 0, 1)[None] + np.cumsum(rng.normal(0, 0.02, (F, U)), 0)
        mv = np.clip(rng.normal(0.5, 0.10, U), 0, 1)[None] + np.cumsum(rng.normal(0, 0.012, (F, U)), 0)
        for a in (mu, mv):
            np.abs(a, out=a)
            a[a > 1] = 2 - a[a > 1]
            np.clip(a, 0, 1, out=a)
    p = np.stack([np.broadcast_to(np.arange(F)[:, None] * 0.1, (F, U)), mu, mv], -1).astype(np.float32)
    if missing:
        p[rng.uniform(size=(F, U)) < missing, 1] = np.nan
    return p


def _engine(cfg, device):
    from viewport_entropy_toolkit_b200 import Engine, EntropyConfig
    return Engine(100, 200, cfg["tcs"], EntropyConfig(fov_angle=90.0, use_weight_distribution=False), device)


def _worker(rank, world, port, cfg, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    ndev = torch.cuda.device_count()
    device = torch.device("cuda", rank % ndev)
    torch.cuda.set_device(device)
    nccl = ndev >= world
    if nccl:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=device)
    else:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    from viewport_entropy_toolkit_b200 import user_transitions_sharded
    video = _video(cfg["F"], cfg["U"], cfg["seed"], cfg["missing"], cfg.get("iid", False))
    eng = _engine(cfg, device)

    def load(b, e):
        return torch.from_numpy(np.ascontiguousarray(video[:, b:e])).to(device)

    res = user_transitions_sharded(eng, load, cfg["U"])
    np.savez(Path(out_dir) / f"r{rank}.npz", entropy=res.entropy.cpu().numpy(), per_k=res.per_k.cpu().numpy(),
             pairs=res.pairs.cpu().numpy(), flags=eng.poll_flags(), nccl=int(nccl))
    dist.destroy_process_group()


CASES = [
    dict(world=2, F=60, U=301, tcs=[200], missing=0.0, seed=1),                    # ragged 151 + 150
    dict(world=3, F=40, U=1001, tcs=[20, 50, 1000], missing=0.1, seed=2),          # missing samples, odd U
    dict(world=4, F=30, U=3, tcs=[200], missing=0.05, seed=3),                     # rank 3 owns no user
    dict(world=4, F=4001, U=37, tcs=[20, 200, 2000], missing=0.02, seed=4, iid=True),  # records past shared memory
]


@pytest.mark.parametrize("cfg", CASES, ids=lambda c: f"w{c['world']}_F{c['F']}_U{c['U']}")
def test_user_transitions_sharded_equals_single_gpu(tmp_path, cfg):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import torch.multiprocessing as mp
    world = cfg["world"]
    port = 35500 + (os.getpid() * 7 + world * 131 + cfg["F"]) % 2000
    mp.spawn(_worker, args=(world, port, cfg, str(tmp_path)), nprocs=world, join=True)

    eng = _engine(cfg, torch.device("cuda", 0))
    video = _video(cfg["F"], cfg["U"], cfg["seed"], cfg["missing"], cfg.get("iid", False))
    one = eng.user_transitions(torch.from_numpy(video).cuda())
    assert eng.poll_flags() == 0
    assert int(one.pairs.max()) > 0
    for r in range(world):
        z = np.load(tmp_path / f"r{r}.npz")
        assert int(z["flags"]) == 0
        assert np.array_equal(z["pairs"], one.pairs.cpu().numpy())
        assert np.array_equal(z["entropy"].view(np.int64), one.entropy.cpu().numpy().view(np.int64))
        assert np.array_equal(z["per_k"].view(np.int64), one.per_k.cpu().numpy().view(np.int64))
    eng.close()
