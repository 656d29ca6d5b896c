"""Multi-rank GPU test of `transition_counts_sharded`: every rank counts the frame pairs of its frames plus the halo
frame, one all_reduce(SUM) adds the int64 counts, every rank finishes them -- the TransitionCountsResult must equal ONE
GPU's Engine.transition_counts on the whole video bit for bit, on every rank (ragged shards, a rank without frames,
missing samples).

Ranks run as separate processes: NCCL with one GPU per rank when the box has `world` GPUs, gloo on a shared GPU
otherwise (the accumulator is then staged through host memory)."""
import os
import sys
from pathlib import Path

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))


def _video(F, U, seed, missing):
    rng = np.random.default_rng(seed)
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
    from viewport_entropy_toolkit_b200 import transition_counts_sharded
    video = _video(cfg["F"], cfg["U"], cfg["seed"], cfg["missing"])
    eng = _engine(cfg, device)

    def load(b, e):
        return torch.from_numpy(np.ascontiguousarray(video[b:e])).to(device)

    res = transition_counts_sharded(eng, load, cfg["F"])
    np.savez(Path(out_dir) / f"r{rank}.npz", entropy=res.entropy.cpu().numpy(), per_k=res.per_k.cpu().numpy(),
             pairs=res.pairs, flags=eng.poll_flags(), nccl=int(nccl),
             **{f"counts{k}": c.cpu().numpy() for k, c in enumerate(res.counts)})
    dist.destroy_process_group()


CASES = [
    dict(world=2, F=9, U=3000, tcs=[200], missing=0.0, seed=1),                    # ragged 5 + 4
    dict(world=3, F=7, U=2001, tcs=[20, 50, 1000], missing=0.1, seed=2),           # missing samples, odd U
    dict(world=4, F=3, U=500, tcs=[200], missing=0.05, seed=3),                    # rank 3 owns no frame
    dict(world=4, F=601, U=257, tcs=[20, 200, 2000], missing=0.02, seed=4),        # long shards, few users, no ranks
]


@pytest.mark.parametrize("cfg", CASES, ids=lambda c: f"w{c['world']}_F{c['F']}_U{c['U']}")
def test_transition_counts_sharded_equals_single_gpu(tmp_path, cfg):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import torch.multiprocessing as mp
    world = cfg["world"]
    port = 33500 + (os.getpid() * 7 + world * 131 + cfg["F"]) % 2000
    mp.spawn(_worker, args=(world, port, cfg, str(tmp_path)), nprocs=world, join=True)

    eng = _engine(cfg, torch.device("cuda", 0))
    one = eng.transition_counts(torch.from_numpy(_video(cfg["F"], cfg["U"], cfg["seed"], cfg["missing"])).cuda())
    assert eng.poll_flags() == 0
    assert one.pairs > 0
    for r in range(world):
        z = np.load(tmp_path / f"r{r}.npz")
        assert int(z["flags"]) == 0
        assert int(z["pairs"]) == one.pairs
        assert np.array_equal(z["entropy"], one.entropy.cpu().numpy())
        assert np.array_equal(z["per_k"], one.per_k.cpu().numpy())
        for k, c in enumerate(one.counts):
            assert np.array_equal(z[f"counts{k}"], c.cpu().numpy()), (r, k)
    eng.close()
