"""`bench.py --dump-outputs DIR`: after the timed steps the benchmark writes what its timed path returned in the
last step, for its own seeded input, as float32 / float64 .npy files (assign0 for a fixed sample of users)."""
import json
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("transition", [False, True], ids=["spatial", "analyze"])
def test_bench_dumps_the_outputs_of_its_timed_path(tmp_path, transition):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    cmd = [sys.executable, str(ROOT / "bench.py"), "--workload", "tiny", "--steps", "3", "--warmup", "1", "--no-e2e",
           "--no-cpu", "--no-extra", "--no-c5", "--sustained-seconds", "0", "--dump-outputs", str(tmp_path)]
    if transition:
        cmd.append("--transition")
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=str(ROOT))
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 3

    got = {p.stem: np.load(p) for p in tmp_path.glob("*.npy")}
    names = {"entropy", "hist0", "assign0", "assign0_users"} | ({"tr_entropy", "tr_prev_count0"} if transition else set())
    assert set(got) == names
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20

    import bench
    from viewport_entropy_toolkit_b200 import EntropyConfig, get_engine
    wl = bench.WORKLOADS["tiny"]
    dev = torch.device("cuda")
    packed = bench.synth_on_device(torch, wl["F"], wl["U"], 20260000 + 3000, dev)
    eng = get_engine(100, 200, wl["tile_counts"], EntropyConfig(fov_angle=wl["fov"], use_weight_distribution=wl["use_w"],
                                                               power_factor=wl["pf"]), dev)
    if transition:
        sp, tr = eng.analyze(packed, want_per_k=False, want_pairs0=False)
        np.testing.assert_allclose(got["tr_entropy"], tr.entropy.cpu().numpy(), rtol=1e-12, atol=0, equal_nan=True)
        assert np.array_equal(got["tr_prev_count0"], tr.prev_count0.cpu().numpy())
    else:
        sp = eng.spatial(packed, want_per_k=False)
    assert eng.poll_flags() == 0
    users = got["assign0_users"].astype(np.int64)
    assert len(users) == min(wl["U"], bench.DUMP_USERS) and np.array_equal(users, np.unique(users))
    np.testing.assert_allclose(got["entropy"], sp.entropy.cpu().numpy(), rtol=1e-12, atol=0)
    np.testing.assert_allclose(got["hist0"], sp.hist0.cpu().numpy(), rtol=1e-12, atol=0)
    assert np.array_equal(got["assign0"], sp.assign0.cpu().numpy()[:, users].astype(np.float32))
