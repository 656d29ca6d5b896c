"""Timing of vet_analyze / vet_transition on the configs[4] shard (1M users x 450 frames, 200 tiles, weighted),
with the handle options of the transition stage switched (vet_set_option):
python tools/time_analyze.py [frames] [users]"""
import sys
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import torch
import bench
from viewport_entropy_toolkit_b200 import EntropyConfig, get_engine

F = int(sys.argv[1]) if len(sys.argv) > 1 else 450
U = int(sys.argv[2]) if len(sys.argv) > 2 else 1_000_000
dev = torch.device("cuda")
torch.cuda.set_stream(torch.cuda.Stream(dev))   # a capturable stream: repeated calls replay as CUDA graphs
p = bench.synth_on_device(torch, F, U, 20265000, dev, chunk=32 if U > 200_000 else 256)
eng = get_engine(100, 200, [200], EntropyConfig(fov_angle=90.0, power_factor=2.0), dev)


def timed(fn, n=5):
    for _ in range(4):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


for tk, overlap, cl in (("auto", "on", "auto"), ("auto", "on", "off"), ("v3", "on", "off"), ("v3", "off", "off")):
    eng.set_option("transition_kernel", tk)   # auto: one-pass kernel (cluster_tail: its clusters for the last pairs); v3: two-pass kernel alone
    eng.set_option("analyze_overlap", overlap)
    eng.set_option("cluster_tail", cl)
    eng.profile(True)
    t_an = timed(lambda: eng.analyze(p, want_per_k=False, want_assign0=True, want_pairs0=False))
    prof = eng.profile_read()
    eng.profile(False)
    t_tr = timed(lambda: eng.transition(p, want_pairs0=False, want_per_k=False))
    print(f"F={F} U={U} transition_kernel={tk} overlap={overlap} cluster_tail={cl}: analyze {t_an:.4f} ms, transition {t_tr:.4f} ms, "
          f"per kernel (ms, launches over 7 calls) {prof}", flush=True)
