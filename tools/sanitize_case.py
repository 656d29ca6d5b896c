"""Small end-to-end case for compute-sanitizer (memcheck / racecheck / initcheck / synccheck):
every kernel family once, sizes of a few thousand samples."""
import sys
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import numpy as np
import torch
from viewport_entropy_toolkit_b200 import Engine, EntropyConfig

rng = np.random.default_rng(3)


def packed(F, U, dtype=np.float32):
    p = np.stack([np.zeros((F, U)), rng.uniform(0, 1, (F, U)), rng.uniform(0, 1, (F, U))], -1).astype(dtype)
    p[0, 0, 1] = np.nan
    return torch.from_numpy(p).cuda()


e = Engine(100, 200, [200, 20], EntropyConfig(fov_angle=90.0))
r = e.spatial(packed(70, 2501))                     # k_stream_tma (odd U: unaligned tile heads) + k_whist + k_entropy_rows
t = e.transition(packed(4, 9000))                   # k_stream_tma<cells> + k_relabel_rows + k_transition4 (iid samples: lists overflow) +
                                                    # k_transition3 (dense) over the flagged pairs, per tile count + k_mean_rows
walk = packed(4, 16384)
walk[1:, :, 1:] = (walk[:1, :, 1:] + 0.004 * torch.arange(1, 4, device="cuda")[:, None, None]).clamp_(0, 1)   # small steps
tw = e.transition(walk)                             # k_transition4 on its tables (ranked tile deltas), list of a few users
e.set_option("cluster_tail", "force")
twc = e.transition(walk)                            # k_transition4<cluster>: tables merged into CTA 0 through DSMEM atomics
tc = e.transition(packed(3, 16384))                 # k_transition4<cluster>: a frame pair per cluster of 2 CTAs, iid samples
sa, ta = e.analyze(packed(3, 16384))                # the same with the spatial epilogue on the side stream beside it
e.set_option("cluster_tail", "auto")
e.set_option("weighted_kernel", "i8")
hot = packed(140, 2504)
hot[:, :600, 1:] = 0.5                              # 600 users in one cell: second count plane
r5 = e.spatial(hot)                                 # k_stream_tma (byte planes) + k_whist_i8 (TMA, tcgen05, TMEM), both passes
r6 = e.spatial(packed(3, 70001))                    # frames in chunks: k_cnt_planes + k_whist_i8
e.set_option("weighted_kernel", "auto")
e.set_option("transition_kernel", "v2")
t4 = e.transition(packed(4, 9000))                  # k_transition2 (dense)
e.set_option("transition_kernel", "auto")
e.close()
e = Engine(100, 200, [1], EntropyConfig(), naive_tiles=(30, 30))
r7 = e.spatial(packed(5, 999))                      # grid tiling: k_stream_tiles with the grid-code table
n1 = e.naive_points(torch.rand((3, 500, 2), dtype=torch.float64, device="cuda") * 90.0, 30, 30, True)   # k_naive_points
e.close()
e = Engine(100, 200, [20, 50, 1000], EntropyConfig(use_weight_distribution=False))
r2 = e.spatial(packed(9, 3001, np.float64))         # k_stream_tiles (direct unweighted) + k_entropy_rows
r3 = e.spatial(packed(3, 90001))                    # cells path: k_stream_tma + k_epilogue, several chunks per frame
t2 = e.transition(packed(3, 20000))                 # k_transition3 hash, overflow -> rows redone by k_transition2 (global tables)
t3 = e.transition(packed(5, 700), mode="textbook")  # k_transition (shared-memory table)
tcn = e.transition_counts(packed(6, 3001))          # k_tc_count (ranked deltas for 21/51 tiles, global atomics for 1001) +
                                                    # k_tc_rows + k_tc_entropy
ut = e.user_transitions(packed(3801, 7))            # k_ut_rows + k_ut_entropy (records past shared memory: global slices)
e.close()
e = Engine(200, 400, [20], EntropyConfig())
r4 = e.spatial(packed(2, 300))                      # global-table regime, weighted: k_stream_frame16 + k_whist
e.close()
e = Engine(200, 400, [20, 50], EntropyConfig(use_weight_distribution=False))
r8 = e.spatial(packed(2, 300))                      # global-table regime, unweighted: k_stream_global + k_entropy_rows
e.close()
e = Engine(200, 400, [20], EntropyConfig(), regime="direct")
r9 = e.spatial(packed(2, 300))                      # direct regime: k_decode + k_nearest + k_spatial_vectors
e.close()
torch.cuda.synchronize()
print("sanitize case ok", float(r.entropy[0]), float(t.entropy[0]), float(r2.entropy[0]), float(r3.entropy[0]),
      float(t2.entropy[0]), float(t3.entropy[0]), float(r4.entropy[0]), float(tc.entropy[0]), float(ta.entropy[0]))
