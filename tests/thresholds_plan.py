"""Constants and launch-planning formulas of the sources that tests/test_gpu_thresholds.py places its boundary cases
around.  No torch and no GPU: tests/test_thresholds_host.py checks them against the sources on any machine."""

MAX_T = 16384           # kMaxT (vet_host_core.inl): tiles per tile set
LUT8_MAX_T = 255        # T <= 255: u8 LUT (vet_host_tables.inl and the streaming / transition / count / user-row kernels)
T4_RANK_MAX_T = 1092    # build_delta_ranks: a delta ranking only while 15 * T * 4 < 0xFFFF
RELABEL_GROUP = 4       # kRelabelGroup (vet_transition4.cuh): tile counts relabelled per pass
TC_GROUP = 6            # kTcGroup (vet_transition_counts.cuh): tile counts per k_tc_count launch
MAX_TILE_COUNTS = 16    # kMaxTileCounts (vet_stream.cuh)
PACKED_LUT_MAX_K = 4    # d_lut_packed (vet_api_core.inl): K <= 4 and every T <= 255
ENTROPY_FRAMES_BYTES = 40 * 1024   # launch_entropy_kernel: k_entropy_frames while sum ceil(T/32) * 32 * 16 B fit
T4_RANKS = 16           # kT4Ranks (vet_transition4.cuh)
T4_OVF_CAP = 1024       # kT4OvfCap: unranked users per frame pair in k_transition4's shared memory
T4_WIN = 160            # build_delta_ranks: deltas ranked within +-160 tiles
T3_TILE_BYTES = 42      # kT3TileBytes (vet_transition3.cuh)
T3_SLOTS = 16384        # kT3Slots: the hash table of k_transition3
STATIC_SLACK = 1024     # kStaticSmemSlack (vet_host_core.inl)
TC_THREADS = 512        # kTcThreads: users per k_tc_count CTA
UT_ROWS_USERS = 32      # kUtRowsUsers: users per k_ut_rows CTA
USER_ROW_BUDGET = 96 * 1024   # vet_users_accumulate: user rows per CTA within 96 KB
USER_UB_WEIGHTED, USER_UB_UNWEIGHTED = 64, 512
I8_MIN_FRAMES = 384     # VET_I8_MIN_FRAMES: the automatic dispatch takes the tensor-core histogram from here on
TR_TILE_BYTES = 24      # launch_transition's tile_bytes per tile: the per-tile shared-memory arrays of k_transition2


def transition_max_t(optin):
    """transition_tiles_supported (vet_host_core.inl): the largest tile set the transition entry points accept."""
    return (optin - STATIC_SLACK - 64) // TR_TILE_BYTES


def t3_row_stride(T):
    return T + (T & 1)


def t3_mode(T, optin):
    """plan_transition (vet_host_transition.inl): the table k_transition3 gives a tile count of T tiles."""
    budget = optin - STATIC_SLACK
    tab_off = (T * T3_TILE_BYTES + 16 + 15) & ~15
    if tab_off + T * t3_row_stride(T) * 4 <= budget:
        return "dense"
    if tab_off + 2 * T3_SLOTS * 4 <= budget:
        return "hash"
    return "v2"


def t3_boundaries(optin):
    """(last dense T, last hash T); the first hash T and the first k_transition2 T follow them."""
    last = {}
    for T in range(2, 4096):
        last[t3_mode(T, optin)] = T
    return last["dense"], last["hash"]


def pair_table_in_smem(U, Tmax, optin):
    """launch_transition: frames whose pair table fits shared memory go to k_transition<true> (no k_transition3/4)."""
    cap = 1024
    while cap < 2 * min(U, Tmax * Tmax):
        cap <<= 1
    return Tmax * 24 + cap * 16 + 64 + STATIC_SLACK <= optin


def user_hist_ub(S, weighted):
    """vet_users_accumulate: users per k_user_hist CTA for a row of S tiles."""
    row = (S + 1) * (8 if weighted else 4)
    return max(1, min(USER_UB_WEIGHTED if weighted else USER_UB_UNWEIGHTED, USER_ROW_BUDGET // row))


def entropy_frames_bytes(Ts):
    return sum((T + 31) // 32 * 32 for T in Ts) * 16


def t4_plan_smem(T):
    """plan_transition4 (vet_host_transition.inl) with the band layout of build_delta_ranks (vet_host_tables.inl): the
    shared memory k_transition4 needs for a ranked tile set of T tiles."""
    s = 0
    while (T + (1 << s) - 1) >> s > 32:
        s += 1
    bands = (T + (1 << s) - 1) >> s
    win = min(T - 1, T4_WIN)
    key_off = 3 * (T4_RANKS * T + 4) * 4
    term_off = key_off + T4_OVF_CAP * 8
    rdelta_off = term_off + T * 8
    drank_off = (rdelta_off + bands * T4_RANKS * 4 + 15) & ~15
    return (drank_off + bands * (2 * win + 2) * 2 + 15) & ~15


def t4_runs(T, optin):
    """k_transition4 runs in front of k_transition3 (auto): the tile set is ranked and its tables fit."""
    return 2 <= T <= T4_RANK_MAX_T and t4_plan_smem(T) <= optin - STATIC_SLACK


def unit_staged_max_t(optin):
    """unit_smem (vet_host_core.inl): the largest T whose unit centres k_nearest / k_tile_weights stage in shared memory."""
    return (optin - STATIC_SLACK) // (3 * 8)

