"""The constants the boundary cases of tests/test_gpu_thresholds.py are placed around, read back from the sources.

If a constant moves, the GPU cases would keep passing while testing the interior of a range; these checks fail
instead, on any machine.  Each expression is matched as written in the source, so a rewritten rule fails here too
and has to be looked at together with the GPU case that depends on it.
"""
import re
from pathlib import Path

import pytest

import thresholds_plan as G

CSRC = Path(__file__).resolve().parents[1] / "viewport_entropy_toolkit_b200" / "csrc"


def _src(name):
    return (CSRC / name).read_text()


def _const(name, src):
    m = re.search(r"constexpr\s+[\w:]+\s+" + name + r"\s*=\s*([^;]+);", _src(src))
    assert m, f"{name} not found in {src}"
    return eval(m.group(1).replace("u", "").replace("(size_t)", ""), {}, {})


@pytest.mark.parametrize("name,src,want", [
    ("kMaxT", "host/vet_host_core.inl", G.MAX_T),
    ("kStaticSmemSlack", "host/vet_host_core.inl", G.STATIC_SLACK),
    ("kRelabelGroup", "vet_transition4.cuh", G.RELABEL_GROUP),
    ("kTcGroup", "vet_transition_counts.cuh", G.TC_GROUP),
    ("kMaxTileCounts", "vet_stream.cuh", G.MAX_TILE_COUNTS),
    ("kT3TileBytes", "vet_transition3.cuh", G.T3_TILE_BYTES),
    ("kT3Slots", "vet_transition3.cuh", G.T3_SLOTS),
    ("kTcThreads", "vet_transition_counts.cuh", G.TC_THREADS),
    ("kUtRowsUsers", "vet_user_transitions.cuh", G.UT_ROWS_USERS),
])
def test_constant(name, src, want):
    assert _const(name, src) == want


def test_t3_tile_set_limits():
    # the 14-bit tile fields of k_transition3: T = 16384 (tile id 0x3FFF) must never get a k_transition3 table
    assert _const("kNoTile", "vet_transition3.cuh") == 0x3FFF == G.MAX_T - 1
    assert "uint32_t t3_row_stride(uint32_t T) { return T + (T & 1u); }" in _src("vet_transition3.cuh")
    assert [G.t3_row_stride(T) for T in (1, 2, 233, 234)] == [2, 2, 234, 234]
    plan = _src("host/vet_host_transition.inl")
    assert "pl.tab_off = (T * vet::kT3TileBytes + 16 + 15) & ~(size_t)15;" in plan
    assert "const size_t dense = T * vet::t3_row_stride((uint32_t)T) * 4, hash = (size_t)2 * vet::kT3Slots * 4;" in plan
    assert "if (pl.tab_off + dense <= budget) {" in plan and "} else if (pl.tab_off + hash <= budget) {" in plan
    assert "const size_t budget = h->smem_optin - kStaticSmemSlack;" in plan
    # the pair table of k_transition<true> (pair_table_in_smem)
    assert "const size_t tile_bytes = (size_t)Tmax * (8 + 4 * 4);" in plan
    assert "const size_t smem_tab = tile_bytes + (size_t)cap * 16 + 64;" in plan
    # at the B200's 227 KB of opt-in shared memory per block
    assert G.t3_boundaries(227 * 1024) == (234, 2388)
    assert G.t3_mode(G.MAX_T, 227 * 1024) == "v2"
    # the transition entry points refuse tile sets whose 24 B per-tile arrays do not fit (transition_tiles_supported)
    core = (CSRC / "host" / "vet_host_core.inl").read_text()
    assert "if ((size_t)h->maxT * (8 + 4 * 4) + 64 + kStaticSmemSlack > h->smem_optin)" in core
    assert G.TR_TILE_BYTES == 8 + 4 * 4 and G.transition_max_t(227 * 1024) == 9640


def test_lut_width_rule():
    tables = _src("host/vet_host_tables.inl")
    assert tables.count("T <= 255") == 2 and "if (T <= 255) {" in tables and "if (t.T <= 255) {" in tables
    assert "if (h->K <= 4 && h->maxT <= 255) {" in _src("host/vet_api_core.inl")
    assert G.LUT8_MAX_T == 255 and G.PACKED_LUT_MAX_K == 4


def test_transition4_plan():
    plan = _src("host/vet_host_transition.inl")
    for line in ("p.key_off = (size_t)3 * (vet::kT4Ranks * T + 4) * 4;",
                 "p.term_off = p.key_off + (size_t)vet::kT4OvfCap * 8;",
                 "p.rdelta_off = p.term_off + T * 8;",
                 "p.drank_off = (p.rdelta_off + (size_t)ts.bands * vet::kT4Ranks * 4 + 15) & ~(size_t)15;",
                 "p.smem = (p.drank_off + (size_t)ts.bands * (2 * ts.win + 2) * 2 + 15) & ~(size_t)15;",
                 "if (p.smem > budget) return p;", "if (!ts.d_drank) return p;"):
        assert line in plan, line
    tables = _src("host/vet_host_tables.inl")
    assert "while (((T + (1 << s) - 1) >> s) > 32) ++s;" in tables
    assert "const int bands = (T + (1 << s) - 1) >> s;" in tables
    assert "const int win = std::min(T - 1, 160), L = 2 * win + 1;" in tables
    assert _const("kT4OvfCap", "vet_transition4.cuh") == G.T4_OVF_CAP
    assert _const("kT4Ranks", "vet_transition4.cuh") == G.T4_RANKS
    # at 227 KB: k_transition4 runs for T <= 1002 and 1025 <= T <= 1055
    runs = [T for T in range(2, 1200) if G.t4_runs(T, 227 * 1024)]
    assert runs == list(range(2, 1003)) + list(range(1025, 1056))


def test_unit_centre_staging():
    core = _src("host/vet_host_core.inl")
    assert "const size_t bytes = (size_t)T * 3 * sizeof(double);" in core
    assert "return bytes + kStaticSmemSlack <= h->smem_optin ? bytes : 0;" in core
    assert G.unit_staged_max_t(227 * 1024) == 9642


def test_delta_rank_limit():
    assert "15 * T * 4 >= 0xFFFF || T < 2) return VET_OK;" in _src("host/vet_host_tables.inl")
    T = G.T4_RANK_MAX_T
    assert 15 * T * 4 < 0xFFFF <= 15 * (T + 1) * 4
    assert _const("kT4Ranks", "vet_transition4.cuh") == 16


def test_entropy_frames_limit():
    src = _src("host/vet_host_spatial.inl")
    assert "if (e.K >= 2 && smem <= 40 * 1024) {" in src
    assert "const size_t smem = (size_t)fp.soff[e.K] * 16;" in src
    assert "fp.soff[k + 1] = fp.soff[k] + units * 32;" in src and "const int units = (e.T[k] + 31) / 32;" in src
    assert G.ENTROPY_FRAMES_BYTES == 40 * 1024
    assert G.entropy_frames_bytes([201, 2001]) <= G.ENTROPY_FRAMES_BYTES < G.entropy_frames_bytes([201, 2501])


def test_user_hist_users_per_cta():
    src = _src("host/vet_host_users.inl")
    assert "a.Ub = (int)std::max<size_t>(1, std::min<size_t>(weighted ? 64 : 512, (96u << 10) / row));" in src
    assert "return (size_t)(S + 1) * (weighted ? 8 : 4); }" in _src("vet_users.cuh")
    # a row above 96 KB: sum T > 24575 unweighted (4 B per column), > 12287 weighted (8 B); one user per CTA then
    assert (24575 + 1) * 4 == G.USER_ROW_BUDGET and (12287 + 1) * 8 == G.USER_ROW_BUDGET
    assert G.user_hist_ub(16383, True) == 1 and G.user_hist_ub(24576, False) == 1
    assert G.user_hist_ub(222, True) == 55 and G.user_hist_ub(222, False) == 110


def test_transition_counts_limits():
    src = _src("host/vet_host_transition_counts.inl")
    assert "constexpr uint64_t kTcMaxEntries = (uint64_t)1 << 28;" in src
    assert G.MAX_T * G.MAX_T == 1 << 28


def test_user_transitions_radix_passes():
    src = _src("vet_user_transitions.cuh")
    assert _const("kUtDigitBits", "vet_user_transitions.cuh") == 4
    assert "const int bits = T > 1 ? 32 - __clz(T * T - 1) : 0;" in src
    bits = (G.MAX_T * G.MAX_T - 1).bit_length()
    assert bits == 28 and -(-bits // 4) == 7
