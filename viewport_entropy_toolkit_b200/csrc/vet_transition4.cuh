// Stage 4, ONE-pass kernel (literal mode, one tile count per launch).
//
// Same closed form as vet_transition3.cuh, but the users of a frame pair are walked once.  What makes one pass
// possible is the size of the pair table: a user moves a few cells per frame, and the lattice neighbours of a
// tile sit at a handful of tile-index offsets that change slowly with latitude, so nearly every transition
// (p, c) has c - p among the 16 RANKED deltas of p's latitude band (rank 0 = staying in the tile; bands of
// 2^s consecutive tiles; ranking from the cell -> tile LUT, built once per handle: build_delta_ranks).  The table
// is [16][T] instead of [T][T] -- small enough for three copies in shared memory:
//     s_cnt[k][p]      users of (p, c = p + delta_k)                     one increment per user
//     s_first[k][p]    smallest user index of the pair                   } behind ONE pre-checked load of `second`:
//     s_second[k][p]   second smallest user index                        } old = atomicMin(first, u) leaves
//                                                                          max(old, u) as the candidate for `second`
// From row p of the three tables: D_p, m_p, (f_p, c_f) = the column of the smallest first user, (x_p, l'_p) = the
// latest first user among the other columns, cnt_cf, cnt_l, and "early" = [second user of (p, c_f) < x_p] -- the one
// thing the two-pass kernel needed its second walk for.  Users with an unranked delta (reflections at the video
// borders, large jumps) go to a list of <= 1024 entries in shared memory, sorted by (p, c, user) and read as extra
// columns.  A pair whose list overflows (adversarial inputs: iid samples) is flagged in `redo` and recomputed by
// k_transition3 / k_transition2, so every input stays exact.  The ranking never changes a result, only which path
// a user takes.
//
// One CTA per frame pair, 512 threads when several CTAs fit an SM (T = 201: 47 KB of tables, four CTAs -- all 449
// pairs of a 450-frame shard are resident at once, no partial last round), 1024 otherwise.  Order enters only
// through minima of user indices -> deterministic, counts bit-exact; the entropy sum runs in the order of
// k_transition3's block_sum, so both kernels return the same bits.
#pragma once
#include <cooperative_groups.h>

#include <type_traits>

#include "vet_stream_tma.cuh"
#include "vet_transition3.cuh"

namespace vet {

constexpr int kT4Ranks = 16;
constexpr int kT4OvfCap = 1024;       // unranked users per frame pair held in shared memory
constexpr uint32_t kT4Unranked = 0xFFu;

struct Transition4Args {
  Transition3Args t;          // rows of TILE ids (cell16), sizes, outputs; tab_off: the [3][16][T] tables
  const uint16_t* drank;      // [bands][2 win + 2]: for p in band p >> band_shift and delta c - p at index
                              // min(c - p + win, 2 win + 1): rank * T * 4 (byte offset of the rank's row in a table),
                              // kT4Unranked16 = no rank (the last entry of a row is always that: deltas outside the window)
  const int* rank_delta;      // [bands][16] delta of every rank
  int band_shift, win, bands;
  int rdelta_off;             // byte offset of the staged rank deltas (int[bands][16])
  int key_off;                // byte offset of the list of unranked users (uint64[kT4OvfCap]) in dynamic shared memory
  int drank_off;              // byte offset of the staged delta ranks
  int term_off;               // byte offset of the per-tile entropy terms (double[T])
  uint32_t* redo_count;       // pairs flagged in t.redo by this launch
  int ovf_cap;                // capacity of the list of unranked users (<= kT4OvfCap)
};

constexpr uint32_t kT4Unranked16 = 0xFFFFu;

// The three shared-memory accesses of the hot loop on 32-bit shared-space addresses (no generic-address arithmetic).
__device__ __forceinline__ uint32_t t4_lds_u16(uint32_t addr) {
  uint32_t v;
  asm("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint32_t t4_lds_volatile(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void t4_inc(uint32_t addr) {
  asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(addr) : "memory");
}

// CL: one frame pair per thread-block CLUSTER (the pairs left after the full rounds of one pair per SM): the CTAs of
// a cluster take interleaved steps of the users into their own tables, then push their non-empty entries into the
// tables of CTA 0 through distributed shared memory (add / two-level min -- the same integers as one CTA would
// have collected), and CTA 0 finishes the pair.
template <bool CL>
__global__ void __launch_bounds__(kT3Threads) k_transition4(Transition4Args A) {
  namespace cg = cooperative_groups;
  const Transition3Args& a = A.t;
  const uint32_t S = CL ? cg::this_cluster().num_blocks() : 1u, crank = CL ? cg::this_cluster().block_rank() : 0u;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  // three tables of [16][T] entries + one DUMMY entry each (index TR): users without a ranked pair (unranked delta, or
  // a missing sample) are pointed at it instead of being branched around -- its `second` stays 0, so nobody takes it
  // for an entry that needs an update, and its counter is never read
  const uint32_t T = (uint32_t)a.T, TR = T * kT4Ranks, TRp = TR + 4u;
  uint32_t* s_first = reinterpret_cast<uint32_t*>(smem_raw + a.tab_off);
  uint32_t* s_second = s_first + TRp;
  uint32_t* s_cnt = s_second + TRp;
  unsigned long long* s_key = reinterpret_cast<unsigned long long*>(smem_raw + A.key_off);
  double* s_term = reinterpret_cast<double*>(smem_raw + A.term_off);
  __shared__ double s_red[32];
  __shared__ uint32_t s_novf, s_valid;
  const uint32_t tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, NT = blockDim.x;
  const double qnan = __longlong_as_double(0x7ff8000000000000LL);

  if (a.only_rows && __ldg(a.only_count) == 0u) return;
  for (uint32_t i = tid; i < TRp; i += NT) {
    s_first[i] = kEmpty;
    s_second[i] = i < TR ? kEmpty : 0u;
    s_cnt[i] = 0u;
  }
  const uint32_t win = (uint32_t)A.win, Lc = 2u * win + 1u, Lp = Lc + 1u, bsh = (uint32_t)A.band_shift;
  {
    const uint4* __restrict__ src = reinterpret_cast<const uint4*>(A.drank);
    uint4* dst = reinterpret_cast<uint4*>(smem_raw + A.drank_off);
    for (uint32_t i = tid; i < ((uint32_t)A.bands * Lp * 2u + 15u) / 16u; i += NT) dst[i] = __ldg(src + i);
  }
  int* rdelta = reinterpret_cast<int*>(smem_raw + A.rdelta_off);
  for (uint32_t i = tid; i < (uint32_t)A.bands * kT4Ranks; i += NT) rdelta[i] = __ldg(A.rank_delta + i);
  if (tid == 0) {
    s_novf = 0u;
    s_valid = 0u;
  }
  __syncthreads();
  const uint32_t U = a.U;
  const bool vec = (U & 7u) == 0u;
  const uint32_t sa_second = smem_u32(s_second), sa_cnt = smem_u32(s_cnt), sa_drank = smem_u32(smem_raw + A.drank_off);

  for (int64_t r = blockIdx.x / S; r < a.F - 1; r += gridDim.x / S) {
    if (a.only_rows && __ldg(a.only_rows + r) == 0u) continue;  // uniform over the CTA
    const uint16_t* __restrict__ prow = a.cell16 + r * (int64_t)U;
    const uint16_t* __restrict__ crow = prow + U;
    // both frames complete (no missing user): the 0xFFFF tests drop out (block-uniform)
    const bool full = a.nvalid && __ldg(a.nvalid + r) == U && __ldg(a.nvalid + r + 1) == U;

    // ---- the pass: one table update per common user ----
    uint32_t nvalid = 0;
    // byte offset of rank(p, c)'s row in a table, kT4Unranked16 when c - p has no rank in p's band
    auto row_of = [&](uint32_t p, uint32_t c) -> uint32_t {
      const uint32_t dw = min(c - p + win, Lc);  // deltas outside the window (also "negative" ones) land on the last entry
      return t4_lds_u16(sa_drank + (((p >> bsh) * Lp + dw) << 1));
    };
    auto two_min = [&](uint32_t off, uint32_t u) {  // u is one of the two smallest users of the entry so far
      uint32_t* f = reinterpret_cast<uint32_t*>(reinterpret_cast<unsigned char*>(s_first) + off);
      uint32_t* g = reinterpret_cast<uint32_t*>(reinterpret_cast<unsigned char*>(s_second) + off);
      const uint32_t old = atomicMin(f, u);
      const uint32_t cand = max(old, u);
      if (cand < lds_u32(g)) atomicMin(g, cand);
    };
    auto to_list = [&](uint32_t u, uint32_t p, uint32_t c) {
      const uint32_t pos = atomicAdd(&s_novf, 1u);
      if (pos < (uint32_t)A.ovf_cap) s_key[pos] = ((unsigned long long)p << 48) | ((unsigned long long)c << 32) | u;
    };
    auto visit = [&](uint32_t u, uint32_t p, uint32_t c) {
      const uint32_t e = row_of(p, c);
      if (e != kT4Unranked16) {
        const uint32_t off = e + (p << 2);  // rank-major: the entries of rank 0 (most users) spread over all banks
        const uint32_t s2 = t4_lds_volatile(sa_second + off);
        t4_inc(sa_cnt + off);
        if (u < s2) two_min(off, u);  // users arrive in roughly increasing order: rare
      } else {
        to_list(u, p, c);
      }
    };
    auto pass = [&](auto full_c) {
      constexpr bool FULL = decltype(full_c)::value;
      if (vec) {
        const uint32_t kStep = NT * 8u;
        const uint32_t dummy = TR * 4u;
        // 8 users per step, in phases, so that the 8 dependent chains (rank load -> entry load) overlap; no branch
        // per user: one test per step sends the step to the slow path when any of its users needs it
        auto step = [&](const uint32_t u0, const uint4& vp, const uint4& vc) {
          const uint32_t wp[4] = {vp.x, vp.y, vp.z, vp.w}, wc[4] = {vc.x, vc.y, vc.z, vc.w};
          uint32_t e[8], s2[8];
          uint32_t slow = 0u;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const uint32_t p = (j & 1) ? (wp[j >> 1] >> 16) : (wp[j >> 1] & 0xFFFFu);
            const uint32_t c = (j & 1) ? (wc[j >> 1] >> 16) : (wc[j >> 1] & 0xFFFFu);
            uint32_t r16;
            if (FULL) {
              r16 = row_of(p, c);
            } else {
              const bool ok = max(p, c) != 0xFFFFu;  // neither of the two is the missing marker
              r16 = row_of(ok ? p : 0u, ok ? c : 0u);
              nvalid += ok ? 1u : 0u;
              r16 = ok ? r16 : 0x10000u;  // no common user here
            }
            slow |= r16 == kT4Unranked16 ? 1u : 0u;
            e[j] = r16 < kT4Unranked16 ? r16 + (p << 2) : dummy;
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) s2[j] = t4_lds_volatile(sa_second + e[j]);
#pragma unroll
          for (int j = 0; j < 8; ++j) t4_inc(sa_cnt + e[j]);
#pragma unroll
          for (int j = 0; j < 8; ++j) slow |= u0 + j < s2[j] ? 1u : 0u;
          if (slow) {  // rare: a user among the two smallest of its entry so far, or one for the list
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              if (u0 + j < s2[j]) two_min(e[j], u0 + j);
              if (e[j] == dummy) {
                const uint32_t p = (j & 1) ? (wp[j >> 1] >> 16) : (wp[j >> 1] & 0xFFFFu);
                const uint32_t c = (j & 1) ? (wc[j >> 1] >> 16) : (wc[j >> 1] & 0xFFFFu);
                if (FULL || max(p, c) != 0xFFFFu) to_list(u0 + j, p, c);
              }
            }
          }
        };
        // rows of 1M-user frames come from DRAM: two register buffers, refilled for step i + 2 right after step i
        uint4 bp[2], bc[2];
        const uint32_t first = crank * kStep + tid * 8u, stride = S * kStep;  // CTA `crank` of S takes every S-th step
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          bp[j] = bc[j] = make_uint4(0u, 0u, 0u, 0u);
          if (first + j * stride < U) {
            bp[j] = __ldg(reinterpret_cast<const uint4*>(prow + first + j * stride));
            bc[j] = __ldg(reinterpret_cast<const uint4*>(crow + first + j * stride));
          }
        }
        for (uint32_t base = first; base < U; base += 2u * stride) {
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const uint32_t u0 = base + j * stride;
            if (u0 < U) {
              step(u0, bp[j], bc[j]);
              if (u0 + 2u * stride < U) {
                bp[j] = __ldg(reinterpret_cast<const uint4*>(prow + u0 + 2u * stride));
                bc[j] = __ldg(reinterpret_cast<const uint4*>(crow + u0 + 2u * stride));
              }
            }
          }
        }
      } else {
        for (uint32_t u = crank * NT + tid; u < U; u += S * NT) {
          const uint32_t p = prow[u], c = crow[u];
          if (p != 0xFFFFu && c != 0xFFFFu) {
            ++nvalid;
            visit(u, p, c);
          }
        }
      }
    };
    const bool counted = !(vec && full);
    if (vec && full) pass(std::true_type{});
    else pass(std::false_type{});
    if (counted) {
      nvalid = __reduce_add_sync(kFull, nvalid);
      if (lane == 0 && nvalid) atomicAdd(&s_valid, nvalid);
    }
    __syncthreads();
    if (CL) {
      cg::cluster_group cluster = cg::this_cluster();
      cluster.sync();  // every CTA of the cluster has finished its steps
      if (crank != 0u) {
        uint32_t* rf = cluster.map_shared_rank(s_first, 0);
        uint32_t* rs = cluster.map_shared_rank(s_second, 0);
        uint32_t* rc = cluster.map_shared_rank(s_cnt, 0);
        for (uint32_t i = tid; i < TR; i += NT) {
          const uint32_t c = s_cnt[i];
          if (c) {
            const uint32_t f = s_first[i], s2 = s_second[i];
            s_cnt[i] = 0u;
            s_first[i] = kEmpty;
            s_second[i] = kEmpty;
            atomicAdd(rc + i, c);
            const uint32_t old = atomicMin(rf + i, f);  // the larger of (old, f) is a candidate for `second`
            const uint32_t cand = min(max(old, f), s2);
            if (cand != kEmpty) atomicMin(rs + i, cand);
          }
        }
        __shared__ uint32_t s_base;
        const uint32_t mine = s_novf;
        if (tid == 0) {
          s_base = mine ? atomicAdd(cluster.map_shared_rank(&s_novf, 0), mine) : 0u;
          if (counted && s_valid) atomicAdd(cluster.map_shared_rank(&s_valid, 0), s_valid);
        }
        __syncthreads();
        unsigned long long* rk = cluster.map_shared_rank(s_key, 0);
        for (uint32_t i = tid; i < min(mine, (uint32_t)A.ovf_cap); i += NT)
          if (s_base + i < (uint32_t)A.ovf_cap) rk[s_base + i] = s_key[i];
      }
      cluster.sync();  // the tables of CTA 0 are complete
      if (crank != 0u) {
        if (tid == 0) {
          s_novf = 0u;
          s_valid = 0u;
        }
        __syncthreads();
        continue;
      }
    }
    const double total = counted ? (double)s_valid : (double)U;
    const uint32_t novf = s_novf;
    if (novf > (uint32_t)A.ovf_cap) {
      // more unranked users than the list holds: wipe the tables, leave the pair to the two-pass kernels
      for (uint32_t i = tid; i < TR; i += NT) {
        s_first[i] = kEmpty;
        s_second[i] = kEmpty;
        s_cnt[i] = 0u;
      }
      __syncthreads();
      if (tid == 0) {
        a.redo[r] = 1u;
        atomicAdd(A.redo_count, 1u);
        s_novf = 0u;
        s_valid = 0u;
      }
      __syncthreads();
      continue;
    }
    if (novf && novf <= 256u) {
      // the unranked users sorted by (prev, cur, user).  Usually a few dozen: every thread ranks its key against all
      // others (the keys are distinct: one per user) and stores it at its rank -- two barriers instead of the ~25 of
      // the bitonic sort below, which is ~10 % of a 100k-user pair
      const unsigned long long mine = tid < novf ? s_key[tid] : 0ull;
      uint32_t rank = 0;
      if (tid < novf)
        for (uint32_t j = 0; j < novf; ++j) rank += s_key[j] < mine ? 1u : 0u;
      __syncthreads();
      if (tid < novf) s_key[rank] = mine;
      __syncthreads();
    } else if (novf) {  // bitonic sort over the next power of two
      uint32_t n2 = 2;
      while (n2 < novf) n2 <<= 1;
      for (uint32_t i = novf + tid; i < n2; i += NT) s_key[i] = ~0ull;
      __syncthreads();
      for (uint32_t k = 2; k <= n2; k <<= 1)
        for (uint32_t j = k >> 1; j > 0; j >>= 1) {
          for (uint32_t i = tid; i < n2; i += NT) {
            const uint32_t o = i ^ j;
            if (o > i) {
              const unsigned long long x = s_key[i], y = s_key[o];
              if ((x > y) == ((i & k) == 0)) {
                s_key[i] = y;
                s_key[o] = x;
              }
            }
          }
          __syncthreads();
        }
    }

    // ---- closed form per previous tile (EU:278-318): two sweeps over the columns of row p -- the ranked entries,
    // then the groups of the sorted list; the row's entries are left empty for the next pair ----
    for (uint32_t p = tid; p < T; p += NT) {
      uint32_t cnt[kT4Ranks], fst[kT4Ranks];
      const int* rd = rdelta + (p >> bsh) * kT4Ranks;
      uint32_t D = 0, m = 0, ncf = 0, ncl = 0, sec_cf = kEmpty;
      unsigned long long best = ~0ull, top = 0ull;
#pragma unroll
      for (int k = 0; k < kT4Ranks; ++k) {
        cnt[k] = s_cnt[k * T + p];
        fst[k] = s_first[k * T + p];
      }
      uint32_t lo = 0, hi = novf;
      if (novf) {
        const unsigned long long want = (unsigned long long)p << 48;
        while (lo < hi) {
          const uint32_t mid = (lo + hi) >> 1;
          if (s_key[mid] < want) lo = mid + 1;
          else hi = mid;
        }
        hi = lo;
        while (hi < novf && (uint32_t)(s_key[hi] >> 48) == p) ++hi;
      }
      // sweep 1: D_p, m_p, (f_p, c_f)
#pragma unroll
      for (int k = 0; k < kT4Ranks; ++k)
        if (cnt[k]) {
          ++D;
          m += cnt[k];
          best = min(best, ((unsigned long long)fst[k] << 32) | (uint32_t)((int)p + rd[k]));
        }
      for (uint32_t i = lo; i < hi;) {
        const uint32_t c = (uint32_t)(s_key[i] >> 32) & 0xFFFFu;
        uint32_t j = i;
        while (j < hi && ((uint32_t)(s_key[j] >> 32) & 0xFFFFu) == c) ++j;
        ++D;
        m += j - i;
        best = min(best, ((unsigned long long)(uint32_t)s_key[i] << 32) | c);
        i = j;
      }
      double term = 0.0;
      if (m) {
        // sweep 2: (x_p, l'_p) = the latest first appearance among the other columns; counts of c_f and l'_p
        const uint32_t cf = (uint32_t)best;
#pragma unroll
        for (int k = 0; k < kT4Ranks; ++k)
          if (cnt[k]) {
            const uint32_t c = (uint32_t)((int)p + rd[k]);
            if (c == cf) {
              ncf = cnt[k];
              sec_cf = s_second[k * T + p];
            } else {
              const unsigned long long v = ((unsigned long long)(fst[k] + 1u) << 32) | c;
              if (v > top) {
                top = v;
                ncl = cnt[k];
              }
            }
            s_cnt[k * T + p] = 0u;
            s_first[k * T + p] = kEmpty;
            s_second[k * T + p] = kEmpty;
          }
        for (uint32_t i = lo; i < hi;) {
          const uint32_t c = (uint32_t)(s_key[i] >> 32) & 0xFFFFu;
          uint32_t j = i;
          while (j < hi && ((uint32_t)(s_key[j] >> 32) & 0xFFFFu) == c) ++j;
          if (c == cf) {
            ncf = j - i;
            sec_cf = j - i >= 2 ? (uint32_t)s_key[i + 1] : kEmpty;
          } else {
            const unsigned long long v = ((unsigned long long)((uint32_t)s_key[i] + 1u) << 32) | c;
            if (v > top) {
              top = v;
              ncl = j - i;
            }
          }
          i = j;
        }
        // EU:297-330 in the arrangement of k_transition3 (same expressions, same order)
        const bool has2 = ncf >= 2u;
        const double Kp = 1.0 + (double)(D - 1u + (has2 ? 1u : 0u));
        double wp = 1.0;
        if (m > 1u) {
          const bool early = top != 0ull && sec_cf < (uint32_t)(top >> 32) - 1u;
          const bool cf_latest = has2 && (top == 0ull || !early);
          wp = cf_latest ? (double)(ncf - 1u) : (double)ncl;
        }
        const double tp = wp / (double)m;
        term = -((double)m / total) * (Kp * (tp * log2(tp)));
      }
      s_term[p] = term;
      if (a.prev_count0) a.prev_count0[r * (int64_t)T + p] = (int32_t)m;
    }
    __syncthreads();
    // the sum of the terms in the order of k_transition3 (block_sum over 1024 threads, thread = p mod 1024): a
    // butterfly inside every group of 32 consecutive tiles, then a butterfly over the 32 group sums
    for (uint32_t v = wid; v < 32u; v += NT >> 5) {
      double acc = 0.0;
      for (uint32_t p = v * 32u + lane; p < T; p += kT3Threads) acc += s_term[p];
      acc = warp_sum(acc);
      if (lane == 0) s_red[v] = acc;
    }
    __syncthreads();
    if (wid == 0) {
      const double Hs = warp_sum(s_red[lane]);
      const double n = (total > (double)T) ? (double)T : total;
      const double q = 1.0 / n;
      double e = Hs / (n * -q * log2(q));
      if (total == 0.0) {
        e = qnan;
        if (lane == 0) atomicOr(a.flags, (uint32_t)VET_FLAG_NO_COMMON_USER);
      }
      if (lane == 0) {
        a.out[r] = e;
        s_novf = 0u;
        s_valid = 0u;
      }
    }
    __syncthreads();
  }
}

// tile ids of one tile count from the cell ids the streaming kernel wrote (several tile counts per handle): the
// one-pass kernel then needs no lookups of its own.  8 samples per thread; n is padded to 8 by the caller's buffers.
__global__ void k_relabel_rows(const uint16_t* __restrict__ cells, const uint16_t* __restrict__ lut, int64_t n,
                               uint16_t* __restrict__ tiles) {
  const int64_t n8 = n >> 3;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(cells) + i);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t lo = w[j] & 0xFFFFu, hi = w[j] >> 16;
      const uint32_t tl = lo != 0xFFFFu ? (uint32_t)__ldg(lut + lo) : 0xFFFFu;
      const uint32_t th = hi != 0xFFFFu ? (uint32_t)__ldg(lut + hi) : 0xFFFFu;
      o[j] = tl | (th << 16);
    }
    reinterpret_cast<uint4*>(tiles)[i] = make_uint4(o[0], o[1], o[2], o[3]);
  }
  for (int64_t i = (n8 << 3) + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t c = cells[i];
    tiles[i] = c != 0xFFFFu ? __ldg(lut + c) : (uint16_t)0xFFFF;
  }
}

// The same for up to kRelabelGroup tile counts in one pass over the cell ids: the lookup tables sit in shared memory
// (entry C = 0xFFFF for a missing sample, so no branch), every cell id is read once and one row per tile count written.
// Three separate passes with lookups through L1 took 3 x 0.43 ms on 100k users x 3600 frames (configs[3]); this one
// takes 0.55 ms for its 0.72 GB in + 3 x 0.72 GB out (5.1 TB/s on a stream that is three quarters writes).  Measured and
// not kept: the tile ids of the three tile counts packed into one 32-bit entry (one lookup per sample instead of three:
// 0.58 ms) and four 16-byte loads in flight per thread (0.57 ms) -- neither the lookups nor the latency bound it.
constexpr int kRelabelGroup = 4;
constexpr int kRelabelThreads = 1024;
struct RelabelArgs {
  const uint16_t* cells;             // [n] cell ids, 0xFFFF = missing
  const uint16_t* lut[kRelabelGroup];  // [C] tile of each cell
  uint16_t* tiles[kRelabelGroup];    // [n] out
  int G;                             // tile counts of this launch
  int C;
  int cp;                            // entries per table in shared memory (>= C + 1, multiple of 8)
  int64_t n;
};

__global__ void __launch_bounds__(kRelabelThreads, 1) k_relabel_rows_group(RelabelArgs a) {
  extern __shared__ __align__(16) uint16_t s_rl[];  // [G][cp]
#pragma unroll
  for (int g = 0; g < kRelabelGroup; ++g) {
    if (g < a.G) {
      uint16_t* dst = s_rl + g * a.cp;
      for (int c = threadIdx.x; c < a.cp; c += blockDim.x) dst[c] = c < a.C ? __ldg(a.lut[g] + c) : (uint16_t)0xFFFF;
    }
  }
  __syncthreads();
  const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(s_rl);
  const uint32_t cmax = (uint32_t)a.C;
  const int64_t n8 = a.n >> 3;
  const int64_t step = (int64_t)gridDim.x * blockDim.x;
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  uint4 v = i < n8 ? __ldg(reinterpret_cast<const uint4*>(a.cells) + i) : make_uint4(0u, 0u, 0u, 0u);
  for (; i < n8; i += step) {
    const uint4 cur = v;
    if (i + step < n8) v = __ldg(reinterpret_cast<const uint4*>(a.cells) + i + step);  // next item in flight
    const uint32_t w[4] = {cur.x, cur.y, cur.z, cur.w};
    uint32_t off[8];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      off[2 * j] = min(w[j] & 0xFFFFu, cmax) << 1;
      off[2 * j + 1] = min(w[j] >> 16, cmax) << 1;
    }
#pragma unroll
    for (int g = 0; g < kRelabelGroup; ++g) {
      if (g < a.G) {
        const uint32_t tb = sbase + (uint32_t)(g * a.cp) * 2u;
        uint32_t o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = (uint32_t)t4_lds_u16(tb + off[2 * j]) | ((uint32_t)t4_lds_u16(tb + off[2 * j + 1]) << 16);
        __stcs(reinterpret_cast<uint4*>(a.tiles[g]) + i, make_uint4(o[0], o[1], o[2], o[3]));
      }
    }
  }
  for (int64_t t = (n8 << 3) + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < a.n; t += step) {
    const uint32_t c = min((uint32_t)a.cells[t], cmax);
#pragma unroll
    for (int g = 0; g < kRelabelGroup; ++g)
      if (g < a.G) a.tiles[g][t] = s_rl[g * a.cp + c];
  }
}

// pairs0[r][u] = (prev, cur) tiles of user u for the frame pair (r, r + 1), 0xFFFF 0xFFFF when the user misses a frame
__global__ void k_pairs_from_rows(const uint16_t* __restrict__ rows, int64_t F, int64_t U, uint32_t* __restrict__ pairs0) {
  const int64_t n = (F - 1) * U;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t p = rows[i], c = rows[i + U];
    pairs0[i] = (p != 0xFFFFu && c != 0xFFFFu) ? (p | (c << 16)) : kNoPair;
  }
}

}  // namespace vet
