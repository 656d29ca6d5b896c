// Tile transition matrix of a video: exact [T, T] counts per tile count over all frame pairs and users, and their
// pooled conditional entropy (vet_transition_counts_accumulate / vet_transition_counts_finish).
//
// Semantics.  For tile count k (T = T_k tiles) n_k[p, c] = the number of (frame pair (f, f+1) of the call, user u) such
// that u is present in both frames, lut_k[cell(f, u)] = p and lut_k[cell(f+1, u)] = c -- the common users and
// (prev_idx, cur_idx) pairs of EU:271-276, unweighted like the reference's transition counts (a weighted and an
// unweighted handle with the same tiles give the same counts).  Missing = NaN in 2dmu or 2dmv; out-of-range coordinates
// set VET_FLAG_OUT_OF_RANGE and count as missing (as in k_user_hist); a frame or frame pair without a common user is
// normal and raises no flag.  A call counts the pairs inside the tensor it is given, so consecutive batches that overlap
// by one frame (the halo) add up to the whole video; integer sums do not depend on order, so any batching or sharding
// gives the same bits as one call.
//
// From the counts: H_k = -sum_{p,c} (n_pc / N) log2(n_pc / n_p), n_p = sum_c n_pc, N = sum n_pc, normalised by log2 T
// if N > T else by log2 N (the textbook mode's rule, EU:321-327) -- by construction transition_entropy_textbook of the
// concatenated (p, c) pairs of all frame pairs.  entropy = the sequential mean over k (SA:151-156).  N = 0 gives NaN
// (the reference would divide by zero), as do N = 1 and T = 1 (0 / 0, as in the textbook mode).
//
// acc is int64, the [T_k][T_k] matrices of all tile counts concatenated in k order (row = previous tile).
#pragma once

#include "vet_common.cuh"
#include "vet_transition4.cuh"

namespace vet {

constexpr int kTcThreads = 512;  // one user per thread; two CTAs per SM
constexpr int kTcGroup = 6;      // tile counts per launch
constexpr uint32_t kTcNone = 0xFFFFu;

struct TcCountArgs {
  int64_t F = 0, U = 0;  // frames of this call, users
  int W = 0, H = 0;
  int G = 0;             // tile counts of this launch
  int64_t pairs_per_cta = 0;  // frame pairs of one CTA's run (the last run may be shorter)
  struct Tc {
    const uint8_t* lut8 = nullptr;    // cell -> tile when T <= 255 (half the L1 footprint), else null
    const uint16_t* lut = nullptr;    // cell -> tile
    int T = 0;
    int cnt_off = -1;                 // byte offset of the [16][T] u32 counters in shared memory, -1 = no ranked deltas
    const uint16_t* drank = nullptr;  // build_delta_ranks: [bands][2 win + 2] rank * T * 4, 0xFFFF = unranked
    const int* rank_delta = nullptr;  // [bands][16] delta of every rank
    int band_shift = 0, win = 0;
    int64_t acc_off = 0;              // first entry of the tile count's matrix in acc
  } k[kTcGroup];
  unsigned long long* acc = nullptr;
  uint32_t* flags = nullptr;
};

// Shared-memory bytes of the counters of one tile count with ranked deltas.
__host__ __device__ inline size_t tc_table_bytes(int T) { return (size_t)kT4Ranks * T * 4; }

// A CTA owns the users [blockIdx.x * kTcThreads, +kTcThreads) and the frame pairs [r0, r1) of its run y = blockIdx.y
// (frames r0 .. r1: consecutive runs share their boundary frame, so each pair is counted once).  A thread owns one
// user and walks the frames in order with the samples of 8 (float) or 4 (double) frames in flight (the loads of one frame are
// coalesced over the CTA's users, 12 B apart); per tile count it keeps the user's previous tile and a pending run of
// one repeated (p, c) pair in registers.  Staying in the tile is the common case along one user's frames, so a run is
// only counted when the pair changes (or the user goes missing and comes back with another pair, or at the end):
// through the ranked deltas of k_transition4 (rank = drank[(p >> s)][c - p + win], one red.shared.add.u32 of the run
// length into cnt[rank][p]), or straight into acc as a 64-bit global atomic when the delta has no rank or the tile
// count has no ranking at all (global-table regime, T > 1092, T = 1).  At the end the non-zero counters are mapped back
// through rank_delta to (p, p + delta) and added into acc with 64-bit atomics.  A counter adds at most
// kTcThreads * pairs_per_cta < 2^32 (pairs_per_cta < 2^16, host-checked).
template <typename TIN>
__global__ void __launch_bounds__(kTcThreads, 2) k_tc_count(const TIN* __restrict__ packed, const TcCountArgs a) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ uint32_t s_oor;
  const uint32_t tid = threadIdx.x;
  for (int g = 0; g < a.G; ++g) {
    if (a.k[g].cnt_off < 0) continue;
    uint32_t* cnt = reinterpret_cast<uint32_t*>(smem + a.k[g].cnt_off);
    for (uint32_t i = tid; i < (uint32_t)kT4Ranks * a.k[g].T; i += blockDim.x) cnt[i] = 0u;
  }
  if (tid == 0) s_oor = 0u;
  __syncthreads();
  const uint32_t sbase = smem_u32(smem);
  const int64_t u = (int64_t)blockIdx.x * kTcThreads + tid;
  const int64_t r0 = (int64_t)blockIdx.y * a.pairs_per_cta;
  const int64_t r1 = min(r0 + a.pairs_per_cta, a.F - 1);  // last frame of the run
  const float Wf = (float)a.W, Hf = (float)a.H;
  bool oor = false;
  if (u < a.U && r0 < r1) {
    // per tile count: st = (previous tile << 16) | length of the pending run (<= pairs_per_cta < 2^16), pend = its pair
    uint32_t st[kTcGroup], pend[kTcGroup];
#pragma unroll
    for (int g = 0; g < kTcGroup; ++g) {
      st[g] = kTcNone << 16;
      pend[g] = 0u;
    }
    auto flush = [&](const TcCountArgs::Tc& t, uint32_t key, uint32_t n) {
      const uint32_t p = key >> 16, c = key & 0xFFFFu;
      if (t.cnt_off >= 0) {
        const uint32_t Lc = 2u * (uint32_t)t.win + 1u;
        const uint32_t dw = min(c - p + (uint32_t)t.win, Lc);  // deltas outside the window land on the last entry
        const uint32_t e = __ldg(t.drank + (p >> t.band_shift) * (Lc + 1u) + dw);
        if (e != kT4Unranked16) {
          asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(sbase + (uint32_t)t.cnt_off + e + (p << 2)), "r"(n) : "memory");
          return;
        }
      }
      atomicAdd(a.acc + t.acc_off + (int64_t)p * t.T + c, (unsigned long long)n);
    };
    auto visit = [&](const TIN mu, const TIN mv) {
      int cell;
      if (decode_cell(mu, mv, Wf, Hf, a.W, a.H, cell) == kOutOfRange) oor = true;
#pragma unroll
      for (int g = 0; g < kTcGroup; ++g) {
        if (g < a.G) {
          const TcCountArgs::Tc& t = a.k[g];
          const uint32_t c = cell < 0 ? kTcNone : (t.lut8 ? (uint32_t)__ldg(t.lut8 + cell) : (uint32_t)__ldg(t.lut + cell));
          const uint32_t p = st[g] >> 16;
          uint32_t run = st[g] & 0xFFFFu;
          if (p != kTcNone && c != kTcNone) {
            const uint32_t key = (p << 16) | c;
            if (key == pend[g]) {
              ++run;
            } else {
              if (run) flush(t, pend[g], run);
              pend[g] = key;
              run = 1u;
            }
          }
          st[g] = (c << 16) | run;
        }
      }
    };
    const int64_t stride = a.U * 3;
    const TIN* __restrict__ src = packed + r0 * stride + u * 3 + 1;  // the next frame to load
    constexpr int kDepth = 32 / (int)sizeof(TIN);  // frames in flight: 8 (float), 4 (double)
    const int n = (int)(r1 - r0) + 1;              // frames of the run
    TIN bu[kDepth], bv[kDepth];
#pragma unroll
    for (int j = 0; j < kDepth; ++j) {
      if (j < n) {
        bu[j] = __ldg(src);
        bv[j] = __ldg(src + 1);
        src += stride;
      }
    }
    for (int f = 0; f < n; f += kDepth) {
#pragma unroll
      for (int j = 0; j < kDepth; ++j) {
        if (f + j < n) {
          const TIN mu = bu[j], mv = bv[j];
          if (f + j + kDepth < n) {
            bu[j] = __ldg(src);
            bv[j] = __ldg(src + 1);
            src += stride;
          }
          visit(mu, mv);
        }
      }
    }
#pragma unroll
    for (int g = 0; g < kTcGroup; ++g)
      if (g < a.G && (st[g] & 0xFFFFu)) flush(a.k[g], pend[g], st[g] & 0xFFFFu);
  }
  if (oor) s_oor = 1u;
  __syncthreads();
  if (tid == 0 && s_oor) atomicOr(a.flags, (uint32_t)VET_FLAG_OUT_OF_RANGE);
  for (int g = 0; g < a.G; ++g) {
    const TcCountArgs::Tc& t = a.k[g];
    if (t.cnt_off < 0) continue;
    const uint32_t* cnt = reinterpret_cast<const uint32_t*>(smem + t.cnt_off);
    const uint32_t T = (uint32_t)t.T;
    for (uint32_t i = tid; i < (uint32_t)kT4Ranks * T; i += blockDim.x) {
      const uint32_t n = cnt[i];
      if (n) {
        const uint32_t rank = i / T, p = i - rank * T;
        const int c = (int)p + __ldg(t.rank_delta + (p >> t.band_shift) * kT4Ranks + rank);
        atomicAdd(a.acc + t.acc_off + (int64_t)p * T + c, (unsigned long long)n);
      }
    }
  }
}

struct TcEntropyArgs {
  int K = 0;
  int T[kMaxTileCounts] = {};
  int64_t acc_off[kMaxTileCounts] = {};
  int row_off[kMaxTileCounts + 1] = {};  // first row of tile count k in the row scratch (sum_j<k T_j)
  const int64_t* acc = nullptr;
  long long* row_n = nullptr;            // [sum T] n_p
  double* row_t = nullptr;               // [sum T] sum_c n_pc log2(n_pc / n_p)
  double* entropy = nullptr;
  double* per_k = nullptr;               // [K] or null
  int64_t* pairs = nullptr;              // [1] N or null
};

// One warp per row p of one tile count: the exact int64 row sum n_p (lane = c mod 32, butterfly), then the fp64 terms
// sum_c n_pc log2(n_pc / n_p) in the same order.
__global__ void __launch_bounds__(256) k_tc_rows(const TcEntropyArgs a) {
  const int lane = threadIdx.x & 31;
  const int row = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (row >= a.row_off[a.K]) return;
  int k = 0;
  while (row >= a.row_off[k + 1]) ++k;
  const int T = a.T[k], p = row - a.row_off[k];
  const int64_t* r = a.acc + a.acc_off[k] + (int64_t)p * T;
  unsigned long long n = 0;
  for (int c = lane; c < T; c += 32) n += (unsigned long long)r[c];
  n = warp_sum(n);
  double t = 0.0;
  if (n) {
    const double np = (double)(long long)n;
    for (int c = lane; c < T; c += 32) {
      const long long v = r[c];
      if (v) t = fma((double)v, log2((double)v / np), t);
    }
    t = warp_sum(t);
  }
  if (lane == 0) {
    a.row_n[row] = (long long)n;
    a.row_t[row] = t;
  }
}

// One warp per tile count over its rows in a fixed order (lane = p mod 32, butterfly): N and the sum of the row terms;
// then the sequential mean over k.
__global__ void __launch_bounds__(kMaxTileCounts * 32) k_tc_entropy(const TcEntropyArgs a) {
  __shared__ double s_e[kMaxTileCounts];
  __shared__ long long s_n;
  const int lane = threadIdx.x & 31, k = threadIdx.x >> 5;
  const double qnan = __longlong_as_double(0x7ff8000000000000LL);
  if (k < a.K) {
    unsigned long long n = 0;
    double t = 0.0;
    for (int p = a.row_off[k] + lane; p < a.row_off[k + 1]; p += 32) {
      n += (unsigned long long)a.row_n[p];
      t += a.row_t[p];
    }
    n = warp_sum(n);
    t = warp_sum(t);
    if (lane == 0) {
      const double N = (double)(long long)n, T = (double)a.T[k];
      const double mx = N > T ? log2(T) : log2(N);
      s_e[k] = n ? (-t / N) / mx : qnan;
      if (k == 0) s_n = (long long)n;
      if (a.per_k) a.per_k[k] = s_e[k];
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double mean = 0.0;
    for (int j = 0; j < a.K; ++j) mean = mean + s_e[j];
    a.entropy[0] = mean / (double)a.K;
    if (a.pairs) a.pairs[0] = s_n;
  }
}

}  // namespace vet
