// Per-viewer transition entropy: the conditional entropy of a user's next tile given the current one, over that
// user's own frames (vet_user_transitions).
//
// Semantics.  For user u and tile count k (T = T_k tiles) a pair is a frame f with u present in frames f and f+1
// (missing = NaN in 2dmu or 2dmv; out-of-range coordinates set VET_FLAG_OUT_OF_RANGE and count as missing, as in
// k_user_hist and k_tc_count).  p = lut_k[cell(f, u)], c = lut_k[cell(f+1, u)]; n_pc counts the user's pairs (p, c),
// n_p = sum_c n_pc, N_u = sum n_pc -- unweighted, so a weighted and an unweighted handle with the same tiles give the
// same bits.  per_k[k, u] = -sum (n_pc / N_u) log2(n_pc / n_p), normalised by log2 T if N_u > T, else by log2 N_u: the
// textbook mode (EU:321-327) of that user's pairs, or transition_counts(packed[:, u:u+1]).per_k[k].  N_u = 0 gives NaN
// (the textbook mode would divide by zero), as do N_u = 1 and T = 1 (0 / 0, as in the textbook mode).  entropy[u] is
// the sequential mean over k (SA:151-156); pairs[u] = N_u.
//
// Exactness.  A user's result depends on that user's samples only: the counts are exact integers and the entropy is
// evaluated from them in an order fixed by the user's records alone (sorted keys, contiguous record ranges per
// thread, a fixed tree), so a user's outputs are the same bits whatever other users share the call, in any user
// order, batching or sharding.
//
// k_ut_rows decodes the samples of a block of users once and writes user-major tile rows rows[k][u][f] (u16, 0xFFFF =
// missing) through shared memory; k_ut_entropy turns one user's rows into its entropies, one CTA per user.
#pragma once

#include "vet_common.cuh"
#include "vet_stream.cuh"

namespace vet {

constexpr int kUtRowsFrames = 64;   // k_ut_rows tile: frames x users, staged as cells in shared memory
constexpr int kUtRowsUsers = 32;
constexpr int kUtRowsThreads = 256;
constexpr int kUtThreads = 256;     // k_ut_entropy: three CTAs per SM
constexpr int kUtDigitBits = 4;     // radix digit of the record sort
constexpr int kUtDigits = 1 << kUtDigitBits;
constexpr uint32_t kUtCap = VET_UT_SMEM_RECORDS;  // records a CTA sorts in shared memory; more go to its global slice
constexpr uint32_t kUtNoKey = 0xFFFFFFFFu;

// Dynamic shared memory of k_ut_entropy: the [digit][thread] counters and two (key, length) record buffers.
constexpr size_t kUtSmem = (size_t)kUtDigits * kUtThreads * 4 + (size_t)4 * kUtCap * 4;

struct UtArgs {
  int64_t F = 0, U = 0;   // frames and users of the call
  int64_t u0 = 0, Ub = 0; // the user block of this launch: users [u0, u0 + Ub) of the call
  int64_t pitch = 0;      // u16 entries per row (F rounded up to 8)
  int W = 0, H = 0, K = 0;
  int T[kMaxTileCounts] = {};
  const uint8_t* lut8[kMaxTileCounts] = {};   // cell -> tile when T <= 255, else null
  const uint16_t* lut[kMaxTileCounts] = {};   // cell -> tile
  uint16_t* rows = nullptr;   // [K][Ub][pitch]
  uint32_t* spill = nullptr;  // [gridDim.x][4][F - 1] record buffers of users with more than kUtCap records
  double* entropy = nullptr;  // [U]
  double* per_k = nullptr;    // [K, U] or null
  int32_t* pairs = nullptr;   // [U] or null
  uint32_t* flags = nullptr;
};

// A CTA decodes kUtRowsFrames frames x kUtRowsUsers users: the loads of one frame are 12 B apart over the users
// (coalesced), the cells go to shared memory, and each tile count's rows leave as u16 pairs along the frames of one
// user (coalesced).  Frames past F (up to the pitch) get 0xFFFF.
template <typename TIN>
__global__ void __launch_bounds__(kUtRowsThreads) k_ut_rows(const TIN* __restrict__ packed, const UtArgs a) {
  constexpr int kPer = kUtRowsFrames * kUtRowsUsers / kUtRowsThreads;
  __shared__ int32_t s_cell[kUtRowsUsers][kUtRowsFrames + 1];
  __shared__ uint32_t s_oor;
  const int tid = threadIdx.x;
  const int64_t f0 = (int64_t)blockIdx.x * kUtRowsFrames;
  const int64_t ub0 = (int64_t)blockIdx.y * kUtRowsUsers;
  const float Wf = (float)a.W, Hf = (float)a.H;
  if (tid == 0) s_oor = 0u;
  TIN mu[kPer], mv[kPer];
#pragma unroll
  for (int j = 0; j < kPer; ++j) {
    const int i = j * kUtRowsThreads + tid, f = i / kUtRowsUsers, u = i % kUtRowsUsers;
    mu[j] = mv[j] = TIN(NAN);
    if (f0 + f < a.F && ub0 + u < a.Ub) {
      const TIN* p = packed + ((f0 + f) * a.U + a.u0 + ub0 + u) * 3;
      mu[j] = __ldg(p + 1);
      mv[j] = __ldg(p + 2);
    }
  }
  bool oor = false;
#pragma unroll
  for (int j = 0; j < kPer; ++j) {
    const int i = j * kUtRowsThreads + tid, f = i / kUtRowsUsers, u = i % kUtRowsUsers;
    int cell;
    if (decode_cell(mu[j], mv[j], Wf, Hf, a.W, a.H, cell) == kOutOfRange) oor = true;
    s_cell[u][f] = cell;
  }
  __syncthreads();
  if (oor) s_oor = 1u;
  for (int k = 0; k < a.K; ++k) {
    const uint8_t* l8 = a.lut8[k];
    const uint16_t* l16 = a.lut[k];
    uint32_t* dst = reinterpret_cast<uint32_t*>(a.rows + (int64_t)k * a.Ub * a.pitch);
    for (int i = tid; i < kUtRowsUsers * kUtRowsFrames / 2; i += kUtRowsThreads) {
      const int u = i / (kUtRowsFrames / 2), fp = i % (kUtRowsFrames / 2);
      const int64_t f = f0 + 2 * fp;
      if (ub0 + u >= a.Ub || f >= a.pitch) continue;
      uint32_t t[2];
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        const int c = s_cell[u][2 * fp + s];
        t[s] = c < 0 ? 0xFFFFu : (l8 ? (uint32_t)__ldg(l8 + c) : (uint32_t)__ldg(l16 + c));
      }
      dst[((ub0 + u) * a.pitch + f) >> 1] = t[0] | (t[1] << 16);
    }
  }
  __syncthreads();
  if (tid == 0 && s_oor) atomicOr(a.flags, (uint32_t)VET_FLAG_OUT_OF_RANGE);
}

// Exclusive prefix sum over the threads of the block (thread order); `total` receives the block's sum.  s_warp holds
// kUtThreads / 32 words.
__device__ __forceinline__ unsigned long long ut_exclusive_scan(unsigned long long v, unsigned long long* s_warp,
                                                                unsigned long long& total) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  unsigned long long x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long y = __shfl_up_sync(kFull, x, o);
    if (lane >= o) x += y;
  }
  __syncthreads();  // the previous scan's reads of s_warp are done
  if (lane == 31) s_warp[wid] = x;
  __syncthreads();
  unsigned long long off = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < kUtThreads / 32; ++w) {
    const unsigned long long s = s_warp[w];
    off += w < wid ? s : 0ull;
    tot += s;
  }
  total = tot;
  return off + x - v;
}

// One CTA per user (persistent: CTA b takes users b, b + gridDim.x, ...), the tile counts in order.  Per tile count:
//  1. Records.  Thread t walks the frame pairs [t L, (t+1) L) of the user's row; a run of one repeated pair (p, c) is
//     one record (key = p T + c, length) -- staying in the tile is the common case -- and a scan over the threads
//     places the records in frame order.  Up to kUtCap records live in shared memory, more in the CTA's slice of
//     global scratch; the same code handles both.
//  2. A stable LSD radix sort of the records by key, kUtDigitBits per pass over ceil(log2 T^2) bits: thread t owns a
//     contiguous range of records, counts its digits into cnt[digit][t], one scan in (digit, thread) order gives every
//     thread's first slot per digit, and it scatters its range in order.
//  3. The records of one p are contiguous now.  Thread t takes the p whose first record lies in its range: n_p = the
//     sum of their lengths, then per run of one key n_pc and the term n_pc log2(n_pc / n_p), added in key order;
//     the threads' sums meet in block_sum's fixed tree.  Each term is evaluated on its own: the difference
//     sum n_p log n_p - sum n_pc log n_pc would cancel for near-deterministic viewers.
__global__ void __launch_bounds__(kUtThreads, 3) k_ut_entropy(const UtArgs a) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ unsigned long long s_scan[kUtThreads / 32];
  __shared__ double s_red[32];
  uint32_t* s_cnt = reinterpret_cast<uint32_t*>(smem);  // [kUtDigits][kUtThreads]
  uint32_t* s_rec = s_cnt + kUtDigits * kUtThreads;      // [4][kUtCap]: keys A, lengths A, keys B, lengths B
  const uint32_t tid = threadIdx.x;
  const int64_t R = a.F > 1 ? a.F - 1 : 0;  // frame pairs (< 2^31, host-checked)
  const uint32_t L = (uint32_t)((R + kUtThreads - 1) / kUtThreads);
  const uint32_t b0 = (uint32_t)min((int64_t)tid * L, R), b1 = (uint32_t)min((int64_t)b0 + L, R);
  uint32_t* spill = a.spill ? a.spill + (int64_t)blockIdx.x * 4 * R : nullptr;
  const double qnan = __longlong_as_double(0x7ff8000000000000LL);
  for (int64_t u = blockIdx.x; u < a.Ub; u += gridDim.x) {
    double mean = 0.0;
    uint32_t N = 0;
    for (int k = 0; k < a.K; ++k) {
      const uint32_t T = (uint32_t)a.T[k];
      const uint16_t* __restrict__ row = a.rows + ((int64_t)k * a.Ub + u) * a.pitch;
      // 1. records
      uint32_t nrec = 0, npairs = 0;
      {
        uint32_t prev = kUtNoKey, pt = b0 < b1 ? row[b0] : 0xFFFFu;
        for (uint32_t f = b0; f < b1; ++f) {
          const uint32_t ct = row[f + 1];
          uint32_t key = kUtNoKey;
          if (pt != 0xFFFFu && ct != 0xFFFFu) {
            key = pt * T + ct;
            ++npairs;
            nrec += key != prev ? 1u : 0u;
          }
          prev = key;
          pt = ct;
        }
      }
      unsigned long long tot;
      const uint32_t rec0 = (uint32_t)ut_exclusive_scan(((unsigned long long)npairs << 32) | nrec, s_scan, tot);
      const uint32_t n = (uint32_t)tot;
      if (k == 0) N = (uint32_t)(tot >> 32);
      const bool big = n > kUtCap;
      const uint32_t cap = big ? (uint32_t)R : kUtCap;
      uint32_t* base = big ? spill : s_rec;
      uint32_t *sk = base, *sl = base + cap, *dk = base + 2 * (size_t)cap, *dl = base + 3 * (size_t)cap;
      {
        uint32_t pos = rec0, prev = kUtNoKey, cur = kUtNoKey, run = 0, pt = b0 < b1 ? row[b0] : 0xFFFFu;
        for (uint32_t f = b0; f < b1; ++f) {
          const uint32_t ct = row[f + 1];
          uint32_t key = kUtNoKey;
          if (pt != 0xFFFFu && ct != 0xFFFFu) {
            key = pt * T + ct;
            if (key == prev) {
              ++run;
            } else {
              if (run) {
                sk[pos] = cur;
                sl[pos++] = run;
              }
              cur = key;
              run = 1;
            }
          }
          prev = key;
          pt = ct;
        }
        if (run) {
          sk[pos] = cur;
          sl[pos] = run;
        }
      }
      // 2. sort by key
      const uint32_t Lr = (n + kUtThreads - 1) / kUtThreads;
      const uint32_t r0 = min(tid * Lr, n), r1 = min(r0 + Lr, n);
      const int bits = T > 1 ? 32 - __clz(T * T - 1) : 0;
      for (int shift = 0; shift < bits && n > 1; shift += kUtDigitBits) {
#pragma unroll
        for (int d = 0; d < kUtDigits; ++d) s_cnt[d * kUtThreads + tid] = 0u;
        __syncthreads();  // the records are written (first pass) or scattered (later passes)
        for (uint32_t i = r0; i < r1; ++i) ++s_cnt[((sk[i] >> shift) & (kUtDigits - 1)) * kUtThreads + tid];
        __syncthreads();
        uint32_t v[kUtDigits], local = 0;
#pragma unroll
        for (int j = 0; j < kUtDigits; ++j) {
          v[j] = s_cnt[tid * kUtDigits + j];
          local += v[j];
        }
        unsigned long long all;
        uint32_t run = (uint32_t)ut_exclusive_scan(local, s_scan, all);
#pragma unroll
        for (int j = 0; j < kUtDigits; ++j) {
          s_cnt[tid * kUtDigits + j] = run;
          run += v[j];
        }
        __syncthreads();
        for (uint32_t i = r0; i < r1; ++i) {
          const uint32_t key = sk[i];
          const uint32_t pos = s_cnt[((key >> shift) & (kUtDigits - 1)) * kUtThreads + tid]++;
          dk[pos] = key;
          dl[pos] = sl[i];
        }
        uint32_t* t0 = sk;
        sk = dk;
        dk = t0;
        t0 = sl;
        sl = dl;
        dl = t0;
      }
      __syncthreads();
      // 3. terms
      double t = 0.0;
      uint32_t h = r0;
      while (h < r1 && h > 0 && sk[h - 1] / T == sk[h] / T) ++h;  // the first p that starts in this range
      while (h < r1) {
        const uint32_t p = sk[h] / T;
        uint32_t j = h, np = 0;
        for (; j < n && sk[j] / T == p; ++j) np += sl[j];
        const double dnp = (double)np;
        for (uint32_t m = h; m < j;) {
          const uint32_t key = sk[m];
          uint32_t c = 0;
          for (; m < j && sk[m] == key; ++m) c += sl[m];
          t = fma((double)c, log2((double)c / dnp), t);
        }
        h = j;
      }
      t = block_sum(t, s_red);
      if (tid == 0) {
        const double Nd = (double)N, Td = (double)T;
        const double mx = Nd > Td ? log2(Td) : log2(Nd);
        const double e = N ? (-t / Nd) / mx : qnan;
        if (a.per_k) a.per_k[(int64_t)k * a.U + a.u0 + u] = e;
        mean = mean + e;
      }
    }
    if (tid == 0) {
      a.entropy[a.u0 + u] = mean / (double)a.K;
      if (a.pairs) a.pairs[a.u0 + u] = (int32_t)N;
    }
  }
}

}  // namespace vet
