// Per-viewer exploration entropy: compute_spatial_entropy (EU:147-211) applied to ONE user's samples over the frames
// of a video instead of one frame's samples over the users, averaged over the tile counts like SA:142-156.
//
// Semantics.  For user u and tile count k let S_u be the frames where the user's sample is present (NaN 2dmu / 2dmv =
// missing, as in vet_spatial).  hist_k[u,t] = sum over f in S_u of w_k(cell(f,u), t): the FOV weight of EU:108-144 on
// weighted handles, 1.0 on the nearest tile on unweighted ones.  per_k[k,u] is the normalised entropy of that row with
// the rule of EU:201-209 (weighted or total > T: divide by log2 T, else by log2 total; one present sample unweighted
// and T == 1 give NaN like the reference).  entropy[u] is the sequential mean of per_k[:,u] over k.  A user with no
// present sample gets entropy NaN, frames 0 and a zero histogram row where the reference would raise "Empty vector
// dictionary": one absent viewer, or a rank that holds none of a viewer's samples, must not fail a whole report.
// A frame without any present user is normal here and raises no flag; out-of-range coordinates set
// VET_FLAG_OUT_OF_RANGE.
//
// Exactness.  The histogram is accumulated as exact integers: weights as q = rint(w * 2^b) (a positive weight below
// half a quantum counts one quantum, the rule of build_i8_tables, so every row keeps the FP64 support), counts as
// plain integers (b = 0 on unweighted handles).  b = 62 - ceil(log2 total_frames) for the GLOBAL frame count of the
// video: w <= 1 keeps every sum below 2^62, and every call, batch and rank of one video uses the same scale, so
// batched, frame-permuted and frame-sharded accumulations are bit-identical to one call.
//
// acc is [U][S + 1] int64, user-major: S = sum_k T_k columns (tile counts concatenated in k order), column S = present
// samples.  k_user_hist adds a frame range into it; k_user_entropy turns finished rows into entropies.
#pragma once
#include <type_traits>

#include "vet_common.cuh"
#include "vet_stream.cuh"

namespace vet {

struct UserHistArgs {
  int64_t F = 0, U = 0;  // frames of this call, users
  int W = 0, H = 0;
  int S = 0;             // columns of the histogram part of a row
  int K = 0;
  int Ub = 0;            // users per CTA
  int Fb = 0;            // frames staged per step (a multiple of kUserDepth)
  int off[kMaxTileCounts] = {};              // first column of tile count k
  const uint16_t* lut[kMaxTileCounts] = {};  // unweighted: cell -> nearest tile of tile count k
  const uint32_t* row_ptr = nullptr;         // weighted: [C + 1] entries of every cell, all tile counts
  const uint32_t* ent_col = nullptr;         // column (off_k + tile) of every entry
  const long long* ent_q = nullptr;          // quantised weight rint(w * 2^b) of every entry (k_user_quantise)
  int64_t* acc = nullptr;
  uint32_t* flags = nullptr;
};

constexpr int kUserThreads = 512;    // 16 warps; two CTAs per SM
constexpr int kUserDepth = 8;        // weighted: samples whose entries a warp loads before it adds them
constexpr int kUserStageLoads = 4;   // staged samples a thread loads before it decodes them

// Shared-memory bytes of one CTA: the users' rows (int64 weighted, uint32 unweighted -- a CTA adds at most F < 2^31
// counts to a column) and the staged samples (weighted: the entry range of each sample's cell; unweighted: its cell).
__host__ __device__ inline size_t user_hist_row_bytes(int S, bool weighted) { return (size_t)(S + 1) * (weighted ? 8 : 4); }
__host__ __device__ inline size_t user_hist_smem(int S, int Ub, int Fb, bool weighted) {
  const size_t rows = ((size_t)Ub * user_hist_row_bytes(S, weighted) + 15) & ~(size_t)15;
  return rows + (size_t)Fb * Ub * (weighted ? 8 : 4);
}

// q = rint(w * 2^b) of every entry, a positive weight below half a quantum raised to one quantum (the rule of
// build_i8_tables: every row keeps the FP64 support).  Run once per (handle, b), not per sample.
__global__ void k_user_quantise(const double* __restrict__ w, uint64_t n, double scale, long long* __restrict__ q) {
  for (uint64_t j = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; j < n; j += (uint64_t)gridDim.x * blockDim.x)
    q[j] = max(__double2ll_rn(__dmul_rn(w[j], scale)), 1ll);
}

// A CTA owns users [blockIdx.x * Ub, +Ub) and the frames [F * y / Y, F * (y+1) / Y) of its y = blockIdx.y.  Per step it
// stages Fb frames of its users (12 * Ub contiguous bytes per frame, one frame every 12 * U bytes), decoded to cells;
// each thread issues the loads of kUserStageLoads samples before it decodes them.
// Weighted: warp w owns the users w, w + warps, ... and walks their samples in frame order; the lanes take the entries
// of the sample's cell row (distinct tiles), so no two threads ever add to the same word and no atomics are needed.
// The column and quantised weight of the entries of kUserDepth samples are loaded (independent L2 reads) before they
// are added: the adds of one sample depend on a gather from the L2-resident entry table, and that latency, not the
// shared-memory traffic, is what the warps wait for.
// Unweighted: one thread per staged sample, K + 1 shared 32-bit atomic increments.
// At the end the non-zero words of the rows are added into acc with 64-bit integer atomics (exact, order-free).
template <typename TIN, bool WEIGHTED>
__global__ void __launch_bounds__(kUserThreads, 2) k_user_hist(const TIN* __restrict__ packed, const UserHistArgs a) {
  using Acc = typename std::conditional<WEIGHTED, unsigned long long, uint32_t>::type;
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ uint32_t s_oor;
  const int Ub = a.Ub, stride = a.S + 1;
  Acc* rows = (Acc*)smem;
  void* stage = smem + (((size_t)Ub * stride * sizeof(Acc) + 15) & ~(size_t)15);
  uint2* s_rng = (uint2*)stage;      // weighted: [Fb][Ub] entry range [j0, j1) of the cell; (1, 0) = missing sample
  int32_t* s_cell = (int32_t*)stage;  // unweighted: [Fb][Ub] cell, -1 for missing samples
  const int64_t u0 = (int64_t)blockIdx.x * Ub;
  const int nu = (int)(a.U - u0 < Ub ? a.U - u0 : (int64_t)Ub);
  const int64_t fb0 = a.F * blockIdx.y / gridDim.y, fb1 = a.F * (blockIdx.y + 1) / gridDim.y;
  const float Wf = (float)a.W, Hf = (float)a.H;
  for (int i = threadIdx.x; i < Ub * stride; i += blockDim.x) rows[i] = 0;
  if (threadIdx.x == 0) s_oor = 0;
  for (int64_t f0 = fb0; f0 < fb1; f0 += a.Fb) {
    const int nf = (int)(fb1 - f0 < a.Fb ? fb1 - f0 : (int64_t)a.Fb);
    const int n = nf * Ub;
    __syncthreads();  // the previous step's samples are consumed (first step: rows zeroed)
    for (int i0 = threadIdx.x; i0 < n; i0 += kUserStageLoads * blockDim.x) {
      TIN mu[kUserStageLoads], mv[kUserStageLoads];
#pragma unroll
      for (int s = 0; s < kUserStageLoads; ++s) {
        const int i = i0 + s * blockDim.x, f = i / Ub, u = i - f * Ub;
        mu[s] = mv[s] = TIN(NAN);
        if (i < n && u < nu) {
          const TIN* p = packed + ((f0 + f) * a.U + u0 + u) * 3;
          mu[s] = p[1];
          mv[s] = p[2];
        }
      }
      int cell[kUserStageLoads];
#pragma unroll
      for (int s = 0; s < kUserStageLoads; ++s)
        if (decode_cell(mu[s], mv[s], Wf, Hf, a.W, a.H, cell[s]) == kOutOfRange) s_oor = 1;
#pragma unroll
      for (int s = 0; s < kUserStageLoads; ++s) {
        const int i = i0 + s * blockDim.x;
        if (i >= n) continue;
        if (WEIGHTED)
          s_rng[i] = cell[s] >= 0 ? make_uint2(a.row_ptr[cell[s]], a.row_ptr[cell[s] + 1]) : make_uint2(1u, 0u);
        else
          s_cell[i] = cell[s];
      }
    }
    __syncthreads();
    if (WEIGHTED) {
      const int lane = threadIdx.x & 31, warps = blockDim.x >> 5;
      for (int u = threadIdx.x >> 5; u < nu; u += warps) {
        Acc* row = rows + (size_t)u * stride;
        uint32_t present = 0;
        for (int f = 0; f < nf; f += kUserDepth) {
          uint32_t col[kUserDepth];
          long long q[kUserDepth];
          uint2 rg[kUserDepth];
#pragma unroll
          for (int s = 0; s < kUserDepth; ++s) {
            rg[s] = f + s < nf ? s_rng[(f + s) * Ub + u] : make_uint2(1u, 0u);
            const uint32_t j = rg[s].x + lane;
            col[s] = 0xFFFFFFFFu;
            q[s] = 0;
            if (j < rg[s].y) {
              col[s] = a.ent_col[j];
              q[s] = a.ent_q[j];
            }
          }
#pragma unroll
          for (int s = 0; s < kUserDepth; ++s) {
            if (col[s] != 0xFFFFFFFFu) row[col[s]] += (Acc)q[s];
            __syncwarp();
            // rows with more than 32 entries (wide FOV, fine lattices): the rest, 32 at a time
            for (uint32_t j = rg[s].x + 32 + lane; j < rg[s].y; j += 32) row[a.ent_col[j]] += (Acc)a.ent_q[j];
            __syncwarp();
            present += rg[s].y >= rg[s].x ? 1u : 0u;  // a present sample may have no tile inside its FOV
          }
        }
        if (lane == 0) row[a.S] += present;
      }
    } else {
      for (int i0 = threadIdx.x; i0 < n; i0 += kUserStageLoads * blockDim.x) {
        int cell[kUserStageLoads];
#pragma unroll
        for (int s = 0; s < kUserStageLoads; ++s) {
          const int i = i0 + s * blockDim.x;
          cell[s] = i < n ? s_cell[i] : -1;
        }
        for (int k = 0; k < a.K; ++k) {
          uint16_t t[kUserStageLoads];
#pragma unroll
          for (int s = 0; s < kUserStageLoads; ++s) t[s] = cell[s] >= 0 ? a.lut[k][cell[s]] : 0;
#pragma unroll
          for (int s = 0; s < kUserStageLoads; ++s)
            if (cell[s] >= 0) atomicAdd(&rows[(size_t)((i0 + s * blockDim.x) % Ub) * stride + a.off[k] + t[s]], (Acc)1);
        }
#pragma unroll
        for (int s = 0; s < kUserStageLoads; ++s)
          if (cell[s] >= 0) atomicAdd(&rows[(size_t)((i0 + s * blockDim.x) % Ub) * stride + a.S], (Acc)1);
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0 && s_oor) atomicOr(a.flags, (uint32_t)VET_FLAG_OUT_OF_RANGE);
  unsigned long long* dst = (unsigned long long*)a.acc + u0 * stride;
  for (int i = threadIdx.x; i < nu * stride; i += blockDim.x) {
    const Acc v = rows[i];
    if (v) atomicAdd(dst + i, (unsigned long long)v);
  }
}

struct UserEntropyArgs {
  int64_t U = 0;
  int S = 0, K = 0, use_weight = 1, b = 0;
  int off[kMaxTileCounts] = {};
  int T[kMaxTileCounts] = {};
  const int64_t* acc = nullptr;
  double* entropy = nullptr;
  double* per_k = nullptr;  // [K, U] or null
  double* hist0 = nullptr;  // [U, T_0] or null
};

// One warp per user row: fixed point -> fp64, normalised entropy per tile count in k_entropy_rows' order (lane = t mod 32,
// fma(-p, log2 p, acc), butterfly), sequential mean over k.  The total of a row is a fixed-order fp64 sum of the same
// values.  The conversion (double)sum rounds once a sum passes 2^53 (after ~8 full-weight frames at b = 50): a relative
// 2^-53 per entry on top of the quantisation, deterministic, so results stay bit-reproducible; ldexp by -b is exact.
__global__ void __launch_bounds__(256) k_user_entropy(const UserEntropyArgs a) {
  const int lane = threadIdx.x & 31;
  const int64_t u = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (u >= a.U) return;
  const int64_t* row = a.acc + u * (int64_t)(a.S + 1);
  const bool empty = row[a.S] == 0;
  const double qnan = __longlong_as_double(0x7ff8000000000000LL);
  double mean = 0.0;
  for (int k = 0; k < a.K; ++k) {
    const int T = a.T[k];
    const int64_t* h = row + a.off[k];
    double total = 0.0;
    for (int t = lane; t < T; t += 32) total += ldexp((double)h[t], -a.b);
    total = warp_sum(total);
    double acc = 0.0;
    for (int t = lane; t < T; t += 32) {
      const double w = ldexp((double)h[t], -a.b);
      if (w > 0.0) {
        const double p = w / total;
        acc = fma(-p, log2(p), acc);
      }
      if (k == 0 && a.hist0) a.hist0[u * T + t] = w;
    }
    acc = warp_sum(acc);
    const double n = (a.use_weight || total > (double)T) ? (double)T : total;
    const double mp = 1.0 / n;
    const double mx = -n * mp * log2(mp);
    const double e = empty ? qnan : acc / mx;
    if (lane == 0 && a.per_k) a.per_k[(int64_t)k * a.U + u] = e;
    mean = mean + e;
  }
  if (lane == 0) a.entropy[u] = empty ? qnan : mean / (double)a.K;
}

// Rows by cell of the FOV weight table (the handle keeps it by tile, CSC): count, then fill through per-cell cursors.
// The order of the entries inside a row is whatever the atomics give; the sums they feed are integers.
__global__ void k_user_rows_count(const uint32_t* __restrict__ cell_idx, uint64_t nnz, uint32_t* __restrict__ count) {
  for (uint64_t j = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; j < nnz; j += (uint64_t)gridDim.x * blockDim.x)
    atomicAdd(&count[cell_idx[j]], 1u);
}
// one block per tile of one tile count
__global__ void k_user_rows_fill(const uint32_t* __restrict__ col_ptr, const uint32_t* __restrict__ cell_idx,
                                 const double* __restrict__ w_val, uint32_t col_off, uint32_t* __restrict__ cursor,
                                 uint32_t* __restrict__ ent_col, double* __restrict__ ent_w) {
  const int t = blockIdx.x;
  for (uint32_t j = col_ptr[t] + threadIdx.x; j < col_ptr[t + 1]; j += blockDim.x) {
    const uint32_t pos = atomicAdd(&cursor[cell_idx[j]], 1u);
    ent_col[pos] = col_off + (uint32_t)t;
    ent_w[pos] = w_val[j];
  }
}

}  // namespace vet
