// Handle-construction kernels: per-cell direction table, brute-force fp64 nearest
// tile (north_star stage 2), dense FOV weights, and the column-compressed weight
// tables used by the weighted histogram.
#pragma once
#include "vet_common.cuh"

namespace vet {

// Direction vector of every cell (py*(W+1)+px) -> out[C,3].
__global__ void k_cell_vectors(const double* __restrict__ cosT, const double* __restrict__ sinT,
                               const double* __restrict__ sinP, const double* __restrict__ cosP, int W, int H,
                               double* __restrict__ out) {
  const int64_t C = (int64_t)(W + 1) * (H + 1);
  for (int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; c < C; c += (int64_t)gridDim.x * blockDim.x) {
    const int py = (int)(c / (W + 1)), px = (int)(c % (W + 1));
    double x, y, z;
    cell_vector(cosT, sinT, sinP, cosP, px, py, x, y, z);
    out[3 * c + 0] = x;
    out[3 * c + 1] = y;
    out[3 * c + 2] = z;
  }
}

// Stage 1 for arbitrary sample lists: packed[n,3] -> vec[n,3] (+ cell index).
template <typename TIN>
__global__ void k_decode(const TIN* __restrict__ packed, int64_t n, int W, int H, const double* __restrict__ cosT,
                         const double* __restrict__ sinT, const double* __restrict__ sinP,
                         const double* __restrict__ cosP, double* __restrict__ vec, int32_t* __restrict__ cell_out,
                         uint32_t* __restrict__ flags) {
  const float Wf = (float)W, Hf = (float)H;
  const double qnan = __longlong_as_double(0x7ff8000000000000LL);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const TIN mu = packed[3 * i + 1], mv = packed[3 * i + 2];
    int cell;
    const int st = decode_cell(mu, mv, Wf, Hf, W, H, cell);
    double x = qnan, y = qnan, z = qnan;
    if (st == kOk) {
      cell_vector(cosT, sinT, sinP, cosP, cell % (W + 1), cell / (W + 1), x, y, z);
    } else if (st == kOutOfRange) {
      atomicOr(flags, (uint32_t)VET_FLAG_OUT_OF_RANGE);
    }
    if (vec) {
      vec[3 * i + 0] = x;
      vec[3 * i + 1] = y;
      vec[3 * i + 2] = z;
    }
    if (cell_out) cell_out[i] = cell;
  }
}

// The unit centres [3 T] of a tile set for the kernels below: copied to shared memory when the launch gave room for
// them (staged != 0, block-uniform), else read from global memory -- above ~9.6k tiles they do not fit the 227 KB of
// opt-in shared memory (unit_smem on the host).  The values and so the results are the same either way.
__device__ __forceinline__ const double* stage_units(const double* __restrict__ unit, int T, double* s_buf, int staged) {
  if (!staged) return unit;
  for (int i = threadIdx.x; i < 3 * T; i += blockDim.x) s_buf[i] = unit[i];
  __syncthreads();
  return s_buf;
}

// Stage 2: brute-force exact nearest tile.  Four lanes share one vector: lane j
// scans tiles j, j+4, ... keeping the first strict maximum of the fp64 dot
// (== first minimum of arccos, EU:104); the four partial winners are merged with
// two shuffle steps, larger dot first and lower tile index on ties.  Unit tile
// centres sit in shared memory (broadcast reads) where they fit (stage_units).
template <typename TOUT>
__global__ void k_nearest(const double* __restrict__ vec, int64_t n, const double* __restrict__ unit, int T,
                          TOUT* __restrict__ idx_out, int staged) {
  extern __shared__ double s_buf[];
  const double* s_unit = stage_units(unit, T, s_buf, staged);
  const int sub = threadIdx.x & 3;
  const int64_t per_block = blockDim.x >> 2;
  const int64_t rounds = (n + per_block - 1) / per_block;
  for (int64_t r = blockIdx.x; r < rounds; r += gridDim.x) {
    const int64_t i = r * per_block + (threadIdx.x >> 2);
    const bool live = i < n;
    double ax = 0.0, ay = 0.0, az = 0.0;
    if (live) {
      ax = vec[3 * i + 0];
      ay = vec[3 * i + 1];
      az = vec[3 * i + 2];
    }
    const bool isnan_v = (ax != ax) || (ay != ay) || (az != az);
    normalize3(ax, ay, az);
    double best = -2.0;
    int best_t = 0x7fffffff;
    for (int t = sub; t < T; t += 4) {
      const double d = clip1(dot3(ax, ay, az, s_unit[3 * t], s_unit[3 * t + 1], s_unit[3 * t + 2]));
      if (d > best) {
        best = d;
        best_t = t;
      }
    }
#pragma unroll
    for (int o = 1; o <= 2; o <<= 1) {
      const double ob = __shfl_xor_sync(kFull, best, o);
      const int ot = __shfl_xor_sync(kFull, best_t, o);
      if (ob > best || (ob == best && ot < best_t)) {
        best = ob;
        best_t = ot;
      }
    }
    if (live && sub == 0) idx_out[i] = isnan_v ? (TOUT)(-1) : (TOUT)best_t;
  }
}

// calculate_tile_weights (EU:108-144), dense rows for arbitrary vectors (unit centres as in k_nearest).
__global__ void k_tile_weights(const double* __restrict__ vec, int64_t n, const double* __restrict__ unit, int T,
                               double max_d, double pf, int use_weight, double* __restrict__ w_out, int staged) {
  extern __shared__ double s_buf[];
  const double* s_unit = stage_units(unit, T, s_buf, staged);
  // one warp per vector
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = warp; i < n; i += nwarps) {
    double ax = vec[3 * i + 0], ay = vec[3 * i + 1], az = vec[3 * i + 2];
    normalize3(ax, ay, az);
    if (use_weight) {
      for (int t = lane; t < T; t += 32) {
        const double d = dot3(ax, ay, az, s_unit[3 * t], s_unit[3 * t + 1], s_unit[3 * t + 2]);
        w_out[i * T + t] = fov_weight(d, max_d, pf);
      }
    } else {
      double best = -2.0;
      int best_t = 0x7fffffff;
      for (int t = lane; t < T; t += 32) {
        const double d = clip1(dot3(ax, ay, az, s_unit[3 * t], s_unit[3 * t + 1], s_unit[3 * t + 2]));
        if (d > best) {
          best = d;
          best_t = t;
        }
      }
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const double ob = __shfl_xor_sync(kFull, best, o);
        const int ot = __shfl_xor_sync(kFull, best_t, o);
        if (ob > best || (ob == best && ot < best_t)) {
          best = ob;
          best_t = ot;
        }
      }
      for (int t = lane; t < T; t += 32) w_out[i * T + t] = (t == best_t) ? 1.0 : 0.0;  // EU:141-142
    }
  }
}

// Column-compressed FOV weight table of one tile count: for tile t the cells with
// d(cell,t) < fov/2 (EU:133) in ascending cell order, and their weights.
// One block per tile.  FILL=false counts, FILL=true writes (same traversal).
template <bool FILL>
__global__ void k_weight_columns(const double* __restrict__ cellvec, int C, const double* __restrict__ unit, int T,
                                 double max_d, double pf, uint32_t* __restrict__ col_count,
                                 const uint32_t* __restrict__ col_ptr, uint32_t* __restrict__ cell_idx,
                                 double* __restrict__ w_val) {
  __shared__ uint32_t s_warp[32];
  __shared__ uint32_t s_base;
  const int t = blockIdx.x;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const double bx = unit[3 * t], by = unit[3 * t + 1], bz = unit[3 * t + 2];
  if (threadIdx.x == 0) s_base = FILL ? col_ptr[t] : 0u;
  __syncthreads();
  for (int c0 = 0; c0 < C; c0 += blockDim.x) {
    const int c = c0 + threadIdx.x;
    double w = 0.0;
    if (c < C) {
      double ax = cellvec[3 * c], ay = cellvec[3 * c + 1], az = cellvec[3 * c + 2];
      normalize3(ax, ay, az);
      w = fov_weight(dot3(ax, ay, az, bx, by, bz), max_d, pf);
    }
    // inclusion test is d < max_d; a weight of exactly 0 can only come from exclusion
    // (r > 0 strictly when d < max_d, and r*r underflows only below 1e-154)
    const bool in = (c < C) && (w > 0.0);
    const uint32_t m = __ballot_sync(kFull, in);
    if (lane == 0) s_warp[wid] = __popc(m);
    __syncthreads();
    uint32_t off = 0, tot = 0;
    for (int k = 0; k < nw; ++k) {
      const uint32_t v = s_warp[k];
      if (k < wid) off += v;
      tot += v;
    }
    if (FILL && in) {
      const uint32_t pos = s_base + off + __popc(m & ((1u << lane) - 1u));
      cell_idx[pos] = (uint32_t)c;
      w_val[pos] = w;
    }
    __syncthreads();
    if (threadIdx.x == 0) s_base += tot;
    __syncthreads();
  }
  if (!FILL && threadIdx.x == 0) col_count[t] = s_base;
}

}  // namespace vet
