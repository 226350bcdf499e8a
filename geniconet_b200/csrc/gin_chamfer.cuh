// Chamfer distance between two batched point sets: one nearest neighbour per point, both directions, and the exact gradient.
//
// Forward (nn_kernel): brute force on the fp32 CUDA cores.  The cross term x.y has K = 3, which a tensor-core MMA would pad to
// 8 or 16, and at level 5 the squared point spacing (~4e-4) is of the size of a TF32 / 16-bit rounding of x.y: only fp32 can pick
// the neighbour.  A candidate is selected by the expanded score |y|^2 - 2 x.y (|x|^2 is common to all candidates of a query).
// A tile of candidates is staged in shared memory as PAIRS (x_j x_j+1 | y_j y_j+1 | z_j z_j+1 | n_j n_j+1, n = |y|^2), so one
// packed fma.rn.f32x2 (FFMA2) scores two candidates and fminf(best, fminf(a, b)) folds both into the running minimum in one
// FMNMX3: 3 FFMA2 + 1 FMNMX3 per two candidates per query.  Each thread owns kQ queries so that every shared-memory read serves
// kQ queries.  Only the minimum is tracked in the hot loop, plus, per chunk of kChunk candidates, which chunk last lowered it; at
// the end of a tile that one chunk is re-scanned for the index (same instructions, so the score found again is bit-identical; the
// lowest index of equal scores wins).  Re-scanning every improving chunk at once would cost more than the hot loop itself: early
// in a scan nearly every chunk improves some query of a warp.  The reported distance is recomputed in difference form (x - y)^2
// for the chosen index -- the expanded form cancels badly near the surface.
//
// The candidate range is split across CTAs (grid.y) when B * N alone cannot fill the GPU (latent fitting: B = 1, M ~ 1e5);
// splits combine with one 64-bit atomicMin per (query, split) on (distance bits << 32 | index), as gin_dist.cuh does: the
// smallest distance and, among equal distances, the lowest index, whatever the order the CTAs finish in.
//
// Backward: dx_i = 2 g_xy_i (x_i - y_idx_xy(i))  +  sum_{j : idx_yx(j) = i} 2 g_yx_j (x_i - y_j), symmetrically for dy.  The first
// term is a gather.  The second is a scatter, summed without floating-point atomics in exact int64 fixed point (gin_fixed_scatter.cuh):
// scatter_stats_kernel is its first pass, scatter_sum_kernel its second, and finish_kernel reads the sums back.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "gin_fixed_scatter.cuh"

namespace gin {
namespace chamfer {

constexpr int kThreads = 128;
constexpr int kQ = 8;                          // queries per thread
constexpr int kQueries = kThreads * kQ;        // queries per CTA
constexpr int kTile = 2048;                    // candidates staged per pass: 1024 pairs * 32 B = 32 KB of shared memory
constexpr int kChunk = 32;                     // candidates per index-recovery chunk (16 pairs)

struct Pts {                                   // element (b, i, c) at p[b*sb + i*sn + c*sc]
  const float* p;
  long long sb, sn, sc;
  __device__ __forceinline__ float at(int b, int i, int c) const { return __ldg(p + b * sb + i * sn + c * sc); }
};

__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  unsigned long long d;
  const unsigned long long ua = *reinterpret_cast<unsigned long long*>(&a), ub = *reinterpret_cast<unsigned long long*>(&b),
                           uc = *reinterpret_cast<unsigned long long*>(&c);
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(ua), "l"(ub), "l"(uc));
  return *reinterpret_cast<float2*>(&d);
}

// score of the candidate pair (A = x0 x1 y0 y1, C = z0 z1 n0 n1) for the query with coefficients (-2qx, -2qy, -2qz)
__device__ __forceinline__ float2 score2(const float4& A, const float4& C, float2 cx, float2 cy, float2 cz) {
  float2 s = ffma2(cx, make_float2(A.x, A.y), make_float2(C.z, C.w));
  s = ffma2(cy, make_float2(A.z, A.w), s);
  return ffma2(cz, make_float2(C.x, C.y), s);
}

// best[b][i] (i < Nq) must be preset to all ones (cudaMemsetAsync 0xFF).  grid = (ceil(Nq / kQueries), splits, B).
__global__ void __launch_bounds__(kThreads) nn_kernel(Pts q, Pts c, int Nq, int Nc, int split_len, unsigned long long* __restrict__ best) {
  __shared__ float4 tile[kTile];               // pair p: tile[2p] = x0 x1 y0 y1, tile[2p+1] = z0 z1 n0 n1
  const int b = blockIdx.z;
  const int c0 = blockIdx.y * split_len, c1 = min(Nc, c0 + split_len);
  float2 cx[kQ], cy[kQ], cz[kQ];
  float bs[kQ];
  int bi[kQ];
#pragma unroll
  for (int k = 0; k < kQ; ++k) {
    const int i = min(blockIdx.x * kQueries + k * kThreads + (int)threadIdx.x, Nq - 1);
    const float qx = -2.f * q.at(b, i, 0), qy = -2.f * q.at(b, i, 1), qz = -2.f * q.at(b, i, 2);
    cx[k] = make_float2(qx, qx); cy[k] = make_float2(qy, qy); cz[k] = make_float2(qz, qz);
    bs[k] = __int_as_float(0x7f800000); bi[k] = c0;
  }
  for (int t0 = c0; t0 < c1; t0 += kTile) {
    const int nt = min(kTile, c1 - t0);
    __syncthreads();
    for (int p = threadIdx.x; p < kTile / 2; p += kThreads) {     // strided gather; the padding scores +inf
      float v[2][4];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int j = 2 * p + h;
        if (j < nt) {
          const float x = c.at(b, t0 + j, 0), y = c.at(b, t0 + j, 1), z = c.at(b, t0 + j, 2);
          v[h][0] = x; v[h][1] = y; v[h][2] = z; v[h][3] = x * x + y * y + z * z;
        } else {
          v[h][0] = v[h][1] = v[h][2] = 0.f; v[h][3] = __int_as_float(0x7f800000);
        }
      }
      tile[2 * p] = make_float4(v[0][0], v[1][0], v[0][1], v[1][1]);
      tile[2 * p + 1] = make_float4(v[0][2], v[1][2], v[0][3], v[1][3]);
    }
    __syncthreads();
    const int nchunks = (nt + kChunk - 1) / kChunk;
    int bc[kQ];                                    // chunk of this tile that last lowered the running minimum, -1: none
#pragma unroll
    for (int k = 0; k < kQ; ++k) bc[k] = -1;
    for (int ch = 0; ch < nchunks; ++ch) {
      const float4* tp = tile + ch * kChunk;       // kChunk / 2 pairs of 2 float4
      float old[kQ];
#pragma unroll
      for (int k = 0; k < kQ; ++k) old[k] = bs[k];
#pragma unroll 4
      for (int p = 0; p < kChunk / 2; ++p) {
        const float4 A = tp[2 * p], C = tp[2 * p + 1];
#pragma unroll
        for (int k = 0; k < kQ; ++k) {
          const float2 s = score2(A, C, cx[k], cy[k], cz[k]);
          bs[k] = fminf(bs[k], fminf(s.x, s.y));
        }
      }
#pragma unroll
      for (int k = 0; k < kQ; ++k) bc[k] = bs[k] < old[k] ? ch : bc[k];
    }
    // Improvements are strict, so the last chunk that lowered the minimum holds its first index: one re-scan per tile and query.
#pragma unroll
    for (int k = 0; k < kQ; ++k) {
      if (bc[k] >= 0) {
        const float4* tp = tile + bc[k] * kChunk;
        int f = kChunk;
#pragma unroll 1
        for (int p = 0; p < kChunk / 2; ++p) {
          const float2 s = score2(tp[2 * p], tp[2 * p + 1], cx[k], cy[k], cz[k]);
          if (s.x == bs[k]) { f = 2 * p; break; }
          if (s.y == bs[k]) { f = 2 * p + 1; break; }
        }
        bi[k] = t0 + bc[k] * kChunk + f;
      }
    }
  }
#pragma unroll
  for (int k = 0; k < kQ; ++k) {
    const int i = blockIdx.x * kQueries + k * kThreads + (int)threadIdx.x;
    if (i < Nq) {
      const int j = min(bi[k], c1 - 1);
      const float dx = q.at(b, i, 0) - c.at(b, j, 0), dy = q.at(b, i, 1) - c.at(b, j, 1), dz = q.at(b, i, 2) - c.at(b, j, 2);
      const float d = dx * dx + dy * dy + dz * dz;
      atomicMin(best + (long long)b * Nq + i, ((unsigned long long)__float_as_uint(d) << 32) | (unsigned)j);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------- backward
// Scatter workspace, per receiving point r of one side: a fixsum::Acc (32 B), zeroed.
using fixsum::Acc;

// term of entry e (a point of the other side, whose nearest point on this side is r = idx[e]): 2 g_e (S_r - E_e)
__device__ __forceinline__ void scatter_term(const Pts& S, const Pts& E, int b, int e, int r, float g, float t[3]) {
#pragma unroll
  for (int k = 0; k < 3; ++k) t[k] = 2.f * g * (S.at(b, r, k) - E.at(b, e, k));
}

__global__ void scatter_stats_kernel(Pts S, Pts E, const int32_t* __restrict__ idx, const float* __restrict__ g, Acc* __restrict__ acc,
                                     int Ns, int Ne, long long n) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int b = (int)(t / Ne), e = (int)(t - (long long)b * Ne);
  const int r = idx[t];
  float v[3];
  scatter_term(S, E, b, e, r, g[t], v);
  fixsum::note(acc + (long long)b * Ns + r, v);
}

__global__ void scatter_sum_kernel(Pts S, Pts E, const int32_t* __restrict__ idx, const float* __restrict__ g, Acc* __restrict__ acc,
                                   int Ns, int Ne, long long n) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int b = (int)(t / Ne), e = (int)(t - (long long)b * Ne);
  const int r = idx[t];
  float v[3];
  scatter_term(S, E, b, e, r, g[t], v);
  fixsum::add(acc + (long long)b * Ns + r, v);
}

// out[b][d][3] = 2 g_d (D_d - O_idx(d))  (when g != NULL)  +  the fixed-point scatter sum of d (when acc != NULL)
__global__ void finish_kernel(Pts D, Pts O, const int32_t* __restrict__ idx, const float* __restrict__ g, const Acc* __restrict__ acc,
                              float* __restrict__ out, int Nd, long long n) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int b = (int)(t / Nd), d = (int)(t - (long long)b * Nd);
  float v[3] = {0.f, 0.f, 0.f};
  if (g) {
    const int o = idx[t];
    const float gd = g[t];
#pragma unroll
    for (int k = 0; k < 3; ++k) v[k] = 2.f * gd * (D.at(b, d, k) - O.at(b, o, k));
  }
  if (acc) fixsum::read(acc[t], v);
#pragma unroll
  for (int k = 0; k < 3; ++k) out[t * 3 + k] = v[k];
}

}  // namespace chamfer
}  // namespace gin
