// Fused BatchNorm(training) + ReLU + residual add + bf16 operand cast around the hex-convs -- SURVEY 8f rank 1.
//
// models.py:37-39 / 59-61 evaluate  relu(bn(conv(x)))  and  relu(bn01(conv01(.)) + bn10(conv10(.)))  with stock torch modules:
// per conv output that is a BatchNorm statistics pass, a normalise pass, a ReLU pass, an add pass and finally the bf16 cast the
// next tcgen05 conv needs -- about 26 bytes of HBM traffic per element forward and twice that backward.  Here a conv output y
// (fp32, written once by the conv epilogue) is read by
//     bn_stats      sum y, sum y^2 per channel                  (4 B / element)
//     bn_act_fwd    out = relu(y*scale + shift [+ y2*scale2 + shift2]) written ONLY as the bf16 operand copy
//                   [B*P + 2B][C] (pixels + pole-mean rows) that the next conv gathers from      (4-8 B read, 2 B written)
// and backward
//     bn_bwd_reduce sum g, sum g*yhat with g = dout * (out > 0)  (mask from the bf16 copy)       (10 B / element)
//     bn_bwd_apply  dy = scale * (g - mean(g) - yhat * mean(g*yhat)) written as the bf16 copy dgrad / wgrad read
// All reductions are two-stage (per-CTA partials, then a fixed-order fp64 final), hence deterministic.
// Thread layout everywhere: one thread = 8 consecutive channels of one row; (C/8) | 256 so a thread keeps its channels
// for every grid-stride iteration.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <cstdlib>

#include "gin_common.cuh"
#include "gin_resample.cuh"

namespace gin {
namespace bn {

constexpr int MAX_CTAS = 148 * 4;          // upper bound (sizes the partial-sum buffers); the grid actually used: bn_ctas()

struct Src {               // a [rows][C] view inside a wider row-major matrix: fp32, or fp16 (f16 != 0: conv outputs of the fused chains)
  const float* p;          // for f16 sources the pointer is reinterpreted
  long long ld;            // row stride in ELEMENTS
  int f16;
};

// pixel e (0..4) of the ring of `pole` on a level with n = 2^level: chart e, first pixel of row 0 / last pixel of row n-1
GIN_DEVINL int ring_pixel(int n, int pole, int e) { return e * n * 2 * n + (pole ? (n - 1) * 2 * n + 2 * n - 1 : 0); }

GIN_DEVINL void ld8(const float* p, float v[8]) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p + 4));
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
GIN_DEVINL void ld8_bf16(const __nv_bfloat16* p, float v[8]) {
  const uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) { const float2 f = __bfloat1622float2(h[i]); v[2 * i] = f.x; v[2 * i + 1] = f.y; }
}
GIN_DEVINL void st8_bf16(__nv_bfloat16* p, const float v[8]) {
  __nv_bfloat162 h[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
  *reinterpret_cast<uint4*>(p) = *reinterpret_cast<uint4*>(h);
}
// 8 values as a 16-byte group of forward operands (fp16 or bf16)
GIN_DEVINL void st8_op(__nv_bfloat16* p, const float v[8], int f16) {
  uint4 o;
  o.x = pack2_op(v[0], v[1], f16); o.y = pack2_op(v[2], v[3], f16); o.z = pack2_op(v[4], v[5], f16); o.w = pack2_op(v[6], v[7], f16);
  *reinterpret_cast<uint4*>(p) = o;
}
// ReLU mask from an activation copy in EITHER 16-bit format: value > 0  <=>  sign bit clear and any other bit set
GIN_DEVINL void ld8_mask(const __nv_bfloat16* p, bool m[8]) {
  const uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    m[2 * i] = (w[i] & 0x8000u) == 0 && (w[i] & 0x7fffu) != 0;
    m[2 * i + 1] = (w[i] & 0x80000000u) == 0 && (w[i] & 0x7fff0000u) != 0;
  }
}
// 8 operands of either format -> fp32
GIN_DEVINL void ld8_op(const __nv_bfloat16* p, float v[8], int f16) {
  if (!f16) { ld8_bf16(p, v); return; }
  const uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
  const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) { const float2 f = __half22float2(h[i]); v[2 * i] = f.x; v[2 * i + 1] = f.y; }
}
// 8 consecutive channels of row r of a source
GIN_DEVINL void ld8_src(const Src& s, long long r, int c, float v[8]) {
  if (!s.f16) { ld8(s.p + r * s.ld + c, v); return; }
  const uint4 u = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const __half*>(s.p) + r * s.ld + c));
  const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) { const float2 f = __half22float2(h[i]); v[2 * i] = f.x; v[2 * i + 1] = f.y; }
}
GIN_DEVINL void st8(float* p, const float v[8]) {
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}

// block-level: partial[blockIdx][k][C] = sum over this CTA's threads of s_k[8]  (k = 0, 1)
GIN_DEVINL void block_partials(const float s0[8], const float s1[8], int C, float* __restrict__ partial) {
  __shared__ float part[2][256][9];
  const int C8 = C >> 3;
#pragma unroll
  for (int k = 0; k < 8; ++k) { part[0][threadIdx.x][k] = s0[k]; part[1][threadIdx.x][k] = s1[k]; }
  __syncthreads();
  float* mine = partial + (size_t)blockIdx.x * 2 * C;
  for (int i = threadIdx.x; i < 2 * C; i += 256) {
    const int w = i / C, c = i - w * C, g = c >> 3, k = c & 7;
    float acc = 0.f;
    for (int t = g; t < 256; t += C8) acc += part[w][t][k];
    mine[i] = acc;
  }
}

// final[k][c] (double) = sum_b partial[b][k][c] for the 8 channels of this CTA; returned to threads 0..7 (k = 0) and 8..15 (k = 1)
GIN_DEVINL double final_sum(const float* __restrict__ partial, int nblocks, int C, long long ld = 0) {
  if (ld == 0) ld = C;                                         // row stride of the partial-sum rows (a column slice of wider rows)
  __shared__ double red[16][17];
  const int j = threadIdx.x & 15, rg = threadIdx.x >> 4;       // j: (k, channel-in-8), rg: 16 row groups
  const int k = j >> 3, c = blockIdx.x * 8 + (j & 7);
  double acc = 0.0;
  if (c < C) {
    // every load of this thread is issued before the first add (the kernel is pure load latency otherwise)
    float v[(MAX_CTAS + 15) / 16];
#pragma unroll
    for (int i = 0; i < (MAX_CTAS + 15) / 16; ++i) {
      const int b = rg + 16 * i;
      v[i] = b < nblocks ? __ldg(partial + ((size_t)b * 2 + k) * ld + c) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < (MAX_CTAS + 15) / 16; ++i) acc += (double)v[i];
  }
  red[rg][j] = acc;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x < 16)
#pragma unroll
    for (int r = 0; r < 16; ++r) t += red[r][threadIdx.x];
  return t;
}

// ------------------------------------------------------------------------------------------------ forward statistics
__global__ void __launch_bounds__(256) stats_kernel(Src y, long long rows, int C, float* __restrict__ partial) {
  GIN_PDL_SYNC();
  const int C8 = C >> 3;
  const long long n = rows * C8;
  float s0[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, s1[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += gridDim.x * 256LL) {
    const long long r = i / C8;
    const int c = (int)(i - r * C8) * 8;
    float v[8];
    ld8_src(y, r, c, v);
#pragma unroll
    for (int k = 0; k < 8; ++k) { s0[k] += v[k]; s1[k] = fmaf(v[k], v[k], s1[k]); }
  }
  block_partials(s0, s1, C, partial);
}

// One BatchNorm whose statistics a final kernel writes.  The pair kernels take two: the sibling convolutions of a residual block
// run as one GEMM, so their partial sums are column slices of the same rows.
struct StatsTarget {
  const float* partial;      // first column of this BatchNorm inside the partial-sum rows
  const float* gamma;
  const float* beta;
  float* running_mean;
  float* running_var;
  long long* num_batches_tracked;
  float* stat;
  float eps, momentum;
};

// sums[0..7] = sum y, sums[8..15] = sum y^2 of the 8 channels of block blk (shared memory, written before a __syncthreads) ->
// stat[0..3][C] = mean, invstd, scale = gamma*invstd, shift = beta - mean*scale; running statistics updated as torch does
// (momentum, unbiased variance over `rows`).
GIN_DEVINL void stats_write(const double* sums, int blk, long long rows, int C, const StatsTarget& t) {
  const int c = blk * 8 + threadIdx.x;
  if (t.num_batches_tracked && blk == 0 && threadIdx.x == 0) *t.num_batches_tracked += 1;
  if (threadIdx.x < 8 && c < C) {
    const double mean = sums[threadIdx.x] / (double)rows;
    double var = sums[8 + threadIdx.x] / (double)rows - mean * mean;
    if (var < 0.0) var = 0.0;
    const float invstd = (float)(1.0 / sqrt(var + (double)t.eps));
    const float g = t.gamma ? t.gamma[c] : 1.f, be = t.beta ? t.beta[c] : 0.f;
    const float scale = g * invstd;
    t.stat[c] = (float)mean; t.stat[C + c] = invstd; t.stat[2 * C + c] = scale; t.stat[3 * C + c] = be - (float)mean * scale;
    if (t.running_mean) {
      const double unbiased = rows > 1 ? var * (double)rows / (double)(rows - 1) : var;
      t.running_mean[c] = (1.f - t.momentum) * t.running_mean[c] + t.momentum * (float)mean;
      t.running_var[c] = (1.f - t.momentum) * t.running_var[c] + t.momentum * (float)unbiased;
    }
  }
}

// stats_write from per-CTA partials.  grid = C/8, block = 256.
__global__ void __launch_bounds__(256)
stats_final_kernel(const float* __restrict__ partial, int nblocks, long long rows, int C, const float* __restrict__ gamma,
                   const float* __restrict__ beta, float eps, float momentum, float* __restrict__ running_mean, float* __restrict__ running_var,
                   long long* __restrict__ num_batches_tracked, float* __restrict__ stat, long long ld) {
  GIN_PDL_SYNC();
  __shared__ double sums[16];
  const double t = final_sum(partial, nblocks, C, ld);
  if (threadIdx.x < 16) sums[threadIdx.x] = t;
  __syncthreads();
  stats_write(sums, blockIdx.x, rows, C, StatsTarget{partial, gamma, beta, running_mean, running_var, num_batches_tracked, stat, eps, momentum});
}

// Two BatchNorms from column slices of the SAME partial-sum rows in one launch: blockIdx.x < C/8 -> the first, else the second.
__global__ void __launch_bounds__(256)
stats_final2_kernel(StatsTarget a, StatsTarget b, int nblocks, long long rows, int C, long long ld) {
  GIN_PDL_SYNC();
  __shared__ double sums[16];
  const int nb = C / 8;
  const bool second = (int)blockIdx.x >= nb;
  const StatsTarget& t = second ? b : a;
  const int blk = second ? blockIdx.x - nb : blockIdx.x;
  // final_sum indexes channels by blockIdx.x: shift the base pointer instead
  const double s = final_sum(t.partial - (second ? (size_t)nb * 8 : 0), nblocks, C + (second ? nb * 8 : 0), ld);
  if (threadIdx.x < 16) sums[threadIdx.x] = s;
  __syncthreads();
  stats_write(sums, blk, rows, C, t);
}

// ------------------------------------------------------------------------------------------------ synchronised BatchNorm
// A BatchNorm synchronised over W ranks splits each final above in two: this rank's fp64 totals go into a record, the records of
// every rank are all-gathered (a copy), and a final kernel sums them in rank order 0..W-1.  Every rank therefore computes the
// same bits, and with W = 1 the sum is the rank's own total: bit for bit the unsynchronised final.
//   forward record of one BatchNorm: [sum y [C] | sum y^2 [C] | rows], 2C + 1 doubles; of a sibling pair: A's record, then B's
//   backward record of one BatchNorm: [sum g [C] | sum g*yhat [C] | rows]; of a pair: A's record, then B's (sum g is the same in both)
GIN_DEVINL double rank_sum(const double* __restrict__ recs, int world, long long stride, long long off) {
  double s = recs[off];
  for (int w = 1; w < world; ++w) s += recs[(long long)w * stride + off];
  return s;
}

// forward records from per-CTA partials (final_sum's order); grid = nbn * C/8 (nbn = 1, or 2 for a pair: partB, the second record)
__global__ void __launch_bounds__(256)
stats_total_kernel(const float* __restrict__ partA, const float* __restrict__ partB, int nblocks, long long rows, int C, long long ld,
                   double* __restrict__ rec) {
  GIN_PDL_SYNC();
  const int nb = C / 8;
  const bool second = (int)blockIdx.x >= nb;
  const int blk = second ? blockIdx.x - nb : blockIdx.x;
  const double s = second ? final_sum(partB - (size_t)nb * 8, nblocks, C + nb * 8, ld) : final_sum(partA, nblocks, C, ld);
  double* r = rec + (second ? 2LL * C + 1 : 0);
  const int k = threadIdx.x >> 3, c = blk * 8 + (threadIdx.x & 7);
  if (threadIdx.x < 16 && c < C) r[(long long)k * C + c] = s;
  if (blk == 0 && threadIdx.x == 0) r[2LL * C] = (double)rows;
}

// stats_write from the gathered forward records recs[world][nbn * (2C + 1)] with the global row count; grid = nbn * C/8
__global__ void __launch_bounds__(256) stats_sync_final_kernel(const double* __restrict__ recs, int world, int nbn, int C, StatsTarget a, StatsTarget b) {
  GIN_PDL_SYNC();
  __shared__ double sums[16];
  __shared__ long long rows;
  const int nb = C / 8;
  const bool second = (int)blockIdx.x >= nb;
  const int blk = second ? blockIdx.x - nb : blockIdx.x;
  const long long stride = (long long)nbn * (2 * C + 1), base = second ? 2LL * C + 1 : 0;
  const int k = threadIdx.x >> 3, c = blk * 8 + (threadIdx.x & 7);
  if (threadIdx.x < 16) sums[threadIdx.x] = c < C ? rank_sum(recs, world, stride, base + (long long)k * C + c) : 0.0;
  if (threadIdx.x == 16) rows = (long long)rank_sum(recs, world, stride, base + 2LL * C);
  __syncthreads();
  stats_write(sums, blk, rows, C, second ? b : a);
}

// ------------------------------------------------------------------------------------------------ forward apply
// out[row, :] = act(y1*scale1 + shift1 [+ y2*scale2 + shift2]) -> bf16 rows [0, rows) of out_b, per-sample pole means
// (mean over the pole's five ring pixels of the fp32 values) in rows [rows, rows + 2B), optional fp32 copy out_f.
template <bool TWO>
GIN_DEVINL void apply_row(const Src& y1, const Src& y2, long long r, int c, const float sc1[8], const float sh1[8], const float sc2[8],
                          const float sh2[8], int relu, float o[8]) {
  float v[8];
  ld8_src(y1, r, c, v);
#pragma unroll
  for (int k = 0; k < 8; ++k) o[k] = fmaf(v[k], sc1[k], sh1[k]);
  if (TWO) {
    ld8_src(y2, r, c, v);
#pragma unroll
    for (int k = 0; k < 8; ++k) o[k] += fmaf(v[k], sc2[k], sh2[k]);
  }
  if (relu) {
#pragma unroll
    for (int k = 0; k < 8; ++k) o[k] = fmaxf(o[k], 0.f);
  }
}

template <bool TWO>
__global__ void __launch_bounds__(256)
act_fwd_anyc_kernel(Src y1, const float* __restrict__ stat1, Src y2, const float* __restrict__ stat2, int relu, __nv_bfloat16* __restrict__ out_b,
               float* __restrict__ out_f, int nlat, int B, int P, int C, int f16, __nv_bfloat16* __restrict__ out_w) {
  GIN_PDL_SYNC();
  const int C8 = C >> 3;
  const long long rows = (long long)B * P, n_main = rows * C8, n_all = n_main + 2LL * B * C8;
  const int c = (int)(threadIdx.x % C8) * 8;            // fixed for this thread: C8 | 256 | grid stride
  float sc1[8], sh1[8], sc2[8], sh2[8];
  ld8(stat1 + 2 * C + c, sc1); ld8(stat1 + 3 * C + c, sh1);
  if (TWO) { ld8(stat2 + 2 * C + c, sc2); ld8(stat2 + 3 * C + c, sh2); }
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n_all; i += gridDim.x * 256LL) {
    float o[8];
    if (i < n_main) {
      const long long r = i / C8;
      apply_row<TWO>(y1, y2, r, c, sc1, sh1, sc2, sh2, relu, o);
      if (out_f) st8(out_f + r * C + c, o);
    } else {
      const long long j = (i - n_main) / C8;
      const int sample = (int)(j >> 1), pole = (int)(j & 1);
#pragma unroll
      for (int k = 0; k < 8; ++k) o[k] = 0.f;
      for (int e = 0; e < 5; ++e) {
        float t[8];
        apply_row<TWO>(y1, y2, (long long)sample * P + ring_pixel(nlat, pole, e), c, sc1, sh1, sc2, sh2, relu, t);
#pragma unroll
        for (int k = 0; k < 8; ++k) o[k] = fmaf(0.2f, t[k], o[k]);
      }
    }
    if (out_b) st8_op(out_b + (i / C8) * C + c, o, f16);
    if (out_w) st8_op(out_w + (i / C8) * C + c, o, 0);          // the bf16 twin wgrad reads (and the ReLU mask of the backward)
  }
}

// ------------------------------------------------------------------------------------------------ backward
// g = dout * (out > 0) (mask read from the bf16 activation copy; mask == null: no ReLU), yhat = (y - mean) * invstd
GIN_DEVINL void grad_row(const float* __restrict__ dout, long long ldg, const __nv_bfloat16* __restrict__ mask, const Src& y, long long r, int c,
                         int C, const float mean[8], const float invstd[8], float g[8], float yh[8]) {
  ld8(dout + r * ldg + c, g);
  if (mask) {
    bool m[8];
    ld8_mask(mask + r * C + c, m);
#pragma unroll
    for (int k = 0; k < 8; ++k) g[k] = m[k] ? g[k] : 0.f;
  }
  float v[8];
  ld8_src(y, r, c, v);
#pragma unroll
  for (int k = 0; k < 8; ++k) yh[k] = (v[k] - mean[k]) * invstd[k];
}

__global__ void __launch_bounds__(256)
bwd_reduce_kernel(const float* __restrict__ dout, long long ldg, const __nv_bfloat16* __restrict__ mask, Src y, const float* __restrict__ stat,
                  long long rows, int C, float* __restrict__ partial) {
  GIN_PDL_SYNC();
  const int C8 = C >> 3;
  const long long n = rows * C8;
  const int c = (int)(threadIdx.x % C8) * 8;
  float mean[8], invstd[8];
  ld8(stat + c, mean); ld8(stat + C + c, invstd);
  float s0[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, s1[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += gridDim.x * 256LL) {
    float g[8], yh[8];
    grad_row(dout, ldg, mask, y, i / C8, c, C, mean, invstd, g, yh);
#pragma unroll
    for (int k = 0; k < 8; ++k) { s0[k] += g[k]; s1[k] = fmaf(g[k], yh[k], s1[k]); }
  }
  block_partials(s0, s1, C, partial);
}

// bstat[0..3][C] = dbeta = sum g, dgamma = sum g*yhat, c1 = mean(g), c2 = mean(g*yhat).  grid = C/8.
__global__ void __launch_bounds__(256)
bwd_final_kernel(const float* __restrict__ partial, int nblocks, long long rows, int C, float* __restrict__ bstat) {
  GIN_PDL_SYNC();
  const double t = final_sum(partial, nblocks, C);
  if (threadIdx.x < 16) {
    const int k = threadIdx.x >> 3, c = blockIdx.x * 8 + (threadIdx.x & 7);
    if (c < C) { bstat[k * C + c] = (float)t; bstat[(2 + k) * C + c] = (float)(t / (double)rows); }
  }
}

// dy = scale * (g - c1 - yhat*c2) -> bf16 copy (rows + per-sample pole means of dy, row stride ldo) and/or fp32 (row stride ldf)
__global__ void __launch_bounds__(256)
bwd_apply_anyc_kernel(const float* __restrict__ dout, long long ldg, const __nv_bfloat16* __restrict__ mask, Src y, const float* __restrict__ stat,
                 const float* __restrict__ bstat, __nv_bfloat16* __restrict__ dy_b, long long ldo, float* __restrict__ dy_f, long long ldf,
                 int nlat, int B, int P, int C) {
  GIN_PDL_SYNC();
  const int C8 = C >> 3;
  const long long rows = (long long)B * P, n_main = rows * C8, n_all = n_main + (dy_b ? 2LL * B * C8 : 0);
  const int c = (int)(threadIdx.x % C8) * 8;
  float mean[8], invstd[8], scale[8], c1[8], c2[8];
  ld8(stat + c, mean); ld8(stat + C + c, invstd); ld8(stat + 2 * C + c, scale); ld8(bstat + 2 * C + c, c1); ld8(bstat + 3 * C + c, c2);
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n_all; i += gridDim.x * 256LL) {
    float o[8];
    if (i < n_main) {
      const long long r = i / C8;
      float g[8], yh[8];
      grad_row(dout, ldg, mask, y, r, c, C, mean, invstd, g, yh);
#pragma unroll
      for (int k = 0; k < 8; ++k) o[k] = scale[k] * (g[k] - c1[k] - yh[k] * c2[k]);
      if (dy_f) st8(dy_f + r * ldf + c, o);
    } else {
      const long long j = (i - n_main) / C8;
      const int sample = (int)(j >> 1), pole = (int)(j & 1);
#pragma unroll
      for (int k = 0; k < 8; ++k) o[k] = 0.f;
      for (int e = 0; e < 5; ++e) {
        float g[8], yh[8];
        grad_row(dout, ldg, mask, y, (long long)sample * P + ring_pixel(nlat, pole, e), c, C, mean, invstd, g, yh);
#pragma unroll
        for (int k = 0; k < 8; ++k) o[k] = fmaf(0.2f * scale[k], g[k] - c1[k] - yh[k] * c2[k], o[k]);
      }
    }
    if (dy_b) st8_bf16(dy_b + (i / C8) * ldo + c, o);
  }
}

// ------------------------------------------------------------------------------------------------ upsample into the operand copy
// IcoUpsampleS2S whose output exists only as the next convolution's bf16 operand copy [B*Pf + 2B][C] (fine pixels + fine pole
// means).  The source is the fp32 coarse map [B*Pc][C] (F32 = true: one rounding, like the module-wise path) or its bf16
// operand copy [B*Pc + 2B][C] (coarse pole means taken from its pole rows).
template <bool F32>
GIN_DEVINL void up_fetch_any(const void* __restrict__ xin, const int32_t* __restrict__ cring, long long sample, int B, int Pc, int code, int C, int c,
                             float v[8], int f16) {
  if (code == GIN_SRC_ZERO) {
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = 0.f;
    return;
  }
  if (F32) {
    const float* x = reinterpret_cast<const float*>(xin) + (size_t)sample * Pc * C + c;
    if (code >= 0) { ld8(x + (size_t)code * C, v); return; }
    const int pole = (-2 - code) & 1;
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = 0.f;
    for (int e = 0; e < 5; ++e) {
      float t[8];
      ld8(x + (size_t)cring[pole * 5 + e] * C, t);
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = fmaf(0.2f, t[k], v[k]);
    }
  } else {
    const __nv_bfloat16* x = reinterpret_cast<const __nv_bfloat16*>(xin);
    if (code >= 0) ld8_op(x + ((size_t)sample * Pc + code) * C + c, v, f16);
    else ld8_op(x + ((size_t)B * Pc + 2 * sample + ((-2 - code) & 1)) * C + c, v, f16);     // the coarse pole-mean row
  }
}
template <bool F32>
GIN_DEVINL void up_pixel(const int32_t* __restrict__ src, const void* __restrict__ xin, const int32_t* __restrict__ cring, long long sample, int B,
                         int Pc, int f, int C, int c, float o[8], int f16) {
  const int s0 = src[2 * f], s1 = src[2 * f + 1];
  up_fetch_any<F32>(xin, cring, sample, B, Pc, s0, C, c, o, f16);
  if (s0 != s1) {
    float t[8];
    up_fetch_any<F32>(xin, cring, sample, B, Pc, s1, C, c, t, f16);
#pragma unroll
    for (int k = 0; k < 8; ++k) o[k] = 0.5f * (o[k] + t[k]);
  }
}
// Idx: the work-item index type -- unsigned when B*(Pf+2)*C/8 < 2^31 (four 32-bit divisions per item instead of four emulated
// 64-bit ones, which made this kernel instruction-bound: ncu r02 sm throughput 47 % at 47 % of the HBM rate), else long long.
template <bool F32, typename Idx>
__global__ void __launch_bounds__(256)
upsample_bf16_kernel(const int32_t* __restrict__ plan, const void* __restrict__ xin, __nv_bfloat16* __restrict__ out, int nfine, int B, int C, int f16,
                     __nv_bfloat16* __restrict__ out_w) {
  GIN_PDL_SYNC();
  const GinUpPlanHdr* h = reinterpret_cast<const GinUpPlanHdr*>(plan);
  const int Pc = h->Pc, C8 = C >> 3;
  const Idx Pf = (Idx)h->Pf, nC8 = (Idx)C8;
  const int32_t* src = plan + h->fwd_off;
  const int32_t* cring = plan + h->ring_off;
  const Idx n_rows = (Idx)B * Pf, n_main = n_rows * nC8, n_all = n_main + (Idx)(2 * B) * nC8;
  for (Idx i = (Idx)blockIdx.x * 256 + threadIdx.x; i < n_all; i += (Idx)gridDim.x * 256) {
    const Idx row = i / nC8;
    const int c = (int)(i - row * nC8) * 8;
    float o[8];
    if (i < n_main) {
      const Idx sample = row / Pf;
      up_pixel<F32>(src, xin, cring, (long long)sample, B, Pc, (int)(row - sample * Pf), C, c, o, f16);
    } else {
      const int j = (int)(row - n_rows);
      const int pole = j & 1;
#pragma unroll
      for (int k = 0; k < 8; ++k) o[k] = 0.f;
      for (int e = 0; e < 5; ++e) {
        float t[8];
        up_pixel<F32>(src, xin, cring, (long long)(j >> 1), B, Pc, ring_pixel(nfine, pole, e), C, c, t, f16);
#pragma unroll
        for (int k = 0; k < 8; ++k) o[k] = fmaf(0.2f, t[k], o[k]);
      }
    }
    st8_op(out + (size_t)row * C + c, o, f16);
    if (out_w) st8_op(out_w + (size_t)row * C + c, o, 0);
  }
}

// ------------------------------------------------------------------------------------------------ backward of a residual pair
// out = relu(bnA(yA) + bnB(yB)) (models.py:38-39, 60-61): both BatchNorms see the SAME g = dout * (out > 0), so dout and the
// mask are read once for both (10 -> 7 bytes per element and pass).  partial[blk][4][C] = sum g (A), sum g*yhatA, sum g (B: same
// as A, kept for symmetry), sum g*yhatB.
__global__ void __launch_bounds__(256)
bwd_reduce2_anyc_kernel(const float* __restrict__ dout, long long ldg, const __nv_bfloat16* __restrict__ mask, Src yA, const float* __restrict__ statA,
                   Src yB, const float* __restrict__ statB, long long rows, int C, float* __restrict__ partial) {
  GIN_PDL_SYNC();
  __shared__ float part[3][256][9];
  const int C8 = C >> 3;
  const long long n = rows * C8;
  const int c = (int)(threadIdx.x % C8) * 8;
  float meanA[8], invA[8], meanB[8], invB[8];
  ld8(statA + c, meanA); ld8(statA + C + c, invA); ld8(statB + c, meanB); ld8(statB + C + c, invB);
  float s0[8], s1[8], s2[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) s0[k] = s1[k] = s2[k] = 0.f;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += gridDim.x * 256LL) {
    const long long r = i / C8;
    float g[8], yh[8], v[8];
    grad_row(dout, ldg, mask, yA, r, c, C, meanA, invA, g, yh);
    ld8_src(yB, r, c, v);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      s0[k] += g[k];
      s1[k] = fmaf(g[k], yh[k], s1[k]);
      s2[k] = fmaf(g[k], (v[k] - meanB[k]) * invB[k], s2[k]);
    }
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) { part[0][threadIdx.x][k] = s0[k]; part[1][threadIdx.x][k] = s1[k]; part[2][threadIdx.x][k] = s2[k]; }
  __syncthreads();
  float* mine = partial + (size_t)blockIdx.x * 4 * C;
  for (int i = threadIdx.x; i < 4 * C; i += 256) {
    const int w = i / C, cc = i - w * C, g8 = cc >> 3, k = cc & 7;
    const int src = w == 2 ? 0 : (w == 3 ? 2 : w);       // rows: sum g | sum g*yhatA | sum g | sum g*yhatB
    float acc = 0.f;
    for (int t = g8; t < 256; t += C8) acc += part[src][t][k];
    mine[i] = acc;
  }
}

// final[k][c] (double) = sum_b partial[b][k][c] (k = 0..3) for the 8 channels of this CTA; returned to threads 0..31 (k = tid >> 3)
GIN_DEVINL double final_sum4(const float* __restrict__ partial, int nblocks, int C) {
  __shared__ double red[8][33];
  const int j = threadIdx.x & 31, rg = threadIdx.x >> 5;
  const int k = j >> 3, c = blockIdx.x * 8 + (j & 7);
  double acc = 0.0;
  if (c < C) {
    float v[(MAX_CTAS + 7) / 8];
#pragma unroll
    for (int i = 0; i < (MAX_CTAS + 7) / 8; ++i) {
      const int b = rg + 8 * i;
      v[i] = b < nblocks ? __ldg(partial + ((size_t)b * 4 + k) * C + c) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < (MAX_CTAS + 7) / 8; ++i) acc += (double)v[i];
  }
  red[rg][j] = acc;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x < 32)
#pragma unroll
    for (int r = 0; r < 8; ++r) t += red[r][threadIdx.x];
  return t;
}

// bstatA / bstatB [4][C] from partial[nblocks][4][C]; grid = C/8, block = 256 (8 row groups x 32 (sum, channel) lanes)
__global__ void __launch_bounds__(256)
bwd_final2_kernel(const float* __restrict__ partial, int nblocks, long long rows, int C, float* __restrict__ bstatA, float* __restrict__ bstatB) {
  GIN_PDL_SYNC();
  const double t = final_sum4(partial, nblocks, C);
  const int k = (threadIdx.x & 31) >> 3, c = blockIdx.x * 8 + (threadIdx.x & 7);
  if (threadIdx.x < 32 && c < C) {
    float* bs = k < 2 ? bstatA : bstatB;
    const int kk = k & 1;
    bs[kk * C + c] = (float)t;
    bs[(2 + kk) * C + c] = (float)(t / (double)rows);
  }
}

// backward records (layout: see stats_total_kernel) from the partials of bwd_reduce(_s)_kernel (nbn = 1, bwd_final_kernel's order)
// or of bwd_reduce2(_anyc)_kernel (nbn = 2, bwd_final2_kernel's order).  grid = C/8.
__global__ void __launch_bounds__(256)
bwd_total_kernel(const float* __restrict__ partial, int nblocks, int nbn, long long rows, int C, double* __restrict__ rec) {
  GIN_PDL_SYNC();
  const double t = nbn == 1 ? final_sum(partial, nblocks, C) : final_sum4(partial, nblocks, C);
  const int k = threadIdx.x >> 3, c = blockIdx.x * 8 + (threadIdx.x & 7);
  const long long len = 2LL * C + 1;
  if (threadIdx.x < 16 * nbn && c < C) rec[(k >> 1) * len + (k & 1) * C + c] = t;
  if (blockIdx.x == 0 && threadIdx.x < nbn) rec[threadIdx.x * len + 2 * C] = (double)rows;
}

// bstatA (and bstatB of a pair, nbn = 2) from the gathered backward records recs[world][nbn * (2C + 1)]: dbeta, dgamma = the sums of
// rank `rank`, mean(g), mean(g*yhat) = the sums over every rank / the global row count.  grid = C/8.
__global__ void __launch_bounds__(256)
bwd_sync_final_kernel(const double* __restrict__ recs, int world, int rank, int nbn, int C, float* __restrict__ bstatA, float* __restrict__ bstatB) {
  GIN_PDL_SYNC();
  const int k = threadIdx.x >> 3, c = blockIdx.x * 8 + (threadIdx.x & 7);
  if (threadIdx.x >= 16 * nbn || c >= C) return;
  const long long len = 2LL * C + 1, stride = nbn * len, base = (k >> 1) * len, off = base + (k & 1) * C + c;
  const double t = recs[rank * stride + off], s = rank_sum(recs, world, stride, off), rows = rank_sum(recs, world, stride, base + 2 * C);
  float* bs = k < 2 ? bstatA : bstatB;
  const int kk = k & 1;
  bs[kk * C + c] = (float)t;
  bs[(2 + kk) * C + c] = (float)(s / rows);
}

// dyA, dyB as bf16 gradient copies (row strides ldoA / ldoB, pole-mean rows included)
__global__ void __launch_bounds__(256)
bwd_apply2_anyc_kernel(const float* __restrict__ dout, long long ldg, const __nv_bfloat16* __restrict__ mask, Src yA, const float* __restrict__ statA,
                  const float* __restrict__ bstatA, Src yB, const float* __restrict__ statB, const float* __restrict__ bstatB,
                  __nv_bfloat16* __restrict__ dyA, long long ldoA, __nv_bfloat16* __restrict__ dyB, long long ldoB, int nlat, int B, int P, int C) {
  GIN_PDL_SYNC();
  const int C8 = C >> 3;
  const long long rows = (long long)B * P, n_main = rows * C8, n_all = n_main + 2LL * B * C8;
  const int c = (int)(threadIdx.x % C8) * 8;
  float meanA[8], invA[8], scA[8], c1A[8], c2A[8], meanB[8], invB[8], scB[8], c1B[8], c2B[8];
  ld8(statA + c, meanA); ld8(statA + C + c, invA); ld8(statA + 2 * C + c, scA); ld8(bstatA + 2 * C + c, c1A); ld8(bstatA + 3 * C + c, c2A);
  ld8(statB + c, meanB); ld8(statB + C + c, invB); ld8(statB + 2 * C + c, scB); ld8(bstatB + 2 * C + c, c1B); ld8(bstatB + 3 * C + c, c2B);
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n_all; i += gridDim.x * 256LL) {
    float oA[8], oB[8];
    if (i < n_main) {
      const long long r = i / C8;
      float g[8], yh[8], v[8];
      grad_row(dout, ldg, mask, yA, r, c, C, meanA, invA, g, yh);
      ld8_src(yB, r, c, v);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        oA[k] = scA[k] * (g[k] - c1A[k] - yh[k] * c2A[k]);
        oB[k] = scB[k] * (g[k] - c1B[k] - (v[k] - meanB[k]) * invB[k] * c2B[k]);
      }
    } else {
      const long long j = (i - n_main) / C8;
      const int sample = (int)(j >> 1), pole = (int)(j & 1);
#pragma unroll
      for (int k = 0; k < 8; ++k) oA[k] = oB[k] = 0.f;
      for (int e = 0; e < 5; ++e) {
        const long long r = (long long)sample * P + ring_pixel(nlat, pole, e);
        float g[8], yh[8], v[8];
        grad_row(dout, ldg, mask, yA, r, c, C, meanA, invA, g, yh);
        ld8_src(yB, r, c, v);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          oA[k] = fmaf(0.2f * scA[k], g[k] - c1A[k] - yh[k] * c2A[k], oA[k]);
          oB[k] = fmaf(0.2f * scB[k], g[k] - c1B[k] - (v[k] - meanB[k]) * invB[k] * c2B[k], oB[k]);
        }
      }
    }
    st8_bf16(dyA + (i / C8) * ldoA + c, oA);
    st8_bf16(dyB + (i / C8) * ldoB + c, oB);
  }
}

// ------------------------------------------------------------------------------------------------ C <= 256: constants in shared memory
// The streaming kernels above keep every per-channel constant of a thread's 8 channels in registers: 96 (bwd_apply), 98
// (bwd_reduce2) and 162 (bwd_apply2) registers per thread, i.e. 2, 2 and ONE resident CTA per SM -- 8 to 16 warps cannot keep
// enough loads in flight to fill HBM (ncu r02: 37-47 % of the copy bandwidth, profiles/r02_step_dram_traffic.txt).  The versions below
// hold the constants in shared memory (pre-combined once per CTA), re-read them every iteration through `ld.shared` that the
// compiler may not hoist (asm volatile), replace the 64-bit divisions by shifts (C/8 is a power of two) and fit 4 CTAs per SM.
// Measured inside the replayed ico2ico step (profiles/r02_trace_n1.log): bwd_apply2 278 -> 171 us, bwd_apply 240 -> 162,
// bwd_reduce2 203 -> 124, act_fwd 266 -> 201; the step 3.80 -> 3.46 ms.
constexpr int CST_MAX_C = 256;
#ifndef GIN_BN_SMEM_DEFAULT
#define GIN_BN_SMEM_DEFAULT 1
#endif
GIN_DEVINL void cst_put(float (*t)[2][32][4], int k, int ch, float v) { t[k][(ch >> 2) & 1][ch >> 3][ch & 3] = v; }
template <int K>
GIN_DEVINL void lds8(uint32_t base, float v[8]) {          // constant K of this thread's 8 channels; base = &cst[0][0][c8][0]
  // "memory": the compiler must see these as reads of the table (its stores are otherwise dead) -- callers therefore issue ALL
  // their global loads before the first lds8, or the loads would be serialised behind it
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4+%5];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(base), "n"(K * 1024) : "memory");
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4+%5];" : "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]) : "r"(base), "n"(K * 1024 + 512) : "memory");
}
GIN_DEVINL int log2_pow2(int v) { return __ffs(v) - 1; }
// the source format as a template argument: half the loads (and registers) of the run-time switch in ld8_src
template <bool F16>
GIN_DEVINL void ld8_y(const Src& s, long long r, int c, float v[8]) {
  if (!F16) { ld8(s.p + r * s.ld + c, v); return; }
  const uint4 u = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const __half*>(s.p) + r * s.ld + c));
  const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) { const float2 f = __half22float2(h[i]); v[2 * i] = f.x; v[2 * i + 1] = f.y; }
}

// o = y1*sc1 + (sh1 [+ sh2]) [+ y2*sc2], optional ReLU
template <bool TWO, bool F16>
GIN_DEVINL void apply_row_s(const Src& y1, const Src& y2, long long r, int c, uint32_t cb, int relu, float o[8]) {
  float v[8], k[8];
  ld8_y<F16>(y1, r, c, v);
  if (TWO) {
    float w[8];
    ld8_y<F16>(y2, r, c, w);
    // explicit intrinsics (never contracted): the backward kernels re-evaluate exactly this expression for the ReLU mask
    lds8<2>(cb, k);
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = __fmul_rn(w[j], k[j]);
    lds8<1>(cb, k);
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = __fadd_rn(o[j], k[j]);
  } else {
    lds8<1>(cb, o);
  }
  lds8<0>(cb, k);
#pragma unroll
  for (int j = 0; j < 8; ++j) o[j] = __fmaf_rn(v[j], k[j], o[j]);
  if (relu) {
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = fmaxf(o[j], 0.f);
  }
}

template <bool TWO, bool F16>
__global__ void __launch_bounds__(256, 4)
act_fwd_kernel(Src y1, const float* __restrict__ stat1, Src y2, const float* __restrict__ stat2, int relu, __nv_bfloat16* __restrict__ out_b,
               float* __restrict__ out_f, int nlat, int B, int P, int C, int f16, __nv_bfloat16* __restrict__ out_w) {
  GIN_PDL_SYNC();
  __shared__ __align__(16) float cst[3][2][32][4];
  for (int ch = threadIdx.x; ch < C; ch += 256) {
    cst_put(cst, 0, ch, stat1[2 * C + ch]);
    cst_put(cst, 1, ch, stat1[3 * C + ch] + (TWO ? stat2[3 * C + ch] : 0.f));
    if (TWO) cst_put(cst, 2, ch, stat2[2 * C + ch]);
  }
  __syncthreads();
  const int C8 = C >> 3, sh = log2_pow2(C8), c8 = threadIdx.x & (C8 - 1), c = c8 * 8;
  const uint32_t cb = (uint32_t)__cvta_generic_to_shared(&cst[0][0][c8][0]);
  const long long rows = (long long)B * P, n_main = rows << sh, n_all = n_main + ((2LL * B) << sh);
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n_all; i += gridDim.x * 256LL) {
    const long long row = i >> sh;
    float o[8];
    if (i < n_main) {
      apply_row_s<TWO, F16>(y1, y2, row, c, cb, relu, o);
      if (out_f) st8(out_f + row * C + c, o);
    } else {
      const int j = (int)(row - rows), sample = j >> 1, pole = j & 1;
#pragma unroll
      for (int k = 0; k < 8; ++k) o[k] = 0.f;
      for (int e = 0; e < 5; ++e) {
        float t[8];
        apply_row_s<TWO, F16>(y1, y2, (long long)sample * P + ring_pixel(nlat, pole, e), c, cb, relu, t);
#pragma unroll
        for (int k = 0; k < 8; ++k) o[k] = fmaf(0.2f, t[k], o[k]);
      }
    }
    if (out_b) st8_op(out_b + row * C + c, o, f16);
    if (out_w) st8_op(out_w + row * C + c, o, 0);          // the bf16 twin wgrad reads (and the ReLU mask of the backward)
  }
}

// g = dout * (out > 0).  The mask is either READ from an activation copy (mask != null, from_y == 0) or RE-EVALUATED from the
// BatchNorm input(s) and constants exactly as act_fwd_kernel computed out (from_y != 0: saves the 2 B / element of the mask read;
// relu_from_y<> below, called once the y values are in registers); mask == null and from_y == 0: no ReLU.
GIN_DEVINL void masked_grad(const float* __restrict__ dout, long long ldg, const __nv_bfloat16* __restrict__ mask, int from_y, long long r, int c, int C, float g[8]) {
  ld8(dout + r * ldg + c, g);
  if (mask && !from_y) {
    bool m[8];
    ld8_mask(mask + r * C + c, m);
#pragma unroll
    for (int k = 0; k < 8; ++k) g[k] = m[k] ? g[k] : 0.f;
  }
}
// out = relu(y*scale + shift): constants KSC = scale, KSH = shift
template <int KSC, int KSH>
GIN_DEVINL void relu_from_y(uint32_t cb, const float y[8], float g[8]) {
  float k[8], t[8];
  lds8<KSH>(cb, t);
  lds8<KSC>(cb, k);
#pragma unroll
  for (int j = 0; j < 8; ++j) g[j] = __fmaf_rn(y[j], k[j], t[j]) > 0.f ? g[j] : 0.f;
}
// out = relu(yA*scaleA + (yB*scaleB + (shiftA + shiftB))): constants KA = scaleA, KB = scaleB, KSH = shiftA + shiftB
template <int KA, int KB, int KSH>
GIN_DEVINL void relu_from_y2(uint32_t cb, const float yA[8], const float yB[8], float g[8]) {
  float k[8], t[8];
  lds8<KB>(cb, k);
#pragma unroll
  for (int j = 0; j < 8; ++j) t[j] = __fmul_rn(yB[j], k[j]);
  lds8<KSH>(cb, k);
#pragma unroll
  for (int j = 0; j < 8; ++j) t[j] = __fadd_rn(t[j], k[j]);
  lds8<KA>(cb, k);
#pragma unroll
  for (int j = 0; j < 8; ++j) g[j] = __fmaf_rn(yA[j], k[j], t[j]) > 0.f ? g[j] : 0.f;
}
// dy = a*g - b - (y - mean)*e  with  a = scale, b = scale*c1, e = scale*invstd*c2  (constants K0 .. K0+3: a, b, mean, e)
template <int K0>
GIN_DEVINL void bn_dy(uint32_t cb, const float g[8], float o[8]) {          // o: in y, out dy
  float k[8];
  lds8<K0 + 2>(cb, k);
#pragma unroll
  for (int j = 0; j < 8; ++j) o[j] -= k[j];
  lds8<K0 + 3>(cb, k);
#pragma unroll
  for (int j = 0; j < 8; ++j) o[j] *= k[j];
  lds8<K0>(cb, k);
#pragma unroll
  for (int j = 0; j < 8; ++j) o[j] = fmaf(k[j], g[j], -o[j]);
  lds8<K0 + 1>(cb, k);
#pragma unroll
  for (int j = 0; j < 8; ++j) o[j] -= k[j];
}
GIN_DEVINL void bn_dy_consts(float (*cst)[2][32][4], int k0, const float* __restrict__ stat, const float* __restrict__ bstat, int C) {
  for (int ch = threadIdx.x; ch < C; ch += 256) {
    const float scale = stat[2 * C + ch];
    cst_put(cst, k0, ch, scale);
    cst_put(cst, k0 + 1, ch, scale * bstat[2 * C + ch]);
    cst_put(cst, k0 + 2, ch, stat[ch]);
    cst_put(cst, k0 + 3, ch, scale * stat[C + ch] * bstat[3 * C + ch]);
  }
}

template <bool F16>
__global__ void __launch_bounds__(256, 4)
bwd_apply_kernel(const float* __restrict__ dout, long long ldg, const __nv_bfloat16* __restrict__ mask, Src y, const float* __restrict__ stat,
                 const float* __restrict__ bstat, __nv_bfloat16* __restrict__ dy_b, long long ldo, float* __restrict__ dy_f, long long ldf,
                 int nlat, int B, int P, int C, int from_y) {
  GIN_PDL_SYNC();
  __shared__ __align__(16) float cst[5][2][32][4];
  bn_dy_consts(cst, 0, stat, bstat, C);
  for (int ch = threadIdx.x; ch < C; ch += 256) cst_put(cst, 4, ch, stat[3 * C + ch]);
  __syncthreads();
  const int C8 = C >> 3, sh = log2_pow2(C8), c8 = threadIdx.x & (C8 - 1), c = c8 * 8;
  const uint32_t cb = (uint32_t)__cvta_generic_to_shared(&cst[0][0][c8][0]);
  const long long rows = (long long)B * P, n_main = rows << sh, n_all = n_main + (dy_b ? (2LL * B) << sh : 0);
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n_all; i += gridDim.x * 256LL) {
    const long long row = i >> sh;
    float o[8], g[8];
    if (i < n_main) {
      masked_grad(dout, ldg, mask, from_y, row, c, C, g);
      ld8_y<F16>(y, row, c, o);
      if (from_y) relu_from_y<0, 4>(cb, o, g);
      bn_dy<0>(cb, g, o);
      if (dy_f) st8(dy_f + row * ldf + c, o);
    } else {
      const int j = (int)(row - rows), sample = j >> 1, pole = j & 1;
#pragma unroll
      for (int k = 0; k < 8; ++k) o[k] = 0.f;
      for (int e = 0; e < 5; ++e) {
        const long long r = (long long)sample * P + ring_pixel(nlat, pole, e);
        float t[8];
        masked_grad(dout, ldg, mask, from_y, r, c, C, g);
        ld8_y<F16>(y, r, c, t);
        if (from_y) relu_from_y<0, 4>(cb, t, g);
        bn_dy<0>(cb, g, t);
#pragma unroll
        for (int k = 0; k < 8; ++k) o[k] = fmaf(0.2f, t[k], o[k]);
      }
    }
    if (dy_b) st8_bf16(dy_b + row * ldo + c, o);
  }
}

// partial[blk][2][C] = sum g | sum g*yhat (the single-BatchNorm form of bwd_reduce2_kernel below)
template <bool F16>
__global__ void __launch_bounds__(256, 4)
bwd_reduce_s_kernel(const float* __restrict__ dout, long long ldg, const __nv_bfloat16* __restrict__ mask, Src y, const float* __restrict__ stat,
                    long long rows, int C, float* __restrict__ partial, int from_y) {
  GIN_PDL_SYNC();
  __shared__ __align__(16) float cst[3][2][32][4];
  for (int ch = threadIdx.x; ch < C; ch += 256) { cst_put(cst, 0, ch, stat[ch]); cst_put(cst, 1, ch, stat[2 * C + ch]); cst_put(cst, 2, ch, stat[3 * C + ch]); }
  __syncthreads();
  const int C8 = C >> 3, sh = log2_pow2(C8), c8 = threadIdx.x & (C8 - 1), c = c8 * 8;
  const uint32_t cb = (uint32_t)__cvta_generic_to_shared(&cst[0][0][c8][0]);
  const long long n = rows << sh;
  float s0[8], s1[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) s0[k] = s1[k] = 0.f;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += gridDim.x * 256LL) {
    const long long r = i >> sh;
    float g[8], v[8], m[8];
    masked_grad(dout, ldg, mask, from_y, r, c, C, g);
    ld8_y<F16>(y, r, c, v);
    if (from_y) relu_from_y<1, 2>(cb, v, g);
    lds8<0>(cb, m);
#pragma unroll
    for (int k = 0; k < 8; ++k) { s0[k] += g[k]; s1[k] = fmaf(g[k], v[k] - m[k], s1[k]); }
  }
  float inv[8];
  ld8(stat + C + c, inv);
#pragma unroll
  for (int k = 0; k < 8; ++k) s1[k] *= inv[k];
  block_partials(s0, s1, C, partial);
}

// partial[blk][4][C] = sum g | sum g*yhatA | sum g | sum g*yhatB; inside the loop only the means are needed:
// sum g*yhat = invstd * sum g*(y - mean)
template <bool F16>
__global__ void __launch_bounds__(256, 4)
bwd_reduce2_kernel(const float* __restrict__ dout, long long ldg, const __nv_bfloat16* __restrict__ mask, Src yA, const float* __restrict__ statA,
                   Src yB, const float* __restrict__ statB, long long rows, int C, float* __restrict__ partial, int from_y) {
  GIN_PDL_SYNC();
  __shared__ float part[3][256][9];
  __shared__ __align__(16) float cst[5][2][32][4];
  for (int ch = threadIdx.x; ch < C; ch += 256) {
    cst_put(cst, 0, ch, statA[ch]); cst_put(cst, 1, ch, statB[ch]);
    cst_put(cst, 2, ch, statA[2 * C + ch]); cst_put(cst, 3, ch, statB[2 * C + ch]); cst_put(cst, 4, ch, statA[3 * C + ch] + statB[3 * C + ch]);
  }
  __syncthreads();
  const int C8 = C >> 3, sh = log2_pow2(C8), c8 = threadIdx.x & (C8 - 1), c = c8 * 8;
  const uint32_t cb = (uint32_t)__cvta_generic_to_shared(&cst[0][0][c8][0]);
  const long long n = rows << sh;
  float s0[8], s1[8], s2[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) s0[k] = s1[k] = s2[k] = 0.f;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += gridDim.x * 256LL) {
    const long long r = i >> sh;
    float g[8], v[8], w[8], m[8];
    masked_grad(dout, ldg, mask, from_y, r, c, C, g);
    ld8_y<F16>(yA, r, c, v);
    ld8_y<F16>(yB, r, c, w);
    if (from_y) relu_from_y2<2, 3, 4>(cb, v, w, g);
    lds8<0>(cb, m);
#pragma unroll
    for (int k = 0; k < 8; ++k) { s0[k] += g[k]; s1[k] = fmaf(g[k], v[k] - m[k], s1[k]); }
    lds8<1>(cb, m);
#pragma unroll
    for (int k = 0; k < 8; ++k) s2[k] = fmaf(g[k], w[k] - m[k], s2[k]);
  }
  {
    float iA[8], iB[8];
    ld8(statA + C + c, iA); ld8(statB + C + c, iB);
#pragma unroll
    for (int k = 0; k < 8; ++k) { part[0][threadIdx.x][k] = s0[k]; part[1][threadIdx.x][k] = s1[k] * iA[k]; part[2][threadIdx.x][k] = s2[k] * iB[k]; }
  }
  __syncthreads();
  float* mine = partial + (size_t)blockIdx.x * 4 * C;
  for (int i = threadIdx.x; i < 4 * C; i += 256) {
    const int w = i / C, cc = i - w * C, g8 = cc >> 3, k = cc & 7;
    const int src = w == 2 ? 0 : (w == 3 ? 2 : w);       // rows: sum g | sum g*yhatA | sum g | sum g*yhatB
    float acc = 0.f;
    for (int t = g8; t < 256; t += C8) acc += part[src][t][k];
    mine[i] = acc;
  }
}

template <bool F16>
__global__ void __launch_bounds__(256, 4)
bwd_apply2_kernel(const float* __restrict__ dout, long long ldg, const __nv_bfloat16* __restrict__ mask, Src yA, const float* __restrict__ statA,
                  const float* __restrict__ bstatA, Src yB, const float* __restrict__ statB, const float* __restrict__ bstatB,
                  __nv_bfloat16* __restrict__ dyA, long long ldoA, __nv_bfloat16* __restrict__ dyB, long long ldoB, int nlat, int B, int P, int C,
                  int from_y) {
  GIN_PDL_SYNC();
  __shared__ __align__(16) float cst[9][2][32][4];
  bn_dy_consts(cst, 0, statA, bstatA, C);
  bn_dy_consts(cst, 4, statB, bstatB, C);
  for (int ch = threadIdx.x; ch < C; ch += 256) cst_put(cst, 8, ch, statA[3 * C + ch] + statB[3 * C + ch]);
  __syncthreads();
  const int C8 = C >> 3, sh = log2_pow2(C8), c8 = threadIdx.x & (C8 - 1), c = c8 * 8;
  const uint32_t cb = (uint32_t)__cvta_generic_to_shared(&cst[0][0][c8][0]);
  const long long rows = (long long)B * P, n_main = rows << sh, n_all = n_main + ((2LL * B) << sh);
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n_all; i += gridDim.x * 256LL) {
    const long long row = i >> sh;
    float g[8], o[8], oB[8];
    if (i < n_main) {
      masked_grad(dout, ldg, mask, from_y, row, c, C, g);
      ld8_y<F16>(yA, row, c, o);
      ld8_y<F16>(yB, row, c, oB);
      if (from_y) relu_from_y2<0, 4, 8>(cb, o, oB, g);
      bn_dy<0>(cb, g, o);
      bn_dy<4>(cb, g, oB);
      st8_bf16(dyA + row * ldoA + c, o);
      st8_bf16(dyB + row * ldoB + c, oB);
    } else {
      // pole-mean rows (2B of them): one BatchNorm after the other keeps the register count of the main path
      const int j = (int)(row - rows), sample = j >> 1, pole = j & 1;
#pragma unroll
      for (int k = 0; k < 8; ++k) o[k] = oB[k] = 0.f;
      for (int e = 0; e < 10; ++e) {
        const long long r = (long long)sample * P + ring_pixel(nlat, pole, e % 5);
        float t[8];
        masked_grad(dout, ldg, mask, from_y, r, c, C, g);
        if (from_y) {
          float u[8];
          ld8_y<F16>(yA, r, c, t);
          ld8_y<F16>(yB, r, c, u);
          relu_from_y2<0, 4, 8>(cb, t, u, g);
        }
        if (e < 5) {
          ld8_y<F16>(yA, r, c, t);
          bn_dy<0>(cb, g, t);
#pragma unroll
          for (int k = 0; k < 8; ++k) o[k] = fmaf(0.2f, t[k], o[k]);
        } else {
          ld8_y<F16>(yB, r, c, t);
          bn_dy<4>(cb, g, t);
#pragma unroll
          for (int k = 0; k < 8; ++k) oB[k] = fmaf(0.2f, t[k], oB[k]);
        }
      }
      st8_bf16(dyA + row * ldoA + c, o);
      st8_bf16(dyB + row * ldoB + c, oB);
    }
  }
}

// GIN_BN_SMEM=0: the register-constant kernels (*_anyc_kernel) for every C
inline bool smem_consts(int C) {
  static int v = -1;
  if (v < 0) { const char* e = getenv("GIN_BN_SMEM"); v = e ? (e[0] != '0') : GIN_BN_SMEM_DEFAULT; }
  return v == 1 && C <= CST_MAX_C;
}

// CTAs of the streaming BatchNorm kernels: GIN_BN_CTAS (experiments), default 4 per SM
inline int bn_ctas() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("GIN_BN_CTAS"); v = e ? atoi(e) : MAX_CTAS; if (v < 1 || v > MAX_CTAS) v = MAX_CTAS; }
  return v;
}
inline int grid_for_rows(long long n_threads) {
  long long b = (n_threads + 255) / 256;
  if (b < 1) b = 1;
  return (int)(b < bn_ctas() ? b : bn_ctas());
}

// ------------------------------------------------------------------------------------------------ eval mode (inference)
// One BatchNorm of a chain in eval mode (include/geniconet_b200.h: GinBnEvalEntry).
struct EvalEntry {
  const float* gamma;
  const float* beta;
  const float* running_mean;
  const float* running_var;
  const float* conv_bias;
  float* scale;
  float* shift;
  float* stat;
  float eps;
  int C;
};

// grid (ceil(max_C / 256), count): the constants of every BatchNorm of a table, read from the device at run time (a captured graph
// follows in-place updates of the parameters and running statistics)
__global__ void __launch_bounds__(256) eval_consts_kernel(const EvalEntry* __restrict__ table) {
  GIN_PDL_SYNC();
  const EvalEntry t = table[blockIdx.y];
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c >= t.C) return;
  const float mean = t.running_mean[c];
  const float invstd = (float)(1.0 / sqrt((double)t.running_var[c] + (double)t.eps));
  const float g = t.gamma ? t.gamma[c] : 1.f, b = t.beta ? t.beta[c] : 0.f;
  const float scale = g * invstd;
  if (t.scale) t.scale[c] = scale;
  if (t.shift) t.shift[c] = fmaf(scale, (t.conv_bias ? t.conv_bias[c] : 0.f) - mean, b);
  if (t.stat) { t.stat[c] = mean; t.stat[t.C + c] = invstd; t.stat[2 * t.C + c] = scale; t.stat[3 * t.C + c] = b - mean * scale; }
}

// pole-mean rows [rows + 2*sample + pole] of an operand copy from the fp32 ring values the affine conv epilogue stored
// (cv2::Affine::ring, [B][10][C]): the same sum, in the same order, as cast_bf16_kernel over the fp32 map
__global__ void __launch_bounds__(256) pole_mean_kernel(const float* __restrict__ ring, __nv_bfloat16* __restrict__ xb, long long rows, int B, int C,
                                                        int f16) {
  GIN_PDL_SYNC();
  const int C8 = C >> 3;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < 2LL * B * C8; i += gridDim.x * 256LL) {
    const int c = (int)(i % C8) * 8, sp = (int)(i / C8), sample = sp >> 1, pole = sp & 1;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
#pragma unroll
    for (int k = 0; k < 5; ++k) {
      const float* src = ring + ((size_t)sample * 10 + pole * 5 + k) * C + c;
      a = fma4(0.2f, ld4(src), a);
      b = fma4(0.2f, ld4(src + 4), b);
    }
    uint4 o;
    o.x = pack2_op(a.x, a.y, f16); o.y = pack2_op(a.z, a.w, f16); o.z = pack2_op(b.x, b.y, f16); o.w = pack2_op(b.z, b.w, f16);
    *reinterpret_cast<uint4*>(xb + (rows + sp) * C + c) = o;
  }
}

// ------------------------------------------------------------------------------------------------ eval mode backward (frozen BatchNorm)
// out = relu(bn(y) [+ bn'(y')]) with the running statistics: dy = scale * g does not depend on any reduction, so the gradient
// copies and the sums come out of ONE streaming pass (the training backward needs a reduction pass first).  Same thread layout,
// register budget (4 CTAs of 256 threads per SM) and shared-memory constants as bwd_apply_kernel / bwd_reduce2_kernel.  The
// ReLU mask is read (mask != null, from_y == 0) or re-evaluated with relu_from_y / relu_from_y2, bit for bit act_fwd_kernel.
// RED: partial[blk][NS][C] = sum g | sum g*yhatA [| sum g*yhatB]  (main rows only; eval_bwd_final_kernel adds them up).
// dy = __fmul_rn(scale, g), and the pole-mean rows are fmaf(0.2, dy, .) over the five ring pixels from 0: the same sum, in the
// same order, as cast_bf16_kernel over the fp32 dy.

// constants of eval_bwd_kernel: 0 scale, 1 shift, 2 mean
template <bool F16, bool RED>
__global__ void __launch_bounds__(256, 4)
eval_bwd_kernel(const float* __restrict__ dout, long long ldg, const __nv_bfloat16* __restrict__ mask, Src y, const float* __restrict__ stat,
                __nv_bfloat16* __restrict__ dy_b, long long ldo, float* __restrict__ dy_f, long long ldf, float* __restrict__ partial, int nlat,
                int B, int P, int C, int from_y) {
  GIN_PDL_SYNC();
  __shared__ __align__(16) float cst[3][2][32][4];
  for (int ch = threadIdx.x; ch < C; ch += 256) { cst_put(cst, 0, ch, stat[2 * C + ch]); cst_put(cst, 1, ch, stat[3 * C + ch]); cst_put(cst, 2, ch, stat[ch]); }
  __syncthreads();
  const int C8 = C >> 3, sh = log2_pow2(C8), c8 = threadIdx.x & (C8 - 1), c = c8 * 8;
  const uint32_t cb = (uint32_t)__cvta_generic_to_shared(&cst[0][0][c8][0]);
  const long long rows = (long long)B * P, n_main = rows << sh, n_all = n_main + (dy_b ? (2LL * B) << sh : 0);
  float s0[8], s1[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) s0[k] = s1[k] = 0.f;
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n_all; i += gridDim.x * 256LL) {
    const long long row = i >> sh;
    float o[8], g[8], k8[8];
    if (i < n_main) {
      masked_grad(dout, ldg, mask, from_y, row, c, C, g);
      if (RED || from_y) ld8_y<F16>(y, row, c, o);
      if (from_y) relu_from_y<0, 1>(cb, o, g);
      if (RED) {
        lds8<2>(cb, k8);
#pragma unroll
        for (int k = 0; k < 8; ++k) { s0[k] += g[k]; s1[k] = fmaf(g[k], o[k] - k8[k], s1[k]); }
      }
      lds8<0>(cb, k8);
#pragma unroll
      for (int k = 0; k < 8; ++k) o[k] = __fmul_rn(k8[k], g[k]);
      if (dy_f) st8(dy_f + row * ldf + c, o);
    } else {
      const int j = (int)(row - rows), sample = j >> 1, pole = j & 1;
#pragma unroll
      for (int k = 0; k < 8; ++k) o[k] = 0.f;
      for (int e = 0; e < 5; ++e) {
        const long long r = (long long)sample * P + ring_pixel(nlat, pole, e);
        masked_grad(dout, ldg, mask, from_y, r, c, C, g);
        if (from_y) {
          float t[8];
          ld8_y<F16>(y, r, c, t);
          relu_from_y<0, 1>(cb, t, g);
        }
        lds8<0>(cb, k8);
#pragma unroll
        for (int k = 0; k < 8; ++k) o[k] = fmaf(0.2f, __fmul_rn(k8[k], g[k]), o[k]);
      }
    }
    if (dy_b) st8_bf16(dy_b + row * ldo + c, o);
  }
  if constexpr (RED) {
    float inv[8];
    ld8(stat + C + c, inv);
#pragma unroll
    for (int k = 0; k < 8; ++k) s1[k] *= inv[k];
    block_partials(s0, s1, C, partial);
  }
}

// Sums of three per-thread vectors over a CTA in two steps, so that the vectors can die in between: stash_partials3 puts this
// thread's values into shared memory, finish_partials3 (once every thread stashed) writes partial[blockIdx][3][C].
GIN_DEVINL float (*part3_smem())[256][9] {
  __shared__ float part[3][256][9];
  return part;
}
GIN_DEVINL void stash_partials3(const float s0[8], const float s1[8], const float s2[8]) {
  float (*part)[256][9] = part3_smem();
#pragma unroll
  for (int k = 0; k < 8; ++k) { part[0][threadIdx.x][k] = s0[k]; part[1][threadIdx.x][k] = s1[k]; part[2][threadIdx.x][k] = s2[k]; }
}
GIN_DEVINL void finish_partials3(int C, float* __restrict__ partial) {
  float (*part)[256][9] = part3_smem();
  __syncthreads();
  const int C8 = C >> 3;
  float* mine = partial + (size_t)blockIdx.x * 3 * C;
  for (int i = threadIdx.x; i < 3 * C; i += 256) {
    const int w = i / C, cc = i - w * C, g8 = cc >> 3, k = cc & 7;
    float acc = 0.f;
    for (int t = g8; t < 256; t += C8) acc += part[w][t][k];
    mine[i] = acc;
  }
}

// out = relu(bnA(yA) + bnB(yB)); constants: 0 scaleA, 1 scaleB, 2 shiftA + shiftB, 3 meanA, 4 meanB
template <bool F16, bool RED>
__global__ void __launch_bounds__(256, 4)
eval_bwd2_kernel(const float* __restrict__ dout, long long ldg, const __nv_bfloat16* __restrict__ mask, Src yA, const float* __restrict__ statA,
                 Src yB, const float* __restrict__ statB, __nv_bfloat16* __restrict__ dyA, long long ldoA, __nv_bfloat16* __restrict__ dyB,
                 long long ldoB, float* __restrict__ partial, int nlat, int B, int P, int C, int from_y) {
  GIN_PDL_SYNC();
  __shared__ __align__(16) float cst[5][2][32][4];
  for (int ch = threadIdx.x; ch < C; ch += 256) {
    cst_put(cst, 0, ch, statA[2 * C + ch]); cst_put(cst, 1, ch, statB[2 * C + ch]); cst_put(cst, 2, ch, statA[3 * C + ch] + statB[3 * C + ch]);
    cst_put(cst, 3, ch, statA[ch]); cst_put(cst, 4, ch, statB[ch]);
  }
  __syncthreads();
  const int C8 = C >> 3, sh = log2_pow2(C8), c8 = threadIdx.x & (C8 - 1), c = c8 * 8;
  const uint32_t cb = (uint32_t)__cvta_generic_to_shared(&cst[0][0][c8][0]);
  const long long rows = (long long)B * P, n_main = rows << sh, n_all = n_main + ((2LL * B) << sh);
  long long i = blockIdx.x * 256LL + threadIdx.x;
  {
    // the pixel rows (every one of them comes before the pole rows in the grid-stride order): the sums are live only here
    float s0[8], s1[8], s2[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) s0[k] = s1[k] = s2[k] = 0.f;
    for (; i < n_main; i += gridDim.x * 256LL) {
      const long long row = i >> sh;
      float g[8], oA[8], oB[8], k8[8];
      masked_grad(dout, ldg, mask, from_y, row, c, C, g);
      if (RED || from_y) { ld8_y<F16>(yA, row, c, oA); ld8_y<F16>(yB, row, c, oB); }
      if (from_y) relu_from_y2<0, 1, 2>(cb, oA, oB, g);
      if (RED) {
        lds8<3>(cb, k8);
#pragma unroll
        for (int k = 0; k < 8; ++k) { s0[k] += g[k]; s1[k] = fmaf(g[k], oA[k] - k8[k], s1[k]); }
        lds8<4>(cb, k8);
#pragma unroll
        for (int k = 0; k < 8; ++k) s2[k] = fmaf(g[k], oB[k] - k8[k], s2[k]);
      }
      lds8<0>(cb, k8);
#pragma unroll
      for (int k = 0; k < 8; ++k) oA[k] = __fmul_rn(k8[k], g[k]);
      st8_bf16(dyA + row * ldoA + c, oA);
      lds8<1>(cb, k8);
#pragma unroll
      for (int k = 0; k < 8; ++k) oB[k] = __fmul_rn(k8[k], g[k]);
      st8_bf16(dyB + row * ldoB + c, oB);
    }
    if constexpr (RED) {
      float iA[8], iB[8];
      ld8(statA + C + c, iA); ld8(statB + C + c, iB);
#pragma unroll
      for (int k = 0; k < 8; ++k) { s1[k] *= iA[k]; s2[k] *= iB[k]; }
      stash_partials3(s0, s1, s2);
    }
  }
  for (; i < n_all; i += gridDim.x * 256LL) {
    // pole-mean rows (2B of them): one BatchNorm after the other keeps the register count of the pixel rows
    const long long row = i >> sh;
    const int j = (int)(row - rows), sample = j >> 1, pole = j & 1;
    float o[8], g[8], k8[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) o[k] = 0.f;
    for (int e = 0; e < 10; ++e) {
      const long long r = (long long)sample * P + ring_pixel(nlat, pole, e % 5);
      masked_grad(dout, ldg, mask, from_y, r, c, C, g);
      if (from_y) {
        float t[8], u[8];
        ld8_y<F16>(yA, r, c, t);
        ld8_y<F16>(yB, r, c, u);
        relu_from_y2<0, 1, 2>(cb, t, u, g);
      }
      if (e < 5) lds8<0>(cb, k8);
      else lds8<1>(cb, k8);
#pragma unroll
      for (int k = 0; k < 8; ++k) o[k] = fmaf(0.2f, __fmul_rn(k8[k], g[k]), o[k]);
      if (e == 4) {
        st8_bf16(dyA + row * ldoA + c, o);
#pragma unroll
        for (int k = 0; k < 8; ++k) o[k] = 0.f;
      }
    }
    st8_bf16(dyB + row * ldoB + c, o);
  }
  if constexpr (RED) finish_partials3(C, partial);
}

// bsum[3][C] = dbeta = sum g, dgamma = sum g*yhat, conv-bias gradient = scale * sum g, from partial[nblocks][ns][C] (ns = 2: one
// BatchNorm, rows g | g*yhatA; ns = 3: a pair, rows g | g*yhatA | g*yhatB); bsumA / bsumB may be NULL.  Fixed-order fp64 sums.
// grid = C/8, block = 256 (8 row groups x 32 (sum, channel) lanes).
__global__ void __launch_bounds__(256)
eval_bwd_final_kernel(const float* __restrict__ partial, int nblocks, int ns, int C, const float* __restrict__ statA, float* __restrict__ bsumA,
                      const float* __restrict__ statB, float* __restrict__ bsumB) {
  GIN_PDL_SYNC();
  __shared__ double red[8][33];
  const int j = threadIdx.x & 31, rg = threadIdx.x >> 5;
  const int k = j >> 3, c = blockIdx.x * 8 + (j & 7);
  double acc = 0.0;
  if (k < ns && c < C) {
    float v[(MAX_CTAS + 7) / 8];
#pragma unroll
    for (int i = 0; i < (MAX_CTAS + 7) / 8; ++i) {
      const int b = rg + 8 * i;
      v[i] = b < nblocks ? __ldg(partial + ((size_t)b * ns + k) * C + c) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < (MAX_CTAS + 7) / 8; ++i) acc += (double)v[i];
  }
  red[rg][j] = acc;
  __syncthreads();
  if (threadIdx.x < 32 && k < ns && c < C) {
    double t = 0.0;
#pragma unroll
    for (int r = 0; r < 8; ++r) t += red[r][threadIdx.x];
    if (k == 0) {                 // sum g: shared by both BatchNorms of a pair
      if (bsumA) { bsumA[c] = (float)t; bsumA[2 * C + c] = (float)((double)statA[2 * C + c] * t); }
      if (bsumB) { bsumB[c] = (float)t; bsumB[2 * C + c] = (float)((double)statB[2 * C + c] * t); }
    } else if (k == 1) {
      if (bsumA) bsumA[C + c] = (float)t;
    } else if (bsumB) {
      bsumB[C + c] = (float)t;
    }
  }
}

}  // namespace bn
}  // namespace gin
