// Normal and Laplacian terms of the Chamfer loss, matched through the nearest-neighbour indices of gin_chamfer.cuh.
//
// v [B][V][3] are the output vertices (poles included), n_i / L_i their unit vertex normal and uniform Laplacian exactly as
// normals_laplacian_kernel computes them (ring_geom of gin_loss.cuh), tn_j / tl_j the target's normal and Laplacian at point j,
// read with element strides (the rows of a [B][9][V] target in place), i_xy [B][V] / i_yx [B][M] the nearest-neighbour indices:
//
//   nor_xy = mean_{b,i} (1 - cos(n_i, tn_{i_xy(i)}))        nor_yx = mean_{b,j} (1 - cos(tn_j, n_{i_yx(j)}))
//   lap_xy = mean_{b,i,c} (L_i - tl_{i_xy(i)})_c^2           lap_yx = mean_{b,j,c} (tl_j - L_{i_yx(j)})_c^2
//
// with the eps of p2p_fwd_kernel.  n and L are recomputed from the ring where they are needed, never materialised.
// Forward: one grid-stride launch over the B*V vertices (xy) and the B*M target points (yx), fp64 per-CTA partials, a fixed-order
// fp64 final: deterministic.
// Backward: the cotangents g_n = dL/dn, g_L = dL/dL [B][V][3].  The xy part is a per-vertex write; the yx part scatters into i_yx(j)
// through the exact fixed-point sum of gin_fixed_scatter.cuh (integer atomics only).  gin_ring_ops_bwd then takes (g_n, g_L) to dv.
// The nearest-neighbour choice is piecewise constant and not differentiated; the target gets no gradient.
//
// The kernels take one Args struct: no type of namespace chamfer appears in their signatures, so the SASS test that counts the
// Chamfer distance kernels by name sees only those.
#pragma once
#include "gin_loss.cuh"
#include "gin_chamfer.cuh"

namespace gin {
namespace chamfer_terms {

constexpr int kThreads = 256;
constexpr int kMaxParts = 1024;

struct Args {
  const int32_t* plan;                  // loss plan (device)
  const float* v;                       // [B][V][3]
  chamfer::Pts tn, tl;                  // target normals / Laplacians; p == NULL: term off
  const int32_t* idx_xy;                // [B][V] or NULL: direction off
  const int32_t* idx_yx;                // [B][M] or NULL: direction off
  const float* dout;                    // backward: device [4], cotangents of {nor_xy, nor_yx, lap_xy, lap_yx}
  fixsum::Acc* acc_n;                   // backward: [B][V] scatter sums of g_n, g_L (zeroed)
  fixsum::Acc* acc_l;
  float* g_n;                           // backward: [B][V][3]
  float* g_l;
  double* partial;                      // forward: [gridDim.x][4]
  int B, M;
};

struct Geom { F3 n, lap; };

// n_u and L_u exactly as normals_laplacian_kernel writes them
GIN_DEVINL Geom vertex_geom(const float* vb, const int32_t* nbt, int u) {
  const RingGeom g = ring_geom(vb, nbt + (size_t)u * 6);
  const float m = fmaxf(sqrtf(dot(g.nraw, g.nraw)), kNormalEps);
  Geom r;
  r.n = (1.0f / m) * g.nraw;
  r.lap = g.mean - ldv(vb, u);
  return r;
}

GIN_DEVINL F3 row(const chamfer::Pts& t, int b, int j) { return f3(t.at(b, j, 0), t.at(b, j, 1), t.at(b, j, 2)); }

// 1 - cos(n, t), as p2p_fwd_kernel
GIN_DEVINL float one_minus_cos(F3 n, F3 t) {
  const float an = fmaxf(sqrtf(dot(n, n)), kCosEps), at = fmaxf(sqrtf(dot(t, t)), kCosEps);
  return 1.0f - dot(n, t) / (an * at);
}

// d(1 - cos(n, t)) / dn, as p2p_bwd_vertex_kernel
GIN_DEVINL F3 one_minus_cos_dn(F3 n, F3 t) {
  const float a = sqrtf(dot(n, n)), A = fmaxf(a, kCosEps), T = fmaxf(sqrtf(dot(t, t)), kCosEps);
  F3 gn = (-1.0f / (A * T)) * t;
  if (a > kCosEps) gn = gn + (dot(n, t) / (A * A * T * a)) * n;
  return gn;
}

__global__ void __launch_bounds__(kThreads) fwd_kernel(Args a) {
  const GinLossPlanHdr* h = reinterpret_cast<const GinLossPlanHdr*>(a.plan);
  const int V = h->V;
  const int32_t* nbt = a.plan + h->ring_off;
  const long long nxy = a.idx_xy ? (long long)a.B * V : 0, n = nxy + (a.idx_yx ? (long long)a.B * a.M : 0);
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;     // nor_xy, nor_yx, lap_xy, lap_yx: scalars, a runtime-indexed array spills
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n; t += (long long)gridDim.x * blockDim.x) {
    const bool xy = t < nxy;
    int b, u, j;
    if (xy) { b = (int)(t / V); u = (int)(t - (long long)b * V); j = a.idx_xy[t]; }
    else { const long long e = t - nxy; b = (int)(e / a.M); j = (int)(e - (long long)b * a.M); u = a.idx_yx[e]; }
    const Geom g = vertex_geom(a.v + (size_t)b * V * 3, nbt, u);
    if (a.tn.p) {
      const double c = (double)one_minus_cos(g.n, row(a.tn, b, j));
      if (xy) s0 += c; else s1 += c;
    }
    if (a.tl.p) {
      const F3 d = g.lap - row(a.tl, b, j);
      const double q = (double)dot(d, d);
      if (xy) s2 += q; else s3 += q;
    }
  }
  __shared__ double sh[4][kThreads];
  sh[0][threadIdx.x] = s0; sh[1][threadIdx.x] = s1; sh[2][threadIdx.x] = s2; sh[3][threadIdx.x] = s3;
  __syncthreads();
  for (int o = kThreads / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o)
#pragma unroll
      for (int k = 0; k < 4; ++k) sh[k][threadIdx.x] += sh[k][threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x < 4) a.partial[(size_t)blockIdx.x * 4 + threadIdx.x] = sh[threadIdx.x][0];
}

// out[4] = {nor_xy, nor_yx, lap_xy, lap_yx}; a direction or term that is off reads 0
__global__ void __launch_bounds__(kThreads) final_kernel(const double* __restrict__ partial, int nparts, float* __restrict__ out,
                                                         double inv_bv, double inv_bm) {
  __shared__ double sh[4][kThreads];
  double s[4] = {0.0, 0.0, 0.0, 0.0};
  for (int i = threadIdx.x; i < nparts; i += blockDim.x)
#pragma unroll
    for (int k = 0; k < 4; ++k) s[k] += partial[(size_t)i * 4 + k];
#pragma unroll
  for (int k = 0; k < 4; ++k) sh[k][threadIdx.x] = s[k];
  __syncthreads();
  for (int o = kThreads / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o)
#pragma unroll
      for (int k = 0; k < 4; ++k) sh[k][threadIdx.x] += sh[k][threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    out[0] = (float)(sh[0][0] * inv_bv);
    out[1] = (float)(sh[1][0] * inv_bm);
    out[2] = (float)(sh[2][0] * inv_bv / 3.0);
    out[3] = (float)(sh[3][0] * inv_bm / 3.0);
  }
}

// The yx terms of target point e = (b, j) for its vertex u = i_yx(j): tn_ = c_nor * d(1 - cos)/dn_u, tl_ = c_lap * 2 (L_u - tl_j).
GIN_DEVINL void yx_terms(const Args& a, const int32_t* nbt, int V, long long e, int& b, int& u, float tn_[3], float tl_[3]) {
  b = (int)(e / a.M);
  const int j = (int)(e - (long long)b * a.M);
  u = a.idx_yx[e];
  const Geom g = vertex_geom(a.v + (size_t)b * V * 3, nbt, u);
  const float bm = (float)a.B * (float)a.M;
  if (a.tn.p) {
    const F3 d = (a.dout[1] / bm) * one_minus_cos_dn(g.n, row(a.tn, b, j));
    tn_[0] = d.x; tn_[1] = d.y; tn_[2] = d.z;
  }
  if (a.tl.p) {
    const F3 d = (a.dout[3] * 2.0f / (3.0f * bm)) * (g.lap - row(a.tl, b, j));
    tl_[0] = d.x; tl_[1] = d.y; tl_[2] = d.z;
  }
}

// kSum = false: the first pass of the fixed-point scatter over the B*M target points, true: the second
template <bool kSum>
__global__ void __launch_bounds__(kThreads) scatter_kernel(Args a) {
  const GinLossPlanHdr* h = reinterpret_cast<const GinLossPlanHdr*>(a.plan);
  const int V = h->V;
  const int32_t* nbt = a.plan + h->ring_off;
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (long long)a.B * a.M) return;
  int b, u;
  float tn_[3], tl_[3];
  yx_terms(a, nbt, V, e, b, u, tn_, tl_);
  const long long r = (long long)b * V + u;
  if (a.tn.p) { if (kSum) fixsum::add(a.acc_n + r, tn_); else fixsum::note(a.acc_n + r, tn_); }
  if (a.tl.p) { if (kSum) fixsum::add(a.acc_l + r, tl_); else fixsum::note(a.acc_l + r, tl_); }
}

// g_n, g_L of vertex (b, i): the xy term (when i_xy is given) plus the fixed-point yx sum (when i_yx is given)
__global__ void __launch_bounds__(kThreads) cotangent_kernel(Args a) {
  const GinLossPlanHdr* h = reinterpret_cast<const GinLossPlanHdr*>(a.plan);
  const int V = h->V;
  const int32_t* nbt = a.plan + h->ring_off;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)a.B * V) return;
  const int b = (int)(t / V), i = (int)(t - (long long)b * V);
  float gn[3] = {0.f, 0.f, 0.f}, gl[3] = {0.f, 0.f, 0.f};
  if (a.idx_xy) {
    const int k = a.idx_xy[t];
    const Geom g = vertex_geom(a.v + (size_t)b * V * 3, nbt, i);
    const float bv = (float)a.B * (float)V;
    if (a.tn.p) {
      const F3 d = (a.dout[0] / bv) * one_minus_cos_dn(g.n, row(a.tn, b, k));
      gn[0] = d.x; gn[1] = d.y; gn[2] = d.z;
    }
    if (a.tl.p) {
      const F3 d = (a.dout[2] * 2.0f / (3.0f * bv)) * (g.lap - row(a.tl, b, k));
      gl[0] = d.x; gl[1] = d.y; gl[2] = d.z;
    }
  }
  if (a.idx_yx) {
    if (a.tn.p) fixsum::read(a.acc_n[t], gn);
    if (a.tl.p) fixsum::read(a.acc_l[t], gl);
  }
  if (a.tn.p) stv(a.g_n, t, f3(gn[0], gn[1], gn[2]));
  if (a.tl.p) stv(a.g_l, t, f3(gl[0], gl[1], gl[2]));
}

}  // namespace chamfer_terms
}  // namespace gin
