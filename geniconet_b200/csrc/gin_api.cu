// C ABI entry points (include/geniconet_b200.h): argument checking, plan validation, launches.
// No allocation, no device state; the only global is the launch counter and the per-thread
// error string.
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "../../include/geniconet_b200.h"
#include "gin_common.cuh"
#include "gin_gemm_simt.cuh"
#include "gin_gemm_tc.cuh"
#include "gin_gemm_tcp.cuh"
#include "gin_conv2.cuh"
#include "gin_conv2_pair.cuh"
#include "gin_wgrad2.cuh"
#include "gin_wgrad_tcp.cuh"
#include "gin_loss.cuh"
#include "gin_narrow.cuh"
#include "gin_adam.cuh"
#include "gin_bn.cuh"
#include "gin_resample.cuh"
#include "gin_dist.cuh"
#include "gin_chamfer.cuh"
#include "gin_chamfer_terms.cuh"
#include "gin_head.cuh"

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

void gin_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

namespace gin {
int cv2_launch_pair(cv2::Params& p, int nt, cudaStream_t st) { return nt == 128 ? cv2::launch_pair<128>(p, st) : cv2::launch_pair<64>(p, st); }
}  // namespace gin

namespace {

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  g_launches.fetch_add(1, std::memory_order_relaxed);
  if (e != cudaSuccess) return fail(GIN_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
  return GIN_OK;
}

// The launch geometry comes from the HOST copy of the plan (the blob gin_plan_build wrote); the
// kernels read the tables from the device copy.
const int32_t* plan_header(const void* plan_host) {
  const int32_t* w = reinterpret_cast<const int32_t*>(plan_host);
  if (!w || w[0] != GIN_MAGIC) { gin_set_error("plan_host is null or has a bad magic"); return nullptr; }
  return w;
}

int grid_for(long long work_items, int threads, int max_waves = 8) {
  long long blocks = (work_items + threads - 1) / threads;
  long long cap = 148LL * max_waves;
  if (blocks < 1) blocks = 1;
  return (int)(blocks < cap ? blocks : cap);
}

// GIN_TC_MODE (A/B experiments): "gather" forces the gather-mode tcgen05 kernels, "patch1" the first-generation patch kernels
// (three shifted copies); default is the second-generation patch kernels wherever a plan has patch tiles
int tc_mode() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("GIN_TC_MODE"); v = (e && strcmp(e, "gather") == 0) ? 0 : (e && strcmp(e, "patch1") == 0) ? 1 : 2; }
  return v;
}
bool patch_mode_enabled() { return tc_mode() >= 1; }
// Cross-seam remainder of dgrad: the row-gather kernel over signature-sorted slot tiles (default), or GIN_SEAM=patch: the regular
// form (GinPxSide, every tile runs all slots) through the patch kernel.  Measured equal within 5 % at I5 / B = 36 (both are bound
// by the latency of ~20-40 tiny stages per CTA, not by work), so the one that moves less data stays the default.
// GIN_SEAM: "fold" (default, r02): boundary tiles inside the in-chart launch (GinPfSide: complete values, masked in-chart stores,
// one launch); "patch": second launch of the patch kernel over GinPxSide (read-modify-write); "gather": second launch of the
// first-generation row-gather kernel.
int seam_mode() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("GIN_SEAM"); v = (e && strcmp(e, "gather") == 0) ? 0 : (e && strcmp(e, "patch") == 0) ? 1 : 2; }
  return v;
}
bool seam_v2_enabled() { return seam_mode() >= 1; }
bool seam_fold_ok(const GinPfSide& pf) { return seam_mode() == 2 && pf.ntiles > 0 && pf.nslots <= gin::cv2::MAX_PLANES && pf.mask_off > 0; }

// fp32 CUDA-core path
int run_gather_gemm_simt(const int32_t* plan_dev, const GinSide& side, int group, GinSrcView X, const char* packed, int B, int K, int N,
                         bool dgrad, const float* bias, float* Y, cudaStream_t st, int Cin, int Cout) {
  const int groups = (B + group - 1) / group;
  const long long ntiles = (long long)groups * side.ntiles;
  if (ntiles <= 0) return GIN_OK;
  const float* W = reinterpret_cast<const float*>(packed + (dgrad ? packed_off_wd(Cin, Cout) : packed_off_wf(Cin, Cout)));
  dim3 grid((unsigned)ntiles, (unsigned)((N + gin::SIMT_TN - 1) / gin::SIMT_TN));
  const bool vec = X.sc == 1 && (K % 4 == 0) && (X.sp % 4 == 0) && (X.sb % 4 == 0) && ((uintptr_t)X.p % 16 == 0);
  if (vec) gin::gather_gemm_simt_kernel<true><<<grid, gin::SIMT_THREADS, 0, st>>>(plan_dev, side, X, W, bias, Y, group, B, K, N);
  else gin::gather_gemm_simt_kernel<false><<<grid, gin::SIMT_THREADS, 0, st>>>(plan_dev, side, X, W, bias, Y, group, B, K, N);
  return check_launch("gather_gemm_simt");
}

// tcgen05 path on the bf16 activation copy: patch mode for stride 1, gather mode otherwise
int run_gemm_tc(const int32_t* plan_dev, const GinConvPlanHdr* h, const void* Xb, const char* packed, int B, bool dgrad,
                const float* bias, float* Y, cudaStream_t st, int Cin, int Cout, float* stats = nullptr, int* stats_parts = nullptr,
                const gin::Bias2& bias2 = {}) {
  if (stats_parts) *stats_parts = 0;
  const GinSide& side = dgrad ? h->dg : h->fwd;
  const int K = dgrad ? Cout : Cin, N = dgrad ? Cin : Cout;
  const int groups = (B + h->group - 1) / h->group;
  if (!gin::tc_supported(K, N)) return fail(GIN_ERR_UNSUPPORTED, "tcgen05 path needs channel counts that are multiples of 64 (K=%d N=%d)", K, N);
  const void* wb = packed + (dgrad ? packed_off_bd(Cin, Cout) : packed_off_bf(Cin, Cout));
  const GinPSide& ps = dgrad ? h->pdg : h->pfwd;
  int rc;
  // forward: activation copy x forward weight tiles (both the forward format); dgrad: dy copy x dgrad weight tiles (both bf16)
  const bool bf16 = dgrad || !gin::fwd_fp16();
  bool fold;                                          // dgrad: the boundary pixels are part of the in-chart launch
  if (h->stride == 1 && patch_mode_enabled() && gin::tcp_supported(ps, K, N)) {
    fold = dgrad && tc_mode() == 2 && gin::cv2_supported(ps, K, N) && seam_fold_ok(h->pf);
    if (tc_mode() == 2 && gin::cv2_supported(ps, K, N))
      rc = gin::launch_patch_conv2(plan_dev, ps, h->group, side.P_dst, 2 << h->level_in, Xb, wb, bias, bias2, Y, B, K, N, dgrad ? 1 : 0, bf16, st,
                                   dgrad ? nullptr : stats, dgrad ? nullptr : stats_parts, fold ? &h->pf : nullptr);
    else rc = gin::launch_patch_gemm_tc(plan_dev, ps, h->group, side.P_dst, Xb, wb, bias, Y, B, K, N, dgrad ? 1 : 0, bf16, st);
    if (rc != GIN_OK) return fail(rc, "tcgen05 patch-GEMM launch failed: %s", cudaGetErrorString(cudaGetLastError()));
  } else if (h->stride == 2 && tc_mode() == 2 && gin::cv2_supported(h->p2, K, N)) {
    // stride 2 in patch mode on the coarse lattice: four parity planes (gin_plan.h: GinP2Side)
    const int Pf = h->fwd.P_src, Pc = h->fwd.P_dst;
    fold = dgrad && seam_fold_ok(h->pf);
    if (!dgrad)
      rc = gin::launch_patch_conv2_s2_fwd(plan_dev, h->p2, h->group, Pf, Pc, 2 << h->level_out, Xb, wb, bias, bias2, Y, B, K, N, bf16, st, stats,
                                          stats_parts);
    else rc = gin::launch_patch_conv2_s2_dgrad(plan_dev, h->p2, h->group, Pf, Pc, 2 << h->level_in, Xb, wb, Y, B, K, N, bf16, st, fold ? &h->pf : nullptr);
    if (rc != GIN_OK) return fail(rc, "tcgen05 stride-2 patch launch failed: %s", cudaGetErrorString(cudaGetLastError()));
  } else {                                            // gather mode: the one launch covers the seams too
    rc = gin::launch_gather_gemm_tc(plan_dev, side, h->group, Xb, wb, bias, Y, B, K, N, groups * side.ntiles, bf16, st);
    if (rc != GIN_OK) return fail(rc, "tcgen05 gather-GEMM launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return GIN_OK;
  }
  g_launches.fetch_add(1, std::memory_order_relaxed);
  if (!dgrad || fold) return GIN_OK;
  // the cross-seam and pole entries of dgrad, added on top of the in-chart pass (side = h->dg: coarse dy -> fine dx at stride 2)
  if (tc_mode() == 2 && seam_v2_enabled() && gin::cv2_seam_supported(h->px, K, N)) {
    rc = gin::launch_patch_conv2_seam(plan_dev, h->px, h->group, side.P_src, side.P_dst, Xb, wb, Y, B, K, N, bf16, st);
    if (rc != GIN_OK) return fail(rc, "tcgen05 seam pass (v2) launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    g_launches.fetch_add(1, std::memory_order_relaxed);
  } else if (h->dgx.ntiles > 0) {
    rc = gin::launch_gather_gemm_tc(plan_dev, h->dgx, h->group, Xb, wb, nullptr, Y, B, K, N, groups * h->dgx.ntiles, bf16, st, 1);
    if (rc != GIN_OK) return fail(rc, "tcgen05 seam pass launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    g_launches.fetch_add(1, std::memory_order_relaxed);
  }
  return GIN_OK;
}

}  // namespace

extern "C" {

int gin_version(void) { return 200; }
int gin_forward_operand_is_fp16(void) { return gin::fwd_fp16() ? 1 : 0; }
const char* gin_last_error(void) { return g_err; }
int64_t gin_launch_count(void) { return (int64_t)g_launches.load(); }

size_t gin_hexconv_packed_bytes(int Cin, int Cout) {
  if (Cin <= 0 || Cout <= 0) return 0;
  return packed_total(Cin, Cout);
}

int gin_hexconv_pack_weights(const float* weight, void* packed, int Cin, int Cout, void* stream) {
  if (!weight || !packed || Cin <= 0 || Cout <= 0) return fail(GIN_ERR_ARG, "gin_hexconv_pack_weights: bad argument");
  char* pk = reinterpret_cast<char*>(packed);
  const long long n = 7LL * Cin * Cout;
  gin::pack_weights_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(
      weight, reinterpret_cast<float*>(pk + packed_off_wf(Cin, Cout)), reinterpret_cast<float*>(pk + packed_off_wd(Cin, Cout)),
      reinterpret_cast<unsigned short*>(pk + packed_off_bf(Cin, Cout)), reinterpret_cast<unsigned short*>(pk + packed_off_bd(Cin, Cout)),
      Cin, Cout, (int)gin::fwd_fp16());
  return check_launch("pack_weights");
}

int gin_hexconv_pack_weights_bf16(const float* w0, int Cout0, const float* w1, int Cout1, void* packed, int Cin, void* stream) {
  const int Cout = Cout0 + Cout1;
  if (!w0 || Cout0 <= 0 || Cout1 < 0 || (Cout1 > 0 && !w1) || !packed || Cin <= 0 || (Cin & 63) || (Cout & 63))
    return fail(GIN_ERR_ARG, "gin_hexconv_pack_weights_bf16: bad argument (channel counts must be multiples of 64)");
  char* pk = reinterpret_cast<char*>(packed);
  const long long n = 7LL * Cin * Cout;
  gin::launch_pdl(gin::pack_weights_bf16_kernel, dim3(grid_for(n, 256)), dim3(256), 0, (cudaStream_t)stream, 
      w0, Cout0, w1, reinterpret_cast<unsigned short*>(pk + packed_off_bf(Cin, Cout)), reinterpret_cast<unsigned short*>(pk + packed_off_bd(Cin, Cout)),
      Cin, Cout, (int)gin::fwd_fp16());
  return check_launch("pack_weights_bf16");
}

int gin_hexconv_pack_weights_bf16_multi(int n, const float* const* w0, const int* Cout0, const float* const* w1, const int* Cout1,
                                        void* const* packed, const int* Cin, void* stream) {
  if (n <= 0 || n > gin::PACK_MAX_JOBS || !w0 || !Cout0 || !w1 || !Cout1 || !packed || !Cin)
    return fail(GIN_ERR_ARG, "gin_hexconv_pack_weights_bf16_multi: bad argument (1..%d jobs)", gin::PACK_MAX_JOBS);
  gin::PackJobs J{};
  J.n = n; J.fwd_f16 = (int)gin::fwd_fp16();
  int blocks = 0;
  for (int j = 0; j < n; ++j) {
    const int Cout = Cout0[j] + Cout1[j];
    if (!w0[j] || Cout0[j] <= 0 || Cout1[j] < 0 || (Cout1[j] > 0 && !w1[j]) || !packed[j] || Cin[j] <= 0 || (Cin[j] & 63) || (Cout & 63))
      return fail(GIN_ERR_ARG, "gin_hexconv_pack_weights_bf16_multi: job %d: bad argument (channel counts must be multiples of 64)", j);
    char* pk = reinterpret_cast<char*>(packed[j]);
    J.w0[j] = w0[j]; J.w1[j] = w1[j]; J.cin[j] = Cin[j]; J.cout0[j] = Cout0[j]; J.cout[j] = Cout;
    J.bf[j] = reinterpret_cast<unsigned short*>(pk + packed_off_bf(Cin[j], Cout));
    J.bd[j] = reinterpret_cast<unsigned short*>(pk + packed_off_bd(Cin[j], Cout));
    J.first[j] = blocks;
    const long long nel = 7LL * Cin[j] * Cout;
    int nb = (int)((nel / 4 + 256 * 2 - 1) / (256 * 2));       // nel / 4 sixteen-byte chunks (both images), two per thread
    if (nb < 1) nb = 1;
    blocks += nb;
  }
  J.first[n] = blocks;
  gin::launch_pdl(gin::pack_weights_multi_kernel, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, J);
  return check_launch("pack_weights_multi");
}

static int conv_hdr(const void* plan_host, const void* plan_dev, const GinConvPlanHdr** out) {
  if (!plan_dev) return fail(GIN_ERR_ARG, "null plan");
  const int32_t* w = plan_header(plan_host);
  if (!w) return GIN_ERR_PLAN;
  const GinConvPlanHdr* h = reinterpret_cast<const GinConvPlanHdr*>(w);
  if (h->kind != GIN_PLAN_HEXCONV) return fail(GIN_ERR_PLAN, "plan is not a hexconv plan (kind %d)", h->kind);
  *out = h;
  return GIN_OK;
}

// the forward of this plan and size runs the second-generation patch kernel (gin_conv2.cuh)
static bool fwd_v2_ok(const GinConvPlanHdr* h, int Cin, int Cout) {
  return tc_mode() == 2 && gin::tc_supported(Cin, Cout) &&
         (h->stride == 1 ? (patch_mode_enabled() && gin::tcp_supported(h->pfwd, Cin, Cout) && gin::cv2_supported(h->pfwd, Cin, Cout))
                         : gin::cv2_supported(h->p2, Cin, Cout));
}

int gin_hexconv_fwd(const void* plan_host, const void* plan_dev, const float* x, int64_t sb, int64_t sp, int64_t sc, const void* packed,
                    const float* bias, float* y, int B, int Cin, int Cout, int impl, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!x || !packed || !y || B < 0 || Cin <= 0 || Cout <= 0) return fail(GIN_ERR_ARG, "gin_hexconv_fwd: bad argument");
  const GinConvPlanHdr* h;
  int rc = conv_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  if (B == 0) return GIN_OK;
  if (impl == GIN_IMPL_TC) return fail(GIN_ERR_UNSUPPORTED, "the tcgen05 path reads bf16: use gin_cast_bf16 + gin_hexconv_fwd_bf16");
  GinSrcView X{x, (long long)sb, (long long)sp, (long long)sc, h->fwd.P_src};
  if (impl == GIN_IMPL_AUTO && gin::narrow_supported(Cin, Cout, h->fwd)) {     // xyz input layer: warp-level memory-bound kernel
    const float* wf = reinterpret_cast<const float*>(reinterpret_cast<const char*>(packed) + packed_off_wf(Cin, Cout));
    rc = gin::launch_narrow_fwd(plan_words(plan_dev), h->fwd, h->group, X, wf, bias, y, B, Cin, Cout, st);
    if (rc != GIN_OK) return fail(rc, "narrow forward launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return GIN_OK;
  }
  return run_gather_gemm_simt(plan_words(plan_dev), h->fwd, h->group, X, reinterpret_cast<const char*>(packed), B, Cin, Cout, false,
                              bias, y, st, Cin, Cout);
}

size_t gin_hexconv_narrow_stats_ws_bytes(int Cout) { return Cout <= 0 ? 0 : (size_t)148 * 4 * 2 * Cout * 4; }

int gin_hexconv_fwd_narrow_stats(const void* plan_host, const void* plan_dev, const float* x, int64_t sb, int64_t sp, int64_t sc, const void* packed,
                                 const float* bias, void* y, int y_fp16, int B, int Cin, int Cout, float* stats_ws, int* nparts, void* stream) {
  if (!x || !packed || !y || !stats_ws || !nparts || B <= 0 || Cin <= 0 || Cout <= 0) return fail(GIN_ERR_ARG, "gin_hexconv_fwd_narrow_stats: bad argument");
  const GinConvPlanHdr* h;
  int rc = conv_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  if (!gin::narrow_supported(Cin, Cout, h->fwd)) return fail(GIN_ERR_UNSUPPORTED, "gin_hexconv_fwd_narrow_stats: only the xyz input layer (Cin = 3, Cout = 64 | 128)");
  GinSrcView X{x, (long long)sb, (long long)sp, (long long)sc, h->fwd.P_src};
  const float* wf = reinterpret_cast<const float*>(reinterpret_cast<const char*>(packed) + packed_off_wf(Cin, Cout));
  rc = gin::launch_narrow_fwd(plan_words(plan_dev), h->fwd, h->group, X, wf, bias, reinterpret_cast<float*>(y), B, Cin, Cout, (cudaStream_t)stream, stats_ws, nparts,
                              y_fp16 ? 1 : 0);
  if (rc != GIN_OK) return fail(rc, "narrow forward launch failed: %s", cudaGetErrorString(cudaGetLastError()));
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return GIN_OK;
}

int gin_hexconv_dgrad(const void* plan_host, const void* plan_dev, const float* dy, const void* packed, float* dx, int B, int Cin, int Cout, int impl,
                      void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!dy || !packed || !dx || B < 0 || Cin <= 0 || Cout <= 0) return fail(GIN_ERR_ARG, "gin_hexconv_dgrad: bad argument");
  const GinConvPlanHdr* h;
  int rc = conv_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  if (B == 0) return GIN_OK;
  if (impl == GIN_IMPL_TC) return fail(GIN_ERR_UNSUPPORTED, "the tcgen05 path reads bf16: use gin_cast_bf16 + gin_hexconv_dgrad_bf16");
  GinSrcView X{dy, (long long)h->dg.P_src * Cout, (long long)Cout, 1, h->dg.P_src};
  return run_gather_gemm_simt(plan_words(plan_dev), h->dg, h->group, X, reinterpret_cast<const char*>(packed), B, Cout, Cin, true,
                              nullptr, dx, st, Cin, Cout);
}

// workspace: [dWp: 7*Cin*Cout fp32][split-K partial sums of the second-generation tcgen05 wgrad]
size_t gin_hexconv_wgrad_ws_bytes(int Cin, int Cout) {
  if (Cin <= 0 || Cout <= 0) return 0;
  size_t n = (size_t)28 * Cin * Cout;
  if (gin::tc_supported(Cin, Cout)) n += gin::wg2::partial_bytes(Cin, Cout);
  if (Cin == 3) n += gin::narrow::wgrad_partial_bytes(Cin, Cout);       // per-CTA sums of the xyz-layer kernel
  return n;
}

static int wgrad_common(const GinConvPlanHdr* h, const void* plan_dev, const float* x, int64_t sb, int64_t sp, int64_t sc, const void* xb,
                        const void* dyb, const float* dy, float* dW, float* db, void* ws, int B, int Cin, int Cout, cudaStream_t st,
                        int impl = GIN_IMPL_SIMT) {
  float* dWp = reinterpret_cast<float*>(ws);
  int rc;
  const bool bf16 = true;                                  // A = the bf16 twin of the forward activation copy, B = the bf16 dy copy
  const bool wg2_s1 = h->stride == 1 && gin::wg2_supported(h->pfwd, Cin, Cout), wg2_s2 = h->stride == 2 && gin::wg2_supported(h->p2, Cin, Cout);
  if (xb && B > 0 && tc_mode() == 2 && (wg2_s1 || wg2_s2)) {
    // second-generation patch wgrad: split-K partials in the workspace, reduced (and laid out as dW[Cout][Cin][7]) by a second kernel
    float* partial = dWp + (size_t)7 * Cin * Cout;
    if (wg2_s1) rc = gin::launch_wgrad_patch2(plan_words(plan_dev), h->pfwd, h->group, h->fwd.P_dst, xb, dyb, partial, dW, B, Cin, Cout, bf16, st);
    else rc = gin::launch_wgrad_patch2_s2(plan_words(plan_dev), h->p2, h->group, h->fwd.P_src, h->fwd.P_dst, xb, dyb, partial, dW, B, Cin, Cout, bf16, st);
    if (rc != GIN_OK) return fail(rc, "tcgen05 patch wgrad (v2) launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    g_launches.fetch_add(2, std::memory_order_relaxed);
    if (db) {
      if (cudaMemsetAsync(db, 0, (size_t)4 * Cout, st) != cudaSuccess) return fail(GIN_ERR_CUDA, "memset failed");
      const long long rows = (long long)B * h->fwd.P_dst;
      int ctas = (int)((rows + 255) / 256);
      if (ctas > 148 * 2) ctas = 148 * 2;
      gin::bias_grad_kernel<<<ctas, 256, 0, st>>>(dy, db, rows, Cout, (int)((rows + ctas - 1) / ctas));
      if ((rc = check_launch("bias_grad"))) return rc;
    }
    return GIN_OK;
  }
  if (cudaMemsetAsync(dWp, 0, (size_t)28 * Cin * Cout, st) != cudaSuccess) return fail(GIN_ERR_CUDA, "memset failed");
  if (db && cudaMemsetAsync(db, 0, (size_t)4 * Cout, st) != cudaSuccess) return fail(GIN_ERR_CUDA, "memset failed");
  if (B > 0) {
    const GinSide& side = h->fwd;
    const int groups = (B + h->group - 1) / h->group;
    const int total_tiles = groups * side.ntiles;
    if (xb) {
      if (!gin::tc_wgrad_supported(Cin, Cout)) return fail(GIN_ERR_UNSUPPORTED, "tcgen05 wgrad needs Cin %% 64 == 0 and Cout %% 64 == 0");
      if (h->stride == 1 && patch_mode_enabled() && gin::tcwp_supported(h->pfwd, Cin, Cout)) {
        rc = gin::launch_wgrad_patch_tc(plan_words(plan_dev), h->pfwd, h->group, side.P_dst, xb, dyb, dWp, B, Cin, Cout, bf16, st);
        if (rc != GIN_OK) return fail(rc, "tcgen05 patch wgrad launch failed: %s", cudaGetErrorString(cudaGetLastError()));
      } else {
        rc = gin::launch_wgrad_tc(plan_words(plan_dev), side, h->group, xb, dyb, dWp, B, Cin, Cout, total_tiles, bf16, st);
        if (rc != GIN_OK) return fail(rc, "tcgen05 wgrad launch failed: %s", cudaGetErrorString(cudaGetLastError()));
      }
      g_launches.fetch_add(1, std::memory_order_relaxed);
    } else if (impl == GIN_IMPL_AUTO && gin::narrow_supported(Cin, Cout, side)) {
      GinSrcView X{x, (long long)sb, (long long)sp, (long long)sc, side.P_src};
      rc = gin::launch_narrow_wgrad(plan_words(plan_dev), side, h->group, X, dy, dWp, db, dWp + (size_t)7 * Cin * Cout, B, Cin, Cout, st);   // db comes with it
      if (rc != GIN_OK) return fail(rc, "narrow wgrad launch failed: %s", cudaGetErrorString(cudaGetLastError()));
      g_launches.fetch_add(2, std::memory_order_relaxed);
      db = nullptr;
    } else {
      GinSrcView X{x, (long long)sb, (long long)sp, (long long)sc, side.P_src};
      const int nblk = ((Cin + gin::WG_TC - 1) / gin::WG_TC) * ((Cout + gin::WG_TC - 1) / gin::WG_TC);
      int slices = (148 * 4 + 7 * nblk - 1) / (7 * nblk);
      if (slices > total_tiles) slices = total_tiles;
      if (slices < 1) slices = 1;
      const int tiles_per_cta = (total_tiles + slices - 1) / slices;
      dim3 grid((unsigned)((total_tiles + tiles_per_cta - 1) / tiles_per_cta), 7, (unsigned)nblk);
      const bool vec = sc == 1 && (Cin % 4 == 0) && (sp % 4 == 0) && (sb % 4 == 0) && ((uintptr_t)x % 16 == 0);
      if (vec) gin::wgrad_simt_kernel<true><<<grid, 256, 0, st>>>(plan_words(plan_dev), side, X, dy, dWp, h->group, B, Cin, Cout, tiles_per_cta, total_tiles);
      else gin::wgrad_simt_kernel<false><<<grid, 256, 0, st>>>(plan_words(plan_dev), side, X, dy, dWp, h->group, B, Cin, Cout, tiles_per_cta, total_tiles);
      rc = check_launch("wgrad_simt");
      if (rc) return rc;
    }
    if (db) {
      const long long rows = (long long)B * side.P_dst;
      int ctas = (int)((rows + 255) / 256);
      if (ctas > 148 * 2) ctas = 148 * 2;
      const int rows_per_cta = (int)((rows + ctas - 1) / ctas);
      gin::bias_grad_kernel<<<ctas, 256, 0, st>>>(dy, db, rows, Cout, rows_per_cta);
      rc = check_launch("bias_grad");
      if (rc) return rc;
    }
  }
  gin::unpack_wgrad_kernel<<<grid_for(7LL * Cin * Cout, 256), 256, 0, st>>>(dWp, dW, Cin, Cout);
  return check_launch("unpack_wgrad");
}

int gin_hexconv_wgrad(const void* plan_host, const void* plan_dev, const float* x, int64_t sb, int64_t sp, int64_t sc, const float* dy, float* dW,
                      float* db, void* ws, int B, int Cin, int Cout, int impl, void* stream) {
  if (!x || !dy || !dW || !ws || B < 0 || Cin <= 0 || Cout <= 0) return fail(GIN_ERR_ARG, "gin_hexconv_wgrad: bad argument");
  if (impl == GIN_IMPL_TC) return fail(GIN_ERR_UNSUPPORTED, "the tcgen05 path reads bf16: use gin_cast_bf16 + gin_hexconv_wgrad_bf16");
  const GinConvPlanHdr* h;
  int rc = conv_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  return wgrad_common(h, plan_dev, x, sb, sp, sc, nullptr, nullptr, dy, dW, db, ws, B, Cin, Cout, (cudaStream_t)stream, impl);
}

// ------------------------------------------------------------------ bf16 (tcgen05) entry points
size_t gin_cast_bf16_bytes(int B, int level, int C) {
  if (B < 0 || level < 0 || level > 9 || C <= 0) return 0;
  return ((size_t)B * (10 << (2 * level)) + 2 * (size_t)B) * C * 2;
}

int gin_cast_bf16(const void* plan_host, const void* plan_dev, int which, const float* x, void* xb, int B, int C, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!x || !xb || B < 0 || C <= 0 || (C & 7) || which < 0 || which > 2) return fail(GIN_ERR_ARG, "gin_cast_bf16: bad argument (C must be a multiple of 8)");
  const GinConvPlanHdr* h;
  int rc = conv_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  if (B == 0) return GIN_OK;
  const GinSide& side = which != 1 ? h->fwd : h->dg;      // the gathered tensor of the forward / of dgrad
  const long long n8 = (long long)B * side.P_src * (C / 8) + 2LL * B * (C / 8);
  gin::cast_bf16_kernel<<<grid_for(n8, 256, 16), 256, 0, st>>>(x, reinterpret_cast<__nv_bfloat16*>(xb), plan_words(plan_dev) + side.ring_off,
                                                                B, side.P_src, C, (int)(which == 0 && gin::fwd_fp16()));
  return check_launch("cast_bf16");
}

size_t gin_cast_bf16_colsum_ws_bytes(int C) { return C <= 0 ? 0 : (size_t)gin::CAST_COLSUM_MAX_CTAS * C * 4; }

int gin_cast_bf16_colsum(const void* plan_host, const void* plan_dev, int which, const float* x, void* xb, float* colsum, void* ws, int B, int C,
                         void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!x || !xb || !colsum || !ws || B < 0 || C <= 0 || (C & 7) || (256 % (C >> 3)) || (which != 0 && which != 1))
    return fail(GIN_ERR_ARG, "gin_cast_bf16_colsum: bad argument (C/8 must divide 256)");
  const GinConvPlanHdr* h;
  int rc = conv_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  if (B == 0) return cudaMemsetAsync(colsum, 0, (size_t)C * 4, st) == cudaSuccess ? GIN_OK : fail(GIN_ERR_CUDA, "memset failed");
  const GinSide& side = which == 0 ? h->fwd : h->dg;
  const long long n8 = (long long)B * side.P_src * (C / 8) + 2LL * B * (C / 8);
  int ctas = grid_for(n8, 256, 2);
  if (ctas > gin::CAST_COLSUM_MAX_CTAS) ctas = gin::CAST_COLSUM_MAX_CTAS;
  gin::cast_bf16_colsum_kernel<<<ctas, 256, 0, st>>>(x, reinterpret_cast<__nv_bfloat16*>(xb), plan_words(plan_dev) + side.ring_off, B,
                                                      side.P_src, C, reinterpret_cast<float*>(ws), (int)(which == 0 && gin::fwd_fp16()));
  if ((rc = check_launch("cast_bf16_colsum"))) return rc;
  gin::colsum_final_kernel<<<(C + 7) / 8, 256, 0, st>>>(reinterpret_cast<const float*>(ws), colsum, C, ctas);
  return check_launch("colsum_final");
}

int gin_hexconv_fwd_bf16(const void* plan_host, const void* plan_dev, const void* xb, const void* packed, const float* bias, float* y, int B,
                         int Cin, int Cout, void* stream) {
  if (!xb || !packed || !y || B < 0 || Cin <= 0 || Cout <= 0) return fail(GIN_ERR_ARG, "gin_hexconv_fwd_bf16: bad argument");
  const GinConvPlanHdr* h;
  int rc = conv_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  if (B == 0) return GIN_OK;
  return run_gemm_tc(plan_words(plan_dev), h, xb, reinterpret_cast<const char*>(packed), B, false, bias, y, (cudaStream_t)stream, Cin, Cout);
}

int gin_hexconv_fwd_bf16_stats(const void* plan_host, const void* plan_dev, const void* xb, const void* packed, const float* bias, float* y, int B,
                               int Cin, int Cout, float* stats_ws, int* nparts, void* stream) {
  if (!xb || !packed || !y || !stats_ws || !nparts || B <= 0 || Cin <= 0 || Cout <= 0) return fail(GIN_ERR_ARG, "gin_hexconv_fwd_bf16_stats: bad argument");
  const GinConvPlanHdr* h;
  int rc = conv_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  return run_gemm_tc(plan_words(plan_dev), h, xb, reinterpret_cast<const char*>(packed), B, false, bias, y, (cudaStream_t)stream, Cin, Cout, stats_ws,
                     nparts);
}

int gin_hexconv_fwd_bf16_stats2(const void* plan_host, const void* plan_dev, const void* xb, const void* packed, const float* bias0,
                                const float* bias1, int split, void* y, int y_fp16, int B, int Cin, int Cout, float* stats_ws, int* nparts,
                                void* stream) {
  if (!bias0 || (bias1 && (split <= 0 || split >= Cout || (split & 63)))) return fail(GIN_ERR_ARG, "gin_hexconv_fwd_bf16_stats2: bad bias split");
  const GinConvPlanHdr* h;
  int rc = conv_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  if (!fwd_v2_ok(h, Cin, Cout)) return fail(GIN_ERR_UNSUPPORTED, "gin_hexconv_fwd_bf16_stats2: this plan / size does not run the second-generation patch kernel");
  if (!xb || !packed || !y || !stats_ws || !nparts || B <= 0 || Cin <= 0 || Cout <= 0) return fail(GIN_ERR_ARG, "gin_hexconv_fwd_bf16_stats2: bad argument");
  const gin::Bias2 bias2{bias1, bias1 ? split : 0, y_fp16 ? 1 : 0};
  return run_gemm_tc(plan_words(plan_dev), h, xb, reinterpret_cast<const char*>(packed), B, false, bias0, reinterpret_cast<float*>(y), (cudaStream_t)stream,
                     Cin, Cout, stats_ws, nparts, bias2);
}

size_t gin_hexconv_affine_ring_bytes(int B, int Cout) { return (B <= 0 || Cout <= 0) ? 0 : (size_t)B * 10 * Cout * 4; }

int gin_hexconv_fwd_affine(const void* plan_host, const void* plan_dev, const void* xb, const void* packed, const float* scale, const float* shift,
                           int relu_split, const void* res, int64_t ld_res, int res_fp16, int split, void* out0_b, float* out0_f, void* out1_b,
                           float* out1_f, float* ring_ws, int B, int Cin, int Cout, void* stream) {
  const bool two = split < Cout;
  if (!xb || !packed || !scale || !shift || B <= 0 || Cin <= 0 || Cout <= 0 || relu_split < 0 || relu_split > Cout)
    return fail(GIN_ERR_ARG, "gin_hexconv_fwd_affine: bad argument");
  if (split <= 0 || split > Cout || (split & 63)) return fail(GIN_ERR_ARG, "gin_hexconv_fwd_affine: split must be a multiple of 64 in (0, Cout]");
  if ((!out0_b && !out0_f) || (two ? (!out1_b && !out1_f) : (out1_b || out1_f)))
    return fail(GIN_ERR_ARG, "gin_hexconv_fwd_affine: every destination needs an output (and split == Cout has no second one)");
  if (res && (ld_res < Cout || (ld_res & 3))) return fail(GIN_ERR_ARG, "gin_hexconv_fwd_affine: ld_res must be >= Cout and a multiple of 4");
  if ((out0_b || out1_b) && !ring_ws) return fail(GIN_ERR_ARG, "gin_hexconv_fwd_affine: an operand copy needs ring_ws");
  const GinConvPlanHdr* h;
  int rc = conv_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  if (!fwd_v2_ok(h, Cin, Cout)) return fail(GIN_ERR_UNSUPPORTED, "gin_hexconv_fwd_affine: this plan / size does not run the second-generation patch kernel");
  if ((long long)B * h->fwd.P_dst + 2LL * B >= 0x7fffffffLL) return fail(GIN_ERR_UNSUPPORTED, "gin_hexconv_fwd_affine: B*P too large");
  cudaStream_t st = (cudaStream_t)stream;
  const int f16 = (int)gin::fwd_fp16();
  gin::cv2::Affine a{};
  a.scale = scale; a.shift = shift; a.relu_split = relu_split; a.res = res; a.res_ld = ld_res; a.res_f16 = res_fp16 ? 1 : 0; a.split = split;
  a.op[0] = out0_b; a.f32[0] = out0_f; a.ld[0] = split; a.ring[0] = ring_ws;
  a.op[1] = out1_b; a.f32[1] = out1_f; a.ld[1] = Cout - split; a.ring[1] = ring_ws + (size_t)B * 10 * split;
  a.op_f16 = f16;
  const void* wb = reinterpret_cast<const char*>(packed) + packed_off_bf(Cin, Cout);
  if (h->stride == 1)
    rc = gin::launch_patch_conv2(plan_words(plan_dev), h->pfwd, h->group, h->fwd.P_dst, 2 << h->level_in, xb, wb, nullptr, {}, nullptr, B, Cin, Cout, 0,
                                 !f16, st, nullptr, nullptr, nullptr, &a);
  else
    rc = gin::launch_patch_conv2_s2_fwd(plan_words(plan_dev), h->p2, h->group, h->fwd.P_src, h->fwd.P_dst, 2 << h->level_out, xb, wb, nullptr, {},
                                        nullptr, B, Cin, Cout, !f16, st, nullptr, nullptr, &a);
  if (rc != GIN_OK) return fail(rc, "gin_hexconv_fwd_affine: launch failed: %s", cudaGetErrorString(cudaGetLastError()));
  g_launches.fetch_add(1, std::memory_order_relaxed);
  for (int d = 0; d < 2; ++d) {
    if (!a.op[d]) continue;
    const long long work = 2LL * B * (a.ld[d] >> 3);
    gin::launch_pdl(gin::bn::pole_mean_kernel, dim3(grid_for(work, 256)), dim3(256), 0, st, (const float*)a.ring[d],
                    reinterpret_cast<__nv_bfloat16*>(a.op[d]), (long long)B * h->fwd.P_dst, B, a.ld[d], f16);
    if ((rc = check_launch("pole_mean"))) return rc;
  }
  return GIN_OK;
}

int gin_bn_eval_consts(const void* table_dev, int count, int max_C, void* stream) {
  static_assert(sizeof(gin::bn::EvalEntry) == sizeof(GinBnEvalEntry), "GinBnEvalEntry layout");
  if (count == 0) return GIN_OK;
  if (!table_dev || count < 0 || count > 65535 || max_C <= 0) return fail(GIN_ERR_ARG, "gin_bn_eval_consts: bad argument");
  gin::launch_pdl(gin::bn::eval_consts_kernel, dim3((max_C + 255) / 256, count), dim3(256), 0, (cudaStream_t)stream,
                  reinterpret_cast<const gin::bn::EvalEntry*>(table_dev));
  return check_launch("bn_eval_consts");
}

int gin_hexconv_dgrad_bf16(const void* plan_host, const void* plan_dev, const void* dyb, const void* packed, float* dx, int B, int Cin, int Cout,
                           void* stream) {
  if (!dyb || !packed || !dx || B < 0 || Cin <= 0 || Cout <= 0) return fail(GIN_ERR_ARG, "gin_hexconv_dgrad_bf16: bad argument");
  const GinConvPlanHdr* h;
  int rc = conv_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  if (B == 0) return GIN_OK;
  return run_gemm_tc(plan_words(plan_dev), h, dyb, reinterpret_cast<const char*>(packed), B, true, nullptr, dx, (cudaStream_t)stream, Cin, Cout);
}

int gin_hexconv_wgrad_bf16(const void* plan_host, const void* plan_dev, const void* xb, const void* dyb, const float* dy, float* dW, float* db,
                           void* ws, int B, int Cin, int Cout, void* stream) {
  if (!xb || !dyb || !dW || !ws || (db && !dy) || B < 0 || Cin <= 0 || Cout <= 0) return fail(GIN_ERR_ARG, "gin_hexconv_wgrad_bf16: bad argument");
  const GinConvPlanHdr* h;
  int rc = conv_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  return wgrad_common(h, plan_dev, nullptr, 0, 0, 0, xb, dyb, dy, dW, db, ws, B, Cin, Cout, (cudaStream_t)stream);
}

static int up_hdr(const void* plan_host, const void* plan_dev, const GinUpPlanHdr** out) {
  if (!plan_dev) return fail(GIN_ERR_ARG, "null plan");
  const int32_t* w = plan_header(plan_host);
  if (!w) return GIN_ERR_PLAN;
  const GinUpPlanHdr* h = reinterpret_cast<const GinUpPlanHdr*>(w);
  if (h->kind != GIN_PLAN_UPSAMPLE) return fail(GIN_ERR_PLAN, "plan is not an upsample plan (kind %d)", h->kind);
  *out = h;
  return GIN_OK;
}

int gin_upsample_fwd(const void* plan_host, const void* plan_dev, const float* x, float* y, int B, int C, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!x || !y || B < 0 || C <= 0 || (C & 3)) return fail(GIN_ERR_ARG, "gin_upsample_fwd: bad argument (C must be a multiple of 4)");
  const GinUpPlanHdr* h;
  int rc = up_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  if (B == 0) return GIN_OK;
  const long long work = (long long)B * h->Pf * (C / 4);
  gin::upsample_fwd_kernel<<<grid_for(work, 256, 16), 256, 0, st>>>(plan_words(plan_dev), x, y, B, C);
  return check_launch("upsample_fwd");
}

int gin_upsample_bwd(const void* plan_host, const void* plan_dev, const float* dy, float* dx, int B, int C, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!dy || !dx || B < 0 || C <= 0 || (C & 3)) return fail(GIN_ERR_ARG, "gin_upsample_bwd: bad argument (C must be a multiple of 4)");
  const GinUpPlanHdr* h;
  int rc = up_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  if (B == 0) return GIN_OK;
  const long long work = (long long)B * h->Pc * (C / 4);
  if (work < 0x7fffffffLL) gin::upsample_bwd_kernel<unsigned><<<grid_for(work, 256, 16), 256, 0, st>>>(plan_words(plan_dev), dy, dx, B, C);
  else gin::upsample_bwd_kernel<long long><<<grid_for(work, 256, 16), 256, 0, st>>>(plan_words(plan_dev), dy, dx, B, C);
  return check_launch("upsample_bwd");
}

static int reparam_fwd_impl(const float* mu, const float* logvar, float* eps, float* z, int64_t n, uint64_t seed, uint64_t offset,
                            uint64_t* step, void* stream) {
  if (!mu || !logvar || !eps || !z || n < 0) return fail(GIN_ERR_ARG, "gin_reparam_fwd: bad argument");
  if (n == 0) return GIN_OK;
  if (((uintptr_t)mu | (uintptr_t)logvar | (uintptr_t)eps | (uintptr_t)z) % 16) return fail(GIN_ERR_ARG, "gin_reparam_fwd: pointers must be 16-byte aligned");
  gin::reparam_fwd_kernel<<<grid_for((n + 3) / 4, 256), 256, 0, (cudaStream_t)stream>>>(mu, logvar, eps, z, n, seed, offset,
                                                                                        reinterpret_cast<const unsigned long long*>(step));
  int rc = check_launch("reparam_fwd");
  if (rc || !step) return rc;
  gin::counter_inc_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(reinterpret_cast<unsigned long long*>(step));
  return check_launch("counter_inc");
}

int gin_reparam_fwd(const float* mu, const float* logvar, float* eps, float* z, int64_t n, uint64_t seed, uint64_t offset, void* stream) {
  return reparam_fwd_impl(mu, logvar, eps, z, n, seed, offset, nullptr, stream);
}

int gin_reparam_fwd_step(const float* mu, const float* logvar, float* eps, float* z, int64_t n, uint64_t seed, uint64_t offset, uint64_t* step,
                         void* stream) {
  if (!step) return fail(GIN_ERR_ARG, "gin_reparam_fwd_step: null step counter");
  return reparam_fwd_impl(mu, logvar, eps, z, n, seed, offset, step, stream);
}

int gin_reparam_bwd(const float* dz, const float* logvar, const float* eps, float* dmu, float* dlogvar, int64_t n, void* stream) {
  if (!dz || !logvar || !eps || !dmu || !dlogvar || n < 0) return fail(GIN_ERR_ARG, "gin_reparam_bwd: bad argument");
  if (n == 0) return GIN_OK;
  gin::reparam_bwd_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(dz, logvar, eps, dmu, dlogvar, n);
  return check_launch("reparam_bwd");
}

int gin_kld_fwd(const float* mu, const float* logvar, float* out, void* ws, int64_t n, void* stream) {
  if (!mu || !logvar || !out || !ws || n <= 0) return fail(GIN_ERR_ARG, "gin_kld_fwd: bad argument");
  int parts = grid_for(n, 256, 2);
  if (parts > 512) parts = 512;
  gin::kld_partial_kernel<<<parts, 256, 0, (cudaStream_t)stream>>>(mu, logvar, reinterpret_cast<double*>(ws), n);
  int rc = check_launch("kld_partial");
  if (rc) return rc;
  gin::kld_final_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const double*>(ws), parts, out, -0.5 / (double)n);
  return check_launch("kld_final");
}

int gin_kld_bwd(const float* mu, const float* logvar, const float* dout, float scale, float* dmu, float* dlogvar, int64_t n,
                void* stream) {
  if (!mu || !logvar || !dout || !dmu || !dlogvar || n <= 0) return fail(GIN_ERR_ARG, "gin_kld_bwd: bad argument");
  gin::kld_bwd_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(mu, logvar, dout, scale * (float)(-0.5 / (double)n), dmu,
                                                                         dlogvar, n);
  return check_launch("kld_bwd");
}

// ------------------------------------------------------------------ decoder head: 1x1 conv + tanh
size_t gin_head_ws_bytes(void) { return (size_t)gin::head::MAX_CTAS * gin::head::PART * sizeof(float); }

static int head_args_ok(const char* what, int B, int64_t P, int Cin, int Cout) {
  if (B < 0 || P <= 0) return fail(GIN_ERR_ARG, "%s: bad sizes B=%d P=%lld", what, B, (long long)P);
  if (Cin != gin::head::CIN || Cout != gin::head::COUT) return fail(GIN_ERR_UNSUPPORTED, "%s: only %d -> %d channels (got %d -> %d)", what, gin::head::CIN, gin::head::COUT, Cin, Cout);
  return GIN_OK;
}

int gin_head_fwd(const float* x, const float* w, const float* bias, float* y, int B, int64_t P, int Cin, int Cout, void* stream) {
  int rc = head_args_ok("gin_head_fwd", B, P, Cin, Cout);
  if (rc != GIN_OK || B == 0) return rc;
  if (!x || !w || !bias || !y) return fail(GIN_ERR_ARG, "gin_head_fwd: null pointer");
  if (((uintptr_t)x | (uintptr_t)w) & 15) return fail(GIN_ERR_ARG, "gin_head_fwd: x and w must be 16-byte aligned");
  const long long rows = (long long)B * P;
  gin::launch_pdl(gin::head::fwd_kernel, dim3(gin::head::grid_for_rows(rows)), dim3(gin::head::kThreads), 0, (cudaStream_t)stream, x, w, bias, y, rows, P);
  return check_launch("head_fwd");
}

int gin_head_bwd(const float* x, const float* w, const float* y, const float* dy, float* dx, float* dw, float* db, void* ws, int B, int64_t P,
                 int Cin, int Cout, void* stream) {
  int rc = head_args_ok("gin_head_bwd", B, P, Cin, Cout);
  if (rc != GIN_OK) return rc;
  if (!x || !w || !y || !dy || !dx || !dw || !db || !ws) return fail(GIN_ERR_ARG, "gin_head_bwd: null pointer");
  if (((uintptr_t)x | (uintptr_t)w | (uintptr_t)dx) & 15) return fail(GIN_ERR_ARG, "gin_head_bwd: x, w and dx must be 16-byte aligned");
  const long long rows = (long long)B * P;
  cudaStream_t st = (cudaStream_t)stream;
  const int grid = gin::head::grid_for_rows(rows);
  gin::launch_pdl(gin::head::bwd_kernel, dim3(grid), dim3(gin::head::kThreads), 0, st, x, w, y, dy, dx, (float*)ws, rows, P);
  rc = check_launch("head_bwd");
  if (rc != GIN_OK) return rc;
  gin::launch_pdl(gin::head::bwd_final_kernel, dim3((gin::head::COUT * gin::head::CIN + gin::head::COUT + 7) / 8), dim3(256), 0, st, (const float*)ws, grid, dw, db);
  return check_launch("head_bwd_final");
}

// ------------------------------------------------------------------ evaluation metric: point-to-mesh distance
size_t gin_point_mesh_ws_bytes(int B, int N) { return (B <= 0 || N <= 0) ? 0 : (size_t)B * N * sizeof(unsigned long long); }

int gin_point_mesh_distance(const float* points, const float* verts, const int32_t* faces, float* dist, int32_t* face_idx, void* ws, int B,
                            int N, int V, int F, void* stream) {
  if (B < 0 || N < 0 || V <= 0 || F <= 0) return fail(GIN_ERR_ARG, "gin_point_mesh_distance: bad sizes B=%d N=%d V=%d F=%d", B, N, V, F);
  if (B == 0 || N == 0) return GIN_OK;
  if (!points || !verts || !faces || !dist || !ws) return fail(GIN_ERR_ARG, "gin_point_mesh_distance: null pointer");
  if (B > 65535) return fail(GIN_ERR_ARG, "gin_point_mesh_distance: B=%d exceeds 65535", B);
  cudaStream_t st = (cudaStream_t)stream;
  const size_t n = (size_t)B * N;
  if (cudaMemsetAsync(ws, 0xFF, n * sizeof(unsigned long long), st) != cudaSuccess) return fail(GIN_ERR_CUDA, "gin_point_mesh_distance: memset failed");
  dim3 grid((N + gin::dist::kThreads - 1) / gin::dist::kThreads, (F + gin::dist::kChunk - 1) / gin::dist::kChunk, B);
  if (grid.y > 65535) return fail(GIN_ERR_ARG, "gin_point_mesh_distance: F=%d exceeds %d", F, 65535 * gin::dist::kChunk);
  gin::dist::point_mesh_kernel<<<grid, gin::dist::kThreads, 0, st>>>(points, verts, faces, (unsigned long long*)ws, N, V, F);
  int rc = check_launch("point_mesh");
  if (rc != GIN_OK) return rc;
  gin::dist::unpack_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const unsigned long long*)ws, dist, face_idx, (long long)n);
  return check_launch("point_mesh_unpack");
}

// ------------------------------------------------------------------ Chamfer distance (one nearest neighbour, both directions)
size_t gin_chamfer_ws_bytes(int B, int N, int M) {
  if (B <= 0 || N <= 0 || M <= 0) return 0;
  return (size_t)B * (N > M ? N : M) * sizeof(gin::fixsum::Acc);     // >= the forward's 8 B * B * (N + M) of 64-bit keys
}

static int chamfer_args(const char* fn, const float* x, const float* y, void* ws, int B, int N, int M) {
  if (B < 0) return fail(GIN_ERR_ARG, "%s: B=%d is negative", fn, B);
  if (B == 0) return GIN_OK;
  if (N < 1 || M < 1) return fail(GIN_ERR_ARG, "%s: empty point set (N=%d, M=%d)", fn, N, M);
  if (B > 65535) return fail(GIN_ERR_ARG, "%s: B=%d exceeds 65535", fn, B);
  if ((long long)B * (N > M ? N : M) > 0x7fffffffLL) return fail(GIN_ERR_ARG, "%s: B*max(N,M) exceeds 2^31-1", fn);
  if (!x || !y || !ws) return fail(GIN_ERR_ARG, "%s: null pointer (x, y and ws are required)", fn);
  return GIN_OK;
}

// best[b][i] over the queries q of their nearest candidate in c, then unpacked into d / idx
static int chamfer_direction(gin::chamfer::Pts q, gin::chamfer::Pts c, int B, int Nq, int Nc, unsigned long long* keys, float* d,
                             int32_t* idx, cudaStream_t st) {
  namespace ch = gin::chamfer;
  const long long n = (long long)B * Nq;
  if (cudaMemsetAsync(keys, 0xFF, (size_t)n * sizeof(unsigned long long), st) != cudaSuccess) return fail(GIN_ERR_CUDA, "gin_chamfer_fwd: memset failed");
  // Split the candidates when the queries alone give fewer than 4 CTAs per SM, down to one tile per split.
  const int qblocks = (Nq + ch::kQueries - 1) / ch::kQueries;
  const long long want = 4LL * gin::num_sms();
  long long splits = (want + (long long)qblocks * B - 1) / ((long long)qblocks * B);
  const long long max_splits = (Nc + ch::kTile - 1) / ch::kTile;
  splits = splits < 1 ? 1 : (splits > max_splits ? max_splits : splits);
  int split_len = (int)((Nc + splits - 1) / splits);
  split_len = (split_len + ch::kChunk - 1) / ch::kChunk * ch::kChunk;
  splits = (Nc + split_len - 1) / split_len;
  ch::nn_kernel<<<dim3(qblocks, (unsigned)splits, B), ch::kThreads, 0, st>>>(q, c, Nq, Nc, split_len, keys);
  int rc = check_launch("chamfer_nn");
  if (rc != GIN_OK) return rc;
  gin::dist::unpack_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(keys, d, idx, n);
  return check_launch("chamfer_unpack");
}

int gin_chamfer_fwd(const float* x, int64_t xsb, int64_t xsn, int64_t xsc, const float* y, int64_t ysb, int64_t ysn, int64_t ysc,
                    float* d_xy, int32_t* idx_xy, float* d_yx, int32_t* idx_yx, void* ws, int B, int N, int M, void* stream) {
  int rc = chamfer_args("gin_chamfer_fwd", x, y, ws, B, N, M);
  if (rc != GIN_OK || B == 0) return rc;
  if ((idx_xy && !d_xy) || (idx_yx && !d_yx)) return fail(GIN_ERR_ARG, "gin_chamfer_fwd: an index output needs its distance output");
  if (!d_xy && !d_yx) return fail(GIN_ERR_ARG, "gin_chamfer_fwd: null pointer (neither direction has an output)");
  cudaStream_t st = (cudaStream_t)stream;
  const gin::chamfer::Pts px{x, xsb, xsn, xsc}, py{y, ysb, ysn, ysc};
  unsigned long long* keys = (unsigned long long*)ws;
  if (d_xy && (rc = chamfer_direction(px, py, B, N, M, keys, d_xy, idx_xy, st)) != GIN_OK) return rc;
  if (d_yx) rc = chamfer_direction(py, px, B, M, N, keys + (size_t)B * N, d_yx, idx_yx, st);
  return rc;
}

// out = direct term of side D (g_d, idx_d: D's own direction, may be NULL) + scatter from the other side's entries (g_e, idx_e)
static int chamfer_side(gin::chamfer::Pts D, gin::chamfer::Pts O, int B, int Nd, int No, const int32_t* idx_d, const float* g_d,
                        const int32_t* idx_e, const float* g_e, float* out, void* ws, cudaStream_t st) {
  namespace ch = gin::chamfer;
  ch::Acc* acc = nullptr;
  if (g_e) {
    acc = (ch::Acc*)ws;
    if (cudaMemsetAsync(acc, 0, (size_t)B * Nd * sizeof(ch::Acc), st) != cudaSuccess) return fail(GIN_ERR_CUDA, "gin_chamfer_bwd: memset failed");
    const long long ne = (long long)B * No;
    ch::scatter_stats_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, st>>>(D, O, idx_e, g_e, acc, Nd, No, ne);
    int rc = check_launch("chamfer_scatter_stats");
    if (rc != GIN_OK) return rc;
    ch::scatter_sum_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, st>>>(D, O, idx_e, g_e, acc, Nd, No, ne);
    if ((rc = check_launch("chamfer_scatter_sum")) != GIN_OK) return rc;
  }
  const long long nd = (long long)B * Nd;
  ch::finish_kernel<<<(unsigned)((nd + 255) / 256), 256, 0, st>>>(D, O, idx_d, g_d, acc, out, Nd, nd);
  return check_launch("chamfer_finish");
}

int gin_chamfer_bwd(const float* x, int64_t xsb, int64_t xsn, int64_t xsc, const float* y, int64_t ysb, int64_t ysn, int64_t ysc,
                    const int32_t* idx_xy, const float* g_xy, const int32_t* idx_yx, const float* g_yx, float* dx, float* dy, void* ws,
                    int B, int N, int M, void* stream) {
  int rc = chamfer_args("gin_chamfer_bwd", x, y, ws, B, N, M);
  if (rc != GIN_OK || B == 0) return rc;
  if ((g_xy && !idx_xy) || (g_yx && !idx_yx)) return fail(GIN_ERR_ARG, "gin_chamfer_bwd: null pointer (a cotangent needs its indices)");
  if (!g_xy && !g_yx) return fail(GIN_ERR_ARG, "gin_chamfer_bwd: null pointer (neither direction has a cotangent)");
  if (!dx && !dy) return fail(GIN_ERR_ARG, "gin_chamfer_bwd: null pointer (neither dx nor dy is requested)");
  cudaStream_t st = (cudaStream_t)stream;
  const gin::chamfer::Pts px{x, xsb, xsn, xsc}, py{y, ysb, ysn, ysc};
  if (dx && (rc = chamfer_side(px, py, B, N, M, g_xy ? idx_xy : nullptr, g_xy, idx_yx, g_yx, dx, ws, st)) != GIN_OK) return rc;
  if (dy) rc = chamfer_side(py, px, B, M, N, g_yx ? idx_yx : nullptr, g_yx, idx_xy, g_xy, dy, ws, st);
  return rc;
}

// ------------------------------------------------------------------ fused BatchNorm + activation + operand cast
size_t gin_bn_ws_bytes(int C) { return C <= 0 ? 0 : (size_t)gin::bn::MAX_CTAS * 2 * C * 4; }

static bool bn_shape_ok(int C) { return C > 0 && (C & 7) == 0 && 256 % (C >> 3) == 0; }

int gin_bn_stats(const float* y, int64_t ld, int64_t rows, int C, const float* gamma, const float* beta, float eps, float momentum,
                 float* running_mean, float* running_var, int64_t* num_batches_tracked, float* stat, void* ws, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!y || !stat || !ws || rows <= 0 || !bn_shape_ok(C) || ld < C || (ld & 3)) return fail(GIN_ERR_ARG, "gin_bn_stats: bad argument (C/8 must divide 256)");
  const int ctas = gin::bn::grid_for_rows(rows * (C >> 3));
  gin::launch_pdl(gin::bn::stats_kernel, dim3(ctas), dim3(256), 0, st, gin::bn::Src{y, (long long)ld, 0}, rows, C, reinterpret_cast<float*>(ws));
  int rc = check_launch("bn_stats");
  if (rc) return rc;
  gin::launch_pdl(gin::bn::stats_final_kernel, dim3(C / 8), dim3(256), 0, st, reinterpret_cast<const float*>(ws), ctas, rows, C, gamma, beta, eps, momentum, running_mean,
                                                     running_var, reinterpret_cast<long long*>(num_batches_tracked), stat, 0);
  return check_launch("bn_stats_final");
}

size_t gin_hexconv_stats_ws_bytes(int Cout) { return Cout <= 0 ? 0 : (size_t)gin::kMaxSMs * 2 * Cout * 4; }   // one row per persistent CTA

int gin_bn_stats_from_parts(const float* parts, int nparts, int64_t ld, int64_t rows, int C, const float* gamma, const float* beta, float eps,
                            float momentum, float* running_mean, float* running_var, int64_t* num_batches_tracked, float* stat, void* stream) {
  if (!parts || nparts <= 0 || nparts > gin::bn::MAX_CTAS || !stat || rows <= 0 || !bn_shape_ok(C) || ld < C)
    return fail(GIN_ERR_ARG, "gin_bn_stats_from_parts: bad argument");
  gin::launch_pdl(gin::bn::stats_final_kernel, dim3(C / 8), dim3(256), 0, (cudaStream_t)stream, parts, nparts, rows, C, gamma, beta, eps, momentum, running_mean, running_var,
                                                                       reinterpret_cast<long long*>(num_batches_tracked), stat, ld);
  return check_launch("bn_stats_final");
}

int gin_bn_stats_from_parts2(const float* parts, int nparts, int64_t ld, int64_t rows, int C, int colA, const float* gammaA, const float* betaA,
                             float epsA, float momentumA, float* rmeanA, float* rvarA, int64_t* nbtA, float* statA, int colB, const float* gammaB,
                             const float* betaB, float epsB, float momentumB, float* rmeanB, float* rvarB, int64_t* nbtB, float* statB, void* stream) {
  if (!parts || nparts <= 0 || nparts > gin::bn::MAX_CTAS || !statA || !statB || rows <= 0 || !bn_shape_ok(C) || colA < 0 || colB < 0 || ld < C + (colA > colB ? colA : colB))
    return fail(GIN_ERR_ARG, "gin_bn_stats_from_parts2: bad argument");
  gin::bn::StatsTarget a{parts + colA, gammaA, betaA, rmeanA, rvarA, reinterpret_cast<long long*>(nbtA), statA, epsA, momentumA};
  gin::bn::StatsTarget b{parts + colB, gammaB, betaB, rmeanB, rvarB, reinterpret_cast<long long*>(nbtB), statB, epsB, momentumB};
  gin::launch_pdl(gin::bn::stats_final2_kernel, dim3(2 * (C / 8)), dim3(256), 0, (cudaStream_t)stream, a, b, nparts, (long long)rows, C, (long long)ld);
  return check_launch("bn_stats_final2");
}

int gin_bn_act_fwd(const void* y1, int64_t ld1, const float* stat1, const void* y2, int64_t ld2, const float* stat2, int y_fp16, int relu, void* out_b,
                   float* out_f, void* out_w, int B, int level, int C, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!y1 || !stat1 || (y2 && !stat2) || (!out_b && !out_f && !out_w) || B <= 0 || level < 0 || level > 9 || !bn_shape_ok(C))
    return fail(GIN_ERR_ARG, "gin_bn_act_fwd: bad argument");
  const int n = 1 << level, P = 10 << (2 * level);
  const int ctas = gin::bn::grid_for_rows(((long long)B * P + 2LL * B) * (C >> 3));
  const gin::bn::Src s1{reinterpret_cast<const float*>(y1), (long long)ld1, y_fp16 ? 1 : 0}, s2{reinterpret_cast<const float*>(y2), (long long)ld2, y_fp16 ? 1 : 0};
  const int f16 = (int)gin::fwd_fp16();          // out_b is the next convolution's FORWARD operand copy
  if (!gin::bn::smem_consts(C)) {
    if (y2) gin::launch_pdl(gin::bn::act_fwd_anyc_kernel<true>, dim3(ctas), dim3(256), 0, st, s1, stat1, s2, stat2, relu, reinterpret_cast<__nv_bfloat16*>(out_b), out_f, n, B, P, C, f16, reinterpret_cast<__nv_bfloat16*>(out_w));
    else gin::launch_pdl(gin::bn::act_fwd_anyc_kernel<false>, dim3(ctas), dim3(256), 0, st, s1, stat1, s2, stat2, relu, reinterpret_cast<__nv_bfloat16*>(out_b), out_f, n, B, P, C, f16, reinterpret_cast<__nv_bfloat16*>(out_w));
  } else {
    auto k = y2 ? (y_fp16 ? gin::bn::act_fwd_kernel<true, true> : gin::bn::act_fwd_kernel<true, false>)
                : (y_fp16 ? gin::bn::act_fwd_kernel<false, true> : gin::bn::act_fwd_kernel<false, false>);
    gin::launch_pdl(k, dim3(ctas), dim3(256), 0, st, s1, stat1, s2, stat2, relu, reinterpret_cast<__nv_bfloat16*>(out_b), out_f, n, B, P, C, f16, reinterpret_cast<__nv_bfloat16*>(out_w));
  }
  return check_launch("bn_act_fwd");
}

// the apply pass of gin_bn_act_bwd / _pair (and of the synchronised backward) from finished bstat
static int bn_bwd_apply(const float* dout, int64_t ldg, const void* mask_b, const void* y, int64_t ld, int y_fp16, const float* stat, const float* bstat,
                        void* dy_b, int64_t ldo, float* dy_f, int64_t ldf, int B, int level, int C, int relu_from_y, cudaStream_t st) {
  const int n = 1 << level, P = 10 << (2 * level);
  const gin::bn::Src sy{reinterpret_cast<const float*>(y), (long long)ld, y_fp16 ? 1 : 0};
  const __nv_bfloat16* mask = reinterpret_cast<const __nv_bfloat16*>(mask_b);
  const int ctas = gin::bn::grid_for_rows((long long)B * P * (C >> 3));
  const bool smem = gin::bn::smem_consts(C);
  const int from_y = (relu_from_y && mask && smem) ? 1 : 0;
  __nv_bfloat16* dyb = reinterpret_cast<__nv_bfloat16*>(dy_b);
  if (!smem) gin::launch_pdl(gin::bn::bwd_apply_anyc_kernel, dim3(ctas), dim3(256), 0, st, dout, ldg, mask, sy, stat, bstat, dyb, ldo, dy_f, ldf, n, B, P, C);
  else gin::launch_pdl(y_fp16 ? gin::bn::bwd_apply_kernel<true> : gin::bn::bwd_apply_kernel<false>, dim3(ctas), dim3(256), 0, st, dout, ldg, mask, sy, stat, bstat, dyb, ldo, dy_f, ldf, n, B, P, C, from_y);
  return check_launch("bn_bwd_apply");
}

static int bn_bwd_apply_pair(const float* dout, int64_t ldg, const void* mask_b, const void* yA, int64_t ldA, const float* statA, const float* bstatA,
                             void* dyA_b, int64_t ldoA, const void* yB, int64_t ldB, const float* statB, const float* bstatB, void* dyB_b, int64_t ldoB,
                             int y_fp16, int B, int level, int C, int relu_from_y, cudaStream_t st) {
  const int n = 1 << level, P = 10 << (2 * level);
  const gin::bn::Src sA{reinterpret_cast<const float*>(yA), (long long)ldA, y_fp16 ? 1 : 0}, sB{reinterpret_cast<const float*>(yB), (long long)ldB, y_fp16 ? 1 : 0};
  const __nv_bfloat16* mask = reinterpret_cast<const __nv_bfloat16*>(mask_b);
  const int ctas = gin::bn::grid_for_rows((long long)B * P * (C >> 3));
  const bool smem = gin::bn::smem_consts(C);
  const int from_y = (relu_from_y && mask && smem) ? 1 : 0;
  __nv_bfloat16 *da = reinterpret_cast<__nv_bfloat16*>(dyA_b), *db = reinterpret_cast<__nv_bfloat16*>(dyB_b);
  if (!smem) gin::launch_pdl(gin::bn::bwd_apply2_anyc_kernel, dim3(ctas), dim3(256), 0, st, dout, ldg, mask, sA, statA, bstatA, sB, statB, bstatB, da, ldoA, db, ldoB, n, B, P, C);
  else gin::launch_pdl(y_fp16 ? gin::bn::bwd_apply2_kernel<true> : gin::bn::bwd_apply2_kernel<false>, dim3(ctas), dim3(256), 0, st, dout, ldg, mask, sA, statA, bstatA, sB, statB, bstatB, da, ldoA, db, ldoB, n, B, P, C, from_y);
  return check_launch("bn_bwd_apply2");
}

// the reduce pass of gin_bn_act_bwd / _pair: per-CTA partials in ws; returns their count in *nparts
static int bn_bwd_reduce(const float* dout, int64_t ldg, const void* mask_b, const void* y, int64_t ld, int y_fp16, const float* stat, void* ws,
                         long long rows, int C, int relu_from_y, cudaStream_t st, int* nparts) {
  const gin::bn::Src sy{reinterpret_cast<const float*>(y), (long long)ld, y_fp16 ? 1 : 0};
  const __nv_bfloat16* mask = reinterpret_cast<const __nv_bfloat16*>(mask_b);
  const int ctas = *nparts = gin::bn::grid_for_rows(rows * (C >> 3));
  const bool smem = gin::bn::smem_consts(C);
  const int from_y = (relu_from_y && mask && smem) ? 1 : 0;      // the register-constant kernels always read the mask
  float* part = reinterpret_cast<float*>(ws);
  if (!smem) gin::launch_pdl(gin::bn::bwd_reduce_kernel, dim3(ctas), dim3(256), 0, st, dout, ldg, mask, sy, stat, rows, C, part);
  else gin::launch_pdl(y_fp16 ? gin::bn::bwd_reduce_s_kernel<true> : gin::bn::bwd_reduce_s_kernel<false>, dim3(ctas), dim3(256), 0, st, dout, ldg, mask, sy, stat, rows, C, part, from_y);
  return check_launch("bn_bwd_reduce");
}

static int bn_bwd_reduce_pair(const float* dout, int64_t ldg, const void* mask_b, const void* yA, int64_t ldA, const float* statA, const void* yB,
                              int64_t ldB, const float* statB, int y_fp16, void* ws, long long rows, int C, int relu_from_y, cudaStream_t st, int* nparts) {
  const gin::bn::Src sA{reinterpret_cast<const float*>(yA), (long long)ldA, y_fp16 ? 1 : 0}, sB{reinterpret_cast<const float*>(yB), (long long)ldB, y_fp16 ? 1 : 0};
  const __nv_bfloat16* mask = reinterpret_cast<const __nv_bfloat16*>(mask_b);
  const int ctas = *nparts = gin::bn::grid_for_rows(rows * (C >> 3));
  const bool smem = gin::bn::smem_consts(C);
  const int from_y = (relu_from_y && mask && smem) ? 1 : 0;
  float* part = reinterpret_cast<float*>(ws);
  if (!smem) gin::launch_pdl(gin::bn::bwd_reduce2_anyc_kernel, dim3(ctas), dim3(256), 0, st, dout, ldg, mask, sA, statA, sB, statB, rows, C, part);
  else gin::launch_pdl(y_fp16 ? gin::bn::bwd_reduce2_kernel<true> : gin::bn::bwd_reduce2_kernel<false>, dim3(ctas), dim3(256), 0, st, dout, ldg, mask, sA, statA, sB, statB, rows, C, part, from_y);
  return check_launch("bn_bwd_reduce2");
}

static bool bn_bwd_args_ok(const float* dout, const void* y, const float* stat, const void* dy_b, const float* dy_f, int B, int level, int C) {
  return dout && y && stat && (dy_b || dy_f) && B > 0 && level >= 0 && level <= 9 && bn_shape_ok(C);
}

static bool bn_bwd_pair_args_ok(const float* dout, const void* yA, const float* statA, const void* dyA_b, const void* yB, const float* statB,
                                const void* dyB_b, int B, int level, int C) {
  return dout && yA && yB && statA && statB && dyA_b && dyB_b && B > 0 && level >= 0 && level <= 9 && bn_shape_ok(C);
}

int gin_bn_act_bwd(const float* dout, int64_t ldg, const void* mask_b, const void* y, int64_t ld, int y_fp16, const float* stat, float* bstat, void* dy_b,
                   int64_t ldo, float* dy_f, int64_t ldf, void* ws, int B, int level, int C, int relu_from_y, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!bstat || !ws || !bn_bwd_args_ok(dout, y, stat, dy_b, dy_f, B, level, C)) return fail(GIN_ERR_ARG, "gin_bn_act_bwd: bad argument");
  const long long rows = (long long)B * (10 << (2 * level));
  int ctas, rc = bn_bwd_reduce(dout, ldg, mask_b, y, ld, y_fp16, stat, ws, rows, C, relu_from_y, st, &ctas);
  if (rc) return rc;
  gin::launch_pdl(gin::bn::bwd_final_kernel, dim3(C / 8), dim3(256), 0, st, reinterpret_cast<const float*>(ws), ctas, rows, C, bstat);
  if ((rc = check_launch("bn_bwd_final"))) return rc;
  return bn_bwd_apply(dout, ldg, mask_b, y, ld, y_fp16, stat, bstat, dy_b, ldo, dy_f, ldf, B, level, C, relu_from_y, st);
}

size_t gin_bn_pair_ws_bytes(int C) { return C <= 0 ? 0 : (size_t)gin::bn::MAX_CTAS * 4 * C * 4; }

int gin_bn_act_bwd_pair(const float* dout, int64_t ldg, const void* mask_b, const void* yA, int64_t ldA, const float* statA, float* bstatA,
                        void* dyA_b, int64_t ldoA, const void* yB, int64_t ldB, const float* statB, float* bstatB, void* dyB_b, int64_t ldoB,
                        int y_fp16, void* ws, int B, int level, int C, int relu_from_y, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!bstatA || !bstatB || !ws || !bn_bwd_pair_args_ok(dout, yA, statA, dyA_b, yB, statB, dyB_b, B, level, C))
    return fail(GIN_ERR_ARG, "gin_bn_act_bwd_pair: bad argument");
  const long long rows = (long long)B * (10 << (2 * level));
  int ctas, rc = bn_bwd_reduce_pair(dout, ldg, mask_b, yA, ldA, statA, yB, ldB, statB, y_fp16, ws, rows, C, relu_from_y, st, &ctas);
  if (rc) return rc;
  gin::launch_pdl(gin::bn::bwd_final2_kernel, dim3(C / 8), dim3(256), 0, st, reinterpret_cast<const float*>(ws), ctas, rows, C, bstatA, bstatB);
  if ((rc = check_launch("bn_bwd_final2"))) return rc;
  return bn_bwd_apply_pair(dout, ldg, mask_b, yA, ldA, statA, bstatA, dyA_b, ldoA, yB, ldB, statB, bstatB, dyB_b, ldoB, y_fp16, B, level, C, relu_from_y, st);
}

// ------------------------------------------------------------------ synchronised BatchNorm (records all-gathered by the caller)
size_t gin_bn_sync_record_bytes(int C, int pair) { return C <= 0 ? 0 : (size_t)8 * (pair ? 2 : 1) * (2 * (size_t)C + 1); }

int gin_bn_sync_stats_total(const float* y, int64_t ld, int64_t rows, int C, double* rec, void* ws, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!y || !rec || !ws || rows <= 0 || !bn_shape_ok(C) || ld < C || (ld & 3)) return fail(GIN_ERR_ARG, "gin_bn_sync_stats_total: bad argument (C/8 must divide 256)");
  const int ctas = gin::bn::grid_for_rows(rows * (C >> 3));
  gin::launch_pdl(gin::bn::stats_kernel, dim3(ctas), dim3(256), 0, st, gin::bn::Src{y, (long long)ld, 0}, rows, C, reinterpret_cast<float*>(ws));
  int rc = check_launch("bn_stats");
  if (rc) return rc;
  gin::launch_pdl(gin::bn::stats_total_kernel, dim3(C / 8), dim3(256), 0, st, reinterpret_cast<const float*>(ws), (const float*)nullptr, ctas, (long long)rows, C,
                  (long long)C, rec);
  return check_launch("bn_stats_total");
}

int gin_bn_sync_stats_total_from_parts(const float* parts, int nparts, int64_t ld, int64_t rows, int C, int colA, int colB, double* rec, void* stream) {
  if (!parts || nparts <= 0 || nparts > gin::bn::MAX_CTAS || !rec || rows <= 0 || !bn_shape_ok(C) || colA < 0 || colB < -1 ||
      ld < C + (colA > colB ? colA : colB))
    return fail(GIN_ERR_ARG, "gin_bn_sync_stats_total_from_parts: bad argument");
  const int nbn = colB >= 0 ? 2 : 1;
  gin::launch_pdl(gin::bn::stats_total_kernel, dim3(nbn * (C / 8)), dim3(256), 0, (cudaStream_t)stream, parts + colA, colB >= 0 ? parts + colB : nullptr,
                  nparts, (long long)rows, C, (long long)ld, rec);
  return check_launch("bn_stats_total");
}

int gin_bn_sync_stats_final(const double* recs, int world, int C, const float* gammaA, const float* betaA, float epsA, float momentumA, float* rmeanA,
                            float* rvarA, int64_t* nbtA, float* statA, const float* gammaB, const float* betaB, float epsB, float momentumB, float* rmeanB,
                            float* rvarB, int64_t* nbtB, float* statB, void* stream) {
  if (!recs || world <= 0 || !statA || !bn_shape_ok(C)) return fail(GIN_ERR_ARG, "gin_bn_sync_stats_final: bad argument");
  const int nbn = statB ? 2 : 1;
  gin::bn::StatsTarget a{nullptr, gammaA, betaA, rmeanA, rvarA, reinterpret_cast<long long*>(nbtA), statA, epsA, momentumA};
  gin::bn::StatsTarget b{nullptr, gammaB, betaB, rmeanB, rvarB, reinterpret_cast<long long*>(nbtB), statB, epsB, momentumB};
  gin::launch_pdl(gin::bn::stats_sync_final_kernel, dim3(nbn * (C / 8)), dim3(256), 0, (cudaStream_t)stream, recs, world, nbn, C, a, b);
  return check_launch("bn_stats_sync_final");
}

int gin_bn_sync_bwd_reduce(const float* dout, int64_t ldg, const void* mask_b, const void* y, int64_t ld, int y_fp16, const float* stat, double* rec,
                           void* ws, int B, int level, int C, int relu_from_y, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!rec || !ws || !bn_bwd_args_ok(dout, y, stat, rec, nullptr, B, level, C)) return fail(GIN_ERR_ARG, "gin_bn_sync_bwd_reduce: bad argument");
  const long long rows = (long long)B * (10 << (2 * level));
  int ctas, rc = bn_bwd_reduce(dout, ldg, mask_b, y, ld, y_fp16, stat, ws, rows, C, relu_from_y, st, &ctas);
  if (rc) return rc;
  gin::launch_pdl(gin::bn::bwd_total_kernel, dim3(C / 8), dim3(256), 0, st, reinterpret_cast<const float*>(ws), ctas, 1, rows, C, rec);
  return check_launch("bn_bwd_total");
}

int gin_bn_sync_bwd_reduce_pair(const float* dout, int64_t ldg, const void* mask_b, const void* yA, int64_t ldA, const float* statA, const void* yB,
                                int64_t ldB, const float* statB, int y_fp16, double* rec, void* ws, int B, int level, int C, int relu_from_y, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!rec || !ws || !bn_bwd_pair_args_ok(dout, yA, statA, rec, yB, statB, rec, B, level, C)) return fail(GIN_ERR_ARG, "gin_bn_sync_bwd_reduce_pair: bad argument");
  const long long rows = (long long)B * (10 << (2 * level));
  int ctas, rc = bn_bwd_reduce_pair(dout, ldg, mask_b, yA, ldA, statA, yB, ldB, statB, y_fp16, ws, rows, C, relu_from_y, st, &ctas);
  if (rc) return rc;
  gin::launch_pdl(gin::bn::bwd_total_kernel, dim3(C / 8), dim3(256), 0, st, reinterpret_cast<const float*>(ws), ctas, 2, rows, C, rec);
  return check_launch("bn_bwd_total");
}

int gin_bn_sync_bwd_final(const double* recs, int world, int rank, int C, float* bstatA, float* bstatB, void* stream) {
  if (!recs || world <= 0 || rank < 0 || rank >= world || !bstatA || !bn_shape_ok(C)) return fail(GIN_ERR_ARG, "gin_bn_sync_bwd_final: bad argument");
  gin::launch_pdl(gin::bn::bwd_sync_final_kernel, dim3(C / 8), dim3(256), 0, (cudaStream_t)stream, recs, world, rank, bstatB ? 2 : 1, C, bstatA, bstatB);
  return check_launch("bn_bwd_sync_final");
}

int gin_bn_bwd_apply(const float* dout, int64_t ldg, const void* mask_b, const void* y, int64_t ld, int y_fp16, const float* stat, const float* bstat,
                     void* dy_b, int64_t ldo, float* dy_f, int64_t ldf, int B, int level, int C, int relu_from_y, void* stream) {
  if (!bstat || !bn_bwd_args_ok(dout, y, stat, dy_b, dy_f, B, level, C)) return fail(GIN_ERR_ARG, "gin_bn_bwd_apply: bad argument");
  return bn_bwd_apply(dout, ldg, mask_b, y, ld, y_fp16, stat, bstat, dy_b, ldo, dy_f, ldf, B, level, C, relu_from_y, (cudaStream_t)stream);
}

int gin_bn_bwd_apply_pair(const float* dout, int64_t ldg, const void* mask_b, const void* yA, int64_t ldA, const float* statA, const float* bstatA,
                          void* dyA_b, int64_t ldoA, const void* yB, int64_t ldB, const float* statB, const float* bstatB, void* dyB_b, int64_t ldoB,
                          int y_fp16, int B, int level, int C, int relu_from_y, void* stream) {
  if (!bstatA || !bstatB || !bn_bwd_pair_args_ok(dout, yA, statA, dyA_b, yB, statB, dyB_b, B, level, C))
    return fail(GIN_ERR_ARG, "gin_bn_bwd_apply_pair: bad argument");
  return bn_bwd_apply_pair(dout, ldg, mask_b, yA, ldA, statA, bstatA, dyA_b, ldoA, yB, ldB, statB, bstatB, dyB_b, ldoB, y_fp16, B, level, C, relu_from_y,
                           (cudaStream_t)stream);
}

// ------------------------------------------------------------------ eval-mode BatchNorm backward (frozen statistics)
size_t gin_bn_eval_bwd_ws_bytes(int C) { return C <= 0 ? 0 : (size_t)gin::bn::MAX_CTAS * 3 * C * 4; }

static bool eval_bwd_shape_ok(int C) { return bn_shape_ok(C) && C <= gin::bn::CST_MAX_C; }

int gin_bn_eval_bwd(const float* dout, int64_t ldg, const void* mask_b, const void* y, int64_t ld, int y_fp16, const float* stat, float* bsum,
                    void* dy_b, int64_t ldo, float* dy_f, int64_t ldf, void* ws, int B, int level, int C, int relu_from_y, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!dout || !y || !stat || (!dy_b && !dy_f) || (bsum && !ws) || B <= 0 || level < 0 || level > 9 || !eval_bwd_shape_ok(C))
    return fail(GIN_ERR_ARG, "gin_bn_eval_bwd: bad argument (C/8 must divide 256, C <= %d)", gin::bn::CST_MAX_C);
  if (ldg < C || ld < C || (dy_b && ldo < C) || (dy_f && ldf < C) || ((ldg | ld | (dy_b ? ldo : 0) | (dy_f ? ldf : 0)) & 7))
    return fail(GIN_ERR_ARG, "gin_bn_eval_bwd: bad row stride (each must be >= C and a multiple of 8)");
  const int n = 1 << level, P = 10 << (2 * level);
  const long long rows = (long long)B * P;
  const gin::bn::Src sy{reinterpret_cast<const float*>(y), (long long)ld, y_fp16 ? 1 : 0};
  const __nv_bfloat16* mask = relu_from_y ? nullptr : reinterpret_cast<const __nv_bfloat16*>(mask_b);
  const int from_y = relu_from_y ? 1 : 0;
  const int ctas = gin::bn::grid_for_rows((rows + (dy_b ? 2LL * B : 0)) * (C >> 3));
  float* part = reinterpret_cast<float*>(ws);
  __nv_bfloat16* dyb = reinterpret_cast<__nv_bfloat16*>(dy_b);
  auto k = bsum ? (y_fp16 ? gin::bn::eval_bwd_kernel<true, true> : gin::bn::eval_bwd_kernel<false, true>)
                : (y_fp16 ? gin::bn::eval_bwd_kernel<true, false> : gin::bn::eval_bwd_kernel<false, false>);
  gin::launch_pdl(k, dim3(ctas), dim3(256), 0, st, dout, (long long)ldg, mask, sy, stat, dyb, (long long)ldo, dy_f, (long long)ldf, part, n, B, P, C, from_y);
  int rc = check_launch("bn_eval_bwd");
  if (rc || !bsum) return rc;
  gin::launch_pdl(gin::bn::eval_bwd_final_kernel, dim3(C / 8), dim3(256), 0, st, (const float*)part, ctas, 2, C, stat, bsum, (const float*)nullptr,
                  (float*)nullptr);
  return check_launch("bn_eval_bwd_final");
}

int gin_bn_eval_bwd_pair(const float* dout, int64_t ldg, const void* mask_b, const void* yA, int64_t ldA, const float* statA, float* bsumA,
                         void* dyA_b, int64_t ldoA, const void* yB, int64_t ldB, const float* statB, float* bsumB, void* dyB_b, int64_t ldoB,
                         int y_fp16, void* ws, int B, int level, int C, int relu_from_y, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!dout || !yA || !yB || !statA || !statB || !dyA_b || !dyB_b || ((bsumA || bsumB) && !ws) || B <= 0 || level < 0 || level > 9 ||
      !eval_bwd_shape_ok(C))
    return fail(GIN_ERR_ARG, "gin_bn_eval_bwd_pair: bad argument (C/8 must divide 256, C <= %d)", gin::bn::CST_MAX_C);
  if (ldg < C || ldA < C || ldB < C || ldoA < C || ldoB < C || ((ldg | ldA | ldB | ldoA | ldoB) & 7))
    return fail(GIN_ERR_ARG, "gin_bn_eval_bwd_pair: bad row stride (each must be >= C and a multiple of 8)");
  const int n = 1 << level, P = 10 << (2 * level);
  const long long rows = (long long)B * P;
  const gin::bn::Src sA{reinterpret_cast<const float*>(yA), (long long)ldA, y_fp16 ? 1 : 0}, sB{reinterpret_cast<const float*>(yB), (long long)ldB, y_fp16 ? 1 : 0};
  const __nv_bfloat16* mask = relu_from_y ? nullptr : reinterpret_cast<const __nv_bfloat16*>(mask_b);
  const int from_y = relu_from_y ? 1 : 0;
  const bool red = bsumA || bsumB;
  const int ctas = gin::bn::grid_for_rows((rows + 2LL * B) * (C >> 3));
  float* part = reinterpret_cast<float*>(ws);
  __nv_bfloat16 *da = reinterpret_cast<__nv_bfloat16*>(dyA_b), *db = reinterpret_cast<__nv_bfloat16*>(dyB_b);
  auto k = red ? (y_fp16 ? gin::bn::eval_bwd2_kernel<true, true> : gin::bn::eval_bwd2_kernel<false, true>)
               : (y_fp16 ? gin::bn::eval_bwd2_kernel<true, false> : gin::bn::eval_bwd2_kernel<false, false>);
  gin::launch_pdl(k, dim3(ctas), dim3(256), 0, st, dout, (long long)ldg, mask, sA, statA, sB, statB, da, (long long)ldoA, db, (long long)ldoB, part, n, B,
                  P, C, from_y);
  int rc = check_launch("bn_eval_bwd2");
  if (rc || !red) return rc;
  gin::launch_pdl(gin::bn::eval_bwd_final_kernel, dim3(C / 8), dim3(256), 0, st, (const float*)part, ctas, 3, C, statA, bsumA, statB, bsumB);
  return check_launch("bn_eval_bwd_final");
}

// ------------------------------------------------------------------ optimizer step (run.py:446, 250)
int gin_adam_chunk(void) { return gin::adam::CHUNK; }

int gin_adam_step(const void* table_dev, const int32_t* chunk_first_dev, int count, int total_chunks, float lr, const float* lr_dev, float beta1,
                  float beta2, float eps, float weight_decay, void* ticket_dev, void* stream) {
  static_assert(sizeof(gin::adam::Tensor) == sizeof(GinAdamTensor), "GinAdamTensor layout");
  if (count == 0) return GIN_OK;
  if (!table_dev || !chunk_first_dev || !ticket_dev || count < 0 || total_chunks < count || !(beta1 >= 0.f && beta1 < 1.f) || !(beta2 >= 0.f && beta2 < 1.f) ||
      !(eps >= 0.f) || !(weight_decay >= 0.f) || (!lr_dev && !(lr >= 0.f)))
    return fail(GIN_ERR_ARG, "gin_adam_step: bad argument");
  const gin::adam::Hyper h{lr, beta1, beta2, eps, weight_decay};
  gin::adam::step_kernel<<<total_chunks, gin::adam::THREADS, 0, (cudaStream_t)stream>>>(reinterpret_cast<const gin::adam::Tensor*>(table_dev), chunk_first_dev, count, h,
                                                                                          lr_dev, reinterpret_cast<unsigned int*>(ticket_dev));
  return check_launch("adam_step");
}

static int up_hdr(const void* plan_host, const void* plan_dev, const GinUpPlanHdr** out);

int gin_upsample_bf16(const void* plan_host, const void* plan_dev, const void* in, int in_is_f32, void* out_b, void* out_w, int B, int C, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!in || !out_b || B <= 0 || C <= 0 || (C & 7)) return fail(GIN_ERR_ARG, "gin_upsample_bf16: bad argument (C must be a multiple of 8)");
  const GinUpPlanHdr* h;
  int rc = up_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  const int ctas = gin::bn::grid_for_rows(((long long)B * h->Pf + 2LL * B) * (C >> 3));
  const int grid = ctas * 4 > 148 * 8 ? 148 * 8 : ctas * 4;
  const int f16 = (int)gin::fwd_fp16();          // both the source copy (when 16-bit) and the result are forward operands
  const bool small = ((long long)B * h->Pf + 2LL * B) * (C >> 3) < 0x7fffffffLL;
  auto k = in_is_f32 ? (small ? gin::bn::upsample_bf16_kernel<true, unsigned> : gin::bn::upsample_bf16_kernel<true, long long>)
                     : (small ? gin::bn::upsample_bf16_kernel<false, unsigned> : gin::bn::upsample_bf16_kernel<false, long long>);
  gin::launch_pdl(k, dim3(grid), dim3(256), 0, st, plan_words(plan_dev), in, reinterpret_cast<__nv_bfloat16*>(out_b), 2 << h->level, B, C, f16, reinterpret_cast<__nv_bfloat16*>(out_w));
  return check_launch("upsample_bf16");
}

static int loss_hdr(const void* plan_host, const void* plan_dev, const GinLossPlanHdr** out) {
  if (!plan_dev) return fail(GIN_ERR_ARG, "null plan");
  const int32_t* w = plan_header(plan_host);
  if (!w) return GIN_ERR_PLAN;
  const GinLossPlanHdr* h = reinterpret_cast<const GinLossPlanHdr*>(w);
  if (h->kind != GIN_PLAN_LOSS) return fail(GIN_ERR_PLAN, "plan is not a loss plan (kind %d)", h->kind);
  *out = h;
  return GIN_OK;
}

int gin_pole_vertices_fwd(const void* plan_host, const void* plan_dev, const float* x, int64_t sb, int64_t sp, int64_t sc, float* v, int B, int C,
                          void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!x || !v || B < 0 || C <= 0) return fail(GIN_ERR_ARG, "gin_pole_vertices_fwd: bad argument");
  const GinLossPlanHdr* h;
  int rc = loss_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  if (B == 0) return GIN_OK;
  GinSrcView X{x, (long long)sb, (long long)sp, (long long)sc, h->P};
  gin::pole_vertices_fwd_kernel<<<grid_for((long long)B * h->V * C, 256), 256, 0, st>>>(plan_words(plan_dev), X, v, B, C);
  return check_launch("pole_vertices_fwd");
}

int gin_pole_vertices_bwd(const void* plan_host, const void* plan_dev, const float* dv, float* dx, int64_t sb, int64_t sp, int64_t sc, int B, int C,
                          void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!dv || !dx || B < 0 || C <= 0) return fail(GIN_ERR_ARG, "gin_pole_vertices_bwd: bad argument");
  const GinLossPlanHdr* h;
  int rc = loss_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  if (B == 0) return GIN_OK;
  gin::pole_vertices_bwd_kernel<<<grid_for((long long)B * h->P * C, 256), 256, 0, st>>>(plan_words(plan_dev), dv, dx, sb, sp, sc, B, C);
  return check_launch("pole_vertices_bwd");
}

int gin_vertex_normals_fwd(const void* plan_host, const void* plan_dev, const float* v, float* nrm, int B, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!v || !nrm || B < 0) return fail(GIN_ERR_ARG, "gin_vertex_normals_fwd: bad argument");
  const GinLossPlanHdr* h;
  int rc = loss_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  if (B == 0) return GIN_OK;
  gin::normals_laplacian_kernel<<<grid_for((long long)B * h->V, 256), 256, 0, st>>>(plan_words(plan_dev), v, nrm, nullptr, B);
  return check_launch("vertex_normals_fwd");
}

int gin_laplacian_fwd(const void* plan_host, const void* plan_dev, const float* v, float* lap, int B, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!v || !lap || B < 0) return fail(GIN_ERR_ARG, "gin_laplacian_fwd: bad argument");
  const GinLossPlanHdr* h;
  int rc = loss_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  if (B == 0) return GIN_OK;
  gin::normals_laplacian_kernel<<<grid_for((long long)B * h->V, 256), 256, 0, st>>>(plan_words(plan_dev), v, nullptr, lap, B);
  return check_launch("laplacian_fwd");
}

size_t gin_ring_ops_ws_bytes(int B, int level) {
  if (B < 0 || level < 0 || level > 9) return 0;
  return (size_t)B * ((size_t)(10 << (2 * level)) + 2) * 6 * 4;
}

int gin_ring_ops_bwd(const void* plan_host, const void* plan_dev, const float* v, const float* g_nrm, const float* g_lap, float* dv, void* ws, int B,
                     void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!v || (!g_nrm && !g_lap) || !dv || !ws || B < 0) return fail(GIN_ERR_ARG, "gin_ring_ops_bwd: bad argument");
  const GinLossPlanHdr* h;
  int rc = loss_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  if (B == 0) return GIN_OK;
  const long long BV = (long long)B * h->V;
  float* g = reinterpret_cast<float*>(ws);
  gin::ring_ops_bwd_vertex_kernel<<<grid_for(BV, 256), 256, 0, st>>>(plan_words(plan_dev), v, g_nrm, g_lap, g, dv, B);
  if ((rc = check_launch("ring_ops_bwd_vertex"))) return rc;
  gin::p2p_bwd_gather_kernel<<<grid_for(BV, 256), 256, 0, st>>>(plan_words(plan_dev), v, g, dv, B);
  return check_launch("ring_ops_bwd_gather");
}

// workspace layout: [v: B*V*3 f32][g: B*V*6 f32][dv: B*V*3 f32][partials: 1024*3 f64]
size_t gin_p2p_ws_bytes(int B, int level) {
  if (B < 0 || level < 0 || level > 9) return 0;
  const size_t V = (size_t)(10 << (2 * level)) + 2;
  return (size_t)B * V * 12 * 4 + 1024 * 3 * 8 + 64;
}

int gin_p2p_loss_fwd(const void* plan_host, const void* plan_dev, const float* x, int64_t sb, int64_t sp, int64_t sc, const float* target, float f_pos,
                     float f_nor, float f_lap, float* out, void* ws, int B, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!x || !target || !out || !ws || B <= 0) return fail(GIN_ERR_ARG, "gin_p2p_loss_fwd: bad argument");
  const GinLossPlanHdr* h;
  int rc = loss_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  const size_t BV = (size_t)B * h->V;
  float* v = reinterpret_cast<float*>(ws);
  double* partial = reinterpret_cast<double*>(reinterpret_cast<char*>(ws) + ((BV * 12 * 4 + 63) / 64) * 64);
  GinSrcView X{x, (long long)sb, (long long)sp, (long long)sc, h->P};
  gin::pole_vertices_fwd_kernel<<<grid_for((long long)BV * 3, 256), 256, 0, st>>>(plan_words(plan_dev), X, v, B, 3);
  if ((rc = check_launch("pole_vertices_fwd"))) return rc;
  int parts = grid_for((long long)BV, 256, 4);
  if (parts > 1024) parts = 1024;
  gin::p2p_fwd_kernel<<<parts, 256, 0, st>>>(plan_words(plan_dev), v, target, partial, B);
  if ((rc = check_launch("p2p_fwd"))) return rc;
  gin::p2p_final_kernel<<<1, 256, 0, st>>>(partial, parts, out, 1.0 / (double)BV, f_pos, f_nor, f_lap);
  return check_launch("p2p_final");
}

int gin_p2p_loss_bwd(const void* plan_host, const void* plan_dev, const float* x, int64_t sb, int64_t sp, int64_t sc, const float* target, float f_pos,
                     float f_nor, float f_lap, const float* dout, float* dx, void* ws, int B, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!x || !target || !dout || !dx || !ws || B <= 0) return fail(GIN_ERR_ARG, "gin_p2p_loss_bwd: bad argument");
  const GinLossPlanHdr* h;
  int rc = loss_hdr(plan_host, plan_dev, &h);
  if (rc) return rc;
  const size_t BV = (size_t)B * h->V;
  float* v = reinterpret_cast<float*>(ws);
  float* g = v + BV * 3;
  float* dv = g + BV * 6;
  GinSrcView X{x, (long long)sb, (long long)sp, (long long)sc, h->P};
  gin::pole_vertices_fwd_kernel<<<grid_for((long long)BV * 3, 256), 256, 0, st>>>(plan_words(plan_dev), X, v, B, 3);
  if ((rc = check_launch("pole_vertices_fwd"))) return rc;
  gin::p2p_bwd_vertex_kernel<<<grid_for((long long)BV, 256), 256, 0, st>>>(plan_words(plan_dev), v, target, dout, f_pos, f_nor, f_lap, g, dv, B);
  if ((rc = check_launch("p2p_bwd_vertex"))) return rc;
  gin::p2p_bwd_gather_kernel<<<grid_for((long long)BV, 256), 256, 0, st>>>(plan_words(plan_dev), v, g, dv, B);
  if ((rc = check_launch("p2p_bwd_gather"))) return rc;
  gin::pole_vertices_bwd_kernel<<<grid_for((long long)B * h->P * 3, 256), 256, 0, st>>>(plan_words(plan_dev), dv, dx, sb, sp, sc, B, 3);
  return check_launch("pole_vertices_bwd");
}


// ------------------------------------------------------------------ Chamfer normal and Laplacian terms (matched through the indices)
// workspace layout: forward [partials: 1024*4 f64]; backward [g_n: B*V*3 f32][g_L: B*V*3 f32][acc_n: B*V Acc][acc_L: B*V Acc], the
// gin_ring_ops_bwd workspace (B*V*6 f32) reusing acc_n once the cotangents are formed
size_t gin_chamfer_terms_ws_bytes(int B, int level, int M) {
  if (B <= 0 || level < 0 || level > 9 || M < 1) return 0;
  const size_t BV = (size_t)B * ((size_t)(10 << (2 * level)) + 2);
  const size_t bwd = BV * (2 * 3 * 4 + 2 * sizeof(gin::fixsum::Acc));
  const size_t fwd = (size_t)gin::chamfer_terms::kMaxParts * 4 * 8;
  return bwd > fwd ? bwd : fwd;
}

static int chamfer_terms_args(const char* fn, const void* plan_host, const void* plan_dev, const float* v, const float* tn, const float* tl,
                              const int32_t* idx_xy, const int32_t* idx_yx, const void* out, void* ws, int B, int M,
                              const GinLossPlanHdr** h) {
  if (B < 0) return fail(GIN_ERR_ARG, "%s: B=%d is negative", fn, B);
  if (M < 1) return fail(GIN_ERR_ARG, "%s: M=%d, the target needs at least one point", fn, M);
  int rc = loss_hdr(plan_host, plan_dev, h);
  if (rc) return rc;
  if ((*h)->level < 0 || (*h)->level > 9) return fail(GIN_ERR_ARG, "%s: bad level %d", fn, (*h)->level);
  if ((long long)B * ((*h)->V > M ? (*h)->V : M) > 0x7fffffffLL) return fail(GIN_ERR_ARG, "%s: B*max(V,M) exceeds 2^31-1", fn);
  if (B == 0) return GIN_OK;
  if (!v || !out || !ws) return fail(GIN_ERR_ARG, "%s: null pointer (v, the output and ws are required)", fn);
  if (!tn && !tl) return fail(GIN_ERR_ARG, "%s: null pointer (neither target normals nor target Laplacians)", fn);
  if (!idx_xy && !idx_yx) return fail(GIN_ERR_ARG, "%s: null pointer (neither direction has indices)", fn);
  return GIN_OK;
}

int gin_chamfer_terms_fwd(const void* plan_host, const void* plan_dev, const float* v, const float* tn, int64_t tnsb, int64_t tnsn,
                          int64_t tnsc, const float* tl, int64_t tlsb, int64_t tlsn, int64_t tlsc, const int32_t* idx_xy,
                          const int32_t* idx_yx, float* out, void* ws, int B, int M, void* stream) {
  namespace ct = gin::chamfer_terms;
  const GinLossPlanHdr* h;
  int rc = chamfer_terms_args("gin_chamfer_terms_fwd", plan_host, plan_dev, v, tn, tl, idx_xy, idx_yx, out, ws, B, M, &h);
  if (rc != GIN_OK || B == 0) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  ct::Args a{};
  a.plan = plan_words(plan_dev); a.v = v;
  a.tn = gin::chamfer::Pts{tn, tnsb, tnsn, tnsc}; a.tl = gin::chamfer::Pts{tl, tlsb, tlsn, tlsc};
  a.idx_xy = idx_xy; a.idx_yx = idx_yx;
  a.partial = reinterpret_cast<double*>(ws);
  a.B = B; a.M = M;
  const long long BV = (long long)B * h->V, BM = (long long)B * M;
  int parts = grid_for((idx_xy ? BV : 0) + (idx_yx ? BM : 0), ct::kThreads, 4);
  if (parts > ct::kMaxParts) parts = ct::kMaxParts;
  ct::fwd_kernel<<<parts, ct::kThreads, 0, st>>>(a);
  if ((rc = check_launch("chamfer_terms_fwd"))) return rc;
  ct::final_kernel<<<1, ct::kThreads, 0, st>>>(a.partial, parts, out, 1.0 / (double)BV, 1.0 / (double)BM);
  return check_launch("chamfer_terms_final");
}

int gin_chamfer_terms_bwd(const void* plan_host, const void* plan_dev, const float* v, const float* tn, int64_t tnsb, int64_t tnsn,
                          int64_t tnsc, const float* tl, int64_t tlsb, int64_t tlsn, int64_t tlsc, const int32_t* idx_xy,
                          const int32_t* idx_yx, const float* dout, float* dv, void* ws, int B, int M, void* stream) {
  namespace ct = gin::chamfer_terms;
  const GinLossPlanHdr* h;
  int rc = chamfer_terms_args("gin_chamfer_terms_bwd", plan_host, plan_dev, v, tn, tl, idx_xy, idx_yx, dv, ws, B, M, &h);
  if (rc != GIN_OK || B == 0) return rc;
  if (!dout) return fail(GIN_ERR_ARG, "gin_chamfer_terms_bwd: null pointer (dout is required)");
  cudaStream_t st = (cudaStream_t)stream;
  const long long BV = (long long)B * h->V, BM = (long long)B * M;
  ct::Args a{};
  a.plan = plan_words(plan_dev); a.v = v;
  a.tn = gin::chamfer::Pts{tn, tnsb, tnsn, tnsc}; a.tl = gin::chamfer::Pts{tl, tlsb, tlsn, tlsc};
  a.idx_xy = idx_xy; a.idx_yx = idx_yx; a.dout = dout;
  a.g_n = reinterpret_cast<float*>(ws);
  a.g_l = a.g_n + BV * 3;
  a.acc_n = reinterpret_cast<gin::fixsum::Acc*>(a.g_l + BV * 3);
  a.acc_l = a.acc_n + BV;
  a.B = B; a.M = M;
  if (idx_yx) {
    if (cudaMemsetAsync(a.acc_n, 0, (size_t)BV * 2 * sizeof(gin::fixsum::Acc), st) != cudaSuccess)
      return fail(GIN_ERR_CUDA, "gin_chamfer_terms_bwd: memset failed");
    const unsigned blocks = (unsigned)((BM + ct::kThreads - 1) / ct::kThreads);
    ct::scatter_kernel<false><<<blocks, ct::kThreads, 0, st>>>(a);
    if ((rc = check_launch("chamfer_terms_scatter_stats"))) return rc;
    ct::scatter_kernel<true><<<blocks, ct::kThreads, 0, st>>>(a);
    if ((rc = check_launch("chamfer_terms_scatter_sum"))) return rc;
  }
  ct::cotangent_kernel<<<(unsigned)((BV + ct::kThreads - 1) / ct::kThreads), ct::kThreads, 0, st>>>(a);
  if ((rc = check_launch("chamfer_terms_cotangents"))) return rc;
  return gin_ring_ops_bwd(plan_host, plan_dev, v, tn ? a.g_n : nullptr, tl ? a.g_l : nullptr, dv, a.acc_n, B, stream);
}

}  // extern "C"
