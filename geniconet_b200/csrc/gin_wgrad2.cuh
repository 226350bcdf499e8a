// Patch-mode tcgen05 wgrad for stride-1 layers, second generation:
//
//     dW[co][ci][tap] = sum over pixels  bf16(x~[pixel + tap, ci]) * bf16(dY[pixel, co])
//
// GEMM with K = pixels.  The A operand is the SAME single-copy patch image the forward kernel stages (gin_conv2.cuh: row u
// of the plan's source table at u*128 bytes, 64 input channels wide), read "MN-major": K runs down the pixel rows (8-row
// groups 1280 bytes apart), M across the 64 channels of a row.  One UMMA covers TWO taps (M = 128 = two 64-channel atoms
// whose distance, the descriptor's leading byte offset, is the difference of the taps' start rows), so the seven taps cost
// four UMMA groups and the input is fetched once per tile instead of seven times.  B is the dY tile (128 pixels x N_BLK).
// A CTA owns one (ci-block, co-block) unit and a contiguous slice of the pixel tiles; its 4 x N_BLK fp32 accumulators stay
// in TMEM for the whole slice.
//
// Against the first generation (gin_wgrad_tcp.cuh; 152 us for 128->64 @ I5, tensor pipe 14 % busy, profiles/r01b_wgrad*):
// single-copy patch (25 KB instead of 72 KB per tile, 3 stages), warp-uniform MMA issue loop, gather tables resolved by a
// table warp several tiles ahead, cp.async.cg, and NO atomics: every CTA writes its partial sums once and a small second
// kernel adds the slices in a fixed order and writes dW in its final [Cout][Cin][7] layout (deterministic; the 4.8 M fp32
// REDs of the old epilogue were 20 % of its samples).
#pragma once
#include "gin_conv2.cuh"

namespace gin {
namespace wg2 {
using namespace tc;

constexpr int PROD_WARPS = 8, PROD_THREADS = PROD_WARPS * 32;
constexpr int W_MMA = PROD_WARPS, W_TABLE = PROD_WARPS + 1;
constexpr int NWARPS = PROD_WARPS + 2, NTHREADS = NWARPS * 32;
constexpr int MAX_ITEMS = 8;
constexpr int MAX_STAGES = 4;
constexpr int TAB_SLOTS = 8, TAB_SRC = 256, TAB_ROWS = TAB_SRC + BM, TAB_BATCH = 4;
constexpr int ATOM = BM * 128;               // one 64-channel atom of the dY tile: 128 pixel rows x 128 bytes
constexpr int SMEM_LIMIT = 227 * 1024;
constexpr int MAX_CTAS = kMaxSMs;

// A tile is `nplanes` stages (gin_conv2.cuh: Params): stride 1 has one image and four tap pairs, stride 2 has one image per
// parity plane of the fine input and ONE tap pair per plane (taps {1,2} {5,6} {0,0} {3,4}); either way four accumulators.
struct Params {
  const int32_t* plan;
  uint32_t fmt;               // operand-format bits of the instruction descriptor (gin_common.cuh: idesc_fmt_bits)
  int U, Q, ntiles;
  int group, B, Cin, Cout;
  int P_src, P_dst;            // pixels per sample of the x map / of the dy map
  const __nv_bfloat16* X;      // [B*P_src + 2B][Cin] bf16
  const __nv_bfloat16* dY;     // [B*P_dst (+2B)][Cout] bf16
  float* partial;              // [gridDim.x][4][128][N_BLK] fp32
  int nplanes;
  int npairs[4];
  int16_t pair_row[4][4];      // start row of the pair's first tap inside the image
  int16_t pair_lbo[4][4];      // rows from the first to the second tap (>= 0: the descriptor's leading byte offset is unsigned)
  int8_t pair_acc[4][4];       // accumulator (0..3) of the pair
  int8_t tap_acc[8], tap_half[8];   // where tap t ends up: accumulator and half (rows 0-63 / 64-127)
  int tab_off, tab_tstride, tab_pstride, rows_off;
  int total_tiles, tiles_per_cta, slices, n_cblk;   // unit = blockIdx.x / slices: ci-block = unit % n_cblk, co-block = unit / n_cblk
  int a_bytes, stages;
};

GIN_DEVINL uint64_t desc_mnmajor(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(lbo_bytes >> 4) << 16;          // distance between the 64-element atoms along M / N
  d |= (uint64_t)(sbo_bytes >> 4) << 32;          // distance between 8-row groups along K
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

constexpr int NBARS = 2 * MAX_STAGES + 1 + 2 * TAB_SLOTS;
constexpr int BAR_BYTES = NBARS * 8 + 16;

template <int N_BLK>
__global__ void __launch_bounds__(NTHREADS, 1) wgrad_patch_kernel(const Params p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  constexpr int NB = N_BLK / 64;
  constexpr int B_BYTES = NB * ATOM;
  const int stage_bytes = p.a_bytes + B_BYTES;
  int32_t* tab = reinterpret_cast<int32_t*>(smem + p.stages * stage_bytes);      // [TAB_SLOTS][TAB_ROWS]
  uint64_t* bars = reinterpret_cast<uint64_t*>(tab + TAB_SLOTS * TAB_ROWS);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = full_bar + MAX_STAGES;
  uint64_t* accum_bar = empty_bar + MAX_STAGES;
  uint64_t* tab_full = accum_bar + 1;
  uint64_t* tab_empty = tab_full + TAB_SLOTS;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tab_empty + TAB_SLOTS);

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int unit = blockIdx.x / p.slices, slice = blockIdx.x % p.slices;
  const int ci0 = (unit % p.n_cblk) * 64, co0 = (unit / p.n_cblk) * N_BLK;
  const int T0 = slice * p.tiles_per_cta, T1 = min(T0 + p.tiles_per_cta, p.total_tiles);
  const int U = p.U, NS = p.stages, NP = p.nplanes;
  constexpr uint32_t TM_COLS = (4 * N_BLK <= 256) ? 256 : 512;

  if (warp == W_MMA) {
    if (lane == 0) {
      for (int s = 0; s < MAX_STAGES; ++s) { mbar_init(&full_bar[s], PROD_THREADS); mbar_init(&empty_bar[s], 1); }
      mbar_init(accum_bar, 1);
      for (int s = 0; s < TAB_SLOTS; ++s) { mbar_init(&tab_full[s], 1); mbar_init(&tab_empty[s], PROD_THREADS); }
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc(tmem_slot, TM_COLS);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  GIN_PDL_SYNC();

  if (warp < PROD_WARPS) {
    // =========================================================== producers: patch rows + dY rows, then the epilogue
    const int sub = lane >> 3, c8 = lane & 7;
    const __nv_bfloat16* __restrict__ Xc = p.X + ci0 + c8 * 8;
    const __nv_bfloat16* __restrict__ Yc = p.dY + co0 + c8 * 8;
    int s = 0, ts = 0;
    uint32_t ph = 0, tph = 0;
    for (int VT = T0 * NP; VT < T1 * NP; ++VT) {
      int v[MAX_ITEMS], dv[4];
      mbar_wait(&tab_full[ts], tph);
#pragma unroll
      for (int it = 0; it < MAX_ITEMS; ++it) v[it] = tab[ts * TAB_ROWS + it * 32 + warp * 4 + sub];
#pragma unroll
      for (int ps = 0; ps < 4; ++ps) dv[ps] = tab[ts * TAB_ROWS + TAB_SRC + ps * 32 + warp * 4 + sub];
      mbar_arrive(&tab_empty[ts]);
      if (++ts == TAB_SLOTS) { ts = 0; tph ^= 1u; }
      mbar_wait(&empty_bar[s], ph ^ 1u);
      const uint32_t st = smem_u32(smem + s * stage_bytes);
#pragma unroll
      for (int it = 0; it < MAX_ITEMS; ++it) {
        const int u = it * 32 + warp * 4 + sub;
        if (u < U) {
          const bool ok = v[it] >= 0;
          cp_async16_cg(st + swz(u, c8), Xc + (size_t)(ok ? v[it] : 0) * p.Cin, ok);
        }
      }
#pragma unroll
      for (int j = 0; j < NB; ++j)
#pragma unroll
        for (int ps = 0; ps < 4; ++ps) {
          const int r = ps * 32 + warp * 4 + sub;
          const bool ok = dv[ps] >= 0;
          cp_async16_cg(st + p.a_bytes + j * ATOM + swz(r, c8), Yc + (size_t)(ok ? dv[ps] : 0) * p.Cout + j * 64, ok);
        }
      cp_async_arrive(&full_bar[s]);
      if (++s == NS) { s = 0; ph ^= 1u; }
    }
    // ---- epilogue: TMEM -> this CTA's slot of the partial-sum workspace (no atomics)
    if (T1 > T0) {
      mbar_wait(accum_bar, 0);
      tc_fence_after();
    }
    const int q = warp & 3, half = warp >> 2;
    const int row = q * 32 + lane;                 // 0..63 first tap of the pair, 64..127 second tap
    float* out = p.partial + (size_t)blockIdx.x * 4 * BM * N_BLK;
    for (int pr = 0; pr < 4; ++pr) {
      float* dst = out + ((size_t)pr * BM + row) * N_BLK;
#pragma unroll 1
      for (int cb = 0; cb < N_BLK / 2; cb += 32) {
        const int col = half * (N_BLK / 2) + cb;
        uint32_t v[32];
        if (T1 > T0) {
          tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(pr * N_BLK + col), v);
          tmem_ld_wait();
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0u;
        }
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          *reinterpret_cast<float4*>(dst + col + j) =
              make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
      }
    }
    tc_fence_before();
  } else if (warp == W_MMA) {
    // =========================================================== MMA issuer (warp-uniform loop, one elected lane issues)
    const uint32_t idesc = make_idesc_f16kind(N_BLK, 1, 1) | p.fmt;
    const bool leader = elect_one();
    int s = 0;
    uint32_t ph = 0;
    for (int T = T0; T < T1; ++T)
      for (int pl = 0; pl < NP; ++pl) {
        mbar_wait(&full_bar[s], ph);
        fence_async_smem();
        tc_fence_after();
        const uint32_t a_addr = smem_u32(smem + s * stage_bytes), b_addr = a_addr + p.a_bytes;
        const int np = p.npairs[pl];
        for (int j = 0; j < np; ++j) {
          const uint32_t ta = (uint32_t)p.pair_row[pl][j] * 128u, lbo = (uint32_t)p.pair_lbo[pl][j] * 128u;
          const uint32_t d_tmem = tmem_base + (uint32_t)(p.pair_acc[pl][j] * N_BLK);
#pragma unroll
          for (int k = 0; k < BM / 16; ++k) {        // 16 pixel rows per MMA = two 8-row groups, 1280 bytes apart in the patch
            const uint64_t da = desc_mnmajor(a_addr + ta + k * 2560, lbo, 1280);
            const uint64_t db = desc_mnmajor(b_addr + k * 2048, ATOM, 1024);
            if (leader) umma_bf16(d_tmem, da, db, idesc, (T > T0) || (k != 0));
          }
        }
        if (leader) umma_commit(&empty_bar[s]);
        __syncwarp();
        if (++s == NS) { s = 0; ph ^= 1u; }
      }
    if (leader && T1 > T0) umma_commit(accum_bar);
    __syncwarp();
  } else {
    // =========================================================== gather tables (source rows + dY rows), several stages ahead
    const long long total_src = (long long)p.B * p.P_src, total_dst = (long long)p.B * p.P_dst;
    int ts = 0;
    uint32_t tph = 0;
    for (int Vb = T0 * NP; Vb < T1 * NP; Vb += TAB_BATCH) {
      int code[TAB_BATCH][MAX_ITEMS], rowc[TAB_BATCH][4];
#pragma unroll
      for (int j = 0; j < TAB_BATCH; ++j) {
        const int VT = Vb + j;
        if (VT < T1 * NP) {
          const int T = VT / NP, pl = VT - T * NP, t = T % p.ntiles;
          const int32_t* __restrict__ src_tab = p.plan + p.tab_off + (size_t)t * p.tab_tstride + (size_t)pl * p.tab_pstride;
          const int32_t* __restrict__ row_tab = p.plan + p.rows_off + t * BM;
#pragma unroll
          for (int it = 0; it < MAX_ITEMS; ++it) {
            const int u = it * 32 + lane;
            code[j][it] = (u < U) ? __ldg(src_tab + u) : GIN_SRC_ZERO;
          }
#pragma unroll
          for (int ps = 0; ps < 4; ++ps) rowc[j][ps] = __ldg(row_tab + ps * 32 + lane);
        }
      }
#pragma unroll
      for (int j = 0; j < TAB_BATCH; ++j) {
        const int VT = Vb + j;
        if (VT < T1 * NP) {
          const int G = (VT / NP) / p.ntiles;
          const long long base_s = (long long)G * p.group * p.P_src, base_d = (long long)G * p.group * p.P_dst;
          mbar_wait(&tab_empty[ts], tph ^ 1u);
#pragma unroll
          for (int it = 0; it < MAX_ITEMS; ++it)
            tab[ts * TAB_ROWS + it * 32 + lane] = resolve_row(code[j][it], base_s, total_src, G * p.group, p.B);
#pragma unroll
          for (int ps = 0; ps < 4; ++ps) {
            const long long gd = base_d + rowc[j][ps];
            tab[ts * TAB_ROWS + TAB_SRC + ps * 32 + lane] = (rowc[j][ps] >= 0 && gd < total_dst) ? (int)gd : -1;
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&tab_full[ts]);
          if (++ts == TAB_SLOTS) { ts = 0; tph ^= 1u; }
        }
      }
    }
  }
  __syncthreads();
  if (warp == W_MMA) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TM_COLS);
  }
}

struct TapMap { int8_t acc[8], half[8]; };

// dW[co][ci][tap] = sum over the slices of a unit (fixed order: deterministic); one thread per output, co runs fastest so the
// partial-sum reads are coalesced rows.  (Splitting the slice loop over several lanes measured slower, and so did eight loads in
// flight per thread instead of two -- 146 vs 117 us per step: the kernel is bound by the 20-40 MB of partials it streams from
// L2, not by latency.)
__global__ void __launch_bounds__(256)
wgrad_reduce_kernel(const float* __restrict__ partial, float* __restrict__ dW, int Cin, int Cout, int n_blk, int slices, int n_cblk, TapMap tm) {
  GIN_PDL_SYNC();
  const long long n = 7LL * Cin * Cout;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int co = (int)(i % Cout);
    const long long r = i / Cout;
    const int ci = (int)(r % Cin), tap = (int)(r / Cin);
    const int pr = tm.acc[tap], h = tm.half[tap];
    const int unit = (ci >> 6) + n_cblk * (co / n_blk);
    const float* src = partial + ((size_t)unit * slices * 4 + pr) * BM * n_blk + (size_t)(h * 64 + (ci & 63)) * n_blk + (co % n_blk);
    float a0 = 0.f, a1 = 0.f;
    int s = 0;
    for (; s + 1 < slices; s += 2) {
      a0 += __ldg(src + (size_t)s * 4 * BM * n_blk);
      a1 += __ldg(src + (size_t)(s + 1) * 4 * BM * n_blk);
    }
    if (s < slices) a0 += __ldg(src + (size_t)s * 4 * BM * n_blk);
    dW[((size_t)co * Cin + ci) * 7 + tap] = a0 + a1;
  }
}

template <int N_BLK>
int launch(Params p, float* dW, cudaStream_t st) {
  auto kern = wgrad_patch_kernel<N_BLK>;
  static PerDeviceFlag configured_on;
  bool& configured = configured_on.here();
  if (!configured) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT) != cudaSuccess) return -3;
    configured = true;
  }
  p.a_bytes = ((p.U * 128 + 1023) / 1024) * 1024;
  const int stage_bytes = p.a_bytes + (N_BLK / 64) * ATOM;
  const int fixed = TAB_SLOTS * TAB_ROWS * 4 + BAR_BYTES + 1024;
  p.stages = (SMEM_LIMIT - fixed) / stage_bytes;
  if (p.stages > MAX_STAGES) p.stages = MAX_STAGES;
  if (p.stages < 2) return -4;
  p.n_cblk = p.Cin / 64;
  const int units = p.n_cblk * (p.Cout / N_BLK);
  int slices = num_sms() / units;              // <= MAX_CTAS / units: the partial-sum workspace is sized for MAX_CTAS
  if (slices > p.total_tiles) slices = p.total_tiles;
  if (slices < 1) slices = 1;
  p.slices = slices;
  p.tiles_per_cta = (p.total_tiles + slices - 1) / slices;
  launch_pdl(kern, dim3(units * slices), dim3(NTHREADS), p.stages * stage_bytes + fixed, st, p);
  if (cudaGetLastError() != cudaSuccess) return -3;
  const long long n = 7LL * p.Cin * p.Cout;
  int blocks = (int)((n + 255) / 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  TapMap tm;
  for (int t = 0; t < 8; ++t) { tm.acc[t] = p.tap_acc[t]; tm.half[t] = p.tap_half[t]; }
  launch_pdl(wgrad_reduce_kernel, dim3(blocks), dim3(256), 0, st, (const float*)p.partial, dW, p.Cin, p.Cout, N_BLK, slices, p.n_cblk, tm);
  return cudaGetLastError() == cudaSuccess ? 0 : -3;
}

inline int pick_nblk(int Cout) { return Cout % 128 == 0 ? 128 : 64; }
// fp32 partial sums: at most MAX_CTAS CTAs x 4 pairs x 128 rows x N_BLK columns
inline size_t partial_bytes(int Cin, int Cout) {
  const int nblk = pick_nblk(Cout), units = (Cin / 64) * (Cout / nblk);
  const int ctas = units > MAX_CTAS ? units : (MAX_CTAS / units) * units;
  return (size_t)ctas * 4 * BM * nblk * 4;
}

}  // namespace wg2

inline bool wg2_supported(const GinPSide& ps, int Cin, int Cout) { return ps.ntiles > 0 && ps.U <= wg2::TAB_SRC && tc_supported(Cin, Cout); }
inline bool wg2_supported(const GinP2Side& ps, int Cin, int Cout) { return ps.ntiles > 0 && ps.U <= wg2::TAB_SRC && tc_supported(Cin, Cout); }

inline int wg2_dispatch(wg2::Params& p, float* dW, cudaStream_t st) {
  const int groups = (p.B + p.group - 1) / p.group;
  p.total_tiles = groups * p.ntiles;
  if ((long long)p.B * (p.P_src > p.P_dst ? p.P_src : p.P_dst) + 2LL * p.B >= 0x7fffffffLL) return -4;
  if (wg2::pick_nblk(p.Cout) == 128) return wg2::launch<128>(p, dW, st);
  return wg2::launch<64>(p, dW, st);
}

// stride 1.  Taps sorted by start row inside the single-copy patch (1, 2, 10Q, 10Q+1, 10Q+2, 20Q, 20Q+1 for taps 1 5 3 0 4 6 2) and
// paired so that the second tap of a pair never starts before the first: (1,5) (3,0) (4,6) (2,2).
// Writes dW[Cout][Cin][7] directly; `partial` needs wg2::partial_bytes(Cin, Cout) bytes.
inline int launch_wgrad_patch2(const int32_t* plan_dev, const GinPSide& ps, int group, int P, const void* Xb, const void* dYb, float* partial,
                               float* dW, int B, int Cin, int Cout, bool bf16, cudaStream_t st) {
  static const int pairs[4][2] = {{1, 5}, {3, 0}, {4, 6}, {2, 2}};
  wg2::Params p{};
  p.plan = plan_dev; p.fmt = idesc_fmt_bits(bf16); p.U = ps.U; p.Q = ps.Q; p.ntiles = ps.ntiles; p.group = group; p.B = B; p.Cin = Cin; p.Cout = Cout; p.P_src = P; p.P_dst = P;
  p.X = reinterpret_cast<const __nv_bfloat16*>(Xb); p.dY = reinterpret_cast<const __nv_bfloat16*>(dYb); p.partial = partial;
  p.nplanes = 1; p.npairs[0] = 4;
  for (int j = 0; j < 4; ++j) {
    const int a = pairs[j][0], b = pairs[j][1];
    const int ra = (1 + cv2::kDi[a]) * ps.Q * 10 + (1 + cv2::kDj[a]), rb = (1 + cv2::kDi[b]) * ps.Q * 10 + (1 + cv2::kDj[b]);
    p.pair_row[0][j] = (int16_t)ra; p.pair_lbo[0][j] = (int16_t)(rb - ra); p.pair_acc[0][j] = (int8_t)j;
    p.tap_acc[a] = (int8_t)j; p.tap_half[a] = 0;
    if (b != a) { p.tap_acc[b] = (int8_t)j; p.tap_half[b] = 1; }
  }
  p.tab_off = ps.src_off; p.tab_tstride = ps.U; p.tab_pstride = 0; p.rows_off = ps.rows_off;
  return wg2_dispatch(p, dW, st);
}

// stride 2: one tap pair per parity plane of the fine input: plane 0 (1,2), plane 1 (5,6), plane 2 (0,0), plane 3 (3,4)
inline int launch_wgrad_patch2_s2(const int32_t* plan_dev, const GinP2Side& ps, int group, int P_f, int P_c, const void* Xb, const void* dYb,
                                  float* partial, float* dW, int B, int Cin, int Cout, bool bf16, cudaStream_t st) {
  static const int pairs[4][2] = {{1, 2}, {5, 6}, {0, 0}, {3, 4}};
  wg2::Params p{};
  p.plan = plan_dev; p.fmt = idesc_fmt_bits(bf16); p.U = ps.U; p.Q = ps.Q; p.ntiles = ps.ntiles; p.group = group; p.B = B; p.Cin = Cin; p.Cout = Cout; p.P_src = P_f; p.P_dst = P_c;
  p.X = reinterpret_cast<const __nv_bfloat16*>(Xb); p.dY = reinterpret_cast<const __nv_bfloat16*>(dYb); p.partial = partial;
  p.nplanes = 4;
  for (int pl = 0; pl < 4; ++pl) {
    const int a = pairs[pl][0], b = pairs[pl][1];
    const int ra = (1 + kS2A[a]) * ps.Q * 10 + (1 + kS2B[a]), rb = (1 + kS2A[b]) * ps.Q * 10 + (1 + kS2B[b]);
    if (rb < ra) return -4;
    p.npairs[pl] = 1;
    p.pair_row[pl][0] = (int16_t)ra; p.pair_lbo[pl][0] = (int16_t)(rb - ra); p.pair_acc[pl][0] = (int8_t)pl;
    p.tap_acc[a] = (int8_t)pl; p.tap_half[a] = 0;
    if (b != a) { p.tap_acc[b] = (int8_t)pl; p.tap_half[b] = 1; }
  }
  p.tab_off = ps.src_off; p.tab_tstride = 4 * ps.U; p.tab_pstride = ps.U; p.rows_off = ps.rows_off;
  return wg2_dispatch(p, dW, st);
}

}  // namespace gin
