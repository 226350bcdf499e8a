// Patch-mode tcgen05 wgrad for stride-1 layers:
//
//     dWp[tap][ci][co] += sum over pixels  bf16(x~[pixel + tap, ci]) * bf16(dY[pixel, co])
//
// GEMM with K = pixels.  The A operand is the SAME shared-memory patch the forward kernel stages (three
// column-shifted copies of the padded neighbourhood, 64 input channels wide), read "MN-major": K runs down the
// pixel rows, M across the 64 channels of a row.  One UMMA covers TWO taps at once (M = 128 = two 64-channel atoms
// whose distance is the descriptor's leading byte offset), so the seven taps cost four UMMA groups and the input is
// fetched once per tile instead of seven times.  The B operand is the dY tile (128 pixels x N_BLK channels).
// A CTA owns one (ci-block, co-block) unit and a contiguous slice of the pixel tiles; its 4 x N_BLK fp32
// accumulators stay in TMEM for the whole slice and are added to dWp with fp32 atomics at the end.
#pragma once
#include "gin_gemm_tcp.cuh"

namespace gin {
namespace tcwp {
using namespace tc;

constexpr int COPY_BYTES = tcp::COPY_BYTES;
constexpr int A_BYTES_ = 3 * COPY_BYTES;
constexpr int ATOM = BM * 128;                   // 128 pixel rows x 64 bf16
constexpr int MAX_ITEMS = tcp::MAX_ITEMS;

struct Params {
  const int32_t* plan;
  uint32_t fmt;               // operand-format bits of the instruction descriptor (gin_common.cuh: idesc_fmt_bits)
  GinPSide ps;
  int group, B, Cin, Cout, P;
  const __nv_bfloat16* X;      // [B*P + 2B][Cin] bf16
  const __nv_bfloat16* dY;     // [B*P (+2B)][Cout] bf16
  float* dWp;          // [7][Cin][Cout]
  int total_tiles, tiles_per_cta, slices, n_cblk;   // unit = blockIdx.x / slices: ci-block = unit % n_cblk, co-block = unit / n_cblk
};

template <int N_BLK>
struct Smem {
  static constexpr int B_BYTES = (N_BLK / 64) * ATOM;
  static constexpr int STAGE = A_BYTES_ + B_BYTES;
  static constexpr int BAR_OFF = 2 * STAGE;                 // full[2] empty[2] accum | tmem slot
  static constexpr int TOTAL = BAR_OFF + 5 * 8 + 16 + 1024;
};

// tap order by ascending start address inside a stage, paired: (3,6) (1,0) (2,5) (4,4)
__device__ __constant__ int8_t kPairTap[4][2] = {{3, 6}, {1, 0}, {2, 5}, {4, 4}};

GIN_DEVINL uint32_t tap_addr(int tap, int Q) {
  return (uint32_t)((tcp::kTapDj[tap] + 1) * COPY_BYTES + (1 + tcp::kTapDi[tap]) * Q * 1024);
}

template <int N_BLK>
__global__ void __launch_bounds__(THREADS, 1) wgrad_patch_tc_kernel(const Params p) {
  using L = Smem<N_BLK>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);
  uint64_t* empty_bar = full_bar + 2;
  uint64_t* accum_bar = empty_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_bar + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int unit = blockIdx.x / p.slices, slice = blockIdx.x % p.slices;
  const int ci0 = (unit % p.n_cblk) * 64, co0 = (unit / p.n_cblk) * N_BLK;
  const int T0 = slice * p.tiles_per_cta, T1 = min(T0 + p.tiles_per_cta, p.total_tiles);
  const int ntile = T1 - T0;
  const int Q = p.ps.Q, U = p.ps.U;
  constexpr uint32_t TM_COLS = (4 * N_BLK <= 256) ? 256 : 512;
  constexpr int NB = N_BLK / 64;

  if (warp == PRODUCER_WARPS) {
    if (lane == 0) {
      for (int s = 0; s < 2; ++s) { mbar_init(&full_bar[s], PRODUCER_THREADS); mbar_init(&empty_bar[s], 1); }
      mbar_init(accum_bar, 1);
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc(tmem_slot, TM_COLS);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (ntile <= 0) {
    __syncthreads();
    if (warp == PRODUCER_WARPS) tmem_dealloc(tmem_base, TM_COLS);
    return;
  }

  if (warp < PRODUCER_WARPS) {
    const int sub = lane >> 3, c8 = lane & 7;
    const __nv_bfloat16* __restrict__ Xc = p.X + ci0 + c8 * 8;
    const __nv_bfloat16* __restrict__ Yc = p.dY + co0 + c8 * 8;
    const long long total_pix = (long long)p.B * p.P;
    for (int ti = 0; ti < ntile; ++ti) {
      const int T = T0 + ti, G = T / p.ps.ntiles, t = T % p.ps.ntiles;
      const long long base = (long long)G * p.group * p.P;
      const int32_t* __restrict__ src_tab = p.plan + p.ps.src_off + (size_t)t * U;
      const int32_t* __restrict__ row_tab = p.plan + p.ps.rows_off + t * BM;
      int v[MAX_ITEMS], dv[4];
#pragma unroll
      for (int it = 0; it < MAX_ITEMS; ++it) {
        const int u = it * 32 + warp * 4 + sub;
        v[it] = (u < U) ? resolve_row(__ldg(src_tab + u), base, total_pix, G * p.group, p.B) : -1;
      }
#pragma unroll
      for (int ps = 0; ps < 4; ++ps) {
        const long long gd = base + __ldg(row_tab + ps * 32 + warp * 4 + sub);
        dv[ps] = (gd < total_pix) ? (int)gd : -1;
      }
      const int s = ti & 1;
      mbar_wait(&empty_bar[s], (((uint32_t)ti >> 1) & 1u) ^ 1u);
      const uint32_t st = smem_u32(smem + s * L::STAGE);
#pragma unroll
      for (int it = 0; it < MAX_ITEMS; ++it) {
        const int u = it * 32 + warp * 4 + sub;
        if (u < U) {
          const int cell = u / 10, c = u - cell * 10;
          const bool ok = v[it] >= 0;
          const __nv_bfloat16* src = Xc + (size_t)(ok ? v[it] : 0) * p.Cin;
          const uint32_t oct = st + cell * 1024;
          if (c <= 7) cp_async16(oct + swz(c, c8), src, ok);
          if (c >= 1 && c <= 8) cp_async16(oct + COPY_BYTES + swz(c - 1, c8), src, ok);
          if (c >= 2) cp_async16(oct + 2 * COPY_BYTES + swz(c - 2, c8), src, ok);
        }
      }
#pragma unroll
      for (int j = 0; j < NB; ++j)
#pragma unroll
        for (int ps = 0; ps < 4; ++ps) {
          const int r = ps * 32 + warp * 4 + sub;
          const bool ok = dv[ps] >= 0;
          cp_async16(st + A_BYTES_ + j * ATOM + swz(r, c8), Yc + (size_t)(ok ? dv[ps] : 0) * p.Cout + j * 64, ok);
        }
      cp_async_arrive(&full_bar[s]);
    }
    // ---- epilogue: TMEM -> atomics into dWp
    mbar_wait(accum_bar, 0);
    tc_fence_after();
    const int q = warp & 3, half = warp >> 2;
    const int row = q * 32 + lane;                 // 0..63 first tap of the pair, 64..127 second tap
    for (int pr = 0; pr < 4; ++pr) {
      const int tap = kPairTap[pr][row >> 6];
      const bool ok = !(pr == 3 && row >= 64);     // the duplicated half of the last pair
      float* dst = p.dWp + ((size_t)tap * p.Cin + ci0 + (row & 63)) * p.Cout + co0;
#pragma unroll 1
      for (int cb = 0; cb < N_BLK / 2; cb += 32) {
        const int col = half * (N_BLK / 2) + cb;
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(pr * N_BLK + col), v);
        tmem_ld_wait();
        if (ok) {
#pragma unroll
          for (int j = 0; j < 32; ++j) atomicAdd(dst + col + j, __uint_as_float(v[j]));
        }
      }
    }
    tc_fence_before();
  } else {
    const uint32_t idesc = make_idesc_f16kind(N_BLK, 1, 1) | p.fmt;
    if (lane == 0) {
      for (int ti = 0; ti < ntile; ++ti) {
        const int s = ti & 1;
        mbar_wait(&full_bar[s], ((uint32_t)ti >> 1) & 1u);
        fence_async_smem();
        tc_fence_after();
        const uint32_t a_addr = smem_u32(smem + s * L::STAGE), b_addr = a_addr + A_BYTES_;
#pragma unroll
        for (int pr = 0; pr < 4; ++pr) {
          const uint32_t ta = tap_addr(kPairTap[pr][0], Q), tb = tap_addr(kPairTap[pr][1], Q);
#pragma unroll
          for (int k = 0; k < BM / 16; ++k) {
            const uint64_t da = tcw::make_desc_mnmajor_sw128(a_addr + ta + k * 2048, tb - ta);
            const uint64_t db = tcw::make_desc_mnmajor_sw128(b_addr + k * 2048, ATOM);
            umma_bf16(tmem_base + (uint32_t)(pr * N_BLK), da, db, idesc, (ti | k) != 0);
          }
        }
        umma_commit(&empty_bar[s]);
      }
      umma_commit(accum_bar);
    }
    __syncwarp();
  }
  __syncthreads();
  if (warp == PRODUCER_WARPS) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TM_COLS);
  }
}

template <int N_BLK>
int launch(Params p, cudaStream_t st) {
  using L = Smem<N_BLK>;
  auto kern = wgrad_patch_tc_kernel<N_BLK>;
  static PerDeviceFlag configured_on;
  bool& configured = configured_on.here();
  if (!configured) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL) != cudaSuccess) return -3;
    configured = true;
  }
  p.n_cblk = p.Cin / 64;
  const int units = p.n_cblk * (p.Cout / N_BLK);
  int slices = (148 + units - 1) / units;
  if (units * slices > 148 && slices > 1) --slices;          // one wave
  if (slices > p.total_tiles) slices = p.total_tiles;
  if (slices < 1) slices = 1;
  p.slices = slices;
  p.tiles_per_cta = (p.total_tiles + slices - 1) / slices;
  kern<<<units * slices, THREADS, L::TOTAL, st>>>(p);
  return cudaGetLastError() == cudaSuccess ? 0 : -3;
}
}  // namespace tcwp

inline bool tcwp_supported(const GinPSide& ps, int Cin, int Cout) { return tcp_supported(ps, Cin, Cout); }

inline int launch_wgrad_patch_tc(const int32_t* plan_dev, const GinPSide& ps, int group, int P, const void* Xb, const void* dYb,
                                 float* dWp, int B, int Cin, int Cout, bool bf16, cudaStream_t st) {
  tcwp::Params p;
  p.plan = plan_dev; p.fmt = idesc_fmt_bits(bf16); p.ps = ps; p.group = group; p.B = B; p.Cin = Cin; p.Cout = Cout; p.P = P;
  p.X = reinterpret_cast<const __nv_bfloat16*>(Xb); p.dY = reinterpret_cast<const __nv_bfloat16*>(dYb); p.dWp = dWp;
  const int groups = (B + group - 1) / group;
  p.total_tiles = groups * ps.ntiles;
  if ((long long)B * P + 2LL * B >= 0x7fffffffLL) return -4;
  if (Cout % 128 == 0) return tcwp::launch<128>(p, st);
  return tcwp::launch<64>(p, st);
}

}  // namespace gin
