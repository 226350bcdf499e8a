// Patch-mode tcgen05 hex-conv for stride-1 layers (forward, and the in-chart part of dgrad).
//
// Measured fact that shapes this kernel (profiles/r01_*): on B200 the L2 -> SM path saturates at about the HBM
// rate (~5.7 TB/s), so re-reading every input row once per tap (7x, gather mode) makes the conv L2-bound.  Here
// the (R+2) x (8Q+2) padded neighbourhood of an R x 8Q pixel tile is fetched ONCE per 64-channel chunk
// (1.4x instead of 7x) from the bf16 activation copy and laid out in shared memory as three column-shifted copies
// (dj = -1, 0, +1).  Every tap (di, dj) is then the SAME shared-memory image read through a UMMA descriptor whose
// start address is moved by (1+di)*Q octets inside copy dj -- no data movement per tap at all.
//
// Persistent CTAs, one per SM:  8 producer warps | 1 MMA warp | 1 weight-copy warp | 4 epilogue warps.
//   A stage  = one 64-channel chunk of the patch (3 copies, 72 KB), double buffered
//   B stage  = one (tap, chunk) weight tile, bulk-copied from the pre-swizzled packed weights, 2-4 deep ring
//   TMEM     = two accumulators of N_TILE fp32 columns: the epilogue of tile i overlaps the MMAs of tile i+1
#pragma once
#include "gin_gemm_tc.cuh"

namespace gin {
namespace tcp {
using namespace tc;

constexpr int COPY_BYTES = 24 * 1024;            // (R+2)*Q octets of 1 KB; 24 KB covers (R,Q) = (4,4) and (8,2)
constexpr int A_STAGE_BYTES = 3 * COPY_BYTES;
constexpr int A_STAGES = 2;
constexpr int EPI_WARPS = 4;
constexpr int NWARPS = PRODUCER_WARPS + 2 + EPI_WARPS;
constexpr int NTHREADS = NWARPS * 32;
constexpr int MAX_ITEMS = 8;                     // source rows per producer thread and chunk: ceil(240 / 32)

struct Params {
  const int32_t* plan;
  uint32_t fmt;               // operand-format bits of the instruction descriptor (gin_common.cuh: idesc_fmt_bits)
  GinPSide ps;
  int group, B, K, N, P;      // P = pixels per sample (stride 1: same on both sides)
  const __nv_bfloat16* X;     // [B*P + 2B][K] bf16 (pixels, then pole-mean rows)
  const __nv_bfloat16* W;     // pre-swizzled bf16 tiles [7][K/64][N][64]
  const float* bias;
  float* Y;                   // [B*P][N] fp32
  int mirror;                 // 0 forward: tap (di,dj) reads cell (+di,+dj);  1 dgrad: reads (-di,-dj)
  int total_work, n_blocks;   // work item = (tile, n block)
};

template <int N_TILE, int B_STAGES>
struct Smem {
  static constexpr int B_BYTES = N_TILE * 128;
  static constexpr int B_OFF = A_STAGES * A_STAGE_BYTES;
  static constexpr int BAR_OFF = B_OFF + B_STAGES * B_BYTES;
  // a_full[2] a_empty[2] b_full[BS] b_empty[BS] acc_full[2] acc_empty[2] | tmem slot
  static constexpr int NBARS = 2 * A_STAGES + 2 * B_STAGES + 4;
  static constexpr int TOTAL = BAR_OFF + NBARS * 8 + 16 + 1024;
};

__device__ __constant__ int8_t kTapDi[7] = {0, -1, 1, 0, 0, -1, 1};
__device__ __constant__ int8_t kTapDj[7] = {0, 0, 0, -1, 1, 1, -1};

template <int N_TILE, int B_STAGES>
__global__ void __launch_bounds__(NTHREADS, 1) patch_gemm_tc_kernel(const Params p) {
  using L = Smem<N_TILE, B_STAGES>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* a_full = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);
  uint64_t* a_empty = a_full + A_STAGES;
  uint64_t* b_full = a_empty + A_STAGES;
  uint64_t* b_empty = b_full + B_STAGES;
  uint64_t* acc_full = b_empty + B_STAGES;
  uint64_t* acc_empty = acc_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int kchunks = p.K / BK;
  const int Q = p.ps.Q, U = p.ps.U;
  constexpr uint32_t TM_COLS = (2 * N_TILE <= 32) ? 32 : 2 * N_TILE;

  if (warp == PRODUCER_WARPS) {
    if (lane == 0) {
      for (int s = 0; s < A_STAGES; ++s) { mbar_init(&a_full[s], PRODUCER_THREADS); mbar_init(&a_empty[s], 1); }
      for (int s = 0; s < B_STAGES; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 1); }
      for (int s = 0; s < 2; ++s) { mbar_init(&acc_full[s], 1); mbar_init(&acc_empty[s], EPI_WARPS * 32); }
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc(tmem_slot, TM_COLS);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < PRODUCER_WARPS) {
    // =========================================================== producers: asynchronous patch gather
    // every 16-byte piece (8 channels of one source pixel) is copied by cp.async to its place in up to three of the
    // column-shifted copies; nothing passes through registers and both A stages can be in flight at once.
    const int sub = lane >> 3, c8 = lane & 7;
    const __nv_bfloat16* __restrict__ Xc = p.X + c8 * 8;
    const long long total_pix = (long long)p.B * p.P;
    uint32_t ac = 0;                                   // running A-stage counter
    for (int w = blockIdx.x; w < p.total_work; w += gridDim.x) {
      const int T = w / p.n_blocks;
      const int G = T / p.ps.ntiles, t = T % p.ps.ntiles;
      const long long base = (long long)G * p.group * p.P;
      const int32_t* __restrict__ src_tab = p.plan + p.ps.src_off + (size_t)t * U;
      int v[MAX_ITEMS];                                // this thread's source rows: u = it*32 + warp*4 + sub
#pragma unroll
      for (int it = 0; it < MAX_ITEMS; ++it) {
        const int u = it * 32 + warp * 4 + sub;
        v[it] = (u < U) ? resolve_row(__ldg(src_tab + u), base, total_pix, G * p.group, p.B) : -1;
      }
      for (int kc = 0; kc < kchunks; ++kc, ++ac) {
        const int s = ac & 1;
        mbar_wait(&a_empty[s], ((ac >> 1) & 1u) ^ 1u);
        const uint32_t st = smem_u32(smem + s * A_STAGE_BYTES);
#pragma unroll
        for (int it = 0; it < MAX_ITEMS; ++it) {
          const int u = it * 32 + warp * 4 + sub;
          if (u < U) {
            const int cell = u / 10, c = u - cell * 10;       // cell = i'*Q + q (octet of the padded patch), c = column 0..9
            const bool ok = v[it] >= 0;
            const __nv_bfloat16* src = Xc + (size_t)(ok ? v[it] : 0) * p.K + kc * BK;
            const uint32_t oct = st + cell * 1024;
            // copy 0 holds column j0+px-1, copy 1 column j0+px, copy 2 column j0+px+1   (c = column - (j0-1))
            if (c <= 7) cp_async16(oct + swz(c, c8), src, ok);                                   // dj = -1: px = c
            if (c >= 1 && c <= 8) cp_async16(oct + COPY_BYTES + swz(c - 1, c8), src, ok);        // dj =  0: px = c-1
            if (c >= 2) cp_async16(oct + 2 * COPY_BYTES + swz(c - 2, c8), src, ok);              // dj = +1: px = c-2
          }
        }
        cp_async_arrive(&a_full[s]);
      }
    }
  } else if (warp == PRODUCER_WARPS) {
    // =========================================================== MMA issuer
    const uint32_t idesc = make_idesc_f16kind(N_TILE) | p.fmt;
    if (lane == 0) {
      uint32_t ac = 0, bc = 0, wc = 0;
      for (int w = blockIdx.x; w < p.total_work; w += gridDim.x, ++wc) {
        const uint32_t ab = wc & 1;
        mbar_wait(&acc_empty[ab], ((wc >> 1) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + ab * N_TILE;
        for (int kc = 0; kc < kchunks; ++kc, ++ac) {
          const int s = ac & 1;
          mbar_wait(&a_full[s], (ac >> 1) & 1u);
          fence_async_smem();                          // cp.async (generic proxy) writes -> visible to the async proxy
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem + s * A_STAGE_BYTES);
          for (int tap = 0; tap < 7; ++tap, ++bc) {
            const int bs = bc % B_STAGES;
            mbar_wait(&b_full[bs], (bc / B_STAGES) & 1u);
            tc_fence_after();
            int di = kTapDi[tap], dj = kTapDj[tap];
            if (p.mirror) { di = -di; dj = -dj; }
            const uint64_t da = make_desc_kmajor_sw128(a_addr + (dj + 1) * COPY_BYTES + (1 + di) * Q * 1024);
            const uint64_t db = make_desc_kmajor_sw128(smem_u32(smem + L::B_OFF + bs * L::B_BYTES));
#pragma unroll
            for (int k = 0; k < BK / 16; ++k)
              umma_bf16(d_tmem, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, (kc | tap | k) != 0);
            umma_commit(&b_empty[bs]);
          }
          umma_commit(&a_empty[s]);
        }
        umma_commit(&acc_full[ab]);
      }
    }
    __syncwarp();
  } else if (warp == PRODUCER_WARPS + 1) {
    // =========================================================== weight tiles
    if (lane == 0) {
      uint32_t bc = 0;
      for (int w = blockIdx.x; w < p.total_work; w += gridDim.x) {
        const int n0 = (w % p.n_blocks) * N_TILE;
        for (int kc = 0; kc < kchunks; ++kc)
          for (int tap = 0; tap < 7; ++tap, ++bc) {
            const int bs = bc % B_STAGES;
            mbar_wait(&b_empty[bs], ((bc / B_STAGES) & 1u) ^ 1u);
            mbar_arrive_expect_tx(&b_full[bs], L::B_BYTES);
            const __nv_bfloat16* wsrc = p.W + (((size_t)tap * kchunks + kc) * p.N + n0) * BK;
            bulk_g2s(smem + L::B_OFF + bs * L::B_BYTES, wsrc, L::B_BYTES, &b_full[bs]);
          }
      }
    }
    __syncwarp();
  } else {
    // =========================================================== epilogue: TMEM -> registers -> global
    const int q = warp & 3;                         // TMEM lane quarter this warp may touch
    const int row = q * 32 + lane;
    uint32_t wc = 0;
    for (int w = blockIdx.x; w < p.total_work; w += gridDim.x, ++wc) {
      const int T = w / p.n_blocks, n0 = (w % p.n_blocks) * N_TILE;
      const int G = T / p.ps.ntiles, t = T % p.ps.ntiles;
      const long long gd = (long long)G * p.group * p.P + __ldg(p.plan + p.ps.rows_off + t * BM + row);
      const bool ok = gd < (long long)p.B * p.P;
      const uint32_t ab = wc & 1;
      mbar_wait(&acc_full[ab], (wc >> 1) & 1u);
      tc_fence_after();
      float* yp = p.Y + (size_t)gd * p.N + n0;
#pragma unroll 1
      for (int col = 0; col < N_TILE; col += 32) {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ab * N_TILE + col), v);
        tmem_ld_wait();
        if (ok) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            float4 o = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
            if (p.bias) {
              const float4 bb = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + col + j));
              o.x += bb.x; o.y += bb.y; o.z += bb.z; o.w += bb.w;
            }
            *reinterpret_cast<float4*>(yp + col + j) = o;
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&acc_empty[ab]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == PRODUCER_WARPS) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TM_COLS);
  }
}

template <int N_TILE, int B_STAGES>
int launch(const Params& p, cudaStream_t st) {
  using L = Smem<N_TILE, B_STAGES>;
  auto kern = patch_gemm_tc_kernel<N_TILE, B_STAGES>;
  static PerDeviceFlag configured_on;
  bool& configured = configured_on.here();
  if (!configured) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL) != cudaSuccess) return -3;
    configured = true;
  }
  const int grid = p.total_work < 148 ? p.total_work : 148;
  kern<<<grid, NTHREADS, L::TOTAL, st>>>(p);
  return cudaGetLastError() == cudaSuccess ? 0 : -3;
}

}  // namespace tcp

inline bool tcp_supported(const GinPSide& ps, int K, int N) {
  return ps.ntiles > 0 && ps.U <= tcp::MAX_ITEMS * 32 && (ps.R + 2) * ps.Q * 1024 <= tcp::COPY_BYTES && tc_supported(K, N);
}

inline int launch_patch_gemm_tc(const int32_t* plan_dev, const GinPSide& ps, int group, int P, const void* Xb, const void* Wb,
                                const float* bias, float* Y, int B, int K, int N, int mirror, bool bf16, cudaStream_t st) {
  tcp::Params p;
  p.plan = plan_dev; p.fmt = idesc_fmt_bits(bf16); p.ps = ps; p.group = group; p.B = B; p.K = K; p.N = N; p.P = P;
  p.X = reinterpret_cast<const __nv_bfloat16*>(Xb); p.W = reinterpret_cast<const __nv_bfloat16*>(Wb); p.bias = bias; p.Y = Y; p.mirror = mirror;
  if ((long long)B * P + 2LL * B >= 0x7fffffffLL) return -4;
  const int groups = (B + group - 1) / group;
  const long long tiles = (long long)groups * ps.ntiles;
  int rc;
  if (N % 256 == 0 && tiles * (N / 256) >= 148) { p.n_blocks = N / 256; p.total_work = (int)(tiles * p.n_blocks); rc = tcp::launch<256, 2>(p, st); }
  else if (N % 128 == 0 && tiles * (N / 128) >= 148) { p.n_blocks = N / 128; p.total_work = (int)(tiles * p.n_blocks); rc = tcp::launch<128, 3>(p, st); }
  else { p.n_blocks = N / 64; p.total_work = (int)(tiles * p.n_blocks); rc = tcp::launch<64, 4>(p, st); }
  return rc;
}

}  // namespace gin
