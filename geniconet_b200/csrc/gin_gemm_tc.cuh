// tcgen05 implicit-GEMM hex-conv (forward and dgrad; rows a1+a2+a3+a5 of SURVEY 8a).
//
//   dst[row, n] = bias[n] + sum_{slot} sum_k  bf16(X[src[slot][row], k]) * bf16(W[tap(slot)][n][k])
//
// One CTA owns one 128-row tile x N_TILE output channels.  The accumulator lives in TMEM
// (128 lanes x N_TILE fp32 columns); the A operand is GATHERED: eight producer warps read the
// source rows named by the plan (chart padding, pole means, stride-2 lattice and the adjoint
// tables are all just row indices), convert fp32 -> bf16 in registers and write the
// 128-byte-swizzled K-major tile that the UMMA smem descriptor expects.  The B operand is the
// pre-packed bf16 weight slice W[tap][n0:n0+N_TILE][k0:k0+64].  A single elected thread issues
// tcgen05.mma; stages are recycled through mbarriers signalled by tcgen05.commit.
//
// The K loop runs k-chunk outer / tap inner, so the seven taps of one 64-channel chunk re-read
// the same few source rows back to back (L1-resident), and HBM/L2 see each row about once.
#pragma once
#include <cuda_bf16.h>

#include "gin_common.cuh"

namespace gin {
namespace tc {

constexpr int BM = 128;              // rows per tile (UMMA M)
constexpr int BK = 64;               // channels per stage: 64 bf16 = one 128-byte swizzle row
constexpr int PRODUCER_WARPS = 8;
constexpr int PRODUCER_THREADS = PRODUCER_WARPS * 32;
constexpr int THREADS = PRODUCER_THREADS + 32;   // + the MMA / TMEM warp
constexpr int A_BYTES = BM * BK * 2;             // 16 KB

// ------------------------------------------------------------------ PTX wrappers
GIN_DEVINL uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

GIN_DEVINL void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
GIN_DEVINL void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
GIN_DEVINL void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity)
      : "memory");
}
// true on exactly one (elected) lane of a fully converged warp
GIN_DEVINL bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
// non-blocking: has the phase with this parity completed?
GIN_DEVINL bool mbar_test(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
GIN_DEVINL void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
GIN_DEVINL void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
GIN_DEVINL void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
GIN_DEVINL void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

GIN_DEVINL void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
GIN_DEVINL void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], bf16 x bf16 -> fp32, issued by ONE thread
GIN_DEVINL void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc),
      "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier once every previously issued tcgen05.mma of this thread has completed
GIN_DEVINL void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread (thread t = TMEM lane base+t)
GIN_DEVINL void tmem_ld32(uint32_t taddr, uint32_t v[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
        "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
        "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
        "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
GIN_DEVINL void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128-byte-swizzled operand tile: rows of 128 B, 8-row atoms of 1024 B (SBO), LBO unused.
GIN_DEVINL uint64_t make_desc_kmajor_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);   // start address
  d |= (uint64_t)0 << 16;                         // leading byte offset (ignored for swizzled K-major)
  d |= (uint64_t)(1024u >> 4) << 32;              // stride byte offset: 8 rows x 128 B
  d |= (uint64_t)1 << 46;                         // descriptor version (sm_100)
  d |= (uint64_t)2 << 61;                         // SWIZZLE_128B
  return d;
}
// kind::f16 instruction descriptor WITHOUT the operand-format bits (those come from Params::fmt, see gin_common.cuh
// idesc_fmt_bits): D = f32, M = 128, operands K-major unless flagged
__host__ __device__ constexpr uint32_t make_idesc_f16kind(int n, int a_mn_major = 0, int b_mn_major = 0) {
  return (1u << 4) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}
// bf16 x bf16 (experiments under tools/exp)
__host__ __device__ constexpr uint32_t make_idesc_bf16(int n, int a_mn_major = 0, int b_mn_major = 0) {
  return make_idesc_f16kind(n, a_mn_major, b_mn_major) | (1u << 7) | (1u << 10);
}

GIN_DEVINL uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

// byte offset of 16-byte chunk `c` of row `r` inside a 128B-swizzled tile whose base is 1024-aligned
GIN_DEVINL uint32_t swz(int r, int c) { return (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4)); }

// 16-byte asynchronous global -> shared copy (LDGSTS); src_bytes == 0 writes zeros instead of reading
GIN_DEVINL void cp_async16(uint32_t dst_smem, const void* src, bool valid) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(dst_smem), "l"(src), "r"(valid ? 16 : 0) : "memory");
}
// same, bypassing L1 (the data is read once; with ~200 KB of the SM's 228 KB configured as shared memory the L1 is too small to hold
// the lines of the cp.async in flight, and allocating them throttles the whole gather)
GIN_DEVINL void cp_async16_cg(uint32_t dst_smem, const void* src, bool valid) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst_smem), "l"(src), "r"(valid ? 16 : 0) : "memory");
}
// the mbarrier receives one (pre-counted) arrival once every cp.async issued so far by this thread has landed
GIN_DEVINL void cp_async_arrive(uint64_t* bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
GIN_DEVINL void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// contiguous global -> shared bulk copy (TMA engine, no tensor map); completion is counted in bytes on `bar`
GIN_DEVINL void bulk_g2s(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// Source rows of the bf16 activation copy made by cast_bf16_kernel: rows [0, B*P) are the pixels, rows
// B*P + 2*sample + pole hold the pole means (corner_mode 'average'), so a pole cell is an ordinary row.
GIN_DEVINL int resolve_row(int code, long long base, long long total_pix, int sample0, int B) {
  if (code >= 0) { const long long gp = base + code; return gp < total_pix ? (int)gp : -1; }
  if (code <= -2) { const int q = -2 - code, sample = sample0 + (q >> 1); return sample < B ? (int)(total_pix + 2 * sample + (q & 1)) : -1; }
  return -1;
}

struct Params {
  const int32_t* plan;
  uint32_t fmt;               // operand-format bits of the instruction descriptor (gin_common.cuh: idesc_fmt_bits)
  GinSide side;
  int group, B, K, N;
  const __nv_bfloat16* X;    // [B*P_src + 2B][K] bf16 (pixels, then pole-mean rows)
  const __nv_bfloat16* W;    // pre-swizzled bf16 tiles [7][K/64][N][64] (see pack_weights_kernel)
  const float* bias;         // [N] or null
  float* Y;                  // [B*P_dst][N] fp32
  int accumulate;            // 1: Y += result; 2: atomic Y += result (seam pass of a split dgrad: rows may share a pixel)
};

constexpr int WARPS = PRODUCER_WARPS + 2;        // + MMA/TMEM warp + weight-copy warp
constexpr int THREADS2 = WARPS * 32;

template <int N_TILE, int STAGES>
struct Smem {
  static constexpr int B_BYTES = N_TILE * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int BAR_OFF = STAGES * STAGE_BYTES;                       // full[STAGES], empty[STAGES], accum
  static constexpr int SRC_OFF = BAR_OFF + (2 * STAGES + 1) * 8 + 8;         // + tmem ptr
  static constexpr int TOTAL = SRC_OFF + GIN_MAX_SLOTS * BM * 4 + BM * 8 + 1024;  // + src table + dst rows + align slack
};

// Gather-mode kernel: one CTA = one 128-row tile x N_TILE channels; every (slot, 64-channel chunk) is a stage whose
// 128 rows are fetched by cp.async straight into the swizzled tile.  Used for stride-2 convs and the seam pass.
template <int N_TILE, int STAGES>
__global__ void __launch_bounds__(THREADS2, (N_TILE <= 128 ? 2 : 1)) gather_gemm_tc_kernel(const Params p) {
  using L = Smem<N_TILE, STAGES>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* accum_bar = empty_bar + STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_bar + 1);
  int32_t* src_s = reinterpret_cast<int32_t*>(smem + L::SRC_OFF);            // [nslots][128] resolved source rows
  long long* dst_s = reinterpret_cast<long long*>(src_s + GIN_MAX_SLOTS * BM);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int G = blockIdx.x / p.side.ntiles, t = blockIdx.x % p.side.ntiles;
  const int n0 = blockIdx.y * N_TILE;
  const GinTileDesc* desc = reinterpret_cast<const GinTileDesc*>(p.plan + p.side.tiles_off) + t;
  const int nslots = desc->nslots;
  const int kchunks = p.K / BK;
  const int total_stages = nslots * kchunks;

  if (warp == PRODUCER_WARPS) {
    if (lane == 0) {
      for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], PRODUCER_THREADS + 1); mbar_init(&empty_bar[s], 1); }
      mbar_init(accum_bar, 1);
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc(tmem_slot, N_TILE < 32 ? 32 : N_TILE);
  } else if (warp < PRODUCER_WARPS) {
    const long long base_src = (long long)G * p.group * p.side.P_src, total_src = (long long)p.B * p.side.P_src;
    const int32_t* src_tab = p.plan + p.side.src_off + desc->src_off;
    for (int i = tid; i < nslots * BM; i += PRODUCER_THREADS) src_s[i] = resolve_row(src_tab[i], base_src, total_src, G * p.group, p.B);
    if (tid < BM) {
      const long long base_dst = (long long)G * p.group * p.side.P_dst, total_dst = (long long)p.B * p.side.P_dst;
      const int r = p.plan[p.side.rows_off + t * BM + tid];
      const long long d = (r >= 0) ? base_dst + r : -1;
      dst_s[tid] = (d >= 0 && d < total_dst) ? d : -1;
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < PRODUCER_WARPS) {
    // =========================================================== producers: asynchronous row gather
    const int sub = lane >> 3, c8 = lane & 7;
    const __nv_bfloat16* __restrict__ Xc = p.X + c8 * 8;
    for (int it = 0; it < total_stages; ++it) {
      const int s = it % STAGES;
      const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
      const int kc = it / nslots, slot = it - kc * nslots;
      mbar_wait(&empty_bar[s], ph ^ 1u);
      const uint32_t a_tile = smem_u32(smem + s * L::STAGE_BYTES);
#pragma unroll
      for (int ps = 0; ps < 4; ++ps) {
        const int r = ps * 32 + warp * 4 + sub;
        const int v = src_s[slot * BM + r];
        cp_async16(a_tile + swz(r, c8), Xc + (size_t)(v < 0 ? 0 : v) * p.K + kc * BK, v >= 0);
      }
      cp_async_arrive(&full_bar[s]);
    }
    // =========================================================== epilogue: TMEM -> registers -> global
    mbar_wait(accum_bar, 0);
    tc_fence_after();
    const int q = warp & 3;                         // TMEM lane quarter this warp may touch
    const int half = warp >> 2;                     // column half
    const int row = q * 32 + lane;
    const long long d = dst_s[row];
    constexpr int COLS_PER_WARP = N_TILE / 2;
#pragma unroll 1
    for (int cb = 0; cb < COLS_PER_WARP; cb += 32) {
      const int col = half * COLS_PER_WARP + cb;
      uint32_t v[32];
      tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)col, v);
      tmem_ld_wait();
      if (d >= 0) {
        float* yp = p.Y + (size_t)d * p.N + n0 + col;
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          float4 o = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
          if (p.bias) {
            const float4 bb = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + col + j));
            o.x += bb.x; o.y += bb.y; o.z += bb.z; o.w += bb.w;
          }
          if (p.accumulate == 2) {          // several rows (of this or other tiles) may share a destination pixel
            atomicAdd(yp + j, o.x); atomicAdd(yp + j + 1, o.y); atomicAdd(yp + j + 2, o.z); atomicAdd(yp + j + 3, o.w);
          } else {
            if (p.accumulate) {
              const float4 old = *reinterpret_cast<const float4*>(yp + j);
              o.x += old.x; o.y += old.y; o.z += old.z; o.w += old.w;
            }
            *reinterpret_cast<float4*>(yp + j) = o;
          }
        }
      }
    }
    tc_fence_before();
  } else if (warp == PRODUCER_WARPS) {
    // =========================================================== MMA issuer (one elected thread)
    const uint32_t idesc = make_idesc_f16kind(N_TILE) | p.fmt;
    if (lane == 0) {
      for (int it = 0; it < total_stages; ++it) {
        const int s = it % STAGES;
        const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
        mbar_wait(&full_bar[s], ph);
        fence_async_smem();                  // cp.async (generic proxy) writes -> visible to the tensor-core (async) proxy
        tc_fence_after();
        const uint32_t a_addr = smem_u32(smem + s * L::STAGE_BYTES);
        const uint64_t da = make_desc_kmajor_sw128(a_addr), db = make_desc_kmajor_sw128(a_addr + A_BYTES);
#pragma unroll
        for (int k = 0; k < BK / 16; ++k)   // UMMA_K = 16 bf16 = 32 bytes inside the swizzle atom
          umma_bf16(tmem_base, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, (it | k) != 0);
        umma_commit(&empty_bar[s]);          // frees the stage once these MMAs have read it
      }
      umma_commit(accum_bar);                // accumulator complete
    }
    __syncwarp();
  } else {
    // =========================================================== weight tiles: one bulk copy per stage
    if (lane == 0) {
      for (int it = 0; it < total_stages; ++it) {
        const int s = it % STAGES;
        const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
        const int kc = it / nslots, slot = it - kc * nslots;
        const int tap = desc->tap[slot];
        mbar_wait(&empty_bar[s], ph ^ 1u);
        mbar_arrive_expect_tx(&full_bar[s], L::B_BYTES);
        const __nv_bfloat16* wsrc = p.W + (((size_t)tap * kchunks + kc) * p.N + n0) * BK;
        bulk_g2s(smem + s * L::STAGE_BYTES + A_BYTES, wsrc, L::B_BYTES, &full_bar[s]);
      }
    }
    __syncwarp();
  }
  __syncthreads();
  if (warp == PRODUCER_WARPS) {
    tc_fence_after();
    tmem_dealloc(tmem_base, N_TILE < 32 ? 32 : N_TILE);
  }
}

template <int N_TILE, int STAGES>
int launch(const Params& p, int ntiles, cudaStream_t st) {
  using L = Smem<N_TILE, STAGES>;
  auto kern = gather_gemm_tc_kernel<N_TILE, STAGES>;
  static PerDeviceFlag configured_on;
  bool& configured = configured_on.here();
  if (!configured) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL) != cudaSuccess) return -3;
    configured = true;
  }
  dim3 grid((unsigned)ntiles, (unsigned)(p.N / N_TILE));
  kern<<<grid, THREADS2, L::TOTAL, st>>>(p);
  return cudaGetLastError() == cudaSuccess ? 0 : -3;
}

}  // namespace tc

inline bool tc_supported(int K, int N) { return K % 64 == 0 && N % 64 == 0 && K >= 64 && N >= 64; }

inline int launch_gather_gemm_tc(const int32_t* plan_dev, const GinSide& side, int group, const void* Xb, const void* Wb,
                                 const float* bias, float* Y, int B, int K, int N, int ntiles, bool bf16, cudaStream_t st, int accumulate = 0) {
  tc::Params p;
  p.plan = plan_dev; p.fmt = idesc_fmt_bits(bf16); p.side = side; p.group = group; p.B = B; p.K = K; p.N = N;
  p.X = reinterpret_cast<const __nv_bfloat16*>(Xb); p.W = reinterpret_cast<const __nv_bfloat16*>(Wb); p.bias = bias; p.Y = Y;
  p.accumulate = accumulate;
  if ((long long)B * side.P_src + 2LL * B >= 0x7fffffffLL) return -4;
  // widest N tile that still gives every SM a CTA
  if (N % 256 == 0 && (long long)ntiles * (N / 256) >= 148) return tc::launch<256, 3>(p, ntiles, st);
  if (N % 128 == 0 && (long long)ntiles * (N / 128) >= 148) return tc::launch<128, 3>(p, ntiles, st);
  return tc::launch<64, 4>(p, ntiles, st);
}

// ======================================================================================= wgrad (gather mode)
//   dWp[tap][ci][co] += sum_rows X[src_tap[row], ci] * dY[row, co]          (bf16 operands, fp32 accumulate)
//
// GEMM with K = pixels.  Both operands are "MN-major" for the tensor core: a staged tile is
// [pixel row][64 channels = 128 swizzled bytes] read by UMMA with K running down the rows.  M = 128 is a PAIR of
// 64-channel atoms (tap, ci-block): two ci-blocks of one tap when Cin >= 128, two taps when Cin == 64.
// A CTA owns `npairs` pairs x N_BLK output channels (npairs * N_BLK <= 512 TMEM columns) and a slice of the pixel
// tiles; partial sums are added to dWp with fp32 atomics.  Used for the stride-2 layers.
namespace tcw {
using namespace tc;

struct Params {
  const int32_t* plan;
  uint32_t fmt;               // operand-format bits of the instruction descriptor (gin_common.cuh: idesc_fmt_bits)
  GinSide side;
  int group, B, Cin, Cout;
  const __nv_bfloat16* X;     // [B*P_src + 2B][Cin]
  const __nv_bfloat16* dY;    // [B*P_dst (+2B)][Cout]
  float* dWp;                 // [7][Cin][Cout]
  int total_tiles, tiles_per_cta, units_m;   // units_m: number of pair-groups along M
};

constexpr int ATOM_BYTES = BM * 128;          // 128 pixel rows x 64 bf16

template <int N_BLK, int NPAIRS, int STAGES>
struct Smem {
  static constexpr int A_STAGE = 2 * ATOM_BYTES;                 // one pair
  static constexpr int B_BYTES_ = (N_BLK / 64) * ATOM_BYTES;     // dY tile, double buffered
  static constexpr int B_OFF = STAGES * A_STAGE;
  static constexpr int BAR_OFF = B_OFF + 2 * B_BYTES_;
  // a_full[STAGES], a_empty[STAGES], b_full[2], b_empty[2], accum, tmem slot, then the per-tile row tables
  static constexpr int TAB_OFF = BAR_OFF + (2 * STAGES + 5) * 8 + 16;
  static constexpr int TOTAL = TAB_OFF + 8 * BM * 4 + 1024;
};

GIN_DEVINL uint64_t make_desc_mnmajor_sw128(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(lbo_bytes >> 4) << 16;          // stride between 64-element atoms along M/N
  d |= (uint64_t)(1024u >> 4) << 32;              // stride between 8-row groups along K
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// atom index a in [0, 7*Cin/64): tap = a / (Cin/64), ci-block = a % (Cin/64)  (Cin >= 128: consecutive atoms pair up
// inside one tap because Cin/64 is even; Cin == 64: consecutive taps pair up, atom 7 is an all-zero dummy)
template <int N_BLK, int NPAIRS, int STAGES>
__global__ void __launch_bounds__(THREADS, 1) wgrad_tc_kernel(const Params p) {
  using L = Smem<N_BLK, NPAIRS, STAGES>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* a_full = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);
  uint64_t* a_empty = a_full + STAGES;
  uint64_t* b_full = a_empty + STAGES;
  uint64_t* b_empty = b_full + 2;
  uint64_t* accum_bar = b_empty + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_bar + 1);
  int32_t* tab_s = reinterpret_cast<int32_t*>(smem + L::TAB_OFF);     // [8][128]: rows 0..6 = per-tap source row, row 7 = dst pixel

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int cblocks = p.Cin / 64, natoms = 7 * cblocks;
  const int unit_m = blockIdx.y % p.units_m, unit_n = blockIdx.y / p.units_m;
  const int pair0 = unit_m * NPAIRS;                       // first pair of this CTA
  const int total_pairs = (natoms + 1) / 2;
  const int npairs = min(NPAIRS, total_pairs - pair0);
  const int n0 = unit_n * N_BLK;
  const int T0 = blockIdx.x * p.tiles_per_cta, T1 = min(T0 + p.tiles_per_cta, p.total_tiles);
  const int ntile = T1 - T0;
  constexpr int TM_COLS = (NPAIRS * N_BLK <= 32) ? 32 : (NPAIRS * N_BLK <= 64) ? 64 : (NPAIRS * N_BLK <= 128) ? 128 : (NPAIRS * N_BLK <= 256) ? 256 : 512;
  constexpr int NB = N_BLK / 64;                            // dY atoms per pixel tile

  if (warp == PRODUCER_WARPS) {
    if (lane == 0) {
      for (int s = 0; s < STAGES; ++s) { mbar_init(&a_full[s], PRODUCER_THREADS); mbar_init(&a_empty[s], 1); }
      for (int s = 0; s < 2; ++s) { mbar_init(&b_full[s], PRODUCER_THREADS); mbar_init(&b_empty[s], 1); }
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
  if (ntile <= 0 || npairs <= 0) {
    __syncthreads();
    if (warp == PRODUCER_WARPS) tmem_dealloc(tmem_base, TM_COLS);
    return;
  }

  if (warp < PRODUCER_WARPS) {
    const long long total_src = (long long)p.B * p.side.P_src, total_dst = (long long)p.B * p.side.P_dst;
    const int sub = lane >> 3, c8 = lane & 7;
    uint32_t it = 0;                                        // running A-pair counter (stage ring)
    for (int ti = 0; ti < ntile; ++ti) {
      const int T = T0 + ti, G = T / p.side.ntiles, t = T % p.side.ntiles;
      const GinTileDesc* desc = reinterpret_cast<const GinTileDesc*>(p.plan + p.side.tiles_off) + t;
      const int32_t* src_tab = p.plan + p.side.src_off + desc->src_off;
      const long long base_src = (long long)G * p.group * p.side.P_src, base_dst = (long long)G * p.group * p.side.P_dst;
      // resolve this tile's tables into shared memory (producers only; addresses are consumed at issue time)
      asm volatile("bar.sync 1, %0;" ::"n"(PRODUCER_THREADS) : "memory");
      for (int i = tid; i < 8 * BM; i += PRODUCER_THREADS) {
        const int trow = i >> 7, r = i & (BM - 1);
        const int dr = p.plan[p.side.rows_off + t * BM + r];
        const long long d = (dr >= 0) ? base_dst + dr : -1;
        const bool row_ok = d >= 0 && d < total_dst;
        int v = -1;
        if (trow == 7) v = row_ok ? (int)d : -1;
        else if (row_ok) {
          int slot = -1;
          for (int q = 0; q < desc->nslots; ++q) if (desc->tap[q] == trow) { slot = q; break; }
          if (slot >= 0) v = resolve_row(src_tab[slot * BM + r], base_src, total_src, G * p.group, p.B);
        }
        tab_s[i] = v;
      }
      asm volatile("bar.sync 1, %0;" ::"n"(PRODUCER_THREADS) : "memory");
      // dY tile (double buffered)
      {
        const int bs = ti & 1;
        mbar_wait(&b_empty[bs], (((uint32_t)ti >> 1) & 1u) ^ 1u);
        const uint32_t bt = smem_u32(smem + L::B_OFF + bs * L::B_BYTES_);
#pragma unroll
        for (int j = 0; j < NB; ++j)
#pragma unroll
          for (int ps = 0; ps < 4; ++ps) {
            const int r = ps * 32 + warp * 4 + sub;
            const int v = tab_s[7 * BM + r];
            cp_async16(bt + j * ATOM_BYTES + swz(r, c8), p.dY + (size_t)(v < 0 ? 0 : v) * p.Cout + n0 + j * 64 + c8 * 8, v >= 0);
          }
        cp_async_arrive(&b_full[bs]);
      }
      for (int pr = 0; pr < npairs; ++pr, ++it) {
        const int s = it % STAGES;
        mbar_wait(&a_empty[s], ((it / STAGES) & 1u) ^ 1u);
        const uint32_t at = smem_u32(smem + s * L::A_STAGE);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int atom = (pair0 + pr) * 2 + h;
          const bool dummy = atom >= natoms;
          const int tap = dummy ? 0 : atom / cblocks, cb = dummy ? 0 : atom % cblocks;
#pragma unroll
          for (int ps = 0; ps < 4; ++ps) {
            const int r = ps * 32 + warp * 4 + sub;
            const int v = dummy ? -1 : tab_s[tap * BM + r];
            cp_async16(at + h * ATOM_BYTES + swz(r, c8), p.X + (size_t)(v < 0 ? 0 : v) * p.Cin + cb * 64 + c8 * 8, v >= 0);
          }
        }
        cp_async_arrive(&a_full[s]);
      }
    }
    // ---- epilogue: TMEM -> atomics into dWp
    mbar_wait(accum_bar, 0);
    tc_fence_after();
    const int q = warp & 3, half = warp >> 2;
    const int row = q * 32 + lane;                 // row of the pair: atom = row / 64, channel = row % 64
    for (int pr = 0; pr < npairs; ++pr) {
      const int atom = (pair0 + pr) * 2 + (row >> 6);
      const bool ok = atom < natoms;
      const int tap = ok ? atom / cblocks : 0, ci = ok ? (atom % cblocks) * 64 + (row & 63) : 0;
      float* dst = p.dWp + ((size_t)tap * p.Cin + ci) * p.Cout + n0;
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
      uint32_t it = 0;
      for (int ti = 0; ti < ntile; ++ti) {
        const int bs = ti & 1;
        mbar_wait(&b_full[bs], ((uint32_t)ti >> 1) & 1u);
        const uint32_t b_addr = smem_u32(smem + L::B_OFF + bs * L::B_BYTES_);
        for (int pr = 0; pr < npairs; ++pr, ++it) {
          const int s = it % STAGES;
          mbar_wait(&a_full[s], (it / STAGES) & 1u);
          fence_async_smem();
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem + s * L::A_STAGE);
#pragma unroll
          for (int k = 0; k < BM / 16; ++k) {      // 16 pixel rows per MMA = 2048 bytes down the tile
            const uint64_t da = make_desc_mnmajor_sw128(a_addr + k * 2048, ATOM_BYTES);
            const uint64_t db = make_desc_mnmajor_sw128(b_addr + k * 2048, ATOM_BYTES);
            umma_bf16(tmem_base + (uint32_t)(pr * N_BLK), da, db, idesc, (ti | k) != 0);
          }
          umma_commit(&a_empty[s]);
        }
        umma_commit(&b_empty[bs]);
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

template <int N_BLK, int NPAIRS, int STAGES>
int launch(Params p, cudaStream_t st) {
  using L = Smem<N_BLK, NPAIRS, STAGES>;
  auto kern = wgrad_tc_kernel<N_BLK, NPAIRS, STAGES>;
  static PerDeviceFlag configured_on;
  bool& configured = configured_on.here();
  if (!configured) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL) != cudaSuccess) return -3;
    configured = true;
  }
  const int total_pairs = (7 * (p.Cin / 64) + 1) / 2;
  p.units_m = (total_pairs + NPAIRS - 1) / NPAIRS;
  const int units = p.units_m * (p.Cout / N_BLK);
  int slices = (148 + units - 1) / units;
  if (slices > p.total_tiles) slices = p.total_tiles;
  if (slices < 1) slices = 1;
  p.tiles_per_cta = (p.total_tiles + slices - 1) / slices;
  dim3 grid((unsigned)((p.total_tiles + p.tiles_per_cta - 1) / p.tiles_per_cta), (unsigned)units);
  kern<<<grid, THREADS, L::TOTAL, st>>>(p);
  return cudaGetLastError() == cudaSuccess ? 0 : -3;
}
}  // namespace tcw

inline bool tc_wgrad_supported(int Cin, int Cout) { return Cin % 64 == 0 && Cout % 64 == 0 && Cin >= 64 && Cout >= 64; }

inline int launch_wgrad_tc(const int32_t* plan_dev, const GinSide& side, int group, const void* Xb, const void* dYb, float* dWp,
                           int B, int Cin, int Cout, int total_tiles, bool bf16, cudaStream_t st) {
  tcw::Params p;
  p.plan = plan_dev; p.fmt = idesc_fmt_bits(bf16); p.side = side; p.group = group; p.B = B; p.Cin = Cin; p.Cout = Cout;
  p.X = reinterpret_cast<const __nv_bfloat16*>(Xb); p.dY = reinterpret_cast<const __nv_bfloat16*>(dYb); p.dWp = dWp;
  p.total_tiles = total_tiles; p.tiles_per_cta = 1; p.units_m = 1;
  if ((long long)B * side.P_src + 2LL * B >= 0x7fffffffLL) return -4;
  if (Cout % 256 == 0) return tcw::launch<256, 2, 2>(p, st);
  if (Cout % 128 == 0) return tcw::launch<128, 4, 3>(p, st);
  return tcw::launch<64, 7, 4>(p, st);
}

}  // namespace gin
