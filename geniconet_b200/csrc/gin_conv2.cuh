// Patch-mode tcgen05 hex-conv, second generation (forward and the in-chart part of dgrad of stride-1 layers).
//
// What changed against gin_gemm_tcp.cuh, each item with the measurement that drove it (gpurun_out/dbg_matrix*.log,
// profiles/r01b_*):
//   * ONE shared-memory copy of the padded patch instead of three column-shifted ones.  tools/exp/umma_shift_test.cu
//     shows that the SWIZZLE_128B pattern of a UMMA operand is a pure function of the shared-memory ADDRESS (bits 4-6 ^=
//     bits 7-9): a descriptor may start at any 128-byte row and its 8-row groups may be any distance apart (SBO) as long
//     as the data was written with the same address-based XOR.  The patch is stored densely in plan order (row u of the
//     plan's source table = 128 bytes at u*128) and tap (di, dj) is the SAME image read from start row
//     (1+di)*Q*10 + (1+dj) with a group stride of 10 rows.  A stage is <= 30 KB instead of 72 KB.
//   * The MMA issuer loop runs WARP-UNIFORM (role index via shuffle, all 32 lanes in lock step, one elected lane issues):
//     descriptors and counters then live in uniform registers, which is what UTCHMMA takes.  With the loop under
//     `if (lane == 0)` every tcgen05.mma cost five R2UR conversions and the issuing thread, not the tensor pipe, set the pace
//     (~140 clk per MMA against 32 clk of tensor work at N = 64).
//   * Weights stay RESIDENT in shared memory when the [7][K/64] x N_TILE slice fits (<= 112 KB: the 64-wide layers);
//     otherwise they stream through a ring that holds >= 96 KB (2-4 tiles in flight could not cover the L2 latency).
//   * A dedicated TABLE warp resolves the plan's gather tables several tiles ahead into a shared-memory ring.  A global
//     load costs ~1 us on B200; with the table fetched one tile ahead by the producers themselves that latency was paid
//     once per tile (24 of 76 us).
//   * The epilogue transposes through shared memory so that every global store instruction writes whole 256-byte rows
//     (the direct TMEM-lane-per-row stores touched 32 different rows per instruction and bounded the kernel), and the
//     output row of a tile is computed from Q base pixels per tile (kept in shared memory for all tiles), not looked up.
//   * cp.async.cg: the patch is read once, and L1 is only ~20 KB next to 200 KB of shared memory.
//
// Warp roles (608 threads, one CTA per SM, persistent, every CTA keeps one n-block):
//   8 producer warps (cp.async patch gather) | 1 MMA warp | 1 weight warp (cp.async.bulk) | 1 table warp |
//   8 epilogue warps (tcgen05.ld -> smem transpose -> +bias -> coalesced fp32 stores).
// Two TMEM accumulators of N_TILE columns: the epilogue of tile i overlaps the MMAs of tile i+1.
#pragma once
#include <cuda_fp16.h>

#include "gin_gemm_tc.cuh"

namespace gin {
namespace cv2 {
using namespace tc;

constexpr int PROD_WARPS = 8, PROD_THREADS = PROD_WARPS * 32;
constexpr int EPI_WARPS = 8;                 // two per TMEM lane quarter: each takes every other 32-column slab
constexpr int W_MMA = PROD_WARPS, W_WEIGHT = PROD_WARPS + 1, W_TABLE = PROD_WARPS + 2, W_EPI0 = PROD_WARPS + 3;
constexpr int NWARPS = W_EPI0 + EPI_WARPS;
constexpr int NTHREADS = NWARPS * 32;
constexpr int MAX_ITEMS = 8;                 // patch rows per producer thread: ceil(256 / 32)
constexpr int MAX_A_STAGES = 4, MAX_B_STAGES = 8;
constexpr int TAB_SLOTS = 8, TAB_ROWS = 256, TAB_BATCH = 4;
constexpr int STAGE_PITCH = 144;             // epilogue staging: 32 fp32 + 16 bytes of padding per row (conflict-free both ways)
constexpr int STAGE_BYTES = EPI_WARPS * 32 * STAGE_PITCH;
constexpr int SMEM_LIMIT = 227 * 1024;
constexpr int MAX_PLANES = 16;

// Eval-mode BatchNorm in the epilogue (forward-only inference, gin_hexconv_fwd_affine): per output column
//   o = acc*scale[col] + shift[col]  (conv bias folded into shift);  ReLU on columns < relu_split;
//   with res: o = relu(o + R[row][col])  (conv01 of a residual block: relu(bn01(conv01) + bn10(conv10)));
// columns < split go to destination 0, the others to destination 1 (column col - split).  A destination is any combination of
// the 16-bit forward operand copy [B*P + 2B][ld] and an fp32 map [B*P][ld] (ld = its width).  Where an operand copy is written,
// the fp32 values of the ten pole-ring pixels of every sample also go to ring[d] = [B][10][ld]; pole_mean_kernel then forms the
// pole-mean rows from them exactly as cast_bf16_kernel would from the fp32 output.
struct Affine {
  const float* scale;
  const float* shift;
  int relu_split;
  const void* res;            // may be null; fp32, or fp16 when res_f16
  long long res_ld;
  int res_f16;
  int split;                  // N when there is one destination
  void* op[2];                // 16-bit operand copies (forward format: op_f16)
  float* f32[2];
  float* ring[2];
  int ld[2];
  int op_f16;
};

// A tile is processed as `nplanes` segments.  Each segment stages ONE image (its own source table) per 64-channel chunk and
// applies its own short tap list to it.  Stride 1: one segment with all seven taps.  Stride-2 forward: four parity planes of
// the fine input, 1-2 taps each, all accumulated into one output tile.  Stride-2 dgrad: the four parity classes of the fine
// output, each its own output tile (flush_each) gathered from the same coarse dy image.  (gin_plan.h: GinPSide / GinP2Side.)
struct Params {
  const int32_t* plan;
  uint32_t fmt;               // operand-format bits of the instruction descriptor (gin_common.cuh: idesc_fmt_bits)
  int U, Q, ntiles;           // patch rows per image, octets per patch row, tiles per sample group
  int group, B, K, N;
  int P_src, P_dst;           // pixels per sample of the gathered / written map
  const __nv_bfloat16* X;     // [B*P_src + 2B][K] bf16 (pixels, then pole-mean rows)
  const __nv_bfloat16* Wt;    // pre-swizzled bf16 tiles [7][K/64][N][64]
  const float* bias;
  const float* bias1;         // optional: columns >= bias_split take bias1[col - bias_split] (two sibling convolutions as one GEMM)
  int bias_split;
  float* Y;                   // [B*P_dst][N] fp32, or fp16 when y_f16 (forward outputs that only a BatchNorm reads: half the bytes)
  int y_f16;
  float* stats;               // optional [gridDim.x / n_blocks][2][N]: per-CTA column sums of y and y^2 (BatchNorm statistics)
  int nplanes, flush_each;    // nplanes <= MAX_PLANES
  int group_bytes;            // distance between the 8-row groups of a tile inside the image: 1280 (patch) or 1024 (gathered rows)
  int accumulate;             // epilogue adds into Y (read-modify-write; every destination pixel belongs to one tile row only)
  int dst_tab_off;            // >= 0: destination pixel of tile row r = plan[dst_tab_off + t*128 + r] (-1: none) instead of base + arithmetic
  int ntaps[MAX_PLANES];
  int8_t tap_id[MAX_PLANES][8];    // weight index of each tap of a segment
  int16_t tap_row[MAX_PLANES][8];  // its start row inside the image
  int tab_off, tab_tstride, tab_pstride;      // source table of (tile t, segment pl): plan[tab_off + t*tab_tstride + pl*tab_pstride ...]
  int base_off, base_tstride, base_qstride;   // first destination pixel of octet column q of tile t
  int dst_row_stride, dst_px_stride, dst_plane_off[MAX_PLANES];
  int total_tiles, n_blocks;  // CTA c owns n-block c % n_blocks and tiles c / n_blocks + k * (gridDim.x / n_blocks)
  int a_stage_bytes, a_stages, b_stages, resident;
  int cl;                     // CTAs per cluster (1, 2 or 4): > 1 only with streamed weights
  // Second tile class (SEAM kernels: dgrad in one launch, gin_plan.h GinPfSide): x_total boundary tiles in regular form --
  // x_nslots segments of 128 gathered rows with one tap each, destination pixels from a table -- appended to the tile list after
  // the total_tiles patch tiles.  mask_off >= 0: plan words [ntiles][nflush][4], bit r set = the patch tile does not store row r.
  int x_total, x_ntiles, x_nslots, x_src_off, x_dst_off, mask_off, x_all;   // x_all: no patch tiles at all (every pixel is a boundary-form row)
  int8_t x_tap[MAX_PLANES];
  int* stats_parts;           // host: receives the number of per-CTA statistics rows written (0: none)
  int dbg;                    // GIN_DBG bit mask (experiments only): 1 no epilogue stores, 2 no patch loads, 4 no MMAs
  Affine aff;                 // eval-mode BatchNorm epilogue (aff.scale != null: the AFFINE instantiations; bias / Y / stats unused)
};

constexpr int kDi[7] = {0, -1, 1, 0, 0, -1, 1};
constexpr int kDj[7] = {0, 0, 0, -1, 1, 1, -1};

GIN_DEVINL uint64_t desc_kmajor(uint32_t smem_addr, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(sbo_bytes >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;                         // SWIZZLE_128B, base offset 0 (address-based pattern)
  return d;
}

// ---- thread-block clusters: the CTAs of a cluster (p.cl = 2 or 4) work on consecutive tiles of the same class in lock step and
// SHARE the weight stream: every CTA fetches 1/cl of each weight tile and multicasts it into the shared memory of all of them,
// so a weight tile crosses the L2 -> SM fabric once per cluster instead of once per CTA (that stream, ~10 TB/s aggregate, is what
// bounded the streamed-weight layers: profiles/r01_bottleneck_matrix_v2_kernel.log, profiles/r02_ncu_conv_kernels.txt).
GIN_DEVINL uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
GIN_DEVINL void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// bulk copy whose bytes (and mbarrier completion) land at the same shared-memory offsets in every CTA of `mask`
GIN_DEVINL void bulk_g2s_mc(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar, uint16_t mask) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(dst_smem)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar)), "h"(mask)
               : "memory");
}
// tcgen05.commit arriving on the barrier at this offset in every CTA of `mask`
GIN_DEVINL void umma_commit_mc(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)), "h"(mask)
               : "memory");
}

// barrier block: a_full[4] a_empty[4] b_full[8] b_empty[8] acc_full[2] acc_empty[2] tab_full[8] tab_empty[8] | tmem slot
constexpr int NBARS = 2 * MAX_A_STAGES + 2 * MAX_B_STAGES + 4 + 2 * TAB_SLOTS;
constexpr int BAR_BYTES = NBARS * 8 + 16;

// -DGIN_PROF: per-role cycle counters (time blocked on each barrier, time per phase) printed by CTA 0; diagnostics only
#ifdef GIN_PROF
#define PROF_T0() const long long _t0 = clock64()
#define PROF_ADD(acc) (acc) += clock64() - _t0
#else
#define PROF_T0()
#define PROF_ADD(acc)
#endif

// store of one 4-column group by the affine epilogue; ri = ring slot (sample*10 + pole*5 + e) of the row, or -1
GIN_DEVINL void affine_store(const Affine& a, int d, int gd, int ri, int dcol, float4 o) {
  const size_t off = (size_t)gd * a.ld[d] + dcol;
  if (a.f32[d]) *reinterpret_cast<float4*>(a.f32[d] + off) = o;
  if (a.op[d]) {
    *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(a.op[d]) + off) = make_uint2(pack2_op(o.x, o.y, a.op_f16), pack2_op(o.z, o.w, a.op_f16));
    if (ri >= 0) *reinterpret_cast<float4*>(a.ring[d] + (size_t)ri * a.ld[d] + dcol) = o;
  }
}

template <int N_TILE, bool RESIDENT, bool STATS, bool SEAM, bool AFFINE = false>
__global__ void __launch_bounds__(NTHREADS, 1) patch_conv_kernel(const Params p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  constexpr int B_TILE = N_TILE * 128;
  const int kchunks = p.K / BK;
  const int b_tiles = RESIDENT ? 7 * kchunks : p.b_stages;
  uint8_t* a_smem = smem;
  uint8_t* b_smem = smem + p.a_stages * p.a_stage_bytes;
  uint8_t* stage_smem = b_smem + (size_t)b_tiles * B_TILE;
  int32_t* tab = reinterpret_cast<int32_t*>(stage_smem + STAGE_BYTES);           // [TAB_SLOTS][TAB_ROWS] resolved source rows
  uint64_t* bars = reinterpret_cast<uint64_t*>(tab + TAB_SLOTS * TAB_ROWS);
  uint64_t* a_full = bars;
  uint64_t* a_empty = a_full + MAX_A_STAGES;
  uint64_t* b_full = a_empty + MAX_A_STAGES;
  uint64_t* b_empty = b_full + MAX_B_STAGES;
  uint64_t* acc_full = b_empty + MAX_B_STAGES;
  uint64_t* acc_empty = acc_full + 2;
  uint64_t* tab_full = acc_empty + 2;
  uint64_t* tab_empty = tab_full + TAB_SLOTS;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tab_empty + TAB_SLOTS);
  int32_t* tile_base = reinterpret_cast<int32_t*>(reinterpret_cast<uint8_t*>(bars) + BAR_BYTES);   // [ntiles][Q] first pixel of each octet column

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);      // warp-UNIFORM role index: keeps the issuer loops in uniform registers
  const int U = p.U, Q = p.Q, NP = p.nplanes;
  const int AS = p.a_stages, BS = p.b_stages;
  constexpr uint32_t TM_COLS = (2 * N_TILE <= 32) ? 32 : 2 * N_TILE;
  // Tiles are handed out in GROUPS of CL consecutive tiles of one class (CL = cluster size; 1: a group is a tile): cluster c keeps
  // n-block c % n_blocks and the groups c / n_blocks + k * (clusters / n_blocks); its CTA of rank r takes tile r of each group (a
  // "ghost" -- all rows zero, nothing stored -- where a class does not fill its last group).  Groups >= groups0 are boundary tiles.
  const int CL = RESIDENT ? 1 : p.cl;
  const int crank = CL > 1 ? (int)cluster_ctarank() : 0;
  const uint16_t cmask = (uint16_t)((1u << CL) - 1u);
  const int cid = blockIdx.x / CL;
  const int nb = cid % p.n_blocks, n0 = nb * N_TILE;
  const int q_first = cid / p.n_blocks, q_step = (gridDim.x / CL) / p.n_blocks;
  const int groups0 = (p.total_tiles + CL - 1) / CL;
  const int NG = groups0 + (SEAM ? (p.x_total + CL - 1) / CL : 0);

  if (warp == W_MMA) {
    if (lane == 0) {
      for (int s = 0; s < MAX_A_STAGES; ++s) { mbar_init(&a_full[s], PROD_THREADS); mbar_init(&a_empty[s], 1); }
      for (int s = 0; s < MAX_B_STAGES; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], CL); }   // a slot is free once EVERY CTA of the cluster has used it
      for (int s = 0; s < 2; ++s) { mbar_init(&acc_full[s], 1); mbar_init(&acc_empty[s], EPI_WARPS * 32); }
      for (int s = 0; s < TAB_SLOTS; ++s) { mbar_init(&tab_full[s], 1); mbar_init(&tab_empty[s], PROD_THREADS); }
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc(tmem_slot, TM_COLS);
  }
  if (p.dst_tab_off < 0)
    for (int i = tid; i < p.ntiles * Q; i += NTHREADS)
      tile_base[i] = __ldg(p.plan + p.base_off + (i / Q) * p.base_tstride + (i % Q) * p.base_qstride);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (CL > 1) cluster_sync_all();                    // every CTA's barriers exist before a peer multicasts into them
  const uint32_t tmem_base = *tmem_slot;
  GIN_PDL_SYNC();                                    // everything above touched only shared memory, TMEM and the constant plan
#ifdef GIN_PROF
  long long pw[6] = {0, 0, 0, 0, 0, 0};
  const long long t_begin = clock64();
#endif

  if (warp < PROD_WARPS) {
    // =========================================================== producers: asynchronous patch gather (one copy)
    const int sub = lane >> 3, c8 = lane & 7;
    const __nv_bfloat16* __restrict__ Xc = p.X + c8 * 8;
    int s = 0, ts = 0;
    uint32_t ph = 0, tph = 0;
    for (int g = q_first; g < NG; g += q_step) {
      const bool sx = SEAM && g >= groups0;
      const int NPt = sx ? p.x_nslots : NP, Ut = sx ? BM : U;
      for (int pl = 0; pl < NPt; ++pl) {
        int v[MAX_ITEMS];
        { PROF_T0(); mbar_wait(&tab_full[ts], tph); PROF_ADD(pw[0]); }
#pragma unroll
        for (int it = 0; it < MAX_ITEMS; ++it) v[it] = tab[ts * TAB_ROWS + it * 32 + warp * 4 + sub];
        mbar_arrive(&tab_empty[ts]);                   // the row ids are in registers now
        if (++ts == TAB_SLOTS) { ts = 0; tph ^= 1u; }
        for (int kc = 0; kc < kchunks; ++kc) {
          { PROF_T0(); mbar_wait(&a_empty[s], ph ^ 1u); PROF_ADD(pw[1]); }
          const uint32_t st = smem_u32(a_smem + s * p.a_stage_bytes);
#pragma unroll
          for (int it = 0; it < MAX_ITEMS; ++it) {
            const int u = it * 32 + warp * 4 + sub;
            if (u < Ut && !(p.dbg & 2)) {
              const bool ok = v[it] >= 0;
              cp_async16_cg(st + swz(u, c8), Xc + (size_t)(ok ? v[it] : 0) * p.K + kc * BK, ok);
            }
          }
          cp_async_arrive(&a_full[s]);
          if (++s == AS) { s = 0; ph ^= 1u; }
        }
      }
    }
#ifdef GIN_PROF
    if (blockIdx.x == 0 && tid == 0) printf("producer: total %lld wait_tab %lld wait_a_empty %lld\n", clock64() - t_begin, pw[0], pw[1]);
#endif
  } else if (warp == W_MMA) {
    // =========================================================== MMA issuer
    // The whole warp runs this loop in lock step (addresses, descriptors and counters stay in uniform registers);
    // only the elected lane issues tcgen05.mma / tcgen05.commit.
    const uint32_t idesc = make_idesc_f16kind(N_TILE) | p.fmt;
    const bool leader = elect_one();
    int s = 0, bs = 0;
    uint32_t ph = 0, bph = 0, wc = 0;
    if (RESIDENT) mbar_wait(&b_full[0], 0);          // the whole weight slice, loaded once
    // The tensor pipe only holds a few MMAs in its queue: whenever this warp stops issuing for longer than they take (an
    // mbarrier try_wait alone is 60-90 clk, a proxy fence more) the pipe runs dry.  So just before the LAST tap group of a chunk
    // is issued -- while the earlier tap groups still execute -- the barriers that open the NEXT chunk are tested WITHOUT
    // blocking (its a_full + proxy fence, and the accumulator hand-back when it starts a new output); whatever is already
    // complete then costs nothing at the chunk boundary.
    bool a_ready = false, acc_ready = false;
    for (int g = q_first; g < NG; g += q_step) {
      const bool sx = SEAM && g >= groups0;
      const int NPt = sx ? p.x_nslots : NP;
      const uint32_t gbytes = sx ? 1024u : (uint32_t)p.group_bytes;
      uint32_t fresh = 1;                            // the next MMA starts a new accumulation
      for (int pl = 0; pl < NPt; ++pl) {
        const uint32_t ab = wc & 1;
        if (fresh && !acc_ready) {
          PROF_T0();
          mbar_wait(&acc_empty[ab], ((wc >> 1) & 1u) ^ 1u);
          PROF_ADD(pw[0]);
          tc_fence_after();
        }
        acc_ready = false;
        const uint32_t d_tmem = tmem_base + ab * N_TILE;
        const int nt = sx ? 1 : p.ntaps[pl];
        const bool flush = sx ? pl == NPt - 1 : (p.flush_each || pl == NP - 1);
        for (int kc = 0; kc < kchunks; ++kc) {
          if (!a_ready) {
            { PROF_T0(); mbar_wait(&a_full[s], ph); PROF_ADD(pw[1]); }
            { PROF_T0(); fence_async_smem(); tc_fence_after(); PROF_ADD(pw[3]); }
          }
          a_ready = false;
          const uint32_t a_addr = smem_u32(a_smem + s * p.a_stage_bytes);
          const bool last_chunk_of_cta = kc == kchunks - 1 && pl == NPt - 1 && g + q_step >= NG;
          for (int j = 0; j < nt; ++j) {
            if (j == nt - 1 && !last_chunk_of_cta) {  // open the next chunk while the earlier tap groups execute
              const int sn = (s + 1 == AS) ? 0 : s + 1;
              const uint32_t phn = (s + 1 == AS) ? ph ^ 1u : ph;
              if (mbar_test(&a_full[sn], phn)) {
                PROF_T0(); fence_async_smem(); tc_fence_after(); PROF_ADD(pw[3]);
                a_ready = true;
              }
              if (kc == kchunks - 1 && flush) {       // ... and it starts a new output tile: is its accumulator back already?
                const uint32_t wn = wc + 1;
                if (mbar_test(&acc_empty[wn & 1], ((wn >> 1) & 1u) ^ 1u)) {
                  tc_fence_after();
                  acc_ready = true;
                }
              }
            }
            const int tap = sx ? p.x_tap[pl] : p.tap_id[pl][j];
            const uint32_t trow = sx ? 0u : (uint32_t)p.tap_row[pl][j];
            uint32_t b_addr;
            if (RESIDENT) b_addr = smem_u32(b_smem + (size_t)(tap * kchunks + kc) * B_TILE);
            else {
              { PROF_T0(); mbar_wait(&b_full[bs], bph); PROF_ADD(pw[2]); }
              tc_fence_after();
              b_addr = smem_u32(b_smem + (size_t)bs * B_TILE);
            }
            const uint64_t da = desc_kmajor(a_addr + trow * 128u, gbytes), db = desc_kmajor(b_addr, 1024);
            {
              PROF_T0();
#pragma unroll
              for (int k = 0; k < BK / 16; ++k) {
                if (leader && !(p.dbg & 4)) umma_bf16(d_tmem, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc, fresh ^ 1u);
                fresh = 0;
              }
              PROF_ADD(pw[4]);
            }
            if (!RESIDENT) {
              if (leader) { if (CL > 1) umma_commit_mc(&b_empty[bs], cmask); else umma_commit(&b_empty[bs]); }
              if (++bs == BS) { bs = 0; bph ^= 1u; }
            }
          }
          { PROF_T0(); if (leader) umma_commit(&a_empty[s]); __syncwarp(); PROF_ADD(pw[5]); }
          if (++s == AS) { s = 0; ph ^= 1u; }
        }
        if (flush) {
          if (leader) umma_commit(&acc_full[ab]);
          __syncwarp();
          ++wc;
          fresh = 1;
        }
      }
    }
#ifdef GIN_PROF
    if (blockIdx.x == 0 && lane == 0)
      printf("mma: total %lld wait_acc_empty %lld wait_a_full %lld wait_b_full %lld fences %lld issue %lld commit %lld\n", clock64() - t_begin, pw[0], pw[1],
             pw[2], pw[3], pw[4], pw[5]);
#endif
  } else if (warp == W_WEIGHT) {
    // =========================================================== weight tiles
    if (lane == 0) {
      if (RESIDENT) {
        mbar_arrive_expect_tx(&b_full[0], (uint32_t)(7 * kchunks * B_TILE));
        for (int i = 0; i < 7 * kchunks; ++i)        // i = tap * kchunks + kc
          bulk_g2s(b_smem + (size_t)i * B_TILE, p.Wt + ((size_t)i * p.N + n0) * BK, B_TILE, &b_full[0]);
      } else {
        int bs = 0;
        uint32_t bph = 0;
        const uint32_t part = (uint32_t)B_TILE / (uint32_t)CL;      // this CTA's share of every weight tile
        for (int g = q_first; g < NG; g += q_step) {
          const bool sx = SEAM && g >= groups0;
          const int NPt = sx ? p.x_nslots : NP;
          for (int pl = 0; pl < NPt; ++pl)
            for (int kc = 0; kc < kchunks; ++kc)
              for (int j = 0; j < (sx ? 1 : p.ntaps[pl]); ++j) {
                const int tap = sx ? p.x_tap[pl] : p.tap_id[pl][j];
                mbar_wait(&b_empty[bs], bph ^ 1u);            // completed by the MMA commits of all CL CTAs
                mbar_arrive_expect_tx(&b_full[bs], B_TILE);   // the whole tile: this CTA's share + the shares multicast by its peers
                const uint8_t* src = reinterpret_cast<const uint8_t*>(p.Wt + (((size_t)tap * kchunks + kc) * p.N + n0) * BK);
                if (CL > 1) bulk_g2s_mc(b_smem + (size_t)bs * B_TILE + crank * part, src + crank * part, part, &b_full[bs], cmask);
                else bulk_g2s(b_smem + (size_t)bs * B_TILE, src, B_TILE, &b_full[bs]);
                if (++bs == BS) { bs = 0; bph ^= 1u; }
              }
        }
      }
    }
    __syncwarp();
  } else if (warp == W_TABLE) {
    // =========================================================== gather tables, resolved TAB_BATCH segments at a time, up to 8 ahead
    const long long total_src = (long long)p.B * p.P_src;
    int ts = 0;
    uint32_t tph = 0;
    int gn = q_first, pn = 0;                        // the next (group, segment) in the producers' order
    while (gn < NG) {
      int code[TAB_BATCH][MAX_ITEMS], grp[TAB_BATCH], sgrp[TAB_BATCH];      // sgrp: sample group of the tile, -1 for a ghost
#pragma unroll
      for (int j = 0; j < TAB_BATCH; ++j) {
        grp[j] = -1;
        if (gn < NG) {
          grp[j] = gn;
          const bool sx = SEAM && gn >= groups0;
          const int loc = (sx ? gn - groups0 : gn) * CL + crank, per = sx ? p.x_ntiles : p.ntiles;
          const bool ghost = loc >= (sx ? p.x_total : p.total_tiles);
          sgrp[j] = ghost ? -1 : loc / per;
          const int32_t* __restrict__ src_tab =
              sx ? p.plan + p.x_src_off + ((size_t)(loc % per) * p.x_nslots + pn) * BM
                 : p.plan + p.tab_off + (size_t)(loc % per) * p.tab_tstride + (size_t)pn * p.tab_pstride;
          const int Ut = (sx ? BM : U);
#pragma unroll
          for (int it = 0; it < MAX_ITEMS; ++it) {
            const int u = it * 32 + lane;
            code[j][it] = (u < Ut && !ghost) ? __ldg(src_tab + u) : GIN_SRC_ZERO;
          }
          if (++pn == (sx ? p.x_nslots : NP)) { pn = 0; gn += q_step; }
        }
      }
#pragma unroll
      for (int j = 0; j < TAB_BATCH; ++j) {
        if (grp[j] >= 0) {
          const int G = sgrp[j] < 0 ? 0 : sgrp[j];
          const long long base = (long long)G * p.group * p.P_src;
          mbar_wait(&tab_empty[ts], tph ^ 1u);
#pragma unroll
          for (int it = 0; it < MAX_ITEMS; ++it)
            tab[ts * TAB_ROWS + it * 32 + lane] = resolve_row(code[j][it], base, total_src, G * p.group, p.B);
          __syncwarp();
          if (lane == 0) mbar_arrive(&tab_full[ts]);
          if (++ts == TAB_SLOTS) { ts = 0; tph ^= 1u; }
        }
      }
    }
  } else {
    // =========================================================== epilogue: TMEM -> smem transpose -> coalesced global stores
    const int e = warp - W_EPI0;
    const int q = warp & 3;                           // TMEM lane quarter this warp may touch
    const int hslab = e >> 2;                         // which of the two warps of this quarter: takes 32-column slabs hslab, hslab+2, ...
    const int row = q * 32 + lane;                    // tile row of this thread: group g = row / 8 = r * Q + oq, pixel px = row % 8
    const int g = row >> 3, r_in = g / Q, oq = g - r_in * Q;
    const int row_off = r_in * p.dst_row_stride + (row & 7) * p.dst_px_stride;
    uint8_t* my_stage = stage_smem + (size_t)e * 32 * STAGE_PITCH;
    const int rsub = lane >> 3, c4 = (lane & 7) * 4;  // store phase: one instruction = four whole 128-byte row segments
    const long long total_pix = (long long)p.B * p.P_dst;
    uint32_t wc = 0;
    const int nflush = p.flush_each ? NP : 1;
    constexpr int NS = N_TILE / 64;                   // 32-column slabs this warp handles
    float ssum[STATS ? NS : 1][4], ssq[STATS ? NS : 1][4];
#pragma unroll
    for (int si = 0; si < (STATS ? NS : 1); ++si)
#pragma unroll
      for (int k = 0; k < 4; ++k) { ssum[si][k] = 0.f; ssq[si][k] = 0.f; }
    for (int g0 = q_first; g0 < NG; g0 += q_step) {
    const bool sx = SEAM && g0 >= groups0;
    const bool tabdst = sx || p.dst_tab_off >= 0;   // destination pixels from a table (boundary tiles / the stand-alone seam form)
    const int Tl = (sx ? g0 - groups0 : g0) * CL + crank, per = sx ? p.x_ntiles : p.ntiles;
    const bool ghost = Tl >= (sx ? p.x_total : p.total_tiles);
    for (int fl = 0; fl < (sx ? 1 : nflush); ++fl, ++wc) {
      const int G = Tl / per, t = Tl - G * per;
      long long gdl;
      bool extra_row = false;
      if (ghost) gdl = total_pix;                    // a ghost tile stores nothing
      else if (tabdst) {
        const int dr = __ldg(p.plan + (sx ? p.x_dst_off : p.dst_tab_off) + t * BM + row);
        extra_row = dr == -3;                         // a further row of the pixel above (same 32-row group): folded in below
        gdl = dr >= 0 ? (long long)G * p.group * p.P_dst + dr : total_pix;
      } else {
        gdl = (long long)G * p.group * p.P_dst + tile_base[t * Q + oq] + row_off + p.dst_plane_off[fl];
        if (SEAM && p.mask_off >= 0) {                // boundary pixels are written by the boundary tiles
          const uint32_t mw = (uint32_t)__ldg(p.plan + p.mask_off + (t * nflush + fl) * 4 + q);
          if ((mw >> lane) & 1u) gdl = total_pix;
        }
      }
      const int gd = extra_row ? -3 : (gdl < total_pix ? (int)gdl : -1);       // B*P < 2^31 is checked by the launcher
      int ri = -1;                                    // AFFINE: ring slot of this row (gin_bn.cuh ring_pixel: first / last pixel of a chart)
      if (AFFINE && gd >= 0) {
        const int sample = gd / p.P_dst, pix = gd - sample * p.P_dst, A = p.P_dst / 5, e = pix / A, li = pix - e * A;
        ri = li == 0 ? sample * 10 + e : li == A - 1 ? sample * 10 + 5 + e : -1;
      }
      const uint32_t ab = wc & 1;
      { PROF_T0(); mbar_wait(&acc_full[ab], (wc >> 1) & 1u); PROF_ADD(pw[0]); }
      tc_fence_after();
#pragma unroll
      for (int si = 0; si < NS; ++si) {
        const int slab = hslab * 32 + si * 64;
        uint32_t v[32];
        { PROF_T0();
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ab * N_TILE + slab), v);
        tmem_ld_wait();
        PROF_ADD(pw[1]); }
        float4* dst = reinterpret_cast<float4*>(my_stage + lane * STAGE_PITCH);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          dst[j] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
        if (slab + 64 >= N_TILE) {                    // this warp has read its last columns of the accumulator
          tc_fence_before();
          mbar_arrive(&acc_empty[ab]);
        }
        __syncwarp();
        if (AFFINE) {
          const int col = n0 + slab + c4;
          const float4 sc = __ldg(reinterpret_cast<const float4*>(p.aff.scale + col)), sh = __ldg(reinterpret_cast<const float4*>(p.aff.shift + col));
          const bool relu = col < p.aff.relu_split;
          const int d = col >= p.aff.split ? 1 : 0, dcol = col - (d ? p.aff.split : 0);
          // the residual rows of four stores are loaded before any of them is written: the compiler cannot move a load across a
          // store through another pointer, and one load latency per store bounded the residual launches
#pragma unroll
          for (int i0 = 0; i0 < 8; i0 += 4) {
            float4 r[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int gd2 = __shfl_sync(0xffffffffu, gd, 4 * (i0 + k) + rsub);
              r[k] = make_float4(0.f, 0.f, 0.f, 0.f);
              if (p.aff.res && gd2 >= 0) {
                if (p.aff.res_f16) {
                  const uint2 u = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const __half*>(p.aff.res) + (size_t)gd2 * p.aff.res_ld + col));
                  const float2 lo = __half22float2(*reinterpret_cast<const __half2*>(&u.x)), hi = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
                  r[k] = make_float4(lo.x, lo.y, hi.x, hi.y);
                } else r[k] = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.aff.res) + (size_t)gd2 * p.aff.res_ld + col));
              }
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int r2 = 4 * (i0 + k) + rsub;
              const int gd2 = __shfl_sync(0xffffffffu, gd, r2), ri2 = __shfl_sync(0xffffffffu, ri, r2);
              const float4 a = *reinterpret_cast<const float4*>(my_stage + r2 * STAGE_PITCH + c4 * 4);
              float4 o = make_float4(fmaf(a.x, sc.x, sh.x), fmaf(a.y, sc.y, sh.y), fmaf(a.z, sc.z, sh.z), fmaf(a.w, sc.w, sh.w));
              if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
              if (p.aff.res) {
                o.x = fmaxf(o.x + r[k].x, 0.f); o.y = fmaxf(o.y + r[k].y, 0.f); o.z = fmaxf(o.z + r[k].z, 0.f); o.w = fmaxf(o.w + r[k].w, 0.f);
              }
              if (gd2 >= 0) affine_store(p.aff, d, gd2, ri2, dcol, o);
            }
          }
          __syncwarp();
          continue;
        }
        float4 bb = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.bias) {
          const int col = n0 + slab + c4;
          bb = __ldg(reinterpret_cast<const float4*>((p.bias1 && col >= p.bias_split) ? p.bias1 + (col - p.bias_split) : p.bias + col));
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int r2 = 4 * i + rsub;
          const int gd2 = __shfl_sync(0xffffffffu, gd, r2);
          float4 o = *reinterpret_cast<const float4*>(my_stage + r2 * STAGE_PITCH + c4 * 4);
          o.x += bb.x; o.y += bb.y; o.z += bb.z; o.w += bb.w;
          if (tabdst) {                                   // table form: up to two extra rows below belong to this pixel
            const int x1 = __shfl_sync(0xffffffffu, gd, (r2 + 1) & 31), x2 = __shfl_sync(0xffffffffu, gd, (r2 + 2) & 31);
            if (r2 + 1 < 32 && x1 == -3) {
              const float4 u = *reinterpret_cast<const float4*>(my_stage + (r2 + 1) * STAGE_PITCH + c4 * 4);
              o.x += u.x; o.y += u.y; o.z += u.z; o.w += u.w;
              if (r2 + 2 < 32 && x2 == -3) {
                const float4 w2 = *reinterpret_cast<const float4*>(my_stage + (r2 + 2) * STAGE_PITCH + c4 * 4);
                o.x += w2.x; o.y += w2.y; o.z += w2.z; o.w += w2.w;
              }
            }
          }
          if (p.accumulate && gd2 >= 0) {
            const float4 old = *reinterpret_cast<const float4*>(p.Y + (size_t)gd2 * p.N + n0 + slab + c4);
            o.x += old.x; o.y += old.y; o.z += old.z; o.w += old.w;
          }
          if (gd2 >= 0 && !(p.dbg & 1)) {
            if (p.y_f16) *reinterpret_cast<uint2*>(reinterpret_cast<__half*>(p.Y) + (size_t)gd2 * p.N + n0 + slab + c4) = make_uint2(pack2_f16(o.x, o.y), pack2_f16(o.z, o.w));
            else *reinterpret_cast<float4*>(p.Y + (size_t)gd2 * p.N + n0 + slab + c4) = o;
          }
          if (STATS && gd2 >= 0) {
            ssum[si][0] += o.x; ssum[si][1] += o.y; ssum[si][2] += o.z; ssum[si][3] += o.w;
            ssq[si][0] = fmaf(o.x, o.x, ssq[si][0]); ssq[si][1] = fmaf(o.y, o.y, ssq[si][1]);
            ssq[si][2] = fmaf(o.z, o.z, ssq[si][2]); ssq[si][3] = fmaf(o.w, o.w, ssq[si][3]);
          }
        }
        __syncwarp();
      }
    }
    }
    if (STATS) {
      // column sums of this CTA's rows: lanes that share (lane & 7) hold the same columns; the four TMEM-quarter warps of a
      // slab set meet in shared memory (the staging area is free now); one plain store per column, no global atomics
      float* sred = reinterpret_cast<float*>(stage_smem);              // [4 quarters][2][N_TILE]
      // one slot per (TMEM quarter, column): every slot is written exactly once, the four quarters are then added in a fixed
      // order -- no atomics, so the statistics (and everything downstream of them) are reproducible run to run
      asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
#pragma unroll
      for (int si = 0; si < NS; ++si)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          float a = ssum[si][k], b = ssq[si][k];
          a += __shfl_xor_sync(0xffffffffu, a, 8); a += __shfl_xor_sync(0xffffffffu, a, 16);
          b += __shfl_xor_sync(0xffffffffu, b, 8); b += __shfl_xor_sync(0xffffffffu, b, 16);
          if (lane < 8) {
            const int col = hslab * 32 + si * 64 + c4 + k;
            sred[(q * 2) * N_TILE + col] = a;
            sred[(q * 2 + 1) * N_TILE + col] = b;
          }
        }
      asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
      float* out = p.stats + (size_t)((cid / p.n_blocks) * CL + crank) * 2 * p.N + n0;
      for (int i = (warp - W_EPI0) * 32 + lane; i < 2 * N_TILE; i += EPI_WARPS * 32)
        out[(i / N_TILE) * p.N + (i % N_TILE)] = (sred[i] + sred[2 * N_TILE + i]) + (sred[4 * N_TILE + i] + sred[6 * N_TILE + i]);
    }
#ifdef GIN_PROF
    if (blockIdx.x == 0 && lane == 0 && e == 0) printf("epilogue: total %lld wait_acc_full %lld tmem_ld %lld tiles %u\n", clock64() - t_begin, pw[0], pw[1], wc);
#endif
  }
  tc_fence_before();
  __syncthreads();
  if (CL > 1) cluster_sync_all();                    // no CTA leaves while a peer may still multicast into it / arrive on its barriers
  if (warp == W_MMA) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TM_COLS);
  }
}

// shared-memory plan for one launch; returns false when nothing fits
inline bool plan_smem(int n_tile, int K, int U, int ntiles, int Q, Params& p, int& total) {
  const int b_tile = n_tile * 128, kchunks = K / 64;
  p.a_stage_bytes = ((U * 128 + 1023) / 1024) * 1024;
  const int fixed = STAGE_BYTES + TAB_SLOTS * TAB_ROWS * 4 + BAR_BYTES + ntiles * Q * 4 + 16;
  const int budget = SMEM_LIMIT - 1024 - fixed;
  const int resident_bytes = 7 * kchunks * b_tile;
  p.resident = resident_bytes <= 114688 && resident_bytes + 2 * p.a_stage_bytes <= budget;
  int b_bytes;
  if (p.resident) { p.b_stages = 1; b_bytes = resident_bytes; }
  else {
    p.b_stages = 98304 / b_tile;                    // >= 96 KB of weights in flight
    if (p.b_stages > MAX_B_STAGES) p.b_stages = MAX_B_STAGES;
    if (p.b_stages < 2) p.b_stages = 2;
    b_bytes = p.b_stages * b_tile;
  }
  p.a_stages = (budget - b_bytes) / p.a_stage_bytes;
  if (p.a_stages > MAX_A_STAGES) p.a_stages = MAX_A_STAGES;
  if (p.a_stages < 2) return false;
  total = p.a_stages * p.a_stage_bytes + b_bytes + fixed + 1024;
  return true;
}

constexpr int B_TILE_OF(int n_tile) { return n_tile * 128; }

template <int N_TILE>
int launch(Params p, cudaStream_t st) {
  int smem_total = 0;
  if (!plan_smem(N_TILE, p.K, p.U, p.ntiles, p.Q, p, smem_total)) return -4;
  static PerDeviceFlag configured_on;
  bool& configured = configured_on.here();
  if (!configured) {
    if (cudaFuncSetAttribute(patch_conv_kernel<N_TILE, true, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT) != cudaSuccess ||
        cudaFuncSetAttribute(patch_conv_kernel<N_TILE, false, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT) != cudaSuccess ||
        cudaFuncSetAttribute(patch_conv_kernel<N_TILE, true, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT) != cudaSuccess ||
        cudaFuncSetAttribute(patch_conv_kernel<N_TILE, false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT) != cudaSuccess ||
        cudaFuncSetAttribute(patch_conv_kernel<N_TILE, true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT) != cudaSuccess ||
        cudaFuncSetAttribute(patch_conv_kernel<N_TILE, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT) != cudaSuccess ||
        cudaFuncSetAttribute(patch_conv_kernel<N_TILE, true, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT) != cudaSuccess ||
        cudaFuncSetAttribute(patch_conv_kernel<N_TILE, false, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT) != cudaSuccess) return -3;
    configured = true;
  }
  p.n_blocks = p.N / N_TILE;
  const bool seam = p.x_total > 0;
  const bool affine = p.aff.scale != nullptr;        // the launcher of the affine form allows no seam tiles, statistics or accumulation
  const bool stats = p.stats != nullptr && !p.flush_each && !seam && !affine;
  const int sms = num_sms();
  void (*kern)(const Params);
  if (affine) kern = p.resident ? patch_conv_kernel<N_TILE, true, false, false, true> : patch_conv_kernel<N_TILE, false, false, false, true>;
  else if (seam) kern = p.resident ? patch_conv_kernel<N_TILE, true, false, true> : patch_conv_kernel<N_TILE, false, false, true>;
  else if (p.resident) kern = stats ? patch_conv_kernel<N_TILE, true, true, false> : patch_conv_kernel<N_TILE, true, false, false>;
  else kern = stats ? patch_conv_kernel<N_TILE, false, true, false> : patch_conv_kernel<N_TILE, false, false, false>;
  // Streamed weights: clusters of CL CTAs share the weight stream (GIN_CLUSTER = 1 switches it off, 4 asks for clusters of four).
  int CL = 1;
  if (!p.resident) {
    static int want = -1;
    // Measured (profiles/r02_cluster_multicast_experiment.md): no gain -- the weight ring is bound by the LATENCY of a tile's round trip
    // (96 KB in flight / ~1.5 us), not by L2 bandwidth, and multicast does not shorten that -- so clusters stay opt-in.
    if (want < 0) { const char* e = getenv("GIN_CLUSTER"); want = e ? atoi(e) : 1; if (want != 1 && want != 2 && want != 4) want = 1; }
    CL = want;
    while (CL > 1 && (B_TILE_OF(N_TILE) / CL) % 16) CL /= 2;
  }
  int grid = 0;
  while (true) {
    const long long groups = ((long long)p.total_tiles + CL - 1) / CL + ((long long)p.x_total + CL - 1) / CL;
    const long long want_clusters = groups * p.n_blocks;
    int cap = sms / CL;                                // clusters that can be resident at once
    if (CL > 1) {
      static PerDeviceFlag probed_on[3];
      static int cap_cl[kMaxDevices][3];
      const int slot = CL == 2 ? 1 : 2, d = current_device();
      if (!probed_on[slot].here()) {
        // the limit is set by shared memory (1 CTA per SM) and by how the SMs pair up inside their GPCs: ask the driver
        cap_cl[d][slot] = max_active_clusters(patch_conv_kernel<N_TILE, false, false, false>, CL, NTHREADS, SMEM_LIMIT);
        probed_on[slot].here() = true;
      }
      cap = cap_cl[d][slot] < cap ? cap_cl[d][slot] : cap;
    }
    long long clusters = want_clusters < cap ? want_clusters : cap;
    clusters -= clusters % p.n_blocks;                 // every cluster keeps one n-block
    if (clusters < p.n_blocks) {
      if (CL > 1) { CL /= 2; continue; }               // not even one cluster per n-block fits: smaller clusters
      clusters = p.n_blocks;
    }
    grid = (int)clusters * CL;
    break;
  }
  p.cl = CL;
  if (p.stats_parts) *p.stats_parts = stats ? grid / p.n_blocks : 0;
  if (CL > 1) launch_cluster(kern, CL, dim3(grid), dim3(NTHREADS), smem_total, st, p);
  else launch_pdl(kern, dim3(grid), dim3(NTHREADS), smem_total, st, p);
  return cudaGetLastError() == cudaSuccess ? 0 : -3;
}

}  // namespace cv2

inline bool cv2_supported(int U, int ntiles, int Q, int K, int N) {
  cv2::Params tmp;
  int total;
  return ntiles > 0 && U <= cv2::TAB_ROWS && tc_supported(K, N) && cv2::plan_smem(64, K, U, ntiles, Q, tmp, total);
}
inline bool cv2_supported(const GinPSide& ps, int K, int N) { return cv2_supported(ps.U, ps.ntiles, ps.Q, K, N); }
inline bool cv2_supported(const GinP2Side& ps, int K, int N) { return cv2_supported(ps.U, ps.ntiles, ps.Q, K, N); }

// N tile: minimise (rounds of 148 CTAs) x (MMA time per item); a 64-wide tile is shared-memory-bandwidth bound (A 128 B/clk +
// B 64 B/clk against 128 B/clk), hence the 1.5 penalty
inline int cv2_pick_ntile(long long tiles, int N) {
  int best = 0;
  double best_cost = 0;
  for (int nt : {256, 128, 64}) {
    if (N % nt) continue;
    const long long items = tiles * (N / nt);
    const int sms = num_sms();
    int ctas = (int)(items < sms ? items : sms);
    ctas -= ctas % (N / nt);
    if (ctas < N / nt) ctas = N / nt;
    const long long rounds = (items + ctas - 1) / ctas;
    const double cost = (double)rounds * nt * (nt == 64 ? 1.5 : 1.0);
    if (!best || cost < best_cost * 0.999) { best = nt; best_cost = cost; }
  }
  return best;
}

// Tile-pair mode (gin_conv2_pair.cuh): for streamed weights, when pairing the tiles costs no extra round of CTAs.
int cv2_launch_pair(cv2::Params& p, int nt, cudaStream_t st);
inline bool cv2_pair_ok(const cv2::Params& p, int nt) {
  static int enabled = -1;
  if (enabled < 0) { const char* e = getenv("GIN_PAIR"); enabled = e ? atoi(e) : 1; }      // 0 off, 1 when it costs no extra round, 2 always
  // the affine epilogue exists in the single-tile kernel only (DESIGN: Inference)
  if (!enabled || p.flush_each || p.accumulate || p.dst_tab_off >= 0 || p.nplanes > 4 || p.x_total > 0 || p.aff.scale) return false;
  const int ntp = nt < 128 ? nt : 128;
  if (7 * (p.K / 64) * ntp * 128 <= 114688) return false;                   // the weights fit: the resident single-tile kernel is better
  auto rounds = [&](long long items, int n_blocks) {
    const int sms = num_sms();
    int ctas = (int)(items < sms ? items : sms);
    ctas -= ctas % n_blocks;
    if (ctas < n_blocks) ctas = n_blocks;
    return (items + ctas - 1) / ctas;
  };
  const long long r1 = rounds((long long)p.total_tiles * (p.N / nt), p.N / nt) * nt;                       // ~ MMA time, single tiles
  const long long r2 = rounds((long long)((p.total_tiles + 1) / 2) * (p.N / ntp), p.N / ntp) * 2 * ntp;   // ~ MMA time, tile pairs
  return enabled == 2 || r2 <= r1;
}

inline int cv2_dispatch(cv2::Params& p, int max_ntile, cudaStream_t st) {
  if ((long long)p.B * (p.P_src > p.P_dst ? p.P_src : p.P_dst) + 2LL * p.B >= 0x7fffffffLL) return -4;
  const int groups = (p.B + p.group - 1) / p.group;
  p.total_tiles = (p.x_ntiles > 0 && p.x_all) ? 0 : groups * p.ntiles;
  p.x_total = p.x_ntiles > 0 ? groups * p.x_ntiles : 0;
  { const char* e = getenv("GIN_DBG"); p.dbg = e ? atoi(e) : 0; }
  int nt = cv2_pick_ntile(p.total_tiles + p.x_total, p.N);
  { static int cap = -1; if (cap < 0) { const char* e = getenv("GIN_NTILE_MAX"); cap = e ? atoi(e) : 256; } if (cap < max_ntile && cap >= 64) max_ntile = cap; }
  while (nt > max_ntile) nt /= 2;
  if (cv2_pair_ok(p, nt)) {
    const int rc = cv2_launch_pair(p, nt < 128 ? nt : 128, st);
    if (rc != -4) return rc;          // -4: the pair kernel's shared-memory plan does not fit this patch size: single tiles
  }
  switch (nt) {
    case 256: return cv2::launch<256>(p, st);
    case 128: return cv2::launch<128>(p, st);
    default: return cv2::launch<64>(p, st);
  }
}

// forward epilogue options: a second bias when two sibling convolutions run as one GEMM (columns >= split take p[col - split];
// none when p is null), and y_f16: write Y as fp16 instead of fp32
struct Bias2 { const float* p = nullptr; int split = 0; int y_f16 = 0; };

// `pf` (dgrad only): fold the boundary tiles of the plan into the same launch
inline void cv2_attach_boundary(cv2::Params& p, const GinPfSide* pf) {
  p.mask_off = -1;
  if (!pf || pf->ntiles <= 0 || pf->nslots > cv2::MAX_PLANES) return;
  p.x_ntiles = pf->ntiles; p.x_nslots = pf->nslots; p.x_src_off = pf->src_off; p.x_dst_off = pf->dst_off; p.mask_off = pf->mask_off;
  for (int s = 0; s < pf->nslots; ++s) p.x_tap[s] = pf->tap[s];
  p.x_all = pf->all;
}

// stride 1: forward (mirror 0) / in-chart dgrad (mirror 1: tap (di,dj) reads cell (-di,-dj)); W = 2n pixels per chart row
inline int launch_patch_conv2(const int32_t* plan_dev, const GinPSide& ps, int group, int P, int W, const void* Xb, const void* Wb,
                              const float* bias, const Bias2& bias2, float* Y, int B, int K, int N, int mirror, bool bf16, cudaStream_t st,
                              float* stats = nullptr, int* stats_parts = nullptr, const GinPfSide* pf = nullptr, const cv2::Affine* aff = nullptr) {
  cv2::Params p{};
  cv2_attach_boundary(p, pf);
  if (aff) p.aff = *aff;
  p.stats = stats; p.stats_parts = stats_parts;
  p.plan = plan_dev; p.fmt = idesc_fmt_bits(bf16); p.U = ps.U; p.Q = ps.Q; p.ntiles = ps.ntiles; p.group = group; p.B = B; p.K = K; p.N = N; p.P_src = P; p.P_dst = P;
  p.X = reinterpret_cast<const __nv_bfloat16*>(Xb); p.Wt = reinterpret_cast<const __nv_bfloat16*>(Wb); p.bias = bias; p.Y = Y;
  p.bias1 = bias2.p; p.bias_split = bias2.split; p.y_f16 = bias2.y_f16;
  p.nplanes = 1; p.flush_each = 0; p.ntaps[0] = 7; p.group_bytes = 1280; p.dst_tab_off = -1;
  for (int t = 0; t < 7; ++t) {
    const int di = mirror ? -cv2::kDi[t] : cv2::kDi[t], dj = mirror ? -cv2::kDj[t] : cv2::kDj[t];
    p.tap_id[0][t] = (int8_t)t;
    p.tap_row[0][t] = (int16_t)((1 + di) * ps.Q * 10 + (1 + dj));
  }
  p.tab_off = ps.src_off; p.tab_tstride = ps.U; p.tab_pstride = 0;
  p.base_off = ps.rows_off; p.base_tstride = GIN_TILE_M; p.base_qstride = 8;
  p.dst_row_stride = W; p.dst_px_stride = 1;
  return cv2_dispatch(p, 256, st);
}

// forward tap -> (parity plane, coarse offset a, b) of a stride-2 convolution (gin_plan.h: GinP2Side)
constexpr int kS2Plane[7] = {2, 0, 0, 3, 3, 1, 1};
constexpr int kS2A[7] = {0, 0, 1, 0, 0, 0, 1};
constexpr int kS2B[7] = {0, 0, 0, -1, 0, 0, -1};

// stride 2 forward: X is the FINE map (P_f pixels per sample), Y the coarse one; Wc = 2n of the coarse level
inline int launch_patch_conv2_s2_fwd(const int32_t* plan_dev, const GinP2Side& ps, int group, int P_f, int P_c, int Wc, const void* Xb,
                                     const void* Wb, const float* bias, const Bias2& bias2, float* Y, int B, int K, int N, bool bf16,
                                     cudaStream_t st, float* stats = nullptr, int* stats_parts = nullptr, const cv2::Affine* aff = nullptr) {
  cv2::Params p{};
  p.mask_off = -1;
  if (aff) p.aff = *aff;
  p.stats = stats; p.stats_parts = stats_parts;
  p.plan = plan_dev; p.fmt = idesc_fmt_bits(bf16); p.U = ps.U; p.Q = ps.Q; p.ntiles = ps.ntiles; p.group = group; p.B = B; p.K = K; p.N = N; p.P_src = P_f; p.P_dst = P_c;
  p.X = reinterpret_cast<const __nv_bfloat16*>(Xb); p.Wt = reinterpret_cast<const __nv_bfloat16*>(Wb); p.bias = bias; p.Y = Y;
  p.bias1 = bias2.p; p.bias_split = bias2.split; p.y_f16 = bias2.y_f16;
  p.nplanes = 4; p.flush_each = 0; p.group_bytes = 1280; p.dst_tab_off = -1;
  for (int t = 0; t < 7; ++t) {
    const int pl = kS2Plane[t], j = p.ntaps[pl]++;
    p.tap_id[pl][j] = (int8_t)t;
    p.tap_row[pl][j] = (int16_t)((1 + kS2A[t]) * ps.Q * 10 + (1 + kS2B[t]));
  }
  p.tab_off = ps.src_off; p.tab_tstride = 4 * ps.U; p.tab_pstride = ps.U;
  p.base_off = ps.rows_off; p.base_tstride = GIN_TILE_M; p.base_qstride = 8;
  p.dst_row_stride = Wc; p.dst_px_stride = 1;
  return cv2_dispatch(p, 256, st);
}

// stride 2 dgrad, in-chart part: X is the coarse dy (K = Cout channels), Y the fine dx; Wf = 2n of the fine level
inline int launch_patch_conv2_s2_dgrad(const int32_t* plan_dev, const GinP2Side& ps, int group, int P_f, int P_c, int Wf, const void* dYb,
                                       const void* Wb, float* dX, int B, int K, int N, bool bf16, cudaStream_t st, const GinPfSide* pf = nullptr) {
  cv2::Params p{};
  cv2_attach_boundary(p, pf);
  p.plan = plan_dev; p.fmt = idesc_fmt_bits(bf16); p.U = ps.U; p.Q = ps.Q; p.ntiles = ps.ntiles; p.group = group; p.B = B; p.K = K; p.N = N; p.P_src = P_c; p.P_dst = P_f;
  p.X = reinterpret_cast<const __nv_bfloat16*>(dYb); p.Wt = reinterpret_cast<const __nv_bfloat16*>(Wb); p.bias = nullptr; p.Y = dX;
  p.nplanes = 4; p.flush_each = 1; p.group_bytes = 1280; p.dst_tab_off = -1;
  for (int t = 0; t < 7; ++t) {
    const int pl = kS2Plane[t], j = p.ntaps[pl]++;
    p.tap_id[pl][j] = (int8_t)t;
    p.tap_row[pl][j] = (int16_t)((1 - kS2A[t]) * ps.Q * 10 + (1 - kS2B[t]));
  }
  p.tab_off = ps.dsrc_off; p.tab_tstride = ps.U; p.tab_pstride = 0;
  p.base_off = ps.frows_off; p.base_tstride = ps.Q; p.base_qstride = 1;
  p.dst_row_stride = 2 * Wf; p.dst_px_stride = 2;
  for (int pl = 0; pl < 4; ++pl) p.dst_plane_off[pl] = (pl >> 1) * Wf + (pl & 1);
  return cv2_dispatch(p, 256, st);     // two accumulators of N_TILE columns, as everywhere
}

// The cross-seam / pole remainder of dgrad (GinPxSide), added into dX after the in-chart pass: every tile = `nslots` segments of
// 128 gathered dy rows with one tap each, all accumulated into one tile, destination pixels from the plan, read-modify-write.
inline bool cv2_seam_supported(const GinPxSide& px, int K, int N) {
  return px.ntiles > 0 && px.nslots <= cv2::MAX_PLANES && cv2_supported(GIN_TILE_M, px.ntiles, 1, K, N);
}
inline int launch_patch_conv2_seam(const int32_t* plan_dev, const GinPxSide& px, int group, int P_src, int P_dst, const void* dYb, const void* Wb,
                                   float* dX, int B, int K, int N, bool bf16, cudaStream_t st) {
  cv2::Params p{};
  p.mask_off = -1;
  p.plan = plan_dev; p.fmt = idesc_fmt_bits(bf16); p.U = GIN_TILE_M; p.Q = 1; p.ntiles = px.ntiles; p.group = group; p.B = B; p.K = K; p.N = N; p.P_src = P_src; p.P_dst = P_dst;
  p.X = reinterpret_cast<const __nv_bfloat16*>(dYb); p.Wt = reinterpret_cast<const __nv_bfloat16*>(Wb); p.bias = nullptr; p.Y = dX;
  p.nplanes = px.nslots; p.flush_each = 0; p.group_bytes = 1024; p.accumulate = 1; p.dst_tab_off = px.dst_off;
  for (int s = 0; s < px.nslots; ++s) { p.ntaps[s] = 1; p.tap_id[s][0] = px.tap[s]; p.tap_row[s][0] = 0; }
  p.tab_off = px.src_off; p.tab_tstride = px.nslots * GIN_TILE_M; p.tab_pstride = GIN_TILE_M;
  return cv2_dispatch(p, 256, st);
}

}  // namespace gin
