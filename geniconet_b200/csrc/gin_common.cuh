// Shared device helpers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "gin_plan.h"

#define GIN_DEVINL __device__ __forceinline__

// Programmatic dependent launch (GIN_PDL=1): a kernel launched through launch_pdl may start while its predecessor in the stream is
// still draining; its CTAs set up (barriers, TMEM, constant tables) and then block in GIN_PDL_SYNC() until the predecessor grid has
// completed and its memory is visible.  EVERY kernel launched through launch_pdl must execute GIN_PDL_SYNC() in all threads before
// its first access to memory another kernel produces or consumes (completion of a grid then implies completion of everything
// before it in the stream).  Without the launch attribute the instructions are no-ops.
#define GIN_PDL_SYNC() asm volatile("griddepcontrol.wait;\n\tgriddepcontrol.launch_dependents;" ::: "memory")

struct GinSrcView {      // a gathered fp32 tensor with arbitrary element strides
  const float* p;
  long long sb, sp, sc;  // element (b, pixel, channel) -> p[b*sb + pixel*sp + channel*sc]
  int P;                 // pixels per sample
};

namespace gin {
// Per-device host state: function attributes (dynamic shared-memory size) are per context, so "configured once" must be
// tracked per device; persistent grids size themselves from the device's SM count (148 on B200; capped there because the
// per-CTA workspaces are sized for 148).
constexpr int kMaxDevices = 64, kMaxSMs = 148;
inline int current_device() { int d = 0; cudaGetDevice(&d); return d & (kMaxDevices - 1); }
inline int num_sms() {
  static int n[kMaxDevices] = {};
  const int d = current_device();
  if (!n[d]) {
    int v = kMaxSMs;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, d) != cudaSuccess || v <= 0) v = kMaxSMs;
    // GIN_SMS: leave some SMs to a concurrent kernel (data-parallel training: the NCCL all-reduce).  The persistent kernels own an SM
    // per CTA and hand tiles out statically, so a kernel that takes SMs from them would push CTAs into a second wave.
    if (const char* e = getenv("GIN_SMS")) { const int cap = atoi(e); if (cap >= 8 && cap < v) v = cap; }
    n[d] = v < kMaxSMs ? v : kMaxSMs;
  }
  return n[d];
}
struct PerDeviceFlag {
  bool done[kMaxDevices] = {};
  bool& here() { return done[current_device()]; }
};

// 16-bit operand formats of the tcgen05 path.  FORWARD-side operands (activation copies, forward weight tiles) are fp16 by
// default: post-BatchNorm activations and weights are O(1), far inside fp16's range (conversions saturate to +-65504 anyway),
// and its 10-bit mantissa leaves 1/8 of bf16's rounding noise in the network output -- which is what the normal / Laplacian
// loss terms differentiate (profiles/r02_precision_study.md).  GRADIENT-side operands (dy copies, dgrad weight tiles) stay
// bf16: their magnitudes span many decades.  GIN_FWD_FP16=0 switches the forward side back to bf16 (A/B experiments).
// The instruction descriptor carries the A and B formats separately (bits 7-9 / 10-12: 0 = fp16, 1 = bf16), but a kind::f16 MMA
// whose two operands differ in format traps as an illegal instruction on sm_100a (measured, r02).  wgrad multiplies a forward
// activation by a gradient, so every forward activation copy is ALSO written in bf16 by its producer (2 more bytes per element);
// wgrad sums over ~10^5 pixels, so the rounding of that copy averages out -- the forward pass is where the mantissa matters.
inline bool fwd_fp16() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("GIN_FWD_FP16"); v = (e && e[0] == '0') ? 0 : 1; }
  return v == 1;
}
// operand-format bits of a tcgen05 launch's instruction descriptor: both operands bf16, or both fp16 (the two must agree)
inline uint32_t idesc_fmt_bits(bool bf16) { return bf16 ? (1u << 7) | (1u << 10) : 0u; }

inline bool pdl_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("GIN_PDL"); v = (e && e[0] == '1') ? 1 : 0; }
  return v == 1;
}

template <typename... KArgs, typename... Args>
inline void launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  if (pdl_enabled()) {
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
  }
  cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// The same as a launch of thread-block clusters of `cluster` CTAs (grid.x must be a multiple of it).
template <typename... KArgs, typename... Args>
inline void launch_cluster(void (*kernel)(KArgs...), int cluster, dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int na = 0;
  attr[na].id = cudaLaunchAttributeClusterDimension;
  attr[na].val.clusterDim.x = (unsigned)cluster; attr[na].val.clusterDim.y = 1; attr[na].val.clusterDim.z = 1;
  ++na;
  if (pdl_enabled()) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr; cfg.numAttrs = na;
  cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// how many clusters of `cluster` CTAs of this kernel can be resident at once (0 on error)
template <typename... KArgs>
inline int max_active_clusters(void (*kernel)(KArgs...), int cluster, int block, size_t smem) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)cluster); cfg.blockDim = dim3((unsigned)block); cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)cluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, kernel, &cfg) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}
}  // namespace gin

__host__ GIN_DEVINL const int32_t* plan_words(const void* plan) { return reinterpret_cast<const int32_t*>(plan); }

// Packed-weight blob layout (gin_hexconv_pack_weights), offsets in bytes from the start:
//   [0]                      float wf[7][Cin][Cout]   forward   B operand (SIMT)
//   [28*Cin*Cout]            float wd[7][Cout][Cin]   dgrad     B operand (SIMT)
//   [56*Cin*Cout]            bf16  bf[7][Cin/64][Cout][64]  forward B tiles (tcgen05), pre-swizzled smem image
//   [70*Cin*Cout]            bf16  bd[7][Cout/64][Cin][64]  dgrad   B tiles (tcgen05), pre-swizzled smem image
GIN_DEVINL __host__ size_t packed_off_wf(int, int) { return 0; }
GIN_DEVINL __host__ size_t packed_off_wd(int Cin, int Cout) { return (size_t)28 * Cin * Cout; }
GIN_DEVINL __host__ size_t packed_off_bf(int Cin, int Cout) { return (size_t)56 * Cin * Cout; }
GIN_DEVINL __host__ size_t packed_off_bd(int Cin, int Cout) { return (size_t)70 * Cin * Cout; }
GIN_DEVINL __host__ size_t packed_total(int Cin, int Cout) { return (size_t)84 * Cin * Cout; }

// two fp32 -> one packed pair of 16-bit operands: fp16 (round to nearest, saturating to the largest finite value) or bf16
GIN_DEVINL uint32_t pack2_f16(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
GIN_DEVINL uint32_t pack2_bf16(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
GIN_DEVINL uint32_t pack2_op(float lo, float hi, int f16) { return f16 ? pack2_f16(lo, hi) : pack2_bf16(lo, hi); }
GIN_DEVINL unsigned short cvt_op(float v, int f16) { return (unsigned short)(pack2_op(v, 0.f, f16) & 0xffffu); }

GIN_DEVINL float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
