// Exact scatter-add of fp32 3-vectors without floating-point atomics, shared by the Chamfer backward (gin_chamfer.cuh) and the
// Chamfer normal / Laplacian terms (gin_chamfer_terms.cuh).
//
// Every receiving point r owns an Acc, zeroed before use.  Pass 1 (note) takes, per receiving point, the largest exponent of its
// terms and their count (integer atomicMax / atomicAdd).  Pass 2 (add) rounds every term to the grid 2^-s of its point (s chosen
// so that count terms cannot overflow 62 bits) and adds the integers with 64-bit integer atomics: integer addition is associative,
// so the sum is the same bits whatever the order.  read() converts it back.  Every term within 2^-38 of its point's largest term
// keeps all of its fp32 bits.  Pass 2 must recompute exactly the terms of pass 1.
#pragma once
#include <cuda_runtime.h>

namespace gin {
namespace fixsum {

struct Acc { long long s[3]; int e; int n; };     // int64 sums [3], biased exponent, count (32 B)

// biased fp32 exponent of the largest component (0 for zeros)
__device__ __forceinline__ int max_exponent(const float t[3]) {
  const unsigned m = max(max(__float_as_uint(t[0]) & 0x7fffffffu, __float_as_uint(t[1]) & 0x7fffffffu), __float_as_uint(t[2]) & 0x7fffffffu);
  return (int)(m >> 23);
}

// 2^shift such that count terms below 2^(e - 126) (biased exponent e) sum to less than 2^62
__device__ __forceinline__ int fixed_shift(const Acc& a) { return 61 - (a.e - 127) - (32 - __clz(max(a.n, 1))); }

// pass 1: register the term t with its receiving point
__device__ __forceinline__ void note(Acc* a, const float t[3]) {
  atomicMax(&a->e, max_exponent(t));
  atomicAdd(&a->n, 1);
}

// pass 2: add the term t in fixed point
__device__ __forceinline__ void add(Acc* a, const float t[3]) {
  if (a->e == 0) return;                           // every term of this point is zero
  const int sh = fixed_shift(*a);
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const long long q = __double2ll_rn(ldexp((double)t[k], sh));      // exact scaling, one rounding to the grid
    atomicAdd(reinterpret_cast<unsigned long long*>(&a->s[k]), (unsigned long long)q);
  }
}

// v += the sum of the point's terms
__device__ __forceinline__ void read(const Acc& a, float v[3]) {
  if (a.e == 0) return;
  const int sh = fixed_shift(a);
#pragma unroll
  for (int k = 0; k < 3; ++k) v[k] += (float)ldexp((double)a.s[k], -sh);
}

}  // namespace fixsum
}  // namespace gin
