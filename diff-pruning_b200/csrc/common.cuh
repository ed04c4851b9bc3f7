// common.cuh — shared helpers for libdpb200 (sm_100a only).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include "dpb200.h"

extern int g_dp_last_cuda_error;
extern long long g_dp_launch_count;

static inline int dp_check_launch() {
  ++g_dp_launch_count;
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) {
    g_dp_last_cuda_error = (int)e;
    (void)cudaGetLastError();
    return DP_ERR_CUDA;
  }
  return DP_OK;
}

#define DP_REQUIRE(cond, code) \
  do {                         \
    if (!(cond)) return (code); \
  } while (0)

static inline int ilog2_exact(int v) {  // log2 if power of two, else -1
  if (v <= 0 || (v & (v - 1))) return -1;
  int l = 0;
  while ((1 << l) < v) ++l;
  return l;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// max |v| of the values a thread wrote -> the output tensor's amax slot (dp_amax semantics: atomicMax on the bit pattern of a
// non-negative float is order-independent, so slots are run-to-run identical); one atomic per converged warp
__device__ __forceinline__ void amax_commit(uint32_t* slot, float m) {
  const unsigned mask = __activemask();
  const uint32_t r = __reduce_max_sync(mask, __float_as_uint(m));
  if ((threadIdx.x & 31) == (unsigned)(__ffs(mask) - 1) && r) atomicMax(slot, r);
}
// 1 / (1 + exp(-x)): __frcp_rn is the correctly rounded reciprocal, i.e. the same bits as the IEEE division 1.0f / y, without the
// division's slow-path check
__device__ __forceinline__ float sigmoidf_acc(float x) { return __frcp_rn(1.0f + expf(-x)); }

// 3 x fp16 split operands (conv_tc.cu, and the split output of the GroupNorm forward that feeds them).
// amax slot -> power-of-two scale.  E = biased exponent of the bound (|v| < 2^(E-126)), clamped so that both factors are normal floats;
// up = 2^(140-E) brings the operand below 2^14 (fp16 overflows at 65504), dn = 2^(E-140) undoes it in the epilogue.
__device__ __forceinline__ int amax_exponent_bits(uint32_t bound_bits) { return min(max((int)((bound_bits >> 23) & 0xFFu), 14), 254); }
__device__ __forceinline__ int amax_exponent(const uint32_t* slot) { return amax_exponent_bits(__ldg(slot)); }
__device__ __forceinline__ float scale_up(int E) { return __uint_as_float((uint32_t)(267 - E) << 23); }
__device__ __forceinline__ float scale_dn(int E) { return __uint_as_float((uint32_t)(E - 13) << 23); }
constexpr float LO_SCALE = 2048.f, LO_UNSCALE = 1.f / 2048.f;   // lo' = lo * 2^11 keeps the residual in fp16's normal range
// two scaled values -> packed fp16 hi pair and lo' pair (low half = first element = lower address)
__device__ __forceinline__ void split2(float a, float b, uint32_t& h, uint32_t& l) {
  const __half2 hh = __floats2half2_rn(a, b);
  const float2 hf = __half22float2(hh);
  const __half2 ll = __floats2half2_rn((a - hf.x) * LO_SCALE, (b - hf.y) * LO_SCALE);
  h = *reinterpret_cast<const uint32_t*>(&hh);
  l = *reinterpret_cast<const uint32_t*>(&ll);
}
