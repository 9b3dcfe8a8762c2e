// Shared helpers for the sm_100a kernels of the YOLO-Nano forward path.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "yolonano_b200.h"

namespace ynb {

constexpr int kNumSMs = 148;   // B200: 2 dies x 74 SMs

// ---- activation epilogues (utils/modules.py:14, backbone/shufflenetv2.py:48) -----------
__device__ __forceinline__ float apply_act(float v, int act) {
  if (act == YNB_ACT_RELU) return fmaxf(v, 0.0f);
  if (act == YNB_ACT_LEAKY) return v > 0.0f ? v : 0.1f * v;   // LeakyReLU(0.1)
  return v;
}

// Class softmax pieces shared by decode_level_kernel and the fused decode epilogue of the head
// GEMM (models/yolo_nano.py:362-365).  d = logit - max <= 0; the denominator only needs ~1e-6
// relative accuracy (scores are compared at rtol 1e-4), so ex2.approx on d*log2(e) is used:
// 2 instructions instead of expf's 7.
__device__ __forceinline__ float softmax_exp(float d) { return __expf(d); }
__device__ __forceinline__ float class_score(float sum, float obj) { return __fmul_rn(__fdiv_rn(1.0f, sum), obj); }

// ---- activation storage type: float32 (parity / tf32 modes) or bfloat16 (YNB_GEMM_TC_BF16) ---------------
// Arithmetic is always fp32 (depthwise taps, bias, activation, accumulators); only what sits in HBM between
// kernels changes.  4 consecutive channels are the unit every HBM-bound kernel moves: 16 bytes as float, 8 as bf16.
using bf16 = __nv_bfloat16;

__device__ __forceinline__ float4 load4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 load4(const bf16* p) {
  const uint2 u = *reinterpret_cast<const uint2*>(p);
  return make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u), __uint_as_float(u.y << 16),
                     __uint_as_float(u.y & 0xffff0000u));
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {     // round to nearest even, lo in bits [0,16)
  const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&v);
}
__device__ __forceinline__ void store4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void store4(bf16* p, float4 v) {
  *reinterpret_cast<uint2*>(p) = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
}
__device__ __forceinline__ float to_float(float v) { return v; }
__device__ __forceinline__ float to_float(bf16 v) { return __bfloat162float(v); }

inline int round_up(int v, int m) { return (v + m - 1) / m * m; }
inline int64_t round_up64(int64_t v, int64_t m) { return (v + m - 1) / m * m; }

// Launch bookkeeping: every kernel launch of the library goes through LAUNCH so that
// ynb_launch_count() is a true count.
struct LaunchCounter {
  int64_t n = 0;
};
extern thread_local LaunchCounter* g_counter;   // set by the engine around a forward

// Programmatic dependent launch: every kernel of the forward is launched with the
// programmatic-stream-serialization attribute, lets its successor start early
// (pdl_trigger at the top) and waits for its predecessor's results right before its first
// dependent global access (pdl_wait) — prologues (barrier init, TMEM alloc, weight loads)
// overlap the previous kernel's tail instead of adding to the critical path.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

inline bool pdl_enabled() {
  static int v = -1;
  if (v < 0) v = getenv("YNB_NO_PDL") ? 0 : 1;
  return v == 1;
}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

#define YNB_COUNT_LAUNCH()                  \
  do {                                      \
    if (::ynb::g_counter) ::ynb::g_counter->n++; \
  } while (0)

}  // namespace ynb
