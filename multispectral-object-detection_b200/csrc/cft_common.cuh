// Shared host/device helpers of libcft_b200 (sm_100a only).
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/cft_b200.h"

namespace cft {

// ---------------------------------------------------------------- host-side bookkeeping
void set_error(const char* fmt, ...);
int fail_arg(const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what);

// Wraps one kernel launch: launch counter + optional CUDA-event profiling per kernel id.
struct LaunchScope {
  int id;
  cudaStream_t stream;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  LaunchScope(int kernel_id, cudaStream_t s);
  int finish(const char* what);  // call right after the <<<>>>; returns CFT_* code
};

int sm_count();

// Launch helper of the small kernels (plain stream order; programmatic dependent launch for them was measured at +0.2 ms
// per step in round 1 and removed -- every kernel still starts with pdl_prologue(), a no-op for a plain launch).
template <typename... KArgs, typename... Args>
inline cudaError_t launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                          Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// attention_tcgen05.cu: CFT_E_UNSUPPORTED when the shape is outside the tensor-core kernel.
int attention_tcgen05(const void* qkv, void* out, int B, int T, int C, int heads, cudaStream_t stream);

#define CFT_REQUIRE(cond, ...)                      \
  do {                                              \
    if (!(cond)) return ::cft::fail_arg(__VA_ARGS__); \
  } while (0)

// ---------------------------------------------------------------- device helpers
// First statement of every small kernel: let the next kernel in the stream begin launching, then wait until all
// predecessor kernels have completed and their writes are visible (both are no-ops for a plain launch).
__device__ __forceinline__ void pdl_prologue() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
}
// relative error <= (2.4 |x| + 10) * 2^-24: __expf (2 + 1.173 |x| ulp), 1 + e, __fdividef (2 ulp)
__device__ __forceinline__ float silu_f(float v) { return __fdividef(v, 1.0f + __expf(-v)); }
// SiLU on the SFU: x * rcp(1 + 2^(-x*log2e)); 2 MUFU + 3 FP32 ops, relative error <= (|x| + 8) * 2^-24 (the rounding of
// x * log2e puts |x| * 2^-24 into 2^(...), ex2 2^-22, rcp 2^-23): 1e-6 at |x| = 9, far below bf16's 2^-9.
__device__ __forceinline__ float silu_fast(float v) {
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(v * -1.4426950408889634f));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
  return v * r;
}
// SiLU with ONE SFU op: x*sigmoid(x) = h + h*tanh(h), h = x/2 (tanh.approx.f32: abs error ~5e-4 -> |err| <= |x| * 2.5e-4).
__device__ __forceinline__ float silu_tanh(float v) {
  const float h = 0.5f * v;
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}
__device__ __forceinline__ float silu_tanh_h(float h) {   // h = v / 2 already formed
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}
// |err| <= |x| * 1.5e-7: erff (2 ulp), the rounding of x / sqrt2 and of 1 + erf (no more than 2^-23 absolute)
__device__ __forceinline__ float gelu_f(float v) { return 0.5f * v * (1.0f + erff(v * 0.70710678118654752440f)); }
// erf-GELU with erf from Abramowitz & Stegun 7.1.26 (|err| <= 1.5e-7), written through erfc so that the negative tail
// has no cancellation: q = erfc(|v|/sqrt2)/2, gelu = v - v*q (v >= 0) or v*q (v < 0).  2 SFU ops + ~10 FP32 ops per
// element (erff: ~30); abs error vs the exact erf form <= 4e-7, far below the bf16 rounding of the result.
__device__ __forceinline__ float gelu_fast(float v) {
  const float ax = fabsf(v) * 0.70710678118654752440f;
  float t, e;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, ax, 1.0f)));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(ax * ax * -1.4426950408889634f));
  float poly = fmaf(0.5f * 1.061405429f, t, 0.5f * -1.453152027f);
  poly = fmaf(poly, t, 0.5f * 1.421413741f);
  poly = fmaf(poly, t, 0.5f * -0.284496736f);
  poly = fmaf(poly, t, 0.5f * 0.254829592f);
  const float q = poly * t * e;
  return v >= 0.f ? fmaf(-v, q, v) : v * q;
}
__device__ __forceinline__ float apply_act(float v, int act) {
  if (act == CFT_ACT_SILU) return silu_f(v);
  if (act == CFT_ACT_GELU) return gelu_f(v);
  return v;
}

// 8 bf16 = one 16-byte memory transaction.  The payload is a uint4 on purpose: a struct of four __nv_bfloat162 is copied
// member by member (four 4-byte LDG / STG per copy -- measured: every mover of the path issued 4x the memory instructions
// and, with one row per lane, 4x the L2 sector requests), a uint4 member is one LDG.128 / STG.128.
struct __align__(16) bf16x8 {
  uint4 u;
  __device__ __forceinline__ __nv_bfloat162 get(int i) const {
    const uint32_t w = i == 0 ? u.x : (i == 1 ? u.y : (i == 2 ? u.z : u.w));
    return *reinterpret_cast<const __nv_bfloat162*>(&w);
  }
  __device__ __forceinline__ void set(int i, __nv_bfloat162 h) {
    const uint32_t w = *reinterpret_cast<const uint32_t*>(&h);
    if (i == 0) u.x = w;
    else if (i == 1) u.y = w;
    else if (i == 2) u.z = w;
    else u.w = w;
  }
};

__device__ __forceinline__ void unpack8(const bf16x8& p, float* f) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t = __bfloat1622float2(p.get(i));
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ bf16x8 pack8(const float* f) {
  bf16x8 p;
#pragma unroll
  for (int i = 0; i < 4; ++i) p.set(i, __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]));
  return p;
}

}  // namespace cft
