// Helpers shared by the x3 disparity-head kernels (disp_head_x3.cuh, disp_head_x3r.cuh, disp_head_x3w.cuh):
// packed-FP32 wrappers (FFMA2 / FADD2 / FMUL2 on sm_100a) and the geometry of the shared-memory window of the
// tiled forward kernel.
#pragma once
#include "common.cuh"

namespace rag {

constexpr float kX3NegLog2e = -1.4426950408889634f;
constexpr float kX3Tau = 24.0f;  // lazy-rescale threshold (log2 units) of the first-generation kernel
// window of the tiled forward kernel: 32 block columns + a 4-column halo on each side = 40 floats per row
constexpr int kTCols = 40;

__device__ __forceinline__ float2 f2(float a, float b) { return make_float2(a, b); }
__device__ __forceinline__ float2 f2b(float a) { return make_float2(a, a); }
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 ex2_2(float2 z) { return make_float2(ex2_approx(z.x), ex2_approx(z.y)); }

}  // namespace rag
