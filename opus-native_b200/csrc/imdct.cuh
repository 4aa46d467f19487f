// imdct.cuh -- complex arithmetic shared by the IMDCT kernels, and the out-of-place comb filter.
//
// Arithmetic contract of every float kernel in this library: each sum and product is evaluated in
// the same order and with the same single roundings as the reference; the translation unit is
// compiled with -fmad=false so nvcc never contracts a*b+c (Rust does not either).  Data placement
// (registers / shared memory / which lane owns which butterfly) is free and is what the B200 design
// changes: see imdct_warp.cuh.
#pragma once
#include "opn_device.cuh"
#include "opn_internal.h"

namespace opn {

// Packed FP32 adds (sm_100 FADD2, PTX add.rn.f32x2): one instruction, both halves rounded to nearest once -- the same two
// values two scalar FADDs give.  The SASS operand may swap its halves and negate either one for free, which ptxas
// recovers from the way the operand is put together here (p_add(a, make_float2(s.y, -s.x)) is ONE FADD2).
// Only sums are packed.  ptxas contracts mul.rn.f32x2 followed by add.rn.f32x2 into FFMA2 even under --fmad=false
// (checked on 12.9), which would change roundings; a scalar FMUL is never contracted, so every product that feeds a sum
// stays scalar.  tests/test_host_logic.py::test_no_fma_in_the_fused_float_kernels looks at the SASS.
__device__ __forceinline__ float2 p_add(float2 a, float2 b)
{
    float2 r;
    asm("{.reg .b64 ra, rb, rc; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%5}; add.rn.f32x2 rc, ra, rb; mov.b64 {%0,%1}, rc;}"
        : "=f"(r.x), "=f"(r.y)
        : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return r;
}
__device__ __forceinline__ float2 c_add(float2 a, float2 b) { return p_add(a, b); }
__device__ __forceinline__ float2 c_sub(float2 a, float2 b) { return p_add(a, make_float2(-b.x, -b.y)); }  // x - y == x + (-y), exactly
// (a.x + s.y, a.y - s.x) and (a.x - s.y, a.y + s.x): a -/+ i s, the rotated sums of the butterflies
__device__ __forceinline__ float2 c_add_mrot(float2 a, float2 s) { return p_add(a, make_float2(s.y, -s.x)); }
__device__ __forceinline__ float2 c_sub_mrot(float2 a, float2 s) { return p_add(a, make_float2(-s.y, s.x)); }
// src/math.rs:115-124: (a.x b.x - a.y b.y, a.x b.y + a.y b.x); four scalar products, one packed sum
__device__ __forceinline__ float2 c_mul(float2 a, float2 b) { return p_add(make_float2(a.x * b.x, a.x * b.y), make_float2(-(a.y * b.y), a.y * b.x)); }
__device__ __forceinline__ float2 c_scale(float2 a, float s) { return make_float2(a.x * s, a.y * s); }

#define OPN_FRAC_1_SQRT_2 0.70710678118654752440f

// ---------------------------------------------------------------------------------------------
// Operator-level kernel (tests call it through opn_op_comb_filter).
// comb_filter (out of place, FIR; comb_filter/mod.rs:59-127, fallback.rs:6-29): no recursion, so
// every output sample is independent.
__global__ void __launch_bounds__(IM_TPC)
k_op_comb(float *__restrict__ y, const float *__restrict__ x, size_t row_stride, int offset, int n,
          const int32_t *__restrict__ params4, const float *__restrict__ gains2, int overlap)
{
    const float *xr = x + (size_t)blockIdx.x * row_stride + offset;
    float *yr = y + (size_t)blockIdx.x * row_stride + offset;
    int t0 = params4[4 * blockIdx.x], t1 = params4[4 * blockIdx.x + 1];
    const int tap0 = params4[4 * blockIdx.x + 2], tap1 = params4[4 * blockIdx.x + 3];
    const float g0 = gains2[2 * blockIdx.x], g1 = gains2[2 * blockIdx.x + 1];
    if (g0 == 0.0f && g1 == 0.0f) {
        for (int i = threadIdx.x; i < n; i += IM_TPC) yr[i] = xr[i];
        return;
    }
    t0 = max(t0, 15);
    t1 = max(t1, 15);
    const float g00 = g0 * g_tab.comb_gains[tap0 * 3], g01 = g0 * g_tab.comb_gains[tap0 * 3 + 1],
                g02 = g0 * g_tab.comb_gains[tap0 * 3 + 2];
    const float g10 = g1 * g_tab.comb_gains[tap1 * 3], g11 = g1 * g_tab.comb_gains[tap1 * 3 + 1],
                g12 = g1 * g_tab.comb_gains[tap1 * 3 + 2];
    if (fabsf(g0 - g1) < 1.1920929e-7f && t0 == t1 && tap0 == tap1) overlap = 0;
    for (int i = threadIdx.x; i < n; i += IM_TPC) {
        float acc = xr[i];
        if (i < overlap) {
            const float f = __ldg(&g_tab.window_sq[i]);
            acc = acc + (((1.0f - f) * g00) * xr[i - t0]);
            acc = acc + (((1.0f - f) * g01) * (xr[i - t0 + 1] + xr[i - t0 - 1]));
            acc = acc + (((1.0f - f) * g02) * (xr[i - t0 + 2] + xr[i - t0 - 2]));
            acc = acc + ((f * g10) * xr[i - t1]);
            acc = acc + ((f * g11) * (xr[i - t1 + 1] + xr[i - t1 - 1]));
            acc = acc + ((f * g12) * (xr[i - t1 + 2] + xr[i - t1 - 2]));
        } else if (g1 != 0.0f) {
            acc = acc + (g10 * xr[i - t1]) + (g11 * (xr[i - t1 + 1] + xr[i - t1 - 1])) +
                  (g12 * (xr[i - t1 + 2] + xr[i - t1 - 2]));
        }
        yr[i] = acc;
    }
}

}  // namespace opn
