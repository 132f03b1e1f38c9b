// front_packed.cuh — building blocks shared by the packed-FP32 front kernels (front3.cu, front4.cu): f32x2 wrappers and the blur
// core on pairs, the exact division on pairs, Sobel in half precision with fp32 magnitude^2, floor(sqrt)^2 on exact fp32 integers.
//
// Why the products use the flush-to-zero form: the reference's rounding order (src/utils.cpp:41-47,56-62: every product rounded,
// every accumulation rounded, ascending taps) forbids fused multiply-adds, and ptxas 12.9 contracts mul.rn.f32x2 + add.rn.f32x2 into
// FFMA2 whatever the PTX says — unless the two instructions disagree on flush-to-zero: a compiler that fused mul.rn.FTZ.f32x2 with
// add.rn.f32x2 would change results for subnormal products, so it must not (SASS: FMUL2.FTZ + FADD2, no FFMA2 in the blur).
// Flushing never happens: every product is 0 or >= 2^-90 (these kernels are only used when the smallest weight squared is >= 2^-90;
// prepare_gauss, GaussTables::tiny), so the values are those of plain mul.rn.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace cb {
namespace pk {

// ---- packed FP32 (two IEEE lanes per instruction; a "pair" is a 64-bit register {lo, hi}) ----
typedef unsigned long long u64;
__device__ __forceinline__ u64 pack2(float lo, float hi) { u64 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void unpack2(u64 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
// products: flush-to-zero form (never flushes here, see the file header) so that ptxas cannot contract them with the sums
__device__ __forceinline__ u64 mul2_ftz(u64 a, u64 b) { u64 r; asm("mul.rn.ftz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ u64 add2(u64 a, u64 b) { u64 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ u64 add2_rz(u64 a, u64 b) { u64 r; asm("add.rz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) { u64 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }

// The blur core of front_common.cuh (blur_run) on pairs: S consecutive outputs, ascending taps, one rounding per product and per sum
// (src/utils.cpp:41-46 / 56-61); ws2[j] = {w[R+j], w[R+j]}.
template <int R, int S, typename Fetch, typename Emit>
static __device__ __forceinline__ void blur_run2(const u64 (&ws2)[R + 1], Fetch fetch, Emit emit) {
    u64 acc[S];
#pragma unroll
    for (int i = 0; i < S + 2 * R; ++i) {
        const u64 x = fetch(i);
        u64 q[R + 1];
#pragma unroll
        for (int j = 0; j <= R; ++j) q[j] = mul2_ftz(x, ws2[j]);  // unused ones are dead code
#pragma unroll
        for (int t = 0; t <= 2 * R; ++t) {
            const int o = i - t;
            if (o >= 0 && o < S) {
                const int j = t < R ? R - t : t - R;
                acc[o] = (t == 0) ? q[j] : add2(acc[o], q[j]);  // 0 + q == q exactly
            }
        }
        if (i >= 2 * R) emit(i - 2 * R, acc[i - 2 * R]);
    }
}

// RN(a / b) for the interior count on pairs.  The 1- and 3-instruction forms are only used when the host has checked on the
// device, for this very b and every float mantissa, that they give the IEEE quotient (check_div_mode_device).
// nb2 = {-b, -b}, y2 = {RN(1/b)} x 2, c2 = {RN(1/b - 1)} x 2
template <int DIV>
__device__ __forceinline__ u64 div_const2(u64 a, u64 nb2, u64 y2, u64 c2) {
    if (DIV == 1) return fma2(a, c2, a);
    u64 q = mul2_ftz(a, y2);               // a is 0 or >= 2^-45 here and y ~ 1: nothing to flush
    u64 r = fma2(nb2, q, a);
    q = fma2(r, y2, q);
    if (DIV == 3) return q;
    r = fma2(nb2, q, a);
    return fma2(r, y2, q);
}

// ---- exact Sobel in half precision ----
__device__ __forceinline__ uint32_t hfma2(uint32_t a, uint32_t b, uint32_t c) { uint32_t r; asm("fma.rn.f16x2 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
// half2(lo = v, hi = u) from two exact small integers held in floats
__device__ __forceinline__ uint32_t pack_half2(float lo, float hi) { uint32_t r; asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo)); return r; }
constexpr uint32_t kHM1P1 = 0x3C00BC00u;   // half2(lo = -1, hi = +1)
constexpr uint32_t kH0P2 = 0x40000000u;    // half2(lo =  0, hi = +2)
// (gx, gy) = (v[c+1] - v[c-1], u[c-1] + 2u[c] + u[c+1]) as half2 from the three words around column c
__device__ __forceinline__ uint32_t sobel_h(uint32_t wl, uint32_t wc, uint32_t wr) { return hfma2(wc, kH0P2, hfma2(wl, kHM1P1, wr)); }
// gx*gx + gy*gy, gx*gx and gx*gy in fp32 from the half pair (mixed-precision FMA, exact: |g| <= 1020)
__device__ __forceinline__ float norm2_h(uint32_t g) {
    float n;
    asm("{ .reg .f16 a, b; .reg .f32 z;\n\tmov.b32 {a, b}, %1;\n\tfma.rn.f32.f16 z, b, b, 0f00000000;\n\tfma.rn.f32.f16 %0, a, a, z; }" : "=f"(n) : "r"(g));
    return n;
}
__device__ __forceinline__ void gx2_gxy_h(uint32_t g, float& gx2, float& gxy) {
    asm("{ .reg .f16 a, b;\n\tmov.b32 {a, b}, %2;\n\tfma.rn.f32.f16 %0, a, a, 0f00000000;\n\tfma.rn.f32.f16 %1, a, b, 0f00000000; }" : "=f"(gx2), "=f"(gxy) : "r"(g));
}
// floor(sqrt(n))^2 for an exact fp32 integer 0 <= n < 2^24: MUFU.SQRT estimate (within 2^-22 relative, i.e. its truncation is off by at
// most one) + one correction in each direction, all in exact fp32 integer arithmetic; == ((int)sqrt((double)n))^2 of src/utils.cpp:212
__device__ __forceinline__ float isqrt_sq_f(float n) {
    float s;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(s) : "f"(n));   // n is 0 or >= 1: nothing to flush, and no denormal scaling around the MUFU
    const float m = __fsub_rn(__fadd_rz(s, 8388608.0f), 8388608.0f);   // trunc(s)
    const float m2 = __fmul_rn(m, m);
    const float up = __fadd_rn(__fmaf_rn(m, 2.0f, m2), 1.0f);         // (m+1)^2
    const float dn = __fadd_rn(__fmaf_rn(m, -2.0f, m2), 1.0f);        // (m-1)^2
    return (m2 > n) ? dn : ((up <= n) ? up : m2);
}

}  // namespace pk
}  // namespace cb
