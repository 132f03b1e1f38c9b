// front_common.cuh — pieces of the front kernels (front.cu: generic / spilling variant, front3.cu: the lean fused variant):
// mbarrier + TMA wrappers, the scalar blur core.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace cb {

// ---------------------------------------------------------------------------------------------
// small PTX wrappers (mbarrier + TMA)
// ---------------------------------------------------------------------------------------------
static __device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
static __device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
static __device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
static __device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a TMA that never lands (bad descriptor) must become an error, not a hung GPU.
static __device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    for (int spin = 0; spin < (1 << 26); ++spin)
        if (mbar_try_wait(bar, parity)) return;
    __trap();
}
static __device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int x, int y, int z) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(x), "r"(y), "r"(z)
        : "memory");
}

// The shared blur core.  S consecutive outputs o = 0..S-1; output o is
//     ((x[o]*w[0] + x[o+1]*w[1]) + ... ) + x[o+2R]*w[2R]          (ascending taps, RN after every op)
// exactly as src/utils.cpp:41-46 / 56-61.  ws[j] = w[R+j] = w[R-j].
template <int R, int S, typename Fetch, typename Emit>
static __device__ __forceinline__ void blur_run(const float (&ws)[R + 1], Fetch fetch, Emit emit) {
    float acc[S];
#pragma unroll
    for (int i = 0; i < S + 2 * R; ++i) {
        const float x = fetch(i);
        float q[R + 1];
#pragma unroll
        for (int j = 0; j <= R; ++j) q[j] = __fmul_rn(x, ws[j]);  // unused ones are dead code
#pragma unroll
        for (int t = 0; t <= 2 * R; ++t) {
            const int o = i - t;
            if (o >= 0 && o < S) {
                const int j = t < R ? R - t : t - R;
                acc[o] = (t == 0) ? q[j] : __fadd_rn(acc[o], q[j]);  // 0 + q == q exactly
            }
        }
        if (i >= 2 * R) emit(i - 2 * R, acc[i - 2 * R]);
    }
}


}  // namespace cb
