// EXPERIMENT, NOT BUILT INTO libcanny_b200.so (kept for the record: DESIGN.md section 8, profiles/r02_front4_*_phase_budget.txt).
// Bit-exact in the GPU suite; 4 % more per-SM throughput than front3.cu's kernel when launched alone (0.338 against 0.353 ms per 9
// 4K frames), but one 768-thread CTA per SM leaves no registers for the previous chunk's hysteresis blocks, so the three-stream batch
// pipeline is slower with it (246 against 268 Gpix/s).  To try it again: copy back to canny_edge_b200/csrc/front4.cu, add it to
// build.py's SOURCES and dispatch to launch_front4 in front.cu's launch_front.
//
// front4.cu — the fused front kernel, warp-specialised: u8 gray -> u8 class map (0 / 1 weak / 255 strong) for sm_100a.
//
// Same contract and the same arithmetic as front3.cu (stages 1-3 of the reference's CPU path, src/utils.cpp:26-68,106-187,201-236,
// 248-308 + the two thresholds of :327-340; packed-FP32 blur with separately rounded products and sums, exact half-precision Sobel,
// candidates-only NMS on exact fp32 magnitudes^2).  What changes is WHO does what, after profiles/r02_front3_*: in front3 every
// warp runs the blur phases (bound by the FP32 pipe: two lanes per instruction, one instruction per two cycles) and then the NMS
// phases (integer / latency bound: dependent shared-memory gathers, divergent tails), separated by six CTA-wide barriers per slab;
// the two kinds of work overlap only by the luck of two co-resident CTAs being out of step, and the machine issues on 53 % of its
// cycles.  Here ONE CTA of 20 warps owns an SM and the two kinds of work run concurrently by construction:
//
//   * 4 PRODUCER warps (one per scheduler) blur: row pass and column pass on packed FP32 with runs of 32 outputs per thread (longer
//     runs than front3's 16: fewer products at run ends, fewer loads) — throughput-bound work whose 11 independent accumulator
//     chains per thread keep the FP32 pipe busy from a single warp per scheduler.  They write one slab's Sobel words (half2(v, u) per
//     pixel) into one of TWO buffers.
//   * 16 CONSUMER warps (four per scheduler) do the horizontal Sobel, the magnitude^2 plane, the candidate lists, direction / NMS /
//     thresholds for the candidates and the weak-pixel hand-over of the PREVIOUS slab's buffer — latency-bound work that needs warps
//     to hide its dependent gathers, and that issues in the slots the half-rate packed instructions leave free.
//   * the two groups meet only at two mbarriers per buffer ("full": producers -> consumers, "free": consumers -> producers); inside
//     a group, named barriers (bar.sync id, count) replace __syncthreads().
//
// Shared memory (radius 5): staged input 2 x 11 KB (TMA, mbarrier complete_tx), f32 row-blurred lines 40 KB, Sobel words 2 x 34 KB,
// magnitude^2 plane 33 KB (it can no longer alias the temp rows: they are being refilled), candidate lists 8 KB: 176 KB, one CTA per
// SM, <= 96 registers x 640 threads.
//
// Used for compile-time radii without spill planes; everything else stays on front.cu's kernel.
#include <cuda.h>

#include "canny_math.h"
#include "exact_math.cuh"
#include "front_common.cuh"
#include "front_packed.cuh"
#include "internal.h"

namespace cb {
namespace f4 {

using namespace pk;

#ifndef F4_WARPS_A
#define F4_WARPS_A 8
#endif
#ifndef F4_WARPS_B
#define F4_WARPS_B 16
#endif
constexpr int kWarpsA = F4_WARPS_A, kWarpsB = F4_WARPS_B;
static_assert(kWarpsA == 4 || kWarpsA == 8, "producer mappings: 128 or 256 threads");
constexpr int kThreadsA = 32 * kWarpsA, kThreadsB = 32 * kWarpsB, kThreads = kThreadsA + kThreadsB;
constexpr int kSlab = 64;        // rows per marching step (one TMA box)
constexpr int kTC = 128;         // computed columns per strip (temp / VU lines); column j <-> image x = x0 - 2 + j
constexpr int kTW = kTC - 4;     // class-map columns produced per strip (Sobel + NMS eat 2 per side)
constexpr int kTempPitch = 132;  // floats; == 4 mod 32: the row pass's 128-bit stores (lane = row) hit 8 distinct bank groups
constexpr int kVuPitch = 132;    // words; lane 31 of phase 3a reads 4 words past column 127
constexpr int kVuRows = kSlab + 2;
constexpr int kVuWords = kVuRows * kVuPitch;
constexpr int kNpPitch = 128;    // magnitude^2 plane: (kSlab + 2) rows x 128 floats
constexpr int kRowsPerWarpB = kSlab / kWarpsB;      // class rows a consumer warp owns in phase 3a
constexpr int kEntPerWarp = kRowsPerWarpB * 64;     // at most one 16-bit entry per (class row, lane, pixel pair)
static_assert(kSlab % kWarpsB == 0, "consumer warps share the slab's rows evenly");

__host__ __device__ constexpr int in_pitch_for(int radius) {
    // bytes per staged input row: up to 15 leading bytes (the TMA box must start on a 16 B boundary of the image row: a tile
    // coordinate that is not a multiple of 16 bytes traps — tools/probes/tma_probe.cu), 128 + 2R needed ones; a multiple of 16
    // (TMA) and an ODD multiple so lane = row 128-bit loads spread over 8 distinct bank groups
    int k = (15 + kTC + 2 * radius + 15) / 16;
    if ((k & 1) == 0) k += 1;
    return 16 * k;
}
__host__ __device__ constexpr int temp_rows_for(int radius) { return 2 * radius + 2 + kSlab; }

struct SmemLayout {
    int in_off, temp_off, vu_off, np_off, ent_off, bits_off, tab_off, w_off, bar_off, total;
};
__host__ __device__ constexpr SmemLayout smem_layout(int radius) {
    SmemLayout L{};
    int o = 0;
    L.in_off = o;   o += 2 * kSlab * in_pitch_for(radius);
    o = (o + 127) & ~127;
    L.temp_off = o; o += temp_rows_for(radius) * kTempPitch * 4;
    L.vu_off = o;   o += 2 * kVuWords * 4;
    L.np_off = o;   o += kVuRows * kNpPitch * 4;
    L.ent_off = o;  o += kWarpsB * kEntPerWarp * 2;
    L.bits_off = o; o += kSlab * 4 * 4;                        // weak-pixel bitmap of the slab's class rows: 4 words per row
    L.tab_off = o;  o += 2 * (radius + 1) * (radius + 1) * 4;  // count table, reciprocal table
    L.w_off = o;    o += (2 * radius + 1) * 4;
    o = (o + 15) & ~15;
    L.bar_off = o;  o += 6 * 8;                                // tma[2], full[2], free[2]
    L.total = o;
    return L;
}

static __device__ __forceinline__ void bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
static __device__ __forceinline__ void mbar_arrive(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
// One thread of a group polls the mbarrier; the others wait at the group's named barrier, where they cost no issue slots (a whole
// group spinning on try_wait took a third of the SM's issue slots from the other group: profiles/r02_front4_spinning_phase_budget.txt).  The
// barrier also carries the acquire: the poller's observation of the phase is ordered before everyone's reads after the barrier.
static __device__ __forceinline__ void group_wait(bool poller, uint32_t bar, uint32_t parity, int bar_id, int n) {
    if (poller) mbar_wait(bar, parity);
    bar_sync(bar_id, n);
}

template <int R, bool USE_TMA, int DIV>
__global__ void __launch_bounds__(kThreads, 1)
front4_kernel(const FrontParams p, const __grid_constant__ CUtensorMap tmap) {
    extern __shared__ __align__(1024) unsigned char smem[];
    static_assert(2 * R + 2 <= kSlab, "the saved tail must not overlap the rows it is copied from");
    constexpr SmemLayout L = smem_layout(R);
    constexpr int in_pitch = in_pitch_for(R);
    constexpr int T0 = 2 * R + 2;  // temp buffer row of the first row of the current slab

    unsigned char* s_in = smem + L.in_off;
    float* s_temp = reinterpret_cast<float*>(smem + L.temp_off);
    int32_t* s_vu = reinterpret_cast<int32_t*>(smem + L.vu_off);
    float* s_np = reinterpret_cast<float*>(smem + L.np_off);
    float* s_cnt = reinterpret_cast<float*>(smem + L.tab_off);
    float* s_rcp = s_cnt + (R + 1) * (R + 1);
    float* s_w = reinterpret_cast<float*>(smem + L.w_off);
    const uint32_t bar_tma = smem_u32(smem + L.bar_off), bar_full = bar_tma + 16, bar_free = bar_tma + 32;
    uint16_t* s_ent = reinterpret_cast<uint16_t*>(smem + L.ent_off);
    uint32_t* s_bits = reinterpret_cast<uint32_t*>(smem + L.bits_off);
    const bool sparse = p.kept_list != nullptr;                  // uniform: also fill parent[] and the weak-pixel list

    const int tid = threadIdx.x;
    const int lane = tid & 31;

    // ---- which strip / band / frame ----
    const int strip = blockIdx.x, band = blockIdx.y, frame = blockIdx.z;
    const int x0 = strip * kTW;
    const int rows_per_band = (p.out_rows + p.tiles_y - 1) / p.tiles_y;
    const int yb = p.out_row0 + band * rows_per_band;
    const int ye = min(p.out_row0 + p.out_rows, yb + rows_per_band);
    if (yb >= ye) return;
    const int W = p.width, H = p.height;
    const int n_slabs = (ye - yb + 2 * R + 4 + kSlab - 1) / kSlab;
    const int in_y0 = yb - 2 - R;                 // global row of slab 0, line 0
    const int lead = (x0 - 2 - R) & 15;           // bytes between the 16 B aligned box origin and the first needed column
    const int in_x0 = x0 - 2 - R - lead;          // global column of staged byte 0 (a multiple of 16, may be negative)

    for (int i = tid; i < (R + 1) * (R + 1); i += kThreads) {
        s_cnt[i] = p.count[i];
        s_rcp[i] = p.count[(R + 1) * (R + 1) + i];
    }
    for (int i = tid; i < 2 * R + 1; i += kThreads) s_w[i] = p.w[i];
    if (tid < 4 * kSlab) s_bits[tid] = 0;
    if (tid == 0) {
#pragma unroll
        for (int b = 0; b < 6; ++b) mbar_init(bar_tma + 8 * b, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();   // the last CTA-wide barrier: from here on the two groups only meet at the full / free mbarriers

    // strips that contain image column -1 or W need the virtual Sobel columns patched in (see the patch pass)
    const bool x_edge = (x0 - 2 < 0) || (x0 - 2 + kTC - 1 >= W);

    if (tid < kThreadsA) {
        // =====================================================================================================================
        // PRODUCERS: staged input -> f32 row-blurred lines -> Sobel words of slab k in buffer k & 1
        // =====================================================================================================================
        const int warp = tid >> 5;
        u64 ws2[R + 1];
#pragma unroll
        for (int j = 0; j <= R; ++j) ws2[j] = pack2(s_w[R + j], s_w[R + j]);
        const float cnt_full = s_cnt[0], rcp_full = s_rcp[0];
        const u64 ncnt2 = pack2(-cnt_full, -cnt_full), rcp2 = pack2(rcp_full, rcp_full), divc2 = pack2(p.div_c, p.div_c);
        const u64 kBias2 = pack2(8388608.0f, 8388608.0f), kNegBias2 = pack2(-8388608.0f, -8388608.0f);
        const u64 kTwo2 = pack2(2.0f, 2.0f), kNegOne2 = pack2(-1.0f, -1.0f);
        // strips whose every computed column has all its taps inside the image divide by the constant count
        const bool x_interior = (x0 - 2 - R >= 0) && (x0 - 2 + kTC - 1 + R <= W - 1);
        const uint8_t* in_frame = p.in + (long long)frame * p.in_frame_stride;
        constexpr uint32_t slab_bytes = (uint32_t)(kSlab * in_pitch);
        constexpr int kSegPairs = kThreadsA / kSlab;        // segment pairs per row in the row pass: 64 rows x 2 (or 4) = the producer threads
        constexpr int kRunRow = (kTC / 2) / kSegPairs;      // outputs per thread and segment: 32 (or 16)
        constexpr int kGroups = kThreadsA / (kTC / 2);      // row groups in the column pass: 64 column pairs x 2 (or 4) = the producer threads
        constexpr int kRunV = kSlab / kGroups;              // Sobel (VU) rows per thread: 32 (or 16)
        constexpr int kRunCol = kRunV + 2;         // ... which need two more blurred rows

        auto issue_slab = [&](int k) {
            const int gy = in_y0 + k * kSlab;
            unsigned char* dst = s_in + (k & 1) * slab_bytes;
            if (USE_TMA) {
                if (tid == 0) {
                    const uint32_t bar = bar_tma + 8 * (k & 1);
                    mbar_expect_tx(bar, slab_bytes);
                    tma_load_3d(smem_u32(dst), &tmap, bar, in_x0, gy - p.in_row0, frame);
                }
            } else {
                // generic staging (image pitch not a multiple of 16 B): byte loads, zero outside the image / buffer
                for (int i = tid; i < kSlab * in_pitch; i += kThreadsA) {
                    const int r = i / in_pitch, c = i - r * in_pitch;
                    const int y = gy + r, x = in_x0 + c;
                    const int by = y - p.in_row0;
                    unsigned char v = 0;
                    if (y >= 0 && y < H && by >= 0 && by < p.in_rows && x >= 0 && x < W) v = in_frame[(long long)by * W + x];
                    dst[i] = v;
                }
            }
        };
        if (USE_TMA) {
            issue_slab(0);
            if (n_slabs > 1) issue_slab(1);
        }

        for (int k = 0; k < n_slabs; ++k) {
            const int I_k = in_y0 + k * kSlab;  // global row of this slab's first input line
            if (USE_TMA) {
                group_wait(tid == 0, bar_tma + 8 * (k & 1), (uint32_t)((k >> 1) & 1), 1, kThreadsA);
            } else {
                issue_slab(k);
                bar_sync(1, kThreadsA);
            }
            const unsigned char* slab = s_in + (k & 1) * slab_bytes;
            int32_t* vu_k = s_vu + (k & 1) * kVuWords;

            // ===================== phase 1: row blur, u8 -> f32 (src/utils.cpp:37-49), two column segments per thread ==================
            // thread = (slab row 32*(warp>>1) + lane, columns 32*sp .. +31 AND 64 + 32*sp .. +31, sp = warp & 1).  A pair = {column c,
            // column c + 64} of the row, and that is also how the temp buffer keeps a line: float 2c <-> column c, float 2c+1 <->
            // column c + 64 (c < 64), so two outputs are one 128-bit store and the column pass loads a pair as one 64-bit word.
            {
                const int srow = 32 * (warp / kSegPairs) + lane;
                const int sp = warp % kSegPairs;
                // needed bytes of a segment: [32*seg + lead, 32*seg + lead + 32 + 2R).  lead = 4*dq + DR with DR a compile-time
                // constant (x0 is a multiple of 4) and dq uniform over the CTA: load aligned 128-bit vectors, shift by dq WORDS with a
                // uniform switch, pick bytes with static selectors.
                constexpr int DR = (((-2 - R) % 4) + 4) % 4;
                constexpr int KW = (DR + kRunRow + 2 * R + 3) / 4;   // words holding the needed bytes
                constexpr int NV = (KW + 3 + 3) / 4;                 // vectors covering KW + 3 words
                static_assert(kTC / 2 + kRunRow + 16 * NV <= in_pitch, "row pass would read past the staged line");
                uint32_t va[NV * 4], vb[NV * 4];
                const uint4* src_a = reinterpret_cast<const uint4*>(slab + srow * in_pitch + sp * kRunRow);
                const uint4* src_b = reinterpret_cast<const uint4*>(slab + srow * in_pitch + sp * kRunRow + kTC / 2);
#pragma unroll
                for (int v = 0; v < NV; ++v) {
                    const uint4 ta = src_a[v], tb = src_b[v];
                    va[4 * v + 0] = ta.x; va[4 * v + 1] = ta.y; va[4 * v + 2] = ta.z; va[4 * v + 3] = ta.w;
                    vb[4 * v + 0] = tb.x; vb[4 * v + 1] = tb.y; vb[4 * v + 2] = tb.z; vb[4 * v + 3] = tb.w;
                }
                uint32_t wa[KW], wb[KW];
                switch (lead >> 2) {
                    case 0:
#pragma unroll
                        for (int q = 0; q < KW; ++q) { wa[q] = va[q]; wb[q] = vb[q]; }
                        break;
                    case 1:
#pragma unroll
                        for (int q = 0; q < KW; ++q) { wa[q] = va[q + 1]; wb[q] = vb[q + 1]; }
                        break;
                    case 2:
#pragma unroll
                        for (int q = 0; q < KW; ++q) { wa[q] = va[q + 2]; wb[q] = vb[q + 2]; }
                        break;
                    default:
#pragma unroll
                        for (int q = 0; q < KW; ++q) { wa[q] = va[q + 3]; wb[q] = vb[q + 3]; }
                        break;
                }
                float* trow = s_temp + (T0 + srow) * kTempPitch + 2 * sp * kRunRow;   // interleaved line: output o of the pair at floats 2o, 2o+1
                int gx_first = x0 - 2 + sp * kRunRow;   // image column of output 0 of the first segment (the second: + 64)
                asm volatile("" : "+r"(gx_first));      // keeps the border strips' table indices from being hoisted out of the slab loop (registers)
                auto fetch = [&](int i) {
                    // {byte, 0, 0, 0x4B} = 2^23 + byte for both columns, then ONE packed subtraction of 2^23
                    const uint32_t sel = 0x7650 + ((i + DR) & 3);
                    const uint32_t ba = __byte_perm(wa[(i + DR) >> 2], 0x4B000000u, sel);
                    const uint32_t bb = __byte_perm(wb[(i + DR) >> 2], 0x4B000000u, sel);
                    return add2(pack2(__uint_as_float(ba), __uint_as_float(bb)), kNegBias2);
                };
                u64 prev = 0;
                // two straight-line copies: the WARP-uniform choice of the division is made once, not inside the unrolled run.  Only the
                // warps whose two segments touch the image border take the per-column weight sums.
                const bool seg_interior = x_interior || ((gx_first - R >= 0) && (gx_first + kTC / 2 + kRunRow - 1 + R <= W - 1));
                if (seg_interior) {
                    blur_run2<R, kRunRow>(ws2, fetch, [&](int o, u64 sum) {
                        const u64 q = div_const2<DIV>(sum, ncnt2, rcp2, divc2);      // divide by the weight sum (src/utils.cpp:47)
                        if (o & 1) {
                            float a0, a1, b0, b1;
                            unpack2(prev, a0, a1);
                            unpack2(q, b0, b1);
                            *reinterpret_cast<float4*>(trow + 2 * (o - 1)) = make_float4(a0, a1, b0, b1);
                        }
                        prev = q;
                    });
                } else {
                    blur_run2<R, kRunRow>(ws2, fetch, [&](int o, u64 sum) {
                        // strips at the left / right image border: per-column in-image weight sums
                        float r01[2];
                        unpack2(sum, r01[0], r01[1]);
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const int gx = gx_first + o + e * (kTC / 2);
                            if (gx < 0 || gx >= W) { r01[e] = 0.f; continue; }
                            const int ta = max(0, R - gx), tb = max(0, gx + R - (W - 1));
                            const int ti = ta * (R + 1) + tb;
                            r01[e] = div_exact(r01[e], s_cnt[ti], s_rcp[ti]);
                        }
                        const u64 q = pack2(r01[0], r01[1]);
                        if (o & 1) {
                            float a0, a1;
                            unpack2(prev, a0, a1);
                            *reinterpret_cast<float4*>(trow + 2 * (o - 1)) = make_float4(a0, a1, r01[0], r01[1]);
                        }
                        prev = q;
                    });
                }
            }
            bar_sync(1, kThreadsA);  // (A) this slab's temp lines are complete; staged buffer k&1 is free again
            if (USE_TMA && k + 2 < n_slabs) issue_slab(k + 2);
            // the consumers have finished with this buffer's previous slab (k - 2)
            if (k >= 2) group_wait(tid == 0, bar_free + 8 * (k & 1), (uint32_t)(((k >> 1) - 1) & 1), 1, kThreadsA);
            // VU rows 64, 65 of the previous slab (blurred-row neighbours of this slab's first class rows) -> rows 0, 1 of this buffer
            if (k > 0) {
                const int32_t* prev_vu = s_vu + ((k - 1) & 1) * kVuWords + kSlab * kVuPitch;
                for (int i = tid; i < 2 * kTC; i += kThreadsA) vu_k[(i >> 7) * kVuPitch + (i & 127)] = prev_vu[(i >> 7) * kVuPitch + (i & 127)];
            }

            // ===================== phase 2: column blur f32 -> int (src/utils.cpp:52-64) + vertical half of Sobel, two columns per thread =
            // thread = (columns c = tid&63 and c + 64; row group tid>>6).  Blurred rows Bg(o) = I_k - R - 2 + 32*group + o, o = 0..33, from
            // temp buffer rows 32*group + o .. + 2R; VU rows Bg(1..32) go to VU buffer rows 2 + 32*group + (o-2).  A pair = the two columns,
            // one 64-bit word of the interleaved temp line.
            {
                const int c = tid & 63;
                const int group = tid >> 6;
                const float* tcol = s_temp + (kRunV * group) * kTempPitch + 2 * c;
                uint32_t* vcol = reinterpret_cast<uint32_t*>(vu_k) + (2 + kRunV * group) * kVuPitch + c;
                const int bg0 = I_k - R - 2 + kRunV * group;  // global row of blurred output 0
                // interior run: every blurred row has all 2R+1 taps inside the image, and every VU row has both vertical neighbours
                const bool y_interior = (bg0 - R >= 0) && (bg0 + kRunCol - 1 + R <= H - 1);
                if (y_interior) {
                    u64 b0 = 0, b1 = 0;  // blurred values (exact integers in fp32) of rows o-2, o-1, both columns
                    blur_run2<R, kRunCol>(
                        ws2, [&](int i) { return *reinterpret_cast<const u64*>(tcol + i * kTempPitch); },
                        [&](int o, u64 sum) {
                            // (short)(sum / count) of src/utils.cpp:62: adding 2^23 toward zero leaves 2^23 + trunc(q); subtracting it
                            // again (exact) gives trunc(q) as a float
                            const u64 b2 = add2(add2_rz(div_const2<DIV>(sum, ncnt2, rcp2, divc2), kBias2), kNegBias2);
                            if (o >= 2) {
                                float v0, v1, u0, u1;
                                unpack2(add2(fma2(b1, kTwo2, b0), b2), v0, v1);   // B[r-1] + 2 B[r] + B[r+1]
                                unpack2(fma2(b0, kNegOne2, b2), u0, u1);          // B[r+1] - B[r-1]
                                vcol[(o - 2) * kVuPitch] = pack_half2(v0, u0);
                                vcol[(o - 2) * kVuPitch + kTC / 2] = pack_half2(v1, u1);
                            }
                            b0 = b1; b1 = b2;
                        });
                } else {
                    // border run (first / last slabs of the image only): a compact loop — direct 2R+1-tap sums per output, per-row counts,
                    // rows outside the image, replicate / drop rules of src/utils.cpp:117-184.  Same products and sums, same order.
                    float pm[2] = {0.f, 0.f}, pc[2] = {0.f, 0.f};
#pragma unroll 1
                    for (int o = 0; o < kRunCol; ++o) {
                        u64 sum = 0;
#pragma unroll
                        for (int t = 0; t <= 2 * R; ++t) {
                            const u64 q = mul2_ftz(*reinterpret_cast<const u64*>(tcol + (o + t) * kTempPitch), ws2[t < R ? R - t : t - R]);
                            sum = (t == 0) ? q : add2(sum, q);
                        }
                        const int gy = bg0 + o;
                        float s01[2], cur[2] = {0.f, 0.f};
                        unpack2(sum, s01[0], s01[1]);
                        if (gy >= 0 && gy < H) {
                            const int ta = max(0, R - gy), tb = max(0, gy + R - (H - 1));
                            const int ti = ta * (R + 1) + tb;
#pragma unroll
                            for (int e = 0; e < 2; ++e)
                                cur[e] = __fsub_rn(__fadd_rz(div_exact(s01[e], s_cnt[ti], s_rcp[ti]), 8388608.0f), 8388608.0f);
                        }
                        if (o >= 2) {
                            const int r = gy - 1;  // the VU row: blurred rows r-1 (pm), r (pc), r+1 (cur)
                            uint32_t word[2] = {0u, 0u};
                            if (r >= 0 && r < H) {
#pragma unroll
                                for (int e = 0; e < 2; ++e) {
                                    const float up = (r > 0) ? pm[e] : pc[e], dn = (r < H - 1) ? cur[e] : pc[e];        // vertical replicate (gy term)
                                    const float u = dn - up;
                                    const float v = 2.f * pc[e] + ((r > 0) ? pm[e] : 0.f) + ((r < H - 1) ? cur[e] : 0.f);  // vertical drop (gx term)
                                    word[e] = pack_half2(v, u);
                                }
                            }
                            vcol[(o - 2) * kVuPitch] = word[0];
                            vcol[(o - 2) * kVuPitch + kTC / 2] = word[1];
                        }
                        pm[0] = pc[0]; pm[1] = pc[1]; pc[0] = cur[0]; pc[1] = cur[1];
                    }
                }
            }
            bar_sync(1, kThreadsA);  // (B) VU rows 2..65 complete; every read of the temp buffer is done

            // keep the last 2R+2 temp lines for the next slab (rows 64.. -> rows 0..): disjoint source / destination
            if (k + 1 < n_slabs) {
                constexpr int n4 = T0 * (kTC / 4);
                for (int i = tid; i < n4; i += kThreadsA) {
                    const int r = i / (kTC / 4), q = i - r * (kTC / 4);
                    reinterpret_cast<float4*>(s_temp + r * kTempPitch)[q] = reinterpret_cast<const float4*>(s_temp + (kSlab + r) * kTempPitch)[q];
                }
            }
            // strips that contain image column -1 or W: the reference replicates horizontally for gx and drops for gy
            // (src/utils.cpp:117-147 vs :158-184).  gx only reads the v half of a neighbour word and gy only the u half, so ONE
            // virtual word {v = v[edge], u = 0} in the out-of-image column serves both.  (Rows 0, 1 were patched in the previous slab.)
            if (x_edge) {
                for (int r = tid; r < kSlab; r += kThreadsA) {
                    int32_t* row = vu_k + (2 + r) * kVuPitch;
                    if (x0 - 2 < 0) row[1] = row[2] & 0xFFFF;                       // x0 == 0: column j=1 is x=-1, j=2 is x=0
                    const int jw = W - (x0 - 2);                                    // column index of image x = W
                    if (jw >= 1 && jw < kTC) row[jw] = row[jw - 1] & 0xFFFF;
                }
            }
            bar_sync(1, kThreadsA);  // (B2) temp tail saved, virtual columns patched: VU rows 0..65 of this buffer are final
            if (tid == 0) mbar_arrive(bar_full + 8 * (k & 1));
        }
    } else {
        // =====================================================================================================================
        // CONSUMERS: Sobel words of slab k -> magnitude^2 plane + candidate lists -> class bytes + weak-pixel hand-over
        // =====================================================================================================================
        const int tb = tid - kThreadsA;
        const int warp = tb >> 5;      // 0 .. kWarpsB-1
        const float lo2f = (float)p.lo2, hi2f = (float)p.hi2;   // thresholds on the exact fp32 magnitude^2 (n < 2^22; INT_MAX rounds to 2^31: never reached)

        // weak-pixel list entries of the previous slab, waiting for their reservation (see the end of the loop body)
        uint32_t pend_bits = 0;
        unsigned int pend_base = 0;
        int pend_off = 0, pend_g0 = 0;
        auto flush_pending = [&]() {
            const unsigned int base = __shfl_sync(0xffffffffu, pend_base, 0);
            uint32_t* dst = p.kept_list + base + pend_off;
            uint32_t m = pend_bits;
            while (m) {
                const int b = __ffs(m) - 1;
                m &= m - 1;
                *dst++ = (uint32_t)(pend_g0 + b);
            }
            pend_bits = 0;
        };

        for (int k = 0; k < n_slabs; ++k) {
            const int I_k = in_y0 + k * kSlab;
            const int32_t* vu_k = s_vu + (k & 1) * kVuWords;
            group_wait(tb == 0, bar_full + 8 * (k & 1), (uint32_t)((k >> 1) & 1), 2, kThreadsB);
            // the previous slab's list entries: their reservation (a global atomic) has had the whole wait to come back
            if (sparse) flush_pending();

            // ===================== phase 3a: horizontal half of Sobel, magnitude^2 plane, candidate lists =====================
            // n-plane row q (0..65) <-> VU buffer row q <-> global row y_base + q - 1.
            // thread = columns j = 4*lane + 1 + e (e = 0..3) of one row; n[j] is stored at word j-1 so the store is one aligned
            // 128-bit write.  Class pixels are j = 2..125 of the class rows.  A thread with a candidate (n >= minVal^2) among its
            // four pixels appends ONE 16-bit entry {row, lane} to its WARP's list (no atomics: the count is a warp-uniform
            // register); phase 3b lets every warp work through its own list with all lanes busy.
            const int y_base = I_k - R - 2;                           // global row of class row rr = 0 (n-plane row 1)
            int my_count = 0;                                         // entries in this warp's list (uniform over the warp)
            uint16_t* my_ent = s_ent + warp * kEntPerWarp;
            // class rows of this slab: n-plane rows cq_lo..cq_hi (always inside the image); the rows just above and below
            // them are neighbour-only rows and may lie outside the image
            const int cq_lo = max(1, yb - y_base + 1), cq_hi = min(kSlab, ye - y_base);
            {
                auto n_of_row = [&](const int32_t* vrow) -> float4 {
                    const uint4 qa = *reinterpret_cast<const uint4*>(vrow);
                    const uint2 qb = *reinterpret_cast<const uint2*>(vrow + 4);
                    const uint32_t wd[6] = {qa.x, qa.y, qa.z, qa.w, qb.x, qb.y};
                    float nv[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) nv[e] = norm2_h(sobel_h(wd[e], wd[e + 1], wd[e + 2]));   // gx^2 + gy^2, exact
                    if (x_edge) {                                 // uniform: columns outside the image never suppress (src/utils.cpp:253-304)
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const int x = x0 - 2 + 4 * lane + 1 + e;
                            if (x < 0 || x >= W) nv[e] = -1.f;
                        }
                    }
                    return make_float4(nv[0], nv[1], nv[2], nv[3]);
                };
                if (cq_lo <= cq_hi) {
                    // the two neighbour-only rows: the last two warps (the first ones get the ragged rows of a partial slab)
                    if (warp >= kWarpsB - 2) {
                        const int q = warp == kWarpsB - 2 ? cq_lo - 1 : cq_hi + 1;
                        const int y = y_base + q - 1;
                        float4 nq = make_float4(-1.f, -1.f, -1.f, -1.f);      // rows outside the image never suppress
                        if (y >= 0 && y < H) nq = n_of_row(vu_k + q * kVuPitch + 4 * lane);
                        *reinterpret_cast<float4*>(s_np + q * kNpPitch + 4 * lane) = nq;
                    }
                    const uint32_t zero_word = 0x01010101u * (uint32_t)p.cls_zero;
                    const bool word_ok = ((W & 3) == 0) && lane < kTW / 4 && (x0 + 4 * lane + 3 < W);  // the aligned 32-bit store applies
                    const bool tail_ok = !word_ok && lane < kTW / 4 && (x0 + 4 * lane < W);            // ragged right edge: byte stores
                    const unsigned lt_mask = (1u << lane) - 1u;
                    int q = cq_lo + ((warp - cq_lo) & (kWarpsB - 1));         // first class row of this warp (rows q = warp mod 16)
                    const int32_t* vrow = vu_k + q * kVuPitch + 4 * lane;
                    float* nrow = s_np + q * kNpPitch + 4 * lane;
                    uint8_t* o = p.cls + (long long)frame * p.out_frame_stride + (long long)(y_base + q - 1 - p.plane_row0) * W + (x0 + 4 * lane);
                    int ent = ((q - 1) << 6) | (lane << 1);
                    const long long o_step = (long long)kWarpsB * W;
                    auto class_row = [&](const int32_t* vr, float* nr, int e16) {
                        const float4 nq = n_of_row(vr);
                        *reinterpret_cast<float4*>(nr) = nq;
                        // one entry per PAIR of pixels (columns 4*lane+1.. +2 and 4*lane+3.. +4) that holds a candidate: candidates
                        // come in bands a few pixels wide, so pairs leave fewer idle pixel slots in phase 3b than whole quads
                        const bool any_lo = fmaxf(nq.x, nq.y) >= lo2f, any_hi = fmaxf(nq.z, nq.w) >= lo2f;
                        const unsigned vote_lo = __ballot_sync(0xffffffffu, any_lo), vote_hi = __ballot_sync(0xffffffffu, any_hi);
                        const int n_lo = __popc(vote_lo);
                        if (any_lo) my_ent[my_count + __popc(vote_lo & lt_mask)] = (uint16_t)e16;
                        if (any_hi) my_ent[my_count + n_lo + __popc(vote_hi & lt_mask)] = (uint16_t)(e16 | 1);
                        my_count += n_lo + __popc(vote_hi);
                    };
                    // every class word starts out as "suppressed"; phase 3b overwrites the bytes of surviving pixels
                    if (cq_lo == 1 && cq_hi == kSlab && ((W & 3) == 0)) {
                        // the common slab (all 64 class rows, image width a multiple of 4): the warp's rows unrolled, every address an
                        // immediate offset from the first row's (word_ok is false for the columns past a ragged right edge)
#pragma unroll
                        for (int i = 0; i < kRowsPerWarpB; ++i) {
                            class_row(vrow + kWarpsB * i * kVuPitch, nrow + kWarpsB * i * kNpPitch, ent + ((kWarpsB * i) << 6));
                            if (word_ok) *reinterpret_cast<uint32_t*>(o + i * o_step) = zero_word;
                        }
                    } else {
                        for (; q <= cq_hi; q += kWarpsB, vrow += kWarpsB * kVuPitch, nrow += kWarpsB * kNpPitch, o += o_step, ent += kWarpsB << 6) {
                            class_row(vrow, nrow, ent);
                            if (word_ok) {
                                *reinterpret_cast<uint32_t*>(o) = zero_word;
                            } else if (tail_ok) {
                                for (int e = 0; e < 4 && x0 + 4 * lane + e < W; ++e) o[e] = (uint8_t)p.cls_zero;
                            }
                        }
                    }
                }
            }
            bar_sync(2, kThreadsB);  // (C1) n-plane complete; the zero words are ordered before phase 3b's byte stores

            // ===================== phase 3b: direction, NMS and thresholds for the candidates only =====================
            {
                const long long out_off = (long long)frame * p.out_frame_stride + (long long)(y_base - p.plane_row0) * W + (x0 - 2) + 1;
                uint8_t* out_base = p.cls + out_off;
                int32_t* par_base = p.parent + out_off;                           // only dereferenced when `sparse`
                const int idx_base = (int)out_off;                                // launch-relative pixel index of (class row 0, column j = 1)
                for (int i = lane; i < my_count; i += 32) {
                    const int ent = my_ent[i];
                    const int rr = ent >> 6, c0 = 2 * (ent & 63);              // pixels j = c0 + 1 and c0 + 2 of class row rr
                    const int32_t* vrow = vu_k + (rr + 1) * kVuPitch + c0;     // VU words j-1 .. j+2 = c0 .. c0+3
                    const uint2 qa = *reinterpret_cast<const uint2*>(vrow);
                    const uint2 qb = *reinterpret_cast<const uint2*>(vrow + 2);
                    const uint32_t wd[4] = {qa.x, qa.y, qb.x, qb.y};
                    const float* nrow = s_np + (rr + 1) * kNpPitch + c0;       // n[j] lives at word j - 1
                    const float2 n2 = *reinterpret_cast<const float2*>(nrow);
                    const float nc[2] = {n2.x, n2.y};
                    uint8_t* orow = out_base + (long long)rr * W + c0;
                    // branch-free up to the local-maximum test so the two pixels' chains overlap
                    float na[2], nb[2];
                    bool pass[2];
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const float n = nc[e];
                        float gx2, pxy;
                        gx2_gxy_h(sobel_h(wd[e], wd[e + 1], wd[e + 2]), gx2, pxy);
                        // direction_code() of canny_math.h in product form (same integer tests as src/utils.cpp:215-231's bins), on
                        // exact fp32 integers:
                        //   0   <=> (ay+ax)^2 < 2ax^2           <=> ax^2 - ay^2 > 2 ax ay
                        //   90  <=> ay > ax and (ay-ax)^2 > 2ax^2 <=> ay^2 - ax^2 > 2 ax ay
                        //   else a diagonal: 45 when gx and gy have the same sign (gx*gy > 0; both are non-zero there).
                        // gx = gy = 0 lands on "45" instead of 0, which cannot change the class: such a pixel is a candidate only when
                        // minVal <= 0, and then kept and suppressed pixels get the same class (see fill_thresholds()).
                        const float dd = __fmaf_rn(gx2, 2.0f, -n);   // ax^2 - ay^2  (n = ax^2 + ay^2)
                        const float p2 = 2.0f * fabsf(pxy);
                        const bool is0 = dd > p2;
                        const bool is90 = -dd > p2;
                        const bool same = pxy >= 0.f;
                        // neighbour pair along the quantised direction (src/utils.cpp:253-304); out-of-image neighbours hold -1
                        const int off = is0 ? 1 : (is90 ? kNpPitch : (same ? (1 - kNpPitch) : (1 + kNpPitch)));
                        na[e] = nrow[e + off];
                        nb[e] = nrow[e - off];
                        const int j = c0 + 1 + e;
                        pass[e] = (n >= lo2f) && (j >= 2) && (j <= kTC - 3) && (na[e] < n) && (nb[e] < n);   // j = 1, j >= 126: neighbour-only columns
                    }
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        if (pass[e]) {
                            // the reference compares truncated magnitudes: keep iff floor(sqrt(n_nb)) < floor(sqrt(n)) <=> n_nb < mag^2
                            const float n = nc[e];
                            const float m2 = isqrt_sq_f(n);
                            if (na[e] < m2 && nb[e] < m2) {
                                const bool strong = n >= hi2f;
                                orow[e] = strong ? (uint8_t)255 : (uint8_t)1;
                                if (sparse && !strong) {
                                    // hand-over to the list-driven hysteresis kernels: only WEAK pixels need any work there (a strong
                                    // pixel is final; its neighbours find it through the class map).  The weak pixel gets its union-
                                    // find slot (itself) and a bit in the slab's bitmap, from which the list entries are made once
                                    // the slab is finished
                                    const int rel = rr * W + c0 + e;
                                    par_base[rel] = idx_base + rel;
                                    const int col = c0 + e - 1;                   // class column within the strip: j - 2
                                    atomicOr(&s_bits[rr * 4 + (col >> 5)], 1u << (col & 31));
                                }
                            }
                        }
                    }
                }
            }
            bar_sync(2, kThreadsB);  // (C) VU, n-plane and list reads done; the slab's weak-pixel bitmap is complete
            if (tb == 0) mbar_arrive(bar_free + 8 * (k & 1));   // the producers may refill this buffer (slab k + 2)
            if (sparse && warp < (4 * kSlab) / 32) {
                // append this slab's weak pixels to the launch-wide list: every warp that owns bitmap words counts their bits and
                // reserves room with ONE global atomicAdd.  The atomic's round trip is hidden behind the wait for the next slab: the
                // entries are written by flush_pending() after it (and once more after the last slab).
                pend_bits = s_bits[tb];
                s_bits[tb] = 0;
                const int cnt = __popc(pend_bits);
                int incl = cnt;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const int t = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= d) incl += t;
                }
                const int total = __shfl_sync(0xffffffffu, incl, 31);
                pend_base = 0;
                if (total && lane == 0) pend_base = atomicAdd(p.kept_count, (unsigned int)total);
                pend_off = incl - cnt;
                // word tb <-> class row rr = tb >> 2, columns 32*(tb & 3) .. of the strip
                pend_g0 = (int)((long long)frame * p.out_frame_stride + (long long)(y_base + (tb >> 2) - p.plane_row0) * W + x0 + 32 * (tb & 3));
            }
        }
        if (sparse) flush_pending();
    }
}

}  // namespace f4

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
template <int R, bool USE_TMA, int DIV>
static int launch_one4(b200_ctx* ctx, cudaStream_t st, const FrontParams& p, const CUtensorMap& tmap, dim3 grid) {
    const f4::SmemLayout L = f4::smem_layout(R);
    static bool configured[64] = {false};  // per instantiation, per device
    if (!configured[ctx->device & 63]) {
        CB_CUDA(cudaFuncSetAttribute(f4::front4_kernel<R, USE_TMA, DIV>, cudaFuncAttributeMaxDynamicSharedMemorySize, L.total));
        CB_CUDA(cudaFuncSetAttribute(f4::front4_kernel<R, USE_TMA, DIV>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
        configured[ctx->device & 63] = true;
    }
    {
        ProfScope ps(ctx, st, 0);
        f4::front4_kernel<R, USE_TMA, DIV><<<grid, f4::kThreads, L.total, st>>>(p, tmap);
    }
    CB_CUDA(cudaGetLastError());
    ctx->launches++;
    return B200_OK;
}

template <int R>
static int launch_r4(b200_ctx* ctx, cudaStream_t st, const FrontParams& p, const CUtensorMap& tmap, dim3 grid, bool use_tma, int div) {
    if (use_tma) {
        if (div == 1) return launch_one4<R, true, 1>(ctx, st, p, tmap, grid);
        if (div == 3) return launch_one4<R, true, 3>(ctx, st, p, tmap, grid);
        return launch_one4<R, true, 5>(ctx, st, p, tmap, grid);
    }
    // generic staging (odd widths) is not a throughput path: one instantiation, the always-valid division
    return launch_one4<R, false, 5>(ctx, st, p, tmap, grid);
}

bool front4_supports(int radius) {
    switch (radius) {
        case 2: case 3: case 5: case 6: case 9: case 15: return true;
        default: return false;
    }
}

// Bands per frame: every band pays 2R+4 warm-up rows and is processed in 64-row slabs, so pick the band count that minimises
// (slabs per band) x (waves of CTAs) — enough CTAs to fill the machine (ONE CTA per SM), few enough that the warm-up and the last
// partly-filled slab stay small.
static int choose_bands4(const b200_ctx* ctx, int out_rows, int strips, int frames, int radius) {
    const int slots = ctx->sm_count > 0 ? ctx->sm_count : 148;
    const long long per_band = (long long)strips * frames;
    int best = 1;
    double best_cost = 1e300;
    const int max_bands = out_rows / 64 > 0 ? out_rows / 64 : 1;
    for (int b = 1; b <= max_bands && b <= 64; ++b) {
        const int rows = (out_rows + b - 1) / b;
        const int slabs = (rows + 2 * radius + 4 + f4::kSlab - 1) / f4::kSlab;
        const long long ctas = per_band * b;
        const long long waves = (ctas + slots - 1) / slots;
        const double cost = (double)waves * slabs;  // time ~ waves x slabs marched per CTA
        if (cost < best_cost * 0.999) { best_cost = cost; best = b; }
    }
    return best;
}

int launch_front4(b200_ctx* ctx, cudaStream_t st, const FrontParams& p_in) {
    FrontParams p = p_in;
    const int radius = p.radius;
    const int strips = (p.width + f4::kTW - 1) / f4::kTW;
    p.tiles_x = strips;
    if (p.tiles_y <= 0) p.tiles_y = choose_bands4(ctx, p.out_rows, strips, p.n_frames, radius);
    dim3 grid(strips, p.tiles_y, p.n_frames);
    CUtensorMap tmap;
    bool use_tma = false;
    CB_TRY(make_input_tensor_map(p, f4::in_pitch_for(radius), f4::kSlab, &tmap, &use_tma));
    const int div3 = ctx->gauss.div_mode;
    p.div_c = ctx->gauss.div_c;
    switch (radius) {
        case 2: return launch_r4<2>(ctx, st, p, tmap, grid, use_tma, div3);
        case 3: return launch_r4<3>(ctx, st, p, tmap, grid, use_tma, div3);
        case 5: return launch_r4<5>(ctx, st, p, tmap, grid, use_tma, div3);
        case 6: return launch_r4<6>(ctx, st, p, tmap, grid, use_tma, div3);
        case 9: return launch_r4<9>(ctx, st, p, tmap, grid, use_tma, div3);
        case 15: return launch_r4<15>(ctx, st, p, tmap, grid, use_tma, div3);
        default: break;
    }
    set_error("front4 kernel not built for radius %d", radius);
    return B200_ERR_UNSUPPORTED;
}

}  // namespace cb
