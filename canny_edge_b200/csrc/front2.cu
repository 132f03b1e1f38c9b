// front2.cu — the lean fused front kernel: u8 gray -> u8 class map (0 / 1 weak / 255 strong) for sm_100a.
//
// Same contract and the same arithmetic as front.cu's front_kernel (stages 1-3 of the reference's CPU path,
// src/utils.cpp:26-68,106-187,201-236,248-308 + the two thresholds of :327-340), restructured so that the
// per-pixel instruction count is close to the arithmetic the reference's rounding order makes unavoidable
// (profiles/r01_front_opcode_mix.txt: the first kernel spent 76 % of its issue slots on integer addressing,
// predicates and branches).  Differences in structure, not in results:
//
//   * slabs of 64 rows x 128 columns, one TMA box each, double buffered (mbarrier complete_tx);
//   * every intermediate sits in a LINEAR shared-memory buffer whose tail rows are copied to the head once per
//     slab, so all addresses inside the unrolled blur runs are base + compile-time immediate;
//   * runs of 32 outputs per thread (register sliding window, symmetric-weight product sharing);
//   * the column pass also does the vertical half of Sobel in registers and stores ONE packed word per pixel,
//     (u << 16) + v with  v = B[r-1] + 2B[r] + B[r+1]  and  u = B[r+1] - B[r-1],  so the last phase gets
//     gx = v[c+1] - v[c-1] and gy = u[c-1] + 2u[c] + u[c+1] from three packed integer adds;
//   * image borders are handled by uniform (per-CTA / per-run) variants, never per pixel in the hot path;
//   * magnitude^2 is compared against the squared thresholds; direction, the exact integer square root and the
//     neighbour magnitudes are only evaluated for candidate pixels (n >= minVal^2).
//
// Used for compile-time radii without spill planes; everything else (run-time radius, `steps` planes, sigma so
// small that sums approach the subnormal range) stays on front.cu's kernel.
#include <cuda.h>

#include "canny_math.h"
#include "exact_math.cuh"
#include "front_common.cuh"
#include "internal.h"

namespace cb {
namespace f2 {

constexpr int kThreads = 256;
// rows per marching step (one TMA box) is the template parameter SLAB (64; 32 also builds, see launch_front2)
constexpr int kTC = 128;         // computed columns per strip (temp / VU lines); column j <-> image x = x0 - 2 + j
constexpr int kTW = kTC - 4;     // class-map columns produced per strip (Sobel + NMS eat 2 per side)
constexpr int kTempPitch = 132;  // floats; == 4 mod 32: the row pass's 128-bit stores (lane = row) hit 8 distinct bank groups
constexpr int kVuPitch = 132;    // int32 words; lane 31 of the last phase reads 4 words past column 127
// outputs per thread: SLAB/2 in the row pass, SLAB/2 VU rows = SLAB/2 + 2 blurred rows in the column pass

__host__ __device__ constexpr int in_pitch_for(int radius) {
    // bytes per staged input row: up to 15 leading bytes (the TMA box starts on a 16 B boundary of the image
    // row), 128 + 2R needed ones; a multiple of 16 (TMA) and an ODD multiple so lane = row 128-bit loads spread
    // over 8 distinct bank groups
    int k = (15 + kTC + 2 * radius + 15) / 16;
    if ((k & 1) == 0) k += 1;
    return 16 * k;
}
constexpr int kNpPitch = 128;    // n-plane words per row: (SLAB+2) rows x 128 words live in the temp rows phase 1 refills next slab
__host__ __device__ constexpr int temp_rows_for(int radius, int slab) {
    // 2R+2 tail rows + the slab's rows, and enough of them that the n-plane fits behind the tail
    const int need = ((slab + 2) * kNpPitch + kTempPitch - 1) / kTempPitch;
    return 2 * radius + 2 + (need > slab ? need : slab);
}

struct SmemLayout {
    int in_off, temp_off, vu_off, ent_off, bits_off, tab_off, w_off, bar_off, total;
};
// staged input slabs: two (the next slab's TMA is in flight while this one is blurred) unless the wide temp buffer of a large
// radius would then push a CTA past half an SM's shared memory — with one buffer the next slab is requested as soon as the row
// pass has read this one and lands during the column pass and phase 3
__host__ __device__ constexpr int in_bufs_for(int radius) { return radius > 9 ? 1 : 2; }
__host__ __device__ constexpr SmemLayout smem_layout(int radius, int slab) {
    SmemLayout L{};
    int o = 0;
    L.in_off = o;   o += in_bufs_for(radius) * slab * in_pitch_for(radius);
    o = (o + 127) & ~127;
    L.temp_off = o; o += temp_rows_for(radius, slab) * kTempPitch * 4;
    L.vu_off = o;   o += (slab + 2) * kVuPitch * 4;
    L.ent_off = o;  o += slab * 64 * 2;                        // candidate lists: at most one 16-bit entry per (class row, lane, pixel pair)
    L.bits_off = o; o += slab * 4 * 4;                         // weak-pixel bitmap of the slab's class rows: 4 words per row
    L.tab_off = o;  o += 2 * (radius + 1) * (radius + 1) * 4;  // count table, reciprocal table
    L.w_off = o;    o += (2 * radius + 1) * 4;
    o = (o + 15) & ~15;
    L.bar_off = o;  o += 2 * 8;
    L.total = o;
    return L;
}

// RN(a / b) for the interior count: y = RN(1/b), c = RN(1/b - 1).  The 1- and 3-instruction forms are only used when the host
// has checked on the device, for this very b and every float mantissa, that they give the IEEE quotient (check_div_mode_device).
template <int DIV>
__device__ __forceinline__ float div_const(float a, float b, float y, float c) {
    if (DIV == 1) return __fmaf_rn(a, c, a);
    if (DIV == 3) {
        const float q = __fmul_rn(a, y);
        const float r = __fmaf_rn(-b, q, a);
        return __fmaf_rn(r, y, q);
    }
    return div_exact(a, b, y);
}

// (short)(q) of src/utils.cpp:62 for 0 <= q < 2^22 without the conversion pipe: adding 2^23 with round-toward-zero
// leaves 2^23 + trunc(q) exactly, i.e. the integer sits in the low mantissa bits.  Returns 0x4B000000 + trunc(q).
__device__ __forceinline__ int trunc_biased(float q) { return __float_as_int(__fadd_rz(q, 8388608.0f)); }
constexpr int kBias = 0x4B000000;
constexpr int kBias4 = (int)(4u * 0x4B000000u);  // 4 * bias mod 2^32 = 0x2C000000

// Register cap: 96 (no spills at any radius; the kernel takes 128 when left alone).  Two resident CTAs then leave a quarter of the
// register file free, so blocks of the small latency-bound hysteresis kernels of the PREVIOUS chunk (other stream) become
// resident next to them instead of waiting for a front CTA to retire: the front kernel alone gets 1.7 % slower, the chunk
// pipeline 2.3 % faster on the bench frames and 8 % faster on photographic content (112 / 104 / 88 / 80 measured too: 96 wins).
template <int R, bool USE_TMA, int DIV, int SLAB>
__global__ void __maxnreg__(SLAB == 64 ? 96 : 64)
front2_kernel(const FrontParams p, const __grid_constant__ CUtensorMap tmap) {
    extern __shared__ __align__(1024) unsigned char smem[];
    constexpr int kSlab = SLAB;
    constexpr int kRunRow = SLAB / 2;          // outputs per thread in the row pass: (SLAB rows) x (128 / kRunRow segments) = 256 threads
    constexpr int kRunV = SLAB / 2;            // VU rows per thread in the column pass: 128 columns x 2 halves = 256 threads
    constexpr int kRunCol = kRunV + 2;         // ... which need two more blurred rows
    constexpr int kVuRows = SLAB + 2;
    constexpr int kEntPerWarp = (SLAB / 8) * 64;
    static_assert(SLAB == 32 || SLAB == 64, "row/column pass mappings are written for 32- and 64-row slabs");
    static_assert(2 * R + 2 <= SLAB, "the saved tail must not overlap the rows it is copied from");
    constexpr SmemLayout L = smem_layout(R, SLAB);
    constexpr int in_pitch = in_pitch_for(R);
    constexpr int T0 = 2 * R + 2;  // temp buffer row of the first row of the current slab

    unsigned char* s_in = smem + L.in_off;
    float* s_temp = reinterpret_cast<float*>(smem + L.temp_off);
    int32_t* s_vu = reinterpret_cast<int32_t*>(smem + L.vu_off);
    float* s_cnt = reinterpret_cast<float*>(smem + L.tab_off);
    float* s_rcp = s_cnt + (R + 1) * (R + 1);
    float* s_w = reinterpret_cast<float*>(smem + L.w_off);
    const uint32_t bar0 = smem_u32(smem + L.bar_off);
    uint16_t* s_ent = reinterpret_cast<uint16_t*>(smem + L.ent_off);
    uint32_t* s_bits = reinterpret_cast<uint32_t*>(smem + L.bits_off);
    const bool sparse = p.kept_list != nullptr;                  // uniform: also fill parent[] and the weak-pixel list
    int32_t* s_np = reinterpret_cast<int32_t*>(s_temp + T0 * kTempPitch);   // n-plane: the temp rows phase 1 refills next slab

    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;

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
    if (USE_TMA && tid == 0) {
        mbar_init(bar0, 1);
        mbar_init(bar0 + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();

    float ws[R + 1];
#pragma unroll
    for (int j = 0; j <= R; ++j) ws[j] = s_w[R + j];
    const float cnt_full = s_cnt[0], rcp_full = s_rcp[0];
    // strips whose every computed column has all its taps inside the image divide by the constant count
    const bool x_interior = (x0 - 2 - R >= 0) && (x0 - 2 + kTC - 1 + R <= W - 1);
    // strips that contain image column -1 or W need the virtual Sobel columns patched in (see the patch pass)
    const bool x_edge = (x0 - 2 < 0) || (x0 - 2 + kTC - 1 >= W);

    const uint8_t* in_frame = p.in + (long long)frame * p.in_frame_stride;
    constexpr uint32_t slab_bytes = (uint32_t)(kSlab * in_pitch);

    constexpr int kInBufs = in_bufs_for(R);
    auto issue_slab = [&](int k) {
        const int gy = in_y0 + k * kSlab;
        unsigned char* dst = s_in + (k % kInBufs) * slab_bytes;
        if (USE_TMA) {
            if (tid == 0) {
                const uint32_t bar = bar0 + 8 * (k % kInBufs);
                mbar_expect_tx(bar, slab_bytes);
                tma_load_3d(smem_u32(dst), &tmap, bar, in_x0, gy - p.in_row0, frame);
            }
        } else {
            // generic staging (image pitch not a multiple of 16 B): byte loads, zero outside the image / buffer
            for (int i = tid; i < kSlab * in_pitch; i += kThreads) {
                const int r = i / in_pitch, c = i - r * in_pitch;
                const int y = gy + r, x = in_x0 + c;
                const int by = y - p.in_row0;
                unsigned char v = 0;
                if (y >= 0 && y < H && by >= 0 && by < p.in_rows && x >= 0 && x < W) v = in_frame[(long long)by * p.in_pitch + x];
                dst[i] = v;
            }
        }
    };

    if (USE_TMA) {
        issue_slab(0);
        if (kInBufs > 1 && n_slabs > 1) issue_slab(1);
    }

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
        const int I_k = in_y0 + k * kSlab;  // global row of this slab's first input line
        if (USE_TMA) {
            mbar_wait(bar0 + 8 * (k % kInBufs), (uint32_t)((k / kInBufs) & 1));
        } else {
            issue_slab(k);
            __syncthreads();
        }
        const unsigned char* slab = s_in + (k % kInBufs) * slab_bytes;

        // ===================== phase 1: row blur, u8 -> f32 (src/utils.cpp:37-49) =====================
        // thread = (slab row 32*(warp>>2) + lane, 32 columns starting at 32*(warp&3)); temp buffer row T0 + slab row
        {
            constexpr int kSegs = kTC / kRunRow;              // 4 segments of 32 columns (SLAB 64) or 8 of 16 (SLAB 32)
            const int srow = 32 * (warp / kSegs) + lane;
            const int seg = warp % kSegs;
            // needed bytes of this line: [32*seg + lead, 32*seg + lead + 32 + 2R).  lead = 4*dq + DR with DR a compile-time
            // constant (x0 is a multiple of 4) and dq uniform over the CTA: load aligned 128-bit vectors, shift by dq
            // WORDS with a uniform switch, pick bytes with static selectors.
            constexpr int DR = (((-2 - R) % 4) + 4) % 4;
            constexpr int KW = (DR + kRunRow + 2 * R + 3) / 4;   // words holding the needed bytes
            constexpr int NV = (KW + 3 + 3) / 4;                 // vectors covering KW + 3 words
            static_assert((kTC - kRunRow) + 16 * NV <= in_pitch, "row pass would read past the staged line");
            uint32_t wv[NV * 4];
            const uint4* src = reinterpret_cast<const uint4*>(slab + srow * in_pitch + seg * kRunRow);
#pragma unroll
            for (int v = 0; v < NV; ++v) {
                const uint4 t4 = src[v];
                wv[4 * v + 0] = t4.x; wv[4 * v + 1] = t4.y; wv[4 * v + 2] = t4.z; wv[4 * v + 3] = t4.w;
            }
            uint32_t w2[KW];
            switch (lead >> 2) {
                case 0:
#pragma unroll
                    for (int q = 0; q < KW; ++q) w2[q] = wv[q];
                    break;
                case 1:
#pragma unroll
                    for (int q = 0; q < KW; ++q) w2[q] = wv[q + 1];
                    break;
                case 2:
#pragma unroll
                    for (int q = 0; q < KW; ++q) w2[q] = wv[q + 2];
                    break;
                default:
#pragma unroll
                    for (int q = 0; q < KW; ++q) w2[q] = wv[q + 3];
                    break;
            }
            float* trow = s_temp + (T0 + srow) * kTempPitch + seg * kRunRow;
            const int gx_first = x0 - 2 + seg * kRunRow;  // image column of output 0
            float grp[4];
            blur_run<R, kRunRow>(
                ws,
                [&](int i) {
                    const uint32_t word = w2[(i + DR) >> 2];
                    const uint32_t bits = __byte_perm(word, 0x4B000000u, 0x7650 + ((i + DR) & 3));  // {byte, 0, 0, 0x4B} = 2^23 + byte
                    return __fsub_rn(__uint_as_float(bits), 8388608.0f);
                },
                [&](int o, float s) {
                    grp[o & 3] = s;
                    if ((o & 3) == 3) {
                        // divide by the in-image weight sum (src/utils.cpp:47) and store four outputs
                        if (x_interior) {
#pragma unroll
                            for (int e = 0; e < 4; ++e) grp[e] = div_const<DIV>(grp[e], cnt_full, rcp_full, p.div_c);
                        } else {
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                const int gx = gx_first + (o - 3) + e;
                                if (gx < 0 || gx >= W) { grp[e] = 0.f; continue; }
                                const int a = max(0, R - gx), b = max(0, gx + R - (W - 1));
                                const int ti = a * (R + 1) + b;
                                grp[e] = div_exact(grp[e], s_cnt[ti], s_rcp[ti]);
                            }
                        }
                        *reinterpret_cast<float4*>(trow + (o - 3)) = make_float4(grp[0], grp[1], grp[2], grp[3]);
                    }
                });
        }
        if (sparse) flush_pending();
        __syncthreads();  // (A) this slab's temp lines are complete; staged buffer k&1 is free again
        if (USE_TMA && k + kInBufs < n_slabs) issue_slab(k + kInBufs);

        // ===================== phase 2: column blur f32 -> int (src/utils.cpp:52-64) + vertical half of Sobel =====================
        // thread = (column tid&127, half tid>>7).  Blurred rows Bg(o) = I_k - R - 2 + 32*half + o, o = 0..33, from temp buffer
        // rows 32*half + o .. + 2R; VU rows Bg(1..32) go to VU buffer rows 2 + 32*half + (o-2).
        {
            const int c = tid & (kTC - 1);
            const int half = tid >> 7;
            const float* tcol = s_temp + (kRunV * half) * kTempPitch + c;
            int32_t* vcol = s_vu + (2 + kRunV * half) * kVuPitch + c;
            const int bg0 = I_k - R - 2 + kRunV * half;  // global row of blurred output 0
            // interior run: every blurred row has all 2R+1 taps inside the image, and every VU row has both vertical neighbours
            const bool y_interior = (bg0 - R >= 0) && (bg0 + kRunCol - 1 + R <= H - 1);
            int t0 = 0, t1 = 0;  // biased blurred values of rows o-2, o-1
            if (y_interior) {
                blur_run<R, kRunCol>(
                    ws, [&](int i) { return tcol[i * kTempPitch]; },
                    [&](int o, float s) {
                        const int t2 = trunc_biased(div_const<DIV>(s, cnt_full, rcp_full, p.div_c));
                        if (o >= 2) {
                            const int u = t2 - t0;                        // B[r+1] - B[r-1]
                            const int v4 = t0 + 2 * t1 + t2 - kBias4;     // B[r-1] + 2 B[r] + B[r+1]
                            vcol[(o - 2) * kVuPitch] = (u << 16) + v4;
                        }
                        t0 = t1; t1 = t2;
                    });
            } else {
                // border run: per-row counts, rows outside the image, replicate / drop rules of src/utils.cpp:117-184
                blur_run<R, kRunCol>(
                    ws, [&](int i) { return tcol[i * kTempPitch]; },
                    [&](int o, float s) {
                        const int gy = bg0 + o;
                        int t2 = kBias;
                        if (gy >= 0 && gy < H) {
                            const int a = max(0, R - gy), b = max(0, gy + R - (H - 1));
                            const int ti = a * (R + 1) + b;
                            t2 = trunc_biased(div_exact(s, s_cnt[ti], s_rcp[ti]));
                        }
                        if (o >= 2) {
                            const int r = gy - 1;  // the VU row: blurred rows r-1 (t0), r (t1), r+1 (t2)
                            int word = 0;
                            if (r >= 0 && r < H) {
                                const int bm = t0 - kBias, bc = t1 - kBias, bp = t2 - kBias;
                                const int up = (r > 0) ? bm : bc, dn = (r < H - 1) ? bp : bc;          // vertical replicate (gy term)
                                const int u = dn - up;
                                const int v = 2 * bc + ((r > 0) ? bm : 0) + ((r < H - 1) ? bp : 0);    // vertical drop (gx term)
                                word = (u << 16) + v;
                            }
                            vcol[(o - 2) * kVuPitch] = word;
                        }
                        t0 = t1; t1 = t2;
                    });
            }
        }
        __syncthreads();  // (B) VU rows 2..65 complete; every read of the temp buffer is done

        // keep the last 2R+2 temp lines for the next slab (rows 64.. -> rows 0..): disjoint source / destination
        if (k + 1 < n_slabs) {
            constexpr int n4 = T0 * (kTC / 4);
            for (int i = tid; i < n4; i += kThreads) {
                const int r = i / (kTC / 4), q = i - r * (kTC / 4);
                reinterpret_cast<float4*>(s_temp + r * kTempPitch)[q] = reinterpret_cast<const float4*>(s_temp + (kSlab + r) * kTempPitch)[q];
            }
        }
        // strips that contain image column -1 or W: the reference replicates horizontally for gx and drops for gy
        // (src/utils.cpp:117-147 vs :158-184).  gx only reads the v half of a neighbour word and gy only the u half, so ONE
        // virtual word {v = v[edge], u = 0} in the out-of-image column serves both.  (Uniform branch: the barrier is legal.)
        if (x_edge) {
            for (int r = tid; r < kSlab; r += kThreads) {
                int32_t* row = s_vu + (2 + r) * kVuPitch;
                if (x0 - 2 < 0) row[1] = row[2] & 0xFFFF;                       // x0 == 0: column j=1 is x=-1, j=2 is x=0
                const int jw = W - (x0 - 2);                                    // column index of image x = W
                if (jw >= 1 && jw < kTC) row[jw] = row[jw - 1] & 0xFFFF;
            }
        }

        __syncthreads();  // (B2) temp tail saved, virtual columns patched: temp rows T0.. are free, VU rows 0..65 final

        // ===================== phase 3a: horizontal half of Sobel, magnitude^2 plane, candidate lists =====================
        // n-plane row q (0..65) <-> VU buffer row q <-> global row y_base + q - 1; it lives in the free part of the temp buffer.
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
            auto n_of_row = [&](const int32_t* vrow) -> int4 {
                const int4 qa = *reinterpret_cast<const int4*>(vrow);
                const int2 qb = *reinterpret_cast<const int2*>(vrow + 4);
                const int wd[6] = {qa.x, qa.y, qa.z, qa.w, qb.x, qb.y};
                int nv[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int wl = wd[e], wc = wd[e + 1], wr = wd[e + 2];
                    const int gx = (int)(short)(wr - wl);    // low halves: v[c+1] - v[c-1] (a borrow only disturbs the high half)
                    const int gy = (wl + wr + 2 * wc) >> 16; // high halves: u[c-1] + 2u[c] + u[c+1] (low-half sum < 2^16: no carry)
                    nv[e] = gx * gx + gy * gy;
                }
                if (x_edge) {                                 // uniform: columns outside the image never suppress (src/utils.cpp:253-304)
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int x = x0 - 2 + 4 * lane + 1 + e;
                        if (x < 0 || x >= W) nv[e] = -1;
                    }
                }
                return make_int4(nv[0], nv[1], nv[2], nv[3]);
            };
            if (cq_lo <= cq_hi) {
                // the two neighbour-only rows: warps 0 and 1
                if (warp < 2) {
                    const int q = warp == 0 ? cq_lo - 1 : cq_hi + 1;
                    const int y = y_base + q - 1;
                    int4 nq = make_int4(-1, -1, -1, -1);      // rows outside the image never suppress
                    if (y >= 0 && y < H) nq = n_of_row(s_vu + q * kVuPitch + 4 * lane);
                    *reinterpret_cast<int4*>(s_np + q * kNpPitch + 4 * lane) = nq;
                }
                const uint32_t zero_word = 0x01010101u * (uint32_t)p.cls_zero;
                const bool word_ok = p.cls_words && lane < kTW / 4 && (x0 + 4 * lane + 3 < W);  // the aligned 32-bit store applies
                const bool tail_ok = !word_ok && lane < kTW / 4 && (x0 + 4 * lane < W);            // ragged right edge: byte stores
                const unsigned lt_mask = (1u << lane) - 1u;
                int q = cq_lo + ((warp - cq_lo) & 7);         // first class row of this warp (rows q = warp mod 8)
                const int32_t* vrow = s_vu + q * kVuPitch + 4 * lane;
                int32_t* nrow = s_np + q * kNpPitch + 4 * lane;
                uint8_t* o = p.cls + (long long)frame * p.cls_frame_stride + (long long)(y_base + q - 1 - p.plane_row0) * p.cls_pitch + (x0 + 4 * lane);
                int ent = ((q - 1) << 6) | (lane << 1);
                const long long o_step = 8LL * p.cls_pitch;
                // two copies of the loop so the store form is decided once, not per row: the aligned 32-bit store (every strip of
                // a class map whose base, pitch and frame stride are multiples of 4, except a ragged last strip) or byte stores
                auto class_row = [&](const int32_t* vr, int32_t* nr, int e16) {
                    const int4 nq = n_of_row(vr);
                    *reinterpret_cast<int4*>(nr) = nq;
                    // one entry per PAIR of pixels (columns 4*lane+1.. +2 and 4*lane+3.. +4) that holds a candidate: candidates
                    // come in bands a few pixels wide, so pairs leave fewer idle pixel slots in phase 3b than whole quads
                    const bool any_lo = max(nq.x, nq.y) >= p.lo2, any_hi = max(nq.z, nq.w) >= p.lo2;
                    const unsigned vote_lo = __ballot_sync(0xffffffffu, any_lo), vote_hi = __ballot_sync(0xffffffffu, any_hi);
                    const int n_lo = __popc(vote_lo);
                    if (any_lo) my_ent[my_count + __popc(vote_lo & lt_mask)] = (uint16_t)e16;
                    if (any_hi) my_ent[my_count + n_lo + __popc(vote_hi & lt_mask)] = (uint16_t)(e16 | 1);
                    my_count += n_lo + __popc(vote_hi);
                };
                // every class word starts out as "suppressed"; phase 3b overwrites the bytes of surviving pixels
                if (__all_sync(0xffffffffu, word_ok || lane >= kTW / 4)) {
                    for (; q <= cq_hi; q += 8, vrow += 8 * kVuPitch, nrow += 8 * kNpPitch, o += o_step, ent += 8 << 6) {
                        class_row(vrow, nrow, ent);
                        if (lane < kTW / 4) *reinterpret_cast<uint32_t*>(o) = zero_word;
                    }
                } else {
                    for (; q <= cq_hi; q += 8, vrow += 8 * kVuPitch, nrow += 8 * kNpPitch, o += o_step, ent += 8 << 6) {
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
        __syncthreads();  // (C1) n-plane complete; the zero words are ordered before phase 3b's byte stores

        // ===================== phase 3b: direction, NMS and thresholds for the candidates only =====================
        {
            const long long out_off = (long long)frame * p.out_frame_stride + (long long)(y_base - p.plane_row0) * W + (x0 - 2) + 1;
            uint8_t* out_base = p.cls + (long long)frame * p.cls_frame_stride + (long long)(y_base - p.plane_row0) * p.cls_pitch + (x0 - 2) + 1;
            int32_t* par_base = p.parent + out_off;                           // only dereferenced when `sparse`
            const int idx_base = (int)out_off;                                // launch-relative pixel index of (class row 0, column j = 1)
            for (int i = lane; i < my_count; i += 32) {
                const int ent = my_ent[i];
                const int rr = ent >> 6, c0 = 2 * (ent & 63);              // pixels j = c0 + 1 and c0 + 2 of class row rr
                const int32_t* vrow = s_vu + (rr + 1) * kVuPitch + c0;     // VU words j-1 .. j+2 = c0 .. c0+3
                const int2 qa = *reinterpret_cast<const int2*>(vrow);
                const int2 qb = *reinterpret_cast<const int2*>(vrow + 2);
                const int wd[4] = {qa.x, qa.y, qb.x, qb.y};
                const int32_t* nrow = s_np + (rr + 1) * kNpPitch + c0;     // n[j] lives at word j - 1
                const int2 n2 = *reinterpret_cast<const int2*>(nrow);
                const int nc[2] = {n2.x, n2.y};
                uint8_t* orow = out_base + (long long)rr * p.cls_pitch + c0;
                // branch-free up to the local-maximum test so the two pixels' chains overlap
                int na[2], nb[2];
                bool pass[2];
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int n = nc[e];
                    const int wl = wd[e], wc = wd[e + 1], wr = wd[e + 2];
                    const int gx = (int)(short)(wr - wl), gy = (wl + wr + 2 * wc) >> 16;
                    // direction_code() of canny_math.h in product form (same integer tests as src/utils.cpp:215-231's bins):
                    //   0   <=> (ay+ax)^2 < 2ax^2           <=> ax^2 - ay^2 > 2 ax ay
                    //   90  <=> ay > ax and (ay-ax)^2 > 2ax^2 <=> ay^2 - ax^2 > 2 ax ay
                    //   else a diagonal: 45 when gx and gy have the same sign (gx*gy > 0; both are non-zero there).
                    // gx = gy = 0 lands on "45" instead of 0, which cannot change the class: such a pixel is a candidate only when
                    // minVal <= 0, and then kept and suppressed pixels get the same class (see fill_thresholds()).
                    const int pxy = gx * gy;
                    const int dd = 2 * gx * gx - n;           // ax^2 - ay^2  (n = ax^2 + ay^2)
                    const int p2 = 2 * abs(pxy);
                    const bool is0 = dd > p2;
                    const bool is90 = -dd > p2;
                    const bool same = pxy >= 0;
                    // neighbour pair along the quantised direction (src/utils.cpp:253-304); out-of-image neighbours hold -1
                    const int off = is0 ? 1 : (is90 ? kNpPitch : (same ? (1 - kNpPitch) : (1 + kNpPitch)));
                    na[e] = nrow[e + off];
                    nb[e] = nrow[e - off];
                    const int j = c0 + 1 + e;
                    pass[e] = (n >= p.lo2) && (j >= 2) && (j <= kTC - 3) && (na[e] < n) && (nb[e] < n);   // j = 1, j >= 126: neighbour-only columns
                }
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    if (pass[e]) {
                        // the reference compares truncated magnitudes: keep iff floor(sqrt(n_nb)) < floor(sqrt(n)) <=> n_nb < mag^2
                        const int n = nc[e];
                        const int mag = isqrt_floor(n);
                        const int m2 = mag * mag;
                        if (na[e] < m2 && nb[e] < m2) {
                            const bool strong = n >= p.hi2;
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
        __syncthreads();  // (C) VU, n-plane and list reads done; the slab's weak-pixel bitmap is complete
        if (sparse) {
            // append this slab's weak pixels to the launch-wide list: every warp counts the bits of its 32 bitmap words and reserves
            // room with ONE global atomicAdd.  The atomic's round trip is hidden behind the next slab's row pass: the entries are
            // written by flush_pending() after it (and once more after the last slab).
            pend_bits = 0;
            if (tid < 4 * kSlab) { pend_bits = s_bits[tid]; s_bits[tid] = 0; }
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
            // word tid <-> class row rr = tid >> 2, columns 32*(tid & 3) .. of the strip
            pend_g0 = (int)((long long)frame * p.out_frame_stride + (long long)(y_base + (tid >> 2) - p.plane_row0) * W + x0 + 32 * (tid & 3));
        }
        // VU rows 64,65 (blurred-row neighbours of the next slab's first class rows) -> rows 0,1
        if (k + 1 < n_slabs) s_vu[(tid >> 7) * kVuPitch + (tid & 127)] = s_vu[(kSlab + (tid >> 7)) * kVuPitch + (tid & 127)];
        // the next iteration's barrier (A) orders this copy before phase 2 rewrites rows 2..65 and phase 3 reads rows 0,1
    }
    if (sparse) flush_pending();
}

}  // namespace f2

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
template <int R, bool USE_TMA, int DIV, int SLAB>
static int launch_one2(b200_ctx* ctx, cudaStream_t st, const FrontParams& p, const CUtensorMap& tmap, dim3 grid) {
    const f2::SmemLayout L = f2::smem_layout(R, SLAB);
    static bool configured[64] = {false};  // per instantiation, per device
    if (!configured[ctx->device & 63]) {
        CB_CUDA(cudaFuncSetAttribute(f2::front2_kernel<R, USE_TMA, DIV, SLAB>, cudaFuncAttributeMaxDynamicSharedMemorySize, L.total));
        CB_CUDA(cudaFuncSetAttribute(f2::front2_kernel<R, USE_TMA, DIV, SLAB>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
        configured[ctx->device & 63] = true;
    }
    {
        ProfScope ps(ctx, st, 0);
        f2::front2_kernel<R, USE_TMA, DIV, SLAB><<<grid, f2::kThreads, L.total, st>>>(p, tmap);
    }
    CB_CUDA(cudaGetLastError());
    ctx->launches++;
    return B200_OK;
}

template <int R, int SLAB>
static int launch_r2(b200_ctx* ctx, cudaStream_t st, const FrontParams& p, const CUtensorMap& tmap, dim3 grid, bool use_tma, int div) {
    if (use_tma) {
        if (div == 1) return launch_one2<R, true, 1, SLAB>(ctx, st, p, tmap, grid);
        if (div == 3) return launch_one2<R, true, 3, SLAB>(ctx, st, p, tmap, grid);
        return launch_one2<R, true, 5, SLAB>(ctx, st, p, tmap, grid);
    }
    // generic staging (odd widths) is not a throughput path: one instantiation, the always-valid division
    return launch_one2<R, false, 5, SLAB>(ctx, st, p, tmap, grid);
}

bool front2_supports(int radius) {
    switch (radius) {
        case 2: case 3: case 5: case 6: case 9: case 15: return true;
        default: return false;
    }
}

// Bands per frame: every band pays 2R+4 warm-up rows and is processed in 64-row slabs, so pick the band count
// that minimises (slabs per band) x (waves of CTAs) — enough CTAs to fill the machine, few enough that the
// warm-up and the last partly-filled slab stay small.
static int choose_bands2(const b200_ctx* ctx, int out_rows, int strips, int frames, int radius, int slab) {
    const int slots = (slab == 64 ? 2 : 4) * (ctx->sm_count > 0 ? ctx->sm_count : 148);
    const long long per_band = (long long)strips * frames;
    int best = 1;
    double best_cost = 1e300;
    const int max_bands = out_rows / 64 > 0 ? out_rows / 64 : 1;
    for (int b = 1; b <= max_bands && b <= 64; ++b) {
        const int rows = (out_rows + b - 1) / b;
        const int slabs = (rows + 2 * radius + 4 + slab - 1) / slab;
        const long long ctas = per_band * b;
        const long long waves = (ctas + slots - 1) / slots;
        const double cost = (double)waves * slabs * slab;  // time ~ waves x rows marched per CTA
        if (cost < best_cost * 0.999) { best_cost = cost; best = b; }
    }
    return best;
}

int launch_front2(b200_ctx* ctx, cudaStream_t st, const FrontParams& p_in) {
    FrontParams p = p_in;
    const int radius = p.radius;
    const int strips = (p.width + f2::kTW - 1) / f2::kTW;
    p.tiles_x = strips;
    // 64-row slabs, 2 CTAs per SM.  The kernel also builds with 32-row slabs (4 CTAs per SM, 63 registers; ncu: issue slots 74 %
    // busy instead of 63 %) but then executes 19 % more instructions (shorter runs share fewer products, twice the tail copies and
    // per-slab set-up) and ends up 2-3 % slower on the 4K batch, so only the 64-row form is instantiated.
    constexpr int slab = 64;
    if (p.tiles_y <= 0) p.tiles_y = choose_bands2(ctx, p.out_rows, strips, p.n_frames, radius, slab);
    dim3 grid(strips, p.tiles_y, p.n_frames);
    CUtensorMap tmap;
    bool use_tma = false;
    CB_TRY(make_input_tensor_map(p, f2::in_pitch_for(radius), slab, &tmap, &use_tma));
    const int div3 = ctx->gauss.div_mode;
    p.div_c = ctx->gauss.div_c;
    switch (radius) {
        case 2: return launch_r2<2, 64>(ctx, st, p, tmap, grid, use_tma, div3);
        case 3: return launch_r2<3, 64>(ctx, st, p, tmap, grid, use_tma, div3);
        case 5: return launch_r2<5, 64>(ctx, st, p, tmap, grid, use_tma, div3);
        case 6: return launch_r2<6, 64>(ctx, st, p, tmap, grid, use_tma, div3);
        case 9: return launch_r2<9, 64>(ctx, st, p, tmap, grid, use_tma, div3);
        case 15: return launch_r2<15, 64>(ctx, st, p, tmap, grid, use_tma, div3);
        default: break;
    }
    set_error("front2 kernel not built for radius %d", radius);
    return B200_ERR_UNSUPPORTED;
}

}  // namespace cb
