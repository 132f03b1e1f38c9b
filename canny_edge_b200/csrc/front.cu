// front.cu — fused stages 1-3 of the Canny hot path for sm_100a, GENERAL variant:
//   u8 gray  --row blur-->  f32  --column blur + truncate-->  i16 blur  --Sobel-->  (gx,gy)
//            --magnitude / direction / non-max suppression / double threshold-->  u8 class map
// It serves what the lean kernel of front3.cu does not: run-time radii (sigma outside the compiled set), the int16 spill planes
// of the stage API / `steps` (blur, magnitude, angle, nms), and sigma so small that sums approach the subnormal range.  The
// dispatcher launch_front() at the end of this file picks between the two; both are parity-tested against the oracle.
//
// Replaces the reference's three kernels gaussian_util / sobel_util / nonmaximal_utility
// (src/cuda.cu:32-73,104-218,249-363) and the host round trips between them
// (src/cuda.cu:90,96,229,240-241,376-377,385).  Semantics are those of the CPU path
// (src/utils.cpp:26-68,106-187,201-236,248-308), bit for bit — see DESIGN.md for why the reference
// GPU kernels are not a valid model (flipped gy, racy border tiles).
//
// Shape of the kernel (one CTA = one 124-px-wide column strip x one band of rows):
//   the CTA marches DOWN its strip in 32-row slabs.  Each slab is brought in by ONE TMA box load
//   (cp.async.bulk.tensor.3d, zero fill outside the image == "skip the tap" for the weighted sum),
//   double buffered on mbarriers.  Intermediates never leave shared memory: they live in row RINGS
//   (f32 row-blurred lines, i16 blurred lines, packed (gx,gy) lines), so there is no vertical halo
//   re-computation — only window/2+2 warm-up rows at the top of a band.
//
// Bit-exactness of the blur (the only float stage): the reference accumulates
//   sum += float(px) * w[k]   for k ascending, separate roundings, then sum / count
// (src/utils.cpp:41-47,56-62).  Here every product is one FMUL (__fmul_rn, never contracted), every
// accumulation one FADD in the same ascending-tap order, and the quotient is an exactly-rounded
// division.  Because w[k] == w[-k] exactly (src/utils.cpp:86-88 squares x), each input's product with
// |k| serves two outputs: blur_run() computes radius+1 products per input and feeds up to 2*radius+1
// accumulators — same roundings, ~45 % fewer multiplies.
#include <cuda.h>

#include "canny_math.h"
#include "exact_math.cuh"
#include "internal.h"
#include "front_common.cuh"

namespace cb {

constexpr int kThreads = 256;
constexpr int kSlab = 32;      // rows per marching step
constexpr int kTC = 128;       // computed columns per strip (temp/blur lines)
constexpr int kTW = kTC - 4;   // class-map columns produced per strip (Sobel + NMS eat 2 per side)
constexpr int kTempPitch = 132;  // floats; == 4 mod 32 so the row pass's 128-bit stores (lane = row) do not conflict
constexpr int kBlurPitch = 128;  // int16
constexpr int kNdPitch = 132;    // int32; column j <-> image x = x0 - 4 + j (class word loads stay 16 B aligned)
constexpr int kRunS = 16;        // outputs per blur_run

__host__ __device__ constexpr int in_pitch_for(int radius) {
    // Bytes per staged input row.  TMA needs the box's first column to sit on a 16-byte boundary of the image
    // row (measured: an unaligned innermost coordinate raises an illegal-instruction fault), so the box starts
    // at the aligned column at or before x0-2-radius and carries up to 15 extra leading bytes.  The pitch is
    // a multiple of 16 (TMA box rule) and an ODD multiple, so that lane = row 128-bit shared loads spread over
    // 8 distinct bank groups.
    int k = (15 + kTC + 2 * radius + 15) / 16;
    if ((k & 1) == 0) k += 1;
    return 16 * k;
}
__host__ __device__ constexpr int temp_cap_for(int radius) {  // ring capacity (rows), power of two >= 32+2R
    return (kSlab + 2 * radius) <= 64 ? 64 : ((kSlab + 2 * radius) <= 128 ? 128 : 256);
}
constexpr int kRingCap = 64;  // blur / nd rings

struct SmemLayout {
    int in_off, temp_off, blur_off, nd_off, tab_off, w_off, bar_off, total;
};
__host__ __device__ inline SmemLayout smem_layout(int radius) {
    SmemLayout L;
    int o = 0;
    L.in_off = o;   o += 2 * kSlab * in_pitch_for(radius);          // two slabs of u8
    o = (o + 127) & ~127;
    L.temp_off = o; o += temp_cap_for(radius) * kTempPitch * 4;
    L.blur_off = o; o += kRingCap * kBlurPitch * 2;
    L.nd_off = o;   o += kRingCap * kNdPitch * 4;
    L.tab_off = o;  o += (radius + 1) * (radius + 1) * 4;           // count table (+ reciprocal right after)
    o += (radius + 1) * (radius + 1) * 4;
    L.w_off = o;    o += (2 * radius + 1) * 4;
    o = (o + 15) & ~15;
    L.bar_off = o;  o += 2 * 8;
    L.total = o;
    return L;
}

// ---------------------------------------------------------------------------------------------
// the kernel
// ---------------------------------------------------------------------------------------------
// R > 0: compile-time radius, fully unrolled blur_run.  R == 0: any radius <= B200_MAX_RADIUS at run time.
template <int R, bool USE_TMA, bool SPILL>
__global__ void __launch_bounds__(kThreads, (R == 0 ? 1 : 2))
front_kernel(const FrontParams p, const __grid_constant__ CUtensorMap tmap) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const int radius = R ? R : p.radius;
    const SmemLayout L = smem_layout(radius);
    const int in_pitch = in_pitch_for(radius);
    const int temp_mask = temp_cap_for(radius) - 1;

    unsigned char* s_in = smem + L.in_off;
    float* s_temp = reinterpret_cast<float*>(smem + L.temp_off);
    int16_t* s_blur = reinterpret_cast<int16_t*>(smem + L.blur_off);
    int32_t* s_nd = reinterpret_cast<int32_t*>(smem + L.nd_off);
    float* s_cnt = reinterpret_cast<float*>(smem + L.tab_off);
    float* s_rcp = s_cnt + (radius + 1) * (radius + 1);
    float* s_w = reinterpret_cast<float*>(smem + L.w_off);
    const uint32_t bar0 = smem_u32(smem + L.bar_off);

    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;

    // ---- which strip / band / frame ----
    const int strip = blockIdx.x;
    const int band = blockIdx.y;
    const int frame = blockIdx.z;
    const int x0 = strip * kTW;                      // first class-map column of this strip
    const int rows_per_band = (p.out_rows + p.tiles_y - 1) / p.tiles_y;
    const int yb = p.out_row0 + band * rows_per_band;                       // first output row (global)
    const int ye = min(p.out_row0 + p.out_rows, yb + rows_per_band);        // one past the last
    if (yb >= ye) return;
    const int W = p.width, H = p.height;
    const int n_slabs = (ye - yb + 2 * radius + 4 + kSlab - 1) / kSlab;
    const int in_y0 = yb - 2 - radius;               // global row of slab 0, line 0
    const int lead = (x0 - 2 - radius) & 15;         // bytes between the 16 B aligned box origin and the first needed column
    const int in_x0 = x0 - 2 - radius - lead;        // global column of staged byte 0 (a multiple of 16, may be negative)
    // ring rows are addressed by (global row + kBias) & mask; kBias keeps the operand positive
    constexpr int kBias = 1 << 20;

    // ---- one-time setup ----
    for (int i = tid; i < (radius + 1) * (radius + 1); i += kThreads) {
        float c = p.count[i];
        s_cnt[i] = c;
        s_rcp[i] = p.count[(radius + 1) * (radius + 1) + i];
    }
    for (int i = tid; i < 2 * radius + 1; i += kThreads) s_w[i] = p.w[i];
    if (USE_TMA && tid == 0) {
        mbar_init(bar0, 1);
        mbar_init(bar0 + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();

    float ws[(R ? R : 1) + 1];
    if (R) {
#pragma unroll
        for (int j = 0; j <= R; ++j) ws[j] = s_w[R + j];
    }
    const bool ieee = p.ieee_div != 0;  // uniform; only for sigma < ~0.15 (see exact_math.cuh)
    auto divq = [&](float a, float b, float y) { return ieee ? __fdiv_rn(a, b) : div_exact(a, b, y); };
    const float cnt_full = s_cnt[0], rcp_full = s_rcp[0];
    // strips whose every computed column has all its taps inside the image use the constant count
    const bool x_interior = (x0 - 2 - radius >= 0) && (x0 - 2 + kTC - 1 + radius <= W - 1);

    const uint8_t* in_frame = p.in + (long long)frame * p.in_frame_stride;
    const uint32_t slab_bytes = (uint32_t)(kSlab * in_pitch);

    auto issue_slab = [&](int k) {  // thread 0 only (TMA) or all threads (fallback)
        const int gy = in_y0 + k * kSlab;
        unsigned char* dst = s_in + (k & 1) * slab_bytes;
        if (USE_TMA) {
            if (tid == 0) {
                const uint32_t bar = bar0 + 8 * (k & 1);
                mbar_expect_tx(bar, slab_bytes);
                tma_load_3d(smem_u32(dst), &tmap, bar, in_x0, gy - p.in_row0, frame);
            }
        } else {
            // generic staging (image pitch not a multiple of 16 B, or TMA disabled): byte loads, zero outside
            for (int i = tid; i < kSlab * in_pitch; i += kThreads) {
                const int r = i / in_pitch, c = i - r * in_pitch;
                const int y = gy + r, x = in_x0 + c;
                const int by = y - p.in_row0;
                unsigned char v = 0;
                if (y >= 0 && y < H && by >= 0 && by < p.in_rows && x >= 0 && x < W)
                    v = in_frame[(long long)by * p.in_pitch + x];
                dst[i] = v;
            }
        }
    };

    if (USE_TMA) {
        issue_slab(0);
        if (n_slabs > 1) issue_slab(1);
    }

    for (int k = 0; k < n_slabs; ++k) {
        const int I_k = in_y0 + k * kSlab;  // global row of this slab's first line
        if (USE_TMA) {
            mbar_wait(bar0 + 8 * (k & 1), (uint32_t)((k >> 1) & 1));
        } else {
            issue_slab(k);
            __syncthreads();
        }
        const unsigned char* slab = s_in + (k & 1) * slab_bytes;

        // ===================== phase 1: row blur, u8 -> f32 (src/utils.cpp:37-49) =====================
        // thread = (line `lane` of the slab, column group `warp` of 16 outputs)
        {
            const int gy = I_k + lane;
            float* trow = s_temp + ((gy + kBias) & temp_mask) * kTempPitch + warp * kRunS;
            const int gx_first = x0 - 2 + warp * kRunS;  // image column of output 0
            float outv[kRunS];
            if (R) {
                // needed bytes of this line: [16*warp + lead, 16*warp + lead + 16 + 2R).  lead = 4*dq + DR where DR is
                // a compile-time constant (x0 is a multiple of 4) and dq in 0..3 is uniform over the CTA: load whole
                // aligned 128-bit vectors, shift by dq WORDS with a uniform switch, pick bytes with static selectors.
                constexpr int RR = R ? R : 1;
                constexpr int DR = (((-2 - RR) % 4) + 4) % 4;
                constexpr int KW = (DR + kRunS + 2 * RR + 3) / 4;       // words holding the needed bytes
                constexpr int NV = (KW + 3 + 3) / 4;                    // vectors covering KW + 3 words
                uint32_t wv[NV * 4];
                const uint4* src = reinterpret_cast<const uint4*>(slab + lane * in_pitch + warp * kRunS);
#pragma unroll
                for (int v = 0; v < NV; ++v) {
                    uint4 t4 = src[v];
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
                blur_run<RR, kRunS>(
                    ws,
                    [&](int i) {
                        const uint32_t word = w2[(i + DR) >> 2];
                        const uint32_t bits = __byte_perm(word, 0x4B000000u, 0x7650 + ((i + DR) & 3));
                        return __fsub_rn(__uint_as_float(bits), 8388608.0f);
                    },
                    [&](int o, float s) { outv[o] = s; });
            } else {
                const unsigned char* src = slab + lane * in_pitch + warp * kRunS + lead;
                for (int o = 0; o < kRunS; ++o) {
                    float s = 0.f;
                    for (int t = 0; t <= 2 * radius; ++t) s = __fadd_rn(s, __fmul_rn((float)src[o + t], s_w[t]));
                    outv[o] = s;
                }
            }
            // divide by the in-image weight sum (src/utils.cpp:47)
            if (x_interior) {
#pragma unroll
                for (int o = 0; o < kRunS; ++o) outv[o] = divq(outv[o], cnt_full, rcp_full);
            } else {
#pragma unroll
                for (int o = 0; o < kRunS; ++o) {
                    const int gx = gx_first + o;
                    if (gx < 0 || gx >= W) { outv[o] = 0.f; continue; }
                    const int a = max(0, radius - gx), b = max(0, gx + radius - (W - 1));
                    const int ti = a * (radius + 1) + b;
                    outv[o] = divq(outv[o], s_cnt[ti], s_rcp[ti]);
                }
            }
#pragma unroll
            for (int v = 0; v < kRunS / 4; ++v)
                reinterpret_cast<float4*>(trow)[v] = make_float4(outv[4 * v], outv[4 * v + 1], outv[4 * v + 2], outv[4 * v + 3]);
        }
        __syncthreads();  // (A) temp lines of this slab visible; staged buffer k&1 is free again
        if (USE_TMA && k + 2 < n_slabs) issue_slab(k + 2);

        // ===================== phase 2: column blur, f32 -> i16 (src/utils.cpp:52-64) =====================
        // window of blurred rows that just became computable: [I_k - radius, I_k - radius + 32)
        // thread = (column tid&127, 16-row half tid>>7)
        {
            const int c = tid & (kTC - 1);
            const int half = tid >> 7;
            const int b0 = I_k - radius + half * kRunS;  // first blurred row of this run (global)
            const int gx = x0 - 2 + c;
            float outv[kRunS];
            if (R) {
                blur_run<(R ? R : 1), kRunS>(
                    ws,
                    [&](int i) { return s_temp[((b0 - (R ? R : 1) + i + kBias) & temp_mask) * kTempPitch + c]; },
                    [&](int o, float s) { outv[o] = s; });
            } else {
                for (int o = 0; o < kRunS; ++o) {
                    float s = 0.f;
                    for (int t = 0; t <= 2 * radius; ++t)
                        s = __fadd_rn(s, __fmul_rn(s_temp[((b0 - radius + o + t + kBias) & temp_mask) * kTempPitch + c], s_w[t]));
                    outv[o] = s;
                }
            }
            const bool y_interior = (b0 - radius >= 0) && (b0 + kRunS - 1 + radius <= H - 1);
#pragma unroll
            for (int o = 0; o < kRunS; ++o) {
                const int gy = b0 + o;
                float q;
                if (y_interior) {
                    q = divq(outv[o], cnt_full, rcp_full);
                } else if (gy < 0 || gy >= H) {
                    q = 0.f;
                } else {
                    const int a = max(0, radius - gy), b = max(0, gy + radius - (H - 1));
                    const int ti = a * (radius + 1) + b;
                    q = divq(outv[o], s_cnt[ti], s_rcp[ti]);
                }
                const int bi = (int)q;  // (short)(sum/count): C truncation, values are >= 0
                s_blur[((gy + kBias) & (kRingCap - 1)) * kBlurPitch + c] = (int16_t)bi;
                if (SPILL) {
                    if (p.blur && gy >= yb && gy < ye && c >= 2 && c < 2 + kTW && gx < W)
                        p.blur[(long long)frame * p.out_frame_stride + (long long)(gy - p.plane_row0) * W + gx] = (int16_t)bi;
                }
            }
        }
        __syncthreads();  // (B)

        // ===================== phase 3: Sobel gx/gy (src/utils.cpp:106-187) =====================
        // rows [I_k - radius - 1, +32); thread = (column c in 1..126, 16-row half), marching down with a
        // 3-row register window of horizontal differences d and horizontal smooths s.
        {
            const int c = tid & (kTC - 1);
            const int half = tid >> 7;
            const int r0 = I_k - radius - 1 + half * kRunS;
            const int gx = x0 - 2 + c;
            const bool col_ok = (c >= 1) && (c <= kTC - 2) && gx >= 0 && gx < W;
            // horizontal neighbours with the reference's border rule: replicate (gx term) / drop (gy term)
            const int cl = (gx > 0) ? c - 1 : c;
            const int cr = (gx < W - 1) ? c + 1 : c;
            const bool has_l = gx > 0, has_r = gx < W - 1;
            int d_m = 0, d_c = 0, s_m = 0, s_c = 0;  // rows y-1 and y
            auto load_row = [&](int y, int& d, int& s) {
                // contributions of image row y; rows outside the image give d = 0 and replicate for s (handled by caller)
                const int16_t* brow = s_blur + ((y + kBias) & (kRingCap - 1)) * kBlurPitch;
                const int l = brow[cl], m = brow[c], r = brow[cr];
                d = r - l;
                s = 2 * m + (has_l ? l : 0) + (has_r ? r : 0);
            };
            if (col_ok) {
                // prime rows r0-1 and r0 (clamped into the image for the replicate rule of gy)
                const int ym = min(max(r0 - 1, 0), H - 1), yc = min(max(r0, 0), H - 1);
                load_row(ym, d_m, s_m);
                load_row(yc, d_c, s_c);
#pragma unroll 4
                for (int o = 0; o < kRunS; ++o) {
                    const int y = r0 + o;
                    int d_p, s_p;
                    const int yp = min(y + 1, H - 1);
                    load_row(max(yp, 0), d_p, s_p);
                    int packed = 0;
                    if (y >= 0 && y < H) {
                        // gx: 2*d(y) + d(y+1) [if y < H-1] + d(y-1) [if y > 0]      (src/utils.cpp:117-147)
                        const int gxv = 2 * d_c + ((y < H - 1) ? d_p : 0) + ((y > 0) ? d_m : 0);
                        // gy: s(min(y+1,H-1)) - s(max(y-1,0)), s with dropped side columns   (src/utils.cpp:158-184)
                        const int gyv = s_p - s_m;
                        packed = (gxv & 0xFFFF) | (gyv << 16);
                    }
                    s_nd[((y + kBias) & (kRingCap - 1)) * kNdPitch + c + 2] = packed;
                    // slide: row y becomes y-1.  At the top border the "row above" of row 0 is row 0 itself
                    // (already primed that way); at the bottom yp clamps.
                    d_m = d_c; s_m = s_c; d_c = d_p; s_c = s_p;
                    if (y < 0) { d_m = d_c; s_m = s_c; }  // rows above the image: keep the window parked on row 0
                }
            }
        }
        __syncthreads();  // (C)

        // ===================== phase 4: magnitude, direction, NMS, thresholds =====================
        // rows [I_k - radius - 2, +32) clipped to [yb, ye); thread = 4 consecutive pixels (one class word)
        {
            const int word = lane;            // 31 words of 4 px = 124 columns
            if (word < kTW / 4) {
                for (int rr = warp; rr < kSlab; rr += kThreads / 32) {
                    const int y = I_k - radius - 2 + rr;
                    if (y < yb || y >= ye) continue;
                    const int xw = x0 + 4 * word;
                    if (xw >= W) continue;
                    const int32_t* nrow = s_nd + ((y + kBias) & (kRingCap - 1)) * kNdPitch;
                    const int32_t* nup = s_nd + ((y - 1 + kBias) & (kRingCap - 1)) * kNdPitch;
                    const int32_t* ndn = s_nd + ((y + 1 + kBias) & (kRingCap - 1)) * kNdPitch;
                    const int4 ctr = *reinterpret_cast<const int4*>(nrow + 4 + 4 * word);
                    const int cv[4] = {ctr.x, ctr.y, ctr.z, ctr.w};
                    uint32_t cls_word = 0;
                    int16_t magv[4], angv[4], nmsv[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int x = xw + e;
                        const int gxv = (int)(int16_t)(cv[e] & 0xFFFF), gyv = cv[e] >> 16;
                        const int n = gxv * gxv + gyv * gyv;
                        int cls = p.cls_zero;
                        int mag = 0, dir = 0, keep = 0;
                        if (SPILL || n >= p.lo2) {
                            mag = isqrt_floor(n);
                            dir = direction_code<int>(gxv, gyv);
                            // neighbour pair along the quantised direction (src/utils.cpp:253-304)
                            const int dx = (dir == DIR_90) ? 0 : 1;
                            const int dy = (dir == DIR_0) ? 0 : ((dir == DIR_45) ? -1 : 1);
                            const int j = 4 + 4 * word + e;
                            const int m2 = mag * mag;
                            keep = 1;
                            {   // neighbour (y+dy, x+dx)
                                const int yy = y + dy, xx = x + dx;
                                if (yy >= 0 && yy < H && xx < W) {
                                    const int32_t* rowp = (dy == 0) ? nrow : ((dy < 0) ? nup : ndn);
                                    const int v = rowp[j + dx];
                                    const int a = (int)(int16_t)(v & 0xFFFF), b = v >> 16;
                                    if (m2 <= a * a + b * b) keep = 0;  // mag <= mag_nb  <=>  mag^2 <= n_nb
                                }
                            }
                            {   // neighbour (y-dy, x-dx)
                                const int yy = y - dy, xx = x - dx;
                                if (yy >= 0 && yy < H && xx >= 0) {
                                    const int32_t* rowp = (dy == 0) ? nrow : ((dy < 0) ? ndn : nup);
                                    const int v = rowp[j - dx];
                                    const int a = (int)(int16_t)(v & 0xFFFF), b = v >> 16;
                                    if (m2 <= a * a + b * b) keep = 0;
                                }
                            }
                            if (keep) cls = (n >= p.hi2 && n >= p.lo2) ? 255 : ((n >= p.lo2) ? 1 : 0);
                        }
                        if (x >= W) cls = 0;
                        cls_word |= (uint32_t)cls << (8 * e);
                        if (SPILL) { magv[e] = (int16_t)mag; angv[e] = (int16_t)(dir * 45); nmsv[e] = keep ? (int16_t)mag : (int16_t)0; }
                    }
                    const long long o = (long long)frame * p.out_frame_stride + (long long)(y - p.plane_row0) * W + xw;
                    uint8_t* oc = p.cls + (long long)frame * p.cls_frame_stride + (long long)(y - p.plane_row0) * p.cls_pitch + xw;
                    if (p.cls_words && xw + 3 < W) {
                        *reinterpret_cast<uint32_t*>(oc) = cls_word;
                    } else {
                        for (int e = 0; e < 4 && xw + e < W; ++e) oc[e] = (uint8_t)(cls_word >> (8 * e));
                    }
                    if (SPILL) {
                        for (int e = 0; e < 4 && xw + e < W; ++e) {
                            if (p.mag) p.mag[o + e] = magv[e];
                            if (p.ang) p.ang[o + e] = angv[e];
                            if (p.nms) p.nms[o + e] = nmsv[e];
                        }
                    }
                }
            }
        }
        // no barrier needed here: the next iteration's (A) orders phase 4 reads before phase 3 rewrites the nd ring,
        // and phase 1 of the next slab only touches the temp ring and the other staged buffer.
    }
}

// ---------------------------------------------------------------------------------------------
// host side: tensor map + launch
// ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* sym = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(sym);
    }
    return fn;
}

template <int R, bool USE_TMA, bool SPILL>
static int launch_one(b200_ctx* ctx, cudaStream_t st, const FrontParams& p, const CUtensorMap& tmap, dim3 grid) {
    const int radius = R ? R : p.radius;
    const SmemLayout L = smem_layout(radius);
    static int configured_bytes[64] = {0};  // per instantiation, per device
    int& conf = configured_bytes[ctx->device & 63];
    if (conf < L.total) {
        CB_CUDA(cudaFuncSetAttribute(front_kernel<R, USE_TMA, SPILL>, cudaFuncAttributeMaxDynamicSharedMemorySize, L.total));
        conf = L.total;
    }
    {
        ProfScope ps(ctx, st, 0);
        front_kernel<R, USE_TMA, SPILL><<<grid, kThreads, L.total, st>>>(p, tmap);
    }
    CB_CUDA(cudaGetLastError());
    ctx->launches++;
    return B200_OK;
}

template <int R>
static int launch_r(b200_ctx* ctx, cudaStream_t st, const FrontParams& p, const CUtensorMap& tmap, dim3 grid,
                    bool use_tma, bool spill) {
    if (use_tma) return spill ? launch_one<R, true, true>(ctx, st, p, tmap, grid) : launch_one<R, true, false>(ctx, st, p, tmap, grid);
    return spill ? launch_one<R, false, true>(ctx, st, p, tmap, grid) : launch_one<R, false, false>(ctx, st, p, tmap, grid);
}

int choose_bands(const b200_ctx* ctx, int out_rows, int strips, int frames, int radius) {
    // One CTA marches a whole band; every band pays 2*radius+4 warm-up rows, so use as few bands as keep
    // the machine full: aim for >= 4 CTAs per resident slot (2 per SM) when the launch is that big anyway.
    const int slots = 2 * (ctx->sm_count > 0 ? ctx->sm_count : 148);
    const long long ctas_one_band = (long long)strips * frames;
    int bands = 1;
    if (ctas_one_band < 4LL * slots) bands = (int)((4LL * slots + ctas_one_band - 1) / ctas_one_band);
    const int min_rows = 2 * kSlab;  // below this the warm-up dominates
    const int max_bands = out_rows / min_rows > 0 ? out_rows / min_rows : 1;
    if (bands > max_bands) bands = max_bands;
    if (bands < 1) bands = 1;
    // prefer band heights with (rows + 2R + 4) a multiple of the slab
    (void)radius;
    return bands;
}

// Builds the 3-D u8 tensor map {width, rows in the buffer, frames} with a box of box_cols x box_rows x 1.  TMA needs a
// 16 B aligned base, row pitch and frame stride (input_tma_layout_ok); *use_tma is false when the image does not qualify
// (the kernels then run their generic staging variant — same kernel, byte loads instead of the bulk copy).  Columns past
// `width` (a padded pitch) arrive as zeros like those left of the image.
int make_input_tensor_map(const FrontParams& p, int box_cols, int box_rows, CUtensorMap* tmap, bool* use_tma) {
    static const bool tma_env_off = [] { const char* e = getenv("B200_CANNY_NO_TMA"); return e && e[0] == '1'; }();
    memset(tmap, 0, sizeof(*tmap));
    *use_tma = !tma_env_off && input_tma_layout_ok(p) && get_encode_fn() != nullptr;
    if (!*use_tma) return B200_OK;
    const cuuint64_t dims[3] = {(cuuint64_t)p.width, (cuuint64_t)p.in_rows, (cuuint64_t)p.n_frames};
    const cuuint64_t strides[2] = {(cuuint64_t)p.in_pitch, (cuuint64_t)input_tma_frame_stride(p)};
    const cuuint32_t box[3] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = get_encode_fn()(tmap, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<uint8_t*>(p.in), dims, strides, box, estr,
                                 CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                 CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed (%d) for %dx%dx%d", (int)r, p.width, p.in_rows, p.n_frames);
        return B200_ERR_CUDA;
    }
    return B200_OK;
}

// Interleaved B,G,R frames as a tensor of 32-bit elements (a box row of a u8 map holds at most 256 bytes; the staged row is 528):
// 3*width/4 elements per row (rows in_pitch bytes apart), out-of-range elements zero-filled like the gray map's.
int make_bgr_tensor_map(const FrontParams& p, int box_words, int box_rows, CUtensorMap* tmap) {
    memset(tmap, 0, sizeof(*tmap));
    if (get_encode_fn() == nullptr) { set_error("cuTensorMapEncodeTiled is not available"); return B200_ERR_UNSUPPORTED; }
    const cuuint64_t dims[3] = {(cuuint64_t)(3 * (long long)p.width / 4), (cuuint64_t)p.in_rows, (cuuint64_t)p.n_frames};
    const cuuint64_t strides[2] = {(cuuint64_t)p.in_pitch, (cuuint64_t)input_tma_frame_stride(p)};
    const cuuint32_t box[3] = {(cuuint32_t)box_words, (cuuint32_t)box_rows, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = get_encode_fn()(tmap, CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, const_cast<uint8_t*>(p.in), dims, strides, box, estr,
                                 CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                 CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed (%d) for BGR %dx%dx%d", (int)r, p.width, p.in_rows, p.n_frames);
        return B200_ERR_CUDA;
    }
    return B200_OK;
}

static int launch_front_v1(b200_ctx* ctx, cudaStream_t st, const FrontParams& p_in) {
    FrontParams p = p_in;
    const int radius = p.radius;
    const int strips = (p.width + kTW - 1) / kTW;
    p.tiles_x = strips;
    if (p.tiles_y <= 0) p.tiles_y = choose_bands(ctx, p.out_rows, strips, p.n_frames, radius);
    dim3 grid(strips, p.tiles_y, p.n_frames);
    const bool spill = p.blur || p.mag || p.ang || p.nms;
    CUtensorMap tmap;
    bool use_tma = false;
    CB_TRY(make_input_tensor_map(p, in_pitch_for(radius), kSlab, &tmap, &use_tma));
    switch (radius) {
        case 2: return launch_r<2>(ctx, st, p, tmap, grid, use_tma, spill);
        case 3: return launch_r<3>(ctx, st, p, tmap, grid, use_tma, spill);
        case 5: return launch_r<5>(ctx, st, p, tmap, grid, use_tma, spill);
        case 6: return launch_r<6>(ctx, st, p, tmap, grid, use_tma, spill);
        case 9: return launch_r<9>(ctx, st, p, tmap, grid, use_tma, spill);
        case 15: return launch_r<15>(ctx, st, p, tmap, grid, use_tma, spill);
        default: return launch_r<0>(ctx, st, p, tmap, grid, use_tma, spill);
    }
}

// Dispatcher: front3.cu's kernel for the hot configuration — no spill planes and a sigma it takes (front3_supports);
// front_kernel above for everything else.
int launch_front(b200_ctx* ctx, cudaStream_t st, const FrontParams& p_in, bool* sparse_out) {
    FrontParams p = p_in;
    if (sparse_out) *sparse_out = false;
    p.ieee_div = ctx->gauss.tiny ? 1 : 0;
    if (p.in_pitch < (p.in_bgr ? 3LL : 1LL) * p.width || p.cls_pitch < p.width) {
        set_error("internal: front launch without input / class-map pitch (%lld, %lld for width %d)", p.in_pitch, p.cls_pitch, p.width);
        return B200_ERR_INVALID_ARG;
    }
    p.cls_words = ((reinterpret_cast<uintptr_t>(p.cls) | (uintptr_t)p.cls_pitch | (uintptr_t)p.cls_frame_stride) & 3) == 0;
    const int radius = p.radius;
    if (radius < 1 || radius > B200_MAX_RADIUS) {
        set_error("gaussian radius %d outside [1,%d]", radius, B200_MAX_RADIUS);
        return B200_ERR_UNSUPPORTED;
    }
    const bool spill = p.blur || p.mag || p.ang || p.nms;
    if (p.in_bgr && (spill || !front3_bgr_supports(ctx->gauss, p))) {
        set_error("interleaved B,G,R input is only taken by the fused front kernel (callers check front3_bgr_supports)");
        return B200_ERR_UNSUPPORTED;
    }
    if (!spill && front3_supports(ctx->gauss)) {
        // the sparse hand-over lists KEPT pixels; with minVal <= 0 suppressed pixels are candidates too (src/utils.cpp:328), so the
        // whole-plane labelling has to run
        const bool sparse = p.parent != nullptr && p.kept_list != nullptr && p.kept_count != nullptr && p.cls_zero == 0 &&
                            (long long)p.n_frames * p.out_frame_stride < (1LL << 31);
        if (!sparse) { p.parent = nullptr; p.kept_list = nullptr; p.kept_count = nullptr; }
        if (sparse_out) *sparse_out = sparse;
        ctx->front_fast++;
        return launch_front3(ctx, st, p);
    }
    // The generic kernel is 3-4x slower than the lean ones.  It is the right one for spill planes (stage API, `steps`); for a plain
    // map it means sigma's half-window is not in the compiled set {2,3,5,6,9,15}: say so once per context instead of silently
    // running at a quarter of the speed (b200_ctx_front_kernel_stats counts both kinds).
    if (!spill && ctx->front_generic == 0 && getenv("B200_CANNY_QUIET") == nullptr)
        fprintf(stderr, "libcanny_b200: gaussian half-window %d (sigma %g) has no specialised front kernel (built: 2, 3, 5, 6, 9, 15)%s; "
                        "using the generic kernel (about 4x slower). Set B200_CANNY_QUIET=1 to silence.\n",
                radius, (double)ctx->gauss.sigma, ctx->gauss.tiny ? " and its weights reach the subnormal range" : "");
    ctx->front_generic++;
    return launch_front_v1(ctx, st, p);
}

}  // namespace cb
