// front_cv.cu — the front kernel of the OpenCV-compatible path (b200_cv_canny_aperture_device_strided, and
// b200_cv_canny_aperture_frames_device through the RAGGED variant below): 1- or 3-channel u8 frames -> class map (0 / 1 weak / 255
// strong) plus the weak-pixel hand-over of the list-driven hysteresis kernels, with cv::Canny's arithmetic (apertureSize K = 3, 5 or
// 7) bit for bit.  No blur: the K x K Sobel kernels on the input, BORDER_REPLICATE for both derivatives.  With a blur class BR > 0
// (b200_cv_gaussian_canny_*: BR = 3 for radii up to 3, 15 up to 15; the radii and taps in CvBlurParams), phase 1 is stage_blurred:
// cv::GaussianBlur's 8-bit fixed-point blur on the staged tile, so s_in holds the blurred frame and phases 2-4 are the same code.
//
// One CTA = one 128 x 64 tile of one frame, 288 threads (9 warps); R = K / 2:
//   1. staging: input rows y0-1-R .. y0+64+R, pixels x0-16 .. x0+143 (C bytes each) into shared memory, with the coordinates
//      clamped into the image (BORDER_REPLICATE then needs nothing else).  16-byte chunks that lie inside the row and are 16-byte
//      aligned in global memory are one vector load; the others (image edges, pitches or bases off a 16-byte boundary) take byte
//      loads of the same clamped bytes.  The columns read are x0-1-R .. x0+128+R, inside the staged ones for R <= 3.
//   2. gradients: threads 0..259 take one column of the 130 x 66 magnitude region (tile + 1 pixel each side, what the non-maximum
//      test reads) and slide down 33 rows of it with the separable Sobel sums of K staged rows in registers: per staged row the
//      derivative taps across the row (for dx) and the smoothing taps (for dy), then down the K rows the smoothing taps for dx and
//      the derivative taps for dy.  K = 7 divides both by 16, rounding half to even (cvRound), as cv::Canny scales them.  Per
//      channel: dx, dy, magnitude (L1: |dx|+|dy|, L2: dx^2+dy^2); the channel of the largest magnitude wins (the first one on ties,
//      as OpenCV).  The magnitude and the direction class are stored as one word, m << 2 | code.  Magnitude outside the image is 0.
//   3. non-maximum suppression and thresholds: warps 0..7, a lane takes 4 adjacent pixels of a row (one 32-bit class store) in 8
//      rows.  The row's 6-word neighbourhood comes from one 128-bit shared load per row plus shuffles.
//   4. hand-over: each thread's 32 pixels fit one bitmask of weak pixels; one atomicAdd per CTA reserves room in the list, and
//      every weak pixel gets its union-find slot (its own dense launch-relative index) and its list entry.
//
// RAGGED (b200_cv_canny_aperture_frames_device): frames of different sizes in one launch.  A 1-D grid over work items (p.ritems),
// each naming a frame and one 128 x 64 tile of it (RaggedItem: x0, yb; ye is not read, rows past the frame's height are clipped as
// in a uniform launch); the frame's descriptor (p.rframes) replaces in / in_pitch / width / height / cls / cls_pitch / cls_words and
// its slot base replaces frame * out_frame_stride.  Staging is per frame as above: 16-byte loads where the chunk is aligned, byte
// loads elsewhere.
//
// Integer bounds.  K = 3: |dx|, |dy| <= 4 * 255 = 1020.  K = 5: the derivative taps' positive sum is 3, the smoothing taps' sum
// 16, so |dx|, |dy| <= 255 * 3 * 16 = 12240, and a staged row's sums are at most 255 * 3 and 255 * 16.  K = 7: the exact sums
// are at most 255 * 10 * 64 = 163 200, so |dx|, |dy| <= 10 200 after the division; a staged row's sums are at most 255 * 10 and
// 255 * 64 = 16 320.  So |dx|, |dy| <= 12240 for every K: L1 m <= 24 480; L2 m <= 2 * 12240^2 = 299 635 200, and m << 2 | code
// <= 1 198 540 803 < 2^31.  In the direction test x = |dx| <= 12240: x * TG22 + (x << 16) <= 968 294 160 and |dy| << 15 <=
// 401 080 320 fit in int32.
#include <string.h>

#include <algorithm>

#include "internal.h"

namespace cb {
namespace fcv {

constexpr int kTW = 128;                 // class columns per tile
constexpr int kTH = 64;                  // class rows per tile
constexpr int kThreads = 288;            // 9 warps: 260 gradient columns in phase 2, 8 warps of 32 x 4 pixels in phase 3
constexpr int kSW = kTW + 32;            // staged pixels per row: x0-16 .. x0+143 (16-pixel aligned chunks; 128 + K - 1 are read)
constexpr int kMR = kTH + 2;             // magnitude rows: y0-1 .. y0+64
constexpr int kMP = 136;                 // magnitude words per row; column j (-1 .. 128) at word j + 4, so column 0 is 16-byte aligned
constexpr int kGroupRows = kMR / 2;      // magnitude rows per phase-2 thread
constexpr int TG22 = 13573;              // (int)(tan(22.5 deg) * 2^15 + 0.5), imgproc/src/canny.cpp

// Sobel taps of cv::getDerivKernels for aperture K: t-th smoothing and derivative tap
__host__ __device__ constexpr int smooth_tap(int K, int t) {
    return K == 3 ? (t == 1 ? 2 : 1) : K == 5 ? (t == 2 ? 6 : (t & 1) ? 4 : 1) : (t == 3 ? 20 : t == 2 || t == 4 ? 15 : t == 1 || t == 5 ? 6 : 1);
}
__host__ __device__ constexpr int deriv_tap(int K, int t) {
    return K == 3 ? t - 1 : K == 5 ? (t == 0 ? -1 : t == 1 ? -2 : t == 2 ? 0 : t == 3 ? 2 : 1)
                  : (t == 0 ? -1 : t == 1 ? -4 : t == 2 ? -5 : t == 3 ? 0 : t == 4 ? 5 : t == 5 ? 4 : 1);
}

template <int C, int K, int BR = 0>
struct Smem {
    static constexpr int kSH = kTH + 2 + 2 * (K / 2);          // staged rows: y0-1-R .. y0+64+R
    static constexpr int in_row = C * kSW;                     // bytes per staged row, a multiple of 16
    static constexpr int in_bytes = kSH * in_row;
    static constexpr int m_off = (in_bytes + 15) & ~15;
    static constexpr int sum_off = m_off + kMR * kMP * 4;      // per-warp weak counts, then the CTA's list base
    // Gaussian pre-blur (BR = 3 or 15, the largest radius of the class; 0: none): the raw rows and one strip of column sums alias
    // s_m and s_sum, which phase 2 writes only after the blur has filled s_in.  Raw pixel u of a row is x0 - kXOff + u; the column
    // pass covers raw pixels kULo .. kUHi-1 (every pixel the row pass reads for staged pixels 8 .. 151, a superset of what phase 2
    // reads); the row pass writes staged pixels 8 .. 151.
    static constexpr int kXOff = BR <= 3 ? 16 : 32;
    static constexpr int raw_row = C * (kSW - 32 + 2 * kXOff);  // 160 or 192 pixels, a multiple of 16 bytes
    static constexpr int raw_rows = kSH + 2 * BR;
    static constexpr int raw_bytes = raw_rows * raw_row;
    static constexpr int kULo = BR <= 3 ? 4 : 8, kUHi = BR <= 3 ? 156 : 184;
    static constexpr int v_row = C * (kUHi - kULo);            // u16 column sums per strip row
    // strip rows: every staged row for gray; for 3 channels as many as keep 3 CTAs per SM (radius <= 3) or 2 (radius <= 15)
    static constexpr int strip = C == 1 ? kSH : BR <= 3 ? 4 : 16;
    static constexpr int blur_bytes = raw_bytes + strip * v_row * 2;
    static constexpr int total = BR == 0 ? sum_off + 16 * 4 : std::max(sum_off + 16 * 4, m_off + blur_bytes);
};

// reflect-101 index into 0 .. n-1 (OpenCV's BORDER_REFLECT_101 / BORDER_DEFAULT), repeated with period 2(n - 1) when the kernel is
// wider than the frame; a 1-pixel side always maps to 0
__device__ __forceinline__ int reflect101(int x, int n) {
    if ((unsigned)x < (unsigned)n) return x;
    if (n == 1) return 0;
    const int per = 2 * (n - 1);
    x %= per;
    if (x < 0) x += per;
    return x < n ? x : per - x;
}

// Phase 1 with cv::GaussianBlur before the Sobel stage: s_in receives, at every staged position phase 2 reads, the blurred pixel B at
// the position's clamped coordinates (cv::Canny's BORDER_REPLICATE applies to B, not to the raw frame), so phases 2-4 are unchanged.
//   a. raw rows y0-1-R-ry .. y0+64+R+ry and pixels x0-kXOff .. through reflect101 into s_raw: 16-byte loads where the chunk lies
//      inside the row and is aligned (no reflection needed there), byte loads elsewhere;
//   b. per strip of staged rows: the column pass (8.8 taps of fy, folded: each tap multiplies the sum of the two mirrored rows) of
//      each staged row's clamped row into u16 sums (<= 255 * 256), then the row pass over them with fx, (sum + 2^15) >> 16 into s_in.
// Every sum is an exact integer below 2^24, so the order of summation does not matter.
template <int C, int K, int BR>
__device__ __forceinline__ void stage_blurred(const CvBlurParams& b, unsigned char* smem, const uint8_t* in_f, long long in_pitch,
                                              int x0, int y0, int W, int H) {
    using S = Smem<C, K, BR>;
    constexpr int R = K / 2;
    const int tid = threadIdx.x;
    const int rx = b.rx, ry = b.ry;
    unsigned char* s_in = smem;
    unsigned char* s_raw = smem + S::m_off;
    uint16_t* s_v = reinterpret_cast<uint16_t*>(smem + S::m_off + S::raw_bytes);
    {
        constexpr int kChunks = S::raw_row / 16;
        const long long row_bytes = (long long)C * W;
        const long long xb = (long long)(x0 - S::kXOff) * C;
        const int n_rows = S::kSH + 2 * ry;
        for (int i = tid; i < n_rows * kChunks; i += kThreads) {
            const int r = i / kChunks, q = i - r * kChunks;
            const int y = reflect101(y0 - 1 - R - ry + r, H);
            const uint8_t* row = in_f + (long long)y * in_pitch;
            const long long b0 = xb + 16 * q;
            uint4 v;
            if (b0 >= 0 && b0 + 16 <= row_bytes && ((reinterpret_cast<uintptr_t>(row + b0) & 15) == 0)) {
                v = __ldg(reinterpret_cast<const uint4*>(row + b0));
            } else {
                uint32_t wd[4] = {0, 0, 0, 0};
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                    const int s = 16 * q + e;
                    const int x = reflect101(x0 - S::kXOff + s / C, W);
                    wd[e >> 2] |= (uint32_t)row[(long long)x * C + (s % C)] << (8 * (e & 3));
                }
                v = make_uint4(wd[0], wd[1], wd[2], wd[3]);
            }
            *reinterpret_cast<uint4*>(s_raw + r * S::raw_row + 16 * q) = v;
        }
    }
    __syncthreads();
    constexpr int kVGroups = S::v_row / 4;                      // 4 column sums per thread and step
    constexpr int kOutLo = 8, kOutGroups = C * 144 / 4;          // staged pixels 8 .. 151, 4 bytes per thread and step
#pragma unroll 1
    for (int r0 = 0; r0 < S::kSH; r0 += S::strip) {
        // column pass: strip row sr holds the sums of staged row r0 + sr, centred on its clamped row (raw row qc + ry)
        for (int i = tid; i < S::strip * kVGroups; i += kThreads) {
            const int sr = i / kVGroups, g = i - sr * kVGroups;
            if (r0 + sr >= S::kSH) break;
            const int qc = min(max(y0 - 1 - R + r0 + sr, 0), H - 1) - (y0 - 1 - R);
            const unsigned char* src = s_raw + (qc + ry) * S::raw_row + C * S::kULo + 4 * g;
            const uint32_t w0 = *reinterpret_cast<const uint32_t*>(src);
            int a[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) a[e] = b.hy[0] * (int)((w0 >> (8 * e)) & 255);
#pragma unroll
            for (int t = 1; t <= BR; ++t) {
                if (t > ry) break;
                const uint32_t wu = *reinterpret_cast<const uint32_t*>(src - t * S::raw_row);
                const uint32_t wd = *reinterpret_cast<const uint32_t*>(src + t * S::raw_row);
#pragma unroll
                for (int e = 0; e < 4; ++e) a[e] += b.hy[t] * (int)(((wu >> (8 * e)) & 255) + ((wd >> (8 * e)) & 255));
            }
            *reinterpret_cast<uint2*>(s_v + sr * S::v_row + 4 * g) =
                make_uint2((uint32_t)a[0] | (uint32_t)a[1] << 16, (uint32_t)a[2] | (uint32_t)a[3] << 16);
        }
        __syncthreads();
        // row pass: staged pixel s of staged row r0 + sr is B at the clamped column, raw pixel xc - x0 + kXOff
        for (int i = tid; i < S::strip * kOutGroups; i += kThreads) {
            const int sr = i / kOutGroups, g = i - sr * kOutGroups;
            if (r0 + sr >= S::kSH) break;
            uint32_t word = 0;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int ob = C * kOutLo + 4 * g + e, s = ob / C, c = ob - s * C;
                const int u = min(max(x0 - 16 + s, 0), W - 1) - x0 + S::kXOff;
                const uint16_t* vp = s_v + sr * S::v_row + (u - S::kULo) * C + c;
                int acc = b.hx[0] * (int)vp[0];
#pragma unroll
                for (int t = 1; t <= BR; ++t) {
                    if (t > rx) break;
                    acc += b.hx[t] * ((int)vp[-t * C] + (int)vp[t * C]);
                }
                word |= (uint32_t)((acc + 32768) >> 16) << (8 * e);
            }
            *reinterpret_cast<uint32_t*>(s_in + (r0 + sr) * S::in_row + C * kOutLo + 4 * g) = word;
        }
        __syncthreads();
    }
}

template <int C, bool L2, bool RAGGED, int K, int BR>
__global__ void __launch_bounds__(kThreads)
front_cv_kernel(const FrontParams p, const CvBlurParams blur) {
    extern __shared__ __align__(16) unsigned char smem[];
    using S = Smem<C, K>;
    constexpr int R = K / 2;
    unsigned char* s_in = smem;
    int* s_m = reinterpret_cast<int*>(smem + S::m_off);
    unsigned int* s_sum = reinterpret_cast<unsigned int*>(smem + S::sum_off);
    // the list-driven hysteresis kernel behind this one may be launched programmatically (HystParams::pdl)
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    RaggedItem item;
    RaggedFrame fd;
    if (RAGGED) {
        item = p.ritems[blockIdx.x];
        fd = p.rframes[item.frame];
    }
    const int x0 = RAGGED ? item.x0 : blockIdx.x * kTW, y0 = RAGGED ? item.yb : blockIdx.y * kTH, frame = RAGGED ? 0 : blockIdx.z;
    const int W = RAGGED ? fd.width : p.width, H = RAGGED ? fd.height : p.height;
    const uint8_t* in_f = RAGGED ? fd.in : p.in + (long long)frame * p.in_frame_stride;
    const long long in_pitch = RAGGED ? fd.in_pitch : p.in_pitch;

    // ---- 1. staging, clamped coordinates (BR > 0: of the blurred frame, stage_blurred) ----
    if constexpr (BR > 0) {
        stage_blurred<C, K, BR>(blur, smem, in_f, in_pitch, x0, y0, W, H);
    } else {
        constexpr int kChunks = S::in_row / 16;
        const long long row_bytes = (long long)C * W;
        const long long xb = (long long)(x0 - 16) * C;         // byte of staged pixel 0 within its row (a multiple of 16 - 48C)
        for (int i = tid; i < S::kSH * kChunks; i += kThreads) {
            const int r = i / kChunks, q = i - r * kChunks;
            const int y = min(max(y0 - 1 - R + r, 0), H - 1);
            const uint8_t* row = in_f + (long long)y * in_pitch;
            const long long b0 = xb + 16 * q;
            uint4 v;
            if (b0 >= 0 && b0 + 16 <= row_bytes && ((reinterpret_cast<uintptr_t>(row + b0) & 15) == 0)) {
                v = __ldg(reinterpret_cast<const uint4*>(row + b0));
            } else {
                uint32_t wd[4] = {0, 0, 0, 0};
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                    const int s = 16 * q + e;                   // staged byte: pixel s / C, channel s % C
                    const int x = min(max(x0 - 16 + s / C, 0), W - 1);
                    wd[e >> 2] |= (uint32_t)row[(long long)x * C + (s % C)] << (8 * (e & 3));
                }
                v = make_uint4(wd[0], wd[1], wd[2], wd[3]);
            }
            *reinterpret_cast<uint4*>(s_in + r * S::in_row + 16 * q) = v;
        }
        __syncthreads();
    }

    // ---- 2. gradients, magnitude, direction class of the 130 x 66 region ----
    if (tid < 2 * (kTW + 2)) {
        const int grp = tid / (kTW + 2);
        const int j = tid - grp * (kTW + 2) - 1;                // tile column -1 .. 128
        const int x = x0 + j;
        const bool x_in = x >= 0 && x < W;
        const int r0 = grp * kGroupRows - 1;                     // first tile row of this thread: -1 or 32
        if constexpr (K == 3) {
            // aperture 3 keeps its three-row window with the taps written out, so its kernels compile to the SASS DESIGN §4.4
            // measured.  Staged row of tile row r is r + 2; staged pixel of column j is j + 16
            const unsigned char* col = s_in + (j + 15) * C;
            int hp[C], hc[C], vp[C], vc[C];
            auto sums = [&](int sr, int* h, int* v) {            // row sums of staged row sr: h = right - left, v = left + 2 mid + right
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const unsigned char* q = col + sr * S::in_row + c;
                    const int a = q[0], b = q[C], d = q[2 * C];
                    h[c] = d - a;
                    v[c] = a + 2 * b + d;
                }
            };
            sums(r0 + 1, hp, vp);
            sums(r0 + 2, hc, vc);
            int* mrow = s_m + (r0 + 1) * kMP + j + 4;
            for (int k = 0; k < kGroupRows; ++k) {
                const int r = r0 + k;
                int hn[C], vn[C];
                sums(r + 3, hn, vn);
                int best = -1, gx = 0, gy = 0;
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const int dx = hp[c] + 2 * hc[c] + hn[c];
                    const int dy = vn[c] - vp[c];
                    const int n = L2 ? dx * dx + dy * dy : abs(dx) + abs(dy);
                    if (n > best) { best = n; gx = dx; gy = dy; }  // strict: ties keep the first channel
                    hp[c] = hc[c]; hc[c] = hn[c]; vp[c] = vc[c]; vc[c] = vn[c];
                }
                // direction (imgproc/src/canny.cpp): horizontal when |dy| < |dx| tan 22.5, vertical when |dy| > |dx| tan 67.5, else a
                // diagonal, (-1,-1)/(1,1) when dx and dy have the same sign, (-1,1)/(1,-1) otherwise
                const int ax = abs(gx), ay = abs(gy) << 15;
                const int t22 = ax * TG22, t67 = t22 + (ax << 16);
                const int code = ay < t22 ? 0 : (ay > t67 ? 1 : ((gx ^ gy) < 0 ? 3 : 2));
                const int y = y0 + r;
                mrow[k * kMP] = (x_in && y >= 0 && y < H) ? (best << 2 | code) : 0;
            }
        } else {
            // K = 5, 7: a K-row window of row sums; staged row of tile row r is r + 1 + R, staged pixel of column j is j + 16
            const unsigned char* col = s_in + (j + 16 - R) * C;
            int h[K][C], v[K][C];                                // row sums of the window's K staged rows, oldest first
            auto sums = [&](int sr, int* hs, int* vs) {          // hs: derivative taps across staged row sr, vs: smoothing taps
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const unsigned char* q = col + sr * S::in_row + c;
                    int a = 0, b = 0;
#pragma unroll
                    for (int t = 0; t < K; ++t) {
                        const int px = q[t * C];
                        if (deriv_tap(K, t)) a += deriv_tap(K, t) * px;
                        b += smooth_tap(K, t) * px;
                    }
                    hs[c] = a;
                    vs[c] = b;
                }
            };
#pragma unroll
            for (int i = 0; i < K - 1; ++i) sums(r0 + 1 + i, h[i], v[i]);
            int* mrow = s_m + (r0 + 1) * kMP + j + 4;
            for (int k = 0; k < kGroupRows; ++k) {
                const int r = r0 + k;
                sums(r + K, h[K - 1], v[K - 1]);
                int best = -1, gx = 0, gy = 0;
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    int dx = 0, dy = 0;
#pragma unroll
                    for (int i = 0; i < K; ++i) {
                        dx += smooth_tap(K, i) * h[i][c];
                        if (deriv_tap(K, i)) dy += deriv_tap(K, i) * v[i][c];
                    }
                    if (K == 7) {                                // cvRound(sum / 16): floor, then half to even
                        const int qx = dx >> 4, rx = dx & 15, qy = dy >> 4, ry = dy & 15;
                        dx = qx + (rx > 8 || (rx == 8 && (qx & 1)));
                        dy = qy + (ry > 8 || (ry == 8 && (qy & 1)));
                    }
                    const int n = L2 ? dx * dx + dy * dy : abs(dx) + abs(dy);
                    if (n > best) { best = n; gx = dx; gy = dy; }  // strict: ties keep the first channel
#pragma unroll
                    for (int i = 0; i < K - 1; ++i) { h[i][c] = h[i + 1][c]; v[i][c] = v[i + 1][c]; }
                }
                // the direction test of the K = 3 branch
                const int ax = abs(gx), ay = abs(gy) << 15;
                const int t22 = ax * TG22, t67 = t22 + (ax << 16);
                const int code = ay < t22 ? 0 : (ay > t67 ? 1 : ((gx ^ gy) < 0 ? 3 : 2));
                const int y = y0 + r;
                mrow[k * kMP] = (x_in && y >= 0 && y < H) ? (best << 2 | code) : 0;
            }
        }
    }
    __syncthreads();

    // ---- 3. non-maximum suppression, thresholds, class stores ----
    uint32_t weak_mask = 0;                                      // bit 4k + e: pixel e of this lane's quad in row warp + 8k
    if (warp < 8) {
        const int xq = x0 + 4 * lane;
        uint8_t* cls_f = RAGGED ? fd.cls : p.cls + (long long)frame * p.cls_frame_stride;
        const long long cls_pitch = RAGGED ? fd.cls_pitch : p.cls_pitch;
        const bool words = (RAGGED ? fd.cls_words : p.cls_words) && xq + 3 < W;
#pragma unroll 1
        for (int k = 0; k < kTH / 8; ++k) {
            const int r = warp + 8 * k, y = y0 + r;
            const int* c0 = s_m + (r + 1) * kMP + 4 + 4 * lane;   // centre row, column 4*lane
            int u[6], c[6], d[6];
            {
                const uint4 U = *reinterpret_cast<const uint4*>(c0 - kMP);
                const uint4 M = *reinterpret_cast<const uint4*>(c0);
                const uint4 D = *reinterpret_cast<const uint4*>(c0 + kMP);
                u[1] = U.x; u[2] = U.y; u[3] = U.z; u[4] = U.w;
                c[1] = M.x; c[2] = M.y; c[3] = M.z; c[4] = M.w;
                d[1] = D.x; d[2] = D.y; d[3] = D.z; d[4] = D.w;
                u[0] = __shfl_up_sync(0xffffffffu, (int)U.w, 1);
                c[0] = __shfl_up_sync(0xffffffffu, (int)M.w, 1);
                d[0] = __shfl_up_sync(0xffffffffu, (int)D.w, 1);
                u[5] = __shfl_down_sync(0xffffffffu, (int)U.x, 1);
                c[5] = __shfl_down_sync(0xffffffffu, (int)M.x, 1);
                d[5] = __shfl_down_sync(0xffffffffu, (int)D.x, 1);
                if (lane == 0) { u[0] = c0[-kMP - 1]; c[0] = c0[-1]; d[0] = c0[kMP - 1]; }
                if (lane == 31) { u[5] = c0[-kMP + 4]; c[5] = c0[4]; d[5] = c0[kMP + 4]; }
            }
            const int code4 = c[1] & 3 | (c[2] & 3) << 2 | (c[3] & 3) << 4 | (c[4] & 3) << 6;
#pragma unroll
            for (int i = 0; i < 6; ++i) { u[i] >>= 2; c[i] >>= 2; d[i] >>= 2; }
            uint32_t word = 0;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int m = c[e + 1], code = (code4 >> (2 * e)) & 3;
                // the test of every direction, then the one of this pixel's: a per-pixel choice of neighbours would be a divergent
                // branch.  `>` against the first neighbour, `>=` against the second except on the diagonals; never true for m = 0
                // (outside the image too)
                const uint32_t tests = (uint32_t)(m > c[e] && m >= c[e + 2]) | (uint32_t)(m > u[e + 1] && m >= d[e + 1]) << 1 |
                                       (uint32_t)(m > u[e] && m > d[e + 2]) << 2 | (uint32_t)(m > u[e + 2] && m > d[e]) << 3;
                const bool keep = (tests >> code) & 1;
                const bool strong = keep && m > p.hi, weak = keep && !strong && m > p.lo;
                word |= (strong ? 255u : weak ? 1u : 0u) << (8 * e);
                weak_mask |= (uint32_t)weak << (4 * k + e);
            }
            if (y < H) {
                uint8_t* o = cls_f + (long long)y * cls_pitch + xq;
                if (words) {
                    *reinterpret_cast<uint32_t*>(o) = word;
                } else {
                    for (int e = 0; e < 4 && xq + e < W; ++e) o[e] = (uint8_t)(word >> (8 * e));
                }
            }
        }
    }

    // ---- 4. weak pixels: union-find slots and list entries, one reservation per CTA ----
    const int cnt = __popc(weak_mask);
    int incl = cnt;
#pragma unroll
    for (int dlt = 1; dlt < 32; dlt <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, dlt);
        if (lane >= dlt) incl += t;
    }
    if (lane == 31) s_sum[warp] = (unsigned int)incl;
    __syncthreads();
    if (tid == 0) {
        unsigned int total = 0;
        for (int w = 0; w < kThreads / 32; ++w) { const unsigned int t = s_sum[w]; s_sum[w] = total; total += t; }
        s_sum[15] = total ? atomicAdd(p.kept_count, total) : 0u;
    }
    __syncthreads();
    if (weak_mask) {
        uint32_t* dst = p.kept_list + s_sum[15] + s_sum[warp] + (unsigned int)(incl - cnt);
        const long long g0 = (RAGGED ? (long long)fd.base : (long long)frame * p.out_frame_stride) + (long long)y0 * W + x0 + 4 * lane;
        uint32_t m = weak_mask;
        while (m) {
            const int bit = __ffs(m) - 1;
            m &= m - 1;
            const int g = (int)(g0 + (long long)(warp + 8 * (bit >> 2)) * W + (bit & 3));
            p.parent[g] = g;
            *dst++ = (uint32_t)g;
        }
    }
}

template <int C, bool L2, bool RAGGED, int K, int BR>
static int launch_cv(b200_ctx* ctx, cudaStream_t st, const FrontParams& p, const CvBlurParams& blur, dim3 grid) {
    static bool configured[64] = {false};  // per instantiation, per device
    if (!configured[ctx->device & 63]) {
        CB_CUDA(cudaFuncSetAttribute(front_cv_kernel<C, L2, RAGGED, K, BR>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     Smem<C, K, BR>::total));
        configured[ctx->device & 63] = true;
    }
    {
        ProfScope ps(ctx, st, 0);
        front_cv_kernel<C, L2, RAGGED, K, BR><<<grid, kThreads, Smem<C, K, BR>::total, st>>>(p, blur);
    }
    CB_CUDA(cudaGetLastError());
    ctx->launches++;
    return B200_OK;
}

// the instantiation for channels (1 or 3), l2, aperture (3, 5 or 7; checked by the caller) and the blur's radius class (the larger
// of blur.rx and blur.ry: 0 none, <= 3, <= 15)
template <bool RAGGED>
static int launch_cv_any(b200_ctx* ctx, cudaStream_t st, const FrontParams& p, const CvBlurParams& blur, dim3 grid, int channels,
                         bool l2, int aperture) {
    const int br = std::max(blur.rx, blur.ry);
    if (blur.rx < 0 || blur.ry < 0 || br > 15) {
        set_error("OpenCV front kernel: blur radii %d, %d (0 .. 15 are supported)", blur.rx, blur.ry);
        return B200_ERR_UNSUPPORTED;
    }
#define CB_CV_LAUNCH_BR(K, BR)                                                                                                             \
    if (channels == 1) return l2 ? launch_cv<1, true, RAGGED, K, BR>(ctx, st, p, blur, grid) : launch_cv<1, false, RAGGED, K, BR>(ctx, st, p, blur, grid); \
    if (channels == 3) return l2 ? launch_cv<3, true, RAGGED, K, BR>(ctx, st, p, blur, grid) : launch_cv<3, false, RAGGED, K, BR>(ctx, st, p, blur, grid);
#define CB_CV_LAUNCH(K)                                                                                                                  \
    if (aperture == K) {                                                                                                               \
        if (br == 0) { CB_CV_LAUNCH_BR(K, 0) }                                                                                         \
        else if (br <= 3) { CB_CV_LAUNCH_BR(K, 3) }                                                                                    \
        else { CB_CV_LAUNCH_BR(K, 15) }                                                                                                \
    }
    CB_CV_LAUNCH(3)
    CB_CV_LAUNCH(5)
    CB_CV_LAUNCH(7)
#undef CB_CV_LAUNCH
#undef CB_CV_LAUNCH_BR
    set_error("OpenCV front kernel: %d channels, aperture %d (1 or 3 channels, aperture 3, 5 or 7 are supported)", channels, aperture);
    return B200_ERR_UNSUPPORTED;
}

}  // namespace fcv

int launch_front_cv(b200_ctx* ctx, cudaStream_t st, const FrontParams& p_in, const CvBlurParams& blur, int channels, bool l2,
                    int aperture) {
    FrontParams p = p_in;
    if (!p.parent || !p.kept_list || !p.kept_count) { set_error("internal: OpenCV front kernel without a weak-pixel list"); return B200_ERR_INVALID_ARG; }
    // aligned 32-bit class stores need base, row pitch and frame stride on 4-byte boundaries (tile columns are multiples of 4)
    p.cls_words = ((reinterpret_cast<uintptr_t>(p.cls) | (uintptr_t)p.cls_pitch | (uintptr_t)(p.n_frames > 1 ? p.cls_frame_stride : 0)) & 3) == 0;
    const dim3 grid((p.width + fcv::kTW - 1) / fcv::kTW, (p.height + fcv::kTH - 1) / fcv::kTH, p.n_frames);
    ctx->front_fast++;
    return fcv::launch_cv_any<false>(ctx, st, p, blur, grid, channels, l2, aperture);
}

void ragged_items_cv(int frame, int height, int width, std::vector<RaggedItem>& items) {
    for (int y0 = 0; y0 < height; y0 += fcv::kTH)
        for (int x0 = 0; x0 < width; x0 += fcv::kTW) items.push_back(RaggedItem{frame, x0, y0, std::min(height, y0 + fcv::kTH)});
}

int launch_front_cv_ragged(b200_ctx* ctx, cudaStream_t st, const FrontParams& p, const CvBlurParams& blur, int n_items, int channels,
                           bool l2, int aperture) {
    if (!p.parent || !p.kept_list || !p.kept_count || !p.rframes || !p.ritems) {
        set_error("internal: ragged OpenCV front kernel without its table or weak-pixel list");
        return B200_ERR_INVALID_ARG;
    }
    if (n_items <= 0) return B200_OK;
    const dim3 grid(n_items);
    ctx->front_fast++;
    return fcv::launch_cv_any<true>(ctx, st, p, blur, grid, channels, l2, aperture);
}

}  // namespace cb
