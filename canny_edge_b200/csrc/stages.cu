// stages.cu — stand-alone kernels behind the stage-level entry points that take ARBITRARY int16 planes
// (b200_xy_gradient, b200_sobel, b200_nonmaximal).  The fused front kernel (front.cu) is the production
// path; these exist because the reference exposes every stage as a public, individually tested function
// (tests/utils/test_utils.cpp) and callers may feed them planes that never came from a blur (the
// reference's own 3x3 vectors do).  Same exact integer arithmetic (canny_math.h), plain coalesced
// global-memory stencils.
#include <math.h>

#include <algorithm>

#include "canny_math.h"
#include "internal.h"

namespace cb {

// calculateXYGradient, src/utils.cpp:106-187.  Results are truncated to int16 as the reference's `short`
// stores do.
__device__ __forceinline__ void xy_at(const int16_t* __restrict__ b, int h, int w, int r, int c, int& gx, int& gy) {
    const int cl = c > 0 ? c - 1 : c, cr = c < w - 1 ? c + 1 : c;
    const int ru = r > 0 ? r - 1 : r, rd = r < h - 1 ? r + 1 : r;
    const int16_t* row = b + (size_t)r * w;
    int v = 2 * row[cr] - 2 * row[cl];
    if (r != h - 1) v += row[w + cr] - row[w + cl];
    if (r != 0) v += row[cr - w] - row[cl - w];
    const int16_t* up = b + (size_t)ru * w;
    const int16_t* dn = b + (size_t)rd * w;
    int u = 2 * dn[c] - 2 * up[c];
    if (c != w - 1) u += dn[c + 1] - up[c + 1];
    if (c != 0) u += dn[c - 1] - up[c - 1];
    gx = (int16_t)v;
    gy = (int16_t)u;
}

__global__ void xy_gradient_kernel(const int16_t* __restrict__ b, int h, int w, int16_t* __restrict__ gx, int16_t* __restrict__ gy) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y * blockDim.y + threadIdx.y;
    if (c >= w || r >= h) return;
    int x, y;
    xy_at(b, h, w, r, c, x, y);
    gx[(size_t)r * w + c] = (int16_t)x;
    gy[(size_t)r * w + c] = (int16_t)y;
}

// sobelOperator, src/utils.cpp:201-236.
__global__ void sobel_kernel(const int16_t* __restrict__ b, int h, int w, int16_t* __restrict__ mag, int16_t* __restrict__ ang) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y * blockDim.y + threadIdx.y;
    if (c >= w || r >= h) return;
    int x, y;
    xy_at(b, h, w, r, c, x, y);
    const int n = x * x + y * y;  // int, as src/utils.cpp:212
    int m;
    int code;
    const int ax = x < 0 ? -x : x, ay = y < 0 ? -y : y;
    if (ax <= 1020 && ay <= 1020) {
        // the range a blurred 8-bit image can produce: exact integer magnitude and direction
        m = (int)sqrtf((float)n);
        if (m * m > n) --m;
        if ((m + 1) * (m + 1) <= n) ++m;
        code = direction_code<int>(x, y);
    } else {
        // gradients no real image produces (raw int16 test planes): follow the reference's float expressions
        m = (int)sqrt((double)n);
        float th = (float)atan2((double)y, (double)x);
        th = (float)((double)th * (180 / 3.1415926535));
        if (th < 0) th = 360 + th;
        if ((th >= 22.5 && th < 67.5) || (th >= 202.5 && th < 247.5)) code = DIR_45;
        else if ((th >= 112.5 && th < 157.5) || (th >= 292.5 && th < 337.5)) code = DIR_135;
        else if ((th >= 67.5 && th < 112.5) || (th >= 247.5 && th < 292.5)) code = DIR_90;
        else code = DIR_0;
    }
    mag[(size_t)r * w + c] = (int16_t)m;
    ang[(size_t)r * w + c] = (int16_t)dir_code_to_angle(code);
}

// nonmaximalSuppression, src/utils.cpp:248-308.  An angle other than 0/45/90/135 leaves the element
// unwritten in the reference; 0 is written here.
__global__ void nonmaximal_kernel(const int16_t* __restrict__ mag, const int16_t* __restrict__ ang, int h, int w, int16_t* __restrict__ out) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y * blockDim.y + threadIdx.y;
    if (c >= w || r >= h) return;
    const size_t i = (size_t)r * w + c;
    const int a = ang[i];
    int dr, dc;
    if (a == 0) { dr = 0; dc = 1; }
    else if (a == 45) { dr = -1; dc = 1; }
    else if (a == 90) { dr = 1; dc = 0; }
    else if (a == 135) { dr = 1; dc = 1; }
    else { out[i] = 0; return; }
    const int m = mag[i];
    bool keep = true;
    {
        const int rr = r + dr, cc = c + dc;
        if (rr >= 0 && rr < h && cc >= 0 && cc < w && m <= mag[(size_t)rr * w + cc]) keep = false;
    }
    {
        const int rr = r - dr, cc = c - dc;
        if (rr >= 0 && rr < h && cc >= 0 && cc < w && m <= mag[(size_t)rr * w + cc]) keep = false;
    }
    out[i] = keep ? (int16_t)m : (int16_t)0;
}

static dim3 grid2d(int h, int w, dim3 block) { return dim3((w + block.x - 1) / block.x, (h + block.y - 1) / block.y); }

int launch_xy_gradient(b200_ctx* ctx, cudaStream_t st, const int16_t* blur, int h, int w, int16_t* gx, int16_t* gy) {
    dim3 block(64, 4);
    xy_gradient_kernel<<<grid2d(h, w, block), block, 0, st>>>(blur, h, w, gx, gy);
    CB_CUDA(cudaGetLastError());
    ctx->launches++;
    return B200_OK;
}
int launch_sobel(b200_ctx* ctx, cudaStream_t st, const int16_t* blur, int h, int w, int16_t* mag, int16_t* ang) {
    dim3 block(64, 4);
    sobel_kernel<<<grid2d(h, w, block), block, 0, st>>>(blur, h, w, mag, ang);
    CB_CUDA(cudaGetLastError());
    ctx->launches++;
    return B200_OK;
}
int launch_nonmaximal(b200_ctx* ctx, cudaStream_t st, const int16_t* mag, const int16_t* ang, int h, int w, int16_t* out) {
    dim3 block(64, 4);
    nonmaximal_kernel<<<grid2d(h, w, block), block, 0, st>>>(mag, ang, h, w, out);
    CB_CUDA(cudaGetLastError());
    ctx->launches++;
    return B200_OK;
}

// ---------------------------------------------------------------------------------------------
// BGR -> gray: the step right before the hot path in the reference (cvtColor(frame, gray, COLOR_BGR2GRAY), src/main.cpp:113).
// OpenCV's 8-bit path is fixed point: (B*3735 + G*19235 + R*9798 + 2^14) >> 15 (coefficients 0.114 / 0.587 / 0.299 in 15 bits);
// tests/test_bgr.py checks the kernel against cv2.cvtColor itself.  One thread per 4 pixels: three 32-bit loads, one 32-bit store.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t gray_of(uint32_t b, uint32_t g, uint32_t r) { return (b * 3735u + g * 19235u + r * 9798u + 16384u) >> 15; }

__global__ void bgr_to_gray_kernel(const uint8_t* __restrict__ bgr, uint8_t* __restrict__ gray, size_t n_px) {
    const size_t n4 = n_px / 4;
    const bool aligned = ((reinterpret_cast<uintptr_t>(bgr) | reinterpret_cast<uintptr_t>(gray)) & 3) == 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
        if (aligned) {
            const uint32_t* src = reinterpret_cast<const uint32_t*>(bgr) + 3 * i;
            const uint32_t w0 = __ldcs(src), w1 = __ldcs(src + 1), w2 = __ldcs(src + 2);   // B0 G0 R0 B1 | G1 R1 B2 G2 | R2 B3 G3 R3
            const uint32_t g0 = gray_of(w0 & 255, (w0 >> 8) & 255, (w0 >> 16) & 255);
            const uint32_t g1 = gray_of(w0 >> 24, w1 & 255, (w1 >> 8) & 255);
            const uint32_t g2 = gray_of((w1 >> 16) & 255, w1 >> 24, w2 & 255);
            const uint32_t g3 = gray_of((w2 >> 8) & 255, (w2 >> 16) & 255, w2 >> 24);
            reinterpret_cast<uint32_t*>(gray)[i] = g0 | (g1 << 8) | (g2 << 16) | (g3 << 24);
        } else {
            for (int k = 0; k < 4; ++k) {
                const uint8_t* px = bgr + 3 * (4 * i + k);
                gray[4 * i + k] = (uint8_t)gray_of(px[0], px[1], px[2]);
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x < (n_px & 3)) {
        const size_t i = (n_px & ~(size_t)3) + threadIdx.x;
        gray[i] = (uint8_t)gray_of(bgr[3 * i], bgr[3 * i + 1], bgr[3 * i + 2]);
    }
}

int launch_bgr_to_gray(b200_ctx* ctx, cudaStream_t st, const uint8_t* bgr, uint8_t* gray, size_t n_px) {
    size_t blocks = (n_px / 4 + 255) / 256;
    const size_t cap = 32 * (size_t)(ctx->sm_count > 0 ? ctx->sm_count : 148);
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    bgr_to_gray_kernel<<<(int)blocks, 256, 0, st>>>(bgr, gray, n_px);
    CB_CUDA(cudaGetLastError());
    ctx->launches++;
    return B200_OK;
}

// The same conversion from pitched frames (row y of frame f at f*frame_stride + y*pitch) into a dense gray plane: what BGR frames
// the front kernel cannot convert while staging go through.  One block-row per image row; byte loads, so any pitch and offset work.
__global__ void bgr_to_gray_strided_kernel(const uint8_t* __restrict__ bgr, long long pitch, long long frame_stride, int h, int w,
                                           long long rows, uint8_t* __restrict__ gray) {
    for (long long r = blockIdx.x; r < rows; r += gridDim.x) {
        const long long f = r / h, y = r - f * h;
        const uint8_t* src = bgr + f * frame_stride + y * pitch;
        uint8_t* dst = gray + r * w;
        for (int x = threadIdx.x; x < w; x += blockDim.x)
            dst[x] = (uint8_t)gray_of(__ldcs(src + 3 * x), __ldcs(src + 3 * x + 1), __ldcs(src + 3 * x + 2));
    }
}

int launch_bgr_to_gray_strided(b200_ctx* ctx, cudaStream_t st, const uint8_t* bgr, long long pitch, long long frame_stride,
                               int n_frames, int h, int w, uint8_t* gray) {
    const long long rows = (long long)n_frames * h;
    const long long cap = 32LL * (ctx->sm_count > 0 ? ctx->sm_count : 148);
    const int blocks = (int)std::max<long long>(1, std::min(rows, cap));
    bgr_to_gray_strided_kernel<<<blocks, 256, 0, st>>>(bgr, pitch, frame_stride, h, w, rows, gray);
    CB_CUDA(cudaGetLastError());
    ctx->launches++;
    return B200_OK;
}

// The same conversion for the frames of a ragged chunk, driven by the chunk's job table: block-rows walk the chunk's row space,
// and row r belongs to the last job whose row0 is <= r (binary search).
__global__ void bgr_to_gray_ragged_kernel(const RaggedGrayJob* __restrict__ jobs, int n_jobs, long long rows) {
    for (long long r = blockIdx.x; r < rows; r += gridDim.x) {
        int lo = 0, hi = n_jobs - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (jobs[mid].row0 <= r) lo = mid; else hi = mid - 1;
        }
        const RaggedGrayJob j = jobs[lo];
        const long long y = r - j.row0;
        const uint8_t* src = j.bgr + y * j.bgr_pitch;
        uint8_t* dst = j.gray + y * j.gray_pitch;
        for (int x = threadIdx.x; x < j.width; x += blockDim.x)
            dst[x] = (uint8_t)gray_of(__ldcs(src + 3 * x), __ldcs(src + 3 * x + 1), __ldcs(src + 3 * x + 2));
    }
}

int launch_bgr_to_gray_ragged(b200_ctx* ctx, cudaStream_t st, const RaggedGrayJob* jobs, int n_jobs, long long rows) {
    const long long cap = 32LL * (ctx->sm_count > 0 ? ctx->sm_count : 148);
    const int blocks = (int)std::max<long long>(1, std::min(rows, cap));
    bgr_to_gray_ragged_kernel<<<blocks, 256, 0, st>>>(jobs, n_jobs, rows);
    CB_CUDA(cudaGetLastError());
    ctx->launches++;
    return B200_OK;
}

}  // namespace cb
