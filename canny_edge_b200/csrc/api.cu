// api.cu — the extern "C" boundary (include/canny_b200.h): context, workspace pool, Gaussian tables,
// stage entry points on host buffers, batched device/host pipelines.
#include <limits.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <emmintrin.h>  // _mm_stream_si64 / _mm_stream_si128 / _mm_sfence (SSE2, x86-64 baseline): non-temporal stores of the expanded edge map

#include <sched.h>

#include <algorithm>
#include <condition_variable>
#include <fstream>
#include <functional>
#include <sstream>
#include <mutex>
#include <thread>

#include <cuda.h>

#include "canny_math.h"
#include "internal.h"

namespace cb {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

// ---- Gaussian weights: the reference's host code, expression for expression (src/utils.cpp:77-95) ----
int host_window(float sigma) {
    const float t = 3 * sigma;            // float product
    return (int)(1 + 2 * ceilf(t));       // std::ceil(float) -> float; 1 + 2*c in float; truncation to int
}
void host_gaussian_kernel(float sigma, std::vector<float>& w) {
    const int n = host_window(sigma);
    const int mid = n / 2;
    w.assign((size_t)n, 0.f);
    float total = 0.0f;
    for (int i = 0; i < n; i++) {
        const float x = (float)(i - mid);
        const float e = expf(-((x * x) / (2 * sigma * sigma)));  // std::exp(float)
        const float pr = (float)((double)e / (sqrt(6.2831853) * (double)sigma));
        w[(size_t)i] = pr;
        total += pr;
    }
    for (int i = 0; i < n; i++) w[(size_t)i] /= total;
}

int ensure_ws(Workspace& ws, size_t bytes, bool pinned_host) {
    if (ws.bytes >= bytes && ws.ptr) return B200_OK;
    if (ws.ptr) {
        if (pinned_host) cudaFreeHost(ws.ptr); else cudaFree(ws.ptr);
        ws.ptr = nullptr;
        ws.bytes = 0;
    }
    const size_t want = bytes + bytes / 8 + 256;  // slack so slowly growing requests do not realloc each time
    cudaError_t e = pinned_host ? cudaMallocHost(&ws.ptr, want) : cudaMalloc(&ws.ptr, want);
    if (e != cudaSuccess) {
        ws.ptr = nullptr;
        set_error("workspace allocation of %zu bytes failed: %s", want, cudaGetErrorString(e));
        cudaGetLastError();
        return B200_ERR_NOMEM;
    }
    ws.bytes = want;
    if (!pinned_host) {
        // the head of a fresh device workspace is zero: the weak-pixel lists keep their counter block there (HystParams::ctr).
        // Synchronous on purpose (allocation is rare): the context's streams do not order themselves after the null stream.
        e = cudaMemset(ws.ptr, 0, 64);
        if (e == cudaSuccess) e = cudaStreamSynchronize(0);
        if (e != cudaSuccess) { set_error("workspace initialisation failed: %s", cudaGetErrorString(e)); cudaGetLastError(); return B200_ERR_CUDA; }
    }
    return B200_OK;
}

// Builds (or reuses) the weight / count / reciprocal tables for `sigma` and uploads them.
int prepare_gauss(b200_ctx* ctx, float sigma) {
    GaussTables& g = ctx->gauss;
    if (g.sigma == sigma && g.d_w) return B200_OK;
    if (!(sigma > 0.f) || !isfinite(sigma)) {
        set_error("sigma must be a finite positive float (got %g)", (double)sigma);
        return B200_ERR_INVALID_ARG;
    }
    const int window = host_window(sigma);
    const int radius = window / 2;
    if (radius < 1 || radius > B200_MAX_RADIUS) {
        set_error("sigma %g gives window %d; supported half-window is 1..%d", (double)sigma, window, B200_MAX_RADIUS);
        return B200_ERR_UNSUPPORTED;
    }
    host_gaussian_kernel(sigma, g.w);
    const int n1 = radius + 1;
    g.count.assign((size_t)2 * n1 * n1, 0.f);
    for (int a = 0; a <= radius; ++a) {
        for (int b = 0; b <= radius; ++b) {
            float c = 0.f;  // `count += kernel[center+k]` over the in-image taps, ascending (src/utils.cpp:44,59)
            for (int t = a; t <= 2 * radius - b; ++t) c += g.w[(size_t)t];
            g.count[(size_t)a * n1 + b] = c;
            // RN(1/c): the double quotient rounds to the same float as an exact one (53 >= 2*24+2 bits)
            g.count[(size_t)n1 * n1 + (size_t)a * n1 + b] = (c != 0.f) ? (float)(1.0 / (double)c) : 0.f;
        }
    }
    // one device allocation for both tables, sized for the largest radius so it is made once
    if (!g.d_w) {
        const size_t cap = sizeof(float) * ((2 * B200_MAX_RADIUS + 1) + 2 * (B200_MAX_RADIUS + 1) * (B200_MAX_RADIUS + 1));
        CB_CUDA(cudaMalloc(reinterpret_cast<void**>(&g.d_w), cap));
        g.d_count = g.d_w + (2 * B200_MAX_RADIUS + 1);
    }
    // the tables may still be in use by kernels of a previous sigma: order the upload after them
    CB_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int s = 0; s < 3; ++s) CB_CUDA(cudaStreamSynchronize(ctx->side[s]));
    CB_CUDA(cudaMemcpyAsync(g.d_w, g.w.data(), sizeof(float) * g.w.size(), cudaMemcpyHostToDevice, ctx->stream));
    CB_CUDA(cudaMemcpyAsync(g.d_count, g.count.data(), sizeof(float) * g.count.size(), cudaMemcpyHostToDevice, ctx->stream));
    CB_CUDA(cudaStreamSynchronize(ctx->stream));
    {
        float wmin = g.w[0];
        for (float v : g.w) wmin = v < wmin ? v : wmin;
        g.tiny = !((double)wmin * (double)wmin >= 8.077935669463161e-28);  // 2^-90
    }
    g.div_mode = 5;
    g.div_c = (float)(1.0 / (double)g.count[0] - 1.0);
    if (!g.tiny) CB_TRY(check_div_mode_device(ctx, g.count[0], g.count[(size_t)n1 * n1], &g.div_c, &g.div_mode));
    g.sigma = sigma;
    g.window = window;
    g.radius = radius;
    return B200_OK;
}

// ---- host side of the transfers: a small thread pool -------------------------------------------------------------
// b200_canny_batch_host sends the edge map over PCIe as 1 bit per pixel (the link is the bottleneck of the host path: with both
// directions carrying 1 B/px it saturates at ~46 GB/s each way) and expands it to the 0 / 255 bytes (or int16 values) of the
// reference's result on the host, with a small pool of threads that runs while the GPU works on the following chunks.  The same
// pool copies PAGEABLE caller buffers into the context's pinned staging memory: a cudaMemcpy from pageable memory goes through
// the driver's own single-threaded staging (~10 GB/s); several threads filling a pinned buffer that is then DMA'd are 2-3x faster.
struct HostPool {
    enum Job { kUnpackU8, kUnpackI16, kCopy };
    std::vector<std::thread> workers;
    std::mutex mu;
    std::condition_variable cv_go, cv_done;
    Job job = kCopy;
    const uint8_t* src = nullptr;
    uint8_t* dst = nullptr;
    size_t n_items = 0;   // pixels (unpack jobs) or bytes (copy)
    int generation = 0, pending = 0;
    bool stop = false;
    uint64_t lut[256];                    // bit pattern -> eight 0 / 255 bytes
    alignas(16) int16_t lut16[256][8];    // bit pattern -> eight 0 / 255 int16 values

    explicit HostPool(int n_threads) {
        for (int b = 0; b < 256; ++b) {
            uint64_t v = 0;
            for (int i = 0; i < 8; ++i) {
                if (b & (1 << i)) v |= 0xFFull << (8 * i);
                lut16[b][i] = (b & (1 << i)) ? 255 : 0;
            }
            lut[b] = v;
        }
        for (int t = 0; t < n_threads; ++t) workers.emplace_back([this, t] { loop(t); });
    }
    ~HostPool() {
        { std::lock_guard<std::mutex> lk(mu); stop = true; }
        cv_go.notify_all();
        for (auto& w : workers) w.join();
    }
    int parts() const { return (int)workers.size() + 1; }
    // units [u0, u1) of the current job: a unit is one packed input byte (8 pixels) for the unpack jobs, 64 bytes for a copy
    void range(size_t u0, size_t u1) {
        if (job == kCopy) {
            const size_t b0 = std::min(n_items, u0 * 64), b1 = std::min(n_items, u1 * 64);
            memcpy(dst + b0, src + b0, b1 - b0);
        } else if (job == kUnpackU8) {
            if ((reinterpret_cast<uintptr_t>(dst) & 7) == 0) {
                // streaming stores: the 64 bytes made from 8 input bytes fill one cache line, so the line is written without
                // first being read (the host path is bound by host-memory traffic: PCIe reads the frames from the same DRAM)
                long long* out = reinterpret_cast<long long*>(dst);
                for (size_t i = u0; i < u1; ++i) _mm_stream_si64(out + i, (long long)lut[src[i]]);
                _mm_sfence();
            } else {
                for (size_t i = u0; i < u1; ++i) memcpy(dst + 8 * i, &lut[src[i]], 8);
            }
        } else {
            if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
                __m128i* out = reinterpret_cast<__m128i*>(dst);
                for (size_t i = u0; i < u1; ++i) _mm_stream_si128(out + i, _mm_load_si128(reinterpret_cast<const __m128i*>(lut16[src[i]])));
                _mm_sfence();
            } else {
                for (size_t i = u0; i < u1; ++i) memcpy(dst + 16 * i, lut16[src[i]], 16);
            }
        }
    }
    size_t units() const { return job == kCopy ? (n_items + 63) / 64 : n_items / 8; }
    void tail() {  // the last few pixels of an unpack job whose pixel count is not a multiple of 8
        if (job == kCopy) return;
        for (size_t px = 8 * (n_items / 8); px < n_items; ++px) {
            const int v = ((src[px >> 3] >> (px & 7)) & 1) ? 255 : 0;
            if (job == kUnpackU8) dst[px] = (uint8_t)v; else reinterpret_cast<int16_t*>(dst)[px] = (int16_t)v;
        }
    }
    void slice(int part) {  // part-th of parts() slices, on multiples of 8 units
        const size_t n = units();
        const size_t per = ((n + parts() - 1) / parts() + 7) & ~(size_t)7;
        const size_t u0 = std::min(n, per * (size_t)part), u1 = std::min(n, u0 + per);
        range(u0, u1);
    }
    void loop(int t) {
        int seen = 0;
        while (true) {
            {
                std::unique_lock<std::mutex> lk(mu);
                cv_go.wait(lk, [&] { return stop || generation != seen; });
                if (stop) return;
                seen = generation;
            }
            slice(t);
            {
                std::lock_guard<std::mutex> lk(mu);
                if (--pending == 0) cv_done.notify_one();
            }
        }
    }
    // runs one job over n items and returns when it is done; the caller's thread takes a slice too.  Jobs too small to be worth
    // waking the workers (a few microseconds of work) run on the caller's thread alone.
    void run(Job j, const void* s, void* d, size_t n) {
        const size_t out_bytes = j == kCopy ? n : (j == kUnpackU8 ? n : 2 * n);
        if (workers.empty() || out_bytes < (256u << 10)) {
            job = j; src = static_cast<const uint8_t*>(s); dst = static_cast<uint8_t*>(d); n_items = n;
            range(0, units());
            tail();
            return;
        }
        {
            std::lock_guard<std::mutex> lk(mu);
            job = j; src = static_cast<const uint8_t*>(s); dst = static_cast<uint8_t*>(d); n_items = n;
            pending = (int)workers.size();
            ++generation;
        }
        cv_go.notify_all();
        slice(parts() - 1);
        tail();
        std::unique_lock<std::mutex> lk(mu);
        cv_done.wait(lk, [&] { return pending == 0; });
    }
};

// measured on the B200 hosts (tools/e2e_probe.py, tools/e2e_multi.sh): 4 threads (3 workers + the caller) keep up with the link
// when one process owns the host (e2e 52.7 Gpix/s with 4, 50 with 6-8, 45 with 10, 34 with 16 threads: more of them only fight
// the DMA engine for host-memory bandwidth); with 8 processes on a 32-vCPU host 2 each are best (aggregate 131 Gpix/s against 87
// with 4 and 104 with 1).  LOCAL_WORLD_SIZE is what torchrun exports.
static HostPool* get_pool(b200_ctx* ctx) {
    if (!ctx->pool) {
        unsigned hc = std::thread::hardware_concurrency();
        int local_world = 1;
        if (const char* e = getenv("LOCAL_WORLD_SIZE")) local_world = std::max(1, atoi(e));
        int n_threads = (int)std::min<unsigned>(std::max<unsigned>((hc ? hc : 4) / (2u * (unsigned)local_world), 1), 4) - 1;
        // eight processes saturate the host's memory system with 2 threads each however many cores there are (a later 8-GPU bench
        // run on a host with more vCPUs, 4 threads per rank by the rule above, reproduced the 87 Gpix/s of the 4-thread probe)
        if (local_world >= 8) n_threads = std::min(n_threads, 1);
        if (const char* e = getenv("B200_CANNY_UNPACK_THREADS")) n_threads = std::max(0, atoi(e) - 1);
        ctx->pool = new HostPool(std::max(0, n_threads));
    }
    return ctx->pool;
}

// Staging pageable memory through the pool pays for large jobs only (measured on the B200 hosts, tools/latency_probe.py: an
// 8192x8192 frame from / to pageable memory 13.6 -> 6.3 ms with int16 output, 8.5 -> 5.8 ms with byte output; a 1080p or 4K frame
// gets slower, the thread wake-ups and the hosts' modest per-core memory bandwidth cost more than the driver's own pageable path)
constexpr long long kStageMinBytes = 32LL << 20;

// true when `p` is ordinary pageable host memory (not pinned / registered / managed): such buffers are staged by the pool
static bool is_pageable(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return true;
    }
    return a.type == cudaMemoryTypeUnregistered;
}

static std::mutex g_default_mu;
static b200_ctx* g_default_ctx = nullptr;

static int resolve_ctx(b200_ctx*& ctx) {
    if (ctx) {
        CB_CUDA(cudaSetDevice(ctx->device));
        return B200_OK;
    }
    std::lock_guard<std::mutex> lk(g_default_mu);
    if (!g_default_ctx) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) {
            cudaGetLastError();
            set_error("no CUDA device available (libcanny_b200 has no CPU fallback)");
            return B200_ERR_NO_DEVICE;
        }
        CB_TRY(b200_ctx_create(dev, &g_default_ctx));
    }
    ctx = g_default_ctx;
    CB_CUDA(cudaSetDevice(ctx->device));
    return B200_OK;
}

// min_side: 2 for the reference's semantics, 1 for the OpenCV-compatible path (cv::Canny takes any image of at least one pixel)
static int check_image(const void* in, const void* out, int h, int w, int min_side = 2) {
    if (!in || !out) { set_error("null image pointer"); return B200_ERR_INVALID_ARG; }
    if (h < min_side || w < min_side) { set_error("height and width must be >= %d (got %dx%d)", min_side, h, w); return B200_ERR_INVALID_ARG; }
    if ((long long)h * w >= (1LL << 31)) { set_error("image of %dx%d pixels exceeds int indexing", h, w); return B200_ERR_UNSUPPORTED; }
    return B200_OK;
}

static int check_thresholds(int lo, int hi) {
    if (!thresholds_supported(lo, hi)) {
        set_error("thresholds minVal=%d > 255 >= maxVal=%d: the reference's result depends on its flood order there (src/utils.cpp:327-340); not reproduced", lo, hi);
        return B200_ERR_UNSUPPORTED;
    }
    return B200_OK;
}

// Byte strides of the caller's frames and edge maps (b200_canny_batch_device_strided); null means dense: rows of width (3*width
// for BGR) bytes, frames of height rows
struct FrameLayout {
    long long in_pitch, in_frame_stride, out_pitch, out_frame_stride;
};

// Runs front + hysteresis on device-resident frames [f0, f0+nf) using workspace slot `slot` on stream st.
// bgr: d_in holds interleaved B,G,R frames (3 bytes per pixel) and the front kernel converts while staging (front3_bgr_supports)
// bands_hint > 0: row bands per frame for the front kernel's grid (0: the launcher's own choice)
// lay: strides of d_in and d_out (null: dense).  The union-find slots and the weak-pixel list stay dense whatever they are.
static int run_frames_device(b200_ctx* ctx, cudaStream_t st, int slot, const uint8_t* d_in, uint8_t* d_out, int nf, int h,
                             int w, int lo, int hi, int16_t* blur, int16_t* mag, int16_t* ang, int16_t* nms, bool bgr = false,
                             int bands_hint = 0, const FrameLayout* lay = nullptr) {
    const long long px = (long long)h * w;
    const int bpp = bgr ? 3 : 1;
    const FrameLayout dense_layout = {bpp * (long long)w, bpp * px, w, px};
    if (!lay) lay = &dense_layout;
    FrontParams fp;
    memset(&fp, 0, sizeof(fp));
    fp.in = d_in; fp.in_pitch = lay->in_pitch; fp.in_frame_stride = lay->in_frame_stride; fp.in_bgr = bgr ? 1 : 0;
    fp.in_row0 = 0; fp.in_rows = h; fp.width = w; fp.height = h;
    fp.out_row0 = 0; fp.out_rows = h; fp.n_frames = nf; fp.out_frame_stride = px;
    fp.cls = d_out; fp.cls_pitch = lay->out_pitch; fp.cls_frame_stride = lay->out_frame_stride;
    fp.blur = blur; fp.mag = mag; fp.ang = ang; fp.nms = nms;
    fp.tiles_y = bands_hint;
    fp.w = ctx->gauss.d_w; fp.count = ctx->gauss.d_count; fp.radius = ctx->gauss.radius;
    fill_thresholds(fp, lo, hi);
    // sparse hand-over to hysteresis (used when the lean front kernel runs): union-find slots + weak-pixel list
    fp.parent = reinterpret_cast<int32_t*>(ctx->ws_parent[slot].ptr);
    fp.kept_count = reinterpret_cast<unsigned int*>(ctx->ws_list[slot].ptr);
    fp.kept_list = reinterpret_cast<uint32_t*>(ctx->ws_list[slot].ptr) + 16;
    // the list's counter block is zero here: zeroed at allocation and retired by the previous launch's kernels (HystParams::ctr);
    // only a launch that failed half-way leaves it dirty
    if (ctx->list_dirty[slot]) CB_CUDA(cudaMemsetAsync(fp.kept_count, 0, 64, st));
    ctx->list_dirty[slot] = true;
    bool sparse = false;
    CB_TRY(launch_front(ctx, st, fp, &sparse));
    static const long long dense_div = [] { const char* e = getenv("B200_CANNY_DENSE_DIV"); return e ? atoll(e) : 8LL; }();
    // weak-pixel count of the previous launch of this slot (written into mapped pinned memory by its kernels, never waited for)
    const unsigned int prev_kept = *reinterpret_cast<volatile unsigned int*>(&ctx->h_kept[slot]);
    const bool dense = ctx->kept_px[slot] > 0 && (long long)prev_kept * dense_div > ctx->kept_px[slot];
    if (sparse) ctx->kept_px[slot] = (long long)nf * px;
    const long long thresh = (long long)nf * px / dense_div;   // n * dense_div > px  <=>  n > floor(px / dense_div)
    HystParams hp;
    memset(&hp, 0, sizeof(hp));
    hp.cls = d_out; hp.cls_pitch = lay->out_pitch; hp.cls_frame_stride = lay->out_frame_stride;
    hp.list = (sparse && !dense) ? fp.kept_list : nullptr;
    hp.ctr = sparse ? fp.kept_count : nullptr;
    hp.h_kept = ctx->d_kept + slot;
    hp.kept_prev = prev_kept;
    hp.kept_thresh = (unsigned int)std::min<long long>(thresh, 0xffffffffLL);
    hp.parent = reinterpret_cast<int32_t*>(ctx->ws_parent[slot].ptr);
    hp.frame_stride = px; hp.rows = h; hp.width = w; hp.row0 = 0; hp.n_frames = nf;
    // Small launches (the single-frame latency configuration) chain front -> link -> resolve by programmatic dependent launch: the
    // next kernel's blocks are resident before its predecessor has drained.  Not for batch chunks: parked blocks would hold the
    // SM resources the PREVIOUS chunk's hysteresis kernels (other stream) are meant to use next to the front kernel's CTAs.
    static const int pdl_env = [] { const char* e = getenv("B200_CANNY_PDL"); return e ? atoi(e) : -1; }();
    hp.pdl = pdl_env >= 0 ? pdl_env : ((long long)nf * px <= (4LL << 20) ? 1 : 0);
    if (ctx->prof.on) hp.pdl = 0;   // per-kernel event pairs need the kernels apart
    CB_TRY(launch_hysteresis(ctx, st, hp));
    ctx->list_dirty[slot] = false;
    return B200_OK;
}

// whether launch_front takes these interleaved B,G,R frames directly (fused conversion) under the context's current sigma
static bool bgr_fused_ok(const b200_ctx* ctx, const uint8_t* d_bgr, int n, int h, int w, long long pitch, long long frame_stride) {
    FrontParams fp;
    memset(&fp, 0, sizeof(fp));
    fp.in = d_bgr; fp.in_pitch = pitch; fp.in_frame_stride = frame_stride; fp.n_frames = n; fp.in_rows = h; fp.width = w;
    return front3_bgr_supports(ctx->gauss, fp);
}

// The OpenCV-compatible path (b200_cv_canny_aperture_device_strided): cv::Canny's thresholds as integers in magnitude space
// (divided by 16 for aperture 7, swapped, clamped and squared for L2, floored), the input's channel count and the Sobel aperture
struct CvSpec {
    int lo, hi;
    int channels;
    bool l2;
    int aperture;   // 3, 5 or 7
};

// Front + hysteresis with cv::Canny's semantics on frames [f0, f0+nf) of slot `slot` (run_frames_device's counterpart): the
// OpenCV front kernel, then always the list-driven hysteresis kernels with plain 8-connectivity.  The uniform path's density state
// (h_kept, kept_px) is neither read nor written.
static int run_frames_cv(b200_ctx* ctx, cudaStream_t st, int slot, const uint8_t* d_in, uint8_t* d_out, int nf, int h, int w,
                         const CvSpec& cv, const FrameLayout& lay) {
    const long long px = (long long)h * w;
    FrontParams fp;
    memset(&fp, 0, sizeof(fp));
    fp.in = d_in; fp.in_pitch = lay.in_pitch; fp.in_frame_stride = lay.in_frame_stride; fp.in_bgr = 0;
    fp.in_rows = h; fp.width = w; fp.height = h; fp.out_rows = h; fp.n_frames = nf; fp.out_frame_stride = px;
    fp.cls = d_out; fp.cls_pitch = lay.out_pitch; fp.cls_frame_stride = lay.out_frame_stride;
    fp.lo = cv.lo; fp.hi = cv.hi;
    fp.parent = reinterpret_cast<int32_t*>(ctx->ws_parent[slot].ptr);
    fp.kept_count = reinterpret_cast<unsigned int*>(ctx->ws_list[slot].ptr);
    fp.kept_list = reinterpret_cast<uint32_t*>(ctx->ws_list[slot].ptr) + 16;
    // the list's counter block is zero here (see run_frames_device)
    if (ctx->list_dirty[slot]) CB_CUDA(cudaMemsetAsync(fp.kept_count, 0, 64, st));
    ctx->list_dirty[slot] = true;
    CB_TRY(launch_front_cv(ctx, st, fp, cv.channels, cv.l2, cv.aperture));
    HystParams hp;
    memset(&hp, 0, sizeof(hp));
    hp.cls = d_out; hp.cls_pitch = lay.out_pitch; hp.cls_frame_stride = lay.out_frame_stride;
    hp.list = fp.kept_list; hp.ctr = fp.kept_count;
    hp.parent = fp.parent;
    hp.frame_stride = px; hp.rows = h; hp.width = w; hp.row0 = 0; hp.n_frames = nf;
    hp.opencv = 1;
    static const int pdl_env = [] { const char* e = getenv("B200_CANNY_PDL"); return e ? atoi(e) : -1; }();
    hp.pdl = pdl_env >= 0 ? pdl_env : ((long long)nf * px <= (4LL << 20) ? 1 : 0);   // as run_frames_device
    if (ctx->prof.on) hp.pdl = 0;
    CB_TRY(launch_hysteresis(ctx, st, hp));
    ctx->list_dirty[slot] = false;
    return B200_OK;
}

// bytes of the weak-pixel list for nf frames of h x w: a counter block + one 32-bit entry per pixel (worst case: all weak)
static size_t list_bytes(int nf, int h, int w) { return 64 + (size_t)nf * (size_t)h * (size_t)w * 4; }

constexpr int kMaxChunkFrames = 65535;
static int auto_chunk_frames(const b200_ctx* ctx, int h, int w, int n_frames) {
    // a chunk's frame count is gridDim.z of the front kernel (gridDim.y of the tile merge / final kernels): at most 65535
    if (ctx->chunk_frames > 0) return std::min(std::min(ctx->chunk_frames, n_frames), kMaxChunkFrames);
    const long long px = (long long)h * w;
    // ~75 Mpix per chunk (9 frames of 4K): measured best on the 512-frame batch (213 Gpix/s against 189 at 4 frames and 204 at
    // 16): long enough launches that the front kernel's last partly-filled wave matters little, short enough that the two
    // streams still interleave one chunk's small hysteresis kernels with the next chunk's front kernel, and the class map of
    // a chunk (75 MB) still fits the 126 MB L2 when hysteresis reads it
    long long f = (75LL << 20) / px;
    if (f < 1) f = 1;
    // NOT equalised over the batch: a 4K chunk of 9 frames is 279 CTAs for 296 slots, 8 frames are 248 CTAs that take just as long
    // (measured at 64 frames per GPU: 8 x 8 frames 2.27 ms, 7 x 9 + 1 frames faster); the remainder chunk is cut into row bands by the
    // front kernel's launcher, so it costs in proportion to its frames
    return (int)std::min<long long>(std::min<long long>(f, n_frames), kMaxChunkFrames);
}

}  // namespace cb

using namespace cb;

// =====================================================================================================
extern "C" {

int b200_version(void) { return 1; }
const char* b200_last_error(void) { return g_err; }

int b200_ctx_create(int device, b200_ctx** out) {
    if (!out) { set_error("null out pointer"); return B200_ERR_INVALID_ARG; }
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
        cudaGetLastError();
        set_error("no CUDA device available (libcanny_b200 has no CPU fallback)");
        return B200_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= n) { set_error("device %d out of range (have %d)", device, n); return B200_ERR_INVALID_ARG; }
    cudaDeviceProp prop;
    CB_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_error("device %d is sm_%d%d; this library ships sm_100a code only", device, prop.major, prop.minor);
        return B200_ERR_NO_DEVICE;
    }
    CB_CUDA(cudaSetDevice(device));
    b200_ctx* c = new b200_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    auto init = [&]() -> int {
        CB_CUDA(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
        c->stream = c->own_stream;
        for (int i = 0; i < 3; ++i) {
            CB_CUDA(cudaStreamCreateWithFlags(&c->side[i], cudaStreamNonBlocking));
            CB_CUDA(cudaEventCreateWithFlags(&c->ev_join[i], cudaEventDisableTiming));
            CB_CUDA(cudaEventCreateWithFlags(&c->ev_chunk[i], cudaEventDisableTiming | cudaEventBlockingSync));
            CB_CUDA(cudaEventCreateWithFlags(&c->ev_in[i], cudaEventDisableTiming));
            CB_CUDA(cudaEventCreateWithFlags(&c->ev_ragged[i], cudaEventDisableTiming));
        }
        CB_CUDA(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
        CB_CUDA(cudaEventCreateWithFlags(&c->ev_switch, cudaEventDisableTiming));
        CB_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&c->h_kept), 4 * sizeof(unsigned int), cudaHostAllocMapped));
        memset(c->h_kept, 0, 4 * sizeof(unsigned int));
        CB_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&c->d_kept), c->h_kept, 0));
        return B200_OK;
    };
    const int rc = init();
    if (rc != B200_OK) {   // release whatever was created (the destroy path skips null members)
        b200_ctx_destroy(c);
        return rc;
    }
    *out = c;
    return B200_OK;
}

int b200_ctx_destroy(b200_ctx* c) {
    if (!c) return B200_OK;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    auto rel = [](Workspace& w, bool pinned) { if (w.ptr) { if (pinned) cudaFreeHost(w.ptr); else cudaFree(w.ptr); w.ptr = nullptr; w.bytes = 0; } };
    for (int i = 0; i < 3; ++i) { rel(c->ws_parent[i], false); rel(c->ws_list[i], false); rel(c->dev_in[i], false); rel(c->dev_out[i], false); }
    rel(c->ws_planes, false); rel(c->ws_misc, false); rel(c->ws_band_parent, false); rel(c->ws_band_list, false); rel(c->ws_band_aux, false);
    if (c->gauss.d_w) cudaFree(c->gauss.d_w);
    if (c->h_kept) cudaFreeHost(c->h_kept);
    for (int i = 0; i < 3; ++i) {
        if (c->side[i]) cudaStreamDestroy(c->side[i]);
        if (c->ev_join[i]) cudaEventDestroy(c->ev_join[i]);
        if (c->ev_chunk[i]) cudaEventDestroy(c->ev_chunk[i]);
        if (c->ev_in[i]) cudaEventDestroy(c->ev_in[i]);
        if (c->ev_ragged[i]) cudaEventDestroy(c->ev_ragged[i]);
        rel(c->ws_ragged[i], false);
        rel(c->host_ragged[i], true);
        rel(c->host_in[i], true);
        rel(c->dev_bits[i], false);
        rel(c->host_bits[i], true);
    }
    delete c->pool;
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_switch) cudaEventDestroy(c->ev_switch);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    {
        std::lock_guard<std::mutex> lk(g_default_mu);
        if (g_default_ctx == c) g_default_ctx = nullptr;
    }
    delete c;
    return B200_OK;
}

// ---- host placement ------------------------------------------------------------------------------------
// Pins the CALLING thread (and every thread it creates afterwards: the context's host pool, pinned allocations made by first
// touch) to the CPUs of the NUMA node the GPU hangs off, read from sysfs.  One process per GPU on a multi-socket host otherwise
// stages half of its frames through the remote socket's memory.
int b200_host_bind_numa(int device, int* node_out) {
    if (node_out) *node_out = -1;
    char bus[32] = "";
    if (cudaDeviceGetPCIBusId(bus, (int)sizeof(bus), device) != cudaSuccess) {
        cudaGetLastError();
        set_error("no PCI bus id for device %d", device);
        return B200_ERR_NO_DEVICE;
    }
    for (char* c = bus; *c; ++c) *c = (char)tolower(*c);
    int node = -1;
    { std::ifstream f(std::string("/sys/bus/pci/devices/") + bus + "/numa_node"); if (f) f >> node; }
    if (node < 0) return B200_OK;                                   // single-node host (or no sysfs): nothing to do
    std::ifstream f("/sys/devices/system/node/node" + std::to_string(node) + "/cpulist");
    std::string list;
    if (!f || !std::getline(f, list)) return B200_OK;
    cpu_set_t set;
    CPU_ZERO(&set);
    std::stringstream ss(list);
    std::string tok;
    int n_cpus = 0;
    while (std::getline(ss, tok, ',')) {                            // "0-15,64-79"
        int a = 0, b = 0;
        if (sscanf(tok.c_str(), "%d-%d", &a, &b) == 2) { for (int c = a; c <= b && c < CPU_SETSIZE; ++c) { CPU_SET(c, &set); ++n_cpus; } }
        else if (sscanf(tok.c_str(), "%d", &a) == 1 && a < CPU_SETSIZE) { CPU_SET(a, &set); ++n_cpus; }
    }
    if (n_cpus == 0) return B200_OK;
    // only narrow the affinity: keep the intersection with what the process is allowed to use (cgroups, taskset)
    cpu_set_t cur, both;
    if (sched_getaffinity(0, sizeof(cur), &cur) == 0) {
        CPU_AND(&both, &cur, &set);
        if (CPU_COUNT(&both) == 0) return B200_OK;
        set = both;
    }
    if (sched_setaffinity(0, sizeof(set), &set) != 0) return B200_OK;   // not permitted: leave the placement to the OS
    if (node_out) *node_out = node;
    return B200_OK;
}

int b200_ctx_front_kernel_stats(const b200_ctx* ctx, long long* fast_launches, long long* generic_launches) {
    if (!ctx) ctx = g_default_ctx;
    if (!ctx || !fast_launches || !generic_launches) { set_error("bad argument"); return B200_ERR_INVALID_ARG; }
    *fast_launches = ctx->front_fast;
    *generic_launches = ctx->front_generic;
    return B200_OK;
}

int b200_ctx_set_stream(b200_ctx* ctx, void* cuda_stream) {
    CB_TRY(resolve_ctx(ctx));
    cudaStream_t next = cuda_stream ? reinterpret_cast<cudaStream_t>(cuda_stream) : ctx->own_stream;
    if (next != ctx->stream) {
        // Work already issued through the context (every call joins its side streams back into ctx->stream) uses the context's
        // workspace — union-find slots, weak-pixel lists and their counters: the new stream starts after it, so calls on two
        // streams never run on the same slots at once.
        CB_CUDA(cudaEventRecord(ctx->ev_switch, ctx->stream));
        CB_CUDA(cudaStreamWaitEvent(next, ctx->ev_switch, 0));
        ctx->stream = next;
    }
    return B200_OK;
}
int b200_ctx_synchronize(b200_ctx* ctx) {
    CB_TRY(resolve_ctx(ctx));
    CB_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < 3; ++i) CB_CUDA(cudaStreamSynchronize(ctx->side[i]));
    return B200_OK;
}
int b200_ctx_set_chunk_frames(b200_ctx* ctx, int frames) {
    CB_TRY(resolve_ctx(ctx));
    ctx->chunk_frames = frames < 0 ? 0 : frames;
    return B200_OK;
}
int b200_ctx_transfer_bytes(const b200_ctx* ctx, unsigned long long* h2d, unsigned long long* d2h) {
    if (!ctx) ctx = g_default_ctx;
    if (!ctx || !h2d || !d2h) { set_error("bad argument"); return B200_ERR_INVALID_ARG; }
    *h2d = ctx->h2d_bytes;
    *d2h = ctx->d2h_bytes;
    return B200_OK;
}
long long b200_ctx_kernel_launches(const b200_ctx* ctx) {
    if (!ctx) ctx = g_default_ctx;
    return ctx ? ctx->launches : 0;
}

// ---- host-side helpers ------------------------------------------------------------------------------
int b200_gaussian_window(float sigma) { return host_window(sigma); }
int b200_gaussian_kernel(float sigma, float* w, int* window) {
    if (!w || !window || !(sigma > 0.f) || !isfinite(sigma)) { set_error("bad argument to b200_gaussian_kernel"); return B200_ERR_INVALID_ARG; }
    std::vector<float> k;
    host_gaussian_kernel(sigma, k);
    memcpy(w, k.data(), sizeof(float) * k.size());
    *window = (int)k.size();
    return B200_OK;
}
int b200_direction_host(int gx, int gy) { return dir_code_to_angle(direction_code<long long>(gx, gy)); }
int b200_isqrt_host(int n) { return isqrt_floor_host(n); }

// ---- stage API on host buffers ------------------------------------------------------------------------
// Scratch layout in ws_planes for one frame of px pixels: [u8 in | u8 cls | i16 a | i16 b | i16 c | i16 d | i16 e]
struct Planes {
    uint8_t *in, *cls;
    int16_t* p16[5];
};
static int get_planes(b200_ctx* ctx, long long px, Planes& pl) {
    const size_t pxa = ((size_t)px + 255) & ~(size_t)255;
    CB_TRY(ensure_ws(ctx->ws_planes, pxa * 2 + pxa * 2 * 5));
    uint8_t* base = reinterpret_cast<uint8_t*>(ctx->ws_planes.ptr);
    pl.in = base;
    pl.cls = base + pxa;
    for (int i = 0; i < 5; ++i) pl.p16[i] = reinterpret_cast<int16_t*>(base + 2 * pxa + (size_t)i * 2 * pxa);
    return B200_OK;
}

int b200_gaussian(b200_ctx* ctx, const uint8_t* img, float sigma, int h, int w, int16_t* blur) {
    CB_TRY(check_image(img, blur, h, w));
    CB_TRY(resolve_ctx(ctx));
    CB_TRY(prepare_gauss(ctx, sigma));
    const long long px = (long long)h * w;
    Planes pl;
    CB_TRY(get_planes(ctx, px, pl));
    cudaStream_t st = ctx->stream;
    CB_CUDA(cudaMemcpyAsync(pl.in, img, (size_t)px, cudaMemcpyHostToDevice, st));
    FrontParams fp;
    memset(&fp, 0, sizeof(fp));
    fp.in = pl.in; fp.in_pitch = w; fp.in_frame_stride = px; fp.in_rows = h; fp.width = w; fp.height = h; fp.out_rows = h; fp.n_frames = 1;
    fp.cls = pl.cls; fp.cls_pitch = w; fp.cls_frame_stride = px; fp.out_frame_stride = px; fp.blur = pl.p16[0];
    fp.w = ctx->gauss.d_w; fp.count = ctx->gauss.d_count; fp.radius = ctx->gauss.radius;
    fill_thresholds(fp, 1 << 20, 1 << 20);  // nothing is a candidate: the later phases do the minimum
    CB_TRY(launch_front(ctx, st, fp));
    CB_CUDA(cudaMemcpyAsync(blur, pl.p16[0], (size_t)px * 2, cudaMemcpyDeviceToHost, st));
    CB_CUDA(cudaStreamSynchronize(st));
    return B200_OK;
}

int b200_xy_gradient(b200_ctx* ctx, const int16_t* blur, int h, int w, int16_t* gx, int16_t* gy) {
    CB_TRY(check_image(blur, gx, h, w));
    if (!gy) { set_error("null grad_y"); return B200_ERR_INVALID_ARG; }
    CB_TRY(resolve_ctx(ctx));
    const long long px = (long long)h * w;
    Planes pl;
    CB_TRY(get_planes(ctx, px, pl));
    cudaStream_t st = ctx->stream;
    CB_CUDA(cudaMemcpyAsync(pl.p16[0], blur, (size_t)px * 2, cudaMemcpyHostToDevice, st));
    CB_TRY(launch_xy_gradient(ctx, st, pl.p16[0], h, w, pl.p16[1], pl.p16[2]));
    CB_CUDA(cudaMemcpyAsync(gx, pl.p16[1], (size_t)px * 2, cudaMemcpyDeviceToHost, st));
    CB_CUDA(cudaMemcpyAsync(gy, pl.p16[2], (size_t)px * 2, cudaMemcpyDeviceToHost, st));
    CB_CUDA(cudaStreamSynchronize(st));
    return B200_OK;
}

int b200_sobel(b200_ctx* ctx, const int16_t* blur, int h, int w, int16_t* magnitude, int16_t* angle) {
    CB_TRY(check_image(blur, magnitude, h, w));
    if (!angle) { set_error("null angle"); return B200_ERR_INVALID_ARG; }
    CB_TRY(resolve_ctx(ctx));
    const long long px = (long long)h * w;
    Planes pl;
    CB_TRY(get_planes(ctx, px, pl));
    cudaStream_t st = ctx->stream;
    CB_CUDA(cudaMemcpyAsync(pl.p16[0], blur, (size_t)px * 2, cudaMemcpyHostToDevice, st));
    CB_TRY(launch_sobel(ctx, st, pl.p16[0], h, w, pl.p16[1], pl.p16[2]));
    CB_CUDA(cudaMemcpyAsync(magnitude, pl.p16[1], (size_t)px * 2, cudaMemcpyDeviceToHost, st));
    CB_CUDA(cudaMemcpyAsync(angle, pl.p16[2], (size_t)px * 2, cudaMemcpyDeviceToHost, st));
    CB_CUDA(cudaStreamSynchronize(st));
    return B200_OK;
}

int b200_nonmaximal(b200_ctx* ctx, const int16_t* magnitude, const int16_t* angle, int h, int w, int16_t* nms) {
    CB_TRY(check_image(magnitude, nms, h, w));
    if (!angle) { set_error("null angle"); return B200_ERR_INVALID_ARG; }
    CB_TRY(resolve_ctx(ctx));
    const long long px = (long long)h * w;
    Planes pl;
    CB_TRY(get_planes(ctx, px, pl));
    cudaStream_t st = ctx->stream;
    CB_CUDA(cudaMemcpyAsync(pl.p16[0], magnitude, (size_t)px * 2, cudaMemcpyHostToDevice, st));
    CB_CUDA(cudaMemcpyAsync(pl.p16[1], angle, (size_t)px * 2, cudaMemcpyHostToDevice, st));
    CB_TRY(launch_nonmaximal(ctx, st, pl.p16[0], pl.p16[1], h, w, pl.p16[2]));
    CB_CUDA(cudaMemcpyAsync(nms, pl.p16[2], (size_t)px * 2, cudaMemcpyDeviceToHost, st));
    CB_CUDA(cudaStreamSynchronize(st));
    return B200_OK;
}

int b200_hysteresis(b200_ctx* ctx, int16_t* nms_inout, int h, int w, int lo, int hi) {
    CB_TRY(check_image(nms_inout, nms_inout, h, w));
    CB_TRY(check_thresholds(lo, hi));
    CB_TRY(resolve_ctx(ctx));
    const long long px = (long long)h * w;
    Planes pl;
    CB_TRY(get_planes(ctx, px, pl));
    CB_TRY(ensure_ws(ctx->ws_parent[0], (size_t)px * 4));
    cudaStream_t st = ctx->stream;
    CB_CUDA(cudaMemcpyAsync(pl.p16[0], nms_inout, (size_t)px * 2, cudaMemcpyHostToDevice, st));
    CB_TRY(launch_classify_i16(ctx, st, pl.p16[0], pl.cls, (size_t)px, lo, effective_hi(hi)));
    HystParams hp;
    memset(&hp, 0, sizeof(hp));
    hp.cls = pl.cls; hp.cls_pitch = w; hp.cls_frame_stride = px; hp.parent = reinterpret_cast<int32_t*>(ctx->ws_parent[0].ptr);
    hp.frame_stride = px; hp.rows = h; hp.width = w; hp.row0 = 0; hp.n_frames = 1;
    CB_TRY(launch_hysteresis(ctx, st, hp));
    CB_TRY(launch_expand_u8_to_i16(ctx, st, pl.cls, pl.p16[1], (size_t)px));
    CB_CUDA(cudaMemcpyAsync(nms_inout, pl.p16[1], (size_t)px * 2, cudaMemcpyDeviceToHost, st));
    CB_CUDA(cudaStreamSynchronize(st));
    return B200_OK;
}

int b200_canny_steps(b200_ctx* ctx, const uint8_t* img, float sigma, int lo, int hi, int h, int w, int16_t* blur,
                     int16_t* magnitude, int16_t* angle, int16_t* nms, int16_t* edges) {
    CB_TRY(check_image(img, edges, h, w));
    CB_TRY(check_thresholds(lo, hi));
    CB_TRY(resolve_ctx(ctx));
    CB_TRY(prepare_gauss(ctx, sigma));
    const long long px = (long long)h * w;
    Planes pl;
    CB_TRY(get_planes(ctx, px, pl));
    CB_TRY(ensure_ws(ctx->ws_parent[0], (size_t)px * 4));
    CB_TRY(ensure_ws(ctx->ws_list[0], list_bytes(1, h, w)));
    cudaStream_t st = ctx->stream;
    CB_CUDA(cudaMemcpyAsync(pl.in, img, (size_t)px, cudaMemcpyHostToDevice, st));
    CB_TRY(run_frames_device(ctx, st, 0, pl.in, pl.cls, 1, h, w, lo, hi, blur ? pl.p16[0] : nullptr,
                             magnitude ? pl.p16[1] : nullptr, angle ? pl.p16[2] : nullptr, nms ? pl.p16[3] : nullptr));
    CB_TRY(launch_expand_u8_to_i16(ctx, st, pl.cls, pl.p16[4], (size_t)px));
    if (blur) CB_CUDA(cudaMemcpyAsync(blur, pl.p16[0], (size_t)px * 2, cudaMemcpyDeviceToHost, st));
    if (magnitude) CB_CUDA(cudaMemcpyAsync(magnitude, pl.p16[1], (size_t)px * 2, cudaMemcpyDeviceToHost, st));
    if (angle) CB_CUDA(cudaMemcpyAsync(angle, pl.p16[2], (size_t)px * 2, cudaMemcpyDeviceToHost, st));
    if (nms) CB_CUDA(cudaMemcpyAsync(nms, pl.p16[3], (size_t)px * 2, cudaMemcpyDeviceToHost, st));
    CB_CUDA(cudaMemcpyAsync(edges, pl.p16[4], (size_t)px * 2, cudaMemcpyDeviceToHost, st));
    CB_CUDA(cudaStreamSynchronize(st));
    return B200_OK;
}

static int batch_host_impl(b200_ctx* ctx, const uint8_t* frames, int n_frames, int h, int w, int lo, int hi, uint8_t* edges8,
                           int16_t* edges16, bool packed, uint32_t* bits_out = nullptr);
static bool packed_transfer_off();

int b200_canny(b200_ctx* ctx, const uint8_t* img, float sigma, int lo, int hi, int h, int w, int16_t* edges) {
    // large frames in pageable memory take the pipelined host path: the frame is staged through pinned memory by the host pool,
    // the map crosses PCIe bit-packed (1/16 of the int16 plane) and is expanded to the reference's 0 / 255 int16 values by the pool
    if ((long long)h * w >= kStageMinBytes && !packed_transfer_off() && img && edges && (is_pageable(img) || is_pageable(edges))) {
        CB_TRY(check_image(img, edges, h, w));
        CB_TRY(check_thresholds(lo, hi));
        CB_TRY(resolve_ctx(ctx));
        CB_TRY(prepare_gauss(ctx, sigma));
        return batch_host_impl(ctx, img, 1, h, w, lo, hi, nullptr, edges, true);
    }
    return b200_canny_steps(ctx, img, sigma, lo, hi, h, w, nullptr, nullptr, nullptr, nullptr, edges);
}

int b200_bgr_to_gray_device(b200_ctx* ctx, const uint8_t* d_bgr, size_t n_px, uint8_t* d_gray) {
    if (!d_bgr || !d_gray || n_px == 0) { set_error("bad argument to b200_bgr_to_gray_device"); return B200_ERR_INVALID_ARG; }
    CB_TRY(resolve_ctx(ctx));
    return launch_bgr_to_gray(ctx, ctx->stream, d_bgr, d_gray, n_px);
}

int b200_canny_bgr(b200_ctx* ctx, const uint8_t* bgr, float sigma, int lo, int hi, int h, int w, uint8_t* gray_out, int16_t* edges) {
    CB_TRY(check_image(bgr, edges, h, w));
    CB_TRY(check_thresholds(lo, hi));
    CB_TRY(resolve_ctx(ctx));
    CB_TRY(prepare_gauss(ctx, sigma));
    const long long px = (long long)h * w;
    Planes pl;
    CB_TRY(get_planes(ctx, px, pl));
    CB_TRY(ensure_ws(ctx->ws_parent[0], (size_t)px * 4));
    CB_TRY(ensure_ws(ctx->ws_list[0], list_bytes(1, h, w)));
    cudaStream_t st = ctx->stream;
    // large frames in pageable memory: staged through pinned memory by the host pool, edge map back bit-packed (see
    // batch_host_impl); everything else takes the plain copies
    const bool fast = 3 * px >= kStageMinBytes && !packed_transfer_off() && (is_pageable(bgr) || is_pageable(edges));
    HostPool* pool = fast ? get_pool(ctx) : nullptr;
    // the 3-byte frame is staged in the int16 scratch planes (p16[0..1] hold 4*px bytes >= 3*px)
    uint8_t* d_bgr = reinterpret_cast<uint8_t*>(pl.p16[0]);
    const uint8_t* h_src = bgr;
    if (fast && is_pageable(bgr)) {
        CB_TRY(ensure_ws(ctx->host_in[0], (size_t)px * 3, /*pinned_host=*/true));
        if (ctx->in_busy[0]) { CB_CUDA(cudaEventSynchronize(ctx->ev_in[0])); ctx->in_busy[0] = false; }
        pool->run(HostPool::kCopy, bgr, ctx->host_in[0].ptr, (size_t)px * 3);
        h_src = reinterpret_cast<const uint8_t*>(ctx->host_in[0].ptr);
    }
    CB_CUDA(cudaMemcpyAsync(d_bgr, h_src, (size_t)px * 3, cudaMemcpyHostToDevice, st));
    if (!gray_out && bgr_fused_ok(ctx, d_bgr, 1, h, w, 3LL * w, 3 * px)) {
        // nobody wants the gray plane: the front kernel converts while it stages (no 4 B/px pass, no gray plane in HBM)
        CB_TRY(run_frames_device(ctx, st, 0, d_bgr, pl.cls, 1, h, w, lo, hi, nullptr, nullptr, nullptr, nullptr, /*bgr=*/true));
    } else {
        CB_TRY(launch_bgr_to_gray(ctx, st, d_bgr, pl.in, (size_t)px));
        CB_TRY(run_frames_device(ctx, st, 0, pl.in, pl.cls, 1, h, w, lo, hi, nullptr, nullptr, nullptr, nullptr));
    }
    if (!fast) {
        CB_TRY(launch_expand_u8_to_i16(ctx, st, pl.cls, pl.p16[4], (size_t)px));
        if (gray_out) CB_CUDA(cudaMemcpyAsync(gray_out, pl.in, (size_t)px, cudaMemcpyDeviceToHost, st));
        CB_CUDA(cudaMemcpyAsync(edges, pl.p16[4], (size_t)px * 2, cudaMemcpyDeviceToHost, st));
        CB_CUDA(cudaStreamSynchronize(st));
        return B200_OK;
    }
    const size_t bits_bytes = (((size_t)px + 31) / 32) * 4;
    CB_TRY(ensure_ws(ctx->dev_bits[0], bits_bytes));
    CB_TRY(ensure_ws(ctx->host_bits[0], bits_bytes, /*pinned_host=*/true));
    CB_TRY(launch_pack_edges(ctx, st, pl.cls, reinterpret_cast<uint32_t*>(ctx->dev_bits[0].ptr), (size_t)px));
    CB_CUDA(cudaMemcpyAsync(ctx->host_bits[0].ptr, ctx->dev_bits[0].ptr, bits_bytes, cudaMemcpyDeviceToHost, st));
    const bool stage_gray = gray_out && is_pageable(gray_out);
    if (stage_gray) {
        CB_TRY(ensure_ws(ctx->host_in[1], (size_t)px, /*pinned_host=*/true));
        CB_CUDA(cudaMemcpyAsync(ctx->host_in[1].ptr, pl.in, (size_t)px, cudaMemcpyDeviceToHost, st));
    } else if (gray_out) {
        CB_CUDA(cudaMemcpyAsync(gray_out, pl.in, (size_t)px, cudaMemcpyDeviceToHost, st));
    }
    CB_CUDA(cudaStreamSynchronize(st));
    pool->run(HostPool::kUnpackI16, ctx->host_bits[0].ptr, edges, (size_t)px);
    if (stage_gray) pool->run(HostPool::kCopy, ctx->host_in[1].ptr, gray_out, (size_t)px);
    return B200_OK;
}

// ---- batched --------------------------------------------------------------------------------------------
// Argument checks of a strided device batch; all of them run before any device work.  bpp: bytes per input pixel.
static int check_strided(const uint8_t* in, long long in_pitch, long long in_fs, int n, int h, int w, const uint8_t* out,
                         long long out_pitch, long long out_fs, int bpp, int min_side = 2) {
    CB_TRY(check_image(in, out, h, w, min_side));
    if (n <= 0) { set_error("n_frames must be positive"); return B200_ERR_INVALID_ARG; }
    if (in_pitch < 0 || in_fs < 0 || out_pitch < 0 || out_fs < 0) {
        set_error("negative stride (in: pitch %lld, frame %lld; out: pitch %lld, frame %lld)", in_pitch, in_fs, out_pitch, out_fs);
        return B200_ERR_INVALID_ARG;
    }
    const long long in_row = (long long)bpp * w;
    if (in_pitch < in_row) { set_error("input row pitch %lld is smaller than a row (%lld bytes)", in_pitch, in_row); return B200_ERR_INVALID_ARG; }
    if (out_pitch < w) { set_error("output row pitch %lld is smaller than a row (%d bytes)", out_pitch, w); return B200_ERR_INVALID_ARG; }
    // extents in 128-bit arithmetic: no stride, however large, can wrap a product and slip past the checks below
    typedef __int128 i128;
    const i128 in_frame = (i128)(h - 1) * in_pitch + in_row, out_frame = (i128)(h - 1) * out_pitch + w;
    if (n > 1 && in_fs < in_frame) { set_error("input frames overlap: frame stride %lld < %.0f bytes per frame", in_fs, (double)in_frame); return B200_ERR_INVALID_ARG; }
    if (n > 1 && out_fs < out_frame) { set_error("output frames overlap: frame stride %lld < %.0f bytes per frame", out_fs, (double)out_frame); return B200_ERR_INVALID_ARG; }
    // the extents: first byte of frame 0 to one past the last byte of frame n-1
    const i128 in_ext = (i128)(n - 1) * in_fs + in_frame, out_ext = (i128)(n - 1) * out_fs + out_frame;
    const i128 kMaxExtent = (i128)1 << 48;   // more than any device address space
    if (in_ext > kMaxExtent || out_ext > kMaxExtent) {
        set_error("strides span more than 2^48 bytes (input %.3g, output %.3g bytes)", (double)in_ext, (double)out_ext);
        return B200_ERR_INVALID_ARG;
    }
    const i128 in_lo = (i128)reinterpret_cast<uintptr_t>(in), out_lo = (i128)reinterpret_cast<uintptr_t>(out);
    if (in_lo < out_lo + out_ext && out_lo < in_lo + in_ext) { set_error("the output's extent overlaps the input's"); return B200_ERR_INVALID_ARG; }
    return B200_OK;
}

// bpp: bytes per input pixel — 1 gray, 3 interleaved B,G,R (converted by the front kernel while staging when it can, else chunk by
// chunk into a gray scratch plane first).  Strides in bytes (b200_canny_batch_device_strided); the dense entry points pass
// pitch = bpp*width and frame stride = height*pitch.
// cv: the OpenCV-compatible path (b200_cv_canny_device_strided; its thresholds are checked by the caller, sigma, lo and hi are
// unused): the same chunks, slots and workspace, each chunk through run_frames_cv.  Null: the reference's semantics.
static int batch_device_impl(b200_ctx* ctx, const uint8_t* d_frames, long long in_pitch, long long in_fs, int n_frames, int h, int w,
                             float sigma, int lo, int hi, uint8_t* d_edges, long long out_pitch, long long out_fs, int bpp,
                             const CvSpec* cv = nullptr) {
    CB_TRY(check_strided(d_frames, in_pitch, in_fs, n_frames, h, w, d_edges, out_pitch, out_fs, bpp, cv ? 1 : 2));
    if (!cv) CB_TRY(check_thresholds(lo, hi));
    CB_TRY(resolve_ctx(ctx));
    if (!cv) CB_TRY(prepare_gauss(ctx, sigma));
    // a single frame's stride is never used: make it the one that keeps the tensor map and the word stores eligible
    if (n_frames == 1) { in_fs = (long long)h * in_pitch; out_fs = (long long)h * out_pitch; }
    const FrameLayout lay = {in_pitch, in_fs, out_pitch, out_fs};
    const long long px = (long long)h * w;
    const int chunk = auto_chunk_frames(ctx, h, w, n_frames);
    const int n_chunks = (n_frames + chunk - 1) / chunk;
    // three slots: while one chunk's small, latency-bound hysteresis kernels wait for SM resources, the front kernels of the TWO
    // following chunks are already queued on their own streams, so the machine never waits for a front kernel that is itself
    // waiting (same slot) for those hysteresis kernels (226 against 219 Gpix/s with two slots; running the hysteresis kernels on
    // high-priority streams on top of that measured 222)
    const int n_slots = std::min(3, n_chunks);
    const bool bgr = bpp == 3 && !cv;   // the OpenCV kernel reads 3-channel frames itself
    const bool fused = bgr && bgr_fused_ok(ctx, d_frames, std::min(chunk, n_frames), h, w, in_pitch, in_fs);
    const bool bgr_dense = in_pitch == 3LL * w && in_fs == 3 * px;
    for (int s = 0; s < n_slots; ++s) {
        CB_TRY(ensure_ws(ctx->ws_parent[s], (size_t)px * 4 * (size_t)chunk));
        CB_TRY(ensure_ws(ctx->ws_list[s], list_bytes(chunk, h, w)));
        if (bgr && !fused) CB_TRY(ensure_ws(ctx->dev_in[s], (size_t)px * (size_t)chunk));   // gray scratch of one chunk
    }
    auto run_chunk = [&](cudaStream_t st, int s, int f0, int nf) -> int {
        const uint8_t* src = d_frames + (long long)f0 * in_fs;
        if (cv) return run_frames_cv(ctx, st, s, src, d_edges + (long long)f0 * out_fs, nf, h, w, *cv, lay);
        FrameLayout cl = lay;
        if (bgr && !fused) {
            // the gray scratch plane is dense whatever the B,G,R frames' strides
            uint8_t* gray = reinterpret_cast<uint8_t*>(ctx->dev_in[s].ptr);
            if (bgr_dense) CB_TRY(launch_bgr_to_gray(ctx, st, src, gray, (size_t)px * (size_t)nf));
            else CB_TRY(launch_bgr_to_gray_strided(ctx, st, src, in_pitch, in_fs, nf, h, w, gray));
            src = gray;
            cl.in_pitch = w; cl.in_frame_stride = px;
        }
        // The last full chunk of a call is cut into four row bands per frame: a front CTA otherwise marches a whole strip of a frame
        // (0.3 ms at 4K) and the call ends with SMs idling while the last of those finish.  Measured on 64-frame calls (one GPU's
        // share of the 512-frame job at 8 GPUs): 2.118 -> 2.075 ms; 512-frame calls unchanged (tools/chunk_sweep.py).
        static const int tail_bands = [] { const char* e = getenv("B200_CANNY_TAIL_BANDS"); return e ? atoi(e) : 4; }();
        static const int tail_chunks = [] { const char* e = getenv("B200_CANNY_TAIL_CHUNKS"); return e ? atoi(e) : 1; }();
        int bands = 0;
        if (n_chunks > 1 && f0 + nf > n_frames - tail_chunks * chunk && nf == chunk && tail_bands > 1 && h / tail_bands >= 256) bands = tail_bands;
        return run_frames_device(ctx, st, s, src, d_edges + (long long)f0 * out_fs, nf, h, w, lo, hi, nullptr, nullptr, nullptr, nullptr,
                                 fused, bands, &cl);
    };
    if (n_slots == 1) return run_chunk(ctx->stream, 0, 0, n_frames);
    // the side streams take the chunks in turn so one chunk's tail waves overlap the next chunks' heads
    CB_CUDA(cudaEventRecord(ctx->ev_fork, ctx->stream));
    for (int s = 0; s < n_slots; ++s) CB_CUDA(cudaStreamWaitEvent(ctx->side[s], ctx->ev_fork, 0));
    for (int c = 0; c < n_chunks; ++c) {
        const int f0 = c * chunk, nf = std::min(chunk, n_frames - f0);
        const int s = c % n_slots;
        CB_TRY(run_chunk(ctx->side[s], s, f0, nf));
    }
    for (int s = 0; s < n_slots; ++s) {
        CB_CUDA(cudaEventRecord(ctx->ev_join[s], ctx->side[s]));
        CB_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_join[s], 0));
    }
    return B200_OK;
}

int b200_canny_batch_device(b200_ctx* ctx, const uint8_t* d_frames, int n_frames, int h, int w, float sigma, int lo,
                            int hi, uint8_t* d_edges) {
    const long long px = (long long)h * w;
    return batch_device_impl(ctx, d_frames, w, px, n_frames, h, w, sigma, lo, hi, d_edges, w, px, 1);
}

int b200_canny_batch_device_bgr(b200_ctx* ctx, const uint8_t* d_bgr, int n_frames, int h, int w, float sigma, int lo,
                                int hi, uint8_t* d_edges) {
    const long long px = (long long)h * w;
    return batch_device_impl(ctx, d_bgr, 3LL * w, 3 * px, n_frames, h, w, sigma, lo, hi, d_edges, w, px, 3);
}

int b200_canny_batch_device_strided(b200_ctx* ctx, const uint8_t* d_frames, int64_t in_row_pitch, int64_t in_frame_stride,
                                    int n_frames, int h, int w, float sigma, int lo, int hi, uint8_t* d_edges,
                                    int64_t out_row_pitch, int64_t out_frame_stride) {
    return batch_device_impl(ctx, d_frames, in_row_pitch, in_frame_stride, n_frames, h, w, sigma, lo, hi, d_edges, out_row_pitch,
                             out_frame_stride, 1);
}

int b200_canny_batch_device_bgr_strided(b200_ctx* ctx, const uint8_t* d_bgr, int64_t in_row_pitch, int64_t in_frame_stride,
                                        int n_frames, int h, int w, float sigma, int lo, int hi, uint8_t* d_edges,
                                        int64_t out_row_pitch, int64_t out_frame_stride) {
    return batch_device_impl(ctx, d_bgr, in_row_pitch, in_frame_stride, n_frames, h, w, sigma, lo, hi, d_edges, out_row_pitch,
                             out_frame_stride, 3);
}

// ---- cv::Canny semantics ----------------------------------------------------------------------------------
// Thresholds as cv::Canny uses them (imgproc/src/canny.cpp): divided by 16 for aperture 7 (whose derivatives are scaled by 1/16)
// before anything else; swapped when low > high; for L2 clamped to 32767 and squared when positive; floored.  NaN / inf:
// B200_ERR_INVALID_ARG.  A floor outside int32: B200_ERR_UNSUPPORTED (OpenCV's cvFloor overflows there and its result is not the
// comparison the thresholds describe).
constexpr int kCvMaxHeight = 65535 * 64;   // the OpenCV front kernel's grid: one row of CTAs per 64 rows, gridDim.y <= 65535

static int cv_thresholds(double t1, double t2, bool l2, int aperture, int* lo, int* hi) {
    if (!isfinite(t1) || !isfinite(t2)) { set_error("thresholds must be finite (got %g, %g)", t1, t2); return B200_ERR_INVALID_ARG; }
    if (aperture == 7) { t1 /= 16; t2 /= 16; }
    double a = std::min(t1, t2), b = std::max(t1, t2);
    if (l2) {
        a = std::min(32767.0, a); b = std::min(32767.0, b);
        if (a > 0) a *= a;
        if (b > 0) b *= b;
    }
    a = floor(a); b = floor(b);
    const double kMin = -2147483648.0, kMax = 2147483647.0;
    if (a < kMin || a > kMax || b < kMin || b > kMax) {
        set_error("thresholds %g, %g: their floor does not fit in int32", t1, t2);
        return B200_ERR_UNSUPPORTED;
    }
    *lo = (int)a; *hi = (int)b;
    return B200_OK;
}

// The checks of the OpenCV calls that come before the layout's: channel count (UNSUPPORTED), aperture (INVALID_ARG, as cv::Canny
// rejects it), the uniform call's height (max_height; UNSUPPORTED), thresholds
static int cv_spec(int channels, int aperture, int height, int max_height, double t1, double t2, int l2_gradient, CvSpec* cv) {
    if (channels != 1 && channels != 3) { set_error("channels must be 1 or 3 (got %d)", channels); return B200_ERR_UNSUPPORTED; }
    if (aperture != 3 && aperture != 5 && aperture != 7) {
        set_error("aperture size must be 3, 5 or 7 (got %d)", aperture);
        return B200_ERR_INVALID_ARG;
    }
    if (height > max_height) { set_error("height %d: at most %d rows (65535 tiles of 64)", height, max_height); return B200_ERR_UNSUPPORTED; }
    cv->channels = channels;
    cv->l2 = l2_gradient != 0;
    cv->aperture = aperture;
    return cv_thresholds(t1, t2, cv->l2, aperture, &cv->lo, &cv->hi);
}

int b200_cv_canny_aperture_device_strided(b200_ctx* ctx, const uint8_t* d_in, int64_t in_row_pitch, int64_t in_frame_stride,
                                          int n_frames, int height, int width, int channels, double threshold1, double threshold2,
                                          int aperture_size, int l2_gradient, uint8_t* d_edges, int64_t out_row_pitch,
                                          int64_t out_frame_stride) {
    CvSpec cv;
    CB_TRY(cv_spec(channels, aperture_size, height, kCvMaxHeight, threshold1, threshold2, l2_gradient, &cv));
    return batch_device_impl(ctx, d_in, in_row_pitch, in_frame_stride, n_frames, height, width, 0.f, 0, 0, d_edges, out_row_pitch,
                             out_frame_stride, channels, &cv);
}

int b200_cv_canny_device_strided(b200_ctx* ctx, const uint8_t* d_in, int64_t in_row_pitch, int64_t in_frame_stride, int n_frames,
                                 int height, int width, int channels, double threshold1, double threshold2, int l2_gradient,
                                 uint8_t* d_edges, int64_t out_row_pitch, int64_t out_frame_stride) {
    return b200_cv_canny_aperture_device_strided(ctx, d_in, in_row_pitch, in_frame_stride, n_frames, height, width, channels, threshold1,
                                                 threshold2, 3, l2_gradient, d_edges, out_row_pitch, out_frame_stride);
}

// ---- ragged lists: frames of different sizes in one call ------------------------------------------------
// Argument checks of b200_canny_frames_device[_bgr] and b200_cv_canny_frames_device; all of them run before any device work.  Overlaps
// are found by sorting the extents (a list can hold thousands of frames): the outputs among themselves, then every output against
// the merged inputs.  bpp: bytes per input pixel; min_side as check_image.
static int check_frames(const b200_frame* fr, int n, int bpp, int min_side = 2) {
    if (!fr) { set_error("null frame list"); return B200_ERR_INVALID_ARG; }
    if (n <= 0) { set_error("n_frames must be positive"); return B200_ERR_INVALID_ARG; }
    typedef __int128 i128;
    struct Ext { i128 lo, hi; int idx; };
    std::vector<Ext> ins((size_t)n), outs((size_t)n);
    for (int i = 0; i < n; ++i) {
        const b200_frame& f = fr[i];
        if (!f.in || !f.out) { set_error("frame %d: null image pointer", i); return B200_ERR_INVALID_ARG; }
        if (f.height < min_side || f.width < min_side) {
            set_error("frame %d: height and width must be >= %d (got %dx%d)", i, min_side, f.height, f.width);
            return B200_ERR_INVALID_ARG;
        }
        if (f.in_row_pitch < 0 || f.out_row_pitch < 0) {
            set_error("frame %d: negative row pitch (in %lld, out %lld)", i, (long long)f.in_row_pitch, (long long)f.out_row_pitch);
            return B200_ERR_INVALID_ARG;
        }
        const long long in_row = (long long)bpp * f.width;
        if (f.in_row_pitch < in_row) { set_error("frame %d: input row pitch %lld is smaller than a row (%lld bytes)", i, (long long)f.in_row_pitch, in_row); return B200_ERR_INVALID_ARG; }
        if (f.out_row_pitch < f.width) { set_error("frame %d: output row pitch %lld is smaller than a row (%d bytes)", i, (long long)f.out_row_pitch, f.width); return B200_ERR_INVALID_ARG; }
        // extents in 128-bit arithmetic, as check_strided
        const i128 in_ext = (i128)(f.height - 1) * f.in_row_pitch + in_row, out_ext = (i128)(f.height - 1) * f.out_row_pitch + f.width;
        const i128 kMaxExtent = (i128)1 << 48;
        if (in_ext > kMaxExtent || out_ext > kMaxExtent) {
            set_error("frame %d: pitches span more than 2^48 bytes (input %.3g, output %.3g bytes)", i, (double)in_ext, (double)out_ext);
            return B200_ERR_INVALID_ARG;
        }
        if ((long long)f.height * f.width >= (1LL << 31)) { set_error("frame %d: %dx%d pixels exceed int indexing", i, f.height, f.width); return B200_ERR_UNSUPPORTED; }
        const i128 in_lo = (i128)reinterpret_cast<uintptr_t>(f.in), out_lo = (i128)reinterpret_cast<uintptr_t>(f.out);
        ins[(size_t)i] = Ext{in_lo, in_lo + in_ext, i};
        outs[(size_t)i] = Ext{out_lo, out_lo + out_ext, i};
    }
    auto by_lo = [](const Ext& a, const Ext& b) { return a.lo < b.lo || (a.lo == b.lo && a.idx < b.idx); };
    std::sort(outs.begin(), outs.end(), by_lo);
    for (size_t k = 1; k < outs.size(); ++k)
        if (outs[k].lo < outs[k - 1].hi) { set_error("the outputs of frames %d and %d overlap", outs[k - 1].idx, outs[k].idx); return B200_ERR_INVALID_ARG; }
    // inputs may overlap each other: merge them, then look up each output's first merged run that ends after its start
    std::sort(ins.begin(), ins.end(), by_lo);
    std::vector<Ext> runs;
    for (const Ext& e : ins) {
        if (!runs.empty() && e.lo < runs.back().hi) { if (e.hi > runs.back().hi) runs.back().hi = e.hi; }
        else runs.push_back(e);
    }
    for (const Ext& o : outs) {
        auto it = std::upper_bound(runs.begin(), runs.end(), o.lo, [](i128 v, const Ext& r) { return v < r.hi; });
        if (it != runs.end() && it->lo < o.hi) { set_error("the output of frame %d overlaps an input", o.idx); return B200_ERR_INVALID_ARG; }
    }
    return B200_OK;
}

constexpr long long kRaggedChunkPx = 75LL << 20;   // the uniform path's chunk budget (auto_chunk_frames): a chunk's class map fits L2

static size_t align16(size_t v) { return (v + 15) & ~(size_t)15; }

// A ragged chunk's table is built on the host in the slot's pinned staging and sent up with one copy.  The staging is rewritten only
// once the copy out of it (previous chunk or call on this slot) has completed: this waits for ev_ragged[s], lets fill(h) write the
// `bytes` bytes at h, copies them to the slot's device table (*d) and records ev_ragged[s] behind the copy.
static int upload_ragged_table(b200_ctx* ctx, cudaStream_t st, int s, size_t bytes, const std::function<void(uint8_t*)>& fill,
                               uint8_t** d) {
    if (ctx->ragged_busy[s]) { CB_CUDA(cudaEventSynchronize(ctx->ev_ragged[s])); ctx->ragged_busy[s] = false; }
    CB_TRY(ensure_ws(ctx->host_ragged[s], bytes, /*pinned_host=*/true));
    CB_TRY(ensure_ws(ctx->ws_ragged[s], bytes));
    uint8_t* h = reinterpret_cast<uint8_t*>(ctx->host_ragged[s].ptr);
    *d = reinterpret_cast<uint8_t*>(ctx->ws_ragged[s].ptr);
    fill(h);
    CB_CUDA(cudaMemcpyAsync(*d, h, bytes, cudaMemcpyHostToDevice, st));
    CB_CUDA(cudaEventRecord(ctx->ev_ragged[s], st));
    ctx->ragged_busy[s] = true;
    return B200_OK;
}

// The frame descriptors and dense slot bases of a chunk.  src / src_pitch: what each frame's front kernel reads (null: the caller's
// frames themselves).
static void fill_ragged_frames(const b200_frame* fr, int nf, const uint8_t* const* src, const long long* src_pitch, RaggedFrame* hf,
                               uint32_t* hb) {
    long long base = 0;
    for (int i = 0; i < nf; ++i) {
        const b200_frame& f = fr[i];
        RaggedFrame& r = hf[i];
        r.in = src ? src[i] : f.in; r.in_pitch = src_pitch ? src_pitch[i] : f.in_row_pitch;
        r.cls = f.out; r.cls_pitch = f.out_row_pitch;
        r.height = f.height; r.width = f.width;
        r.base = (int)base;
        r.cls_words = ((reinterpret_cast<uintptr_t>(f.out) | (uintptr_t)f.out_row_pitch) & 3) == 0;
        hb[i] = (uint32_t)base;
        base += (long long)f.height * f.width;
    }
}

// One chunk of a ragged list on slot s / stream st: table (descriptors, tensor maps, work items, B,G,R jobs) built on the host into
// the slot's pinned staging and sent up with one copy; then [B,G,R -> gray], the front kernel (one launch per staging form, both
// appending to the same weak-pixel list) and the list-driven hysteresis kernels.
static int run_ragged_chunk(b200_ctx* ctx, cudaStream_t st, int s, const b200_frame* fr, int nf, int lo, int hi, bool bgr) {
    const int radius = ctx->gauss.radius;
    std::vector<int> hs((size_t)nf), ws((size_t)nf);
    std::vector<const uint8_t*> src((size_t)nf);
    std::vector<long long> src_pitch((size_t)nf), gray_off((size_t)nf);
    long long px = 0, gray_bytes = 0;
    for (int i = 0; i < nf; ++i) {
        hs[(size_t)i] = fr[i].height; ws[(size_t)i] = fr[i].width;
        px += (long long)fr[i].height * fr[i].width;
        if (bgr) {
            // every converted frame takes TMA: 16-byte aligned base and row pitch in the chunk's gray scratch
            const long long pitch = (fr[i].width + 15) & ~15LL;
            gray_off[(size_t)i] = gray_bytes;
            src[(size_t)i] = reinterpret_cast<const uint8_t*>(ctx->dev_in[s].ptr) + gray_bytes;
            src_pitch[(size_t)i] = pitch;
            gray_bytes += pitch * fr[i].height;
        } else {
            src[(size_t)i] = fr[i].in;
            src_pitch[(size_t)i] = fr[i].in_row_pitch;
        }
    }
    std::vector<CUtensorMap> maps((size_t)nf);
    std::vector<RaggedItem> items_tma, items_byte;
    const int band_rows = ragged_band_rows3(ctx, hs.data(), ws.data(), nf, radius);
    for (int i = 0; i < nf; ++i) {
        bool use_tma = false;
        CB_TRY(ragged_tensor_map3(src[(size_t)i], src_pitch[(size_t)i], hs[(size_t)i], ws[(size_t)i], radius, &maps[(size_t)i], &use_tma));
        ragged_items3(i, hs[(size_t)i], ws[(size_t)i], band_rows, use_tma ? items_tma : items_byte);
    }
    // the longest CTAs first (frames shorter than the band height have shorter ones): the launch ends on short CTAs
    auto longer = [](const RaggedItem& a, const RaggedItem& b) { return a.ye - a.yb > b.ye - b.yb; };
    std::stable_sort(items_tma.begin(), items_tma.end(), longer);
    std::stable_sort(items_byte.begin(), items_byte.end(), longer);
    const size_t n_items = items_tma.size() + items_byte.size();
    // table: tensor maps (128 B, 64-byte aligned) | frame descriptors | bases | work items | B,G,R jobs
    const size_t off_frames = (size_t)nf * sizeof(CUtensorMap);
    const size_t off_bases = align16(off_frames + (size_t)nf * sizeof(RaggedFrame));
    const size_t off_items = align16(off_bases + (size_t)nf * sizeof(uint32_t));
    const size_t off_jobs = align16(off_items + n_items * sizeof(RaggedItem));
    const size_t bytes = off_jobs + (bgr ? (size_t)nf * sizeof(RaggedGrayJob) : 0);
    long long row0 = 0;
    uint8_t* d = nullptr;
    CB_TRY(upload_ragged_table(ctx, st, s, bytes, [&](uint8_t* h) {
        memcpy(h, maps.data(), off_frames);
        fill_ragged_frames(fr, nf, src.data(), src_pitch.data(), reinterpret_cast<RaggedFrame*>(h + off_frames),
                           reinterpret_cast<uint32_t*>(h + off_bases));
        RaggedGrayJob* hj = reinterpret_cast<RaggedGrayJob*>(h + off_jobs);
        for (int i = 0; bgr && i < nf; ++i) {
            const b200_frame& f = fr[i];
            hj[i] = RaggedGrayJob{f.in, f.in_row_pitch, const_cast<uint8_t*>(src[(size_t)i]), src_pitch[(size_t)i], (int)row0, f.width};
            row0 += f.height;
        }
        memcpy(h + off_items, items_tma.data(), items_tma.size() * sizeof(RaggedItem));
        memcpy(h + off_items + items_tma.size() * sizeof(RaggedItem), items_byte.data(), items_byte.size() * sizeof(RaggedItem));
    }, &d));
    if (bgr) CB_TRY(launch_bgr_to_gray_ragged(ctx, st, reinterpret_cast<const RaggedGrayJob*>(d + off_jobs), nf, row0));

    FrontParams fp;
    memset(&fp, 0, sizeof(fp));
    fp.out_rows = 1; fp.tiles_y = 1;
    fp.w = ctx->gauss.d_w; fp.count = ctx->gauss.d_count; fp.radius = radius;
    fill_thresholds(fp, lo, hi);
    fp.parent = reinterpret_cast<int32_t*>(ctx->ws_parent[s].ptr);
    fp.kept_count = reinterpret_cast<unsigned int*>(ctx->ws_list[s].ptr);
    fp.kept_list = reinterpret_cast<uint32_t*>(ctx->ws_list[s].ptr) + 16;
    fp.rframes = reinterpret_cast<const RaggedFrame*>(d + off_frames);
    fp.rtmaps = reinterpret_cast<const CUtensorMap*>(d);
    // the list's counter block is zero here (see run_frames_device)
    if (ctx->list_dirty[s]) CB_CUDA(cudaMemsetAsync(fp.kept_count, 0, 64, st));
    ctx->list_dirty[s] = true;
    const RaggedItem* d_items = reinterpret_cast<const RaggedItem*>(d + off_items);
    fp.ritems = d_items;
    CB_TRY(launch_front3_ragged(ctx, st, fp, (int)items_tma.size(), true));
    fp.ritems = d_items + items_tma.size();
    CB_TRY(launch_front3_ragged(ctx, st, fp, (int)items_byte.size(), false));
    RaggedHystParams hp;
    memset(&hp, 0, sizeof(hp));
    hp.frames = fp.rframes;
    hp.bases = reinterpret_cast<const uint32_t*>(d + off_bases);
    hp.n_frames = nf;
    hp.parent = fp.parent; hp.list = fp.kept_list; hp.ctr = fp.kept_count;
    hp.px = px;
    CB_TRY(launch_hysteresis_ragged(ctx, st, hp));
    ctx->list_dirty[s] = false;
    return B200_OK;
}

// One chunk of an OpenCV-compatible list (b200_cv_canny_frames_device) on slot s / stream st: table (frame descriptors | bases | tile
// items) sent up as run_ragged_chunk's, then the OpenCV front kernel over every frame's 128 x 64 tiles and the list-driven hysteresis
// kernels with plain 8-connectivity.  No Gaussian tables, tensor maps, band height or B,G,R jobs: the kernel stages the caller's 1 or
// 3 interleaved bytes per pixel itself, 16-byte loads where a chunk of a row is aligned and byte loads elsewhere.  As run_frames_cv,
// the uniform path's density state (h_kept, kept_px) is neither read nor written.
static int run_ragged_cv_chunk(b200_ctx* ctx, cudaStream_t st, int s, const b200_frame* fr, int nf, const CvSpec& cv) {
    std::vector<RaggedItem> items;
    long long px = 0;
    for (int i = 0; i < nf; ++i) {
        ragged_items_cv(i, fr[i].height, fr[i].width, items);
        px += (long long)fr[i].height * fr[i].width;
    }
    const size_t off_bases = align16((size_t)nf * sizeof(RaggedFrame));
    const size_t off_items = align16(off_bases + (size_t)nf * sizeof(uint32_t));
    const size_t bytes = off_items + items.size() * sizeof(RaggedItem);
    uint8_t* d = nullptr;
    CB_TRY(upload_ragged_table(ctx, st, s, bytes, [&](uint8_t* h) {
        fill_ragged_frames(fr, nf, nullptr, nullptr, reinterpret_cast<RaggedFrame*>(h), reinterpret_cast<uint32_t*>(h + off_bases));
        memcpy(h + off_items, items.data(), items.size() * sizeof(RaggedItem));
    }, &d));

    FrontParams fp;
    memset(&fp, 0, sizeof(fp));
    fp.lo = cv.lo; fp.hi = cv.hi;
    fp.parent = reinterpret_cast<int32_t*>(ctx->ws_parent[s].ptr);
    fp.kept_count = reinterpret_cast<unsigned int*>(ctx->ws_list[s].ptr);
    fp.kept_list = reinterpret_cast<uint32_t*>(ctx->ws_list[s].ptr) + 16;
    fp.rframes = reinterpret_cast<const RaggedFrame*>(d);
    fp.ritems = reinterpret_cast<const RaggedItem*>(d + off_items);
    // the list's counter block is zero here (see run_frames_device)
    if (ctx->list_dirty[s]) CB_CUDA(cudaMemsetAsync(fp.kept_count, 0, 64, st));
    ctx->list_dirty[s] = true;
    CB_TRY(launch_front_cv_ragged(ctx, st, fp, (int)items.size(), cv.channels, cv.l2, cv.aperture));
    RaggedHystParams hp;
    memset(&hp, 0, sizeof(hp));
    hp.frames = fp.rframes;
    hp.bases = reinterpret_cast<const uint32_t*>(d + off_bases);
    hp.n_frames = nf;
    hp.parent = fp.parent; hp.list = fp.kept_list; hp.ctr = fp.kept_count;
    hp.px = px;
    hp.opencv = 1;
    CB_TRY(launch_hysteresis_ragged(ctx, st, hp));
    ctx->list_dirty[s] = false;
    return B200_OK;
}

// cv: an OpenCV-compatible list (b200_cv_canny_frames_device; its channel count and thresholds are checked by the caller, sigma, lo
// and hi are unused): the same checks (frames from 1 x 1), chunks, slots and workspace, each chunk through run_ragged_cv_chunk.  It
// needs no sigma, so it never prepares Gaussian tables and never takes the per-frame fallback.  Null: the reference's semantics.
static int frames_device_impl(b200_ctx* ctx, const b200_frame* fr, int n, float sigma, int lo, int hi, int bpp,
                              const CvSpec* cv = nullptr) {
    CB_TRY(check_frames(fr, n, bpp, cv ? 1 : 2));
    if (!cv) CB_TRY(check_thresholds(lo, hi));
    CB_TRY(resolve_ctx(ctx));
    if (!cv) {
        CB_TRY(prepare_gauss(ctx, sigma));
        if (!front3_supports(ctx->gauss)) {
            // no ragged kernel for this sigma: each frame through the strided path
            for (int i = 0; i < n; ++i) {
                const b200_frame& f = fr[i];
                CB_TRY(batch_device_impl(ctx, f.in, f.in_row_pitch, f.height * f.in_row_pitch, 1, f.height, f.width, sigma, lo, hi, f.out,
                                         f.out_row_pitch, f.height * f.out_row_pitch, bpp));
            }
            return B200_OK;
        }
    }
    // chunks in call order: about the uniform path's pixel budget each, at most chunk_frames (b200_ctx_set_chunk_frames) frames;
    // a frame above the budget has a chunk of its own
    const int cap = std::min(ctx->chunk_frames > 0 ? ctx->chunk_frames : kMaxChunkFrames, kMaxChunkFrames);
    std::vector<int> starts;
    long long chunk_px = 0, max_px = 0, max_gray = 0, gray = 0;
    for (int i = 0; i < n; ++i) {
        const long long fpx = (long long)fr[i].height * fr[i].width;
        if (i == 0 || (chunk_px + fpx > kRaggedChunkPx || i - starts.back() >= cap)) {
            starts.push_back(i);
            chunk_px = 0;
            gray = 0;
        }
        chunk_px += fpx;
        gray += ((fr[i].width + 15) & ~15LL) * fr[i].height;
        max_px = std::max(max_px, chunk_px);
        max_gray = std::max(max_gray, gray);
    }
    starts.push_back(n);
    const int n_chunks = (int)starts.size() - 1;
    const int n_slots = std::min(3, n_chunks);
    const bool gray_scratch = bpp == 3 && !cv;   // the OpenCV kernel reads 3-channel frames itself
    for (int s = 0; s < n_slots; ++s) {
        CB_TRY(ensure_ws(ctx->ws_parent[s], (size_t)max_px * 4));
        CB_TRY(ensure_ws(ctx->ws_list[s], 64 + (size_t)max_px * 4));
        if (gray_scratch) CB_TRY(ensure_ws(ctx->dev_in[s], (size_t)max_gray));
    }
    auto run_chunk = [&](cudaStream_t st, int s, int c) -> int {
        const b200_frame* f = fr + starts[(size_t)c];
        const int nf = starts[(size_t)c + 1] - starts[(size_t)c];
        return cv ? run_ragged_cv_chunk(ctx, st, s, f, nf, *cv) : run_ragged_chunk(ctx, st, s, f, nf, lo, hi, bpp == 3);
    };
    if (n_slots == 1) return run_chunk(ctx->stream, 0, 0);
    // the same three stream slots and fork / join as batch_device_impl
    CB_CUDA(cudaEventRecord(ctx->ev_fork, ctx->stream));
    for (int s = 0; s < n_slots; ++s) CB_CUDA(cudaStreamWaitEvent(ctx->side[s], ctx->ev_fork, 0));
    for (int c = 0; c < n_chunks; ++c) CB_TRY(run_chunk(ctx->side[c % n_slots], c % n_slots, c));
    for (int s = 0; s < n_slots; ++s) {
        CB_CUDA(cudaEventRecord(ctx->ev_join[s], ctx->side[s]));
        CB_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_join[s], 0));
    }
    return B200_OK;
}

int b200_canny_frames_device(b200_ctx* ctx, const b200_frame* frames, int n_frames, float sigma, int min_val, int max_val) {
    return frames_device_impl(ctx, frames, n_frames, sigma, min_val, max_val, 1);
}

int b200_canny_frames_device_bgr(b200_ctx* ctx, const b200_frame* frames, int n_frames, float sigma, int min_val, int max_val) {
    return frames_device_impl(ctx, frames, n_frames, sigma, min_val, max_val, 3);
}

int b200_cv_canny_aperture_frames_device(b200_ctx* ctx, const b200_frame* frames, int n_frames, int channels, double threshold1,
                                         double threshold2, int aperture_size, int l2_gradient) {
    CvSpec cv;
    // a list's 1-D grid has no height limit
    CB_TRY(cv_spec(channels, aperture_size, 0, INT_MAX, threshold1, threshold2, l2_gradient, &cv));
    return frames_device_impl(ctx, frames, n_frames, 0.f, 0, 0, channels, &cv);
}

int b200_cv_canny_frames_device(b200_ctx* ctx, const b200_frame* frames, int n_frames, int channels, double threshold1,
                                double threshold2, int l2_gradient) {
    return b200_cv_canny_aperture_frames_device(ctx, frames, n_frames, channels, threshold1, threshold2, 3, l2_gradient);
}

// Host buffers in, host buffers out: frames -> 0 / 255 edge maps, as bytes (edges8) or as the reference's int16 (edges16).
// Chunks of frames are pipelined over three stream slots (H2D | kernels | D2H + host expansion).  Pageable caller memory is staged
// through pinned buffers by the host pool; the maps come back bit-packed unless the job is small AND the output buffer is pinned.
// bits_out: the caller takes the maps PACKED (b200_canny_batch_host_packed): frame f's bits start at word f * ceil(px / 32); the
// packed chunks are copied straight into the caller's buffer and no host pass runs.
static int batch_host_impl(b200_ctx* ctx, const uint8_t* frames, int n_frames, int h, int w, int lo, int hi, uint8_t* edges8,
                           int16_t* edges16, bool packed, uint32_t* bits_out) {
    const long long px = (long long)h * w;
    const size_t frame_words = ((size_t)px + 31) / 32;
    // chunks of ~64 MB: big enough for full PCIe rate, small enough that three are in flight
    int chunk = ctx->chunk_frames > 0 ? ctx->chunk_frames : (int)std::max<long long>(1, (64LL << 20) / px);
    chunk = std::min(std::min(chunk, n_frames), kMaxChunkFrames);
    const int n_chunks = (n_frames + chunk - 1) / chunk;
    const int n_slots = std::min(3, n_chunks);
    const bool stage_in = is_pageable(frames) && (long long)n_frames * px >= kStageMinBytes;
    if (edges16 && !packed) { set_error("internal: int16 output needs the packed path"); return B200_ERR_INVALID_ARG; }
    const size_t chunk_bits_bytes = bits_out ? (size_t)chunk * frame_words * 4 : (((size_t)px * (size_t)chunk + 31) / 32) * 4;
    for (int s = 0; s < n_slots; ++s) {
        CB_TRY(ensure_ws(ctx->ws_parent[s], (size_t)px * 4 * (size_t)chunk));
        CB_TRY(ensure_ws(ctx->ws_list[s], list_bytes(chunk, h, w)));
        CB_TRY(ensure_ws(ctx->dev_in[s], (size_t)px * (size_t)chunk));
        CB_TRY(ensure_ws(ctx->dev_out[s], (size_t)px * (size_t)chunk));
        if (packed) {
            CB_TRY(ensure_ws(ctx->dev_bits[s], chunk_bits_bytes));
            if (!bits_out) CB_TRY(ensure_ws(ctx->host_bits[s], chunk_bits_bytes, /*pinned_host=*/true));
        }
        if (stage_in) CB_TRY(ensure_ws(ctx->host_in[s], (size_t)px * (size_t)chunk, /*pinned_host=*/true));
    }
    HostPool* pool = ((packed && !bits_out) || stage_in) ? get_pool(ctx) : nullptr;
    CB_CUDA(cudaEventRecord(ctx->ev_fork, ctx->stream));
    for (int s = 0; s < n_slots; ++s) CB_CUDA(cudaStreamWaitEvent(ctx->side[s], ctx->ev_fork, 0));
    auto finish_chunk = [&](int c) -> int {  // host side of chunk c: wait for its packed map, expand it into the caller's buffer
        const int f0 = c * chunk, nf = std::min(chunk, n_frames - f0);
        const int s = c % n_slots;
        CB_CUDA(cudaEventSynchronize(ctx->ev_chunk[s]));
        const uint8_t* bits = reinterpret_cast<const uint8_t*>(ctx->host_bits[s].ptr);
        if (edges16) pool->run(HostPool::kUnpackI16, bits, edges16 + (long long)f0 * px, (size_t)px * nf);
        else pool->run(HostPool::kUnpackU8, bits, edges8 + (long long)f0 * px, (size_t)px * nf);
        return B200_OK;
    };
    for (int c = 0; c < n_chunks; ++c) {
        const int f0 = c * chunk, nf = std::min(chunk, n_frames - f0);
        const int s = c % n_slots;
        cudaStream_t st = ctx->side[s];
        uint8_t* din = reinterpret_cast<uint8_t*>(ctx->dev_in[s].ptr);
        uint8_t* dout = reinterpret_cast<uint8_t*>(ctx->dev_out[s].ptr);
        // slot reuse: chunk c's device buffers are ordered by the stream; its pinned host_bits[s] was consumed by
        // finish_chunk(c - n_slots), which ran before this iteration (see below); host_in[s] is free once ev_in[s] has fired
        const uint8_t* h_src = frames + (long long)f0 * px;
        if (stage_in) {
            if (ctx->in_busy[s]) { CB_CUDA(cudaEventSynchronize(ctx->ev_in[s])); ctx->in_busy[s] = false; }
            pool->run(HostPool::kCopy, h_src, ctx->host_in[s].ptr, (size_t)px * nf);
            h_src = reinterpret_cast<const uint8_t*>(ctx->host_in[s].ptr);
        }
        CB_CUDA(cudaMemcpyAsync(din, h_src, (size_t)px * nf, cudaMemcpyHostToDevice, st));
        if (stage_in) { CB_CUDA(cudaEventRecord(ctx->ev_in[s], st)); ctx->in_busy[s] = true; }
        ctx->h2d_bytes += (unsigned long long)px * nf;
        ctx->d2h_bytes += packed ? (unsigned long long)(((size_t)px * nf + 31) / 32) * 4 : (unsigned long long)px * nf;
        CB_TRY(run_frames_device(ctx, st, s, din, dout, nf, h, w, lo, hi, nullptr, nullptr, nullptr, nullptr));
        if (bits_out) {
            uint32_t* dbits = reinterpret_cast<uint32_t*>(ctx->dev_bits[s].ptr);
            if ((px & 31) == 0) {
                CB_TRY(launch_pack_edges(ctx, st, dout, dbits, (size_t)px * nf));           // frames are whole words: one launch
            } else {
                for (int f = 0; f < nf; ++f) CB_TRY(launch_pack_edges(ctx, st, dout + (size_t)f * px, dbits + (size_t)f * frame_words, (size_t)px));
            }
            CB_CUDA(cudaMemcpyAsync(bits_out + (size_t)f0 * frame_words, dbits, (size_t)nf * frame_words * 4, cudaMemcpyDeviceToHost, st));
            ctx->d2h_bytes += (unsigned long long)nf * frame_words * 4 - (unsigned long long)(((size_t)px * nf + 31) / 32) * 4;
        } else if (packed) {
            uint32_t* dbits = reinterpret_cast<uint32_t*>(ctx->dev_bits[s].ptr);
            CB_TRY(launch_pack_edges(ctx, st, dout, dbits, (size_t)px * nf));
            CB_CUDA(cudaMemcpyAsync(ctx->host_bits[s].ptr, dbits, (((size_t)px * nf + 31) / 32) * 4, cudaMemcpyDeviceToHost, st));
            CB_CUDA(cudaEventRecord(ctx->ev_chunk[s], st));
            // keep n_slots chunks in flight on the GPU; expand the oldest one while they run
            if (c >= n_slots - 1) CB_TRY(finish_chunk(c - (n_slots - 1)));
        } else {
            CB_CUDA(cudaMemcpyAsync(edges8 + (long long)f0 * px, dout, (size_t)px * nf, cudaMemcpyDeviceToHost, st));
        }
    }
    if (packed && !bits_out)
        for (int c = std::max(0, n_chunks - (n_slots - 1)); c < n_chunks; ++c) CB_TRY(finish_chunk(c));
    for (int s = 0; s < n_slots; ++s) {
        CB_CUDA(cudaEventRecord(ctx->ev_join[s], ctx->side[s]));
        CB_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_join[s], 0));
    }
    CB_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int s = 0; s < 3; ++s) ctx->in_busy[s] = false;   // everything issued above has completed
    return B200_OK;
}

static bool packed_transfer_off() {
    static const bool off = [] { const char* e = getenv("B200_CANNY_NO_PACKED_D2H"); return e && e[0] == '1'; }();
    return off;
}

int b200_canny_batch_host(b200_ctx* ctx, const uint8_t* frames, int n_frames, int h, int w, float sigma, int lo, int hi,
                          uint8_t* edges) {
    CB_TRY(check_image(frames, edges, h, w));
    CB_TRY(check_thresholds(lo, hi));
    if (n_frames <= 0) { set_error("n_frames must be positive"); return B200_ERR_INVALID_ARG; }
    CB_TRY(resolve_ctx(ctx));
    CB_TRY(prepare_gauss(ctx, sigma));
    const long long total = (long long)n_frames * h * w;
    // small jobs are latency-bound: the byte map goes back directly (no pack kernel, no host pass)
    const bool packed = !packed_transfer_off() && total >= (8LL << 20);
    return batch_host_impl(ctx, frames, n_frames, h, w, lo, hi, edges, nullptr, packed);
}

int b200_canny_batch_host_packed(b200_ctx* ctx, const uint8_t* frames, int n_frames, int h, int w, float sigma, int lo, int hi,
                                 uint32_t* edge_bits) {
    CB_TRY(check_image(frames, edge_bits, h, w));
    CB_TRY(check_thresholds(lo, hi));
    if (n_frames <= 0) { set_error("n_frames must be positive"); return B200_ERR_INVALID_ARG; }
    CB_TRY(resolve_ctx(ctx));
    CB_TRY(prepare_gauss(ctx, sigma));
    return batch_host_impl(ctx, frames, n_frames, h, w, lo, hi, nullptr, nullptr, true, edge_bits);
}

int b200_pack_edges_device(b200_ctx* ctx, const uint8_t* d_edges, size_t n_px, uint32_t* d_bits) {
    if (!d_edges || !d_bits || n_px == 0) { set_error("bad argument to b200_pack_edges_device"); return B200_ERR_INVALID_ARG; }
    CB_TRY(resolve_ctx(ctx));
    return launch_pack_edges(ctx, ctx->stream, d_edges, d_bits, n_px);
}

int b200_unpack_edges_host(const uint8_t* bits, size_t n_px, void* out, int elem_size, int threads) {
    if (!bits || !out || (elem_size != 1 && elem_size != 2)) { set_error("bad argument to b200_unpack_edges_host"); return B200_ERR_INVALID_ARG; }
    if (n_px == 0) return B200_OK;
    if (threads <= 0) {
        const unsigned hc = std::thread::hardware_concurrency();
        threads = (int)std::min<unsigned>(std::max<unsigned>((hc ? hc : 4) / 2u, 1), 4);
    }
    HostPool pool(std::min(threads, 64) - 1);   // short-lived: this entry point has no context to keep one in
    pool.run(elem_size == 1 ? HostPool::kUnpackU8 : HostPool::kUnpackI16, bits, out, n_px);
    return B200_OK;
}

static int profile_impl(b200_ctx* ctx, const uint8_t* d_frames, int n_frames, int h, int w, float sigma, int lo, int hi,
                        uint8_t* d_edges, float* ms_out, int* launches_out, bool pipelined);
int b200_profile_stages_device(b200_ctx* ctx, const uint8_t* d_frames, int n_frames, int h, int w, float sigma, int lo, int hi,
                               uint8_t* d_edges, float* ms_out, int* launches_out) {
    return profile_impl(ctx, d_frames, n_frames, h, w, sigma, lo, hi, d_edges, ms_out, launches_out, false);
}
int b200_profile_pipeline_device(b200_ctx* ctx, const uint8_t* d_frames, int n_frames, int h, int w, float sigma, int lo, int hi,
                                 uint8_t* d_edges, float* ms_out, int* launches_out) {
    return profile_impl(ctx, d_frames, n_frames, h, w, sigma, lo, hi, d_edges, ms_out, launches_out, true);
}
static int profile_impl(b200_ctx* ctx, const uint8_t* d_frames, int n_frames, int h, int w, float sigma, int lo, int hi,
                        uint8_t* d_edges, float* ms_out, int* launches_out, bool pipelined) {
    CB_TRY(check_image(d_frames, d_edges, h, w));
    CB_TRY(check_thresholds(lo, hi));
    if (!ms_out || !launches_out || n_frames <= 0) { set_error("bad argument"); return B200_ERR_INVALID_ARG; }
    CB_TRY(resolve_ctx(ctx));
    CB_TRY(prepare_gauss(ctx, sigma));
    const long long px = (long long)h * w;
    const int chunk = auto_chunk_frames(ctx, h, w, n_frames);
    CB_TRY(ensure_ws(ctx->ws_parent[0], (size_t)px * 4 * (size_t)chunk));
    CB_TRY(ensure_ws(ctx->ws_list[0], list_bytes(chunk, h, w)));
    CB_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->prof.recs.clear();
    ctx->prof.on = true;
    int status = B200_OK;
    if (pipelined) {
        // the production path itself (three stream slots): every kernel's events sit on its own stream, so the durations
        // include whatever the kernel shares the machine with
        status = b200_canny_batch_device(ctx, d_frames, n_frames, h, w, sigma, lo, hi, d_edges);
    } else {
        for (int f0 = 0; f0 < n_frames && status == B200_OK; f0 += chunk) {
            const int nf = std::min(chunk, n_frames - f0);
            status = run_frames_device(ctx, ctx->stream, 0, d_frames + (long long)f0 * px, d_edges + (long long)f0 * px, nf, h, w, lo, hi,
                                       nullptr, nullptr, nullptr, nullptr);
        }
    }
    ctx->prof.on = false;
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    for (int c = 0; c < 5; ++c) { ms_out[c] = 0.f; launches_out[c] = 0; }
    for (auto& r : ctx->prof.recs) {
        float ms = 0.f;
        if (e == cudaSuccess && cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) { ms_out[r.cat] += ms; launches_out[r.cat]++; }
        cudaEventDestroy(r.a);
        cudaEventDestroy(r.b);
    }
    ctx->prof.recs.clear();
    if (e != cudaSuccess) { set_error("profile run failed: %s", cudaGetErrorString(e)); return B200_ERR_CUDA; }
    return status;
}

// ---- synthetic workloads / helpers -------------------------------------------------------------------------
int b200_synth_rows_host(uint8_t* out, int row0, int rows, int width, int kind, uint64_t seed, int frame) {
    if (!out || rows < 0 || width <= 0) { set_error("bad argument to b200_synth_rows_host"); return B200_ERR_INVALID_ARG; }
    for (int r = 0; r < rows; ++r)
        for (int c = 0; c < width; ++c) out[(size_t)r * width + c] = synth_pixel(kind, seed, frame, c, row0 + r);
    return B200_OK;
}
int b200_synth_host(uint8_t* frames, int n_frames, int h, int w, int kind, uint64_t seed, int first_frame) {
    if (!frames || n_frames < 0) { set_error("bad argument to b200_synth_host"); return B200_ERR_INVALID_ARG; }
    for (int f = 0; f < n_frames; ++f) CB_TRY(b200_synth_rows_host(frames + (size_t)f * h * w, 0, h, w, kind, seed, first_frame + f));
    return B200_OK;
}
int b200_synth_rows_device(b200_ctx* ctx, uint8_t* d_rows, int row0, int rows, int width, int kind, uint64_t seed, int frame) {
    if (!d_rows || rows <= 0 || width <= 0) { set_error("bad argument to b200_synth_rows_device"); return B200_ERR_INVALID_ARG; }
    CB_TRY(resolve_ctx(ctx));
    return launch_synth(ctx, ctx->stream, d_rows, 1, row0, rows, width, kind, seed, frame);
}
int b200_synth_device(b200_ctx* ctx, uint8_t* d_frames, int n_frames, int h, int w, int kind, uint64_t seed, int first_frame) {
    if (!d_frames || n_frames <= 0 || h <= 0 || w <= 0) { set_error("bad argument to b200_synth_device"); return B200_ERR_INVALID_ARG; }
    CB_TRY(resolve_ctx(ctx));
    return launch_synth(ctx, ctx->stream, d_frames, n_frames, 0, h, w, kind, seed, first_frame);
}

int b200_count_edges_device(b200_ctx* ctx, const uint8_t* d_edges, size_t n, unsigned long long* count) {
    if (!d_edges || !count) { set_error("null pointer"); return B200_ERR_INVALID_ARG; }
    CB_TRY(resolve_ctx(ctx));
    CB_TRY(ensure_ws(ctx->ws_misc, 256));
    unsigned long long* d = reinterpret_cast<unsigned long long*>(ctx->ws_misc.ptr);
    CB_TRY(launch_count255(ctx, ctx->stream, d_edges, n, d));
    CB_CUDA(cudaMemcpyAsync(count, d, sizeof(*count), cudaMemcpyDeviceToHost, ctx->stream));
    CB_CUDA(cudaStreamSynchronize(ctx->stream));
    return B200_OK;
}

int b200_hash_edges_device(b200_ctx* ctx, const uint8_t* d_edges, size_t n, unsigned long long global_offset, unsigned long long* hash) {
    if (!d_edges || !hash) { set_error("null pointer"); return B200_ERR_INVALID_ARG; }
    CB_TRY(resolve_ctx(ctx));
    CB_TRY(ensure_ws(ctx->ws_misc, 256));
    unsigned long long* d = reinterpret_cast<unsigned long long*>(ctx->ws_misc.ptr) + 8;
    CB_TRY(launch_hash255(ctx, ctx->stream, d_edges, n, global_offset, d));
    CB_CUDA(cudaMemcpyAsync(hash, d, sizeof(*hash), cudaMemcpyDeviceToHost, ctx->stream));
    CB_CUDA(cudaStreamSynchronize(ctx->stream));
    return B200_OK;
}

int b200_device_alloc(b200_ctx* ctx, size_t bytes, void** d_ptr) {
    if (!d_ptr) { set_error("null pointer"); return B200_ERR_INVALID_ARG; }
    CB_TRY(resolve_ctx(ctx));
    cudaError_t e = cudaMalloc(d_ptr, bytes ? bytes : 1);
    if (e != cudaSuccess) { cudaGetLastError(); set_error("cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e)); return B200_ERR_NOMEM; }
    return B200_OK;
}
int b200_device_free(b200_ctx* ctx, void* d_ptr) {
    CB_TRY(resolve_ctx(ctx));
    CB_CUDA(cudaFree(d_ptr));
    return B200_OK;
}
int b200_memcpy_h2d(b200_ctx* ctx, void* d_dst, const void* h_src, size_t bytes) {
    CB_TRY(resolve_ctx(ctx));
    CB_CUDA(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CB_CUDA(cudaStreamSynchronize(ctx->stream));
    return B200_OK;
}
int b200_memcpy_d2h(b200_ctx* ctx, void* h_dst, const void* d_src, size_t bytes) {
    CB_TRY(resolve_ctx(ctx));
    CB_CUDA(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CB_CUDA(cudaStreamSynchronize(ctx->stream));
    return B200_OK;
}
int b200_host_alloc_pinned(size_t bytes, void** h_ptr) {
    if (!h_ptr) { set_error("null pointer"); return B200_ERR_INVALID_ARG; }
    cudaError_t e = cudaMallocHost(h_ptr, bytes ? bytes : 1);
    if (e != cudaSuccess) { cudaGetLastError(); set_error("cudaMallocHost(%zu) failed: %s", bytes, cudaGetErrorString(e)); return B200_ERR_NOMEM; }
    return B200_OK;
}
int b200_host_free_pinned(void* h_ptr) {
    CB_CUDA(cudaFreeHost(h_ptr));
    return B200_OK;
}

}  // extern "C"
