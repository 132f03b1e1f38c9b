// hysteresis.cu — stage 4 as GPU connected components.
//
// Replaces hysteresis() + findEdgePixels() (src/utils.cpp:322-342, 360-427), which the reference runs on
// the CPU even in its CUDA path (src/cuda.cu:436).  The reference floods breadth-first from every pixel
// >= maxVal through 8-connected pixels >= minVal.  Equivalent formulation used here:
//   candidates = class != 0, seeds = class 255; label the 8-connected components of the candidates with a
//   union-find forest; a weak pixel survives iff its component contains a seed.
// "Contains a seed" is folded into the forest itself: every component that holds a seed is linked under
// one virtual root SUPER (-1, smaller than any pixel index, never stored as a slot), so the final test is
// find(p) == SUPER and no separate flag propagation pass exists.
//
// The reference's single missing directed link (src/utils.cpp:399: `current - width > 0` is false for
// current == width) means pixel (1,0) never reaches (0,1) although (0,1) reaches (1,0).  The edge
// (0,1)-(1,0) is therefore left out of the forest and re-applied one-way in the final pass: if (0,1)'s
// component is strong, (1,0)'s becomes strong; not the other way round.
//
// Two kernel families, identical results:
//   list-driven (the default after the lean front kernels, which hand over a list of the WEAK pixels and their union-find slots):
//     ccl_sparse_link     one thread per weak pixel: strong neighbour -> SUPER, unions with its forward weak neighbours; the
//                         last block applies the one-way link and retires the list's counters (HystParams::ctr)
//     ccl_sparse_resolve  every weak pixel chases its root and becomes 0 or 255
//     ragged chunks (frames of different sizes, b200_canny_frames_device and b200_cv_canny_frames_device) always take the list-driven
//     pair, in a form that finds each entry's frame in the chunk's table (ccl_ragged_link / ccl_ragged_resolve; the link kernel
//     has the same OpenCV switch, RaggedHystParams::opencv); the tile-based family below serves uniform batches only
//     launches of the OpenCV-compatible path (HystParams::opencv) take the list-driven pair too, with plain 8-connectivity: no pair
//     is left out and no one-way link is applied
//   tile-based (stage API, minVal <= 0, maps with more than 1/8 weak pixels; reference semantics only):
//     ccl_local   one CTA per 64x64 tile: union-find in shared memory (atomicMin links, row-run seeding
//                 with warp ballots), then writes each candidate's parent (its tile root, or SUPER).
//     ccl_merge   one thread per pixel on a tile boundary: lock-free atomicMin unions in global memory.
//     ccl_final   every weak pixel chases its root; rewrites the class map to 0 / 255 in place.
#include <string.h>

#include <algorithm>

#include "ccl.cuh"
#include "internal.h"

namespace cb {


// ---------------------------------------------------------------------------------------------
// kernel 1: tile-local labelling
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kCclThreads)
ccl_local_kernel(const HystParams p) {
    __shared__ unsigned char s_cls[kTile][kTile + 16];
    __shared__ int s_lab[kTile * kTile];
    __shared__ unsigned char s_strong[kTile * kTile];
    __shared__ int s_any;

    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * kTile, y0 = blockIdx.y * kTile;
    const int frame = blockIdx.z;
    const uint8_t* cls = p.cls + (long long)frame * p.cls_frame_stride;
    int32_t* parent = p.parent + (long long)frame * p.frame_stride;
    const int W = p.width, Hh = p.rows;
    const long long cp = p.cls_pitch;

    if (tid == 0) s_any = 0;
    __syncthreads();

    // ---- load the tile (16 B per thread-iteration when aligned), remember whether it has any candidate ----
    const bool vec_ok = ((cp & 15) == 0) && ((reinterpret_cast<uintptr_t>(cls) & 15) == 0);
    int any = 0;
    for (int i = tid; i < kTile * (kTile / 16); i += kCclThreads) {
        const int r = i >> 2, q = i & 3;
        const int y = y0 + r, x = x0 + 16 * q;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (y < Hh) {
            if (vec_ok && x + 15 < W) {
                v = __ldg(reinterpret_cast<const uint4*>(cls + (long long)y * cp + x));
            } else {
                unsigned char tmp[16];
                for (int e = 0; e < 16; ++e) tmp[e] = (x + e < W) ? cls[(long long)y * cp + x + e] : 0;
                v = *reinterpret_cast<uint4*>(tmp);
            }
        }
        *reinterpret_cast<uint4*>(&s_cls[r][16 * q]) = v;
        any |= (v.x | v.y | v.z | v.w) != 0;
    }
    if (any) s_any = 1;
    __syncthreads();
    if (!s_any) return;  // nothing to label in this tile (the common case on sparse edge maps)

    // ---- seed labels: every candidate starts at the head of its horizontal run ----
    // warp w handles rows w, w+8, ...; lanes cover the 64 columns in two halves, run heads found with ballots
    const int lane = tid & 31, warp = tid >> 5;
    for (int r = warp; r < kTile; r += kCclThreads / 32) {
        const bool c_lo = s_cls[r][lane] != 0, c_hi = s_cls[r][32 + lane] != 0;
        const unsigned m_lo = __ballot_sync(0xffffffffu, c_lo), m_hi = __ballot_sync(0xffffffffu, c_hi);
        const unsigned long long m = ((unsigned long long)m_hi << 32) | m_lo;
        // head of the run containing column c: one past the highest zero bit below c
        {
            const int c = lane;
            int lab = -1;
            if (c_lo) {
                const unsigned long long below = ~m & ((1ull << c) - 1ull);
                const int head = below ? (64 - __clzll(below)) : 0;
                lab = r * kTile + head;
            }
            s_lab[r * kTile + c] = lab;
            s_strong[r * kTile + c] = 0;
        }
        {
            const int c = 32 + lane;
            int lab = -1;
            if (c_hi) {
                const unsigned long long below = ~m & ((1ull << c) - 1ull);
                const int head = below ? (64 - __clzll(below)) : 0;
                lab = r * kTile + head;
            }
            s_lab[r * kTile + c] = lab;
            s_strong[r * kTile + c] = 0;
        }
    }
    __syncthreads();

    // ---- vertical / diagonal unions: only run heads... every candidate whose upper neighbours are candidates ----
    // (left neighbour is already in the same run).  The pair (1,0)-(0,1) of the GLOBAL image is skipped.
    for (int i = tid; i < kTile * kTile; i += kCclThreads) {
        const int r = i >> 6, c = i & 63;
        if (r == 0 || s_cls[r][c] == 0) continue;
        const bool up = s_cls[r - 1][c] != 0;
        if (up) {
            s_union(s_lab, i, i - kTile);
        } else {
            // with `up` set, the two diagonals are already joined to it through their own runs
            if (c > 0 && s_cls[r - 1][c - 1] != 0) s_union(s_lab, i, i - kTile - 1);
            if (c < kTile - 1 && s_cls[r - 1][c + 1] != 0) {
                const bool quirk = (p.row0 + y0 + r == 1) && (x0 + c == 0);
                if (!quirk) s_union(s_lab, i, i - kTile + 1);
            }
        }
    }
    __syncthreads();

    // ---- flatten + mark roots of components that contain a seed ----
    for (int i = tid; i < kTile * kTile; i += kCclThreads) {
        const int r = i >> 6, c = i & 63;
        if (s_cls[r][c] == 0) continue;
        const int root = s_find(s_lab, i);
        s_lab[i] = root;
        if (s_cls[r][c] == 255) s_strong[root] = 1;
    }
    __syncthreads();

    // ---- publish: parent = tile root (as a frame-relative pixel index), or SUPER for the root of a strong component ----
    for (int i = tid; i < kTile * kTile; i += kCclThreads) {
        const int r = i >> 6, c = i & 63;
        if (s_cls[r][c] == 0) continue;
        const int root = s_lab[i];
        const int gi = (y0 + r) * W + (x0 + c);
        int val;
        if (root == i) val = s_strong[i] ? kSuper : gi;
        else val = (y0 + (root >> 6)) * W + (x0 + (root & 63));
        parent[gi] = val;
    }
}

// ---------------------------------------------------------------------------------------------
// kernel 2: unions across tile boundaries
// ---------------------------------------------------------------------------------------------
// work item space: [0, n_hb*W) horizontal boundaries (row 64i-1 | row 64i), then [.., + n_vb*H) vertical ones
__global__ void __launch_bounds__(256)
ccl_merge_kernel(const HystParams p) {
    const int W = p.width, Hh = p.rows;
    const int n_hb = p.tiles_y - 1, n_vb = p.tiles_x - 1;
    const long long n_h = (long long)n_hb * W, n_v = (long long)n_vb * Hh;
    const int frame = blockIdx.y;
    const uint8_t* cls = p.cls + (long long)frame * p.cls_frame_stride;
    int32_t* parent = p.parent + (long long)frame * p.frame_stride;
    const long long cp = p.cls_pitch;
    // a: dense index of the pixel (union-find slots), ca: its class byte
    for (long long it = (long long)blockIdx.x * blockDim.x + threadIdx.x; it < n_h + n_v;
         it += (long long)gridDim.x * blockDim.x) {
        if (it < n_h) {
            const int b = (int)(it / W), x = (int)(it - (long long)b * W);
            const int y = (b + 1) * kTile - 1;  // upper row of the boundary; y+1 < Hh because the tile below exists
            const int a = y * W + x;
            const long long ca = y * cp + x;
            if (cls[ca] == 0) continue;
            const int below = a + W;
            // (0,1)-(1,0), the one pair that must not be joined, never straddles a tile boundary (kTile > 1).
            if (cls[ca + cp] != 0) {
                // the two diagonals sit next to `below` in row y+1, so they reach `a` through it
                g_union(parent, a, below);
            } else {
                if (x > 0 && cls[ca + cp - 1] != 0) g_union(parent, a, below - 1);
                if (x < W - 1 && cls[ca + cp + 1] != 0) g_union(parent, a, below + 1);
            }
        } else {
            const long long j = it - n_h;
            const int b = (int)(j / Hh), y = (int)(j - (long long)b * Hh);
            const int x = (b + 1) * kTile - 1;  // left column of the boundary; x+1 < W because the tile to the right exists
            const int a = y * W + x;
            const long long ca = y * cp + x;
            if (cls[ca] == 0) continue;
            const int right = a + 1;
            if (cls[ca + 1] != 0) {
                g_union(parent, a, right);  // (y-1,x+1) and (y+1,x+1) are vertical neighbours of `right`
            } else {
                if (y > 0 && cls[ca + 1 - cp] != 0) g_union(parent, a, right - W);
                if (y < Hh - 1 && cls[ca + 1 + cp] != 0) g_union(parent, a, right + W);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// kernel 3: resolve weak pixels in place
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
ccl_final_kernel(const HystParams p) {
    __shared__ int s_qroot;
    const int W = p.width, Hh = p.rows;
    const int frame = blockIdx.y;
    uint8_t* cls = p.cls + (long long)frame * p.cls_frame_stride;
    const int32_t* parent = p.parent + (long long)frame * p.frame_stride;
    const long long cp = p.cls_pitch;

    // the one-way link (0,1) -> (1,0) of the global image (see file header)
    if (threadIdx.x == 0) {
        int q = kNone;
        if (p.row0 == 0 && Hh >= 2 && W >= 2 && cls[1] != 0 && cls[cp] != 0) {
            if (g_find(parent, 1) == kSuper) q = g_find(parent, W);
        }
        s_qroot = q;
    }
    __syncthreads();
    const int qroot = s_qroot;

    const long long n = (long long)Hh * W;
    if (cp != W) {
        // class map rows with a pitch of their own: blocks take rows, threads columns; only the rows' own bytes are read and written
        for (int y = blockIdx.x; y < Hh; y += gridDim.x) {
            uint8_t* row = cls + y * cp;
            for (int x = threadIdx.x; x < W; x += blockDim.x) {
                if (row[x] == 1) {
                    const int root = g_find(parent, y * W + x);
                    row[x] = (root == kSuper || root == qroot) ? 255 : 0;
                }
            }
        }
        return;
    }
    // dense rows: the frame is one flat run of bytes, walked 16 at a time (whole vectors are written back)
    const bool vec_ok = ((n & 15) == 0) && ((reinterpret_cast<uintptr_t>(cls) & 15) == 0);
    if (vec_ok) {
        const long long n16 = n >> 4;
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (long long)gridDim.x * blockDim.x) {
            uint4 v = *reinterpret_cast<const uint4*>(cls + 16 * i);
            uint32_t wv[4] = {v.x, v.y, v.z, v.w};
            bool changed = false;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                uint32_t w = wv[k];
                // any byte == 1 ?  (bytes are 0, 1 or 255)
                if (((w & 0x01010101u) & ~(w >> 1)) == 0) continue;
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    if (((w >> (8 * e)) & 0xFF) == 1) {
                        const int idx = (int)(16 * i + 4 * k + e);
                        const int root = g_find(parent, idx);
                        const uint32_t out = (root == kSuper || root == qroot) ? 255u : 0u;
                        w = (w & ~(0xFFu << (8 * e))) | (out << (8 * e));
                    }
                }
                wv[k] = w;
                changed = true;
            }
            if (changed) *reinterpret_cast<uint4*>(cls + 16 * i) = make_uint4(wv[0], wv[1], wv[2], wv[3]);
        }
    } else {
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
            if (cls[i] == 1) {
                const int root = g_find(parent, (int)i);
                cls[i] = (root == kSuper || root == qroot) ? 255 : 0;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// sparse variants: driven by the weak-pixel list front3 (uniform and ragged) and front_cv write (work ~ weak pixels, not pixels)
// ---------------------------------------------------------------------------------------------
// Only weak pixels (class 1) need anything: a strong pixel is final.  The front kernel has initialised parent[] of every weak pixel
// to its own launch-relative index.  One thread per weak pixel: the eight neighbours' class bytes are fetched together; any strong
// neighbour hangs the pixel's component under SUPER; weak "forward" neighbours E, S (or SW / SE when S is not weak: with S weak
// the two diagonals reach the pixel through S's own links) are united with it, so every weak-weak pair is visited exactly once,
// from its earlier endpoint in raster order.  The pair (0,1)-(1,0) of the GLOBAL image is skipped in both directions (see the
// file header): the one-way link is applied by the last block of this kernel, below.
// Programmatic dependent launch (sm_90+): a kernel launched with the programmatic-stream-serialization attribute may become resident
// while its predecessor in the stream still runs; griddepcontrol.wait then blocks until that grid has completed and its writes are
// visible.  launch_dependents lets the NEXT kernel in the stream do the same with this one.  Both are no-ops in ordinary launches.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// The list holds DENSE launch-relative indices g = f*frame_stride + y*width + x (the union-find slots); the class byte of that
// pixel is at f*cls_frame_stride + y*cls_pitch + x, which is g itself when the map is dense.
__device__ __forceinline__ long long cls_index(const HystParams& p, unsigned int g) {
    if (p.cls_pitch == p.width && p.cls_frame_stride == p.frame_stride) return g;
    const unsigned int fs = (unsigned int)p.frame_stride;
    const unsigned int f = g / fs, rel = g - f * fs;
    const unsigned int y = rel / (unsigned int)p.width, x = rel - y * (unsigned int)p.width;
    return (long long)f * p.cls_frame_stride + (long long)y * p.cls_pitch + x;
}

// OPENCV: cv::Canny's plain 8-connectivity (b200_cv_canny_device_strided) — the pair (0,1)-(1,0) is linked like any other and the
// last block applies no one-way link; it only retires the counters.
template <bool OPENCV>
__global__ void __launch_bounds__(256)
ccl_sparse_link_kernel(const HystParams p) {
    pdl_launch_dependents();
    pdl_wait();
    const unsigned int n_all = p.ctr[0];
    const unsigned int n = n_all;
    const uint32_t* const walk = p.list;
    const int W = p.width, Hh = p.rows;
    const unsigned int fs = (unsigned int)p.frame_stride;
    const long long cp = p.cls_pitch;
    for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const unsigned int g = walk[i];
        const unsigned int f = g / fs, rel = g - f * fs;
        const int y = (int)(rel / (unsigned int)W), x = (int)(rel - (unsigned int)y * (unsigned int)W);
        const uint8_t* c = p.cls + ((long long)f * p.cls_frame_stride + y * cp + x);
        const bool has_n = y > 0, has_s = y + 1 < Hh, has_w = x > 0, has_e = x + 1 < W;
        const bool top_rows = !OPENCV && (p.row0 + y) <= 1;
        const bool q01 = top_rows && (p.row0 + y == 0) && (x == 1);   // this pixel is (0,1): its SW neighbour (1,0) is off limits
        const bool q10 = top_rows && (p.row0 + y == 1) && (x == 0);   // this pixel is (1,0): its NE neighbour (0,1) is off limits
        const int c_nw = (has_n && has_w) ? c[-cp - 1] : 0;
        const int c_n = has_n ? c[-cp] : 0;
        const int c_ne = (has_n && has_e && !q10) ? c[-cp + 1] : 0;
        const int c_w = has_w ? c[-1] : 0;
        const int c_e = has_e ? c[1] : 0;
        const int c_sw = (has_s && has_w && !q01) ? c[cp - 1] : 0;
        const int c_s = has_s ? c[cp] : 0;
        const int c_se = (has_s && has_e) ? c[cp + 1] : 0;
        // classes are 0, 1 or 255: a strong neighbour anywhere around makes the component strong
        if (((c_nw | c_n | c_ne | c_w | c_e | c_sw | c_s | c_se) & 0x80) != 0) g_union_halve(p.parent, (int)g, kSuper);
        if (c_e == 1) g_union_halve(p.parent, (int)g, (int)g + 1);
        if (c_s == 1) {
            g_union_halve(p.parent, (int)g, (int)g + W);
        } else {
            if (c_sw == 1) g_union_halve(p.parent, (int)g, (int)g + W - 1);
            if (c_se == 1) g_union_halve(p.parent, (int)g, (int)g + W + 1);
        }
    }
    // The reference's one-way link (0,1) -> (1,0) (src/utils.cpp:399): once EVERY block has finished its unions the forest is
    // final, and the last block to get here hangs (1,0)'s component under SUPER when (0,1) is strong or strong-connected.  The
    // class bytes are still untouched at this point (the resolve kernel runs after this one).
    __shared__ bool s_last;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = atomicAdd(p.ctr + 1, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    if (!OPENCV && p.row0 == 0 && Hh >= 2 && W >= 2) {
        for (int f = threadIdx.x; f < p.n_frames; f += blockDim.x) {
            const unsigned int f0 = (unsigned int)f * fs;
            const uint8_t* cf = p.cls + (long long)f * p.cls_frame_stride;
            const int c01 = cf[1], c10 = cf[cp];
            if (c10 == 1 && (c01 == 255 || (c01 == 1 && g_find_halve(p.parent, (int)f0 + 1) == kSuper)))
                g_union_halve(p.parent, (int)f0 + W, kSuper);
        }
    }
    // every block has read ctr[0] by now: retire the counters (see HystParams::ctr)
    if (threadIdx.x == 0) {
        p.ctr[2] = n_all;
        if (p.h_kept && ((n_all > p.kept_thresh) != (p.kept_prev > p.kept_thresh))) *p.h_kept = n_all;
        p.ctr[0] = 0;
        p.ctr[1] = 0;
    }
}

// tile-based path after a front kernel that built a list nobody walks: publish and reset the counters all the same
__global__ void list_retire_kernel(unsigned int* ctr, unsigned int* h_kept, unsigned int kept_prev, unsigned int kept_thresh) {
    const unsigned int n = ctr[0];
    ctr[2] = n;
    if (h_kept && ((n > kept_thresh) != (kept_prev > kept_thresh))) *h_kept = n;
    ctr[0] = 0;
    ctr[1] = 0;
}

// every weak pixel chases its root: 255 when the component hangs under SUPER, else 0
__global__ void __launch_bounds__(256)
ccl_sparse_resolve_kernel(const HystParams p) {
    pdl_wait();
    const unsigned int n = p.ctr[2];
    for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const unsigned int g = p.list[i];
        p.cls[cls_index(p, g)] = (g_find_halve(p.parent, (int)g) == kSuper) ? 255 : 0;
    }
}

// The list length lives on the device, so the grid is sized from the launch's pixel count: one 256-thread block per 16 Ki pixels
// (1.5 % of them weak = one entry per thread), at least 32 blocks, at most every SM full once; the kernels stride over the list, so
// any grid is correct.  A small frame must not pay for 1184 blocks: every block of the link kernel takes a ticket on ONE counter
// (the last one applies the reference's one-way link), and 1184 serialised atomics alone are ~12 us of a 1080p frame's 45.
static int sparse_grid(const b200_ctx* ctx, const HystParams& p) {
    const long long px = (long long)p.n_frames * p.frame_stride;
    const long long cap = 8LL * (ctx->sm_count > 0 ? ctx->sm_count : 148);
    long long b = px / 16384;
    if (b < 32) b = 32;
    if (b > cap) b = cap;
    return (int)b;
}

// <<<grid, 256, 0, st>>> or, for the latency path, the same launch with the programmatic-stream-serialization attribute
static cudaError_t launch_list_kernel(void (*kernel)(const HystParams), int grid, cudaStream_t st, const HystParams& p) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = 0; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = p.pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, p);
}

static int check_hyst_params(const HystParams& p) {
    if (p.cls_pitch < p.width || p.cls_frame_stride < 0) {
        set_error("internal: hysteresis launch without a class-map pitch (%lld for width %d)", p.cls_pitch, p.width);
        return B200_ERR_INVALID_ARG;
    }
    return B200_OK;
}

int launch_ccl_label(b200_ctx* ctx, cudaStream_t st, const HystParams& p_in) {
    HystParams p = p_in;
    CB_TRY(check_hyst_params(p));
    if (p.list) {
        ProfScope ps(ctx, st, 1);
        CB_CUDA(launch_list_kernel(p.opencv ? ccl_sparse_link_kernel<true> : ccl_sparse_link_kernel<false>, sparse_grid(ctx, p), st, p));
        CB_CUDA(cudaGetLastError());
        ctx->launches++;
        return B200_OK;
    }
    if (p.opencv) { set_error("internal: OpenCV hysteresis runs on the weak-pixel list only"); return B200_ERR_INVALID_ARG; }
    if (p.ctr) {
        list_retire_kernel<<<1, 1, 0, st>>>(p.ctr, p.h_kept, p.kept_prev, p.kept_thresh);
        ctx->launches++;
    }
    p.tiles_x = (p.width + kTile - 1) / kTile;
    p.tiles_y = (p.rows + kTile - 1) / kTile;
    {
        dim3 grid(p.tiles_x, p.tiles_y, p.n_frames);
        ProfScope ps(ctx, st, 1);
        ccl_local_kernel<<<grid, kCclThreads, 0, st>>>(p);
        CB_CUDA(cudaGetLastError());
        ctx->launches++;
    }
    const long long items = (long long)(p.tiles_y - 1) * p.width + (long long)(p.tiles_x - 1) * p.rows;
    if (items > 0) {
        int blocks = (int)((items + 255) / 256);
        if (blocks > 4096) blocks = 4096;
        dim3 grid(blocks, p.n_frames);
        {
            ProfScope ps(ctx, st, 2);
            ccl_merge_kernel<<<grid, 256, 0, st>>>(p);
        }
        CB_CUDA(cudaGetLastError());
        ctx->launches++;
    }
    return B200_OK;
}

int launch_ccl_resolve(b200_ctx* ctx, cudaStream_t st, const HystParams& p_in) {
    HystParams p = p_in;
    CB_TRY(check_hyst_params(p));
    if (p.list) {
        ProfScope ps(ctx, st, 3);
        CB_CUDA(launch_list_kernel(ccl_sparse_resolve_kernel, sparse_grid(ctx, p), st, p));
        CB_CUDA(cudaGetLastError());
        ctx->launches++;
        return B200_OK;
    }
    p.tiles_x = (p.width + kTile - 1) / kTile;
    p.tiles_y = (p.rows + kTile - 1) / kTile;
    const long long n16 = ((long long)p.rows * p.width + 15) / 16;
    int blocks = (int)((n16 + 255) / 256);
    const int cap = 8 * (ctx->sm_count > 0 ? ctx->sm_count : 148);
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    dim3 grid(blocks, p.n_frames);
    {
        ProfScope ps(ctx, st, 3);
        ccl_final_kernel<<<grid, 256, 0, st>>>(p);
    }
    CB_CUDA(cudaGetLastError());
    ctx->launches++;
    return B200_OK;
}

int launch_hysteresis(b200_ctx* ctx, cudaStream_t st, const HystParams& p) {
    CB_TRY(launch_ccl_label(ctx, st, p));
    return launch_ccl_resolve(ctx, st, p);
}

// ---------------------------------------------------------------------------------------------
// ragged chunks: the list-driven kernels over frames of different sizes (b200_canny_frames_device)
// ---------------------------------------------------------------------------------------------
// A list entry g is a launch-relative slot; its frame is the last one whose base is <= g (binary search in the dense base table,
// which stays in L1), and the frame gives W, H and the class-byte address.  Same unions, same neighbour rules, per frame.  Ragged
// chunks always take these kernels, never the tile-based ones: the list holds every weak pixel at any density (every pixel at
// worst, which also covers minVal <= 0), so they are correct everywhere, and the uniform path's density state is left alone.
__device__ __forceinline__ int ragged_frame_of(const RaggedHystParams& p, unsigned int g) {
    int lo = 0, hi = p.n_frames - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(p.bases + mid) <= g) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// OPENCV: cv::Canny's plain 8-connectivity (b200_cv_canny_frames_device), as in ccl_sparse_link_kernel: no pair is left out and the
// last block only retires the counters.  It must not run the one-way fix-up anyway: that reads cls[1] and cls[cls_pitch], which a
// 1-wide or 1-tall frame (accepted on that path) does not have.
template <bool OPENCV>
__global__ void __launch_bounds__(256)
ccl_ragged_link_kernel(const RaggedHystParams p) {
    const unsigned int n = p.ctr[0];
    for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const unsigned int g = p.list[i];
        const RaggedFrame fd = p.frames[ragged_frame_of(p, g)];
        const int W = fd.width, Hh = fd.height;
        const unsigned int rel = g - (unsigned int)fd.base;
        const int y = (int)(rel / (unsigned int)W), x = (int)(rel - (unsigned int)y * (unsigned int)W);
        const long long cp = fd.cls_pitch;
        const uint8_t* c = fd.cls + ((long long)y * cp + x);
        const bool has_n = y > 0, has_s = y + 1 < Hh, has_w = x > 0, has_e = x + 1 < W;
        const bool q01 = !OPENCV && (y == 0) && (x == 1);   // (0,1): its SW neighbour (1,0) is off limits
        const bool q10 = !OPENCV && (y == 1) && (x == 0);   // (1,0): its NE neighbour (0,1) is off limits
        const int c_nw = (has_n && has_w) ? c[-cp - 1] : 0;
        const int c_n = has_n ? c[-cp] : 0;
        const int c_ne = (has_n && has_e && !q10) ? c[-cp + 1] : 0;
        const int c_w = has_w ? c[-1] : 0;
        const int c_e = has_e ? c[1] : 0;
        const int c_sw = (has_s && has_w && !q01) ? c[cp - 1] : 0;
        const int c_s = has_s ? c[cp] : 0;
        const int c_se = (has_s && has_e) ? c[cp + 1] : 0;
        if (((c_nw | c_n | c_ne | c_w | c_e | c_sw | c_s | c_se) & 0x80) != 0) g_union_halve(p.parent, (int)g, kSuper);
        if (c_e == 1) g_union_halve(p.parent, (int)g, (int)g + 1);
        if (c_s == 1) {
            g_union_halve(p.parent, (int)g, (int)g + W);
        } else {
            if (c_sw == 1) g_union_halve(p.parent, (int)g, (int)g + W - 1);
            if (c_se == 1) g_union_halve(p.parent, (int)g, (int)g + W + 1);
        }
    }
    // the last block applies the reference's one-way link (0,1) -> (1,0) of every frame (see ccl_sparse_link_kernel)
    __shared__ bool s_last;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = atomicAdd(p.ctr + 1, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    for (int f = threadIdx.x; !OPENCV && f < p.n_frames; f += blockDim.x) {
        const RaggedFrame fd = p.frames[f];
        const int c01 = fd.cls[1], c10 = fd.cls[fd.cls_pitch];
        if (c10 == 1 && (c01 == 255 || (c01 == 1 && g_find_halve(p.parent, fd.base + 1) == kSuper)))
            g_union_halve(p.parent, fd.base + fd.width, kSuper);
    }
    if (threadIdx.x == 0) {
        p.ctr[2] = n;
        p.ctr[0] = 0;
        p.ctr[1] = 0;
    }
}

__global__ void __launch_bounds__(256)
ccl_ragged_resolve_kernel(const RaggedHystParams p) {
    const unsigned int n = p.ctr[2];
    for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const unsigned int g = p.list[i];
        const RaggedFrame fd = p.frames[ragged_frame_of(p, g)];
        const unsigned int rel = g - (unsigned int)fd.base;
        const unsigned int y = rel / (unsigned int)fd.width, x = rel - y * (unsigned int)fd.width;
        fd.cls[(long long)y * fd.cls_pitch + x] = (g_find_halve(p.parent, (int)g) == kSuper) ? 255 : 0;
    }
}

int launch_hysteresis_ragged(b200_ctx* ctx, cudaStream_t st, const RaggedHystParams& p) {
    const long long cap = 8LL * (ctx->sm_count > 0 ? ctx->sm_count : 148);
    const int grid = (int)std::min(cap, std::max(32LL, p.px / 16384));   // as sparse_grid()
    {
        ProfScope ps(ctx, st, 1);
        (p.opencv ? ccl_ragged_link_kernel<true> : ccl_ragged_link_kernel<false>)<<<grid, 256, 0, st>>>(p);
    }
    CB_CUDA(cudaGetLastError());
    ctx->launches++;
    {
        ProfScope ps(ctx, st, 3);
        ccl_ragged_resolve_kernel<<<grid, 256, 0, st>>>(p);
    }
    CB_CUDA(cudaGetLastError());
    ctx->launches++;
    return B200_OK;
}

// ---------------------------------------------------------------------------------------------
// stage-API helpers: int16 nms plane -> class map, class map -> int16 0/255
// ---------------------------------------------------------------------------------------------
__global__ void classify_i16_kernel(const int16_t* __restrict__ nms, uint8_t* __restrict__ cls, size_t n, int lo, int hi) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int v = nms[i];
        // src/utils.cpp:328-333: below minVal -> dropped; otherwise >= maxVal seeds a flood
        cls[i] = (v < lo) ? 0 : ((v >= hi) ? 255 : 1);
    }
}
__global__ void expand_u8_i16_kernel(const uint8_t* __restrict__ cls, int16_t* __restrict__ out, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        out[i] = cls[i];
}

// 0 / 255 bytes -> 1 bit per pixel (bit i of byte k <-> pixel 8k + i): what b200_canny_batch_host sends over PCIe instead of
// the byte map.  One thread per 32 pixels (two 128-bit loads, one 32-bit store).
__global__ void pack_edges_kernel(const uint8_t* __restrict__ cls, uint32_t* __restrict__ bits, size_t n_px) {
    const size_t n_words = (n_px + 31) / 32;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_words; i += (size_t)gridDim.x * blockDim.x) {
        uint32_t out = 0;
        if (32 * i + 32 <= n_px && ((reinterpret_cast<uintptr_t>(cls) & 15) == 0)) {
            const uint4 a = __ldcs(reinterpret_cast<const uint4*>(cls + 32 * i));
            const uint4 b = __ldcs(reinterpret_cast<const uint4*>(cls + 32 * i) + 1);
            const uint32_t wv[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const uint32_t m = wv[k] & 0x01010101u;                 // bit 0 of each of the four bytes
                const uint32_t nib = (m | (m >> 7) | (m >> 14) | (m >> 21)) & 0xFu;
                out |= nib << (4 * k);
            }
        } else {
            for (int k = 0; k < 32 && 32 * i + k < n_px; ++k) out |= (uint32_t)(cls[32 * i + k] & 1u) << k;
        }
        bits[i] = out;
    }
}

int launch_pack_edges(b200_ctx* ctx, cudaStream_t st, const uint8_t* cls, uint32_t* bits, size_t n_px) {
    const size_t n_words = (n_px + 31) / 32;
    size_t b = (n_words + 255) / 256;
    const size_t cap = 16 * (size_t)(ctx->sm_count > 0 ? ctx->sm_count : 148);
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    pack_edges_kernel<<<(int)b, 256, 0, st>>>(cls, bits, n_px);
    CB_CUDA(cudaGetLastError());
    ctx->launches++;
    return B200_OK;
}

static int grid_for(size_t n, const b200_ctx* ctx) {
    size_t b = (n + 255) / 256;
    size_t cap = 16 * (size_t)(ctx->sm_count > 0 ? ctx->sm_count : 148);
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (int)b;
}

int launch_classify_i16(b200_ctx* ctx, cudaStream_t st, const int16_t* nms, uint8_t* cls, size_t n, int lo, int hi) {
    classify_i16_kernel<<<grid_for(n, ctx), 256, 0, st>>>(nms, cls, n, lo, hi);
    CB_CUDA(cudaGetLastError());
    ctx->launches++;
    return B200_OK;
}
int launch_expand_u8_to_i16(b200_ctx* ctx, cudaStream_t st, const uint8_t* cls, int16_t* out, size_t n) {
    expand_u8_i16_kernel<<<grid_for(n, ctx), 256, 0, st>>>(cls, out, n);
    CB_CUDA(cudaGetLastError());
    ctx->launches++;
    return B200_OK;
}

}  // namespace cb
