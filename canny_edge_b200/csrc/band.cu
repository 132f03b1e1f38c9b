// band.cu — row-band sharding of ONE image across GPUs (BASELINE config 5: 32768^2 over 8 B200).
//
// The reference has nothing like this (one 640x480 frame, one GPU, src/main.cpp:111).  A band owns
// global rows [row0, row0+band_rows).  Stages 1-3 are local once the band holds window/2+2 halo rows
// from its neighbours (exchanged by the caller over NVLink: NCCL send/recv or peer copies); every
// border rule keys off GLOBAL row numbers, so front.cu runs unchanged.  Stage 4 needs one exchange:
//
//   1. each band labels its own candidates (ccl_local + ccl_merge, hysteresis.cu);
//   2. band_export: for every pixel of the band's first and last row (+ the two pixels of the
//      reference's missing-link quirk in band 0) it publishes a RECORD {label, flags}.  `label` is a
//      canonical record index: all boundary pixels of one band-local component carry the same label,
//      so other ranks can tell "same component" without seeing this band's parent array;
//   3. the caller all-gathers the records (NCCL);
//   4. band_finalize: every rank builds the same small forest over ALL bands' records, joins records
//      that touch across a band boundary (8-connectivity: columns x-1, x, x+1), hangs classes that
//      contain a seed under SUPER, then marks its own components whose class became strong and
//      resolves its weak pixels.  One step, no iteration: strength is the OR over the merged class.
#include <string.h>

#include "ccl.cuh"
#include "internal.h"

namespace cb {

constexpr int kRecCand = 2, kRecStrong = 1;

// records per band: first row (W), last row (W), global pixel (0,1), global pixel (1,0)
__host__ __device__ inline int band_records(int width) { return 2 * width + 2; }

// band-relative pixel index of record i, or -1 when the record does not exist in this band
__device__ __forceinline__ int record_pixel(int i, int rows, int W, int row0) {
    if (i < W) return i;
    if (i < 2 * W) return (rows - 1) * W + (i - W);
    if (row0 != 0 || rows < 2 || W < 2) return -1;
    return (i == 2 * W) ? 1 : W;  // (0,1) and (1,0)
}

// pass 1: root of every record's pixel (kNone = not a candidate / absent)
__global__ void band_roots_kernel(const uint8_t* __restrict__ cls, const int32_t* __restrict__ parent, int rows, int W,
                                  int row0, int32_t* __restrict__ roots) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= band_records(W)) return;
    const int px = record_pixel(i, rows, W, row0);
    int r = kNone;
    if (px >= 0) {
        const int c = cls[px];
        if (c == 255) r = kSuper;                 // strong pixels are final (the list-driven path gives them no union-find slot)
        else if (c != 0) r = g_find(parent, px);
    }
    roots[i] = r;
}
// pass 2: every non-strong root is claimed by ONE of the records that reach it (the largest index wins)
__global__ void band_claim_kernel(int32_t* __restrict__ parent, int W, const int32_t* __restrict__ roots) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= band_records(W)) return;
    const int r = roots[i];
    if (r >= 0) atomicMin(parent + r, -2 - i);
}
// pass 3: publish
__global__ void band_export_kernel(const int32_t* __restrict__ parent, int W, const int32_t* __restrict__ roots,
                                   b200_band_record* __restrict__ rec) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= band_records(W)) return;
    const int r = roots[i];
    b200_band_record out;
    if (r == kNone) { out.label = -1; out.flags = 0; }
    else if (r == kSuper) { out.label = -1; out.flags = kRecCand | kRecStrong; }
    else { out.label = -2 - parent[r]; out.flags = kRecCand; }
    rec[i] = out;
}

// node of record i of band b in the cross-band forest: SUPER for strong, else b*S + label; kNone if absent
__device__ __forceinline__ int rec_node(const b200_band_record* all, int S, int b, int i) {
    const b200_band_record r = all[(long long)b * S + i];
    if (!(r.flags & kRecCand)) return kNone;
    if (r.flags & kRecStrong) return kSuper;
    return b * S + r.label;
}

__global__ void band_uf_init_kernel(int32_t* __restrict__ uf, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) uf[i] = i;
}
// one thread per (boundary, column): last row of band b against first row of band b+1
__global__ void band_uf_union_kernel(int32_t* __restrict__ uf, const b200_band_record* __restrict__ all, int n_bands, int W) {
    const int S = band_records(W);
    const long long it = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (it >= (long long)(n_bands - 1) * W) return;
    const int b = (int)(it / W), x = (int)(it - (long long)b * W);
    const int u = rec_node(all, S, b, W + x);
    if (u == kNone) return;
    const int v_mid = rec_node(all, S, b + 1, x);
    if (v_mid != kNone) {
        g_union(uf, u, v_mid);  // x-1 and x+1 of the lower row are in v_mid's run
    } else {
        if (x > 0) { const int v = rec_node(all, S, b + 1, x - 1); if (v != kNone) g_union(uf, u, v); }
        if (x < W - 1) { const int v = rec_node(all, S, b + 1, x + 1); if (v != kNone) g_union(uf, u, v); }
    }
}
// the reference's one-way link (0,1) -> (1,0) (src/utils.cpp:399) at image scope: if (0,1)'s class is
// strong, (1,0)'s whole class (which may continue into other bands) becomes strong.
__global__ void band_uf_quirk_kernel(int32_t* __restrict__ uf, const b200_band_record* __restrict__ all, int W) {
    const int S = band_records(W);
    const int a = rec_node(all, S, 0, 2 * W), b = rec_node(all, S, 0, 2 * W + 1);
    if (a == kNone || b == kNone) return;
    if (g_find(uf, a) == kSuper) g_union(uf, b, kSuper);
}
// every local component whose class hangs under SUPER becomes strong in the band's own forest
__global__ void band_mark_kernel(const int32_t* __restrict__ uf, const b200_band_record* __restrict__ all, int band, int W,
                                 const int32_t* __restrict__ roots, int32_t* __restrict__ parent) {
    const int S = band_records(W);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= S) return;
    const int r = roots[i];
    if (r < 0) return;  // absent, not a candidate, or already strong
    const int node = rec_node(all, S, band, i);
    if (node >= 0 && g_find(uf, node) == kSuper) parent[r] = kSuper;
}


// ---- the band's local stages, in pieces (b200_band_front chains them; bands_mgpu.cu interleaves them with the halo exchange) ----
int band_prepare(b200_ctx* ctx, const BandGeom& g, float sigma) {
    if (!g.d_rows || !g.d_edges) { set_error("null pointer"); return B200_ERR_INVALID_ARG; }
    if (g.rows < 2 || g.width < 2 || g.height < 2 || g.row0 < 0 || g.row0 + g.rows > g.height || g.above < 0 || g.below < 0 ||
        g.above > g.row0 || g.row0 + g.rows + g.below > g.height) {
        set_error("inconsistent band geometry (row0=%d rows=%d halos=%d/%d height=%d)", g.row0, g.rows, g.above, g.below, g.height);
        return B200_ERR_INVALID_ARG;
    }
    if ((long long)g.rows * g.width >= (1LL << 31)) { set_error("band exceeds int indexing"); return B200_ERR_UNSUPPORTED; }
    if (!ctx) { set_error("band calls need an explicit context (they keep per-band state)"); return B200_ERR_INVALID_ARG; }
    if (!thresholds_supported(g.lo, g.hi)) { set_error("thresholds minVal=%d > 255 >= maxVal=%d are not reproduced (src/utils.cpp:327-340)", g.lo, g.hi); return B200_ERR_UNSUPPORTED; }
    CB_CUDA(cudaSetDevice(ctx->device));
    CB_TRY(prepare_gauss(ctx, sigma));
    const int need = ctx->gauss.radius + 2;
    const int need_above = need < g.row0 ? need : g.row0;
    const int rows_after = g.height - (g.row0 + g.rows);
    const int need_below = need < rows_after ? need : rows_after;
    if (g.above < need_above || g.below < need_below) {
        set_error("band needs %d/%d halo rows above/below (got %d/%d)", need_above, need_below, g.above, g.below);
        return B200_ERR_INVALID_ARG;
    }
    const long long px = (long long)g.rows * g.width;
    CB_TRY(ensure_ws(ctx->ws_band_parent, (size_t)px * 4));
    CB_TRY(ensure_ws(ctx->ws_band_list, 64 + (size_t)px * 4));
    // the list's counter block is zero here: zeroed at allocation and retired by the previous band's kernels (HystParams::ctr);
    // only a band that failed between its front launches and its labelling leaves it dirty
    if (ctx->list_dirty[3]) CB_CUDA(cudaMemsetAsync(ctx->ws_band_list.ptr, 0, 64, ctx->stream));
    ctx->list_dirty[3] = false;
    return B200_OK;
}

// stages 1-3 for the band's rows [sub_row0, sub_row0 + sub_rows) (global numbers); several calls may cover one band: they append
// to the same weak-pixel list, which band_label() then consumes
int band_front_rows(b200_ctx* ctx, cudaStream_t st, const BandGeom& g, int sub_row0, int sub_rows) {
    if (sub_rows <= 0) return B200_OK;
    const long long px = (long long)g.rows * g.width;
    FrontParams fp;
    memset(&fp, 0, sizeof(fp));
    fp.in = g.d_rows;
    fp.in_pitch = g.width;
    fp.in_frame_stride = (long long)(g.above + g.rows + g.below) * g.width;
    fp.in_row0 = g.row0 - g.above;
    fp.in_rows = g.above + g.rows + g.below;
    fp.width = g.width; fp.height = g.height;
    fp.out_row0 = sub_row0; fp.out_rows = sub_rows; fp.plane_row0 = g.row0; fp.n_frames = 1;
    fp.cls = g.d_edges; fp.cls_pitch = g.width; fp.cls_frame_stride = px; fp.out_frame_stride = px;
    fp.w = ctx->gauss.d_w; fp.count = ctx->gauss.d_count; fp.radius = ctx->gauss.radius;
    fill_thresholds(fp, g.lo, g.hi);
    fp.parent = reinterpret_cast<int32_t*>(ctx->ws_band_parent.ptr);
    fp.kept_count = reinterpret_cast<unsigned int*>(ctx->ws_band_list.ptr);
    fp.kept_list = reinterpret_cast<uint32_t*>(ctx->ws_band_list.ptr) + 16;
    ctx->list_dirty[3] = true;   // until band_label() has consumed the list
    bool sparse = false;
    CB_TRY(launch_front(ctx, st, fp, &sparse));
    ctx->band_front_sparse = sparse;
    return B200_OK;
}

// band-local connected components over the weak pixels the front launches listed (or the whole plane)
int band_label(b200_ctx* ctx, cudaStream_t st, const BandGeom& g) {
    const long long px = (long long)g.rows * g.width;
    const unsigned int prev_kept = *reinterpret_cast<volatile unsigned int*>(&ctx->h_kept[3]);   // previous band on this context
    const bool dense = ctx->kept_px[3] > 0 && (long long)prev_kept * 8 > ctx->kept_px[3];
    const bool front_sparse = ctx->band_front_sparse;
    if (front_sparse) ctx->kept_px[3] = px;
    const bool sparse = front_sparse && !dense;
    ctx->band_sparse = sparse;
    HystParams hp;
    memset(&hp, 0, sizeof(hp));
    unsigned int* ctr = reinterpret_cast<unsigned int*>(ctx->ws_band_list.ptr);
    hp.list = sparse ? reinterpret_cast<const uint32_t*>(ctr + 16) : nullptr;
    hp.ctr = front_sparse ? ctr : nullptr;
    hp.h_kept = ctx->d_kept + 3;
    hp.kept_prev = prev_kept;
    hp.kept_thresh = (unsigned int)(px / 8);
    hp.cls = g.d_edges; hp.cls_pitch = g.width; hp.cls_frame_stride = px; hp.parent = reinterpret_cast<int32_t*>(ctx->ws_band_parent.ptr);
    hp.frame_stride = px; hp.rows = g.rows; hp.width = g.width; hp.row0 = g.row0; hp.n_frames = 1;
    CB_TRY(launch_ccl_label(ctx, st, hp));
    ctx->list_dirty[3] = false;
    ctx->band_rows = g.rows; ctx->band_width = g.width; ctx->band_row0 = g.row0; ctx->band_cls = g.d_edges;
    return B200_OK;
}

}  // namespace cb

using namespace cb;

extern "C" {

int b200_band_halo_rows(float sigma) { return host_window(sigma) / 2 + 2; }
int b200_band_record_count(int width) { return band_records(width); }

int b200_band_front(b200_ctx* ctx, const uint8_t* d_rows, int halo_above, int halo_below, int band_rows, int row0,
                    int global_height, int width, float sigma, int lo, int hi, uint8_t* d_edges) {
    BandGeom g{d_rows, halo_above, halo_below, band_rows, row0, global_height, width, lo, hi, d_edges};
    CB_TRY(band_prepare(ctx, g, sigma));
    CB_TRY(band_front_rows(ctx, ctx->stream, g, row0, band_rows));
    return band_label(ctx, ctx->stream, g);
}

int b200_band_boundary_export(b200_ctx* ctx, int band_rows, int width, b200_band_record* d_records) {
    if (!ctx || !d_records) { set_error("null pointer"); return B200_ERR_INVALID_ARG; }
    if (ctx->band_rows != band_rows || ctx->band_width != width || !ctx->band_cls) {
        set_error("b200_band_boundary_export: no matching b200_band_front on this context");
        return B200_ERR_INVALID_ARG;
    }
    CB_CUDA(cudaSetDevice(ctx->device));
    const int S = band_records(width);
    CB_TRY(ensure_ws(ctx->ws_band_aux, (size_t)S * 4));
    int32_t* roots = reinterpret_cast<int32_t*>(ctx->ws_band_aux.ptr);
    int32_t* parent = reinterpret_cast<int32_t*>(ctx->ws_band_parent.ptr);
    cudaStream_t st = ctx->stream;
    const int blocks = (S + 255) / 256;
    band_roots_kernel<<<blocks, 256, 0, st>>>(ctx->band_cls, parent, band_rows, width, ctx->band_row0, roots);
    band_claim_kernel<<<blocks, 256, 0, st>>>(parent, width, roots);
    band_export_kernel<<<blocks, 256, 0, st>>>(parent, width, roots, d_records);
    CB_CUDA(cudaGetLastError());
    ctx->launches += 3;
    return B200_OK;
}

int b200_band_finalize(b200_ctx* ctx, const b200_band_record* d_all, int n_bands, int band_index, int band_rows, int width,
                       uint8_t* d_edges) {
    if (!ctx || !d_all || !d_edges) { set_error("null pointer"); return B200_ERR_INVALID_ARG; }
    if (n_bands < 1 || band_index < 0 || band_index >= n_bands) { set_error("bad band index %d of %d", band_index, n_bands); return B200_ERR_INVALID_ARG; }
    if (ctx->band_rows != band_rows || ctx->band_width != width || ctx->band_cls != d_edges) {
        set_error("b200_band_finalize: no matching b200_band_front on this context");
        return B200_ERR_INVALID_ARG;
    }
    CB_CUDA(cudaSetDevice(ctx->device));
    const int S = band_records(width);
    const long long n_nodes = (long long)n_bands * S;
    if (n_nodes >= (1LL << 31)) { set_error("too many boundary records"); return B200_ERR_UNSUPPORTED; }
    // aux layout: [roots: S ints (from export)] [uf: n_nodes ints]
    {
        // grow without losing the roots written by b200_band_boundary_export
        const size_t need = (size_t)(S + n_nodes) * 4;
        if (ctx->ws_band_aux.bytes < need) {
            Workspace bigger;
            CB_TRY(ensure_ws(bigger, need));
            CB_CUDA(cudaMemcpyAsync(bigger.ptr, ctx->ws_band_aux.ptr, (size_t)S * 4, cudaMemcpyDeviceToDevice, ctx->stream));
            CB_CUDA(cudaStreamSynchronize(ctx->stream));
            cudaFree(ctx->ws_band_aux.ptr);
            ctx->ws_band_aux = bigger;
        }
    }
    int32_t* roots = reinterpret_cast<int32_t*>(ctx->ws_band_aux.ptr);
    int32_t* uf = roots + S;
    int32_t* parent = reinterpret_cast<int32_t*>(ctx->ws_band_parent.ptr);
    cudaStream_t st = ctx->stream;
    band_uf_init_kernel<<<(int)((n_nodes + 255) / 256), 256, 0, st>>>(uf, (int)n_nodes);
    ctx->launches++;
    if (n_bands > 1) {
        const long long items = (long long)(n_bands - 1) * width;
        band_uf_union_kernel<<<(int)((items + 255) / 256), 256, 0, st>>>(uf, d_all, n_bands, width);
        ctx->launches++;
    }
    band_uf_quirk_kernel<<<1, 1, 0, st>>>(uf, d_all, width);
    band_mark_kernel<<<(S + 255) / 256, 256, 0, st>>>(uf, d_all, band_index, width, roots, parent);
    ctx->launches += 2;
    CB_CUDA(cudaGetLastError());
    HystParams hp;
    memset(&hp, 0, sizeof(hp));
    hp.cls = d_edges; hp.cls_pitch = width; hp.cls_frame_stride = (long long)band_rows * width; hp.parent = parent;
    hp.list = ctx->band_sparse ? reinterpret_cast<const uint32_t*>(ctx->ws_band_list.ptr) + 16 : nullptr;
    hp.ctr = reinterpret_cast<unsigned int*>(ctx->ws_band_list.ptr);   // the resolve kernel reads the retired count, ctr[2]
    hp.frame_stride = (long long)band_rows * width; hp.rows = band_rows; hp.width = width; hp.row0 = ctx->band_row0; hp.n_frames = 1;
    CB_TRY(launch_ccl_resolve(ctx, st, hp));
    return B200_OK;
}

}  // extern "C"
