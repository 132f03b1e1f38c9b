// internal.h — declarations shared between the translation units of libcanny_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

struct CUtensorMap_st;

#include <string>
#include <vector>

#include "../../include/canny_b200.h"

namespace cb {

// ---- error plumbing -------------------------------------------------------------------------
void set_error(const char* fmt, ...);
#define CB_CUDA(expr)                                                                      \
    do {                                                                                   \
        cudaError_t e_ = (expr);                                                           \
        if (e_ != cudaSuccess) {                                                           \
            cb::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, \
                          __LINE__);                                                       \
            return B200_ERR_CUDA;                                                          \
        }                                                                                  \
    } while (0)
#define CB_TRY(expr)                   \
    do {                               \
        int s_ = (expr);               \
        if (s_ != B200_OK) return s_;  \
    } while (0)

// ---- Gaussian tables (host generated, bit-identical to the reference's float arithmetic) ------
struct GaussTables {
    float sigma = -1.f;
    int window = 0, radius = 0;
    std::vector<float> w;      // window weights, src/utils.cpp:77-95
    std::vector<float> count;  // (radius+1)^2: count[a*(radius+1)+b] = sum of weights with the first a
                               // and last b taps skipped, accumulated in ascending tap order
                               // exactly as src/utils.cpp:44,59 do
    float* d_w = nullptr;      // device copies (owned by the context)
    float* d_count = nullptr;
    bool tiny = false;         // min weight^2 < 2^-90: blur sums may approach the subnormal range
    int div_mode = 5;          // cheapest exact form of RN(a / count_full), checked for EVERY float mantissa on the device when
                               // the tables are built: 1 = fma(a, c, a) with c = RN(1/count - 1); 3 / 5 = one / two Markstein
                               // corrections of a * RN(1/count)
    float div_c = 0.f;         // c of the one-instruction form
};

// ---- parameters of the fused front kernel -----------------------------------------------------
// The kernel works in GLOBAL image coordinates so the same code serves whole frames and row bands.
struct FrontParams {
    const uint8_t* in;      // first byte of buffer row 0 of frame 0
    long long in_frame_stride;  // bytes between frames in `in`
    long long in_pitch;     // bytes between rows of `in` (>= width, >= 3*width for BGR)
    int in_bgr;             // 1: `in` holds interleaved B,G,R bytes (3 per pixel, in_pitch >= 3*width bytes per row):
                            // front3's fused-conversion variant (front3_bgr_supports); 0: one gray byte per pixel
    int in_row0;            // global row index of buffer row 0 (0 for whole frames; row0-halo for bands)
    int in_rows;            // rows present in the buffer
    int width;              // image width == pitch of every internal plane (parent, list indices, spill planes)
    int height;             // GLOBAL image height (border rules key off this)
    int out_row0;           // first global row this launch produces
    int out_rows;           // number of rows produced
    int plane_row0;         // global row of row 0 of every OUTPUT plane below (cls, parent, spill planes).  == out_row0 unless a launch
                            // produces only part of the plane's rows (row bands: interior rows first, the rows that need the
                            // neighbours' halo once it has arrived; bands_mgpu.cu)
    int n_frames;
    uint8_t* cls;           // out: class map (0 / 1 weak / 255 strong) in the caller's layout: pixel (f, y, x) at
                            // f*cls_frame_stride + (y - plane_row0)*cls_pitch + x; no other byte of it is written
    long long cls_pitch;         // bytes between rows of cls
    long long cls_frame_stride;  // bytes between frames of cls
    int cls_words;               // 1: base, pitch and frame stride of cls are multiples of 4, so four pixels at a column that is a
                                 // multiple of 4 are one aligned 32-bit store (set by launch_front from the three; else byte stores)
    long long out_frame_stride;  // elements between frames in the dense internal planes (parent, list indices, spill planes)
    int16_t* blur;          // optional spill planes (steps / stage API); may be null
    int16_t* mag;
    int16_t* ang;
    int16_t* nms;
    const float* w;         // device weights [2*radius+1]
    const float* count;     // device count table [(radius+1)^2]
    int radius;
    int lo2, hi2;           // thresholds in squared-magnitude space (see front.cu)
    int lo, hi;             // raw thresholds (spill / zero-class decisions)
    int cls_zero;           // class of a suppressed pixel (value 0): nonzero only when lo <= 0
    float div_c;            // front3: c of the one-instruction interior division (GaussTables::div_c)
    int ieee_div;           // 1: weights so small that sums can fall below 2^-100 -> use IEEE division instead of div_exact
    int tiles_x, tiles_y;
    // sparse hand-over to the hysteresis kernels (front3.cu and front_cv.cu only; both null -> not produced):
    int32_t* parent;        // union-find slots, dense: every WEAK pixel is initialised to its own launch-relative index
                            // frame*out_frame_stride + (y - plane_row0)*width + x (strong pixels need no slot: they are final)
    uint32_t* kept_list;    // launch-relative indices of all weak pixels, in no particular order
    unsigned int* kept_count;  // number of entries: word 0 of the list's counter block (see HystParams::ctr); zero at launch
    // ragged launches (front3's RAGGED variant, b200_canny_frames_device; front_cv's, b200_cv_canny_frames_device): the chunk's device
    // table.  Work item blockIdx.x names a frame, a strip and a row band (front_cv: one 128 x 64 tile); the frame's descriptor replaces
    // in / in_pitch / width / height / cls / cls_pitch / cls_words and the slot base, and for front3 its tensor map (TMA staging)
    // replaces the `tmap` parameter.
    const struct RaggedFrame* rframes;
    const struct RaggedItem* ritems;
    const CUtensorMap_st* rtmaps;
};

// ---- ragged chunks: frames of different sizes in one launch --------------------------------------
// One frame of a chunk as the kernels see it.  Frames are whole images (row 0 is the image's row 0).  Union-find slots and list
// indices stay dense and launch-relative: pixel (y, x) of the frame is slot base + y*width + x, base being the sum of h*w over
// the frames before it in the chunk (ascending, below 2^31).
struct RaggedFrame {
    const uint8_t* in;      // gray input (a scratch plane for B,G,R lists); for OpenCV-compatible lists (b200_cv_canny_frames_device)
                            // the caller's frame itself, 1 or 3 interleaved bytes per pixel
    long long in_pitch;
    uint8_t* cls;           // the caller's output: class map, then 0 / 255
    long long cls_pitch;
    int height, width;
    int base;
    int cls_words;          // cls and cls_pitch are multiples of 4 (aligned 32-bit class stores)
};
struct RaggedItem { int frame, x0, yb, ye; };   // one front CTA: strip at column x0, class rows [yb, ye) of the frame
// B,G,R -> gray of one frame of a ragged chunk: rows [row0, row0 + height) of the chunk's row space
struct RaggedGrayJob {
    const uint8_t* bgr;
    long long bgr_pitch;
    uint8_t* gray;
    long long gray_pitch;
    int row0, width;
};
struct RaggedHystParams {
    const RaggedFrame* frames;
    const uint32_t* bases;  // frames[i].base, a dense copy for the per-entry binary search (stays in L1)
    int n_frames;
    int32_t* parent;
    const uint32_t* list;
    unsigned int* ctr;      // the list's counter block (HystParams::ctr); h_kept is never written by ragged launches
    long long px;           // pixels of the chunk (sizes the grid)
    int opencv;             // 1: cv::Canny's plain 8-connectivity, without the reference's one-way (0,1)/(1,0) link (as HystParams::opencv;
                            // b200_cv_canny_frames_device)
};

// The input layout a TMA tensor map can describe: base, row pitch and frame stride on 16-byte boundaries, frames that do not
// overlap (a single frame's stride is never used).  Other layouts take the kernels' byte-load staging.
inline bool input_tma_layout_ok(const FrontParams& p) {
    return ((reinterpret_cast<uintptr_t>(p.in) & 15) == 0) && (p.in_pitch % 16 == 0) && (p.in_frame_stride % 16 == 0) &&
           (p.n_frames <= 1 || p.in_frame_stride >= (long long)p.in_rows * p.in_pitch);
}
inline long long input_tma_frame_stride(const FrontParams& p) {
    return p.n_frames <= 1 ? (long long)p.in_rows * p.in_pitch : p.in_frame_stride;
}

// ---- thresholds ---------------------------------------------------------------------------------
// The reference accepts any int pair (only its CLI checks 0 <= minVal < maxVal <= 255, src/main.cpp:63-76).  What
// src/utils.cpp:322-342 then does:
//   * maxVal > 255: every flooded pixel is written as EDGE = 255 (src/utils.cpp:368) and the second scan zeroes everything below
//     maxVal (:336-340) -> the map is ALL ZERO.  Reproduced: no pixel is ever strong (hi2 = INT_MAX), so every weak pixel
//     resolves to 0.
//   * minVal > 255 >= maxVal: the first scan re-zeroes flooded pixels it has not passed yet (255 < minVal, :328-329), so the
//     result depends on the raster order of the flood starts.  Not reproduced: B200_ERR_UNSUPPORTED.
//   * everything else (including minVal >= maxVal and negative values) follows from the two comparisons and is reproduced.
inline bool thresholds_supported(int lo, int hi) { return !(lo > 255 && hi <= 255); }
// maxVal as the classification kernels must see it: above every representable magnitude when the reference's map is all zero
inline int effective_hi(int hi) { return hi > 255 ? 0x7fffffff : hi; }
inline void fill_thresholds(FrontParams& p, int lo, int hi) {
    // class of a kept pixel with squared magnitude n: candidate iff mag >= lo  <=>  n >= lo^2 (lo > 0), always if lo <= 0
    const long long kBig = 0x7fffffff;
    auto sq = [&](int v) -> int { if (v <= 0) return 0; long long s = (long long)v * v; return (int)(s < kBig ? s : kBig); };
    p.lo = lo; p.hi = hi;
    p.lo2 = sq(lo);
    p.hi2 = hi > 255 ? (int)kBig : sq(hi);   // magnitudes stay below 1443, n below 2^22: INT_MAX is never reached
    p.cls_zero = (0 >= lo) ? ((0 >= hi) ? 255 : 1) : 0;  // what a suppressed pixel (value 0) is: src/utils.cpp:328-333
}

// ---- parameters of the hysteresis (connected components) kernels ---------------------------------
struct HystParams {
    uint8_t* cls;          // in/out: 0 / 1 / 255 -> 0 / 255; pixel (f, y, x) at f*cls_frame_stride + y*cls_pitch + x
    long long cls_pitch, cls_frame_stride;   // bytes between rows / frames of cls
    int32_t* parent;       // workspace: union-find parent per pixel (only candidate entries are defined), dense
    long long frame_stride;  // elements between frames of parent (and of the list's pixel indices: f*frame_stride + y*width + x)
    int rows, width;       // rows in this launch's plane (whole frame or band)
    int row0;              // global row of plane row 0 (the missing-link quirk lives at global (1,0)->(0,1))
    int n_frames;
    int tiles_x, tiles_y;
    const uint32_t* list;        // weak-pixel list written by the front kernel (null -> tile-based labelling over the whole plane);
                                 // the list-driven kernels keep LAUNCH-relative indices (frame*frame_stride + pixel) in parent[]
    // Counter block of the list (null when the front kernel did not produce one).  It is zeroed ONCE, when the workspace is
    // allocated, and then kept consistent by the kernels themselves, so a launch needs neither a memset before the front kernel
    // nor a copy after it:
    //   ctr[0]  live entry count (the front kernel's atomicAdd)   ctr[1]  link-kernel blocks that have finished
    //   ctr[2]  entry count of the finished launch: written, with h_kept, by the last block of the link kernel (or by
    //           list_retire_kernel on the tile-based path), which also zeroes ctr[0] and ctr[1] for the next launch
    unsigned int* ctr;
    unsigned int* h_kept;        // mapped pinned host word that receives the entry count (density of the next launch's choice) ...
    int pdl;                     // list-driven kernels only: launch them with programmatic stream serialization (they are resident and
                                 // parked on griddepcontrol.wait while their predecessor drains) — the single-frame latency path
    unsigned int kept_prev, kept_thresh;   // ... but only when it moves across the threshold: the host's last view of it and the
                                           // "tile-based labelling above this many weak pixels" bound (a write to host memory at the
                                           // end of every launch measured 1 % of the batch throughput)
    int opencv;                  // 1: cv::Canny's plain 8-connectivity, without the reference's one-way (0,1)/(1,0) link (list-driven
                                 // kernels only; b200_cv_canny_device_strided)
};

struct HostPool;  // api.cu

// ---- the context ------------------------------------------------------------------------------
struct Workspace {
    void* ptr = nullptr;
    size_t bytes = 0;
};

}  // namespace cb

namespace cb {
// Optional per-kernel timing (b200_profile_stages_device): every launch site brackets its kernel with two
// events on the launching stream; categories: 0 front, 1 ccl_local, 2 ccl_merge, 3 ccl_final, 4 other.
struct ProfRecord { int cat; cudaEvent_t a, b; };
struct Profiler {
    bool on = false;
    std::vector<ProfRecord> recs;
};
}  // namespace cb

struct b200_ctx {
    int device = -1;
    int sm_count = 0;
    cudaStream_t own_stream = nullptr;   // private stream
    cudaStream_t stream = nullptr;       // stream work is issued on (own_stream or the user's)
    cudaStream_t side[3] = {nullptr, nullptr, nullptr};  // chunk pipelining / copy overlap
    cudaEvent_t ev_fork = nullptr, ev_join[3] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_switch = nullptr;     // b200_ctx_set_stream: the new stream waits for what was issued on the old one
    cb::GaussTables gauss;
    cb::Workspace ws_parent[3];   // int32 union-find slots for one chunk, per pipeline slot
    cb::Workspace ws_list[3];     // kept-pixel lists for one chunk ([0..15] = counter block, entries from word 16), per pipeline slot
    cb::Workspace ws_band_list;   // kept-pixel list of the resident band
    cb::Workspace ws_planes;      // stage-API scratch planes
    cb::Workspace ws_misc;
    cb::Workspace dev_in[3], dev_out[3];  // device staging for the batch_host pipeline
    cb::Workspace dev_bits[3], host_bits[3];  // bit-packed edge maps of a chunk: device side and pinned host side
    cudaEvent_t ev_chunk[3] = {nullptr, nullptr, nullptr};  // "chunk's packed map has arrived in host_bits[slot]"
    cb::HostPool* pool = nullptr;         // host threads that expand the packed maps into the caller's buffer and stage pageable memory
    cb::Workspace host_in[3];             // pinned staging for PAGEABLE caller frames, per pipeline slot
    cudaEvent_t ev_in[3] = {nullptr, nullptr, nullptr};     // "the H2D copy out of host_in[slot] is done"
    bool in_busy[3] = {false, false, false};                // ev_in[slot] has been recorded and not waited for yet
    cb::Workspace ws_band_parent;         // union-find slots of the resident band (row-band sharding)
    cb::Workspace ws_band_aux;            // boundary roots of the resident band + the cross-band forest
    int chunk_frames = 0;
    long long launches = 0;
    long long front_fast = 0, front_generic = 0;   // front-kernel launches on the lean kernels (front3 / front_cv) and on front.cu's generic one
    unsigned long long h2d_bytes = 0, d2h_bytes = 0;  // PCIe bytes moved by b200_canny_batch_host so far
    cb::Profiler prof;
    // band state (row-band sharding)
    int band_rows = 0, band_width = 0, band_row0 = 0;
    uint8_t* band_cls = nullptr;          // class map of the resident band (caller's d_edges)
    bool band_sparse = false;             // the resident band's labels were built from the kept-pixel list
    bool band_front_sparse = false;       // the band's front launches produced the kept-pixel list
    // weak-pixel count of the last launch of each pipeline slot, copied back asynchronously (pinned host memory, never waited
    // for): when more than 1/8 of the previous launch's pixels were weak the next one uses the tile-based labelling, whose shared-
    // memory unions win on such maps.  Both give identical results; a stale value only costs speed.
    unsigned int* h_kept = nullptr;       // [4]: slots 0..2 + the band (mapped pinned memory: the kernels write it directly)
    unsigned int* d_kept = nullptr;       // device-side address of h_kept
    bool list_dirty[4] = {false, false, false, false};   // a launch on this slot failed between front and link: re-zero its counters
    long long kept_px[4] = {0, 0, 0, 0};
    // ragged chunks (b200_canny_frames_device): the chunk's table (descriptors, tensor maps, work items) is built in pinned
    // staging per slot and sent up with one copy; the host rewrites the staging only after ev_ragged[slot] (recorded behind it)
    cb::Workspace ws_ragged[3], host_ragged[3];
    cudaEvent_t ev_ragged[3] = {nullptr, nullptr, nullptr};
    bool ragged_busy[3] = {false, false, false};
};

namespace cb {

struct ProfScope {  // RAII: records an event before and after whatever is launched inside its lifetime
    b200_ctx* ctx; cudaStream_t st; cudaEvent_t a = nullptr, b = nullptr; int cat;
    ProfScope(b200_ctx* c, cudaStream_t s, int category) : ctx(c), st(s), cat(category) {
        if (!ctx->prof.on) return;
        cudaEventCreate(&a); cudaEventCreate(&b);
        cudaEventRecord(a, st);
    }
    ~ProfScope() {
        if (!a) return;
        cudaEventRecord(b, st);
        ctx->prof.recs.push_back({cat, a, b});
    }
};

int ensure_ws(Workspace& ws, size_t bytes, bool pinned_host = false);
int prepare_gauss(b200_ctx* ctx, float sigma);
void host_gaussian_kernel(float sigma, std::vector<float>& w);
int host_window(float sigma);

// front.cu
// *sparse_out (optional) tells whether the kernel that ran filled p.parent / p.kept_list
// sparse_out: the kernel produced the weak-pixel list
int launch_front(b200_ctx* ctx, cudaStream_t st, const FrontParams& p, bool* sparse_out = nullptr);
int make_input_tensor_map(const FrontParams& p, int box_cols, int box_rows, CUtensorMap_st* tmap, bool* use_tma);
int make_bgr_tensor_map(const FrontParams& p, int box_words, int box_rows, CUtensorMap_st* tmap);   // 32-bit elements over 3*width-byte rows
// front3.cu (packed-FP32 blur, half-precision Sobel; the default for the radii it is built for)
bool front3_supports(const GaussTables& g);   // front3 takes this sigma: its half-window is compiled and its weights are not tiny
// ... and these interleaved B,G,R frames: p.in / width / in_pitch / in_frame_stride allow the fused BGR -> gray staging
bool front3_bgr_supports(const GaussTables& g, const FrontParams& p);
int launch_front3(b200_ctx* ctx, cudaStream_t st, const FrontParams& p);
// ragged chunks: class-row band height shared by the chunk's frames (the policy is described at its definition), the work items
// of one frame, and the launch over n_items items of p.ritems (all TMA-staged or all byte-staged)
int ragged_band_rows3(const b200_ctx* ctx, const int* heights, const int* widths, int n, int radius);
void ragged_items3(int frame, int height, int width, int band_rows, std::vector<RaggedItem>& items);
int ragged_tensor_map3(const uint8_t* in, long long pitch, int height, int width, int radius, CUtensorMap_st* tmap, bool* use_tma);
int launch_front3_ragged(b200_ctx* ctx, cudaStream_t st, const FrontParams& p, int n_items, bool use_tma);
// front_cv.cu (cv::Canny semantics, b200_cv_canny_aperture_device_strided): class map + weak-pixel list of p's frames, channels 1 or
// 3 interleaved, Sobel aperture 3, 5 or 7, L1 or L2 magnitude against p.lo / p.hi (already divided for aperture 7, floored and, for
// L2, squared)
int launch_front_cv(b200_ctx* ctx, cudaStream_t st, const FrontParams& p, int channels, bool l2, int aperture);
// ragged chunks (b200_cv_canny_aperture_frames_device): the work items of one frame (its 128 x 64 tiles), and the launch over n_items items of
// p.ritems with the frames of p.rframes
void ragged_items_cv(int frame, int height, int width, std::vector<RaggedItem>& items);
int launch_front_cv_ragged(b200_ctx* ctx, cudaStream_t st, const FrontParams& p, int n_items, int channels, bool l2, int aperture);
// selftest.cu
int check_div_mode_device(b200_ctx* ctx, float b, float y, float* c, int* mode);
// hysteresis.cu
int launch_hysteresis(b200_ctx* ctx, cudaStream_t st, const HystParams& p);   // label + resolve
int launch_ccl_label(b200_ctx* ctx, cudaStream_t st, const HystParams& p);    // tile-local forest + tile-boundary unions
int launch_ccl_resolve(b200_ctx* ctx, cudaStream_t st, const HystParams& p);  // weak pixels -> 0/255 in place
int launch_hysteresis_ragged(b200_ctx* ctx, cudaStream_t st, const RaggedHystParams& p);   // list-driven link + resolve
int launch_classify_i16(b200_ctx* ctx, cudaStream_t st, const int16_t* nms, uint8_t* cls, size_t n,
                        int lo, int hi);
int launch_expand_u8_to_i16(b200_ctx* ctx, cudaStream_t st, const uint8_t* cls, int16_t* out, size_t n);
int launch_pack_edges(b200_ctx* ctx, cudaStream_t st, const uint8_t* cls, uint32_t* bits, size_t n_px);
// stages.cu
int launch_xy_gradient(b200_ctx* ctx, cudaStream_t st, const int16_t* blur, int h, int w, int16_t* gx,
                       int16_t* gy);
int launch_sobel(b200_ctx* ctx, cudaStream_t st, const int16_t* blur, int h, int w, int16_t* mag,
                 int16_t* ang);
int launch_nonmaximal(b200_ctx* ctx, cudaStream_t st, const int16_t* mag, const int16_t* ang, int h,
                      int w, int16_t* out);
int launch_bgr_to_gray(b200_ctx* ctx, cudaStream_t st, const uint8_t* bgr, uint8_t* gray, size_t n_px);
// n_frames x h rows of w pixels from a pitched B,G,R source into a dense n_frames*h*w gray plane
int launch_bgr_to_gray_strided(b200_ctx* ctx, cudaStream_t st, const uint8_t* bgr, long long pitch, long long frame_stride,
                               int n_frames, int h, int w, uint8_t* gray);
// the frames of a ragged chunk (jobs: device table, ascending row0) into their gray scratch frames; rows: total rows
int launch_bgr_to_gray_ragged(b200_ctx* ctx, cudaStream_t st, const RaggedGrayJob* jobs, int n_jobs, long long rows);
// band.cu: one row band's local stages in pieces
struct BandGeom {
    const uint8_t* d_rows;   // global row (row0 - above) of the band buffer
    int above, below;        // halo rows present above / below the band
    int rows, row0;          // rows owned, first global row
    int height, width;       // GLOBAL image height, width
    int lo, hi;
    uint8_t* d_edges;        // rows x width class / edge map of the band
};
int band_prepare(b200_ctx* ctx, const BandGeom& g, float sigma);
int band_front_rows(b200_ctx* ctx, cudaStream_t st, const BandGeom& g, int sub_row0, int sub_rows);
int band_label(b200_ctx* ctx, cudaStream_t st, const BandGeom& g);
// synth.cu
int launch_synth(b200_ctx* ctx, cudaStream_t st, uint8_t* d, int n_frames, int row0, int rows, int width,
                 int kind, uint64_t seed, int first_frame);
int launch_count255(b200_ctx* ctx, cudaStream_t st, const uint8_t* d, size_t n, unsigned long long* d_count);
int launch_hash255(b200_ctx* ctx, cudaStream_t st, const uint8_t* d, size_t n, unsigned long long offset, unsigned long long* d_out);

}  // namespace cb
