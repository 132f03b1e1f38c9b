/*
 * canny_b200.h — C ABI of the B200-native Canny hot path (libcanny_b200.so).
 *
 * This is the drop-in boundary for StevenChang5/Canny_Edge's GPU stage API.  Every entry point names
 * the reference interface it replaces (paths relative to the reference checkout).  Plain pointers and
 * sizes only; no C++ or torch types.  All images are row-major, contiguous (pitch == width) exactly
 * as the reference's Mat.data convention (src/utils.cpp:12-15), except in the *_strided device batch
 * calls, which take byte strides for rows and frames.
 *
 * There is NO CPU fallback: every compute entry point runs hand-written sm_100a kernels and returns
 * B200_ERR_NO_DEVICE / B200_ERR_CUDA when that is impossible.
 *
 * Error convention.  The reference returns void and checks no CUDA status (src/cuda.cu:83-101).  The
 * C ABI returns an int status (0 == B200_OK) and keeps a thread-local message readable through
 * b200_last_error().  Argument domains follow the reference: height,width >= 2 (below that the
 * reference's gradient reads out of bounds, src/utils.cpp:117,158), sigma > 0.  Thresholds: the CLI's
 * 0 <= lo < hi <= 255 check lives in src/main.cpp:63-76 and stays there; the library accepts any int pair
 * and behaves as src/utils.cpp:322-342 does — lo >= hi and negative values included, and max_val > 255
 * gives the reference's ALL-ZERO map (its flood writes EDGE = 255, its second scan then removes everything
 * below max_val) — with ONE exception: min_val > 255 >= max_val, where the reference's result depends on
 * the raster order of its flood starts (:327-340), returns B200_ERR_UNSUPPORTED.
 */
#ifndef CANNY_B200_H
#define CANNY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_OK 0
#define B200_ERR_INVALID_ARG 1 /* bad pointer / size / sigma                                    */
#define B200_ERR_NO_DEVICE 2   /* no CUDA device, or the device is not sm_100                    */
#define B200_ERR_CUDA 3        /* a CUDA runtime / driver call failed (see b200_last_error)     */
#define B200_ERR_UNSUPPORTED 4 /* valid in the reference but outside this build's limits         */
#define B200_ERR_NOMEM 5

/* Constants of src/utils.h:5-6. */
#define B200_EDGE 255
#define B200_NOEDGE 0

/* Largest Gaussian half-window (window/2) the kernels are built for: sigma <= 16. */
#define B200_MAX_RADIUS 48

typedef struct b200_ctx b200_ctx; /* opaque: device, streams, workspace pool, cached tables */

/* ------------------------------------------------------------------ library / context ---------- */

int b200_version(void);              /* ABI version, bumped on any signature change             */
const char* b200_last_error(void);   /* thread-local text of the last non-OK status             */

/* Creates a context on CUDA device `device` (>= 0).  Replaces the reference's per-call
 * cudaMalloc/cudaFree (src/cuda.cu:83-86,98-101 and the same pattern in every wrapper) with a
 * persistent workspace pool, streams and pinned staging. */
int b200_ctx_create(int device, b200_ctx** out);
int b200_ctx_destroy(b200_ctx* ctx);
/* Makes the context issue work on an existing cudaStream_t (e.g. torch's current stream) instead of
 * its own; pass NULL to go back to the context's private stream.  When the stream changes, the new one
 * first waits for the work already issued through the context (it shares the context's workspace). */
int b200_ctx_set_stream(b200_ctx* ctx, void* cuda_stream);
/* Blocks until everything issued on the context has finished. */
int b200_ctx_synchronize(b200_ctx* ctx);
/* Frames per internal chunk for batch calls (0 = automatic: sized so a chunk's intermediates stay in
 * the 126 MB L2). */
int b200_ctx_set_chunk_frames(b200_ctx* ctx, int frames);
/* Number of kernels this context has launched so far (bench.py's gpu_launches). */
long long b200_ctx_kernel_launches(const b200_ctx* ctx);
/* Bytes b200_canny_batch_host has moved over PCIe so far on this context, per direction (bench.py's e2e byte counts: the edge
 * maps of jobs >= 8 Mpix come back bit-packed, 1 bit per pixel, and are expanded to 0 / 255 bytes on the host). */
int b200_ctx_transfer_bytes(const b200_ctx* ctx, unsigned long long* h2d_bytes, unsigned long long* d2h_bytes);

/* Front-kernel launches so far on this context: on the specialised kernels (Gaussian half-window 2, 3, 5, 6, 9 or 15 — sigma 1.4
 * is 5, sigma 5 is 15 — and no per-stage planes requested) and on the generic one (any half-window up to B200_MAX_RADIUS, spill
 * planes; about 4x slower).  The first plain-map launch that falls back also prints one line on stderr (B200_CANNY_QUIET=1
 * silences it). */
int b200_ctx_front_kernel_stats(const b200_ctx* ctx, long long* fast_launches, long long* generic_launches);
/* Pins the calling thread — and the threads and first-touch pinned allocations it makes afterwards — to the CPUs of the NUMA node
 * `device` is attached to (sysfs); *node_out = that node, or -1 when nothing was changed (single-node host, no permission).  Call
 * it before b200_ctx_create / before allocating pinned buffers in a one-process-per-GPU deployment. */
int b200_host_bind_numa(int device, int* node_out);

/* In every function below ctx may be NULL: a lazily created process-wide context on the current
 * CUDA device is used (what the reference-signature C++ shims in canny_b200_compat.hpp do). */

/* ------------------------------------------------------------------ host-side helpers ----------- */

/* window = 1 + 2*ceil(3*sigma)                         — src/utils.cpp:78, src/cuda.cu:78 */
int b200_gaussian_window(float sigma);
/* createGaussianKernel(float*&, float, int*)            — src/utils.cpp:77-95 and the host overload
 * src/cuda.cu:15-30.  Host code (as in the reference); w must hold b200_gaussian_window(sigma)
 * floats. */
int b200_gaussian_kernel(float sigma, float* w, int* window);
/* Exact integer form of the reference's atan2 binning (src/utils.cpp:215-231) as the kernels use
 * it, evaluated on the HOST for table tests: returns 0, 45, 90 or 135. Valid for |gx|,|gy| <= 1020. */
int b200_direction_host(int gx, int gy);
/* floor(sqrt(n)) as the kernels compute magnitude (src/utils.cpp:212), host evaluation. */
int b200_isqrt_host(int n);

/* ------------------------------------------------------------------ stage API, host buffers ---- */

/* cuda_gaussian(unsigned char*& img_h, float sigma, int height, int width, short*& result_h)
 *                                                       — src/cuda.h:4, src/cuda.cu:75-102
 * (CPU twin gaussian(), src/utils.cpp:26-68).  blur: caller-allocated height*width int16. */
int b200_gaussian(b200_ctx* ctx, const uint8_t* img, float sigma, int height, int width,
                  int16_t* blur);

/* calculateXYGradient(short*& img, int h, int w, short*& grad_x, short*& grad_y)
 *                                                       — src/utils.h:12, src/utils.cpp:106-187
 * (the reference GPU path fuses this into sobel_util, src/cuda.cu:185-191, with a flipped gy sign;
 * this follows the CPU semantics). */
int b200_xy_gradient(b200_ctx* ctx, const int16_t* blur, int height, int width, int16_t* grad_x,
                     int16_t* grad_y);

/* cuda_sobel(short*& img_h, int height, int width, short*& magnitude_h, short*& angle_h)
 *                                                       — src/cuda.h:6, src/cuda.cu:220-246
 * (CPU twin sobelOperator(), src/utils.cpp:201-236; unlike it the input is NOT freed, matching
 * cuda_sobel).  angle holds 0/45/90/135. */
int b200_sobel(b200_ctx* ctx, const int16_t* blur, int height, int width, int16_t* magnitude,
               int16_t* angle);

/* cuda_nonmaixmal_suppression(short*& magnitude_h, short*& angle_h, int height, int width,
 *                             short*& result_h)         — src/cuda.h:8, src/cuda.cu:366-390
 * (CPU twin nonmaximalSuppression(), src/utils.cpp:248-308; inputs are NOT freed). */
int b200_nonmaximal(b200_ctx* ctx, const int16_t* magnitude, const int16_t* angle, int height,
                    int width, int16_t* nms);

/* hysteresis(short*& edgeCandidates, int height, int width, int minVal, int maxVal)
 *                                                       — src/utils.h:18, src/utils.cpp:322-342
 * + findEdgePixels (src/utils.cpp:360-427).  The reference has no GPU hysteresis (cuda_canny calls
 * the CPU one, src/cuda.cu:436); this runs it as GPU connected components.  In place: on return every
 * element is 0 or 255. */
int b200_hysteresis(b200_ctx* ctx, int16_t* nms_inout, int height, int width, int min_val,
                    int max_val);

/* cuda_canny(unsigned char* img, float sigma, int min_val, int max_val, int height, int width,
 *            bool steps)                                — src/cuda.h:10, src/cuda.cu:392-450
 * (CPU twin canny(), src/utils.cpp:429-492).  The reference only displays its result; here the 0/255
 * map is returned in `edges` (int16, the type of the array the reference shows, src/cuda.cu:439).
 * Fused path: one H2D, two kernel phases, one D2H. */
int b200_canny(b200_ctx* ctx, const uint8_t* img, float sigma, int min_val, int max_val, int height,
               int width, int16_t* edges);

/* The `steps` flag of cuda_canny (src/cuda.cu:400-434): additionally returns the planes the
 * reference would display after each stage.  Any of blur/magnitude/angle/nms may be NULL. */
int b200_canny_steps(b200_ctx* ctx, const uint8_t* img, float sigma, int min_val, int max_val,
                     int height, int width, int16_t* blur, int16_t* magnitude, int16_t* angle,
                     int16_t* nms, int16_t* edges);

/* cvtColor(frame, gray, COLOR_BGR2GRAY) + cuda_canny — what the reference's frame loop does per frame (src/main.cpp:113,128),
 * with the colour conversion moved onto the GPU.  bgr: height*width*3 bytes, interleaved B,G,R as cv::Mat stores them.  The
 * gray values are OpenCV's 8-bit fixed-point ones ((B*3735 + G*19235 + R*9798 + 2^14) >> 15), bit for bit.  gray_out may be
 * NULL (then the front kernel converts while it stages its tiles, see b200_canny_batch_device_bgr); when given it receives the
 * height*width gray plane the pipeline ran on. */
int b200_canny_bgr(b200_ctx* ctx, const uint8_t* bgr, float sigma, int min_val, int max_val, int height, int width,
                   uint8_t* gray_out, int16_t* edges);
/* The conversion alone on DEVICE memory (n_px pixels; d_bgr 3*n_px bytes, d_gray n_px bytes), asynchronous on the
 * context's stream: for callers whose decoder already leaves BGR frames in HBM. */
int b200_bgr_to_gray_device(b200_ctx* ctx, const uint8_t* d_bgr, size_t n_px, uint8_t* d_gray);

/* ------------------------------------------------------------------ batched, u8 edge maps ------ */

/* n_frames independent frames, host memory in, host memory out (u8, 0/255).  What main.cpp's frame
 * loop (src/main.cpp:120-137) becomes for N frames: chunked, H2D / kernels / D2H overlapped on
 * separate streams.  frames: n_frames*height*width bytes.  Pinned (page-locked) buffers give the full
 * PCIe rate; pageable ones work (jobs of >= 32 MB are staged through pinned memory by the library's host
 * threads).  Jobs of >= 8 Mpix return the map over PCIe bit-packed and expand it into `edges` with a few
 * host threads while the GPU works on the next chunk. */
int b200_canny_batch_host(b200_ctx* ctx, const uint8_t* frames, int n_frames, int height, int width,
                          float sigma, int min_val, int max_val, uint8_t* edges);

/* Same, but the caller takes the maps in the PACKED form they cross PCIe in: 1 bit per pixel, bit i of frame f's words <-> pixel
 * i of frame f, every frame starting on a 32-bit word (frame stride ceil(height*width/32) words).  No host expansion pass: on a
 * host whose memory system is shared by several GPUs' transfers this is the scalable form (b200_unpack_edges_host expands a
 * frame when bytes are needed after all). */
int b200_canny_batch_host_packed(b200_ctx* ctx, const uint8_t* frames, int n_frames, int height, int width,
                                 float sigma, int min_val, int max_val, uint32_t* edge_bits);

/* Same with DEVICE pointers (already resident in HBM): d_frames and d_edges are n_frames*height*width
 * bytes each, on the context's device.  Asynchronous on the context's stream.  d_edges may not alias
 * d_frames. */
int b200_canny_batch_device(b200_ctx* ctx, const uint8_t* d_frames, int n_frames, int height,
                            int width, float sigma, int min_val, int max_val, uint8_t* d_edges);

/* b200_canny_batch_device for frames a decoder left in HBM as interleaved B,G,R (cv::Mat's CV_8UC3 layout; d_bgr: n_frames *
 * height*width*3 bytes): cvtColor(frame, gray, COLOR_BGR2GRAY) (src/main.cpp:113) happens INSIDE the front kernel, on the
 * staged tile — no separate conversion pass and no gray plane in HBM — when width % 16 == 0, d_bgr is 16-byte aligned and
 * sigma's half-window is one of 2, 3, 5, 6, 9 (B200_CANNY_BGR_FUSED=0 turns it off); otherwise each chunk is converted into a
 * gray scratch plane first.  Same gray values either way (OpenCV's fixed-point ones, see b200_canny_bgr), same edge maps. */
int b200_canny_batch_device_bgr(b200_ctx* ctx, const uint8_t* d_bgr, int n_frames, int height, int width, float sigma,
                                int min_val, int max_val, uint8_t* d_edges);

/* The two calls above for frames and edge maps with their own strides: pitched buffers (cv::cuda::GpuMat's data / step, a
 * decoder's luma plane), crops and channel views of tensors, frames padded for alignment.  All strides are in BYTES:
 *   pixel (f, y, x) is read from d_frames + f*in_frame_stride + y*in_row_pitch + x (gray) or from the 3 bytes at
 *   d_bgr + f*in_frame_stride + y*in_row_pitch + 3*x (B, G, R), and its 0 / 255 result is written to
 *   d_edges + f*out_frame_stride + y*out_row_pitch + x.
 * No other byte of d_edges is written (not even with the value it holds), so d_edges may be a region of a larger image.  No copy
 * is made: the kernels address the strides themselves.  The front kernel stages its tiles by TMA when the input's base, row pitch
 * and frame stride are multiples of 16 bytes (any width); other layouts take its byte-load staging, with the same results.  BGR
 * frames are converted inside the front kernel under the conditions of b200_canny_batch_device_bgr plus a row pitch that is a
 * multiple of 16; otherwise each chunk is converted into a dense gray scratch plane first.  The frame strides of a single frame
 * are ignored.  Asynchronous on the context's stream.
 * B200_ERR_INVALID_ARG, before any device work: a null pointer; height or width < 2; n_frames <= 0; a negative stride;
 * in_row_pitch < width (3*width for BGR) or out_row_pitch < width; for n_frames > 1, a frame stride smaller than one frame's
 * bytes ((height-1)*pitch + row bytes), i.e. overlapping frames; an input or output extent of more than 2^48 bytes; an output
 * extent that overlaps the input extent.  The dense calls above run the same checks with pitch = row bytes. */
int b200_canny_batch_device_strided(b200_ctx* ctx, const uint8_t* d_frames, int64_t in_row_pitch, int64_t in_frame_stride,
                                    int n_frames, int height, int width, float sigma, int min_val, int max_val,
                                    uint8_t* d_edges, int64_t out_row_pitch, int64_t out_frame_stride);
int b200_canny_batch_device_bgr_strided(b200_ctx* ctx, const uint8_t* d_bgr, int64_t in_row_pitch, int64_t in_frame_stride,
                                        int n_frames, int height, int width, float sigma, int min_val, int max_val,
                                        uint8_t* d_edges, int64_t out_row_pitch, int64_t out_frame_stride);

/* OpenCV semantics: the edge maps of cv::Canny(image, edges, threshold1, threshold2, aperture_size, l2_gradient) (OpenCV 4.x), bit
 * for bit, for 8-bit frames with 1 channel or 3 interleaved channels (in any order: B,G,R as cv::Mat holds them, R,G,B, ...), any
 * size of at least 1 x 1.  The entry points above compute the reference's Canny instead; the differences:
 *   blur            reference: Gaussian from sigma, renormalised at borders      here: none
 *   gradient        reference: Sobel, replicate for gx, drop for gy                here: Sobel of aperture_size 3, 5 or 7,
 *                                                                                        BORDER_REPLICATE for both
 *   magnitude       reference: floor(sqrt(gx^2 + gy^2))                            here: |dx| + |dy|, or dx^2 + dy^2 against squared
 *                                                                                        thresholds when l2_gradient != 0
 *   direction, NMS  reference: atan2 bins, `>` on both sides                       here: fixed-point tan 22.5 deg (13573 / 2^15),
 *                                                                                        `>` on one side and `>=` on the other, `>`
 *                                                                                        on both along the diagonals
 *   thresholds      reference: `>= minVal`, `>= maxVal`, ints                      here: `> low`, `> high`, doubles: swapped when
 *                                                                                        threshold1 > threshold2; for L2 clamped to
 *                                                                                        32767 and squared when positive; floored
 *   hysteresis      reference: 8-connected minus its one-way (1,0)->(0,1) link     here: plain 8-connected
 *   colour          reference: BGR -> gray first                                   here: Sobel on every channel, per pixel the
 *                                                                                        channel of largest magnitude (the first
 *                                                                                        in memory on ties)
 * Strides in BYTES as b200_canny_batch_device_strided: pixel (f, y, x) is the `channels` bytes at d_in + f*in_frame_stride +
 * y*in_row_pitch + channels*x, and its 0 / 255 result is written to d_edges + f*out_frame_stride + y*out_row_pitch + x; no other
 * byte of d_edges is written.  Chunks, stream slots and b200_ctx_set_chunk_frames as the batch calls.  Asynchronous on the
 * context's stream.
 * Apertures, as cv::getDerivKernels builds them (dx: derivative taps across columns, smoothing taps down rows; dy: the transpose):
 *   3: smoothing 1 2 1, derivative -1 0 1;
 *   5: smoothing 1 4 6 4 1, derivative -1 -2 0 2 1; exact integers, |dx|, |dy| <= 12240;
 *   7: smoothing 1 6 15 20 15 6 1, derivative -1 -4 -5 0 5 4 1; both derivatives are scaled by 1/16 and rounded half to even
 *      (cvRound), |dx|, |dy| <= 10200, and both thresholds are divided by 16 before the swap, the L2 clamp, the squaring and the
 *      floor (so the int32 check below applies to the divided value).
 * Before any device work, in this order: B200_ERR_UNSUPPORTED for channels other than 1 and 3; B200_ERR_INVALID_ARG for an
 * aperture_size other than 3, 5 and 7 (cv::Canny rejects those too); B200_ERR_UNSUPPORTED for a height above 4 194 240 (65535 x 64)
 * rows; B200_ERR_INVALID_ARG for a NaN or infinite threshold; B200_ERR_UNSUPPORTED for a threshold whose floor (after the L2
 * squaring) does not fit in int32, where OpenCV's own conversion overflows; then the layout checks of
 * b200_canny_batch_device_strided (in_row_pitch >= channels*width), except that frames of 1 pixel per side are accepted.
 * b200_cv_canny_device_strided is the same call with aperture_size 3.
 * Frames of different sizes in one call: b200_cv_canny_aperture_frames_device, below b200_frame. */
int b200_cv_canny_aperture_device_strided(b200_ctx* ctx, const uint8_t* d_in, int64_t in_row_pitch, int64_t in_frame_stride,
                                          int n_frames, int height, int width, int channels, double threshold1, double threshold2,
                                          int aperture_size, int l2_gradient, uint8_t* d_edges, int64_t out_row_pitch,
                                          int64_t out_frame_stride);
int b200_cv_canny_device_strided(b200_ctx* ctx, const uint8_t* d_in, int64_t in_row_pitch, int64_t in_frame_stride, int n_frames,
                                 int height, int width, int channels, double threshold1, double threshold2, int l2_gradient,
                                 uint8_t* d_edges, int64_t out_row_pitch, int64_t out_frame_stride);

/* A list of frames of DIFFERENT sizes and layouts in one call: dataset images, camera streams of several resolutions, crops of
 * detections, a list of cv::cuda::GpuMat.  Each frame has its own size, input pointer and row pitch and its own output pointer
 * and row pitch; sigma and the thresholds are shared.  Frame i's map is the one b200_canny_batch_device_strided gives for that
 * frame alone, bit for bit.
 *   pixel (y, x) of frame i is read from in + y*in_row_pitch + x (gray) or from the 3 bytes at in + y*in_row_pitch + 3*x
 *   (B, G, R), and its 0 / 255 result is written to out + y*out_row_pitch + x.  No other output byte is written, so the outputs
 *   may be regions of one larger image (a mosaic whose tiles sit in rows of their own: extents may not overlap, see below).
 * `frames` is host memory, read only during the call.  Work is asynchronous on the context's stream.  The list is cut, in call
 * order, into chunks of about 75 Mpix (b200_ctx_set_chunk_frames caps the frames per chunk); a larger frame has a chunk of its own.
 * B200_ERR_INVALID_ARG, before any device work: a null `frames`, `in` or `out`; n_frames <= 0; a frame smaller than 2 x 2; a
 * negative pitch or one below a row (width, 3*width for BGR); an extent ((height-1)*pitch + row bytes) above 2^48 bytes; an
 * output extent that overlaps any input extent or any other output extent.  Inputs may overlap each other (the same frame may be
 * listed twice).  A frame of 2^31 pixels or more: B200_ERR_UNSUPPORTED. */
typedef struct b200_frame {
    const uint8_t* in;        /* device; gray: 1 byte per pixel, BGR: 3 (B,G,R) */
    int64_t in_row_pitch;     /* bytes */
    uint8_t* out;             /* device; 0 / 255 bytes */
    int64_t out_row_pitch;    /* bytes */
    int32_t height, width;
} b200_frame;
int b200_canny_frames_device(b200_ctx* ctx, const b200_frame* frames, int n_frames, float sigma, int min_val, int max_val);
int b200_canny_frames_device_bgr(b200_ctx* ctx, const b200_frame* frames, int n_frames, float sigma, int min_val, int max_val);

/* cv2.Canny(frame_i, threshold1, threshold2, apertureSize=aperture_size, L2gradient=l2_gradient) of a list of frames of different
 * sizes in one call: b200_cv_canny_aperture_device_strided's semantics with b200_canny_frames_device's lists (a dataset of photos of
 * many sizes, prepared for an edge-conditioned model).  Frame i's map is bit for bit the one b200_cv_canny_aperture_device_strided
 * gives for that frame alone.
 *   pixel (y, x) of frame i is the `channels` bytes (1 or 3 interleaved) at in + y*in_row_pitch + channels*x, and its 0 / 255 result
 *   is written to out + y*out_row_pitch + x.  No other output byte is written.
 * Frames of any size from 1 x 1 up; no limit on the height beyond the 2^31 pixels below.  `frames` is host memory, read only during
 * the call.  Chunks (about 75 Mpix, b200_ctx_set_chunk_frames), stream slots and asynchrony as b200_canny_frames_device.
 * Before any device work, in this order: B200_ERR_UNSUPPORTED for channels other than 1 and 3; B200_ERR_INVALID_ARG for an
 * aperture_size other than 3, 5 and 7; the threshold checks of b200_cv_canny_aperture_device_strided (B200_ERR_INVALID_ARG for NaN
 * or inf, B200_ERR_UNSUPPORTED for a floor outside int32, after the division for aperture 7); then the list
 * checks of b200_canny_frames_device with `channels` bytes per input pixel and frames from 1 x 1: B200_ERR_INVALID_ARG for a null
 * `frames`, `in` or `out`, n_frames <= 0, an empty frame, a negative pitch or one below a row (channels*width input bytes, width
 * output bytes), an extent above 2^48 bytes, an output extent that overlaps any input extent or any other output extent (inputs may
 * overlap); B200_ERR_UNSUPPORTED for a frame of 2^31 pixels or more.
 * b200_cv_canny_frames_device is the same call with aperture_size 3. */
int b200_cv_canny_aperture_frames_device(b200_ctx* ctx, const b200_frame* frames, int n_frames, int channels, double threshold1,
                                         double threshold2, int aperture_size, int l2_gradient);
int b200_cv_canny_frames_device(b200_ctx* ctx, const b200_frame* frames, int n_frames, int channels, double threshold1,
                                double threshold2, int l2_gradient);

/* The packed form of an edge map — 1 bit per pixel, bit i of byte k <-> pixel 8k+i, ceil(n_px/32)*4 bytes — is what
 * b200_canny_batch_host moves over PCIe.  Both halves are exported for callers that store or ship maps in that form:
 *   b200_pack_edges_device   0 / 255 bytes in DEVICE memory -> packed words in DEVICE memory, asynchronous on the context's
 *                            stream (d_bits: ceil(n_px/32) 32-bit words);
 *   b200_unpack_edges_host   packed bytes in HOST memory -> 0 / 255 values in HOST memory, as bytes (elem_size 1) or as the
 *                            reference's int16 (elem_size 2), on `threads` host threads (<= 0: the library's default).  Pure
 *                            host code: needs no GPU.  (No reference counterpart: src/utils.cpp:322-342 writes int16 in place.) */
int b200_pack_edges_device(b200_ctx* ctx, const uint8_t* d_edges, size_t n_px, uint32_t* d_bits);
int b200_unpack_edges_host(const uint8_t* bits, size_t n_px, void* out, int elem_size, int threads);

/* The same work as b200_canny_batch_device, issued serially on the context's stream with a CUDA event
 * pair around every kernel; blocks, then returns per-kernel-class totals: ms_out[5] / launches_out[5]
 * indexed 0 = front (blur+Sobel+NMS+classify), 1 = ccl_local, 2 = ccl_merge, 3 = ccl_final, 4 = other.
 * This is how bench.py measures the dominant kernel's launch duration for its roofline entry. */
int b200_profile_stages_device(b200_ctx* ctx, const uint8_t* d_frames, int n_frames, int height,
                               int width, float sigma, int min_val, int max_val, uint8_t* d_edges,
                               float* ms_out, int* launches_out);

/* Same, but through the production path itself (b200_canny_batch_device: three stream slots whose kernels overlap), every
 * kernel bracketed by events on ITS stream: durations of kernels as they run in the timed bench step, sharing the machine. */
int b200_profile_pipeline_device(b200_ctx* ctx, const uint8_t* d_frames, int n_frames, int height,
                                 int width, float sigma, int min_val, int max_val, uint8_t* d_edges,
                                 float* ms_out, int* launches_out);

/* ------------------------------------------------------------------ row-band sharding ---------- */

/* One image of global_height rows split into row bands, one band per GPU/rank (BASELINE config 5).
 * A band owns global rows [row0, row0+band_rows).  Stages 1-3 need b200_band_halo_rows(sigma) input
 * rows beyond each interior band edge (window/2 for the blur + 1 Sobel + 1 NMS).
 *
 * b200_band_front : d_rows points at global row (row0 - halo_above); halo_above/halo_below say how
 *   many real rows are present above/below the band (0 at the image's true top/bottom, otherwise
 *   b200_band_halo_rows).  Runs stages 1-3 + classification and the band-local connected components.
 *   Afterwards d_edges (band_rows*width) holds 0 / 1 (weak) / 255 (strong) and the band's label state
 *   is kept in the context.
 * b200_band_boundary_export : writes this band's first and last row as (label, flags) records into
 *   d_records[b200_band_record_count(width)], ready to be all-gathered (NCCL) by the caller.
 * b200_band_finalize : given ALL bands' records (n_bands*b200_band_record_count(width), band order), merges label
 *   equivalences across every band boundary (8-connectivity across the boundary, including the
 *   reference's missing (1,0)->(0,1) link when that pair straddles nothing — it never does for
 *   band_rows >= 2), decides which local components become strong and rewrites d_edges to 0/255.
 */
typedef struct b200_band_record {
    int32_t label; /* canonical record index of the pixel's band-local component (same label == same
                      component inside that band); -1 when not a candidate or already strong          */
    int32_t flags; /* bit1 = pixel is a candidate (>= minVal); bit0 = its component contains a seed   */
} b200_band_record;

/* records a band exports: its first row (width), its last row (width), and the two pixels (0,1), (1,0)
 * of the reference's missing link (src/utils.cpp:399), present only in the band that owns row 0. */
int b200_band_record_count(int width);
int b200_band_halo_rows(float sigma);
int b200_band_front(b200_ctx* ctx, const uint8_t* d_rows, int halo_above, int halo_below,
                    int band_rows, int row0, int global_height, int width, float sigma, int min_val,
                    int max_val, uint8_t* d_edges);
int b200_band_boundary_export(b200_ctx* ctx, int band_rows, int width, b200_band_record* d_records);
int b200_band_finalize(b200_ctx* ctx, const b200_band_record* d_all_records, int n_bands,
                       int band_index, int band_rows, int width, uint8_t* d_edges);

/* ------------------------------------------------------------------ row bands across GPUs ------- */

/* The whole band pipeline of one rank — halo exchange, stages 1-3, band-local labelling, boundary-record exchange, cross-band
 * merge, finalisation — behind one handle, for a caller in the position of src/main.cpp:128 that owns several B200s (the
 * reference itself is single-GPU and finishes hysteresis on the CPU, src/cuda.cu:436).  One band per GPU, band r of `world` owns
 * global rows [r*H/world ..) (remainder rows go to the low ranks; b200_bands_info tells).
 *
 * Transports (same results; b200_bands_info reports which one is active):
 *   1 = P2P: the neighbours' band buffers are mapped (CUDA IPC between processes, plain pointers inside one process); halo rows
 *       are pulled by the copy engines over NVLink while the front kernel works on the interior rows, and the boundary records
 *       travel sparse (candidate pixels only), read straight from the peers' memory by the merge kernel.  No collective on the
 *       data path; NCCL only bootstraps (all-gather of the IPC handles).
 *   2 = NCCL: ncclSend/ncclRecv of the halo rows + one ncclAllGather of the dense records.  Chosen when a peer cannot be mapped,
 *       or with B200_BANDS_TRANSPORT=nccl in the environment.
 *   0 = a single band (world == 1): no exchange.
 *
 * b200_bands_create: one call per rank (one process per GPU, or one thread per GPU with separate communicators).  Pass EITHER
 *   an existing ncclComm_t of exactly `world` ranks (of the libnccl.so.2 already loaded in the process: the library resolves NCCL
 *   with dlopen and has no link-time dependency on it) OR nccl_comm = NULL and the 128-byte unique id that rank 0 obtained from
 *   b200_bands_unique_id and the caller broadcast by its own means (MPI, a socket, torch.distributed ...).  Collective: every rank
 *   must call it.  world == 1 needs neither.
 * b200_bands_create_group: all bands inside ONE process (ctxs[i] may sit on different devices, peer access is enabled, or on the
 *   same device: the virtual-band mode of the tests); no NCCL at all.  Drive a group with b200_bands_run_group.
 * b200_bands_input: device pointer of the band's own rows inside the handle's persistent [halo | band | halo] buffer: the caller
 *   writes its rows (rows x width bytes) there, on the context's stream or ordered before it, then calls run.
 * b200_bands_run: one step, asynchronous on the context's stream; d_edges (rows x width bytes, device) holds the band's 0 / 255
 *   map afterwards.  Collective: every rank calls it the same number of times.  A rank may overwrite its input rows again as soon
 *   as ITS step has completed (every peer has fetched what it needs by then).
 * b200_bands_check: synchronises and reports a peer that never signalled (bounded waits in the kernels) as B200_ERR_CUDA.
 * b200_bands_set_timing / b200_bands_stage_ms: CUDA-event times (ms) of the last step's stages on this rank:
 *   [0] signal + interior rows, [1] waiting for the halo rows, [2] edge rows + labelling, [3] record export, [4] record exchange,
 *   [5] cross-band merge + finalisation.
 */
typedef struct b200_bands b200_bands;
#define B200_NCCL_UNIQUE_ID_BYTES 128
int b200_bands_unique_id(void* id_out /* B200_NCCL_UNIQUE_ID_BYTES */);
int b200_bands_create(b200_ctx* ctx, void* nccl_comm, const void* unique_id, int rank, int world, int height, int width,
                      float sigma, int min_val, int max_val, b200_bands** out);
int b200_bands_create_group(b200_ctx* const* ctxs, int n_bands, int height, int width, float sigma, int min_val, int max_val,
                            b200_bands** out /* n_bands handles */);
int b200_bands_destroy(b200_bands* bands);
int b200_bands_info(const b200_bands* bands, int* row0, int* rows, int* halo_rows, int* transport);
int b200_bands_input(b200_bands* bands, uint8_t** d_band_rows);
int b200_bands_run(b200_bands* bands, uint8_t* d_edges);
int b200_bands_run_group(b200_bands* const* bands, int n_bands, uint8_t* const* d_edges);
/* the three phases b200_bands_run chains (exported for callers that interleave several bands themselves) */
int b200_bands_begin(b200_bands* bands, uint8_t* d_edges);
int b200_bands_front(b200_bands* bands);
int b200_bands_finish(b200_bands* bands);
int b200_bands_check(b200_bands* bands);
int b200_bands_set_timing(b200_bands* bands, int on);
int b200_bands_stage_ms(b200_bands* bands, float* ms6);

/* ------------------------------------------------------------------ synthetic workloads -------- */

/* Procedural test frames (pure integer hash; identical bytes on host and device) used by bench.py
 * and the parity tests.  kind: 0 = "shapes" (smooth background + discs + mild noise),
 * 1 = uniform noise (hysteresis worst case), 2 = constant 128.  Frame f of a batch uses
 * frame index first_frame + f. */
int b200_synth_host(uint8_t* frames, int n_frames, int height, int width, int kind, uint64_t seed,
                    int first_frame);
int b200_synth_device(b200_ctx* ctx, uint8_t* d_frames, int n_frames, int height, int width,
                      int kind, uint64_t seed, int first_frame);
/* Same generator for a row range [row0, row0+rows) of one frame of global_height rows (band tests). */
int b200_synth_rows_host(uint8_t* rows_out, int row0, int rows, int width, int kind, uint64_t seed,
                         int frame);
int b200_synth_rows_device(b200_ctx* ctx, uint8_t* d_rows, int row0, int rows, int width, int kind,
                           uint64_t seed, int frame);

/* ------------------------------------------------------------------ self-tests ----------------- */
/* Whole-domain dumps of the exact-arithmetic building blocks (tests/): the angle (0/45/90/135) for
 * every (gx,gy) in [-gmax,gmax]^2, row-major by gy then gx, from the host classifier and from the
 * device one; floor(sqrt(n)) for n = 0..n_max as the kernels compute it; and an exhaustive comparison
 * of the kernels' Markstein division against IEEE division for every numerator in [0, 256*count] and
 * every entry of sigma's count table (mismatch count returned). */
int b200_direction_table_host(int gmax, int16_t* out);
int b200_direction_table_device(b200_ctx* ctx, int gmax, int16_t* out_host);
int b200_isqrt_table_device(b200_ctx* ctx, int n_max, int32_t* out_host);
int b200_division_check_device(b200_ctx* ctx, float sigma, unsigned long long* mismatches);
/* Which exact form of sum / count the fused kernel uses for sigma's interior count, as decided by an exhaustive device check
 * over all 2^23 float mantissas when the tables are built: 1 = fma(a, RN(1/count - 1), a), 3 = one Markstein correction of
 * a * RN(1/count), 5 = two corrections (always valid). */
int b200_division_mode_device(b200_ctx* ctx, float sigma, int* mode);

/* Device-side count of 255 bytes in a u8 buffer (edge pixels), written to *count. */
int b200_count_edges_device(b200_ctx* ctx, const uint8_t* d_edges, size_t n, unsigned long long* count);

/* Position-dependent checksum of a device edge map: sum over its 255-pixels of mix64(global_offset + index) mod 2^64 (the
 * splitmix64 finaliser of the frame generator).  Additive: the checksums of the row bands of one image, each taken with its
 * band's global pixel offset, sum to the checksum of the whole map (bench.py's cross-GPU parity field). */
int b200_hash_edges_device(b200_ctx* ctx, const uint8_t* d_edges, size_t n, unsigned long long global_offset,
                           unsigned long long* hash);

/* Raw device memory helpers so non-CUDA hosts (ctypes, cgo, JNI) can stage data without a CUDA
 * binding of their own. */
int b200_device_alloc(b200_ctx* ctx, size_t bytes, void** d_ptr);
int b200_device_free(b200_ctx* ctx, void* d_ptr);
int b200_memcpy_h2d(b200_ctx* ctx, void* d_dst, const void* h_src, size_t bytes);
int b200_memcpy_d2h(b200_ctx* ctx, void* h_dst, const void* d_src, size_t bytes);
int b200_host_alloc_pinned(size_t bytes, void** h_ptr);
int b200_host_free_pinned(void* h_ptr);

#ifdef __cplusplus
}
#endif
#endif /* CANNY_B200_H */
