// front3.cu — the fused front kernel: u8 gray -> u8 class map (0 / 1 weak / 255 strong) for sm_100a.
//
// A CTA marches down one 128-column strip in 64-row slabs (one TMA box each) through linear shared-memory buffers whose tails are
// copied to the head; NMS runs on candidate pixels only.  In scalar FP32 the two blur passes are 60 of the 104 lane-instructions
// per pixel (DESIGN.md §4.1, per-phase budget), hence:
//
//   * BOTH BLUR PASSES RUN ON PACKED FP32 (sm_100's mul/add/fma .f32x2: two lanes' worth of IEEE operations per issue slot).  The
//     reference's rounding order (src/utils.cpp:41-47,56-62: every product rounded, every accumulation rounded, ascending taps)
//     forbids fused multiply-adds, and ptxas 12.9 contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 whatever the PTX says — unless
//     the two instructions disagree on flush-to-zero: the products are formed with mul.rn.FTZ.f32x2, the sums with add.rn.f32x2,
//     and a compiler that fused them would change results for subnormal products, so it must not (SASS: FMUL2.FTZ + FADD2, no
//     FFMA2 in the blur).  Flushing never happens here: every product is 0 or >= 2^-90 (the kernel is only used when the smallest
//     weight squared is >= 2^-90; front3_supports, GaussTables::tiny), so the values are those of plain mul.rn.
//       - row pass: a thread owns TWO rows (r, r+32) x 16 columns; a packed lane pair = the two rows at one column;
//       - column pass: a thread owns TWO adjacent columns x 18 blurred rows (16 Sobel rows); a pair = the two columns of one row,
//         loaded as one 64-bit word.
//   * Sobel in half precision, exactly: the column pass emits ONE word per pixel, half2(v, u) with v = B[r-1] + 2B[r] + B[r+1] and
//     u = B[r+1] - B[r-1] (integers of magnitude <= 1020, exact in fp16), so (gx, gy) of a pixel are two HFMA2 —
//     h[c+1] + h[c-1] * (-1, 1), then + h[c] * (0, 2) — and n = gx^2 + gy^2 is two mixed-precision FMAs with fp32 accumulation
//     (fma.rn.f32.f16, SASS FHFMA): 4 instructions per pixel instead of 7 integer ones.  The magnitude^2 plane, the thresholds, the
//     direction test and the truncated-magnitude comparison all work on these exact fp32 integers (n <= 2 * 1020^2 < 2^24).
//
// Used for compile-time radii without spill planes; everything else (run-time radius, `steps` planes, sigma so small that sums
// approach the subnormal range) stays on front.cu's kernel.
#include <cuda.h>
#include <string.h>

#include <algorithm>

#include "canny_math.h"
#include "exact_math.cuh"
#include "front_common.cuh"
#include "front_packed.cuh"
#include "internal.h"

namespace cb {
namespace f3 {

constexpr int kThreads = 256;
// rows per marching step (one TMA box) is the template parameter SLAB (64; 32 also builds, see launch_front3)
constexpr int kTC = 128;         // computed columns per strip (temp / VU lines); column j <-> image x = x0 - 2 + j
constexpr int kTW = kTC - 4;     // class-map columns produced per strip (Sobel + NMS eat 2 per side)
constexpr int kTempPitch = 132;  // floats; == 4 mod 32: the row pass's 128-bit stores (lane = row) hit 8 distinct bank groups
constexpr int kVuPitch = 132;    // int32 words; lane 31 of the last phase reads 4 words past column 127
// outputs per thread: SLAB/2 in the row pass, SLAB/2 VU rows = SLAB/2 + 2 blurred rows in the column pass

__host__ __device__ constexpr int in_pitch_for(int radius) {
    // bytes per staged input row: up to 15 leading bytes (the TMA box must start on a 16 B boundary of the image row: a tile
    // coordinate that is not a multiple of 16 bytes traps — tools/probes/tma_probe.cu), 128 + 2R needed ones; a multiple of 16
    // (TMA) and an ODD multiple so lane = row 128-bit loads spread over 8 distinct bank groups
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
// bgr: the kernel is fed interleaved B,G,R bytes.  A slab of them (slab rows x 3 * in_pitch bytes) lands by TMA in VU rows 2.. —
// free between the end of phase 3 and the next column pass — and is converted into ONE staged gray buffer, so the variant needs
// less shared memory than the gray one, not more.
__host__ __device__ constexpr SmemLayout smem_layout(int radius, int slab, bool bgr = false) {
    SmemLayout L{};
    int o = 0;
    L.in_off = o;   o += (bgr ? 1 : in_bufs_for(radius)) * slab * in_pitch_for(radius);
    o = (o + 127) & ~127;
    L.temp_off = o; o += temp_rows_for(radius, slab) * kTempPitch * 4;
    if (bgr) while ((o + 2 * kVuPitch * 4) & 127) o += 16;     // the TMA destination (VU row 2) on a 128 B boundary
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

using namespace pk;

// Predicated stores for phase 3b: nvcc turns `if (keep) *p = v;` into a branch around the store (and sinks the address arithmetic
// into it); four pixels per round would be eight short divergent regions.
__device__ __forceinline__ void st_u8_if(bool on, uint8_t* ptr, uint32_t v) {
    asm volatile("{ .reg .pred q;\n\tsetp.ne.b32 q, %0, 0;\n\t@q st.global.u8 [%1], %2; }" ::"r"((int)on), "l"(ptr), "r"(v) : "memory");
}
__device__ __forceinline__ void st_u32_if(bool on, int32_t* ptr, uint32_t v) {
    asm volatile("{ .reg .pred q;\n\tsetp.ne.b32 q, %0, 0;\n\t@q st.global.u32 [%1], %2; }" ::"r"((int)on), "l"(ptr), "r"(v) : "memory");
}
__device__ __forceinline__ void red_or_shared_if(bool on, uint32_t* ptr, uint32_t v) {
    asm volatile("{ .reg .pred q;\n\tsetp.ne.b32 q, %0, 0;\n\t@q red.shared.or.b32 [%1], %2; }" ::"r"((int)on), "r"(smem_u32(ptr)), "r"(v) : "memory");
}

// Register cap: 96 (no spills at any radius; the kernel takes 128 when left alone).  Two resident CTAs then leave a quarter of the
// register file free, so blocks of the small latency-bound hysteresis kernels of the PREVIOUS chunk (other stream) become
// resident next to them instead of waiting for a front CTA to retire: the front kernel alone gets 1.7 % slower, the chunk
// pipeline 2.3 % faster on the bench frames and 8 % faster on photographic content (112 / 104 / 88 / 80 measured too: 96 wins).
// PITCHED: the input or the class map has a row pitch / frame stride of its own, or the map is not word-aligned
// (b200_canny_batch_device_strided; layout_pitched()).  Dense layouts (the batch and host paths) keep the dense addressing, whose
// class and union-find offsets are one and the same, so their instruction stream and register allocation are those of the
// dense-only kernel.
// RAGGED: frames of different sizes in one launch (b200_canny_frames_device).  A 1-D grid over work items (p.ritems): the item names
// the frame, the strip and the row band, and the frame's descriptor (p.rframes) replaces in / in_pitch / width / height / cls /
// cls_pitch / cls_words and the slot base, with the pitched addressing.  Frames are whole images (in_row0 = plane_row0 = 0), so
// every border rule keys off the frame's own H and W.  TMA staging reads the frame's tensor map from the chunk's table in global
// memory.  Gray input, DIV 5 only.
template <int R, bool USE_TMA, int DIV, int SLAB, bool BGR = false, bool PITCHED = false, bool RAGGED = false>
#ifndef F3_MAXREG
#define F3_MAXREG 96
#endif
__global__ void __maxnreg__(SLAB == 64 ? F3_MAXREG : 64)
front3_kernel(const FrontParams p, const __grid_constant__ CUtensorMap tmap) {
    extern __shared__ __align__(1024) unsigned char smem[];
    constexpr int kSlab = SLAB;
    constexpr int kRunRow = 16;                // outputs per thread and row in the row pass: (SLAB/2 row pairs) x (128/16 segments) = 256 threads
    constexpr int kRunV = SLAB / 4;            // Sobel (VU) rows per thread in the column pass: 64 column pairs x 4 row groups = 256 threads
    constexpr int kRunCol = kRunV + 2;         // ... which need two more blurred rows
    constexpr int kVuRows = SLAB + 2;
    constexpr int kEntPerWarp = (SLAB / 8) * 64;
    static_assert(SLAB == 64, "row/column pass mappings are written for 64-row slabs");
    static_assert(2 * R + 2 <= SLAB, "the saved tail must not overlap the rows it is copied from");
    constexpr SmemLayout L = smem_layout(R, SLAB, BGR);
    constexpr int in_pitch = in_pitch_for(R);
    static_assert(!BGR || (USE_TMA && 3 * in_pitch == kVuPitch * 4 && R <= 9), "BGR staging: one TMA box row per VU row, 160 staged columns");
    static_assert(!RAGGED || (!BGR && !PITCHED && DIV == 5), "ragged launches: gray input, their own pitched addressing, DIV 5");
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
    // n-plane (exact fp32 integers, (SLAB+2) x 128 words): temp rows 0 .. SLAB-1.  The last 2R+2 temp lines (rows SLAB ..) — the ones
    // the next slab's column pass needs again — are NOT under it, so nobody has to save them between the column pass and phase 3:
    // the row pass of the next slab moves them to rows 0 .. 2R+1 (see there).
    float* s_np = s_temp;
    static_assert((SLAB + 2) * kNpPitch <= SLAB * kTempPitch, "the n-plane must end before the saved tail");

    const int tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    // latency path: the list-driven hysteresis kernel behind this one may be launched programmatically (HystParams::pdl); it parks
    // on griddepcontrol.wait until this grid has completed.  A no-op for ordinary launches.
#ifndef F3_NO_PDL_TRIGGER
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif

    // ---- which strip / band / frame ----
    RaggedItem item{};
    RaggedFrame fd{};
    if (RAGGED) {
        item = p.ritems[blockIdx.x];
        fd = p.rframes[item.frame];
    }
    const int strip = blockIdx.x, band = blockIdx.y, frame = RAGGED ? item.frame : blockIdx.z;
    const int x0 = RAGGED ? item.x0 : strip * kTW;
    const int rows_per_band = (p.out_rows + p.tiles_y - 1) / p.tiles_y;
    const int yb = RAGGED ? item.yb : p.out_row0 + band * rows_per_band;
    const int ye = RAGGED ? item.ye : min(p.out_row0 + p.out_rows, yb + rows_per_band);
    if (yb >= ye) return;
    const int W = RAGGED ? fd.width : p.width, H = RAGGED ? fd.height : p.height;
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
        // a tensor map in global memory, written by a host copy: acquire it for the tensor-map proxy before its first use (CUDA
        // programming guide, "Using TMA to transfer multi-dimensional arrays": scope .sys after a cudaMemcpy from the host)
        if (RAGGED) asm volatile("fence.proxy.tensormap::generic.acquire.sys [%0], 128;" ::"l"(p.rtmaps + frame) : "memory");
    }
    __syncthreads();

    u64 ws2[R + 1];
#pragma unroll
    for (int j = 0; j <= R; ++j) ws2[j] = pack2(s_w[R + j], s_w[R + j]);
    const float cnt_full = s_cnt[0], rcp_full = s_rcp[0];
    const u64 ncnt2 = pack2(-cnt_full, -cnt_full), rcp2 = pack2(rcp_full, rcp_full), divc2 = pack2(p.div_c, p.div_c);
    const u64 kBias2 = pack2(8388608.0f, 8388608.0f), kNegBias2 = pack2(-8388608.0f, -8388608.0f);
    const u64 kTwo2 = pack2(2.0f, 2.0f), kNegOne2 = pack2(-1.0f, -1.0f);
    const float lo2f = (float)p.lo2, hi2f = (float)p.hi2;   // thresholds on the exact fp32 magnitude^2 (n < 2^22; INT_MAX rounds to 2^31: never reached)
    // strips whose every computed column has all its taps inside the image divide by the constant count
    const bool x_interior = (x0 - 2 - R >= 0) && (x0 - 2 + kTC - 1 + R <= W - 1);
    // strips that contain image column -1 or W need the virtual Sobel columns patched in (see the patch pass)
    const bool x_edge = (x0 - 2 < 0) || (x0 - 2 + kTC - 1 >= W);

    const uint8_t* in_frame = RAGGED ? fd.in : p.in + (long long)frame * p.in_frame_stride;
    constexpr uint32_t slab_bytes = (uint32_t)(kSlab * in_pitch);

    constexpr int kInBufs = BGR ? 1 : in_bufs_for(R);
    auto issue_slab = [&](int k) {
        const int gy = in_y0 + k * kSlab;
        unsigned char* dst = s_in + (k % kInBufs) * slab_bytes;
        if (USE_TMA) {
            if (tid == 0) {
                const uint32_t bar = bar0 + 8 * (k % kInBufs);
                mbar_expect_tx(bar, slab_bytes);
                if (RAGGED) tma_load_3d(smem_u32(dst), p.rtmaps + frame, bar, in_x0, gy, 0);
                else tma_load_3d(smem_u32(dst), &tmap, bar, in_x0, gy - p.in_row0, frame);
            }
        } else {
            // generic staging (image pitch not a multiple of 16 B): byte loads, zero outside the image / buffer
            for (int i = tid; i < kSlab * in_pitch; i += kThreads) {
                const int r = i / in_pitch, c = i - r * in_pitch;
                const int y = gy + r, x = in_x0 + c;
                const int by = y - p.in_row0;
                unsigned char v = 0;
                if (y >= 0 && y < H && by >= 0 && by < (RAGGED ? H : p.in_rows) && x >= 0 && x < W)
                    v = in_frame[(long long)by * (RAGGED ? fd.in_pitch : PITCHED ? p.in_pitch : (long long)W) + x];
                dst[i] = v;
            }
        }
    };
    // ---- BGR input (cvtColor(frame, gray, COLOR_BGR2GRAY) of src/main.cpp:113, folded into the staging) ----
    // One thread issues the TMA of a slab of interleaved bytes (the tensor map sees 32-bit elements, 3W/4 per row; rows and columns
    // outside the image arrive as zeros, whose gray value is 0: the same zero fill the gray path relies on) into VU rows 2 .. SLAB+1.
    unsigned char* s_bgr = reinterpret_cast<unsigned char*>(s_vu + 2 * kVuPitch);
    auto issue_bgr = [&](int k) {   // one thread
        mbar_expect_tx(bar0, 3u * slab_bytes);
        tma_load_3d(smem_u32(s_bgr), &tmap, bar0, (in_x0 * 3) / 4, in_y0 + k * kSlab - p.in_row0, frame);
    };
    // OpenCV's 8-bit BGR2GRAY is fixed point: (B*3735 + G*19235 + R*9798 + 2^14) >> 15.  With doubled coefficients the result sits
    // in byte 2 of 2*(..) + 2^15 (< 2^24), and the three products of a pixel are two 16x8-bit dot products (dp2a) whichever way
    // its bytes straddle the 32-bit words.  A task = 8 pixels = 24 bytes -> two gray words; SLAB x 20 tasks = 5 per thread cover
    // the 160 staged columns the row pass reads.
    auto convert_bgr = [&]() {
        constexpr uint32_t cB = 2 * 3735, cG = 2 * 19235, cR = 2 * 9798;
        constexpr uint32_t kBG = cB | (cG << 16), kR0 = cR, k0B = cB << 16, kGR = cG | (cR << 16), kHalf = 32768;
        auto gray4 = [&](uint32_t w0, uint32_t w1, uint32_t w2) {   // B0 G0 R0 B1 | G1 R1 B2 G2 | R2 B3 G3 R3
            const uint32_t g0 = __dp2a_hi(kR0, w0, __dp2a_lo(kBG, w0, kHalf));
            const uint32_t g1 = __dp2a_lo(kGR, w1, __dp2a_hi(k0B, w0, kHalf));
            const uint32_t g2 = __dp2a_lo(kR0, w2, __dp2a_hi(kBG, w1, kHalf));
            const uint32_t g3 = __dp2a_hi(kGR, w2, __dp2a_lo(k0B, w2, kHalf));
            return __byte_perm(__byte_perm(g0, g1, 0x0062), __byte_perm(g2, g3, 0x0062), 0x5410);
        };
        constexpr int kHU = 20;
        static_assert((kSlab * kHU) % kThreads == 0 && kSlab * 16 % kThreads == 0 && kSlab * 4 == kThreads, "whole rounds");
#pragma unroll
        for (int t0 = 0; t0 < kSlab * kHU; t0 += kThreads) {
            // tasks 0..15 of a row belong to one half-warp (24 B apart: its 64-bit loads touch every bank once); the four left over
            // per row make up the last round
            const int r = t0 < kSlab * 16 ? (t0 + tid) >> 4 : tid >> 2;
            const int hu = t0 < kSlab * 16 ? (tid & 15) : 16 + (tid & 3);
            const uint2* src = reinterpret_cast<const uint2*>(s_bgr + r * (3 * in_pitch) + hu * 24);
            const uint2 a = src[0], b = src[1], c = src[2];
            *reinterpret_cast<uint2*>(s_in + r * in_pitch + hu * 8) = make_uint2(gray4(a.x, a.y, b.x), gray4(b.y, c.x, c.y));
        }
    };

    if (BGR) {
        // slab 0 is converted before the loop; from then on slab k+1 lands during the row pass of slab k and is converted right
        // after it (the single gray buffer is free by then), before the column pass takes the VU rows back
        if (tid == 0) issue_bgr(0);
        mbar_wait(bar0, 0);
        convert_bgr();
        __syncthreads();
        if (n_slabs > 1 && tid == 0) issue_bgr(1);
    } else if (USE_TMA) {
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
        if (BGR) {
            // the staged gray slab was converted in the previous iteration (or before the loop)
        } else if (USE_TMA) {
            mbar_wait(bar0 + 8 * (k % kInBufs), (uint32_t)((k / kInBufs) & 1));
        } else {
            issue_slab(k);
            __syncthreads();
        }
        const unsigned char* slab = s_in + (k % kInBufs) * slab_bytes;

        // ===================== phase 1: row blur, u8 -> f32 (src/utils.cpp:37-49), two column segments per thread =====================
        // thread = (slab row 32*(warp>>2) + lane, columns 16*sp .. +15 AND 64 + 16*sp .. +15, sp = warp & 3).  A pair = {column c,
        // column c + 64} of the row, and that is also how the temp buffer keeps a line: float 2c <-> column c, float 2c+1 <-> column
        // c + 64 (c < 64), so two outputs are one 128-bit store and the column pass loads a pair as one 64-bit word.
        {
            const int srow = 32 * (warp >> 2) + lane;
            const int sp = warp & 3;
            // The previous slab's last 2R+2 temp lines are needed again by this slab's column pass, at rows 0 .. 2R+1.  They sit exactly
            // where the threads of slab rows SLAB-T0 .. SLAB-1 are about to write, so each of those threads first moves the 32 floats it
            // is going to overwrite (no other thread touches them; the destination rows are only read after barrier (A)).
            if (k > 0 && srow >= kSlab - T0) {
                float4* dst = reinterpret_cast<float4*>(s_temp + (T0 + srow - kSlab) * kTempPitch + 2 * sp * kRunRow);
                const float4* src = dst + kSlab * kTempPitch / 4;
#pragma unroll
                for (int q = 0; q < (2 * kRunRow) / 4; ++q) dst[q] = src[q];
            }
            // needed bytes of a segment: [16*seg + lead, 16*seg + lead + 16 + 2R).  lead = 4*dq + DR with DR a compile-time constant
            // (x0 is a multiple of 4) and dq uniform over the CTA: load aligned 128-bit vectors, shift by dq WORDS with a uniform
            // switch, pick bytes with static selectors.
            constexpr int DR = (((-2 - R) % 4) + 4) % 4;
            constexpr int KW = (DR + kRunRow + 2 * R + 3) / 4;   // words holding the needed bytes
            constexpr int NV = (KW + 3 + 3) / 4;                 // vectors covering KW + 3 words
            static_assert((kTC - kRunRow) + 16 * NV <= in_pitch, "row pass would read past the staged line");
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
            // warps whose two segments touch the image border (1 in 4 of a border strip's warps) take the per-column weight sums.
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
        if (sparse) flush_pending();
        __syncthreads();  // (A) this slab's temp lines are complete; staged buffer k&1 is free again
        if (BGR) {
            if (k + 1 < n_slabs) {
                mbar_wait(bar0, (uint32_t)((k + 1) & 1));
                convert_bgr();
                __syncthreads();  // (A') the gray slab of the next iteration is staged; the VU rows belong to the column pass again
            }
        } else if (USE_TMA && k + kInBufs < n_slabs) {
            issue_slab(k + kInBufs);
        }

        // ===================== phase 2: column blur f32 -> int (src/utils.cpp:52-64) + vertical half of Sobel, two columns per thread ====
        // thread = (columns c = tid&63 and c + 64; row group tid>>6).  Blurred rows Bg(o) = I_k - R - 2 + 16*group + o, o = 0..17, from temp
        // buffer rows 16*group + o .. + 2R; VU rows Bg(1..16) go to VU buffer rows 2 + 16*group + (o-2).  A pair = the two columns, one
        // 64-bit word of the interleaved temp line.
        {
            const int c = tid & 63;
            const int group = tid >> 6;
            const float* tcol = s_temp + (kRunV * group) * kTempPitch + 2 * c;
            uint32_t* vcol = reinterpret_cast<uint32_t*>(s_vu) + (2 + kRunV * group) * kVuPitch + c;
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
        __syncthreads();  // (B) VU rows 2..65 complete; every read of the temp buffer is done

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
            __syncthreads();  // (B2) virtual columns patched
        }

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
            auto n_of_words = [&](const uint4 qa, const uint2 qb) -> float4 {
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
            auto n_of_row = [&](const int32_t* vrow) -> float4 {
                return n_of_words(*reinterpret_cast<const uint4*>(vrow), *reinterpret_cast<const uint2*>(vrow + 4));
            };
            if (cq_lo <= cq_hi) {
                // the two neighbour-only rows: warps 0 and 1
                if (warp < 2) {
                    const int q = warp == 0 ? cq_lo - 1 : cq_hi + 1;
                    const int y = y_base + q - 1;
                    float4 nq = make_float4(-1.f, -1.f, -1.f, -1.f);      // rows outside the image never suppress
                    if (y >= 0 && y < H) nq = n_of_row(s_vu + q * kVuPitch + 4 * lane);
                    *reinterpret_cast<float4*>(s_np + q * kNpPitch + 4 * lane) = nq;
                }
                const uint32_t zero_word = 0x01010101u * (uint32_t)p.cls_zero;
                // dense layouts: base aligned (layout_pitched), so word stores need a width that is a multiple of 4
                const bool words = RAGGED ? fd.cls_words != 0 : PITCHED ? p.cls_words != 0 : ((W & 3) == 0);
                const bool word_ok = words && lane < kTW / 4 && (x0 + 4 * lane + 3 < W);  // the aligned 32-bit store applies
                const bool tail_ok = !word_ok && lane < kTW / 4 && (x0 + 4 * lane < W);            // ragged right edge: byte stores
                const unsigned lt_mask = (1u << lane) - 1u;
                int q = cq_lo + ((warp - cq_lo) & 7);         // first class row of this warp (rows q = warp mod 8)
                const int32_t* vrow = s_vu + q * kVuPitch + 4 * lane;
                float* nrow = s_np + q * kNpPitch + 4 * lane;
                uint8_t* o = RAGGED ? fd.cls + (long long)(y_base + q - 1) * fd.cls_pitch + (x0 + 4 * lane)
                           : PITCHED ? p.cls + (long long)frame * p.cls_frame_stride + (long long)(y_base + q - 1 - p.plane_row0) * p.cls_pitch + (x0 + 4 * lane)
                                     : p.cls + (long long)frame * p.out_frame_stride + (long long)(y_base + q - 1 - p.plane_row0) * W + (x0 + 4 * lane);
                int ent = ((q - 1) << 6) | (lane << 1);
                const long long o_step = 8LL * (RAGGED ? fd.cls_pitch : PITCHED ? p.cls_pitch : (long long)W);
                // two copies of the loop so the store form is decided once, not per row: the aligned 32-bit store (every strip of
                // a class map whose base, pitch and frame stride are multiples of 4, except a ragged last strip) or byte stores
                auto class_row_nq = [&](const float4 nq, float* nr, int e16) {
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
                auto class_row = [&](const int32_t* vr, float* nr, int e16) { class_row_nq(n_of_row(vr), nr, e16); };
                // every class word starts out as "suppressed"; phase 3b overwrites the bytes of surviving pixels
                if (cq_lo == 1 && cq_hi == kSlab && words) {
                    // the common slab (all 64 class rows, word-aligned class map): the warp's eight rows unrolled, every address an
                    // immediate offset from the first row's (word_ok is false for the columns past a ragged right edge)
                    // The next row's Sobel words are fetched before this row's stores: the compiler cannot move a shared-memory load
                    // above the n-plane / list stores of the row before (it cannot prove they do not alias), and every row would
                    // otherwise start by waiting for its own loads.
                    uint4 qa = *reinterpret_cast<const uint4*>(vrow);
                    uint2 qb = *reinterpret_cast<const uint2*>(vrow + 4);
#pragma unroll
                    for (int i = 0; i < kSlab / 8; ++i) {
                        uint4 qa_next = qa;
                        uint2 qb_next = qb;
                        if (i + 1 < kSlab / 8) {
                            qa_next = *reinterpret_cast<const uint4*>(vrow + 8 * (i + 1) * kVuPitch);
                            qb_next = *reinterpret_cast<const uint2*>(vrow + 8 * (i + 1) * kVuPitch + 4);
                        }
                        class_row_nq(n_of_words(qa, qb), nrow + 8 * i * kNpPitch, ent + ((8 * i) << 6));
                        if (word_ok) *reinterpret_cast<uint32_t*>(o + i * o_step) = zero_word;
                        qa = qa_next; qb = qb_next;
                    }
                } else if (__all_sync(0xffffffffu, word_ok || lane >= kTW / 4)) {
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
        // A lane takes TWO list entries (four pixels) per round and everything up to the stores is branch-free, so the four
        // dependent chains (entry -> Sobel words -> direction -> neighbours -> truncated-magnitude test) overlap: with 16 warps
        // per SM this phase is bound by those chains, not by issue slots.
        {
            // PITCHED: the class byte is addressed through the caller's pitches; the union-find slot and the list index stay dense
            const long long out_off = RAGGED ? (long long)fd.base + (long long)y_base * W + (x0 - 2) + 1
                                             : (long long)frame * p.out_frame_stride + (long long)(y_base - p.plane_row0) * W + (x0 - 2) + 1;
            uint8_t* out_base = RAGGED ? fd.cls + (long long)y_base * fd.cls_pitch + (x0 - 2) + 1
                              : PITCHED ? p.cls + (long long)frame * p.cls_frame_stride + (long long)(y_base - p.plane_row0) * p.cls_pitch + (x0 - 2) + 1
                                        : p.cls + out_off;
            // ragged launches always hand over the list, also when minVal <= 0 makes every suppressed pixel weak (class cls_zero = 1):
            // then every class pixel that is not kept as strong is listed
            const bool zero_weak = RAGGED && p.cls_zero == 1;
            int32_t* par_base = p.parent + out_off;                           // only dereferenced when `sparse`
            const int idx_base = (int)out_off;                                // launch-relative pixel index of (class row 0, column j = 1)
            for (int i = lane; i < my_count; i += 64) {
                int ent[2];
                ent[0] = my_ent[i];
                const bool have1 = i + 32 < my_count;
                ent[1] = have1 ? my_ent[i + 32] : ent[0];
                float nc[2][2], na[2][2], nb[2][2];
                bool pass[2][2];
                int rel[2];
                uint8_t* orow[2];
                int32_t* prow[2];
                uint32_t* bits[2][2];
                uint32_t mask[2][2];
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int rr = ent[u] >> 6, c0 = 2 * (ent[u] & 63);        // pixels j = c0 + 1 and c0 + 2 of class row rr
                    rel[u] = rr * W + c0;                                      // < 2^31: rr < 64, W < 2^24
                    orow[u] = RAGGED ? out_base + ((long long)rr * fd.cls_pitch + c0)
                            : PITCHED ? out_base + ((long long)rr * p.cls_pitch + c0) : out_base + (unsigned)rel[u];
                    prow[u] = par_base + (unsigned)rel[u];
                    const int32_t* vrow = s_vu + (rr + 1) * kVuPitch + c0;     // VU words j-1 .. j+2 = c0 .. c0+3
                    const uint2 qa = *reinterpret_cast<const uint2*>(vrow);
                    const uint2 qb = *reinterpret_cast<const uint2*>(vrow + 2);
                    const uint32_t wd[4] = {qa.x, qa.y, qb.x, qb.y};
                    const float* nrow = s_np + (rr + 1) * kNpPitch + c0;       // n[j] lives at word j - 1
                    const float2 n2 = *reinterpret_cast<const float2*>(nrow);
                    nc[u][0] = n2.x; nc[u][1] = n2.y;
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const float n = nc[u][e];
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
                        na[u][e] = nrow[e + off];
                        nb[u][e] = nrow[e - off];
                        const int j = c0 + 1 + e;
                        pass[u][e] = (n >= lo2f) && (j >= 2) && (j <= kTC - 3);   // j = 1, j >= 126: neighbour-only columns
                        const int col = j - 2;                                // class column within the strip (bitmap: 4 words per row)
                        bits[u][e] = &s_bits[rr * 4 + ((col >> 5) & 3)];
                        mask[u][e] = 1u << (col & 31);
                    }
                }
                pass[1][0] = pass[1][0] && have1;
                pass[1][1] = pass[1][1] && have1;
#pragma unroll
                for (int u = 0; u < 2; ++u) {
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        // the reference compares truncated magnitudes: keep iff floor(sqrt(n_nb)) < floor(sqrt(n)) <=> n_nb < mag^2
                        // (n_nb < mag^2 <= n implies the plain local-maximum test; n = -1 of an out-of-image column gives NaN: false)
                        const float n = nc[u][e];
                        const float m2 = isqrt_sq_f(n);
                        const bool keep = pass[u][e] && (na[u][e] < m2) && (nb[u][e] < m2);
                        const bool strong = n >= hi2f;
                        st_u8_if(keep, orow[u] + e, strong ? 255u : 1u);
                        // hand-over to the list-driven hysteresis kernels: only WEAK pixels need any work there (a strong pixel is
                        // final; its neighbours find it through the class map).  The weak pixel gets its union-find slot (itself)
                        // and a bit in the slab's bitmap, from which the list entries are made once the slab is finished
                        const bool weak = RAGGED ? sparse && (keep ? !strong : (pass[u][e] && zero_weak)) : sparse && keep && !strong;
                        st_u32_if(weak, prow[u] + e, (uint32_t)(idx_base + rel[u] + e));
                        red_or_shared_if(weak, bits[u][e], mask[u][e]);
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
            // (inline PTX: nvcc turns a plain atomicAdd in divergent code into its warp-aggregated form, whose shuffle needs the
            // atomic's result at once — 2 % of the kernel's warp-time waited on that round trip)
            // ptxas does the same to a PTX atom on an address it can prove uniform, so the address carries threadIdx.z (always 0,
            // but a per-thread value)
            if (total && lane == 0)
                asm volatile("atom.global.add.u32 %0, [%1], %2;" : "=r"(pend_base) : "l"(p.kept_count + threadIdx.z), "r"((unsigned int)total) : "memory");
            pend_off = incl - cnt;
            // word tid <-> class row rr = tid >> 2, columns 32*(tid & 3) .. of the strip
            pend_g0 = RAGGED ? (int)((long long)fd.base + (long long)(y_base + (tid >> 2)) * W + x0 + 32 * (tid & 3))
                             : (int)((long long)frame * p.out_frame_stride + (long long)(y_base + (tid >> 2) - p.plane_row0) * W + x0 + 32 * (tid & 3));
        }
        // VU rows 64,65 (blurred-row neighbours of the next slab's first class rows) -> rows 0,1
        if (!BGR) {
            if (k + 1 < n_slabs) s_vu[(tid >> 7) * kVuPitch + (tid & 127)] = s_vu[(kSlab + (tid >> 7)) * kVuPitch + (tid & 127)];
        } else if (k + 1 < n_slabs && warp == 0) {
            // BGR: the slab after the next one is about to land on VU rows 2 .. SLAB+1, so ONE warp moves the two rows and then
            // issues that TMA (every warp's phase 3 reads are behind barrier (C))
            const uint4 a = *reinterpret_cast<const uint4*>(s_vu + kSlab * kVuPitch + 4 * lane);
            const uint4 b = *reinterpret_cast<const uint4*>(s_vu + (kSlab + 1) * kVuPitch + 4 * lane);
            *reinterpret_cast<uint4*>(s_vu + 4 * lane) = a;
            *reinterpret_cast<uint4*>(s_vu + kVuPitch + 4 * lane) = b;
            __syncwarp();
            if (k + 2 < n_slabs && lane == 0) {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                issue_bgr(k + 2);
            }
        }
        // the next iteration's barrier (A) orders this copy before phase 2 rewrites rows 2..65 and phase 3 reads rows 0,1
    }
    if (sparse) flush_pending();
}

}  // namespace f3

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
template <int R, bool USE_TMA, int DIV, int SLAB, bool BGR = false, bool PITCHED = false, bool RAGGED = false>
static int launch_one3(b200_ctx* ctx, cudaStream_t st, const FrontParams& p, const CUtensorMap& tmap, dim3 grid) {
    const f3::SmemLayout L = f3::smem_layout(R, SLAB, BGR);
    static bool configured[64] = {false};  // per instantiation, per device
    if (!configured[ctx->device & 63]) {
        CB_CUDA(cudaFuncSetAttribute(f3::front3_kernel<R, USE_TMA, DIV, SLAB, BGR, PITCHED, RAGGED>, cudaFuncAttributeMaxDynamicSharedMemorySize, L.total));
        CB_CUDA(cudaFuncSetAttribute(f3::front3_kernel<R, USE_TMA, DIV, SLAB, BGR, PITCHED, RAGGED>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
        configured[ctx->device & 63] = true;
    }
    {
        ProfScope ps(ctx, st, 0);
        f3::front3_kernel<R, USE_TMA, DIV, SLAB, BGR, PITCHED, RAGGED><<<grid, f3::kThreads, L.total, st>>>(p, tmap);
    }
    CB_CUDA(cudaGetLastError());
    ctx->launches++;
    return B200_OK;
}

// whether the kernel needs the pitched addressing: an input whose rows are not `width` bytes (3*width for B,G,R) apart, a class map
// whose rows are not `width` bytes apart or whose frames are not out_frame_stride bytes apart, or a class map off a 4-byte boundary
static bool layout_pitched(const FrontParams& p) {
    return p.in_pitch != (p.in_bgr ? 3LL : 1LL) * p.width || p.cls_pitch != p.width || p.cls_frame_stride != p.out_frame_stride ||
           (reinterpret_cast<uintptr_t>(p.cls) & 3) != 0;
}

template <int R, int SLAB>
static int launch_r3(b200_ctx* ctx, cudaStream_t st, const FrontParams& p, const CUtensorMap& tmap, dim3 grid, bool use_tma, int div) {
    // layouts with pitches of their own: one instantiation per staging form, the always-valid division
    if (layout_pitched(p)) return use_tma ? launch_one3<R, true, 5, SLAB, false, true>(ctx, st, p, tmap, grid)
                                       : launch_one3<R, false, 5, SLAB, false, true>(ctx, st, p, tmap, grid);
    if (use_tma) {
        if (div == 1) return launch_one3<R, true, 1, SLAB>(ctx, st, p, tmap, grid);
        if (div == 3) return launch_one3<R, true, 3, SLAB>(ctx, st, p, tmap, grid);
        return launch_one3<R, true, 5, SLAB>(ctx, st, p, tmap, grid);
    }
    // generic staging (odd widths) is not a throughput path: one instantiation, the always-valid division
    return launch_one3<R, false, 5, SLAB>(ctx, st, p, tmap, grid);
}

// interleaved B,G,R input: TMA only, the three exact divisions
template <int R, int SLAB>
static int launch_r3_bgr(b200_ctx* ctx, cudaStream_t st, const FrontParams& p, const CUtensorMap& tmap, dim3 grid, int div) {
    if (layout_pitched(p)) return launch_one3<R, true, 5, SLAB, true, true>(ctx, st, p, tmap, grid);
    if (div == 1) return launch_one3<R, true, 1, SLAB, true>(ctx, st, p, tmap, grid);
    if (div == 3) return launch_one3<R, true, 3, SLAB, true>(ctx, st, p, tmap, grid);
    return launch_one3<R, true, 5, SLAB, true>(ctx, st, p, tmap, grid);
}

// The kernel is built for these half-windows, and its packed blur flushes subnormal products, so it takes only weights whose
// smallest square is >= 2^-90 (GaussTables::tiny).
bool front3_supports(const GaussTables& g) {
    if (g.tiny) return false;
    switch (g.radius) {
        case 2: case 3: case 5: case 6: case 9: case 15: return true;
        default: return false;
    }
}

// The fused-conversion variant exists for half-windows up to 9 (one staged input buffer is what larger ones use anyway) and needs
// the TMA path: a width that is a multiple of 16 (whole 32-bit elements per staged row), base, row pitch and frame stride on 16 B
// boundaries.
bool front3_bgr_supports(const GaussTables& g, const FrontParams& p) {
    static const bool tma_env_off = [] { const char* e = getenv("B200_CANNY_NO_TMA"); return e && e[0] == '1'; }();
    static const bool fuse_off = [] { const char* e = getenv("B200_CANNY_BGR_FUSED"); return e && e[0] == '0'; }();
    return front3_supports(g) && g.radius <= 9 && !tma_env_off && !fuse_off && (p.width % 16 == 0) && input_tma_layout_ok(p);
}

// Bands per frame: every band pays 2R+4 warm-up rows and is processed in 64-row slabs, so pick the band count
// that minimises (slabs per band) x (waves of CTAs) — enough CTAs to fill the machine, few enough that the
// warm-up and the last partly-filled slab stay small.
static int choose_bands3(const b200_ctx* ctx, int out_rows, int strips, int frames, int radius, int slab) {
    const int slots = (slab == 64 ? 2 : 4) * (ctx->sm_count > 0 ? ctx->sm_count : 148);
    const long long per_band = (long long)strips * frames;
    int best = 1;
    double best_cost = 1e300;
    // bands down to 32 rows: a 256-row frame cut into 6 bands is ONE slab per CTA (43 + 2R + 4 rows) instead of two (256 x 256 frame:
    // 34 -> 26 us); large frames never get there (more CTAs than slots means more waves)
    const int max_bands = out_rows / 32 > 0 ? out_rows / 32 : 1;
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

// ---- ragged chunks ----
// Band policy: one class-row band height T for the whole chunk, every frame cut into ceil(H / T) equal bands, so every CTA marches
// about the same rows (T plus the 2R+4 warm-up rows) whatever its frame's size: large frames get more bands and the CTAs of a chunk
// take similar times.  T is chosen from the heights that fill whole 64-row slabs (64k - 2R - 4) by the list-scheduling estimate
// of the chunk's time: slab-steps of all CTAs over the 2 x SMs CTA slots, plus the longest CTA (the last wave's tail); the largest
// T within 0.1 % of the best wins, since more bands cost warm-up rows.  Measured with this policy on one B200 (1000 W), 2000 frames of
// 320x240 .. 1920x1080 (tools/ragged_probe.py, profiles/r04_ragged_probe.jsonl): 113 Gpix/s for the C call on "shapes" content
// against 281 Gpix/s for the same pixels as uniform 4K frames and 21 Gpix/s for one call per frame; other policies not measured.
int ragged_band_rows3(const b200_ctx* ctx, const int* heights, const int* widths, int n, int radius) {
    const long long slots = 2LL * (ctx->sm_count > 0 ? ctx->sm_count : 148);
    const int warm = 2 * radius + 4, slab = 64;
    int max_h = 0;
    for (int i = 0; i < n; ++i) max_h = std::max(max_h, heights[i]);
    int best = max_h;
    double best_cost = 1e300;
    for (int k = (max_h + warm + slab - 1) / slab; k >= 1; --k) {
        const int t = std::min(max_h, std::max(16, slab * k - warm));
        long long steps = 0;
        int longest = 0;
        for (int i = 0; i < n; ++i) {
            const int bands = (heights[i] + t - 1) / t;
            const int rows = (heights[i] + bands - 1) / bands;
            const int slabs = (rows + warm + slab - 1) / slab;
            steps += (long long)slabs * bands * ((widths[i] + f3::kTW - 1) / f3::kTW);
            longest = std::max(longest, slabs);
        }
        const double cost = (double)steps / (double)slots + longest;
        if (cost < best_cost * 0.999) { best_cost = cost; best = t; }
    }
    return best;
}

void ragged_items3(int frame, int height, int width, int band_rows, std::vector<RaggedItem>& items) {
    const int bands = (height + band_rows - 1) / band_rows;
    const int rows = (height + bands - 1) / bands;
    for (int b = 0; b < bands; ++b) {
        const int yb = b * rows, ye = std::min(height, yb + rows);
        if (yb >= ye) break;
        for (int x0 = 0; x0 < width; x0 += f3::kTW) items.push_back(RaggedItem{frame, x0, yb, ye});
    }
}

// The tensor map of one ragged frame (3-D like the uniform maps, one frame deep); *use_tma is false when its base or pitch is not a
// multiple of 16 bytes (the frame then takes the byte-load staging)
int ragged_tensor_map3(const uint8_t* in, long long pitch, int height, int width, int radius, CUtensorMap_st* tmap, bool* use_tma) {
    FrontParams p;
    memset(&p, 0, sizeof(p));
    p.in = in; p.in_pitch = pitch; p.in_frame_stride = (long long)height * pitch; p.in_rows = height; p.width = width; p.n_frames = 1;
    return make_input_tensor_map(p, f3::in_pitch_for(radius), 64, tmap, use_tma);
}

template <int R>
static int launch_r3_ragged(b200_ctx* ctx, cudaStream_t st, const FrontParams& p, const CUtensorMap& tmap, dim3 grid, bool use_tma) {
    return use_tma ? launch_one3<R, true, 5, 64, false, false, true>(ctx, st, p, tmap, grid)
                   : launch_one3<R, false, 5, 64, false, false, true>(ctx, st, p, tmap, grid);
}

int launch_front3_ragged(b200_ctx* ctx, cudaStream_t st, const FrontParams& p_in, int n_items, bool use_tma) {
    if (n_items <= 0) return B200_OK;
    FrontParams p = p_in;
    p.div_c = ctx->gauss.div_c;
    CUtensorMap tmap;   // unused: every frame's map is in the chunk's table
    memset(&tmap, 0, sizeof(tmap));
    const dim3 grid(n_items);
    ctx->front_fast++;
    switch (p.radius) {
        case 2: return launch_r3_ragged<2>(ctx, st, p, tmap, grid, use_tma);
        case 3: return launch_r3_ragged<3>(ctx, st, p, tmap, grid, use_tma);
        case 5: return launch_r3_ragged<5>(ctx, st, p, tmap, grid, use_tma);
        case 6: return launch_r3_ragged<6>(ctx, st, p, tmap, grid, use_tma);
        case 9: return launch_r3_ragged<9>(ctx, st, p, tmap, grid, use_tma);
        case 15: return launch_r3_ragged<15>(ctx, st, p, tmap, grid, use_tma);
        default: break;
    }
    set_error("front3 kernel not built for radius %d", p.radius);
    return B200_ERR_UNSUPPORTED;
}

int launch_front3(b200_ctx* ctx, cudaStream_t st, const FrontParams& p_in) {
    FrontParams p = p_in;
    const int radius = p.radius;
    const int strips = (p.width + f3::kTW - 1) / f3::kTW;
    p.tiles_x = strips;
    // 64-row slabs, 2 CTAs per SM.  The kernel also builds with 32-row slabs (4 CTAs per SM, 63 registers; ncu: issue slots 74 %
    // busy instead of 63 %) but then executes 19 % more instructions (shorter runs share fewer products, twice the tail copies and
    // per-slab set-up) and ends up 2-3 % slower on the 4K batch, so only the 64-row form is instantiated.
    constexpr int slab = 64;
    static const int bands_env = [] { const char* e = getenv("B200_CANNY_BANDS"); return e ? atoi(e) : 0; }();   // experiments
    if (p.tiles_y <= 0 && bands_env > 0 && p.out_rows / bands_env >= 1) p.tiles_y = bands_env;
    if (p.tiles_y <= 0) p.tiles_y = choose_bands3(ctx, p.out_rows, strips, p.n_frames, radius, slab);
    dim3 grid(strips, p.tiles_y, p.n_frames);
    CUtensorMap tmap;
    bool use_tma = false;
    const int div3 = ctx->gauss.div_mode;
    p.div_c = ctx->gauss.div_c;
    if (p.in_bgr) {
        if (!front3_bgr_supports(ctx->gauss, p)) { set_error("fused BGR input needs width %% 16 == 0, a 16-byte aligned base, row pitch and frame stride and a half-window <= 9"); return B200_ERR_UNSUPPORTED; }
        CB_TRY(make_bgr_tensor_map(p, 3 * f3::in_pitch_for(radius) / 4, slab, &tmap));
        switch (radius) {
            case 2: return launch_r3_bgr<2, 64>(ctx, st, p, tmap, grid, div3);
            case 3: return launch_r3_bgr<3, 64>(ctx, st, p, tmap, grid, div3);
            case 5: return launch_r3_bgr<5, 64>(ctx, st, p, tmap, grid, div3);
            case 6: return launch_r3_bgr<6, 64>(ctx, st, p, tmap, grid, div3);
            default: return launch_r3_bgr<9, 64>(ctx, st, p, tmap, grid, div3);
        }
    }
    CB_TRY(make_input_tensor_map(p, f3::in_pitch_for(radius), slab, &tmap, &use_tma));
    switch (radius) {
        case 2: return launch_r3<2, 64>(ctx, st, p, tmap, grid, use_tma, div3);
        case 3: return launch_r3<3, 64>(ctx, st, p, tmap, grid, use_tma, div3);
        case 5: return launch_r3<5, 64>(ctx, st, p, tmap, grid, use_tma, div3);
        case 6: return launch_r3<6, 64>(ctx, st, p, tmap, grid, use_tma, div3);
        case 9: return launch_r3<9, 64>(ctx, st, p, tmap, grid, use_tma, div3);
        case 15: return launch_r3<15, 64>(ctx, st, p, tmap, grid, use_tma, div3);
        default: break;
    }
    set_error("front3 kernel not built for radius %d", radius);
    return B200_ERR_UNSUPPORTED;
}

}  // namespace cb
