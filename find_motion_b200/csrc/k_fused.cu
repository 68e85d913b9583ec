// K1: fused, time-blocked stencil + background kernel (full-resolution mode, Gaussian k <= 5).
//
// One CTA owns a 128 x FT_H pixel tile of one stream and walks the T frames of the call in order:
//   BGR tile + 2 px halo --(TMA, double buffered)--> gray bytes in shared memory
//   --> horizontal 8.8 fixed-point Gaussian pass as a banded (Toeplitz) u8 x u8 matrix product on the
//       tensor cores (IMMA.16832.U8: A = 16 gray rows x 32 columns via LDSM, B = the taps), sums packed
//       2x16-bit into shared memory
//   --> vertical pass on the packed lanes in registers (sliding 5-row window)
//   --> polygon mask --> bg8 = rne(f32(bg)), |blur - bg8| > threshold --> bit-packed mask out
//   --> bg = fma(bg, 1-alpha, rn(blur*alpha))
// Each thread keeps the float64 background of its 16 pixels (one row, two 8-pixel segments) in registers across all T frames,
// so the background costs one 16 B/px HBM round trip per call instead of per frame.
// Replaces blur_frame + mask_off_areas + find_diff's diff/threshold/accumulateWeighted
// (find_motion/find_motion.py:487-494, 619-635, 246-257, 651-659; SURVEY.md A.2-A.7).
//
// Packed arithmetic: for k in {1,3,5} the taps are g*[b0,b1,b2,b1,b0] with g >= 16, so the
// horizontal sums (<= 255*256/g) and the vertical sums (<= 255*(256/g)^2 <= 65280) fit 16 bits
// and two pixels share one 32-bit IMAD; (ver + 32768) >> 16 == (v' + round) >> shift exactly.
#include <cuda.h>

#include "fm_common.cuh"

#define FT_W 128
#ifndef FT_H
#define FT_H 32            // tile height; a thread owns one row x 16 pixels, a warp 4 rows x 128 columns
#endif
#define FT_PX 16           // pixels (and float64 background values) per thread
#define FUSED_WARPS (FT_H / 4)
#define FG_WORDS 36        // gray words per shared row: cols x0-4 .. x0+139 (18 units of 8 pixels)
#define FG_ROWS (FT_H + 4) // rows y0-2 .. y0+FT_H+1
#define FH_MB ((FG_ROWS + 15) / 16)     // 16-row blocks of the tensor-core pass
#define FH_ROWS (16 * FH_MB)            // rows of the shared planes (the rows past FG_ROWS are scratch: no row guards)
#ifndef FUSED_MIN_CTAS
#define FUSED_MIN_CTAS (1024 / (8 * FT_H))      // 64 registers per thread: 1024 resident threads per SM
#endif
#define FH_WORDS 68         // packed horizontal sums per shared row: 64 pixel pairs + 4 (bank spread for the D-fragment stores)
#define FUSED_THREADS (8 * FT_H)
#define RAW_PITCH 432      // bytes per staged BGR row: bytes x0*3-16 .. x0*3+415 (TMA box of 108 u32)
#define RAW_BYTES (RAW_PITCH * FG_ROWS)                 // bytes one TMA box delivers
#define RAW_STAGE ((RAW_BYTES + 127) / 128 * 128)        // stage stride (TMA destinations are 128 B aligned)
// NV12 (FM_FLAG_NV12): a stage holds two boxes, the luma rows y0-2 .. y0+FT_H+1 and the UV rows (y0-2)/2 .. that cover
// them, each of bytes x0-16 .. x0+143 (40 u32: the box start must be 16 B aligned in global memory)
#define NV_PITCH 160
#define NV_Y_BYTES (NV_PITCH * FG_ROWS)                  // 5760 = 45 * 128: the UV box lands 128 B aligned after it
#define NV_BYTES (NV_Y_BYTES + NV_PITCH * FG_ROWS / 2)   // <= RAW_BYTES: both fit the BGR stage
// Gray (FM_FLAG_GRAY): a stage holds the luma box alone, rows y0-2 .. y0+FT_H+1 of the caller's frame; no conversion
// Four-byte pixels (FM_FLAG_ALPHA): a stage holds one box of the tile's pixels x0-4 .. x0+139 as u32 words, 576-byte
// rows; one 16-byte word of 4 pixels is one gray word, no realignment.  Two such stages make the CTA's shared memory
// FUSED_SMEM_A4 = 61,456 B (BGR: 51,216 B), so three CTAs fit an SM instead of four (DESIGN §4.9)
#define A4_PITCH 576
#define A4_BYTES (A4_PITCH * FG_ROWS)
#define A4_STAGE ((A4_BYTES + 127) / 128 * 128)
enum { FUSED_BGR = 0, FUSED_NV12 = 1, FUSED_GRAY = 2, FUSED_RGB = 3, FUSED_BGRA = 4, FUSED_RGBA = 5 };
// source format of k_fused (RGB, RGBA: the gray weights of bytes 0 and 2 swapped)

struct FusedParams {
    int T, w, h, wpr;           // T = frames per stream of the call
    const int *nvalid;          // [S] real frames of each stream in this call (ragged batches), <= T
    int tilesX, tilesY;
    double *bg;                 // [S][tiles][8 warps][8 pairs][32 lanes] double2 (thread-private, coalesced)
    const uint32_t *maskbits;   // [S][h][wpr]
    uint32_t *tbits;            // [S][T][flatwords]  (row-padded == flat because w % 32 == 0)
    size_t flatwords;
    const int *bg_in;           // [S] bg_valid slot of this call: the stream has a background
    int *bg_out;                // [S] bg_valid slot of the next call
    int *clear_ff;              // filled with -1 after the wait at the end: the other range slot and `any`
    int *clear_zero;            //   ... and zeroed: the contour counters
    int n_ff, n_zero;
    unsigned long long *stamp;  // front-end group stamps of the call (null: timing off)
    int b0, b1, b2, shift, rnd; // taps / g, and the rounding of the final shift (packed in both lanes)
    int threshold;
    double alpha, beta;
    int qoff; uint32_t nthr2; double nC;    // fm_temporal_px's constants: read from the constant bank, not rebuilt per frame
    uint8_t *gray_out, *blur_out;   // [S][T][h][w], only with KEEP
    int *rawrange;                  // [S][T][2] (max y, max h-1-y) of rows with pixels above threshold
    uint4 bfr[32];                  // per lane: B fragments of the horizontal pass (fused_bfr)
#ifdef FM_K1_PROF
    long long *prof;                // development aid: [K1_NPROF] cycles per phase summed over CTAs (thread 0), [K1_NPROF] frames
#endif
};

// Development aid (build with -DFM_K1_PROF, tools/k1_prof.py): clock64 of thread 0 of every CTA per phase of the frame
// loop.  A phase that ends in a barrier includes the wait at it.  Off by default: the shipped code has no trace of it.
enum { K1_WAIT, K1_GRAY, K1_BORDER, K1_HORIZ, K1_VERT, K1_TAIL, K1_NPROF };
#ifdef FM_K1_PROF
#define K1_PROF(slot)                                \
    do {                                             \
        if (tid == 0) {                              \
            const long long now_ = clock64();        \
            k1_prof[slot] += now_ - k1_prof_t;       \
            k1_prof_t = now_;                        \
        }                                            \
    } while (0)
#else
#define K1_PROF(slot) do {} while (0)
#endif

// B fragments of the horizontal pass (constant per call): the banded tap matrix for the two 8-column output blocks of a
// 32-byte window.  Output column n of block nb is gray byte 4 + 16 j + 8 nb + n of its row, window byte k is gray byte
// 16 j + k, so the tap index is k - n - 8 nb - 2 (taps b0 b1 b2 b1 b0).  Lane = 4 g + tq holds bytes k = 16 r + 4 tq + i of
// column n = g: words (nb, r) = (0,0) (0,1) (1,0) (1,1).
static void fused_bfr(FusedParams &p) {
    for (int lane = 0; lane < 32; lane++) {
        const int g = lane >> 2, tq = lane & 3;
        uint32_t v[4];
        for (int nb = 0; nb < 2; nb++)
            for (int r = 0; r < 2; r++) {
                uint32_t x = 0;
                for (int i = 0; i < 4; i++) {
                    const int idx = 16 * r + 4 * tq + i - g - 8 * nb - 2;
                    const int tap = (idx == 2) ? p.b2 : (idx == 1 || idx == 3) ? p.b1 : (idx == 0 || idx == 4) ? p.b0 : 0;
                    x |= (uint32_t)tap << (8 * i);
                }
                v[2 * nb + r] = x;
            }
        p.bfr[lane] = make_uint4(v[0], v[1], v[2], v[3]);
    }
}

// 8x8 transpose of 4-bit elements across the 8 lanes of a lane octet: in: lane i holds e[r] (nibble r)
// = bits of row r; out: lane r holds nibble i = bits of lane i  -> a 32-pixel row word.
__device__ __forceinline__ uint32_t nibble_transpose8(uint32_t x, int lane) {
    uint32_t o = __shfl_xor_sync(0xffffffffu, x, 4);
    x = (lane & 4) ? ((o >> 16) | (x & 0xFFFF0000u)) : ((x & 0x0000FFFFu) | (o << 16));
    o = __shfl_xor_sync(0xffffffffu, x, 2);
    x = (lane & 2) ? (((o >> 8) & 0x00FF00FFu) | (x & 0xFF00FF00u)) : ((x & 0x00FF00FFu) | ((o & 0x00FF00FFu) << 8));
    o = __shfl_xor_sync(0xffffffffu, x, 1);
    x = (lane & 1) ? (((o >> 4) & 0x0F0F0F0Fu) | (x & 0xF0F0F0F0u)) : ((x & 0x0F0F0F0Fu) | ((o & 0x0F0F0F0Fu) << 4));
    return x;
}

// a + b + c as one IADD3: written as C, the compiler adds c after the products of the vertical pass, one add more per word
__device__ __forceinline__ uint32_t add3(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("add.u32 %0, %1, %2;\n\tadd.u32 %0, %0, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

// One thread: 5 rows of packed horizontal sums in -> ONE output row x 16 pixels (two segments of 8 consecutive pixels, 64
// pixels apart, so that the 128-bit shared loads of a quarter-warp are contiguous): vertical pass, mask, threshold bits,
// background update.  The 16 threshold bits of a thread are two bytes of the bit plane: no transposition across lanes.
// INIT: first frame of a stream (ref_frame = blur.astype(float));  MASKED: the warp has masked pixels (M bit j = pixel j);
// SH8: k = 5 (taps 1,4,6,4,1 compiled in, final shift 8 done by byte selection).
template <bool KEEP, bool SAFE, bool INIT, bool MASKED, bool SH8>
__device__ __forceinline__ uint32_t fused_rows(const uint32_t *shw, double (&bg)[FT_PX], uint32_t M, const FusedParams &p,
                                               uint8_t *blur_out, uint32_t vmask) {
    const uint32_t b0 = p.b0, b1 = p.b1, b2 = p.b2;
    uint32_t bits = 0;
#pragma unroll
    for (int seg = 0; seg < 2; seg++) {
        // rows y-2 .. y+2 of the segment, pixels (0,1) (2,3) (4,5) (6,7) per 128-bit load, 16 bits each; accumulated as they
        // arrive (outer rows, then the +-1 rows, then the centre) to keep the live registers low
        const uint32_t *sp = shw + 32 * seg;
        uint32_t v[4];             // the two pixels of a pair in bits [0,8) and [16,24) (SH8: in bytes 1 and 3)
        {
            const uint4 r0 = *reinterpret_cast<const uint4 *>(sp), r4 = *reinterpret_cast<const uint4 *>(sp + 4 * FH_WORDS);
            const uint32_t rn = SH8 ? 0x00800080u : (uint32_t)p.rnd;
            if (SH8) { v[0] = add3(r0.x, r4.x, rn); v[1] = add3(r0.y, r4.y, rn); v[2] = add3(r0.z, r4.z, rn); v[3] = add3(r0.w, r4.w, rn); }
            else { v[0] = b0 * (r0.x + r4.x) + rn; v[1] = b0 * (r0.y + r4.y) + rn; v[2] = b0 * (r0.z + r4.z) + rn; v[3] = b0 * (r0.w + r4.w) + rn; }
        }
        {
            const uint4 r1 = *reinterpret_cast<const uint4 *>(sp + FH_WORDS), r3 = *reinterpret_cast<const uint4 *>(sp + 3 * FH_WORDS);
            const uint32_t m1 = SH8 ? 4u : (uint32_t)b1;
            v[0] += m1 * (r1.x + r3.x); v[1] += m1 * (r1.y + r3.y); v[2] += m1 * (r1.z + r3.z); v[3] += m1 * (r1.w + r3.w);
        }
        {
            const uint4 r2 = *reinterpret_cast<const uint4 *>(sp + 2 * FH_WORDS);
            const uint32_t m2 = SH8 ? 6u : (uint32_t)b2;
            v[0] += m2 * r2.x; v[1] += m2 * r2.y; v[2] += m2 * r2.z; v[3] += m2 * r2.w;
        }
        if (!SH8) {
#pragma unroll
            for (int j = 0; j < 4; j++) v[j] = (v[j] >> p.shift) & 0x00FF00FFu;
        }
        if (KEEP && (vmask & (1u << seg))) {
            uint2 o;
            if (SH8) { o.x = __byte_perm(v[0], v[1], 0x7531); o.y = __byte_perm(v[2], v[3], 0x7531); }
            else { o.x = __byte_perm(v[0], v[1], 0x6420); o.y = __byte_perm(v[2], v[3], 0x6420); }
            const uint32_t mk = (M >> (8 * seg)) & 0xFFu;
            o.x = fm_clear_masked4(o.x, mk & 0xFu);
            o.y = fm_clear_masked4(o.y, (mk >> 4) & 0xFu);
            *reinterpret_cast<uint2 *>(blur_out + 64 * seg) = o;
        }
#pragma unroll
        for (int c = 0; c < 8; c++) {
            const int idx = 8 * seg + c;
            uint32_t sv = SH8 ? __byte_perm(v[c >> 1], 0, (c & 1) ? 0x4443 : 0x4441)
                              : ((c & 1) ? (v[c >> 1] >> 16) : (v[c >> 1] & 0xFFFFu));
            if (MASKED && (M & (1u << idx))) sv = 0;          // mask_off_areas paints BLACK into blur
            fm_temporal_px<SAFE, INIT>(sv, bg[idx], bits, p.threshold, p.qoff, p.nthr2, p.alpha, p.beta, p.nC);
        }
    }
    return __brev(bits) >> (32 - FT_PX);      // the first pixel was pushed first: bit idx = pixel idx
}

// Frame t of stream s has pixels above threshold in the 4 rows y .. y+3 of a warp: widen that frame's rawrange.
__device__ __forceinline__ void rawrange_hit(const FusedParams &p, int s, int t, int y) {
    int *rr = p.rawrange + 2 * ((size_t)s * p.T + t);
    atomicMax(rr, min(y + 3, p.h - 1));
    atomicMax(rr + 1, p.h - 1 - y);
}

// End of every CTA of K1.  K1 of call i+1 is launched as a programmatic dependent of k_decide of call i (fm_host.cu), so
// it starts while the contour stage of call i still runs and may do all its own work then: it reads only the frames,
// the mask, n_valid, its background and bg_valid, and writes the other tflat / rawrange slot.  The wait here keeps the
// chain transitive: K1(i+1) cannot complete before decide(i) has, and decide(i) waits for the labelling kernels of
// call i, which wait for K1(i).  So the contour stage of call i+1 (an ordinary launch after K1(i+1)) never runs ahead
// of call i, and K1(i+2) never writes the slot the contour stage of call i reads.  Past the wait, the contour stage of
// call i is complete, so this is where the per-call result slots are cleared: the range slot call i used (call i+1
// uses it next), `any` and the counters, which the contour stage of call i+1 fills.
__device__ __forceinline__ void fused_exit(const FusedParams &p) {
    fm_stamp_end(p.stamp);                       // this CTA's own work is done; the wait below is not the front end's
    fm_wait_predecessor();
    const int nthreads = gridDim.x * gridDim.y * gridDim.z * FUSED_THREADS;
    for (int i = ((blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * FUSED_THREADS + threadIdx.x;
         i < p.n_ff + p.n_zero; i += nthreads) {
        if (i < p.n_ff) p.clear_ff[i] = -1;
        else p.clear_zero[i - p.n_ff] = 0;
    }
}

// 4 luma bytes of one row and the chroma of their two 2x2 blocks -> 4 gray bytes (fm_nv12_gray: cv2's COLOR_YUV2BGR_NV12)
__device__ __forceinline__ uint32_t nv12_gray4(uint32_t y4, const FmChroma &c0, const FmChroma &c1) {
    return fm_nv12_gray(y4 & 0xFFu, c0) | (fm_nv12_gray((y4 >> 8) & 0xFFu, c0) << 8) |
           (fm_nv12_gray((y4 >> 16) & 0xFFu, c1) << 16) | (fm_nv12_gray(y4 >> 24, c1) << 24);
}

// NV12: frames arrive as the two boxes above (tmap = luma plane, tmap_uv = chroma plane); otherwise tmap_uv is unused.
// GRAY: tmap = the gray frames as one plane of W-byte rows (the NV12 luma box)
template <bool KEEP, bool SAFE, int SRC>
__global__ void __launch_bounds__(FUSED_THREADS, FUSED_MIN_CTAS) k_fused(const __grid_constant__ CUtensorMap tmap, FusedParams p,
                                                                         const __grid_constant__ CUtensorMap tmap_uv) {
    extern __shared__ __align__(128) unsigned char fsm[];
    constexpr bool A4 = SRC == FUSED_BGRA || SRC == FUSED_RGBA, RGBO = SRC == FUSED_RGB || SRC == FUSED_RGBA;
    constexpr int STG = A4 ? A4_STAGE : RAW_STAGE;
    unsigned char *raw = fsm;                                                  // [2][STG] staged BGR rows (TMA)
    uint32_t *sg = reinterpret_cast<uint32_t *>(fsm + 2 * STG);              // [FH_ROWS][FG_WORDS] gray bytes (FG_ROWS used)
    uint32_t *sh = sg + FH_ROWS * FG_WORDS;                                  // [FH_ROWS][FH_WORDS] packed horizontal sums
    uint64_t *bars = reinterpret_cast<uint64_t *>(sh + FH_ROWS * FH_WORDS);
    constexpr bool NV12 = SRC == FUSED_NV12, GRAY = SRC == FUSED_GRAY;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int s = blockIdx.z;
    const int tx = blockIdx.x, ty = blockIdx.y, tile = ty * p.tilesX + tx;
    const int x0 = tx * FT_W, y0 = ty * FT_H;
    const int w = p.w, h = p.h;
    const bool border = (x0 == 0) || (x0 + FT_W >= w) || (y0 == 0) || (y0 + FT_H >= h);
    fm_stamp_start(p.stamp);
    // not StreamState::has_bg: k_decide of the previous call may still be running and writes it
    const bool has_bg = p.bg_in[s] != 0;
    const int Ts = min(p.T, __ldg(p.nvalid + s));            // frames of this stream that are real
    if (tid == 0 && tx == 0 && ty == 0) p.bg_out[s] = has_bg || Ts > 0;
    if (Ts <= 0) {
        fused_exit(p);
        return;
    }

    // this thread's pixels: row y0 + tid / 8, columns x0 + 8 (tid % 8) .. + 7 and the same 64 pixels further right
    const int trow = tid >> 3, xg = tid & 7;
    const int px = x0 + 8 * xg, py = y0 + trow;
    double2 *bgt = reinterpret_cast<double2 *>(p.bg) +
                   ((((size_t)s * p.tilesX * p.tilesY + tile) * FUSED_WARPS + warp) * (FT_PX / 2)) * 32 + lane;
    double bg[FT_PX];
    if (has_bg) {
#pragma unroll
        for (int i = 0; i < FT_PX / 2; i++) {
            double2 v = bgt[i * 32];
            bg[2 * i] = v.x;
            bg[2 * i + 1] = v.y;
        }
    }
    // polygon mask bits of the 16 pixels (bit j = pixel j of the first segment, bit 8 + j of the second), loaded once per call
    uint32_t M = 0;
    const bool okA = py < h && px < w, okB = py < h && px + 64 < w;
    const uint32_t vmask = (okA ? 1u : 0u) | (okB ? 2u : 0u);
    if (okA) M = (__ldg(p.maskbits + ((size_t)s * h + py) * p.wpr + (px >> 5)) >> (px & 31)) & 0xFFu;
    if (okB) M |= ((__ldg(p.maskbits + ((size_t)s * h + py) * p.wpr + ((px + 64) >> 5)) >> (px & 31)) & 0xFFu) << 8;
    const bool wmasked = __any_sync(0xffffffffu, M != 0);       // warp-uniform choice of the masked variant
    // TMA pipeline: frame t+1 lands in the other stage while frame t is being processed
    const int cx = A4 ? x0 - 4 : (x0 * 3) / 4 - 4, cy = y0 - 2;     // box origin in (u32 column, row); OOB is zero-filled
    if (tid == 0) {
        fm_mbar_init(&bars[0], 1);
        fm_mbar_init(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
        if (NV12) {
            fm_mbar_expect_tx(&bars[0], NV_BYTES);
            fm_tma_load_4d(raw, &tmap, &bars[0], x0 / 4 - 4, y0 - 2, 0, s);
            fm_tma_load_4d(raw + NV_Y_BYTES, &tmap_uv, &bars[0], x0 / 4 - 4, y0 / 2 - 1, 0, s);
        } else if (GRAY) {
            fm_mbar_expect_tx(&bars[0], NV_Y_BYTES);
            fm_tma_load_4d(raw, &tmap, &bars[0], x0 / 4 - 4, y0 - 2, 0, s);
        } else {
            fm_mbar_expect_tx(&bars[0], A4 ? A4_BYTES : RAW_BYTES);
            fm_tma_load_4d(raw, &tmap, &bars[0], cx, cy, 0, s);
        }
    }
    // the thread's two bytes of the bit plane (row py, pixels px .. px+7 and px+64 .. px+71)
    uint8_t *tb = reinterpret_cast<uint8_t *>(p.tbits + ((size_t)s * p.T) * p.flatwords + (size_t)py * p.wpr) + (px >> 3);
    // B fragments of the horizontal pass (constant, prepared by the host: fused_bfr)
    uint32_t bfr[2][2];
    {
        const uint4 b = p.bfr[lane];
        bfr[0][0] = b.x; bfr[0][1] = b.y; bfr[1][0] = b.z; bfr[1][1] = b.w;
        // opaque: otherwise the compiler re-reads the (lane-indexed, hence serialised) constant bank in every frame
        asm volatile("" : "+r"(bfr[0][0]), "+r"(bfr[0][1]), "+r"(bfr[1][0]), "+r"(bfr[1][1]));
    }
    // A-fragment row addresses of LDSM.x4 (lane L supplies row L&7 of matrix L>>3; matrices: rows 0-7 / 8-15 of
    // bytes 0-15, then of bytes 16-31) and D-fragment store positions
    const int hwin = warp & 7;                                  // the warp's 16-column window of the horizontal pass
    const uint32_t sg_lane = fm_smem_u32(sg) + ((lane & 7) + 8 * ((lane >> 3) & 1)) * (FG_WORDS * 4) + 16 * hwin + 16 * (lane >> 4);
    uint32_t *sh_lane = sh + (lane >> 2) * FH_WORDS + 8 * hwin + (lane & 3);
    // the thread's first unit of the BGR -> gray conversion: stage bytes 4 + 24 tid .. (see below), gray words 2 tid, 2 tid + 1
    const int rs_tid = 4 + 24 * tid;
    uint2 *const sgt = reinterpret_cast<uint2 *>(sg) + tid;
    // gray: the thread copies word gu of rows gr, gr + GROWS, ... (GROWS rows of FG_WORDS words per step): the offsets of
    // every step are immediates from these two
    constexpr int GROWS = FUSED_THREADS / FG_WORDS;
    const int gr = tid / FG_WORDS, gu = tid - gr * FG_WORDS;
    const int gs_tid = gr * NV_PITCH + 12 + 4 * gu;
    uint32_t *const sgg = sg + gr * FG_WORDS + gu;
    const uint32_t bars_s = fm_smem_u32(bars);
    uint32_t hits = 0;                  // bit t: frame t has a pixel above threshold in this warp's rows (Ts <= 32)
#ifdef FM_K1_PROF
    long long k1_prof[K1_NPROF] = {}, k1_prof_t = clock64();
#endif

    for (int t = 0; t < Ts; t++) {
        // No barrier here: every thread that gets this far has passed the second barrier of frame t-1, i.e. all
        // conversions out of raw stage (t+1)&1 (frame t-1) and all reads of the gray plane are complete.
        if (tid == 0 && t + 1 < Ts) {
            if (NV12) {
                unsigned char *dst = raw + ((t + 1) & 1) * STG;
                fm_mbar_expect_tx(&bars[(t + 1) & 1], NV_BYTES);
                fm_tma_load_4d(dst, &tmap, &bars[(t + 1) & 1], x0 / 4 - 4, y0 - 2, t + 1, s);
                fm_tma_load_4d(dst + NV_Y_BYTES, &tmap_uv, &bars[(t + 1) & 1], x0 / 4 - 4, y0 / 2 - 1, t + 1, s);
            } else if (GRAY) {
                fm_mbar_expect_tx(&bars[(t + 1) & 1], NV_Y_BYTES);
                fm_tma_load_4d(raw + ((t + 1) & 1) * STG, &tmap, &bars[(t + 1) & 1], x0 / 4 - 4, y0 - 2, t + 1, s);
            } else {
                fm_mbar_expect_tx(&bars[(t + 1) & 1], A4 ? A4_BYTES : RAW_BYTES);
                fm_tma_load_4d(raw + ((t + 1) & 1) * STG, &tmap, &bars[(t + 1) & 1], cx, cy, t + 1, s);
            }
        }
        fm_mbar_wait(bars_s + 8 * (t & 1), (t >> 1) & 1);
        K1_PROF(K1_WAIT);
        // ---- staged BGR (or NV12) -> gray bytes in shared memory (tile + halo) ----
        if (NV12) {
            // unit = gray word u of the row pair 2k, 2k+1 (image rows y0-2+2k, +1; y0 is even): two luma words and the UV
            // word of chroma row k (= image UV row y0/2-1+k), all at byte 12 + 4u of their box rows (columns x0-4+4u ..
            // +3); the chroma terms of the word's two 2x2 blocks serve both rows.  Zero-filled bytes outside the image
            // convert to some colour: the border step below overwrites every halo pixel the passes read, as with BGR.
            constexpr int NU = (FG_ROWS / 2) * FG_WORDS, NFULL = NU / FUSED_THREADS;
            const unsigned char *st = raw + (t & 1) * STG;
#pragma unroll
            for (int i = 0; i <= NFULL; i++) {
                if (i < NFULL || tid < NU - NFULL * FUSED_THREADS) {
                    const int un = tid + i * FUSED_THREADS, k = un / FG_WORDS, u = un - k * FG_WORDS;
                    const unsigned char *yq = st + 2 * k * NV_PITCH + 12 + 4 * u;
                    const uint32_t l0 = *reinterpret_cast<const uint32_t *>(yq);
                    const uint32_t l1 = *reinterpret_cast<const uint32_t *>(yq + NV_PITCH);
                    const uint32_t cw = *reinterpret_cast<const uint32_t *>(st + NV_Y_BYTES + k * NV_PITCH + 12 + 4 * u);
                    const FmChroma c0 = fm_nv12_chroma(cw & 0xFFu, (cw >> 8) & 0xFFu);
                    const FmChroma c1 = fm_nv12_chroma((cw >> 16) & 0xFFu, cw >> 24);
                    sg[2 * k * FG_WORDS + u] = nv12_gray4(l0, c0, c1);
                    sg[(2 * k + 1) * FG_WORDS + u] = nv12_gray4(l1, c0, c1);
                }
            }
        } else if (GRAY) {
            // the stage already holds gray bytes: word u of a row (columns x0-4+4u .. +3) is at byte 12 + 4u of its box row.
            // Zero-filled bytes outside the image are overwritten by the border step below, as with BGR.
            const unsigned char *st = raw + (t & 1) * STG + gs_tid;
            if (gr < GROWS) {
#pragma unroll 1                // unrolled, the six loads in flight push the kernel to 40 spilled bytes (rolled: 20)
                for (int i = 0; i < (FG_ROWS + GROWS - 1) / GROWS; i++)
                    if ((i + 1) * GROWS <= FG_ROWS || gr + i * GROWS < FG_ROWS)
                        sgg[i * GROWS * FG_WORDS] = *reinterpret_cast<const uint32_t *>(st + i * GROWS * NV_PITCH);
            }
        } else if (A4) {
            // word u of a gray row (columns x0-4+4u .. +3) is the 16-byte word u of its box row
            const unsigned char *st = raw + (t & 1) * STG;
            for (int un = tid; un < FG_ROWS * FG_WORDS; un += FUSED_THREADS) {
                const int k = un / FG_WORDS, u = un - k * FG_WORDS;
                sg[k * FG_WORDS + u] = fm_gray4a<RGBO>(*reinterpret_cast<const uint4 *>(st + k * A4_PITCH + 16 * u));
            }
        } else {
            // the staged rows are dense (pitch 432 B = 36 groups of 4 pixels = 12 B, the first at byte 4 because the
            // TMA box must start 16 B aligned in global memory -- a box at x0 * 3 - 12 raises "illegal instruction") and
            // so are the gray rows (36 words): group u is raw + 4 + 12 u -> sg[u].
            // two units (8 pixels, 24 bytes -> 2 gray words) per step: half the address arithmetic and loop control.  Unit
            // u = tid + i * FUSED_THREADS: the offsets of all steps are immediates from the thread's own (rs, sgt), and
            // only the last step, which not every thread has, is predicated.
            constexpr int NU = FG_ROWS * FG_WORDS / 2, NFULL = NU / FUSED_THREADS;
            const unsigned char *rs = raw + (t & 1) * STG + rs_tid;
#pragma unroll
            for (int i = 0; i <= NFULL; i++) {
                if (i < NFULL || tid < NU - NFULL * FUSED_THREADS) {
                    // 24 bytes at byte 4 (mod 8) of the stage: 4 + 8 + 8 + 4
                    const unsigned char *q = rs + i * (24 * FUSED_THREADS);
                    const uint32_t a0 = *reinterpret_cast<const uint32_t *>(q), a5 = *reinterpret_cast<const uint32_t *>(q + 20);
                    const uint2 a12 = *reinterpret_cast<const uint2 *>(q + 4), a34 = *reinterpret_cast<const uint2 *>(q + 12);
                    const uint32_t g0 = fm_gray4<RGBO>(a0, a12.x, a12.y), g1 = fm_gray4<RGBO>(a34.x, a34.y, a5);
                    sgt[i * FUSED_THREADS] = make_uint2(g0, g1);
                }
            }
        }
        __syncthreads();
        K1_PROF(K1_GRAY);
        if (border) {               // BORDER_REFLECT_101 for the 2-pixel ring outside the image
            unsigned char *sb = reinterpret_cast<unsigned char *>(sg);
            for (int ry = tid; ry < FG_ROWS; ry += FUSED_THREADS) {
                unsigned char *row = sb + ry * (FG_WORDS * 4) + 4;       // row[c] = column x0 + c
                if (x0 == 0) { row[-1] = row[1]; row[-2] = row[2]; }
                if (x0 + FT_W >= w) { int e = w - x0; row[e] = row[e - 2]; row[e + 1] = row[e - 3]; }
            }
            __syncthreads();
            for (int i = tid; i < FG_WORDS; i += FUSED_THREADS) {
                if (y0 == 0) { sg[1 * FG_WORDS + i] = sg[3 * FG_WORDS + i]; sg[0 * FG_WORDS + i] = sg[4 * FG_WORDS + i]; }
                if (y0 + FT_H >= h) {
                    int e = h - y0 + 2;       // shared row of image row h
                    sg[e * FG_WORDS + i] = sg[(e - 2) * FG_WORDS + i];
                    sg[(e + 1) * FG_WORDS + i] = sg[(e - 3) * FG_WORDS + i];
                }
            }
            __syncthreads();
        }
        K1_PROF(K1_BORDER);
        if (KEEP) {
            for (int u = tid; u < FT_H * (FT_W / 4); u += FUSED_THREADS) {
                int ry = u / (FT_W / 4), ux = u - ry * (FT_W / 4);
                int gy = y0 + ry, gx = x0 + 4 * ux;
                if (gy < h && gx < w)
                    *reinterpret_cast<uint32_t *>(p.gray_out + (((size_t)s * p.T + t) * h + gy) * w + gx) =
                        sg[(ry + 2) * FG_WORDS + ux + 1];
            }
        }
        // ---- horizontal pass on the tensor cores: warp = one 16-column window, every (FUSED_WARPS / 8)-th block of 16 rows ----
        {
            constexpr int MBS = FUSED_WARPS / 8;                 // warps per window
            constexpr int NMB = (FH_MB + MBS - 1) / MBS;         // blocks per warp (the last may not exist for every warp)
            const int mb0 = warp >> 3;
            uint32_t a[NMB][4];
#pragma unroll
            for (int i = 0; i < NMB; i++)
                if (MBS == 1 || mb0 + i * MBS < FH_MB) fm_ldsm_x4(sg_lane + (mb0 + i * MBS) * (16 * FG_WORDS * 4), a[i]);
#pragma unroll
            for (int i = 0; i < NMB; i++) {
                if (MBS == 1 || mb0 + i * MBS < FH_MB) {
                    int d0[4], d1[4];
                    fm_imma0(d0, a[i][0], a[i][1], a[i][2], a[i][3], bfr[0][0], bfr[0][1], 0);
                    fm_imma0(d1, a[i][0], a[i][1], a[i][2], a[i][3], bfr[1][0], bfr[1][1], 0);
                    uint32_t *o = sh_lane + (mb0 + i * MBS) * (16 * FH_WORDS);
                    o[0] = __byte_perm(d0[0], d0[1], 0x5410);
                    o[4] = __byte_perm(d1[0], d1[1], 0x5410);
                    o[8 * FH_WORDS] = __byte_perm(d0[2], d0[3], 0x5410);
                    o[8 * FH_WORDS + 4] = __byte_perm(d1[2], d1[3], 0x5410);
                }
            }
        }
        __syncthreads();
        K1_PROF(K1_HORIZ);
        // ---- vertical pass on packed pairs (5 rows x 16 pixels per thread), then the temporal update ----
        const uint32_t *sgw = sh + trow * FH_WORDS + 4 * xg;
        asm volatile("" : "+r"(M));        // opaque per frame: keeps the 16 single-bit tests of M from being hoisted (and spilled)
        uint8_t *bo = KEEP ? p.blur_out + (((size_t)s * p.T + t) * h + py) * w + px : nullptr;
        uint32_t bits;
        if (t == 0 && !has_bg) bits = fused_rows<KEEP, SAFE, true, true, false>(sgw, bg, M, p, bo, vmask);
        else if (wmasked) bits = p.shift == 8 ? fused_rows<KEEP, SAFE, false, true, true>(sgw, bg, M, p, bo, vmask)
                                              : fused_rows<KEEP, SAFE, false, true, false>(sgw, bg, M, p, bo, vmask);
        else if (p.shift == 8) bits = fused_rows<KEEP, SAFE, false, false, true>(sgw, bg, M, p, bo, vmask);
        else bits = fused_rows<KEEP, SAFE, false, false, false>(sgw, bg, M, p, bo, vmask);
        K1_PROF(K1_VERT);
        // ---- two bytes of the bit plane per thread ----
        if (!okA) bits = 0;
        if (!okB) bits &= 0xFFu;
        if (okA) tb[0] = (uint8_t)bits;
        if (okB) tb[8] = (uint8_t)(bits >> 8);
        // rawrange: whether this warp's 4 rows hold something in frame t.  Up to 32 frames that is bit t of the
        // warp-uniform `hits`, and the atomics of all frames go out once after the loop, one lane per frame.
        const bool any = __any_sync(0xffffffffu, bits != 0);
        if (Ts <= 32) hits |= (any ? 1u : 0u) << t;
        else if (any && lane == 0) rawrange_hit(p, s, t, y0 + 4 * warp);
        tb += 4 * p.flatwords;
        K1_PROF(K1_TAIL);
    }
#ifdef FM_K1_PROF
    if (tid == 0) {
        for (int i = 0; i < K1_NPROF; i++) atomicAdd((unsigned long long *)p.prof + i, (unsigned long long)k1_prof[i]);
        atomicAdd((unsigned long long *)p.prof + K1_NPROF, (unsigned long long)Ts);
    }
#endif
    if (Ts <= 32 && ((hits >> lane) & 1u)) rawrange_hit(p, s, lane, y0 + 4 * warp);
#pragma unroll
    for (int i = 0; i < FT_PX / 2; i++) bgt[i * 32] = make_double2(bg[2 * i], bg[2 * i + 1]);
    fused_exit(p);
}

// tiled background -> row-major float64 plane
__global__ void k_bg_export_fused(const double *__restrict__ bg, double *__restrict__ dst, int w, int h, int tilesX,
                                  int tilesY, int s) {
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= w) return;
    int tx = x / FT_W, ty = y / FT_H, tile = ty * tilesX + tx;
    int lx = x - tx * FT_W, ly = y - ty * FT_H;
    int tid = ly * 8 + ((lx & 63) >> 3);           // thread = row, two 8-pixel segments 64 pixels apart
    int warp = tid >> 5, lane = tid & 31;
    int idx = 8 * (lx >> 6) + (lx & 7);            // pixel index inside the thread
    size_t base = ((((size_t)s * tilesX * tilesY + tile) * FUSED_WARPS + warp) * (FT_PX / 2)) * 32;
    dst[(size_t)y * w + x] = bg[(base + (size_t)(idx >> 1) * 32 + lane) * 2 + (idx & 1)];
}

// NV12 needs nothing more: W % 32 == 0 makes the luma and chroma rows 16 B aligned, and with an even H (fm_ctx_create)
// the frame (W * H * 3 / 2 bytes) and the chroma plane's offset (W * H) too; the caller's pointer and strides are checked
// at launch, as with BGR.  Nor does gray: its rows and frames (W * H bytes) are 16 B aligned with W % 32 == 0
bool fm_fused_supported(const fm_ctx *c) {
    return c->resize_mode == 0 && c->k <= 5 && (c->w % 32) == 0 && c->w >= 4 && c->h >= 4 && c->frame_bytes % 16 == 0;
}

size_t fm_fused_bg_doubles(const fm_ctx *c) {
    size_t tilesX = (c->w + FT_W - 1) / FT_W, tilesY = (c->h + FT_H - 1) / FT_H;
    return (size_t)c->S * tilesX * tilesY * FT_W * FT_H;
}

#ifdef FM_K1_PROF
#include <cstdio>
#include <cstring>

static long long *k1_prof_buffer() {               // [K1_NPROF] cycles, [K1_NPROF] CTA-frames: managed, read by the host
    static long long *buf = nullptr;
    if (!buf && cudaMallocManaged(&buf, (K1_NPROF + 1) * sizeof(long long)) == cudaSuccess)
        memset(buf, 0, (K1_NPROF + 1) * sizeof(long long));
    return buf;
}

// cycles per CTA-frame of each phase since the last call (thread 0 of every CTA), then reset
extern "C" void fm_k1_prof_dump(void) {
    long long *b = k1_prof_buffer();
    if (!b) return;
    cudaDeviceSynchronize();
    const double n = b[K1_NPROF] ? (double)b[K1_NPROF] : 1.0;
    fprintf(stderr, "k1 phases (cycles per CTA-frame, thread 0, %lld CTA-frames): wait %.1f gray %.1f border %.1f "
            "horizontal %.1f vertical %.1f tail %.1f\n", b[K1_NPROF], b[K1_WAIT] / n, b[K1_GRAY] / n, b[K1_BORDER] / n,
            b[K1_HORIZ] / n, b[K1_VERT] / n, b[K1_TAIL] / n);
    memset(b, 0, (K1_NPROF + 1) * sizeof(long long));
}
#endif

#define FUSED_SMEM (2 * RAW_STAGE + FH_ROWS * FG_WORDS * 4 + FH_ROWS * FH_WORDS * 4 + 16)
#define FUSED_SMEM_A4 (2 * A4_STAGE + FH_ROWS * FG_WORDS * 4 + FH_ROWS * FH_WORDS * 4 + 16)
static_assert(FUSED_SMEM_A4 == 61456, "DESIGN §4.9 states this budget");

// one plane of the call's NV12 frames, or the gray frames (rows of W bytes, `pitch` bytes apart), as a 4-D u32 tensor map
// with boxes of NV_PITCH bytes x box_rows
static int nv12_plane_tmap(const fm_ctx *c, const uint8_t *plane, int rows, size_t sstride, size_t fstride, size_t pitch, int T,
                           int box_rows, CUtensorMap *out) {
    PFN_encodeTiled enc = fm_tma_encoder();
    if (!enc) { fm_set_error("cuTensorMapEncodeTiled not available"); return FM_ECUDA; }
    const size_t dense = c->frame_bytes;        // stands in for the stride of a dimension of extent 1 (never applied)
    cuuint64_t dims[4] = {(cuuint64_t)c->W / 4, (cuuint64_t)rows, (cuuint64_t)T, (cuuint64_t)c->S};
    cuuint64_t strides[3] = {(cuuint64_t)pitch, (cuuint64_t)(T > 1 ? fstride : dense),
                             (cuuint64_t)(c->S > 1 ? sstride : (T > 1 ? fstride * T : dense))};
    cuuint32_t box[4] = {NV_PITCH / 4, (cuuint32_t)box_rows, 1, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_UINT32, 4, (void *)plane, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { fm_set_error("cuTensorMapEncodeTiled (NV12 plane) failed (%d)", (int)r); return FM_ECUDA; }
    return FM_OK;
}

int fm_launch_fused(fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, size_t pitch, int64_t uv, int T,
                    cudaStream_t st) {
    CUtensorMap tmap, tmap_uv;
    const bool nv12 = c->nv12_bgr == nullptr && (c->cfg.flags & FM_FLAG_NV12);     // NV12 read directly (no staged slot)
    const bool gray = c->px_bytes == 1;
    int rc;
    if (nv12) {
        if ((((uintptr_t)frames) | sstride | fstride | pitch | (size_t)uv) & 15) {
            fm_set_error("the fused NV12 front end needs 16-byte aligned frames, strides, row pitch and chroma offset");
            return FM_EINVAL;
        }
        if ((rc = nv12_plane_tmap(c, frames, c->H, sstride, fstride, pitch, T, FG_ROWS, &tmap))) return rc;
        if ((rc = nv12_plane_tmap(c, frames + uv, c->H / 2, sstride, fstride, pitch, T, FG_ROWS / 2, &tmap_uv))) return rc;
    } else if (gray) {
        if ((((uintptr_t)frames) | sstride | fstride | pitch) & 15) {
            fm_set_error("the fused gray front end needs 16-byte aligned frames, strides and row pitch");
            return FM_EINVAL;
        }
        if ((rc = nv12_plane_tmap(c, frames, c->H, sstride, fstride, pitch, T, FG_ROWS, &tmap))) return rc;
        tmap_uv = tmap;                          // not read
    } else {
        if ((rc = fm_frames_tmap(c, frames, sstride, fstride, pitch, T, c->px_bytes == 4 ? A4_PITCH / 4 : RAW_PITCH / 4, FG_ROWS,
                                 &tmap)))
            return rc;
        tmap_uv = tmap;                          // not read
    }
    FusedParams p;
    p.T = T; p.nvalid = c->nvalid;
    p.w = c->w; p.h = c->h; p.wpr = c->wpr;
    p.tilesX = (c->w + FT_W - 1) / FT_W; p.tilesY = (c->h + FT_H - 1) / FT_H;
    p.bg = c->bg; p.maskbits = c->maskbits; p.tbits = fm_tflat(c);
    p.flatwords = (size_t)c->ntiles * FM_TILE_WORDS;
    p.bg_in = c->bg_valid + (size_t)c->slot * c->S;
    p.bg_out = c->bg_valid + (size_t)(c->slot ^ 1) * c->S;
    {
        const int Fmax = c->S * c->Tmax;
        p.clear_ff = c->rawrange + (c->slot ? 0 : 2 * Fmax);      // [range slot 0][any] or [any][range slot 1]
        p.n_ff = 6 * Fmax;
        p.clear_zero = c->ncomp;                                   // ncomp, ncounted and the frame counter
        p.n_zero = 2 * Fmax + 4;
    }
    // taps / g for k in {1,3,5}: [0,0,1,0,0] g=256, [0,1,2,1,0] g=64, [1,4,6,4,1] g=16
    int lg;
    if (c->k == 1) { p.b0 = 0; p.b1 = 0; p.b2 = 1; lg = 8; }
    else if (c->k == 3) { p.b0 = 0; p.b1 = 1; p.b2 = 2; lg = 6; }
    else { p.b0 = 1; p.b1 = 4; p.b2 = 6; lg = 4; }
    p.shift = 16 - 2 * lg;
    int r1 = p.shift ? (1 << (p.shift - 1)) : 0;
    p.rnd = r1 | (r1 << 16);
    p.threshold = c->cfg.threshold;
    p.alpha = c->cfg.avg; p.beta = 1.0 - p.alpha;
    p.qoff = (int)(0x4B400000u - (unsigned)p.threshold); p.nthr2 = ~(2u * (unsigned)p.threshold); p.nC = -(4503599627370496.0 * p.alpha);
    p.gray_out = c->gray; p.blur_out = c->blur;
    p.rawrange = fm_rawrange(c);
    p.stamp = c->stamp;
#ifdef FM_K1_PROF
    p.prof = k1_prof_buffer();
    if (!p.prof) return FM_ECUDA;
#endif
    const bool keep = (c->cfg.flags & FM_FLAG_KEEP_PLANES) != 0;
    const bool safe = p.alpha >= 0.0 && p.alpha <= 1.0 && p.threshold >= 0;
    fused_bfr(p);
    dim3 grid(p.tilesX, p.tilesY, c->S);
    typedef void (*FusedKernel)(const CUtensorMap, FusedParams, const CUtensorMap);
#define FM_K1_SRCS(K, S) {k_fused<K, S, FUSED_BGR>, k_fused<K, S, FUSED_NV12>, k_fused<K, S, FUSED_GRAY>, k_fused<K, S, FUSED_RGB>, \
                          k_fused<K, S, FUSED_BGRA>, k_fused<K, S, FUSED_RGBA>}
    const FusedKernel kerns[2][2][6] = {{FM_K1_SRCS(false, false), FM_K1_SRCS(false, true)},
                                        {FM_K1_SRCS(true, false), FM_K1_SRCS(true, true)}};
#undef FM_K1_SRCS
    const int src = nv12 ? FUSED_NV12 : gray ? FUSED_GRAY : c->px_bytes == 4 ? (c->rgb ? FUSED_RGBA : FUSED_BGRA)
                                                 : c->rgb ? FUSED_RGB : FUSED_BGR;
    const FusedKernel kern = kerns[keep][safe][src];
    const int smem = c->px_bytes == 4 ? FUSED_SMEM_A4 : FUSED_SMEM;
    if ((rc = fm_ensure_smem((const void *)kern, smem, c->cfg.device))) return rc;
    // a programmatic dependent of the contour stage of the previous call: see fused_exit.  Not after the NV12 staging
    // kernel (k_nv12.cu, FM_NV12_STAGED builds): K1 reads the frames before its wait, and that kernel writes them
    if (c->nv12_bgr) kern<<<grid, FUSED_THREADS, smem, st>>>(tmap, p, tmap_uv);
    else (void)fm_launch_chained(kern, grid, dim3(FUSED_THREADS), smem, st, tmap, p, tmap_uv);
    FM_LAUNCH_CHECK();
    return FM_OK;
}

int fm_launch_bg_export_fused(fm_ctx *c, int stream, double *dst_dev, cudaStream_t st) {
    dim3 grid((c->w + 127) / 128, c->h);
    k_bg_export_fused<<<grid, 128, 0, st>>>(c->bg, dst_dev, c->w, c->h, (c->w + FT_W - 1) / FT_W,
                                            (c->h + FT_H - 1) / FT_H, stream);
    FM_LAUNCH_CHECK();
    return FM_OK;
}
