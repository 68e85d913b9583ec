// Gaussian blur (3 <= k <= 97) + temporal stage on the 5th-generation tensor cores: both passes of the separable
// 8.8 fixed-point Gaussian are banded (Toeplitz) u8 x u8 -> s32 products issued as tcgen05.mma.kind::i8 with the
// accumulators in tensor memory (SASS: UTCIMMA / LDTM), the gray tile staged by TMA (UTMALDG, 128-byte swizzle).
// Replaces cv2.GaussianBlur + mask_off_areas + VideoFrame.diff/threshold + accumulateWeighted of the reference
// (find_motion/find_motion.py:494, 619-635, 246-257, 651-659; SURVEY.md A.3-A.7) in ONE pass over the image: the
// 16-bit horizontal sums never leave the SM (the two-kernel mma.sync path of k_wide.cu sends them through HBM as two
// byte planes, 2.03x the algorithmic traffic).  Integer arithmetic throughout: bit-exact.
//
// Input: the gray plane with a BORDER_REFLECT_101 apron of 48 pixels materialised (k_pad_gray below: from the BGR
// frames in full-resolution mode, from the resized gray plane otherwise), so no tile needs border logic.
// CTA = 128 x 128 output pixels of one stream, 1024 threads, one CTA per SM, walking the T frames of the call:
//   TMA: gray rows Y0-48 .. Y0+175 x columns X0-48 .. X0+207 -> shared, K-major SWIZZLE_128B (two 128-byte panels)
//   MMA1 (7 x M128 N224 K32): D1[x][y] = sum_q band[x - 32j][q] * gray[y][q]      horizontal pass, TRANSPOSED result:
//        tensor-memory lane = output column, tensor-memory column = row, so a thread reading its lane gets 16
//        consecutive ROWS of one column = one 16-byte chunk of the K-major operand of the vertical pass
//   split: LDTM -> low / high byte planes of the 16-bit sums -> shared (K-major, no swizzle)
//   MMA2 (2 x 7 x M128 N128 K32): D2lo / D2hi[x][y] = sum_q hor_lo/hi[x][q] * band[y - 32j][q]       vertical pass
//   epilogue: LDTM -> blur = (256 hi + lo + 32768) >> 16 -> mask -> bg8, threshold bit (warp ballot = one 32-pixel
//        word of the bit plane), float64 background update; the background of the thread's 16 pixels stays in
//        registers across the T frames.  MMA1 of frame t+1 is issued before the epilogue of frame t and runs under it.
// The band operand is ONE constant matrix: band[u][q] = c[q - u] (c zero-padded to 97 taps), of which every MMA reads
// 128 rows starting at a multiple of 32.
#include <cuda.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "fm_common.cuh"

#define UB_PAD 48                     // apron of the padded gray plane = largest kernel radius
#define UB_T 128                      // output tile edge
#define UB_IN (UB_T + 2 * UB_PAD)     // 224 input rows / columns per tile
#define UB_THREADS 1024
#define UB_GSTAGE (2 * UB_IN * 128)   // bytes of one gray stage: two 128-byte-wide panels of 224 rows
#define UB_YQ (UB_IN / 16)            // 16-row chunks of the horizontal sums
#define UB_PLANE (UB_T * UB_IN)       // bytes of one byte plane of the horizontal sums
#define UB_BROWS 352                  // band rows u in [-224, 128)
#define UB_BOFF 224
#define UB_SMEM (2 * UB_GSTAGE + 2 * UB_PLANE + UB_BROWS * 32 + 1024 /* alignment */ + 64)

// shared-memory matrix descriptors (sm_100 version bit set): K-major, no swizzle (LBO = stride of the two 16-byte K
// chunks, SBO = stride of 8-row groups) and K-major SWIZZLE_128B (rows of 128 bytes, SBO = 1024)
__device__ __forceinline__ uint64_t ub_desc_plain(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo >> 4) & 0x3FFF) << 16) | ((uint64_t)((sbo >> 4) & 0x3FFF) << 32) |
           (1ull << 46);
}
__device__ __forceinline__ uint64_t ub_desc_sw128(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ void ub_mma(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}\n"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}
__device__ __forceinline__ void ub_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(fm_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void ub_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                   "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
}
__device__ __forceinline__ void ub_ld8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}
#define UB_FENCE_BEFORE() asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory")
#define UB_FENCE_AFTER() asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory")

struct UmmaParams {
    const uint8_t *band;        // [UB_BROWS * 32] bytes in the blocked K-major order of the shared copy
    double *bg;                 // [S][tiles][32 warps][8][32 lanes] double2
    const uint32_t *maskbits;   // [S][h][wpr]
    uint32_t *tbits;            // [S][T][flatwords] raw threshold bits
    size_t flatwords;
    const StreamState *state;
    const int *nvalid;
    int *rawrange;              // [S][T][2]
    uint8_t *blur_out;          // [S][T][h][w] parity tap or null
    int T, w, h, wpr, tilesX, tilesY, threshold;
    double alpha, beta;
    int qoff; uint32_t thr2; double nC;         // 0x4B400000 - threshold, 2 threshold, -(2^52 alpha): kept in the constant bank
    long long *prof;            // development aid (FM_UMMA_PROF=1): cycles per phase of CTA (0, 0), thread 0
};
#define UB_PROF(slot)                                                                              \
    do {                                                                                           \
        if (p.prof && (tid == 0 || tid == 992) && blockIdx.x == p.tilesX + 1 && blockIdx.y == 0) { \
            const long long now_ = clock64();                                                      \
            prof_acc[(slot) + (tid ? 16 : 0)] += now_ - prof_t;                                    \
            prof_t = now_;                                                                         \
        }                                                                                          \
    } while (0)

// 16 tensor-memory columns of the thread's lane as 8 registers of two 16-bit values (column 2i in the low half): the
// accumulators of both passes fit 16 bits (sum of taps = 256, operands <= 255), and a packed load moves half the register
// bytes -- tensor-memory reads are bound by the bytes delivered to the register file (profiles/micro/ldtm_rate.log).
__device__ __forceinline__ void ub_ld16p(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.pack::16b.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}

// split: the 16-bit horizontal sums of lane x (tensor-memory columns = rows) -> low / high byte planes in shared memory,
// K-major for the vertical pass: [x >> 3][16-row chunk][x & 7][16 rows].  NU = chunks per column, chunks [yq_lo, yq_hi).
template <int NU>
__device__ __forceinline__ void ub_split(uint32_t tD1lane, unsigned char *sLo, unsigned char *sHi, int xl, int rg, int yq_lo, int yq_hi) {
    for (int yq = yq_lo + rg; yq < yq_hi; yq += 8) {
        uint32_t r[8];
        ub_ld16p(tD1lane + 16 * yq, r);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        uint4 lo, hi;                 // r[i] = bytes [l(2i), h(2i), l(2i+1), h(2i+1)]
        lo.x = __byte_perm(r[0], r[1], 0x6420); hi.x = __byte_perm(r[0], r[1], 0x7531);
        lo.y = __byte_perm(r[2], r[3], 0x6420); hi.y = __byte_perm(r[2], r[3], 0x7531);
        lo.z = __byte_perm(r[4], r[5], 0x6420); hi.z = __byte_perm(r[4], r[5], 0x7531);
        lo.w = __byte_perm(r[6], r[7], 0x6420); hi.w = __byte_perm(r[6], r[7], 0x7531);
        const int off = ((xl >> 3) * NU + yq) * 128 + (xl & 7) * 16;
        *reinterpret_cast<uint4 *>(sLo + off) = lo;
        *reinterpret_cast<uint4 *>(sHi + off) = hi;
    }
}

// epilogue of one frame: 16 consecutive pixels of one row per thread (tensor-memory lane = row, columns = x: low-plane sums
// in columns 0..127, high-plane sums in columns 128..255 of D2).  blur = (256 hi + lo + 32768) >> 16 evaluated on packed pairs:
// u = hi + (lo >> 8) + 128 is exactly (256 hi + lo + 32768) >> 8 and fits 16 bits, blur = u >> 8.
// MASKED: the thread has masked pixels (M = polygon mask bits, bit j = pixel j) or a parity tap is requested.
// Returns the 16 threshold bits (bit j = pixel j).
template <bool SAFE, bool MASKED>
__device__ __forceinline__ uint32_t ub_epilogue(uint32_t tLo16, uint32_t tHi16, double (&bg)[16], uint32_t M, bool init, const UmmaParams &p,
                                                uint8_t *blur_px) {
    uint32_t L[8], Hh[8];
    ub_ld16p(tLo16, L);
    ub_ld16p(tHi16, Hh);
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    uint32_t Uu[8];
#pragma unroll
    for (int k = 0; k < 8; k++) Uu[k] = Hh[k] + __byte_perm(L[k], 0, 0x4341) + 0x00800080u;      // blur of pixels 2k, 2k+1 in bytes 1, 3
    if (MASKED && blur_px) {
        uint4 o;
        o.x = __byte_perm(Uu[0], Uu[1], 0x7531); o.y = __byte_perm(Uu[2], Uu[3], 0x7531);
        o.z = __byte_perm(Uu[4], Uu[5], 0x7531); o.w = __byte_perm(Uu[6], Uu[7], 0x7531);
        uint32_t *ow = &o.x;
#pragma unroll
        for (int wd = 0; wd < 4; wd++) {
            const uint32_t m4 = (M >> (4 * wd)) & 0xFu;
            ow[wd] = fm_clear_masked4(ow[wd], m4);
        }
        *reinterpret_cast<uint4 *>(blur_px) = o;
    }
    uint32_t bits = 0;
    const uint32_t nthr2 = ~p.thr2;
#pragma unroll
    for (int k = 0; k < 8; k++) {
#pragma unroll
        for (int hlf = 0; hlf < 2; hlf++) {
            const int i = 2 * k + hlf;
            uint32_t sv = __byte_perm(Uu[k], 0, hlf ? 0x4443 : 0x4441);
            if (MASKED && (M & (1u << i))) sv = 0;                               // mask_off_areas paints BLACK into blur
            if (init) bg[i] = fm_u8_to_f64(sv);           // ref_frame = blur.astype(float); init is a run-time flag here
            fm_temporal_px<SAFE, false>(sv, bg[i], bits, p.threshold, p.qoff, nthr2, p.alpha, p.beta, p.nC);
        }
    }
    return __brev(bits) >> 16;          // pixel 0 was pushed first
}

// per-frame tail of a thread: epilogue, 16-bit store of the threshold bits, row range of the raw mask
template <bool SAFE>
__device__ __forceinline__ void ub_frame_out(uint32_t tLo16, uint32_t tHi16, double (&bg)[16], uint32_t M, bool ok, bool init, bool masked,
                                             const UmmaParams &p, uint16_t *th16, uint8_t *blur_px, int *rr, int ywarp, int lane) {
    uint32_t bits = masked ? ub_epilogue<SAFE, true>(tLo16, tHi16, bg, M, init, p, blur_px)
                           : ub_epilogue<SAFE, false>(tLo16, tHi16, bg, M, init, p, nullptr);
    if (!ok) bits = 0;
    if (ok) *th16 = (uint16_t)bits;
    if (__any_sync(0xffffffffu, bits != 0) && lane == 0) {       // this warp's 32 rows hold something
        atomicMax(rr, min(ywarp + 31, p.h - 1));
        atomicMax(rr + 1, p.h - 1 - ywarp);
    }
}

template <bool SAFE>
__global__ void __launch_bounds__(UB_THREADS, 1) k_umma_blur(const __grid_constant__ CUtensorMap tmap, UmmaParams p) {
    extern __shared__ unsigned char ub_raw[];
    unsigned char *sm = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(ub_raw) + 1023) & ~(uintptr_t)1023);
    unsigned char *sGray = sm;                                     // [2 stages][2 panels][224][128], written by TMA
    unsigned char *sLo = sm + 2 * UB_GSTAGE;                       // [16 column groups][14 row chunks][8][16]
    unsigned char *sHi = sLo + UB_PLANE;
    unsigned char *sBand = sHi + UB_PLANE;                         // [44 row groups][2][8][16]
    uint64_t *bars = reinterpret_cast<uint64_t *>(sBand + UB_BROWS * 32);      // tma[2], mma1, mma2 (rows 0-63), mma2 (rows 64-127)
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 5);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int s = blockIdx.y, tile = blockIdx.x;
    const int ty = tile / p.tilesX, tx = tile - ty * p.tilesX;
    const int X0 = tx * UB_T, Y0 = ty * UB_T;
    const int Ts = min(p.T, __ldg(p.nvalid + s));
    if (Ts <= 0) return;
    const bool has_bg = p.state[s].has_bg != 0;

    for (int i = tid; i < UB_BROWS * 32 / 16; i += UB_THREADS)
        reinterpret_cast<uint4 *>(sBand)[i] = __ldg(reinterpret_cast<const uint4 *>(p.band) + i);
    if (tid == 0) {
        fm_mbar_init(&bars[0], 1);
        fm_mbar_init(&bars[1], 1);
        fm_mbar_init(&bars[2], 1);
        fm_mbar_init(&bars[3], 1);
        fm_mbar_init(&bars[4], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(fm_smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // the band (generic-proxy writes) is read by the MMAs
    UB_FENCE_BEFORE();
    __syncthreads();
    UB_FENCE_AFTER();
    const uint32_t tmem = *tmem_slot;
    const uint32_t tD1 = tmem, tLo = tmem + 256, tHi = tmem + 384;

    // this thread's pixels: row Y0 + 32 (warp & 3) + lane (= its tensor-memory lane in D2), columns X0 + 16 (warp >> 2) .. + 15;
    // in the split stage the same lane is column 32 (warp & 3) + lane of D1
    const int lq = warp & 3, rg = warp >> 2;
    const int px = X0 + 16 * rg, py = Y0 + 32 * lq + lane;
    double2 *bgt = reinterpret_cast<double2 *>(p.bg) + ((((size_t)s * p.tilesX * p.tilesY + tile) * 32 + warp) * 8) * 32 + lane;
    double bg[16];
    if (has_bg) {
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const double2 v = bgt[i * 32];
            bg[2 * i] = v.x;
            bg[2 * i + 1] = v.y;
        }
    }
    // mask bits of the 16 pixels (bit j = pixel px + j); warp-uniform choice of the masked variant
    const bool ok = py < p.h && px < p.w;
    uint32_t M = 0;
    if (ok) M = (__ldg(p.maskbits + ((size_t)s * p.h + py) * p.wpr + (px >> 5)) >> (px & 31)) & 0xFFFFu;
    const bool masked = __any_sync(0xffffffffu, M != 0) || p.blur_out != nullptr;

    const uint32_t idesc1 = (2u << 4) | ((uint32_t)(UB_IN >> 3) << 17) | ((128u >> 4) << 24);      // S32 += U8 x U8, M128, N224
    const uint32_t idesc2 = (2u << 4) | ((uint32_t)(256 >> 3) << 17) | ((128u >> 4) << 24);        // N256: both byte planes
    const uint32_t aBand = fm_smem_u32(sBand), aGray = fm_smem_u32(sGray), aLo = fm_smem_u32(sLo), aHi = fm_smem_u32(sHi);
    auto issue_tma = [&](int t) {                 // thread 0
        uint64_t *bar = &bars[t & 1];
        unsigned char *dst = sGray + (t & 1) * UB_GSTAGE;
        fm_mbar_expect_tx(bar, UB_GSTAGE);
        fm_tma_load_4d(dst, &tmap, bar, X0, Y0, t, s);
        fm_tma_load_4d(dst + UB_IN * 128, &tmap, bar, X0 + 128, Y0, t, s);
    };
    auto issue_mma1 = [&](int t) {                // thread 0: horizontal pass of frame t into D1
        fm_mbar_wait(&bars[t & 1], (t >> 1) & 1);
        UB_FENCE_AFTER();
        const uint32_t g = aGray + (t & 1) * UB_GSTAGE;
#pragma unroll
        for (int j = 0; j < UB_IN / 32; j++) {
            const uint64_t ad = ub_desc_plain(aBand + (UB_BOFF - 32 * j) * 32, 128, 256);
            const uint64_t bd = ub_desc_sw128(g + (j >> 2) * (UB_IN * 128) + (j & 3) * 32);
            ub_mma(tD1, ad, bd, idesc1, j > 0);
        }
        ub_commit(&bars[2]);
    };
    if (tid == 0) {
        issue_tma(0);
        issue_mma1(0);
    }
    uint16_t *th16 = reinterpret_cast<uint16_t *>(p.tbits + (size_t)s * p.T * p.flatwords + (size_t)py * p.wpr) + (px >> 4);
    const uint32_t lanebase = (uint32_t)(32 * lq) << 16;
    const int xl = 32 * lq + lane;

    __shared__ long long prof_acc[32];
    if (p.prof && tid < 32) prof_acc[tid] = 0;
    long long prof_t = clock64();
    for (int t = 0; t < Ts; t++) {
        fm_mbar_wait(&bars[2], t & 1);            // D1 of frame t is complete (and gray stage t & 1 has been read)
        UB_FENCE_AFTER();
        UB_PROF(0);
        if (tid == 0 && t + 1 < Ts) issue_tma(t + 1);
        UB_PROF(1);
        ub_split<UB_YQ>(tD1 + lanebase, sLo, sHi, xl, rg, 0, UB_YQ);
        UB_PROF(2);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        UB_PROF(3);
        UB_FENCE_BEFORE();
        __syncthreads();
        UB_PROF(4);
        if (tid == 0) {
            UB_FENCE_AFTER();
            // vertical pass: A = band (rows = output rows), B = both byte planes (N = 128 low + 128 high columns)
#pragma unroll
            for (int j = 0; j < UB_IN / 32; j++)
                ub_mma(tLo, ub_desc_plain(aBand + (UB_BOFF - 32 * j) * 32, 128, 256), ub_desc_plain(aLo + 2 * j * 128, 128, UB_YQ * 128), idesc2,
                       j > 0);
            ub_commit(&bars[3]);
            if (t + 1 < Ts) issue_mma1(t + 1);    // runs on the tensor pipe under the epilogue below
        }
        UB_PROF(5);
        fm_mbar_wait(&bars[3], t & 1);
        UB_FENCE_AFTER();
        UB_PROF(6);
        uint8_t *bo = (p.blur_out && ok) ? p.blur_out + (((size_t)s * p.T + t) * p.h + py) * p.w + px : nullptr;
        ub_frame_out<SAFE>(tLo + lanebase + 16 * rg, tHi + lanebase + 16 * rg, bg, M, ok, t == 0 && !has_bg, masked, p, th16, bo,
                           p.rawrange + 2 * ((size_t)s * p.T + t), Y0 + 32 * lq, lane);
        th16 += 2 * p.flatwords;
        UB_PROF(7);
        UB_FENCE_BEFORE();
        __syncthreads();          // D2 and the byte planes are free for frame t + 1
        UB_FENCE_AFTER();
        UB_PROF(8);
    }
#pragma unroll
    for (int i = 0; i < 8; i++) bgt[i * 32] = make_double2(bg[2 * i], bg[2 * i + 1]);
    UB_FENCE_BEFORE();
    __syncthreads();
    if (p.prof && tid < 32 && blockIdx.x == p.tilesX + 1 && blockIdx.y == 0) p.prof[tid] += prof_acc[tid];
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
}

// ---------------------------------------------------------------------------------------------
// k_umma_fused: the same pipeline reading the BGR frames directly (full-resolution mode): no gray plane, no apron
// plane -- DRAM traffic = the algorithmic bytes.  RA = apron of the tile in shared memory (16: k <= 33, 48: k <= 97).
//   TMA ring: BGR rows in chunks of 64 rows x 3 (128 + 2 RA) bytes (u32 tensor map over the caller's frames, rows
//       outside the image zero-filled)
//   convert: 16-pixel units, three LDS.128 -> 32 IDP.2A -> one 16-byte chunk of the gray tile, written straight into the
//       SWIZZLE_128B K-major layout the MMA descriptor expects; BORDER_REFLECT_101 columns / rows are mirrored inside
//       the tile (border tiles only).  Only the rows / columns within the kernel radius of the tile are converted,
//       the rest of the apron meets zero taps.
//   MMA1, split, MMA2, epilogue as above.  Order per frame: split(t), MMA2(t) issued, convert(t+1) under it, MMA1(t+1)
//       issued, epilogue(t) under it -- the tensor pipe and the ALUs never wait for each other.
// ---------------------------------------------------------------------------------------------
template <int RA>
struct UfGeom {
    static constexpr int RC = RA == 16 ? 80 : 64;     // rows per BGR chunk (RA = 16: a frame is two chunks)
    static constexpr int NST = RA == 16 ? 3 : 2;      // ring stages
    static constexpr int IN = UB_T + 2 * RA;          // rows / columns of the gray tile
    static constexpr int KS = IN / 32;                // K steps of either pass
    static constexpr int NU = IN / 16;                // 16-pixel units per row
    static constexpr int RB = 3 * IN;                 // bytes of a staged BGR row
    static constexpr int RSTAGE = RC * RB;            // bytes of one ring stage
    static constexpr int GRAY = 2 * IN * 128;         // two 128-byte panels
    static constexpr int PLANE = UB_T * IN;
    static constexpr int BROWS = 32 * (KS - 1) + 128; // band rows u in [-32 (KS - 1), 128)
    static constexpr int BOFF = 32 * (KS - 1);
    static constexpr int SMEM = GRAY + 2 * PLANE + BROWS * 32 + NST * RSTAGE + 1024 + 128;
};

struct UfParams {
    UmmaParams u;
    int r;                      // kernel radius (k >> 1) <= RA
};

// RGB: R-first frames (FM_FLAG_RGB)
template <int RA, bool SAFE, bool RGB = false>
__global__ void __launch_bounds__(UB_THREADS, 1) k_umma_fused(const __grid_constant__ CUtensorMap tmap, UfParams q) {
    using G = UfGeom<RA>;
    const UmmaParams &p = q.u;
    extern __shared__ unsigned char ub_raw[];
    unsigned char *sm = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(ub_raw) + 1023) & ~(uintptr_t)1023);
    unsigned char *sGray = sm;                                     // [2 panels][IN rows][128], SWIZZLE_128B
    unsigned char *sLo = sGray + G::GRAY;
    unsigned char *sHi = sLo + G::PLANE;
    unsigned char *sBand = sHi + G::PLANE;
    unsigned char *sRaw = sBand + G::BROWS * 32;                   // [NST stages][RC rows][RB]   (128-byte aligned)
    uint64_t *bars = reinterpret_cast<uint64_t *>(sRaw + G::NST * G::RSTAGE);   // mma1, mma2, raw[NST]
    uint64_t *rbar = bars + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(rbar + G::NST);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int s = blockIdx.y, tile = blockIdx.x;
    const int ty = tile / p.tilesX, tx = tile - ty * p.tilesX;
    const int TH = UB_T;
    const int X0 = tx * UB_T, Y0 = ty * TH;
    const int Ts = min(p.T, __ldg(p.nvalid + s));
    if (Ts <= 0) return;
    const bool has_bg = p.state[s].has_bg != 0;
    const int r = q.r;

    for (int i = tid; i < G::BROWS * 32 / 16; i += UB_THREADS)
        reinterpret_cast<uint4 *>(sBand)[i] = __ldg(reinterpret_cast<const uint4 *>(p.band) + i);
    if (tid == 0) {
        fm_mbar_init(&bars[0], 1);
        fm_mbar_init(&bars[1], 1);
        for (int i = 0; i < G::NST; i++) fm_mbar_init(&rbar[i], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(fm_smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    UB_FENCE_BEFORE();
    __syncthreads();
    UB_FENCE_AFTER();
    const uint32_t tmem = *tmem_slot;
    const uint32_t tD1 = tmem, tLo = tmem + 256, tHi = tmem + 384;

    // this thread's pixels: row Y0 + 32 (warp & 3) + lane (= its tensor-memory lane in D2), columns X0 + 16 (warp >> 2) .. + 15
    const int lq = warp & 3, rg = warp >> 2;
    const int px = X0 + 16 * rg, py = Y0 + 32 * lq + lane;
    double2 *bgt = reinterpret_cast<double2 *>(p.bg) + ((((size_t)s * p.tilesX * p.tilesY + tile) * 32 + warp) * 8) * 32 + lane;
    double bg[16];
    if (has_bg) {
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const double2 v = bgt[i * 32];
            bg[2 * i] = v.x;
            bg[2 * i + 1] = v.y;
        }
    }
    // mask bits of the 16 pixels (bit j = pixel px + j); warp-uniform choice of the masked variant
    const bool ok = py < p.h && px < p.w;
    uint32_t M = 0;
    if (ok) M = (__ldg(p.maskbits + ((size_t)s * p.h + py) * p.wpr + (px >> 5)) >> (px & 31)) & 0xFFFFu;
    const bool masked = __any_sync(0xffffffffu, M != 0) || p.blur_out != nullptr;

    const uint32_t idesc1 = (2u << 4) | ((uint32_t)(G::IN >> 3) << 17) | ((128u >> 4) << 24);
    const uint32_t idesc2 = (2u << 4) | ((uint32_t)(256 >> 3) << 17) | ((128u >> 4) << 24);        // N256: both byte planes
    const uint32_t aBand = fm_smem_u32(sBand), aGray = fm_smem_u32(sGray), aLo = fm_smem_u32(sLo), aHi = fm_smem_u32(sHi);

    // rows / columns of the gray tile that meet non-zero taps: tile row p <-> image row Y0 - RA + p
    const int p_lo = RA - r, p_hi = RA + TH + r;                   // [p_lo, p_hi)
    const int NR = p_hi - p_lo;                                    // BGR rows per frame
    const int NCH = (NR + G::RC - 1) / G::RC;                      // chunks per frame
    const int u_lo = (RA - r) >> 4, u_hi = (RA + UB_T + r + 15) >> 4;     // 16-pixel units [u_lo, u_hi)
    const int cx = (3 * (X0 - RA)) / 4;                            // box origin, u32 column (16-byte aligned)
    // chunk g of the call: frame g / NCH, chunk g % NCH -> ring stage g % NST
    const int total_chunks = Ts * NCH;
    auto issue_raw = [&](int g) {                 // thread 0
        const int t = g / NCH, c = g - t * NCH;
        uint64_t *bar = &rbar[g % G::NST];
        fm_mbar_expect_tx(bar, G::RSTAGE);
        fm_tma_load_4d(sRaw + (g % G::NST) * G::RSTAGE, &tmap, bar, cx, Y0 - r + G::RC * c, t, s);
    };
    // BGR -> gray of frame t into the swizzled tile (all threads), chunk by chunk; re-arms the ring as stages drain
    auto convert = [&](int t) {
        for (int c = 0; c < NCH; c++) {
            const int g = t * NCH + c;
            fm_mbar_wait(&rbar[g % G::NST], (g / G::NST) & 1);
            const unsigned char *raw = sRaw + (g % G::NST) * G::RSTAGE;
            const int nun = u_hi - u_lo;
            for (int u = tid; u < G::RC * nun; u += UB_THREADS) {
                const int rr = u / nun, uu = u_lo + (u - rr * nun);
                const int pr = p_lo + G::RC * c + rr;              // tile row
                if (pr < p_hi) {
                    const uint4 *src = reinterpret_cast<const uint4 *>(raw + rr * G::RB + 48 * uu);
                    const uint4 a = src[0], b = src[1], d = src[2];
                    uint4 o;
                    o.x = fm_gray4<RGB>(a.x, a.y, a.z);
                    o.y = fm_gray4<RGB>(a.w, b.x, b.y);
                    o.z = fm_gray4<RGB>(b.z, b.w, d.x);
                    o.w = fm_gray4<RGB>(d.y, d.z, d.w);
                    *reinterpret_cast<uint4 *>(sGray + (uu >> 3) * (G::IN * 128) + pr * 128 + (((uu & 7) ^ (pr & 7)) << 4)) = o;
                }
            }
            __syncthreads();                       // the stage is drained
            if (tid == 0 && g + G::NST < total_chunks) issue_raw(g + G::NST);
        }
        // BORDER_REFLECT_101: mirror inside the tile (tile column / row c <-> image X0 - RA + c)
        auto gaddr = [&](int pr, int qc) { return sGray + (qc >> 7) * (G::IN * 128) + pr * 128 + ((((qc >> 4) & 7) ^ (pr & 7)) << 4) + (qc & 15); };
        const bool bl = X0 == 0, br = X0 + UB_T + r > p.w, bt = Y0 == 0, bb = Y0 + TH + r > p.h;
        if (bl || br) {
            const int e = RA + p.w - X0;           // tile column of image column w
            const int rows_lo = max(p_lo, RA - Y0), rows_hi = min(p_hi, RA + p.h - Y0);      // rows inside the image
            const int nrow = rows_hi - rows_lo, per = (bl ? r : 0) + (br ? r : 0);
            for (int i = tid; i < nrow * per; i += UB_THREADS) {
                const int pr = rows_lo + i / per;
                int j = i % per;
                if (bl && j < r) *gaddr(pr, RA - 1 - j) = *gaddr(pr, RA + 1 + j);
                else { j -= bl ? r : 0; *gaddr(pr, e + j) = *gaddr(pr, e - 2 - j); }
            }
            __syncthreads();
        }
        if (bt || bb) {
            const int e = RA + p.h - Y0;           // tile row of image row h
            const int nun = u_hi - u_lo, per = (bt ? r : 0) + (bb ? r : 0);
            for (int i = tid; i < per * nun; i += UB_THREADS) {
                int j = i / nun;
                const int uu = u_lo + i % nun;
                int dst, src;
                if (bt && j < r) { dst = RA - 1 - j; src = RA + 1 + j; }
                else { j -= bt ? r : 0; dst = e + j; src = e - 2 - j; }
                if (dst < G::IN) {
                    const uint4 v = *reinterpret_cast<const uint4 *>(sGray + (uu >> 3) * (G::IN * 128) + src * 128 + (((uu & 7) ^ (src & 7)) << 4));
                    *reinterpret_cast<uint4 *>(sGray + (uu >> 3) * (G::IN * 128) + dst * 128 + (((uu & 7) ^ (dst & 7)) << 4)) = v;
                }
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        UB_FENCE_BEFORE();
        __syncthreads();
    };
    auto issue_mma1 = [&]() {                     // thread 0: horizontal pass of the gray tile into D1
        UB_FENCE_AFTER();
#pragma unroll
        for (int j = 0; j < G::KS; j++) {
            const uint64_t ad = ub_desc_plain(aBand + (G::BOFF - 32 * j) * 32, 128, 256);
            const uint64_t bd = ub_desc_sw128(aGray + (j >> 2) * (G::IN * 128) + (j & 3) * 32);
            ub_mma(tD1, ad, bd, idesc1, j > 0);
        }
        ub_commit(&bars[0]);
    };
    if (tid == 0)
        for (int g = 0; g < G::NST && g < total_chunks; g++) issue_raw(g);
    // (the part of the apron that is never converted holds arbitrary bytes: they only meet zero taps)
    convert(0);
    if (tid == 0) issue_mma1();

    uint16_t *th16 = reinterpret_cast<uint16_t *>(p.tbits + (size_t)s * p.T * p.flatwords + (size_t)py * p.wpr) + (px >> 4);
    const uint32_t lanebase = (uint32_t)(32 * lq) << 16;
    const int xl = 32 * lq + lane;
    const int yq_lo = p_lo >> 4, yq_hi = (p_hi + 15) >> 4;        // 16-row chunks of the horizontal sums that meet non-zero taps

    for (int t = 0; t < Ts; t++) {
        fm_mbar_wait(&bars[0], t & 1);            // D1 of frame t is complete, the gray tile is free
        UB_FENCE_AFTER();
        ub_split<G::NU>(tD1 + lanebase, sLo, sHi, xl, rg, yq_lo, yq_hi);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        UB_FENCE_BEFORE();
        __syncthreads();
        if (tid == 0) {
            UB_FENCE_AFTER();
#pragma unroll
            for (int j = 0; j < G::KS; j++)
                ub_mma(tLo, ub_desc_plain(aBand + (G::BOFF - 32 * j) * 32, 128, 256), ub_desc_plain(aLo + 2 * j * 128, 128, G::NU * 128), idesc2,
                       j > 0);
            ub_commit(&bars[1]);
        }
        if (t + 1 < Ts) {                         // gray of frame t + 1 while the vertical pass runs
            convert(t + 1);
            if (tid == 0) issue_mma1();           // ... and its horizontal pass under the epilogue below
        }
        fm_mbar_wait(&bars[1], t & 1);
        UB_FENCE_AFTER();
        uint8_t *bo = (p.blur_out && ok) ? p.blur_out + (((size_t)s * p.T + t) * p.h + py) * p.w + px : nullptr;
        ub_frame_out<SAFE>(tLo + lanebase + 16 * rg, tHi + lanebase + 16 * rg, bg, M, ok, t == 0 && !has_bg, masked, p, th16, bo,
                           p.rawrange + 2 * ((size_t)s * p.T + t), Y0 + 32 * lq, lane);
        th16 += 2 * p.flatwords;
        UB_FENCE_BEFORE();
        __syncthreads();
        UB_FENCE_AFTER();
    }
#pragma unroll
    for (int i = 0; i < 8; i++) bgt[i * 32] = make_double2(bg[2 * i], bg[2 * i + 1]);
    UB_FENCE_BEFORE();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
}

// ---------------------------------------------------------------------------------------------
// padded gray plane: gpad[f][yp][xp] = gray(reflect101(yp - 48), reflect101(xp - 48)); BGR: convert on the way
// (find_motion.py:493, SURVEY.md A.2); otherwise src is a gray plane (the context's, or gray frames).  Frame (s, t) starts at
// src + s * sstride + t * fstride, rows rpitch bytes apart.  One thread = 4 padded pixels.  RGB: R-first frames; PX: bytes
// per pixel of the frames (3, or 4 with FM_FLAG_ALPHA)
// ---------------------------------------------------------------------------------------------
template <bool BGR, bool RGB = false, int PX = 3>
__global__ void __launch_bounds__(256) k_pad_gray(const uint8_t *__restrict__ src, size_t sstride, size_t fstride, size_t rpitch, int T,
                                                  uint8_t *__restrict__ gpad, int w, int h, int Wp, int Hp,
                                                  const int *__restrict__ nvalid, int aligned4) {
    const int f = blockIdx.z, s = f / T, t = f - s * T;
    if (t >= __ldg(nvalid + s)) return;
    const int yp = blockIdx.y, xp = 4 * (blockIdx.x * blockDim.x + threadIdx.x);
    if (xp >= Wp) return;
    uint32_t out = 0;
    if (yp < h + 2 * UB_PAD && xp < w + 2 * UB_PAD) {
        const int y = fm_reflect101(yp - UB_PAD, h);
        const uint8_t *row = src + (size_t)s * sstride + (size_t)t * fstride + (size_t)y * rpitch;
        const int x = xp - UB_PAD;
        if (x >= 0 && x + 3 < w && aligned4) {
            if (BGR) {
                const uint32_t *q = reinterpret_cast<const uint32_t *>(row + PX * x);
                if constexpr (PX == 4) out = fm_gray4a<RGB>(make_uint4(__ldg(q), __ldg(q + 1), __ldg(q + 2), __ldg(q + 3)));
                else out = fm_gray4<RGB>(__ldg(q), __ldg(q + 1), __ldg(q + 2));
            } else {
                out = __ldg(reinterpret_cast<const uint32_t *>(row + x));
            }
        } else {
#pragma unroll
            for (int b = 0; b < 4; b++) {
                if (xp + b < w + 2 * UB_PAD) {
                    const int xx = fm_reflect101(x + b, w);
                    out |= (BGR ? fm_gray<RGB>(row[PX * xx], row[PX * xx + 1], row[PX * xx + 2]) : (uint32_t)row[xx]) << (8 * b);
                }
            }
        }
    }
    *reinterpret_cast<uint32_t *>(gpad + ((size_t)f * Hp + yp) * Wp + xp) = out;
}

// tiled background -> row-major float64 plane
__global__ void k_bg_export_umma(const double *__restrict__ bg, double *__restrict__ dst, int w, int h, int tilesX, int tilesY, int s) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= w) return;
    const int tx = x / UB_T, ty = y / UB_T, lx = x % UB_T, ly = y % UB_T;
    const int warp = (ly >> 5) + 4 * (lx >> 4), lane = ly & 31, i = lx & 15;       // thread = row, 16 consecutive columns
    const size_t base = ((((size_t)s * tilesX * tilesY + (size_t)ty * tilesX + tx) * 32 + warp) * 8) * 32;
    dst[(size_t)y * w + x] = bg[(base + (size_t)(i >> 1) * 32 + lane) * 2 + (i & 1)];
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
// bit planes are written a 32-pixel word per warp ballot: needs the flat bit order to equal the row-padded one (w % 32 == 0)
// (k = 1 has the single tap 256, which is not a u8: the identity blur of k_wide.cu takes it)
bool fm_umma_supported(const fm_ctx *c) { return c->k >= 3 && c->k <= 2 * UB_PAD + 1 && (c->w % 32) == 0; }

// Default policy (no FM_FLAG_UMMA / FM_FLAG_NO_UMMA): measured on B200 at 1080p, 8 streams x 16 frames (profiles/r2_*), the
// mma.sync two-pass kernels are still ahead, so the tcgen05 kernel is opt-in.
bool fm_umma_preferred(const fm_ctx *) { return false; }

static void umma_geom(const fm_ctx *c, int *tilesX, int *tilesY, int *Wp, int *Hp) {
    *tilesX = (c->w + UB_T - 1) / UB_T;
    *tilesY = (c->h + UB_T - 1) / UB_T;
    *Wp = *tilesX * UB_T + 128;             // the second panel of the last tile stays inside the plane
    *Hp = *tilesY * UB_T + 2 * UB_PAD;
}

size_t fm_umma_pad_bytes(const fm_ctx *c) {
    int tx, ty, Wp, Hp;
    umma_geom(c, &tx, &ty, &Wp, &Hp);
    return (size_t)c->S * c->Tmax * Wp * Hp;
}

size_t fm_umma_bg_doubles(const fm_ctx *c) {
    int tx, ty, Wp, Hp;
    umma_geom(c, &tx, &ty, &Wp, &Hp);
    return (size_t)c->S * tx * ty * UB_T * UB_T;
}

// band[u][q] = cRA[q - u], u in [-boff, 128), q in [0, 32), cRA = the taps centred in a (2 RA + 1)-tap window; stored in the
// blocked K-major order of the shared copy: [row group of 8][16-byte half][8 rows][16 bytes]
static std::vector<uint8_t> make_band(const fm_ctx *c, const int *taps, int RA, int brows, int boff) {
    std::vector<uint8_t> band((size_t)brows * 32, 0);
    const int shift = RA - (c->k >> 1);
    for (int ur = 0; ur < brows; ur++)
        for (int q = 0; q < 32; q++) {
            const int i = q - (ur - boff) - shift;
            if (i >= 0 && i < c->k) band[((ur >> 3) * 2 + (q >> 4)) * 128 + (ur & 7) * 16 + (q & 15)] = (uint8_t)taps[i];
        }
    return band;
}

// the BGR (and RGB) frames can feed the tcgen05 kernel directly (TMA over the caller's frames, mirroring inside the tile);
// gray and four-byte frames take the apron plane, which k_pad_gray fills from them in place
static bool umma_fused_geometry(const fm_ctx *c) {
    const int r = c->k >> 1;
    return c->resize_mode == 0 && (c->W % 16) == 0 && c->w >= r + 2 && c->h >= r + 2 && c->px_bytes == 3;
}

template <bool RGB>
static int umma_fused_smem(const fm_ctx *c) {
    int rc;
    if ((rc = fm_ensure_smem((const void *)k_umma_fused<16, true, RGB>, UfGeom<16>::SMEM, c->cfg.device))) return rc;
    if ((rc = fm_ensure_smem((const void *)k_umma_fused<16, false, RGB>, UfGeom<16>::SMEM, c->cfg.device))) return rc;
    if ((rc = fm_ensure_smem((const void *)k_umma_fused<48, true, RGB>, UfGeom<48>::SMEM, c->cfg.device))) return rc;
    return fm_ensure_smem((const void *)k_umma_fused<48, false, RGB>, UfGeom<48>::SMEM, c->cfg.device);
}

int fm_umma_init(fm_ctx *c, const int *taps) {
    std::vector<uint8_t> band = make_band(c, taps, UB_PAD, UB_BROWS, UB_BOFF);
    FM_CUDA(cudaMalloc((void **)&c->uband, band.size()));
    FM_CUDA(cudaMemcpy(c->uband, band.data(), band.size(), cudaMemcpyHostToDevice));
    int rc;
    if (!fm_tma_encoder()) { fm_set_error("cuTensorMapEncodeTiled not available"); return FM_ECUDA; }
    c->umma_direct = umma_fused_geometry(c);
    if (c->umma_direct) {
        c->umma_ra = (c->k >> 1) <= 16 ? 16 : 48;
        band = c->umma_ra == 16 ? make_band(c, taps, 16, UfGeom<16>::BROWS, UfGeom<16>::BOFF)
                                : make_band(c, taps, 48, UfGeom<48>::BROWS, UfGeom<48>::BOFF);
        FM_CUDA(cudaMalloc((void **)&c->uband_f, band.size()));
        FM_CUDA(cudaMemcpy(c->uband_f, band.data(), band.size(), cudaMemcpyHostToDevice));
        if ((rc = c->rgb ? umma_fused_smem<true>(c) : umma_fused_smem<false>(c))) return rc;
    } else {
        FM_CUDA(cudaMalloc((void **)&c->gpad, fm_umma_pad_bytes(c)));      // apron plane of the resize modes
    }
    if ((rc = fm_ensure_smem((const void *)k_umma_blur<true>, UB_SMEM, c->cfg.device))) return rc;
    if ((rc = fm_ensure_smem((const void *)k_umma_blur<false>, UB_SMEM, c->cfg.device))) return rc;
    return FM_OK;
}

static void umma_params(fm_ctx *c, int T, int tilesX, int tilesY, UmmaParams &p) {
    p.bg = c->bg; p.maskbits = c->maskbits; p.tbits = c->tflat;
    p.flatwords = (size_t)c->ntiles * FM_TILE_WORDS;
    p.state = c->state; p.nvalid = c->nvalid; p.rawrange = c->rawrange;
    p.blur_out = (c->cfg.flags & FM_FLAG_KEEP_PLANES) ? c->blur : nullptr;
    p.T = T; p.w = c->w; p.h = c->h; p.wpr = c->wpr; p.tilesX = tilesX; p.tilesY = tilesY; p.threshold = c->cfg.threshold;
    p.alpha = c->cfg.avg; p.beta = 1.0 - p.alpha;
    p.qoff = 0x4B400000 - p.threshold; p.thr2 = 2u * (uint32_t)p.threshold; p.nC = -(4503599627370496.0 * p.alpha);
    p.prof = nullptr;
}

static long long *umma_prof_buffer() {              // FM_UMMA_PROF=1: managed buffer, dumped by fm_umma_prof_dump()
    static long long *buf = nullptr;
    if (!buf && getenv("FM_UMMA_PROF")) {
        if (cudaMallocManaged(&buf, 32 * sizeof(long long)) != cudaSuccess) buf = nullptr;
        else memset(buf, 0, 32 * sizeof(long long));
    }
    return buf;
}

extern "C" void fm_umma_prof_dump(void) {
    long long *b = umma_prof_buffer();
    if (!b) return;
    cudaDeviceSynchronize();
    for (int k = 0; k < 2; k++)
        fprintf(stderr, "umma phases (cycles, interior CTA, thread %d): wait_mma1 %lld issue_tma %lld split %lld fence_proxy %lld barrier %lld "
                "mma_issue %lld wait_mma2 %lld epilogue %lld end_sync %lld\n", k ? 992 : 0, b[16 * k + 0], b[16 * k + 1], b[16 * k + 2],
                b[16 * k + 3], b[16 * k + 4], b[16 * k + 5], b[16 * k + 6], b[16 * k + 7], b[16 * k + 8]);
    memset(b, 0, 32 * sizeof(long long));
}

template <bool RGB>
static void umma_fused_launch(int RA, bool safe, dim3 grid, cudaStream_t st, const CUtensorMap &tmap, const UfParams &q) {
    if (RA == 16) {
        if (safe) k_umma_fused<16, true, RGB><<<grid, UB_THREADS, UfGeom<16>::SMEM, st>>>(tmap, q);
        else k_umma_fused<16, false, RGB><<<grid, UB_THREADS, UfGeom<16>::SMEM, st>>>(tmap, q);
    } else {
        if (safe) k_umma_fused<48, true, RGB><<<grid, UB_THREADS, UfGeom<48>::SMEM, st>>>(tmap, q);
        else k_umma_fused<48, false, RGB><<<grid, UB_THREADS, UfGeom<48>::SMEM, st>>>(tmap, q);
    }
}

// full-resolution mode, BGR (or RGB) frames straight into the tcgen05 kernel
static int launch_umma_fused(fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, size_t pitch, int T, cudaStream_t st) {
    int tilesX, tilesY, Wp, Hp;
    umma_geom(c, &tilesX, &tilesY, &Wp, &Hp);
    if (c->cfg.flags & FM_FLAG_KEEP_PLANES) {              // parity tap of the gray conversion
        int rc = fm_launch_gray_plane(c, frames, sstride, fstride, pitch, T, st);
        if (rc) return rc;
    }
    const int RA = c->umma_ra;
    CUtensorMap tmap;
    int rc = fm_frames_tmap(c, frames, sstride, fstride, pitch, T, 3 * (UB_T + 2 * RA) / 4, RA == 16 ? UfGeom<16>::RC : UfGeom<48>::RC, &tmap);
    if (rc) return rc;
    UfParams q;
    umma_params(c, T, tilesX, tilesY, q.u);
    q.u.band = c->uband_f;
    q.r = c->k >> 1;
    const bool safe = q.u.alpha >= 0.0 && q.u.alpha <= 1.0 && q.u.threshold >= 0;
    dim3 grid(tilesX * tilesY, c->S);
    if (c->rgb) umma_fused_launch<true>(RA, safe, grid, st, tmap, q);
    else umma_fused_launch<false>(RA, safe, grid, st, tmap, q);
    FM_LAUNCH_CHECK();
    return FM_OK;
}

// frames != nullptr: full-resolution mode (BGR -> padded gray in one kernel); else the resized gray plane c->gray.  Pitched
// rows that TMA cannot read (not 16-byte aligned) take the apron plane; packed ones keep the direct kernel's refusal.
int fm_launch_umma_blur(fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, size_t pitch, int T, cudaStream_t st) {
    const bool tma_ok = pitch == (size_t)c->W * c->px_bytes || ((((uintptr_t)frames) | sstride | fstride | pitch) & 15) == 0;
    if (frames && c->umma_direct && !(c->cfg.flags & FM_FLAG_UMMA_APRON) && tma_ok)
        return launch_umma_fused(c, frames, sstride, fstride, pitch, T, st);
    if (!c->gpad) {                     // first call that needs the apron plane (A/B flag on a direct-capable context)
        FM_CUDA(cudaStreamSynchronize(st));
        FM_CUDA(cudaMalloc((void **)&c->gpad, fm_umma_pad_bytes(c)));
    }
    int tilesX, tilesY, Wp, Hp;
    umma_geom(c, &tilesX, &tilesY, &Wp, &Hp);
    const int F = c->S * T;
    dim3 pgrid((Wp / 4 + 255) / 256, Hp, F);
    const bool gray_in = frames && c->px_bytes == 1;
    if (frames && (c->cfg.flags & FM_FLAG_KEEP_PLANES)) {      // parity tap of the gray conversion (gray frames: a copy)
        int rc = fm_launch_gray_plane(c, frames, sstride, fstride, pitch, T, st);
        if (rc) return rc;
    }
    if (frames && !gray_in) {
        const int al = ((((uintptr_t)frames) | sstride | fstride | pitch | ((size_t)c->W * c->px_bytes)) & 3) == 0;
        fm_px_dispatch(c->px_bytes, c->rgb, [&](auto Cx, auto RGB) {
            constexpr int P = Cx.value == 4 ? 4 : 3;
            k_pad_gray<true, RGB.value, P><<<pgrid, 256, 0, st>>>(frames, sstride, fstride, pitch, T, c->gpad, c->w, c->h, Wp, Hp,
                                                                  c->nvalid, al);
        });
    } else if (gray_in) {
        const int al = ((((uintptr_t)frames) | sstride | fstride | pitch | ((size_t)c->W * c->px_bytes)) & 3) == 0;
        k_pad_gray<false><<<pgrid, 256, 0, st>>>(frames, sstride, fstride, pitch, T, c->gpad, c->w, c->h, Wp, Hp, c->nvalid, al);
    } else {
        const int al = (c->w & 3) == 0;
        k_pad_gray<false><<<pgrid, 256, 0, st>>>(c->gray, (size_t)T * c->N, (size_t)c->N, (size_t)c->w, T, c->gpad, c->w, c->h, Wp,
                                                 Hp, c->nvalid, al);
    }
    FM_LAUNCH_CHECK();
    CUtensorMap tmap;
    cuuint64_t dims[4] = {(cuuint64_t)Wp, (cuuint64_t)Hp, (cuuint64_t)T, (cuuint64_t)c->S};
    cuuint64_t strides[3] = {(cuuint64_t)Wp, (cuuint64_t)Wp * Hp, (cuuint64_t)Wp * Hp * T};
    cuuint32_t box[4] = {128, UB_IN, 1, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = fm_tma_encoder()(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, (void *)c->gpad, dims, strides, box, estr,
                                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { fm_set_error("cuTensorMapEncodeTiled (padded gray plane) failed (%d)", (int)r); return FM_ECUDA; }
    UmmaParams p;
    umma_params(c, T, tilesX, tilesY, p);
    p.band = c->uband;
    p.prof = umma_prof_buffer();
    const bool safe = p.alpha >= 0.0 && p.alpha <= 1.0 && p.threshold >= 0;
    dim3 grid(tilesX * tilesY, c->S);
    if (safe) k_umma_blur<true><<<grid, UB_THREADS, UB_SMEM, st>>>(tmap, p);
    else k_umma_blur<false><<<grid, UB_THREADS, UB_SMEM, st>>>(tmap, p);
    FM_LAUNCH_CHECK();
    return FM_OK;
}

int fm_launch_bg_export_umma(fm_ctx *c, int stream, double *dst_dev, cudaStream_t st) {
    int tilesX, tilesY, Wp, Hp;
    umma_geom(c, &tilesX, &tilesY, &Wp, &Hp);
    dim3 grid((c->w + 127) / 128, c->h);
    k_bg_export_umma<<<grid, 128, 0, st>>>(c->bg, dst_dev, c->w, c->h, tilesX, tilesY, stream);
    FM_LAUNCH_CHECK();
    return FM_OK;
}
