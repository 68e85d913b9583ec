// Device primitives shared by the front-end kernels (sm_100a only): the TMA / mbarrier and u8 tensor-core (mma.sync)
// wrappers, and the reference's per-pixel arithmetic -- gray (SURVEY.md A.2), BORDER_REFLECT_101, the polygon mask
// painted into the blur (find_motion.py:619-635) and one pixel of the temporal stage (A.4, A.6, A.7).  Every kernel
// that computes one of these calls the copy here, so the bit-exact arithmetic has a single definition.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

// ---- TMA / mbarrier ----
__device__ __forceinline__ uint32_t fm_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void fm_mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(fm_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fm_mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(fm_smem_u32(bar)), "r"(bytes) : "memory");
}
// bar: shared-window address of the barrier (fm_smem_u32), for loops that keep it in a register
__device__ __forceinline__ void fm_mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void fm_mbar_wait(uint64_t *bar, uint32_t parity) { fm_mbar_wait(fm_smem_u32(bar), parity); }
// box (c0, c1, c2, c3) of a 4-D tensor map -> shared memory at `dst`; completes a transaction on `bar`
__device__ __forceinline__ void fm_tma_load_4d(uint32_t dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1, int c2,
                                               int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(dst), "l"(map), "r"(fm_smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void fm_tma_load_4d(void *dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1, int c2, int c3) {
    fm_tma_load_4d(fm_smem_u32(dst), map, bar, c0, c1, c2, c3);
}

// ---- u8 x u8 -> s32 products on the tensor cores (IMMA.16832.U8) ----
__device__ __forceinline__ void fm_ldsm_x4(uint32_t addr, uint32_t (&r)[4]) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
// D += A * B
__device__ __forceinline__ void fm_imma(int (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                        uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+r"(d[0]), "+r"(d[1]), "+r"(d[2]), "+r"(d[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
// D = A * B + c (the same constant in all four lanes): the first step of a chain
__device__ __forceinline__ void fm_imma0(int (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                         uint32_t b1, int c) {
    asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%10,%10,%10};"
                 : "=r"(d[0]), "=r"(d[1]), "=r"(d[2]), "=r"(d[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1), "r"(c));
}

// ---- gray (SURVEY.md A.2): Y = (3735 B + 19235 G + 9798 R + 16384) >> 15 ----
__device__ __forceinline__ uint32_t fm_gray(uint32_t b, uint32_t g, uint32_t r) {
    return (3735u * b + 19235u * g + 9798u * r + 16384u) >> 15;
}
// 4 BGR pixels in 3 words -> 4 gray bytes.  The same Y computed as (7470 B + 38470 G + 19596 R + 32768) >> 16 with two
// 16-bit x 8-bit dot products per pixel (IDP.2A); the lo/hi byte-pair selection of IDP.2A picks each pixel's bytes straight
// out of the three words.  The result is byte 2 of the accumulator.
__device__ __forceinline__ uint32_t fm_gray4(uint32_t w0, uint32_t w1, uint32_t w2) {
    const uint32_t C_BG = 7470u | (38470u << 16), C_R = 19596u;              // byte pairs [B,G], [R,x]
    const uint32_t C_xB = 7470u << 16, C_GR = 38470u | (19596u << 16);       // byte pairs [x,B], [G,R]
    uint32_t t0 = __dp2a_hi(C_R, w0, __dp2a_lo(C_BG, w0, 32768u));           // w0 = [B0,G0,R0,B1]
    uint32_t t1 = __dp2a_hi(C_xB, w0, __dp2a_lo(C_GR, w1, 32768u));          // w1 = [G1,R1,B2,G2]
    uint32_t t2 = __dp2a_hi(C_BG, w1, __dp2a_lo(C_R, w2, 32768u));           // w2 = [R2,B3,G3,R3]
    uint32_t t3 = __dp2a_hi(C_GR, w2, __dp2a_lo(C_xB, w2, 32768u));
    return __byte_perm(__byte_perm(t0, t1, 0x0062), __byte_perm(t2, t3, 0x0062), 0x5410);
}

// ---- NV12 -> BGR exactly as cv2.cvtColor(COLOR_YUV2BGR_NV12): ITU-R BT.601 in 20-bit fixed point ----
//   y' = max(Y - 16, 0) * 1220542,  u = U - 128,  v = V - 128
//   R = sat((y' + 1673527 v + 2^19) >> 20),  G = sat((y' - 852492 v - 409993 u + 2^19) >> 20),  B = sat((y' + 2116026 u + 2^19) >> 20)
// Chroma is nearest-neighbour (pixel (x, y) takes the U, V pair of UV row y/2, column pair x/2), so the chroma terms,
// with the rounding folded in, are computed once per 2x2 block (fm_nv12_chroma) and shared by its four pixels.
// Every intermediate fits an int32: |y'| + |2116026 u| < 2^30.
struct FmChroma {
    int r, g, b;
};
__device__ __forceinline__ FmChroma fm_nv12_chroma(uint32_t u, uint32_t v) {
    const int uu = (int)u - 128, vv = (int)v - 128;
    return FmChroma{1673527 * vv + (1 << 19), -852492 * vv - 409993 * uu + (1 << 19), 2116026 * uu + (1 << 19)};
}
__device__ __forceinline__ uint32_t fm_sat_q20(int x) { return (uint32_t)min(max(x >> 20, 0), 255); }
__device__ __forceinline__ void fm_nv12_bgr(uint32_t y, const FmChroma &c, uint32_t &b, uint32_t &g, uint32_t &r) {
    const int yy = max((int)y - 16, 0) * 1220542;
    b = fm_sat_q20(yy + c.b);
    g = fm_sat_q20(yy + c.g);
    r = fm_sat_q20(yy + c.r);
}
__device__ __forceinline__ uint32_t fm_nv12_gray(uint32_t y, const FmChroma &c) {
    uint32_t b, g, r;
    fm_nv12_bgr(y, c, b, g, r);
    return fm_gray(b, g, r);
}

__device__ __forceinline__ int fm_reflect101(int i, int n) {
    // BORDER_REFLECT_101 for any offset
    if ((unsigned)i < (unsigned)n) return i;
    if (n == 1) return 0;
    int p = 2 * (n - 1);
    i %= p;
    if (i < 0) i += p;
    return i >= n ? p - i : i;
}

// rn(byte i of w * a) in one FFMA: (2^23 + byte) * a - 2^23 * a is exactly byte * a before the single rounding (2^23 * a is
// exact), i.e. the same float32 as the reference's unfused product; na = -(2^23 * a).  The byte is placed into the
// mantissa of 2^23 by PRMT: no byte loads, no XU conversions.
__device__ __forceinline__ float fm_byte_mul(uint32_t w, int i, float a, float na) {
    return __fmaf_rn(__uint_as_float(__byte_perm(w, 0x4B000000u, 0x7540u | (uint32_t)i)), a, na);
}

// mask_off_areas paints BLACK into the blur: byte i of `bytes4` cleared where bit i of m4 (< 16) is set
__device__ __forceinline__ uint32_t fm_clear_masked4(uint32_t bytes4, uint32_t m4) {
    return bytes4 & ~(((m4 * 0x00204081u) & 0x01010101u) * 0xFFu);
}

// ---- temporal stage (SURVEY.md A.4, A.6, A.7) ----
__device__ __forceinline__ double fm_u8_to_f64(uint32_t v) {
    // exact: 2^52 + v, minus 2^52 (avoids the slow I2F.F64 conversion)
    return __hiloint2double(0x43300000, (int)v) - 4503599627370496.0;
}

// bg8 = sat(rne(|float32(bg)|)): convertScaleAbs of the background
__device__ __forceinline__ uint32_t fm_bg8(double bg) {
    float f = fabsf(__double2float_rn(bg));        // double -> float32 first (A.7)
    f = fminf(f, 255.0f);
    // rne to integer through the 1.5*2^23 trick (f in [0, 255])
    return __float_as_uint(__fadd_rn(f, 12582912.0f)) & 0x1FFu;
}

// One pixel of one frame: blur byte sv against the float64 background bg.  Pushes the threshold bit
// (|blur - bg8| > threshold) into bits (bits = 2 bits + bit) and updates bg = fma(bg, 1 - alpha, rn(blur * alpha)).
// INIT: first frame of the stream (ref_frame = blur.astype(float)).
// SAFE: alpha in [0, 1] and threshold >= 0, so bg stays in [0, 255] (no fabs / saturation); then
//   rn(blur * alpha) = fma(2^52 + blur, alpha, nC) exactly, nC = -(2^52 alpha), without an int -> double conversion, and
//   the bit is the carry of (bg8 + 0x4B400000) - qoff - blur + nthr2 (qoff = 0x4B400000 - threshold,
//   nthr2 = ~(2 threshold)): that difference lies in [0, 2 threshold] exactly when |blur - bg8| <= threshold.
// Otherwise: the plain comparison, correct for every threshold (qoff, nthr2 and nC are not used).
template <bool SAFE, bool INIT>
__device__ __forceinline__ void fm_temporal_px(uint32_t sv, double &bg, uint32_t &bits, int threshold, int qoff, uint32_t nthr2,
                                               double alpha, double beta, double nC) {
    if (SAFE) {
        const double X = __hiloint2double(0x43300000, (int)sv);          // 2^52 + blur
        if (INIT) bg = X - 4503599627370496.0;
        const int q = __float_as_int(__fadd_rn(__double2float_rn(bg), 12582912.0f));     // 0x4B400000 + bg8
        asm("{\n .reg .u32 t;\n add.cc.u32 t, %1, %2;\n addc.u32 %0, %0, %0;\n}"
            : "+r"(bits) : "r"((uint32_t)(q - qoff - (int)sv)), "r"(nthr2));
        bg = __fma_rn(bg, beta, __fma_rn(X, alpha, nC));
    } else {
        const double sd = fm_u8_to_f64(sv);
        if (INIT) bg = sd;
        int d = (int)sv - (int)fm_bg8(bg);
        d = d < 0 ? -d : d;
        bits = 2u * bits + (d > threshold ? 1u : 0u);
        bg = __fma_rn(bg, beta, __dmul_rn(sd, alpha));
    }
}
