// Wide-kernel Gaussian blur (any k that the fused kernel does not take: 7 ... 97 ... 193 ... 385 ...) as two
// banded (Toeplitz) u8 x u8 -> s32 matrix products on the tensor cores (IMMA.16832.U8.U8, 1.13 Pop/s measured
// on B200 against 0.15 Pop/s for IDP.4A: profiles/micro/mma_rate.cu).
// Replaces cv2.GaussianBlur(gray, (k,k), 0) of blur_frame (find_motion/find_motion.py:494; SURVEY.md A.3) and the
// polygon masks painted into the blur (fm.py:619-635).  Integer arithmetic throughout: bit-exact.
//
// Pass 1 (k_wide_h), horizontal: D[row][col] = sum_j gray[row][col + j - r] * c[j].
//   A = 16 gray rows x 32 columns (ldmatrix from a shared tile with the BORDER_REFLECT_101 columns and rows
//   materialised), B = the taps as a banded 32 x 8 block that depends only on (window step, column block).
//   The 16-bit sums are split into a low-byte and a high-byte plane, laid out for pass 2:
//     plane[frame][group of 32 padded rows][half][column][4 words],   word (4*half + j) byte i = row j' + 8 i of
//   the group (j' = 4*half + j), i.e. the 16 bytes of a (column, half) are one ldmatrix row.
//   Padded row p holds image row reflect101(p - r), so pass 2 has no border logic.
//   In full-resolution mode the BGR -> gray conversion (fm.py:493, SURVEY.md A.2) is fused into the staging of
//   the shared tile, so no gray plane is written or read.
// Pass 2 (k_wide_v), vertical: out[y][x] = (256 * sum_j hi[y + j][x] c[j] + sum_j lo[y + j][x] c[j] + 32768) >> 16.
//   A = the taps as a banded 16 x 32 block with the k index permuted to the row order of the plane words
//   (k = 4t+i <-> row t + 8i, k = 16+4t+i <-> row 4 + t + 8i), B = 32 padded rows x 8 columns of a byte plane
//   (ldmatrix.x4 = two column blocks).  The columns of a block are permuted (block nb holds columns
//   8t' + 2nb + e) so that a thread ends up with 8 consecutive output bytes of a row: mask, two 32-bit stores.
//   The planes stream through a cp.async double buffer along a strip of column tiles.
#include <cuda.h>

#include <algorithm>
#include <cstdlib>
#include <type_traits>

#include "fm_common.cuh"

#define WH_COLS 256        // pass 1 CTA tile: 32 padded rows (one group) x 256 columns, 8 warps of 32 x 32
#define WH_THREADS 256
#define WV_ROWS 128        // pass 2 CTA tile: 128 output rows x 32 columns per step, 4 warps of 32 x 32
#define WV_COLS 32
#define WV_NT 4            // column tiles per pass-2 CTA (cp.async double buffer)
#define WT_COLS 16         // columns of a k_wide_vt CTA

__device__ __forceinline__ void wcp_async16(uint32_t dst, const void *src, bool valid) {
    const int n = valid ? 16 : 0;                 // src-size 0: the 16 bytes are zero-filled
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(n) : "memory");
}

struct WideGeom {
    int k, r;
    int R16;        // left pad of the pass-1 window, r rounded up to 16
    int Sh;         // 32-column steps of a pass-1 warp window
    int Sv;         // 32-row groups of a pass-2 warp window
    int pitch;      // bytes per row of the pass-1 shared tile
    int NGa;        // allocated row groups per frame
};

static WideGeom wide_geom(const fm_ctx *c) {
    WideGeom g;
    g.k = c->k; g.r = c->k >> 1;
    g.R16 = (g.r + 15) / 16 * 16;
    g.Sh = (g.R16 + 32 + g.r + 31) / 32;
    g.Sv = 1 + (2 * g.r + 31) / 32;
    int L = WH_COLS - 32 + 32 * g.Sh;                                  // the last warp's last step ends here
    while ((L % 128) != 16 && (L % 128) != 48 && (L % 128) != 80 && (L % 128) != 112) L += 16;   // ldmatrix: 8 rows -> 8 bank groups
    g.pitch = L;
    g.NGa = (c->h + 31) / 32 + g.Sv - 1;
    return g;
}

size_t fm_wide_plane_bytes(const fm_ctx *c) {
    WideGeom g = wide_geom(c);
    return (size_t)c->S * c->Tmax * g.NGa * 2 * c->w * 16;          // one byte plane
}

// Tap tables, per lane (g = lane >> 2, t = lane & 3).
// Pass 1 (B operand, uint2): entry d = 4 s - nb + 3 (s = window step, nb = 8-column output block); register rg
//   byte i is the tap 8 (d - 3) + kk - g + r - R16 with kk = 16 rg + 4 t + i.
// Pass 2 (A operand, uint4): entry e = 2 s - mt + 1 (s = row group of the window, mt = 16-row output tile);
//   registers a0..a3 = (m = g, g+8, g, g+8; k = 4t+i, 4t+i, 16+4t+i, 16+4t+i), tap 16 (e - 1) + row(k) - m.
int fm_wide_init(fm_ctx *c, const int *taps) {
    WideGeom g = wide_geom(c);
    {   // shared-memory needs of the three kernels, checked when the context is created
        const size_t smh = (size_t)32 * g.pitch + (size_t)(4 * g.Sh + 3) * 256;
        const size_t smv = (size_t)4 * (4 + g.Sv - 1) * 2 * WV_COLS * 16 + (size_t)2 * g.Sv * 512;
        const size_t smt = (size_t)4 * (4 + g.Sv - 1) * 2 * WT_COLS * 16 + (size_t)2 * g.Sv * 512 + WV_ROWS * 16;
        if (smh > 200 * 1024 || smv > 200 * 1024 || smt > 200 * 1024) {
            fm_set_error("Gaussian kernel %d too wide for the tensor-core blur (%zu / %zu / %zu bytes of shared memory)", c->k,
                         smh, smv, smt);
            return FM_ERANGE;
        }
    }
    const int nh = 4 * g.Sh + 3, nv = 2 * g.Sv;
    const size_t words = (size_t)nh * 32 * 2 + (size_t)nv * 32 * 4;
    uint32_t *hh = (uint32_t *)malloc(words * 4);
    if (!hh) { fm_set_error("out of host memory"); return FM_ENOMEM; }
    uint32_t *hv = hh + (size_t)nh * 32 * 2;
    auto tap = [&](int j) -> uint32_t { return (j >= 0 && j < g.k) ? (uint32_t)(taps[j] & 255) : 0u; };
    for (int d = 0; d < nh; d++)
        for (int lane = 0; lane < 32; lane++) {
            const int gq = lane >> 2, t = lane & 3;
            for (int rg = 0; rg < 2; rg++) {
                uint32_t v = 0;
                for (int i = 0; i < 4; i++) v |= tap(8 * (d - 3) + (16 * rg + 4 * t + i) - gq + g.r - g.R16) << (8 * i);
                hh[((size_t)d * 32 + lane) * 2 + rg] = v;
            }
        }
    for (int e = 0; e < nv; e++)
        for (int lane = 0; lane < 32; lane++) {
            const int gq = lane >> 2, t = lane & 3;
            for (int a = 0; a < 4; a++) {
                const int m = gq + 8 * (a & 1), half = a >> 1;
                uint32_t v = 0;
                for (int i = 0; i < 4; i++) v |= tap(16 * (e - 1) + (4 * half + t + 8 * i) - m) << (8 * i);
                hv[((size_t)e * 32 + lane) * 4 + a] = v;
            }
        }
    cudaError_t er = cudaMalloc((void **)&c->wtab, words * 4);
    if (er == cudaSuccess) er = cudaMemcpy(c->wtab, hh, words * 4, cudaMemcpyHostToDevice);
    free(hh);
    if (er != cudaSuccess) { fm_set_error("wide-blur tap tables: %s", cudaGetErrorString(er)); return FM_ECUDA; }
    return FM_OK;
}

// source row of padded row index i (BORDER_REFLECT_101).  One reflection is enough when the plane is taller than
// the kernel radius; rows past the padded range (their taps are all zero) only have to stay inside the plane.
__device__ __forceinline__ int wrow(int i, int n) {
    if (i >= 0 && i < n) return i;
    const int j = i < 0 ? -i : 2 * n - 2 - i;
    return (j >= 0 && j < n) ? j : fm_reflect101(i, n);
}

// BORDER_REFLECT_101 columns of a staged window from their mirror images inside the window (one reflection)
__device__ __forceinline__ void wide_h_mirror(unsigned char *tile, int X0, int w, int r, int R16, int pitch) {
    const int tid = threadIdx.x;
    const int nl = X0 == 0 ? R16 : 0;                    // shared columns [0, nl) are x < 0
    const int c0 = w - X0 + R16;                         // shared column of x = w
    const int nr = X0 + WH_COLS + r > w ? r : 0;
    for (int i = tid; i < 32 * (nl + nr); i += WH_THREADS) {
        const int rr = i / (nl + nr), j = i - rr * (nl + nr);
        const int c = j < nl ? j : c0 + (j - nl);
        const int cm = j < nl ? 2 * R16 - c : 2 * (c0 - 1) - c;      // x -> -x, x -> 2w - 2 - x
        tile[rr * pitch + c] = tile[rr * pitch + cm];
    }
}

// ---- pass 1, step A: stage the gray window of a CTA (shared column cc <-> image column X0 - R16 + cc, reflected; row rr <->
// padded row 32 G + rr) with register-staged global loads.  BGR: the BGR -> gray conversion is fused in (RGB: R-first
// pixels; PX = 4: four-byte BGRA / RGBA pixels). ----
template <bool BGR, bool RGB = false, int PX = 3>
__device__ __forceinline__ void wide_h_stage(unsigned char *tile, const uint8_t *__restrict__ src, size_t sstride, size_t fstride,
                                             size_t rpitch, int T, int f, int G, int X0, int w, int h, int r, int R16, int pitch) {
    const int tid = threadIdx.x, lane = tid & 31, wq = tid >> 5;
    if (BGR) {
        // warp wq: rows wq, wq+8, wq+16, wq+24; lane: a unit of 16 pixels = 48 BGR bytes (three 128-bit loads; PX = 4:
        // 64 bytes, four); the loads of the four rows are issued before the first conversion
        const uint8_t *fr = src + (size_t)(f / T) * sstride + (size_t)(f % T) * fstride;
        const uint8_t *rp[4];
#pragma unroll
        for (int i = 0; i < 4; i++) rp[i] = fr + (size_t)wrow(32 * G + wq + 8 * i - r, h) * rpitch;
        const int upr = pitch >> 4;
        const int xneed = min(X0 + WH_COLS, w) + r;           // first column no output of this CTA reads
        const bool mirror = R16 < w && R16 + r < WH_COLS;      // border columns are copies of staged columns (one reflection)
        for (int u = lane; u < upr; u += 32) {
            const int x = X0 - R16 + 16 * u;
            if (x >= xneed) continue;
            if (x >= 0 && x + 15 < w) {
                uint4 raw[4][PX];
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const uint4 *q = reinterpret_cast<const uint4 *>(rp[i] + PX * x);
#pragma unroll
                    for (int k = 0; k < PX; k++) raw[i][k] = __ldg(q + k);
                }
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    uint4 o;
                    if constexpr (PX == 4) {
                        o = make_uint4(fm_gray4a<RGB>(raw[i][0]), fm_gray4a<RGB>(raw[i][1]), fm_gray4a<RGB>(raw[i][2]),
                                       fm_gray4a<RGB>(raw[i][3]));
                    } else {
                        o.x = fm_gray4<RGB>(raw[i][0].x, raw[i][0].y, raw[i][0].z);
                        o.y = fm_gray4<RGB>(raw[i][0].w, raw[i][1].x, raw[i][1].y);
                        o.z = fm_gray4<RGB>(raw[i][1].z, raw[i][1].w, raw[i][2].x);
                        o.w = fm_gray4<RGB>(raw[i][2].y, raw[i][2].z, raw[i][2].w);
                    }
                    *reinterpret_cast<uint4 *>(tile + (wq + 8 * i) * pitch + 16 * u) = o;
                }
            } else if (!mirror || (PX == 4 && x >= 0 && x < w)) {
                // PX = 4: rows of 4 W bytes are 16-byte aligned for any W % 4 == 0, so the last unit may straddle the right
                // edge (three-byte rows are aligned only for W % 16 == 0); its columns inside the image are staged here
#pragma unroll 1
                for (int b = 0; b < 16; b++) {
                    const int xx = PX * fm_reflect101(x + b, w);
#pragma unroll
                    for (int i = 0; i < 4; i++) tile[(wq + 8 * i) * pitch + 16 * u + b] = (unsigned char)fm_gray<RGB>(rp[i][xx], rp[i][xx + 1], rp[i][xx + 2]);
                }
            }
        }
        if (mirror && (X0 == 0 || X0 + WH_COLS + r > w)) {       // BORDER_REFLECT_101 columns from their mirror images
            __syncthreads();
            wide_h_mirror(tile, X0, w, r, R16, pitch);
        }
    } else {
        const int words = pitch >> 2;
        const uint8_t *fr = src + (size_t)(f / T) * sstride + (size_t)(f % T) * fstride;
#pragma unroll 1
        for (int rr = wq; rr < 32; rr += WH_THREADS / 32) {
            const uint8_t *row = fr + (size_t)wrow(32 * G + rr - r, h) * rpitch;
            uint32_t *trow = reinterpret_cast<uint32_t *>(tile + rr * pitch);
            for (int cw = lane; cw < words; cw += 32) {
                const int x = X0 - R16 + 4 * cw;
                if (x >= min(X0 + WH_COLS, w) + r) break;
                uint32_t v;
                if (x >= 0 && x + 3 < w && (((uintptr_t)(row + x)) & 3) == 0) v = __ldg(reinterpret_cast<const uint32_t *>(row + x));
                else {
                    v = 0;
#pragma unroll
                    for (int b = 0; b < 4; b++) v |= (uint32_t)row[wrow(x + b, w)] << (8 * b);
                }
                trow[cw] = v;
            }
        }
    }
}

// ---- pass 1, step B: the banded products of the staged window and the byte planes ----
__device__ __forceinline__ void wide_h_products(const unsigned char *tile, const uint2 *tab, int f, int G, int X0, int w, int Sh,
                                                int pitch, int NGa, uint32_t *__restrict__ plo, uint32_t *__restrict__ phi) {
    const int lane = threadIdx.x & 31, wq = threadIdx.x >> 5;
    if (X0 + 32 * wq >= w) return;                            // this warp's 32 columns are outside the image
    int acc[2][4][4];
    const uint32_t abase = fm_smem_u32(tile) + ((lane & 7) + 8 * ((lane >> 3) & 1)) * pitch + 32 * wq + 16 * (lane >> 4);
    auto step = [&](int s, auto first) {
        uint32_t a0[4], a1[4];
        fm_ldsm_x4(abase + 32 * s, a0);
        fm_ldsm_x4(abase + 32 * s + 16 * pitch, a1);
#pragma unroll
        for (int nb = 0; nb < 4; nb++) {
            const uint2 b = tab[(4 * s - nb + 3) * 32 + lane];
            if (decltype(first)::value) {
                fm_imma0(acc[0][nb], a0[0], a0[1], a0[2], a0[3], b.x, b.y, 0);
                fm_imma0(acc[1][nb], a1[0], a1[1], a1[2], a1[3], b.x, b.y, 0);
            } else {
                fm_imma(acc[0][nb], a0[0], a0[1], a0[2], a0[3], b.x, b.y);
                fm_imma(acc[1][nb], a1[0], a1[1], a1[2], a1[3], b.x, b.y);
            }
        }
    };
    step(0, std::true_type());
#pragma unroll 1
    for (int s = 1; s < Sh; s++) step(s, std::false_type());
    // thread (g, t): rows g, g+8 (tile 0), g+16, g+24 (tile 1) of columns 2t, 2t+1 of each block = word g of the group
    const int g = lane >> 2, t = lane & 3;
    const int xb = X0 + 32 * wq + 2 * t;
    const size_t o0 = ((((size_t)f * NGa + G) * 2 + (g >> 2)) * w + xb) * 4 + (g & 3);
    uint32_t *ql = plo + o0, *qh = phi + o0;
#pragma unroll
    for (int nb = 0; nb < 4; nb++)
#pragma unroll
        for (int e = 0; e < 2; e++) {
            if (xb + 8 * nb + e < w) {
                const uint32_t p = __byte_perm(acc[0][nb][e], acc[0][nb][2 + e], 0x5140);     // [r0.b0, r8.b0, r0.b1, r8.b1]
                const uint32_t q = __byte_perm(acc[1][nb][e], acc[1][nb][2 + e], 0x5140);
                ql[(8 * nb + e) * 4] = __byte_perm(p, q, 0x5410);
                qh[(8 * nb + e) * 4] = __byte_perm(p, q, 0x7632);
            }
        }
}

// grid: (ceil(w / 256), NGa, F), 256 threads.  dynamic smem: 32 * pitch + (4 Sh + 3) * 256
// BGR: src = the caller's frames (identity resize, 16-byte aligned rows rpitch bytes apart); otherwise src = a gray plane, rows
// rpitch bytes apart (the context's [F][h][w], or the caller's gray frames with FM_FLAG_GRAY).  RGB: R-first frames; PX:
// bytes per pixel of the frames (3, or 4 with FM_FLAG_ALPHA)
template <bool BGR, bool RGB = false, int PX = 3>
__global__ void __launch_bounds__(WH_THREADS, 4) k_wide_h(const uint8_t *__restrict__ src, size_t sstride, size_t fstride,
                                                       size_t rpitch, int T,
                                                       uint32_t *__restrict__ plo, uint32_t *__restrict__ phi,
                                                       const uint2 *__restrict__ tabg, int w, int h, int r, int R16, int Sh,
                                                       int pitch, int NGa, const int *__restrict__ nvalid) {
    extern __shared__ __align__(16) unsigned char wsm[];
    unsigned char *tile = wsm;                                              // [32][pitch] gray bytes
    uint2 *tab = reinterpret_cast<uint2 *>(wsm + 32 * pitch);             // [4 Sh + 3][32]
    const int tid = threadIdx.x;
    const int f = blockIdx.z, G = blockIdx.y, X0 = blockIdx.x * WH_COLS;
    if (f % T >= __ldg(nvalid + f / T)) return;                             // not a real frame of this (ragged) call
    for (int i = tid; i < (4 * Sh + 3) * 32; i += WH_THREADS) tab[i] = __ldg(tabg + i);
    wide_h_stage<BGR, RGB, PX>(tile, src, sstride, fstride, rpitch, T, f, G, X0, w, h, r, R16, pitch);
    __syncthreads();
    wide_h_products(tile, tab, f, G, X0, w, Sh, pitch, NGa, plo, phi);
}

// The same pass with the BGR window staged by TMA (16-byte aligned frames, one-reflection borders): one thread issues one or two
// boxes of 32 rows x (ubox units of 16 pixels = 48 bytes) for the whole CTA, every lane then converts units out of shared memory
// (no per-thread global addresses, no idle lanes: 22 units per row at k = 97 left 10 of 32 lanes without work above).  Row groups
// that touch the top or bottom border need reflected rows and take the register-staged path.
// dynamic smem: nbox * 32 * ubox * 16 PX (raw pixels)  +  32 * pitch  +  (4 Sh + 3) * 256  +  16.  RGB: R-first frames; PX:
// bytes per pixel (3, or 4 with FM_FLAG_ALPHA: a unit of 16 pixels is four 16-byte words, each one gray word)
template <bool RGB = false, int PX = 3>
__global__ void __launch_bounds__(WH_THREADS, 4) k_wide_h_tma(const __grid_constant__ CUtensorMap tmap, const uint8_t *__restrict__ src,
                                                           size_t sstride, size_t fstride, size_t rpitch, int T,
                                                           uint32_t *__restrict__ plo,
                                                           uint32_t *__restrict__ phi, const uint2 *__restrict__ tabg, int w, int h,
                                                           int r, int R16, int Sh, int pitch, int NGa,
                                                           const int *__restrict__ nvalid, int nunits, int ubox, int nbox, int gp) {
    extern __shared__ __align__(128) unsigned char wsmt[];
    constexpr int UB = 16 * PX;                                              // bytes of a unit of 16 pixels
    const int boxbytes = 32 * ubox * UB;                                     // a multiple of 128
    unsigned char *raw = wsmt;                                               // [nbox][32][ubox * 48] staged BGR rows
    unsigned char *tile = raw + nbox * boxbytes;                             // [32][pitch] gray bytes
    uint2 *tab = reinterpret_cast<uint2 *>(tile + 32 * pitch);              // [4 Sh + 3][32]
    uint64_t *bar = reinterpret_cast<uint64_t *>(tab + (4 * Sh + 3) * 32);
    const int tid = threadIdx.x;
    const int f = blockIdx.z, X0 = blockIdx.x * WH_COLS;
    if (f % T >= __ldg(nvalid + f / T)) return;                             // not a real frame of this (ragged) call
    // the CTA walks gp consecutive row groups: the box of group i + 1 is requested as soon as the conversion of group i has
    // consumed the raw stage, and lands while the products of group i run
    const int Gbeg = blockIdx.y * gp, Gend = min(Gbeg + gp, NGa);
    auto interior = [&](int G) { return 32 * G - r >= 0 && 32 * G - r + 32 <= h; };    // CTA-uniform
    auto issue = [&](int G) {                  // one thread
        fm_mbar_expect_tx(bar, (uint32_t)(nbox * boxbytes));
        const int c0 = (PX * (X0 - R16)) / 4;                                // u32 column (negative / past the row: zero-filled)
        for (int b = 0; b < nbox; b++) fm_tma_load_4d(fm_smem_u32(raw) + b * boxbytes, &tmap, bar, c0 + b * ubox * (UB / 4), 32 * G - r, f % T, f / T);
    };
    if (tid == 0) {
        fm_mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        if (interior(Gbeg)) issue(Gbeg);
    }
    for (int i = tid; i < (4 * Sh + 3) * 32; i += WH_THREADS) tab[i] = __ldg(tabg + i);
    __syncthreads();                                                         // the barrier is initialised for everybody
    const int xneed = min(X0 + WH_COLS, w) + r;                              // first column no output of this CTA reads
    const uint32_t inv = (65536u + nunits - 1) / nunits;                     // u / nunits == (u * inv) >> 16 for u * nunits < 65536
    uint32_t phase = 0;
    for (int G = Gbeg; G < Gend; G++) {
        const bool more = G + 1 < Gend && interior(G + 1);
        if (interior(G)) {
            fm_mbar_wait(bar, phase);
            phase ^= 1;
            for (int u = tid; u < 32 * nunits; u += WH_THREADS) {
                const int rr = (int)(((uint32_t)u * inv) >> 16), j = u - rr * nunits;
                const int x = X0 - R16 + 16 * j;
                if (x < 0 || x >= w || x >= xneed) continue;                 // border columns come from their mirror images below
                const int jb = j >= ubox ? 1 : 0;
                const uint4 *q = reinterpret_cast<const uint4 *>(raw + jb * boxbytes + rr * (ubox * UB) + (j - jb * ubox) * UB);
                uint4 o;
                if constexpr (PX == 4) {
                    o = make_uint4(fm_gray4a<RGB>(q[0]), fm_gray4a<RGB>(q[1]), fm_gray4a<RGB>(q[2]), fm_gray4a<RGB>(q[3]));
                } else {
                    const uint4 r0 = q[0], r1 = q[1], r2 = q[2];
                    o.x = fm_gray4<RGB>(r0.x, r0.y, r0.z);
                    o.y = fm_gray4<RGB>(r0.w, r1.x, r1.y);
                    o.z = fm_gray4<RGB>(r1.z, r1.w, r2.x);
                    o.w = fm_gray4<RGB>(r2.y, r2.z, r2.w);
                }
                *reinterpret_cast<uint4 *>(tile + rr * pitch + 16 * j) = o;
            }
            __syncthreads();                                                 // raw stage consumed, window written
            if (more && tid == 0) issue(G + 1);
            if (X0 == 0 || X0 + WH_COLS + r > w) {
                wide_h_mirror(tile, X0, w, r, R16, pitch);
                __syncthreads();
            }
        } else {
            wide_h_stage<true, RGB, PX>(tile, src, sstride, fstride, rpitch, T, f, G, X0, w, h, r, R16, pitch);
            __syncthreads();
            if (more && tid == 0) issue(G + 1);                              // the raw stage is not in use
        }
        wide_h_products(tile, tab, f, G, X0, w, Sh, pitch, NGa, plo, phi);
        if (G + 1 < Gend) __syncthreads();                                   // every warp is done with the window
    }
}

// shared slot of column c of a 32-column tile: the 8 columns {8t' + 2nb + e} of a block land in 8 different 16-byte lanes
__device__ __forceinline__ int wv_slot(int c) { return (c & 24) | ((c & 7) ^ (((c >> 3) & 3) << 1)); }

// grid: (ceil(w / (32 WV_NT)), ceil(h / 128), F), 128 threads.
// dynamic smem: 2 stages * 2 planes * (4 + Sv - 1) groups * 2 halves * 32 columns * 16 B  +  2 Sv * 512
__global__ void __launch_bounds__(128, 4) k_wide_v(const uint4 *__restrict__ plo, const uint4 *__restrict__ phi,
                                                uint8_t *__restrict__ blur, const uint4 *__restrict__ tabg, int w, int h,
                                                int Sv, int NGa, int wpr, int T, const uint32_t *__restrict__ maskbits,
                                                const int *__restrict__ nvalid) {
    extern __shared__ __align__(16) unsigned char wsm[];
    if ((int)blockIdx.z % T >= __ldg(nvalid + blockIdx.z / T)) return;      // not a real frame of this (ragged) call
    const int NGt = 4 + Sv - 1;
    const int per = NGt * 2 * WV_COLS;                                        // 16-byte chunks per plane and stage
    uint4 *sB = reinterpret_cast<uint4 *>(wsm);                               // [stage][plane][NGt][half][32 slots]
    uint4 *tab = sB + 4 * per;                                                // [2 Sv][32]
    uint4 *sT = tab + 2 * Sv * 32;                                            // [128 rows] 16 blur bytes
    const int tid = threadIdx.x, lane = tid & 31, wq = tid >> 5;
    const int f = blockIdx.z, Y0 = blockIdx.y * WV_ROWS, XS = blockIdx.x * (WV_COLS * WV_NT), G0 = Y0 >> 5;
    for (int i = tid; i < 2 * Sv * 32; i += 128) tab[i] = __ldg(tabg + i);
    const int nt = min(WV_NT, (w - XS + WV_COLS - 1) / WV_COLS);
    // staging: lane = column of the tile, warp = chunk row gh (2 * group + half) modulo 4, both planes
    const uint4 *gsrc = plo + (((size_t)f * NGa + G0) * 2 + wq) * w + XS + lane;
    const size_t pdiff = phi - plo;
    const uint32_t sdst = fm_smem_u32(sB) + (wq * WV_COLS + wv_slot(lane)) * 16;
    const int ghmax = min(2 * NGt, 2 * (NGa - G0));              // chunk rows that exist in the planes
    auto issue = [&](int ct) {
        const bool okx = XS + ct * WV_COLS + lane < w;
        const uint4 *sp = gsrc + ct * WV_COLS;
        uint32_t dp = sdst + (ct & 1) * 2 * per * 16;
#pragma unroll 1
        for (int gh = wq; gh < 2 * NGt; gh += 4) {
            const bool ok = okx && gh < ghmax;
            wcp_async16(dp, ok ? sp : plo, ok);
            wcp_async16(dp + per * 16, ok ? sp + pdiff : plo, ok);
            sp += 4 * (size_t)w;
            dp += 4 * WV_COLS * 16;
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    issue(0);
    const int g = lane >> 2, t = lane & 3;
    // ldmatrix rows of a pair of column blocks (nb = 2 np, 2 np + 1): matrices (nb0, half 0), (nb0, half 1), (nb1, half 0), (nb1, half 1)
    uint32_t boff[2];
#pragma unroll
    for (int np = 0; np < 2; np++) {
        const int mi = lane >> 3, n = lane & 7;
        const int nb = 2 * np + (mi >> 1), half = mi & 1;
        const int col = 8 * (n >> 1) + 2 * nb + (n & 1);
        boff[np] = (half * WV_COLS + wv_slot(col)) * 16;
    }
    for (int ct = 0; ct < nt; ct++) {
        if (ct + 1 < nt) {
            issue(ct + 1);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
        const int X0 = XS + ct * WV_COLS;
        int acc[2][2][4][4];       // [plane][row tile][column block][4]; the low plane starts at the rounding constant
        const uint32_t sbase = fm_smem_u32(sB + (ct & 1) * 2 * per);
        auto step = [&](int s, auto first) {
            uint32_t bq[2][2][4];        // [plane][block pair][4]
#pragma unroll
            for (int pl = 0; pl < 2; pl++)
#pragma unroll
                for (int np = 0; np < 2; np++)
                    fm_ldsm_x4(sbase + (pl * per + (wq + s) * 2 * WV_COLS) * 16 + boff[np], bq[pl][np]);
#pragma unroll
            for (int mt = 0; mt < 2; mt++) {
                const uint4 a = tab[(2 * s - mt + 1) * 32 + lane];
#pragma unroll
                for (int pl = 0; pl < 2; pl++)
#pragma unroll
                    for (int nb = 0; nb < 4; nb++) {
                        const uint32_t b0 = bq[pl][nb >> 1][2 * (nb & 1)], b1 = bq[pl][nb >> 1][2 * (nb & 1) + 1];
                        if (decltype(first)::value) fm_imma0(acc[pl][mt][nb], a.x, a.y, a.z, a.w, b0, b1, pl ? 0 : 32768);
                        else fm_imma(acc[pl][mt][nb], a.x, a.y, a.z, a.w, b0, b1);
                    }
            }
        };
        step(0, std::true_type());
#pragma unroll 1
        for (int s = 1; s < Sv; s++) step(s, std::false_type());
        // epilogue: thread (g, t) holds output rows 16 mt + g (+8), columns 8 t + 2 nb + e
        const int yb = Y0 + 32 * wq + g;
        const uint32_t *mp = maskbits + ((size_t)(f / T) * h + yb) * wpr + (X0 >> 5);
        uint8_t *dp0 = blur + ((size_t)f * h + yb) * w + X0 + 8 * t;
        const bool ok0 = X0 + 8 * t < w, ok1 = X0 + 8 * t + 4 < w;
#pragma unroll
        for (int mt = 0; mt < 2; mt++)
#pragma unroll
            for (int hr = 0; hr < 2; hr++) {
                const int dy = 16 * mt + 8 * hr;
                uint32_t wd[2];
#pragma unroll
                for (int wi = 0; wi < 2; wi++) {
                    uint32_t v[4];
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        const int nb = 2 * wi + (q >> 1), d = 2 * hr + (q & 1);
                        v[q] = (uint32_t)(acc[1][mt][nb][d] * 256 + acc[0][mt][nb][d]);      // blur = byte 2
                    }
                    wd[wi] = __byte_perm(__byte_perm(v[0], v[1], 0x0062), __byte_perm(v[2], v[3], 0x0062), 0x5410);
                }
                if (yb + dy < h) {
                    const uint32_t m = __ldg(mp + dy * wpr) >> (8 * t);
                    uint8_t *dst = dp0 + dy * w;
                    // masked pixels -> 0xFF bytes -> cleared
                    const uint32_t o0 = fm_clear_masked4(wd[0], m & 0xFu);
                    const uint32_t o1 = fm_clear_masked4(wd[1], (m >> 4) & 0xFu);
                    if ((w & 3) == 0) {
                        if (ok0) *reinterpret_cast<uint32_t *>(dst) = o0;
                        if (ok1) *reinterpret_cast<uint32_t *>(dst + 4) = o1;
                    } else {                      // rows are not word aligned: guarded byte stores
#pragma unroll
                        for (int b = 0; b < 8; b++)
                            if (X0 + 8 * t + b < w) dst[b] = (uint8_t)((b < 4 ? o0 : o1) >> (8 * (b & 3)));
                    }
                }
            }
        __syncthreads();       // every warp is done with this stage before the loads of tile ct + 2 overwrite it
    }
}

// ---------------------------------------------------------------------------------------------
// Pass 2 fused with the temporal stage (planes with w % 32 == 0, alpha in [0, 1]): the blur never goes to memory.
// CTA = 128 output rows x 16 columns of ONE stream, walking the T frames of the call in order; the byte planes of
// frame t+1 stream in through cp.async while frame t is multiplied; a thread ends up with 4 rows x 4 consecutive
// pixels whose float64 background stays in registers for all T frames (find_motion.py:246-257, 651-659).
// Background layout: [S][tilesY][tilesX][warp 4][8][lane 32] double2 (thread-private, coalesced).
// ---------------------------------------------------------------------------------------------
// shared slot of column c of a 16-column tile: the 8 columns {4t' + 2nb + e} of a block land in 8 different 16-byte lanes
__device__ __forceinline__ int wt_slot(int c) { return c ^ ((c >> 3) << 1); }

struct WideVtParams {
    const uint4 *plo, *phi;
    const uint4 *tabg;
    double *bg;
    uint32_t *tbits;            // [S][T][flatwords] raw threshold bits (flat order == row-padded order since w % 32 == 0)
    const uint32_t *maskbits;   // [S][h][wpr]
    const StreamState *state;
    const int *nvalid;          // [S] real frames of each stream in this call
    int *rawrange;              // [S][T][2]
    uint8_t *blur_out;          // [S][T][h][w] parity tap (KEEP) or null
    int w, h, Sv, NGa, wpr, T, threshold, tilesX, tilesY;
    size_t flatwords;           // words per frame of tbits
    double alpha, beta;
};

// 16 consecutive pixels of one row (blur bytes q, unmasked): polygon mask, threshold bits (bit j = pixel j), background update.
// MASKED: the warp has masked pixels (M bit j = pixel j) or the parity tap is on; INIT: first frame of the stream.
template <bool INIT, bool MASKED>
__device__ __forceinline__ uint32_t wt_temporal16(uint4 q, uint32_t M, double (&bg)[16], int threshold, int qoff, uint32_t nthr2,
                                                  double alpha, double beta, double nC, uint8_t *blur_px) {
    uint32_t w4[4] = {q.x, q.y, q.z, q.w};
    if (MASKED) {
#pragma unroll
        for (int k = 0; k < 4; k++) w4[k] = fm_clear_masked4(w4[k], (M >> (4 * k)) & 0xFu);
        if (blur_px) *reinterpret_cast<uint4 *>(blur_px) = make_uint4(w4[0], w4[1], w4[2], w4[3]);
    }
    uint32_t bits = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) {
        const uint32_t sv = __byte_perm(w4[i >> 2], 0, 0x4440 + (i & 3));
        fm_temporal_px<true, INIT>(sv, bg[i], bits, threshold, qoff, nthr2, alpha, beta, nC);
    }
    return __brev(bits) >> 16;       // bit j = pixel j
}

// grid: (w / 16, ceil(h / 128), S), 128 threads.
// dynamic smem: 2 stages * 2 planes * (4 + Sv - 1) groups * 2 halves * 16 columns * 16 B  +  2 Sv * 512  +  128 rows * 16 B
// The accumulators leave the tensor cores as 4 rows x 4 pixels per thread; the blur bytes go through a 2 KB shared tile so that
// the temporal stage sees ONE row x 16 pixels per thread (the mapping of K1): no lane shuffles, one 16-bit store of the
// threshold bits and a quarter of the per-row overhead.
__global__ void __launch_bounds__(128, 5) k_wide_vt(WideVtParams p) {
    extern __shared__ __align__(16) unsigned char wsm[];
    const int Sv = p.Sv, w = p.w, h = p.h, NGa = p.NGa, T = p.T;
    const int Ts = min(T, __ldg(p.nvalid + blockIdx.z));                      // real frames of this stream (ragged batches)
    if (Ts <= 0) return;
    const int NGt = 4 + Sv - 1;
    const int per = NGt * 2 * WT_COLS;                                        // 16-byte chunks per plane and stage
    uint4 *sB = reinterpret_cast<uint4 *>(wsm);                               // [stage][plane][NGt][half][16 slots]
    uint4 *tab = sB + 4 * per;                                                // [2 Sv][32]
    uint4 *sT = tab + 2 * Sv * 32;                                            // [128 rows] 16 blur bytes
    const int tid = threadIdx.x, lane = tid & 31, wq = tid >> 5;
    const int s = blockIdx.z, Y0 = blockIdx.y * WV_ROWS, X0 = blockIdx.x * WT_COLS, G0 = Y0 >> 5;
    const int g = lane >> 2, t4 = lane & 3;
    for (int i = tid; i < 2 * Sv * 32; i += 128) tab[i] = __ldg(p.tabg + i);
    // staging: 16 lanes = the columns of the tile, 8 chunk rows gh (2 * group + half) per pass of the CTA, both planes
    const int scol = tid & 15, sgh = tid >> 4;
    const size_t fstride = (size_t)NGa * 2 * w;                               // uint4 per frame and plane
    const uint4 *gsrc = p.plo + ((size_t)s * T * NGa + G0) * 2 * w + (size_t)sgh * w + X0 + scol;
    const size_t pdiff = p.phi - p.plo;
    const uint32_t sdst = fm_smem_u32(sB) + (sgh * WT_COLS + wt_slot(scol)) * 16;
    const int ghmax = min(2 * NGt, 2 * (NGa - G0));
    auto issue = [&](int t) {
        const uint4 *sp = gsrc + (size_t)t * fstride;
        uint32_t dp = sdst + (t & 1) * 2 * per * 16;
#pragma unroll 1
        for (int gh = sgh; gh < 2 * NGt; gh += 8) {
            const bool ok = gh < ghmax;
            wcp_async16(dp, ok ? sp : p.plo, ok);
            wcp_async16(dp + per * 16, ok ? sp + pdiff : p.plo, ok);
            sp += 8 * (size_t)w;
            dp += 8 * WT_COLS * 16;
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    issue(0);
    // ldmatrix rows of the two column blocks: matrices (nb0, half 0), (nb0, half 1), (nb1, half 0), (nb1, half 1)
    uint32_t boff;
    {
        const int mi = lane >> 3, n = lane & 7;
        const int col = 4 * (n >> 1) + 2 * (mi >> 1) + (n & 1);
        boff = ((mi & 1) * WT_COLS + wt_slot(col)) * 16;
    }
    // accumulator fragment of this thread: rows 32 wq + 16 mt + 8 hr + g of the tile, columns 4 t4 .. + 3 (pixel j: block j >> 1,
    // e = j & 1); temporal stage of this thread: row Y0 + 32 wq + lane, columns X0 .. X0 + 15
    uint32_t *sTw = reinterpret_cast<uint32_t *>(sT) + (32 * wq + g) * 4 + t4;
    const uint4 *sTr = sT + 32 * wq + lane;
    const int y = Y0 + 32 * wq + lane;
    uint32_t M = 0;                                                           // polygon mask bits of the 16 pixels
    if (y < h) M = (__ldg(p.maskbits + ((size_t)s * h + y) * p.wpr + (X0 >> 5)) >> (X0 & 31)) & 0xFFFFu;
    const bool masked = __any_sync(0xffffffffu, M != 0) || p.blur_out != nullptr;
    const bool has_bg = p.state[s].has_bg != 0;
    double2 *bgt = reinterpret_cast<double2 *>(p.bg) +
                   ((((size_t)s * p.tilesY + blockIdx.y) * p.tilesX + blockIdx.x) * 4 + wq) * 8 * 32 + lane;
    double bg[16];
    if (has_bg) {
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const double2 v = bgt[i * 32];
            bg[2 * i] = v.x;
            bg[2 * i + 1] = v.y;
        }
    }
    const int qoff = 0x4B400000 - p.threshold;
    const uint32_t nthr2 = ~(2u * (uint32_t)p.threshold);
    const double nC = -(4503599627370496.0 * p.alpha);
    uint16_t *tw = reinterpret_cast<uint16_t *>(p.tbits + (size_t)s * T * p.flatwords) + (size_t)y * p.wpr * 2 + (size_t)2 * (X0 >> 5) + ((X0 >> 4) & 1);
    for (int t = 0; t < Ts; t++) {
        if (t + 1 < Ts) {
            issue(t + 1);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
        int acc[2][2][2][4];       // [plane][row tile][column block][4]; the low plane starts at the rounding constant
        const uint32_t sbase = fm_smem_u32(sB + (t & 1) * 2 * per);
        auto step = [&](int sg, auto first) {
            uint32_t bq[2][4];
#pragma unroll
            for (int pl = 0; pl < 2; pl++) fm_ldsm_x4(sbase + (pl * per + (wq + sg) * 2 * WT_COLS) * 16 + boff, bq[pl]);
#pragma unroll
            for (int mt = 0; mt < 2; mt++) {
                const uint4 a = tab[(2 * sg - mt + 1) * 32 + lane];
#pragma unroll
                for (int pl = 0; pl < 2; pl++)
#pragma unroll
                    for (int nb = 0; nb < 2; nb++) {
                        if (decltype(first)::value) fm_imma0(acc[pl][mt][nb], a.x, a.y, a.z, a.w, bq[pl][2 * nb], bq[pl][2 * nb + 1], pl ? 0 : 32768);
                        else fm_imma(acc[pl][mt][nb], a.x, a.y, a.z, a.w, bq[pl][2 * nb], bq[pl][2 * nb + 1]);
                    }
            }
        };
        step(0, std::true_type());
#pragma unroll 1
        for (int sg = 1; sg < Sv; sg++) step(sg, std::false_type());
        // ---- blur bytes of the fragment -> shared tile (blur = byte 2 of 256 hi + lo, rounding constant already in lo) ----
#pragma unroll
        for (int r = 0; r < 4; r++) {
            const int mt = r >> 1, hr = r & 1;
            uint32_t v[4];
#pragma unroll
            for (int j = 0; j < 4; j++) v[j] = (uint32_t)(acc[1][mt][j >> 1][2 * hr + (j & 1)] * 256 + acc[0][mt][j >> 1][2 * hr + (j & 1)]);
            sTw[(16 * mt + 8 * hr) * 4] = __byte_perm(__byte_perm(v[0], v[1], 0x0062), __byte_perm(v[2], v[3], 0x0062), 0x5410);
        }
        __syncwarp();              // the 32 rows of a warp are produced and consumed by the same warp
        const uint4 q = *sTr;
        // ---- temporal stage: one row x 16 pixels per thread ----
        uint8_t *bo = (p.blur_out && y < h) ? p.blur_out + (((size_t)s * T + t) * h + y) * w + X0 : nullptr;
        asm volatile("" : "+r"(M));        // opaque per frame: keeps the single-bit tests of M from being hoisted
        uint32_t bits;
        if (t == 0 && !has_bg) bits = wt_temporal16<true, true>(q, M, bg, p.threshold, qoff, nthr2, p.alpha, p.beta, nC, bo);
        else if (masked) bits = wt_temporal16<false, true>(q, M, bg, p.threshold, qoff, nthr2, p.alpha, p.beta, nC, bo);
        else bits = wt_temporal16<false, false>(q, M, bg, p.threshold, qoff, nthr2, p.alpha, p.beta, nC, nullptr);
        if (y >= h) bits = 0;
        if (y < h) *tw = (uint16_t)bits;
        if (__any_sync(0xffffffffu, bits != 0) && lane == 0) {       // this warp's 32 rows hold something
            int *rr = p.rawrange + 2 * ((size_t)s * T + t);
            atomicMax(rr, min(Y0 + 32 * wq + 31, h - 1));
            atomicMax(rr + 1, h - 1 - (Y0 + 32 * wq));
        }
        tw += p.flatwords * 2;
        __syncthreads();       // every warp is done with this stage before the loads of frame t + 2 overwrite it
    }
#pragma unroll
    for (int i = 0; i < 8; i++) bgt[i * 32] = make_double2(bg[2 * i], bg[2 * i + 1]);
}

// tiled background of k_wide_vt -> row-major float64 plane
__global__ void k_bg_export_wide(const double *__restrict__ bg, double *__restrict__ dst, int w, int h, int tilesX, int tilesY,
                                 int s) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= w) return;
    const int tx = x / WT_COLS, ty = y / WV_ROWS, lx = x % WT_COLS, ly = y % WV_ROWS;
    const int wq = ly >> 5, lane = ly & 31;                        // thread = row, 16 consecutive columns
    const int i = lx >> 1, j = lx & 1;                             // double2 index of the thread, component
    const size_t base = ((((size_t)s * tilesY + ty) * tilesX + tx) * 4 + wq) * 8 * 32;
    dst[(size_t)y * w + x] = bg[(base + (size_t)i * 32 + lane) * 2 + j];
}

bool fm_wide_fused_supported(const fm_ctx *c) {
    const double a = c->cfg.avg;
    return c->k >= 3 && (c->w % 32) == 0 && a >= 0.0 && a <= 1.0 && c->cfg.threshold >= 0;
}

size_t fm_wide_bg_doubles(const fm_ctx *c) {
    return (size_t)c->S * ((c->w + WT_COLS - 1) / WT_COLS) * ((c->h + WV_ROWS - 1) / WV_ROWS) * WT_COLS * WV_ROWS;
}

int fm_launch_bg_export_wide(fm_ctx *c, int stream, double *dst_dev, cudaStream_t st) {
    dim3 grid((c->w + 127) / 128, c->h);
    k_bg_export_wide<<<grid, 128, 0, st>>>(c->bg, dst_dev, c->w, c->h, (c->w + WT_COLS - 1) / WT_COLS,
                                           (c->h + WV_ROWS - 1) / WV_ROWS, stream);
    FM_LAUNCH_CHECK();
    return FM_OK;
}

// k = 1: GaussianBlur is the identity, only the polygon masks are painted (find_motion.py:494, 619-635).  The gray plane
// of frame (s, t) starts at gray + s * sstride + t * fstride, its rows rpitch bytes apart
__global__ void __launch_bounds__(256) k_blur_identity(const uint8_t *__restrict__ gray, size_t sstride, size_t fstride,
                                                       size_t rpitch, uint8_t *__restrict__ blur,
                                                       const uint32_t *__restrict__ maskbits, int w, int h, int wpr, int T,
                                                       const int *__restrict__ nvalid) {
    const int f = blockIdx.z, y = blockIdx.y, x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= w || f % T >= __ldg(nvalid + f / T)) return;
    const uint32_t m = __ldg(maskbits + ((size_t)(f / T) * h + y) * wpr + (x >> 5));
    const uint8_t v = gray[(size_t)(f / T) * sstride + (size_t)(f % T) * fstride + (size_t)y * rpitch + x];
    blur[((size_t)f * h + y) * w + x] = ((m >> (x & 31)) & 1u) ? (uint8_t)0 : v;
}

// frames != nullptr: full-resolution mode, convert BGR -> gray while staging (no gray plane); else read c->gray.  Gray
// frames (FM_FLAG_GRAY) are the gray plane: read in place, copied to c->gray only as the FM_FLAG_KEEP_PLANES tap
int fm_launch_wide_blur(fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, size_t pitch, int T, cudaStream_t st) {
    const uint8_t *gsrc = c->gray;                                   // the gray plane the passes read, and its layout
    size_t gsstride = (size_t)T * c->N, gfstride = c->N, gpitch = c->w;
    if (frames && c->px_bytes == 1) {
        if (c->cfg.flags & FM_FLAG_KEEP_PLANES) {
            int rc = fm_launch_gray_plane(c, frames, sstride, fstride, pitch, T, st);
            if (rc) return rc;
        }
        gsrc = frames; gsstride = sstride; gfstride = fstride; gpitch = pitch;
        frames = nullptr;
    }
    if (c->k == 1) {
        if (frames) {
            int rc = fm_launch_gray_plane(c, frames, sstride, fstride, pitch, T, st);
            if (rc) return rc;
        }
        dim3 grid((c->w + 255) / 256, c->h, c->S * T);
        k_blur_identity<<<grid, 256, 0, st>>>(gsrc, gsstride, gfstride, gpitch, c->blur, c->maskbits, c->w, c->h, c->wpr, T,
                                              c->nvalid);
        FM_LAUNCH_CHECK();
        return FM_OK;
    }
    const WideGeom g = wide_geom(c);
    const int F = c->S * T;
    uint32_t *plo = reinterpret_cast<uint32_t *>(c->hor);
    uint32_t *phi = plo + fm_wide_plane_bytes(c) / 4;
    const uint2 *tabh = reinterpret_cast<const uint2 *>(c->wtab);
    const uint4 *tabv = reinterpret_cast<const uint4 *>(c->wtab + (size_t)(4 * g.Sh + 3) * 32 * 2);
    const size_t smh = (size_t)32 * g.pitch + (size_t)(4 * g.Sh + 3) * 256;
    const size_t smv = (size_t)4 * (4 + g.Sv - 1) * 2 * WV_COLS * 16 + (size_t)2 * g.Sv * 512;
    int rc;
    if ((rc = fm_ensure_smem((const void *)k_wide_h<false>, smh, c->cfg.device))) return rc;
    if ((rc = fm_ensure_smem((const void *)k_wide_v, smv, c->cfg.device))) return rc;
    dim3 hgrid((c->w + WH_COLS - 1) / WH_COLS, g.NGa, F);
    const bool aligned16 = frames && ((((uintptr_t)frames) | sstride | fstride | pitch | ((size_t)c->W * c->px_bytes)) & 15) == 0;
    if (aligned16) {
        if (c->cfg.flags & FM_FLAG_KEEP_PLANES) {
            int rc = fm_launch_gray_plane(c, frames, sstride, fstride, pitch, T, st);
            if (rc) return rc;
        }
        // TMA-staged pass 1 when the window of a CTA is one or two boxes and the CTA needs <= 100 KB (k <= ~200 at 1080p / 4K: k = 97 runs four CTAs
        // per SM, k = 193 three; measured against the register-staged path in profiles/r2_wide_ab.txt).  A box row is at
        // most 256 words: 21 units of 16 three-byte pixels, 16 of four-byte ones
        const int PX = c->px_bytes, umax = PX == 4 ? 16 : 21;
        const bool mirror = g.R16 < c->w && g.R16 + g.r < WH_COLS;
        const int nunits = (g.R16 + WH_COLS + g.r + 15) / 16;
        const int nbox = nunits > umax ? 2 : 1, ubox = (nunits + nbox - 1) / nbox;
        const size_t smt = (size_t)nbox * 32 * ubox * 16 * PX + smh + 16;
        static const long tma_kb = getenv("FM_WIDE_TMA_KB") ? atol(getenv("FM_WIDE_TMA_KB")) : 100;
        const bool tma = mirror && ubox <= umax && smt <= (size_t)tma_kb * 1024;
        CUtensorMap tmap;
        if (tma && (rc = fm_frames_tmap(c, frames, sstride, fstride, pitch, T, ubox * 4 * PX, 32, &tmap))) return rc;
        static const int gp = getenv("FM_WIDE_GP") ? std::max(1, atoi(getenv("FM_WIDE_GP"))) : 4;     // row groups per CTA (A/B: profiles/r2_wide_ab.txt)
        fm_px_dispatch(c->px_bytes, c->rgb, [&](auto Cx, auto RGB) {
            constexpr int P = Cx.value == 4 ? 4 : 3;
            if (tma) {
                if ((rc = fm_ensure_smem((const void *)k_wide_h_tma<RGB.value, P>, smt, c->cfg.device))) return;
                dim3 tgrid(hgrid.x, (g.NGa + gp - 1) / gp, F);
                k_wide_h_tma<RGB.value, P><<<tgrid, WH_THREADS, smt, st>>>(tmap, frames, sstride, fstride, pitch, T, plo, phi, tabh,
                                                                           c->w, c->h, g.r, g.R16, g.Sh, g.pitch, g.NGa, c->nvalid,
                                                                           nunits, ubox, nbox, gp);
            } else {
                if ((rc = fm_ensure_smem((const void *)k_wide_h<true, RGB.value, P>, smh, c->cfg.device))) return;
                k_wide_h<true, RGB.value, P><<<hgrid, WH_THREADS, smh, st>>>(frames, sstride, fstride, pitch, T, plo, phi, tabh, c->w,
                                                                             c->h, g.r, g.R16, g.Sh, g.pitch, g.NGa, c->nvalid);
            }
        });
        if (rc) return rc;
    } else {
        if (frames) {
            int rc = fm_launch_gray_plane(c, frames, sstride, fstride, pitch, T, st);
            if (rc) return rc;
        }
        k_wide_h<false><<<hgrid, WH_THREADS, smh, st>>>(gsrc, gsstride, gfstride, gpitch, T, plo, phi, tabh, c->w, c->h, g.r,
                                                        g.R16, g.Sh, g.pitch, g.NGa, c->nvalid);
    }
    FM_LAUNCH_CHECK();
    if (c->wide_fused) {
        const size_t smt = (size_t)4 * (4 + g.Sv - 1) * 2 * WT_COLS * 16 + (size_t)2 * g.Sv * 512 + WV_ROWS * 16;
        if ((rc = fm_ensure_smem((const void *)k_wide_vt, smt, c->cfg.device))) return rc;
        WideVtParams p;
        p.plo = reinterpret_cast<const uint4 *>(plo); p.phi = reinterpret_cast<const uint4 *>(phi); p.tabg = tabv;
        p.bg = c->bg; p.tbits = c->tflat; p.maskbits = c->maskbits; p.state = c->state; p.rawrange = c->rawrange;
        p.nvalid = c->nvalid;
        p.blur_out = (c->cfg.flags & FM_FLAG_KEEP_PLANES) ? c->blur : nullptr;
        p.w = c->w; p.h = c->h; p.Sv = g.Sv; p.NGa = g.NGa; p.wpr = c->wpr; p.T = T; p.threshold = c->cfg.threshold;
        p.tilesX = (c->w + WT_COLS - 1) / WT_COLS; p.tilesY = (c->h + WV_ROWS - 1) / WV_ROWS;
        p.flatwords = (size_t)c->ntiles * FM_TILE_WORDS;
        p.alpha = c->cfg.avg; p.beta = 1.0 - p.alpha;
        dim3 tgrid(p.tilesX, p.tilesY, c->S);
        k_wide_vt<<<tgrid, 128, smt, st>>>(p);
        FM_LAUNCH_CHECK();
        return FM_OK;
    }
    dim3 vgrid((c->w + WV_COLS * WV_NT - 1) / (WV_COLS * WV_NT), (c->h + WV_ROWS - 1) / WV_ROWS, F);
    k_wide_v<<<vgrid, 128, smv, st>>>(reinterpret_cast<const uint4 *>(plo), reinterpret_cast<const uint4 *>(phi), c->blur,
                                      tabv, c->w, c->h, g.Sv, g.NGa, c->wpr, T, c->maskbits, c->nvalid);
    FM_LAUNCH_CHECK();
    return FM_OK;
}
