// Generic front end: INTER_AREA resize + gray (K0), gray, separable 8.8 fixed-point Gaussian,
// mask application.  Produces the masked blur plane the temporal kernel consumes.
// Replaces VideoMotion.blur_frame + mask_off_areas (find_motion/find_motion.py:487-494, 619-635).
#include "fm_common.cuh"

// identity-resize mode: one thread per 4 pixels of a frame (12 bytes in, 4 bytes out; C = 1, gray frames: a copy).  Pixel
// i = y * w + x of a frame is at y * pitch + C x; packed rows (pitch == C w) are one flat run, so 4 pixels may then straddle
// a row end.  RGB: R-first pixels (FM_FLAG_RGB)
template <int C, bool RGB = false>
__global__ void __launch_bounds__(256) k_gray(const uint8_t *__restrict__ frames, size_t sstride,
                                              size_t fstride, size_t pitch, int T, int w, int N, uint8_t *__restrict__ gray,
                                              const int *__restrict__ nvalid) {
    int f = blockIdx.y;   // s*T + t
    int s = f / T, t = f - s * T;
    if (t >= __ldg(nvalid + s)) return;       // not a real frame of this (ragged) call
    const uint8_t *src = frames + (size_t)s * sstride + (size_t)t * fstride;
    uint8_t *dst = gray + (size_t)f * N;
    int i4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i4 >= N) return;
    const bool flat = pitch == (size_t)w * C;
    const int y4 = flat ? 0 : i4 / w, x4 = i4 - y4 * w;
    const uint8_t *q4 = flat ? src + (size_t)i4 * C : src + (size_t)y4 * pitch + (size_t)x4 * C;
    if (i4 + 4 <= N && (flat || x4 + 4 <= w) && ((((uintptr_t)q4) & 3) == 0) && ((((uintptr_t)dst) & 3) == 0)) {
        const uint32_t *p = reinterpret_cast<const uint32_t *>(q4);
        *reinterpret_cast<uint32_t *>(dst + i4) = C == 1   ? __ldg(p)
            : C == 4 ? fm_gray4a<RGB>(make_uint4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3)))
                     : fm_gray4<RGB>(__ldg(p), __ldg(p + 1), __ldg(p + 2));
    } else {
        for (int i = i4; i < min(i4 + 4, N); i++) {
            const int y = i / w;
            const uint8_t *p = src + (size_t)y * pitch + (size_t)(i - y * w) * C;
            dst[i] = C == 1 ? p[0] : (uint8_t)fm_gray<RGB>(p[0], p[1], p[2]);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// K0: INTER_AREA resize (float32, unfused, strictly ordered) + gray.  SURVEY.md A.1.
// One CTA per (frame, destination row).  Source rows are staged through shared memory with
// coalesced loads; horizontal chains run per (source row, dx) and the vertical chain per (dx, c).
// ---------------------------------------------------------------------------------------------
struct K0Params {
    const uint8_t *frames;
    size_t sstride, fstride;
    size_t pitch;                // bytes from one source row to the next (>= W * 3)
    int T, W, H, w, h;
    int mode, fx, fy;            // 1 = tables, 2 = integer ratio
    const int *xstart, *xidx;
    const float *xwt;
    const int *ystart, *yidx;
    const float *ywt;
    int max_ytaps;
    uint8_t *gray;
    const int *nvalid;           // [S] real frames of each stream in this call (null: every frame)
    uint8_t *bgr_out;            // [F][h][w][3] resized BGR instead of gray (fm_resize_area: the detector input plane)
};

#define K0_THREADS 512
#define K0_GROUPS 4       // source rows in flight (K0_THREADS/K0_GROUPS threads each)

// oidx (with bgr_out): null, or [F] plane index (-1: skip the frame); frame f's plane then goes to
// bgr_out + s * ostride + oidx[f] * h*w*3 (fm_object_planes).  C: channels of the source (3 BGR, 1 gray); per channel the
// chains are the same, and a gray source's resized byte is stored in all three channels of bgr_out.  RGB: R-first source
// pixels, whose resized bytes go to bgr_out in BGR order
template <int C, bool RGB = false>
__global__ void __launch_bounds__(K0_THREADS) k_resize_gray(K0Params p, const int *__restrict__ oidx, size_t ostride) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int f = blockIdx.y;
    const int s = f / p.T, t = f - s * p.T;
    if (p.nvalid && t >= __ldg(p.nvalid + s)) return;
    const int o = oidx ? __ldg(oidx + f) : 0;
    if (o < 0) return;
    const int dy = blockIdx.x;
    const uint8_t *src = p.frames + (size_t)s * p.sstride + (size_t)t * p.fstride;
    const int rowbytes = p.W * C;
    const int rowpitch = (rowbytes + 16 + 15) & ~15;          // room for a misaligned start
    unsigned char *rowbuf = smem;                               // [K0_GROUPS][rowpitch]
    float *bufs = reinterpret_cast<float *>(smem + (size_t)K0_GROUPS * rowpitch);   // [ny][C w]
    constexpr int NC = C == 4 ? 3 : C;          // chains per column: the fourth byte of BGRA / RGBA is not resized
    const int w3 = p.w * NC;
    const int tid = threadIdx.x;
    const int gsz = K0_THREADS / K0_GROUPS;
    const int grp = tid / gsz, gt = tid - grp * gsz;

    int y0, ny;
    if (p.mode == 1) {
        y0 = p.ystart[dy];
        ny = p.ystart[dy + 1] - y0;
    } else {
        y0 = 0;
        ny = p.fy;
    }

    for (int jb = 0; jb < ny; jb += K0_GROUPS) {
        int j = jb + grp;
        int mis = 0;
        if (j < ny) {
            int sy = (p.mode == 1) ? p.yidx[y0 + j] : dy * p.fy + j;
            const uint8_t *row = src + (size_t)sy * p.pitch;
            mis = (int)((uintptr_t)row & 15);
            const uint4 *row16 = reinterpret_cast<const uint4 *>(row - mis);
            int n16 = (mis + rowbytes + 15) >> 4;
            uint4 *dst16 = reinterpret_cast<uint4 *>(rowbuf + (size_t)grp * rowpitch);
            // partial first/last 16-byte blocks are loaded bytewise so that nothing outside the
            // row (possibly outside the caller's buffer) is touched
            for (int i = gt; i < n16; i += gsz) {
                if ((i == 0 && mis) || (i == n16 - 1 && ((mis + rowbytes) & 15))) {
                    unsigned char *d = reinterpret_cast<unsigned char *>(dst16 + i);
                    for (int b = 0; b < 16; b++) {
                        int o = i * 16 + b - mis;
                        d[b] = (o >= 0 && o < rowbytes) ? row[o] : 0;
                    }
                } else {
                    dst16[i] = __ldg(row16 + i);
                }
            }
        }
        __syncthreads();
        if (j < ny) {
            const unsigned char *rb = rowbuf + (size_t)grp * rowpitch + mis;
            float *out = bufs + (size_t)j * w3;
            if (p.mode == 1) {
                for (int dx = gt; dx < p.w; dx += gsz) {
                    int a = p.xstart[dx], b = p.xstart[dx + 1];
                    float bc[NC];
#pragma unroll
                    for (int ch = 0; ch < NC; ch++) bc[ch] = 0.f;
                    for (int q = a; q < b; q++) {
                        const unsigned char *px = rb + p.xidx[q] * C;
                        float al = p.xwt[q];
#pragma unroll
                        for (int ch = 0; ch < NC; ch++) bc[ch] = __fadd_rn(bc[ch], __fmul_rn((float)px[ch], al));
                    }
#pragma unroll
                    for (int ch = 0; ch < NC; ch++) out[dx * NC + ch] = bc[ch];
                }
            } else {   // integer ratio: exact integer row sums, kept as int bit patterns
                int *outi = reinterpret_cast<int *>(out);
                for (int dx = gt; dx < p.w; dx += gsz) {
                    int sc[NC];
#pragma unroll
                    for (int ch = 0; ch < NC; ch++) sc[ch] = 0;
                    const unsigned char *px = rb + dx * p.fx * C;
                    for (int q = 0; q < p.fx; q++, px += C) {
#pragma unroll
                        for (int ch = 0; ch < NC; ch++) sc[ch] += px[ch];
                    }
#pragma unroll
                    for (int ch = 0; ch < NC; ch++) outi[dx * NC + ch] = sc[ch];
                }
            }
        }
        __syncthreads();
    }
    // vertical chains + rounding + gray
    unsigned char *small = rowbuf;        // reuse: [C w] resized bytes of this row
    for (int i = tid; i < w3; i += K0_THREADS) {
        int v;
        if (p.mode == 1) {
            float sum = __fmul_rn(p.ywt[y0], bufs[i]);
            for (int j = 1; j < ny; j++) sum = __fadd_rn(sum, __fmul_rn(p.ywt[y0 + j], bufs[(size_t)j * w3 + i]));
            v = __float2int_rn(sum);
        } else {
            const int *bi = reinterpret_cast<const int *>(bufs);
            int sum = 0;
            for (int j = 0; j < ny; j++) sum += bi[(size_t)j * w3 + i];
            if (p.fx == 2 && p.fy == 2) {
                v = (sum + 2) >> 2;
            } else {
                float sc = __fdiv_rn(1.f, (float)(p.fx * p.fy));
                v = __float2int_rn(__fmul_rn((float)sum, sc));
            }
        }
        small[i] = (unsigned char)min(max(v, 0), 255);
    }
    __syncthreads();
    if (p.bgr_out) {
        const int wb = p.w * 3;
        uint8_t *out = p.bgr_out + (oidx ? (size_t)s * ostride + ((size_t)o * p.h + dy) * wb : ((size_t)f * p.h + dy) * wb);
        for (int i = tid; i < wb; i += K0_THREADS) out[i] = C == 1 ? small[i / 3] : RGB ? small[i + 2 - 2 * (i % 3)] : small[i];
        return;
    }
    uint8_t *g = p.gray + ((size_t)f * p.h + dy) * p.w;
    for (int dx = tid; dx < p.w; dx += K0_THREADS)
        g[dx] = C == 1 ? small[dx] : (uint8_t)fm_gray<RGB>(small[dx * 3], small[dx * 3 + 1], small[dx * 3 + 2]);
}

// INTER_AREA resize to BGR (device buffers); mode / tables as fm_ctx_create derives them.  One frame (fm_resize_area:
// S = T = 1, oidx null) or the frames of a call with an oidx table (fm_object_planes).  channels: 3 (BGR source) or 1 (gray
// source, its resize stored in B, G and R); rgb: R-first three-byte source
int fm_launch_resize_bgr(int device, const uint8_t *src_dev, size_t sstride, size_t fstride, size_t pitch, int S, int T, int W,
                         int H, int w, int h, int mode, int fx, int fy, const ResizeTab &xt, const ResizeTab &yt, const int *oidx,
                         uint8_t *dst_dev, size_t ostride, cudaStream_t st, int channels, bool rgb) {
    K0Params p;
    p.frames = src_dev; p.sstride = sstride; p.fstride = fstride; p.pitch = pitch;
    p.T = T; p.W = W; p.H = H; p.w = w; p.h = h;
    p.mode = mode; p.fx = fx; p.fy = fy;
    p.xstart = xt.start; p.xidx = xt.idx; p.xwt = xt.wt;
    p.ystart = yt.start; p.yidx = yt.idx; p.ywt = yt.wt;
    p.max_ytaps = mode == 1 ? yt.max_taps : fy;
    p.gray = nullptr; p.nvalid = nullptr; p.bgr_out = dst_dev;
    const int rowpitch = (W * channels + 16 + 15) & ~15;
    const size_t smem = (size_t)K0_GROUPS * rowpitch + (size_t)p.max_ytaps * w * channels * sizeof(float);
    if (smem > 220 * 1024) {
        fm_set_error("resize needs %zu bytes of shared memory (frame too wide / ratio too large)", smem);
        return FM_ERANGE;
    }
    int rc = FM_OK;
    dim3 grid(h, S * T);
    fm_px_dispatch(channels, rgb, [&](auto C, auto RGB) {
        const void *kern = (const void *)k_resize_gray<C.value, RGB.value>;
        if ((rc = fm_ensure_smem(kern, smem, device))) return;
        k_resize_gray<C.value, RGB.value><<<grid, K0_THREADS, smem, st>>>(p, oidx, ostride);
    });
    if (rc) return rc;
    FM_LAUNCH_CHECK();
    return FM_OK;
}

// ---------------------------------------------------------------------------------------------
// K0w: the same INTER_AREA + gray, one WARP per (frame, destination row), no block barriers.
// The warp streams its source rows through a private shared-memory row buffer with 128-bit loads
// (all loads of a row in flight together), each lane owns destination columns lane, lane+32, ... and
// keeps their horizontal and vertical float32 chains in registers.  Used when w <= 128 (tables mode).
// ---------------------------------------------------------------------------------------------
#define K0W_WARPS 8

// task = ((frame * h + dy) * nq + q): the warp produces destination columns q*dxw .. q*dxw+dxw-1 (one per lane).
// C: channels of the source (3 BGR, 1 gray); RGB: R-first three-byte source
template <int C, bool RGB = false>
__global__ void __launch_bounds__(32 * K0W_WARPS) k_resize_gray_warp(K0Params p, int segpitch, int tasks, int nq,
                                                                     int dxw) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int task = blockIdx.x * K0W_WARPS + warp;
    if (task >= tasks) return;
    const int q = task % nq, fd = task / nq;
    const int f = fd / p.h, dy = fd - f * p.h;
    const int s = f / p.T, t = f - s * p.T;
    if (t >= __ldg(p.nvalid + s)) return;
    const uint8_t *src = p.frames + (size_t)s * p.sstride + (size_t)t * p.fstride;
    unsigned char *rowbuf = smem + (size_t)warp * segpitch;
    const int rowbytes = p.W * C;
    const int y0 = p.ystart[dy], ny = p.ystart[dy + 1] - y0;
    const int dxa = q * dxw, dxb = min(dxa + dxw, p.w);
    const int dx = dxa + lane;
    const bool live = lane < dxw && dx < p.w;
    // source byte range of this warp's columns
    const int b_lo = p.xidx[p.xstart[dxa]] * C, b_hi = (p.xidx[p.xstart[dxb] - 1] + 1) * C;
    int xa = 0, xn = 0;
    int xfirst = 0;
    if (live) { xa = p.xstart[dx]; xn = p.xstart[dx + 1] - xa; xfirst = p.xidx[xa]; }
    constexpr int NC = C == 4 ? 3 : C;          // chains per column: the fourth byte of BGRA / RGBA is not resized
    float sc[NC];
    for (int j = 0; j < ny; j++) {
        const int sy = p.yidx[y0 + j];
        const float beta = p.ywt[y0 + j];
        const uint8_t *seg = src + (size_t)sy * p.pitch + b_lo;           // first needed byte
        const int nbytes = b_hi - b_lo;
        const int mis = (int)((uintptr_t)seg & 15);
        const uint4 *seg16 = reinterpret_cast<const uint4 *>(seg - mis);
        const int n16 = (mis + nbytes + 15) >> 4;
        uint4 *dst16 = reinterpret_cast<uint4 *>(rowbuf);
        // 16-byte blocks that are not fully inside the ROW are fetched bytewise (nothing outside the
        // caller's buffer is touched)
        const long row_lo = -(long)b_lo + mis, row_hi = (long)rowbytes - b_lo + mis;   // row extent in buffer coords
        __syncwarp();
        for (int i = lane; i < n16; i += 32) {
            long o0 = (long)i * 16;
            if (o0 >= row_lo && o0 + 16 <= row_hi) {
                dst16[i] = __ldg(seg16 + i);
            } else {
                unsigned char *d = reinterpret_cast<unsigned char *>(dst16 + i);
                for (int b = 0; b < 16; b++) {
                    long o = o0 + b;
                    d[b] = (o >= row_lo && o < row_hi) ? seg[o - mis] : 0;
                }
            }
        }
        __syncwarp();
        const unsigned char *rb = rowbuf + mis - b_lo;                    // rb[C*x + c] = source pixel x
        float bc[NC];
#pragma unroll
        for (int ch = 0; ch < NC; ch++) bc[ch] = 0.f;
        const unsigned char *px = rb + xfirst * C;      // the taps of a column are consecutive source pixels
        const float *wt = p.xwt + xa;
#pragma unroll 4
        for (int qq = 0; qq < xn; qq++, px += C) {
            const float al = __ldg(wt + qq);
#pragma unroll
            for (int ch = 0; ch < NC; ch++) bc[ch] = __fadd_rn(bc[ch], __fmul_rn((float)px[ch], al));
        }
#pragma unroll
        for (int ch = 0; ch < NC; ch++) sc[ch] = j == 0 ? __fmul_rn(beta, bc[ch]) : __fadd_rn(sc[ch], __fmul_rn(beta, bc[ch]));
    }
    if (live) {
        int v[NC];
#pragma unroll
        for (int ch = 0; ch < NC; ch++) v[ch] = min(max(__float2int_rn(sc[ch]), 0), 255);
        p.gray[((size_t)f * p.h + dy) * p.w + dx] = C == 1 ? (uint8_t)v[0] : (uint8_t)fm_gray<RGB>(v[0], v[NC > 1 ? 1 : 0], v[NC - 1]);
    }
}

// Same decomposition for 4-byte aligned rows: every lane walks its taps in groups of 4 source pixels
// (12 bytes = three aligned 32-bit shared loads), the tap list padded to group boundaries with zero
// weights (x + 0*y == x exactly, so the strictly ordered float32 chains are unchanged).  Bytes become
// floats with PRMT into the mantissa of 2^23 (fm_byte_mul) and the bias leaves inside the tap product.
struct K0GParams {
    const int *g4start;      // [w] first source pixel of the column's first group (multiple of 4)
    const int *g4n;          // [w] groups
    const int *g4off;        // [w] offset (in float4) into g4w
    const float4 *g4w;       // padded weights
};

__device__ __noinline__ void copy_partial_block(unsigned char *d, const uint8_t *origin, long o0, long row_lo,
                                                long row_hi) {
#pragma unroll 1
    for (int b = 0; b < 16; b++) {
        long o = o0 + b;
        d[b] = (o >= row_lo && o < row_hi) ? origin[o] : 0;
    }
}

#define K0_RG 7         // tap groups per destination column held in registers
// PF = 16-byte blocks per lane of one source segment (registers used to prefetch the next row).  C: channels of the source
// (3 BGR: a group is 12 bytes; 1 gray: a group is one word); RGB: R-first three-byte source
template <int PF, bool INREG, int C, bool RGB = false>
__global__ void __launch_bounds__(32 * K0W_WARPS) k_resize_gray_g4(K0Params p, K0GParams gp, int segpitch, int tasks,
                                                                   int nq, int dxw) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int task = blockIdx.x * K0W_WARPS + warp;
    if (task >= tasks) return;
    const int q = task % nq, fd = task / nq;
    const int f = fd / p.h, dy = fd - f * p.h;
    const int s = f / p.T, t = f - s * p.T;
    if (t >= __ldg(p.nvalid + s)) return;
    const uint8_t *src = p.frames + (size_t)s * p.sstride + (size_t)t * p.fstride;
    unsigned char *rowbuf = smem + (size_t)warp * segpitch;
    const int rowbytes = p.W * C;
    const int y0 = p.ystart[dy], ny = p.ystart[dy + 1] - y0;
    const int dxa = q * dxw, dxb = min(dxa + dxw, p.w);
    const int dx = dxa + lane;
    const bool live = lane < dxw && dx < p.w;
    const int b_lo = gp.g4start[dxa] * C;
    const int b_hi = min((gp.g4start[dxb - 1] + 4 * gp.g4n[dxb - 1]) * C, rowbytes);
    const int nbytes = b_hi - b_lo;
    int gs = b_lo / C, gn = 0;          // idle lanes walk the start of the segment with zero weights
    const float4 *gw = gp.g4w;
    if (live) { gs = gp.g4start[dx]; gn = gp.g4n[dx]; gw += gp.g4off[dx]; }
    float s0 = 0.f, s1 = 0.f, s2 = 0.f;
    uint4 *dst16 = reinterpret_cast<uint4 *>(rowbuf);
    // software pipeline: the 16-byte blocks of row j+1 are loaded into registers while row j is reduced
    uint4 pre[PF];
    auto seg_of = [&](int j) { return src + (size_t)p.yidx[y0 + j] * p.pitch + b_lo; };
    auto issue = [&](int j) {
        const uint8_t *seg = seg_of(j);
        const int mis = (int)((uintptr_t)seg & 15);
        const uint4 *seg16 = reinterpret_cast<const uint4 *>(seg - mis);
        const int n16 = (mis + nbytes + 15) >> 4;
        const long row_lo = -(long)b_lo + mis, row_hi = (long)rowbytes - b_lo + mis;
#pragma unroll
        for (int k = 0; k < PF; k++) {
            const int i = lane + 32 * k;
            const long o0 = (long)i * 16;
            if (i < n16 && o0 >= row_lo && o0 + 16 <= row_hi) pre[k] = __ldg(seg16 + i);
        }
    };
    auto commit = [&](int j) {           // registers (or, for partial blocks at the row ends, bytes) -> shared
        const uint8_t *seg = seg_of(j);
        const int mis = (int)((uintptr_t)seg & 15);
        const int n16 = (mis + nbytes + 15) >> 4;
        const long row_lo = -(long)b_lo + mis, row_hi = (long)rowbytes - b_lo + mis;
#pragma unroll
        for (int k = 0; k < PF; k++) {
            const int i = lane + 32 * k;
            const long o0 = (long)i * 16;
            if (i < n16) {
                if (o0 >= row_lo && o0 + 16 <= row_hi) {
                    dst16[i] = pre[k];
                } else {
                    copy_partial_block(reinterpret_cast<unsigned char *>(dst16 + i), seg - mis, o0, row_lo, row_hi);
                }
            }
        }
        return mis;
    };
    // columns with at most K0_RG tap groups (1080p -> 100: 6) keep weights and bias terms in registers
    // (INREG: chosen by the host when every column has at most K0_RG groups)
    const int gmax = __reduce_max_sync(0xffffffffu, gn);
    constexpr bool inreg = INREG;
    float4 wr[INREG ? K0_RG : 1], wn[INREG ? K0_RG : 1];
    if (inreg) {
#pragma unroll
        for (int g = 0; g < K0_RG; g++) {
            const float4 a = g < gn ? __ldg(gw + g) : make_float4(0.f, 0.f, 0.f, 0.f);
            wr[g] = a;
            wn[g] = make_float4(__fmul_rn(a.x, -8388608.0f), __fmul_rn(a.y, -8388608.0f), __fmul_rn(a.z, -8388608.0f),
                                __fmul_rn(a.w, -8388608.0f));
        }
    }
    issue(0);
    for (int j = 0; j < ny; j++) {
        const float beta = p.ywt[y0 + j];
        __syncwarp();                      // readers of the previous row are done
        const int mis = commit(j);
        __syncwarp();
        if (j + 1 < ny) issue(j + 1);
        const uint32_t *wp = reinterpret_cast<const uint32_t *>(rowbuf + mis - b_lo + C * gs);
        float b0 = 0.f, b1 = 0.f, b2 = 0.f;
#define FM_G4(W0, W1, W2, a, n)                                                                               \
        b0 = __fadd_rn(b0, fm_byte_mul(W0, 0, a.x, n.x)); b1 = __fadd_rn(b1, fm_byte_mul(W0, 1, a.x, n.x));       \
        b2 = __fadd_rn(b2, fm_byte_mul(W0, 2, a.x, n.x)); b0 = __fadd_rn(b0, fm_byte_mul(W0, 3, a.y, n.y));       \
        b1 = __fadd_rn(b1, fm_byte_mul(W1, 0, a.y, n.y)); b2 = __fadd_rn(b2, fm_byte_mul(W1, 1, a.y, n.y));       \
        b0 = __fadd_rn(b0, fm_byte_mul(W1, 2, a.z, n.z)); b1 = __fadd_rn(b1, fm_byte_mul(W1, 3, a.z, n.z));       \
        b2 = __fadd_rn(b2, fm_byte_mul(W2, 0, a.z, n.z)); b0 = __fadd_rn(b0, fm_byte_mul(W2, 1, a.w, n.w));       \
        b1 = __fadd_rn(b1, fm_byte_mul(W2, 2, a.w, n.w)); b2 = __fadd_rn(b2, fm_byte_mul(W2, 3, a.w, n.w));
#define FM_G4A(W0, W1, W2, W3, a, n)                                                                          \
        b0 = __fadd_rn(b0, fm_byte_mul(W0, 0, a.x, n.x)); b1 = __fadd_rn(b1, fm_byte_mul(W0, 1, a.x, n.x));       \
        b2 = __fadd_rn(b2, fm_byte_mul(W0, 2, a.x, n.x)); b0 = __fadd_rn(b0, fm_byte_mul(W1, 0, a.y, n.y));       \
        b1 = __fadd_rn(b1, fm_byte_mul(W1, 1, a.y, n.y)); b2 = __fadd_rn(b2, fm_byte_mul(W1, 2, a.y, n.y));       \
        b0 = __fadd_rn(b0, fm_byte_mul(W2, 0, a.z, n.z)); b1 = __fadd_rn(b1, fm_byte_mul(W2, 1, a.z, n.z));       \
        b2 = __fadd_rn(b2, fm_byte_mul(W2, 2, a.z, n.z)); b0 = __fadd_rn(b0, fm_byte_mul(W3, 0, a.w, n.w));       \
        b1 = __fadd_rn(b1, fm_byte_mul(W3, 1, a.w, n.w)); b2 = __fadd_rn(b2, fm_byte_mul(W3, 2, a.w, n.w));
#define FM_G1(W0, a, n)                                                                                       \
        b0 = __fadd_rn(b0, fm_byte_mul(W0, 0, a.x, n.x)); b0 = __fadd_rn(b0, fm_byte_mul(W0, 1, a.y, n.y));       \
        b0 = __fadd_rn(b0, fm_byte_mul(W0, 2, a.z, n.z)); b0 = __fadd_rn(b0, fm_byte_mul(W0, 3, a.w, n.w));
        if (C == 4 && inreg) {          // four-byte pixels: a group is 4 words, the fourth byte of each is skipped
#pragma unroll
            for (int g = 0; g < K0_RG; g++) {
                if (g < gmax) {     // braces: the macro is several statements, all of them guarded
                    FM_G4A(wp[4 * g], wp[4 * g + 1], wp[4 * g + 2], wp[4 * g + 3], wr[g], wn[g])
                }
            }
        } else if (C == 4) {
#pragma unroll 2
            for (int g = 0; g < gn; g++) {
                const float4 a = __ldg(gw + g);
                const float4 n = make_float4(__fmul_rn(a.x, -8388608.0f), __fmul_rn(a.y, -8388608.0f),
                                             __fmul_rn(a.z, -8388608.0f), __fmul_rn(a.w, -8388608.0f));
                FM_G4A(wp[4 * g], wp[4 * g + 1], wp[4 * g + 2], wp[4 * g + 3], a, n)
            }
        } else if (C == 1 && inreg) {
#pragma unroll
            for (int g = 0; g < K0_RG; g++) {
                if (g < gmax) FM_G1(wp[g], wr[g], wn[g])
            }
        } else if (C == 1) {
#pragma unroll 2
            for (int g = 0; g < gn; g++) {
                const float4 a = __ldg(gw + g);
                const float4 n = make_float4(__fmul_rn(a.x, -8388608.0f), __fmul_rn(a.y, -8388608.0f),
                                             __fmul_rn(a.z, -8388608.0f), __fmul_rn(a.w, -8388608.0f));
                FM_G1(wp[g], a, n)
            }
        } else if (inreg) {            // the column's weights live in registers for all source rows
#pragma unroll
            for (int g = 0; g < K0_RG; g++) {
                if (g < gmax) {     // warp-uniform: lanes with fewer groups add exact zeros (zero weights, finite bytes)
                    const uint32_t W0 = wp[3 * g], W1 = wp[3 * g + 1], W2 = wp[3 * g + 2];
                    FM_G4(W0, W1, W2, wr[g], wn[g])
                }
            }
        } else {
#pragma unroll 2
            for (int g = 0; g < gn; g++) {
                const uint32_t W0 = wp[3 * g], W1 = wp[3 * g + 1], W2 = wp[3 * g + 2];
                const float4 a = __ldg(gw + g);
                const float4 n = make_float4(__fmul_rn(a.x, -8388608.0f), __fmul_rn(a.y, -8388608.0f),
                                             __fmul_rn(a.z, -8388608.0f), __fmul_rn(a.w, -8388608.0f));
                FM_G4(W0, W1, W2, a, n)
            }
        }
#undef FM_G4
#undef FM_G1
#undef FM_G4A
        if (j == 0) {
            s0 = __fmul_rn(beta, b0); s1 = __fmul_rn(beta, b1); s2 = __fmul_rn(beta, b2);
        } else {
            s0 = __fadd_rn(s0, __fmul_rn(beta, b0));
            s1 = __fadd_rn(s1, __fmul_rn(beta, b1));
            s2 = __fadd_rn(s2, __fmul_rn(beta, b2));
        }
    }
    if (live) {
        int v0 = min(max(__float2int_rn(s0), 0), 255);
        int v1 = min(max(__float2int_rn(s1), 0), 255);
        int v2 = min(max(__float2int_rn(s2), 0), 255);
        p.gray[((size_t)f * p.h + dy) * p.w + dx] = C == 1 ? (uint8_t)v0 : (uint8_t)fm_gray<RGB>(v0, v1, v2);
    }
}

int fm_launch_gray_plane(fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, size_t pitch, int T, cudaStream_t st) {
    dim3 grid(((c->N + 3) / 4 + 255) / 256, c->S * T);
    fm_px_dispatch(c->px_bytes, c->rgb, [&](auto C, auto RGB) {
        k_gray<C.value, RGB.value><<<grid, 256, 0, st>>>(frames, sstride, fstride, pitch, T, c->w, c->N, c->gray, c->nvalid);
    });
    FM_LAUNCH_CHECK();
    return FM_OK;
}

template <int C, bool RGB = false>
static int launch_resize_warps(fm_ctx *c, const K0Params &p, const uint8_t *frames, size_t sstride, size_t fstride, size_t pitch,
                               int F, cudaStream_t st) {
    // one warp per (frame, destination row, group of <= 32 destination columns)
    int nq = (c->w + 31) / 32, dxw = (c->w + nq - 1) / nq;
    int segpitch = ((c->W * C + nq - 1) / nq + C * (c->xtab.max_taps + 10) + 32 + 15) & ~15;
    size_t smemw = (size_t)K0W_WARPS * segpitch;
    int rc;
    if ((rc = fm_ensure_smem((const void *)k_resize_gray_warp<C, RGB>, smemw, c->cfg.device))) return rc;
    int tasks = c->h * F * nq;
    const bool aligned4 = ((((uintptr_t)frames) | sstride | fstride | pitch | ((size_t)c->W * C)) & 3) == 0;
    if (aligned4 && c->g4w) {
        if ((rc = fm_ensure_smem((const void *)k_resize_gray_g4<4, true, C, RGB>, smemw, c->cfg.device))) return rc;
        if ((rc = fm_ensure_smem((const void *)k_resize_gray_g4<4, false, C, RGB>, smemw, c->cfg.device))) return rc;
        if ((rc = fm_ensure_smem((const void *)k_resize_gray_g4<8, true, C, RGB>, smemw, c->cfg.device))) return rc;
        if ((rc = fm_ensure_smem((const void *)k_resize_gray_g4<8, false, C, RGB>, smemw, c->cfg.device))) return rc;
        if ((rc = fm_ensure_smem((const void *)k_resize_gray_g4<16, true, C, RGB>, smemw, c->cfg.device))) return rc;
        if ((rc = fm_ensure_smem((const void *)k_resize_gray_g4<16, false, C, RGB>, smemw, c->cfg.device))) return rc;
        K0GParams gp;
        gp.g4start = c->g4start; gp.g4n = c->g4n; gp.g4off = c->g4off; gp.g4w = c->g4w;
        const int blocks16 = segpitch / 16 + 1;         // upper bound of 16-byte blocks per segment
        const int gridw = (tasks + K0W_WARPS - 1) / K0W_WARPS;
        const bool inreg = c->g4max <= K0_RG;
#define FM_K0(PF)                                                                                                   \
        do {                                                                                                        \
            if (inreg) k_resize_gray_g4<PF, true, C, RGB><<<gridw, 32 * K0W_WARPS, smemw, st>>>(p, gp, segpitch, tasks, nq, dxw); \
            else k_resize_gray_g4<PF, false, C, RGB><<<gridw, 32 * K0W_WARPS, smemw, st>>>(p, gp, segpitch, tasks, nq, dxw);     \
        } while (0)
        if (blocks16 <= 4 * 32) FM_K0(4);
        else if (blocks16 <= 8 * 32) FM_K0(8);
        else if (blocks16 <= 16 * 32) FM_K0(16);
        else k_resize_gray_warp<C, RGB><<<gridw, 32 * K0W_WARPS, smemw, st>>>(p, segpitch, tasks, nq, dxw);
#undef FM_K0
    } else {
        k_resize_gray_warp<C, RGB><<<(tasks + K0W_WARPS - 1) / K0W_WARPS, 32 * K0W_WARPS, smemw, st>>>(p, segpitch, tasks, nq, dxw);
    }
    FM_LAUNCH_CHECK();
    return FM_OK;
}

int fm_launch_frontend(fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, size_t pitch, int T,
                       cudaStream_t st) {
    const int F = c->S * T;
    const int C = c->px_bytes;
    // every Gaussian the fused stencil does not take goes to the tensor-core blur (k_wide.cu)
    if (c->resize_mode == 0)          // gray fused into the first kernel of the blur (gray frames: they are the gray plane)
        return c->umma ? fm_launch_umma_blur(c, frames, sstride, fstride, pitch, T, st)
                       : fm_launch_wide_blur(c, frames, sstride, fstride, pitch, T, st);
    if (c->resize_mode == 3) {        // upscale + gray into the gray plane (k_upscale.cu)
        int rc;
        if ((rc = fm_launch_upscale(c->cfg.device, frames, sstride, fstride, pitch, T, F, c->W, c->H, c->w, c->h, c->uxt, c->uyt,
                                    c->nvalid, c->gray, nullptr, nullptr, 0, st, C, c->rgb)))
            return rc;
    } else {
        K0Params p;
        p.frames = frames; p.sstride = sstride; p.fstride = fstride; p.pitch = pitch;
        p.T = T; p.W = c->W; p.H = c->H; p.w = c->w; p.h = c->h;
        p.mode = c->resize_mode; p.fx = c->fx; p.fy = c->fy;
        p.xstart = c->xtab.start; p.xidx = c->xtab.idx; p.xwt = c->xtab.wt;
        p.ystart = c->ytab.start; p.yidx = c->ytab.idx; p.ywt = c->ytab.wt;
        p.max_ytaps = c->resize_mode == 1 ? c->ytab.max_taps : c->fy;
        p.gray = c->gray; p.nvalid = c->nvalid; p.bgr_out = nullptr;
        int rowpitch = (c->W * C + 16 + 15) & ~15;
        int rc;
        if (c->resize_mode == 1 && fm_rows_usable(c, frames, sstride, fstride, pitch)) {
            // one source row per lane, TMA-staged (k_resize_rows.cu)
            if ((rc = fm_launch_resize_rows(c, frames, sstride, fstride, pitch, T, st))) return rc;
        } else if (c->resize_mode == 1) {
            fm_px_dispatch(c->px_bytes, c->rgb, [&](auto Cx, auto RGB) {
                rc = launch_resize_warps<Cx.value, RGB.value>(c, p, frames, sstride, fstride, pitch, F, st);
            });
            if (rc) return rc;
        } else {
            size_t smem = (size_t)K0_GROUPS * rowpitch + (size_t)p.max_ytaps * c->w * C * sizeof(float);
            if (smem > 220 * 1024) {
                fm_set_error("resize front end needs %zu bytes of shared memory (frame too wide / ratio too large)", smem);
                return FM_ERANGE;
            }
            dim3 grid(c->h, F);
            fm_px_dispatch(c->px_bytes, c->rgb, [&](auto Cx, auto RGB) {
                if ((rc = fm_ensure_smem((const void *)k_resize_gray<Cx.value, RGB.value>, smem, c->cfg.device))) return;
                k_resize_gray<Cx.value, RGB.value><<<grid, K0_THREADS, smem, st>>>(p, nullptr, 0);
            });
            if (rc) return rc;
            FM_LAUNCH_CHECK();
        }
    }
    return c->umma ? fm_launch_umma_blur(c, nullptr, 0, 0, 0, T, st) : fm_launch_wide_blur(c, nullptr, 0, 0, 0, T, st);
}
