// Upscaling front end (resize mode 3): cv2.resize(INTER_AREA) with a destination wider than the source, which cv2
// computes as its fixed-point linear interpolation with area-style offsets (SURVEY.md A.1, tests/upscale_restated.py
// resize_upscale), followed by gray.  Bit-exact with the reference's imutils.resize + cvtColor (find_motion.py:492-493).
//
// Per axis, destination index d reads source indices s = tab[d].x and min(s + 1, n - 1) with 11-bit weights a0, a1
// (tab[d].y = a0 | a1 << 16).  Horizontal: hx = src[s] * a0 + src[s + 1] * a1 (int32, per channel).  Vertical, in the
// form of cv2's VResizeLinear for u8 on every column:
//     v = (((b0 * (hx0 >> 4)) >> 16) + ((b1 * (hx1 >> 4)) >> 16) + 2) >> 2
//
// One CTA per (band of destination rows, frame).  The ratio is >= 1 on both axes, so consecutive destination rows
// read the same or the next source row: the CTA keeps the horizontal pass (hx >> 4, <= 32640, as u16) of two source
// rows in shared memory, computes each source row once, and writes each gray byte once.  Source rows are read
// from global memory once per band (plus the row a band shares with the band above).
#include "fm_common.cuh"

#define UP_THREADS 256
#define UP_BAND_MAX 32          // destination rows per CTA (fewer when the grid would not fill the GPU)

struct UpParams {
    const uint8_t *frames;
    size_t sstride, fstride;
    size_t pitch;               // bytes from one source row to the next (>= W * channels)
    int T, W, H, w, h;
    int band;                   // destination rows per CTA
    const int2 *xt;             // [w] (source x, a0 | a1 << 16)
    const int2 *yt;             // [h] (source y, b0 | b1 << 16)
    const int *nvalid;          // [S] real frames of each stream in this call (null: every frame)
    uint8_t *gray;              // [F][h][w]
    uint8_t *bgr_out;           // [F][h][w][3] resized BGR instead of gray (fm_resize_area: the detector input plane)
    const int *oidx;            // with bgr_out: null, or [F] plane index (-1: skip the frame); frame f's plane then goes to
    size_t ostride;             //   bgr_out + s * ostride + oidx[f] * h*w*3 (fm_object_planes)
};

// horizontal pass of one source row into a staged row of u16 (hx >> 4), 4 destination columns per thread.  C: channels of
// the source (3 BGR, 1 gray; each channel is interpolated the same way)
template <int C>
__device__ __forceinline__ void up_hrow(const UpParams &p, const uint8_t *__restrict__ row, uint16_t *out) {
    const int nq = (p.w + 3) >> 2;
    for (int q = threadIdx.x; q < nq; q += UP_THREADS) {
        const int dx0 = q * 4;
        uint32_t v[4 * C];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int dx = min(dx0 + j, p.w - 1);                       // columns past w: computed, not stored
            const int2 xv = __ldg(p.xt + dx);
            const uint8_t *a = row + C * xv.x;
            const uint8_t *b = row + C * min(xv.x + 1, p.W - 1);
            const uint32_t a0 = (uint32_t)xv.y & 0xffffu, a1 = (uint32_t)xv.y >> 16;
#pragma unroll
            for (int ch = 0; ch < C; ch++) v[C * j + ch] = ((uint32_t)__ldg(a + ch) * a0 + (uint32_t)__ldg(b + ch) * a1) >> 4;
        }
        uint16_t *o = out + 4 * C * q;
        if (dx0 + 4 <= p.w) {                                           // 8 C bytes at a multiple of 8 C: C 8-byte stores
#pragma unroll
            for (int k = 0; k < C; k++)
                reinterpret_cast<uint2 *>(o)[k] = make_uint2(v[4 * k] | (v[4 * k + 1] << 16), v[4 * k + 2] | (v[4 * k + 3] << 16));
        } else {
#pragma unroll
            for (int i = 0; i < 4 * C; i++)
                if (i < C * (p.w - dx0)) o[i] = (uint16_t)v[i];
        }
    }
}

// RGB: R-first three-byte source pixels; their channels are put in BGR order as they leave the vertical pass
template <int C, bool RGB = false>
__global__ void __launch_bounds__(UP_THREADS) k_upscale_gray(UpParams p) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int f = blockIdx.y;                    // s*T + t
    const int s = f / p.T, t = f - s * p.T;
    if (p.nvalid && t >= __ldg(p.nvalid + s)) return;
    const int oi = p.oidx ? __ldg(p.oidx + f) : 0;
    if (oi < 0) return;
    const size_t obase = p.oidx ? (size_t)s * p.ostride + (size_t)oi * p.h * (size_t)(3 * p.w) : (size_t)f * p.h * (size_t)(3 * p.w);
    const uint8_t *src = p.frames + (size_t)s * p.sstride + (size_t)t * p.fstride;
    const size_t rowbytes = p.pitch;
    const int pitch = (C * p.w + 3) & ~3;        // u16 per staged row (rows 8-byte aligned)
    uint16_t *rows = reinterpret_cast<uint16_t *>(smem);    // [2][pitch]: source row y lives in slot y & 1
    const int dy0 = blockIdx.x * p.band, dy1 = min(dy0 + p.band, p.h);
    const int nq = (p.w + 3) >> 2;
    int held0 = -1, held1 = -1;                  // source row in slot 0 / 1 (block-uniform)
    for (int dy = dy0; dy < dy1; dy++) {
        const int2 yv = __ldg(p.yt + dy);
        const int sy0 = yv.x, sy1 = min(yv.x + 1, p.H - 1);
        // the ratio is >= 1: at most one new source row per destination row, except at the top of the band
        const bool need0 = ((sy0 & 1) ? held1 : held0) != sy0;
        const bool need1 = sy1 != sy0 && ((sy1 & 1) ? held1 : held0) != sy1;
        if (need0 || need1) {
            __syncthreads();                     // readers of the slot about to be replaced are done
            if (need0) up_hrow<C>(p, src + (size_t)sy0 * rowbytes, rows + (sy0 & 1) * pitch);
            if (need1) up_hrow<C>(p, src + (size_t)sy1 * rowbytes, rows + (sy1 & 1) * pitch);
            if (need0) { if (sy0 & 1) held1 = sy0; else held0 = sy0; }
            if (need1) { if (sy1 & 1) held1 = sy1; else held0 = sy1; }
            __syncthreads();
        }
        const uint16_t *r0 = rows + (sy0 & 1) * pitch, *r1 = rows + (sy1 & 1) * pitch;
        const uint32_t b0 = (uint32_t)yv.y & 0xffffu, b1 = (uint32_t)yv.y >> 16;
        for (int q = threadIdx.x; q < nq; q += UP_THREADS) {
            const int dx0 = q * 4, n = min(4, p.w - dx0);
            uint32_t h0[4 * C], h1[4 * C];
            if (n == 4) {
#pragma unroll
                for (int k = 0; k < C; k++) {
                    const uint2 u = reinterpret_cast<const uint2 *>(r0 + 4 * C * q)[k];
                    const uint2 l = reinterpret_cast<const uint2 *>(r1 + 4 * C * q)[k];
                    h0[4 * k] = u.x & 0xffffu; h0[4 * k + 1] = u.x >> 16; h0[4 * k + 2] = u.y & 0xffffu; h0[4 * k + 3] = u.y >> 16;
                    h1[4 * k] = l.x & 0xffffu; h1[4 * k + 1] = l.x >> 16; h1[4 * k + 2] = l.y & 0xffffu; h1[4 * k + 3] = l.y >> 16;
                }
            } else {
#pragma unroll
                for (int i = 0; i < 4 * C; i++) {
                    const int ii = min(i, C * n - 1);
                    h0[i] = r0[4 * C * q + ii];
                    h1[i] = r1[4 * C * q + ii];
                }
            }
            uint32_t v[12];                              // 4 pixels x 3 channels, BGR (a gray source: its byte in all three)
#pragma unroll
            for (int i = 0; i < 12; i++) {
                const int k = C == 1 ? i / 3 : C == 4 ? 4 * (i / 3) + (RGB ? 2 - i % 3 : i % 3) : RGB ? i + 2 - 2 * (i % 3) : i;
                v[i] = min((((b0 * h0[k]) >> 16) + ((b1 * h1[k]) >> 16) + 2u) >> 2, 255u);
            }
            if (p.bgr_out) {
                uint8_t *o = p.bgr_out + obase + (size_t)dy * (size_t)(3 * p.w) + 12 * q;
                if (n == 4 && (((uintptr_t)o) & 3) == 0) {
#pragma unroll
                    for (int k = 0; k < 3; k++)
                        reinterpret_cast<uint32_t *>(o)[k] = v[4 * k] | (v[4 * k + 1] << 8) | (v[4 * k + 2] << 16) | (v[4 * k + 3] << 24);
                } else {
#pragma unroll
                    for (int i = 0; i < 12; i++)
                        if (i < 3 * n) o[i] = (uint8_t)v[i];
                }
            } else {
                uint32_t g[4];
#pragma unroll
                for (int j = 0; j < 4; j++) g[j] = C == 1 ? v[3 * j] : fm_gray(v[3 * j], v[3 * j + 1], v[3 * j + 2]);
                uint8_t *o = p.gray + ((size_t)f * p.h + dy) * (size_t)p.w + dx0;
                if (n == 4 && (((uintptr_t)o) & 3) == 0) {
                    *reinterpret_cast<uint32_t *>(o) = g[0] | (g[1] << 8) | (g[2] << 16) | (g[3] << 24);
                } else {
#pragma unroll
                    for (int j = 0; j < 4; j++)
                        if (j < n) o[j] = (uint8_t)g[j];
                }
            }
        }
    }
}

size_t fm_upscale_smem(int w, int channels) {
    return (size_t)2 * (((size_t)(channels > 3 ? channels : 3) * w + 3) & ~(size_t)3) * sizeof(uint16_t);
}

int fm_launch_upscale(int device, const uint8_t *frames, size_t sstride, size_t fstride, size_t pitch, int T, int F, int W, int H,
                      int w, int h, const int2 *xt, const int2 *yt, const int *nvalid, uint8_t *gray, uint8_t *bgr_out,
                      const int *oidx, size_t ostride, cudaStream_t st, int channels, bool rgb) {
    UpParams p;
    p.frames = frames; p.sstride = sstride; p.fstride = fstride; p.pitch = pitch;
    p.T = T; p.W = W; p.H = H; p.w = w; p.h = h;
    p.xt = xt; p.yt = yt; p.nvalid = nvalid; p.gray = gray; p.bgr_out = bgr_out;
    p.oidx = oidx; p.ostride = ostride;
    // taller bands re-read fewer source rows; shorter ones keep every SM busy when there are few frames
    int band = UP_BAND_MAX;
    while (band > 4 && (size_t)((h + band - 1) / band) * F < 4 * 148) band >>= 1;
    p.band = band;
    const size_t smem = fm_upscale_smem(w, channels);
    if (smem > 200 * 1024) {
        fm_set_error("upscale needs %zu bytes of shared memory (destination width %d too large)", smem, w);
        return FM_ERANGE;
    }
    int rc;
    dim3 grid((h + band - 1) / band, F);
    rc = FM_OK;
    fm_px_dispatch(channels, rgb, [&](auto C, auto RGB) {
        if ((rc = fm_ensure_smem((const void *)k_upscale_gray<C.value, RGB.value>, smem, device))) return;
        k_upscale_gray<C.value, RGB.value><<<grid, UP_THREADS, smem, st>>>(p);
    });
    if (rc) return rc;
    FM_LAUNCH_CHECK();
    return FM_OK;
}
