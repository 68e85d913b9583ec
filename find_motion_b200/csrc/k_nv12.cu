// NV12 input (FM_FLAG_NV12), staged path: the valid frames of the call are converted to BGR exactly as
// cv2.cvtColor(COLOR_YUV2BGR_NV12) does it (fm_nv12_bgr, fm_device.cuh) into the context's slot [S][T][H][W][3], packed
// like a dense BGR batch of the call, and the unchanged BGR front end reads that slot.  This serves every configuration
// except the fused full-resolution one (k_fused reads NV12 itself): the wide and tcgen05 blurs, the resize modes,
// integer ratios and the upscale.  One launch, counted in the front-end timing group (the stamps of the chained front
// end, or the events around the front end).
#include "fm_common.cuh"

#define NV12_THREADS 256

// 8 pixels of one row (8 luma bytes, the 4 chroma blocks they fall in) -> 24 BGR bytes as 3 words of 8 bytes
__device__ __forceinline__ void nv12_row8(uint2 yv, const FmChroma (&c)[4], uint2 *dst) {
    uint32_t o[6] = {0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const uint32_t y = ((i < 4 ? yv.x : yv.y) >> (8 * (i & 3))) & 0xFFu;
        uint32_t b, g, r;
        fm_nv12_bgr(y, c[i >> 1], b, g, r);
        o[(3 * i) >> 2] |= b << (8 * ((3 * i) & 3));
        o[(3 * i + 1) >> 2] |= g << (8 * ((3 * i + 1) & 3));
        o[(3 * i + 2) >> 2] |= r << (8 * ((3 * i + 2) & 3));
    }
    dst[0] = make_uint2(o[0], o[1]);
    dst[1] = make_uint2(o[2], o[3]);
    dst[2] = make_uint2(o[4], o[5]);
}

// One thread per (row pair, unit): VEC = 8 columns with 8-byte loads and stores (W % 8 == 0, 8-byte aligned frames,
// strides, pitch and chroma offset), otherwise one 2 x 2 block with byte accesses.  Luma row y of a frame is at y * pitch,
// chroma row y at uv + y * pitch.  blockIdx.y = frame t, blockIdx.z = stream s.  oidx (the
// detector input planes of a fused context, k_objects.cu): null, or [S][T] and only the frames with oidx >= 0 are converted.
template <bool VEC>
__global__ void __launch_bounds__(NV12_THREADS) k_nv12_bgr(const uint8_t *__restrict__ frames, size_t sstride, size_t fstride,
                                                           size_t pitch, int64_t uv_off, int T, int W, int H, const int *__restrict__ nvalid,
                                                           const int *__restrict__ oidx, uint8_t *__restrict__ bgr,
                                                           unsigned long long *stamp) {
    fm_stamp_start(stamp);
    const int t = blockIdx.y, s = blockIdx.z, f = s * T + t;
    const int cols = VEC ? W / 8 : W / 2;
    const int u = blockIdx.x * NV12_THREADS + threadIdx.x;
    if ((oidx ? __ldg(oidx + f) >= 0 : t < __ldg(nvalid + s)) && u < cols * (H / 2)) {
        const int yb = u / cols, x = (u - yb * cols) * (VEC ? 8 : 2);
        const uint8_t *src = frames + (size_t)s * sstride + (size_t)t * fstride;
        const uint8_t *l0 = src + (size_t)(2 * yb) * pitch + x, *l1 = l0 + pitch;
        const uint8_t *uv = src + uv_off + (ptrdiff_t)((size_t)yb * pitch + x);
        uint8_t *d0 = bgr + (((size_t)f * H + 2 * yb) * W + x) * 3, *d1 = d0 + (size_t)W * 3;
        if (VEC) {
            const uint2 cv = __ldg(reinterpret_cast<const uint2 *>(uv));
            FmChroma c[4];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const uint32_t w = j < 2 ? cv.x : cv.y;
                c[j] = fm_nv12_chroma((w >> (16 * (j & 1))) & 0xFFu, (w >> (16 * (j & 1) + 8)) & 0xFFu);
            }
            nv12_row8(__ldg(reinterpret_cast<const uint2 *>(l0)), c, reinterpret_cast<uint2 *>(d0));
            nv12_row8(__ldg(reinterpret_cast<const uint2 *>(l1)), c, reinterpret_cast<uint2 *>(d1));
        } else {
            const FmChroma c = fm_nv12_chroma(uv[0], uv[1]);
#pragma unroll
            for (int i = 0; i < 4; i++) {
                uint32_t b, g, r;
                fm_nv12_bgr((i < 2 ? l0 : l1)[i & 1], c, b, g, r);
                uint8_t *d = (i < 2 ? d0 : d1) + 3 * (i & 1);
                d[0] = (uint8_t)b; d[1] = (uint8_t)g; d[2] = (uint8_t)r;
            }
        }
    }
    fm_stamp_end(stamp);
}

int fm_launch_nv12_bgr(fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, size_t pitch, int64_t uv, int T,
                       const int *oidx, uint8_t *bgr, cudaStream_t st) {
    const bool vec = c->W % 8 == 0 && ((((uintptr_t)frames) | sstride | fstride | pitch | (size_t)uv) & 7) == 0;
    const int units = (vec ? c->W / 8 : c->W / 2) * (c->H / 2);
    const dim3 grid((units + NV12_THREADS - 1) / NV12_THREADS, T, c->S);     // S, T <= 65535: fm_ctx_create
    if (vec) k_nv12_bgr<true><<<grid, NV12_THREADS, 0, st>>>(frames, sstride, fstride, pitch, uv, T, c->W, c->H, c->nvalid, oidx, bgr, c->stamp);
    else k_nv12_bgr<false><<<grid, NV12_THREADS, 0, st>>>(frames, sstride, fstride, pitch, uv, T, c->W, c->H, c->nvalid, oidx, bgr, c->stamp);
    FM_LAUNCH_CHECK();
    return FM_OK;
}
