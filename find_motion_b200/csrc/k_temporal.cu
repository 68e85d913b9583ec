// Temporal kernel: per pixel, over the T frames of a call, in frame order
//   bg8 = sat(rne(|float32(bg)|)); thresh = |blur - bg8| > threshold;
//   bg = fma(bg, 1-alpha, rn(blur*alpha))            (tail elements: fma(blur, alpha, rn(bg*(1-alpha))))
// with the float64 background held in registers across the T frames (one HBM read and one
// write of the background per call).  Replaces find_diff's first-frame init, VideoFrame.diff,
// VideoFrame.threshold and cv2.accumulateWeighted (find_motion/find_motion.py:246-257, 651-659;
// SURVEY.md A.4, A.6, A.7).  Pointwise, so pixels are addressed by their flat index i = y*w + x.
#include "fm_common.cuh"

// One lane owns 16 consecutive pixels; a warp owns a 512-pixel tile.  The background tile is
// stored [8][32] double2 so that every 128-bit access of the warp is one contiguous 512 B run.

// One frame of one lane: 16 pixels (bytes of px[4]) -> 16 threshold bits (bit j = pixel j), background updated.
// TAIL: the lane holds the N mod 16 remainder group (A.6: the product order of the AVX2 tail, any alpha and threshold);
// SAFE, INIT: as in fm_temporal_px.
template <bool TAIL, bool SAFE, bool INIT>
__device__ __forceinline__ uint32_t fm_temporal16(const uint32_t (&px)[4], double (&b)[16], int threshold, double alpha,
                                                  double beta) {
    const double nC = -(4503599627370496.0 * alpha);
    const int qoff = 0x4B400000 - threshold;
    const uint32_t nthr2 = ~(2u * (uint32_t)threshold);
    uint32_t bits = 0;
#pragma unroll
    for (int j = 0; j < 16; j++) {
        const uint32_t src = __byte_perm(px[j >> 2], 0, 0x4440 + (j & 3));
        if (TAIL) {
            const double sd = fm_u8_to_f64(src);
            if (INIT) b[j] = sd;
            int d = (int)src - (int)fm_bg8(b[j]);
            d = d < 0 ? -d : d;
            bits = 2u * bits + (d > threshold ? 1u : 0u);
            b[j] = __fma_rn(sd, alpha, __dmul_rn(b[j], beta));
        } else {
            fm_temporal_px<SAFE, INIT>(src, b[j], bits, threshold, qoff, nthr2, alpha, beta, nC);
        }
    }
    return __brev(bits) >> 16;          // pixel 0 was pushed first
}

template <bool SAFE>
__global__ void __launch_bounds__(256) k_temporal(const uint8_t *__restrict__ blur, double *__restrict__ bg,
                                                  uint32_t *__restrict__ tflat, const StreamState *__restrict__ state,
                                                  int T, int N, int ntiles, int threshold, double alpha,
                                                  double beta, int *__restrict__ rawrange, int w, int h,
                                                  const int *__restrict__ nframes) {
    const int s = blockIdx.y;
    const int Ts = min(T, __ldg(nframes + s));              // real frames of this stream in the call (ragged batches)
    if (Ts <= 0) return;
    const int lane = threadIdx.x & 31;
    const int tile = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (tile >= ntiles) return;
    const int i0 = tile * FM_TILE_PX + lane * 16;          // first flat pixel of this lane
    const int nbody = N - (N & 15);
    const bool active = i0 < N;
    const bool tail = i0 >= nbody;                          // the N mod 16 remainder group
    const int nvalid = active ? min(16, N - i0) : 0;
    double2 *bgt = reinterpret_cast<double2 *>(bg) + ((size_t)s * ntiles + tile) * 256;
    const bool has_bg = state[s].has_bg != 0;

    double b[16];
    if (has_bg) {
#pragma unroll
        for (int j = 0; j < 8; j++) {
            double2 v = bgt[j * 32 + lane];
            b[2 * j] = v.x;
            b[2 * j + 1] = v.y;
        }
    }
    const uint8_t *bl = blur + (size_t)s * T * N + i0;
    uint32_t *tw = tflat + ((size_t)s * T) * ((size_t)ntiles * FM_TILE_WORDS) + tile * FM_TILE_WORDS + (lane >> 1);
    const bool vec = (nvalid == 16) && ((((uintptr_t)bl) & 15) == 0) && ((N & 15) == 0);

    for (int t = 0; t < Ts; t++) {
        uint32_t px[4] = {0, 0, 0, 0};
        if (vec) {
            uint4 v = __ldg(reinterpret_cast<const uint4 *>(bl));
            px[0] = v.x; px[1] = v.y; px[2] = v.z; px[3] = v.w;
        } else {
            for (int j = 0; j < nvalid; j++) px[j >> 2] |= (uint32_t)bl[j] << (8 * (j & 3));
        }
        bl += N;
        uint32_t bits;
        if (t == 0 && !has_bg) bits = tail ? fm_temporal16<true, SAFE, true>(px, b, threshold, alpha, beta)
                                           : fm_temporal16<false, SAFE, true>(px, b, threshold, alpha, beta);
        else if (tail) bits = fm_temporal16<true, SAFE, false>(px, b, threshold, alpha, beta);
        else bits = fm_temporal16<false, SAFE, false>(px, b, threshold, alpha, beta);
        if (nvalid < 16) bits &= (1u << nvalid) - 1u;
        uint32_t hi = __shfl_down_sync(0xffffffffu, bits, 1);
        if ((lane & 1) == 0) *tw = bits | (hi << 16);
        tw += (size_t)ntiles * FM_TILE_WORDS;
        if (__any_sync(0xffffffffu, bits != 0) && lane == 0) {       // rows touched by this 512-pixel tile
            int ya = (tile * FM_TILE_PX) / w, yb = min((tile * FM_TILE_PX + FM_TILE_PX - 1) / w, h - 1);
            int *rr = rawrange + 2 * ((size_t)s * T + t);
            atomicMax(rr, yb);
            atomicMax(rr + 1, h - 1 - ya);
        }
    }
#pragma unroll
    for (int j = 0; j < 8; j++) bgt[j * 32 + lane] = make_double2(b[2 * j], b[2 * j + 1]);
}

// background tile layout -> plain row-major float64 plane (parity tests / export)
__global__ void k_bg_export(const double *__restrict__ bg, double *__restrict__ dst, int N, int ntiles, int s) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    int tile = i / FM_TILE_PX, r = i - tile * FM_TILE_PX;
    int lane = r >> 4, j = r & 15;
    dst[i] = bg[(((size_t)s * ntiles + tile) * 256 + (j >> 1) * 32 + lane) * 2 + (j & 1)];
}

int fm_launch_temporal(fm_ctx *c, int T, cudaStream_t st) {
    double alpha = c->cfg.avg;
    double beta = 1.0 - alpha;
    dim3 grid((c->ntiles + 7) / 8, c->S);
    const bool safe = alpha >= 0.0 && alpha <= 1.0 && c->cfg.threshold >= 0;
    if (safe) k_temporal<true><<<grid, 256, 0, st>>>(c->blur, c->bg, c->tflat, c->state, T, c->N, c->ntiles, c->cfg.threshold,
                                                     alpha, beta, c->rawrange, c->w, c->h, c->nvalid);
    else k_temporal<false><<<grid, 256, 0, st>>>(c->blur, c->bg, c->tflat, c->state, T, c->N, c->ntiles, c->cfg.threshold,
                                                 alpha, beta, c->rawrange, c->w, c->h, c->nvalid);
    FM_LAUNCH_CHECK();
    return FM_OK;
}

int fm_launch_bg_export(fm_ctx *c, int stream, double *dst_dev, cudaStream_t st) {
    k_bg_export<<<(c->N + 255) / 256, 256, 0, st>>>(c->bg, dst_dev, c->N, c->ntiles, stream);
    FM_LAUNCH_CHECK();
    return FM_OK;
}
