// Device-side look-back cache and motion-clip write-back (FM_FLAG_DEVICE_CLIPS, fm_process_clip).
//
// The reference keeps the last cache_frames raw frames in a deque and flushes it into the output when motion starts
// (find_motion.py:415, 561-570, 588).  A write with a non-empty cache always flushes it, and the cache grows only
// while nothing is written, so the cache always holds the last cache_len frames of the stream, consecutive, ending at
// the current frame (SURVEY.md A.9; tests/test_clips_plan.py).  A ring of C = cache_frames slots per stream, indexed
// by absolute frame number mod C, replaces the deque; the schedule of a call follows from the stats k_decide wrote
// and the stream's frame counter `base` (tests/clips_restated.py restates it):
//   * flushed frame b >= base is input frame b - base, b < base is ring slot b mod C;
//   * the frames still cached at the end of the call that the ring does not hold yet, base + Ts - m .. base + Ts - 1
//     with m = min(cache_len of the last valid frame, Ts), are stored to their slots; then base += Ts.
// A store can overwrite a slot a flush earlier in the same call still reads (T > C), so every gather of the call runs
// in one launch and the stores in the next.
//
// Launches: k_clip_plan (one CTA, one warp per stream) writes both copy lists, k_clip_gather runs the gather list, then
// k_clip_store the store list.  Without the flag none of this runs.  Calls whose frames have a row pitch or a chroma
// offset of their own (fm_process_frames) run k_clip_gather_pitched / k_clip_store_pitched instead: entries that read an
// input frame copy its rows into the packed ring slot or output frame, ring slots are copied whole as above.
#include <algorithm>

#include "fm_common.cuh"

#define CLIP_PLAN_THREADS 1024
#define CLIP_COPY_THREADS 256
#define CLIP_VEC_PER_THREAD 8                                            // 16-byte loads in flight per thread
#define CLIP_CHUNK_BYTES (CLIP_COPY_THREADS * CLIP_VEC_PER_THREAD * 16)  // bytes of a frame per (copy, chunk) item

struct ClipPlanArgs {
    const fm_frame_stats *stats;   // [S][T] of this call
    const int *nvalid;             // [S]
    long long *base;               // [S] frame counters (null when C == 0)
    const uint8_t *frames;
    size_t sstride, fstride;
    uint8_t *ring;                 // [S][C] slots of slot_bytes
    size_t slot_bytes;
    uint8_t *out;                  // null: no gather (the plain entry points only keep the ring up to date)
    size_t ostride;
    size_t fb;                     // bytes of one input frame (fm_ctx::frame_bytes)
    int S, T, C;
    FmClipCopy *gather, *store;
    int *count;                    // [2] entries of the gather and of the store list
};

__device__ __forceinline__ const uint8_t *clip_src(const ClipPlanArgs &a, int s, long long b, long long base) {
    if (b >= base) return a.frames + (size_t)s * a.sstride + (size_t)(b - base) * a.fstride;
    return a.ring + ((size_t)s * a.C + (size_t)(b % a.C)) * a.slot_bytes;
}

__global__ void __launch_bounds__(CLIP_PLAN_THREADS) k_clip_plan(ClipPlanArgs a) {
    __shared__ int n_gather, n_store;
    if (threadIdx.x == 0) n_gather = n_store = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int s = warp; s < a.S; s += CLIP_PLAN_THREADS / 32) {
        const int Ts = min(a.T, a.nvalid[s]);
        if (Ts <= 0) continue;
        const long long base = a.base ? a.base[s] : 0;
        if (a.out) {
            int off = 0;                                             // output frames of the stream so far
            for (int tc = 0; tc < Ts; tc += 32) {
                const int t = tc + lane;
                int wrote = 0, nf = 0;
                if (t < Ts) {
                    const fm_frame_stats r = a.stats[(size_t)s * a.T + t];
                    wrote = r.wrote; nf = r.n_flush;
                }
                const int cnt = wrote + nf;
                int incl = cnt;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const int v = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= d) incl += v;
                }
                const int total = __shfl_sync(0xffffffffu, incl, 31);
                int g0 = 0;
                if (lane == 0 && total) g0 = atomicAdd(&n_gather, total);
                g0 = __shfl_sync(0xffffffffu, g0, 0) + incl - cnt;   // this lane's first list entry
                uint8_t *dst = a.out + (size_t)s * a.ostride + (size_t)(off + incl - cnt) * a.fb;
                for (int j = 0; j < cnt; j++) {                      // n_flush cached frames, then the frame itself
                    const long long b = base + t - nf + j;
                    a.gather[g0 + j] = FmClipCopy{clip_src(a, s, b, base), dst + (size_t)j * a.fb};
                }
                off += total;
            }
        }
        if (a.C > 0) {
            const int m = min(a.stats[(size_t)s * a.T + Ts - 1].cache_len, Ts);
            int s0 = 0;
            if (lane == 0 && m) s0 = atomicAdd(&n_store, m);
            s0 = __shfl_sync(0xffffffffu, s0, 0);
            for (int j = lane; j < m; j += 32) {
                const int t = Ts - m + j;
                const long long b = base + t;
                a.store[s0 + j] = FmClipCopy{a.frames + (size_t)s * a.sstride + (size_t)t * a.fstride,
                                             a.ring + ((size_t)s * a.C + (size_t)(b % a.C)) * a.slot_bytes};
            }
            if (lane == 0) a.base[s] = base + Ts;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) { a.count[0] = n_gather; a.count[1] = n_store; }
}

// One frame copy of fb bytes per list entry, cut into chunks of CLIP_CHUNK_BYTES; a grid-stride loop over
// (entry, chunk).  Source and destination with the same offset mod 16 (the ring slots are 256-byte aligned; dense
// frames whose size is a multiple of 16) take 16-byte streaming loads and stores, several in flight per thread, with
// the head and tail bytes done by chunk 0; any other pair is copied byte by byte.
__device__ __forceinline__ void clip_copy(const FmClipCopy *__restrict__ list, const int *__restrict__ count, size_t fb) {
    const size_t nch = (fb + CLIP_CHUNK_BYTES - 1) / CLIP_CHUNK_BYTES;
    const size_t items = (size_t)__ldg(count) * nch;
    for (size_t it = blockIdx.x; it < items; it += gridDim.x) {
        const size_t e = it / nch, ch = it % nch;
        const FmClipCopy cp = list[e];
        const uint8_t *src = cp.src;
        uint8_t *dst = cp.dst;
        if ((((uintptr_t)src ^ (uintptr_t)dst) & 15) == 0) {
            const size_t head = min(fb, (size_t)((16 - ((uintptr_t)dst & 15)) & 15));
            const size_t nv = (fb - head) / 16, tail0 = head + nv * 16;
            if (ch == 0) {
                if (threadIdx.x < head) dst[threadIdx.x] = src[threadIdx.x];
                if (threadIdx.x < fb - tail0) dst[tail0 + threadIdx.x] = src[tail0 + threadIdx.x];
            }
            const int4 *s4 = reinterpret_cast<const int4 *>(src + head);
            int4 *d4 = reinterpret_cast<int4 *>(dst + head);
            const size_t v0 = ch * (CLIP_CHUNK_BYTES / 16) + threadIdx.x;
            int4 r[CLIP_VEC_PER_THREAD];
#pragma unroll
            for (int k = 0; k < CLIP_VEC_PER_THREAD; k++) {
                const size_t v = v0 + (size_t)k * CLIP_COPY_THREADS;
                if (v < nv) r[k] = __ldcs(s4 + v);
            }
#pragma unroll
            for (int k = 0; k < CLIP_VEC_PER_THREAD; k++) {
                const size_t v = v0 + (size_t)k * CLIP_COPY_THREADS;
                if (v < nv) __stcs(d4 + v, r[k]);
            }
        } else {
            const size_t b0 = ch * CLIP_CHUNK_BYTES, b1 = min(fb, b0 + CLIP_CHUNK_BYTES);
            for (size_t b = b0 + threadIdx.x; b < b1; b += CLIP_COPY_THREADS) dst[b] = __ldcs(src + b);
        }
    }
}

// two names, so that a profile tells the gathers of fm_process_clip from the ring stores
__global__ void __launch_bounds__(CLIP_COPY_THREADS) k_clip_gather(const FmClipCopy *__restrict__ list,
                                                                   const int *__restrict__ count, size_t fb) {
    clip_copy(list, count, fb);
}
__global__ void __launch_bounds__(CLIP_COPY_THREADS) k_clip_store(const FmClipCopy *__restrict__ list,
                                                                  const int *__restrict__ count, size_t fb) {
    clip_copy(list, count, fb);
}

// The row layout of a pitched call's input frames: rows of rowbytes, `pitch` apart; rows >= luma_rows (the NV12 chroma
// rows) start at uv + (row - luma_rows) * pitch.  Sources inside [ring, ring_end) are ring slots, dense like the outputs.
struct ClipRows {
    size_t pitch, rowbytes;
    int64_t uv;
    int luma_rows, rows, rows_per_item;
    const uint8_t *ring, *ring_end;
};

// n bytes by the whole CTA: 16-byte streaming accesses when source and destination agree mod 16, bytes otherwise
__device__ __forceinline__ void clip_span(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, size_t n) {
    if ((((uintptr_t)src ^ (uintptr_t)dst) & 15) == 0) {
        const size_t head = min(n, (size_t)((16 - ((uintptr_t)dst & 15)) & 15));
        const size_t nv = (n - head) / 16, tail0 = head + nv * 16;
        if (threadIdx.x < head) dst[threadIdx.x] = src[threadIdx.x];
        if (threadIdx.x < n - tail0) dst[tail0 + threadIdx.x] = src[tail0 + threadIdx.x];
        const int4 *s4 = reinterpret_cast<const int4 *>(src + head);
        int4 *d4 = reinterpret_cast<int4 *>(dst + head);
        for (size_t v = threadIdx.x; v < nv; v += CLIP_COPY_THREADS) __stcs(d4 + v, __ldcs(s4 + v));
    } else {
        for (size_t b = threadIdx.x; b < n; b += CLIP_COPY_THREADS) dst[b] = __ldcs(src + b);
    }
}

// clip_copy for pitched calls: item (entry, ch) is chunk ch of a ring slot, or rows ch * rows_per_item .. of an input frame
__device__ __forceinline__ void clip_copy_pitched(const FmClipCopy *__restrict__ list, const int *__restrict__ count, size_t fb,
                                                  const ClipRows &g) {
    const size_t nch = max((fb + CLIP_CHUNK_BYTES - 1) / CLIP_CHUNK_BYTES,
                           (size_t)((g.rows + g.rows_per_item - 1) / g.rows_per_item));
    const size_t items = (size_t)__ldg(count) * nch;
    for (size_t it = blockIdx.x; it < items; it += gridDim.x) {
        const size_t e = it / nch, ch = it % nch;
        const FmClipCopy cp = list[e];
        if (cp.src >= g.ring && cp.src < g.ring_end) {
            const size_t b0 = ch * CLIP_CHUNK_BYTES;
            if (b0 < fb) clip_span(cp.src + b0, cp.dst + b0, min((size_t)CLIP_CHUNK_BYTES, fb - b0));
        } else {
            const int r0 = (int)ch * g.rows_per_item, r1 = min(g.rows, r0 + g.rows_per_item);
            for (int r = r0; r < r1; r++) {
                const uint8_t *s = r < g.luma_rows ? cp.src + (size_t)r * g.pitch
                                                   : cp.src + g.uv + (ptrdiff_t)((size_t)(r - g.luma_rows) * g.pitch);
                clip_span(s, cp.dst + (size_t)r * g.rowbytes, g.rowbytes);
            }
        }
    }
}

__global__ void __launch_bounds__(CLIP_COPY_THREADS) k_clip_gather_pitched(const FmClipCopy *__restrict__ list,
                                                                           const int *__restrict__ count, size_t fb,
                                                                           ClipRows g) {
    clip_copy_pitched(list, count, fb, g);
}
__global__ void __launch_bounds__(CLIP_COPY_THREADS) k_clip_store_pitched(const FmClipCopy *__restrict__ list,
                                                                          const int *__restrict__ count, size_t fb,
                                                                          ClipRows g) {
    clip_copy_pitched(list, count, fb, g);
}

int fm_clips_alloc(fm_ctx *c) {
    const int C = c->info.cache_frames;
    const size_t fb = c->frame_bytes;
    c->clip_slot_bytes = (fb + 255) & ~(size_t)255;
    if (C > 0) {
        const size_t ring = (size_t)c->S * C * c->clip_slot_bytes;
        cudaError_t e = cudaMalloc((void **)&c->clip_ring, ring);
        if (e != cudaSuccess) {
            cudaGetLastError();
            fm_set_error("device clip ring: cudaMalloc(%zu bytes = %d streams x %d cached frames x %zu) failed: %s", ring,
                         c->S, C, c->clip_slot_bytes, cudaGetErrorString(e));
            return FM_ENOMEM;
        }
        e = cudaMalloc((void **)&c->clip_base, (size_t)c->S * sizeof(long long));
        if (e != cudaSuccess) { cudaGetLastError(); fm_set_error("device clip frame counters: %s", cudaGetErrorString(e)); return FM_ENOMEM; }
        FM_CUDA(cudaMemset(c->clip_base, 0, (size_t)c->S * sizeof(long long)));
    }
    const size_t ng = (size_t)c->S * (C + c->Tmax), ns = (size_t)c->S * std::min(C, c->Tmax);
    FM_CUDA(cudaMalloc((void **)&c->clip_list, (ng + ns) * sizeof(FmClipCopy)));
    FM_CUDA(cudaMalloc((void **)&c->clip_count, 2 * sizeof(int)));
    int dev = 0;
    FM_CUDA(cudaGetDevice(&dev));
    FM_CUDA(cudaDeviceGetAttribute(&c->clip_sms, cudaDevAttrMultiProcessorCount, dev));
    return FM_OK;
}

void fm_clips_free(fm_ctx *c) {
    cudaFree(c->clip_ring); cudaFree(c->clip_base); cudaFree(c->clip_list); cudaFree(c->clip_count);
}

int fm_launch_clips(fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, size_t pitch, int64_t uv, int T,
                    uint8_t *out, size_t ostride, cudaStream_t st) {
    const int C = c->info.cache_frames;
    if (!out && C == 0) return FM_OK;                    // nothing to gather and no ring to keep
    ClipPlanArgs a;
    a.stats = c->stats; a.nvalid = c->nvalid; a.base = c->clip_base;
    a.frames = frames; a.sstride = sstride; a.fstride = fstride;
    a.ring = c->clip_ring; a.slot_bytes = c->clip_slot_bytes;
    a.out = out; a.ostride = ostride;
    a.fb = c->frame_bytes;
    a.S = c->S; a.T = T; a.C = C;
    const size_t ng = (size_t)c->S * (C + c->Tmax);
    a.gather = c->clip_list; a.store = c->clip_list + ng;
    a.count = c->clip_count;
    k_clip_plan<<<1, CLIP_PLAN_THREADS, 0, st>>>(a);
    FM_LAUNCH_CHECK();
    const bool nv12 = (c->cfg.flags & FM_FLAG_NV12) != 0;
    ClipRows g;
    g.rowbytes = c->row_bytes;
    g.pitch = pitch; g.uv = uv;
    g.luma_rows = c->H; g.rows = nv12 ? c->H + c->H / 2 : c->H;
    g.rows_per_item = (int)std::max<size_t>(1, CLIP_CHUNK_BYTES / g.rowbytes);
    g.ring = c->clip_ring; g.ring_end = c->clip_ring ? c->clip_ring + (size_t)c->S * C * c->clip_slot_bytes : nullptr;
    if (pitch != g.rowbytes || (nv12 && uv != (int64_t)(g.rowbytes * c->H))) {
        const size_t nch = std::max((a.fb + CLIP_CHUNK_BYTES - 1) / CLIP_CHUNK_BYTES,
                                    (size_t)((g.rows + g.rows_per_item - 1) / g.rows_per_item));
        auto grid = [&](size_t entries) { return (int)std::max<size_t>(1, std::min<size_t>(entries * nch, (size_t)c->clip_sms * 8)); };
        if (out) {
            k_clip_gather_pitched<<<grid((size_t)c->S * (C + T)), CLIP_COPY_THREADS, 0, st>>>(a.gather, a.count, a.fb, g);
            FM_LAUNCH_CHECK();
        }
        if (C > 0) {
            k_clip_store_pitched<<<grid((size_t)c->S * std::min(C, T)), CLIP_COPY_THREADS, 0, st>>>(a.store, a.count + 1, a.fb, g);
            FM_LAUNCH_CHECK();
        }
        return FM_OK;
    }
    // grid: enough CTAs to keep every SM streaming, never more than the largest list could use
    const size_t nch = (a.fb + CLIP_CHUNK_BYTES - 1) / CLIP_CHUNK_BYTES;
    auto grid = [&](size_t entries) { return (int)std::max<size_t>(1, std::min<size_t>(entries * nch, (size_t)c->clip_sms * 8)); };
    if (out) {
        k_clip_gather<<<grid((size_t)c->S * (C + T)), CLIP_COPY_THREADS, 0, st>>>(a.gather, a.count, a.fb);
        FM_LAUNCH_CHECK();
    }
    if (C > 0) {
        k_clip_store<<<grid((size_t)c->S * std::min(C, T)), CLIP_COPY_THREADS, 0, st>>>(a.store, a.count + 1, a.fb);
        FM_LAUNCH_CHECK();
    }
    return FM_OK;
}
