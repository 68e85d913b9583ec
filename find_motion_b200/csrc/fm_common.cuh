// Shared declarations of libfmgpu.so (sm_100a only).  See include/fm_gpu.h for the C ABI and
// DESIGN.md for the data layout.  Arithmetic follows SURVEY.md Appendix A (verified against the
// reference's cv2 call chain, find_motion/find_motion.py:487-494, 619-700, 549-589).
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <utility>

#include "../../include/fm_gpu.h"
#include "fm_device.cuh"

#define FM_MAX_K 1024          // widest supported Gaussian (taps)
#define FM_TILE_PX 512         // pixels per background tile: 32 lanes x 16 px
#define FM_TILE_WORDS 16       // 32-bit threshold words per tile
#define FM_TIMING_RING 16384
#define FM_MAX_DEVICES 64      // per-device caches of kernel attributes (cudaFuncSetAttribute is per device)

struct StreamState {           // per stream, device resident (find_motion.py:362-371)
    int has_bg;                // ref_frame is not None
    int counter;               // movement_counter
    int decay;                 // movement_decay
    int cache_len;             // len(frame_cache)
};

struct ResizeTab {             // INTER_AREA decimation tables of one axis (SURVEY.md A.1)
    int *start;                // [dst+1] prefix offsets into idx/wt
    int *idx;                  // source index per tap
    float *wt;                 // float32 weight per tap
    int max_taps;
};

struct FmClipCopy {            // one whole-frame copy of the device clip path (k_clips.cu)
    const uint8_t *src;
    uint8_t *dst;
};

struct CclScratch {            // run-based labelling scratch for `frames` frames at a time
    int frames;                // sub-batch capacity
    int cap;                   // run slots per row
    size_t slots;              // per frame: h * cap
    uint16_t *xs, *xe;         // [frames][slots]
    int *rowcnt;               // [frames][h]
    int *parent;               // [frames][1 + slots]   (id 0 = the outside of the image)
    int *area2;                // [frames][slots]
    int *bbox;                 // [frames][slots][4]  xmin, ymin, xmax, ymax
};

struct fm_ctx {
    fm_config cfg;
    fm_info info;
    int S, Tmax, W, H, w, h, k, wpr;
    int N;                     // w*h
    int ntiles;                // ceil(N / FM_TILE_PX)
    int resize_mode;           // 0 identity, 1 general tables, 2 integer ratio, 3 upscale (FM_FLAG_UPSCALE, k_upscale.cu)
    size_t frame_bytes;        // bytes of one input frame: H * W * 3 (BGR) or H * W * 3 / 2 (FM_FLAG_NV12)
    uint8_t *nv12_bgr;         // FM_FLAG_NV12 on the staged path: [S][Tmax][H][W][3] the call's frames converted to BGR
                               // (k_nv12.cu), read by the BGR front end; null when none is needed
    bool fused;                // K1 fused stencil+background kernel drives the front end
    bool wide_fused;           // wide Gaussian: the vertical pass runs the temporal stage too (k_wide_vt)
    bool umma;                 // blur + temporal stage on tcgen05 tensor cores (k_umma.cu), k <= 97
    uint8_t *uband;            // band (Toeplitz) operand of the tcgen05 blur (apron-plane kernel)
    uint8_t *uband_f;          // ... of the kernel that reads the BGR frames directly
    bool umma_direct;          // full-resolution mode with TMA-compatible rows: no gray / apron plane at all
    int umma_ra;               // apron class of the direct kernel (16: k <= 33, 48: k <= 97)
    uint8_t *gpad;             // [S][Tmax][Hp][Wp] gray plane with the BORDER_REFLECT_101 apron materialised
    int fx, fy;                // integer ratios (mode 2)
    int maxc;
    // tables
    int *coef;                 // [k] 8.8 fixed-point Gaussian taps
    uint32_t *wtab;            // tap tables of the tensor-core blur (k_wide.cu): pass 1 (uint2 per lane) then pass 2 (uint4 per lane)
    ResizeTab xtab, ytab;
    int *g4start, *g4n, *g4off;   // x taps regrouped in 4-pixel groups with zero-weight padding (k_resize_gray_g4)
    float4 *g4w;
    int g4max;                    // most tap groups of any destination column
    int2 *uxt, *uyt;              // upscale taps (mode 3): [w] / [h] (source index, a0 | a1 << 16)
    struct RowsPlan *rows;        // plan of the row-per-lane resize kernel (k_resize_rows.cu); null: not applicable
    // planes
    uint8_t *gray;             // [S][Tmax][h][w]
    uint16_t *hor;             // horizontal pass: u16 [S][Tmax][h][w] (naive) or the low/high byte planes of k_wide.cu
    uint8_t *blur;             // [S][Tmax][h][w]  masked blur
    double *bg;                // [S][ntiles][8][32][2]  float64 background, tiled
    uint32_t *maskbits;        // [S][h][wpr]  1 = zero the blur here
    uint32_t *maskflat;        // [S][ntiles*16] same mask, flat bit order (fused kernels)
    uint32_t *tflat;           // [slots][S][Tmax][ntiles*16]  raw threshold, flat bit order (fm_tflat)
    uint32_t *dil;             // [S][Tmax][h][wpr]  dilated threshold, row-padded bit plane
    uint32_t *fill;            // [S][Tmax][h][wpr]  dilated threshold with holes filled
    int *any;                  // [S][Tmax][4] range of set pixels: (max y, max h-1-y, max word column j, max wpr-1-j), -1 = none
    int *rawrange;             // [slots][S][Tmax][2] row range of the RAW threshold (written by the temporal kernels, fm_rawrange)
    int slot;                  // per-call slot of tflat / rawrange the next call uses (alternates with the fused front end)
    int *bg_valid;             // [2][S] the fused front end's own "background exists" flag, indexed by slot
    int *heavy;                // [S][Tmax] frame needs the global-memory labelling kernel
    int *ncomp;                // [S][Tmax]
    int *ncounted;             // [S][Tmax]
    fm_component *comps;       // [S][Tmax][maxc]
    fm_frame_stats *stats;     // [S][Tmax]
    StreamState *state;        // [S]
    int *errflag;              // device error word (capacity overflow), sticky until fm_ctx_check / fm_ctx_reset
    int *nvalid;               // [S] frames of each stream that are real in the current call (ragged batches)
    int *nvalid_host;          // [S] last uploaded copy (uploaded only when it changes)
    CclScratch ccl;
    int *spans;                // mask raster scratch [h][2]
    int last_T;                // frames per stream of the last call
    bool planes_valid;
    // host entry points (fm_process_host, fm_submit_host / fm_wait): two slots, so that the host->device copy of
    // batch i+1 runs on the copy stream while the kernels of batch i run on the compute stream
    uint8_t *stage_dev[2];
    size_t stage_bytes[2];
    fm_frame_stats *stats_pinned[2];   // [S][Tmax] each
    int slot_T[2];             // frames per stream of the batch in flight in the slot (0 = idle)
    int *err_pinned;           // [2] error word of the slot's batch
    cudaStream_t own_stream;   // compute
    cudaStream_t copy_stream;  // host -> device frame copies
    cudaEvent_t ev_copied[2], ev_done[2];
    // device look-back cache (FM_FLAG_DEVICE_CLIPS, k_clips.cu)
    uint8_t *clip_ring;        // [S][cache_frames] raw input frames, slots of clip_slot_bytes; null when cache_frames == 0
    size_t clip_slot_bytes;    // frame_bytes rounded up to 256
    long long *clip_base;      // [S] absolute frame number of the next frame of each stream
    FmClipCopy *clip_list;     // gather list [S * (cache_frames + Tmax)], then store list [S * min(cache_frames, Tmax)]
    int *clip_count;           // [2] entries of the two lists in the current call
    int clip_sms;              // multiprocessors of the device (grid of the copy kernels)
    // detector input planes (FM_FLAG_OBJECT_PLANES, k_objects.cu): W x H -> FM_OBJECT_WIDTH x obj_h
    int obj_h;
    int obj_mode;              // 1 tables, 2 integer ratio (identity: fx = fy = 1), 3 upscale
    int obj_fx, obj_fy;
    ResizeTab obj_xtab, obj_ytab;
    int2 *obj_uxt, *obj_uyt;
    struct RowsPlan *obj_rows;    // BGR-output plan of k_resize_rows; null: not applicable
    int *obj_idx;              // [S][Tmax] plane index of each frame of the last call, -1 = no plane
    uint8_t *obj_bgr;          // FM_FLAG_NV12 on the fused front end: [S][Tmax][H][W][3] the written frames converted
    int obj_src;               // the last hot-path call: 0 none (or failed), 1 a device entry point, 2 a host entry point
    const uint8_t *obj_frames; // ... and its frames, as the caller passed them
    size_t obj_sstride, obj_fstride;
    // timing
    bool timing;               // time the kernel groups: events around them, or stamps with the fused front end (no sync inside fm_process)
    cudaEvent_t *evs;          // [FM_TIMING_RING][4]
    unsigned long long *stamps;   // [FM_TIMING_RING][4] fused front end: %globaltimer of the groups (fm_stamp_*)
    unsigned long long *stamp;    // the stamps of the call being enqueued, null when none are taken
    int ev_pending;
    double t_ms[3];
    int64_t t_calls;
};

extern std::atomic<unsigned long long> g_launches;
// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per device and per function: one mutex-protected cache for
// all kernels, so that host threads driving contexts on different (or the same) devices do not race
int fm_ensure_smem(const void *func, size_t bytes, int device);
void fm_set_error(const char *fmt, ...);

#define FM_CUDA(call)                                                                     \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess) {                                                          \
            fm_set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, \
                         __LINE__);                                                       \
            return FM_ECUDA;                                                              \
        }                                                                                 \
    } while (0)

#define FM_LAUNCH_CHECK()                                                         \
    do {                                                                          \
        g_launches.fetch_add(1, std::memory_order_relaxed);                       \
        cudaError_t e_ = cudaGetLastError();                                      \
        if (e_ != cudaSuccess) {                                                  \
            fm_set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(e_), \
                         __FILE__, __LINE__);                                     \
            return FM_ECUDA;                                                      \
        }                                                                         \
    } while (0)

// The fused front end of call i+1 runs while the contour stage of call i still reads its raw threshold bits and
// ranges, so those two buffers have two slots used by alternate calls (one slot with the other front ends).  Layout of
// `rawrange`: [range slot 0][any][range slot 1], each range slot S*Tmax*2 ints: a range slot and `any` are adjacent in
// both parities, so one fill clears both.
inline uint32_t *fm_tflat(const fm_ctx *c) {
    return c->tflat + (size_t)c->slot * c->S * c->Tmax * c->ntiles * FM_TILE_WORDS;
}
inline int *fm_rawrange(const fm_ctx *c) { return c->rawrange + (size_t)c->slot * 6 * c->S * c->Tmax; }

// Programmatic dependent launch (sm_90+): the kernel may start while the kernel before it in `st` still runs, once
// every CTA of that one has executed griddepcontrol.launch_dependents (or exited).  It must execute
// griddepcontrol.wait before it touches what its predecessor writes; that wait returns when the predecessor has
// completed and its memory is visible.  After any other stream operation it is an ordinary launch.
template <typename... KArgs, typename... Args>
cudaError_t fm_launch_chained(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args &&...args) {
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}
// Group times of a chained call: events recorded between two chained kernels would sit in the chain, so the kernels of a
// group stamp %globaltimer (ns) themselves.  stamp[0] / stamp[2]: NOT of the earliest start of the front end / contour
// stage (atomicMax of ~t is a minimum, and 0 is the cleared value of both kinds), stamp[1] / stamp[3]: latest end.
__device__ __forceinline__ unsigned long long fm_globaltimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void fm_stamp_start(unsigned long long *stamp) {
    if (stamp && threadIdx.x == 0) atomicMax(stamp, ~fm_globaltimer());
}
__device__ __forceinline__ void fm_stamp_end(unsigned long long *stamp) {
    if (stamp && threadIdx.x == 0) atomicMax(stamp + 1, fm_globaltimer());
}
__device__ __forceinline__ void fm_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void fm_wait_predecessor() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// cuTensorMapEncodeTiled of the driver (null when it is not available)
typedef CUresult (*PFN_encodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                    const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_encodeTiled fm_tma_encoder();
// The call's frames as a 4-D u32 tensor map (W*3/4 words, H rows, T frames, S streams) with boxes of box_words x box_rows
// (out-of-range elements are zero-filled).  FM_EINVAL unless the frames, their strides and rows are 16-byte aligned.
int fm_frames_tmap(const fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, int T, int box_words, int box_rows,
                   CUtensorMap *out);

// stage launchers (each enqueues on `st`, returns FM_OK / error)
int fm_launch_frontend(fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, int T,
                       cudaStream_t st);
int fm_launch_temporal(fm_ctx *c, int T, cudaStream_t st);
int fm_launch_fused(fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, int T, cudaStream_t st);
int fm_ccl_configure(fm_ctx *c);
int fm_launch_morph_ccl(fm_ctx *c, int T, cudaStream_t st, fm_frame_stats *stats_out);
int fm_launch_masks(fm_ctx *c, int stream, int n_polys, const int *offs, const int *pts_scaled,
                    int npts, cudaStream_t st);
int fm_launch_bg_export(fm_ctx *c, int stream, double *dst_dev, cudaStream_t st);
int fm_launch_thresh_export(fm_ctx *c, int stream, int t, uint8_t *dst_dev, cudaStream_t st);
int fm_launch_mask_export(fm_ctx *c, int stream, uint8_t *dst_dev, cudaStream_t st);
bool fm_fused_supported(const fm_ctx *c);
size_t fm_wide_plane_bytes(const fm_ctx *c);
int fm_wide_init(fm_ctx *c, const int *taps);
bool fm_wide_fused_supported(const fm_ctx *c);
size_t fm_wide_bg_doubles(const fm_ctx *c);
int fm_launch_bg_export_wide(fm_ctx *c, int stream, double *dst_dev, cudaStream_t st);
int fm_launch_wide_blur(fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, int T, cudaStream_t st);
size_t fm_fused_bg_doubles(const fm_ctx *c);
int fm_launch_bg_export_fused(fm_ctx *c, int stream, double *dst_dev, cudaStream_t st);
int fm_launch_resize_bgr(int device, const uint8_t *src_dev, size_t sstride, size_t fstride, int S, int T, int W, int H,
                         int w, int h, int mode, int fx, int fy, const ResizeTab &xt, const ResizeTab &yt, const int *oidx,
                         uint8_t *dst_dev, size_t ostride, cudaStream_t st);
size_t fm_upscale_smem(int w);
int fm_launch_upscale(int device, const uint8_t *frames, size_t sstride, size_t fstride, int T, int F, int W, int H, int w,
                      int h, const int2 *xt, const int2 *yt, const int *nvalid, uint8_t *gray, uint8_t *bgr_out,
                      const int *oidx, size_t ostride, cudaStream_t st);
int fm_rows_plan(fm_ctx *c, const int *xstart, const int *xidx, const float *xwt, const int *ystart, const int *yidx);
void fm_rows_free(fm_ctx *c);
int fm_rows_plan_describe(int W, int w, int h, const int *xstart, const int *xidx, const float *xwt, const int *ystart,
                          const int *yidx, fm_rows_plan_info *out);
int fm_rows_plan_objects(fm_ctx *c, const int *xstart, const int *xidx, const float *xwt, const int *ystart, const int *yidx);
bool fm_rows_usable(const fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride);
int fm_launch_resize_rows(fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, int T, cudaStream_t st);
int fm_launch_resize_rows_objects(fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, int T, uint8_t *out,
                                  size_t ostride, cudaStream_t st);
int fm_launch_resize_objects(fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, int T, uint8_t *out,
                             size_t ostride, cudaStream_t st);
int fm_launch_object_plan(fm_ctx *c, int T, cudaStream_t st);
bool fm_umma_supported(const fm_ctx *c);
bool fm_umma_preferred(const fm_ctx *c);
int fm_umma_init(fm_ctx *c, const int *taps);
size_t fm_umma_bg_doubles(const fm_ctx *c);
int fm_launch_umma_blur(fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, int T, cudaStream_t st);
int fm_launch_bg_export_umma(fm_ctx *c, int stream, double *dst_dev, cudaStream_t st);
int fm_clips_alloc(fm_ctx *c);
void fm_clips_free(fm_ctx *c);
int fm_launch_clips(fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, int T, uint8_t *out,
                    size_t ostride, cudaStream_t st);
int fm_launch_nv12_bgr(fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, int T, const int *oidx,
                       uint8_t *bgr, cudaStream_t st);
int fm_launch_gray_plane(fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, int T, cudaStream_t st);
int fm_ccl_alloc(CclScratch *s, int frames, int h, int cap);
void fm_ccl_free(CclScratch *s);
int fm_ccl_plane(int device, const uint8_t *plane_host, int w, int h, int max_n, fm_component *out,
                 int *n);
