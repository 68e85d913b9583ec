/*
 * fm_gpu.h -- C ABI of libfmgpu.so, the B200 (sm_100a) implementation of find_motion's
 * per-frame motion-detection hot path.
 *
 * The reference (dmiruke/find_motion) has no FFI of its own: its hot path is the cv2 call chain
 * inside VideoMotion (find_motion/find_motion.py:487-494 blur_frame, :619-635 mask_off_areas,
 * :638-662 find_diff, :246-276 VideoFrame.diff/threshold/find_contours, :665-700 find_movement,
 * :549-589 decide_output) driven by the per-stream loop VideoMotion.find_motion (:852-904) and
 * fanned out one process per stream by run_pool/run_map/run_stream (:1054-1210).  This header
 * is the boundary a maintainer binds instead of those calls (ctypes stub: INTEGRATION.md).
 *
 * Conventions: every entry point returns 0 on success or a negative FM_E* code;
 * fm_last_error() returns a thread-local message.  A context is not thread-safe; distinct
 * contexts are independent.  One context = n_streams streams of identical geometry and tuning
 * (what `partial(run_vid, **tuning)` gives every job, find_motion.py:1323-1331), processed as a
 * batch.  There is no CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef FM_GPU_H
#define FM_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FM_OK 0
#define FM_EINVAL (-1)   /* bad argument */
#define FM_ECUDA (-2)    /* CUDA runtime error (text in fm_last_error) */
#define FM_ENOMEM (-3)
#define FM_ERANGE (-4)   /* configuration outside the supported range */

typedef struct fm_ctx fm_ctx;

/* Tuning options: names, meaning and defaults of VideoMotion.__init__ (find_motion.py:299-307)
 * plus the geometry that _load_video reads from the capture (find_motion.py:413-423). */
typedef struct fm_config {
    int32_t device;          /* CUDA device ordinal */
    int32_t n_streams;       /* streams batched in this context */
    int32_t frame_width;     /* W of the raw BGR (or, with FM_FLAG_NV12, NV12) frames (CAP_PROP_FRAME_WIDTH) */
    int32_t frame_height;    /* H */
    int32_t max_frames;      /* most frames per stream a single fm_process call will carry (T_max) */
    int32_t fps;             /* --fps, default 30 (find_motion.py:1463) */
    int32_t box_size;        /* --box-size, default 100: processing width (find_motion.py:492) */
    int32_t min_box_scale;   /* --min-box-scale, default 50 (find_motion.py:406) */
    int32_t blur_scale;      /* --blur-scale, default 20 (find_motion.py:482-484) */
    int32_t threshold;       /* --threshold, CLI default 12 / ctor default 7 (find_motion.py:257) */
    double avg;              /* --avg, default 0.1 (find_motion.py:659) */
    double min_time;         /* --mintime, default 0.5 s (find_motion.py:335) */
    double cache_time;       /* --cachetime, CLI default 1.0 / ctor default 2.0 (find_motion.py:334) */
    int32_t max_components;  /* per-frame component records kept for fm_get_components (0 -> 256) */
    int32_t flags;           /* FM_FLAG_* */
} fm_config;

#define FM_FLAG_KEEP_PLANES 1   /* keep gray/blur planes of the last call for fm_debug_planes */
#define FM_FLAG_NO_FUSED    2   /* force the generic multi-kernel front end (A/B testing) */
#define FM_FLAG_UMMA_APRON  16  /* tcgen05 blur through the gray plane with a materialised border apron even when the BGR
                                   frames could feed the kernel directly (A/B; it is the path of the resize modes) */
#define FM_FLAG_NO_UMMA     8   /* never take the tcgen05 one-pass Gaussian (k_umma.cu); the mma.sync two-pass kernels instead */
#define FM_FLAG_UMMA        32  /* take the tcgen05 one-pass Gaussian wherever it applies (3 <= k <= 97, w % 32 == 0); without
                                   either flag the library picks the faster path for the geometry (measured: DESIGN.md) */
#define FM_FLAG_NO_ROWS     64  /* default (resize) mode: never take the row-per-lane INTER_AREA kernel (k_resize_rows.cu);
                                   the warp-per-destination-row kernels instead (A/B testing); the same for the planes of
                                   fm_object_planes */
#define FM_FLAG_UPSCALE     128 /* accept box_size > frame_width: cv2's INTER_AREA upscale (a fixed-point linear interpolation,
                                   SURVEY.md A.1), bit-exact, as imutils.resize does it.  Without the flag such a
                                   configuration is refused with FM_ERANGE */
#define FM_FLAG_DEVICE_CLIPS 256 /* keep the look-back cache of raw frames on the device (a ring of cache_frames frames per
                                   stream, n_streams * cache_frames slots of the frame size rounded up to 256 bytes:
                                   H * W * 3, or H * W * 3 / 2 with FM_FLAG_NV12) and accept fm_process_clip.  Every
                                   hot-path call then keeps that ring up to date, so they mix freely with fm_process_clip */
#define FM_FLAG_NV12        512 /* the frames are NV12, as hardware video decoders emit them: (H + H/2) rows of W bytes, the H
                                   luma rows, then H/2 rows of interleaved U, V bytes (U first); W and H even (FM_ERANGE
                                   otherwise).  Every entry point that takes frames reads W*H*3/2 bytes per frame; strides keep
                                   their meaning in bytes.  Results are those of a BGR context on cv2.cvtColor(frame,
                                   COLOR_YUV2BGR_NV12): BT.601 fixed point, chroma of pixel (x, y) from UV row y/2, bytes
                                   2(x/2) and 2(x/2)+1.  With FM_FLAG_DEVICE_CLIPS the ring and the clips hold the NV12 frames.
                                   Memory: the fused full-resolution front end (fm_info.front_end == 0) reads NV12 itself; every
                                   other front end reads the frames converted into a BGR slot the context allocates,
                                   n_streams * max_frames * H * W * 3 bytes (796 MB for 8 x 16 frames of 1080p), so such a
                                   context needs more device memory than a BGR one.  At most 65535 streams and max_frames */
#define FM_FLAG_OBJECT_PLANES 1024 /* accept fm_object_planes: find_objects' detector input of every written frame, on the
                                   device.  fm_ctx_create derives the plane height oh = int(H * (300 / float(W))) (imutils.resize,
                                   FM_OBJECT_WIDTH wide) and builds the INTER_AREA tables of W x H -> 300 x oh once; oh < 1 is
                                   refused with FM_ERANGE before any device query.  Memory: [S][max_frames] ints of plane
                                   indices, and with FM_FLAG_NV12 on the fused front end (fm_info.front_end == 0) a BGR slot
                                   of n_streams * max_frames * H * W * 3 bytes like the staged one.  The hot-path entry
                                   points launch nothing more and return the same results with the flag */
#define FM_OBJECT_WIDTH 300     /* width of the detector input plane (find_motion.py:703-706 hard-codes it) */

/* Derived parameters, exactly as the reference computes them (SURVEY.md A.0). */
typedef struct fm_info {
    int32_t proc_width;            /* w = box_size */
    int32_t proc_height;           /* h = int(H * (box_size / float(W)))  (imutils.resize) */
    int32_t gaussian;              /* odd(int(box_size / blur_scale)) */
    int32_t min_area;              /* int((box_size / min_box_scale) ** 2) */
    int32_t max_area;              /* int(W * H / 2 * scale) */
    int32_t cache_frames;          /* int(cache_time * fps) */
    int32_t min_movement_frames;   /* int(min_time * fps) */
    int32_t words_per_row;         /* 32-bit words per row of the bit planes */
    double scale;                  /* box_size / frame_width */
    int32_t front_end;             /* 0 = fused full-res stencil, 1 = generic blur, 2 = resize front end */
    int32_t max_components;        /* component records kept per frame (fm_config.max_components, 0 -> 256) */
} fm_info;

/* Per-frame result: everything find_movement + decide_output decide (find_motion.py:665-700,
 * 549-589), in frame order.  The host adapter replays `wrote` / `n_flush` on the raw frames. */
typedef struct fm_frame_stats {
    int32_t n_contours;         /* len(frame.contours): external contours of the dilated mask */
    int32_t n_counted;          /* contours not skipped by `max_area < area < min_area` (:684) */
    int32_t movement;           /* self.movement after find_movement */
    int32_t movement_counter;   /* self.movement_counter after find_movement (per CONTOUR, :694) */
    int32_t movement_decay;     /* self.movement_decay after decide_output */
    int32_t cache_len;          /* len(self.frame_cache) after decide_output */
    int32_t wrote;              /* 1 if output_frame() ran for this frame (:583) */
    int32_t n_flush;            /* cached raw frames written before it (:561-570) */
} fm_frame_stats;

/* One external contour: 2*cv2.contourArea (an integer) and cv2.boundingRect (find_motion.py:679, 792). */
typedef struct fm_component {
    int32_t area_x2;
    int32_t x, y, w, h;
} fm_component;

/* Plan of the default-mode resize kernel (k_resize_rows.cu) for one geometry: fm_debug_rows_plan. */
typedef struct fm_rows_plan_info {
    int32_t usable;        /* 0: the warp-per-row kernels take this geometry (rows not TMA-compatible, < 4 taps, band too tall) */
    int32_t band_rows;     /* destination rows per CTA */
    int32_t box_rows;      /* source rows of a TMA box (<= 160 = the CTA's row threads) */
    int32_t chunk_cols;    /* destination columns per TMA box */
    int32_t seg_cols;      /* destination columns per CTA */
    int32_t box_bytes;     /* bytes per box row: an odd multiple of 16, <= 1024 */
    int32_t smem_bytes;    /* dynamic shared memory per CTA */
    int32_t bands, segs;   /* grid.y, grid.x */
    int32_t max_groups;    /* most 4-pixel tap groups of a destination column */
} fm_rows_plan_info;

const char *fm_last_error(void);
int fm_version(void);

/* Replaces VideoMotion.__init__ + _calc_min_area + _make_gaussian + _load_video
 * (find_motion.py:299-380, 402-424, 478-484) for n_streams streams.  box_size > frame_width (a processing plane larger
 * than the frame, which imutils.resize produces with cv2's INTER_AREA upscale) needs FM_FLAG_UPSCALE; without it
 * fm_ctx_create returns FM_ERANGE.  So does an odd frame width or height with FM_FLAG_NV12.  Both checks come before
 * any device query. */
int fm_ctx_create(const fm_config *cfg, fm_ctx **out);
int fm_ctx_destroy(fm_ctx *ctx);
int fm_ctx_info(const fm_ctx *ctx, fm_info *info);

/* Replaces mask_off_areas' per-frame drawing (find_motion.py:619-635): the polygons are
 * rasterised once on the device with cv2.rectangle(FILLED) / cv2.fillConvexPoly semantics.
 * xy holds the user's UNSCALED integer coordinates (x0,y0,x1,y1,...); poly_offsets[i] ..
 * poly_offsets[i+1] index the points of polygon i (2 points = rectangle).  stream < 0 = all. */
int fm_ctx_set_masks(fm_ctx *ctx, int stream, int n_polys, const int32_t *poly_offsets,
                     const int32_t *xy);

/* ref_frame = None, counters = 0, frame cache emptied (find_motion.py:362-371, 414-415). */
int fm_ctx_reset(fm_ctx *ctx, int stream);

/* The hot path: for every stream s < n_streams and t < n_frames (in order), run
 * blur_frame -> mask_off_areas -> find_diff -> find_movement -> decide_output on the BGR frame
 *   frames + s * stream_stride + t * frame_stride          (H*W*3 bytes, HWC, uint8; FM_FLAG_NV12: H*W*3/2 bytes NV12)
 * `frames` is a DEVICE pointer; work is enqueued on `cuda_stream` (a cudaStream_t, 0 = default)
 * and the call returns without synchronising.  stats_dev, if not NULL, is a device buffer of
 * n_streams * n_frames fm_frame_stats ([stream][frame]) filled by the call. */
int fm_process(fm_ctx *ctx, const uint8_t *frames, size_t stream_stride, size_t frame_stride,
               int n_frames, void *cuda_stream, fm_frame_stats *stats_dev);

/* Ragged batch: stream s carries only n_valid[s] <= n_frames real frames in this call (a HOST array of
 * n_streams entries; NULL = all n_frames).  Streams are independent jobs of different lengths
 * (find_motion.py:1071-1075 gives each file / camera its own process): a stream with n_valid[s] == 0 is
 * left untouched (background, counters), the stats of frames t >= n_valid[s] are zero. */
int fm_process_ragged(fm_ctx *ctx, const uint8_t *frames, size_t stream_stride, size_t frame_stride,
                      int n_frames, const int32_t *n_valid, void *cuda_stream, fm_frame_stats *stats_dev);

/* fm_process_ragged that also hands out the frames the reference writes to its *_motion.avi in this call (needs
 * FM_FLAG_DEVICE_CLIPS).  For stream s, with n_out[s] = sum of wrote + n_flush over its valid frames, it writes
 * n_out[s] raw BGR frames densely to the DEVICE buffer
 *   out_dev + s * out_stream_stride + i * H*W*3          (i < n_out[s]; FM_FLAG_NV12: NV12 frames, i * H*W*3/2)
 * in the reference's order: for each frame in order, the n_flush cached frames it flushes (oldest first, taken from the
 * device ring or from this call's input), then the frame itself if `wrote` (find_motion.py:561-570, 583).  n_out
 * follows from the stats.  out_capacity is the room per stream in frames and must be at least cache_frames + n_frames,
 * the most one call can write (the whole cache plus every frame); otherwise, or without the flag, FM_EINVAL.
 * Asynchronous on `cuda_stream` like fm_process. */
int fm_process_clip(fm_ctx *ctx, const uint8_t *frames, size_t stream_stride, size_t frame_stride,
                    int n_frames, const int32_t *n_valid, void *cuda_stream, fm_frame_stats *stats_dev,
                    uint8_t *out_dev, size_t out_stream_stride, int out_capacity);

/* find_objects' input planes (find_motion.py:572, 703-706) of the last hot-path call made through fm_process,
 * fm_process_ragged or fm_process_clip (needs FM_FLAG_OBJECT_PLANES).  The context remembers that call's frames, strides
 * and n_frames.  For stream s, with n_obj[s] = the number of its valid frames with wrote == 1, it writes n_obj[s] dense
 * BGR planes of oh x 300 x 3 bytes (oh as for FM_FLAG_OBJECT_PLANES), in frame order, to the DEVICE buffer
 *   out_dev + s * out_stream_stride + i * oh*300*3          (i < n_obj[s])
 * each byte-identical to cv2.resize(raw, (300, oh), interpolation=cv2.INTER_AREA) of the written frame (the upscale for
 * W < 300, a copy for W == 300).  The masks do not apply (find_objects reads frame.raw).  NV12 contexts resize
 * cv2.cvtColor(frame, COLOR_YUV2BGR_NV12).  out_capacity is the room per stream in planes and must be at least the last
 * call's n_frames.  Asynchronous on `cuda_stream`: the last call's frames must stay untouched until the planes are
 * written, as for the call itself.  FM_EINVAL without the flag, for a short out_capacity, before the first device-entry
 * call, and after fm_process_host / fm_submit_host (their frames live in the context's staging buffers). */
int fm_object_planes(fm_ctx *ctx, void *cuda_stream, uint8_t *out_dev, size_t out_stream_stride, int out_capacity);

/* Same with HOST buffers: copies the frames host->device (pinned memory recommended), runs the
 * path, copies the stats back and synchronises.  This is the call a drop-in adapter makes.  With FM_FLAG_NV12 a frame
 * is H*W*3/2 bytes, half the host->device traffic of BGR. */
int fm_process_host(fm_ctx *ctx, const uint8_t *frames_host, size_t stream_stride,
                    size_t frame_stride, int n_frames, fm_frame_stats *stats_host);

/* Pipelined form of fm_process_host on two slots (0, 1): fm_submit_host enqueues the host->device copy
 * of the batch on the context's copy stream, the hot path and the stats read-back on its compute stream,
 * and returns at once; fm_wait blocks until that slot's batch is done and hands out its stats
 * ([n_streams][n_frames]).  Submitting batch i+1 to the other slot before waiting for batch i overlaps its
 * copy with the kernels of batch i and with the host's replay of decide_output on batch i-1.  Batches run
 * in submission order.  frames_host must stay untouched until fm_wait(slot) returns.  n_valid as in
 * fm_process_ragged (only the real frames are copied). */
int fm_submit_host(fm_ctx *ctx, int slot, const uint8_t *frames_host, size_t stream_stride,
                   size_t frame_stride, int n_frames, const int32_t *n_valid);
int fm_wait(fm_ctx *ctx, int slot, fm_frame_stats *stats_host);
/* fm_ctx_reset(stream) ordered with the submitted batches instead of synchronising: it takes effect after the
 * batches already submitted and before the next one (a slot changes over to the next file, find_motion.py:1075). */
int fm_submit_reset(fm_ctx *ctx, int stream);

/* Pinned (page-locked) host memory for frame batches, first touched from a thread bound to the CPUs that
 * are local to `device` (when the platform exposes the GPU's NUMA node; *numa_node = -1 otherwise). */
int fm_host_alloc(int device, size_t bytes, void **ptr, int *numa_node);
int fm_host_free(void *ptr);

/* Synchronises and reports (then clears) a sticky device-side error of the calls since the last check:
 * FM_ERANGE if a frame exceeded the run capacity of the contour stage.  fm_process is asynchronous and
 * cannot report it; fm_process_host / fm_wait do. */
int fm_ctx_check(fm_ctx *ctx);

/* Components (contours) of frame t of the LAST fm_process call, sorted by (area_x2, x, y, w, h).
 * Writes min(*n, max_n, fm_info.max_components) records and the true count to *n.  Synchronises. */
int fm_get_components(fm_ctx *ctx, int stream, int t, int max_n, fm_component *out, int *n);

/* Parity-test taps for frame t of the last call (host buffers, any may be NULL):
 * gray, blur (masked) and dilated thresh are proc_height*proc_width uint8; bg is float64 and is
 * the background AFTER the whole call (so compare it at t = n_frames-1).  gray/blur need
 * FM_FLAG_KEEP_PLANES (the fused front ends never materialise them otherwise). */
int fm_debug_planes(fm_ctx *ctx, int stream, int t, uint8_t *gray, uint8_t *blur, uint8_t *thresh,
                    double *bg);

/* Parity-test tap for the mask raster: proc_height*proc_width uint8, 1 where blur is zeroed. */
int fm_debug_mask(fm_ctx *ctx, int stream, uint8_t *mask);

/* Parity-test entry for the contour stage alone: label a host uint8 plane (non-zero = set) of
 * size h*w with findContours(RETR_EXTERNAL)+contourArea+boundingRect semantics. */
int fm_debug_components(int device, const uint8_t *plane, int w, int h, int max_n,
                        fm_component *out, int *n);

/* The detector input plane of find_objects (find_motion.py:703-706): imutils.resize(frame.raw, width=300), i.e.
 * cv2.resize(INTER_AREA) of one BGR frame to (width, int(H * width / W)), bit-exact (SURVEY.md A.1), also for width > W
 * (cv2's fixed-point upscale; no flag needed here).  Host buffers;
 * out_host holds width * out_height * 3 bytes.  The detectors themselves stay on the host. */
int fm_resize_area(int device, const uint8_t *bgr_host, int frame_width, int frame_height, int width,
                   uint8_t *out_host, int *out_height);

/* Host-side test entry (no device needed): derives the processing plane and the INTER_AREA tables of a frame size and
 * box_size exactly as fm_ctx_create does (find_motion.py:487-492), lays out the plan of the row-per-lane resize kernel and
 * re-checks, tap by tap, that every read of every column stays inside its TMA box and meets the weight cv2's table gives
 * it.  FM_OK with info->usable = 0 when the geometry is left to the warp-per-row kernels; FM_ERANGE if a check fails. */
int fm_debug_rows_plan(int frame_width, int frame_height, int box_size, fm_rows_plan_info *info);

/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
uint64_t fm_launch_count(void);

/* Mean device time in ms of the kernels of group `which` (0 = front end, 1 = temporal, 2 =
 * dilate+contours+decisions) over the calls since fm_timing_reset; needs fm_timing_enable(1),
 * which brackets each group with CUDA events on the launching stream. */
int fm_timing_enable(fm_ctx *ctx, int on);
int fm_timing_reset(fm_ctx *ctx);
int fm_timing_get(fm_ctx *ctx, int which, double *ms_total, int64_t *n_calls);

#ifdef __cplusplus
}
#endif
#endif /* FM_GPU_H */
