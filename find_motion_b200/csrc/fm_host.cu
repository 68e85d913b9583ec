// Host side of libfmgpu.so: context life cycle, parameter derivation exactly as the reference
// computes it (find_motion/find_motion.py:334-335, 406, 422-423, 482-484; SURVEY.md A.0), table
// construction (Gaussian taps A.3, INTER_AREA taps A.1) and the C-ABI entry points of
// include/fm_gpu.h.
#include <ctype.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <utility>
#include <vector>

#include <sched.h>
#include <unistd.h>

#include "fm_common.cuh"

std::atomic<unsigned long long> g_launches{0};
static thread_local char g_err[512] = "";

int fm_ensure_smem(const void *func, size_t bytes, int device) {
    static std::mutex mu;
    static std::map<std::pair<const void *, int>, size_t> done;
    std::lock_guard<std::mutex> lk(mu);
    size_t &have = done[std::make_pair(func, device)];
    if (bytes <= have) return FM_OK;
    FM_CUDA(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    have = bytes;
    return FM_OK;
}

void fm_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

PFN_encodeTiled fm_tma_encoder() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void *sym = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (PFN_encodeTiled)sym;
    }
    return fn;
}

int fm_frames_tmap(const fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, size_t pitch, int T, int box_words,
                   int box_rows, CUtensorMap *out) {
    const size_t row = (size_t)c->W * c->px_bytes, dense = pitch * c->H;
    if ((((uintptr_t)frames) | sstride | fstride | pitch | row) & 15) {
        fm_set_error("the TMA front ends need 16-byte aligned frames, strides and rows (row pitch %zu)", pitch);
        return FM_EINVAL;
    }
    PFN_encodeTiled enc = fm_tma_encoder();
    if (!enc) { fm_set_error("cuTensorMapEncodeTiled not available"); return FM_ECUDA; }
    // the stride of a dimension of extent 1 is never applied: the dense size stands in for it (the caller's may be 0)
    cuuint64_t dims[4] = {(cuuint64_t)row / 4, (cuuint64_t)c->H, (cuuint64_t)T, (cuuint64_t)c->S};
    cuuint64_t strides[3] = {(cuuint64_t)pitch, (cuuint64_t)(T > 1 ? fstride : dense),
                             (cuuint64_t)(c->S > 1 ? sstride : (T > 1 ? fstride * T : dense))};
    cuuint32_t box[4] = {(cuuint32_t)box_words, (cuuint32_t)box_rows, 1, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_UINT32, 4, (void *)frames, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { fm_set_error("cuTensorMapEncodeTiled (frames) failed (%d)", (int)r); return FM_ECUDA; }
    return FM_OK;
}

extern "C" const char *fm_last_error(void) { return g_err; }
extern "C" int fm_version(void) { return 100; }
extern "C" uint64_t fm_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

// --------------------------------------------------------------------------------------------
// tables
// --------------------------------------------------------------------------------------------
static std::vector<int> gauss_coeffs(int k) {
    // cv2.getGaussianKernel(k, sigma<=0) quantised to 8 fractional bits with error diffusion
    std::vector<double> kern(k);
    static const double small[4][7] = {{1.0},
                                       {0.25, 0.5, 0.25},
                                       {0.0625, 0.25, 0.375, 0.25, 0.0625},
                                       {0.03125, 0.109375, 0.21875, 0.28125, 0.21875, 0.109375, 0.03125}};
    if (k <= 7) {
        for (int i = 0; i < k; i++) kern[i] = small[k >> 1][i];
    } else {
        double sigma = 0.3 * ((k - 1) * 0.5 - 1) + 0.8;
        double scale2x = -0.5 / (sigma * sigma);
        double sum = 0.0;
        for (int i = 0; i < k; i++) {
            double x = i - (k - 1) * 0.5;
            kern[i] = exp(scale2x * x * x);
            sum += kern[i];
        }
        double inv = 1.0 / sum;
        for (int i = 0; i < k; i++) kern[i] *= inv;
    }
    std::vector<int> c(k, 0);
    double err = 0.0;
    int tot = 0;
    for (int i = 0; i < k / 2; i++) {
        double adj = kern[i] * 256.0 + err;
        int v = (int)nearbyint(adj);          // round half to even (default rounding mode)
        err = adj - v;
        c[i] = c[k - 1 - i] = v;
        tot += 2 * v;
    }
    c[k / 2] = 256 - tot;
    return c;
}

struct HostTab {
    std::vector<int> start, idx;
    std::vector<float> wt;
    int max_taps = 0;
};

static HostTab area_tab(int src, int dst) {
    HostTab t;
    double scale = 1.0 / ((double)dst / (double)src);
    t.start.push_back(0);
    for (int d = 0; d < dst; d++) {
        double f1 = d * scale, f2 = f1 + scale;
        double cell = std::min(scale, (double)src - f1);
        int s1 = (int)ceil(f1), s2 = (int)floor(f2);
        s2 = std::min(s2, src - 1);
        s1 = std::min(s1, s2);
        if (s1 - f1 > 1e-3) {
            t.idx.push_back(s1 - 1);
            t.wt.push_back((float)((s1 - f1) / cell));
        }
        for (int s = s1; s < s2; s++) {
            t.idx.push_back(s);
            t.wt.push_back((float)(1.0 / cell));
        }
        if (f2 - s2 > 1e-3) {
            t.idx.push_back(s2);
            t.wt.push_back((float)(std::min(std::min(f2 - s2, 1.0), cell) / cell));
        }
        t.max_taps = std::max(t.max_taps, (int)t.idx.size() - t.start.back());
        t.start.push_back((int)t.idx.size());
    }
    return t;
}

// One axis of INTER_AREA with dst >= src: cv2 takes its linear interpolation with area-style offsets there
// (cv::resize, `area_mode`), fixed point with INTER_RESIZE_COEF_SCALE = 2048.  Per destination index: the first source
// index and the weights a0 | a1 << 16 of it and of the next one (clamped to the border).  float where cv2 uses float.
static std::vector<int2> upscale_tab(int src, int dst) {
    std::vector<int2> t(dst);
    const double inv = (double)dst / (double)src, scale = 1.0 / inv;
    for (int d = 0; d < dst; d++) {
        int sx = (int)floor(d * scale);
        float fx = (float)((d + 1) - (sx + 1) * inv);
        fx = fx <= 0 ? 0.f : fx - (float)(int)floorf(fx);
        if (sx >= src - 1) { fx = 0.f; sx = src - 1; }
        const int a0 = (int)lrintf((1.f - fx) * 2048.f), a1 = (int)lrintf(fx * 2048.f);   // saturate_cast<short>
        t[d] = make_int2(sx, a0 | (a1 << 16));
    }
    return t;
}

template <typename T>
static int upload(T **dst, const std::vector<T> &v) {
    FM_CUDA(cudaMalloc(dst, std::max<size_t>(v.size(), 1) * sizeof(T)));
    if (!v.empty()) FM_CUDA(cudaMemcpy(*dst, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    return FM_OK;
}

static int upload_tab(ResizeTab *d, const HostTab &h) {
    int rc;
    if ((rc = upload(&d->start, h.start))) return rc;
    if ((rc = upload(&d->idx, h.idx))) return rc;
    if ((rc = upload(&d->wt, h.wt))) return rc;
    d->max_taps = h.max_taps;
    return FM_OK;
}

namespace {
struct DevBuf {           // scratch that is released on every return path
    void *p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
};
}

// --------------------------------------------------------------------------------------------
// context
// --------------------------------------------------------------------------------------------
extern "C" int fm_ctx_destroy(fm_ctx *c) {
    if (!c) return FM_OK;
    cudaSetDevice(c->cfg.device);
    cudaDeviceSynchronize();
    cudaFree(c->coef); cudaFree(c->wtab); cudaFree(c->uband); cudaFree(c->uband_f); cudaFree(c->gpad);
    cudaFree(c->g4start); cudaFree(c->g4n); cudaFree(c->g4off); cudaFree(c->g4w);
    cudaFree(c->uxt); cudaFree(c->uyt); cudaFree(c->nv12_bgr);
    cudaFree(c->obj_xtab.start); cudaFree(c->obj_xtab.idx); cudaFree(c->obj_xtab.wt);
    cudaFree(c->obj_ytab.start); cudaFree(c->obj_ytab.idx); cudaFree(c->obj_ytab.wt);
    cudaFree(c->obj_uxt); cudaFree(c->obj_uyt); cudaFree(c->obj_idx); cudaFree(c->obj_bgr);
    fm_rows_free(c);
    fm_clips_free(c);
    cudaFree(c->xtab.start); cudaFree(c->xtab.idx); cudaFree(c->xtab.wt);
    cudaFree(c->ytab.start); cudaFree(c->ytab.idx); cudaFree(c->ytab.wt);
    cudaFree(c->gray); cudaFree(c->hor); cudaFree(c->blur); cudaFree(c->bg);
    cudaFree(c->maskbits); cudaFree(c->maskflat); cudaFree(c->tflat); cudaFree(c->dil); cudaFree(c->fill);
    cudaFree(c->heavy); cudaFree(c->rawrange); cudaFree(c->ncomp); cudaFree(c->comps); cudaFree(c->stats);      // any / ncounted live inside rawrange / ncomp
    cudaFree(c->state); cudaFree(c->bg_valid); cudaFree(c->errflag); cudaFree(c->nvalid);
    free(c->nvalid_host);
    fm_ccl_free(&c->ccl);
    for (int i = 0; i < 2; i++) {
        cudaFree(c->stage_dev[i]);
        if (c->stats_pinned[i]) cudaFreeHost(c->stats_pinned[i]);
        if (c->ev_copied[i]) cudaEventDestroy(c->ev_copied[i]);
        if (c->ev_done[i]) cudaEventDestroy(c->ev_done[i]);
    }
    if (c->err_pinned) cudaFreeHost(c->err_pinned);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->evs) {
        for (int i = 0; i < 4 * FM_TIMING_RING; i++) cudaEventDestroy(c->evs[i]);
        delete[] c->evs;
    }
    cudaFree(c->stamps);
    delete c;
    return FM_OK;
}

// The pixel format the flags select, decided here once for fm_ctx_create and fm_debug_rows_plan_format: bytes per pixel
// of the frames the BGR / gray front ends read (NV12's staged slot is BGR) and whether R comes first.  false (with the
// error set) for two formats at once.
static bool fm_pixel_format(int32_t flags, int *px_bytes, bool *rgb) {
    if ((flags & FM_FLAG_GRAY) && (flags & FM_FLAG_NV12)) {
        fm_set_error("FM_FLAG_GRAY and FM_FLAG_NV12 are two frame formats: set one of them");
        return false;
    }
    for (int32_t f : {FM_FLAG_RGB, FM_FLAG_ALPHA}) {
        if ((flags & f) && (flags & (FM_FLAG_NV12 | FM_FLAG_GRAY))) {
            fm_set_error("%s and %s are two frame formats: set one of them", f == FM_FLAG_RGB ? "FM_FLAG_RGB" : "FM_FLAG_ALPHA",
                         (flags & FM_FLAG_NV12) ? "FM_FLAG_NV12" : "FM_FLAG_GRAY");
            return false;
        }
    }
    *px_bytes = (flags & FM_FLAG_GRAY) ? 1 : (flags & FM_FLAG_ALPHA) ? 4 : 3;
    *rgb = (flags & FM_FLAG_RGB) != 0;
    return true;
}

extern "C" int fm_ctx_create(const fm_config *cfg, fm_ctx **out) {
    if (!cfg || !out) { fm_set_error("null argument"); return FM_EINVAL; }
    *out = nullptr;
    if (cfg->n_streams < 1 || cfg->frame_width < 1 || cfg->frame_height < 1 || cfg->max_frames < 1 ||
        cfg->box_size < 1 || cfg->blur_scale < 1 || cfg->min_box_scale < 1 || cfg->fps < 0) {
        fm_set_error("invalid configuration (streams/geometry/max_frames/box_size/blur_scale/min_box_scale)");
        return FM_EINVAL;
    }
    int px_bytes;
    bool rgb;
    if (!fm_pixel_format(cfg->flags, &px_bytes, &rgb)) return FM_EINVAL;
    if (cfg->box_size > cfg->frame_width && !(cfg->flags & FM_FLAG_UPSCALE)) {
        // INTER_AREA with a destination wider than the source is cv2's fixed-point linear upscale (SURVEY.md A.1):
        // opt-in with FM_FLAG_UPSCALE, so that binders of the earlier ABI keep their range check
        fm_set_error("box_size %d > frame width %d: upscaling resize needs FM_FLAG_UPSCALE", cfg->box_size,
                     cfg->frame_width);
        return FM_ERANGE;
    }
    if ((cfg->flags & FM_FLAG_NV12) && ((cfg->frame_width | cfg->frame_height) & 1)) {
        // the chroma plane has one U, V pair per 2 x 2 block (cv2's COLOR_YUV2BGR_NV12 refuses odd sizes as well)
        fm_set_error("NV12 frames need an even width and height (%d x %d)", cfg->frame_width, cfg->frame_height);
        return FM_ERANGE;
    }
    if ((cfg->flags & FM_FLAG_NV12) && (cfg->n_streams > 65535 || cfg->max_frames > 65535)) {
        // the staging kernel's grid: one z index per stream, one y index per frame
        fm_set_error("NV12 contexts take at most 65535 streams and 65535 frames per call");
        return FM_ERANGE;
    }
    // find_objects' input plane: imutils.resize(frame.raw, width=300) (find_motion.py:703-706)
    const int obj_h = (int)((double)cfg->frame_height * (FM_OBJECT_WIDTH / (double)cfg->frame_width));
    if ((cfg->flags & FM_FLAG_OBJECT_PLANES) && obj_h < 1) {
        fm_set_error("detector input plane of %d x %d frames is %d x 0", cfg->frame_width, cfg->frame_height, FM_OBJECT_WIDTH);
        return FM_ERANGE;
    }
    int ndev = 0;
    FM_CUDA(cudaGetDeviceCount(&ndev));
    if (cfg->device < 0 || cfg->device >= ndev) {
        fm_set_error("CUDA device %d not present (%d devices)", cfg->device, ndev);
        return FM_ECUDA;
    }
    FM_CUDA(cudaSetDevice(cfg->device));

    fm_ctx *c = new fm_ctx();
    memset(c, 0, sizeof(*c));
    c->cfg = *cfg;
    c->S = cfg->n_streams; c->Tmax = cfg->max_frames;
    c->W = cfg->frame_width; c->H = cfg->frame_height;
    c->px_bytes = px_bytes; c->rgb = rgb;
    c->row_bytes = (cfg->flags & FM_FLAG_NV12) ? (size_t)c->W : (size_t)c->W * px_bytes;
    c->frame_bytes = (cfg->flags & FM_FLAG_NV12) ? (size_t)c->W * c->H * 3 / 2 : c->row_bytes * c->H;
    // derived parameters, mirroring the Python expressions (true division on floats, int() truncation)
    const double W = c->W, H = c->H, box = cfg->box_size;
    c->w = cfg->box_size;
    c->h = (int)(H * (box / W));                                   // imutils.resize
    int g = (int)(box / (double)cfg->blur_scale);                  // find_motion.py:482
    c->k = (g % 2 == 0) ? g + 1 : g;                               // :483
    fm_info &inf = c->info;
    inf.proc_width = c->w; inf.proc_height = c->h; inf.gaussian = c->k;
    inf.min_area = (int)pow(box / (double)cfg->min_box_scale, 2.0);    // :406
    inf.scale = box / W;                                           // :422
    inf.max_area = (int)((W * H) / 2.0 * inf.scale);               // :423
    inf.cache_frames = (int)(cfg->cache_time * cfg->fps);          // :334
    inf.min_movement_frames = (int)(cfg->min_time * cfg->fps);     // :335
    if (c->h < 1) { fm_set_error("processing height is zero"); delete c; return FM_ERANGE; }
    if (c->k > FM_MAX_K) { fm_set_error("gaussian size %d too large", c->k); delete c; return FM_ERANGE; }
    if (c->w > 65535 || c->h > 65535) { fm_set_error("processing plane too large"); delete c; return FM_ERANGE; }
    c->wpr = (c->w + 31) / 32;
    inf.words_per_row = c->wpr;
    c->N = c->w * c->h;
    c->ntiles = (c->N + FM_TILE_PX - 1) / FM_TILE_PX;
    c->maxc = cfg->max_components > 0 ? cfg->max_components : 256;
    inf.max_components = c->maxc;

    int rc = FM_OK;
    auto fail = [&](int code) { fm_ctx_destroy(c); return code; };
#define FM_TRY(call)                                                                       \
    do {                                                                                   \
        cudaError_t e_ = (call);                                                           \
        if (e_ != cudaSuccess) {                                                           \
            fm_set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            return fail(FM_ECUDA);                                                         \
        }                                                                                  \
    } while (0)

    // resize mode (cv2::resize INTER_AREA dispatch)
    if (c->w == c->W && c->h == c->H) {
        c->resize_mode = 0;
    } else if (c->w > c->W || c->h > c->H) {
        // imutils.resize keeps the aspect ratio, so h >= H whenever w > W: both axes go up (or stay)
        if (!(cfg->flags & FM_FLAG_UPSCALE) || c->w < c->W || c->h < c->H) {
            fm_set_error("upscaling resize needs FM_FLAG_UPSCALE");
            return fail(FM_ERANGE);
        }
        c->resize_mode = 3;
        if (fm_upscale_smem(c->w, c->px_bytes) > 200 * 1024) { fm_set_error("processing width %d too large to upscale", c->w); return fail(FM_ERANGE); }
        if ((rc = upload(&c->uxt, upscale_tab(c->W, c->w)))) return fail(rc);
        if ((rc = upload(&c->uyt, upscale_tab(c->H, c->h)))) return fail(rc);
    } else {
        double sx = 1.0 / ((double)c->w / W), sy = 1.0 / ((double)c->h / H);
        int isx = (int)nearbyint(sx), isy = (int)nearbyint(sy);
        bool fast = fabs(sx - isx) < 2.220446049250313e-16 && fabs(sy - isy) < 2.220446049250313e-16;
        if (fast) {
            c->resize_mode = 2; c->fx = isx; c->fy = isy;
        } else {
            c->resize_mode = 1;
            HostTab xt = area_tab(c->W, c->w);
            if ((rc = upload_tab(&c->xtab, xt))) return fail(rc);
            {   // the same x taps in groups of 4 consecutive source pixels, zero-weight padded
                std::vector<int> g4s(c->w), g4n(c->w), g4o(c->w);
                std::vector<float4> g4w;
                for (int dx = 0; dx < c->w; dx++) {
                    int a = xt.start[dx], b = xt.start[dx + 1];
                    int first = xt.idx[a], last = xt.idx[b - 1];
                    int gs = first & ~3, ge = (last | 3) + 1;
                    g4s[dx] = gs; g4n[dx] = (ge - gs) / 4; g4o[dx] = (int)g4w.size();
                    for (int g = gs; g < ge; g += 4) {
                        float wv[4];
                        for (int i = 0; i < 4; i++) {
                            int x = g + i;
                            wv[i] = (x >= first && x <= last) ? xt.wt[a + (x - first)] : 0.0f;
                        }
                        g4w.push_back(make_float4(wv[0], wv[1], wv[2], wv[3]));
                    }
                }
                if ((rc = upload(&c->g4start, g4s))) return fail(rc);
                if ((rc = upload(&c->g4n, g4n))) return fail(rc);
                c->g4max = 0;
                for (int v : g4n) c->g4max = std::max(c->g4max, v);
                if ((rc = upload(&c->g4off, g4o))) return fail(rc);
                if ((rc = upload(&c->g4w, g4w))) return fail(rc);
            }
            HostTab yt = area_tab(c->H, c->h);
            if ((rc = upload_tab(&c->ytab, yt))) return fail(rc);
            if ((rc = fm_rows_plan(c, xt.start.data(), xt.idx.data(), xt.wt.data(), yt.start.data(), yt.idx.data())))
                return fail(rc);
        }
    }
    c->fused = fm_fused_supported(c) && !(cfg->flags & FM_FLAG_NO_FUSED);
    c->umma = !c->fused && fm_umma_supported(c) && !(cfg->flags & FM_FLAG_NO_UMMA) &&
              ((cfg->flags & FM_FLAG_UMMA) || fm_umma_preferred(c));
    c->wide_fused = !c->fused && !c->umma && fm_wide_fused_supported(c);
    inf.front_end = c->fused ? 0 : (c->resize_mode == 0 ? 1 : 2);
    {
        std::vector<int> taps = gauss_coeffs(c->k);
        if ((rc = upload(&c->coef, taps))) return fail(rc);
        // the shared-memory needs of the wide blur are checked here, not at the first launch
        if (c->umma && (rc = fm_umma_init(c, taps.data()))) return fail(rc);
        if (!c->fused && !c->umma && (rc = fm_wide_init(c, taps.data()))) return fail(rc);
    }

    const size_t F = (size_t)c->S * c->Tmax;
    const size_t flatw = (size_t)c->ntiles * FM_TILE_WORDS;
#define ALLOC(ptr, bytes)                                                                 \
    do {                                                                                  \
        cudaError_t e_ = cudaMalloc((void **)&(ptr), (bytes));                            \
        if (e_ != cudaSuccess) {                                                          \
            fm_set_error("cudaMalloc(%zu bytes) for %s failed: %s", (size_t)(bytes), #ptr, \
                         cudaGetErrorString(e_));                                         \
            return fail(FM_ENOMEM);                                                       \
        }                                                                                 \
    } while (0)
    // the fused front ends never materialise gray / blur planes (except as parity taps)
    const bool keep = (cfg->flags & FM_FLAG_KEEP_PLANES) != 0;
    // gray frames at full resolution are the gray plane themselves
    const bool need_gray = keep || (!c->fused && !(c->px_bytes == 1 && c->resize_mode == 0));
    const bool need_blur = keep || !c->fused;
    ALLOC(c->gray, need_gray ? F * c->N : 16);
    ALLOC(c->hor, (c->fused || c->umma) ? 16 : 2 * fm_wide_plane_bytes(c));
    ALLOC(c->blur, need_blur ? F * c->N + 64 : 64);
    const size_t bg_doubles = std::max((size_t)c->S * c->ntiles * FM_TILE_PX,
                                       c->fused ? fm_fused_bg_doubles(c)
                                                : (c->umma ? fm_umma_bg_doubles(c) : (c->wide_fused ? fm_wide_bg_doubles(c) : (size_t)0)));
    ALLOC(c->bg, bg_doubles * sizeof(double));
    ALLOC(c->maskbits, (size_t)c->S * c->h * c->wpr * 4);
    ALLOC(c->maskflat, (size_t)c->S * flatw * 4);
    // two slots of the raw threshold bits and ranges with the fused front end, which overlaps the previous call's
    // contour stage (fm_tflat, fm_rawrange)
    const size_t slots = c->fused ? 2 : 1;
    ALLOC(c->tflat, (slots * F * flatw + FM_TILE_WORDS) * 4);
    ALLOC(c->dil, F * c->h * c->wpr * 4);
    ALLOC(c->fill, F * c->h * c->wpr * 4);
    // ranges of the raw ([slots][F][2]) and of the dilated mask ([F][4]) share one allocation, and so do the two
    // counters: one clear each per call
    ALLOC(c->rawrange, F * (4 + 2 * slots) * sizeof(int));
    c->any = c->rawrange + 2 * F;
    ALLOC(c->ncomp, (F * 2 + 4) * sizeof(int));        // + the frame counter of the decision tail
    c->ncounted = c->ncomp + F;
    ALLOC(c->heavy, F * sizeof(int));
    ALLOC(c->comps, F * c->maxc * sizeof(fm_component));
    ALLOC(c->stats, F * sizeof(fm_frame_stats));
    ALLOC(c->state, (size_t)c->S * sizeof(StreamState));
    ALLOC(c->bg_valid, 2 * (size_t)c->S * sizeof(int));
    ALLOC(c->errflag, sizeof(int));
    ALLOC(c->nvalid, (size_t)c->S * sizeof(int));
    c->nvalid_host = (int *)malloc((size_t)c->S * sizeof(int));
    if (!c->nvalid_host) { fm_set_error("out of host memory"); return fail(FM_ENOMEM); }
    for (int s = 0; s < c->S; s++) c->nvalid_host[s] = c->Tmax;
    FM_TRY(cudaMemcpy(c->nvalid, c->nvalid_host, (size_t)c->S * sizeof(int), cudaMemcpyHostToDevice));
    FM_TRY(cudaMemset(c->maskbits, 0, (size_t)c->S * c->h * c->wpr * 4));
    FM_TRY(cudaMemset(c->maskflat, 0, (size_t)c->S * flatw * 4));
    FM_TRY(cudaMemset(c->tflat, 0, (slots * F * flatw + FM_TILE_WORDS) * 4));
    FM_TRY(cudaMemset(c->bg, 0, bg_doubles * sizeof(double)));
    FM_TRY(cudaMemset(c->state, 0, (size_t)c->S * sizeof(StreamState)));
    FM_TRY(cudaMemset(c->bg_valid, 0, 2 * (size_t)c->S * sizeof(int)));
    FM_TRY(cudaMemset(c->rawrange, 0xFF, F * (4 + 2 * slots) * sizeof(int)));      // the fused front end clears them
    FM_TRY(cudaMemset(c->ncomp, 0, (F * 2 + 4) * sizeof(int)));                    //   for the call after it
    FM_TRY(cudaMemset(c->errflag, 0, sizeof(int)));
    FM_TRY(cudaMemset(c->heavy, 0, F * sizeof(int)));
    // contour scratch: a dilated plane has runs >= 3 px separated by >= 1 px, so a row holds at
    // most w/4 + 2 runs of either polarity; sub-batch sized to <= 8 GB (only the slots of existing runs are ever touched)
    int cap = c->w / 4 + 3;
    size_t per_frame = (size_t)c->h * cap * 28 + (size_t)c->h * 4 + 4;
    size_t budget = (size_t)8 << 30;
    int nb = (int)std::min<size_t>(F, std::max<size_t>(1, budget / per_frame));
    if ((rc = fm_ccl_alloc(&c->ccl, nb, c->h, cap))) return fail(rc);
    if ((rc = fm_ccl_configure(c))) return fail(rc);
    if ((cfg->flags & FM_FLAG_DEVICE_CLIPS) && (rc = fm_clips_alloc(c))) return fail(rc);
    // NV12: the fused front end reads the frames directly; every other front end reads them converted into a BGR slot
    // (k_nv12.cu).  FM_NV12_STAGED builds (A/B of the two paths, tools/bench_nv12.py --ab-staged) stage them always.
#ifdef FM_NV12_STAGED
    const bool nv12_staged = true;
#else
    const bool nv12_staged = !c->fused;
#endif
    if ((cfg->flags & FM_FLAG_NV12) && nv12_staged) ALLOC(c->nv12_bgr, F * c->W * c->H * 3);
    if (cfg->flags & FM_FLAG_OBJECT_PLANES) {
        // W x H -> 300 x obj_h, dispatched as cv::resize(INTER_AREA) does it (and as fm_resize_area does)
        const int ow = FM_OBJECT_WIDTH;
        c->obj_h = obj_h;
        if (ow < c->W) {
            const double sx = 1.0 / ((double)ow / W), sy = 1.0 / ((double)obj_h / H);
            const int isx = (int)nearbyint(sx), isy = (int)nearbyint(sy);
            if (fabs(sx - isx) < 2.220446049250313e-16 && fabs(sy - isy) < 2.220446049250313e-16) {
                c->obj_mode = 2; c->obj_fx = isx; c->obj_fy = isy;
            } else {
                c->obj_mode = 1;
                const HostTab xt = area_tab(c->W, ow), yt = area_tab(c->H, obj_h);
                if ((rc = upload_tab(&c->obj_xtab, xt)) || (rc = upload_tab(&c->obj_ytab, yt))) return fail(rc);
                if ((rc = fm_rows_plan_objects(c, xt.start.data(), xt.idx.data(), xt.wt.data(), yt.start.data(), yt.idx.data())))
                    return fail(rc);
            }
        } else if (ow == c->W) {                               // obj_h == H: the integer ratio 1 x 1 is a copy
            c->obj_mode = 2; c->obj_fx = c->obj_fy = 1;
        } else {
            c->obj_mode = 3;
            if ((rc = upload(&c->obj_uxt, upscale_tab(c->W, ow))) || (rc = upload(&c->obj_uyt, upscale_tab(c->H, obj_h))))
                return fail(rc);
        }
        ALLOC(c->obj_idx, F * sizeof(int));
        if ((cfg->flags & FM_FLAG_NV12) && !c->nv12_bgr) ALLOC(c->obj_bgr, F * c->W * c->H * 3);
    }
    FM_TRY(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
    FM_TRY(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; i++) {
        FM_TRY(cudaEventCreateWithFlags(&c->ev_copied[i], cudaEventDisableTiming));
        FM_TRY(cudaEventCreateWithFlags(&c->ev_done[i], cudaEventDisableTiming));
    }
#undef FM_TRY
#undef ALLOC
    *out = c;
    return FM_OK;
}

extern "C" int fm_ctx_info(const fm_ctx *c, fm_info *info) {
    if (!c || !info) { fm_set_error("null argument"); return FM_EINVAL; }
    *info = c->info;
    return FM_OK;
}

extern "C" int fm_ctx_reset(fm_ctx *c, int stream) {
    if (!c) { fm_set_error("null context"); return FM_EINVAL; }
    if (stream >= c->S) { fm_set_error("stream %d out of range", stream); return FM_EINVAL; }
    FM_CUDA(cudaSetDevice(c->cfg.device));
    FM_CUDA(cudaDeviceSynchronize());
    if (stream < 0) {
        FM_CUDA(cudaMemset(c->state, 0, (size_t)c->S * sizeof(StreamState)));
        FM_CUDA(cudaMemset(c->bg_valid, 0, 2 * (size_t)c->S * sizeof(int)));
        FM_CUDA(cudaMemset(c->errflag, 0, sizeof(int)));
    } else {
        FM_CUDA(cudaMemset(c->state + stream, 0, sizeof(StreamState)));
        for (int i = 0; i < 2; i++) FM_CUDA(cudaMemset(c->bg_valid + (size_t)i * c->S + stream, 0, sizeof(int)));
    }
    return FM_OK;
}

extern "C" int fm_ctx_check(fm_ctx *c) {
    if (!c) { fm_set_error("null context"); return FM_EINVAL; }
    FM_CUDA(cudaSetDevice(c->cfg.device));
    FM_CUDA(cudaDeviceSynchronize());
    int err = 0;
    FM_CUDA(cudaMemcpy(&err, c->errflag, sizeof(int), cudaMemcpyDeviceToHost));
    if (err) {
        FM_CUDA(cudaMemset(c->errflag, 0, sizeof(int)));
        fm_set_error("contour stage: run capacity exceeded (results of the affected frames are not valid)");
        return FM_ERANGE;
    }
    return FM_OK;
}

extern "C" int fm_ctx_set_masks(fm_ctx *c, int stream, int n_polys, const int32_t *poly_offsets,
                                const int32_t *xy) {
    if (!c || n_polys < 0 || (n_polys > 0 && (!poly_offsets || !xy))) { fm_set_error("bad mask arguments"); return FM_EINVAL; }
    if (stream >= c->S) { fm_set_error("stream %d out of range", stream); return FM_EINVAL; }
    FM_CUDA(cudaSetDevice(c->cfg.device));
    FM_CUDA(cudaDeviceSynchronize());
    int npts = n_polys ? poly_offsets[n_polys] : 0;
    std::vector<int> pts((size_t)npts * 2);
    const double scale = c->info.scale;
    for (int i = 0; i < npts * 2; i++) pts[i] = (int)((double)xy[i] * scale);   // find_motion.py:616 int(a*scale)
    int s0 = stream < 0 ? 0 : stream, s1 = stream < 0 ? c->S : stream + 1;
    for (int s = s0; s < s1; s++) {
        int rc = fm_launch_masks(c, s, n_polys, poly_offsets, pts.data(), npts, 0);
        if (rc) return rc;
    }
    FM_CUDA(cudaDeviceSynchronize());
    return FM_OK;
}

// --------------------------------------------------------------------------------------------
// the hot path
// --------------------------------------------------------------------------------------------
static int timing_drain(fm_ctx *c) {
    if (c->fused) {     // group stamps taken by the kernels (the chained launches carry no events)
        if (!c->ev_pending) return FM_OK;
        std::vector<unsigned long long> st((size_t)4 * c->ev_pending);
        FM_CUDA(cudaDeviceSynchronize());
        FM_CUDA(cudaMemcpy(st.data(), c->stamps, st.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        FM_CUDA(cudaMemset(c->stamps, 0, st.size() * sizeof(unsigned long long)));
        for (int i = 0; i < c->ev_pending; i++) {
            const unsigned long long *q = &st[4 * (size_t)i];
            c->t_ms[0] += (double)(q[1] - ~q[0]) * 1e-6;     // front end: first CTA start .. last CTA end
            c->t_ms[2] += (double)(q[3] - ~q[2]) * 1e-6;     // contour stage (the temporal stage is inside K1)
            c->t_calls++;
        }
        c->ev_pending = 0;
        return FM_OK;
    }
    for (int i = 0; i < c->ev_pending; i++) {
        cudaEvent_t *ev = c->evs + 4 * i;
        FM_CUDA(cudaEventSynchronize(ev[3]));
        for (int g = 0; g < 3; g++) {
            float ms = 0;
            FM_CUDA(cudaEventElapsedTime(&ms, ev[g], ev[g + 1]));
            c->t_ms[g] += ms;
        }
        c->t_calls++;
    }
    c->ev_pending = 0;
    return FM_OK;
}

// out: the motion-clip frames of fm_process_clip (null from the other entry points, which with FM_FLAG_DEVICE_CLIPS
// still keep the device ring up to date).  pitch / uv: the row pitch and the chroma offset, resolved (packed: W*3, or W
// and W*H with FM_FLAG_NV12)
static int process(fm_ctx *c, const uint8_t *frames, size_t stream_stride, size_t frame_stride, size_t pitch, int64_t uv,
                   int n_frames, const int32_t *n_valid, void *cuda_stream, fm_frame_stats *stats_dev, uint8_t *out,
                   size_t out_stride) {
    if (!c || !frames) { fm_set_error("null argument"); return FM_EINVAL; }
    if (n_frames < 1 || n_frames > c->Tmax) {
        fm_set_error("n_frames %d outside [1, max_frames=%d]", n_frames, c->Tmax);
        return FM_EINVAL;
    }
    FM_CUDA(cudaSetDevice(c->cfg.device));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    int rc;
    c->obj_src = 0;
    {   // frames of each stream that are real in this call (uploaded only when the vector changes)
        bool changed = false;
        for (int s = 0; s < c->S; s++) {
            int v = n_valid ? n_valid[s] : n_frames;
            if (v < 0 || v > n_frames) { fm_set_error("n_valid[%d] = %d outside [0, n_frames=%d]", s, v, n_frames); return FM_EINVAL; }
            if (v != c->nvalid_host[s]) { c->nvalid_host[s] = v; changed = true; }
        }
        // pageable source: the runtime stages the bytes before returning, so nvalid_host may change right after
        if (changed) FM_CUDA(cudaMemcpyAsync(c->nvalid, c->nvalid_host, (size_t)c->S * sizeof(int), cudaMemcpyHostToDevice, st));
    }
    if (!c->fused) {   // per-frame result slots of the call: ranges = -1 (nothing set), counters = 0
        // (the fused front end clears them itself for the call after it, so that no memset ends the launch chain)
        const size_t Fmax = (size_t)c->S * c->Tmax;
        FM_CUDA(cudaMemsetAsync(c->rawrange, 0xFF, Fmax * 6 * sizeof(int), st));
        FM_CUDA(cudaMemsetAsync(c->ncomp, 0, (Fmax * 2 + 4) * sizeof(int), st));
    }
    cudaEvent_t *ev = nullptr;
    c->stamp = nullptr;
    if (c->timing) {
        if (c->ev_pending == FM_TIMING_RING && (rc = timing_drain(c))) return rc;
        if (c->fused) c->stamp = c->stamps + 4 * c->ev_pending++;
        else { ev = c->evs + 4 * c->ev_pending++; FM_CUDA(cudaEventRecord(ev[0], st)); }
    }
    // NV12 on the staged path: the BGR front end reads the call's frames converted into the context's slot, packed as a
    // dense BGR batch of the call; the device ring keeps the caller's NV12 frames
    const uint8_t *fe = frames;
    size_t fe_sstride = stream_stride, fe_fstride = frame_stride, fe_pitch = pitch;
    if (c->nv12_bgr) {
        rc = fm_launch_nv12_bgr(c, frames, stream_stride, frame_stride, pitch, uv, n_frames, nullptr, c->nv12_bgr, st);
        if (rc) { if (c->stamp) c->ev_pending--; c->stamp = nullptr; return rc; }
        fe = c->nv12_bgr;
        fe_pitch = (size_t)c->W * 3;
        fe_fstride = fe_pitch * c->H;
        fe_sstride = fe_fstride * n_frames;
    }
    if (c->fused) {
        rc = fm_launch_fused(c, fe, fe_sstride, fe_fstride, fe_pitch, uv, n_frames, st);
        if (rc) { if (c->stamp) c->ev_pending--; c->stamp = nullptr; return rc; }
    } else {
        if ((rc = fm_launch_frontend(c, fe, fe_sstride, fe_fstride, fe_pitch, n_frames, st))) return rc;
        if (ev) FM_CUDA(cudaEventRecord(ev[1], st));
        if (!c->wide_fused && !c->umma && (rc = fm_launch_temporal(c, n_frames, st))) return rc;
        if (ev) FM_CUDA(cudaEventRecord(ev[2], st));
    }
    rc = fm_launch_morph_ccl(c, n_frames, st, stats_dev);
    c->stamp = nullptr;
    if (rc) return rc;
    if (c->fused) c->slot ^= 1;
    if (ev) FM_CUDA(cudaEventRecord(ev[3], st));
    if ((c->cfg.flags & FM_FLAG_DEVICE_CLIPS) &&
        (rc = fm_launch_clips(c, frames, stream_stride, frame_stride, pitch, uv, n_frames, out, out_stride, st)))
        return rc;
    c->last_T = n_frames;
    c->planes_valid = true;
    c->obj_src = 1;
    c->obj_frames = frames; c->obj_sstride = stream_stride; c->obj_fstride = frame_stride;
    c->obj_pitch = pitch; c->obj_uv = uv;
    return FM_OK;
}

// Every device entry point: the layout checks of fm_process_frames, then the clip rules of fm_process_clip (clip_out
// non-null), all before anything is enqueued
extern "C" int fm_process_frames(fm_ctx *c, const fm_frames *fr, int n_frames, const int32_t *n_valid, void *cuda_stream,
                                 fm_frame_stats *stats_dev, uint8_t *clip_out, size_t clip_stream_stride, int clip_capacity) {
    if (!c || !fr || !fr->data) { fm_set_error("null argument"); return FM_EINVAL; }
    const bool nv12 = (c->cfg.flags & FM_FLAG_NV12) != 0;
    const size_t row = c->row_bytes;
    const size_t pitch = fr->row_pitch ? fr->row_pitch : row;
    if (pitch < row) {
        fm_set_error("row_pitch %zu < %zu bytes of a row", pitch, row);
        return FM_EINVAL;
    }
    if ((c->px_bytes != 3 || c->rgb) && !nv12 && fr->uv_offset) {
        fm_set_error("uv_offset %lld: %s frames have no chroma plane", (long long)fr->uv_offset,
                     c->px_bytes == 1 ? "gray" : c->px_bytes == 4 ? (c->rgb ? "RGBA" : "BGRA") : "RGB");
        return FM_EINVAL;
    }
    const int64_t luma = (int64_t)(pitch * (c->H - 1) + row);           // bytes the luma rows of a frame span
    const int64_t uv = nv12 ? (fr->uv_offset ? fr->uv_offset : (int64_t)(pitch * c->H)) : 0;
    if (nv12 && uv < luma && uv + (int64_t)(pitch * (c->H / 2 - 1) + row) > 0) {
        fm_set_error("uv_offset %lld: the chroma plane overlaps the luma plane (rows %zu bytes apart, luma spans %lld bytes)",
                     (long long)uv, pitch, (long long)luma);
        return FM_EINVAL;
    }
    const bool packed = pitch == row && (!nv12 || uv == (int64_t)(row * c->H));
    if (!packed && c->fused) {      // k_fused reads by TMA only: refused here, before the call changes anything
        const uintptr_t a = (uintptr_t)fr->data | fr->stream_stride | fr->frame_stride | pitch;
        if (a & 15) {
            fm_set_error("the fused front end reads by TMA: data %p, stream_stride %zu, frame_stride %zu and row_pitch %zu "
                         "must be multiples of 16", (const void *)fr->data, fr->stream_stride, fr->frame_stride, pitch);
            return FM_EINVAL;
        }
        if (nv12 && ((uintptr_t)(fr->data + uv) & 15)) {
            fm_set_error("the fused front end reads by TMA: data + uv_offset (%lld) must be 16-byte aligned", (long long)uv);
            return FM_EINVAL;
        }
    }
    if (clip_out) {
        if (!(c->cfg.flags & FM_FLAG_DEVICE_CLIPS)) {
            fm_set_error("fm_process_clip needs a context created with FM_FLAG_DEVICE_CLIPS");
            return FM_EINVAL;
        }
        if ((long long)clip_capacity < (long long)c->info.cache_frames + n_frames) {
            fm_set_error("out_capacity %d < cache_frames %d + n_frames %d (the most frames one call can write)", clip_capacity,
                         c->info.cache_frames, n_frames);
            return FM_EINVAL;
        }
    }
    return process(c, fr->data, fr->stream_stride, fr->frame_stride, pitch, uv, n_frames, n_valid, cuda_stream, stats_dev,
                   clip_out, clip_stream_stride);
}

extern "C" int fm_process_ragged(fm_ctx *c, const uint8_t *frames, size_t stream_stride, size_t frame_stride,
                                 int n_frames, const int32_t *n_valid, void *cuda_stream, fm_frame_stats *stats_dev) {
    const fm_frames fr = {frames, stream_stride, frame_stride, 0, 0};
    return fm_process_frames(c, &fr, n_frames, n_valid, cuda_stream, stats_dev, nullptr, 0, 0);
}

extern "C" int fm_process_clip(fm_ctx *c, const uint8_t *frames, size_t stream_stride, size_t frame_stride,
                               int n_frames, const int32_t *n_valid, void *cuda_stream, fm_frame_stats *stats_dev,
                               uint8_t *out_dev, size_t out_stream_stride, int out_capacity) {
    if (!c || !frames || !out_dev) { fm_set_error("null argument"); return FM_EINVAL; }
    const fm_frames fr = {frames, stream_stride, frame_stride, 0, 0};
    return fm_process_frames(c, &fr, n_frames, n_valid, cuda_stream, stats_dev, out_dev, out_stream_stride, out_capacity);
}

extern "C" int fm_process(fm_ctx *c, const uint8_t *frames, size_t stream_stride, size_t frame_stride,
                          int n_frames, void *cuda_stream, fm_frame_stats *stats_dev) {
    const fm_frames fr = {frames, stream_stride, frame_stride, 0, 0};
    return fm_process_frames(c, &fr, n_frames, nullptr, cuda_stream, stats_dev, nullptr, 0, 0);
}

extern "C" int fm_object_planes(fm_ctx *c, void *cuda_stream, uint8_t *out_dev, size_t out_stream_stride, int out_capacity) {
    if (!c || !out_dev) { fm_set_error("null argument"); return FM_EINVAL; }
    if (!(c->cfg.flags & FM_FLAG_OBJECT_PLANES)) {
        fm_set_error("fm_object_planes needs a context created with FM_FLAG_OBJECT_PLANES");
        return FM_EINVAL;
    }
    if (c->obj_src != 1) {
        fm_set_error(c->obj_src == 2 ? "the last call came through fm_process_host / fm_submit_host: no device frames to resize"
                                     : "no fm_process / fm_process_ragged / fm_process_clip call to take the planes from");
        return FM_EINVAL;
    }
    const int T = c->last_T;
    const size_t plane = (size_t)FM_OBJECT_WIDTH * c->obj_h * 3;
    if (out_capacity < T) {
        fm_set_error("out_capacity %d < n_frames %d of the last call (the most planes it can have)", out_capacity, T);
        return FM_EINVAL;
    }
    if (c->S > 1 && out_stream_stride < (size_t)out_capacity * plane) {
        fm_set_error("out_stream_stride %zu < out_capacity %d x %zu bytes per plane", out_stream_stride, out_capacity, plane);
        return FM_EINVAL;
    }
    FM_CUDA(cudaSetDevice(c->cfg.device));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    int rc;
    if ((rc = fm_launch_object_plan(c, T, st))) return rc;
    const uint8_t *src = c->obj_frames;
    size_t sstride = c->obj_sstride, fstride = c->obj_fstride, pitch = c->obj_pitch;
    if (c->cfg.flags & FM_FLAG_NV12) {      // the call's frames as BGR, packed as a dense batch of the call (k_nv12.cu)
        if (c->obj_bgr && (rc = fm_launch_nv12_bgr(c, src, sstride, fstride, pitch, c->obj_uv, T, c->obj_idx, c->obj_bgr, st)))
            return rc;
        src = c->obj_bgr ? c->obj_bgr : c->nv12_bgr;
        pitch = (size_t)c->W * 3;
        fstride = pitch * c->H;
        sstride = fstride * T;
    }
    return fm_launch_resize_objects(c, src, sstride, fstride, pitch, T, out_dev, out_stream_stride, st);
}

// ---- host buffers: pipelined (submit / wait on two slots) and the blocking form built on it ----
extern "C" int fm_submit_host(fm_ctx *c, int slot, const uint8_t *frames_host, size_t stream_stride, size_t frame_stride,
                              int n_frames, const int32_t *n_valid) {
    if (!c || !frames_host) { fm_set_error("null argument"); return FM_EINVAL; }
    if (slot < 0 || slot > 1) { fm_set_error("slot %d outside [0, 1]", slot); return FM_EINVAL; }
    if (n_frames < 1 || n_frames > c->Tmax) {
        fm_set_error("n_frames %d outside [1, max_frames=%d]", n_frames, c->Tmax);
        return FM_EINVAL;
    }
    if (c->slot_T[slot]) { fm_set_error("slot %d still holds a batch: call fm_wait first", slot); return FM_EINVAL; }
    FM_CUDA(cudaSetDevice(c->cfg.device));
    const size_t fb = c->frame_bytes;
    const size_t need = (size_t)c->S * n_frames * fb;
    if (c->stage_bytes[slot] < need) {
        cudaFree(c->stage_dev[slot]);
        c->stage_dev[slot] = nullptr; c->stage_bytes[slot] = 0;
        const size_t full = (size_t)c->S * c->Tmax * fb;           // sized once for the largest batch
        FM_CUDA(cudaMalloc(&c->stage_dev[slot], full));
        c->stage_bytes[slot] = full;
    }
    if (!c->stats_pinned[slot]) FM_CUDA(cudaMallocHost(&c->stats_pinned[slot], (size_t)c->S * c->Tmax * sizeof(fm_frame_stats)));
    if (!c->err_pinned) { FM_CUDA(cudaMallocHost(&c->err_pinned, 2 * sizeof(int))); c->err_pinned[0] = c->err_pinned[1] = 0; }
    cudaStream_t cs = c->copy_stream, st = c->own_stream;
    uint8_t *dev = c->stage_dev[slot];
    // densely packed device copy [stream][frame][H][W][3]; only the real frames of a ragged batch travel.
    // The staging buffer of this slot was last read by the kernels of the batch fm_wait(slot) already waited for.
    bool ragged = false;
    if (n_valid) for (int s = 0; s < c->S; s++) ragged |= n_valid[s] != n_frames;
    if (!ragged && frame_stride == fb && stream_stride == fb * (size_t)n_frames) {
        FM_CUDA(cudaMemcpyAsync(dev, frames_host, need, cudaMemcpyHostToDevice, cs));
    } else {
        for (int s = 0; s < c->S; s++) {
            const int nv = n_valid ? n_valid[s] : n_frames;
            if (nv <= 0) continue;
            if (frame_stride == fb)
                FM_CUDA(cudaMemcpyAsync(dev + (size_t)s * n_frames * fb, frames_host + s * stream_stride, (size_t)nv * fb,
                                        cudaMemcpyHostToDevice, cs));
            else
                FM_CUDA(cudaMemcpy2DAsync(dev + (size_t)s * n_frames * fb, fb, frames_host + s * stream_stride, frame_stride,
                                          fb, nv, cudaMemcpyHostToDevice, cs));
        }
    }
    FM_CUDA(cudaEventRecord(c->ev_copied[slot], cs));
    FM_CUDA(cudaStreamWaitEvent(st, c->ev_copied[slot], 0));
    int rc = fm_process_ragged(c, dev, fb * (size_t)n_frames, fb, n_frames, n_valid, st, nullptr);
    if (rc) return rc;
    c->obj_src = 2;                                       // fm_object_planes would read a staging buffer that gets reused
    const size_t sb = (size_t)c->S * n_frames * sizeof(fm_frame_stats);
    FM_CUDA(cudaMemcpyAsync(c->stats_pinned[slot], c->stats, sb, cudaMemcpyDeviceToHost, st));
    FM_CUDA(cudaMemcpyAsync(c->err_pinned + slot, c->errflag, sizeof(int), cudaMemcpyDeviceToHost, st));
    FM_CUDA(cudaEventRecord(c->ev_done[slot], st));
    c->slot_T[slot] = n_frames;
    return FM_OK;
}

extern "C" int fm_wait(fm_ctx *c, int slot, fm_frame_stats *stats_host) {
    if (!c || !stats_host) { fm_set_error("null argument"); return FM_EINVAL; }
    if (slot < 0 || slot > 1 || !c->slot_T[slot]) { fm_set_error("no batch in flight in slot %d", slot); return FM_EINVAL; }
    FM_CUDA(cudaSetDevice(c->cfg.device));
    const int T = c->slot_T[slot];
    c->slot_T[slot] = 0;
    FM_CUDA(cudaEventSynchronize(c->ev_done[slot]));
    if (c->err_pinned[slot]) {
        c->err_pinned[slot] = 0;
        cudaMemsetAsync(c->errflag, 0, sizeof(int), c->own_stream);
        fm_set_error("contour stage: run capacity exceeded");
        return FM_ERANGE;
    }
    memcpy(stats_host, c->stats_pinned[slot], (size_t)c->S * T * sizeof(fm_frame_stats));
    return FM_OK;
}

extern "C" int fm_submit_reset(fm_ctx *c, int stream) {
    if (!c) { fm_set_error("null context"); return FM_EINVAL; }
    if (stream < 0 || stream >= c->S) { fm_set_error("stream %d out of range", stream); return FM_EINVAL; }
    FM_CUDA(cudaSetDevice(c->cfg.device));
    FM_CUDA(cudaMemsetAsync(c->state + stream, 0, sizeof(StreamState), c->own_stream));
    for (int i = 0; i < 2; i++)
        FM_CUDA(cudaMemsetAsync(c->bg_valid + (size_t)i * c->S + stream, 0, sizeof(int), c->own_stream));
    return FM_OK;
}

extern "C" int fm_process_host(fm_ctx *c, const uint8_t *frames_host, size_t stream_stride, size_t frame_stride,
                               int n_frames, fm_frame_stats *stats_host) {
    if (!c || !frames_host || !stats_host) { fm_set_error("null argument"); return FM_EINVAL; }
    int rc = fm_submit_host(c, 0, frames_host, stream_stride, frame_stride, n_frames, nullptr);
    if (rc) return rc;
    return fm_wait(c, 0, stats_host);
}

// ---- pinned host memory next to the context's GPU ----
// cudaHostAlloc places pages by the calling thread's memory policy (first touch by default), so the thread is moved to
// the CPUs the kernel lists as local to the GPU's PCI function (/sys/bus/pci/devices/<bdf>/local_cpulist) for the
// duration of the allocation and the first touch; on platforms that expose a single NUMA node this is a no-op.
static bool parse_cpulist(const char *txt, cpu_set_t *set) {
    CPU_ZERO(set);
    bool any = false;
    const char *p = txt;
    while (*p) {
        char *e;
        long a = strtol(p, &e, 10);
        if (e == p) break;
        long b = a;
        if (*e == '-') { p = e + 1; b = strtol(p, &e, 10); }
        for (long i = a; i <= b && i < CPU_SETSIZE; i++) { CPU_SET((int)i, set); any = true; }
        p = (*e == ',') ? e + 1 : e;
        if (*e != ',') break;
    }
    return any;
}

static bool gpu_local_cpus(int device, cpu_set_t *set, int *node) {
    char bdf[32] = "";
    if (cudaDeviceGetPCIBusId(bdf, sizeof(bdf), device) != cudaSuccess) return false;
    for (char *q = bdf; *q; q++) *q = (char)tolower(*q);
    char path[128], buf[4096];
    *node = -1;
    snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/numa_node", bdf);
    if (FILE *f = fopen(path, "r")) { if (fscanf(f, "%d", node) != 1) *node = -1; fclose(f); }
    snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/local_cpulist", bdf);
    FILE *f = fopen(path, "r");
    if (!f) return false;
    bool ok = fgets(buf, sizeof(buf), f) != nullptr && parse_cpulist(buf, set);
    fclose(f);
    return ok;
}

extern "C" int fm_host_alloc(int device, size_t bytes, void **ptr, int *numa_node) {
    if (!ptr || bytes == 0) { fm_set_error("bad argument"); return FM_EINVAL; }
    *ptr = nullptr;
    FM_CUDA(cudaSetDevice(device));
    cpu_set_t old, local, both;
    int node = -1;
    bool moved = false;
    if (sched_getaffinity(0, sizeof(old), &old) == 0 && gpu_local_cpus(device, &local, &node)) {
        CPU_AND(&both, &old, &local);                     // stay inside the cpuset the process was given
        if (CPU_COUNT(&both) > 0 && !CPU_EQUAL(&both, &old)) moved = sched_setaffinity(0, sizeof(both), &both) == 0;
    }
    if (numa_node) *numa_node = node;
    cudaError_t e = cudaHostAlloc(ptr, bytes, cudaHostAllocPortable);
    if (e == cudaSuccess) {                               // first touch while the thread sits next to the GPU
        volatile unsigned char *p = (volatile unsigned char *)*ptr;
        const size_t page = (size_t)sysconf(_SC_PAGESIZE);
        for (size_t o = 0; o < bytes; o += page) p[o] = 0;
    }
    if (moved) sched_setaffinity(0, sizeof(old), &old);
    if (e != cudaSuccess) {
        fm_set_error("cudaHostAlloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
        return FM_ENOMEM;
    }
    return FM_OK;
}

extern "C" int fm_host_free(void *ptr) {
    if (ptr) FM_CUDA(cudaFreeHost(ptr));
    return FM_OK;
}

extern "C" int fm_get_components(fm_ctx *c, int stream, int t, int max_n, fm_component *out, int *n) {
    if (!c || !n || (max_n > 0 && !out)) { fm_set_error("null argument"); return FM_EINVAL; }
    if (!c->planes_valid || stream < 0 || stream >= c->S || t < 0 || t >= c->last_T) {
        fm_set_error("no such frame in the last call");
        return FM_EINVAL;
    }
    FM_CUDA(cudaSetDevice(c->cfg.device));
    FM_CUDA(cudaDeviceSynchronize());
    size_t f = (size_t)stream * c->last_T + t;
    int cnt = 0;
    FM_CUDA(cudaMemcpy(&cnt, c->ncomp + f, sizeof(int), cudaMemcpyDeviceToHost));
    *n = cnt;
    int m = std::min(cnt, c->maxc);                       // records the device kept (fm_info.max_components)
    std::vector<fm_component> v(m);
    if (m) FM_CUDA(cudaMemcpy(v.data(), c->comps + f * c->maxc, (size_t)m * sizeof(fm_component), cudaMemcpyDeviceToHost));
    std::sort(v.begin(), v.end(), [](const fm_component &a, const fm_component &b) {
        if (a.area_x2 != b.area_x2) return a.area_x2 < b.area_x2;
        if (a.x != b.x) return a.x < b.x;
        if (a.y != b.y) return a.y < b.y;
        if (a.w != b.w) return a.w < b.w;
        return a.h < b.h;
    });
    for (int i = 0; i < std::min(m, max_n); i++) out[i] = v[i];
    return FM_OK;
}

extern "C" int fm_debug_planes(fm_ctx *c, int stream, int t, uint8_t *gray, uint8_t *blur, uint8_t *thresh,
                               double *bg) {
    if (!c) { fm_set_error("null context"); return FM_EINVAL; }
    if (!c->planes_valid || stream < 0 || stream >= c->S || t < 0 || t >= c->last_T) {
        fm_set_error("no such frame in the last call");
        return FM_EINVAL;
    }
    FM_CUDA(cudaSetDevice(c->cfg.device));
    FM_CUDA(cudaDeviceSynchronize());
    size_t f = (size_t)stream * c->last_T + t;
    if ((gray || blur) && !(c->cfg.flags & FM_FLAG_KEEP_PLANES)) {
        fm_set_error("gray/blur planes are only materialised with FM_FLAG_KEEP_PLANES");
        return FM_EINVAL;
    }
    if (gray) FM_CUDA(cudaMemcpy(gray, c->gray + f * c->N, c->N, cudaMemcpyDeviceToHost));
    if (blur) FM_CUDA(cudaMemcpy(blur, c->blur + f * c->N, c->N, cudaMemcpyDeviceToHost));
    if (thresh) {
        DevBuf d;
        FM_CUDA(cudaMalloc(&d.p, c->N));
        int rc = fm_launch_thresh_export(c, stream, t, (uint8_t *)d.p, 0);
        if (rc) return rc;
        FM_CUDA(cudaMemcpy(thresh, d.p, c->N, cudaMemcpyDeviceToHost));
    }
    if (bg) {
        DevBuf d;
        FM_CUDA(cudaMalloc(&d.p, (size_t)c->N * sizeof(double)));
        int rc = c->fused ? fm_launch_bg_export_fused(c, stream, (double *)d.p, 0)
                 : c->umma ? fm_launch_bg_export_umma(c, stream, (double *)d.p, 0)
                 : c->wide_fused ? fm_launch_bg_export_wide(c, stream, (double *)d.p, 0)
                                 : fm_launch_bg_export(c, stream, (double *)d.p, 0);
        if (rc) return rc;
        FM_CUDA(cudaMemcpy(bg, d.p, (size_t)c->N * sizeof(double), cudaMemcpyDeviceToHost));
    }
    return FM_OK;
}

extern "C" int fm_debug_mask(fm_ctx *c, int stream, uint8_t *mask) {
    if (!c || !mask || stream < 0 || stream >= c->S) { fm_set_error("bad argument"); return FM_EINVAL; }
    FM_CUDA(cudaSetDevice(c->cfg.device));
    DevBuf d;
    FM_CUDA(cudaMalloc(&d.p, c->N));
    int rc = fm_launch_mask_export(c, stream, (uint8_t *)d.p, 0);
    if (rc) return rc;
    FM_CUDA(cudaMemcpy(mask, d.p, c->N, cudaMemcpyDeviceToHost));
    return FM_OK;
}

// find_objects' input plane (find_motion.py:703-706): imutils.resize(frame.raw, width=300) = INTER_AREA, BGR out
// the self-checked rows plan of a geometry for px_bytes-byte pixels (1, 3 or 4)
static int rows_plan_px(int W, int H, int box_size, int channels, fm_rows_plan_info *info) {
    if (!info || W < 1 || H < 1 || box_size < 1 || box_size > W) { fm_set_error("bad geometry"); return FM_EINVAL; }
    const int w = box_size, h = (int)((double)H * ((double)box_size / (double)W));          // imutils.resize
    memset(info, 0, sizeof(*info));
    if (h < 1 || (w == W && h == H)) return FM_OK;
    const double sx = 1.0 / ((double)w / W), sy = 1.0 / ((double)h / H);
    if (fabs(sx - nearbyint(sx)) < 2.220446049250313e-16 && fabs(sy - nearbyint(sy)) < 2.220446049250313e-16) return FM_OK;   // integer ratio
    const HostTab xt = area_tab(W, w), yt = area_tab(H, h);
    return fm_rows_plan_describe(W, w, h, channels, xt.start.data(), xt.idx.data(), xt.wt.data(), yt.start.data(), yt.idx.data(),
                                 info);
}

extern "C" int fm_debug_rows_plan_channels(int W, int H, int box_size, int channels, fm_rows_plan_info *info) {
    if (channels != 1 && channels != 3) { fm_set_error("channels %d: 3 (BGR) or 1 (gray)", channels); return FM_EINVAL; }
    return rows_plan_px(W, H, box_size, channels, info);
}

extern "C" int fm_debug_rows_plan(int W, int H, int box_size, fm_rows_plan_info *info) {
    return fm_debug_rows_plan_channels(W, H, box_size, 3, info);
}

extern "C" int fm_debug_rows_plan_format(int W, int H, int box_size, int32_t flags, fm_rows_plan_info *info) {
    if (flags & ~(FM_FLAG_RGB | FM_FLAG_ALPHA | FM_FLAG_GRAY)) {
        fm_set_error("flags %d: a combination of FM_FLAG_RGB and FM_FLAG_ALPHA, or FM_FLAG_GRAY", (int)flags);
        return FM_EINVAL;
    }
    int px_bytes;
    bool rgb;
    if (!fm_pixel_format(flags, &px_bytes, &rgb)) return FM_EINVAL;
    return rows_plan_px(W, H, box_size, px_bytes, info);
}

extern "C" int fm_resize_area(int device, const uint8_t *bgr_host, int W, int H, int width, uint8_t *out_host, int *out_height) {
    if (!bgr_host || !out_host || W < 1 || H < 1 || width < 1) { fm_set_error("bad argument"); return FM_EINVAL; }
    int ndev = 0;
    FM_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) { fm_set_error("CUDA device %d not present", device); return FM_ECUDA; }
    FM_CUDA(cudaSetDevice(device));
    const int h = (int)((double)H * ((double)width / (double)W));            // imutils.resize: int(h * r)
    if (h < 1) { fm_set_error("resized height is zero"); return FM_ERANGE; }
    if (out_height) *out_height = h;
    if (width == W && h == H) { memcpy(out_host, bgr_host, (size_t)W * H * 3); return FM_OK; }
    if (width > W) {                                                          // h >= H: cv2's fixed-point linear upscale
        struct UpTabs {
            int2 *x = nullptr, *y = nullptr;
            ~UpTabs() { cudaFree(x); cudaFree(y); }
        } ut;
        int rc;
        if ((rc = upload(&ut.x, upscale_tab(W, width)))) return rc;
        if ((rc = upload(&ut.y, upscale_tab(H, h)))) return rc;
        DevBuf src, dst;
        FM_CUDA(cudaMalloc(&src.p, (size_t)W * H * 3));
        FM_CUDA(cudaMalloc(&dst.p, (size_t)width * h * 3));
        FM_CUDA(cudaMemcpy(src.p, bgr_host, (size_t)W * H * 3, cudaMemcpyHostToDevice));
        if ((rc = fm_launch_upscale(device, (const uint8_t *)src.p, 0, 0, (size_t)W * 3, 1, 1, W, H, width, h, ut.x, ut.y, nullptr, nullptr,
                                    (uint8_t *)dst.p, nullptr, 0, 0, 3)))
            return rc;
        FM_CUDA(cudaMemcpy(out_host, dst.p, (size_t)width * h * 3, cudaMemcpyDeviceToHost));
        return FM_OK;
    }
    const double sx = 1.0 / ((double)width / W), sy = 1.0 / ((double)h / H);
    const int isx = (int)nearbyint(sx), isy = (int)nearbyint(sy);
    const bool fast = fabs(sx - isx) < 2.220446049250313e-16 && fabs(sy - isy) < 2.220446049250313e-16;
    struct Tabs {
        ResizeTab x{}, y{};
        ~Tabs() { cudaFree(x.start); cudaFree(x.idx); cudaFree(x.wt); cudaFree(y.start); cudaFree(y.idx); cudaFree(y.wt); }
    } tb;
    int rc;
    if (!fast) {
        if ((rc = upload_tab(&tb.x, area_tab(W, width)))) return rc;
        if ((rc = upload_tab(&tb.y, area_tab(H, h)))) return rc;
    }
    DevBuf src, dst;
    FM_CUDA(cudaMalloc(&src.p, (size_t)W * H * 3));
    FM_CUDA(cudaMalloc(&dst.p, (size_t)width * h * 3));
    FM_CUDA(cudaMemcpy(src.p, bgr_host, (size_t)W * H * 3, cudaMemcpyHostToDevice));
    if ((rc = fm_launch_resize_bgr(device, (const uint8_t *)src.p, 0, 0, (size_t)W * 3, 1, 1, W, H, width, h, fast ? 2 : 1, isx, isy, tb.x,
                                   tb.y, nullptr, (uint8_t *)dst.p, 0, 0, 3)))
        return rc;
    FM_CUDA(cudaMemcpy(out_host, dst.p, (size_t)width * h * 3, cudaMemcpyDeviceToHost));
    return FM_OK;
}

extern "C" int fm_debug_components(int device, const uint8_t *plane, int w, int h, int max_n, fm_component *out,
                                   int *n) {
    if (!plane || !n || w < 1 || h < 1 || w > 65535) { fm_set_error("bad argument"); return FM_EINVAL; }
    int ndev = 0;
    FM_CUDA(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) { fm_set_error("CUDA device %d not present", device); return FM_ECUDA; }
    std::vector<fm_component> v(std::max(max_n, 1));
    int rc = fm_ccl_plane(device, plane, w, h, max_n, v.data(), n);
    if (rc) return rc;
    int m = std::min(*n, max_n);
    std::sort(v.begin(), v.begin() + m, [](const fm_component &a, const fm_component &b) {
        if (a.area_x2 != b.area_x2) return a.area_x2 < b.area_x2;
        if (a.x != b.x) return a.x < b.x;
        if (a.y != b.y) return a.y < b.y;
        if (a.w != b.w) return a.w < b.w;
        return a.h < b.h;
    });
    for (int i = 0; i < m; i++) out[i] = v[i];
    return FM_OK;
}

extern "C" int fm_timing_enable(fm_ctx *c, int on) {
    if (!c) return FM_EINVAL;
    FM_CUDA(cudaSetDevice(c->cfg.device));
    if (on && c->fused && !c->stamps) {
        FM_CUDA(cudaMalloc(&c->stamps, (size_t)4 * FM_TIMING_RING * sizeof(unsigned long long)));
        FM_CUDA(cudaMemset(c->stamps, 0, (size_t)4 * FM_TIMING_RING * sizeof(unsigned long long)));
    }
    if (on && !c->fused && !c->evs) {
        c->evs = new cudaEvent_t[4 * FM_TIMING_RING];
        for (int i = 0; i < 4 * FM_TIMING_RING; i++) FM_CUDA(cudaEventCreate(&c->evs[i]));
    }
    if (!on && c->ev_pending) { int rc = timing_drain(c); if (rc) return rc; }
    c->timing = on != 0;
    return FM_OK;
}
extern "C" int fm_timing_reset(fm_ctx *c) {
    if (!c) return FM_EINVAL;
    if (c->ev_pending) { int rc = timing_drain(c); if (rc) return rc; }
    c->t_ms[0] = c->t_ms[1] = c->t_ms[2] = 0;
    c->t_calls = 0;
    return FM_OK;
}
extern "C" int fm_timing_get(fm_ctx *c, int which, double *ms_total, int64_t *n_calls) {
    if (!c || which < 0 || which > 2) return FM_EINVAL;
    if (c->ev_pending) { int rc = timing_drain(c); if (rc) return rc; }
    if (ms_total) *ms_total = c->t_ms[which];
    if (n_calls) *n_calls = c->t_calls;
    return FM_OK;
}

