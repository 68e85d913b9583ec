// Detector input planes (FM_FLAG_OBJECT_PLANES, fm_object_planes): the reference's decide_output calls find_objects on
// every frame it writes (find_motion.py:572), and find_objects starts with imutils.resize(frame.raw, width=300)
// (find_motion.py:703-706), i.e. cv2.resize(INTER_AREA) to 300 x oh.  Those planes are made here from the frames of the
// last hot-path call, with the frame list taken from that call's own decisions on the device.
//
// Launches: k_object_plan (one CTA, one warp per stream) turns the `wrote` flags of the call's stats into one plane
// index per frame (oidx, -1 = no plane).  The resize kernels of the processing plane then run with BGR output, skip the
// frames with oidx < 0 and address their output through oidx (SURVEY.md A.1):
//   * k_resize_rows<true> when the context has a usable rows plan for W -> 300 and the frames are 16-byte aligned;
//   * otherwise k_resize_gray with bgr_out (tables, integer ratios, and the identity as the integer ratio 1 x 1);
//   * k_upscale_gray with bgr_out for W < 300.
// NV12 contexts resize the BGR slot: the staged front ends already hold the call's frames converted there; a fused
// context first converts its written frames into its own slot with k_nv12_bgr.
#include "fm_common.cuh"

#define OBJ_PLAN_THREADS 1024

__global__ void __launch_bounds__(OBJ_PLAN_THREADS) k_object_plan(const fm_frame_stats *__restrict__ stats,
                                                                  const int *__restrict__ nvalid, int S, int T,
                                                                  int *__restrict__ oidx) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int s = warp; s < S; s += OBJ_PLAN_THREADS / 32) {
        const int Ts = min(T, __ldg(nvalid + s));
        int off = 0;                                              // planes of the stream so far
        for (int tc = 0; tc < T; tc += 32) {
            const int t = tc + lane;
            const bool wrote = t < Ts && stats[(size_t)s * T + t].wrote;
            const unsigned m = __ballot_sync(0xffffffffu, wrote);
            if (t < T) oidx[(size_t)s * T + t] = wrote ? off + __popc(m & ((1u << lane) - 1)) : -1;
            off += __popc(m);
        }
    }
}

int fm_launch_object_plan(fm_ctx *c, int T, cudaStream_t st) {
    k_object_plan<<<1, OBJ_PLAN_THREADS, 0, st>>>(c->stats, c->nvalid, c->S, T, c->obj_idx);
    FM_LAUNCH_CHECK();
    return FM_OK;
}

int fm_launch_resize_objects(fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, int T, uint8_t *out,
                             size_t ostride, cudaStream_t st) {
    const int w = FM_OBJECT_WIDTH, h = c->obj_h;
    if (c->obj_mode == 3)
        return fm_launch_upscale(c->cfg.device, frames, sstride, fstride, T, c->S * T, c->W, c->H, w, h, c->obj_uxt,
                                 c->obj_uyt, nullptr, nullptr, out, c->obj_idx, ostride, st);
    if (c->obj_rows && ((((uintptr_t)frames) | sstride | fstride) & 15) == 0)
        return fm_launch_resize_rows_objects(c, frames, sstride, fstride, T, out, ostride, st);
    return fm_launch_resize_bgr(c->cfg.device, frames, sstride, fstride, c->S, T, c->W, c->H, w, h, c->obj_mode, c->obj_fx,
                                c->obj_fy, c->obj_xtab, c->obj_ytab, c->obj_idx, out, ostride, st);
}
