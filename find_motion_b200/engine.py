"""MotionEngine: thin Python handle on an fm_ctx (include/fm_gpu.h).

One engine = n_streams streams of equal geometry and tuning processed as a batch on one GPU,
the B200 replacement of one `partial(run_vid, **tuning)` job set (find_motion.py:1323-1331).
torch is used only for device memory, streams and pinned host buffers.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib

STATS_DTYPE = np.dtype([(n, np.int32) for n in ("n_contours", "n_counted", "movement", "movement_counter",
                                                "movement_decay", "cache_len", "wrote", "n_flush")])


class MotionEngine:
    def __init__(self, frame_width, frame_height, n_streams=1, max_frames=8, device=0, fps=30, box_size=100,
                 min_box_scale=50, cache_time=2.0, min_time=0.5, threshold=7, avg=0.1, blur_scale=20,
                 mask_areas=None, max_components=256, keep_planes=False, no_fused=False, no_umma=False, umma_apron=False, umma=False, no_rows=False,
                 upscale=False, device_clips=False, nv12=False, object_planes=False):
        """upscale: accept box_size > frame_width (cv2's INTER_AREA upscale, bit-exact, as imutils.resize does it);
        without it such a geometry raises, as in earlier releases.
        device_clips: keep the look-back cache of raw frames on the GPU (n_streams x cache_frames frames) so that
        process_clip can hand out the frames the reference writes to its *_motion.avi.
        nv12: the frames are NV12 as GPU video decoders emit them, each [H * 3 // 2, W] uint8 (the luma rows, then the
        interleaved U, V rows; W and H even), with the results of a BGR engine on cv2.cvtColor(frame,
        cv2.COLOR_YUV2BGR_NV12).  process, process_clip, submit_host and process_host then take [S, T, H * 3 // 2, W],
        and the clips are NV12 frames too.
        object_planes: accept object_planes(), the input planes of the reference's find_objects for the frames each
        process / process_clip call writes (imutils.resize(frame.raw, width=300), made on the GPU)."""
        self._lib = _lib.load()
        self._ctx = C.c_void_p()
        cfg = _lib.fm_config(
            device=device, n_streams=n_streams, frame_width=frame_width, frame_height=frame_height,
            max_frames=max_frames, fps=int(fps), box_size=int(box_size), min_box_scale=int(min_box_scale),
            blur_scale=int(blur_scale), threshold=int(threshold), avg=float(avg), min_time=float(min_time),
            cache_time=float(cache_time), max_components=max_components,
            flags=(_lib.FLAG_KEEP_PLANES if keep_planes else 0) | (_lib.FLAG_NO_FUSED if no_fused else 0) |
            (_lib.FLAG_NO_UMMA if no_umma else 0) | (_lib.FLAG_UMMA_APRON if umma_apron else 0) | (_lib.FLAG_UMMA if umma else 0) |
            (_lib.FLAG_NO_ROWS if no_rows else 0) | (_lib.FLAG_UPSCALE if upscale else 0) |
            (_lib.FLAG_DEVICE_CLIPS if device_clips else 0) | (_lib.FLAG_NV12 if nv12 else 0) |
            (_lib.FLAG_OBJECT_PLANES if object_planes else 0))
        _lib.check(self._lib.fm_ctx_create(C.byref(cfg), C.byref(self._ctx)))
        self.device = device
        self.n_streams, self.max_frames = n_streams, max_frames
        self.W, self.H = frame_width, frame_height
        self.nv12 = bool(nv12)
        # shape of one input frame
        self.frame_shape = (frame_height * 3 // 2, frame_width) if nv12 else (frame_height, frame_width, 3)
        inf = _lib.fm_info()
        _lib.check(self._lib.fm_ctx_info(self._ctx, C.byref(inf)))
        self.info = {f: getattr(inf, f) for f, _ in _lib.fm_info._fields_}
        self.w, self.h = inf.proc_width, inf.proc_height
        self.max_components = inf.max_components
        self._stats_dev = None
        self._clips_out = None
        self._objects_out = None
        self._last_T = None              # frames per stream of the last process / process_clip call
        # shape of one detector input plane (find_objects: imutils.resize(frame.raw, width=300))
        self.object_shape = (int(frame_height * (_lib.OBJECT_WIDTH / float(frame_width))), _lib.OBJECT_WIDTH, 3)
        self._inflight = {}
        if mask_areas:
            self.set_masks(mask_areas)

    # -- life cycle ---------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx.value:
            self._lib.fm_ctx_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- configuration --------------------------------------------------------------------------
    def set_masks(self, mask_areas, stream=-1):
        """mask_areas: the reference's list of areas, each a tuple of (x, y) points in SOURCE
        pixels; two points = rectangle, more = polygon (find_motion.py:619-635)."""
        offs, xy = [0], []
        for area in mask_areas or []:
            for (x, y) in area:
                xy += [int(x), int(y)]
            offs.append(len(xy) // 2)
        n = len(offs) - 1
        offs_a = (C.c_int32 * len(offs))(*offs)
        xy_a = (C.c_int32 * max(len(xy), 1))(*xy)
        _lib.check(self._lib.fm_ctx_set_masks(self._ctx, stream, n, offs_a, xy_a))

    def reset(self, stream=-1):
        _lib.check(self._lib.fm_ctx_reset(self._ctx, stream))

    # -- hot path ---------------------------------------------------------------------------------
    @staticmethod
    def _nvalid(n_valid, S, T):
        if n_valid is None:
            return None
        nv = [int(v) for v in n_valid]
        assert len(nv) == S and all(0 <= v <= T for v in nv), "n_valid: one count in [0, T] per stream"
        return (C.c_int32 * S)(*nv)

    def _check_batch(self, shape):
        """-> (S, T) of a batch [n_streams, T, *frame_shape]"""
        assert len(shape) == 2 + len(self.frame_shape) and shape[0] == self.n_streams and \
            tuple(shape[2:]) == self.frame_shape, f"frame geometry mismatch: want [{self.n_streams}, T, {self.frame_shape}]"
        return shape[0], shape[1]

    def process(self, frames, sync=True, n_valid=None):
        """frames: CUDA uint8 tensor [n_streams, T, H, W, 3] (BGR; nv12: [n_streams, T, H * 3 // 2, W]).  Returns the
        per-frame stats as a structured numpy array [n_streams, T] (or the device tensor if sync=False).
        n_valid: optional per-stream count of real frames in this call (ragged batch)."""
        import torch

        assert frames.is_cuda and frames.dtype == torch.uint8, "uint8 CUDA frames"
        S, T = self._check_batch(frames.shape)
        assert frames[0, 0].is_contiguous()
        need = S * T * STATS_DTYPE.itemsize
        if self._stats_dev is None or self._stats_dev.numel() < need:
            self._stats_dev = torch.empty(S * self.max_frames * STATS_DTYPE.itemsize, dtype=torch.uint8,
                                          device=frames.device)
        st = torch.cuda.current_stream(frames.device).cuda_stream
        _lib.check(self._lib.fm_process_ragged(self._ctx, frames.data_ptr(), frames.stride(0), frames.stride(1), T,
                                               self._nvalid(n_valid, S, T), C.c_void_p(st), self._stats_dev.data_ptr()))
        self._last_T = T
        if not sync:
            return self._stats_dev[:need]
        host = self._stats_dev[:need].cpu().numpy()
        self.check()
        return host.view(STATS_DTYPE).reshape(S, T)

    def process_clip(self, frames, n_valid=None, out=None):
        """process() that also returns the frames the reference writes to its *_motion.avi in this call (needs
        device_clips=True).  frames: CUDA uint8 tensor [n_streams, T, *frame_shape] (frame_shape = (H, W, 3), or
        (H * 3 // 2, W) with nv12).  out: optional CUDA uint8 tensor [n_streams, >= cache_frames + T, *frame_shape]
        (dense frames) for them; by default one of [n_streams, cache_frames + max_frames, *frame_shape] is allocated once
        and reused, so the views returned by one call are overwritten by the next.  Runs on the current torch stream and
        synchronises.
        Returns (stats [n_streams, T], clips): clips[s] is a view [n_out, *frame_shape] of `out` holding, in order, the
        cached frames each frame of stream s flushes and the frame itself where it is written."""
        import torch

        assert frames.is_cuda and frames.dtype == torch.uint8, "uint8 CUDA frames"
        S, T = self._check_batch(frames.shape)
        assert frames[0, 0].is_contiguous()
        if out is None:
            if self._clips_out is None:
                self._clips_out = torch.empty((S, self.info["cache_frames"] + self.max_frames) + self.frame_shape,
                                              dtype=torch.uint8, device=frames.device)
            out = self._clips_out
        assert out.is_cuda and out.dtype == torch.uint8 and out.dim() == 2 + len(self.frame_shape) and \
            out.shape[0] == S and tuple(out.shape[2:]) == self.frame_shape and out[0].is_contiguous(), \
            "uint8 CUDA [S, capacity, *frame_shape]"
        need = S * T * STATS_DTYPE.itemsize
        if self._stats_dev is None or self._stats_dev.numel() < need:
            self._stats_dev = torch.empty(S * self.max_frames * STATS_DTYPE.itemsize, dtype=torch.uint8,
                                          device=frames.device)
        st = torch.cuda.current_stream(frames.device).cuda_stream
        _lib.check(self._lib.fm_process_clip(self._ctx, frames.data_ptr(), frames.stride(0), frames.stride(1), T,
                                             self._nvalid(n_valid, S, T), C.c_void_p(st), self._stats_dev.data_ptr(),
                                             out.data_ptr(), out.stride(0), out.shape[1]))
        self._last_T = T
        stats = self._stats_dev[:need].cpu().numpy().view(STATS_DTYPE).reshape(S, T)
        self.check()
        n_out = (stats["wrote"].astype(np.int64) + stats["n_flush"]).sum(axis=1)
        return stats, [out[s, :int(n_out[s])] for s in range(S)]

    def object_planes(self, out=None):
        """The input planes of the reference's find_objects (find_motion.py:572, 703-706) for the frames the last
        process / process_clip call wrote (needs object_planes=True): cv2.resize(raw, (300, oh), INTER_AREA) of each,
        bit-exact, made on the GPU from that call's frames (which must still hold them).  NV12 engines resize
        cv2.cvtColor(frame, COLOR_YUV2BGR_NV12).  out: optional CUDA uint8 tensor [n_streams, >= T, *object_shape]; by
        default one of [n_streams, max_frames, *object_shape] is allocated once and reused, so the views returned by one
        call are overwritten by the next.  Runs on the current torch stream and synchronises.
        Returns, per stream, (frame_indices, planes): the indices t of the written frames in the call, in order, and a
        view [len(frame_indices), *object_shape] of `out` holding their planes."""
        import torch

        dev = torch.device("cuda", self.device)
        if out is None:
            if self._objects_out is None:
                self._objects_out = torch.empty((self.n_streams, self.max_frames) + self.object_shape, dtype=torch.uint8,
                                                device=dev)
            out = self._objects_out
        assert out.is_cuda and out.dtype == torch.uint8 and out.dim() == 5 and out.shape[0] == self.n_streams and \
            tuple(out.shape[2:]) == self.object_shape and out[0].is_contiguous(), "uint8 CUDA [S, capacity, oh, 300, 3]"
        st = torch.cuda.current_stream(out.device).cuda_stream
        _lib.check(self._lib.fm_object_planes(self._ctx, C.c_void_p(st), out.data_ptr(), out.stride(0), out.shape[1]))
        T = self._last_T
        stats = self._stats_dev[:self.n_streams * T * STATS_DTYPE.itemsize].cpu().numpy().view(STATS_DTYPE)
        self.check()
        res = []
        for s, wrote in enumerate(stats.reshape(self.n_streams, T)["wrote"]):
            idx = np.flatnonzero(wrote)
            res.append((idx, out[s, :len(idx)]))
        return res

    def check(self):
        """Synchronise and raise if a call since the last check hit a device-side capacity error."""
        _lib.check(self._lib.fm_ctx_check(self._ctx))

    @staticmethod
    def _host_view(frames):
        """-> (object that owns the memory, pointer, shape, stream stride, frame stride); frames must be dense."""
        if hasattr(frames, "data_ptr"):
            assert frames[0, 0].is_contiguous()
            return frames, frames.data_ptr(), tuple(frames.shape), frames.stride(0), frames.stride(1)
        frames = np.asarray(frames)
        if frames.dtype != np.uint8 or not frames[0, 0].flags["C_CONTIGUOUS"]:
            frames = np.ascontiguousarray(frames, np.uint8)
        return frames, frames.ctypes.data, frames.shape, frames.strides[0], frames.strides[1]

    def submit_host(self, slot, frames, n_valid=None):
        """Pipelined host entry: enqueue the batch [n_streams, T, *frame_shape] (host array / pinned tensor) on slot 0
        or 1 and return; wait_host(slot) gives its stats.  The buffer must stay untouched until then."""
        frames, ptr, shape, s0, s1 = self._host_view(frames)
        S, T = self._check_batch(shape)
        _lib.check(self._lib.fm_submit_host(self._ctx, slot, C.c_void_p(ptr), s0, s1, T, self._nvalid(n_valid, S, T)))
        self._inflight[slot] = (T, frames)          # keeps the buffer alive

    def submit_reset(self, stream):
        """reset(stream) ordered with the submitted batches: takes effect after the batches already submitted and
        before the next one (a slot of a batched context changing over to the next file)."""
        _lib.check(self._lib.fm_submit_reset(self._ctx, stream))

    def wait_host(self, slot):
        T, _ = self._inflight.pop(slot)
        out = np.empty((self.n_streams, T), STATS_DTYPE)
        _lib.check(self._lib.fm_wait(self._ctx, slot, C.c_void_p(out.ctypes.data)))
        return out

    def process_host(self, frames):
        """frames: host uint8 array / pinned tensor [n_streams, T, *frame_shape].  Copies in, runs,
        copies the stats out (the end-to-end call of the drop-in adapter)."""
        frames, ptr, shape, s0, s1 = self._host_view(frames)
        S, T = self._check_batch(shape)
        out = np.empty((S, T), STATS_DTYPE)
        _lib.check(self._lib.fm_process_host(self._ctx, C.c_void_p(ptr), s0, s1, T, C.c_void_p(out.ctypes.data)))
        return out

    # -- taps ---------------------------------------------------------------------------------------
    def components(self, stream, t, max_n=None):
        max_n = max_n or 4096
        buf = (_lib.fm_component * max_n)()
        n = C.c_int(0)
        _lib.check(self._lib.fm_get_components(self._ctx, stream, t, max_n, buf, C.byref(n)))
        m = min(n.value, max_n, self.max_components)     # records the device kept; n is the true count
        return n.value, [(buf[i].area_x2, (buf[i].x, buf[i].y, buf[i].w, buf[i].h)) for i in range(m)]

    def motion_boxes(self, stream, t):
        """The rectangles `--show` would draw for frame t (find_motion.py:690-692, 787-813): for every contour
        that find_movement counts, make_area_from_rect(boundingRect) scaled back to source pixels with
        scale_area(area, 1 / scale) (int() truncation).  Sorted."""
        n, comps = self.components(stream, t)
        if n > len(comps):
            raise _lib.FmError(-4, f"frame has {n} contours, only {len(comps)} kept: raise max_components")
        inv = 1 / self.info["scale"]
        out = []
        for area2, (x, y, w, h) in comps:
            area = area2 / 2.0
            if self.info["max_area"] < area < self.info["min_area"]:      # find_motion.py:684
                continue
            out.append(((int(x * inv), int(y * inv)), (int((x + w) * inv), int((y + h) * inv))))
        return sorted(out)

    def planes(self, stream, t, gray=True, blur=True, thresh=True, bg=True):
        out = {}
        arrs = {}
        for key, want, dt in (("gray", gray, np.uint8), ("blur", blur, np.uint8), ("thresh", thresh, np.uint8),
                              ("bg", bg, np.float64)):
            arrs[key] = np.empty((self.h, self.w), dt) if want else None
        ptr = lambda a: C.c_void_p(a.ctypes.data) if a is not None else None  # noqa: E731
        _lib.check(self._lib.fm_debug_planes(self._ctx, stream, t, ptr(arrs["gray"]), ptr(arrs["blur"]),
                                             ptr(arrs["thresh"]), ptr(arrs["bg"])))
        out.update({k: v for k, v in arrs.items() if v is not None})
        return out

    def mask(self, stream=0):
        m = np.empty((self.h, self.w), np.uint8)
        _lib.check(self._lib.fm_debug_mask(self._ctx, stream, C.c_void_p(m.ctypes.data)))
        return m

    def timing(self, enable=None, reset=False):
        if enable is not None:
            _lib.check(self._lib.fm_timing_enable(self._ctx, int(enable)))
        if reset:
            _lib.check(self._lib.fm_timing_reset(self._ctx))
        res = {}
        for i, name in enumerate(("front_end", "temporal", "contours")):
            ms, n = C.c_double(0), C.c_int64(0)
            _lib.check(self._lib.fm_timing_get(self._ctx, i, C.byref(ms), C.byref(n)))
            res[name] = (ms.value, n.value)
        return res


def label_components(plane: np.ndarray, device=0, max_n=65536):
    """findContours(RETR_EXTERNAL)+contourArea+boundingRect of a host uint8 plane on the GPU."""
    lib = _lib.load()
    plane = np.ascontiguousarray(plane, np.uint8)
    h, w = plane.shape
    buf = (_lib.fm_component * max_n)()
    n = C.c_int(0)
    _lib.check(lib.fm_debug_components(device, C.c_void_p(plane.ctypes.data), w, h, max_n, buf, C.byref(n)))
    return [(buf[i].area_x2, (buf[i].x, buf[i].y, buf[i].w, buf[i].h)) for i in range(min(n.value, max_n))]


class PinnedBatch:
    """uint8 numpy array in pinned host memory next to `device` (fm_host_alloc), for frame batches."""

    def __init__(self, shape, device=0):
        self._lib = _lib.load()
        n = int(np.prod(shape))
        p, node = C.c_void_p(), C.c_int(-1)
        _lib.check(self._lib.fm_host_alloc(device, n, C.byref(p), C.byref(node)))
        self._ptr, self.numa_node = p, node.value
        self.array = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(n,)).reshape(shape)

    def free(self):
        if self._ptr is not None and self._ptr.value:
            self.array = None
            self._lib.fm_host_free(self._ptr)
            self._ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def resize_area(frame: np.ndarray, width: int = 300, device: int = 0) -> np.ndarray:
    """imutils.resize(frame, width=width) (cv2.INTER_AREA) of one BGR frame on the GPU: the input plane of the
    reference's find_objects (find_motion.py:703-706).  Bit-exact with cv2, also for width > frame width (upscale)."""
    lib = _lib.load()
    frame = np.ascontiguousarray(frame, np.uint8)
    H, W, ch = frame.shape
    assert ch == 3
    h = int(H * (width / float(W)))
    out = np.empty((max(h, 1), width, 3), np.uint8)
    oh = C.c_int(0)
    _lib.check(lib.fm_resize_area(device, C.c_void_p(frame.ctypes.data), W, H, width, C.c_void_p(out.ctypes.data), C.byref(oh)))
    return out[:oh.value]


def launch_count() -> int:
    return int(_lib.load().fm_launch_count())
