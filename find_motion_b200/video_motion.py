"""Drop-in mirror of the reference's per-stream surface: VideoMotion and run_vid
(find_motion/find_motion.py:299-380, 852-904, 1021-1037), with the per-frame cv2 call chain
replaced by the B200 path (libfmgpu.so through MotionEngine).

Same constructor keywords, same derived parameters, same `(wrote_frames, err_msg, seen_objects)`
result, same output files: decode (`cap.read`) and encode (`outfile.write(frame.raw)`) stay on
the host exactly as in the reference; frames are batched `chunk` at a time into pinned host memory,
the GPU returns the per-frame decisions, and the adapter replays decide_output's cache/flush/write
actions in frame order on the raw frames.  Batches are pipelined: while batch i is on the GPU the
host decodes batch i+1 and replays batch i-1.  Many files / cameras are batched into one context per
GPU by find_motion_b200.jobs (run_pool / run_map / run_stream).  Display (`show`), Haar cascades and YOLO are outside the hot
path (SURVEY.md section 2 rows 6, 10, 11) and are ignored with a warning.
"""
from __future__ import annotations

import logging
import os
import typing
from collections import deque

import numpy as np

from .engine import MotionEngine, PinnedBatch

log = logging.getLogger("find_motion")


class VideoError(Exception):
    """find_motion.py:173-178"""


class VideoMotion(object):
    def __init__(self, filename: typing.Union[str, int, typing.Any] = None, outdir: str = '', fps: int = 30,
                 box_size: int = 100, min_box_scale: int = 50, cache_time: float = 2.0, min_time: float = 0.5,
                 threshold: int = 7, avg: float = 0.1, blur_scale: int = 20,
                 mask_areas: list = None, show: bool = False,
                 codec: str = 'MJPG', log_level: int = logging.INFO,
                 mem: bool = False, cleanup: bool = False,
                 multiprocess: bool = False,
                 cascades: typing.List[str] = None,
                 yolo_tiny: bool = False, *,
                 device: int = 0, chunk: int = 16, engine: typing.Any = None) -> None:
        self.filename = filename
        if self.filename is None:
            raise Exception('Filename required')                      # find_motion.py:311
        self.log = logging.getLogger('find_motion.VideoMotion')
        self.log.setLevel(log_level)
        self.multiprocess = multiprocess
        self.outfile = None
        self.outfiles = 0
        self.outfile_name = ''
        self.outdir = os.path.normpath(outdir)                        # :326 ('' becomes '.', as in the reference)
        self.fps = fps
        self.box_size = box_size
        self.min_box_scale = min_box_scale
        self.gaussian_scale = blur_scale
        self.cache_frames = int(cache_time * fps)                     # :334
        self.min_movement_frames = int(min_time * fps)                # :335
        self.delta_thresh = threshold
        self.avg = avg
        self.mask_areas = mask_areas if mask_areas is not None else []
        self.show = show
        self.codec = codec
        self.debug = log_level == logging.DEBUG
        self.mem = mem
        self.cleanup_flag = cleanup
        if show or cascades or yolo_tiny:
            self.log.warning('show / cascades / yolo_tiny are outside the GPU hot path and are ignored')
        self._tuning = dict(fps=fps, box_size=box_size, min_box_scale=min_box_scale, cache_time=cache_time,
                            min_time=min_time, threshold=threshold, avg=avg, blur_scale=blur_scale)
        self.device = device
        self.chunk = max(1, int(chunk))

        self.amount_of_frames = -1
        self.frame_width = -1
        self.frame_height = -1
        self.scale = -1.0
        self.frame_cache: typing.Deque[np.ndarray] = deque()
        self.wrote_frames: typing.Optional[bool] = False
        self.err_msg = ''
        self.movement = False
        self.movement_decay = 0
        self.movement_counter = 0
        self.seen_objects: typing.Set[str] = set()
        self.frames_read = 0
        self.frames_written = 0
        # engine=False: the stream is one slot of a batched context driven by find_motion_b200.jobs
        self._own_engine = engine is None
        self.engine: typing.Optional[MotionEngine] = engine if engine not in (None, False) else None
        self.loaded = self._load_video()

    # -- I/O (host side, as in the reference) ---------------------------------------------------
    def _open_capture(self):
        self._cv_capture = False
        if hasattr(self.filename, 'read') and hasattr(self.filename, 'get'):
            return self.filename                                     # capture-like object (tests, cameras)
        import cv2
        self._cv_capture = True
        return cv2.VideoCapture(self.filename)                        # :413

    def _get_video_info(self) -> None:
        import cv2
        self.amount_of_frames = int(self.cap.get(cv2.CAP_PROP_FRAME_COUNT))       # :430-432
        self.frame_width = int(self.cap.get(cv2.CAP_PROP_FRAME_WIDTH))
        self.frame_height = int(self.cap.get(cv2.CAP_PROP_FRAME_HEIGHT))
        if self.frame_width == 0 or self.frame_height == 0:
            broken = 'width' if self.frame_width == 0 else 'height'
            raise VideoError("Video info malformed - {} is 0: {}".format(broken, self.filename))

    def _load_video(self) -> bool:
        self.cap = self._open_capture()
        self.frame_cache = deque(maxlen=self.cache_frames)            # :415
        try:
            self._get_video_info()
        except VideoError as e:
            self.log.error(str(e))
            return False
        if self._own_engine:
            self.engine = MotionEngine(self.frame_width, self.frame_height, n_streams=1, max_frames=self.chunk,
                                       device=self.device, mask_areas=self.mask_areas, upscale=True, **self._tuning)
        if self.engine is not None:
            self._adopt_info(self.engine.info)
        return True

    def _adopt_info(self, inf) -> None:
        self.scale = inf["scale"]
        self.max_area = inf["max_area"]
        self.min_area = inf["min_area"]
        self.gaussian = (inf["gaussian"], inf["gaussian"])

    def _make_outfile(self) -> None:                                   # :443-475
        import cv2
        self.outfiles += 1
        if self.outfiles > 1 and self.outfile is not None:
            self.outfile.release()
        outname = str(self.filename) + '_' + str(self.outfiles)
        if self.outdir == '':
            self.outfile_name = outname + '_motion.avi'
        else:
            self.outfile_name = os.path.join(self.outdir, os.path.basename(outname)) + '_motion.avi'
        self.outfile = cv2.VideoWriter(self.outfile_name, cv2.VideoWriter_fourcc(*self.codec), self.fps,
                                       (self.frame_width, self.frame_height))

    def output_raw_frame(self, frame: np.ndarray = None) -> None:      # :533-546 (and :509-530 without show)
        if not self.wrote_frames:
            self._make_outfile()
            self.wrote_frames = True
        try:
            self.outfile.write(frame)
        except Exception as e:
            self.log.warning('Having to create output file due to exception: {}'.format(e))
            self._make_outfile()
            self.outfile.write(frame)
        self.frames_written += 1

    def is_open(self) -> bool:
        return self.cap.isOpened()

    def cleanup(self) -> None:                                         # :907-926
        if getattr(self, 'cap', None) is not None and not hasattr(self.filename, 'read'):
            self.cap.release()
        if self.outfile is not None:
            self.outfile.release()
        if self.engine is not None and self._own_engine:
            self.engine.close()
        self.engine = None

    # -- main loop ----------------------------------------------------------------------------------
    def _replay(self, raws, stats) -> None:
        """decide_output's actions on the raw frames, in frame order (find_motion.py:549-589).  `raws` may be views
        of a staging buffer that is about to be reused: frames that go into the cache are copied (the reference
        copies every frame, find_motion.py:236), frames that are written are written from where they lie."""
        for raw, st in zip(raws, stats):
            self.movement = bool(st["movement"])
            self.movement_counter = int(st["movement_counter"])
            self.movement_decay = int(st["movement_decay"])
            if st["wrote"]:
                if st["n_flush"]:
                    assert int(st["n_flush"]) == len(self.frame_cache), "frame cache out of step with the device"
                    for cached in self.frame_cache:
                        self.output_raw_frame(cached)
                    self.frame_cache.clear()
                self.output_raw_frame(raw)
            elif self.cache_frames > 0:
                self.frame_cache.append(raw.copy() if self._copy_cached else raw)
            assert len(self.frame_cache) == int(st["cache_len"]), "frame cache out of step with the device"

    _copy_cached = True

    def read_chunk(self, dst: np.ndarray) -> int:
        """Decode up to len(dst) frames into dst ([n, H, W, 3] uint8, e.g. a slice of a pinned batch); returns
        the number read (fewer than len(dst) = end of stream).  find_motion.py:497-506."""
        n = 0
        shape = (self.frame_height, self.frame_width, 3)
        while n < len(dst):
            if self._cv_capture:
                ret, frame = self.cap.read(dst[n])                   # decoded straight into the batch when cv2 can
            else:
                ret, frame = self.cap.read()
            if not ret:
                break
            if frame.shape != shape or frame.dtype != np.uint8:
                raise VideoError('frame geometry changed mid-stream: {}'.format(frame.shape))
            if frame.ctypes.data != dst[n].ctypes.data:
                dst[n] = frame
            n += 1
        self.frames_read += n
        return n

    def find_motion(self) -> tuple:
        """Main loop (find_motion.py:852-904): returns (wrote_frames, err_msg, seen_objects)."""
        if self.engine is None:
            raise VideoError('this stream is a slot of a batched context: drive it through find_motion_b200.jobs')
        shape = (1, self.chunk, self.frame_height, self.frame_width, 3)
        bufs = [PinnedBatch(shape, self.device) for _ in range(3)]
        try:
            pending = None                                            # (slot, host buffer, frames) of the batch in flight
            i = 0
            while True:
                host = bufs[i % 3].array
                n = self.read_chunk(host[0]) if self.is_open() else 0
                if n:
                    self.engine.submit_host(i & 1, host[:, :n])
                if pending is not None:                               # replay batch i-1 while batch i is on the GPU
                    pslot, phost, pn = pending
                    self._replay(phost[0, :pn], self.engine.wait_host(pslot)[0])
                pending = (i & 1, host, n) if n else None
                if n < self.chunk:
                    break
                i += 1
            if pending is not None:
                pslot, phost, pn = pending
                self._replay(phost[0, :pn], self.engine.wait_host(pslot)[0])
        finally:
            self.cleanup()
            for b in bufs:
                b.free()
        return self.wrote_frames, self.err_msg, tuple(self.seen_objects)


def run_vid(filename: typing.Union[str, int], **kwargs) -> tuple:
    """find_motion.py:1021-1037: the job `run()` binds with functools.partial."""
    seen_objects = None
    try:
        vid = VideoMotion(filename=filename, **kwargs)
        if vid.loaded:
            wrote_frames, err_msg, seen_objects = vid.find_motion()
        else:
            wrote_frames = None
            seen_objects = None
            err_msg = 'Video did not load successfully'
    except Exception as e:
        err_msg = 'Error processing video {}: {}'.format(filename, e)
        wrote_frames = None
    return (wrote_frames, filename, err_msg, seen_objects)
