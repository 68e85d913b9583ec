"""Job scheduling on B200s: the replacement of the reference's one-process-per-stream fan-out
(run_pool / run_map / run_stream, find_motion/find_motion.py:1054-1210).

The reference starts `multiprocessing.Pool(processes)` and gives every file (or camera) to a worker
process that runs `job(filename)` = `run_vid(filename, **tuning)` (fm.py:1071-1075, 1174-1177,
1323-1331).  Here the same `job` (a functools.partial carrying the tuning keywords) is taken apart
and the streams are batched instead: inputs of equal geometry share ONE context of `streams`
slots per GPU (libfmgpu.so processes the slots of a context in one launch), one driver thread per
GPU pulls files from a shared queue as slots fall free (the dynamic assignment a Pool gives), and
per batch of `chunk` frames per slot

    decode batch i+1 (host threads, straight into pinned memory next to the GPU)
    H2D + kernels of batch i (fm_submit_host: copy stream + compute stream)
    replay decide_output of batch i-1 on the raw frames (cache / flush / write, fm.py:549-589)

run concurrently.  Streams of different lengths make ragged batches (n_valid per slot); a slot is
reset (fm_submit_reset) and handed to the next file when its stream ends.  The result contract is
the reference's: one `(wrote_frames, filename, err_msg, seen_objects)` tuple per input, progress-log
lines `"<filename> // <seen_objects>"` for the successful ones (fm.py:1105-1106, 1151-1152).
There is no data-path collective: streams are independent (SURVEY.md 8e).
"""
from __future__ import annotations

import functools
import logging
import queue
import threading
import time
import typing
from concurrent.futures import ThreadPoolExecutor

from . import engine as _engine
from .engine import MotionEngine, PinnedBatch
from .video_motion import VideoMotion

log = logging.getLogger("find_motion")

# find_motion.py:124: workers wait on this Event once per frame when multiprocess (fm.py:858-860); here the
# drivers wait on it once per batch.  Set = running.
unpaused = threading.Event()
unpaused.set()

ENGINE_KEYS = ("fps", "box_size", "min_box_scale", "cache_time", "min_time", "threshold", "avg", "blur_scale")


def _job_kwargs(job) -> dict:
    """The tuning keywords `run()` bound into the job with functools.partial (fm.py:1323-1331)."""
    kw = dict(getattr(job, "keywords", None) or {})
    return kw


def visible_devices() -> typing.List[int]:
    import torch
    return list(range(torch.cuda.device_count()))


def _open_stream(filename, kw, stream_cls) -> typing.Tuple[typing.Optional[VideoMotion], typing.Optional[tuple]]:
    """VideoMotion(filename, **kw) without an engine of its own; mirrors run_vid's error handling (fm.py:1025-1037)."""
    try:
        vid = stream_cls(filename=filename, engine=False, **kw)
    except Exception as e:
        return None, (None, filename, 'Error processing video {}: {}'.format(filename, e), None)
    if not vid.loaded:
        try:
            vid.cleanup()
        except Exception:
            pass
        return None, (None, filename, 'Video did not load successfully', None)
    return vid, None


class _GroupDriver:
    """One GPU, one geometry: S slots, three pinned host batches, two device slots."""

    def __init__(self, device, geom, kw, streams, chunk, source_q, results, stream_cls, max_latency=None,
                 engine_factory=None, buffer_factory=None):
        factory = engine_factory or MotionEngine
        if factory is _engine.MotionEngine:
            # the reference upscales frames narrower than box_size (imutils.resize): so does the library's engine
            factory = functools.partial(factory, upscale=True)
        self.engine_factory = factory
        self.buffer_factory = buffer_factory or PinnedBatch
        self.device, self.geom, self.kw = device, geom, kw
        self.S, self.T = streams, chunk
        self.q, self.results, self.stream_cls = source_q, results, stream_cls
        self.max_latency = max_latency
        self.first: typing.List[VideoMotion] = []        # streams opened by the scheduler while probing

    def _finish(self, vid: VideoMotion, err: str = '') -> None:
        try:
            vid.cleanup()
        except Exception as e:           # a failing release must not lose the result
            err = err or str(e)
        if err:
            self.results.put((None, vid.filename, 'Error processing video {}: {}'.format(vid.filename, err), None))
        else:
            self.results.put((vid.wrote_frames, vid.filename, vid.err_msg, tuple(vid.seen_objects)))

    def _next_stream(self) -> typing.Optional[VideoMotion]:
        while True:
            if self.first:
                return self.first.pop()
            try:
                filename = self.q.get_nowait()
            except queue.Empty:
                return None
            vid, err = _open_stream(filename, self.kw, self.stream_cls)
            if err is not None:
                self.results.put(err)
                continue
            if (vid.frame_width, vid.frame_height) != self.geom:
                # another geometry: back to the scheduler (it opens a context of that shape later)
                vid.cleanup()
                self.requeue(filename, (vid.frame_width, vid.frame_height))
                continue
            return vid

    def requeue(self, filename, geom):      # replaced by the scheduler
        raise NotImplementedError

    def run(self) -> None:
        W, H = self.geom
        S, T = self.S, self.T
        ekw = {k: self.kw[k] for k in ENGINE_KEYS if k in self.kw}
        eng = self.engine_factory(W, H, n_streams=S, max_frames=T, device=self.device,
                                  mask_areas=self.kw.get("mask_areas"), **ekw)
        bufs = [self.buffer_factory((S, T, H, W, 3), self.device) for _ in range(3)]
        pool = ThreadPoolExecutor(max_workers=2 * S)
        slots: typing.List[typing.Optional[VideoMotion]] = [None] * S
        pending = None            # (device slot, host batch, [(s, vid, n, ended)]) of the batch on the GPU
        i = 0

        def read(vid: VideoMotion, dst, deadline):
            # bounded latency for live sources: stop filling the batch at the deadline (ragged batch)
            if deadline is None:
                return vid.read_chunk(dst)
            n = 0
            while n < len(dst) and (n == 0 or time.monotonic() < deadline):
                if vid.read_chunk(dst[n:n + 1]) == 0:
                    break
                n += 1
            return n

        def start_replay(batch):
            pslot, phost, entries = batch
            stats = eng.wait_host(pslot)
            return [pool.submit(self._replay_one, vid, phost[s, :n], stats[s, :n], ended) for s, vid, n, ended in entries]

        try:
            while True:
                unpaused.wait()
                for s in range(S):                       # free slots take the next inputs
                    if slots[s] is None:
                        vid = self._next_stream()
                        if vid is None:
                            break
                        vid._adopt_info(eng.info)
                        eng.submit_reset(s)              # ordered after the batches already submitted
                        slots[s] = vid
                active = [s for s in range(S) if slots[s] is not None]
                if not active:
                    break
                # decode batch i (one thread per slot) while batch i-1 is replayed (its kernels are done or about to be)
                host = bufs[i % 3].array
                deadline = time.monotonic() + self.max_latency if self.max_latency else None
                futs = {s: pool.submit(read, slots[s], host[s], deadline) for s in active}
                replays = start_replay(pending) if pending is not None else []
                pending = None
                n_valid = [0] * S
                entries = []
                for s in active:
                    vid = slots[s]
                    try:
                        n = futs[s].result()
                    except Exception as e:               # decode error: the stream ends here, like run_vid's except
                        for f in replays:
                            f.result()
                        replays = []
                        self._finish(vid, str(e))
                        slots[s] = None
                        continue
                    ended = (n < T and deadline is None) or n == 0 or not vid.is_open()
                    n_valid[s] = n
                    entries.append((s, vid, n, ended))
                    if ended:
                        slots[s] = None                  # the device slot is free from the next batch on
                if any(n_valid):
                    eng.submit_host(i & 1, host, n_valid)
                for f in replays:
                    f.result()
                if any(n_valid):
                    pending = (i & 1, host, entries)
                    i += 1
                else:
                    for s, vid, n, ended in entries:
                        if ended:
                            self._finish(vid)
            if pending is not None:
                for f in start_replay(pending):
                    f.result()
        finally:
            for vid in slots:
                if vid is not None:
                    self._finish(vid, 'interrupted')
            pool.shutdown(wait=True)
            eng.close()
            for b in bufs:
                b.free()

    def _replay_one(self, vid: VideoMotion, raws, stats, ended: bool) -> None:
        err = ''
        try:
            vid._replay(raws, stats)
        except Exception as e:
            err = str(e)
        if ended or err:
            self._finish(vid, err)


class BatchScheduler:
    """Files / cameras -> geometry groups -> one _GroupDriver per (GPU, geometry), run by one thread per GPU."""

    def __init__(self, job, devices=None, streams=8, chunk=16, stream_cls=None, max_latency=None,
                 engine_factory=None, buffer_factory=None):
        self.engine_factory, self.buffer_factory = engine_factory, buffer_factory
        self.kw = _job_kwargs(job)
        for k in ("device", "chunk", "engine"):
            self.kw.pop(k, None)
        self.devices = list(devices) if devices is not None else visible_devices()
        if not self.devices:
            raise RuntimeError("no CUDA device (there is no CPU fallback)")
        self.streams, self.chunk = int(streams), int(chunk)
        self.stream_cls, self.max_latency = stream_cls or VideoMotion, max_latency

    def run(self, sources, on_result=None) -> list:
        """Process every source; returns the result tuples in completion order."""
        sources = list(sources)
        results: "queue.Queue[tuple]" = queue.Queue()
        out: typing.List[tuple] = []
        failures: typing.List[BaseException] = []
        groups: typing.Dict[tuple, "queue.Queue"] = {}
        lock = threading.Lock()
        pending_q: "queue.Queue" = queue.Queue()
        for f in sources:
            pending_q.put(f)

        def drain():
            while True:
                try:
                    r = results.get_nowait()
                except queue.Empty:
                    return
                out.append(r)
                if on_result:
                    on_result(r)

        def worker(device):
            # each GPU thread: take an unseen source to learn a geometry, then drive that geometry until the shared
            # queue has no more sources of it; sources of other shapes are parked for a later context
            while True:
                geom, q, first = None, None, None
                with lock:
                    for g, gq in groups.items():
                        if not gq.empty():
                            geom, q = g, gq
                            break
                if geom is None:
                    try:
                        filename = pending_q.get_nowait()
                    except queue.Empty:
                        return
                    vid, err = _open_stream(filename, self.kw, self.stream_cls)
                    if err is not None:
                        results.put(err)
                        continue
                    geom, first = (vid.frame_width, vid.frame_height), vid
                    q = pending_q
                drv = _GroupDriver(device, geom, self.kw, self.streams, self.chunk, q, results, self.stream_cls,
                                   self.max_latency, self.engine_factory, self.buffer_factory)
                if first is not None:
                    drv.first.append(first)

                def requeue(filename, g):
                    with lock:
                        groups.setdefault(g, queue.Queue()).put(filename)
                drv.requeue = requeue
                try:
                    drv.run()
                except Exception as e:           # e.g. the context could not be created: loud, not a silent skip
                    log.error('GPU {} driver failed: {}'.format(device, e))
                    for vid in drv.first:
                        results.put((None, vid.filename, 'Error processing video {}: {}'.format(vid.filename, e), None))
                    failures.append(e)
                    return

        threads = [threading.Thread(target=worker, args=(d,), name=f"fm-gpu{d}", daemon=True) for d in self.devices]
        for t in threads:
            t.start()
        while any(t.is_alive() for t in threads):
            drain()
            time.sleep(0.02)
        for t in threads:
            t.join()
        drain()
        if failures:
            raise failures[0]
        return out


class _NoBar:
    def update(self, n):
        pass


def _report(progress_log, on_done):
    state = {"done": 0, "err": 0, "wrote": 0}

    def cb(res):
        wrote_frames, filename, err_msg, seen_objects = res
        state["done"] += 1
        log.debug('Done {}{}'.format(filename, '' if wrote_frames else ' (no output)'))
        if err_msg:
            log.error('Error processing {}: {}'.format(filename, err_msg))
            log.debug('Saw objects: {}'.format(seen_objects))
            state["err"] += 1
        elif progress_log is not None:
            print("{} // {}".format(filename, seen_objects), file=progress_log)       # fm.py:1105-1106
        if wrote_frames:
            state["wrote"] += 1
        on_done(state["done"])
    return cb, state


def run_pool(job: typing.Callable[..., typing.Any], processes: int, files: typing.Iterable[str] = None,
             pbar=None, progress_log: typing.IO[str] = None, *, devices=None, streams: int = None,
             chunk: int = 16) -> list:
    """find_motion.py:1054-1122.  `processes` (the reference's worker count) is the number of streams in flight:
    they are spread over the visible GPUs as slots of batched contexts instead of OS processes."""
    if not files:
        raise ValueError('More than 0 files needed')
    files = list(files)
    devices = list(devices) if devices is not None else visible_devices()
    if streams is None:
        streams = max(1, min(16, -(-max(int(processes), 1) // max(len(devices), 1))))
    pbar = pbar if pbar is not None else _NoBar()
    cb, state = _report(progress_log, pbar.update)
    try:
        out = BatchScheduler(job, devices, streams, chunk).run(files, cb)
        log.debug("All processes completed. {} errors, wrote {} files".format(state["err"], state["wrote"]))
        return out
    except KeyboardInterrupt:
        log.warning('Ending processing at user request')
        return []


def run_map(job: typing.Callable, files: typing.Iterable[str], pbar=None, progress_log: typing.IO[str] = None, *,
            device: int = 0, chunk: int = 16) -> list:
    """find_motion.py:1125-1155: files one by one (one stream in flight, on one GPU), results in input order."""
    if not files:
        raise ValueError('More than 0 files needed')
    log.debug('Processing each file one-by-one')
    pbar = pbar if pbar is not None else _NoBar()
    cb, _ = _report(progress_log, pbar.update)
    out = []
    try:
        for f in files:
            out += BatchScheduler(job, [device], 1, chunk).run([f], cb)
    except KeyboardInterrupt:
        log.warning('Ending processing at user request')
    return out


def run_stream(job: typing.Callable, processes: int, cameras: typing.List[int], progress_log: typing.IO[str] = None, *,
               devices=None, chunk: int = 2, max_latency: float = 0.25) -> list:
    """find_motion.py:1158-1210: live sources.  Small batches and a deadline per batch bound the latency between a
    frame being captured and its decision: a batch closes when every camera delivered `chunk` frames or
    `max_latency` seconds after it was opened, whichever comes first (ragged batch)."""
    if not cameras:
        raise ValueError('More than 0 cameras needed')
    cameras = list(cameras)
    log.debug('Cameras: {}'.format(cameras))
    devices = list(devices) if devices is not None else visible_devices()
    streams = max(1, -(-len(cameras) // max(len(devices), 1)))

    def cb(res):
        status, stream, err_msg, seen_objects = res
        log.debug('Done {}{}'.format(stream, '' if status else ' (no output)'))
        if err_msg:
            log.error('Ended processing camera {}: {}'.format(stream, err_msg))
            log.debug('Saw objects: {}'.format(seen_objects))
        print('Finished streaming from camera {}'.format(stream), file=progress_log)       # fm.py:1200
    try:
        return BatchScheduler(job, devices, streams, chunk, max_latency=max_latency).run(cameras, cb)
    except KeyboardInterrupt:
        log.warning('Ending processing at user request')
        return []
