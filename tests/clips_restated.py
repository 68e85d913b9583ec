"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the device-side look-back cache (FM_FLAG_DEVICE_CLIPS,
csrc/k_clips.cu): which frames fm_process_clip writes, from where, and which frames each call stores into the ring.

The invariant it rests on (SURVEY.md A.9, oracle.restated.Decision): a write with a non-empty cache always flushes it,
and the cache only grows while nothing is written, so the cache always holds the last `cache_len` frames of the
stream, consecutive, ending at the current frame.  A ring of C = cache_frames slots per stream, indexed by absolute
frame number mod C, therefore replaces the reference's deque(maxlen=C).  Checked by tests/test_clips_plan.py; the
GPU tests map these frame ids back to the synthetic frames.

Frame ids are absolute per-stream frame numbers: frame t of a call is `base + t`, and `base` advances by the
stream's valid frame count.
"""
from __future__ import annotations


def schedule(stats, n_valid, base, C):
    """One call of one stream.  stats: per-frame records (mappings with "wrote", "n_flush", "cache_len") of at least
    n_valid frames; base: the stream's frame counter before the call; C: cache_frames.

    Returns (gather, store, new_base):
      gather  [(src, id)] in output order, src = ("in", t) for input frame t of the call or ("ring", slot);
      store   [(t, slot)] input frames the call leaves in the ring, applied after every gather;
      new_base = base + n_valid.
    """
    gather = []
    for t in range(n_valid):
        r = stats[t]
        nf = int(r["n_flush"])
        for j in range(nf):
            b = base + t - nf + j
            gather.append((("in", b - base) if b >= base else ("ring", b % C), b))
        if int(r["wrote"]):
            gather.append((("in", t), base + t))
    store = []
    if n_valid > 0 and C > 0:
        m = min(int(stats[n_valid - 1]["cache_len"]), n_valid)
        store = [(t, (base + t) % C) for t in range(n_valid - m, n_valid)]
    return gather, store, base + n_valid


class RingSim:
    """Ring of frame ids of one stream (what the device ring holds), driven call by call by `schedule`."""

    def __init__(self, C):
        self.C = C
        self.slots = [None] * C
        self.base = 0

    def call(self, stats, n_valid, stores_first=False):
        """-> the frame ids the call writes, in order.  stores_first applies the stores before the gathers (the
        wrong order, kept so that a test can show it matters)."""
        gather, store, new_base = schedule(stats, n_valid, self.base, self.C)
        ids_in = [self.base + t for t in range(n_valid)]

        def do_store():
            for t, slot in store:
                self.slots[slot] = ids_in[t]

        if stores_first:
            do_store()
        out = [ids_in[src[1]] if src[0] == "in" else self.slots[src[1]] for src, _ in gather]
        if not stores_first:
            do_store()
        self.base = new_base
        return out


class DequeReplay:
    """The reference's frame cache as a deque(maxlen=C) of frame ids, replaying the per-frame records."""

    def __init__(self, C):
        from collections import deque
        self.C = C
        self.cache = deque(maxlen=C) if C > 0 else None
        self.next_id = 0

    def reset(self):
        if self.cache is not None:
            self.cache.clear()

    def frame(self, rec):
        fid = self.next_id
        self.next_id += 1
        out = []
        if int(rec["wrote"]):
            if int(rec["n_flush"]):
                assert len(self.cache) == int(rec["n_flush"])
                out += list(self.cache)
                self.cache.clear()
            out.append(fid)
        elif self.cache is not None:
            self.cache.append(fid)
        return out
