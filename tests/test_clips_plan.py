"""CPU: the look-back cache of the reference (a deque of raw frames, find_motion.py:415, 561-570, 588) can live in a
ring of cache_frames slots per stream indexed by absolute frame number, and the per-call schedule of
tests/clips_restated.py (the one csrc/k_clips.cu implements) emits exactly the frames the deque would."""
import random

import pytest

from oracle import restated as R
from tests import clips_restated as CR

GRID = [(C, M) for C in (0, 1, 2, 3, 5, 30) for M in (0, 1, 2, 4, 15)]


def _records(C, M, counts):
    dec = R.Decision(min_area=0, max_area=10 ** 9, cache_frames=C, min_movement_frames=M)
    out = []
    for n in counts:
        r = dec.step([2] * n)
        out.append({"wrote": int(r["wrote"]), "n_flush": r["n_flush"], "cache_len": r["cache_len"]})
    return out


def _counts(rng, n, p_move):
    """Contour counts with runs of motion and quiet, so that caches fill, overflow and flush."""
    out, moving = [], False
    for _ in range(n):
        if rng.random() < 0.15:
            moving = not moving
        out.append(rng.choice((1, 1, 2, 3)) if (moving and rng.random() < p_move) else 0)
    return out


@pytest.mark.parametrize("C,M", GRID)
def test_cache_is_last_frames_consecutive(C, M):
    """Invariant: the deque, as explicit frame ids, always holds the last cache_len ids, ending at the current one."""
    rng = random.Random(1000 * C + M)
    for trial in range(20):
        counts = _counts(rng, 300, rng.choice((0.3, 0.7, 1.0)))
        replay = CR.DequeReplay(C)
        for t, rec in enumerate(_records(C, M, counts)):
            replay.frame(rec)
            cache = list(replay.cache) if replay.cache is not None else []
            assert len(cache) == rec["cache_len"], (trial, t)
            assert cache == list(range(t + 1 - len(cache), t + 1)), (trial, t, cache)


def _run_calls(C, M, counts, calls, resets=(), stores_first=False):
    """calls: list of (T, n_valid).  Returns (ids from the ring schedule, ids from the deque replay), call by call."""
    dec = R.Decision(min_area=0, max_area=10 ** 9, cache_frames=C, min_movement_frames=M)
    ring, replay = CR.RingSim(C), CR.DequeReplay(C)
    got, want, k = [], [], 0
    for ci, (T, nv) in enumerate(calls):
        if ci in resets:                                   # fm_ctx_reset / fm_submit_reset: counters and cache
            dec.counter = dec.decay = dec.cache_len = 0
            replay.reset()
        recs = []
        for t in range(nv):
            r = dec.step([2] * counts[k])
            k += 1
            recs.append({"wrote": int(r["wrote"]), "n_flush": r["n_flush"], "cache_len": r["cache_len"]})
        recs += [{"wrote": 0, "n_flush": 0, "cache_len": 0}] * (T - nv)     # the device zeroes frames past n_valid
        got.append(ring.call(recs, nv, stores_first=stores_first))
        want.append([i for rec in recs[:nv] for i in replay.frame(rec)])
    return got, want


@pytest.mark.parametrize("C,M", GRID)
@pytest.mark.parametrize("T", [1, 2, 7, 16, 40])
def test_ring_schedule_matches_deque(C, M, T):
    rng = random.Random(C * 7919 + M * 104729 + T)
    for trial in range(8):
        calls = [(T, T if rng.random() < 0.6 else rng.randint(0, T)) for _ in range(30)]
        counts = _counts(rng, sum(nv for _, nv in calls), rng.choice((0.3, 0.8)))
        resets = {i for i in range(1, len(calls)) if rng.random() < 0.08}
        got, want = _run_calls(C, M, counts, calls, resets)
        assert got == want, (trial, C, M, T)


def test_flushes_reach_back_across_calls():
    """C = 30 > T = 16: a flush takes frames of the two calls before."""
    counts = [0] * 40 + [1] + [0] * 7
    got, want = _run_calls(30, 1, counts, [(16, 16)] * 3)
    assert got == want
    assert got[2][:31] == list(range(10, 41)), got[2]
    assert min(got[2]) < 16                          # two calls back


def test_several_flushes_and_overflow_in_one_call():
    """C = 3, T = 32: the cache overflows inside the call, and three episodes flush in it."""
    counts = [0] * 8 + [1] + [0] * 9 + [1] + [0] * 5 + [1] + [0] * 7
    got, want = _run_calls(3, 1, counts, [(32, 32)])
    assert got == want
    flushes = [g for g in got[0]]
    assert flushes[:4] == [5, 6, 7, 8]
    recs = _records(3, 1, counts)
    assert sum(1 for r in recs if r["n_flush"]) == 3


def test_gather_before_store_matters():
    """C = 3, min_movement_frames = 1, T = 7, a full cache at the start: motion at frame 1 flushes base-2 .. base
    (base-2, base-1 from the ring), frames 2-3 are written on decay, 4-6 are cached and go to the slots of base-2 and
    base-1.  Storing before gathering hands out the new frames instead of the old ones."""
    counts = [0] * 3 + [0, 1, 0, 0, 0, 0, 0]
    calls = [(3, 3), (7, 7)]
    got, want = _run_calls(3, 1, counts, calls)
    assert got == want == [[], [1, 2, 3, 4, 5, 6]]
    bad, _ = _run_calls(3, 1, counts, calls, stores_first=True)
    assert bad != want


def test_store_list():
    """The stores of a call are the frames still cached at its end that the ring does not hold yet, each in slot
    id mod C; base advances by the stream's valid frames only."""
    recs = _records(5, 2, [0, 0, 0, 0, 0, 0, 0])
    gather, store, nb = CR.schedule(recs, 3, base=10, C=5)
    assert gather == [] and store == [(0, 0), (1, 1), (2, 2)] and nb == 13
    recs2 = recs[3:]
    gather, store, nb = CR.schedule(recs2, 4, base=13, C=5)
    assert store == [(0, 3), (1, 4), (2, 0), (3, 1)] and nb == 17
    _, store, nb = CR.schedule(recs2, 0, base=17, C=5)
    assert store == [] and nb == 17
