"""Designed motion planes for the contour stage as fm_process runs it (CPU only: numpy, scipy; no GPU import).

With k = 1 (blur_scale >= box_size / 1.99...), a black first frame and frame t painted as 255 * P_t in every channel, the
threshold bits the front ends produce are known without running an image pipeline:
  avg = 0: the background stays the black first frame, so raw_t = P_t for any threshold in [0, 254];
  avg = 1: the background becomes the previous frame, so raw_t = P_t xor P_(t-1);
  threshold = 255: no bit is ever set.
Masked pixels are painted black into the blurred plane, so raw_t loses the mask in both modes.  The designed planes are
therefore the raw planes themselves: `Painter` turns them into the planes to paint, the encoders into BGR, NV12 or
default-mode frames, and `replay` gives what every valid frame must produce: the 5x5-dilated plane, the sorted contour
records, the true contour count and the decision counters.  Every front end fed the same raw planes must produce the same
outputs, so `expected_plane` is computed once per distinct plane.

`labelling` restates which labelling path k_morph_ccl.cu takes for a frame (shared-memory tables or the global-memory
fallback, window rows cached in shared memory or read from L2), so that a scenario can assert that it reaches the path it
claims to test.
"""
from __future__ import annotations

import hashlib
from dataclasses import dataclass, field

import numpy as np

from oracle import restated as R

CCL2_CAP = 4096                  # runs of one polarity the shared-memory tables hold (k_morph_ccl.cu)
TILE_PX = 512                    # pixels of one k_temporal tile (FM_TILE_PX)


# ---------------------------------------------------------------------------------------------------------------------
# the labelling path of a frame (k_morph_ccl.cu: ccl_smem_plan, ccl_window, ccl_frame_lanes, fm_launch_morph_ccl)
# ---------------------------------------------------------------------------------------------------------------------
def smem_cache_words(h: int, wpr: int):
    """Words of the shared-memory row cache of k_ccl_frame_smem, or None when the plane has no shared-memory plan."""
    tables = 2 * h * 8 + 2 * (CCL2_CAP + 2) * 4 + 6 * CCL2_CAP * 2
    budget = 200 * 1024
    if wpr > 128 or tables + 4096 > budget:
        return None
    return min(budget - tables, 128 * 1024) // 4


def _runs(rows: np.ndarray) -> int:
    """Number of runs of True in the rows of a 2-D bool array."""
    if rows.size == 0:
        return 0
    return int((np.diff(rows.astype(np.int8), axis=1, prepend=0) == 1).sum())


def _filled(fg: np.ndarray) -> np.ndarray:
    """Foreground with its holes filled (background 4-connected to the outside removed)."""
    from scipy import ndimage
    h, w = fg.shape
    pad = np.zeros((h + 2, w + 2), bool)
    pad[1:-1, 1:-1] = fg
    lab, _ = ndimage.label(~pad, structure=np.array([[0, 1, 0], [1, 1, 1], [0, 1, 0]], bool))
    return (lab != lab[0, 0])[1:-1, 1:-1]


def labelling(dil: np.ndarray):
    """The window k_ccl_frame_smem labels for the dilated plane `dil` and the runs it holds.  Returns None for a quiet
    frame, else a dict: rows (ylo, yhi), words (jlo, jhi), bg_runs / fg_runs in the window (background of the dilated
    plane, foreground of the hole-filled one), heavy (more runs of a polarity than CCL2_CAP: the global-memory
    k_ccl_frame labels the frame), cached (the window rows fit the shared-memory row cache), plan (the plane has a
    shared-memory plan at all)."""
    fg = dil != 0
    h, w = fg.shape
    wpr = (w + 31) // 32
    rows = np.flatnonzero(fg.any(axis=1))
    if rows.size == 0:
        return None
    cols = np.flatnonzero(fg.any(axis=0))
    jlo, jhi = int(cols[0]) // 32, int(cols[-1]) // 32
    ylo, yhi = max(int(rows[0]) - 1, 0), min(int(rows[-1]) + 1, h - 1)
    x0, x1 = 32 * jlo, min(w, 32 * (jhi + 1))
    win = fg[ylo:yhi + 1, x0:x1]
    bg_runs, fg_runs = _runs(~win), _runs(_filled(win))
    cw = smem_cache_words(h, wpr)
    nwords = jhi - jlo + 1
    return {"rows": (ylo, yhi), "words": (jlo, jhi), "bg_runs": bg_runs, "fg_runs": fg_runs,
            "heavy": max(bg_runs, fg_runs) > CCL2_CAP, "plan": cw is not None,
            "cached": cw is not None and (yhi - ylo + 1) * (nwords | 1) <= cw}


# ---------------------------------------------------------------------------------------------------------------------
# plane families (bool [h, w]; True = a raw threshold bit)
# ---------------------------------------------------------------------------------------------------------------------
def dots(h, w, pts):
    p = np.zeros((h, w), bool)
    for y, x in pts:
        p[y, x] = True
    return p


def edge_planes(h, w):
    """Single pixels on every edge: the four corners, row 0, row h-1, column 0, column w-1 (the last valid bit of a
    partial word when w % 32 != 0), (y, w-1) alone and (y+1, 0) alone (adjacent bits of the flat layout k_temporal
    writes), the four corners together, and, on planes narrower than a 512-pixel k_temporal tile, the last pixel of
    the tile that spans the most rows (its last row is the one the tile's range must report)."""
    y = h // 3
    out = {"corner_tl": dots(h, w, [(0, 0)]), "corner_tr": dots(h, w, [(0, w - 1)]),
           "corner_bl": dots(h, w, [(h - 1, 0)]), "corner_br": dots(h, w, [(h - 1, w - 1)]),
           "row_first": dots(h, w, [(0, w // 2)]), "row_last": dots(h, w, [(h - 1, w // 3)]),
           "col_first": dots(h, w, [(h // 2, 0)]), "col_last": dots(h, w, [(h // 2, w - 1)]),
           "row_end": dots(h, w, [(y, w - 1)]), "next_row_start": dots(h, w, [(y + 1, 0)]),
           "all_corners": dots(h, w, [(0, 0), (0, w - 1), (h - 1, 0), (h - 1, w - 1)])}
    if w < TILE_PX:
        N = w * h
        best = max(range(N // TILE_PX), key=lambda k: ((k * TILE_PX + TILE_PX - 1) // w - (k * TILE_PX) // w, -k),
                   default=None)
        if best is not None:
            i = best * TILE_PX + TILE_PX - 1
            if i // w + 2 < h:                      # its dilation reaches two rows further down
                out["tile_end"] = dots(h, w, [(i // w, i % w)])
    return out


def _outline(p, y0, x0, y1, x1):
    """1-px rectangle outline with corners (y0, x0), (y1, x1) (after the 5x5 dilation a ring 5 px thick)."""
    p[y0, x0:x1 + 1] = True
    p[y1, x0:x1 + 1] = True
    p[y0:y1 + 1, x0] = True
    p[y0:y1 + 1, x1] = True


def topology_planes(h, w):
    """Window topology (needs h >= 38 and w >= 160): U shapes open to the image border and to the window's first and
    last word column, a ring with a dot, nested rings (with a dot), and a ring whose dilation spans exactly whole word
    columns (it touches the window's first and last word column)."""
    assert h >= 38 and w >= 160, (h, w)
    cy = h // 2
    out = {}
    p = np.zeros((h, w), bool)                      # U open to the left image border, and one open upwards to row 0
    p[cy - 8, 0:20] = p[cy + 8, 0:20] = True
    p[cy - 8:cy + 9, 20] = True
    p[0:14, 40] = p[0:14, 60] = True
    p[14, 40:61] = True
    out["u_border"] = p
    p = np.zeros((h, w), bool)                      # U open to the right; its arms end at the window's last bit
    x1 = 32 * 4 + 29                                # dilated to 32 * 4 + 31
    p[cy - 8, 66:x1 + 1] = p[cy + 8, 66:x1 + 1] = True
    p[cy - 8:cy + 9, 66] = True                     # dilated from 64: the window's first bit
    out["u_window_right"] = p
    p = np.zeros((h, w), bool)                      # U open to the left at the window's first word column
    p[cy - 8, 66:120] = p[cy + 8, 66:120] = True
    p[cy - 8:cy + 9, 120] = True
    out["u_window_left"] = p
    p = np.zeros((h, w), bool)
    _outline(p, cy - 7, 70, cy + 7, 84)
    p[cy, 77] = True
    out["ring_dot"] = p
    p = np.zeros((h, w), bool)
    _outline(p, cy - 15, 40, cy + 15, 70)
    _outline(p, cy - 7, 48, cy + 7, 62)
    p[cy, 55] = True
    out["nested_rings"] = p
    p = np.zeros((h, w), bool)
    _outline(p, cy - 8, 32 * 2 + 2, cy + 8, 32 * 3 + 29)      # dilated: x 64 .. 127, words 2 .. 3 exactly
    out["ring_word_edges"] = p
    return out


def corner_planes(h, w):
    """One component in the top-left corner (a small window) against two in opposite corners (the whole plane)."""
    one = np.zeros((h, w), bool)
    one[1:4, 1:4] = True
    two = one.copy()
    two[h - 4:h - 1, w - 4:w - 1] = True
    return {"corner_one": one, "corners_two": two}


def comb(h, w, y0, y1, x0=0, x1=None, step=6):
    """Vertical 1-px lines `step` px apart in rows [y0, y1), columns [x0, x1): after the dilation 5-px bars with 1-px
    gaps, about (x1 - x0) / step runs of each polarity per row."""
    p = np.zeros((h, w), bool)
    p[y0:y1, x0:x1:step] = True
    return p


def random_plane(h, w, density, seed):
    return np.random.default_rng(seed).random((h, w)) < density


def grid_dots(h, w, n, step=8, y0=2, x0=2):
    """n isolated dots (n components after the dilation), row by row."""
    pts = []
    for y in range(y0, h - 2, step):
        for x in range(x0, w - 2, step):
            if len(pts) < n:
                pts.append((y, x))
    assert len(pts) == n, (h, w, n)
    return dots(h, w, pts)


def one_frame_plane(h, w, y):
    """A 3 x 5 blob whose lowest row is y (use y % 4 == 3: the last row of a 4-row warp group of k_fused)."""
    p = np.zeros((h, w), bool)
    p[y - 2:y + 1, w // 2:w // 2 + 5] = True
    return p


# ---------------------------------------------------------------------------------------------------------------------
# encoders
# ---------------------------------------------------------------------------------------------------------------------
def encode_bgr(P):
    return np.repeat((P.astype(np.uint8) * 255)[..., None], 3, axis=2)


def encode_nv12(P):
    """Y = 255 P, U = V = 128 (cv2's COLOR_YUV2BGR_NV12 gives gray 255 and 0)."""
    h, w = P.shape
    out = np.full((h * 3 // 2, w), 128, np.uint8)
    out[:h] = P.astype(np.uint8) * 255
    return out


def encode_area(P, f):
    """Default-mode frame at the integer ratio f: every plane pixel painted as its f x f footprint (INTER_AREA exact)."""
    return encode_bgr(np.repeat(np.repeat(P, f, axis=0), f, axis=1))


def encoder(kind, f=1):
    return {"bgr": encode_bgr, "nv12": encode_nv12, "area": lambda P: encode_area(P, f)}[kind]


class Painter:
    """The planes to paint for designed raw planes of one stream.  avg = 0: P_t = raw_t (the background stays black);
    avg = 1: P_t = P_(t-1) xor raw_t (the background is the previous frame)."""

    def __init__(self, h, w, avg):
        assert avg in (0, 1)
        self.avg = avg
        self.prev = np.zeros((h, w), bool)

    def reset(self):
        self.prev = np.zeros_like(self.prev)

    def paint(self, raw):
        P = raw.copy() if self.avg == 0 else self.prev ^ raw
        self.prev = P
        return P


# ---------------------------------------------------------------------------------------------------------------------
# expected outputs
# ---------------------------------------------------------------------------------------------------------------------
def components(dil: np.ndarray):
    """R.external_components of `dil`, computed on the bounding box of its set pixels (everything outside is background
    connected to the outside, so the records are those of the whole plane shifted by the box origin)."""
    ys, xs = np.flatnonzero(dil.any(axis=1)), np.flatnonzero(dil.any(axis=0))
    if ys.size == 0:
        return []
    y0, x0 = int(ys[0]), int(xs[0])
    sub = dil[y0:int(ys[-1]) + 1, x0:int(xs[-1]) + 1]
    return sorted((a, (x + x0, y + y0, bw, bh)) for a, (x, y, bw, bh) in R.external_components(sub))


_EXPECTED = {}


def expected_plane(raw: np.ndarray):
    """(dilated uint8 plane, sorted contour records) of one raw plane; computed once per distinct plane."""
    key = (raw.shape, hashlib.sha1(np.packbits(raw).tobytes()).hexdigest())
    if key not in _EXPECTED:
        dil = R.dilate5(raw.astype(np.uint8) * 255) if raw.any() else np.zeros(raw.shape, np.uint8)
        _EXPECTED[key] = (dil, components(dil))
    return _EXPECTED[key]


# ---------------------------------------------------------------------------------------------------------------------
# scenarios: a context configuration and a sequence of calls of designed raw planes
# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class Call:
    raws: list                      # [S][T]: a bool [h, w] plane or None (quiet)
    n_valid: tuple = None           # per stream, or None: all T frames
    fill: dict = field(default_factory=dict)     # (s, t) -> plane painted into a frame past n_valid (not processed)
    reset: tuple = ()               # streams reset before the call
    claims: dict = field(default_factory=dict)   # (s, t) -> set of labelling claims ("heavy", "smem", "cached", ...)

    @property
    def T(self):
        return len(self.raws[0])


@dataclass
class Scenario:
    name: str
    W: int
    H: int
    kind: str                       # "bgr", "nv12" or "area"
    S: int
    Tmax: int
    threshold: int
    avg: int
    calls: list
    box_size: int = None            # default: W (full resolution)
    engine: dict = field(default_factory=dict)   # extra MotionEngine arguments
    fps: int = 10
    min_time: float = 0.3
    cache_time: float = 0.5
    mask_areas: list = None
    max_components: int = 8192

    @property
    def box(self):
        return self.box_size or self.W

    @property
    def ratio(self):
        return self.W // self.box

    @property
    def hw(self):
        p = self.params()
        return p["h"], p["w"]

    def tuning(self):
        """MotionEngine / StreamOracle tuning: k = 1 (blur_scale = box_size)."""
        return dict(fps=self.fps, box_size=self.box, blur_scale=self.box, threshold=self.threshold, avg=float(self.avg),
                    min_time=self.min_time, cache_time=self.cache_time, mask_areas=self.mask_areas)

    def params(self):
        return R.derive_params(self.W, self.H, self.fps, self.box, 50, self.cache_time, self.min_time, self.box)

    def mask(self):
        h, w = self.hw
        return R.rasterise_masks(w, h, self.mask_areas, self.params()["scale"])


def frames(sc: Scenario):
    """The input batch of every call: uint8 [S, T, *frame_shape] (frames past n_valid hold the call's fill planes)."""
    h, w = sc.hw
    enc = encoder(sc.kind, sc.ratio)
    painters = [Painter(h, w, sc.avg) for _ in range(sc.S)]
    for c in sc.calls:
        for s in c.reset:
            painters[s].reset()
        nv = c.n_valid or (c.T,) * sc.S
        batch = None
        for s in range(sc.S):
            for t in range(c.T):
                if t < nv[s]:
                    raw = c.raws[s][t]
                    P = painters[s].paint(raw if raw is not None else np.zeros((h, w), bool))
                else:
                    P = c.fill.get((s, t), np.zeros((h, w), bool))
                fr = enc(P)
                if batch is None:
                    batch = np.empty((sc.S, c.T) + fr.shape, np.uint8)
                batch[s, t] = fr
        yield batch


@dataclass
class Frame:
    dil: np.ndarray
    comps: list
    stats: dict                     # the fm_frame_stats fields


def replay(sc: Scenario):
    """What every call must produce: per call, [S] lists of Frame for the valid frames, and per stream the expected
    float64 background after the call (None: the stream has not started)."""
    h, w = sc.hw
    p = sc.params()
    keep = ~sc.mask()
    decs = [R.Decision(p["min_area"], p["max_area"], p["cache_frames"], p["min_movement_frames"]) for _ in range(sc.S)]
    painters = [Painter(h, w, sc.avg) for _ in range(sc.S)]
    started = [False] * sc.S
    bgs = [None] * sc.S
    out = []
    for c in sc.calls:
        for s in c.reset:
            decs[s] = R.Decision(p["min_area"], p["max_area"], p["cache_frames"], p["min_movement_frames"])
            painters[s].reset()
            started[s] = False
        nv = c.n_valid or (c.T,) * sc.S
        res = []
        for s in range(sc.S):
            fr = []
            for t in range(nv[s]):
                raw = c.raws[s][t]
                raw = np.zeros((h, w), bool) if raw is None else raw
                if not started[s]:
                    assert not raw.any(), f"{sc.name}: the first frame of a stream must be black"
                    started[s] = True
                P = painters[s].paint(raw)
                eff = raw & keep if sc.threshold <= 254 else np.zeros_like(raw)
                dil, comps = expected_plane(eff)
                rec = decs[s].step([a for a, _ in comps])
                n_counted = sum(1 for a, _ in comps if not (p["max_area"] < a / 2.0 < p["min_area"]))
                fr.append(Frame(dil, comps, {
                    "n_contours": len(comps), "n_counted": n_counted, "movement": int(rec["movement"]),
                    "movement_counter": rec["counter"], "movement_decay": rec["decay"], "cache_len": rec["cache_len"],
                    "wrote": int(rec["wrote"]), "n_flush": rec["n_flush"]}))
                # avg = 0: the background stays the black first frame; avg = 1: it is the last (masked) frame
                bgs[s] = np.zeros((h, w)) if sc.avg == 0 else (P & keep) * 255.0
            res.append(fr)
        out.append((res, list(bgs)))
    return out


def contour_path(sc: Scenario, T: int):
    """The contour-stage path fm_launch_morph_ccl takes for a call of T frames: "smem_dilate" (k_ccl_frame_smem dilates
    the raw bits itself: F = S T >= 32), "k_dilate+smem" (F < 32) or "k_dilate+global" (no shared-memory plan)."""
    h, w = sc.hw
    if smem_cache_words(h, (w + 31) // 32) is None:
        return "k_dilate+global"
    return "smem_dilate" if sc.S * T >= 32 else "k_dilate+smem"


def check_claims(sc: Scenario):
    """Assert every labelling claim of the scenario's frames (so that no case silently stops testing what it claims)."""
    h, w = sc.hw
    keep = ~sc.mask()
    for i, c in enumerate(sc.calls):
        for (s, t), claims in c.claims.items():
            raw = c.raws[s][t]
            raw = np.zeros((h, w), bool) if raw is None else raw
            eff = raw & keep if sc.threshold <= 254 else np.zeros_like(raw)
            lab = labelling(expected_plane(eff)[0])
            where = (sc.name, i, s, t, claims, lab and {k: lab[k] for k in ("bg_runs", "fg_runs", "rows", "words")})
            for cl in claims:
                if cl == "quiet":
                    assert lab is None, where
                    continue
                assert lab is not None, where
                if cl == "heavy":
                    assert lab["plan"] and lab["heavy"], where
                elif cl == "smem":
                    assert lab["plan"] and not lab["heavy"], where
                elif cl == "cached":
                    assert lab["plan"] and not lab["heavy"] and lab["cached"], where
                elif cl == "uncached":
                    assert lab["plan"] and not lab["heavy"] and not lab["cached"], where
                elif cl == "clamped":
                    assert len(expected_plane(eff)[1]) > sc.max_components, where
                elif cl.startswith("touch:"):
                    side = cl[6:]
                    sl = {"top": eff[0], "bottom": eff[-1], "left": eff[:, 0], "right": eff[:, -1]}[side]
                    assert sl.any(), where
                else:
                    raise AssertionError(f"unknown claim {cl}")


# ---------------------------------------------------------------------------------------------------------------------
# the scenarios of tests/test_gpu_contour_stage.py
# ---------------------------------------------------------------------------------------------------------------------
def _seq(T, items, start=1):
    """[T] frame list: None (quiet) except items placed from frame `start` on (frame 0 stays black)."""
    out = [None] * T
    for i, p in enumerate(items):
        out[start + i] = p
    return out


def _fill(n_valid, T, plane):
    """The frames past n_valid, each holding `plane`."""
    return {(s, t): plane for s, nv in enumerate(n_valid) for t in range(nv, T)}


def _claims(call, s, start, tags):
    for i, tag in enumerate(tags):
        if tag:
            call.claims[(s, start + i)] = set(tag.split(","))


def _mixed_1080(name, kind, threshold, avg, engine=None):
    """1920 x 1080, two streams of 16 frames (F = 32: k_ccl_frame_smem dilates the raw bits itself, 60 words per row):
    a corner component (small cached window) against opposite corners (whole, uncached window), window topology,
    random planes straddling CCL2_CAP runs, combs, heavy / light / quiet frames mixed inside calls and across streams,
    and a ragged call whose frames past n_valid hold heavy planes."""
    h, w = 1080, 1920
    cor, top, edg = corner_planes(h, w), topology_planes(h, w), edge_planes(h, w)
    light, heavy = random_plane(h, w, 0.0002, 1), random_plane(h, w, 0.00035, 2)
    heavier = random_plane(h, w, 0.0005, 3)
    comb_l, comb_h = comb(h, w, 500, 512, 600, 1300), comb(h, w, 300, 360, 100, 1000)
    fill = {k: random_plane(h, w, 0.002, 10 + k) for k in range(11)}
    c0 = Call([_seq(16, [cor["corner_one"], cor["corners_two"], top["u_border"], top["u_window_right"],
                         top["u_window_left"], top["ring_dot"], top["nested_rings"], top["ring_word_edges"],
                         edg["all_corners"], edg["row_last"], edg["col_last"], None, light, None]),
               _seq(16, [light, heavy, comb_l, comb_h, None, heavier, None, None, edg["corner_br"], cor["corner_one"],
                         None, None, None, None])])
    _claims(c0, 0, 1, ["cached", "uncached", "cached,touch:left,touch:top", "cached", "cached", "cached", "cached",
                       "cached", "uncached,touch:top,touch:bottom", "touch:bottom", "touch:right", "quiet", "uncached"])
    _claims(c0, 1, 1, ["uncached", "heavy", "cached", "heavy", "quiet", "heavy"])
    c1 = Call([_seq(16, [heavy, None, cor["corners_two"], light, None, None, comb_h, None, None, top["ring_dot"],
                         None, None, None, None, None], start=0),
               _seq(16, [comb_h, None, light, heavier], start=0)],
              n_valid=(16, 5), fill={(1, t): fill[t - 5] for t in range(5, 16)})
    _claims(c1, 0, 0, ["heavy", "quiet", "uncached"])
    c2 = Call([_seq(16, [None, None, None, light, heavy, None, None, cor["corner_one"]], start=0),
               _seq(16, [None, cor["corners_two"], None, None, None, heavy, None, None, None, None, None, None, None,
                         None, None, comb_l], start=0)])
    return Scenario(name, w, h, kind, 2, 16, threshold, avg, [c0, c1, c2], engine=engine or {})


def _one_frame_index():
    """Motion in exactly one frame index per stream, quiet elsewhere: t in {0, 15, 16, 31} of a T = 32 call (k_fused's
    `hits` mask, one rawrange atomic per frame after the frame loop) and t in {31, 32, 33, 39} of a T = 40 call (the
    per-frame atomics), in the last row of a 4-row warp group; then the edges and the window topology, and a ragged
    call with a stream that takes no part (256 x 146: h % 4 == 2)."""
    h, w = 146, 256
    c0 = Call([[None] * 32 for _ in range(4)])
    c1 = Call([[one_frame_plane(h, w, 83) if t == ts else None for t in range(32)] for ts in (0, 15, 16, 31)])
    c2 = Call([[one_frame_plane(h, w, 123) if t == ts else None for t in range(40)] for ts in (31, 32, 33, 39)])
    edg, top = list(edge_planes(h, w).values()), list(topology_planes(h, w).values())
    c3 = Call([_seq(40, edg, start=0), _seq(40, top, start=3), _seq(40, edg[::-1] + top, start=5),
               _seq(40, top + edg, start=20)])
    hv = comb(h, w, 10, 140)
    c4 = Call([_seq(32, edg[:6], start=0), [None] * 32, _seq(32, top, start=8), _seq(32, [hv, None, hv], start=28)],
              n_valid=(32, 0, 17, 31), fill=_fill((32, 0, 17, 31), 32, hv))
    _claims(c4, 3, 28, ["heavy"])
    return Scenario("fused_256x146_one_frame_index", w, h, "bgr", 4, 40, 254, 1, [c0, c1, c2, c3, c4])


def _generic_200x75():
    """200 x 75 (w % 32 == 8, N % 16 == 8, h % 4 == 3): k_gray + k_blur_identity + k_temporal, and the unaligned
    (flat bit order) dilation inside k_ccl_frame_smem (F = 32); the last pixel of the 512-pixel k_temporal tile that
    spans four rows; more components than max_components (24)."""
    h, w = 75, 200
    edg, top = edge_planes(h, w), topology_planes(h, w)
    dense = random_plane(h, w, 0.01, 4)
    c0 = Call([_seq(16, list(edg.values()), start=1),
               _seq(16, list(top.values()) + [dense, grid_dots(h, w, 40), None, dense], start=1)])
    _claims(c0, 1, 7, ["clamped", "clamped"])
    c1 = Call([_seq(16, [edg["tile_end"], None, edg["corner_br"]], start=0), _seq(16, [top["ring_dot"]], start=0)],
              n_valid=(9, 3), fill=_fill((9, 3), 16, dense))
    c2 = Call([_seq(16, [edg["row_end"], edg["next_row_start"], None, edg["tile_end"]], start=0),
               _seq(16, [None, dense, None, edg["all_corners"]], start=0)])
    return Scenario("generic_200x75", w, h, "bgr", 2, 16, 0, 0, [c0, c1, c2], max_components=24)


def _generic_masked():
    """200 x 75, one stream of 8 frames (F < 32: k_dilate<false>), README_MASKS: motion in the masked top-left corner
    disappears."""
    from find_motion_b200 import synth
    h, w = 75, 200
    edg = edge_planes(h, w)
    inside = np.zeros((h, w), bool)
    inside[20:30, 20:40] = True                     # inside the square mask (0, 0) .. (100, 100)
    c0 = Call([_seq(8, [edg["corner_tl"], edg["all_corners"], inside, inside | edg["corner_br"], None, edg["col_last"],
                        edg["row_last"]])])
    _claims(c0, 0, 1, ["quiet", "touch:right", "quiet", "touch:bottom"])
    return Scenario("generic_200x75_masked", w, h, "bgr", 1, 8, 254, 1, [c0], mask_areas=synth.README_MASKS)


def _nofused_256x147():
    """256 x 147 with no_fused (aligned k_temporal), one stream of 8 frames (F < 32: k_dilate<true> + the shared-memory
    labelling, heavy frames to the global-memory fallback), h % 4 == 3."""
    h, w = 147, 256
    edg, top = list(edge_planes(h, w).values()), list(topology_planes(h, w).values())
    hv = comb(h, w, 5, 140)
    c0 = Call([_seq(8, edg[:7], start=1)])
    c1 = Call([_seq(8, edg[7:] + [hv], start=0)])
    c2 = Call([_seq(8, top + [hv, None], start=0)], n_valid=(7,), fill={(0, 7): hv})
    c3 = Call([_seq(8, [hv, None, hv, edg[0]], start=0)])
    _claims(c2, 0, 6, ["heavy"])
    return Scenario("nofused_256x147", w, h, "bgr", 1, 8, 0, 1, [c0, c1, c2, c3], engine=dict(no_fused=True))


def _area_320x242():
    """Default mode at the integer ratio 2 (320 x 242 -> 160 x 121, h % 4 == 1), k = 1."""
    h, w = 121, 160
    edg, top = list(edge_planes(h, w).values()), list(topology_planes(h, w).values())
    rnd = random_plane(h, w, 0.02, 5)
    c0 = Call([_seq(16, edg[:12] + [rnd], start=1), _seq(16, top + [rnd, None, rnd], start=1)])
    c1 = Call([_seq(16, edg[::-1], start=0), _seq(16, [rnd] + top, start=2)], n_valid=(16, 9),
              fill={(1, t): rnd for t in range(9, 16)})
    return Scenario("area_320x242", 320, 242, "area", 2, 16, 254, 1, [c0, c1], box_size=160)


def _wide_4096x38():
    """4096 x 38: 128 words per row (the widest plane with a shared-memory plan), F = 32, h % 4 == 2."""
    h, w = 38, 4096
    edg, top = list(edge_planes(h, w).values()), list(topology_planes(h, w).values())
    hv, lt = comb(h, w, 4, 34), random_plane(h, w, 0.004, 6)
    c0 = Call([_seq(16, edg + [hv, lt], start=1), _seq(16, [hv, None, lt] + top + [hv], start=1)])
    _claims(c0, 0, 12, ["heavy", "smem"])
    _claims(c0, 1, 1, ["heavy", "quiet", "smem"])
    c1 = Call([_seq(16, [lt, None, hv], start=0), _seq(16, edg, start=2)], n_valid=(16, 14),
              fill={(1, t): hv for t in range(14, 16)})
    return Scenario("fused_4096x38", w, h, "bgr", 2, 16, 0, 1, [c0, c1])


def _no_plan(name, w, h, S, T):
    """Planes without a shared-memory plan (129 words per row, or h >= 7424): k_dilate and the global-memory
    k_ccl_frame label every frame; more components than max_components (32)."""
    edg = list(edge_planes(h, w).values())
    rnd = random_plane(h, w, 0.01, 7)
    extra = [grid_dots(h, w, 60), rnd] + (list(topology_planes(h, w).values()) if w >= 160 and h >= 38 else [])
    calls = [Call([_seq(T, (edg + extra)[s::S][:T - 1], start=1) for s in range(S)])]
    calls.append(Call([_seq(T, (extra + edg)[s::S][:T], start=0) for s in range(S)]))
    return Scenario(name, w, h, "bgr", S, T, 254, 0, calls, max_components=32)


def _quiet_255():
    """threshold 255: no raw bit is ever set, whatever the frames hold."""
    h, w = 146, 256
    hv = comb(h, w, 10, 140)
    c0 = Call([_seq(8, [hv, random_plane(h, w, 0.05, 8), hv])])
    _claims(c0, 0, 1, ["quiet", "quiet", "quiet"])
    return Scenario("fused_256x146_threshold_255", w, h, "bgr", 1, 8, 255, 0, [c0, c0])


def chained_scenario():
    """Eight calls of 256 x 146, two streams of 16 frames on the fused path: heavy frames, border frames, resets and
    ragged calls."""
    h, w = 146, 256
    edg, top = list(edge_planes(h, w).values()), list(topology_planes(h, w).values())
    hv, rnd = comb(h, w, 10, 140), random_plane(h, w, 0.01, 9)
    calls = [Call([_seq(16, edg[:11]), _seq(16, top + [hv])]),
             Call([_seq(16, [hv, None, rnd], start=0), _seq(16, edg, start=4)]),
             Call([_seq(16, top, start=2), _seq(16, [None] * 3 + [rnd, hv], start=0)], n_valid=(16, 6),
                  fill={(1, t): hv for t in range(6, 16)}),
             Call([_seq(16, [None, hv] + edg[:5]), _seq(16, top, start=1)], reset=(1,)),
             Call([_seq(16, [rnd, rnd, None, hv], start=0), [None] * 16], n_valid=(4, 0), fill=_fill((4, 0), 16, hv)),
             Call([_seq(16, edg, start=0), _seq(16, [hv] + top, start=0)]),
             Call([_seq(16, [None] * 15), _seq(16, [rnd] * 3, start=10)], reset=(0,)),
             Call([_seq(16, top + [hv], start=0), _seq(16, edg[::-1], start=0)], n_valid=(16, 13),
                  fill={(1, t): rnd for t in range(13, 16)})]
    _claims(calls[0], 1, 7, ["heavy"])
    return Scenario("chained_256x146", w, h, "bgr", 2, 16, 254, 0, calls)


def scenarios():
    """Scenario builders by name: the contour paths (F >= 32 with the in-kernel dilation, aligned and not, up to 32, 64
    and 128 words per row; F < 32 with k_dilate; no shared-memory plan) through the front ends (fused BGR and NV12,
    generic, no_fused, default mode), with threshold 0 / 254 / 255 and avg 0 / 1."""
    return {
        "fused_bgr_1080": lambda: _mixed_1080("fused_bgr_1080", "bgr", 254, 0),
        "fused_nv12_1080": lambda: _mixed_1080("fused_nv12_1080", "nv12", 0, 1),
        "fused_256x146_one_frame_index": _one_frame_index,
        "generic_200x75": _generic_200x75,
        "generic_200x75_masked": _generic_masked,
        "nofused_256x147": _nofused_256x147,
        "area_320x242": _area_320x242,
        "fused_4096x38": _wide_4096x38,
        "no_plan_4128x48": lambda: _no_plan("no_plan_4128x48", 4128, 48, 2, 16),
        "no_plan_64x7440": lambda: _no_plan("no_plan_64x7440", 64, 7440, 1, 16),
        "fused_256x146_threshold_255": _quiet_255,
        "chained_256x146": chained_scenario,
    }
