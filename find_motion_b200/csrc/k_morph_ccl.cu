// Dilation, external-contour extraction and the per-frame decision logic on bit planes.
// Replaces VideoFrame.find_contours (cv2.dilate x2 + cv2.findContours RETR_EXTERNAL), the
// cv2.contourArea / boundingRect calls of find_movement, and the counters of find_movement /
// decide_output (find_motion/find_motion.py:260-276, 665-700, 549-589; SURVEY.md A.8, A.9).
//
// Contours are obtained without border following (SURVEY.md A.8):
//   O  = background 4-connected to the outside of the image
//   F  = not O  (foreground with its holes filled)
//   external contours <-> 8-connected components of F
//   contourArea = Q4 + Q3/2 over the 2x2 windows of the component (4 resp. 3 pixels set)
// Both labellings are run-based union-find with one warp per row: lanes hold the 32-bit words
// of the row, run starts/ends come from shifted-word logic and are enumerated with warp prefix
// sums, unions are lock-free atomicMin links between runs of adjacent rows.
#include "fm_common.cuh"

#define WARPS_PER_BLOCK 8

__device__ __forceinline__ uint32_t ld_word(const uint32_t *row, int j, int wpr) {
    return ((unsigned)j < (unsigned)wpr) ? __ldg(row + j) : 0u;
}

// ---------------------------------------------------------------------------------------------
// dilate: flat raw threshold bits -> row-padded 5x5-dilated bit plane (+ any flag)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t flat_row_word(const uint32_t *flat, int y, int j, int w, int h, int wpr) {
    // 32 pixels x = 32j .. 32j+31 of row y as a word (bits beyond w cleared)
    if ((unsigned)y >= (unsigned)h || (unsigned)j >= (unsigned)wpr) return 0u;
    long long b0 = (long long)y * w + 32 * j;
    int wi = (int)(b0 >> 5), sh = (int)(b0 & 31);
    uint32_t lo = __ldg(flat + wi);
    uint32_t v = lo;
    if (sh) {
        uint32_t hi = __ldg(flat + wi + 1);      // flat planes are padded by one tile
        v = __funnelshift_r(lo, hi, sh);
    }
    int rem = w - 32 * j;
    if (rem < 32) v &= (1u << rem) - 1u;
    return v;
}

// one row of the 5x5 dilation (two iterations of the 3x3 default kernel, out-of-image pixels ignored): lanes hold the
// words of the row; returns the OR of the lane's words and the lane's first / last non-empty word column
template <bool ALIGNED>
__device__ __forceinline__ uint32_t dilate_vor(const uint32_t *__restrict__ flat, int y, int j, int w, int h, int wpr) {
    // OR of word j over rows y-2 .. y+2 (rows outside the image ignored)
    uint32_t v = 0;
    if (j >= wpr) return 0u;
#pragma unroll
    for (int dy = -2; dy <= 2; dy++) {
        const int yy = y + dy;
        if (ALIGNED) {                  // w % 32 == 0: flat order == row-padded order
            if ((unsigned)yy < (unsigned)h) v |= __ldcg(flat + (size_t)yy * wpr + j);
        } else {
            v |= flat_row_word(flat, yy, j, w, h, wpr);
        }
    }
    return v;
}

template <bool ALIGNED>
__device__ __forceinline__ uint32_t dilate_row(const uint32_t *__restrict__ flat, uint32_t *__restrict__ out, int y, int w,
                                               int h, int wpr, int lane, int &jmin, int &jmax) {
    // vertical OR first (5 loads per word), then the horizontal +-2 from the neighbouring lanes' words
    uint32_t anyw = 0, vprev = 0, vc = dilate_vor<ALIGNED>(flat, y, lane, w, h, wpr);
    for (int j0 = 0; j0 < wpr; j0 += 32) {
        const int j = j0 + lane;
        const uint32_t vnext = dilate_vor<ALIGNED>(flat, y, j + 32, w, h, wpr);
        uint32_t vm = __shfl_up_sync(0xffffffffu, vc, 1), vp = __shfl_down_sync(0xffffffffu, vc, 1);
        const uint32_t pl = __shfl_sync(0xffffffffu, vprev, 31), nf = __shfl_sync(0xffffffffu, vnext, 0);
        if (lane == 0) vm = pl;
        if (lane == 31) vp = nf;
        if (j < wpr) {
            uint32_t d = vc | (vc << 1) | (vc << 2) | (vc >> 1) | (vc >> 2) | (vm >> 31) | (vm >> 30) | (vp << 31) | (vp << 30);
            const int rem = w - 32 * j;
            if (rem < 32) d &= (1u << rem) - 1u;
            out[j] = d;
            anyw |= d;
            if (d) { jmax = max(jmax, j); jmin = min(jmin, j); }      // a lane walks several words and (in the labelling kernel) several rows
        }
        vprev = vc;
        vc = vnext;
    }
    return anyw;
}

// The same dilation for a BLOCK of consecutive rows [ya, yb) walked by one warp: the vertical OR slides (one new row per
// step instead of five loads), the raw rows of the next four steps are requested before the current four are combined
// (the steps of a row block would otherwise pay one L2 round trip each), and all word columns of a lane (NCH = words per
// row / 32, rounded up) are carried together so that the +-2 pixel neighbours come from registers.
template <bool ALIGNED, int NCH>
__device__ __noinline__ void dilate_rows(const uint32_t *flat, uint32_t *dplane, int ya, int yb, int w, int h, int wpr, int lane,
                                            int &jmin, int &jmax, int &ymn, int &ymx) {
    auto raw = [&](int y, int c) -> uint32_t {
        const int j = lane + 32 * c;
        if ((unsigned)y >= (unsigned)h || j >= wpr) return 0u;
        return ALIGNED ? __ldcg(flat + (size_t)y * wpr + j) : flat_row_word(flat, y, j, w, h, wpr);
    };
    uint32_t win[NCH][4];            // raw rows y-2 .. y+1 of the row about to be produced
#pragma unroll
    for (int c = 0; c < NCH; c++)
#pragma unroll
        for (int i = 0; i < 4; i++) win[c][i] = raw(ya - 2 + i, c);
    for (int y0 = ya; y0 < yb; y0 += 4) {
        uint32_t nxt[NCH][4];        // raw rows y0+2 .. y0+5: the new row of each of the next four steps
#pragma unroll
        for (int c = 0; c < NCH; c++)
#pragma unroll
            for (int i = 0; i < 4; i++) nxt[c][i] = raw(y0 + 2 + i, c);
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int y = y0 + i;
            if (y >= yb) break;
            uint32_t v[NCH];
#pragma unroll
            for (int c = 0; c < NCH; c++) {
                v[c] = win[c][0] | win[c][1] | win[c][2] | win[c][3] | nxt[c][i];
                win[c][0] = win[c][1]; win[c][1] = win[c][2]; win[c][2] = win[c][3]; win[c][3] = nxt[c][i];
            }
            uint32_t anyw = 0;
#pragma unroll
            for (int c = 0; c < NCH; c++) {
                uint32_t vm = __shfl_up_sync(0xffffffffu, v[c], 1), vp = __shfl_down_sync(0xffffffffu, v[c], 1);
                const uint32_t pl = c > 0 ? __shfl_sync(0xffffffffu, v[c > 0 ? c - 1 : 0], 31) : 0u;
                const uint32_t nf = c + 1 < NCH ? __shfl_sync(0xffffffffu, v[c + 1 < NCH ? c + 1 : c], 0) : 0u;
                if (lane == 0) vm = pl;
                if (lane == 31) vp = nf;
                const int j = lane + 32 * c;
                if (j < wpr) {
                    uint32_t d = v[c] | (v[c] << 1) | (v[c] << 2) | (v[c] >> 1) | (v[c] >> 2) | (vm >> 31) | (vm >> 30) | (vp << 31) | (vp << 30);
                    const int rem = w - 32 * j;
                    if (rem < 32) d &= (1u << rem) - 1u;
                    dplane[(size_t)y * wpr + j] = d;
                    anyw |= d;
                    if (d) { jmax = max(jmax, j); jmin = min(jmin, j); }
                }
            }
            if (__any_sync(0xffffffffu, anyw != 0)) { ymx = max(ymx, y); ymn = min(ymn, y); }
        }
    }
}

// rowrange[4f] = max y with a set pixel (-1: none), [4f+1] = max (h-1-y), [4f+2] = max word column j with a set
// pixel, [4f+3] = max (wpr-1-j)   (memset 0xFF before)
template <bool ALIGNED>
__global__ void __launch_bounds__(32 * WARPS_PER_BLOCK) k_dilate(const uint32_t *__restrict__ tflat,
                                                                 uint32_t *__restrict__ dil, int *__restrict__ rowrange,
                                                                 const int *__restrict__ rawrange, int F, int w, int h,
                                                                 int wpr, int flatwords, int T, int t0, int Th,
                                                                 unsigned long long *stamp) {
    fm_stamp_start(stamp);
    // F = S*Th local frames: local frame lf is frame t0 + lf % Th of stream lf / Th, stored at s*T + t
    int warp = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
    int lane = threadIdx.x & 31;
    if (warp >= F * h) return;
    int lf = warp / h, y = warp - lf * h;
    int f = (lf / Th) * T + t0 + lf % Th;
    if (rawrange) {      // rows further than 2 from any pixel above threshold stay untouched (nobody reads them)
        int rmax = rawrange[2 * f], rmin = h - 1 - rawrange[2 * f + 1];
        if (rmax < 0 || y < rmin - 3 || y > rmax + 3) return;   // +-2 for the dilation, +-1 for the zero rows the labelling reads
    }
    const uint32_t *flat = tflat + (size_t)f * flatwords;
    uint32_t *out = dil + ((size_t)f * h + y) * wpr;
    int jmax = -1, jmin = wpr;
    const uint32_t anyw = dilate_row<ALIGNED>(flat, out, y, w, h, wpr, lane, jmin, jmax);
    if (__any_sync(0xffffffffu, anyw != 0)) {
        jmax = __reduce_max_sync(0xffffffffu, jmax);
        jmin = __reduce_min_sync(0xffffffffu, jmin);
        if (lane == 0) {
            atomicMax(rowrange + 4 * f, y);
            atomicMax(rowrange + 4 * f + 1, h - 1 - y);
            atomicMax(rowrange + 4 * f + 2, jmax);
            atomicMax(rowrange + 4 * f + 3, wpr - 1 - jmin);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// run extraction
// ---------------------------------------------------------------------------------------------
struct CclArgs {
    const uint32_t *plane;     // [F][h][wpr] dilated bit plane
    uint32_t *fill;            // [F][h][wpr] dilated plane with holes filled (written by the kernel)
    const int *rowrange;       // [F][4] from k_dilate (NULL: label every row and column of every frame)
    const uint32_t *raw;       // [F][flatwords] raw threshold bits: the shared-memory kernel dilates them into `plane`
    const int *rawrange;       //   itself (rows of [F][2] rawrange +- 3) and writes the ranges to `rangeout`;
    int *rangeout;             //   NULL: `plane` is already dilated
    uint32_t *planeout;
    int flatwords, aligned;
    int cache_words;           // shared-memory words available for staging the window rows
    int f0, nf;                // local frames [f0, f0+nf) of the range are in this sub-batch
    int T, t0, Th;             // local frame l -> stream l / Th, frame t0 + l % Th, stored at s*T + t
    int w, h, wpr, cap;
    size_t slots;
    uint16_t *xs, *xe;
    int *rowcnt, *parent, *area2, *bbox;
    int *errflag;
    int *ncomp, *ncounted;     // [F]
    fm_component *comps;       // [F][maxc]
    int maxc, min_area, max_area;
    unsigned long long *stamp; // contour-stage stamps of the call (null: timing off): &stamps[2]
};

// INVERT: runs of zeros (background pass).  Planes written earlier in the same kernel are read
// with ld.global.cg (L2), never through the non-coherent path.
template <bool INVERT>
__device__ __forceinline__ uint32_t plane_word(const uint32_t *row, int j, int w, int wpr) {
    if ((unsigned)j >= (unsigned)wpr) return 0u;
    uint32_t v = __ldcg(row + j);
    if (INVERT) {
        v = ~v;
        int rem = w - 32 * j;
        if (rem < 32) v &= (1u << rem) - 1u;
    }
    return v;
}

template <bool INVERT>
__device__ __forceinline__ void runs_row(const CclArgs &a, const uint32_t *plane, int lf, int f, int y, int lane) {
    const uint32_t *row = plane + ((size_t)f * a.h + y) * a.wpr;
    size_t base = (size_t)lf * a.slots + (size_t)y * a.cap;
    int *parent = a.parent + (size_t)lf * (a.slots + 1);
    int nstart = 0, nend = 0;
    for (int j0 = 0; j0 < a.wpr; j0 += 32) {
        int j = j0 + lane;
        uint32_t B = plane_word<INVERT>(row, j, a.w, a.wpr);
        uint32_t Bp = plane_word<INVERT>(row, j - 1, a.w, a.wpr);
        uint32_t Bn = plane_word<INVERT>(row, j + 1, a.w, a.wpr);
        uint32_t S = B & ~((B << 1) | (Bp >> 31));
        uint32_t E = B & ~((B >> 1) | (Bn << 31));
        if (!__any_sync(0xffffffffu, (S | E) != 0)) continue;      // no run starts or ends in these 1024 pixels
        int cs = __popc(S), ce = __popc(E);
        int ps = cs, pe = ce;     // inclusive warp scans
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int vs = __shfl_up_sync(0xffffffffu, ps, o);
            int ve = __shfl_up_sync(0xffffffffu, pe, o);
            if (lane >= o) { ps += vs; pe += ve; }
        }
        int is = nstart + ps - cs, ie = nend + pe - ce;
        while (S) {
            int bit = __ffs(S) - 1;
            S &= S - 1;
            if (is < a.cap) {
                a.xs[base + is] = (uint16_t)(32 * j + bit);
                parent[1 + (size_t)y * a.cap + is] = 1 + y * a.cap + is;
                a.area2[base + is] = 0;
                int *bb = a.bbox + (base + is) * 4;
                bb[0] = 0x7fffffff; bb[1] = 0x7fffffff; bb[2] = -1; bb[3] = -1;
            }
            is++;
        }
        while (E) {
            int bit = __ffs(E) - 1;
            E &= E - 1;
            if (ie < a.cap) a.xe[base + ie] = (uint16_t)(32 * j + bit);
            ie++;
        }
        nstart += __shfl_sync(0xffffffffu, ps, 31);
        nend += __shfl_sync(0xffffffffu, pe, 31);
    }
    if (lane == 0) {
        if (nstart > a.cap) { atomicExch(a.errflag, 1); nstart = a.cap; }
        a.rowcnt[(size_t)lf * a.h + y] = nstart;
    }
}

// ---------------------------------------------------------------------------------------------
// union-find on run ids (id 0 = outside, run (y, i) = 1 + y*cap + i); roots are minimal ids
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int uf_find(const int *parent, int x) {
    int p = __ldcg(parent + x);
    while (p != x) {
        x = p;
        p = __ldcg(parent + x);
    }
    return x;
}

// find with path halving: every visited node is re-pointed at its grandparent.  Links only ever
// decrease (atomicMin), so concurrent unions stay correct.
__device__ __forceinline__ int uf_find_compress(int *parent, int x) {
    int p = __ldcg(parent + x);
    while (p != x) {
        int gp = __ldcg(parent + p);
        if (gp != p) atomicMin(parent + x, gp);
        x = p;
        p = gp;
    }
    return x;
}

__device__ __forceinline__ void uf_union(int *parent, int a, int b) {
    while (true) {
        a = uf_find_compress(parent, a);
        b = uf_find_compress(parent, b);
        if (a == b) return;
        if (a < b) { int t = a; a = b; b = t; }
        int old = atomicMin(parent + a, b);
        if (old == a) return;
        a = old;
    }
}

// CONN8: runs of adjacent rows touch if their x ranges overlap after growing by one pixel.
// OUTSIDE: runs that touch the image border are linked to the outside node (background pass).
// ylo: first labelled row (runs of row ylo have no labelled predecessor row).
template <bool CONN8, bool OUTSIDE>
__device__ __forceinline__ void union_row(const CclArgs &a, int lf, int y, int ylo, int lane) {
    int n = a.rowcnt[(size_t)lf * a.h + y];
    if (n == 0) return;
    size_t base = (size_t)lf * a.slots + (size_t)y * a.cap;
    int *parent = a.parent + (size_t)lf * (a.slots + 1);
    int np = y > ylo ? a.rowcnt[(size_t)lf * a.h + y - 1] : 0;
    const uint16_t *pxs = a.xs + base - a.cap, *pxe = a.xe + base - a.cap;
    const int d = CONN8 ? 1 : 0;
    for (int i = lane; i < n; i += 32) {
        int xs = a.xs[base + i], xe = a.xe[base + i];
        int id = 1 + y * a.cap + i;
        if (OUTSIDE && (y == 0 || y == a.h - 1 || xs == 0 || xe == a.w - 1)) uf_union(parent, id, 0);
        if (np) {
            // first run of the previous row whose end reaches xs - d
            int lo = 0, hi = np;
            while (lo < hi) {
                int mid = (lo + hi) >> 1;
                if ((int)pxe[mid] < xs - d) lo = mid + 1; else hi = mid;
            }
            for (int q = lo; q < np && (int)pxs[q] <= xe + d; q++) uf_union(parent, id, 1 + (y - 1) * a.cap + q);
        }
    }
}

// background pass epilogue: F = plane | (background runs not connected to the outside)
__device__ __forceinline__ void fill_row(const CclArgs &a, int lf, int f, int y, int lane) {
    const uint32_t *row = a.plane + ((size_t)f * a.h + y) * a.wpr;
    uint32_t *out = a.fill + ((size_t)f * a.h + y) * a.wpr;
    for (int j = lane; j < a.wpr; j += 32) out[j] = __ldcg(row + j);
    __syncwarp();
    int n = a.rowcnt[(size_t)lf * a.h + y];
    size_t base = (size_t)lf * a.slots + (size_t)y * a.cap;
    const int *parent = a.parent + (size_t)lf * (a.slots + 1);
    for (int i = lane; i < n; i += 32) {
        if (uf_find(parent, 1 + y * a.cap + i) == 0) continue;
        int xs = a.xs[base + i], xe = a.xe[base + i];
        for (int j = xs >> 5; j <= (xe >> 5); j++) {
            int lo = max(xs - 32 * j, 0), hi = min(xe - 32 * j, 31);
            uint32_t m = (hi == 31 ? 0xffffffffu : ((1u << (hi + 1)) - 1u)) & ~((1u << lo) - 1u);
            atomicOr(out + j, m);
        }
    }
}

// per run: bit-quad area contribution (windows whose lower row is y) and bounding box -> root
__device__ __forceinline__ void stats_row(const CclArgs &a, int lf, int f, int y, int lane) {
    int n = a.rowcnt[(size_t)lf * a.h + y];
    if (n == 0) return;
    size_t base = (size_t)lf * a.slots + (size_t)y * a.cap;
    const int *parent = a.parent + (size_t)lf * (a.slots + 1);
    const uint32_t *up = a.fill + ((size_t)f * a.h + (y > 0 ? y - 1 : 0)) * a.wpr;   // row y-1 (unused for y == 0)
    for (int i = lane; i < n; i += 32) {
        int xs = a.xs[base + i], xe = a.xe[base + i];
        int root = uf_find(parent, 1 + y * a.cap + i) - 1;
        int q = 0;
        if (y > 0) {
            // windows x in [xs, xe-1] have both lower pixels set: count upper pairs
            if (xe > xs) {
                int x0 = xs, x1 = xe - 1;
                for (int j = x0 >> 5; j <= (x1 >> 5); j++) {
                    uint32_t U = plane_word<false>(up, j, a.w, a.wpr), Un = plane_word<false>(up, j + 1, a.w, a.wpr);
                    uint32_t Us = (U >> 1) | (Un << 31);            // bit i = pixel x+1
                    int lo = max(x0 - 32 * j, 0), hi = min(x1 - 32 * j, 31);
                    uint32_t m = (hi == 31 ? 0xffffffffu : ((1u << (hi + 1)) - 1u)) & ~((1u << lo) - 1u);
                    q += 2 * __popc(U & Us & m) + __popc((U ^ Us) & m);
                }
            }
            // windows x = xs-1 (lower 0,1) and x = xe (lower 1,0): need both upper pixels
            auto ubit = [&](int x) -> uint32_t {
                if (x < 0 || x >= a.w) return 0u;
                return (__ldcg(up + (x >> 5)) >> (x & 31)) & 1u;
            };
            q += (int)(ubit(xs - 1) & ubit(xs)) + (int)(ubit(xe) & ubit(xe + 1));
        }
        size_t r = (size_t)lf * a.slots + root;
        if (q) atomicAdd(a.area2 + r, q);
        int *bb = a.bbox + r * 4;
        atomicMin(bb + 0, xs);
        atomicMin(bb + 1, y);
        atomicMax(bb + 2, xe);
        atomicMax(bb + 3, y);
    }
}

__device__ __forceinline__ void collect_row(const CclArgs &a, int lf, int f, int y, int lane) {
    int n = a.rowcnt[(size_t)lf * a.h + y];
    size_t base = (size_t)lf * a.slots + (size_t)y * a.cap;
    const int *parent = a.parent + (size_t)lf * (a.slots + 1);
    for (int i = lane; i < n; i += 32) {
        int id = 1 + y * a.cap + i;
        if (__ldcg(parent + id) != id) continue;
        int area2 = __ldcg(a.area2 + base + i);
        const int *bb = a.bbox + (base + i) * 4;
        int slot = atomicAdd(a.ncomp + f, 1);
        // find_motion.py:684  `if self.max_area < area < self.min_area: continue`  (area = area2/2)
        bool skipped = (2LL * a.max_area < area2) && (area2 < 2LL * a.min_area);
        if (!skipped) atomicAdd(a.ncounted + f, 1);
        if (slot < a.maxc) {
            fm_component c;
            c.area_x2 = area2;
            int x0 = __ldcg(bb), y0 = __ldcg(bb + 1), x1 = __ldcg(bb + 2), y1 = __ldcg(bb + 3);
            c.x = x0; c.y = y0; c.w = x1 - x0 + 1; c.h = y1 - y0 + 1;
            a.comps[(size_t)f * a.maxc + slot] = c;
        }
    }
}

// One CTA labels one frame: seven row-parallel phases separated by block barriers (all traffic
// between phases goes through L2: atomics and ld.global.cg).  Only the rows around the set
// pixels are visited; quiet frames exit at once.
#define CCL_THREADS 1024
// all CCL_THREADS threads of the CTA; rows [ylo, yhi] of frame f (scratch slot lf)
__device__ __forceinline__ void ccl_frame_global(const CclArgs &a, int lf, int f, int ylo, int yhi) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = CCL_THREADS / 32;
    if (threadIdx.x == 0) a.parent[(size_t)lf * (a.slots + 1)] = 0;      // the outside node
    // pass 1: background runs, 4-connected, linked to the outside -> holes
    for (int y = ylo + warp; y <= yhi; y += nw) runs_row<true>(a, a.plane, lf, f, y, lane);
    __syncthreads();
    for (int y = ylo + warp; y <= yhi; y += nw) union_row<false, true>(a, lf, y, ylo, lane);
    __syncthreads();
    for (int y = ylo + warp; y <= yhi; y += nw) fill_row(a, lf, f, y, lane);
    __syncthreads();
    // pass 2: hole-filled foreground, 8-connected
    for (int y = ylo + warp; y <= yhi; y += nw) runs_row<false>(a, a.fill, lf, f, y, lane);
    __syncthreads();
    for (int y = ylo + warp; y <= yhi; y += nw) union_row<true, false>(a, lf, y, ylo, lane);
    __syncthreads();
    for (int y = ylo + warp; y <= yhi; y += nw) stats_row(a, lf, f, y, lane);
    __syncthreads();
    for (int y = ylo + warp; y <= yhi; y += nw) collect_row(a, lf, f, y, lane);
}

// decision state machine of one stream over the frames of the call (SURVEY.md A.9; find_motion.py:665-700, 549-589)
struct DecideArgs {
    StreamState *state;
    fm_frame_stats *stats, *stats_out;
    const int *nvalid;
    int *done;                 // frames labelled so far in this call (cleared with the counters)
    unsigned long long *stamp; // contour-stage stamps of the call (null: timing off): &stamps[2]
    int S, T, total, cache_frames, min_movement_frames;
};

__device__ __forceinline__ void decide_stream(const DecideArgs &d, const int *ncomp, const int *ncounted, int s) {
    StreamState st = d.state[s];
    const int T = d.T;
    const int Ts = min(T, d.nvalid[s]);           // real frames of this stream in the call (ragged batches)
    for (int t = Ts; t < T; t++) {
        fm_frame_stats z = {0, 0, 0, 0, 0, 0, 0, 0};
        d.stats[s * T + t] = z;
        if (d.stats_out) d.stats_out[s * T + t] = z;
    }
    if (Ts <= 0) return;                        // the stream did not take part: state untouched
    for (int tc = 0; tc < Ts; tc += 16) {
        // the counts of 16 frames first (independent loads: one L2 round trip per chunk instead of one per frame)
        int nco[16], ncd[16];
#pragma unroll
        for (int i = 0; i < 16; i++) {
            const bool in = tc + i < Ts;
            nco[i] = in ? __ldcg(ncomp + s * T + tc + i) : 0;
            ncd[i] = in ? __ldcg(ncounted + s * T + tc + i) : 0;
        }
#pragma unroll
        for (int i = 0; i < 16; i++) {
            if (tc + i >= Ts) break;
            const int f = s * T + tc + i;
            fm_frame_stats r;
            r.n_contours = nco[i];
            r.n_counted = ncd[i];
            if (st.decay > 0) st.decay -= 1;                       // find_motion.py:672
            bool movement = r.n_counted > 0;
            st.counter = movement ? st.counter + r.n_counted : 0;   // :694 per contour, :697-698
            r.wrote = 0;
            r.n_flush = 0;
            if (st.counter >= d.min_movement_frames || st.decay > 0) {   // :555
                if (movement) {
                    st.decay = d.cache_frames;                      // :559
                    r.n_flush = st.cache_len;                       // :561-570
                    st.cache_len = 0;
                }
                r.wrote = 1;                                        // :583
            } else {
                st.cache_len = min(st.cache_len + 1, d.cache_frames); // deque(maxlen), :415, :588
            }
            r.movement = movement ? 1 : 0;
            r.movement_counter = st.counter;
            r.movement_decay = st.decay;
            r.cache_len = st.cache_len;
            d.stats[f] = r;
            if (d.stats_out) d.stats_out[f] = r;
        }
    }
    st.has_bg = 1;
    d.state[s] = st;
}

// decisions of the call, one thread per stream (measured: a "last CTA done" tail inside the labelling kernel and an in-kernel
// call of the global-memory fallback made the labelling kernel 15 us slower than these two tiny extra launches cost)
// The contour stage is a chain of programmatic dependent launches (fm_launch_chained): each kernel lets the next one
// start at its entry and waits for its predecessor before its first read of it, so the next call's fused front end can
// take the SMs this stage leaves idle (see fused_exit in k_fused.cu).
__global__ void k_decide(DecideArgs d, const int *__restrict__ ncomp, const int *__restrict__ ncounted) {
    fm_launch_dependents();
    fm_wait_predecessor();
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < d.S) decide_stream(d, ncomp, ncounted, s);
    fm_stamp_end(d.stamp);                            // the last kernel of the stage: its end is the stage's
}

// One CTA per frame, or, as the fallback of k_ccl_frame_smem (heavy != null), CCL_FALLBACK_CTAS CTAs that take the frames
// in turn: the fallback is a programmatic dependent of k_ccl_frame_smem, and a CTA waiting for it holds a whole SM
// (1024 threads x 56 registers), so one CTA per frame would take every SM the labelling kernel leaves free, and the next
// call's front end, further down the chain, could not start before the labelling kernel ends.
#define CCL_FALLBACK_CTAS 16
__global__ void __launch_bounds__(CCL_THREADS, 1) k_ccl_frame(CclArgs a, const int *__restrict__ heavy) {
    fm_launch_dependents();
    fm_stamp_start(a.stamp);
    fm_wait_predecessor();
    for (int lf = blockIdx.x; lf < a.nf; lf += gridDim.x) {
        const int lg = a.f0 + lf, f = (lg / a.Th) * a.T + a.t0 + lg % a.Th;
        if (heavy && !heavy[f]) continue;           // already labelled by k_ccl_frame_smem
        int ylo = 0, yhi = a.h - 1;
        bool work = true;
        if (a.rowrange) {
            int ymax = a.rowrange[4 * f], ymin = a.h - 1 - a.rowrange[4 * f + 1];
            if (ymax < 0) work = false;             // no set pixel in this frame
            ylo = max(ymin - 1, 0);
            yhi = min(ymax + 1, a.h - 1);
        }
        if (work) ccl_frame_global(a, lf, f, ylo, yhi);     // scratch slot lf: frames share nothing
    }
}

// ---------------------------------------------------------------------------------------------
// K2: the same labelling with the run tables and the union-find forests in SHARED memory, one CTA per frame.
// Frames whose active rows hold more than CCL2_CAP runs (or planes wider than 4096 px) are flagged "heavy" and
// left to k_ccl_frame.  The kernel works on the window of rows and word columns that holds the motion (background
// touching a window edge is connected to the outside exactly as background touching the image border is: there is
// no foreground beyond the window to enclose it), staged into shared memory when it fits:
//   row extraction     one row per lane (a lane walks the words of its row; rows hold a handful of runs, so
//                      spreading one row over a warp would idle most lanes); slots in row order by a CTA-wide scan
//   unions             one thread per run: first partner by plain store (ids grow with the row, so the link points
//                      to a smaller id and nobody chases pointers while 1000 rows build their chains concurrently),
//                      pointer-jumping flatten, remaining partners by lock-free union, flatten
//   holes              background runs whose root is not the outside are OR-ed into the plane (in place)
//   statistics         one thread per run: bit-quad area over the run's 2x2 windows, bounding box -> root
// ---------------------------------------------------------------------------------------------
#define CCL2_THREADS 1024
#define CCL2_WARPS (CCL2_THREADS / 32)
#define CCL2_CAP 4096

struct RunTable {
    int2 *row;        // [rows] (first slot, run count) of each row
    int *parent;      // [CCL2_CAP + 1]; for the background table id 0 = outside
    uint16_t *xs, *xe;
    uint16_t *rowof;  // [CCL2_CAP] window row of each run
};

__device__ __forceinline__ int suf_find(int *parent, int x) {
    int p = parent[x];
    while (p != x) {
        int gp = parent[p];
        if (gp != p) atomicMin(parent + x, gp);      // path halving
        x = p;
        p = gp;
    }
    return x;
}

__device__ __forceinline__ void suf_union(int *parent, int a, int b) {
    while (true) {
        a = suf_find(parent, a);
        b = suf_find(parent, b);
        if (a == b) return;
        if (a < b) { int t = a; a = b; b = t; }
        int old = atomicMin(parent + a, b);
        if (old == a) return;
        a = old;
    }
}

template <bool INVERT>
__device__ __forceinline__ uint32_t win_word(const uint32_t *row, int j, int ww, int wprw) {
    if ((unsigned)j >= (unsigned)wprw) return 0u;
    uint32_t v = row[j];
    if (INVERT) {
        v = ~v;
        const int rem = ww - 32 * j;
        if (rem < 32) v &= (1u << rem) - 1u;
    }
    return v;
}

// Runs of rows [r0, r0 + 1024) -> run table, one row per thread: count pass, CTA-wide prefix sum (slots are handed
// out in ROW ORDER, so run ids grow with the row and a link "run -> run of the row above" always points to a
// smaller id), emit pass.  Returns false when the table is full.  Called by all threads of the CTA.
template <bool INVERT>
__device__ __forceinline__ bool lane_extract(const uint32_t *row, bool act, int yr, int id0, const RunTable &t, int *cursor,
                                             int *wsum, int ww, int wprw) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int n = 0;
    if (act) {
        uint32_t carry = 0;
        for (int j = 0; j < wprw; j++) {
            const uint32_t B = win_word<INVERT>(row, j, ww, wprw);
            n += __popc(B & ~((B << 1) | carry));
            carry = B >> 31;
        }
    }
    int incl = n;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    const int wv = wsum[lane];                               // CCL2_WARPS == 32: one total per lane
    int winc = wv;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, winc, o);
        if (lane >= o) winc += v;
    }
    const int tot = __shfl_sync(0xffffffffu, winc, 31);
    const int wbase = __shfl_sync(0xffffffffu, winc - wv, warp);
    const int start = *cursor;
    const int off = start + wbase + incl - n;
    __syncthreads();                                         // everybody has read wsum and the cursor
    if (threadIdx.x == 0) *cursor = start + tot;
    if (act) t.row[yr] = make_int2(off, n);
    if (start + tot > CCL2_CAP) return false;
    if (act && n) {
        int is = off, ie = off;
        uint32_t carry = 0, B = win_word<INVERT>(row, 0, ww, wprw);
        for (int j = 0; j < wprw; j++) {
            const uint32_t Bn = win_word<INVERT>(row, j + 1, ww, wprw);
            uint32_t S = B & ~((B << 1) | carry), E = B & ~((B >> 1) | (Bn << 31));
            carry = B >> 31;
            while (S) {
                const int bit = __ffs(S) - 1;
                S &= S - 1;
                t.xs[is] = (uint16_t)(32 * j + bit);
                t.rowof[is] = (uint16_t)yr;
                t.parent[id0 + is] = id0 + is;
                is++;
            }
            while (E) {
                const int bit = __ffs(E) - 1;
                E &= E - 1;
                t.xe[ie++] = (uint16_t)(32 * j + bit);
            }
            B = Bn;
        }
    }
    return true;
}

// Unions of run i (one thread per run: rows with hundreds of runs -- noise at a fading edge -- must not serialise on
// one lane) with the outside (OUTSIDE: background touching the window / image border, id 0) and with the runs of the
// row above that it touches (binary search for the first one).
// FIRST pass: the run stores its first partner as its parent -- a plain store, nobody else writes the parent of
// this run in this pass, and the partner's id is smaller (row order), so no find and no pointer chasing while the
// chains are being built concurrently.  REST pass (after the forest has been flattened by pointer jumping): the
// remaining partners through the lock-free union, whose finds are now one step.  Returns true if it did a union.
template <bool CONN8, bool OUTSIDE, bool FIRST>
__device__ __forceinline__ bool run_union(const RunTable &t, int id0, int i, int ylo, int w, int h) {
    const int yr = t.rowof[i], y = ylo + yr;
    const int xs = t.xs[i], xe = t.xe[i], id = id0 + i;
    bool linked = false, did = false;
    if (OUTSIDE && (y == 0 || y == h - 1 || xs == 0 || xe == w - 1)) {
        if (FIRST) t.parent[id] = 0;
        linked = true;
    }
    if (yr == 0) return false;
    const int2 prv = t.row[yr - 1];
    const int d = CONN8 ? 1 : 0;
    int lo = 0, hi = prv.y;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if ((int)t.xe[prv.x + mid] < xs - d) lo = mid + 1; else hi = mid;
    }
    for (int q = lo; q < prv.y && (int)t.xs[prv.x + q] <= xe + d; q++) {
        if (!linked) {
            if (FIRST) t.parent[id] = id0 + prv.x + q;
            linked = true;
        } else if (!FIRST) {
            suf_union(t.parent, id, id0 + prv.x + q);
            did = true;
        }
    }
    return did;
}

// pointer jumping until every run points at its root (called by all threads of the CTA; ids 0 .. n-1):
// four hops per round, one barrier-with-vote per round
__device__ __forceinline__ void flatten_forest(int *parent, int n) {
    __syncthreads();
    while (true) {
        bool ch = false;
        for (int i = threadIdx.x; i < n; i += CCL2_THREADS) {
            const int p = parent[i];
            int q = parent[p];
            if (q != p) {
                q = parent[parent[q]];
                parent[i] = q;
                ch = true;
            }
        }
        if (!__syncthreads_or(ch)) break;
    }
}

// returns false when the frame has more runs than the shared tables hold (nothing has been published then)
__device__ __forceinline__ bool ccl_frame_lanes(const CclArgs &a, unsigned char *csm, int f, int lf,
                                                int ylo, int yhi, int jlo, int wprw) {
    const int ww = min(a.w - 32 * jlo, 32 * wprw);           // window width in pixels
    const int nrows = yhi - ylo + 1;
    RunTable bg, fg;
    bg.row = reinterpret_cast<int2 *>(csm);
    fg.row = bg.row + a.h;
    bg.parent = reinterpret_cast<int *>(fg.row + a.h);
    fg.parent = bg.parent + CCL2_CAP + 2;
    bg.xs = reinterpret_cast<uint16_t *>(fg.parent + CCL2_CAP + 2);
    bg.xe = bg.xs + CCL2_CAP;
    fg.xs = bg.xe + CCL2_CAP;
    fg.xe = fg.xs + CCL2_CAP;
    bg.rowof = fg.xe + CCL2_CAP;
    fg.rowof = bg.rowof + CCL2_CAP;
    __shared__ int cur_bg, cur_fg, overflow, wsum[CCL2_WARPS];
    if (threadIdx.x == 0) { cur_bg = 0; cur_fg = 0; overflow = 0; bg.parent[0] = 0; }
    __syncthreads();
    // The window rows are walked seven times by single lanes: when they fit they are staged into shared memory (odd
    // pitch: lanes of a warp read different rows at the same word index) and the hole filling happens in place;
    // otherwise the walks go to the planes in global memory (L2).  Generic pointers serve both.
    uint32_t *cache = reinterpret_cast<uint32_t *>(fg.rowof + CCL2_CAP);
    const int cpitch = wprw | 1;
    const bool cached = (size_t)nrows * cpitch <= (size_t)a.cache_words;
    const uint32_t *dil;
    uint32_t *fil;
    size_t pitch;
    if (cached) {
        const uint32_t *src = a.plane + ((size_t)f * a.h + ylo) * a.wpr + jlo;
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        for (int yr = warp; yr < nrows; yr += CCL2_WARPS)
            for (int j = lane; j < wprw; j += 32) cache[yr * cpitch + j] = __ldcg(src + (size_t)yr * a.wpr + j);
        dil = cache; fil = cache; pitch = cpitch;
        __syncthreads();
    } else {
        dil = a.plane + ((size_t)f * a.h + ylo) * a.wpr + jlo;
        fil = a.fill + ((size_t)f * a.h + ylo) * a.wpr + jlo;
        pitch = a.wpr;
    }

    // ---- pass 1: background runs (4-connected, linked to the outside) ----
    for (int r0 = 0; r0 < nrows; r0 += CCL2_THREADS) {
        const int yr = r0 + threadIdx.x;
        const bool act = yr < nrows;
        if (!lane_extract<true>(dil + (size_t)(act ? yr : 0) * pitch, act, yr, 1, bg, &cur_bg, wsum, ww, wprw)) overflow = 1;
    }
    __syncthreads();
    if (overflow) return false;
    const int nbg = cur_bg;
    for (int i = threadIdx.x; i < nbg; i += CCL2_THREADS) run_union<false, true, true>(bg, 1, i, ylo, ww, a.h);
    flatten_forest(bg.parent, nbg + 1);
    {
        bool did = false;
        for (int i = threadIdx.x; i < nbg; i += CCL2_THREADS) did |= run_union<false, true, false>(bg, 1, i, ylo, ww, a.h);
        if (__syncthreads_or(did)) flatten_forest(bg.parent, nbg + 1);
    }
    // ---- holes (background runs whose root is not the outside) -> filled plane; then its foreground runs ----
    if (!cached) {
        for (int yr = threadIdx.x; yr < nrows; yr += CCL2_THREADS)
            for (int j = 0; j < wprw; j++) fil[(size_t)yr * pitch + j] = dil[(size_t)yr * pitch + j];
        __syncthreads();
    }
    for (int i = threadIdx.x; i < nbg; i += CCL2_THREADS) {
        if (bg.parent[1 + i] == 0) continue;                               // connected to the outside: not a hole
        const int xs = bg.xs[i], xe = bg.xe[i];
        uint32_t *frow = fil + (size_t)bg.rowof[i] * pitch;
        for (int j = xs >> 5; j <= (xe >> 5); j++) {
            const int lo = max(xs - 32 * j, 0), hi = min(xe - 32 * j, 31);
            atomicOr(frow + j, (hi == 31 ? 0xffffffffu : ((1u << (hi + 1)) - 1u)) & ~((1u << lo) - 1u));
        }
    }
    __syncthreads();
    for (int r0 = 0; r0 < nrows; r0 += CCL2_THREADS) {
        const int yr = r0 + threadIdx.x;
        const bool act = yr < nrows;
        if (!lane_extract<false>(fil + (size_t)(act ? yr : 0) * pitch, act, yr, 0, fg, &cur_fg, wsum, ww, wprw)) overflow = 1;
    }
    __syncthreads();
    if (overflow) return false;
    const int total = cur_fg;
    int *area2 = a.area2 + (size_t)lf * a.slots, *bbox = a.bbox + (size_t)lf * a.slots * 4;
    for (int i = threadIdx.x; i < total; i += CCL2_THREADS) {
        area2[i] = 0;
        reinterpret_cast<int4 *>(bbox)[i] = make_int4(0x7fffffff, 0x7fffffff, -1, -1);
    }
    // ---- pass 2: filled foreground, 8-connected ----
    for (int i = threadIdx.x; i < total; i += CCL2_THREADS) run_union<true, false, true>(fg, 0, i, ylo, ww, a.h);
    flatten_forest(fg.parent, total);
    {
        bool did = false;
        for (int i = threadIdx.x; i < total; i += CCL2_THREADS) did |= run_union<true, false, false>(fg, 0, i, ylo, ww, a.h);
        if (__syncthreads_or(did)) flatten_forest(fg.parent, total);
    }
    // ---- per-run bit-quad area and bounding box -> root (one thread per run) ----
    for (int i = threadIdx.x; i < total; i += CCL2_THREADS) {
        const int yr = fg.rowof[i], y = ylo + yr;
        const bool has_up = yr > 0;      // row ylo is empty unless ylo == 0, where there is no row above
        const uint32_t *lrow = fil + (size_t)yr * pitch, *urow = lrow - pitch;
        const int xs = fg.xs[i], xe = fg.xe[i];
        const int root = fg.parent[i];
        int q = 0;
        if (has_up) {
            const int x0 = max(xs - 1, 0), x1 = xe;         // 2x2 windows owned by this run
            uint32_t L = win_word<false>(lrow, x0 >> 5, ww, wprw), U = win_word<false>(urow, x0 >> 5, ww, wprw);
            for (int j = x0 >> 5; j <= (x1 >> 5); j++) {
                const uint32_t Ln = win_word<false>(lrow, j + 1, ww, wprw), Un = win_word<false>(urow, j + 1, ww, wprw);
                const uint32_t l1 = (L >> 1) | (Ln << 31), u1 = (U >> 1) | (Un << 31);
                const uint32_t q4 = L & l1 & U & u1, q3 = (L & l1 & (U ^ u1)) | (U & u1 & (L ^ l1));
                const int lo = max(x0 - 32 * j, 0), hi = min(x1 - 32 * j, 31);
                const uint32_t m = (hi == 31 ? 0xffffffffu : ((1u << (hi + 1)) - 1u)) & ~((1u << lo) - 1u);
                q += 2 * __popc(q4 & m) + __popc(q3 & m);
                L = Ln; U = Un;
            }
        }
        if (q) atomicAdd(area2 + root, q);
        int *bb = bbox + (size_t)root * 4;
        atomicMin(bb + 0, xs);
        atomicMin(bb + 1, y);
        atomicMax(bb + 2, xe);
        atomicMax(bb + 3, y);
    }
    __syncthreads();
    // ---- roots -> component records ----
    for (int i = threadIdx.x; i < total; i += CCL2_THREADS) {
        if (fg.parent[i] != i) continue;
        const int ar = __ldcg(area2 + i);
        const int4 bb = __ldcg(reinterpret_cast<const int4 *>(bbox) + i);
        const int slot = atomicAdd(a.ncomp + f, 1);
        const bool skipped = (2LL * a.max_area < ar) && (ar < 2LL * a.min_area);   // find_motion.py:684
        if (!skipped) atomicAdd(a.ncounted + f, 1);
        if (slot < a.maxc) {
            fm_component c;
            c.area_x2 = ar; c.x = bb.x + 32 * jlo; c.y = bb.y; c.w = bb.z - bb.x + 1; c.h = bb.w - bb.y + 1;
            a.comps[(size_t)f * a.maxc + slot] = c;
        }
    }
    return true;
}

// dilation (optional) + window of frame f; false = quiet frame
__device__ __forceinline__ bool ccl_window(const CclArgs &a, int f, int &ylo, int &yhi, int &jlo, int &jhi) {
    ylo = 0; yhi = a.h - 1; jlo = 0; jhi = a.wpr - 1;
    if (a.raw) {
        // ---- 5x5 dilation of the raw threshold bits of this frame (rows within 3 of a pixel above threshold) ----
        const int rmax = a.rawrange[2 * f], rmin = a.h - 1 - a.rawrange[2 * f + 1];
        if (rmax < 0) return false;                                        // quiet frame: rangeout stays (-1, ...)
        __shared__ int rng[4];
        if (threadIdx.x < 4) rng[threadIdx.x] = -1;
        __syncthreads();
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        const uint32_t *flat = a.raw + (size_t)f * a.flatwords;
        uint32_t *dplane = a.planeout + (size_t)f * a.h * a.wpr;
        int jmax = -1, jmin = a.wpr, ymx = -1, ymn = a.h;
        {   // every warp takes a block of consecutive rows
            const int y0 = max(rmin - 3, 0), y1 = min(rmax + 3, a.h - 1) + 1;
            const int B = (y1 - y0 + CCL2_WARPS - 1) / CCL2_WARPS;
            const int ya = y0 + warp * B, yb = min(ya + B, y1);
            if (ya < yb) {
#define FM_DIL(AL, N) dilate_rows<AL, N>(flat, dplane, ya, yb, a.w, a.h, a.wpr, lane, jmin, jmax, ymn, ymx)
                if (a.aligned) { if (a.wpr <= 32) FM_DIL(true, 1); else if (a.wpr <= 64) FM_DIL(true, 2); else FM_DIL(true, 4); }
                else { if (a.wpr <= 32) FM_DIL(false, 1); else if (a.wpr <= 64) FM_DIL(false, 2); else FM_DIL(false, 4); }
#undef FM_DIL
            }
        }
        jmax = __reduce_max_sync(0xffffffffu, jmax);
        jmin = __reduce_min_sync(0xffffffffu, jmin);
        if (lane == 0 && ymx >= 0) {
            atomicMax(&rng[0], ymx);
            atomicMax(&rng[1], a.h - 1 - ymn);
            atomicMax(&rng[2], jmax);
            atomicMax(&rng[3], a.wpr - 1 - jmin);
        }
        __syncthreads();
        if (threadIdx.x < 4) a.rangeout[4 * f + threadIdx.x] = rng[threadIdx.x];
        if (rng[0] < 0) return false;
        ylo = max(a.h - 1 - rng[1] - 1, 0);
        yhi = min(rng[0] + 1, a.h - 1);
        jhi = rng[2];
        jlo = a.wpr - 1 - rng[3];
    } else if (a.rowrange) {
        int ymax = a.rowrange[4 * f], ymin = a.h - 1 - a.rowrange[4 * f + 1];
        if (ymax < 0) return false;
        ylo = max(ymin - 1, 0);
        yhi = min(ymax + 1, a.h - 1);
        jhi = a.rowrange[4 * f + 2];
        jlo = a.wpr - 1 - a.rowrange[4 * f + 3];
    }
    return true;
}

__global__ void __launch_bounds__(CCL2_THREADS, 1) k_ccl_frame_smem(CclArgs a, int *__restrict__ heavy) {
    extern __shared__ __align__(16) unsigned char csm[];
    fm_launch_dependents();                           // an ordinary launch: what it reads is complete
    fm_stamp_start(a.stamp);
    const int lf = blockIdx.x, lg = a.f0 + lf, f = (lg / a.Th) * a.T + a.t0 + lg % a.Th;
    int ylo, yhi, jlo, jhi;
    bool is_heavy = false;
    // frames with more runs than the shared tables hold are left to k_ccl_frame (tables in global memory)
    if (ccl_window(a, f, ylo, yhi, jlo, jhi)) is_heavy = !ccl_frame_lanes(a, csm, f, lf, ylo, yhi, jlo, jhi - jlo + 1);
    if (threadIdx.x == 0) heavy[f] = is_heavy;
}

// ---------------------------------------------------------------------------------------------
// exports for the parity tests
// ---------------------------------------------------------------------------------------------
// rowrange (optional): rows outside [h-1-rowrange[1], rowrange[0]] were never written and read as zero
__global__ void k_bits_to_u8(const uint32_t *__restrict__ plane, uint8_t *__restrict__ dst, int w, int h, int wpr,
                             uint8_t on, const int *__restrict__ rowrange) {
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= w) return;
    bool live = true;
    if (rowrange) live = rowrange[0] >= 0 && y <= rowrange[0] && y >= h - 1 - rowrange[1];
    dst[(size_t)y * w + x] = (live && ((plane[(size_t)y * wpr + (x >> 5)] >> (x & 31)) & 1u)) ? on : 0;
}

__global__ void k_u8_to_bits(const uint8_t *__restrict__ src, uint32_t *__restrict__ plane, int w, int h, int wpr) {
    int j = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (j >= wpr) return;
    uint32_t v = 0;
    for (int b = 0; b < 32; b++) {
        int x = 32 * j + b;
        if (x < w && src[(size_t)y * w + x]) v |= 1u << b;
    }
    plane[(size_t)y * wpr + j] = v;
}

int fm_launch_thresh_export(fm_ctx *c, int stream, int t, uint8_t *dst_dev, cudaStream_t st) {
    const uint32_t *pl = c->dil + ((size_t)stream * c->last_T + t) * c->h * c->wpr;
    dim3 grid((c->w + 127) / 128, c->h);
    k_bits_to_u8<<<grid, 128, 0, st>>>(pl, dst_dev, c->w, c->h, c->wpr, 255, c->any + 4 * ((size_t)stream * c->last_T + t));
    FM_LAUNCH_CHECK();
    return FM_OK;
}

int fm_launch_mask_export(fm_ctx *c, int stream, uint8_t *dst_dev, cudaStream_t st) {
    const uint32_t *pl = c->maskbits + (size_t)stream * c->h * c->wpr;
    dim3 grid((c->w + 127) / 128, c->h);
    k_bits_to_u8<<<grid, 128, 0, st>>>(pl, dst_dev, c->w, c->h, c->wpr, 1, nullptr);
    FM_LAUNCH_CHECK();
    return FM_OK;
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
int fm_ccl_alloc(CclScratch *s, int frames, int h, int cap) {
    s->frames = frames;
    s->cap = cap;
    s->slots = (size_t)h * cap;
    size_t n = (size_t)frames * s->slots;
    FM_CUDA(cudaMalloc(&s->xs, n * sizeof(uint16_t)));
    FM_CUDA(cudaMalloc(&s->xe, n * sizeof(uint16_t)));
    FM_CUDA(cudaMalloc(&s->rowcnt, (size_t)frames * h * sizeof(int)));
    FM_CUDA(cudaMalloc(&s->parent, (size_t)frames * (s->slots + 1) * sizeof(int)));
    FM_CUDA(cudaMalloc(&s->area2, n * sizeof(int)));
    FM_CUDA(cudaMalloc(&s->bbox, n * 4 * sizeof(int)));
    return FM_OK;
}

void fm_ccl_free(CclScratch *s) {
    cudaFree(s->xs); cudaFree(s->xe); cudaFree(s->rowcnt); cudaFree(s->parent); cudaFree(s->area2);
    cudaFree(s->bbox);
    s->xs = s->xe = nullptr; s->rowcnt = s->parent = s->area2 = s->bbox = nullptr;
}

// Shared-memory budget of k_ccl_frame_smem: the run tables (16 B per row + 80 KB) plus a row cache.  Planes that are
// too tall for the tables (or wider than 4096 px) are labelled by the global-memory kernel alone.
static bool ccl_smem_plan(int h, int wpr, size_t *smem, int *cache_words) {
    const size_t tables = (size_t)2 * h * sizeof(int2) + (size_t)2 * (CCL2_CAP + 2) * sizeof(int) +
                          (size_t)6 * CCL2_CAP * sizeof(uint16_t);
    const size_t budget = 200 * 1024;
    if (wpr > 128 || tables + 4096 > budget) return false;
    const size_t room = budget - tables;                                           // shared-memory row cache
    *smem = tables + (room < 128 * 1024 ? room : 128 * 1024);
    *cache_words = (int)((*smem - tables) / 4);
    return true;
}

int fm_ccl_configure(fm_ctx *c) {          // fm_ctx_create: fail here, not at the first call
    size_t smem = 0;
    int cw = 0;
    if (!ccl_smem_plan(c->h, c->wpr, &smem, &cw)) return FM_OK;
    return fm_ensure_smem((const void *)k_ccl_frame_smem, smem, c->cfg.device);
}

// labels frames [0, F) of `plane` (dilated) using `fill` as the hole-filled plane; `heavy` != null: tables in shared memory,
// frames that overflow them are flagged and labelled by the global-memory kernel that follows
static int ccl_run(const CclScratch &sc, const uint32_t *plane, uint32_t *fill, int *rowrange, int F, int w,
                   int h, int wpr, int *ncomp, int *ncounted, fm_component *comps, int maxc, int min_area,
                   int max_area, int *errflag, int *heavy, int T, int t0, int Th, cudaStream_t st,
                   const uint32_t *raw = nullptr, const int *rawrange = nullptr, int flatwords = 0,
                   unsigned long long *stamp = nullptr) {
    for (int f0 = 0; f0 < F; f0 += sc.frames) {
        int nf = F - f0 < sc.frames ? F - f0 : sc.frames;
        CclArgs a;
        a.plane = plane; a.fill = fill; a.rowrange = rowrange;
        a.raw = raw; a.rawrange = rawrange; a.rangeout = rowrange; a.planeout = const_cast<uint32_t *>(plane);
        a.flatwords = flatwords; a.aligned = (w % 32) == 0;
        a.T = T; a.t0 = t0; a.Th = Th;
        a.f0 = f0; a.nf = nf; a.w = w; a.h = h; a.wpr = wpr; a.cap = sc.cap; a.slots = sc.slots;
        a.xs = sc.xs; a.xe = sc.xe; a.rowcnt = sc.rowcnt; a.parent = sc.parent; a.area2 = sc.area2;
        a.bbox = sc.bbox; a.errflag = errflag;
        a.ncomp = ncomp; a.ncounted = ncounted; a.comps = comps; a.maxc = maxc;
        a.min_area = min_area; a.max_area = max_area;
        a.cache_words = 0;
        a.stamp = stamp;
        size_t smem = 0;
        if (heavy && ccl_smem_plan(h, wpr, &smem, &a.cache_words)) {
            int dev = 0;
            FM_CUDA(cudaGetDevice(&dev));
            int rc = fm_ensure_smem((const void *)k_ccl_frame_smem, smem, dev);
            if (rc) return rc;
            k_ccl_frame_smem<<<nf, CCL2_THREADS, smem, st>>>(a, heavy);
            FM_LAUNCH_CHECK();
            // the global-memory kernel takes the frames that overflowed the shared tables; on small planes (default mode:
            // 100 x 56) no frame can hold more than CCL2_CAP runs of either polarity, and the idle launch is left out
            if ((size_t)h * (w / 2 + 2) > CCL2_CAP)
                (void)fm_launch_chained(k_ccl_frame, nf < CCL_FALLBACK_CTAS ? nf : CCL_FALLBACK_CTAS, CCL_THREADS, 0, st, a, (const int *)heavy);
        } else {
            a.raw = nullptr;
            (void)fm_launch_chained(k_ccl_frame, nf, CCL_THREADS, 0, st, a, (const int *)nullptr);
        }
        FM_LAUNCH_CHECK();
    }
    return FM_OK;
}

// Dilation + contours + decisions of a T-frame call.  The per-frame result slots (ranges, counts, the frame counter of
// the decision tail) are cleared before this stage runs (by fm_process, or by the fused front end: fused_exit); frames
// beyond a stream's n_valid keep an empty range and leave at once.
int fm_launch_morph_ccl(fm_ctx *c, int T, cudaStream_t st, fm_frame_stats *stats_out) {
    const int F = c->S * T;
    size_t smem_plan = 0;
    int cw_plan = 0, rc;
    const bool smem_ok = ccl_smem_plan(c->h, c->wpr, &smem_plan, &cw_plan);
    unsigned long long *stamp = c->stamp ? c->stamp + 2 : nullptr;
    // With enough frames to fill the GPU (one CTA per frame) the shared-memory labelling kernel dilates the raw
    // threshold bits of its frame itself; with few frames the grid-wide k_dilate (one warp per row) is faster.
    if (smem_ok && F >= 32) {
        rc = ccl_run(c->ccl, c->dil, c->fill, c->any, F, c->w, c->h, c->wpr, c->ncomp, c->ncounted, c->comps, c->maxc,
                     c->info.min_area, c->info.max_area, c->errflag, c->heavy, T, 0, T, st, fm_tflat(c), fm_rawrange(c),
                     c->ntiles * FM_TILE_WORDS, stamp);
    } else {
        int blocks = (F * c->h + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
        if (c->w % 32 == 0)
            k_dilate<true><<<blocks, 32 * WARPS_PER_BLOCK, 0, st>>>(fm_tflat(c), c->dil, c->any, fm_rawrange(c), F, c->w, c->h,
                                                                   c->wpr, c->ntiles * FM_TILE_WORDS, T, 0, T, stamp);
        else
            k_dilate<false><<<blocks, 32 * WARPS_PER_BLOCK, 0, st>>>(fm_tflat(c), c->dil, c->any, fm_rawrange(c), F, c->w, c->h,
                                                                    c->wpr, c->ntiles * FM_TILE_WORDS, T, 0, T, stamp);
        FM_LAUNCH_CHECK();
        rc = ccl_run(c->ccl, c->dil, c->fill, c->any, F, c->w, c->h, c->wpr, c->ncomp, c->ncounted, c->comps, c->maxc,
                     c->info.min_area, c->info.max_area, c->errflag, smem_ok ? c->heavy : nullptr, T, 0, T, st, nullptr,
                     nullptr, 0, stamp);
    }
    if (rc) return rc;
    DecideArgs d;
    d.state = c->state; d.stats = c->stats; d.stats_out = stats_out; d.nvalid = c->nvalid; d.done = nullptr;
    d.stamp = stamp;
    d.S = c->S; d.T = T; d.total = F; d.cache_frames = c->info.cache_frames; d.min_movement_frames = c->info.min_movement_frames;
    (void)fm_launch_chained(k_decide, (c->S + 127) / 128, 128, 0, st, d, (const int *)c->ncomp, (const int *)c->ncounted);
    FM_LAUNCH_CHECK();
    return FM_OK;
}

// standalone labelling of one host plane (parity tests of the contour stage)
namespace {
struct PlaneScratch {                       // released on every return path
    CclScratch sc{};
    uint8_t *d8 = nullptr;
    uint32_t *pl = nullptr, *fill = nullptr;
    int *cnt = nullptr;
    fm_component *comps = nullptr;
    ~PlaneScratch() {
        cudaFree(d8); cudaFree(pl); cudaFree(fill); cudaFree(cnt); cudaFree(comps);
        fm_ccl_free(&sc);
    }
};
}

int fm_ccl_plane(int device, const uint8_t *plane_host, int w, int h, int max_n, fm_component *out, int *n) {
    FM_CUDA(cudaSetDevice(device));
    int wpr = (w + 31) / 32;
    PlaneScratch q;
    int rc = fm_ccl_alloc(&q.sc, 1, h, w / 2 + 2);
    if (rc) return rc;
    int maxc = max_n > 0 ? max_n : 1;
    FM_CUDA(cudaMalloc(&q.d8, (size_t)w * h));
    FM_CUDA(cudaMalloc(&q.pl, (size_t)wpr * h * 4));
    FM_CUDA(cudaMalloc(&q.fill, (size_t)wpr * h * 4));
    FM_CUDA(cudaMalloc(&q.cnt, 4 * sizeof(int)));
    FM_CUDA(cudaMalloc(&q.comps, (size_t)maxc * sizeof(fm_component)));
    FM_CUDA(cudaMemcpy(q.d8, plane_host, (size_t)w * h, cudaMemcpyHostToDevice));
    FM_CUDA(cudaMemset(q.cnt, 0, 4 * sizeof(int)));
    dim3 grid((wpr + 63) / 64, h);
    k_u8_to_bits<<<grid, 64>>>(q.d8, q.pl, w, h, wpr);
    FM_LAUNCH_CHECK();
    rc = ccl_run(q.sc, q.pl, q.fill, nullptr, 1, w, h, wpr, q.cnt, q.cnt + 1, q.comps, maxc, 0, 0, q.cnt + 2, q.cnt + 3, 1, 0, 1, 0);
    if (rc) return rc;
    FM_CUDA(cudaDeviceSynchronize());
    int hc[3];
    FM_CUDA(cudaMemcpy(hc, q.cnt, sizeof(hc), cudaMemcpyDeviceToHost));
    if (hc[2]) {
        fm_set_error("contour stage: run capacity exceeded");
        return FM_ERANGE;
    }
    *n = hc[0];
    int m = hc[0] < maxc ? hc[0] : maxc;
    if (max_n > 0 && m > 0) FM_CUDA(cudaMemcpy(out, q.comps, (size_t)m * sizeof(fm_component), cudaMemcpyDeviceToHost));
    return FM_OK;
}
