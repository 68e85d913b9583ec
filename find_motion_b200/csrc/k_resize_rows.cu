// K0r: INTER_AREA resize + gray for the decimating default mode (frame -> box_size wide plane), "one source row per lane".
// Replaces imutils.resize(frame, width=box_size) + cv2.cvtColor of blur_frame (find_motion/find_motion.py:487-493;
// SURVEY.md A.1, A.2).  Same float32 arithmetic in the same order as cv2's resizeArea_ (products rounded one by one,
// summed left to right along x, then top to bottom along y), so the result is bit-identical.
//
// Why rows across lanes: the horizontal chain of a (source row, destination column) is strictly sequential, and every
// source row runs the SAME chain (same taps, same weights, same byte alignment).  With a lane per source row a warp is
// fully converged: no lane idles because the plane is 100 and not 128 columns wide, no zero-weight padding to a common
// group count across lanes, and the weights are warp-uniform (one broadcast load instead of 56 registers per lane).
//
// One CTA = (frame, band of D destination rows, segment of destination columns).  The band's source rows (<= 160) are
// the CTA's threads.  The source bytes of CX destination columns at a time ("chunk") arrive by TMA as a box of
// NR rows x BW bytes, double buffered; BW / 16 is odd, so the 128-bit shared loads of a quarter warp (8 rows) hit 8
// different bank groups.
//   phase 1: thread = source row: horizontal chains of the chunk's columns -> hs[column, channel][row]   (float32)
//   phase 2: thread = (destination row, column, channel): vertical chain over the rows of its cell -> BGR byte
// and at the end of the segment the BGR bytes become gray bytes of the processing plane (or, in the BGR variant, are stored
// as they are: the detector input plane of fm_object_planes, k_objects.cu).
#include <cuda.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "fm_common.cuh"

#define RR_THREADS 160     // source rows of a band (5 warps)
#define RR_GMAX 6          // tap groups (4 source pixels = 12 bytes) per pass of a column
#ifndef RR_MIN_CTAS
#define RR_MIN_CTAS 4
#endif

struct RowsPlan {
    int D, NR, NRp, CX, NCHU, BW, nbands, segs;
    uint32_t stage_stride;
    size_t smem;
    int4 *coltab;      // [w] {byte offset of the first tap in the chunk's box, tap groups, first float4 of the weights, 0}
    int *cstartw;      // [chunks] first u32 column of the chunk's box (multiple of 4: 16-byte aligned for TMA)
    float4 *rw;        // per group: {a0..a3}, {-(2^23 a0) .. -(2^23 a3)}
};

struct RowsParams {
    int T, w, h;
    int D, NR, NRp, CX, NCHU, BW;
    uint32_t stage_stride;
    const int4 *coltab;
    const int *cstartw;
    const float4 *rw;
    const int *ystart, *yidx;
    const float *ywt;
    uint8_t *gray;
    const int *nvalid;
    // BGR variant (detector input planes, k_objects.cu): frame f's plane goes to out + s * ostride + oidx[f] * h*w*3
    const int *oidx;
    uint8_t *out;
    size_t ostride;
};

__device__ __forceinline__ uint4 rr_lds128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}

// One pass of a column: NPG (<= RR_GMAX) groups of 4 source pixels starting at word WO of the 16-byte block at shared
// address `blk`, bytes realigned by `sel` (PRMT selector 0x3210 + 0x1111 * (byte offset & 3)); weights are warp-uniform
// (broadcast loads).  The last block may reach past the column's last tap (other columns, the next row, the next shared
// buffer): finite bytes that only meet zero weights or nothing at all.
template <int WO, int NPG>
__device__ __forceinline__ void rr_col_pass(uint32_t blk, uint32_t sel, const float4 *__restrict__ wp, float &b0, float &b1,
                                            float &b2) {
    constexpr int NL = (WO + 3 * NPG) / 4 + 1;           // 16-byte blocks that hold words WO .. WO + 3 NPG
    uint32_t W[4 * NL];
#pragma unroll
    for (int k = 0; k < NL; k++) {
        const uint4 v = rr_lds128(blk + 16 * k);
        W[4 * k] = v.x; W[4 * k + 1] = v.y; W[4 * k + 2] = v.z; W[4 * k + 3] = v.w;
    }
#pragma unroll
    for (int g = 0; g < NPG; g++) {          // straight-line code: the compiler schedules the weight loads ahead of their use
        const float4 a = __ldg(wp + 2 * g), n = __ldg(wp + 2 * g + 1);
        const uint32_t X0 = __byte_perm(W[WO + 3 * g], W[WO + 3 * g + 1], sel);
        const uint32_t X1 = __byte_perm(W[WO + 3 * g + 1], W[WO + 3 * g + 2], sel);
        const uint32_t X2 = __byte_perm(W[WO + 3 * g + 2], W[WO + 3 * g + 3], sel);
        // pixels in source order, channels B G R of each: the strictly ordered chains of resizeArea_
        b0 = __fadd_rn(b0, fm_byte_mul(X0, 0, a.x, n.x)); b1 = __fadd_rn(b1, fm_byte_mul(X0, 1, a.x, n.x));
        b2 = __fadd_rn(b2, fm_byte_mul(X0, 2, a.x, n.x)); b0 = __fadd_rn(b0, fm_byte_mul(X0, 3, a.y, n.y));
        b1 = __fadd_rn(b1, fm_byte_mul(X1, 0, a.y, n.y)); b2 = __fadd_rn(b2, fm_byte_mul(X1, 1, a.y, n.y));
        b0 = __fadd_rn(b0, fm_byte_mul(X1, 2, a.z, n.z)); b1 = __fadd_rn(b1, fm_byte_mul(X1, 3, a.z, n.z));
        b2 = __fadd_rn(b2, fm_byte_mul(X2, 0, a.z, n.z)); b0 = __fadd_rn(b0, fm_byte_mul(X2, 1, a.w, n.w));
        b1 = __fadd_rn(b1, fm_byte_mul(X2, 2, a.w, n.w)); b2 = __fadd_rn(b2, fm_byte_mul(X2, 3, a.w, n.w));
    }
}

template <int WO>
__device__ __forceinline__ void rr_col_pass_n(uint32_t blk, uint32_t sel, int npg, const float4 *__restrict__ wp, float &b0,
                                              float &b1, float &b2) {
    switch (npg) {                            // warp-uniform
    case 1: rr_col_pass<WO, 1>(blk, sel, wp, b0, b1, b2); break;
    case 2: rr_col_pass<WO, 2>(blk, sel, wp, b0, b1, b2); break;
    case 3: rr_col_pass<WO, 3>(blk, sel, wp, b0, b1, b2); break;
    case 4: rr_col_pass<WO, 4>(blk, sel, wp, b0, b1, b2); break;
    case 5: rr_col_pass<WO, 5>(blk, sel, wp, b0, b1, b2); break;
    default: rr_col_pass<WO, RR_GMAX>(blk, sel, wp, b0, b1, b2); break;
    }
}

// named barriers with immediate ids (a register id makes ptxas reserve all 16 barriers for the CTA)
template <int ID> __device__ __forceinline__ void rr_bar_sync_id(int count) { asm volatile("bar.sync %0, %1;" ::"n"(ID), "r"(count) : "memory"); }
template <int ID> __device__ __forceinline__ void rr_bar_arrive_id(int count) { asm volatile("bar.arrive %0, %1;" ::"n"(ID), "r"(count) : "memory"); }
__device__ __forceinline__ void rr_bar_sync(int id, int count) {
    if (id == 1) rr_bar_sync_id<1>(count); else if (id == 2) rr_bar_sync_id<2>(count);
    else if (id == 3) rr_bar_sync_id<3>(count); else rr_bar_sync_id<4>(count);
}
__device__ __forceinline__ void rr_bar_arrive(int id, int count) {
    if (id == 1) rr_bar_arrive_id<1>(count); else if (id == 2) rr_bar_arrive_id<2>(count);
    else if (id == 3) rr_bar_arrive_id<3>(count); else rr_bar_arrive_id<4>(count);
}

// grid: (column segments, bands, F), RR_THREADS + 32 threads: warps 0..4 = the band's source rows (phase 1), warp 5 = TMA
// producer + vertical chains (phase 2) + gray.  Named barriers 1 + (i & 1): "hs of chunk i complete and stage i & 1 read"
// (row warps arrive, warp 5 waits); 3 + (i & 1): "hs buffer i & 1 consumed" (warp 5 arrives, row warps wait before chunk
// i + 2), so the row warps run up to two chunks ahead of the vertical warp and never wait for each other.
// BGR: warp 5 stores the band's BGR bytes as they are (the detector input plane) for the frames with oidx >= 0.
template <bool BGR>
__global__ void __launch_bounds__(RR_THREADS + 32, RR_MIN_CTAS) k_resize_rows(const __grid_constant__ CUtensorMap tmap, RowsParams p) {
    extern __shared__ __align__(128) unsigned char rsm[];
    const int tid = threadIdx.x;
    const int f = blockIdx.z, s = f / p.T, t = f - s * p.T;
    if constexpr (BGR) {
        if (__ldg(p.oidx + f) < 0) return;                  // no plane for this frame
    } else {
        if (t >= __ldg(p.nvalid + s)) return;               // not a real frame of this (ragged) call
    }
    const int CX = p.CX, BW = p.BW, NRp = p.NRp;
    const int DXU = CX * p.NCHU;
    const int dy0 = blockIdx.y * p.D, dy1 = min(dy0 + p.D, p.h), Dn = dy1 - dy0;
    const int dxa = blockIdx.x * DXU, dxb = min(dxa + DXU, p.w), dxun = dxb - dxa;
    const int nch = (dxun + CX - 1) / CX, ch0 = dxa / CX;
    const int yb = __ldg(p.ystart + dy0), ytn = __ldg(p.ystart + dy1) - yb;       // the band's y taps
    const int R0 = __ldg(p.yidx + yb);                                             // first source row of the band
    const int nrows = __ldg(p.yidx + yb + ytn - 1) - R0 + 1;

    unsigned char *stage = rsm;                                                    // [2][stage_stride]
    float *hs = reinterpret_cast<float *>(rsm + 2 * (size_t)p.stage_stride);       // [2][CX * 3][NRp]
    const int hsbuf = CX * 3 * NRp;
    float *yw = hs + 2 * hsbuf;                                                    // [2 NR] y weights of the band
    uint64_t *bars = reinterpret_cast<uint64_t *>((reinterpret_cast<uintptr_t>(yw + 2 * p.NR) + 7) & ~(uintptr_t)7);
    unsigned char *bgr = reinterpret_cast<unsigned char *>(bars + 2);              // [D][DXU][3]
    constexpr int NT = RR_THREADS + 32;

    if (tid == 0) {
        fm_mbar_init(&bars[0], 1);
        fm_mbar_init(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    if (tid < RR_THREADS) {
        // =========================== phase 1: one source row per thread ===========================
        const bool rowlive = (tid & ~31) < nrows;           // warp-uniform: this warp holds rows of the band
        for (int i = 0; i < nch; i++) {
            fm_mbar_wait(&bars[i & 1], (i >> 1) & 1);
            if (i >= 2) rr_bar_sync(3 + (i & 1), NT);       // phase 2 of chunk i - 2 has consumed this hs buffer
            const int dx0 = dxa + i * CX, cxn = min(CX, dxb - dx0);
            if (rowlive) {
                const uint32_t myrow = fm_smem_u32(stage) + (uint32_t)(i & 1) * p.stage_stride + (uint32_t)min(tid, p.NR - 1) * BW;
                float *hw = hs + (i & 1) * hsbuf + tid;
                int4 cnext = __ldg(p.coltab + dx0);
#pragma unroll 1
                for (int dxl = 0; dxl < cxn; dxl++) {
                    const int4 ci = cnext;
                    cnext = __ldg(p.coltab + dx0 + dxl + 1);          // the table has one entry more than columns
                    const float4 *wp = p.rw + ci.z;
                    const uint32_t sel = 0x3210u + 0x1111u * (uint32_t)(ci.x & 3);
                    float b0 = 0.f, b1 = 0.f, b2 = 0.f;
#pragma unroll 1
                    for (int g0 = 0; g0 < ci.y; g0 += RR_GMAX) {
                        const int off = ci.x + 12 * g0;
                        const int npg = min(RR_GMAX, ci.y - g0);
                        const uint32_t blk = myrow + (uint32_t)(off & ~15);
                        switch ((off >> 2) & 3) {
                        case 0: rr_col_pass_n<0>(blk, sel, npg, wp + 2 * g0, b0, b1, b2); break;
                        case 1: rr_col_pass_n<1>(blk, sel, npg, wp + 2 * g0, b0, b1, b2); break;
                        case 2: rr_col_pass_n<2>(blk, sel, npg, wp + 2 * g0, b0, b1, b2); break;
                        default: rr_col_pass_n<3>(blk, sel, npg, wp + 2 * g0, b0, b1, b2); break;
                        }
                    }
                    if (tid < nrows) {        // lanes past the band's last row ran on rows of the box that nobody reads
                        hw[(3 * dxl) * NRp] = b0;
                        hw[(3 * dxl + 1) * NRp] = b1;
                        hw[(3 * dxl + 2) * NRp] = b2;
                    }
                }
            }
            __threadfence_block();
            rr_bar_arrive(1 + (i & 1), NT);                 // hs of chunk i is complete, stage i & 1 is no longer read
        }
        return;
    }
    // =========================== warp 5: TMA producer, phase 2, gray ===========================
    const int lane = tid - RR_THREADS;
    for (int i = lane; i < ytn; i += 32) yw[i] = __ldg(p.ywt + yb + i);
    const uint32_t box_bytes = (uint32_t)p.NR * (uint32_t)BW;
    auto issue = [&](int i) {                 // chunk i of the segment -> stage i & 1 (rows past the image are zero-filled)
        fm_mbar_expect_tx(&bars[i & 1], box_bytes);
        fm_tma_load_4d(stage + (size_t)(i & 1) * p.stage_stride, &tmap, &bars[i & 1], __ldg(p.cstartw + ch0 + i), R0, t, s);
    };
    if (lane == 0) {
        issue(0);
        if (nch > 1) issue(1);
    }
    __syncwarp();
    for (int i = 0; i < nch; i++) {
        const int dx0 = dxa + i * CX, cxn = min(CX, dxb - dx0);
        rr_bar_sync(1 + (i & 1), NT);
        if (lane == 0 && i + 2 < nch) issue(i + 2);
        // vertical chains of the chunk's cells: task = (destination row, column, channel)
        const float *hb = hs + (i & 1) * hsbuf;
        const int nq = cxn * 3, ntask = Dn * nq;
        for (int task = lane; task < ntask; task += 32) {
            const int dyl = task / nq, q = task - dyl * nq;
            const int y0 = __ldg(p.ystart + dy0 + dyl), ny = __ldg(p.ystart + dy0 + dyl + 1) - y0;
            const float *hp = hb + q * NRp + (__ldg(p.yidx + y0) - R0);
            const float *wy = yw + (y0 - yb);
            float sum = __fmul_rn(wy[0], hp[0]);
            for (int j = 1; j < ny; j++) sum = __fadd_rn(sum, __fmul_rn(wy[j], hp[j]));
            const int v = min(max(__float2int_rn(sum), 0), 255);
            bgr[(dyl * DXU + (dx0 - dxa)) * 3 + q] = (unsigned char)v;
        }
        if (i + 2 < nch) {
            __threadfence_block();
            rr_bar_arrive(3 + (i & 1), NT);                 // the row warps may overwrite this hs buffer (chunk i + 2)
        }
    }
    __syncwarp();
    if constexpr (BGR) {
        uint8_t *o = p.out + (size_t)s * p.ostride + ((size_t)__ldg(p.oidx + f) * p.h + dy0) * p.w * 3 + (size_t)dxa * 3;
        const int rb = dxun * 3;
        for (int i = lane; i < Dn * rb; i += 32) {
            const int dyl = i / rb, b = i - dyl * rb;
            o[(size_t)dyl * p.w * 3 + b] = bgr[dyl * DXU * 3 + b];
        }
    } else {
        // ---- BGR -> gray (SURVEY.md A.2) ----
        for (int i = lane; i < Dn * dxun; i += 32) {
            const int dyl = i / dxun, dxo = i - dyl * dxun;
            const unsigned char *q = bgr + (dyl * DXU + dxo) * 3;
            p.gray[((size_t)f * p.h + dy0 + dyl) * p.w + dxa + dxo] =
                (uint8_t)fm_gray(q[0], q[1], q[2]);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// host: plan + launch
// ---------------------------------------------------------------------------------------------
static void rr_free(RowsPlan *&r) {
    if (!r) return;
    cudaFree(r->coltab); cudaFree(r->cstartw); cudaFree(r->rw);
    delete r;
    r = nullptr;
}

void fm_rows_free(fm_ctx *c) {
    rr_free(c->rows);
    rr_free(c->obj_rows);
}

template <typename T>
static bool rr_upload(T **dst, const std::vector<T> &v) {
    if (cudaMalloc((void **)dst, std::max<size_t>(v.size(), 1) * sizeof(T)) != cudaSuccess) return false;
    return v.empty() || cudaMemcpy(*dst, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice) == cudaSuccess;
}

static_assert(RR_GMAX == 6, "rr_col_pass_n dispatches 1 .. 6 groups");
static int rr_env(const char *name, int dflt) {
    const char *e = getenv(name);
    return (e && *e) ? atoi(e) : dflt;
}

// Host arithmetic of the plan (no CUDA): fills r and the three tables for the decimation tables of a geometry.  false: the
// geometry does not fit the kernel (source rows not TMA-compatible, bands taller than the CTA, tiny ratios) and the
// warp-per-row kernels stay in charge.
static bool rr_layout(int W, int w, int h, const int *xstart, const int *xidx, const float *xwt, const int *ystart,
                      const int *yidx, RowsPlan *r, std::vector<int4> &col, std::vector<float4> &rw, std::vector<int> &cstartw) {
    memset(r, 0, sizeof(*r));
    if (((size_t)W * 3) % 16 != 0) return false;
    // band height: the most destination rows whose source rows fit the CTA
    auto band_rows = [&](int D) {
        int mx = 0;
        for (int d0 = 0; d0 < h; d0 += D) {
            const int d1 = std::min(d0 + D, h);
            mx = std::max(mx, yidx[ystart[d1] - 1] - yidx[ystart[d0]] + 1);
        }
        return mx;
    };
    int D = 0;
    for (int d = 1; d <= h; d++) {
        if (band_rows(d) <= RR_THREADS) D = d; else break;
    }
    if (D == 0) return false;
    // tiny ratios (a handful of taps per cell) are not what this kernel is for
    int max_xt = 0;
    for (int dx = 0; dx < w; dx++) max_xt = std::max(max_xt, xstart[dx + 1] - xstart[dx]);
    if (max_xt < 4) return false;
    r->D = D; r->NR = band_rows(D); r->NRp = r->NR | 1;
    for (int d0 = 0; d0 < h; d0 += D)          // the band's y weights are staged in 2 NR floats
        if (ystart[std::min(d0 + D, h)] - ystart[d0] > 2 * r->NR) return false;
    r->nbands = (h + D - 1) / D;
    // columns per chunk: two when the CTA then still fits four to an SM (the measured optimum at 1080p -> 100: A/B log in
    // profiles/), else one (large ratios: a chunk of two columns would take > 56 KB); FM_K0_CX / FM_K0_DXU override (tuning)
    auto layout = [&](int cx) -> bool {       // fills r, col, rw, cstartw for chunks of cx columns; false: does not fit
        col.assign(w, make_int4(0, 0, 0, 0)); rw.clear(); cstartw.clear();
        r->CX = cx;
        const int dxu = std::max(cx, rr_env("FM_K0_DXU", 20));
        r->NCHU = std::max(1, (dxu + cx / 2) / cx);
        const int DXU = cx * r->NCHU;
        r->segs = (w + DXU - 1) / DXU;
        int BW = 16;
        const int nchunks = (w + cx - 1) / cx;
        for (int ch = 0; ch < nchunks; ch++) {
            const int dxa = ch * cx, dxb = std::min(dxa + cx, w);
            const int cstart = (3 * xidx[xstart[dxa]]) & ~15;
            cstartw.push_back(cstart / 4);
            for (int dx = dxa; dx < dxb; dx++) {
                const int a = xstart[dx], b = xstart[dx + 1], first = xidx[a], nt = b - a;
                for (int q = a; q < b; q++)
                    if (xidx[q] != first + (q - a)) return false;              // taps are consecutive pixels (always, for INTER_AREA)
                // groups of 4 consecutive source pixels from the first tap on, zero-weight padded at the end
                const int ng = (nt + 3) / 4, off = 3 * first - cstart;
                col[dx] = make_int4(off, ng, (int)rw.size(), 0);
                for (int g = 0; g < ng; g++) {
                    float wv[4];
                    for (int i = 0; i < 4; i++) wv[i] = (4 * g + i < nt) ? xwt[a + 4 * g + i] : 0.0f;
                    rw.push_back(make_float4(wv[0], wv[1], wv[2], wv[3]));
                    rw.push_back(make_float4(-8388608.0f * wv[0], -8388608.0f * wv[1], -8388608.0f * wv[2], -8388608.0f * wv[3]));
                }
                // 16-byte blocks the passes of this column read: block (off >> 4) + ((WO + 3 npg) >> 2) of the last pass
                for (int g0 = 0; g0 < ng; g0 += RR_GMAX) {
                    const int o = off + 12 * g0, npg = std::min(RR_GMAX, ng - g0);
                    const int last = (o >> 4) + ((((o >> 2) & 3) + 3 * npg) >> 2);
                    BW = std::max(BW, 16 * (last + 1));
                }
            }
        }
        col.push_back(col.back());                                              // the kernel reads one entry ahead
        if ((BW / 16) % 2 == 0) BW += 16;      // odd number of 16-byte blocks per row: conflict-free 128-bit loads down a column of rows
        if (BW / 4 > 256) return false;        // TMA box limit
        r->BW = BW;
        r->stage_stride = (uint32_t)(((size_t)r->NR * BW + 127) / 128 * 128);
        r->smem = 2 * (size_t)r->stage_stride + ((size_t)2 * cx * 3 * r->NRp + 2 * r->NR) * sizeof(float) + 8 + 16 +
                  (size_t)r->D * DXU * 3;
        return r->smem <= 200 * 1024;
    };
    const int forced = rr_env("FM_K0_CX", 0);
    if (forced > 0) return layout(std::min(forced, w));
    return (w >= 2 && layout(2) && r->smem <= 56 * 1024) || layout(1);
}

// Builds the plan of a W -> w x h decimation into *out; leaves it null when the geometry does not fit (rr_layout) or
// FM_FLAG_NO_ROWS is set.
static int rr_build(fm_ctx *c, const void *kern, int w, int h, const int *xstart, const int *xidx, const float *xwt,
                    const int *ystart, const int *yidx, RowsPlan **out) {
    *out = nullptr;
    if (c->cfg.flags & FM_FLAG_NO_ROWS) return FM_OK;
    RowsPlan *r = new RowsPlan();
    std::vector<int4> col;
    std::vector<float4> rw;
    std::vector<int> cstartw;
    if (!rr_layout(c->W, w, h, xstart, xidx, xwt, ystart, yidx, r, col, rw, cstartw)) { delete r; return FM_OK; }
    if (!rr_upload(&r->coltab, col) || !rr_upload(&r->cstartw, cstartw) || !rr_upload(&r->rw, rw)) {
        cudaFree(r->coltab); cudaFree(r->cstartw); cudaFree(r->rw);
        delete r;
        fm_set_error("resize plan: out of device memory");
        return FM_ENOMEM;
    }
    *out = r;
    return fm_ensure_smem(kern, r->smem, c->cfg.device);
}

// the processing plane (gray out) and the detector input plane (BGR out)
int fm_rows_plan(fm_ctx *c, const int *xstart, const int *xidx, const float *xwt, const int *ystart, const int *yidx) {
    return rr_build(c, (const void *)k_resize_rows<false>, c->w, c->h, xstart, xidx, xwt, ystart, yidx, &c->rows);
}
int fm_rows_plan_objects(fm_ctx *c, const int *xstart, const int *xidx, const float *xwt, const int *ystart, const int *yidx) {
    return rr_build(c, (const void *)k_resize_rows<true>, FM_OBJECT_WIDTH, c->obj_h, xstart, xidx, xwt, ystart, yidx,
                    &c->obj_rows);
}

// Plan of a geometry without a device (include/fm_gpu.h: fm_debug_rows_plan): the layout plus a re-check, tap by tap, that
// every shared-memory read of every column pass stays inside the chunk's box and meets the weight the tables give it.
int fm_rows_plan_describe(int W, int w, int h, const int *xstart, const int *xidx, const float *xwt, const int *ystart,
                          const int *yidx, fm_rows_plan_info *out) {
    RowsPlan r;
    std::vector<int4> col;
    std::vector<float4> rw;
    std::vector<int> cstartw;
    memset(out, 0, sizeof(*out));
    if (!rr_layout(W, w, h, xstart, xidx, xwt, ystart, yidx, &r, col, rw, cstartw)) return FM_OK;
    out->usable = 1;
    out->band_rows = r.D; out->box_rows = r.NR; out->chunk_cols = r.CX; out->seg_cols = r.CX * r.NCHU;
    out->box_bytes = r.BW; out->smem_bytes = (int32_t)r.smem; out->bands = r.nbands; out->segs = r.segs;
    for (int dx = 0; dx < w; dx++) {
        const int ch = dx / r.CX, a = xstart[dx], nt = xstart[dx + 1] - a;
        const int4 ci = col[dx];
        out->max_groups = std::max(out->max_groups, ci.y);
        if (4 * cstartw[ch] + ci.x != 3 * xidx[a] || (cstartw[ch] & 3) || ci.x < 0) { fm_set_error("rows plan: column %d misplaced", dx); return FM_ERANGE; }
        for (int g = 0; g < ci.y; g++)
            for (int i = 0; i < 4; i++) {
                const float wv = (&rw[ci.z + 2 * g].x)[i], nv = (&rw[ci.z + 2 * g + 1].x)[i];
                const float want = 4 * g + i < nt ? xwt[a + 4 * g + i] : 0.0f;
                if (wv != want || nv != -8388608.0f * want) { fm_set_error("rows plan: weight of column %d tap %d", dx, 4 * g + i); return FM_ERANGE; }
                if (ci.x + 3 * (4 * g + i) + 2 >= r.BW) { fm_set_error("rows plan: column %d reads past the box", dx); return FM_ERANGE; }
            }
        for (int g0 = 0; g0 < ci.y; g0 += RR_GMAX) {           // the 128-bit loads of a pass
            const int o = ci.x + 12 * g0, npg = std::min(RR_GMAX, ci.y - g0);
            if (16 * ((o >> 4) + ((((o >> 2) & 3) + 3 * npg) >> 2) + 1) > r.BW) { fm_set_error("rows plan: pass of column %d reads past the box", dx); return FM_ERANGE; }
        }
    }
    for (int b = 0; b < r.nbands; b++) {
        const int d0 = b * r.D, d1 = std::min(d0 + r.D, h);
        if (yidx[ystart[d1] - 1] - yidx[ystart[d0]] + 1 > r.NR || r.NR > RR_THREADS) { fm_set_error("rows plan: band %d taller than the box", b); return FM_ERANGE; }
    }
    return FM_OK;
}

bool fm_rows_usable(const fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride) {
    return c->rows && ((((uintptr_t)frames) | sstride | fstride) & 15) == 0;
}

template <bool BGR>
static int rr_launch(const fm_ctx *c, const RowsPlan *r, int w, int h, const ResizeTab &yt, const uint8_t *frames,
                     size_t sstride, size_t fstride, int T, uint8_t *out, size_t ostride, cudaStream_t st) {
    CUtensorMap tmap;
    int rc = fm_frames_tmap(c, frames, sstride, fstride, T, r->BW / 4, r->NR, &tmap);
    if (rc) return rc;
    RowsParams p;
    p.T = T; p.w = w; p.h = h;
    p.D = r->D; p.NR = r->NR; p.NRp = r->NRp; p.CX = r->CX; p.NCHU = r->NCHU; p.BW = r->BW;
    p.stage_stride = r->stage_stride;
    p.coltab = r->coltab; p.cstartw = r->cstartw; p.rw = r->rw;
    p.ystart = yt.start; p.yidx = yt.idx; p.ywt = yt.wt;
    p.gray = c->gray; p.nvalid = c->nvalid;
    p.oidx = c->obj_idx; p.out = out; p.ostride = ostride;
    dim3 grid(r->segs, r->nbands, c->S * T);
    k_resize_rows<BGR><<<grid, RR_THREADS + 32, r->smem, st>>>(tmap, p);
    FM_LAUNCH_CHECK();
    return FM_OK;
}

int fm_launch_resize_rows(fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, int T, cudaStream_t st) {
    return rr_launch<false>(c, c->rows, c->w, c->h, c->ytab, frames, sstride, fstride, T, nullptr, 0, st);
}

int fm_launch_resize_rows_objects(fm_ctx *c, const uint8_t *frames, size_t sstride, size_t fstride, int T, uint8_t *out,
                                  size_t ostride, cudaStream_t st) {
    return rr_launch<true>(c, c->obj_rows, FM_OBJECT_WIDTH, c->obj_h, c->obj_ytab, frames, sstride, fstride, T, out,
                           ostride, st);
}
