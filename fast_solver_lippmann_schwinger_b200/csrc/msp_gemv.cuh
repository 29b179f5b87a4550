// Batched, ragged matrix-vector kernel of the device-resident Msp^-1 solve (msp.cu, solver 2).
//
// One launch sweeps the stored blocks of all nodes of one dissection depth:
//     val[t][r] = y0(t, r) + sign * sum_{c < ncols[t]} M_t[r][c] * X(t, c),        r < nrows[t]
// M_t is node t's block, row-major nrows[t] x ncols[t] at M + moff[t] (tightly packed: the nodes of a depth differ
// by a row or a column, and near the leaves the identity padding of a uniform batch would be more than half of the
// bytes).  The vectors keep the uniform (padded) strides rows_p / cols_p.
//   X  : xmode 0  x[t*xstride + c]
//        xmode 1  xg[xidx[t*cols_p + c]]                  (u_B picked out of the global solution, downward sweep)
//        xmode 2  assembled right-hand side g_S           (upward sweep with the gather fused in:
//                 f[sidx[t*cols_p + c]] + tchild[(2t)*Bpc + pmap[(2t)*Fp + c]] + tchild[(2t+1)*Bpc + pmap[(2t+1)*Fp + c]])
//   y0 : ymode 0  none;   ymode 1  y0[t*y0stride + r];   ymode 2  assembled g_B (p = cols_p + r, children's terms only)
//   out: oidx ? og[oidx[t*rows_p + r]] : out[t*ostride + r]
// Thread mapping: a group of LANES lanes owns UNR consecutive rows of one node and strides over the columns; a CTA of
// 256 threads holds 256/LANES groups which are either `npc` whole nodes (small blocks) or one of `cpn` row chunks of a
// single node (large blocks), so that with XS the CTA stages X for its node(s) in shared memory once instead of every
// group fetching (and, for xmode 1 / 2, index-chasing) it again.  LANES, UNR and XS are chosen per launch - by a fixed
// rule or by timing the candidates once at factorisation time (msp.cu, LS_MSP_TUNE).  For a given LANES the summation
// order of a row does not depend on UNR / XS: lane l adds columns l, l + LANES, ... in order, then an xor tree.
//
// The index logic lives in __host__ __device__ functions so that tests/test_msp_gemv_emulation.py can run the very
// same code on the CPU (scripts/msp_gemv_emu.cu executes the CTA phases thread by thread).
#pragma once
#include <cuda_runtime.h>

namespace lsmsp {

typedef double2 cd;

#define LSMSP_HD __host__ __device__ __forceinline__

struct Gemv2 {
    const cd* M; const long* moff; const int* nrows; const int* ncols;
    int rows_p, cols_p, nodes;
    int xmode; const cd* x; long xstride; const int* xidx; const cd* xg;
    const cd* f; const int* sidx; const int* pmap; const cd* tchild; int Fp, Bpc;
    int ymode; const cd* y0; long y0stride; double sign;
    cd* out; long ostride; const int* oidx; cd* og;
};

struct Geo { unsigned rblocks, npc, cpn; };      // row blocks per node; nodes per CTA (cpn == 1) or CTAs per node (npc == 1)

template <class T> LSMSP_HD T ldg_(const T* p) {
#ifdef __CUDA_ARCH__
    return __ldg(p);
#else
    return *p;
#endif
}

LSMSP_HD cd czero() { cd z; z.x = 0.0; z.y = 0.0; return z; }

// children's contributions to entry p of node t's assembled vector (k_msp_gather's order: child 0 first)
LSMSP_HD void add_children(const Gemv2& a, unsigned t, int p, cd& v) {
    if (a.pmap == nullptr) return;
    const int k0 = ldg_(&a.pmap[((long)t * 2 + 0) * a.Fp + p]);
    const int k1 = ldg_(&a.pmap[((long)t * 2 + 1) * a.Fp + p]);
    if (k0 >= 0) { const cd w = a.tchild[(2L * t) * a.Bpc + k0]; v.x += w.x; v.y += w.y; }
    if (k1 >= 0) { const cd w = a.tchild[(2L * t + 1) * a.Bpc + k1]; v.x += w.x; v.y += w.y; }
}

LSMSP_HD cd fetch_x(const Gemv2& a, unsigned t, int c) {
    if (a.xmode == 0) return a.x[(long)t * a.xstride + c];
    if (a.xmode == 1) {
        const int gi = ldg_(&a.xidx[(long)t * a.cols_p + c]);
        return gi >= 0 ? a.xg[gi] : czero();
    }
    cd v = czero();
    const int gi = ldg_(&a.sidx[(long)t * a.cols_p + c]);
    if (gi >= 0) v = a.f[gi];
    add_children(a, t, c, v);
    return v;
}

LSMSP_HD cd fetch_y0(const Gemv2& a, unsigned t, int r) {
    if (a.ymode == 1) return a.y0[(long)t * a.y0stride + r];
    cd v = czero();
    if (a.ymode == 2) add_children(a, t, a.cols_p + r, v);
    return v;
}

struct ThreadMap {
    bool work;          // this group has rows to compute
    unsigned t;         // node
    unsigned tn;        // node index inside the CTA (shared-memory slot of its X)
    int r0, lane, nr, nc;
};

template <int LANES, int UNR>
LSMSP_HD ThreadMap map_thread(const Gemv2& a, const Geo& g, unsigned bid, unsigned tid) {
    constexpr unsigned GPC = 256 / LANES;
    ThreadMap m;
    const unsigned lg = tid / LANES;
    m.lane = (int)(tid % LANES);
    unsigned rb;
    bool live;
    if (g.cpn == 1) {
        m.tn = lg / g.rblocks;
        rb = lg - m.tn * g.rblocks;
        m.t = bid * g.npc + m.tn;
        live = m.tn < g.npc && m.t < (unsigned)a.nodes;
    } else {
        m.tn = 0;
        m.t = bid / g.cpn;
        rb = (bid - m.t * g.cpn) * GPC + lg;
        live = rb < g.rblocks;
    }
    m.r0 = (int)rb * UNR;
    m.nr = 0; m.nc = 0;
    if (live) { m.nr = ldg_(&a.nrows[m.t]); m.nc = ldg_(&a.ncols[m.t]); }
    m.work = live && m.r0 < m.nr;
    return m;
}

// phase 1 (XS): the CTA's X vectors -> xs[tn*cols_p + c]
LSMSP_HD void stage_x(const Gemv2& a, const Geo& g, unsigned bid, unsigned tid, cd* xs) {
    unsigned tfirst, cnt;
    if (g.cpn == 1) {
        tfirst = bid * g.npc;
        cnt = (unsigned)a.nodes - tfirst < g.npc ? (unsigned)a.nodes - tfirst : g.npc;
    } else {
        tfirst = bid / g.cpn;
        cnt = 1;
    }
    const unsigned total = cnt * (unsigned)a.cols_p;
    for (unsigned i = tid; i < total; i += 256u) {
        const unsigned tn = i / (unsigned)a.cols_p;
        const int c = (int)(i - tn * (unsigned)a.cols_p);
        const unsigned t = tfirst + tn;
        xs[i] = c < ldg_(&a.ncols[t]) ? fetch_x(a, t, c) : czero();
    }
}

// phase 2: per-lane partial sums of the group's UNR rows
template <int LANES, int UNR, bool XS>
LSMSP_HD void accumulate(const Gemv2& a, const ThreadMap& m, const cd* xs, double (&sr)[UNR], double (&si)[UNR]) {
#pragma unroll
    for (int u = 0; u < UNR; ++u) { sr[u] = 0.0; si[u] = 0.0; }
    if (!m.work) return;
    const cd* base = a.M + ldg_(&a.moff[m.t]) + (long)m.r0 * m.nc;
    const int nrow = (m.nr - m.r0) < UNR ? (m.nr - m.r0) : UNR;
    const cd* xsn = XS ? xs + (long)m.tn * a.cols_p : nullptr;
    // UC column steps per trip, their 8 independent 16-byte loads issued as one batch before the first multiply.  ptxas
    // keeps that order only when the launch bounds allow the registers (minBlocksPerSM = 2 below); with the default
    // bound it sinks every load next to its use to save registers and two loads per thread are in flight (SASS checked)
    constexpr int UC = (8 / UNR) > 0 ? (8 / UNR) : 1;
    for (int c0 = m.lane; c0 < m.nc; c0 += LANES * UC) {
        cd e[UC][UNR];
        cd v[UC];
        // loads past the end of the row (or of the node's rows) are clamped onto a valid element and zeroed afterwards:
        // unconditional loads are scheduled as one batch, predicated ones are sunk next to their first use
#pragma unroll
        for (int k = 0; k < UC; ++k) {
            const int c = c0 + k * LANES;
            const int cc = c < m.nc ? c : m.nc - 1;
#pragma unroll
            for (int u = 0; u < UNR; ++u) e[k][u] = ldg_(&base[(long)(u < nrow ? u : nrow - 1) * m.nc + cc]);
            if (!XS) v[k] = fetch_x(a, m.t, cc);
        }
#pragma unroll
        for (int k = 0; k < UC; ++k) {
            const int c = c0 + k * LANES;
            if (XS) v[k] = xsn[c < m.nc ? c : m.nc - 1];
            if (c >= m.nc) v[k] = czero();
#pragma unroll
            for (int u = 0; u < UNR; ++u) if (u >= nrow) e[k][u] = czero();
#pragma unroll
            for (int u = 0; u < UNR; ++u) {
                sr[u] = fma(e[k][u].x, v[k].x, sr[u]);
                sr[u] = fma(-e[k][u].y, v[k].y, sr[u]);
                si[u] = fma(e[k][u].x, v[k].y, si[u]);
                si[u] = fma(e[k][u].y, v[k].x, si[u]);
            }
        }
    }
}

// phase 4 (after the cross-lane reduction: every lane of the group holds the row sums): lane l stores rows l, l + LANES, ...
template <int LANES, int UNR>
LSMSP_HD void store_rows(const Gemv2& a, const ThreadMap& m, const double (&sr)[UNR], const double (&si)[UNR]) {
    if (!m.work) return;
#pragma unroll
    for (int u = 0; u < UNR; ++u) {
        if ((u % LANES) != m.lane || m.r0 + u >= m.nr) continue;
        const int r = m.r0 + u;
        cd val;
        val.x = a.sign * sr[u]; val.y = a.sign * si[u];
        if (a.ymode != 0) { const cd y = fetch_y0(a, m.t, r); val.x += y.x; val.y += y.y; }
        if (a.oidx) {
            const int gi = a.oidx[(long)m.t * a.rows_p + r];
            if (gi >= 0) a.og[gi] = val;
        } else {
            a.out[(long)m.t * a.ostride + r] = val;
        }
    }
}

#ifdef __CUDACC__
template <int LANES, int UNR, bool XS>
__global__ void __launch_bounds__(256, 2) k_msp_gemv2(const Gemv2 a, const Geo g) {
    extern __shared__ double2 lsmsp_xs[];
    if (XS) {
        stage_x(a, g, blockIdx.x, threadIdx.x, lsmsp_xs);
        __syncthreads();
    }
    const ThreadMap m = map_thread<LANES, UNR>(a, g, blockIdx.x, threadIdx.x);
    double sr[UNR], si[UNR];
    accumulate<LANES, UNR, XS>(a, m, lsmsp_xs, sr, si);
#pragma unroll
    for (int u = 0; u < UNR; ++u)
#pragma unroll
        for (int o = LANES / 2; o > 0; o >>= 1) {
            sr[u] += __shfl_xor_sync(0xffffffffu, sr[u], o, LANES);
            si[u] += __shfl_xor_sync(0xffffffffu, si[u], o, LANES);
        }
    store_rows<LANES, UNR>(a, m, sr, si);
}
#endif

// ---- multi-column variant: NRHS right-hand sides per factor read ---------------------------------------------------
// The same sweep for NRHS vectors at once (msp.cu, ls_msp_solve_batch): every matrix element loaded from HBM feeds NRHS
// complex FMAs.  Column j of each vector the sweep addresses lies at (column-0 address) + j * (its column stride); the
// index arrays (xidx, sidx, pmap, oidx) are shared by all columns.  Per column, lane l adds columns l, l + LANES, ... in
// the order of k_msp_gemv2 and the xor tree is the same, so for a given LANES every column of the result has the bits of
// the single-vector kernel, whatever UNR, XS and NRHS are.
struct Cols { long f, x, xg, tchild, y0, out; };

template <int NRHS>
LSMSP_HD void add_children_cols(const Gemv2& a, const Cols& cs, unsigned t, int p, cd (&v)[NRHS]) {
    if (a.pmap == nullptr) return;
    const int k0 = ldg_(&a.pmap[((long)t * 2 + 0) * a.Fp + p]);
    const int k1 = ldg_(&a.pmap[((long)t * 2 + 1) * a.Fp + p]);
    if (k0 >= 0)
#pragma unroll
        for (int j = 0; j < NRHS; ++j) { const cd w = a.tchild[(2L * t) * a.Bpc + k0 + j * cs.tchild]; v[j].x += w.x; v[j].y += w.y; }
    if (k1 >= 0)
#pragma unroll
        for (int j = 0; j < NRHS; ++j) { const cd w = a.tchild[(2L * t + 1) * a.Bpc + k1 + j * cs.tchild]; v[j].x += w.x; v[j].y += w.y; }
}

// X(t, c) of every column; the index is chased once for all of them
template <int NRHS>
LSMSP_HD void fetch_x_cols(const Gemv2& a, const Cols& cs, unsigned t, int c, cd (&v)[NRHS]) {
    if (a.xmode == 0) {
#pragma unroll
        for (int j = 0; j < NRHS; ++j) v[j] = a.x[(long)t * a.xstride + c + j * cs.x];
        return;
    }
    if (a.xmode == 1) {
        const int gi = ldg_(&a.xidx[(long)t * a.cols_p + c]);
#pragma unroll
        for (int j = 0; j < NRHS; ++j) v[j] = gi >= 0 ? a.xg[gi + j * cs.xg] : czero();
        return;
    }
    const int gi = ldg_(&a.sidx[(long)t * a.cols_p + c]);
#pragma unroll
    for (int j = 0; j < NRHS; ++j) v[j] = gi >= 0 ? a.f[gi + j * cs.f] : czero();
    add_children_cols<NRHS>(a, cs, t, c, v);
}

// X(t, c) of column j alone (the groups that fetch X themselves: one column live at a time)
LSMSP_HD cd fetch_x_col(const Gemv2& a, const Cols& cs, unsigned t, int c, int j) {
    if (a.xmode == 0) return a.x[(long)t * a.xstride + c + j * cs.x];
    if (a.xmode == 1) {
        const int gi = ldg_(&a.xidx[(long)t * a.cols_p + c]);
        return gi >= 0 ? a.xg[gi + j * cs.xg] : czero();
    }
    cd v = czero();
    const int gi = ldg_(&a.sidx[(long)t * a.cols_p + c]);
    if (gi >= 0) v = a.f[gi + j * cs.f];
    if (a.pmap != nullptr) {
        const int k0 = ldg_(&a.pmap[((long)t * 2 + 0) * a.Fp + c]);
        const int k1 = ldg_(&a.pmap[((long)t * 2 + 1) * a.Fp + c]);
        if (k0 >= 0) { const cd w = a.tchild[(2L * t) * a.Bpc + k0 + j * cs.tchild]; v.x += w.x; v.y += w.y; }
        if (k1 >= 0) { const cd w = a.tchild[(2L * t + 1) * a.Bpc + k1 + j * cs.tchild]; v.x += w.x; v.y += w.y; }
    }
    return v;
}

template <int NRHS>
LSMSP_HD void fetch_y0_cols(const Gemv2& a, const Cols& cs, unsigned t, int r, cd (&v)[NRHS]) {
#pragma unroll
    for (int j = 0; j < NRHS; ++j) v[j] = a.ymode == 1 ? a.y0[(long)t * a.y0stride + r + j * cs.y0] : czero();
    if (a.ymode == 2) add_children_cols<NRHS>(a, cs, t, a.cols_p + r, v);
}

// phase 1 (XS): column j of the CTA's X -> xs[j * npc * cols_p + tn * cols_p + c] (a block per column: the lanes of a
// group read consecutive c, as in k_msp_gemv2)
template <int NRHS>
LSMSP_HD void stage_x_cols(const Gemv2& a, const Cols& cs, const Geo& g, unsigned bid, unsigned tid, cd* xs) {
    unsigned tfirst, cnt;
    if (g.cpn == 1) {
        tfirst = bid * g.npc;
        cnt = (unsigned)a.nodes - tfirst < g.npc ? (unsigned)a.nodes - tfirst : g.npc;
    } else {
        tfirst = bid / g.cpn;
        cnt = 1;
    }
    const unsigned total = cnt * (unsigned)a.cols_p;
    const long cstride = (long)g.npc * a.cols_p;
    for (unsigned i = tid; i < total; i += 256u) {
        const unsigned tn = i / (unsigned)a.cols_p;
        const int c = (int)(i - tn * (unsigned)a.cols_p);
        const unsigned t = tfirst + tn;
        cd v[NRHS];
        if (c < ldg_(&a.ncols[t])) fetch_x_cols<NRHS>(a, cs, t, c, v);
        else
#pragma unroll
            for (int j = 0; j < NRHS; ++j) v[j] = czero();
#pragma unroll
        for (int j = 0; j < NRHS; ++j) xs[j * cstride + i] = v[j];
    }
}

// phase 2: per-lane partial sums of the group's UNR rows for every column.  The UC * UNR matrix loads of a trip are issued
// as one batch (as in accumulate); X is read one column at a time next to its use, so the registers held across the trip
// are the matrix elements and the NRHS x UNR sums
template <int LANES, int UNR, bool XS, int NRHS>
LSMSP_HD void accumulate_cols(const Gemv2& a, const Cols& cs, const Geo& g, const ThreadMap& m, const cd* xs,
                              double (&sr)[NRHS][UNR], double (&si)[NRHS][UNR]) {
#pragma unroll
    for (int j = 0; j < NRHS; ++j)
#pragma unroll
        for (int u = 0; u < UNR; ++u) { sr[j][u] = 0.0; si[j][u] = 0.0; }
    if (!m.work) return;
    const cd* base = a.M + ldg_(&a.moff[m.t]) + (long)m.r0 * m.nc;
    const int nrow = (m.nr - m.r0) < UNR ? (m.nr - m.r0) : UNR;
    const long cstride = (long)g.npc * a.cols_p;
    const cd* xsn = XS ? xs + (long)m.tn * a.cols_p : nullptr;
    constexpr int UC = (8 / UNR) > 0 ? (8 / UNR) : 1;
    for (int c0 = m.lane; c0 < m.nc; c0 += LANES * UC) {
        cd e[UC][UNR];
#pragma unroll
        for (int k = 0; k < UC; ++k) {
            const int c = c0 + k * LANES;
            const int cc = c < m.nc ? c : m.nc - 1;
#pragma unroll
            for (int u = 0; u < UNR; ++u) e[k][u] = ldg_(&base[(long)(u < nrow ? u : nrow - 1) * m.nc + cc]);
        }
#pragma unroll
        for (int k = 0; k < UC; ++k) {
            const int c = c0 + k * LANES;
            const int cc = c < m.nc ? c : m.nc - 1;
#pragma unroll
            for (int u = 0; u < UNR; ++u) if (u >= nrow) e[k][u] = czero();
#pragma unroll
            for (int j = 0; j < NRHS; ++j) {
                cd v = XS ? xsn[j * cstride + cc] : fetch_x_col(a, cs, m.t, cc, j);
                if (c >= m.nc) v = czero();
#pragma unroll
                for (int u = 0; u < UNR; ++u) {
                    sr[j][u] = fma(e[k][u].x, v.x, sr[j][u]);
                    sr[j][u] = fma(-e[k][u].y, v.y, sr[j][u]);
                    si[j][u] = fma(e[k][u].x, v.y, si[j][u]);
                    si[j][u] = fma(e[k][u].y, v.x, si[j][u]);
                }
            }
        }
    }
}

// phase 4: lane l stores rows l, l + LANES, ... of every column
template <int LANES, int UNR, int NRHS>
LSMSP_HD void store_rows_cols(const Gemv2& a, const Cols& cs, const ThreadMap& m, const double (&sr)[NRHS][UNR],
                              const double (&si)[NRHS][UNR]) {
    if (!m.work) return;
#pragma unroll
    for (int u = 0; u < UNR; ++u) {
        if ((u % LANES) != m.lane || m.r0 + u >= m.nr) continue;
        const int r = m.r0 + u;
        cd y[NRHS];
        if (a.ymode != 0) fetch_y0_cols<NRHS>(a, cs, m.t, r, y);
        const int gi = a.oidx ? a.oidx[(long)m.t * a.rows_p + r] : 0;
#pragma unroll
        for (int j = 0; j < NRHS; ++j) {
            cd val;
            val.x = a.sign * sr[j][u]; val.y = a.sign * si[j][u];
            if (a.ymode != 0) { val.x += y[j].x; val.y += y[j].y; }
            if (a.oidx) {
                if (gi >= 0) a.og[gi + j * cs.out] = val;
            } else {
                a.out[(long)m.t * a.ostride + r + j * cs.out] = val;
            }
        }
    }
}

#ifdef __CUDACC__
template <int LANES, int UNR, bool XS, int NRHS>
__global__ void __launch_bounds__(256, 2) k_msp_gemv2_cols(const Gemv2 a, const Cols cs, const Geo g) {
    extern __shared__ double2 lsmsp_xs[];
    if (XS) {
        stage_x_cols<NRHS>(a, cs, g, blockIdx.x, threadIdx.x, lsmsp_xs);
        __syncthreads();
    }
    const ThreadMap m = map_thread<LANES, UNR>(a, g, blockIdx.x, threadIdx.x);
    double sr[NRHS][UNR], si[NRHS][UNR];
    accumulate_cols<LANES, UNR, XS, NRHS>(a, cs, g, m, lsmsp_xs, sr, si);
#pragma unroll
    for (int j = 0; j < NRHS; ++j)
#pragma unroll
        for (int u = 0; u < UNR; ++u)
#pragma unroll
            for (int o = LANES / 2; o > 0; o >>= 1) {
                sr[j][u] += __shfl_xor_sync(0xffffffffu, sr[j][u], o, LANES);
                si[j][u] += __shfl_xor_sync(0xffffffffu, si[j][u], o, LANES);
            }
    store_rows_cols<LANES, UNR, NRHS>(a, cs, m, sr, si);
}
#endif

// ---- launch geometry (host) -------------------------------------------------------------------------------------
struct Choice { int lanes_log2, unr_log2, xs; };       // LANES = 1 << lanes_log2 (1..32), UNR = 1 << unr_log2 (1..8)

struct LaunchGeo { Geo g; unsigned grid; size_t smem; };

inline LaunchGeo launch_geo(int rows_p, int cols_p, int nodes, const Choice& ch) {
    const unsigned lanes = 1u << ch.lanes_log2, unr = 1u << ch.unr_log2;
    const unsigned gpc = 256u / lanes;
    LaunchGeo L;
    L.g.rblocks = ((unsigned)rows_p + unr - 1) / unr;
    if (L.g.rblocks < 1) L.g.rblocks = 1;
    if (L.g.rblocks <= gpc) {
        L.g.cpn = 1;
        L.g.npc = gpc / L.g.rblocks;
        L.grid = ((unsigned)nodes + L.g.npc - 1) / L.g.npc;
    } else {
        L.g.npc = 1;
        L.g.cpn = (L.g.rblocks + gpc - 1) / gpc;
        L.grid = (unsigned)nodes * L.g.cpn;
    }
    L.smem = ch.xs ? (size_t)L.g.npc * (size_t)cols_p * sizeof(cd) : 0;
    return L;
}

// the fixed rule (LS_MSP_TUNE=0): about eight column steps per lane, four rows per group, X staged when it is index-chased
inline Choice default_choice(int cols_p, int xmode) {
    Choice ch;
    int lg = 2;
    while (lg < 5 && (1 << lg) * 8 < cols_p) ++lg;
    ch.lanes_log2 = lg;
    ch.unr_log2 = 2;
    ch.xs = xmode != 0 ? 1 : 0;
    return ch;
}

// The multi-column kernel keeps NRHS x UNR complex sums per lane next to the 8 matrix elements in flight: UNR * NRHS <= 8
// keeps them within the 128 registers of __launch_bounds__(256, 2) (ptxas reports no spills).
constexpr int COLS_MAX = 8;                              // widest compiled NRHS; wider batches go in chunks
LSMSP_HD int cols_unr_cap_log2(int nrhs) { return nrhs >= 8 ? 0 : nrhs >= 4 ? 1 : nrhs >= 2 ? 2 : 3; }

// Geometry of the multi-column sweep: the LANES of the single-vector plan (the bits depend on it), UNR capped as above,
// X staged whenever the single plan stages it or X is index-chased (one fetch then serves NRHS columns), provided the
// staging buffer of NRHS columns fits in `limit` bytes
inline Choice cols_choice(const Choice& single, int nrhs, int rows_p, int cols_p, int nodes, int xmode, size_t limit) {
    Choice ch = single;
    const int cap = cols_unr_cap_log2(nrhs);
    if (ch.unr_log2 > cap) ch.unr_log2 = cap;
    ch.xs = (single.xs || xmode != 0) ? 1 : 0;
    if (ch.xs && launch_geo(rows_p, cols_p, nodes, ch).smem * (size_t)nrhs > limit) ch.xs = 0;
    return ch;
}

}  // namespace lsmsp
