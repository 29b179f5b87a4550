// Device-resident direct solve with the sparsified system matrix  Msp = As + k^2 AG diag(nu)  (2-D and 3-D).
//
// Stands behind `MspInv = lu(Msp)` (preconditioner.jl:35, UMFPACK; :41-55 MKL PARDISO) and the solve that runs in
// every GMRES iteration, `MspInv \ (As*b)` (preconditioner.jl:138,142,159,163).  Upstream that solve is a CPU
// sparse LU; with the Krylov basis resident on the GPU it would cost a PCIe round trip of N complex numbers plus a
// host triangular solve per iteration (SURVEY.md hard part H1), so the factorisation lives on the device here.
//
// Msp is a 9-point stencil matrix on the n x m grid (unknown i + n*j couples to (i+-1, j+-1); buildSparseA /
// buildSparseAG, SparsifyingMatrix2D.jl:806-884, :351-438) or a 27-point one on the n x m x l grid (example3D.jl:56-61).
// Geometric nested dissection (msp_symbolic.h): the grid is bisected recursively by separators one cell thick into a
// complete binary tree of depth D; the leaves are boxes of at most LEAF unknowns per side.  Node t eliminates its own
// unknowns S (separator, or the whole leaf box) against the ring B of ancestor-separator unknowns around its region
// (multifrontal method):
//      F = [F_SS F_SB; F_BS F_BB] = (entries of Msp) + (update matrices of the two children)
//      Sinv = F_SS^-1 (partial pivoting),   Y = Sinv F_SB,   update U = F_BB - F_BS Y  -> parent.
// All nodes of one depth have sizes within +-1 of each other, so a depth is one uniform batch (padded with identity
// rows): the factorisation is cuBLAS batched LU / inverse / GEMM calls (one-time set-up, like `lu(Msp)`; on a 3-D grid
// the depths with large, few fronts take cuSOLVER's LU one node at a time instead), the
// per-iteration SOLVE is hand-written: per depth three batched matrix-vector kernels on the way up
//      g = [f_S; 0] + extend(t_child0) + extend(t_child1);   z = Sinv g_S;   t = g_B - F_BS z
// and one on the way down,  u_S = z - Y u_B,  all memory-bound sweeps over the stored blocks (about 200 N complex
// numbers for a square grid: 13 GB at 2048^2, read once per solve).  Reductions run in a fixed order: deterministic.
#include "ls_common.cuh"
#include "spmv.cuh"
#include "msp_gemv.cuh"
#include "msp_symbolic.h"
#include "line_kernels.cuh"
#include <cublas_v2.h>
#include <cusolverDn.h>
#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>

using namespace ls;

namespace {

struct Level {                            // all 2^d nodes of one depth
    int count = 0, Sp = 0, Bp = 0;        // padded sizes of S and B
    bool leaf = false;
    int axis = 0;                         // split axis of this depth (0: x, 1: y, 2: z), internal levels
    bool lu_cusolver = false;             // F_SS factorised by cuSOLVER one node at a time (else cuBLAS batched)
    bool gather_s = false, gather_y = false;   // X of sweep 0 / 2 longer than the shared memory: assembled by k_msp_gather
    int* d_Sidx = nullptr;                // [count][Sp]  global unknown, -1 = padding
    int* d_Bidx = nullptr;                // [count][Bp]
    int* d_pmap = nullptr;                // [count][2][Sp+Bp]  position in child's B list, -1 = none (internal levels)
    cd* d_Sinv = nullptr;                 // [count][Sp][Sp]  row-major
    cd* d_FBS = nullptr;                  // [count][Bp][Sp]
    cd* d_Y = nullptr;                    // [count][Sp][Bp]
    cd* d_g = nullptr;                    // [count][Sp+Bp]   assembled right-hand side
    cd* d_z = nullptr;                    // [count][Sp]
    cd* d_t = nullptr;                    // [count][Bp]      update vector passed to the parent
    // solver 2: blocks packed tightly with the nodes' actual sizes (msp_gemv.cuh); d_Sinv / d_FBS / d_Y then hold
    // node t's ns x ns, nb x ns and ns x nb blocks at offS[t], offB[t], offB[t]
    int* d_ns = nullptr; int* d_nb = nullptr;
    long* d_offS = nullptr; long* d_offB = nullptr;
    lsmsp::Choice ch_sinv{2, 2, 0}, ch_fbs{2, 2, 0}, ch_y{2, 2, 1};   // kernel geometry of the three sweeps of this depth
};

struct Msp : MspBase {
    long gn = 0, gm = 0, gl = 1;
    std::vector<Level> lev;
    cd* d_in = nullptr; cd* d_out = nullptr;      // staging for host-pointer solves
    size_t factor_bytes = 0;
    double factor_seconds = 0.0;
    cublasHandle_t cublas = nullptr;
    cusolverDnHandle_t cusolver = nullptr;
    size_t smem_max = 48 * 1024;                  // the device's opt-in shared memory per block
    // solver 1: uniform (identity-padded) batches, k_msp_gather + k_msp_gemv (round-2 first version, kept selectable);
    // solver 2 (default): tightly packed blocks, gather fused into the sweeps, per-launch geometry (msp_gemv.cuh).
    // LS_MSP_SOLVER / LS_MSP_FUSE / LS_MSP_TUNE are read when the handle is created.
    int solver = 2;
    bool fuse = true, tune = true;
    double tune_seconds = 0.0;
    int solve_dev(const cd* rhs, cd* out, cudaStream_t s) override;
    int solve_launch(const cd* rhs, cd* out, cudaStream_t s);
    int solve_launch2(const cd* rhs, cd* out, cudaStream_t s);
    int tune_sweeps();
    size_t xs_limit(int cols_p) const;
    // the 4 x (depth + 1) dependent launches of one solve, captured once per (rhs, out) pair and replayed as a CUDA graph
    // (GMRES calls the solve with at most restart + 2 different pairs): removes the launch gaps between the small kernels
    struct Captured { const cd* rhs; cd* out; cudaGraphExec_t exec; };
    std::vector<Captured> graphs;
    int use_graph = -1;

    // ---- several right-hand sides (ls_msp_solve_batch) ----
    // Columns go in chunks of cols_max (4), ..., 2 and 1; a chunk of w >= 2 runs the multi-column sweeps (one factor read for w
    // columns) on work arrays of its own (per depth: w columns of g, z, t), allocated on first use and kept; a chunk of 1
    // is the single-vector solve.  Each chunk is captured and replayed as a CUDA graph per (pointers, strides, width).
    struct BatchWork { std::vector<cd*> g, z, t; };
    BatchWork bwork[4];                           // index log2(w): 1, 2, 3
    cd* d_bstage = nullptr;                       // host-pointer calls: cols_max columns of staging
    bool cols_optin = false;
    struct CapturedB { const cd* rhs; long ldr; cd* out; long ldx; int w; cudaGraphExec_t exec; };
    std::vector<CapturedB> bgraphs;
    int use_graph_cols = -1;                      // own flag: a failed batched capture leaves ls_msp_solve's graphs alone
    // widest chunk (LS_MSP_BATCH_COLS = 2, 4 or 8, read when the handle is created).  Default 4: measured on B200, one
    // chunk of 8 columns takes longer than two chunks of 4 at 2048^2, 48^3 and 64^3 (DESIGN.md 3.5)
    int cols_max = 4;
    int chunk_width(int left) const { for (int w = cols_max; w > 1; w >>= 1) if (left >= w) return w; return 1; }
    // chunk widths (bit log2 w) a batch of nrhs columns uses; with `subsets` also those of every smaller count (the
    // lockstep GMRES solves fewer columns as its systems converge)
    unsigned width_mask(int nrhs, bool subsets) const {
        unsigned m = 0;
        if (subsets) { for (int w = 2; w <= cols_max && w <= nrhs; w <<= 1) m |= 1u << log2w(w); return m; }
        for (int left = nrhs; left > 0;) { const int w = chunk_width(left); left -= w; if (w > 1) m |= 1u << log2w(w); }
        return m;
    }
    static int log2w(int w) { return w >= 8 ? 3 : w >= 4 ? 2 : 1; }
    // bw: the work arrays of a multi-column chunk (null: the level's own); their column strides, and ldr / ldx for the
    // caller's vectors, go to *cs
    int sweep_args(int d, int which, const cd* rhs, cd* out, lsmsp::Gemv2& a, const BatchWork* bw = nullptr,
                   lsmsp::Cols* cs = nullptr, long ldr = 0, long ldx = 0) const;
    size_t work_bytes(int w) const;
    size_t batch_bytes(int nrhs, bool host, bool subsets) const override;
    int batch_reserve(int nrhs, bool host, bool subsets) override;
    int solve_batch_dev(const cd* rhs, long ldr, cd* out, long ldx, int nrhs, cudaStream_t s) override;
    int solve_launch_cols(int w, const cd* rhs, long ldr, cd* out, long ldx, cudaStream_t s);
    lsmsp::Choice cols_choice(int d, int which, int w) const;
    // staging bytes a multi-column launch may use: half the opt-in limit, so that two CTAs still share an SM
    size_t cols_limit() const { return std::max<size_t>(48 * 1024, smem_max / 2); }

    ~Msp() override {
        for (auto& g : graphs) cudaGraphExecDestroy(g.exec);
        for (auto& g : bgraphs) cudaGraphExecDestroy(g.exec);
        if (cublas) cublasDestroy(cublas);
        if (cusolver) cusolverDnDestroy(cusolver);
    }
};

// ---- solve kernels ------------------------------------------------------------------------------------------
// g[t][p] = (p < Sp ? f[Sidx[t][p]] : 0) + t_child0[pmap0[p]] + t_child1[pmap1[p]]
__global__ void __launch_bounds__(256)
k_msp_gather(const cd* __restrict__ f, const int* __restrict__ Sidx, const int* __restrict__ pmap, const cd* __restrict__ tchild,
             int Sp, int Fp, int Bpc, long total, cd* __restrict__ g) {
    for (long e = (long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long)gridDim.x * blockDim.x) {
        const long t = e / Fp;
        const int p = (int)(e % Fp);
        cd v = make_double2(0.0, 0.0);
        if (p < Sp) {
            const int gi = Sidx[t * Sp + p];
            if (gi >= 0) v = f[gi];
        }
        if (pmap != nullptr) {
            const int k0 = pmap[(t * 2 + 0) * Fp + p], k1 = pmap[(t * 2 + 1) * Fp + p];
            if (k0 >= 0) { const cd a = tchild[(2 * t) * (long)Bpc + k0]; v.x += a.x; v.y += a.y; }
            if (k1 >= 0) { const cd a = tchild[(2 * t + 1) * (long)Bpc + k1]; v.x += a.x; v.y += a.y; }
        }
        g[e] = v;
    }
}

// Batched matrix-vector product over the nodes of one depth; one group of LANES lanes per row.
//   val = y0[t][r] + sign * sum_c M[t][r][c] * X(t, c)
//   X(t, c) = xidx ? xg[xidx[t][c]] (0 where the index is -1) : x[t*xstride + c]
//   result -> oidx ? og[oidx[t][r]] (skipped where -1) : out[t*ostride + r]
struct GemvArgs {
    const cd* M; int rows, cols; long ntasks;
    const cd* x; long xstride; const int* xidx; const cd* xg;
    const cd* y0; long y0stride; double sign;
    cd* out; long ostride; const int* oidx; cd* og;
};

// One group of LANES lanes handles UNR consecutive rows of one node: UNR independent 16-byte loads per lane and
// column step are in flight before the first multiply (the kernels are pure streaming: with one row per group a warp
// had 512 bytes outstanding and the sweep ran at 30 % of the HBM peak), and x is fetched once per UNR rows.
template <int LANES, int UNR>
__global__ void __launch_bounds__(256)
k_msp_gemv(const GemvArgs a, unsigned rblocks, unsigned ngroups) {
    const unsigned g = (blockIdx.x * 256u + threadIdx.x) / LANES;
    const int lane = threadIdx.x % LANES;
    const bool live = g < ngroups;
    const unsigned t = live ? g / rblocks : 0u;
    const int r0 = live ? (int)(g - t * rblocks) * UNR : 0;
    double sr[UNR], si[UNR];
#pragma unroll
    for (int u = 0; u < UNR; ++u) { sr[u] = 0.0; si[u] = 0.0; }
    if (live) {
        const cd* base = a.M + ((long)t * a.rows + r0) * (long)a.cols;
        const cd* xv = a.x ? a.x + (long)t * a.xstride : nullptr;
        const int* xi = a.xidx ? a.xidx + (long)t * a.cols : nullptr;
        const int nrow = min(UNR, a.rows - r0);
#pragma unroll 2
        for (int c = lane; c < a.cols; c += LANES) {
            cd m[UNR];
#pragma unroll
            for (int u = 0; u < UNR; ++u) m[u] = (u < nrow) ? __ldg(&base[(long)u * a.cols + c]) : make_double2(0.0, 0.0);
            cd v;
            if (xi) {
                const int gi = __ldg(&xi[c]);
                v = gi >= 0 ? a.xg[gi] : make_double2(0.0, 0.0);
            } else {
                v = xv[c];
            }
#pragma unroll
            for (int u = 0; u < UNR; ++u) {
                sr[u] += m[u].x * v.x - m[u].y * v.y;
                si[u] += m[u].x * v.y + m[u].y * v.x;
            }
        }
    }
#pragma unroll
    for (int u = 0; u < UNR; ++u)
#pragma unroll
        for (int o = LANES / 2; o > 0; o >>= 1) {
            sr[u] += __shfl_xor_sync(0xffffffffu, sr[u], o, LANES);
            si[u] += __shfl_xor_sync(0xffffffffu, si[u], o, LANES);
        }
    if (live && lane < UNR && r0 + lane < a.rows) {
        const int r = r0 + lane;
        double vr = 0.0, vi = 0.0;
#pragma unroll
        for (int u = 0; u < UNR; ++u) if (u == lane) { vr = sr[u]; vi = si[u]; }
        cd val = make_double2(a.sign * vr, a.sign * vi);
        if (a.y0) { const cd y = a.y0[(long)t * a.y0stride + r]; val.x += y.x; val.y += y.y; }
        if (a.oidx) {
            const int gi = a.oidx[(long)t * a.rows + r];
            if (gi >= 0) a.og[gi] = val;
        } else {
            a.out[(long)t * a.ostride + r] = val;
        }
    }
}

int launch_gemv(const GemvArgs& a, cudaStream_t s) {
    if (a.ntasks <= 0) return LS_OK;
    constexpr int UNR = 4;
    // lanes per row group: about `cpl` column steps per lane - the cross-lane reduction costs 4 log2(lanes) shuffles per
    // row, which dominates the small blocks when every lane owns a single column (measured: 16 x 16 leaf blocks)
    static int cpl = -1;
    if (cpl < 0) { const char* e = getenv("LS_MSP_COLS_PER_LANE"); cpl = e ? atoi(e) : 8; if (cpl < 1) cpl = 1; }
    int lanes = 4;
    while (lanes < 32 && lanes * cpl < a.cols) lanes *= 2;
    const unsigned rblocks = (unsigned)((a.rows + UNR - 1) / UNR);
    const long nodes = a.ntasks / a.rows;
    const long ngroups = nodes * rblocks;
    const long threads = ngroups * lanes;
    const unsigned blocks = (unsigned)((threads + 255) / 256);
    switch (lanes) {
        case 4:  k_msp_gemv<4, UNR><<<blocks, 256, 0, s>>>(a, rblocks, (unsigned)ngroups); break;
        case 8:  k_msp_gemv<8, UNR><<<blocks, 256, 0, s>>>(a, rblocks, (unsigned)ngroups); break;
        case 16: k_msp_gemv<16, UNR><<<blocks, 256, 0, s>>>(a, rblocks, (unsigned)ngroups); break;
        default: k_msp_gemv<32, UNR><<<blocks, 256, 0, s>>>(a, rblocks, (unsigned)ngroups); break;
    }
    return LS_OK;
}

// ---- solver 2: ragged batches, launch geometry per sweep (msp_gemv.cuh) --------------------------------------------
typedef void (*gemv2_fn)(const lsmsp::Gemv2, const lsmsp::Geo);
#define LS_G2_U(L, U) { lsmsp::k_msp_gemv2<L, U, false>, lsmsp::k_msp_gemv2<L, U, true> }
#define LS_G2_L(L) { LS_G2_U(L, 1), LS_G2_U(L, 2), LS_G2_U(L, 4), LS_G2_U(L, 8) }
const gemv2_fn gemv2_table[6][4][2] = { LS_G2_L(1), LS_G2_L(2), LS_G2_L(4), LS_G2_L(8), LS_G2_L(16), LS_G2_L(32) };
constexpr size_t GEMV2_SMEM_MAX = 48 * 1024;      // the default dynamic shared-memory limit: no per-device opt-in needed

// `limit`: the staging bytes a launch may use (Msp::xs_limit)
inline bool gemv2_valid(const lsmsp::Gemv2& a, const lsmsp::Choice& ch, size_t limit) {
    if (ch.lanes_log2 < 0 || ch.lanes_log2 > 5 || ch.unr_log2 < 0 || ch.unr_log2 > 3) return false;
    return lsmsp::launch_geo(a.rows_p, a.cols_p, a.nodes, ch).smem <= limit;
}

int launch_gemv2(const lsmsp::Gemv2& a, lsmsp::Choice ch, size_t limit, cudaStream_t s) {
    if (a.nodes <= 0 || a.rows_p <= 0) return LS_OK;
    if (!gemv2_valid(a, ch, limit)) ch.xs = 0;         // X too long for the staging buffer: every group fetches it itself
    const lsmsp::LaunchGeo L = lsmsp::launch_geo(a.rows_p, a.cols_p, a.nodes, ch);
    gemv2_table[ch.lanes_log2][ch.unr_log2][ch.xs ? 1 : 0]<<<L.grid, 256, L.smem, s>>>(a, L.g);
    return LS_OK;
}

// lets every staging kernel use `smem` bytes of dynamic shared memory on the current device (done once, at
// factorisation: the solve launches are captured into a graph)
int optin_staging(size_t smem) {
    static unsigned long long done[6][4] = {};
    for (int ll = 0; ll < 6; ++ll)
        for (int ul = 0; ul < 4; ++ul) LS_CUDA_TRY(lsk::smem_optin(gemv2_table[ll][ul][1], (int)smem, done[ll][ul]));
    return LS_OK;
}

// multi-column sweeps, NRHS = 2, 4, 8: [log2(NRHS) - 1][lanes_log2][unr_log2][xs]; UNR past lsmsp::cols_unr_cap_log2 maps
// onto the capped instantiation (cols_choice never asks for it)
typedef void (*gemv2c_fn)(const lsmsp::Gemv2, const lsmsp::Cols, const lsmsp::Geo);
#define LS_G2C_UR(L, U, R) lsmsp::k_msp_gemv2_cols<L, ((U) * (R) <= 8 ? (U) : 8 / (R)), false, R>, \
                           lsmsp::k_msp_gemv2_cols<L, ((U) * (R) <= 8 ? (U) : 8 / (R)), true, R>
#define LS_G2C_U(L, U, R) { LS_G2C_UR(L, U, R) }
#define LS_G2C_L(L, R) { LS_G2C_U(L, 1, R), LS_G2C_U(L, 2, R), LS_G2C_U(L, 4, R), LS_G2C_U(L, 8, R) }
#define LS_G2C_R(R) { LS_G2C_L(1, R), LS_G2C_L(2, R), LS_G2C_L(4, R), LS_G2C_L(8, R), LS_G2C_L(16, R), LS_G2C_L(32, R) }
const gemv2c_fn gemv2c_table[3][6][4][2] = { LS_G2C_R(2), LS_G2C_R(4), LS_G2C_R(8) };

inline int log2_width(int w) { return w >= 8 ? 3 : w >= 4 ? 2 : 1; }

int launch_gemv2_cols(const lsmsp::Gemv2& a, const lsmsp::Cols& cs, const lsmsp::Choice& ch, int w, cudaStream_t s) {
    if (a.nodes <= 0 || a.rows_p <= 0) return LS_OK;
    lsmsp::LaunchGeo L = lsmsp::launch_geo(a.rows_p, a.cols_p, a.nodes, ch);
    L.smem *= (size_t)w;
    gemv2c_table[log2_width(w) - 1][ch.lanes_log2][ch.unr_log2][ch.xs ? 1 : 0]<<<L.grid, 256, L.smem, s>>>(a, cs, L.g);
    return LS_OK;
}

int optin_staging_cols(size_t smem) {
    static unsigned long long done[3][6][4] = {};
    for (int wl = 0; wl < 3; ++wl)
        for (int ll = 0; ll < 6; ++ll)
            for (int ul = 0; ul < 4; ++ul) LS_CUDA_TRY(lsk::smem_optin(gemv2c_table[wl][ll][ul][1], (int)smem, done[wl][ll][ul]));
    return LS_OK;
}

// column-major factor blocks of the uniform batch -> tightly packed row-major blocks of the nodes' actual sizes
__global__ void k_msp_pack_tight(const cd* __restrict__ Cinv, const cd* __restrict__ Ytmp, const cd* __restrict__ F, int Sp, int Bp,
                                 long count, const int* __restrict__ ns, const int* __restrict__ nb,
                                 const long* __restrict__ offS, const long* __restrict__ offB, cd* Sinv, cd* FBS, cd* Y) {
    const int Fp = Sp + Bp;
    const long nS = (long)Sp * Sp, nB = (long)Sp * Bp;
    const long per = nS + 2 * nB;
    for (long e = (long)blockIdx.x * blockDim.x + threadIdx.x; e < count * per; e += (long)gridDim.x * blockDim.x) {
        const long t = e / per;
        long r = e % per;
        const int s_t = ns[t], b_t = nb[t];
        if (r < nS) {
            const int i = (int)(r / Sp), j = (int)(r % Sp);
            if (i < s_t && j < s_t) Sinv[offS[t] + (long)i * s_t + j] = Cinv[t * nS + i + (long)j * Sp];
        } else if (r < nS + nB) {
            r -= nS;
            const int b = (int)(r / Sp), sidx = (int)(r % Sp);
            if (b < b_t && sidx < s_t) FBS[offB[t] + (long)b * s_t + sidx] = F[t * (long)Fp * Fp + (Sp + b) + (long)sidx * Fp];
        } else {
            r -= nS + nB;
            const int sidx = (int)(r / Bp), b = (int)(r % Bp);
            if (b < b_t && sidx < s_t) Y[offB[t] + (long)sidx * b_t + b] = Ytmp[t * nB + sidx + (long)b * Sp];
        }
    }
}

// ---- factorisation kernels ------------------------------------------------------------------------------------
__global__ void k_msp_ptrs(cd** ptrs, cd* base, long stride, int count) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) ptrs[i] = base + (long)i * stride;
}
// identity on the padded diagonal entries of F_SS
__global__ void k_msp_pad_diag(cd* F, const int* __restrict__ Sidx, int Sp, int Fp, long total) {
    for (long e = (long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long)gridDim.x * blockDim.x) {
        const long t = e / Sp;
        const int i = (int)(e % Sp);
        if (Sidx[e] < 0) F[t * (long)Fp * Fp + i + (long)i * Fp] = make_double2(1.0, 0.0);
    }
}
__global__ void k_msp_scatter_entries(cd* F, const long* __restrict__ dest, const int* __restrict__ src, const cd* __restrict__ nz, long cnt) {
    for (long e = (long)blockIdx.x * blockDim.x + threadIdx.x; e < cnt; e += (long)gridDim.x * blockDim.x) {
        const cd v = nz[src[e]];
        cd* p = F + dest[e];
        p->x += v.x;
        p->y += v.y;
    }
}
// F_parent[cmap[k1], cmap[k2]] += U_child[k1, k2] for the children of one side (even or odd child index)
__global__ void k_msp_extend_add(cd* Fpar, int Fp, const cd* __restrict__ Fch, int Spc, int Bpc, const int* __restrict__ cmap,
                                 int side, long nparents) {
    const int Fpc = Spc + Bpc;
    const long per = (long)Bpc * Bpc;
    for (long e = (long)blockIdx.x * blockDim.x + threadIdx.x; e < nparents * per; e += (long)gridDim.x * blockDim.x) {
        const long t = e / per;
        const long r = e % per;
        const int k1 = (int)(r % Bpc), k2 = (int)(r / Bpc);
        const long c = 2 * t + side;
        const int pr = cmap[c * Bpc + k1], pc = cmap[c * Bpc + k2];
        if (pr < 0 || pc < 0) continue;
        const cd v = Fch[c * (long)Fpc * Fpc + (Spc + k1) + (long)(Spc + k2) * Fpc];
        cd* p = Fpar + t * (long)Fp * Fp + pr + (long)pc * Fp;
        p->x += v.x;
        p->y += v.y;
    }
}
// column-major factor blocks -> the row-major blocks the solve kernels sweep
__global__ void k_msp_pack(const cd* __restrict__ Cinv, const cd* __restrict__ Ytmp, const cd* __restrict__ F, int Sp, int Bp,
                           long count, cd* Sinv, cd* FBS, cd* Y) {
    const int Fp = Sp + Bp;
    const long nS = (long)Sp * Sp, nB = (long)Sp * Bp;
    const long per = nS + 2 * nB;
    for (long e = (long)blockIdx.x * blockDim.x + threadIdx.x; e < count * per; e += (long)gridDim.x * blockDim.x) {
        const long t = e / per;
        long r = e % per;
        if (r < nS) {
            const int i = (int)(r / Sp), j = (int)(r % Sp);
            Sinv[t * nS + r] = Cinv[t * nS + i + (long)j * Sp];
        } else if (r < nS + nB) {
            r -= nS;
            const int b = (int)(r / Sp), sidx = (int)(r % Sp);
            FBS[t * nB + r] = F[t * (long)Fp * Fp + (Sp + b) + (long)sidx * Fp];
        } else {
            r -= nS + nB;
            const int sidx = (int)(r / Bp), b = (int)(r % Bp);
            Y[t * nB + r] = Ytmp[t * nB + sidx + (long)b * Sp];
        }
    }
}

#define LS_CUBLAS_TRY(expr)                                                                        \
    do {                                                                                           \
        cublasStatus_t _s = (expr);                                                                \
        if (_s != CUBLAS_STATUS_SUCCESS) {                                                         \
            set_error("%s failed at %s:%d: cuBLAS status %d", #expr, __FILE__, __LINE__, (int)_s); \
            return LS_ERR_CUDA;                                                                    \
        }                                                                                          \
    } while (0)

inline unsigned grid_for(long total) { return (unsigned)std::min<long>((total + 255) / 256, 148L * 32); }

#define LS_CUSOLVER_TRY(expr)                                                                        \
    do {                                                                                             \
        cusolverStatus_t _s = (expr);                                                                \
        if (_s != CUSOLVER_STATUS_SUCCESS) {                                                         \
            set_error("%s failed at %s:%d: cuSOLVER status %d", #expr, __FILE__, __LINE__, (int)_s); \
            return LS_ERR_CUDA;                                                                      \
        }                                                                                            \
    } while (0)

__global__ void k_msp_eye(cd* C, int Sp, long total) {
    for (long e = (long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long)gridDim.x * blockDim.x) {
        const long t = e / Sp;
        const int i = (int)(e % Sp);
        C[t * (long)Sp * Sp + i + (long)i * Sp] = make_double2(1.0, 0.0);
    }
}

// Pivot blocks of at least this many unknowns on a 3-D grid go through cuSOLVER's blocked LU one node at a time:
// the batched cuBLAS LU / inverse are built for small matrices, and in 3-D the upper depths hold a few fronts of
// thousands of unknowns.  Depths with more nodes than LU_CUSOLVER_MAX_NODES keep the batched route (per-node calls
// would be launch-bound).  2-D handles keep the batched route at every depth.
constexpr int LU_CUSOLVER_MIN_SP = 128;
constexpr int LU_CUSOLVER_MAX_NODES = 1024;

// `sym` has been analysed and its memory need checked; builds the lists, routes the entries and factorises
int msp_factor(Msp* M, lsmsp::Symbolic& sym, const int64_t* colptr, const int64_t* rowval, const cd* nzval) {
    const auto t_start = std::chrono::steady_clock::now();
    const int64_t nnz = colptr[sym.N()] - 1;
    const int D = sym.D;
    M->lev.assign((size_t)D + 1, Level());
    cudaStream_t s = M->stream;
    int rc;
    if ((rc = sym.lists()) || (rc = sym.route(colptr, rowval)) || (rc = sym.maps())) {
        set_error("%s", sym.err.c_str());
        return rc;
    }
    for (int d = 0; d <= D; ++d) {
        Level& L = M->lev[d];
        const lsmsp::LevelShape& S = sym.lev[d];
        L.count = S.count; L.Sp = S.Sp; L.Bp = S.Bp; L.leaf = S.leaf; L.axis = S.axis;
        L.lu_cusolver = M->gl > 1 && L.Sp >= LU_CUSOLVER_MIN_SP && L.count <= LU_CUSOLVER_MAX_NODES;
    }
    const auto& hSidx = sym.Sidx;
    const auto& hBidx = sym.Bidx;
    const auto& hpmap = sym.pmap;
    const auto& hcmap = sym.cmap;
    const auto& edest = sym.edest;
    const auto& esrc = sym.esrc;

    // ---- device: index maps, solve storage ----
    size_t fbytes = 0;
    for (int d = 0; d <= D; ++d) {
        Level& L = M->lev[d];
        const size_t cnt = (size_t)L.count, Sp = (size_t)L.Sp, Bp = (size_t)L.Bp, Fp = Sp + Bp;
        if ((rc = M->dupload((void**)&L.d_Sidx, hSidx[d].data(), cnt * Sp * sizeof(int)))) return rc;
        if ((rc = M->dupload((void**)&L.d_Bidx, hBidx[d].data(), cnt * std::max<size_t>(Bp, 1) * sizeof(int)))) return rc;
        if (d < D && (rc = M->dupload((void**)&L.d_pmap, hpmap[d].data(), cnt * 2 * Fp * sizeof(int)))) return rc;
        size_t totS = cnt * Sp * Sp, totB = cnt * Sp * Bp;
        if (M->solver == 2) {
            // actual sizes (the valid entries lead every node's list) and the offsets of the tightly packed blocks
            std::vector<int> hns(cnt), hnb(cnt);
            std::vector<long> hoffS(cnt), hoffB(cnt);
            totS = 0; totB = 0;
            for (size_t t = 0; t < cnt; ++t) {
                int s_t = 0, b_t = 0;
                while (s_t < (int)Sp && hSidx[d][t * Sp + s_t] >= 0) ++s_t;
                while (b_t < (int)Bp && hBidx[d][t * Bp + b_t] >= 0) ++b_t;
                hns[t] = s_t; hnb[t] = b_t;
                hoffS[t] = (long)totS; hoffB[t] = (long)totB;
                totS += (size_t)s_t * s_t; totB += (size_t)s_t * b_t;
            }
            if ((rc = M->dupload((void**)&L.d_ns, hns.data(), cnt * sizeof(int)))) return rc;
            if ((rc = M->dupload((void**)&L.d_nb, hnb.data(), cnt * sizeof(int)))) return rc;
            if ((rc = M->dupload((void**)&L.d_offS, hoffS.data(), cnt * sizeof(long)))) return rc;
            if ((rc = M->dupload((void**)&L.d_offB, hoffB.data(), cnt * sizeof(long)))) return rc;
        }
        if ((rc = M->dmalloc((void**)&L.d_Sinv, std::max<size_t>(totS, 1) * sizeof(cd)))) return rc;
        if ((rc = M->dmalloc((void**)&L.d_FBS, std::max<size_t>(totB, 1) * sizeof(cd)))) return rc;
        if ((rc = M->dmalloc((void**)&L.d_Y, std::max<size_t>(totB, 1) * sizeof(cd)))) return rc;
        if ((rc = M->dmalloc((void**)&L.d_g, cnt * Fp * sizeof(cd)))) return rc;
        if ((rc = M->dmalloc((void**)&L.d_z, cnt * Sp * sizeof(cd)))) return rc;
        if ((rc = M->dmalloc((void**)&L.d_t, std::max<size_t>(cnt * Bp, 1) * sizeof(cd)))) return rc;
        fbytes += (totS + 2 * totB) * sizeof(cd);
    }
    M->factor_bytes = fbytes;

    // ---- numeric factorisation, leaves first ----
    cd* d_nz = nullptr;
    if ((rc = M->dupload((void**)&d_nz, nzval, (size_t)std::max<int64_t>(nnz, 1) * sizeof(cd)))) return rc;
    LS_CUBLAS_TRY(cublasCreate(&M->cublas));
    LS_CUBLAS_TRY(cublasSetStream(M->cublas, s));
    const cuDoubleComplex one = make_cuDoubleComplex(1.0, 0.0), zero = make_cuDoubleComplex(0.0, 0.0), mone = make_cuDoubleComplex(-1.0, 0.0);
    cd* Fchild = nullptr;
    for (int d = D; d >= 0; --d) {
        Level& L = M->lev[d];
        const long cnt = L.count, Sp = L.Sp, Bp = L.Bp, Fp = Sp + Bp;
        cd* F = nullptr;
        if ((rc = M->dmalloc((void**)&F, (size_t)cnt * Fp * Fp * sizeof(cd)))) return rc;
        LS_CUDA_TRY(cudaMemsetAsync(F, 0, (size_t)cnt * Fp * Fp * sizeof(cd), s));
        k_msp_pad_diag<<<grid_for(cnt * Sp), 256, 0, s>>>(F, L.d_Sidx, (int)Sp, (int)Fp, cnt * Sp);
        if (!edest[d].empty()) {
            long* d_dest = nullptr; int* d_src = nullptr;
            if ((rc = M->dupload((void**)&d_dest, edest[d].data(), edest[d].size() * sizeof(long)))) return rc;
            if ((rc = M->dupload((void**)&d_src, esrc[d].data(), esrc[d].size() * sizeof(int)))) return rc;
            k_msp_scatter_entries<<<grid_for((long)edest[d].size()), 256, 0, s>>>(F, d_dest, d_src, d_nz, (long)edest[d].size());
            LS_CUDA_TRY(cudaStreamSynchronize(s));
            M->dfree(d_dest); M->dfree(d_src);
        }
        if (d < D) {
            const Level& Lc = M->lev[d + 1];
            int* d_cmap = nullptr;
            if ((rc = M->dupload((void**)&d_cmap, hcmap[d + 1].data(), hcmap[d + 1].size() * sizeof(int)))) return rc;
            for (int side = 0; side < 2; ++side)
                k_msp_extend_add<<<grid_for(cnt * (long)Lc.Bp * Lc.Bp), 256, 0, s>>>(F, (int)Fp, Fchild, Lc.Sp, Lc.Bp, d_cmap, side, cnt);
            LS_CUDA_TRY(cudaStreamSynchronize(s));
            M->dfree(d_cmap);
            M->dfree(Fchild);
            Fchild = nullptr;
        }
        // batched LU with partial pivoting and explicit inverse of F_SS
        cd *Cinv = nullptr, *Ytmp = nullptr;
        cd **pA = nullptr, **pC = nullptr;
        int *piv = nullptr, *info = nullptr;
        if ((rc = M->dmalloc((void**)&Cinv, (size_t)cnt * Sp * Sp * sizeof(cd)))) return rc;
        if ((rc = M->dmalloc((void**)&Ytmp, std::max<size_t>((size_t)cnt * Sp * Bp, 1) * sizeof(cd)))) return rc;
        if ((rc = M->dmalloc((void**)&pA, (size_t)cnt * sizeof(cd*)))) return rc;
        if ((rc = M->dmalloc((void**)&pC, (size_t)cnt * sizeof(cd*)))) return rc;
        if ((rc = M->dmalloc((void**)&piv, (size_t)cnt * Sp * sizeof(int)))) return rc;
        if ((rc = M->dmalloc((void**)&info, (size_t)cnt * 2 * sizeof(int)))) return rc;
        if (L.lu_cusolver) {
            // F_SS = P L U in place (as the batched route), then Sinv = getrs(F_SS, I)
            if (!M->cusolver) {
                LS_CUSOLVER_TRY(cusolverDnCreate(&M->cusolver));
                LS_CUSOLVER_TRY(cusolverDnSetStream(M->cusolver, s));
            }
            int lwork = 0;
            LS_CUSOLVER_TRY(cusolverDnZgetrf_bufferSize(M->cusolver, (int)Sp, (int)Sp, reinterpret_cast<cuDoubleComplex*>(F), (int)Fp, &lwork));
            cd* work = nullptr;
            if ((rc = M->dmalloc((void**)&work, (size_t)std::max(lwork, 1) * sizeof(cd)))) return rc;
            LS_CUDA_TRY(cudaMemsetAsync(Cinv, 0, (size_t)cnt * Sp * Sp * sizeof(cd), s));
            k_msp_eye<<<grid_for(cnt * Sp), 256, 0, s>>>(Cinv, (int)Sp, cnt * Sp);
            for (long t = 0; t < cnt; ++t) {
                cuDoubleComplex* A = reinterpret_cast<cuDoubleComplex*>(F + t * Fp * Fp);
                LS_CUSOLVER_TRY(cusolverDnZgetrf(M->cusolver, (int)Sp, (int)Sp, A, (int)Fp, reinterpret_cast<cuDoubleComplex*>(work),
                                                 piv + t * Sp, info + t));
                LS_CUSOLVER_TRY(cusolverDnZgetrs(M->cusolver, CUBLAS_OP_N, (int)Sp, (int)Sp, A, (int)Fp, piv + t * Sp,
                                                 reinterpret_cast<cuDoubleComplex*>(Cinv + t * Sp * Sp), (int)Sp, info + cnt + t));
            }
            LS_CUDA_TRY(cudaStreamSynchronize(s));
            M->dfree(work);
        } else {
            k_msp_ptrs<<<(unsigned)((cnt + 255) / 256), 256, 0, s>>>(pA, F, Fp * Fp, (int)cnt);
            k_msp_ptrs<<<(unsigned)((cnt + 255) / 256), 256, 0, s>>>(pC, Cinv, Sp * Sp, (int)cnt);
            LS_CUBLAS_TRY(cublasZgetrfBatched(M->cublas, (int)Sp, reinterpret_cast<cuDoubleComplex**>(pA), (int)Fp, piv, info, (int)cnt));
            LS_CUBLAS_TRY(cublasZgetriBatched(M->cublas, (int)Sp, reinterpret_cast<cuDoubleComplex**>(pA), (int)Fp, piv,
                                              reinterpret_cast<cuDoubleComplex**>(pC), (int)Sp, info + cnt, (int)cnt));
        }
        {
            std::vector<int> hinfo((size_t)cnt * 2);
            LS_CUDA_TRY(cudaMemcpyAsync(hinfo.data(), info, hinfo.size() * sizeof(int), cudaMemcpyDeviceToHost, s));
            LS_CUDA_TRY(cudaStreamSynchronize(s));
            for (size_t q = 0; q < hinfo.size(); ++q)
                LS_REQUIRE(hinfo[q] == 0, LS_ERR_INVALID, "ls_msp_factor: singular pivot block at depth %d, node %ld (info %d)",
                           d, (long)(q % cnt), hinfo[q]);
        }
        if (Bp > 0) {
            // Y = Sinv F_SB ;  U = F_BB - F_BS Y (in place in the front, read by the parent's extend-add)
            LS_CUBLAS_TRY(cublasZgemmStridedBatched(M->cublas, CUBLAS_OP_N, CUBLAS_OP_N, (int)Sp, (int)Bp, (int)Sp, &one,
                                                    reinterpret_cast<cuDoubleComplex*>(Cinv), (int)Sp, Sp * Sp,
                                                    reinterpret_cast<cuDoubleComplex*>(F + Sp * Fp), (int)Fp, Fp * Fp, &zero,
                                                    reinterpret_cast<cuDoubleComplex*>(Ytmp), (int)Sp, Sp * Bp, (int)cnt));
            LS_CUBLAS_TRY(cublasZgemmStridedBatched(M->cublas, CUBLAS_OP_N, CUBLAS_OP_N, (int)Bp, (int)Bp, (int)Sp, &mone,
                                                    reinterpret_cast<cuDoubleComplex*>(F + Sp), (int)Fp, Fp * Fp,
                                                    reinterpret_cast<cuDoubleComplex*>(Ytmp), (int)Sp, Sp * Bp, &one,
                                                    reinterpret_cast<cuDoubleComplex*>(F + Sp + Sp * Fp), (int)Fp, Fp * Fp, (int)cnt));
        }
        if (M->solver == 2)
            k_msp_pack_tight<<<grid_for(cnt * (Sp * Sp + 2 * Sp * Bp)), 256, 0, s>>>(Cinv, Ytmp, F, (int)Sp, (int)Bp, cnt, L.d_ns, L.d_nb,
                                                                                    L.d_offS, L.d_offB, L.d_Sinv, L.d_FBS, L.d_Y);
        else
            k_msp_pack<<<grid_for(cnt * (Sp * Sp + 2 * Sp * Bp)), 256, 0, s>>>(Cinv, Ytmp, F, (int)Sp, (int)Bp, cnt, L.d_Sinv, L.d_FBS, L.d_Y);
        LS_CUDA_TRY(cudaStreamSynchronize(s));
        LS_CUDA_TRY(cudaGetLastError());
        M->dfree(Cinv); M->dfree(Ytmp); M->dfree(pA); M->dfree(pC); M->dfree(piv); M->dfree(info);
        Fchild = F;
    }
    M->dfree(Fchild);
    M->dfree(d_nz);
    M->launches_per_solve = 4 * (D + 1);
    M->factor_seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
    return LS_OK;
}

}  // namespace

int Msp::solve_dev(const cd* rhs, cd* out, cudaStream_t s) {
    auto launch = [this](const cd* r, cd* o, cudaStream_t st) { return solver == 2 ? solve_launch2(r, o, st) : solve_launch(r, o, st); };
    if (use_graph < 0) { const char* e = getenv("LS_MSP_GRAPH"); use_graph = e ? atoi(e) : 1; }
    if (!use_graph) return launch(rhs, out, s);
    for (auto& g : graphs)
        if (g.rhs == rhs && g.out == out) {
            LS_CUDA_TRY(cudaGraphLaunch(g.exec, s));
            launches += launches_per_solve;
            return LS_OK;
        }
    if (graphs.size() >= 64) return launch(rhs, out, s);
    cudaGraph_t graph = nullptr;
    if (cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
        cudaGetLastError();
        use_graph = 0;
        return launch(rhs, out, s);
    }
    const int rc = launch(rhs, out, s);
    const cudaError_t ce = cudaStreamEndCapture(s, &graph);
    if (rc != LS_OK || ce != cudaSuccess || graph == nullptr) {
        cudaGetLastError();
        if (graph) cudaGraphDestroy(graph);
        use_graph = 0;
        return launch(rhs, out, s);
    }
    cudaGraphExec_t exec = nullptr;
    const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ie != cudaSuccess) { cudaGetLastError(); use_graph = 0; return launch(rhs, out, s); }
    graphs.push_back(Captured{rhs, out, exec});
    LS_CUDA_TRY(cudaGraphLaunch(exec, s));
    return LS_OK;
}

int Msp::solve_launch(const cd* rhs, cd* out, cudaStream_t s) {
    const int D = (int)lev.size() - 1;
    // upward pass: leaves -> root
    for (int d = D; d >= 0; --d) {
        Level& L = lev[d];
        const int Fp = L.Sp + L.Bp;
        const long total = (long)L.count * Fp;
        const Level* Lc = d < D ? &lev[d + 1] : nullptr;
        k_msp_gather<<<grid_for(total), 256, 0, s>>>(rhs, L.d_Sidx, Lc ? L.d_pmap : nullptr, Lc ? Lc->d_t : nullptr, L.Sp, Fp,
                                                     Lc ? Lc->Bp : 0, total, L.d_g);
        GemvArgs a{};
        a.M = L.d_Sinv; a.rows = L.Sp; a.cols = L.Sp; a.ntasks = (long)L.count * L.Sp;
        a.x = L.d_g; a.xstride = Fp; a.sign = 1.0;
        a.out = L.d_z; a.ostride = L.Sp;
        launch_gemv(a, s);
        if (L.Bp > 0) {
            GemvArgs b{};
            b.M = L.d_FBS; b.rows = L.Bp; b.cols = L.Sp; b.ntasks = (long)L.count * L.Bp;
            b.x = L.d_z; b.xstride = L.Sp; b.sign = -1.0;
            b.y0 = L.d_g + L.Sp; b.y0stride = Fp;
            b.out = L.d_t; b.ostride = L.Bp;
            launch_gemv(b, s);
        }
    }
    // downward pass: root -> leaves; u_S = z - Y u_B, written straight into `out`
    for (int d = 0; d <= D; ++d) {
        Level& L = lev[d];
        GemvArgs a{};
        a.M = L.d_Y; a.rows = L.Sp; a.cols = L.Bp; a.ntasks = (long)L.count * L.Sp;
        a.xidx = L.d_Bidx; a.xg = out; a.sign = -1.0;
        a.y0 = L.d_z; a.y0stride = L.Sp;
        a.oidx = L.d_Sidx; a.og = out;
        launch_gemv(a, s);
    }
    launches += launches_per_solve;
    LS_CUDA_TRY(cudaGetLastError());
    return LS_OK;
}

// ---- solver 2 ----------------------------------------------------------------------------------------------------
// Staging bytes a sweep with cols_p columns may use: the default 48 KB, or the device's opt-in limit (227 KB on B200)
// when one node's X alone is longer than 48 KB (separators and rings of more than 3072 unknowns, 3-D grids).  Beyond
// that, sweeps 0 and 2 read X assembled once by k_msp_gather (Level::gather_s / gather_y).
size_t Msp::xs_limit(int cols_p) const {
    return (size_t)cols_p * sizeof(cd) > GEMV2_SMEM_MAX ? smem_max : GEMV2_SMEM_MAX;
}

// arguments of sweep `which` of depth d:  0  z = Sinv g_S   1  t = g_B - F_BS z   2  u_S = z - Y u_B
int Msp::sweep_args(int d, int which, const cd* rhs, cd* out, lsmsp::Gemv2& a, const BatchWork* bw, lsmsp::Cols* cs,
                    long ldr, long ldx) const {
    const int D = (int)lev.size() - 1;
    const Level& L = lev[d];
    const Level* Lc = d < D ? &lev[d + 1] : nullptr;
    const int Fp = L.Sp + L.Bp;
    cd* g = bw ? bw->g[d] : L.d_g;
    cd* z = bw ? bw->z[d] : L.d_z;
    cd* t = bw ? bw->t[d] : L.d_t;
    cd* tc = Lc ? (bw ? bw->t[d + 1] : Lc->d_t) : nullptr;
    // column strides of the work arrays: their per-column sizes (work_bytes)
    const long gcs = (long)L.count * Fp, zcs = (long)L.count * L.Sp, tcs = std::max<long>((long)L.count * L.Bp, 1);
    const long tccs = Lc ? std::max<long>((long)Lc->count * Lc->Bp, 1) : 0;
    a = lsmsp::Gemv2{};
    lsmsp::Cols c{};
    c.f = ldr; c.xg = ldx; c.tchild = tccs;
    a.nodes = L.count;
    a.pmap = Lc ? L.d_pmap : nullptr; a.tchild = tc; a.Fp = Fp; a.Bpc = Lc ? Lc->Bp : 0;
    if (which == 0) {
        a.M = L.d_Sinv; a.moff = L.d_offS; a.nrows = L.d_ns; a.ncols = L.d_ns; a.rows_p = L.Sp; a.cols_p = L.Sp;
        if (fuse && !L.gather_s) { a.xmode = 2; a.f = rhs; a.sidx = L.d_Sidx; }
        else { a.xmode = 0; a.x = g; a.xstride = Fp; c.x = gcs; }
        a.ymode = 0; a.sign = 1.0;
        a.out = z; a.ostride = L.Sp; c.out = zcs;
    } else if (which == 1) {
        a.M = L.d_FBS; a.moff = L.d_offB; a.nrows = L.d_nb; a.ncols = L.d_ns; a.rows_p = L.Bp; a.cols_p = L.Sp;
        a.xmode = 0; a.x = z; a.xstride = L.Sp; c.x = zcs;
        if (fuse) a.ymode = 2;
        else { a.ymode = 1; a.y0 = g + L.Sp; a.y0stride = Fp; c.y0 = gcs; }
        a.sign = -1.0;
        a.out = t; a.ostride = L.Bp; c.out = tcs;
    } else {
        a.M = L.d_Y; a.moff = L.d_offB; a.nrows = L.d_ns; a.ncols = L.d_nb; a.rows_p = L.Sp; a.cols_p = L.Bp;
        if (L.gather_y) { a.xmode = 0; a.x = g; a.xstride = L.Bp; c.x = gcs; }
        else { a.xmode = 1; a.xidx = L.d_Bidx; a.xg = out; }
        a.ymode = 1; a.y0 = z; a.y0stride = L.Sp; a.sign = -1.0; c.y0 = zcs;
        a.oidx = L.d_Sidx; a.og = out; c.out = ldx;
    }
    if (cs) *cs = c;
    return LS_OK;
}

int Msp::solve_launch2(const cd* rhs, cd* out, cudaStream_t s) {
    const int D = (int)lev.size() - 1;
    lsmsp::Gemv2 a;
    for (int d = D; d >= 0; --d) {                      // upward: leaves -> root
        Level& L = lev[d];
        if (!fuse || L.gather_s) {
            const int Fp = L.Sp + L.Bp;
            const long total = (long)L.count * Fp;
            const Level* Lc = d < D ? &lev[d + 1] : nullptr;
            k_msp_gather<<<grid_for(total), 256, 0, s>>>(rhs, L.d_Sidx, Lc ? L.d_pmap : nullptr, Lc ? Lc->d_t : nullptr, L.Sp, Fp,
                                                         Lc ? Lc->Bp : 0, total, L.d_g);
        }
        sweep_args(d, 0, rhs, out, a);
        launch_gemv2(a, L.ch_sinv, xs_limit(a.cols_p), s);
        if (L.Bp > 0) {
            sweep_args(d, 1, rhs, out, a);
            launch_gemv2(a, L.ch_fbs, xs_limit(a.cols_p), s);
        }
    }
    for (int d = 0; d <= D; ++d) {                      // downward: root -> leaves, u_S written straight into `out`
        const Level& L = lev[d];
        if (L.gather_y) {                               // u_B = out[Bidx] into d_g (free once the upward pass is done)
            const long total = (long)L.count * L.Bp;
            k_msp_gather<<<grid_for(total), 256, 0, s>>>(out, L.d_Bidx, nullptr, nullptr, L.Bp, L.Bp, 0, total, L.d_g);
        }
        sweep_args(d, 2, rhs, out, a);
        launch_gemv2(a, L.ch_y, xs_limit(a.cols_p), s);
    }
    launches += launches_per_solve;
    LS_CUDA_TRY(cudaGetLastError());
    return LS_OK;
}

// Times every admissible (LANES, UNR, XS) of every sweep once, on the blocks just factorised (cold L2: a buffer larger
// than the L2 is cleared before each timed launch, as in a solve every block arrives from HBM), and keeps the fastest.
// The sweeps are idempotent on fixed inputs, so the candidates simply run one after the other in solve order.
int Msp::tune_sweeps() {
    const auto t_start = std::chrono::steady_clock::now();
    const int D = (int)lev.size() - 1;
    cudaStream_t s = stream;
    cd *f = nullptr, *u = nullptr;
    void* flush = nullptr;
    int rc;
    const size_t vb = (size_t)n * sizeof(cd);
    const size_t flush_bytes = factor_bytes > ((size_t)64 << 20) ? ((size_t)192 << 20) : 0;    // small factors live in the L2 anyway
    if ((rc = dmalloc((void**)&f, vb))) return rc;
    if ((rc = dmalloc((void**)&u, vb))) return rc;
    if (flush_bytes && dmalloc(&flush, flush_bytes) != LS_OK) flush = nullptr;      // no room for the flush buffer: time warm
    LS_CUDA_TRY(cudaMemsetAsync(f, 0, vb, s));
    LS_CUDA_TRY(cudaMemsetAsync(u, 0, vb, s));
    for (Level& L : lev) {
        LS_CUDA_TRY(cudaMemsetAsync(L.d_g, 0, (size_t)L.count * (L.Sp + L.Bp) * sizeof(cd), s));
        LS_CUDA_TRY(cudaMemsetAsync(L.d_z, 0, (size_t)L.count * L.Sp * sizeof(cd), s));
        LS_CUDA_TRY(cudaMemsetAsync(L.d_t, 0, std::max<size_t>((size_t)L.count * L.Bp, 1) * sizeof(cd), s));
    }
    struct Events {
        cudaEvent_t a = nullptr, b = nullptr;
        ~Events() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
    } ev;
    LS_CUDA_TRY(cudaEventCreate(&ev.a));
    LS_CUDA_TRY(cudaEventCreate(&ev.b));
    const cudaEvent_t e0 = ev.a, e1 = ev.b;
    auto tune_one = [&](int d, int which, lsmsp::Choice& best) -> int {
        lsmsp::Gemv2 a;
        sweep_args(d, which, f, u, a);
        if (a.nodes <= 0 || a.rows_p <= 0) return LS_OK;
        const lsmsp::Choice def = lsmsp::default_choice(a.cols_p, a.xmode);
        const size_t limit = xs_limit(a.cols_p);
        float best_ms = 1e30f;
        lsmsp::Choice pick = def;
        if (!gemv2_valid(a, pick, limit)) pick.xs = 0;
        for (int ll = std::max(0, def.lanes_log2 - 2); ll <= std::min(5, def.lanes_log2 + 1); ++ll)
            for (int ul = 0; ul <= 3; ++ul)
                for (int xs = 0; xs <= 1; ++xs) {
                    const lsmsp::Choice ch{ll, ul, xs};
                    if (!gemv2_valid(a, ch, limit)) continue;
                    if ((1 << ul) > std::max(a.rows_p, 1) * 2) continue;          // more rows per group than the block has
                    launch_gemv2(a, ch, limit, s);                                 // warm-up: instruction cache, first touch
                    float ms = 1e30f;
                    for (int rep = 0; rep < 2; ++rep) {
                        if (flush) LS_CUDA_TRY(cudaMemsetAsync(flush, 0, flush_bytes, s));
                        LS_CUDA_TRY(cudaEventRecord(e0, s));
                        launch_gemv2(a, ch, limit, s);
                        LS_CUDA_TRY(cudaEventRecord(e1, s));
                        LS_CUDA_TRY(cudaEventSynchronize(e1));
                        float t = 0.f;
                        LS_CUDA_TRY(cudaEventElapsedTime(&t, e0, e1));
                        ms = std::min(ms, t);
                    }
                    if (ms < best_ms) { best_ms = ms; pick = ch; }
                }
        best = pick;
        return LS_OK;
    };
    for (int d = D; d >= 0 && rc == LS_OK; --d) {
        rc = tune_one(d, 0, lev[d].ch_sinv);
        if (rc == LS_OK && lev[d].Bp > 0) rc = tune_one(d, 1, lev[d].ch_fbs);
    }
    for (int d = 0; d <= D && rc == LS_OK; ++d) rc = tune_one(d, 2, lev[d].ch_y);
    if (rc == LS_OK) {
        cudaError_t ce = cudaStreamSynchronize(s);
        if (ce == cudaSuccess) ce = cudaGetLastError();
        if (ce != cudaSuccess) { set_error("ls_msp_factor: tuning the solve sweeps failed: %s", cudaGetErrorString(ce)); rc = LS_ERR_CUDA; }
    }
    dfree(f); dfree(u); dfree(flush);
    tune_seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
    return rc;
}

// ---- several right-hand sides ----------------------------------------------------------------------------------------
// geometry of sweep `which` of depth d for chunks of w columns: the LANES of the single-vector plan, so that every column
// has the single solve's bits (msp_gemv.cuh), UNR / XS by lsmsp::cols_choice
lsmsp::Choice Msp::cols_choice(int d, int which, int w) const {
    lsmsp::Gemv2 a;
    sweep_args(d, which, nullptr, nullptr, a);
    const Level& L = lev[d];
    const lsmsp::Choice& single = which == 0 ? L.ch_sinv : which == 1 ? L.ch_fbs : L.ch_y;
    return lsmsp::cols_choice(single, w, a.rows_p, a.cols_p, a.nodes, a.xmode, cols_limit());
}

size_t Msp::work_bytes(int w) const {
    size_t b = 0;
    for (const Level& L : lev)
        b += (size_t)w * ((size_t)L.count * (L.Sp + L.Bp) + (size_t)L.count * L.Sp + std::max<size_t>((size_t)L.count * L.Bp, 1));
    return b * sizeof(cd);
}

size_t Msp::batch_bytes(int nrhs, bool host, bool subsets) const {
    size_t b = 0;
    if (solver == 2) {
        const unsigned m = width_mask(nrhs, subsets);
        for (int wl = 1; wl <= 3; ++wl)
            if ((m >> wl & 1u) && bwork[wl].g.empty()) b += work_bytes(1 << wl);
    }
    if (host && !d_bstage) b += (size_t)n * cols_max * sizeof(cd);
    return b;
}

int Msp::batch_reserve(int nrhs, bool host, bool subsets) {
    int rc;
    if (host && !d_bstage && (rc = dmalloc((void**)&d_bstage, (size_t)n * cols_max * sizeof(cd)))) return rc;
    if (solver != 2) return LS_OK;
    if (!cols_optin && smem_max > 48 * 1024) {
        if ((rc = optin_staging_cols(cols_limit()))) return rc;
        cols_optin = true;
    }
    const unsigned m = width_mask(nrhs, subsets);
    for (int wl = 1; wl <= 3; ++wl) {
        BatchWork& W = bwork[wl];
        if (!(m >> wl & 1u) || !W.g.empty()) continue;
        const int w = 1 << wl;
        for (const Level& L : lev) {
            const size_t nb[3] = {(size_t)w * L.count * (L.Sp + L.Bp), (size_t)w * L.count * L.Sp,
                                  (size_t)w * std::max<size_t>((size_t)L.count * L.Bp, 1)};
            cd* p[3];
            for (int q = 0; q < 3; ++q) {
                if ((rc = dmalloc((void**)&p[q], std::max<size_t>(nb[q], 1) * sizeof(cd)))) return rc;
                LS_CUDA_TRY(cudaMemsetAsync(p[q], 0, std::max<size_t>(nb[q], 1) * sizeof(cd), stream));
            }
            W.g.push_back(p[0]); W.z.push_back(p[1]); W.t.push_back(p[2]);
        }
        LS_CUDA_TRY(cudaStreamSynchronize(stream));
    }
    return LS_OK;
}

// the solve_launch2 sequence for w columns: the same sweeps, gathers and order, on the chunk's work arrays
int Msp::solve_launch_cols(int w, const cd* rhs, long ldr, cd* out, long ldx, cudaStream_t s) {
    const int D = (int)lev.size() - 1;
    const BatchWork& W = bwork[log2_width(w)];
    lsmsp::Gemv2 a;
    lsmsp::Cols cs;
    for (int d = D; d >= 0; --d) {                      // upward: leaves -> root
        const Level& L = lev[d];
        // the separate gathers (unfused solves, separators too long to stage) run once per column: they read N-sized
        // vectors, not factor blocks, and take no part in the sweeps' sharing of the factor reads
        if (!fuse || L.gather_s) {
            const int Fp = L.Sp + L.Bp;
            const long total = (long)L.count * Fp;
            const Level* Lc = d < D ? &lev[d + 1] : nullptr;
            const long tccs = Lc ? std::max<long>((long)Lc->count * Lc->Bp, 1) : 0;
            for (int j = 0; j < w; ++j)
                k_msp_gather<<<grid_for(total), 256, 0, s>>>(rhs + j * ldr, L.d_Sidx, Lc ? L.d_pmap : nullptr,
                                                             Lc ? W.t[d + 1] + j * tccs : nullptr, L.Sp, Fp, Lc ? Lc->Bp : 0,
                                                             total, W.g[d] + j * total);
        }
        sweep_args(d, 0, rhs, out, a, &W, &cs, ldr, ldx);
        launch_gemv2_cols(a, cs, cols_choice(d, 0, w), w, s);
        if (L.Bp > 0) {
            sweep_args(d, 1, rhs, out, a, &W, &cs, ldr, ldx);
            launch_gemv2_cols(a, cs, cols_choice(d, 1, w), w, s);
        }
    }
    for (int d = 0; d <= D; ++d) {                      // downward: root -> leaves, u_S written straight into `out`
        const Level& L = lev[d];
        if (L.gather_y) {
            const long total = (long)L.count * L.Bp;
            const long gcs = (long)L.count * (L.Sp + L.Bp);
            for (int j = 0; j < w; ++j)
                k_msp_gather<<<grid_for(total), 256, 0, s>>>(out + j * ldx, L.d_Bidx, nullptr, nullptr, L.Bp, L.Bp, 0, total,
                                                             W.g[d] + j * gcs);
        }
        sweep_args(d, 2, rhs, out, a, &W, &cs, ldr, ldx);
        launch_gemv2_cols(a, cs, cols_choice(d, 2, w), w, s);
    }
    LS_CUDA_TRY(cudaGetLastError());
    return LS_OK;
}

int Msp::solve_batch_dev(const cd* rhs, long ldr, cd* out, long ldx, int nrhs, cudaStream_t s) {
    // solver 1 (the first version, uniform batches) has no multi-column sweeps: its columns are solved one by one
    if (solver != 2) {
        for (int j = 0; j < nrhs; ++j) {
            int rc = solve_dev(rhs + j * ldr, out + j * ldx, s);
            if (rc) return rc;
        }
        return LS_OK;
    }
    if (use_graph_cols < 0) { const char* e = getenv("LS_MSP_GRAPH"); use_graph_cols = e ? atoi(e) : 1; }
    for (int j0 = 0; j0 < nrhs;) {
        const int w = chunk_width(nrhs - j0);
        const cd* r = rhs + j0 * ldr;
        cd* o = out + j0 * ldx;
        j0 += w;
        int rc;
        if (w == 1) {
            if ((rc = solve_dev(r, o, s))) return rc;
            continue;
        }
        LS_REQUIRE(!bwork[log2_width(w)].g.empty(), LS_ERR_INVALID,
                   "Msp batched solve: no work arrays for chunks of %d columns (batch_reserve first)", w);
        const int per = launches_per_solve + (w - 1) * (int)std::count_if(lev.begin(), lev.end(), [this](const Level& L) {
            return !fuse || L.gather_s; }) + (w - 1) * (int)std::count_if(lev.begin(), lev.end(), [](const Level& L) { return L.gather_y; });
        bool done = false;
        if (use_graph_cols) {
            for (auto& g : bgraphs)
                if (g.rhs == r && g.ldr == ldr && g.out == o && g.ldx == ldx && g.w == w) {
                    LS_CUDA_TRY(cudaGraphLaunch(g.exec, s));
                    done = true;
                    break;
                }
            if (!done && bgraphs.size() < 64) {
                cudaGraph_t graph = nullptr;
                cudaGraphExec_t exec = nullptr;
                if (cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
                    rc = solve_launch_cols(w, r, ldr, o, ldx, s);
                    const cudaError_t ce = cudaStreamEndCapture(s, &graph);
                    if (rc == LS_OK && ce == cudaSuccess && graph && cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess) {
                        bgraphs.push_back(CapturedB{r, ldr, o, ldx, w, exec});
                        LS_CUDA_TRY(cudaGraphLaunch(exec, s));
                        done = true;
                    }
                    if (graph) cudaGraphDestroy(graph);
                }
                if (!done) { cudaGetLastError(); use_graph_cols = 0; }
            }
        }
        if (!done && (rc = solve_launch_cols(w, r, ldr, o, ldx, s))) return rc;
        launches += per;
    }
    return LS_OK;
}

// ls_msp_factor (l = 1) and ls_msp_factor3d.  Refusals come as early and as cheaply as possible: arguments (no device
// needed), then the memory the dissection needs against the free device memory (before anything is allocated), then
// the entries as they are routed (pattern, duplicates).
static int msp_factor_entry(const char* fn, ls_handle* out, int64_t n, int64_t m, int64_t l, const int64_t* colptr,
                            const int64_t* rowval, const ls_cdouble* nzval) {
    char grid[96];
    if (l == 1) snprintf(grid, sizeof grid, "%ld x %ld", (long)n, (long)m);
    else snprintf(grid, sizeof grid, "%ld x %ld x %ld", (long)n, (long)m, (long)l);
    LS_REQUIRE(out && colptr && rowval && nzval, LS_ERR_INVALID, "%s: null pointer", fn);
    const int64_t I32 = 2147483647;
    LS_REQUIRE(n > 0 && m > 0 && l > 0 && n < I32 && m < I32 && l < I32 && n * m < I32 && n * m * l < I32, LS_ERR_INVALID,
               "%s: bad grid %s", fn, grid);
    const int64_t N = n * m * l;
    LS_REQUIRE(colptr[0] == 1, LS_ERR_INVALID, "%s: colptr must be 1-based (Julia SparseMatrixCSC)", fn);
    LS_REQUIRE(colptr[N] >= 1, LS_ERR_INVALID, "%s: colptr[end] = %ld is not a 1-based column pointer", fn, (long)colptr[N]);
    LS_REQUIRE(colptr[N] - 1 < I32, LS_ERR_UNSUPPORTED, "%s: nnz exceeds the 32-bit index range", fn);
    int leaf = 4;
    if (const char* e = getenv("LS_MSP_LEAF")) { const int v = atoi(e); if (v >= 3 && v <= 16) leaf = v; }
    int solver = 2;
    bool fuse = true, tune = true;
    if (const char* e = getenv("LS_MSP_SOLVER")) solver = atoi(e) == 1 ? 1 : 2;
    if (const char* e = getenv("LS_MSP_FUSE")) fuse = atoi(e) != 0;
    if (const char* e = getenv("LS_MSP_TUNE")) tune = atoi(e) != 0;

    lsmsp::Symbolic sym;
    sym.fn = fn;
    int rc = sym.analyse((int)n, (int)m, (int)l, leaf);
    if (rc) { set_error("%s", sym.err.c_str()); return rc; }
    {
        // cuBLAS / cuSOLVER handles and work space, allocation granularity
        const size_t reserve = (size_t)256 << 20;
        const size_t need = sym.need_bytes(colptr[N] - 1, solver == 2);
        size_t free_b = 0, total_b = 0;
        LS_CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
        LS_REQUIRE(need + reserve <= free_b, LS_ERR_NOMEM,
                   "%s: factorising the %s grid needs %zu bytes of device memory (plus %zu reserved for library work space); "
                   "%zu of %zu bytes are free", fn, grid, need, reserve, free_b, total_b);
    }

    Msp* M = new Msp();
    rc = M->init_base(KIND_MSP);
    if (rc) { delete M; return rc; }
    M->n = N; M->gn = n; M->gm = m; M->gl = l;
    M->solver = solver; M->fuse = fuse; M->tune = tune;
    if (const char* e = getenv("LS_MSP_BATCH_COLS")) { const int v = atoi(e); if (v == 2 || v == 4 || v == 8) M->cols_max = v; }
    {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, M->device) == cudaSuccess && (size_t)v > M->smem_max)
            M->smem_max = (size_t)v;
        cudaGetLastError();
    }
    rc = msp_factor(M, sym, colptr, rowval, reinterpret_cast<const cd*>(nzval));
    if (rc) { delete M; return rc; }
    if (M->solver == 2) {
        bool wide = false;
        for (Level& L : M->lev) {
            L.gather_s = M->fuse && (size_t)L.Sp * sizeof(cd) > M->smem_max;
            L.gather_y = (size_t)L.Bp * sizeof(cd) > M->smem_max;
            wide = wide || M->xs_limit(L.Sp) > GEMV2_SMEM_MAX || M->xs_limit(L.Bp) > GEMV2_SMEM_MAX;
            L.ch_sinv = lsmsp::default_choice(L.Sp, (M->fuse && !L.gather_s) ? 2 : 0);
            L.ch_fbs = lsmsp::default_choice(L.Sp, 0);
            L.ch_y = lsmsp::default_choice(L.Bp, L.gather_y ? 0 : 1);
        }
        if (wide && (rc = optin_staging(M->smem_max))) { delete M; return rc; }
        M->launches_per_solve = 0;
        for (const Level& L : M->lev)
            M->launches_per_solve += ((M->fuse && !L.gather_s) ? 0 : 1) + 2 + (L.Bp > 0 ? 1 : 0) + (L.gather_y ? 1 : 0);
        if (M->tune) rc = M->tune_sweeps();
        if (rc) { delete M; return rc; }
    }
    *out = reinterpret_cast<ls_handle>(M);
    return LS_OK;
}

extern "C" {

int ls_msp_factor(ls_handle* out, int64_t n, int64_t m, const int64_t* colptr, const int64_t* rowval, const ls_cdouble* nzval) {
    return msp_factor_entry("ls_msp_factor", out, n, m, 1, colptr, rowval, nzval);
}

int ls_msp_factor3d(ls_handle* out, int64_t n, int64_t m, int64_t l, const int64_t* colptr, const int64_t* rowval,
                    const ls_cdouble* nzval) {
    return msp_factor_entry("ls_msp_factor3d", out, n, m, l, colptr, rowval, nzval);
}

int ls_msp_solve(ls_handle h, const ls_cdouble* rhs, ls_cdouble* x, int memloc) {
    LS_REQUIRE(h && rhs && x, LS_ERR_INVALID, "ls_msp_solve: null argument");
    Msp* M = reinterpret_cast<Msp*>(h);
    LS_REQUIRE(M->kind == KIND_MSP, LS_ERR_INVALID, "ls_msp_solve: not an Msp factorisation handle");
    LS_CUDA_TRY(cudaSetDevice(M->device));
    if (memloc == LS_MEM_DEVICE)
        return M->solve_dev(reinterpret_cast<const cd*>(rhs), reinterpret_cast<cd*>(x), M->stream);
    LS_REQUIRE(memloc == LS_MEM_HOST, LS_ERR_INVALID, "ls_msp_solve: unknown memloc %d", memloc);
    const size_t bytes = (size_t)M->n * sizeof(cd);
    if (!M->d_in) {
        int rc;
        if ((rc = M->dmalloc((void**)&M->d_in, bytes))) return rc;
        if ((rc = M->dmalloc((void**)&M->d_out, bytes))) return rc;
    }
    LS_CUDA_TRY(cudaMemcpyAsync(M->d_in, rhs, bytes, cudaMemcpyHostToDevice, M->stream));
    int rc = M->solve_dev(M->d_in, M->d_out, M->stream);
    if (rc) return rc;
    LS_CUDA_TRY(cudaMemcpyAsync(x, M->d_out, bytes, cudaMemcpyDeviceToHost, M->stream));
    LS_CUDA_TRY(cudaStreamSynchronize(M->stream));
    return LS_OK;
}

// Refusals before any CUDA call: arguments, then the device memory the work arrays of this column count still need.
int ls_msp_solve_batch(ls_handle h, const ls_cdouble* rhs, int64_t ldr, ls_cdouble* x, int64_t ldx, int nrhs, int memloc) {
    LS_REQUIRE(nrhs >= 1, LS_ERR_INVALID, "ls_msp_solve_batch: nrhs = %d, at least one right-hand side needed", nrhs);
    LS_REQUIRE(h && rhs && x, LS_ERR_INVALID, "ls_msp_solve_batch: null argument");
    Msp* M = reinterpret_cast<Msp*>(h);
    LS_REQUIRE(M->kind == KIND_MSP, LS_ERR_INVALID, "ls_msp_solve_batch: not an Msp factorisation handle");
    LS_REQUIRE(memloc == LS_MEM_HOST || memloc == LS_MEM_DEVICE, LS_ERR_INVALID, "ls_msp_solve_batch: unknown memloc %d", memloc);
    const int64_t N = M->n;
    LS_REQUIRE(ldr >= N && ldx >= N, LS_ERR_INVALID, "ls_msp_solve_batch: leading dimensions ldr = %ld, ldx = %ld must be >= N = %ld",
               (long)ldr, (long)ldx, (long)N);
    {
        // x may alias rhs only column for column (same start, same leading dimension)
        const char* r0 = reinterpret_cast<const char*>(rhs);
        const char* x0 = reinterpret_cast<const char*>(x);
        const char* r1 = r0 + ((size_t)ldr * (nrhs - 1) + N) * sizeof(cd);
        const char* x1 = x0 + ((size_t)ldx * (nrhs - 1) + N) * sizeof(cd);
        const bool overlap = r0 < x1 && x0 < r1;
        LS_REQUIRE(!overlap || (r0 == x0 && ldr == ldx), LS_ERR_INVALID,
                   "ls_msp_solve_batch: x overlaps rhs other than in place (x == rhs needs ldx == ldr; ldr = %ld, ldx = %ld)",
                   (long)ldr, (long)ldx);
    }
    const bool host = memloc == LS_MEM_HOST;
    LS_CUDA_TRY(cudaSetDevice(M->device));
    const size_t need = M->batch_bytes(nrhs, host, false);
    if (need > 0) {
        size_t free_b = 0, total_b = 0;
        LS_CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
        LS_REQUIRE(need <= free_b, LS_ERR_NOMEM,
                   "ls_msp_solve_batch: work arrays for %d right-hand sides need %zu bytes of device memory; %zu of %zu bytes are free",
                   nrhs, need, free_b, total_b);
    }
    int rc = M->batch_reserve(nrhs, host, false);
    if (rc) return rc;
    if (!host)
        return M->solve_batch_dev(reinterpret_cast<const cd*>(rhs), (long)ldr, reinterpret_cast<cd*>(x), (long)ldx, nrhs, M->stream);
    // host pointers: chunks of cols_max columns through the staging buffer, solved in place there
    const cd* hr = reinterpret_cast<const cd*>(rhs);
    cd* hx = reinterpret_cast<cd*>(x);
    const size_t vb = (size_t)N * sizeof(cd);
    for (int j0 = 0; j0 < nrhs; j0 += M->cols_max) {
        const int w = std::min(nrhs - j0, M->cols_max);
        LS_CUDA_TRY(cudaMemcpy2DAsync(M->d_bstage, vb, hr + (size_t)j0 * ldr, (size_t)ldr * sizeof(cd), vb, (size_t)w,
                                      cudaMemcpyHostToDevice, M->stream));
        if ((rc = M->solve_batch_dev(M->d_bstage, (long)N, M->d_bstage, (long)N, w, M->stream))) return rc;
        LS_CUDA_TRY(cudaMemcpy2DAsync(hx + (size_t)j0 * ldx, (size_t)ldx * sizeof(cd), M->d_bstage, vb, vb, (size_t)w,
                                      cudaMemcpyDeviceToHost, M->stream));
        LS_CUDA_TRY(cudaStreamSynchronize(M->stream));
    }
    return LS_OK;
}

int ls_msp_info(ls_handle h, int64_t* factor_bytes, int* depth, double* factor_seconds) {
    LS_REQUIRE(h, LS_ERR_INVALID, "ls_msp_info: null handle");
    Msp* M = reinterpret_cast<Msp*>(h);
    LS_REQUIRE(M->kind == KIND_MSP, LS_ERR_INVALID, "ls_msp_info: not an Msp factorisation handle");
    if (factor_bytes) *factor_bytes = (int64_t)M->factor_bytes;
    if (depth) *depth = (int)M->lev.size() - 1;
    if (factor_seconds) *factor_seconds = M->factor_seconds;
    return LS_OK;
}

int ls_msp_plan(ls_handle h, char* buf, int64_t cap) {
    LS_REQUIRE(h && buf && cap > 0, LS_ERR_INVALID, "ls_msp_plan: null argument");
    Msp* M = reinterpret_cast<Msp*>(h);
    LS_REQUIRE(M->kind == KIND_MSP, LS_ERR_INVALID, "ls_msp_plan: not an Msp factorisation handle");
    std::string out;
    char line[256];
    snprintf(line, sizeof line, "solver %d fuse %d tune %d tune_seconds %.3f launches_per_solve %d factor_bytes %zu\n", M->solver,
             M->fuse ? 1 : 0, M->tune ? 1 : 0, M->tune_seconds, M->launches_per_solve, M->factor_bytes);
    out += line;
    for (size_t d = 0; d < M->lev.size(); ++d) {
        const Level& L = M->lev[d];
        snprintf(line, sizeof line, "depth %zu nodes %d Sp %d Bp %d", d, L.count, L.Sp, L.Bp);
        out += line;
        if (M->solver == 2) {
            const lsmsp::Choice* ch[3] = {&L.ch_sinv, &L.ch_fbs, &L.ch_y};
            const char* nm[3] = {"sinv", "fbs", "y"};
            for (int w = 0; w < 3; ++w) {
                snprintf(line, sizeof line, " %s L%d U%d X%d", nm[w], 1 << ch[w]->lanes_log2, 1 << ch[w]->unr_log2, ch[w]->xs);
                out += line;
                // the multi-column kernel of ls_msp_solve_batch (same LANES): UNR and XS for 2, 4 and 8 columns
                const lsmsp::Choice c2 = M->cols_choice((int)d, w, 2), c4 = M->cols_choice((int)d, w, 4), c8 = M->cols_choice((int)d, w, 8);
                snprintf(line, sizeof line, " cols U%dX%d/U%dX%d/U%dX%d", 1 << c2.unr_log2, c2.xs, 1 << c4.unr_log2, c4.xs,
                         1 << c8.unr_log2, c8.xs);
                out += line;
            }
        }
        if (M->gl > 1) out += L.lu_cusolver ? " lu cusolver" : " lu batched";
        out += "\n";
    }
    const size_t ncopy = std::min<size_t>(out.size(), (size_t)cap - 1);
    memcpy(buf, out.data(), ncopy);
    buf[ncopy] = 0;
    return LS_OK;
}

}  // extern "C"
