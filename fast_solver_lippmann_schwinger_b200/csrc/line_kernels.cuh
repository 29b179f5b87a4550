// Pruned-FFT line kernels of the Lippmann-Schwinger apply (shared by the 2-D and 3-D operators).
//
// The reference transforms the full zero-padded array (FastConvolution.jl:89-98).  With the
// Greengard-Vico padding factor 4 only 1/4 of every padded line is non-zero on the way in and
// only 1/4 is kept on the way out, and a length-4N DFT of an N-point signal splits exactly
// into four length-N DFTs of the modulated signal:
//     X[4q + r] = FFT_N( x[j] * w_{4N}^{r j} )[q],        r = 0..3
//     y[j]      = 1/4 * sum_r conj(w_{4N}^{r j}) * IFFT_N( Y[4q + r] )[j],   j < N.
// A padded line is therefore stored as 4 blocks (r) of N "slots" (the engine's output order).
//
// Line addressing: point p of line L sits at base + L*ls + p*es (elements of 16 B).
//   mode A kernels: the threads of one line are consecutive lanes (contiguous lines);
//   mode B kernels: eight adjacent lines are interleaved across lanes (lane%8 = line) so that
//                   strided lines (es large, ls == 1) are read/written as 128-byte segments.
#pragma once
#include <cuda.h>   // CUtensorMap (the type only: the maps are encoded through the runtime's driver entry point)
#include "fft_engine.cuh"

namespace lsk {
using namespace lsfft;

template <int N> struct GeoA {
    static constexpr int E = Cfg<N>::E;
    static constexpr int T = N / E;
    static constexpr int LPC = (T >= 128) ? 1 : 128 / T;   // lines per CTA
    static constexpr int THREADS = T * LPC;
};
template <int N> struct GeoB {
    static constexpr int E = Cfg<N>::E;
    static constexpr int T = N / E;
    static constexpr int LB = LinesB<N>::value;             // lines interleaved across lanes (8; 4 for 512-point lines)
    static constexpr int GPC = (LB * T >= 128) ? 1 : 128 / (LB * T);     // groups of LB lines per CTA
    static constexpr int LPC = LB * GPC;
    static constexpr int THREADS = LB * T * GPC;
};
// resident CTAs per SM asked of ptxas: 128-thread CTAs 3 (168 registers); the 256-thread CTAs of the 4-line mode-B
// geometry 2 (128 registers: E = 8 points per thread there); everything else 1
template <int N, bool MODE_B> struct MinB {
    static constexpr int TH = MODE_B ? GeoB<N>::THREADS : GeoA<N>::THREADS;
    static constexpr int value = (TH <= 128) ? 3 : ((MODE_B && GeoB<N>::LB == 4 && TH == 256) ? 2 : 1);
};
// the inverse pass keeps E accumulators next to the E working values: at 512 points (E = 16 since r2) the 168-register
// cap of three CTAs per SM spills inside the loop, so it asks for two.  Measured on B200
// (profiles/r2_l_512_variants.log): 512^3 P4 3.67 -> 3.19 ms, 2-D 512^2 apply 0.0353 -> 0.0332 ms.
template <int N, bool MODE_B> struct MinBInv {
    static constexpr int value = (N == 512 && MinB<N, MODE_B>::value == 3) ? 2 : MinB<N, MODE_B>::value;
};

// thread -> (line within CTA, thread within line, smem layout)
template <int N, bool MODE_B> struct Map;
template <int N> struct Map<N, false> {
    typedef GeoA<N> G;
    typedef LayA<N> Lay;
    int line, t;
    Lay lay;
    __device__ __forceinline__ Map() {
        line = threadIdx.x / G::T;
        t = threadIdx.x % G::T;
        lay.base = line * N;
    }
    __device__ __forceinline__ int lay_lam() const { return 0; }
};
template <int N> struct Map<N, true> {
    typedef GeoB<N> G;
    typedef LayB<N> Lay;
    int line, t;
    Lay lay;
    __device__ __forceinline__ Map() {
        constexpr int LB = G::LB;
        int grp = threadIdx.x / (LB * G::T);
        int w = threadIdx.x % (LB * G::T);
        lay.lam = w % LB;
        t = w / LB;
        line = grp * LB + lay.lam;
        smoff = grp * LB * N;
    }
    int smoff;
    __device__ __forceinline__ int lay_lam() const { return lay.lam; }
};
template <int N> __device__ __forceinline__ int sm_group_off(const Map<N, false>&) { return 0; }
template <int N> __device__ __forceinline__ int sm_group_off(const Map<N, true>& m) { return m.smoff; }

// Two-level line addressing: line L = l0 + ldim0*l1 starts at l0*ls0 + l1*ls1; its points/slots
// are `es` elements apart.  (2-D uses one level; 3-D y-lines are indexed by (x slot, z plane).)
struct LineAddr {
    long ldim0;
    long in_ls0, in_ls1, in_es;
    long out_ls0, out_ls1, out_es;
    // slab split of the 4N-slot axis (multi-GPU transposes): slot s lives at
    // (s & (2^shift - 1))*es + (s >> shift)*split_stride.  shift = 62 disables it.
    int split_shift = 62;
    // MASK instantiations only: lines >= mask_lines read as zero (forward) / are not written (inverse).  32 bits (3-D
    // line counts reach 2^19) in the alignment gap after split_shift: no other member moves.
    int mask_lines = 0;
    long split_stride = 0;
    // optional second level (x-slot chunks inside a rank's slab, pipelined transposes): bits
    // [split_shift, split2_shift) select the chunk (stride split_stride), bits >= split2_shift the
    // rank (stride split2_stride).  split2_shift = 62 leaves the one-level rule above.
    int split2_shift = 62;
    long split2_stride = 0;
    // padding factor of the line: nr = 4 sub-transforms r = 0..3 (the reference's 4N zero padding) or
    // nr = 2 (r = 0, 2 in units of w_4N: a 2N padding, enough once the kernel is restricted to lags (-N, N))
    int nr = 4;
    int cblock = 0;     // inverse: which N-block [cblock*N, (cblock+1)*N) of the padded output line is kept
    int full2 = 0;      // forward: the input line has 2N points (no zero padding), nr must be 2
    // MASK instantiations only (zero-embedded sizes, op2d.cu, op3d.cu): points >= mask_pts of a line read as zero
    // (forward) / are not written (inverse).  16 bits suffice (<= 4096) and fill the tail padding: the struct stays
    // 104 bytes, so the parameter layout of every unmasked kernel is unchanged.
    int16_t mask_pts = 0;
};
static_assert(sizeof(LineAddr) == 104, "LineAddr: kernel parameter layout");
static_assert(offsetof(LineAddr, split_stride) == 64 && offsetof(LineAddr, nr) == 88, "LineAddr: member offsets");
__device__ __forceinline__ long slot_off(const LineAddr& a, long s, long es) {
    return (s & ((1L << a.split_shift) - 1)) * es
         + ((s & ((1L << a.split2_shift) - 1)) >> a.split_shift) * a.split_stride
         + (s >> a.split2_shift) * a.split2_stride;
}
// Column pointers of k_fwd_pruned and k_inv_pruned: column c reads its lines at in[c] (and b at b[c]) and writes them
// at out[c], with the one LineAddr of the launch.  The COLS instantiations serve a launch over several columns
// (ls_op_apply_batch), column c = blockIdx.y; the others read column 0 at fixed parameter offsets.  A pointer loaded by
// block index has to live in registers, which costs the single apply spills at the 168-register cap (ptxas: 2-D P1 at
// 2048 points 140 -> 164 bytes), so the single apply keeps the fixed-offset instantiation.
constexpr int MAX_COLS = 8;
struct ColPtrs {
    const cd* in[MAX_COLS];
    const cd* b[MAX_COLS];
    cd* out[MAX_COLS];
};
__device__ __forceinline__ long line_in(const LineAddr& a, long L) { return (L % a.ldim0) * a.in_ls0 + (L / a.ldim0) * a.in_ls1; }
__device__ __forceinline__ long line_out(const LineAddr& a, long L) { return (L % a.ldim0) * a.out_ls0 + (L / a.ldim0) * a.out_ls1; }

// per-CTA shared memory: [exchange: LPC*N][(mid only) x copy: LPC*N][(mid, mode B only) spectrum: LPC*N][tw1][mbarrier]
// (k_mid_swap: [exchange][lines: LPC*N][tw1][mbarrier], sized in launch_mid_swap)
template <int N, bool MODE_B> struct Smem {
    static constexpr int LPC = MODE_B ? GeoB<N>::LPC : GeoA<N>::LPC;
    static constexpr int TW1N = EngTab<N>::TW1N;
    static constexpr int fwd_bytes = (LPC * N + TW1N) * (int)sizeof(cd);
    static constexpr int mid_bytes = ((MODE_B ? 3 : 2) * LPC * N + TW1N) * (int)sizeof(cd) + 16;
};

// ---- forward, pruned: N inputs -> 4N slots -------------------------------------------
// in  : line L point j at in[L*in_ls + j*in_es], optionally scaled by the real nu (same addressing)
// out : line L slot  s at out[L*out_ls + s*out_es], s = r*N + slot
// MASK: points >= la.mask_pts and lines >= la.mask_lines are zeros (not read); their slots are written
template <int N, bool MODE_B, bool MASK = false, bool COLS = false>
__global__ void __launch_bounds__(MODE_B ? GeoB<N>::THREADS : GeoA<N>::THREADS, MinB<N, MODE_B>::value)
k_fwd_pruned(const ColPtrs cp, const double* __restrict__ nu, const cd* __restrict__ TAB, const LineAddr la, long line0) {
    typedef Map<N, MODE_B> M;
    const cd* __restrict__ in = cp.in[COLS ? blockIdx.y : 0];
    cd* __restrict__ out = cp.out[COLS ? blockIdx.y : 0];
    constexpr int E = Cfg<N>::E, T = N / E, LPC = M::G::LPC;
    extern __shared__ __align__(128) cd sm[];
    M mp;
    cd* ex = sm + sm_group_off(mp);
    cd* tw1 = sm + LPC * N;
    load_tw1<N>(tw1, TAB);
    const long L = line0 + (long)blockIdx.x * LPC + mp.line;
    const int t = mp.t;
    const TwState<N> tw = make_tw<N>(t, TAB, tw1);
    const long in_base = line_in(la, L), out_base = line_out(la, L);
    const long in_es = la.in_es, out_es = la.out_es;
    const int npts = (!MASK || L < la.mask_lines) ? la.mask_pts : 0;   // MASK: valid points of this line
    cd x[E];
#pragma unroll
    for (int a = 0; a < E; ++a) {
        if (MASK && a * T + t >= npts) {
            x[a] = make_double2(0.0, 0.0);
            continue;
        }
        long off = in_base + (long)(a * T + t) * in_es;
        cd val = in[off];
        if (nu != nullptr) {
            double s = nu[off];
            val.x *= s;
            val.y *= s;
        }
        x[a] = val;
    }
    __syncthreads();   // tw1 visible
    const int nr = la.nr, rstep = 4 / la.nr;
#pragma unroll 1
    for (int rr = 0; rr < nr; ++rr) {
        const int r = rr * rstep;
        cd v[E];
        if (la.full2) {
            // unpadded 2N-point line (setup only): first DIF stage x[j] +- x[j + N]
#pragma unroll
            for (int a = 0; a < E; ++a) {
                const cd hi = in[in_base + (long)(N + a * T + t) * in_es];
                v[a] = rr == 0 ? cadd(x[a], hi) : csub(x[a], hi);
            }
        } else {
#pragma unroll
            for (int a = 0; a < E; ++a) v[a] = x[a];
        }
        fft_fwd<N>(v, t, r, ex, mp.lay, tw);
        cd* o = out + out_base;
#pragma unroll
        for (int e = 0; e < E; ++e) o[slot_off(la, (long)(rr * N + t + T * e), out_es)] = v[e];
        __syncthreads();   // next forward rewrites the exchange buffer at other addresses
    }
}

// ---- middle, fused: 4x (forward, multiply by the Green's spectrum, inverse) --------------
// in  : line L point j at in[L*in_ls + j*in_es]
// G   : spectrum of line L, block r, slot s at G[(L*4 + r)*N + s]                 (mode A)
//       or at G[((L/8)*4 + r)*8N + s*8 + L%8]                                     (mode B)
//       mode A: the values go straight from memory into registers, requested before the last butterfly stage
//       mode B: per (unit, r) one contiguous chunk, fetched by TMA bulk copy into shared memory
//               while the previous block's inverse transform runs.
// out : line L point j at out[L*out_ls + j*out_es]  (may alias in when strides agree)
// Several columns (ncol > 1, mode B: the 3-D z pass): column c's lines start at in + c*cs / out + c*cs.  CTA x = g*ncol + c
// serves the line group g of column c: the ncol CTAs that read the same spectrum chunk are dispatched together, and all
// but the first find it in L2.  Mode A (the 2-D middle pass with LS_FLAG_PAD4) runs one column: the column arithmetic
// costs it spills (ptxas: 24 - 52 bytes at 1024 - 4096 points).
template <int N, bool MODE_B, int MINB = 1>
__global__ void __launch_bounds__(MODE_B ? GeoB<N>::THREADS : GeoA<N>::THREADS, MINB)
k_mid_fused(const cd* in, cd* out, const cd* __restrict__ G, const cd* __restrict__ TAB,
            const LineAddr la, long line0, int ncol, long cs) {
    typedef Map<N, MODE_B> M;
    constexpr int E = Cfg<N>::E, T = N / E, LPC = M::G::LPC;
    constexpr int LBK = MODE_B ? GeoB<N>::LB : 1;     // lines interleaved in a spectrum chunk
    constexpr int UNIT = LBK * N;                     // points per spectrum chunk
    constexpr int UPC = LPC * N / UNIT;               // chunks per CTA and r
    extern __shared__ __align__(128) cd sm[];
    M mp;
    cd* ex = sm + sm_group_off(mp);
    cd* xs = sm + LPC * N + sm_group_off(mp);   // thread-private copy of the input line
    cd* gb = sm + 2 * LPC * N;                  // spectrum chunk(s) of the current r (mode B only)
    cd* tw1 = sm + (MODE_B ? 3 : 2) * LPC * N;
    unsigned long long* bar = reinterpret_cast<unsigned long long*>(tw1 + Smem<N, MODE_B>::TW1N);
    long grp = blockIdx.x;
    if constexpr (MODE_B) {
        const int col = (int)(blockIdx.x % (unsigned)ncol);
        in += col * cs;
        out += col * cs;
        grp = blockIdx.x / (unsigned)ncol;
    }
    const long Lcta = line0 + grp * LPC;
    const long L = Lcta + mp.line;
    const int t = mp.t;
    const int nr = la.nr, rstep = 4 / la.nr;
    const cd* gsrc = G + (Lcta / LBK) * (long)nr * UNIT;   // chunk (unit u, rr) at gsrc + (u*nr + rr)*UNIT

    auto issue_g = [&](int rr) {
        mbar_expect_tx(bar, (unsigned)(UPC * UNIT * sizeof(cd)));
#pragma unroll
        for (int u = 0; u < UPC; ++u)
            bulk_g2s(gb + u * UNIT, gsrc + ((long)u * nr + rr) * UNIT, (unsigned)(UNIT * sizeof(cd)), bar);
    };
    if (MODE_B && threadIdx.x == 0) {
        mbar_init(bar, 1);
        fence_proxy_async();
        issue_g(0);
    }
    load_tw1<N>(tw1, TAB);
    const TwState<N> tw = make_tw<N>(t, TAB, tw1);
    {
        const cd* p = in + line_in(la, L) + (long)t * la.in_es;
#pragma unroll
        for (int a = 0; a < E; ++a) xs[mp.lay.phys(a * T + t)] = p[(long)(a * T) * la.in_es];
    }
    // mode A: pull spectrum chunk r into L2 one r ahead (one request per 128-byte line)
    auto prefetch_g = [&](int rr) {
        if (!MODE_B && rr < nr) {
            const cd* g = gsrc + ((long)mp.line * nr + rr) * UNIT;
            if ((t & 7) == 0) {
#pragma unroll
                for (int e = 0; e < E; ++e) prefetch_l2(&g[t + T * e]);
            }
        }
    };
    prefetch_g(0);
    __syncthreads();   // tw1 + mbarrier init visible
    cd acc[E];
#pragma unroll 1
    for (int rr = 0; rr < nr; ++rr) {
        const int r = rr * rstep;
        cd v[E];
#pragma unroll
        for (int a = 0; a < E; ++a) v[a] = xs[mp.lay.phys(a * T + t)];
        prefetch_g(rr + 1);
        if (MODE_B) {
            fft_fwd<N>(v, t, r, ex, mp.lay, tw);
            mbar_wait(bar, (unsigned)(rr & 1));
            const cd* g = gb + sm_group_off(mp);
#pragma unroll
            for (int e = 0; e < E; ++e) v[e] = cmul(v[e], g[(t + T * e) * LBK + mp.lay_lam()]);
        } else {
            // spectrum values are requested before the last butterfly stage and consumed after it
            cd gv[E];
            fft_fwd<N>(v, t, r, ex, mp.lay, tw, [&]() {
                const cd* g = gsrc + ((long)mp.line * nr + rr) * UNIT;
#pragma unroll
                for (int e = 0; e < E; ++e) gv[e] = __ldg(&g[t + T * e]);
            });
#pragma unroll
            for (int e = 0; e < E; ++e) v[e] = cmul(v[e], gv[e]);
        }
        fft_inv<N>(v, t, r, ex, mp.lay, tw, [&]() {
            // every thread has consumed gb (the multiply precedes this barrier): refill it
            if (MODE_B && rr + 1 < nr && threadIdx.x == 0) {
                fence_proxy_async();
                issue_g(rr + 1);
            }
        });
        demod_accumulate<N>(acc, v, r);
    }
    cd* o = out + line_out(la, L) + (long)t * la.out_es;
#pragma unroll
    for (int a = 0; a < E; ++a) o[(long)(a * T) * la.out_es] = acc[a];
}

// ---- middle, fused, 2x padding, no accumulator registers ("swap" variant, mode A) ----------------------------
// Same arithmetic and the same bits as k_mid_fused with nr = 2 in mode A.  k_mid_fused keeps the input line in shared
// memory AND 16 accumulators in registers.  With two sub-transforms only one thread-private buffer is needed: it
// holds the input line x while r = 0 is transformed, then x and the r = 0 result trade places (each thread swaps
// its own 16 elements, no barrier), and the r = 2 result is combined with the held one on the way out.  The spectrum
// values are requested before the last butterfly stage and held in registers across it.
// The lines move by tensor copies, not through the load/store pipe: their points are one x-slot (16 bytes) wide in
// A and CW-interleaved in C, so an LSU access of a line used 16 bytes of every 128-byte (A) or 64-byte (C) line.
// tmA: 3-D map of A as FLOAT64 {2 pn, lm, cols}; line L of column c is the boxes {2, BOX, 1} at (2L, j0, c).  tmC: 4-D
// map of C {2 CW, lm, pn/CW, cols}; line L of column c is the boxes {2, BOX, 1, 1} at (2 (L % CW), j0, L / CW, c),
// CW = 2^CWS.  Column c's C starts at C + c*ccs.  The grid is {columns, pn / LPC}: the CTAs of one line group, which
// read the same spectrum lines, are dispatched together, and all but the first find those lines in L2.  BOX = min(N, 256);
// each line of the CTA has its own N / BOX boxes.  Thread 0 issues the loads into the buffer first thing (the table
// set-up runs under them) and, after the combine has been written back into the same buffer, the stores.
// With one resident CTA per SM (MINB = 1: N = 4096) the stores go through the load/store pipe instead: the CTA has to
// wait until the tensor stores have read its shared memory before it exits, and no second CTA on the SM covers that
// wait.  Measured on B200 (1000 W) at 4096^2 (apply, profiles/r4_p2_tma.log): TMA loads + LSU stores 1.498 ms, TMA both
// ways 1.640 ms, LSU both ways 1.568 ms; at 2048^2 TMA both ways is the fastest (0.3025 / 0.309 / 0.336 ms).
template <int N, int MINB, int CWS>
__global__ void __launch_bounds__(GeoA<N>::THREADS, MINB)
k_mid_swap(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmC, cd* C, long ccs,
           const cd* __restrict__ G, const cd* __restrict__ TAB) {
    typedef Map<N, false> M;
    constexpr int E = Cfg<N>::E, T = N / E, LPC = M::G::LPC;
    constexpr int BOX = N < 256 ? N : 256, NBOX = N / BOX;
    constexpr bool TMA_STORE = MINB > 1;
    extern __shared__ __align__(128) cd sm[];
    M mp;
    cd* ex = sm;
    cd* lines = sm + LPC * N;                       // line l of the CTA, point j at lines[l*N + j]
    cd* hold = lines + mp.line * N + mp.t;          // element a of this thread at hold[a*T]
    cd* tw1 = sm + 2 * LPC * N;
    unsigned long long* bar = reinterpret_cast<unsigned long long*>(tw1 + EngTab<N>::TW1N);
    const int L0 = blockIdx.y * LPC;        // column blockIdx.x (read where used: nothing holds it across the transforms)
    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        fence_proxy_async();
        mbar_expect_tx(bar, (unsigned)(LPC * N * sizeof(cd)));
#pragma unroll
        for (int l = 0; l < LPC; ++l)
#pragma unroll
            for (int b = 0; b < NBOX; ++b) tma_load_3d(lines + l * N + b * BOX, &tmA, 2 * (L0 + l), b * BOX, blockIdx.x, bar);
    }
    load_tw1<N>(tw1, TAB);
    const long L = L0 + mp.line;
    const int t = mp.t;
    const TwState<N> tw = make_tw<N>(t, TAB, tw1);
    const cd* gline = G + L * 2L * N;               // chunk rr of line L at gline + rr*N
    __syncthreads();   // tw1 and the mbarrier initialisation visible
    mbar_wait(bar, 0);
    cd v[E];
#pragma unroll
    for (int a = 0; a < E; ++a) v[a] = hold[a * T];
#pragma unroll 1
    for (int rr = 0; rr < 2; ++rr) {
        const int r = 2 * rr;
        const cd* g = gline + (long)rr * N;
        cd gv[E];
        fft_fwd<N>(v, t, r, ex, mp.lay, tw, [&]() {
#pragma unroll
            for (int e = 0; e < E; ++e) gv[e] = __ldg(&g[t + T * e]);
        });
#pragma unroll
        for (int e = 0; e < E; ++e) v[e] = cmul(v[e], gv[e]);
        fft_inv<N>(v, t, r, ex, mp.lay, tw);
        if (rr == 0) {
            // x and the r = 0 result trade places
#pragma unroll
            for (int a = 0; a < E; ++a) {
                const cd xa = hold[a * T];
                hold[a * T] = v[a];
                v[a] = xa;
            }
        }
    }
    if constexpr (!TMA_STORE) {
        // point j of line L at C[(L / CW)*(CW*N) + CW*j + L % CW] (< 2^25 elements: int offsets)
        const int l = (int)L;
        cd* o = C + blockIdx.x * ccs + (((l >> CWS) * N) << CWS) + (l & ((1 << CWS) - 1)) + (t << CWS);
        o[0] = cadd(hold[0], v[0]);
#pragma unroll
        for (int a = 1; a < E; ++a) o[(a * T) << CWS] = cfmac(v[a], c64(2 * a * (16 / E)), hold[a * T]);
        return;
    }
    hold[0] = cadd(hold[0], v[0]);
#pragma unroll
    for (int a = 1; a < E; ++a) hold[a * T] = cfmac(v[a], c64(2 * a * (16 / E)), hold[a * T]);
    fence_proxy_async();   // these shared-memory writes before the tensor stores read them
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
        for (int l = 0; l < LPC; ++l)
#pragma unroll
            for (int b = 0; b < NBOX; ++b)
                tma_store_4d(&tmC, 2 * ((L0 + l) & ((1 << CWS) - 1)), b * BOX, (L0 + l) >> CWS, blockIdx.x, lines + l * N + b * BOX);
        bulk_store_drain();   // the CTA's shared memory must outlive the stores' reads of it
    }
}

// cp.async helpers (inverse pass staging)
__device__ __forceinline__ void cp_async16(void* dst_smem, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int K> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(K) : "memory"); }

// ---- inverse, pruned: 4N slots -> N outputs, optional identity-plus-contrast combine --
// in  : line L slot s at in[L*in_ls + s*in_es]
// out : line L point j at out[L*out_ls + j*out_es];  if bsrc: out = bsrc + scale*result
// STAGED: the next slot block (at the end, the b values) is staged in shared memory by cp.async while the current
// block is transformed (each thread stages exactly the elements it consumes: no extra barrier), which takes two of
// the kernel's three exposed DRAM latencies off the critical path.  The applies run staged; the set-up passes of the
// compact spectrum do not.
// MASK: only points < la.mask_pts of lines < la.mask_lines are written (and only their b values staged)
template <int N, bool MODE_B, bool STAGED = false, bool MASK = false, bool COLS = false>
__global__ void __launch_bounds__(MODE_B ? GeoB<N>::THREADS : GeoA<N>::THREADS, MinBInv<N, MODE_B>::value)
k_inv_pruned(const ColPtrs cp, const cd* __restrict__ TAB, double scale, const LineAddr la, long line0) {
    typedef Map<N, MODE_B> M;
    const cd* __restrict__ in = cp.in[COLS ? blockIdx.y : 0];
    const cd* bsrc = cp.b[COLS ? blockIdx.y : 0];
    cd* out = cp.out[COLS ? blockIdx.y : 0];
    constexpr int E = Cfg<N>::E, T = N / E, LPC = M::G::LPC;
    extern __shared__ __align__(128) cd sm[];
    M mp;
    cd* ex = sm + sm_group_off(mp);
    cd* tw1 = sm + LPC * N;
    load_tw1<N>(tw1, TAB);
    const long L = line0 + (long)blockIdx.x * LPC + mp.line;
    const int t = mp.t;
    const TwState<N> tw = make_tw<N>(t, TAB, tw1);
    __syncthreads();
    const long in_base = line_in(la, L), out_base = line_out(la, L);
    cd acc[E];
    const int nr = la.nr, rstep = 4 / la.nr;
    constexpr int TH = MODE_B ? GeoB<N>::THREADS : GeoA<N>::THREADS;
    cd* stg = sm + LPC * N + EngTab<N>::TW1N + threadIdx.x;      // STAGED: element e of this thread at stg[TH*e]
    const int npts = (!MASK || L < la.mask_lines) ? la.mask_pts : 0;   // MASK: kept points of this line
#pragma unroll 1
    for (int rr = 0; rr < nr; ++rr) {
        const int r = rr * rstep;
        cd v[E];
        const cd* p = in + in_base;
        if (STAGED && rr > 0) {
            cp_async_wait<0>();
#pragma unroll
            for (int e = 0; e < E; ++e) v[e] = stg[TH * e];
        } else {
#pragma unroll
            for (int e = 0; e < E; ++e) v[e] = p[slot_off(la, (long)(rr * N + t + T * e), la.in_es)];
        }
        if (STAGED) {
            if (rr + 1 < nr) {
#pragma unroll
                for (int e = 0; e < E; ++e) cp_async16(&stg[TH * e], &p[slot_off(la, (long)((rr + 1) * N + t + T * e), la.in_es)]);
                cp_async_commit();
            } else if (bsrc != nullptr) {
#pragma unroll
                for (int a = 0; a < E; ++a)
                    if (!MASK || a * T + t < npts) cp_async16(&stg[TH * a], &bsrc[out_base + (long)(a * T + t) * la.out_es]);
                cp_async_commit();
            }
        }
        fft_inv<N>(v, t, r, ex, mp.lay, tw);
        if (la.cblock == 0) demod_accumulate<N>(acc, v, r);
        else demod_accumulate_block<N>(acc, v, r, 16 * r * la.cblock);     // kept block c: extra factor w_4^(-r c)
        __syncthreads();
    }
    if (MASK && STAGED && bsrc != nullptr) cp_async_wait<0>();
#pragma unroll
    for (int a = 0; a < E; ++a) {
        if (MASK && a * T + t >= npts) continue;
        long off = out_base + (long)(a * T + t) * la.out_es;
        cd res = cscale(acc[a], scale);
        if (bsrc != nullptr) {
            if (STAGED && a == 0) cp_async_wait<0>();
            const cd bv = STAGED ? stg[TH * a] : bsrc[off];
            res = make_double2(__fma_rn(acc[a].x, scale, bv.x), __fma_rn(acc[a].y, scale, bv.y));   // one rounding, same bits staged or not
        }
        out[off] = res;
    }
}

}  // namespace lsk

// ---- host-side launchers ----------------------------------------------------------------
namespace lsk {

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device attribute and a process may hold handles on several
// GPUs (ls_set_device): opt in once per (kernel instantiation, device).  `done` = the call site's static bit mask.
template <class K> inline cudaError_t smem_optin(K kernel, int smem, unsigned long long& done) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const unsigned long long bit = 1ull << (dev & 63);
    if (done & bit) return cudaSuccess;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) done |= bit;
    return e;
}

// MASK launchers cover ceil(nlines / LPC) CTAs: nlines need not be a multiple of the lines per CTA (the lines past
// nlines in the last CTA are masked by la.mask_lines and must still be addressable for the unmasked side)
// the pointer list of one column
inline ColPtrs one_col(const cd* in, const cd* b, cd* out) {
    ColPtrs cp = {};
    cp.in[0] = in; cp.b[0] = b; cp.out[0] = out;
    return cp;
}

template <int N, bool B, bool MASK = false>
inline cudaError_t launch_fwd_cols(cudaStream_t s, long nlines, const ColPtrs& cp, int ncol, const double* nu, const cd* TAB,
                                   const LineAddr& la) {
    constexpr int smem = Smem<N, B>::fwd_bytes;
    constexpr int LPC = Smem<N, B>::LPC, TH = B ? GeoB<N>::THREADS : GeoA<N>::THREADS;
    static unsigned long long optin = 0;
    const long grid = MASK ? (nlines + LPC - 1) / LPC : nlines / LPC;
    if (ncol == 1) {
        { cudaError_t e = smem_optin(k_fwd_pruned<N, B, MASK>, smem, optin); if (e != cudaSuccess) return e; }
        k_fwd_pruned<N, B, MASK><<<(unsigned)grid, TH, smem, s>>>(cp, nu, TAB, la, 0);
    } else {
        static unsigned long long optin_cols = 0;
        { cudaError_t e = smem_optin(k_fwd_pruned<N, B, MASK, true>, smem, optin_cols); if (e != cudaSuccess) return e; }
        k_fwd_pruned<N, B, MASK, true><<<dim3((unsigned)grid, (unsigned)ncol), TH, smem, s>>>(cp, nu, TAB, la, 0);
    }
    return cudaPeekAtLastError();
}
template <int N, bool B, bool MASK = false>
inline cudaError_t launch_fwd(cudaStream_t s, long nlines, const cd* in, const double* nu, cd* out, const cd* TAB,
                              const LineAddr& la) {
    return launch_fwd_cols<N, B, MASK>(s, nlines, one_col(in, nullptr, out), 1, nu, TAB, la);
}

template <int N, bool B>
inline cudaError_t launch_mid(cudaStream_t s, long nlines, const cd* in, cd* out, const cd* G, const cd* TAB,
                              const LineAddr& la, int ncol = 1, long cs = 0) {
    constexpr int smem = Smem<N, B>::mid_bytes;
    constexpr int LPC = Smem<N, B>::LPC, TH = B ? GeoB<N>::THREADS : GeoA<N>::THREADS;
    static unsigned long long optin = 0;
    constexpr int MB = (B && GeoB<N>::LB == 4) ? 2 : 1;      // 4-line geometry: two CTAs per SM (128 registers)
    if (!B && ncol != 1) return cudaErrorInvalidValue;         // mode A runs one column (k_mid_fused)
    { cudaError_t e = smem_optin(k_mid_fused<N, B, MB>, smem, optin); if (e != cudaSuccess) return e; }
    k_mid_fused<N, B, MB><<<(unsigned)(nlines / LPC * ncol), TH, smem, s>>>(in, out, G, TAB, la, 0, ncol, cs);
    return cudaPeekAtLastError();
}

// CTAs per SM asked of ptxas: 3 up to N = 256, 2 from 512 to 2048, 1 at 4096 (256-thread CTAs).  Measured on B200
// (profiles/r2_e_notes.md) before the lines moved by tensor copies: at N >= 1024 three CTAs were slower than two
// (168-register cap -> spills, and 3 x 66 KB of shared memory left 30 KB of L1 for the then strided LSU line loads:
// 2048^2 0.297 vs 0.211 ms); at small N several lines share a CTA and three CTAs win.  At the 168-register cap of three
// CTAs the 256- and 128-point kernels still spill (ptxas: 76 and 4 bytes; 116 and 84 before the tensor copies); the
// others do not spill (2048: 254 registers).
template <int N, int CWS>
inline cudaError_t launch_mid_swap(cudaStream_t s, long nlines, const CUtensorMap& tmA, const CUtensorMap& tmC, cd* C,
                                   const cd* G, const cd* TAB, int ncol = 1, long ccs = 0) {
    constexpr int MINB = GeoA<N>::THREADS > 128 ? 1 : (N <= 256 ? 3 : 2);
    constexpr int smem = (2 * GeoA<N>::LPC * N + EngTab<N>::TW1N) * (int)sizeof(cd) + 8;
    static unsigned long long optin = 0;
    { cudaError_t e = smem_optin(k_mid_swap<N, MINB, CWS>, smem, optin); if (e != cudaSuccess) return e; }
    k_mid_swap<N, MINB, CWS><<<dim3((unsigned)ncol, (unsigned)(nlines / GeoA<N>::LPC)), GeoA<N>::THREADS, smem, s>>>(tmA, tmC, C, ccs, G, TAB);
    return cudaPeekAtLastError();
}

template <int N, bool B, bool STAGED = false, bool MASK = false>
inline cudaError_t launch_inv_cols(cudaStream_t s, long nlines, const ColPtrs& cp, int ncol, const cd* TAB, double scale,
                                   const LineAddr& la) {
    constexpr int smem = Smem<N, B>::fwd_bytes + (STAGED ? Smem<N, B>::LPC * N * (int)sizeof(cd) : 0);
    constexpr int LPC = Smem<N, B>::LPC, TH = B ? GeoB<N>::THREADS : GeoA<N>::THREADS;
    static unsigned long long optin = 0;
    const long grid = MASK ? (nlines + LPC - 1) / LPC : nlines / LPC;
    if (ncol == 1) {
        { cudaError_t e = smem_optin(k_inv_pruned<N, B, STAGED, MASK>, smem, optin); if (e != cudaSuccess) return e; }
        k_inv_pruned<N, B, STAGED, MASK><<<(unsigned)grid, TH, smem, s>>>(cp, TAB, scale, la, 0);
    } else {
        static unsigned long long optin_cols = 0;
        { cudaError_t e = smem_optin(k_inv_pruned<N, B, STAGED, MASK, true>, smem, optin_cols); if (e != cudaSuccess) return e; }
        k_inv_pruned<N, B, STAGED, MASK, true><<<dim3((unsigned)grid, (unsigned)ncol), TH, smem, s>>>(cp, TAB, scale, la, 0);
    }
    return cudaPeekAtLastError();
}
template <int N, bool B, bool STAGED = false, bool MASK = false>
inline cudaError_t launch_inv(cudaStream_t s, long nlines, const cd* in, const cd* bsrc, cd* out, const cd* TAB,
                              double scale, const LineAddr& la) {
    return launch_inv_cols<N, B, STAGED, MASK>(s, nlines, one_col(in, bsrc, out), 1, TAB, scale, la);
}

}  // namespace lsk
