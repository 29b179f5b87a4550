// Register-resident complex128 line-FFT engine for sm_100a.
//
// One line of N points (N = 2^6..2^12) is owned by T = N/E threads, E = 8 or 16 points per
// thread.  Stages are radix 8/16 butterflies done entirely in registers; between stages
// the points are exchanged through shared memory *in place* (stage i reads and writes the
// same set of addresses per thread), so one __syncthreads() per exchange is enough and
// the forward -> spectrum multiply -> inverse chain of the Lippmann-Schwinger apply never
// needs a reorder:
//   forward  = decimation in frequency: natural order in, "slot" order out;
//   inverse  = the exact adjoint network: slot order in, natural order out.
// The Green's spectrum is permuted once at create time into slot order, so no bit/digit
// reversal ever runs on the device hot path.
//
// Shared-memory exchange patterns were checked bank-conflict free for every size with the
// XOR swizzle below (128-bit accesses are served per quarter warp = 8 lanes).
#pragma once
#include <cuda_runtime.h>
#include "w64_table.cuh"

namespace lsfft {

typedef double2 cd;

__device__ __forceinline__ cd cadd(cd a, cd b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ cd csub(cd a, cd b) { return make_double2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ cd cmul(cd a, cd b) {
    return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
// a * conj(b)
__device__ __forceinline__ cd cmulc(cd a, cd b) {
    return make_double2(a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y);
}
__device__ __forceinline__ cd cscale(cd a, double s) { return make_double2(a.x * s, a.y * s); }
// a + b*c
__device__ __forceinline__ cd cfma(cd b, cd c, cd a) {
    return make_double2(a.x + (b.x * c.x - b.y * c.y), a.y + (b.x * c.y + b.y * c.x));
}
// a + b*conj(c)
__device__ __forceinline__ cd cfmac(cd b, cd c, cd a) {
    return make_double2(a.x + (b.x * c.x + b.y * c.y), a.y + (b.y * c.x - b.x * c.y));
}

// DIR = -1: forward kernel e^{-2 pi i jk/N};  DIR = +1: inverse (unnormalised).
// multiply by DIR*i
template <int DIR> __device__ __forceinline__ cd mul_i(cd a) {
    if (DIR < 0) return make_double2(a.y, -a.x);
    return make_double2(-a.y, a.x);
}

// multiply by exp(DIR * 2 pi i * K / 16), K compile time
template <int DIR, int K> __device__ __forceinline__ cd mul_w16(cd a) {
    constexpr int k = ((K % 16) + 16) % 16;
    constexpr double c1 = 0.92387953251128673848;   // cos(pi/8)
    constexpr double s1 = 0.38268343236508978178;   // sin(pi/8)
    constexpr double h = 0.70710678118654752440;    // sqrt(1/2)
    if (k == 0) return a;
    if (k == 4) return mul_i<DIR>(a);
    if (k == 8) return make_double2(-a.x, -a.y);
    if (k == 12) return mul_i<-DIR>(a);
    // general: w = cos(th) + DIR*i*sin(th), th = 2 pi k/16
    constexpr double cs[16] = {1, c1, h, s1, 0, -s1, -h, -c1, -1, -c1, -h, -s1, 0, s1, h, c1};
    constexpr double sn[16] = {0, s1, h, c1, 1, c1, h, s1, 0, -s1, -h, -c1, -1, -c1, -h, -s1};
    constexpr double wr = cs[k];
    constexpr double wi = (DIR < 0 ? -1.0 : 1.0) * sn[k];
    if (k == 2 || k == 6 || k == 10 || k == 14) {
        // |wr| == |wi| == h : two adds + two muls
        constexpr double sr = wr > 0 ? 1.0 : -1.0;
        constexpr double si = wi > 0 ? 1.0 : -1.0;
        // (a.x + i a.y)(wr + i wi) = (a.x wr - a.y wi) + i (a.x wi + a.y wr)
        return make_double2(h * (sr * a.x - si * a.y), h * (si * a.x + sr * a.y));
    }
    return make_double2(a.x * wr - a.y * wi, a.x * wi + a.y * wr);
}

template <int DIR> __device__ __forceinline__ void dft2(cd& a0, cd& a1) {
    cd t = a0;
    a0 = cadd(t, a1);
    a1 = csub(t, a1);
}

template <int DIR> __device__ __forceinline__ void dft4(cd& a0, cd& a1, cd& a2, cd& a3) {
    cd t0 = cadd(a0, a2), t1 = csub(a0, a2);
    cd t2 = cadd(a1, a3), t3 = mul_i<DIR>(csub(a1, a3));
    a0 = cadd(t0, t2);
    a1 = cadd(t1, t3);
    a2 = csub(t0, t2);
    a3 = csub(t1, t3);
}

// natural order in, natural order out
template <int DIR> __device__ __forceinline__ void dft8(cd* v) {
    // n = 2 n1 + n2 ; k = k1 + 4 k2
    dft4<DIR>(v[0], v[2], v[4], v[6]);   // y0[k1] in v[0],v[2],v[4],v[6]
    dft4<DIR>(v[1], v[3], v[5], v[7]);   // y1[k1] in v[1],v[3],v[5],v[7]
    cd y1_1 = mul_w16<DIR, 2>(v[3]);
    cd y1_2 = mul_w16<DIR, 4>(v[5]);
    cd y1_3 = mul_w16<DIR, 6>(v[7]);
    cd y0_0 = v[0], y0_1 = v[2], y0_2 = v[4], y0_3 = v[6], y1_0 = v[1];
    v[0] = cadd(y0_0, y1_0); v[4] = csub(y0_0, y1_0);
    v[1] = cadd(y0_1, y1_1); v[5] = csub(y0_1, y1_1);
    v[2] = cadd(y0_2, y1_2); v[6] = csub(y0_2, y1_2);
    v[3] = cadd(y0_3, y1_3); v[7] = csub(y0_3, y1_3);
}

template <int DIR> __device__ __forceinline__ void dft16(cd* v) {
    // n = 4 n1 + n2 ; k = k1 + 4 k2
    dft4<DIR>(v[0], v[4], v[8], v[12]);    // n2 = 0 : y[0][k1] at v[4 k1 + 0]
    dft4<DIR>(v[1], v[5], v[9], v[13]);    // n2 = 1
    dft4<DIR>(v[2], v[6], v[10], v[14]);   // n2 = 2
    dft4<DIR>(v[3], v[7], v[11], v[15]);   // n2 = 3
    // y[n2][k1] lives at v[4 k1 + n2]; twiddle W16^{n2 k1}
    v[5] = mul_w16<DIR, 1>(v[5]);
    v[6] = mul_w16<DIR, 2>(v[6]);
    v[7] = mul_w16<DIR, 3>(v[7]);
    v[9] = mul_w16<DIR, 2>(v[9]);
    v[10] = mul_w16<DIR, 4>(v[10]);
    v[11] = mul_w16<DIR, 6>(v[11]);
    v[13] = mul_w16<DIR, 3>(v[13]);
    v[14] = mul_w16<DIR, 6>(v[14]);
    v[15] = mul_w16<DIR, 9>(v[15]);
    // for each k1: 4-point DFT over n2 -> X[k1 + 4 k2] ; result k2 lands at v[4 k1 + k2]
    dft4<DIR>(v[0], v[1], v[2], v[3]);
    dft4<DIR>(v[4], v[5], v[6], v[7]);
    dft4<DIR>(v[8], v[9], v[10], v[11]);
    dft4<DIR>(v[12], v[13], v[14], v[15]);
    // now v[4 k1 + k2] = X[k1 + 4 k2]: transpose the 4x4 register tile (pure renaming)
    cd t;
    t = v[1]; v[1] = v[4]; v[4] = t;
    t = v[2]; v[2] = v[8]; v[8] = t;
    t = v[3]; v[3] = v[12]; v[12] = t;
    t = v[6]; v[6] = v[9]; v[9] = t;
    t = v[7]; v[7] = v[13]; v[13] = t;
    t = v[11]; v[11] = v[14]; v[14] = t;
}

template <int DIR, int R> __device__ __forceinline__ void dftR(cd* v) {
    if (R == 16) dft16<DIR>(v);
    else if (R == 8) dft8<DIR>(v);
    else if (R == 4) dft4<DIR>(v[0], v[1], v[2], v[3]);
    else dft2<DIR>(v[0], v[1]);
}

// ------------------------------------------------------------------------------------
// size configuration: E points per thread, up to three stages (every radix is 8 or 16)
// ------------------------------------------------------------------------------------
template <int N> struct Cfg;
template <> struct Cfg<64>   { static constexpr int E = 8,  S = 2, R0 = 8,  R1 = 8,  R2 = 1; };
template <> struct Cfg<128>  { static constexpr int E = 16, S = 2, R0 = 16, R1 = 8,  R2 = 1; };
template <> struct Cfg<256>  { static constexpr int E = 16, S = 2, R0 = 16, R1 = 16, R2 = 1; };
// 512 = 16 x 16 x 2: the closing radix-2 stage pairs values that sit in lane partners t, t^1 at the same register index
// (addresses 32 D + 2a + b after stage 1, b = t & 1), so it runs on warp shuffles: one shared-memory exchange and one
// barrier per transform instead of the two of the former 8 x 8 x 8 plan (the 512-point z / y passes of the 512^3 apply
// were shared-memory bound at 47-56 % of the HBM roofline).
template <> struct Cfg<512>  { static constexpr int E = 16, S = 3, R0 = 16, R1 = 16, R2 = 2; };
template <> struct Cfg<1024> { static constexpr int E = 16, S = 3, R0 = 16, R1 = 8,  R2 = 8; };
template <> struct Cfg<2048> { static constexpr int E = 16, S = 3, R0 = 16, R1 = 16, R2 = 8; };
template <> struct Cfg<4096> { static constexpr int E = 16, S = 3, R0 = 16, R1 = 16, R2 = 16; };

constexpr int ilog2(int x) { return x <= 1 ? 0 : 1 + ilog2(x >> 1); }

// the last stage is a radix-2 done across lane partners (no shared-memory exchange in front of it)
template <int N> struct ShflLast { static constexpr bool value = (Cfg<N>::S == 3 && Cfg<N>::R2 == 2); };

template <int N, int I> struct Stage {
    typedef Cfg<N> C;
    static constexpr int E = C::E;
    static constexpr int T = N / E;
    static constexpr int R = (I == 0) ? C::R0 : (I == 1 ? C::R1 : C::R2);
    static constexpr int PRE = (I == 0) ? 1 : (I == 1 ? C::R0 : C::R0 * C::R1);
    static constexpr int Mprev = N / PRE;
    static constexpr int M = Mprev / R;
    static constexpr int NB = E / R;            // butterflies per thread
    static constexpr bool LAST = (I == C::S - 1);
    static constexpr int RLAST = (C::S == 2) ? C::R1 : C::R2;
    // logical (unswizzled) in-place address of point a of butterfly u, thread t
    __device__ __forceinline__ static int addr(int t, int u, int a) {
        int beta = t + T * u;
        int D = beta / M, b = beta % M;
        return D * Mprev + a * M + b;
    }
    __device__ __forceinline__ static int bidx(int t, int u) { return (t + T * u) % M; }
};

// shared-memory layouts --------------------------------------------------------------
// A: one line contiguous at `base`, XOR swizzle keyed on the last radix
template <int N> struct LayA {
    static constexpr int XOR_LANE = 1;           // lane distance of the threads t, t^1 of one line
    int base;
    __device__ __forceinline__ int phys(int l) const {
        if constexpr (ShflLast<N>::value) {
            // only stages 0 and 1 touch shared memory.  Stage 1 reads 32 D + 2a + b with D = t/2, b = t&1: the four D of a
            // quarter warp would hit the same eight banks; XOR bits 1-2 with D mod 4 spreads them (stage 0, 32a + t, only
            // sees a permutation inside aligned groups of eight)
            constexpr int sh = ilog2(Stage<N, 1>::Mprev);
            return base + (l ^ (((l >> sh) & 3) << 1));
        } else {
            constexpr int sh = ilog2(Stage<N, 0>::RLAST);
            return base + (l ^ ((l >> sh) & 7));
        }
    }
};
// B: LB adjacent lines interleaved point by point (lane % LB = line).  LB = 8: a quarter warp reads one point of eight
// lines = 128 contiguous bytes, conflict free by construction.  LB = 4 (512-point lines: half the shared memory and
// threads per CTA, so two CTAs fit an SM): a quarter warp spans two points t, t+1 (t even) of four lines, i.e. two
// 64-byte pieces that must fall into different halves of the 32 banks - true when the two logical addresses differ in
// parity, which the XOR with bit log2(RLAST) arranges for the last stage (addresses 8t + a and 8(t+1) + a there).
// Measured on B200 (profiles/r2_l_512_variants.log): 512^3 apply 18.9 ms with LB = 4 against 21.2 ms with LB = 8.
constexpr int lines_b512 = 4;
template <int N> struct LinesB { static constexpr int value = (N == 512) ? lines_b512 : 8; };
template <int N> struct LayB {
    static constexpr int LB = LinesB<N>::value;
    static constexpr int XOR_LANE = LB;          // lane = t * LB + line
    int lam;
    __device__ __forceinline__ int phys(int l) const {
        if (LB == 8 || ShflLast<N>::value) return l * LB + lam;     // stages 0 / 1 of the shuffle plan: l, l+1 for t, t+1
        constexpr int sh = ilog2(Stage<N, 0>::RLAST);
        return (l ^ ((l >> sh) & 1)) * LB + lam;
    }
};

template <int N, int I, class Lay>
__device__ __forceinline__ void st_stage(const cd* v, int t, cd* sm, const Lay& lay) {
    typedef Stage<N, I> St;
#pragma unroll
    for (int u = 0; u < St::NB; ++u)
#pragma unroll
        for (int a = 0; a < St::R; ++a) sm[lay.phys(St::addr(t, u, a))] = v[u * St::R + a];
}
template <int N, int I, class Lay>
__device__ __forceinline__ void ld_stage(cd* v, int t, const cd* sm, const Lay& lay) {
    typedef Stage<N, I> St;
    // issue order = consumption order of the butterfly's first layer (dft4 over a, a+R/4, a+R/2, a+3R/4)
#pragma unroll
    for (int u = 0; u < St::NB; ++u)
#pragma unroll
        for (int i = 0; i < St::R; ++i) {
            const int a = (St::R >= 4) ? (i % 4) * (St::R / 4) + i / 4 : i;
            v[u * St::R + a] = sm[lay.phys(St::addr(t, u, a))];
        }
}

// ------------------------------------------------------------------------------------
// Twiddles.  No per-point table lookups on the hot path:
//  * stage 0 carries the pruned-FFT modulation with it.  For sub-transform r (0..3) of a line
//    zero-padded to 4N the input is x[j] * w_{4N}^{r j}, j = a*T + t.  The a-dependent part
//    w_{4E}^{r a} is a warp-uniform constant (constant bank); the t-dependent part merges
//    with the DIF twiddle w_N^{t d} into q^(4d + r), q = w_{4N}^t, generated from two
//    per-thread constants (q, s = q^4) by a short product recurrence in registers.
//  * middle stages (3-stage sizes only) read a tiny [d][b] table staged in shared memory.
// ------------------------------------------------------------------------------------
template <int N> struct TwState {
    cd q;            // w_{4N}^t
    cd s;            // w_N^t  (= q^4, taken from the table for accuracy)
    cd s2;           // s^2
    const cd* tw1;   // shared-memory table of stage 1, entry [d*M1 + b] = w_{Mprev1}^{b d}
};

// engine table for size N (built on the host, ls::engine_table):
//   [0, T)            q_t = exp(-2 pi i t/(4N))
//   [T, 2T)           s_t = exp(-2 pi i t/N)
//   [2T, 2T + TW1N)   stage-1 table (3-stage sizes), TW1N = N/R0
template <int N> struct EngTab {
    static constexpr int T = N / Cfg<N>::E;
    static constexpr int TW1N = (Cfg<N>::S == 3) ? N / Cfg<N>::R0 : 0;
    static constexpr int TOTAL = 2 * T + TW1N;
};

// cooperative copy of the stage-1 table into shared memory (call before the first sync)
template <int N>
__device__ __forceinline__ void load_tw1(cd* tw1_sm, const cd* __restrict__ tab) {
    for (int i = threadIdx.x; i < EngTab<N>::TW1N; i += blockDim.x) tw1_sm[i] = tab[2 * EngTab<N>::T + i];
}
template <int N>
__device__ __forceinline__ TwState<N> make_tw(int t, const cd* __restrict__ tab, const cd* tw1_sm) {
    TwState<N> tw;
    tw.q = tab[t];
    tw.s = tab[EngTab<N>::T + t];
    tw.s2 = cmul(tw.s, tw.s);
    tw.tw1 = tw1_sm;
    return tw;
}

__device__ __forceinline__ cd c64(int k) { return make_double2(C64_RE[k & 63], C64_IM[k & 63]); }

// v[d] *= q^(4d + r)  (CONJ: by the conjugate), d = 0..E-1; two interleaved product chains
template <int N, bool CONJ>
__device__ __forceinline__ void mul_stage0_twiddles(cd* v, int r, const TwState<N>& tw) {
    constexpr int E = Cfg<N>::E;
    cd pe;   // q^r
    if (r == 0) pe = make_double2(1.0, 0.0);
    else if (r == 1) pe = tw.q;
    else {
        cd q2 = cmul(tw.q, tw.q);
        pe = (r == 2) ? q2 : cmul(q2, tw.q);
    }
    cd po = cmul(pe, tw.s);
    if (r != 0) v[0] = CONJ ? cmulc(v[0], pe) : cmul(v[0], pe);
    v[1] = CONJ ? cmulc(v[1], po) : cmul(v[1], po);
#pragma unroll
    for (int d = 2; d < E; d += 2) {
        pe = cmul(pe, tw.s2);
        po = cmul(po, tw.s2);
        v[d] = CONJ ? cmulc(v[d], pe) : cmul(v[d], pe);
        v[d + 1] = CONJ ? cmulc(v[d + 1], po) : cmul(v[d + 1], po);
    }
}

// stage 0, forward, sub-transform r:  in v[a] = x[a*T + t] (unmodulated)
template <int N>
__device__ __forceinline__ void fwd_stage0(cd* v, int r, const TwState<N>& tw) {
    constexpr int E = Cfg<N>::E;
    if (r != 0) {
#pragma unroll
        for (int a = 1; a < E; ++a) v[a] = cmul(v[a], c64(r * a * (16 / E)));
    }
    dftR<-1, E>(v);
    mul_stage0_twiddles<N, false>(v, r, tw);
}
// adjoint of fwd_stage0 without the final demodulation constants: out v[a] = sum_d ...;
// the caller accumulates acc[a] += v[a] * conj(c64(r a 16/E)).
template <int N>
__device__ __forceinline__ void inv_stage0(cd* v, int r, const TwState<N>& tw) {
    constexpr int E = Cfg<N>::E;
    mul_stage0_twiddles<N, true>(v, r, tw);
    dftR<+1, E>(v);
}
template <int N>
__device__ __forceinline__ void demod_accumulate(cd* acc, const cd* v, int r) {
    constexpr int E = Cfg<N>::E;
    if (r == 0) {
#pragma unroll
        for (int a = 0; a < E; ++a) acc[a] = v[a];
    } else {
        acc[0] = cadd(acc[0], v[0]);
#pragma unroll
        for (int a = 1; a < E; ++a) acc[a] = cfmac(v[a], c64(r * a * (16 / E)), acc[a]);
    }
}

// same for an output block other than the first: every term carries the extra factor conj(w_64^shift)
template <int N>
__device__ __forceinline__ void demod_accumulate_block(cd* acc, const cd* v, int r, int shift) {
    constexpr int E = Cfg<N>::E;
    if (r == 0) {
#pragma unroll
        for (int a = 0; a < E; ++a) acc[a] = v[a];
    } else {
#pragma unroll
        for (int a = 0; a < E; ++a) acc[a] = cfmac(v[a], c64(r * a * (16 / E) + shift), acc[a]);
    }
}

// middle / last stages ------------------------------------------------------------------
// Middle-stage twiddles w^d, d = 1..R-1, w = w_{Mprev}^b.  LS_TW_TABLE: every factor read from the shared-memory
// table (R-1 LDS.128 per butterfly - a fifth of the engine's shared-memory traffic at N = 2048).  Default: only w is
// read, the powers come from a product tree of depth <= 4 (w2 = w^2, w4 = w2^2, w8 = w4^2, the rest one product of
// two of those), about 4 ulp instead of the table's 0.5 ulp - still four orders below the 1e-12 parity bar - and
// FP64 work on the otherwise idle per-quadrant pipe instead of wavefronts on the SM-wide shared-memory pipe.
template <int R, bool CONJ>
__device__ __forceinline__ void mul_twiddle_powers(cd* v, const cd w1) {
    auto ap = [](cd a, cd w) { return CONJ ? cmulc(a, w) : cmul(a, w); };
    const cd w2 = cmul(w1, w1);
    const cd w4 = cmul(w2, w2);
    if constexpr (R == 16) {
        const cd w8 = cmul(w4, w4);
        v[8] = ap(v[8], w8);
        v[1] = ap(v[1], w1);  v[9] = ap(v[9], cmul(w8, w1));
        v[2] = ap(v[2], w2);  v[10] = ap(v[10], cmul(w8, w2));
        const cd w3 = cmul(w2, w1);
        v[3] = ap(v[3], w3);  v[11] = ap(v[11], cmul(w8, w3));
        v[4] = ap(v[4], w4);  v[12] = ap(v[12], cmul(w8, w4));
        const cd w5 = cmul(w4, w1);
        v[5] = ap(v[5], w5);  v[13] = ap(v[13], cmul(w8, w5));
        const cd w6 = cmul(w4, w2);
        v[6] = ap(v[6], w6);  v[14] = ap(v[14], cmul(w8, w6));
        const cd w7 = cmul(w4, w3);
        v[7] = ap(v[7], w7);  v[15] = ap(v[15], cmul(w8, w7));
    } else {
        static_assert(R == 8, "middle stages are radix 8 or 16");
        v[1] = ap(v[1], w1);
        v[2] = ap(v[2], w2);
        const cd w3 = cmul(w2, w1);
        v[3] = ap(v[3], w3);
        v[4] = ap(v[4], w4);
        v[5] = ap(v[5], cmul(w4, w1));
        v[6] = ap(v[6], cmul(w4, w2));
        v[7] = ap(v[7], cmul(w4, w3));
    }
}

template <int N, int I>
__device__ __forceinline__ void fwd_stage(cd* v, int t, const TwState<N>& tw) {
    typedef Stage<N, I> St;
#pragma unroll
    for (int u = 0; u < St::NB; ++u) {
        dftR<-1, St::R>(v + u * St::R);
        if (!St::LAST) {
            int b = St::bidx(t, u);
#ifdef LS_TW_TABLE
#pragma unroll
            for (int d = 1; d < St::R; ++d) v[u * St::R + d] = cmul(v[u * St::R + d], tw.tw1[d * St::M + b]);
#else
            if constexpr (false && St::M == 2) {   // measured slower (divergent constant-bank reads): 512^3 apply 18.7 -> 19.4 ms; the product tree stays
                // w_Mprev^(b d) are entries of the 64th-root table in the constant bank (512 = 16 x 16 x 2: Mprev = 32,
                // b = t & 1): no product tree, no shared-memory read - this pass is FP64-bound at 512 points
#pragma unroll
                for (int d = 1; d < St::R; ++d) v[u * St::R + d] = cmul(v[u * St::R + d], c64((64 / St::Mprev) * b * d));
            } else {
                mul_twiddle_powers<St::R, false>(v + u * St::R, tw.tw1[St::M + b]);
            }
#endif
        }
    }
}
template <int N, int I>
__device__ __forceinline__ void inv_stage(cd* v, int t, const TwState<N>& tw) {
    typedef Stage<N, I> St;
#pragma unroll
    for (int u = 0; u < St::NB; ++u) {
        if (!St::LAST) {
            int b = St::bidx(t, u);
#ifdef LS_TW_TABLE
#pragma unroll
            for (int d = 1; d < St::R; ++d) v[u * St::R + d] = cmulc(v[u * St::R + d], tw.tw1[d * St::M + b]);
#else
            if constexpr (false && St::M == 2) {   // measured slower (divergent constant-bank reads): 512^3 apply 18.7 -> 19.4 ms; the product tree stays
#pragma unroll
                for (int d = 1; d < St::R; ++d) v[u * St::R + d] = cmulc(v[u * St::R + d], c64((64 / St::Mprev) * b * d));
            } else {
                mul_twiddle_powers<St::R, true>(v + u * St::R, tw.tw1[St::M + b]);
            }
#endif
        }
        dftR<+1, St::R>(v + u * St::R);
    }
}

struct NoHook { __device__ __forceinline__ void operator()() const {} };

// closing / opening radix-2 stage of the shuffle plans: thread t (even) holds p = value at address 2D, its partner
// t^1 holds q at 2D + 1, for every register index a.  Forward and adjoint are the same butterfly: even keeps p + q,
// odd keeps p - q.
template <int N, class Lay>
__device__ __forceinline__ void shfl_radix2(cd* v, int t) {
    constexpr int E = Cfg<N>::E;
    const bool odd = (t & 1) != 0;
#pragma unroll
    for (int a = 0; a < E; ++a) {
        const double qx = __shfl_xor_sync(0xffffffffu, v[a].x, Lay::XOR_LANE);
        const double qy = __shfl_xor_sync(0xffffffffu, v[a].y, Lay::XOR_LANE);
        v[a] = odd ? make_double2(qx - v[a].x, qy - v[a].y) : make_double2(v[a].x + qx, v[a].y + qy);
    }
}

// Forward FFT of sub-transform r of one line.  In: v[a] = x[a*T + t].  Out: v[e] = X_r[freq(t + T*e)],
// X_r = FFT_N(x[j] w_{4N}^{r j}).  sm/lay = this line's exchange buffer (N points).
// `pre_last` runs on every thread just before the butterflies of the last stage (the place to issue
// global loads whose latency should hide behind them).
template <int N, class Lay, class Hook = NoHook>
__device__ __forceinline__ void fft_fwd(cd* v, int t, int r, cd* sm, const Lay& lay, const TwState<N>& tw,
                                        Hook pre_last = Hook()) {
    typedef Cfg<N> C;
    fwd_stage0<N>(v, r, tw);
    st_stage<N, 0>(v, t, sm, lay);
    __syncthreads();
    ld_stage<N, 1>(v, t, sm, lay);
    if constexpr (ShflLast<N>::value) {
        pre_last();                      // the closing stage is a handful of shuffles: issue the loads ahead of stage 1
        fwd_stage<N, 1>(v, t, tw);
        shfl_radix2<N, Lay>(v, t);
    } else if constexpr (C::S == 3) {
        fwd_stage<N, 1>(v, t, tw);
        st_stage<N, 1>(v, t, sm, lay);
        __syncthreads();
        ld_stage<N, 2>(v, t, sm, lay);
        pre_last();
        fwd_stage<N, 2>(v, t, tw);
    } else {
        pre_last();
        fwd_stage<N, 1>(v, t, tw);
    }
}

// Adjoint network (unnormalised inverse) up to, not including, the demodulation constants.
// In: v[e] = Y_r[freq(t + T*e)].  Out: v[a]; then y[a*T+t] += v[a]*conj(c64(..)) (demod_accumulate).
// `hook` runs on every thread right after the first __syncthreads() of the inverse.
template <int N, class Lay, class Hook = NoHook>
__device__ __forceinline__ void fft_inv(cd* v, int t, int r, cd* sm, const Lay& lay, const TwState<N>& tw,
                                        Hook hook = Hook()) {
    typedef Cfg<N> C;
    if constexpr (ShflLast<N>::value) {
        shfl_radix2<N, Lay>(v, t);
        inv_stage<N, 1>(v, t, tw);
        st_stage<N, 1>(v, t, sm, lay);
        __syncthreads();
        hook();
    } else if constexpr (C::S == 3) {
        inv_stage<N, 2>(v, t, tw);
        st_stage<N, 2>(v, t, sm, lay);
        __syncthreads();
        hook();
        ld_stage<N, 1>(v, t, sm, lay);
        inv_stage<N, 1>(v, t, tw);
        st_stage<N, 1>(v, t, sm, lay);
        __syncthreads();
    } else {
        inv_stage<N, 1>(v, t, tw);
        st_stage<N, 1>(v, t, sm, lay);
        __syncthreads();
        hook();
    }
    ld_stage<N, 0>(v, t, sm, lay);
    inv_stage0<N>(v, r, tw);
}

// ---- two sub-transforms in flight per thread --------------------------------------------------
// The four sub-transforms r = 0..3 of a padded line are independent.  Running two of them through the
// stages together lets one transform's shared-memory exchange (stores, barrier, loads in flight)
// overlap the other's FP64 butterflies inside the same warp - the FP64 pipe and the shared-memory
// pipe are both ~50 % loaded in the fused middle pass and otherwise take turns.
template <int N, class Lay>
__device__ __forceinline__ void fft_fwd_dual(cd* vA, cd* vB, int t, int rA, int rB, cd* sm, const Lay& layA, const Lay& layB,
                                             const TwState<N>& tw) {
    typedef Cfg<N> C;
    fwd_stage0<N>(vA, rA, tw);
    st_stage<N, 0>(vA, t, sm, layA);
    fwd_stage0<N>(vB, rB, tw);
    st_stage<N, 0>(vB, t, sm, layB);
    __syncthreads();
    ld_stage<N, 1>(vA, t, sm, layA);
    ld_stage<N, 1>(vB, t, sm, layB);
    if constexpr (C::S == 3) {
        fwd_stage<N, 1>(vA, t, tw);
        st_stage<N, 1>(vA, t, sm, layA);
        fwd_stage<N, 1>(vB, t, tw);
        st_stage<N, 1>(vB, t, sm, layB);
        __syncthreads();
        ld_stage<N, 2>(vA, t, sm, layA);
        ld_stage<N, 2>(vB, t, sm, layB);
        fwd_stage<N, 2>(vA, t, tw);
        fwd_stage<N, 2>(vB, t, tw);
    } else {
        fwd_stage<N, 1>(vA, t, tw);
        fwd_stage<N, 1>(vB, t, tw);
    }
}
template <int N, class Lay>
__device__ __forceinline__ void fft_inv_dual(cd* vA, cd* vB, int t, int rA, int rB, cd* sm, const Lay& layA, const Lay& layB,
                                             const TwState<N>& tw) {
    typedef Cfg<N> C;
    if constexpr (C::S == 3) {
        inv_stage<N, 2>(vA, t, tw);
        st_stage<N, 2>(vA, t, sm, layA);
        inv_stage<N, 2>(vB, t, tw);
        st_stage<N, 2>(vB, t, sm, layB);
        __syncthreads();
        ld_stage<N, 1>(vA, t, sm, layA);
        ld_stage<N, 1>(vB, t, sm, layB);
    }
    inv_stage<N, 1>(vA, t, tw);
    st_stage<N, 1>(vA, t, sm, layA);
    inv_stage<N, 1>(vB, t, tw);
    st_stage<N, 1>(vB, t, sm, layB);
    __syncthreads();
    ld_stage<N, 0>(vA, t, sm, layA);
    ld_stage<N, 0>(vB, t, sm, layB);
    inv_stage0<N>(vA, rA, tw);
    inv_stage0<N>(vB, rB, tw);
}

// ---- TMA bulk copy + mbarrier helpers (sm_90+/sm_100a PTX) -------------------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    unsigned ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// tensor copies of one box through a tensor map (a __grid_constant__ kernel parameter): a 3-D load into shared memory
// that completes on `bar`, and a 4-D store from shared memory in this thread's bulk group
__device__ __forceinline__ void tma_load_3d(void* dst_smem, const void* map, int c0, int c1, int c2, unsigned long long* bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 ::"r"(smem_u32(dst_smem)), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_store_4d(const void* map, int c0, int c1, int c2, int c3, const void* src_smem) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%1, %2, %3, %4}], [%5];"
                 ::"l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(smem_u32(src_smem)) : "memory");
}
// commit this thread's bulk stores and wait until their shared-memory sources have been read
__device__ __forceinline__ void bulk_store_drain() {
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

}  // namespace lsfft
