// General-size 2-D Lippmann-Schwinger operator: any n, m and both quadratures.
//
// Serves what the power-of-two fast path (op2d.cu) cannot: the sizes the reference actually ships
// (examples/example.jl: n = 201, Greengard_Vico padded 804 = 2^2*3*67) and the Duan-Rokhlin
// trapezoidal rule (FastConvolution.jl:64-83: padded 2n-1, crop [n:2n-1]).  Every line DFT of
// arbitrary length Lf is evaluated exactly by Bluestein's identity
//       X_q = conj(c_q) * sum_j [x_j conj(c_j)] c_{q-j},      c_t = exp(i pi t^2 / Lf)
// as a circular convolution of power-of-two length Nb >= Lf + nin - 1 on the same register-resident
// engine (forward -> multiply by the chirp spectrum -> adjoint inverse, all inside one CTA).
// Zero padding is still pruned: only the nin non-zero inputs are read and only the nout kept outputs
// are formed.  Three launches per apply, like the fast path:
//   G1 k_bs_fwd   columns: b, nu          -> A [ne x m]     (natural frequency order)
//   G2 k_bs_mid   rows: A, spectrum       -> C [m x ne]     (forward, x GFFT, inverse, crop)
//   G3 k_bs_inv   columns: C, b           -> y              (inverse, crop, b + omega^2 *)
// In G2 the post-chirp of the forward and the pre-chirp of the inverse cancel exactly.
#include "ls_common.cuh"
#include "op2d_base.cuh"
#include "line_kernels.cuh"
#include "bluestein.cuh"

using namespace ls;
using namespace lsk;
using namespace lsb;

namespace {

struct Op2DGeneric : Op2DBase {
    BsDim X, Y;
    double* d_nu = nullptr;
    cd* d_G = nullptr;     // [kx][ky] natural order, shift folded, scaled
    cd* d_A = nullptr;     // ne x m
    cd* d_C = nullptr;     // m x ne
    int apply_dev(const cd* b, cd* y, int mode) override;
    // the spectrum is the reference's: padded 4n (Greengard_Vico) or 2n - 1 (trapezoidal)
    void info(int* route, int64_t* n_line, int64_t* m_line, int* padding) const override {
        *route = 1; *n_line = X.Nb; *m_line = Y.Nb; *padding = quadrule == LS_QUAD_TRAPEZOIDAL ? 2 : 4;
    }
};

// Gd[kx*me + ky] = GFFT[(kx + sx) % ne, (ky + sy) % me] * scale   (sx = ne/2 for Greengard_Vico, 0 otherwise)
__global__ void k_bs_permute_g(const cd* __restrict__ gin, cd* __restrict__ gout, long ne, long me, long sx, long sy,
                               double scale) {
    const long total = ne * me;
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const long ky = idx % me, kx = idx / me;
        const cd v = gin[(kx + sx) % ne + ne * ((ky + sy) % me)];
        gout[idx] = make_double2(v.x * scale, v.y * scale);
    }
}

}  // namespace

int Op2DGeneric::apply_dev(const cd* b, cd* y, int mode) {
    const bool full = (mode == LS_APPLY_FASTCONVOLUTION);
    const bool trap = (quadrule == LS_QUAD_TRAPEZOIDAL);
    // Q2: FFTconvolution multiplies by nu in the trapezoidal branch only (FastConvolution.jl:122 vs :141)
    const double* nuptr = (full || trap) ? d_nu : nullptr;
    const long big = 1L << 40;
    {   // G1: columns j: in b[n*j + i]; out A[ne*j + kx]
        LineAddr la{big, n, 0, 1, ne, 0, 1};
        phase_begin(0);
#define CALL1(NB)                                                                                             \
        {                                                                                                     \
            LS_CUDA_TRY(bs_attr(k_bs_fwd<NB>, BsGeo<NB>::smem));                                              \
            const long grid = (m + BsGeo<NB>::LPC - 1) / BsGeo<NB>::LPC;                                      \
            k_bs_fwd<NB><<<(unsigned)grid, BsGeo<NB>::THREADS, BsGeo<NB>::smem, stream>>>(                    \
                b, nuptr, d_A, X.d_tab, X.d_ch, X.d_hf, (int)n, (int)ne, m, la);                              \
        }
        BS_DISPATCH(X.Nb, CALL1);
        phase_end(); launches++;
    }
    {   // G2: rows kx: in A[kx + ne*j]; out C[m*kx + j]
        LineAddr la{big, 1, 0, ne, m, 0, 1};
        phase_begin(1);
#define CALL2(NB)                                                                                             \
        {                                                                                                     \
            LS_CUDA_TRY(bs_attr(k_bs_mid<NB>, BsGeo<NB>::smem));                                              \
            const long grid = (ne + BsGeo<NB>::LPC - 1) / BsGeo<NB>::LPC;                                     \
            k_bs_mid<NB><<<(unsigned)grid, BsGeo<NB>::THREADS, BsGeo<NB>::smem, stream>>>(                    \
                d_A, d_C, d_G, Y.d_tab, Y.d_ch, Y.d_hf, Y.d_hi, (int)m, (int)me, (int)Y.o0, ne, la);          \
        }
        BS_DISPATCH(Y.Nb, CALL2);
        phase_end(); launches++;
    }
    {   // G3: columns j: in C[j + m*kx]; out y[n*j + i]
        LineAddr la{big, 1, 0, m, n, 0, 1};
        phase_begin(2);
#define CALL3(NB)                                                                                             \
        {                                                                                                     \
            LS_CUDA_TRY(bs_attr(k_bs_inv<NB>, BsGeo<NB>::smem));                                              \
            const long grid = (m + BsGeo<NB>::LPC - 1) / BsGeo<NB>::LPC;                                      \
            k_bs_inv<NB><<<(unsigned)grid, BsGeo<NB>::THREADS, BsGeo<NB>::smem, stream>>>(                    \
                d_C, full ? b : nullptr, y, X.d_tab, X.d_ch, X.d_hi, (int)n, (int)ne, (int)X.o0,              \
                full ? omega * omega : 1.0, m, la);                                                           \
        }
        BS_DISPATCH(X.Nb, CALL3);
        phase_end(); launches++;
    }
    LS_CUDA_TRY(cudaGetLastError());
    return LS_OK;
}

namespace ls {

int create_op2d_generic(ls_handle* out, int64_t n, int64_t m, int64_t ne, int64_t me, const double* nu,
                        const ls_cdouble* gfft, double omega, int quadrule, const cd* gfft_dev) {
    // size check first (no CUDA call needed to refuse)
    LS_REQUIRE(ne + n - 1 <= 4096 && me + m - 1 <= 4096, LS_ERR_UNSUPPORTED,
               "ls_op2d_create: n=%ld, m=%ld (padded %ld x %ld): the general-size GPU path serves ne + n - 1 <= 4096; "
               "larger grids need the power-of-two Greengard_Vico fast path", (long)n, (long)m, (long)ne, (long)me);
    Op2DGeneric* op = new Op2DGeneric();
    int rc = op->init_base(KIND_OP2D);
    if (rc) { delete op; return rc; }
    op->n = n; op->m = m; op->ne = ne; op->me = me; op->omega = omega; op->quadrule = quadrule;
    const bool trap = (quadrule == LS_QUAD_TRAPEZOIDAL);
#define TRY(x) do { rc = (x); if (rc) { delete op; return rc; } } while (0)
    // kept outputs: Greengard_Vico [1:n] (FastConvolution.jl:101), trapezoidal [n:2n-1] (:82)
    TRY(setup_dim(op, op->X, n, ne, trap ? n - 1 : 0));
    TRY(setup_dim(op, op->Y, m, me, trap ? m - 1 : 0));
    const size_t N = (size_t)n * m, NE = (size_t)ne * me;
    TRY(op->dupload((void**)&op->d_nu, nu, N * sizeof(double)));
    {
        cd* d_gin = nullptr;
        if (gfft_dev) d_gin = const_cast<cd*>(gfft_dev);
        else TRY(op->dupload((void**)&d_gin, gfft, NE * sizeof(cd)));
        TRY(op->dmalloc((void**)&op->d_G, NE * sizeof(cd)));
        // ifft normalisation 1/(ne me) and the 1/Nb of each of the four circular convolutions
        const double scale = 1.0 / ((double)ne * (double)me) / ((double)op->X.Nb * (double)op->X.Nb)
                             / ((double)op->Y.Nb * (double)op->Y.Nb);
        // fftshift/ifftshift pair (FastConvolution.jl:94,98): for even ne a roll by ne/2; none for trapezoidal
        const long sx = trap ? 0 : ne / 2, sy = trap ? 0 : me / 2;
        k_bs_permute_g<<<148 * 8, 256, 0, op->stream>>>(d_gin, op->d_G, ne, me, sx, sy, scale);
        cudaError_t e = cudaStreamSynchronize(op->stream);
        if (e != cudaSuccess) { set_error("spectrum permutation failed: %s", cudaGetErrorString(e)); delete op; return LS_ERR_CUDA; }
        if (!gfft_dev) op->dfree(d_gin);
    }
    TRY(op->dmalloc((void**)&op->d_A, (size_t)ne * m * sizeof(cd)));
    TRY(op->dmalloc((void**)&op->d_C, (size_t)ne * m * sizeof(cd)));
    TRY(op->dmalloc((void**)&op->d_b, N * sizeof(cd)));
    TRY(op->dmalloc((void**)&op->d_y, N * sizeof(cd)));
#undef TRY
    *out = reinterpret_cast<ls_handle>(op);
    return LS_OK;
}

}  // namespace ls
