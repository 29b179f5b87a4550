// General-size 3-D Lippmann-Schwinger operator (any n = m, l): the reference's own 3-D example ships
// n = 48 (examples/example3D.jl:20-31, padded 192^3).  Same five passes as op3d.cu, every line DFT
// evaluated by Bluestein's identity on the power-of-two engine (bluestein.cuh); padding still pruned.
//   G1 x lines  b, nu [n m l]  -> A1 [ne m l]     G2 y lines  A1 -> A2 [ne me l]
//   G3 z lines  A2 (x spectrum, in place, kept planes [1:l])      G4 y lines  A2 -> A1     G5 x lines A1, b -> y
// Strided lines are read and written 16 bytes at a time (lane mapping A): this path is for the small and
// odd sizes the fast path does not serve, not for throughput.
#include "ls_common.cuh"
#include "line_kernels.cuh"
#include "bluestein.cuh"
#include "gv_spectrum.cuh"

using namespace ls;
using namespace lsk;
using namespace lsb;

namespace {

struct Op3DGeneric : HandleBase {
    long n = 0, m = 0, l = 0, ne = 0, me = 0, le = 0;
    double omega = 0;
    BsDim X, Y, Z;
    double* d_nu = nullptr;
    cd* d_G = nullptr;      // [(kx + ne*ky)*le + kz], shift folded, scaled
    cd* d_A1 = nullptr;     // ne x m x l
    cd* d_A2 = nullptr;     // ne x me x l
    cd* d_b = nullptr; cd* d_y = nullptr;
    int64_t op_size() const override { return n * m * l; }
    int apply_dev(const cd* b, cd* y, int mode) override;
};

// Gd[(kx + ne*ky)*le + kz] = GFFT[(kx+ne/2)%ne, (ky+me/2)%me, (kz+le/2)%le] * scale, gathered or generated
__global__ void k_bs_fill_g3d(const cd* __restrict__ gin, cd* __restrict__ gout, long ne, long me, long le,
                              double dk, double L, double k, double eLk_re, double eLk_im, double scale) {
    const long total = ne * me * le;
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const long kz = idx % le;
        const long Lxy = idx / le;
        const long kx = Lxy % ne, ky = Lxy / ne;
        const long ix = (kx + ne / 2) % ne, iy = (ky + me / 2) % me, iz = (kz + le / 2) % le;
        cd v;
        if (gin != nullptr) v = gin[ix + ne * (iy + me * iz)];
        else v = gtrunc3d_eval(gv_radius(dk, ix, iy, iz, ne, me, le), L, k, eLk_re, eLk_im);
        gout[idx] = make_double2(v.x * scale, v.y * scale);
    }
}

}  // namespace

int Op3DGeneric::apply_dev(const cd* b, cd* y, int mode) {
    const bool full = (mode == LS_APPLY_FASTCONVOLUTION);
    const long big = 1L << 40;
#define BS_LAUNCH(KERN, NBV, NLINES, ...)                                                                     \
    {                                                                                                         \
        LS_CUDA_TRY(bs_attr(KERN<NBV>, BsGeo<NBV>::smem));                                                    \
        const long grid = ((NLINES) + BsGeo<NBV>::LPC - 1) / BsGeo<NBV>::LPC;                                 \
        KERN<NBV><<<(unsigned)grid, BsGeo<NBV>::THREADS, BsGeo<NBV>::smem, stream>>>(__VA_ARGS__);            \
    }
    {   // G1: x lines (j,p)
        LineAddr la{big, n, 0, 1, ne, 0, 1};
        phase_begin(0);
#define G1(NB) BS_LAUNCH(k_bs_fwd, NB, m * l, b, full ? d_nu : nullptr, d_A1, X.d_tab, X.d_ch, X.d_hf, (int)n, (int)ne, m * l, la)
        BS_DISPATCH(X.Nb, G1);
        phase_end(); launches++;
    }
    {   // G2: y lines (kx,p): in A1[kx + ne*m*p + ne*j]; out A2[kx + ne*me*p + ne*ky]
        LineAddr la{ne, 1, ne * m, ne, 1, ne * me, ne};
        phase_begin(1);
#define G2(NB) BS_LAUNCH(k_bs_fwd, NB, ne * l, d_A1, nullptr, d_A2, Y.d_tab, Y.d_ch, Y.d_hf, (int)m, (int)me, ne * l, la)
        BS_DISPATCH(Y.Nb, G2);
        phase_end(); launches++;
    }
    {   // G3: z lines L = kx + ne*ky, point p at A2[L + ne*me*p], in place
        LineAddr la{big, 1, 0, ne * me, 1, 0, ne * me};
        phase_begin(2);
#define G3(NB) BS_LAUNCH(k_bs_mid, NB, ne * me, d_A2, d_A2, d_G, Z.d_tab, Z.d_ch, Z.d_hf, Z.d_hi, (int)l, (int)le, 0, ne * me, la)
        BS_DISPATCH(Z.Nb, G3);
        phase_end(); launches++;
    }
    {   // G4: inverse y lines (kx,p): in A2[kx + ne*me*p + ne*ky]; out A1[kx + ne*m*p + ne*j]
        LineAddr la{ne, 1, ne * me, ne, 1, ne * m, ne};
        phase_begin(3);
#define G4(NB) BS_LAUNCH(k_bs_inv, NB, ne * l, d_A2, nullptr, d_A1, Y.d_tab, Y.d_ch, Y.d_hi, (int)m, (int)me, 0, 1.0, ne * l, la)
        BS_DISPATCH(Y.Nb, G4);
        phase_end(); launches++;
    }
    {   // G5: inverse x lines (j,p) + combine
        LineAddr la{big, ne, 0, 1, n, 0, 1};
        phase_begin(4);
#define G5(NB) BS_LAUNCH(k_bs_inv, NB, m * l, d_A1, full ? b : nullptr, y, X.d_tab, X.d_ch, X.d_hi, (int)n, (int)ne, 0, full ? omega * omega : 1.0, m * l, la)
        BS_DISPATCH(X.Nb, G5);
        phase_end(); launches++;
    }
    LS_CUDA_TRY(cudaGetLastError());
    return LS_OK;
}

namespace ls {

void op3d_generic_lines(const HandleBase* h, int64_t* n_line, int64_t* m_line, int64_t* l_line) {
    const Op3DGeneric* op = static_cast<const Op3DGeneric*>(h);
    *n_line = op->X.Nb; *m_line = op->Y.Nb; *l_line = op->Z.Nb;
}

int create_op3d_generic(ls_handle* out, int64_t n, int64_t m, int64_t l, int64_t ne, int64_t me, int64_t le,
                        const double* nu, const ls_cdouble* gfft, double omega, double L, double Lp) {
    LS_REQUIRE(ne + n - 1 <= 4096 && me + m - 1 <= 4096 && le + l - 1 <= 4096, LS_ERR_UNSUPPORTED,
               "ls_op3d_create: n=%ld m=%ld l=%ld - the general-size GPU path serves 5n - 1 <= 4096", (long)n, (long)m, (long)l);
    Op3DGeneric* op = new Op3DGeneric();
    int rc = op->init_base(KIND_OP3D);
    if (rc) { delete op; return rc; }
    op->n = n; op->m = m; op->l = l; op->ne = ne; op->me = me; op->le = le; op->omega = omega;
#define TRY(x) do { rc = (x); if (rc) { delete op; return rc; } } while (0)
    TRY(setup_dim(op, op->X, n, ne, 0));
    TRY(setup_dim(op, op->Y, m, me, 0));
    TRY(setup_dim(op, op->Z, l, le, 0));
    const size_t N = (size_t)n * m * l, NE = (size_t)ne * me * le;
    TRY(op->dupload((void**)&op->d_nu, nu, N * sizeof(double)));
    {
        cd* d_gin = nullptr;
        if (gfft) TRY(op->dupload((void**)&d_gin, gfft, NE * sizeof(cd)));
        TRY(op->dmalloc((void**)&op->d_G, NE * sizeof(cd)));
        // ifft normalisation and the 1/Nb of the six circular convolutions of an apply (x, y, z: forward + inverse)
        const double scale = 1.0 / ((double)ne * (double)me * (double)le)
                             / ((double)op->X.Nb * op->X.Nb) / ((double)op->Y.Nb * op->Y.Nb) / ((double)op->Z.Nb * op->Z.Nb);
        k_bs_fill_g3d<<<148 * 8, 256, 0, op->stream>>>(d_gin, op->d_G, ne, me, le, gfft ? 0.0 : 2.0 * 3.141592653589793 / Lp,
                                                       L, omega, cos(L * omega), sin(L * omega), scale);
        cudaError_t e = cudaStreamSynchronize(op->stream);
        if (e != cudaSuccess) { set_error("spectrum setup failed: %s", cudaGetErrorString(e)); delete op; return LS_ERR_CUDA; }
        if (d_gin) op->dfree(d_gin);
    }
    TRY(op->dmalloc((void**)&op->d_A1, (size_t)ne * m * l * sizeof(cd)));
    TRY(op->dmalloc((void**)&op->d_A2, (size_t)ne * me * l * sizeof(cd)));
#undef TRY
    *out = reinterpret_cast<ls_handle>(op);
    return LS_OK;
}

}  // namespace ls
