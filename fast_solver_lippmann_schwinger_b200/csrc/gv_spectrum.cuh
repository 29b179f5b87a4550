// Greengard-Vico truncated-kernel spectrum in 3-D, evaluated on the device.
// Gtruncated3D(L, k, s) = (-1 + e^{iLk} (cos(Ls) - i k L sinc(Ls/pi))) / (k^2 - s^2)   (Functions.jl:49-51;
// Julia's sinc(x) = sin(pi x)/(pi x)).  The sinc argument goes through pi*(Ls/pi) exactly like the
// oracle's numpy.sinc so that both round the same way at arguments ~1e3.
#pragma once
#include "ls_common.cuh"

namespace ls {

__device__ __forceinline__ lsfft::cd gtrunc3d_eval(double s, double L, double k, double eLk_re, double eLk_im) {
    const double PI = 3.141592653589793;
    // Q7: removable singularity at s == k (Functions.jl:50 divides by k^2 - s^2); a grid frequency that hits k exactly is
    // moved by sqrt(eps) relative instead of producing NaN
    if (s == k) s = k * (1.0 + 1.4901161193847656e-08);
    const double Ls = L * s;
    const double c = cos(Ls);
    double sinc;
    {
        const double xs = Ls / PI;
        const double yv = PI * xs;
        sinc = (xs == 0.0) ? 1.0 : sin(yv) / yv;
    }
    const double ar = c, ai = -(k * L * sinc);
    const double nr = -1.0 + (eLk_re * ar - eLk_im * ai);
    const double ni = eLk_re * ai + eLk_im * ar;
    const double den = k * k - s * s;
    return make_double2(nr / den, ni / den);
}

// |kappa| on the centred grid (2 pi/Lp)(-N/2 .. N/2-1), summed like numpy: (kx^2 + ky^2) + kz^2, no FMA contraction
__device__ __forceinline__ double gv_radius(double dk, long ix, long iy, long iz, long ne, long me, long le) {
    const double kxv = dk * (double)(ix - ne / 2);
    const double kyv = dk * (double)(iy - me / 2);
    const double kzv = dk * (double)(iz - le / 2);
    return sqrt(__dadd_rn(__dadd_rn(__dmul_rn(kxv, kxv), __dmul_rn(kyv, kyv)), __dmul_rn(kzv, kzv)));
}

int create_op3d_generic(ls_handle* out, int64_t n, int64_t m, int64_t l, int64_t ne, int64_t me, int64_t le,
                        const double* nu, const ls_cdouble* gfft, double omega, double L, double Lp);
// ls_op3d_lines of a general-size handle: its Bluestein convolution lengths
void op3d_generic_lines(const HandleBase* h, int64_t* n_line, int64_t* m_line, int64_t* l_line);

// Zero-embedded 3-D route, create time (op3d_embed.cu): the lags (-n, n)^2 x (-l, l) of the spatial kernel
// g = ifftn(GFFT) wrapped onto the zeroed n2 x n2 x l2 grid (negative lags at the end), this rank's z slab of it:
// g2[jx + n2*(jy + n2*jz_loc)], planes [rank*l2/P, (rank+1)*l2/P).  gin: the 4n x 4n x 4l centred spectrum on the
// device, or nullptr to evaluate Gtruncated3D(L, omega) on the grid of period Lp.  Rank r contracts the x-slots
// [r*4n/P, (r+1)*4n/P) of the spectrum; P > 1 sums the partial grids with one ncclReduceScatter over `comm`.
// chunk_slots > 0 sets the x-slots per chunk of the contraction (0: as many as 8 GB of spectrum hold).
int embed_lag_grid3d(HandleBase* op, const lsfft::cd* gin, long n, long l, double omega, double L, double Lp,
                     int rank, int P, ncclComm_t comm, lsfft::cd* g2, long n2, long l2, long chunk_slots);

}  // namespace ls
