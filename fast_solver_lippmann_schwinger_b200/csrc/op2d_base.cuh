// Common part of the 2-D operator implementations (power-of-two pruned path and its zero-embedded use for
// any size, op2d.cu + op2d_embed.cu; general-size Bluestein path, op2d_generic.cu).
#pragma once
#include "ls_common.cuh"

namespace ls {

struct Op2DBase : HandleBase {
    long n = 0, m = 0, ne = 0, me = 0;
    double omega = 0;
    int quadrule = 0;
    cd* d_b = nullptr; cd* d_y = nullptr;   // staging for host-pointer applies
    int64_t op_size() const override { return n * m; }
    // ls_op2d_info: route (0 power of two, 1 Bluestein, 2 zero-embedded), the line lengths the kernels run, and the
    // padding factor of the spectrum the applies use
    virtual void info(int* route, int64_t* n_line, int64_t* m_line, int* padding) const = 0;
};

// Zero-embedded route, create time: the lags (-n, n) x (-m, m) of the spatial kernel g = ifft2(GFFT) wrapped onto the
// zeroed n2 x m2 grid g2[jx + n2*jy] (negative lags at the end), n2 >= 2n, m2 >= 2m.  gin: the ne x me spectrum on
// the device in the reference's layout (centred for Greengard_Vico).  Two cuBLAS ZGEMMs against DFT matrices built on
// the device; temporaries are allocated and freed through `op`.
int embed_lag_grid(HandleBase* op, const cd* gin, long n, long m, long ne, long me, bool trapezoidal,
                   cd* g2, long n2, long m2);

// general sizes / trapezoidal rule: line DFTs of arbitrary length by Bluestein's algorithm on the
// power-of-two engine.  Returns LS_ERR_UNSUPPORTED when a padded line does not fit the engine.
// gfft: host array in the reference's layout, or nullptr with gfft_dev = the same array already on the device.
int create_op2d_generic(ls_handle* out, int64_t n, int64_t m, int64_t ne, int64_t me, const double* nu,
                        const ls_cdouble* gfft, double omega, int quadrule, const cd* gfft_dev = nullptr);

}  // namespace ls
