// Lag DFT matrices and cuBLAS plumbing shared by the zero-embedded routes' create-time lag extraction
// (op2d_embed.cu, op3d_embed.cu).
#pragma once
#include "ls_common.cuh"
#include <cublas_v2.h>

namespace {

using ls::cd;

#define LS_CUBLAS_TRY(expr)                                                                        \
    do {                                                                                           \
        cublasStatus_t _s = (expr);                                                                \
        if (_s != CUBLAS_STATUS_SUCCESS) {                                                         \
            set_error("%s failed at %s:%d: cuBLAS status %d", #expr, __FILE__, __LINE__, (int)_s); \
            return LS_ERR_CUDA;                                                                    \
        }                                                                                          \
    } while (0)

// F[k + K*dd], k < K, dd < 2nv - 1 (lag d = dd - (nv - 1))
__global__ void k_dft_lags(cd* __restrict__ F, long K, long nv, long shift, int trapezoidal) {
    const long nl = 2 * nv - 1, total = K * nl;
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const long k = idx % K, dd = idx / K;
        const long col = trapezoidal ? dd : ((dd - (nv - 1)) % K + K) % K;
        const long row = ((k - shift) % K + K) % K;
        const long r = (row * col) % K;
        double s, c;
        sincospi(2.0 * (double)r / (double)K, &s, &c);
        F[idx] = make_double2(c, s);
    }
}

struct CublasGuard {
    cublasHandle_t h = nullptr;
    ~CublasGuard() { if (h) cublasDestroy(h); }
};

}  // namespace
