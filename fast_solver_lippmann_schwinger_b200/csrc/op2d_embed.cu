// Zero-embedded 2-D route (LS_FLAG_EMBED), create time: the lags of the spatial kernel an n x m apply touches, exactly.
//
// The apply is a Toeplitz product: output point i only ever meets input point j through g[i - j], lags (-n, n) x
// (-m, m).  With the reference's spectrum GFFT (ne x me; centred for Greengard_Vico, ne = 4n; natural order for the
// trapezoidal rule, ne = 2n - 1 and the crop [n:2n-1]) and Gd[kx, ky] = GFFT[(kx + sx) % ne, (ky + sy) % me]
// (sx = ne/2 for Greengard_Vico, 0 otherwise; the shift of k_bs_permute_g):
//     g[dx, dy] = 1/(ne me) sum_{kx,ky} Gd[kx, ky] exp(+2 pi i (kx ix(dx) / ne + ky iy(dy) / me))
// with ix(d) = d mod ne (Greengard_Vico) or n - 1 + d (trapezoidal: the crop offset; no wrap, all 2n - 1 lags).
// Only 2n - 1 of the ne output points per dimension are needed, so instead of an ne x me inverse FFT the lags come
// out of two dense products with the (2n - 1)-column DFT matrices, y first, then x:
//     T1 = GFFT * Fy   (ne x (2m-1)),      g = Fx^T * T1 / (ne me)   ((2n-1) x (2m-1))
// F[k, dd] = exp(+2 pi i ((k - s) mod K) * idx(dd) / K): the shift is folded into the matrix, the angle is reduced
// exactly in integers before sincospi.  Native FP64 ZGEMM in cuBLAS's default math mode.  At n = m = 4096
// (Greengard_Vico) that is about 2.6e13 flop and 12 GB of temporaries (estimates).  op2d.cu then places g on the
// 2n' x 2m' grid of the power-of-two apply and transforms it (lag_spectrum).
#include "ls_common.cuh"
#include "op2d_base.cuh"
#include "lag_dft.cuh"

using namespace ls;

namespace {

// g2[(dx mod n2) + n2 * (dy mod m2)] = g[ddx + (2n-1) ddy],  d = dd - (n - 1)
__global__ void k_place_lags(const cd* __restrict__ g, cd* __restrict__ g2, long n, long m, long n2, long m2) {
    const long lx = 2 * n - 1, total = lx * (2 * m - 1);
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const long dx = idx % lx - (n - 1), dy = idx / lx - (m - 1);
        g2[(dx < 0 ? dx + n2 : dx) + n2 * (dy < 0 ? dy + m2 : dy)] = g[idx];
    }
}

}  // namespace

namespace ls {

int embed_lag_grid(HandleBase* op, const cd* gin, long n, long m, long ne, long me, bool trapezoidal,
                   cd* g2, long n2, long m2) {
    cudaStream_t s = op->stream;
    const long lx = 2 * n - 1, ly = 2 * m - 1;
    const long sx = trapezoidal ? 0 : ne / 2, sy = trapezoidal ? 0 : me / 2;
    CublasGuard cb;
    LS_CUBLAS_TRY(cublasCreate(&cb.h));
    LS_CUBLAS_TRY(cublasSetStream(cb.h, s));
    LS_CUBLAS_TRY(cublasSetMathMode(cb.h, CUBLAS_DEFAULT_MATH));
    const cuDoubleComplex one = make_cuDoubleComplex(1.0, 0.0), zero = make_cuDoubleComplex(0.0, 0.0);
    const cuDoubleComplex scale = make_cuDoubleComplex(1.0 / ((double)ne * (double)me), 0.0);
    int rc;
    cd *Fy = nullptr, *T1 = nullptr, *Fx = nullptr, *g = nullptr;
    // y first: T1 = Gin * Fy
    if ((rc = op->dmalloc((void**)&Fy, (size_t)me * ly * sizeof(cd)))) return rc;
    if ((rc = op->dmalloc((void**)&T1, (size_t)ne * ly * sizeof(cd)))) return rc;
    k_dft_lags<<<148 * 8, 256, 0, s>>>(Fy, me, m, sy, trapezoidal ? 1 : 0);
    LS_CUDA_TRY(cudaGetLastError());
    LS_CUBLAS_TRY(cublasZgemm(cb.h, CUBLAS_OP_N, CUBLAS_OP_N, (int)ne, (int)ly, (int)me, &one,
                              reinterpret_cast<const cuDoubleComplex*>(gin), (int)ne,
                              reinterpret_cast<const cuDoubleComplex*>(Fy), (int)me, &zero,
                              reinterpret_cast<cuDoubleComplex*>(T1), (int)ne));
    LS_CUDA_TRY(cudaStreamSynchronize(s));
    op->dfree(Fy);
    // then x: g = Fx^T * T1 / (ne me)
    if ((rc = op->dmalloc((void**)&Fx, (size_t)ne * lx * sizeof(cd)))) return rc;
    if ((rc = op->dmalloc((void**)&g, (size_t)lx * ly * sizeof(cd)))) return rc;
    k_dft_lags<<<148 * 8, 256, 0, s>>>(Fx, ne, n, sx, trapezoidal ? 1 : 0);
    LS_CUDA_TRY(cudaGetLastError());
    LS_CUBLAS_TRY(cublasZgemm(cb.h, CUBLAS_OP_T, CUBLAS_OP_N, (int)lx, (int)ly, (int)ne, &scale,
                              reinterpret_cast<const cuDoubleComplex*>(Fx), (int)ne,
                              reinterpret_cast<const cuDoubleComplex*>(T1), (int)ne, &zero,
                              reinterpret_cast<cuDoubleComplex*>(g), (int)lx));
    LS_CUDA_TRY(cudaStreamSynchronize(s));
    op->dfree(T1);
    op->dfree(Fx);
    // wrap onto the zeroed n2 x m2 grid
    LS_CUDA_TRY(cudaMemsetAsync(g2, 0, (size_t)n2 * m2 * sizeof(cd), s));
    k_place_lags<<<148 * 8, 256, 0, s>>>(g, g2, n, m, n2, m2);
    LS_CUDA_TRY(cudaGetLastError());
    LS_CUDA_TRY(cudaStreamSynchronize(s));
    op->dfree(g);
    return LS_OK;
}

}  // namespace ls
