// Zero-embedded 3-D route (LS_FLAG_EMBED), create time: the lags of the spatial kernel an n x n x l apply touches,
// exactly.  3-D version of op2d_embed.cu.
//
// The apply only ever meets g at the lags (-n, n)^2 x (-l, l).  With the reference's centred spectrum GFFT
// (ne = me = 4n, le = 4l) those (2n - 1)^2 (2l - 1) values are three dense contractions with the lag DFT matrices
// F[k, dd] = exp(+2 pi i ((k - K/2) mod K) (d mod K) / K) of k_dft_lags:
//     T1 = S  *_z Fz   (one ZGEMM),   T2 = T1 *_y Fy   (strided-batched over the z lags),   g += Fx^T *_x T2 / (ne me le)
// Native FP64 ZGEMM in cuBLAS's default math mode.  The 4n x 4n x 4l spectrum S (136 GB at n = l = 511) is never
// resident: it is generated (Gtruncated3D, as k_fill_g3d does) or gathered from the uploaded GFFT in x-slot chunks of
// at most CHUNK_BYTES (LS_OP3D_EMBED_CHUNK_SLOTS forces the width), and the x contraction accumulates over the chunks.  About 1.2e14 flop at n = l = 511, 5e13 at
// 400 (estimates).  Sharded, rank r contracts only its x-slots [r*4n/P, (r+1)*4n/P): its partial lags are placed on
// the whole 2n' x 2n' x 2l' grid and one ncclReduceScatter over z-plane blocks leaves every rank its 2l'/P summed
// planes, the slab op3d.cu's lag_spectrum3d transforms.
#include "ls_common.cuh"
#include "gv_spectrum.cuh"
#include "lag_dft.cuh"
#include <algorithm>

using namespace ls;

namespace {

constexpr double CHUNK_BYTES = 8e9;     // spectrum chunk S; the z contraction's output T1 is about half of it

// S[ixl + cw*(iy + me*iz)] = GFFT[x0 + ixl, iy, iz] (centred), gathered from gin or evaluated (Gtruncated3D)
__global__ void k_fill_xchunk(const cd* __restrict__ gin, cd* __restrict__ S, long x0, long cw, long ne, long me, long le,
                              double dk, double L, double k, double eLk_re, double eLk_im) {
    const long total = cw * me * le;
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const long ix = x0 + idx % cw, q = idx / cw;
        const long iy = q % me, iz = q / me;
        S[idx] = gin != nullptr ? gin[ix + ne * (iy + me * iz)]
                                : gtrunc3d_eval(gv_radius(dk, ix, iy, iz, ne, me, le), L, k, eLk_re, eLk_im);
    }
}

// g2[(dx mod n2) + n2*((dy mod n2) + n2*(dz mod l2))] = g[ddx + lx*(ddy + lx*ddz)],  d = dd - (n - 1) (z: l - 1)
__global__ void k_place_lags3(const cd* __restrict__ g, cd* __restrict__ g2, long n, long l, long n2, long l2) {
    const long lx = 2 * n - 1, total = lx * lx * (2 * l - 1);
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const long dx = idx % lx - (n - 1), dy = (idx / lx) % lx - (n - 1), dz = idx / (lx * lx) - (l - 1);
        g2[(dx < 0 ? dx + n2 : dx) + n2 * ((dy < 0 ? dy + n2 : dy) + n2 * (dz < 0 ? dz + l2 : dz))] = g[idx];
    }
}

}  // namespace

namespace ls {

int embed_lag_grid3d(HandleBase* op, const cd* gin, long n, long l, double omega, double L, double Lp,
                     int rank, int P, ncclComm_t comm, cd* g2, long n2, long l2, long chunk_slots) {
    cudaStream_t s = op->stream;
    const long ne = 4 * n, me = 4 * n, le = 4 * l;
    const long lx = 2 * n - 1, lz = 2 * l - 1;
    const long x0 = ne * rank / P, x1 = ne * (rank + 1) / P;          // this rank's x-slots of the spectrum
    const long by_size = (long)(CHUNK_BYTES / ((double)me * le * sizeof(cd)));
    const long cw = std::max(1L, std::min(x1 - x0, chunk_slots > 0 ? chunk_slots : by_size));
    const double dk = gin ? 0.0 : 2.0 * 3.141592653589793 / Lp;
    CublasGuard cb;
    LS_CUBLAS_TRY(cublasCreate(&cb.h));
    LS_CUBLAS_TRY(cublasSetStream(cb.h, s));
    LS_CUBLAS_TRY(cublasSetMathMode(cb.h, CUBLAS_DEFAULT_MATH));
    const cuDoubleComplex one = make_cuDoubleComplex(1.0, 0.0), zero = make_cuDoubleComplex(0.0, 0.0);
    const cuDoubleComplex scale = make_cuDoubleComplex(1.0 / ((double)ne * (double)me * (double)le), 0.0);
    int rc;
    cd *Fx = nullptr, *Fy = nullptr, *Fz = nullptr, *S = nullptr, *T1 = nullptr, *T2 = nullptr, *g = nullptr;
    if ((rc = op->dmalloc((void**)&Fx, (size_t)ne * lx * sizeof(cd)))) return rc;
    if ((rc = op->dmalloc((void**)&Fy, (size_t)me * lx * sizeof(cd)))) return rc;
    if ((rc = op->dmalloc((void**)&Fz, (size_t)le * lz * sizeof(cd)))) return rc;
    if ((rc = op->dmalloc((void**)&S, (size_t)cw * me * le * sizeof(cd)))) return rc;
    if ((rc = op->dmalloc((void**)&T1, (size_t)cw * me * lz * sizeof(cd)))) return rc;
    if ((rc = op->dmalloc((void**)&T2, (size_t)cw * lx * lz * sizeof(cd)))) return rc;
    if ((rc = op->dmalloc((void**)&g, (size_t)lx * lx * lz * sizeof(cd)))) return rc;
    k_dft_lags<<<148 * 8, 256, 0, s>>>(Fx, ne, n, ne / 2, 0);
    k_dft_lags<<<148 * 8, 256, 0, s>>>(Fy, me, n, me / 2, 0);
    k_dft_lags<<<148 * 8, 256, 0, s>>>(Fz, le, l, le / 2, 0);
    LS_CUDA_TRY(cudaGetLastError());
    LS_CUDA_TRY(cudaMemsetAsync(g, 0, (size_t)lx * lx * lz * sizeof(cd), s));
    for (long c0 = x0; c0 < x1; c0 += cw) {
        const long w = std::min(cw, x1 - c0);
        k_fill_xchunk<<<148 * 16, 256, 0, s>>>(gin, S, c0, w, ne, me, le, dk, L, omega, cos(L * omega), sin(L * omega));
        LS_CUDA_TRY(cudaGetLastError());
        // z: T1[ixl + w*iy, dz] = sum_iz S[ixl + w*iy, iz] Fz[iz, dz]
        LS_CUBLAS_TRY(cublasZgemm(cb.h, CUBLAS_OP_N, CUBLAS_OP_N, (int)(w * me), (int)lz, (int)le, &one,
                                  reinterpret_cast<const cuDoubleComplex*>(S), (int)(w * me),
                                  reinterpret_cast<const cuDoubleComplex*>(Fz), (int)le, &zero,
                                  reinterpret_cast<cuDoubleComplex*>(T1), (int)(w * me)));
        // y, per z lag: T2[ixl + w*dy + w*lx*dz] = sum_iy T1[ixl + w*iy + w*me*dz] Fy[iy, dy]
        LS_CUBLAS_TRY(cublasZgemmStridedBatched(cb.h, CUBLAS_OP_N, CUBLAS_OP_N, (int)w, (int)lx, (int)me, &one,
                                                reinterpret_cast<const cuDoubleComplex*>(T1), (int)w, (long long)w * me,
                                                reinterpret_cast<const cuDoubleComplex*>(Fy), (int)me, 0LL, &zero,
                                                reinterpret_cast<cuDoubleComplex*>(T2), (int)w, (long long)w * lx, (int)lz));
        // x, accumulated over the chunks: g[dx, (dy, dz)] += sum_ixl Fx[c0 + ixl, dx] T2[ixl, (dy, dz)] / (ne me le)
        LS_CUBLAS_TRY(cublasZgemm(cb.h, CUBLAS_OP_T, CUBLAS_OP_N, (int)lx, (int)(lx * lz), (int)w, &scale,
                                  reinterpret_cast<const cuDoubleComplex*>(Fx + c0), (int)ne,
                                  reinterpret_cast<const cuDoubleComplex*>(T2), (int)w, &one,
                                  reinterpret_cast<cuDoubleComplex*>(g), (int)lx));
    }
    LS_CUDA_TRY(cudaStreamSynchronize(s));
    op->dfree(S); op->dfree(T1); op->dfree(T2);
    op->dfree(Fx); op->dfree(Fy); op->dfree(Fz);
    // wrap onto the zeroed grid: the whole grid on every rank when P > 1 (partial sums), reduced into the z slabs
    const size_t grid = (size_t)n2 * n2 * l2;
    cd* full = g2;
    if (P > 1 && (rc = op->dmalloc((void**)&full, grid * sizeof(cd)))) return rc;
    LS_CUDA_TRY(cudaMemsetAsync(full, 0, grid * sizeof(cd), s));
    k_place_lags3<<<148 * 8, 256, 0, s>>>(g, full, n, l, n2, l2);
    LS_CUDA_TRY(cudaGetLastError());
    if (P > 1) {
        ncclResult_t r = ncclReduceScatter(full, g2, 2 * grid / P, ncclDouble, ncclSum, comm, s);
        if (r != ncclSuccess) { set_error("lag reduce-scatter failed: %s", ncclGetErrorString(r)); return LS_ERR_NCCL; }
    }
    LS_CUDA_TRY(cudaStreamSynchronize(s));
    op->dfree(g);
    if (full != g2) op->dfree(full);
    return LS_OK;
}

}  // namespace ls
