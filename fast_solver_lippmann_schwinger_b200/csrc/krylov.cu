// GMRES Arnoldi vector kernels and a device-resident restarted GMRES driver.
//
// The reference calls IterativeSolvers.jl `gmres!` (examples/example.jl:85,91; example3D.jl:78;
// tests/plasma_example.jl:164,176); that package is not vendored, its algorithm (restart 20,
// modified Gram-Schmidt, left preconditioner, null-vector residual estimate) is restated in
// oracle/gmres_is.py and reproduced here step for step so residual histories agree.
//
//   zdotc  : sum conj(x) y      (BLAS zdotc: conjugates the FIRST argument, like Julia's dot)
//   dznrm2 : sqrt(sum |x|^2)
//   zaxpy / zscal, and the fused modified-Gram-Schmidt passes
//        k_axpy_dot  : w -= h_prev * V_prev ;  h = conj(V_i) . w      (one sweep: 64 B/elt)
//        k_axpy_nrm2 : w -= h_prev * V_prev ;  s = |w|^2              (48 B/elt)
//   All reductions: 128-bit loads, per-thread partial sums, warp shuffles, one partial per CTA,
//   the last CTA (ticket) folds the partials in a fixed order -> bitwise reproducible.
//   Scalars stay on the device between the passes of one Gram-Schmidt sweep; one D2H copy of the
//   Hessenberg column per GMRES iteration.
#include "ls_common.cuh"
#include "spmv.cuh"
#include <algorithm>
#include <chrono>
#include <cstring>

using namespace ls;

namespace {

constexpr int RED_THREADS = 256;
constexpr int RED_BLOCKS = 148 * 8;

struct RedOut {       // where a reduction result goes (device)
    double* re;       // receives sum.x (or sqrt(sum.x) if take_sqrt)
    double* im;       // receives sum.y (may be null)
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// block-level fold + "last block finalises" (deterministic order)
__device__ __forceinline__ void block_finish(double sx, double sy, double2* partials, unsigned* ticket,
                                             double* out_re, double* out_im, int take_sqrt) {
    __shared__ double shx[RED_THREADS / 32], shy[RED_THREADS / 32];
    __shared__ bool is_last;
    sx = warp_sum(sx);
    sy = warp_sum(sy);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) { shx[w] = sx; shy[w] = sy; }
    __syncthreads();
    if (w == 0) {
        sx = (l < RED_THREADS / 32) ? shx[l] : 0.0;
        sy = (l < RED_THREADS / 32) ? shy[l] : 0.0;
        sx = warp_sum(sx);
        sy = warp_sum(sy);
        if (l == 0) {
            partials[blockIdx.x] = make_double2(sx, sy);
            __threadfence();
            unsigned t = atomicInc(ticket, gridDim.x - 1);
            is_last = (t == gridDim.x - 1);
        }
    }
    __syncthreads();
    if (is_last) {
        __threadfence();
        double ax = 0.0, ay = 0.0;
        for (int i = threadIdx.x; i < (int)gridDim.x; i += RED_THREADS) {
            double2 p = __ldcg(&partials[i]);
            ax += p.x;
            ay += p.y;
        }
        ax = warp_sum(ax);
        ay = warp_sum(ay);
        if (l == 0) { shx[w] = ax; shy[w] = ay; }
        __syncthreads();
        if (threadIdx.x == 0) {
            double tx = 0.0, ty = 0.0;
            for (int i = 0; i < RED_THREADS / 32; ++i) { tx += shx[i]; ty += shy[i]; }
            *out_re = take_sqrt ? sqrt(tx) : tx;
            if (out_im) *out_im = ty;
        }
    }
}

// ---- L2 residency hints (LS_MGS_L2HINT=1, experiment) --------------------------------------------------------------
// A modified Gram-Schmidt sweep re-reads and re-writes w in every one of its k steps while the basis columns stream by
// once each.  At 2048^2 w is 67 MB against 126 MB of L2: loading / storing w with an evict_last policy and the basis
// columns with evict_first asks the L2 to keep w resident across the sweep (64 -> 32 bytes of HBM traffic per element
// and step if it does).
__device__ __forceinline__ unsigned long long l2_policy_last() {
    unsigned long long p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ unsigned long long l2_policy_first() {
    unsigned long long p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
template <bool HINT> __device__ __forceinline__ cd ld_pol(const cd* p, unsigned long long pol) {
    if (!HINT) return *p;
    cd v;
    asm volatile("ld.global.L2::cache_hint.v2.f64 {%0, %1}, [%2], %3;" : "=d"(v.x), "=d"(v.y) : "l"(p), "l"(pol));
    return v;
}
template <bool HINT> __device__ __forceinline__ void st_pol(cd* p, cd v, unsigned long long pol) {
    if (!HINT) { *p = v; return; }
    asm volatile("st.global.L2::cache_hint.v2.f64 [%0], {%1, %2}, %3;" ::"l"(p), "d"(v.x), "d"(v.y), "l"(pol) : "memory");
}

// h = conj(x) . y
__global__ void __launch_bounds__(RED_THREADS)
k_dot(const cd* __restrict__ x, const cd* __restrict__ y, long n, double2* partials, unsigned* ticket,
      double* out_re, double* out_im) {
    double sx = 0.0, sy = 0.0;
    for (long i = (long)blockIdx.x * RED_THREADS + threadIdx.x; i < n; i += (long)gridDim.x * RED_THREADS) {
        const cd a = x[i], b = y[i];
        sx += a.x * b.x + a.y * b.y;
        sy += a.x * b.y - a.y * b.x;
    }
    block_finish(sx, sy, partials, ticket, out_re, out_im, 0);
}

__global__ void k_sqrt1(double* v) { *v = sqrt(*v); }

__global__ void __launch_bounds__(RED_THREADS)
k_nrm2(const cd* __restrict__ x, long n, double2* partials, unsigned* ticket, double* out, int take_sqrt) {
    double sx = 0.0;
    for (long i = (long)blockIdx.x * RED_THREADS + threadIdx.x; i < n; i += (long)gridDim.x * RED_THREADS) {
        const cd a = x[i];
        sx += a.x * a.x + a.y * a.y;
    }
    block_finish(sx, 0.0, partials, ticket, out, nullptr, take_sqrt);
}

// w -= h_prev * vprev ;  h = conj(vi) . w
template <bool HINT>
__global__ void __launch_bounds__(RED_THREADS)
k_axpy_dot(const cd* __restrict__ vprev, const double* hprev_re, const double* hprev_im,
           const cd* __restrict__ vi, cd* w, long n, double2* partials, unsigned* ticket,
           double* out_re, double* out_im) {
    const double hr = *hprev_re, hi = *hprev_im;
    const unsigned long long keep = HINT ? l2_policy_last() : 0ull, stream = HINT ? l2_policy_first() : 0ull;
    double sx = 0.0, sy = 0.0;
    for (long i = (long)blockIdx.x * RED_THREADS + threadIdx.x; i < n; i += (long)gridDim.x * RED_THREADS) {
        const cd p = ld_pol<HINT>(&vprev[i], stream);
        cd ww = ld_pol<HINT>(&w[i], keep);
        ww.x -= hr * p.x - hi * p.y;
        ww.y -= hr * p.y + hi * p.x;
        st_pol<HINT>(&w[i], ww, keep);
        const cd a = ld_pol<HINT>(&vi[i], stream);
        sx += a.x * ww.x + a.y * ww.y;
        sy += a.x * ww.y - a.y * ww.x;
    }
    block_finish(sx, sy, partials, ticket, out_re, out_im, 0);
}

// w -= h_prev * vprev ;  out = sqrt(sum |w|^2)
template <bool HINT>
__global__ void __launch_bounds__(RED_THREADS)
k_axpy_nrm2(const cd* __restrict__ vprev, const double* hprev_re, const double* hprev_im, cd* w, long n,
            double2* partials, unsigned* ticket, double* out, int take_sqrt) {
    const double hr = *hprev_re, hi = *hprev_im;
    const unsigned long long keep = HINT ? l2_policy_last() : 0ull, stream = HINT ? l2_policy_first() : 0ull;
    double sx = 0.0;
    for (long i = (long)blockIdx.x * RED_THREADS + threadIdx.x; i < n; i += (long)gridDim.x * RED_THREADS) {
        const cd p = ld_pol<HINT>(&vprev[i], stream);
        cd ww = ld_pol<HINT>(&w[i], keep);
        ww.x -= hr * p.x - hi * p.y;
        ww.y -= hr * p.y + hi * p.x;
        st_pol<HINT>(&w[i], ww, keep);
        sx += ww.x * ww.x + ww.y * ww.y;
    }
    block_finish(sx, 0.0, partials, ticket, out, nullptr, take_sqrt);
}

// ---- classical Gram-Schmidt (orth_meth = ClassicalGramSchmidt / DGKS upstream): BLAS-2 style sweeps ----
constexpr int KC = 8;     // columns per multi-dot pass

// h[c0 + i] = conj(V[:, c0 + i]) . w for i < kc <= KC, one sweep over w and kc columns
__global__ void __launch_bounds__(RED_THREADS)
k_multi_dot(const cd* __restrict__ V, long ldv, int c0, int kc, const cd* __restrict__ w, long n,
            double2* partials /* [KC][gridDim.x] */, unsigned* ticket, double* out /* 2*(c0+i) */) {
    double sx[KC], sy[KC];
#pragma unroll
    for (int i = 0; i < KC; ++i) { sx[i] = 0.0; sy[i] = 0.0; }
    for (long e = (long)blockIdx.x * RED_THREADS + threadIdx.x; e < n; e += (long)gridDim.x * RED_THREADS) {
        const cd b = w[e];
#pragma unroll
        for (int i = 0; i < KC; ++i) {
            if (i < kc) {
                const cd a = V[e + (long)(c0 + i) * ldv];
                sx[i] += a.x * b.x + a.y * b.y;
                sy[i] += a.x * b.y - a.y * b.x;
            }
        }
    }
    __shared__ double shx[KC][RED_THREADS / 32], shy[KC][RED_THREADS / 32];
    __shared__ bool is_last;
    const int wp = threadIdx.x >> 5, l = threadIdx.x & 31;
#pragma unroll
    for (int i = 0; i < KC; ++i) {
        const double a = warp_sum(sx[i]), b = warp_sum(sy[i]);
        if (l == 0) { shx[i][wp] = a; shy[i][wp] = b; }
    }
    __syncthreads();
    if (threadIdx.x < KC) {
        double a = 0.0, b = 0.0;
        for (int q = 0; q < RED_THREADS / 32; ++q) { a += shx[threadIdx.x][q]; b += shy[threadIdx.x][q]; }
        partials[(long)threadIdx.x * gridDim.x + blockIdx.x] = make_double2(a, b);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned tk = atomicInc(ticket, gridDim.x - 1);
        is_last = (tk == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) {
        __threadfence();
        for (int i = 0; i < kc; ++i) {
            double ax = 0.0, ay = 0.0;
            for (int q = threadIdx.x; q < (int)gridDim.x; q += RED_THREADS) {
                const double2 p = __ldcg(&partials[(long)i * gridDim.x + q]);
                ax += p.x;
                ay += p.y;
            }
            ax = warp_sum(ax);
            ay = warp_sum(ay);
            __syncthreads();
            if (l == 0) { shx[0][wp] = ax; shy[0][wp] = ay; }
            __syncthreads();
            if (threadIdx.x == 0) {
                double tx = 0.0, ty = 0.0;
                for (int q = 0; q < RED_THREADS / 32; ++q) { tx += shx[0][q]; ty += shy[0][q]; }
                out[2 * (c0 + i)] = tx;
                out[2 * (c0 + i) + 1] = ty;
            }
        }
    }
}

// w -= sum_{i<k} h_i V_i ;  out = sqrt(sum |w|^2)   (h: k complex values on the device)
__global__ void __launch_bounds__(RED_THREADS)
k_multi_axpy_nrm2(const cd* __restrict__ V, long ldv, int k, const double* __restrict__ h, cd* w, long n,
                  double2* partials, unsigned* ticket, double* out, int take_sqrt) {
    __shared__ double hs[128];
    for (int i = threadIdx.x; i < 2 * k; i += RED_THREADS) hs[i] = h[i];
    __syncthreads();
    double sx = 0.0;
    for (long e = (long)blockIdx.x * RED_THREADS + threadIdx.x; e < n; e += (long)gridDim.x * RED_THREADS) {
        cd ww = w[e];
        for (int i = 0; i < k; ++i) {
            const cd p = V[e + (long)i * ldv];
            ww.x -= hs[2 * i] * p.x - hs[2 * i + 1] * p.y;
            ww.y -= hs[2 * i] * p.y + hs[2 * i + 1] * p.x;
        }
        w[e] = ww;
        sx += ww.x * ww.x + ww.y * ww.y;
    }
    block_finish(sx, 0.0, partials, ticket, out, nullptr, take_sqrt);
}

// y += alpha*x  (alpha by value)
__global__ void __launch_bounds__(256)
k_axpy(cd alpha, const cd* __restrict__ x, cd* y, long n) {
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        const cd a = x[i];
        cd b = y[i];
        b.x += alpha.x * a.x - alpha.y * a.y;
        b.y += alpha.x * a.y + alpha.y * a.x;
        y[i] = b;
    }
}
__global__ void __launch_bounds__(256)
k_scal(cd alpha, cd* x, long n) {
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        const cd a = x[i];
        x[i] = make_double2(alpha.x * a.x - alpha.y * a.y, alpha.x * a.y + alpha.y * a.x);
    }
}
// x *= 1/(*nrm)   (nrm on the device); optionally also writes the scaled vector to `copy`
__global__ void __launch_bounds__(256)
k_scal_inv_dev(const double* nrm, cd* x, long n) {
    const double s = 1.0 / *nrm;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        cd a = x[i];
        a.x *= s;
        a.y *= s;
        x[i] = a;
    }
}
// r = b - ax
__global__ void __launch_bounds__(256)
k_sub(const cd* __restrict__ b, const cd* __restrict__ ax, cd* r, long n) {
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        const cd p = b[i], q = ax[i];
        r[i] = make_double2(p.x - q.x, p.y - q.y);
    }
}
// x += V[:, 0:k] * y   (y: k complex values on the device; V column-major, leading dimension ldv)
__global__ void __launch_bounds__(256)
k_update_solution(const cd* __restrict__ V, long ldv, int k, const cd* __restrict__ y, cd* x, long n) {
    __shared__ cd ys[64];
    if (threadIdx.x < k) ys[threadIdx.x] = y[threadIdx.x];
    __syncthreads();
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        cd acc = x[i];
        for (int j = 0; j < k; ++j) {
            const cd v = V[i + (long)j * ldv];
            acc.x += v.x * ys[j].x - v.y * ys[j].y;
            acc.y += v.x * ys[j].y + v.y * ys[j].x;
        }
        x[i] = acc;
    }
}

struct Krylov : HandleBase {
    long n = 0;
    double2* d_partials = nullptr;
    unsigned* d_ticket = nullptr;
    double* d_scal = nullptr;     // 2*(64+2) doubles: Hessenberg column (re, im interleaved) + scratch
    double* h_scal = nullptr;     // pinned mirror
    cd* d_y = nullptr;            // least-squares solution for the x update
    cd* d_V = nullptr; long v_cols = 0;
    cd* d_ax = nullptr; cd* d_b = nullptr; cd* d_x = nullptr;
    cd* h_stage = nullptr;        // pinned staging for the preconditioner callback
    // ls_gmres_msp_batch: the systems' Krylov bases, the columns of the batched Msp solve, host-pointer b / x staging
    cd* d_Vb = nullptr; size_t Vb_bytes = 0;
    cd* d_Pb = nullptr; size_t Pb_bytes = 0;
    cd* d_bxb = nullptr; size_t bxb_bytes = 0;
    // (re)allocates *p when it holds fewer than `bytes`
    int ensure(cd** p, size_t& have, size_t bytes) {
        if (have >= bytes) return LS_OK;
        if (*p) dfree(*p);
        *p = nullptr; have = 0;
        int rc = dmalloc((void**)p, bytes);
        if (rc) return rc;
        have = bytes;
        return LS_OK;
    }
    double t_precond_host_s = 0.0; // last ls_gmres: wall time inside D2H + callback + H2D of the Msp solve

    int grid_stream(long nn) const { long b = (nn + 255) / 256; return (int)(b < 148 * 16 ? (b > 0 ? b : 1) : 148 * 16); }

    // sharded vectors (z slabs, one process per GPU): local sums are all-reduced as scalars
    ncclComm_t comm = nullptr;
    int allreduce(double* v, int count, cudaStream_t s) {
        if (!comm) return LS_OK;
        ncclResult_t r = ncclAllReduce(v, v, count, ncclDouble, ncclSum, comm, s);
        if (r != ncclSuccess) { set_error("ncclAllReduce failed: %s", ncclGetErrorString(r)); return LS_ERR_NCCL; }
        return LS_OK;
    }
    int finish_norm(double* v, cudaStream_t s) {
        if (!comm) return LS_OK;
        int rc = allreduce(v, 1, s);
        if (rc) return rc;
        k_sqrt1<<<1, 1, 0, s>>>(v);
        launches++;
        return LS_OK;
    }
    int dot(const cd* x, const cd* y, double* out2, cudaStream_t s) {
        k_dot<<<RED_BLOCKS, RED_THREADS, 0, s>>>(x, y, n, d_partials, d_ticket, out2, out2 + 1);
        launches++;
        return allreduce(out2, 2, s);
    }
    int nrm2(const cd* x, double* out, cudaStream_t s) {
        k_nrm2<<<RED_BLOCKS, RED_THREADS, 0, s>>>(x, n, d_partials, d_ticket, out, comm ? 0 : 1);
        launches++;
        return finish_norm(out, s);
    }
    // modified Gram-Schmidt of w against V[:,0..k-1] and normalisation; h (k+1 complex) lands in d_scal
    int mgs(const cd* V, long ldv, int k, cd* w, cudaStream_t s) {
        double* h = d_scal;
        int rc;
        if (k == 0) {
            if ((rc = nrm2(w, h, s))) return rc;
            cudaMemsetAsync(h + 1, 0, sizeof(double), s);
        } else {
            // L2 residency hints: on when w (16 n bytes) can live in the 126 MB L2 next to the streaming columns.
            // Measured at 2048^2 (w = 67 MB, profiles/r2_m_mgs.log): sweep k = 20 0.986 -> 0.868 ms, GMRES 0.896 -> 0.845 ms/iter
            static int l2env = -2;
            if (l2env == -2) { const char* e = getenv("LS_MGS_L2HINT"); l2env = e ? atoi(e) : -1; }
            const int l2hint = l2env >= 0 ? l2env : ((size_t)n * sizeof(cd) <= ((size_t)96 << 20) ? 1 : 0);
            if ((rc = dot(V, w, h, s))) return rc;
            for (int i = 1; i < k; ++i) {
                if (l2hint)
                    k_axpy_dot<true><<<RED_BLOCKS, RED_THREADS, 0, s>>>(V + (long)(i - 1) * ldv, h + 2 * (i - 1), h + 2 * (i - 1) + 1,
                                                                        V + (long)i * ldv, w, n, d_partials, d_ticket, h + 2 * i, h + 2 * i + 1);
                else
                    k_axpy_dot<false><<<RED_BLOCKS, RED_THREADS, 0, s>>>(V + (long)(i - 1) * ldv, h + 2 * (i - 1), h + 2 * (i - 1) + 1,
                                                                         V + (long)i * ldv, w, n, d_partials, d_ticket, h + 2 * i, h + 2 * i + 1);
                launches++;
                if ((rc = allreduce(h + 2 * i, 2, s))) return rc;
            }
            if (l2hint)
                k_axpy_nrm2<true><<<RED_BLOCKS, RED_THREADS, 0, s>>>(V + (long)(k - 1) * ldv, h + 2 * (k - 1), h + 2 * (k - 1) + 1, w, n,
                                                                     d_partials, d_ticket, h + 2 * k, comm ? 0 : 1);
            else
            k_axpy_nrm2<false><<<RED_BLOCKS, RED_THREADS, 0, s>>>(V + (long)(k - 1) * ldv, h + 2 * (k - 1), h + 2 * (k - 1) + 1, w, n,
                                                           d_partials, d_ticket, h + 2 * k, comm ? 0 : 1);
            launches++;
            if ((rc = finish_norm(h + 2 * k, s))) return rc;
            cudaMemsetAsync(h + 2 * k + 1, 0, sizeof(double), s);
        }
        k_scal_inv_dev<<<grid_stream(n), 256, 0, s>>>(h + 2 * k, w, n);
        launches++;
        return LS_OK;
    }

    // orth_meth: 0 ModifiedGramSchmidt (default, what the reference's call sites use), 1 ClassicalGramSchmidt,
    // 2 DGKS (classical + conditional re-orthogonalisation) - IterativeSolvers.jl orthogonalize.jl
    int orth_meth = 0;
    double2* d_partials_multi = nullptr;
    double* d_corr = nullptr;
    int multi_dot(const cd* V, long ldv, int k, const cd* w, double* out, cudaStream_t s) {
        for (int c0 = 0; c0 < k; c0 += KC) {
            const int kc = (k - c0) < KC ? (k - c0) : KC;
            k_multi_dot<<<RED_BLOCKS, RED_THREADS, 0, s>>>(V, ldv, c0, kc, w, n, d_partials_multi, d_ticket, out);
            launches++;
        }
        return allreduce(out, 2 * k, s);
    }
    // classical Gram-Schmidt (+ DGKS) of w against V[:,0..k-1] and normalisation; h lands in d_scal
    int cgs(const cd* V, long ldv, int k, cd* w, cudaStream_t s) {
        double* h = d_scal;
        int rc;
        if ((rc = multi_dot(V, ldv, k, w, h, s))) return rc;
        k_multi_axpy_nrm2<<<RED_BLOCKS, RED_THREADS, 0, s>>>(V, ldv, k, h, w, n, d_partials, d_ticket, h + 2 * k, comm ? 0 : 1);
        launches++;
        if ((rc = finish_norm(h + 2 * k, s))) return rc;
        cudaMemsetAsync(h + 2 * k + 1, 0, sizeof(double), s);
        if (orth_meth == 2) {
            std::vector<double> hh(2 * (size_t)k + 2), cc(2 * (size_t)k + 2);
            LS_CUDA_TRY(cudaMemcpyAsync(h_scal, h, (2 * (size_t)k + 1) * sizeof(double), cudaMemcpyDeviceToHost, s));
            LS_CUDA_TRY(cudaStreamSynchronize(s));
            memcpy(hh.data(), h_scal, (2 * (size_t)k + 1) * sizeof(double));
            double nrm = hh[2 * k], proj = 0.0;
            for (int i = 0; i < 2 * k; ++i) proj += hh[i] * hh[i];
            proj = sqrt(proj);
            const double eta = 1.0 / sqrt(2.0);
            bool changed = false;
            while (nrm < eta * proj) {
                if ((rc = multi_dot(V, ldv, k, w, d_corr, s))) return rc;
                k_multi_axpy_nrm2<<<RED_BLOCKS, RED_THREADS, 0, s>>>(V, ldv, k, d_corr, w, n, d_partials, d_ticket, d_corr + 2 * k, comm ? 0 : 1);
                launches++;
                if ((rc = finish_norm(d_corr + 2 * k, s))) return rc;
                LS_CUDA_TRY(cudaMemcpyAsync(h_scal, d_corr, (2 * (size_t)k + 1) * sizeof(double), cudaMemcpyDeviceToHost, s));
                LS_CUDA_TRY(cudaStreamSynchronize(s));
                memcpy(cc.data(), h_scal, (2 * (size_t)k + 1) * sizeof(double));
                proj = 0.0;
                for (int i = 0; i < 2 * k; ++i) { proj += cc[i] * cc[i]; hh[i] += cc[i]; }
                proj = sqrt(proj);
                nrm = cc[2 * k];
                changed = true;
            }
            if (changed) {
                hh[2 * k] = nrm; hh[2 * k + 1] = 0.0;
                memcpy(h_scal + 144, hh.data(), (2 * (size_t)k + 2) * sizeof(double));     // pinned scratch beyond the live part
                LS_CUDA_TRY(cudaMemcpyAsync(h, h_scal + 144, (2 * (size_t)k + 2) * sizeof(double), cudaMemcpyHostToDevice, s));
            }
        }
        k_scal_inv_dev<<<grid_stream(n), 256, 0, s>>>(h + 2 * k, w, n);
        launches++;
        return LS_OK;
    }
    int orthogonalize(const cd* V, long ldv, int k, cd* w, cudaStream_t s) {
        return (orth_meth == 0 || k == 0) ? mgs(V, ldv, k, w, s) : cgs(V, ldv, k, w, s);
    }
};

int krylov_alloc(Krylov* K, long n) {
    K->n = n;
    int rc;
    if ((rc = K->dmalloc((void**)&K->d_partials, RED_BLOCKS * sizeof(double2)))) return rc;
    if ((rc = K->dmalloc((void**)&K->d_ticket, sizeof(unsigned)))) return rc;
    if ((rc = K->dmalloc((void**)&K->d_scal, 2 * 72 * sizeof(double)))) return rc;
    if ((rc = K->dmalloc((void**)&K->d_corr, 2 * 72 * sizeof(double)))) return rc;
    if ((rc = K->dmalloc((void**)&K->d_partials_multi, (size_t)KC * RED_BLOCKS * sizeof(double2)))) return rc;
    if ((rc = K->dmalloc((void**)&K->d_y, 64 * sizeof(cd)))) return rc;
    LS_CUDA_TRY(cudaMemsetAsync(K->d_ticket, 0, sizeof(unsigned), K->stream));
    LS_CUDA_TRY(cudaMallocHost((void**)&K->h_scal, 4 * 72 * sizeof(double)));
    K->host_allocs.push_back(K->h_scal);
    LS_CUDA_TRY(cudaStreamSynchronize(K->stream));
    return LS_OK;
}

// host-side Givens least squares (hessenberg.jl ldiv!): H is (k+1) x k column-major with ld = ldh
struct cplx { double re, im; };
inline cplx cmulh(cplx a, cplx b) { return {a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re}; }
inline cplx caddh(cplx a, cplx b) { return {a.re + b.re, a.im + b.im}; }
inline cplx csubh(cplx a, cplx b) { return {a.re - b.re, a.im - b.im}; }
inline cplx conjh(cplx a) { return {a.re, -a.im}; }
inline cplx scaleh(cplx a, double s) { return {a.re * s, a.im * s}; }
inline double absh(cplx a) { return hypot(a.re, a.im); }
inline cplx cdivh(cplx a, cplx b) {
    double d = b.re * b.re + b.im * b.im;
    return {(a.re * b.re + a.im * b.im) / d, (a.im * b.re - a.re * b.im) / d};
}

void givens(cplx f, cplx g, double& c, cplx& s) {
    if (g.re == 0.0 && g.im == 0.0) { c = 1.0; s = {0.0, 0.0}; return; }
    if (f.re == 0.0 && f.im == 0.0) { c = 0.0; s = scaleh(conjh(g), 1.0 / absh(g)); return; }
    const double nf = absh(f), d = hypot(nf, absh(g));
    c = nf / d;
    s = scaleh(cmulh(scaleh(f, 1.0 / nf), conjh(g)), 1.0 / d);
}

void solve_least_squares(std::vector<cplx>& H, int ldh, double beta, int k, std::vector<cplx>& y) {
    // k = number of columns; solves min || H[0:k+1, 0:k] y - beta e1 ||
    std::vector<cplx> rhs((size_t)k + 1, cplx{0.0, 0.0});
    rhs[0] = {beta, 0.0};
    for (int i = 0; i < k; ++i) {
        double c; cplx s;
        givens(H[i + (size_t)i * ldh], H[i + 1 + (size_t)i * ldh], c, s);
        H[i + (size_t)i * ldh] = caddh(scaleh(H[i + (size_t)i * ldh], c), cmulh(s, H[i + 1 + (size_t)i * ldh]));
        for (int j = i + 1; j < k; ++j) {
            cplx a = H[i + (size_t)j * ldh], b = H[i + 1 + (size_t)j * ldh];
            H[i + 1 + (size_t)j * ldh] = caddh(cmulh(scaleh(conjh(s), -1.0), a), scaleh(b, c));
            H[i + (size_t)j * ldh] = caddh(scaleh(a, c), cmulh(s, b));
        }
        cplx a = rhs[i], b = rhs[i + 1];
        rhs[i + 1] = caddh(cmulh(scaleh(conjh(s), -1.0), a), scaleh(b, c));
        rhs[i] = caddh(scaleh(a, c), cmulh(s, b));
    }
    y.assign((size_t)k, cplx{0.0, 0.0});
    for (int i = k - 1; i >= 0; --i) {
        cplx acc = rhs[i];
        for (int j = i + 1; j < k; ++j) acc = csubh(acc, cmulh(H[i + (size_t)j * ldh], y[j]));
        y[i] = cdivh(acc, H[i + (size_t)i * ldh]);
    }
}

}  // namespace

extern "C" {

int ls_krylov_create(ls_handle* out, int64_t n) {
    LS_REQUIRE(out && n > 0, LS_ERR_INVALID, "ls_krylov_create: bad argument");
    Krylov* K = new Krylov();
    int rc = K->init_base(KIND_VEC);
    if (rc) { delete K; return rc; }
    rc = krylov_alloc(K, n);
    if (rc) { delete K; return rc; }
    *out = reinterpret_cast<ls_handle>(K);
    return LS_OK;
}

#define KRYLOV_HANDLE(K, h, fn)                                                                \
    LS_REQUIRE(h, LS_ERR_INVALID, fn ": null handle");                                         \
    Krylov* K = reinterpret_cast<Krylov*>(h);                                                  \
    LS_REQUIRE(K->kind == KIND_VEC, LS_ERR_INVALID, fn ": not a Krylov workspace handle");     \
    LS_CUDA_TRY(cudaSetDevice(K->device))

int ls_krylov_set_orth(ls_handle h, int orth_meth) {
    KRYLOV_HANDLE(K, h, "ls_krylov_set_orth");
    LS_REQUIRE(orth_meth >= 0 && orth_meth <= 2, LS_ERR_INVALID,
               "ls_krylov_set_orth: 0 ModifiedGramSchmidt, 1 ClassicalGramSchmidt, 2 DGKS");
    K->orth_meth = orth_meth;
    return LS_OK;
}

int ls_zdotc(ls_handle h, const ls_cdouble* x, const ls_cdouble* y, ls_cdouble* result) {
    KRYLOV_HANDLE(K, h, "ls_zdotc");
    LS_REQUIRE(x && y && result, LS_ERR_INVALID, "ls_zdotc: null pointer");
    { int rc = K->dot((const cd*)x, (const cd*)y, K->d_scal, K->stream); if (rc) return rc; }
    LS_CUDA_TRY(cudaMemcpyAsync(K->h_scal, K->d_scal, 2 * sizeof(double), cudaMemcpyDeviceToHost, K->stream));
    LS_CUDA_TRY(cudaStreamSynchronize(K->stream));
    result->re = K->h_scal[0];
    result->im = K->h_scal[1];
    return LS_OK;
}

int ls_dznrm2(ls_handle h, const ls_cdouble* x, double* result) {
    KRYLOV_HANDLE(K, h, "ls_dznrm2");
    LS_REQUIRE(x && result, LS_ERR_INVALID, "ls_dznrm2: null pointer");
    { int rc = K->nrm2((const cd*)x, K->d_scal, K->stream); if (rc) return rc; }
    LS_CUDA_TRY(cudaMemcpyAsync(K->h_scal, K->d_scal, sizeof(double), cudaMemcpyDeviceToHost, K->stream));
    LS_CUDA_TRY(cudaStreamSynchronize(K->stream));
    *result = K->h_scal[0];
    return LS_OK;
}

int ls_zaxpy(ls_handle h, ls_cdouble alpha, const ls_cdouble* x, ls_cdouble* y) {
    KRYLOV_HANDLE(K, h, "ls_zaxpy");
    LS_REQUIRE(x && y, LS_ERR_INVALID, "ls_zaxpy: null pointer");
    k_axpy<<<K->grid_stream(K->n), 256, 0, K->stream>>>(make_double2(alpha.re, alpha.im), (const cd*)x, (cd*)y, K->n);
    K->launches++;
    LS_CUDA_TRY(cudaGetLastError());
    return LS_OK;
}

int ls_zscal(ls_handle h, ls_cdouble alpha, ls_cdouble* x) {
    KRYLOV_HANDLE(K, h, "ls_zscal");
    LS_REQUIRE(x, LS_ERR_INVALID, "ls_zscal: null pointer");
    k_scal<<<K->grid_stream(K->n), 256, 0, K->stream>>>(make_double2(alpha.re, alpha.im), (cd*)x, K->n);
    K->launches++;
    LS_CUDA_TRY(cudaGetLastError());
    return LS_OK;
}

int ls_mgs_step(ls_handle h, const ls_cdouble* V, int64_t ldv, int k, ls_cdouble* w, ls_cdouble* hcol) {
    KRYLOV_HANDLE(K, h, "ls_mgs_step");
    LS_REQUIRE(V && w && hcol, LS_ERR_INVALID, "ls_mgs_step: null pointer");
    LS_REQUIRE(k >= 0 && k <= 64 && ldv >= K->n, LS_ERR_INVALID, "ls_mgs_step: k must be in [0,64] and ldv >= n");
    { int rc = K->orthogonalize((const cd*)V, ldv, k, (cd*)w, K->stream); if (rc) return rc; }
    LS_CUDA_TRY(cudaGetLastError());
    LS_CUDA_TRY(cudaMemcpyAsync(K->h_scal, K->d_scal, 2 * (size_t)(k + 1) * sizeof(double), cudaMemcpyDeviceToHost, K->stream));
    LS_CUDA_TRY(cudaStreamSynchronize(K->stream));
    memcpy(hcol, K->h_scal, 2 * (size_t)(k + 1) * sizeof(double));
    return LS_OK;
}

// Common driver behind ls_gmres (host callback for Msp^-1) and ls_gmres_msp (device-resident Msp^-1).
static int gmres_driver(Krylov* K, HandleBase* op, SpM* As, MspBase* msp, ls_solve_cb msp_solve, void* user,
                        const ls_cdouble* b, ls_cdouble* x, int restart, int64_t maxiter, double reltol, double abstol,
                        int initially_zero, double* resnorm_hist, int64_t hist_cap, int64_t* niter, int* converged,
                        int64_t* mv_products, int memloc) {
    LS_REQUIRE(op->op_size() == K->n, LS_ERR_INVALID, "ls_gmres: operator size %ld != workspace size %ld",
               (long)op->op_size(), (long)K->n);
    if (As) LS_REQUIRE(As->kind == KIND_SPM && As->nrows == K->n && As->x_len() == K->n, LS_ERR_INVALID,
                       "ls_gmres: As must be an N x N sparse-matrix handle (or the row slab of one, ls_spm_create_dist)");
    if (msp) LS_REQUIRE(msp->kind == KIND_MSP && msp->n == K->n, LS_ERR_INVALID,
                        "ls_gmres_msp: the Msp factorisation has %ld unknowns, the operator %ld", (long)msp->n, (long)K->n);
    const long n = K->n;
    if (restart <= 0) restart = 20;
    LS_REQUIRE(restart <= 64, LS_ERR_UNSUPPORTED, "ls_gmres: restart > 64 is not supported");
    if (maxiter < 0) maxiter = n;      // default; callers with sharded vectors pass the global N.  0 = no iteration.
    // all work is enqueued on the operator's stream so that its apply orders with our kernels
    cudaStream_t s = op->stream;
    // sharded operator: dots / norms are all-reduced on its communicator for the duration of this solve only
    struct CommScope { Krylov* K; ~CommScope() { K->comm = nullptr; } } comm_scope{K};
    K->comm = op->nccl_comm();
    if (K->comm) {
        // Sharded vectors.  As must be the row slab living on the same communicator (its halo exchange is a
        // collective); the Msp solve is not sharded: only a host callback (which may gather / scatter) is accepted.
        LS_REQUIRE(!As || (As->halo > 0 && As->comm == K->comm), LS_ERR_INVALID,
                   "ls_gmres: with a sharded operator As must come from ls_spm_create_dist on the same operator");
        LS_REQUIRE(!msp, LS_ERR_UNSUPPORTED, "ls_gmres_msp: the device Msp factorisation is single-GPU");
    } else if (As) {
        LS_REQUIRE(As->halo == 0, LS_ERR_INVALID, "ls_gmres: a row-slab As needs the sharded operator it was created on");
    }
    const size_t vb = (size_t)n * sizeof(cd);
    if (K->v_cols < restart + 1) {
        if (K->d_V) K->dfree(K->d_V);
        K->d_V = nullptr;
        int rc = K->dmalloc((void**)&K->d_V, vb * (size_t)(restart + 1));
        if (rc) return rc;
        K->v_cols = restart + 1;
    }
    if (!K->d_ax) {
        int rc;
        if ((rc = K->dmalloc((void**)&K->d_ax, vb))) return rc;
        if ((rc = K->dmalloc((void**)&K->d_b, vb))) return rc;
        if ((rc = K->dmalloc((void**)&K->d_x, vb))) return rc;
    }
    if (msp_solve && !K->h_stage) {
        LS_CUDA_TRY(cudaMallocHost((void**)&K->h_stage, vb));
        K->host_allocs.push_back(K->h_stage);
    }
    const cd* db; cd* dx;
    if (memloc == LS_MEM_HOST) {
        LS_CUDA_TRY(cudaMemcpyAsync(K->d_b, b, vb, cudaMemcpyHostToDevice, s));
        LS_CUDA_TRY(cudaMemcpyAsync(K->d_x, x, vb, cudaMemcpyHostToDevice, s));
        db = K->d_b; dx = K->d_x;
    } else {
        LS_REQUIRE(memloc == LS_MEM_DEVICE, LS_ERR_INVALID, "ls_gmres: unknown memloc %d", memloc);
        db = (const cd*)b; dx = (cd*)x;
    }
    cd* V = K->d_V;
    const long ldv = n;
    const int gs = K->grid_stream(n);
    K->t_precond_host_s = 0.0;

    // ldiv!(Pl, v):  v <- Msp^-1 (As v)   (preconditioner.jl:147-166).  As on the GPU; Msp^-1 either on the GPU
    // (msp: the factorisation of ls_msp_factor, no PCIe traffic) or through the host callback.
    auto precond = [&](cd* v) -> int {
        if (!As && !msp_solve && !msp) return LS_OK;
        cd* cur = v;
        if (As) {
            int rc = As->mv_dev(make_double2(1.0, 0.0), v, make_double2(0.0, 0.0), K->d_ax, s);
            if (rc) return rc;
            K->launches++;
            cur = K->d_ax;
        }
        if (msp) {
            int rc = msp->solve_dev(cur, v, s);
            if (rc) return rc;
            K->launches += msp->launches_per_solve;
        } else if (msp_solve) {
            const auto t0 = std::chrono::steady_clock::now();
            LS_CUDA_TRY(cudaMemcpyAsync(K->h_stage, cur, vb, cudaMemcpyDeviceToHost, s));
            LS_CUDA_TRY(cudaStreamSynchronize(s));
            int crc = msp_solve(user, reinterpret_cast<ls_cdouble*>(K->h_stage), n);
            LS_REQUIRE(crc == 0, LS_ERR_CALLBACK, "ls_gmres: the Msp solve callback returned %d", crc);
            LS_CUDA_TRY(cudaMemcpyAsync(v, K->h_stage, vb, cudaMemcpyHostToDevice, s));
            LS_CUDA_TRY(cudaStreamSynchronize(s));
            K->t_precond_host_s += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        } else {
            LS_CUDA_TRY(cudaMemcpyAsync(v, cur, vb, cudaMemcpyDeviceToDevice, s));
        }
        return LS_OK;
    };
    int64_t mv = initially_zero ? 1 : 0;
    // init!: V1 = Pl^-1 (b - A x); beta = ||V1||; V1 /= beta
    auto init = [&](bool first, double& beta) -> int {
        if (first && initially_zero) {
            LS_CUDA_TRY(cudaMemcpyAsync(V, db, vb, cudaMemcpyDeviceToDevice, s));
        } else {
            int rc = op->apply_dev(dx, K->d_ax, LS_APPLY_FASTCONVOLUTION);
            if (rc) return rc;
            k_sub<<<gs, 256, 0, s>>>(db, K->d_ax, V, n);
            K->launches++;
        }
        int rc = precond(V);
        if (rc) return rc;
        rc = K->nrm2(V, K->d_scal, s);
        if (rc) return rc;
        k_scal_inv_dev<<<gs, 256, 0, s>>>(K->d_scal, V, n);
        K->launches++;
        LS_CUDA_TRY(cudaMemcpyAsync(K->h_scal, K->d_scal, sizeof(double), cudaMemcpyDeviceToHost, s));
        LS_CUDA_TRY(cudaStreamSynchronize(s));
        beta = K->h_scal[0];
        return LS_OK;
    };

    const int ldh = restart + 1;
    std::vector<cplx> H((size_t)ldh * restart, cplx{0.0, 0.0});
    std::vector<cplx> nullvec((size_t)restart + 1, cplx{1.0, 0.0});
    double beta = 0.0;
    int rc = init(true, beta);
    if (rc) return rc;
    double current = beta, accumulator = 1.0, rbeta = beta;
    const double tol = fmax(reltol * current, abstol);
    int k = 1;
    int64_t iteration = 0, nh = 0;
    // IterativeSolvers gmres.jl: converged(g) = residual <= tol; done(g, it) = it >= maxiter || converged(g)
    auto is_converged = [&]() { return current <= tol; };
    std::vector<cplx> y;
    while (!(iteration >= maxiter || is_converged())) {
        // expand!: V_{k+1} = Pl^-1 (A V_k)
        cd* w = V + (long)k * ldv;
        rc = op->apply_dev(V + (long)(k - 1) * ldv, w, LS_APPLY_FASTCONVOLUTION);
        if (rc) return rc;
        rc = precond(w);
        if (rc) return rc;
        mv++;
        // orthogonalize_and_normalize! (modified Gram-Schmidt), Hessenberg column -> host
        rc = K->orthogonalize(V, ldv, k, w, s);
        if (rc) return rc;
        LS_CUDA_TRY(cudaMemcpyAsync(K->h_scal, K->d_scal, 2 * (size_t)(k + 1) * sizeof(double), cudaMemcpyDeviceToHost, s));
        LS_CUDA_TRY(cudaStreamSynchronize(s));
        for (int i = 0; i <= k; ++i) H[i + (size_t)(k - 1) * ldh] = {K->h_scal[2 * i], K->h_scal[2 * i + 1]};
        // update_residual!
        cplx acc = {0.0, 0.0};
        for (int i = 0; i < k; ++i) acc = caddh(acc, cmulh(conjh(nullvec[i]), H[i + (size_t)(k - 1) * ldh]));
        cplx q = cdivh(acc, H[k + (size_t)(k - 1) * ldh]);
        nullvec[k] = {-q.re, q.im};     // -conj(q)
        accumulator += nullvec[k].re * nullvec[k].re + nullvec[k].im * nullvec[k].im;
        current = rbeta / sqrt(accumulator);
        k++;
        // gmres.jl iterate(): x is formed at a restart or at convergence only - when maxiter lands inside a cycle the
        // caller gets the x of the last restart, exactly as upstream - and the cycle restarts whenever not converged.
        if (k == restart + 1 || is_converged()) {
            std::vector<cplx> Hc(H);
            solve_least_squares(Hc, ldh, beta, k - 1, y);
            LS_CUDA_TRY(cudaMemcpyAsync(K->d_y, y.data(), (size_t)(k - 1) * sizeof(cd), cudaMemcpyHostToDevice, s));
            k_update_solution<<<gs, 256, 0, s>>>(V, ldv, k - 1, K->d_y, dx, n);
            K->launches++;
            LS_CUDA_TRY(cudaStreamSynchronize(s));   // y (host vector) must outlive the H2D copy
            k = 1;
            if (!is_converged()) {
                rc = init(false, beta);
                if (rc) return rc;
                accumulator = 1.0;
                rbeta = beta;
                mv++;
            }
        }
        iteration++;
        if (resnorm_hist && nh < hist_cap) resnorm_hist[nh++] = current;
    }
    LS_CUDA_TRY(cudaGetLastError());
    if (memloc == LS_MEM_HOST) LS_CUDA_TRY(cudaMemcpyAsync(x, dx, vb, cudaMemcpyDeviceToHost, s));
    LS_CUDA_TRY(cudaStreamSynchronize(s));
    if (niter) *niter = iteration;
    if (converged) *converged = current <= tol ? 1 : 0;
    if (mv_products) *mv_products = mv;
    return LS_OK;
}

// ls_gmres_msp_batch / ls_gmres_batch: nrhs independent GMRES(restart) runs of gmres_driver side by side with one
// operator and, with msp, one As and Msp (msp == nullptr: Pl = Identity, no As).  Every system keeps its own basis,
// Hessenberg matrix, restarts, tolerance and history, and goes through exactly the steps gmres_driver takes for it (same
// kernels, same inputs), so its history, counts and x have the bits of a run on its own.  In each lockstep iteration the
// operator applies of all active systems go through the multi-column apply (chunks of batch_cols columns at the
// systems' basis columns), the SpMVs and Gram-Schmidt steps run system by system, and the Msp^-1 of all active systems
// is one batched solve (ls_msp_solve_batch: each factor block is read once per chunk of columns).  All active systems
// share the iteration count and the position k in the restart cycle; a system that converges or reaches maxiter drops
// out of the later applies and solves.
static int gmres_batch_driver(Krylov* K, HandleBase* op, SpM* As, MspBase* msp, int nrhs, const ls_cdouble* b, int64_t ldb,
                              ls_cdouble* x, int64_t ldx, int restart, int64_t maxiter, double reltol, double abstol,
                              int initially_zero, double* resnorm_hist, int64_t hist_cap, int64_t* niter, int* converged,
                              int64_t* mv_products, int memloc) {
    const char* fn = msp ? "ls_gmres_msp_batch" : "ls_gmres_batch";
    LS_REQUIRE(op->op_size() == K->n, LS_ERR_INVALID, "%s: operator size %ld != workspace size %ld", fn, (long)op->op_size(), (long)K->n);
    LS_REQUIRE(op->nccl_comm() == nullptr, LS_ERR_UNSUPPORTED, "%s: several right-hand sides are served on one GPU", fn);
    if (As) LS_REQUIRE(As->kind == KIND_SPM && As->nrows == K->n && As->x_len() == K->n && As->halo == 0, LS_ERR_INVALID,
                       "%s: As must be an N x N sparse-matrix handle", fn);
    if (msp) LS_REQUIRE(msp->kind == KIND_MSP && msp->n == K->n, LS_ERR_INVALID, "%s: the Msp factorisation has %ld unknowns, the operator %ld",
                        fn, (long)msp->n, (long)K->n);
    const long n = K->n;
    if (restart <= 0) restart = 20;
    LS_REQUIRE(restart <= 64, LS_ERR_UNSUPPORTED, "%s: restart > 64 is not supported", fn);
    if (maxiter < 0) maxiter = n;
    cudaStream_t s = op->stream;
    const size_t vb = (size_t)n * sizeof(cd);
    const bool host = memloc == LS_MEM_HOST;

    // memory: nrhs bases of restart + 1 columns, nrhs columns for the batched solve, host staging of b and x, the
    // batched solve's and the multi-column apply's work arrays - checked against the free device memory before anything
    // is allocated
    const int wcols = std::min(nrhs, op->batch_cols());
    const size_t needV = vb * (size_t)(restart + 1) * nrhs, needP = msp ? vb * nrhs : 0, needBX = host ? 2 * vb * nrhs : 0;
    size_t need = (K->Vb_bytes < needV ? needV : 0) + (K->Pb_bytes < needP ? needP : 0) + (K->bxb_bytes < needBX ? needBX : 0) +
                  (K->d_ax ? 0 : 3 * vb) + (msp ? msp->batch_bytes(nrhs, false, true) : 0) + op->batch_bytes(wcols);
    if (need > 0) {
        size_t free_b = 0, total_b = 0;
        LS_CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
        LS_REQUIRE(need <= free_b, LS_ERR_NOMEM,
                   "%s: %d systems of %ld unknowns with restart %d need %zu more bytes of device memory; %zu of %zu bytes are free",
                   fn, nrhs, n, restart, need, free_b, total_b);
    }
    int rc;
    if ((rc = K->ensure(&K->d_Vb, K->Vb_bytes, needV))) return rc;
    if (msp && (rc = K->ensure(&K->d_Pb, K->Pb_bytes, needP))) return rc;
    if (host && (rc = K->ensure(&K->d_bxb, K->bxb_bytes, needBX))) return rc;
    if (!K->d_ax) {
        if ((rc = K->dmalloc((void**)&K->d_ax, vb))) return rc;
        if ((rc = K->dmalloc((void**)&K->d_b, vb))) return rc;
        if ((rc = K->dmalloc((void**)&K->d_x, vb))) return rc;
    }
    if (msp && (rc = msp->batch_reserve(nrhs, false, true))) return rc;
    if ((rc = op->batch_reserve(wcols))) return rc;

    struct Sys {
        cd* V; const cd* db; cd* dx;
        std::vector<cplx> H, nullvec;
        double beta = 0.0, current = 0.0, accumulator = 1.0, rbeta = 0.0, tol = 0.0;
        int k = 1;
        int64_t iteration = 0, nh = 0, mv = 0;
        bool active = true;
    };
    const int ldh = restart + 1;
    std::vector<Sys> sys((size_t)nrhs);
    for (int q = 0; q < nrhs; ++q) {
        Sys& S = sys[q];
        S.V = K->d_Vb + (size_t)q * (restart + 1) * n;
        if (host) {
            cd* db = K->d_bxb + (size_t)q * n;
            S.dx = K->d_bxb + (size_t)(nrhs + q) * n;
            LS_CUDA_TRY(cudaMemcpyAsync(db, b + (size_t)q * ldb, vb, cudaMemcpyHostToDevice, s));
            LS_CUDA_TRY(cudaMemcpyAsync(S.dx, x + (size_t)q * ldx, vb, cudaMemcpyHostToDevice, s));
            S.db = db;
        } else {
            S.db = reinterpret_cast<const cd*>(b) + (size_t)q * ldb;
            S.dx = reinterpret_cast<cd*>(x) + (size_t)q * ldx;
        }
        S.H.assign((size_t)ldh * restart, cplx{0.0, 0.0});
        S.nullvec.assign((size_t)restart + 1, cplx{1.0, 0.0});
        S.mv = initially_zero ? 1 : 0;
    }
    const int gs = K->grid_stream(n);

    // ldiv!(Pl, v) for the listed vectors: As v into the solve's columns, one batched Msp^-1 in place, back into v
    auto precond = [&](const std::vector<cd*>& vs) -> int {
        const int na = (int)vs.size();
        if (na == 0 || !msp) return LS_OK;
        for (int i = 0; i < na; ++i) {
            cd* col = K->d_Pb + (size_t)i * n;
            if (As) {
                int r = As->mv_dev(make_double2(1.0, 0.0), vs[i], make_double2(0.0, 0.0), col, s);
                if (r) return r;
                K->launches++;
            } else {
                LS_CUDA_TRY(cudaMemcpyAsync(col, vs[i], vb, cudaMemcpyDeviceToDevice, s));
            }
        }
        int r = msp->solve_batch_dev(K->d_Pb, n, K->d_Pb, n, na, s);
        if (r) return r;
        K->launches += (int64_t)msp->launches_per_solve * na;
        for (int i = 0; i < na; ++i) LS_CUDA_TRY(cudaMemcpyAsync(vs[i], K->d_Pb + (size_t)i * n, vb, cudaMemcpyDeviceToDevice, s));
        return LS_OK;
    };
    // init! of the listed systems: V1 = Pl^-1 (b - A x); beta = ||V1||; V1 /= beta
    auto init = [&](const std::vector<int>& which, bool first) -> int {
        std::vector<cd*> vs;
        for (int q : which) {
            Sys& S = sys[q];
            if (first && initially_zero) {
                LS_CUDA_TRY(cudaMemcpyAsync(S.V, S.db, vb, cudaMemcpyDeviceToDevice, s));
            } else {
                int r = op->apply_dev(S.dx, K->d_ax, LS_APPLY_FASTCONVOLUTION);
                if (r) return r;
                k_sub<<<gs, 256, 0, s>>>(S.db, K->d_ax, S.V, n);
                K->launches++;
            }
            vs.push_back(S.V);
        }
        int r = precond(vs);
        if (r) return r;
        for (int q : which) {
            Sys& S = sys[q];
            if ((r = K->nrm2(S.V, K->d_scal, s))) return r;
            k_scal_inv_dev<<<gs, 256, 0, s>>>(K->d_scal, S.V, n);
            K->launches++;
            LS_CUDA_TRY(cudaMemcpyAsync(K->h_scal, K->d_scal, sizeof(double), cudaMemcpyDeviceToHost, s));
            LS_CUDA_TRY(cudaStreamSynchronize(s));
            S.beta = K->h_scal[0];
        }
        return LS_OK;
    };

    std::vector<int> all((size_t)nrhs);
    for (int q = 0; q < nrhs; ++q) all[q] = q;
    if ((rc = init(all, true))) return rc;
    for (Sys& S : sys) {
        S.current = S.beta; S.accumulator = 1.0; S.rbeta = S.beta;
        S.tol = fmax(reltol * S.current, abstol);
        S.active = !(S.iteration >= maxiter || S.current <= S.tol);
    }
    std::vector<cplx> y;
    for (;;) {
        std::vector<int> act;
        for (int q = 0; q < nrhs; ++q) if (sys[q].active) act.push_back(q);
        if (act.empty()) break;
        // expand!: V_{k+1} = Pl^-1 (A V_k) for every active system
        std::vector<const cd*> vk;
        std::vector<cd*> ws;
        for (int q : act) {
            Sys& S = sys[q];
            vk.push_back(S.V + (long)(S.k - 1) * n);
            ws.push_back(S.V + (long)S.k * n);
        }
        if ((rc = op->apply_list_dev(vk.data(), ws.data(), (int)act.size(), LS_APPLY_FASTCONVOLUTION))) return rc;
        if ((rc = precond(ws))) return rc;
        std::vector<int> restarting;
        for (size_t i = 0; i < act.size(); ++i) {
            Sys& S = sys[act[i]];
            const int k = S.k;
            S.mv++;
            if ((rc = K->orthogonalize(S.V, n, k, ws[i], s))) return rc;
            LS_CUDA_TRY(cudaMemcpyAsync(K->h_scal, K->d_scal, 2 * (size_t)(k + 1) * sizeof(double), cudaMemcpyDeviceToHost, s));
            LS_CUDA_TRY(cudaStreamSynchronize(s));
            for (int r = 0; r <= k; ++r) S.H[r + (size_t)(k - 1) * ldh] = {K->h_scal[2 * r], K->h_scal[2 * r + 1]};
            cplx acc = {0.0, 0.0};
            for (int r = 0; r < k; ++r) acc = caddh(acc, cmulh(conjh(S.nullvec[r]), S.H[r + (size_t)(k - 1) * ldh]));
            const cplx qv = cdivh(acc, S.H[k + (size_t)(k - 1) * ldh]);
            S.nullvec[k] = {-qv.re, qv.im};
            S.accumulator += S.nullvec[k].re * S.nullvec[k].re + S.nullvec[k].im * S.nullvec[k].im;
            S.current = S.rbeta / sqrt(S.accumulator);
            S.k++;
            const bool conv = S.current <= S.tol;
            if (S.k == restart + 1 || conv) {
                std::vector<cplx> Hc(S.H);
                solve_least_squares(Hc, ldh, S.beta, S.k - 1, y);
                LS_CUDA_TRY(cudaMemcpyAsync(K->d_y, y.data(), (size_t)(S.k - 1) * sizeof(cd), cudaMemcpyHostToDevice, s));
                k_update_solution<<<gs, 256, 0, s>>>(S.V, n, S.k - 1, K->d_y, S.dx, n);
                K->launches++;
                LS_CUDA_TRY(cudaStreamSynchronize(s));
                S.k = 1;
                if (!conv) restarting.push_back(act[i]);
            }
            S.iteration++;
            if (resnorm_hist && S.nh < hist_cap) resnorm_hist[(size_t)act[i] * hist_cap + S.nh++] = S.current;
        }
        // restart of the unconverged systems at the end of a cycle (init does not change `current`: the history entry
        // above is the one gmres_driver logs after its init)
        if (!restarting.empty()) {
            if ((rc = init(restarting, false))) return rc;
            for (int q : restarting) { Sys& S = sys[q]; S.accumulator = 1.0; S.rbeta = S.beta; S.mv++; }
        }
        for (int q : act) { Sys& S = sys[q]; S.active = !(S.iteration >= maxiter || S.current <= S.tol); }
    }
    LS_CUDA_TRY(cudaGetLastError());
    if (host)
        for (int q = 0; q < nrhs; ++q)
            LS_CUDA_TRY(cudaMemcpyAsync(x + (size_t)q * ldx, sys[q].dx, vb, cudaMemcpyDeviceToHost, s));
    LS_CUDA_TRY(cudaStreamSynchronize(s));
    for (int q = 0; q < nrhs; ++q) {
        if (niter) niter[q] = sys[q].iteration;
        if (converged) converged[q] = sys[q].current <= sys[q].tol ? 1 : 0;
        if (mv_products) mv_products[q] = sys[q].mv;
    }
    return LS_OK;
}

int ls_gmres(ls_handle kh, ls_handle op_h, ls_handle as_h, ls_solve_cb msp_solve, void* user,
             const ls_cdouble* b, ls_cdouble* x, int restart, int64_t maxiter, double reltol, double abstol,
             int initially_zero, double* resnorm_hist, int64_t hist_cap, int64_t* niter, int* converged,
             int64_t* mv_products, int memloc) {
    KRYLOV_HANDLE(K, kh, "ls_gmres");
    LS_REQUIRE(op_h && b && x, LS_ERR_INVALID, "ls_gmres: null argument");
    return gmres_driver(K, reinterpret_cast<HandleBase*>(op_h), reinterpret_cast<SpM*>(as_h), nullptr, msp_solve, user, b, x,
                        restart, maxiter, reltol, abstol, initially_zero, resnorm_hist, hist_cap, niter, converged,
                        mv_products, memloc);
}

int ls_gmres_msp(ls_handle kh, ls_handle op_h, ls_handle as_h, ls_handle msp_h,
                 const ls_cdouble* b, ls_cdouble* x, int restart, int64_t maxiter, double reltol, double abstol,
                 int initially_zero, double* resnorm_hist, int64_t hist_cap, int64_t* niter, int* converged,
                 int64_t* mv_products, int memloc) {
    KRYLOV_HANDLE(K, kh, "ls_gmres_msp");
    LS_REQUIRE(op_h && msp_h && b && x, LS_ERR_INVALID, "ls_gmres_msp: null argument");
    return gmres_driver(K, reinterpret_cast<HandleBase*>(op_h), reinterpret_cast<SpM*>(as_h), reinterpret_cast<MspBase*>(msp_h),
                        nullptr, nullptr, b, x, restart, maxiter, reltol, abstol, initially_zero, resnorm_hist, hist_cap,
                        niter, converged, mv_products, memloc);
}

// Argument refusals come before any CUDA call.
int ls_gmres_msp_batch(ls_handle kh, ls_handle op_h, ls_handle as_h, ls_handle msp_h, int nrhs, const ls_cdouble* b, int64_t ldb,
                       ls_cdouble* x, int64_t ldx, int restart, int64_t maxiter, double reltol, double abstol, int initially_zero,
                       double* resnorm_hist, int64_t hist_cap, int64_t* niter, int* converged, int64_t* mv_products, int memloc) {
    LS_REQUIRE(nrhs >= 1, LS_ERR_INVALID, "ls_gmres_msp_batch: nrhs = %d, at least one system needed", nrhs);
    LS_REQUIRE(kh && op_h && msp_h && b && x, LS_ERR_INVALID, "ls_gmres_msp_batch: null argument");
    LS_REQUIRE(!resnorm_hist || hist_cap >= 0, LS_ERR_INVALID, "ls_gmres_msp_batch: hist_cap = %ld", (long)hist_cap);
    Krylov* K = reinterpret_cast<Krylov*>(kh);
    LS_REQUIRE(K->kind == KIND_VEC, LS_ERR_INVALID, "ls_gmres_msp_batch: not a Krylov workspace handle");
    LS_REQUIRE(ldb >= K->n && ldx >= K->n, LS_ERR_INVALID, "ls_gmres_msp_batch: leading dimensions ldb = %ld, ldx = %ld must be >= N = %ld",
               (long)ldb, (long)ldx, (long)K->n);
    LS_REQUIRE(memloc == LS_MEM_HOST || memloc == LS_MEM_DEVICE, LS_ERR_INVALID, "ls_gmres_msp_batch: unknown memloc %d", memloc);
    LS_CUDA_TRY(cudaSetDevice(K->device));
    return gmres_batch_driver(K, reinterpret_cast<HandleBase*>(op_h), reinterpret_cast<SpM*>(as_h), reinterpret_cast<MspBase*>(msp_h),
                              nrhs, b, ldb, x, ldx, restart, maxiter, reltol, abstol, initially_zero, resnorm_hist, hist_cap, niter,
                              converged, mv_products, memloc);
}

// Argument refusals come before any CUDA call.
int ls_gmres_batch(ls_handle kh, ls_handle op_h, int nrhs, const ls_cdouble* b, int64_t ldb, ls_cdouble* x, int64_t ldx, int restart,
                   int64_t maxiter, double reltol, double abstol, int initially_zero, double* resnorm_hist, int64_t hist_cap,
                   int64_t* niter, int* converged, int64_t* mv_products, int memloc) {
    LS_REQUIRE(nrhs >= 1, LS_ERR_INVALID, "ls_gmres_batch: nrhs = %d, at least one system needed", nrhs);
    LS_REQUIRE(kh && op_h && b && x, LS_ERR_INVALID, "ls_gmres_batch: null argument");
    LS_REQUIRE(!resnorm_hist || hist_cap >= 0, LS_ERR_INVALID, "ls_gmres_batch: hist_cap = %ld", (long)hist_cap);
    Krylov* K = reinterpret_cast<Krylov*>(kh);
    LS_REQUIRE(K->kind == KIND_VEC, LS_ERR_INVALID, "ls_gmres_batch: not a Krylov workspace handle");
    LS_REQUIRE(ldb >= K->n && ldx >= K->n, LS_ERR_INVALID, "ls_gmres_batch: leading dimensions ldb = %ld, ldx = %ld must be >= N = %ld",
               (long)ldb, (long)ldx, (long)K->n);
    LS_REQUIRE(memloc == LS_MEM_HOST || memloc == LS_MEM_DEVICE, LS_ERR_INVALID, "ls_gmres_batch: unknown memloc %d", memloc);
    HandleBase* op = reinterpret_cast<HandleBase*>(op_h);
    LS_REQUIRE(op->kind == KIND_OP2D || op->kind == KIND_OP3D, LS_ERR_INVALID, "ls_gmres_batch: not an operator handle");
    LS_REQUIRE(op->dist_size() == 1, LS_ERR_UNSUPPORTED, "ls_gmres_batch: several right-hand sides are served on one GPU");
    LS_CUDA_TRY(cudaSetDevice(K->device));
    return gmres_batch_driver(K, op, nullptr, nullptr, nrhs, b, ldb, x, ldx, restart, maxiter, reltol, abstol, initially_zero,
                              resnorm_hist, hist_cap, niter, converged, mv_products, memloc);
}

// ---- sparsifier sampling on the device (SURVEY.md 8(f) row 2) --------------------------------------------------------
// sampleGConv (FastConvolution.jl:278-306) / sampleG3D (FastConvolution3D.jl:136-160): row i of the discrete Green's
// operator = FFTconvolution(fastconv, e_{indS[i]}).  The rows stay on the device (column i of V), so the far-field
// Gram matrix of entriesSparseAConv (SparsifyingMatrix2D.jl:104-201: svd of the s x N block) is a handful of fused
// multi-dot sweeps and only s^2 numbers reach the host.
namespace {
__global__ void k_set_unit(cd* e, long idx_prev, long idx) {
    if (idx_prev >= 0) e[idx_prev] = make_double2(0.0, 0.0);
    e[idx] = make_double2(1.0, 0.0);
}
__global__ void k_gather_rows(const cd* __restrict__ V, long ldv, int s, const long* __restrict__ idx, int nidx, cd* out) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < s * nidx) out[e] = V[idx[e % nidx] + (long)(e / nidx) * ldv];
}
}  // namespace

int ls_sample_rows(ls_handle kh, ls_handle op_h, const int64_t* indS, int s, ls_cdouble* V_dev, int64_t ldv) {
    KRYLOV_HANDLE(K, kh, "ls_sample_rows");
    LS_REQUIRE(op_h && indS && V_dev && s > 0, LS_ERR_INVALID, "ls_sample_rows: bad argument");
    HandleBase* op = reinterpret_cast<HandleBase*>(op_h);
    LS_REQUIRE(op->op_size() == K->n && ldv >= K->n, LS_ERR_INVALID, "ls_sample_rows: operator size %ld, workspace %ld, ldv %ld",
               (long)op->op_size(), (long)K->n, (long)ldv);
    LS_REQUIRE(op->nccl_comm() == nullptr, LS_ERR_UNSUPPORTED, "ls_sample_rows: single-GPU operators only");
    const size_t vb = (size_t)K->n * sizeof(cd);
    if (!K->d_ax) {
        int rc;
        if ((rc = K->dmalloc((void**)&K->d_ax, vb))) return rc;
        if ((rc = K->dmalloc((void**)&K->d_b, vb))) return rc;
        if ((rc = K->dmalloc((void**)&K->d_x, vb))) return rc;
    }
    cudaStream_t st = op->stream;
    LS_CUDA_TRY(cudaMemsetAsync(K->d_b, 0, vb, st));
    long prev = -1;
    for (int i = 0; i < s; ++i) {
        LS_REQUIRE(indS[i] >= 1 && indS[i] <= K->n, LS_ERR_INVALID, "ls_sample_rows: stencil index %ld outside the grid", (long)indS[i]);
        k_set_unit<<<1, 1, 0, st>>>(K->d_b, prev, indS[i] - 1);
        prev = indS[i] - 1;
        int rc = op->apply_dev(K->d_b, reinterpret_cast<cd*>(V_dev) + (long)i * ldv, LS_APPLY_FFTCONVOLUTION);
        if (rc) return rc;
        K->launches++;
    }
    LS_CUDA_TRY(cudaStreamSynchronize(st));
    return LS_OK;
}

// gram[i + s*j] = sum_c conj(V[c, i]) V[c, j]   (host, column-major s x s); V: device, N x s, leading dimension ldv
int ls_gram(ls_handle kh, const ls_cdouble* V_dev, int64_t ldv, int s, ls_cdouble* gram_host) {
    KRYLOV_HANDLE(K, kh, "ls_gram");
    LS_REQUIRE(V_dev && gram_host && s > 0 && s <= 64 && ldv >= K->n, LS_ERR_INVALID, "ls_gram: bad argument (s in [1, 64], ldv >= n)");
    const cd* V = reinterpret_cast<const cd*>(V_dev);
    for (int j = 0; j < s; ++j) {
        int rc = K->multi_dot(V, ldv, s, V + (long)j * ldv, K->d_scal, K->stream);
        if (rc) return rc;
        LS_CUDA_TRY(cudaMemcpyAsync(K->h_scal, K->d_scal, 2 * (size_t)s * sizeof(double), cudaMemcpyDeviceToHost, K->stream));
        LS_CUDA_TRY(cudaStreamSynchronize(K->stream));
        memcpy(gram_host + (size_t)j * s, K->h_scal, 2 * (size_t)s * sizeof(double));
    }
    return LS_OK;
}

// out[j + nidx*i] = V[idx[j] - 1, i]  (idx 1-based, host; out host): the s x s near-field blocks of the sampled rows
int ls_gather_rows(ls_handle kh, const ls_cdouble* V_dev, int64_t ldv, int s, const int64_t* idx, int nidx, ls_cdouble* out_host) {
    KRYLOV_HANDLE(K, kh, "ls_gather_rows");
    LS_REQUIRE(V_dev && idx && out_host && s > 0 && nidx > 0, LS_ERR_INVALID, "ls_gather_rows: bad argument");
    std::vector<long> h((size_t)nidx);
    for (int j = 0; j < nidx; ++j) {
        LS_REQUIRE(idx[j] >= 1 && idx[j] <= K->n, LS_ERR_INVALID, "ls_gather_rows: index %ld outside the grid", (long)idx[j]);
        h[(size_t)j] = idx[j] - 1;
    }
    long* d_idx = nullptr; cd* d_out = nullptr;
    int rc;
    if ((rc = K->dupload((void**)&d_idx, h.data(), h.size() * sizeof(long)))) return rc;
    if ((rc = K->dmalloc((void**)&d_out, (size_t)s * nidx * sizeof(cd)))) return rc;
    k_gather_rows<<<(s * nidx + 127) / 128, 128, 0, K->stream>>>(reinterpret_cast<const cd*>(V_dev), ldv, s, d_idx, nidx, d_out);
    LS_CUDA_TRY(cudaMemcpyAsync(out_host, d_out, (size_t)s * nidx * sizeof(cd), cudaMemcpyDeviceToHost, K->stream));
    LS_CUDA_TRY(cudaStreamSynchronize(K->stream));
    K->dfree(d_idx); K->dfree(d_out);
    return LS_OK;
}

int ls_krylov_last_precond_host_seconds(ls_handle kh, double* seconds) {
    KRYLOV_HANDLE(K, kh, "ls_krylov_last_precond_host_seconds");
    LS_REQUIRE(seconds, LS_ERR_INVALID, "ls_krylov_last_precond_host_seconds: null pointer");
    *seconds = K->t_precond_host_s;
    return LS_OK;
}

}  // extern "C"
