/* libls_cuda.so - C ABI of the B200-native Lippmann-Schwinger hot path.
 *
 * The reference (tanderson92/Fast_solver_Lippmann_Schwinger, pure Julia) has no FFI for
 * this path; its boundary is Julia multiple dispatch on the operator objects.  Each entry
 * point below names the reference method it stands behind (file:line under the reference's
 * src/), and INTEGRATION.md shows the `ccall` stubs a maintainer adds on the Julia side
 * (julia/LSCuda.jl).  The only ccall precedent upstream is sparseblas.jl:14-25
 * (mkl_zcscmv_: y <- alpha*A*x + beta*y on CSC arrays), which ls_spm_mv mirrors.
 *
 * Conventions: complex128 = two doubles (re, im); arrays are Julia column-major, x fastest;
 * sparse matrices arrive as Julia SparseMatrixCSC{ComplexF64,Int64} (1-based colptr /
 * rowval).  Every function returns 0 (LS_OK) or a negative error code; ls_last_error()
 * returns a thread-local message.  No C++ exception and no torch type crosses this ABI.
 * Handles are opaque, not thread-safe, own their CUDA stream(s) and are freed by
 * ls_destroy.  `memloc` tells whether data pointers are host or device memory.  Calls with
 * host pointers are synchronous; calls with device pointers are enqueued on the handle's
 * stream (ls_sync waits for it).  There is no CPU fallback anywhere in this library.
 */
#ifndef LS_CUDA_H
#define LS_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct { double re, im; } ls_cdouble;
typedef struct ls_handle_s* ls_handle;

#define LS_OK               0
#define LS_ERR_INVALID     -1   /* bad argument / shape mismatch (reference would throw DimensionMismatch) */
#define LS_ERR_UNSUPPORTED -2   /* valid for the reference, not (yet) served by the GPU path */
#define LS_ERR_CUDA        -3
#define LS_ERR_NOMEM       -4
#define LS_ERR_NCCL        -5
#define LS_ERR_CALLBACK    -6

/* create flags */
#define LS_FLAG_FORCE_GENERIC 1   /* take the general-size (Bluestein) path even for power-of-two grids (tests) */
#define LS_FLAG_PAD4          2   /* evaluate with the reference's literal 4x zero padding; default: the handle restricts
                                     the kernel to the lags the cropped apply touches and runs with 2x padding (same
                                     operator to rounding, see csrc/op2d.cu) */
#define LS_FLAG_EMBED         4   /* 2-D, any n, m <= 4096, both quadratures: the lags the apply touches are extracted once
                                     and the apply runs on the power-of-two kernels of n' = max(64, nextpow2(n)) (and m')
                                     with the grid zero-embedded (csrc/op2d_embed.cu).  With LS_FLAG_PAD4 ->
                                     LS_ERR_UNSUPPORTED, with LS_FLAG_FORCE_GENERIC -> LS_ERR_INVALID.
                                     3-D (ls_op3d_create, ls_op3d_create_dist), any n = m, l <= 512: the apply runs on
                                     the kernels of n' = m' = max(64, nextpow2(n)), l' = max(64, nextpow2(l))
                                     (csrc/op3d_embed.cu), sharded too when l is divisible by the rank count.  The same
                                     two refusals; n or l > 512 -> LS_ERR_UNSUPPORTED */

#define LS_MEM_HOST   0
#define LS_MEM_DEVICE 1

/* FastM.quadRule, FastConvolution.jl:22-26 */
#define LS_QUAD_TRAPEZOIDAL    0
#define LS_QUAD_GREENGARD_VICO 1

/* which reference method an apply reproduces */
#define LS_APPLY_FASTCONVOLUTION 0   /* fastconvolution(M,b) = M*b, FastConvolution.jl:58-107; FastM3D `*`, FastConvolution3D.jl:31-37 */
#define LS_APPLY_FFTCONVOLUTION  1   /* FFTconvolution(M,b), FastConvolution.jl:110-154; FastConvolution3D.jl:39-63 */

/* ---- library ------------------------------------------------------------------------ */
int         ls_version(void);
const char* ls_last_error(void);
int         ls_device_count(int* count);
int         ls_set_device(int device);          /* one process per GPU: call with LOCAL_RANK first */

/* ---- raw device buffers (for callers that keep Krylov vectors resident) --------------- */
int ls_dev_alloc(void** dptr, size_t bytes);
int ls_dev_free(void* dptr);
int ls_memcpy_h2d(void* dst_dev, const void* src_host, size_t bytes);
int ls_memcpy_d2h(void* dst_host, const void* src_dev, size_t bytes);
int ls_host_alloc_pinned(void** hptr, size_t bytes);
int ls_host_free_pinned(void* hptr);

/* ---- 2-D operator: struct FastM, FastConvolution.jl:11-27 ----------------------------- *
 * create copies nu (n*m doubles) and GFFT (ne*me complex, column-major, the reference's
 * centred ordering for Greengard_Vico - the fftshift/ifftshift pair of FastConvolution.jl:94,98
 * is folded into a one-time permutation) to the device.  Nothing of the caller's memory is
 * kept.  Fast path: Greengard_Vico with ne = 4n, me = 4m and n, m in {64,...,4096} powers of
 * two (pruned radix-8/16 transforms).  Every other case the reference accepts - any n, m
 * (examples/example.jl ships n = 201, ne = 804) and the trapezoidal rule (ne = 2n-1, crop
 * [n:2n-1], FastConvolution.jl:64-83) - runs on the general path: arbitrary-length line DFTs
 * by Bluestein's algorithm on the same engine, as long as ne + n - 1 <= 4096 (Greengard_Vico
 * n <= 819, trapezoidal n <= 1366); larger sizes are refused (LS_ERR_UNSUPPORTED).  With
 * LS_FLAG_EMBED every such grid up to n, m <= 4096 (h = 1/1000: n = 1001) runs instead on the
 * power-of-two kernels of n' = max(64, nextpow2(n)), zero-embedded.                        */
int ls_op2d_create(ls_handle* out, int64_t n, int64_t m, int64_t ne, int64_t me,
                   const double* nu, const ls_cdouble* gfft, double omega,
                   int quadrule, int flags);
/* The same operator with the Greengard_Vico spectrum GFFT = Gtruncated2D(L, k, S) (Functions.jl:40-42) on the grid
 * S = (2 pi/Lp) |(-2n:2n-1, -2m:2m-1)| of buildFastConvolution (FastConvolution.jl:185-231; there L = 1.5 (x[end]-x[1]+h),
 * Lp = 4 (x[end]-x[1]+h)) evaluated on the device straight into the kernel layout: no host Bessel evaluation and no
 * 16*ne*me-byte upload (4.3 GB at n = 4096).  omega = k.  Power-of-two fast path and the general-size path alike.   */
int ls_op2d_create_gv(ls_handle* out, int64_t n, int64_t m, const double* nu, double omega, double L, double Lp, int flags);
/* y = M*b (mode 0; `*` FastConvolution.jl:43-48, mul! :50-54) or FFTconvolution(M,b) (mode 1).
 * b and y hold n*m complex values and may alias.                                          */
int ls_op2d_apply(ls_handle h, const ls_cdouble* b, ls_cdouble* y, int mode, int memloc);
/* how the handle evaluates: route (0 power-of-two fast path, 1 Bluestein general path, 2 zero-embedded), the line
 * lengths its kernels run (n, m; the Bluestein convolution lengths Nb; n', m') and the padding factor of the spectrum
 * the applies use (2 compact, 4 literal; Bluestein: the reference's, 4 Greengard_Vico / 2 trapezoidal).  Any pointer
 * may be NULL.                                                                             */
int ls_op2d_info(ls_handle h, int* route, int64_t* n_line, int64_t* m_line, int* padding_factor);
/* size(M,dim) / eltype, FastConvolution.jl:31-41: writes N = n*m */
int ls_op_size(ls_handle h, int64_t* N);

/* ---- 3-D operator: struct FastM3D, FastConvolution3D.jl:7-26 ----------------------------- *
 * GFFT (ne*me*le complex, column-major, centred ordering) may be NULL: the Greengard-Vico
 * spectrum Gtruncated3D(L, k, |kappa|) (Functions.jl:49-51; grid kappa = (2 pi/Lp)(-2n:2n-1),
 * FastConvolution3D.jl:72-99) is then evaluated on the device straight into the kernel layout
 * (at 256^3 the array is 17 GB, at 512^3 137 GB - too big to ship from the host).
 * Served: n == m (the reference pads (ne, ne, le), :48).  Fast path: n, m, l in {64,128,256,512};
 * any other size with 5n - 1 <= 4096 (examples/example3D.jl ships n = 48) runs on the general path
 * (Bluestein lines, single GPU).  With LS_FLAG_EMBED every n = m, l <= 512 runs instead on the
 * power-of-two kernels of n' = max(64, nextpow2(n)) and l', zero-embedded, on one GPU or sharded. */
int ls_op3d_create(ls_handle* out, int64_t n, int64_t m, int64_t l, int64_t ne, int64_t me, int64_t le,
                   const double* nu, const ls_cdouble* gfft_or_null, double omega, double L, double Lp,
                   int flags);
/* Sharded 3-D operator, one process per GPU (P = 2, 4 or 8 ranks of one NVLink/NVSwitch box).
 * Rank r owns the z planes [r*l/P, (r+1)*l/P): nu_slab, and the b / y of ls_op3d_apply, are that
 * contiguous range of n*m*l/P values.  The padded FFT is slab-decomposed; its two transposes push contiguous blocks
 * into the peers' IPC-mapped exchange buffers with the copy engines over NVLink (LS_OP3D_XCHG=nccl: grouped
 * ncclSend/ncclRecv instead), synchronised on the communicator created here from `nccl_unique_id` (128 bytes obtained
 * with ls_nccl_unique_id on rank 0 and broadcast by the host: torch.distributed / MPI /
 * Distributed.jl).  Collective: every rank must call create and each apply.                   */
int ls_nccl_unique_id(void* out128);
int ls_op3d_create_dist(ls_handle* out, int64_t n, int64_t m, int64_t l, const double* nu_slab,
                        double omega, double L, double Lp, int rank, int nranks,
                        const void* nccl_unique_id, int flags);
/* how the handle evaluates: padding factor in use (2 compact / 4 literal), x-slot chunks of the pipelined transposes,
 * transpose route (0: single GPU, 1: NCCL grouped send/recv, 2: copy-engine pushes into IPC-mapped peer buffers)      */
int ls_op3d_info(ls_handle h, int* padding_factor, int* x_slot_chunks, int* exchange);
/* which route the handle runs (0 power-of-two fast path, 1 Bluestein general path, 2 zero-embedded; numbered as in
 * ls_op2d_info) and the line lengths its kernels run along x, y and z (n, m, l; the Bluestein convolution lengths;
 * n', m', l').  Any 3-D handle, sharded or not.  Any pointer may be NULL.                   */
int ls_op3d_lines(ls_handle h, int* route, int64_t* n_line, int64_t* m_line, int64_t* l_line);
/* mode 0: `*(M::FastM3D, b)` = b + omega^2 FFTconvolution(M, nu.*b)  (FastConvolution3D.jl:31-37)
 * mode 1: FFTconvolution(M, b)                                      (FastConvolution3D.jl:39-63) */
int ls_op3d_apply(ls_handle h, const ls_cdouble* b, ls_cdouble* y, int mode, int memloc);

/* ---- several right-hand sides through one operator ------------------------------------------ *
 * Y[:, j] = M*B[:, j] (mode 0) or FFTconvolution(M, B[:, j]) (mode 1) for j < nrhs: b and y are column-major N x nrhs
 * arrays (leading dimensions ldb, ldy >= N); y may alias b only in place (y == b, ldy == ldb).  Any single-GPU 2-D or
 * 3-D operator handle; every column gets the bits of ls_op2d_apply / ls_op3d_apply of it.  The 2x-padded power-of-two
 * routes (route 0 and 2 of ls_op2d_info / ls_op3d_lines) run ls_op_batch_cols columns per launch of each pass, so that
 * the pass that reads the Green's spectrum reads each part of it from HBM once per chunk of columns; every other handle
 * applies the columns one by one.  The work arrays of the extra columns (64 N bytes per column in 2-D, 96 N in 3-D; with
 * host pointers also 32 N of staging) are allocated on first use, kept by the handle and freed by ls_destroy; too
 * little free device memory -> LS_ERR_NOMEM before anything is allocated.  nrhs < 1, ld < N, a null pointer, an overlap
 * other than in place or a handle that is not an operator -> LS_ERR_INVALID, a sharded operator (ls_op3d_create_dist)
 * -> LS_ERR_UNSUPPORTED, both before any CUDA call.                                                                    */
int ls_op_apply_batch(ls_handle op, const ls_cdouble* b, int64_t ldb, ls_cdouble* y, int64_t ldy, int nrhs, int mode,
                      int memloc);
/* columns per multi-column apply of the handle (1: ls_op_apply_batch applies its columns one by one) */
int ls_op_batch_cols(ls_handle op, int* cols);

/* ---- sparsifying matrix As: SparseMatrixCSC{ComplexF64,Int64}, preconditioner.jl:27-30 ------ *
 * Arrays exactly as Julia holds them (A.colptr, A.rowval, A.nzval; 1-based).  Converted once
 * to CSR/int32 on the device.                                                              */
int ls_spm_create(ls_handle* out, int64_t nrows, int64_t ncols, const int64_t* colptr,
                  const int64_t* rowval, const ls_cdouble* nzval);
/* Row slab of As for the slab-decomposed 3-D operator `op` (ls_op3d_create_dist; SURVEY.md 8(e): the 27-point
 * sparsifier of SparsifyingMatrix3D.jl:1410-1653 couples a row only to rows within n*m + n + 1, i.e. to the
 * neighbouring z planes).  The CSC arrays (1-based, as ls_spm_create) hold the block
 * A[row0 : row0 + nrows_local, row0 - halo : row0 + nrows_local + halo), nrows_local + 2*halo columns, columns
 * outside the global matrix empty; row0 = first row of this rank's slab, halo <= nrows_local and equal on every
 * rank.  ls_spm_mv then takes x and y as this rank's slabs and fetches the halo of x from the z-neighbours on
 * the operator's communicator (collective: every rank calls it).  `op` must outlive the matrix.            */
int ls_spm_create_dist(ls_handle* out, ls_handle op, int64_t nrows_local, int64_t halo, const int64_t* colptr,
                       const int64_t* rowval, const ls_cdouble* nzval);
/* y <- alpha*A*x + beta*y : `M.As*b` (preconditioner.jl:138,142,159,163) is alpha=1, beta=0;
 * same meaning as SparseBLAS.cscmv!('N', alpha, "GXXF", A, x, beta, y), sparseblas.jl:14-25.
 * x and y must not alias.                                                                  */
int ls_spm_mv(ls_handle A, ls_cdouble alpha, const ls_cdouble* x, ls_cdouble beta, ls_cdouble* y, int memloc);
/* device format: 0 = CSR (sub-warp per row), 1 = stencil classes (rows grouped by identical
 * (relative offsets, values) - the structure buildSparseA produces; exact detection at create) */
int ls_spm_info(ls_handle A, int64_t* nrows, int64_t* ncols, int64_t* nnz, int* format, int* nclasses);

/* ---- GMRES Arnoldi vector kernels (IterativeSolvers.jl gmres!, un-vendored; call sites ------ *
 * examples/example.jl:85,91).  A Krylov workspace owns the reduction buffers for vectors of
 * length n.  All vector pointers below are DEVICE pointers (ls_dev_alloc).                  */
int ls_krylov_create(ls_handle* out, int64_t n);
/* orth_meth keyword of gmres! (IterativeSolvers.jl orthogonalize.jl): 0 ModifiedGramSchmidt (upstream default,
 * used by every call site of the reference), 1 ClassicalGramSchmidt, 2 DGKS.  1 and 2 sweep the basis with
 * BLAS-2 style multi-dot / multi-axpy kernels: half the HBM traffic of the Gram-Schmidt step.              */
int ls_krylov_set_orth(ls_handle k, int orth_meth);
int ls_zdotc(ls_handle k, const ls_cdouble* x, const ls_cdouble* y, ls_cdouble* result);   /* sum conj(x) y */
int ls_dznrm2(ls_handle k, const ls_cdouble* x, double* result);
int ls_zaxpy(ls_handle k, ls_cdouble alpha, const ls_cdouble* x, ls_cdouble* y);           /* y += alpha x */
int ls_zscal(ls_handle k, ls_cdouble alpha, ls_cdouble* x);
/* orthogonalize_and_normalize!(V[:,1:k], w, h) with ModifiedGramSchmidt: for i<k: h[i] = dot(V_i,w),
 * w -= h[i] V_i; h[k] = norm(w); w /= h[k].  V is column-major with leading dimension ldv.
 * hcol receives k+1 complex values (the last one real).                                     */
int ls_mgs_step(ls_handle k, const ls_cdouble* V, int64_t ldv, int kcols, ls_cdouble* w, ls_cdouble* hcol);

/* Host callback applying Msp^-1 in place on a HOST vector of n complex values (the sparse direct
 * solve `MspInv \ .` of preconditioner.jl:138,159 stays with the caller: UMFPACK / PARDISO /
 * SuperLU).  Return 0 on success.                                                           */
typedef int (*ls_solve_cb)(void* user, ls_cdouble* v_inout, int64_t n);

/* gmres!(x, A, b; Pl, abstol, reltol, restart, maxiter, log=true, initially_zero) with the Krylov
 * basis resident on the GPU.  A = operator handle; left preconditioner ldiv!(Pl, v) =
 * msp_solve(As*v) (preconditioner.jl:147-166): `As` nullable, `msp_solve` nullable.
 * restart <= 0 -> min(20, N); maxiter < 0 -> N (inner iterations), maxiter == 0 -> no iteration;
 * reltol as given (upstream default sqrt(eps)).  resnorm_hist receives the logged residual per
 * inner iteration (history[:resnorm], example.jl:86).  b, x: host or device per memloc.
 * As upstream, x is formed at a restart or at convergence only: when maxiter lands inside a cycle
 * the x of the last restart is returned.  With a sharded operator (ls_op3d_create_dist) the vectors
 * are this rank's slabs, dots and norms are all-reduced on the operator's communicator, `As` must
 * come from ls_spm_create_dist on the same operator and `msp_solve` receives the rank's slab
 * (gathering it is the callback's business; the Msp solve itself is not sharded).            */
int ls_gmres(ls_handle krylov, ls_handle op, ls_handle As, ls_solve_cb msp_solve, void* user,
             const ls_cdouble* b, ls_cdouble* x, int restart, int64_t maxiter, double reltol,
             double abstol, int initially_zero, double* resnorm_hist, int64_t hist_cap,
             int64_t* niter, int* converged, int64_t* mv_products, int memloc);

/* ---- device-resident Msp^-1: `MspInv = lu(Msp)` preconditioner.jl:35 (UMFPACK; :41-55 PARDISO) and the solve
 * `MspInv \ (As*b)` of every GMRES iteration (:138,142,159,163).  Msp = As + k^2 AG diag(nu) (examples/example.jl:67)
 * is a 9-point stencil matrix on the n x m grid (unknown i + n*j, x fastest), given as Julia holds it (1-based CSC).
 * Factorised on the GPU by geometric nested dissection (multifrontal, partial pivoting inside the pivot blocks);
 * every solve is a fixed sequence of batched matrix-vector kernels - no PCIe traffic, no host work per iteration.
 * 2-D grids; ls_msp_factor3d serves the 27-point matrices of 3-D grids.  Entries outside the 9-point pattern ->
 * LS_ERR_UNSUPPORTED, a duplicate (row, col) entry -> LS_ERR_INVALID, a singular pivot block -> LS_ERR_INVALID (depth
 * and node named), more device memory needed than is free -> LS_ERR_NOMEM before anything is allocated.           */
int ls_msp_factor(ls_handle* out, int64_t n, int64_t m, const int64_t* colptr, const int64_t* rowval,
                  const ls_cdouble* nzval);
/* the same for Msp = As + k^2 AG diag(nu) of examples/example3D.jl:56-61: a 27-point stencil matrix on the n x m x l grid
 * (unknown i + n*(j + m*p), x fastest), 1-based CSC.  Nested dissection by separator planes; the handle works with
 * ls_msp_solve / ls_msp_info / ls_msp_plan / ls_gmres_msp unchanged.  l = 1 is exactly ls_msp_factor.              */
int ls_msp_factor3d(ls_handle* out, int64_t n, int64_t m, int64_t l, const int64_t* colptr, const int64_t* rowval,
                    const ls_cdouble* nzval);
/* x <- Msp^-1 rhs (x may alias rhs); host or device pointers per memloc */
int ls_msp_solve(ls_handle msp, const ls_cdouble* rhs, ls_cdouble* x, int memloc);
/* X <- Msp^-1 RHS for nrhs right-hand sides at once (several incident fields with one preconditioner): rhs and x are
 * column-major N x nrhs arrays with leading dimensions ldr, ldx >= N; x may alias rhs when ldx == ldr (in place).
 * Each stored factor block is read once per chunk of columns and applied to all of them (multi-column sweeps,
 * csrc/msp_gemv.cuh): chunks of 4, 2 and 1 (LS_MSP_BATCH_COLS=8 / =2 at handle creation: chunks of up to 8 / 2).  Every column is bit-identical to ls_msp_solve of
 * that column.  Work arrays for each chunk width are allocated on first use and kept by the handle; when the device
 * has too little free memory for them -> LS_ERR_NOMEM before anything is allocated.  nrhs < 1, ld < N, a null pointer
 * or an overlap of x and rhs other than in place -> LS_ERR_INVALID before any CUDA call.  Host or device pointers per
 * memloc; with device pointers each chunk is replayed as a CUDA graph per (pointers, leading dimensions, width).      */
int ls_msp_solve_batch(ls_handle msp, const ls_cdouble* rhs, int64_t ldr, ls_cdouble* x, int64_t ldx, int nrhs, int memloc);
int ls_msp_info(ls_handle msp, int64_t* factor_bytes, int* depth, double* factor_seconds);
/* one line per dissection depth: node count, padded block sizes and the kernel geometry (lanes per row group, rows per
 * group, X staged in shared memory) chosen for its three sweeps, each followed by "cols UuXx/UuXx/UuXx": rows per group
 * and staging of the multi-column kernel of ls_msp_solve_batch for 2, 4 and 8 columns (same lanes); first line: solver
 * version, fusion, tuning time.
 * Writes at most `cap` bytes including the terminator into `buf` (diagnostics for bench / profiles).               */
int ls_msp_plan(ls_handle msp, char* buf, int64_t cap);
/* ls_gmres with ldiv!(Pl, v) = Msp^-1 (As v) entirely on the device (`msp` from ls_msp_factor / ls_msp_factor3d, `As`
 * nullable); single-GPU: a sharded operator -> LS_ERR_UNSUPPORTED                                                  */
int ls_gmres_msp(ls_handle krylov, ls_handle op, ls_handle As, ls_handle msp,
                 const ls_cdouble* b, ls_cdouble* x, int restart, int64_t maxiter, double reltol,
                 double abstol, int initially_zero, double* resnorm_hist, int64_t hist_cap,
                 int64_t* niter, int* converged, int64_t* mv_products, int memloc);
/* nrhs independent ls_gmres_msp runs side by side with one op, As and msp (several incident fields): b and x are
 * column-major N x nrhs arrays (leading dimensions ldb, ldx >= N), resnorm_hist is hist_cap x nrhs (column q: system q's
 * history), niter / converged / mv_products hold nrhs entries (each pointer nullable).  Each system keeps its own Krylov
 * basis, Hessenberg matrix, restarts and tolerance and gets the bits ls_gmres_msp gives it alone; per lockstep iteration
 * the operator applies of all active systems are ls_op_apply_batch chunks, the SpMVs and Gram-Schmidt steps run system
 * by system and the Msp^-1 of all active systems is one ls_msp_solve_batch.  A system that converged or reached maxiter drops out; its x is formed as ls_gmres_msp forms it.
 * Memory for nrhs bases of restart + 1 vectors (and the batched solve's work arrays) is checked against the free device
 * memory before anything is allocated -> LS_ERR_NOMEM; nrhs < 1, ld < N, null pointers -> LS_ERR_INVALID before any
 * CUDA call; a sharded operator -> LS_ERR_UNSUPPORTED.                                                               */
int ls_gmres_msp_batch(ls_handle krylov, ls_handle op, ls_handle As, ls_handle msp, int nrhs,
                       const ls_cdouble* b, int64_t ldb, ls_cdouble* x, int64_t ldx, int restart, int64_t maxiter,
                       double reltol, double abstol, int initially_zero, double* resnorm_hist, int64_t hist_cap,
                       int64_t* niter, int* converged, int64_t* mv_products, int memloc);
/* nrhs independent ls_gmres runs with Pl = Identity side by side with one op (several incident fields without a
 * preconditioner); arguments as ls_gmres_msp_batch without As and msp.  Each system gets the bits ls_gmres (no As, no
 * callback) gives it alone; per lockstep iteration the operator applies of all active systems are ls_op_apply_batch
 * chunks and the Gram-Schmidt steps run system by system.  Same memory check and refusals as ls_gmres_msp_batch.     */
int ls_gmres_batch(ls_handle krylov, ls_handle op, int nrhs, const ls_cdouble* b, int64_t ldb, ls_cdouble* x, int64_t ldx,
                   int restart, int64_t maxiter, double reltol, double abstol, int initially_zero, double* resnorm_hist,
                   int64_t hist_cap, int64_t* niter, int* converged, int64_t* mv_products, int memloc);
/* wall time the last ls_gmres spent in D2H + msp_solve callback + H2D (the "Msp-solve" column of SURVEY.md H1) */
int ls_krylov_last_precond_host_seconds(ls_handle krylov, double* seconds);

/* ---- sparsifier sampling on the device: sampleGConv (FastConvolution.jl:278-306), sampleG3D (FastConvolution3D.jl:136-160).
 * V[:, i] = FFTconvolution(op, e_{indS[i]}) for the s stencil indices (1-based), kept on the device (N x s, column-major).   */
int ls_sample_rows(ls_handle krylov, ls_handle op, const int64_t* indS, int s, ls_cdouble* V_dev, int64_t ldv);
/* gram[i + s*j] = sum_c conj(V[c,i]) V[c,j] (host, s x s): what entriesSparseAConv's svd(GSampled) needs of the rows
 * (SparsifyingMatrix2D.jl:119-127) - its last left singular vector is the eigenvector of the smallest eigenvalue.   */
int ls_gram(ls_handle krylov, const ls_cdouble* V_dev, int64_t ldv, int s, ls_cdouble* gram_host);
/* out[j + nidx*i] = V[idx[j], i] (idx 1-based): the near-field block sampleGConv(...)[:, ind] of entriesSparseGConv (:278-350) */
int ls_gather_rows(ls_handle krylov, const ls_cdouble* V_dev, int64_t ldv, int s, const int64_t* idx, int nidx, ls_cdouble* out_host);

/* ---- handle services ------------------------------------------------------------------ */
int ls_destroy(ls_handle h);
int ls_sync(ls_handle h);
/* CUDA-event timer on the handle's own stream (the stream its kernels are launched on) */
int ls_timer_start(ls_handle h);
int ls_timer_stop(ls_handle h, float* elapsed_ms);
/* number of kernels this handle has launched since creation (bench `gpu_launches`) */
int ls_launch_count(ls_handle h, int64_t* count);

/* per-phase CUDA-event profile of the handle's launches (phase ids are listed per operator
 * in DESIGN.md; 2-D: 0 = P1 forward columns, 1 = P2 fused rows, 2 = P3 inverse columns).
 * ls_profile_read synchronises and returns cumulative milliseconds and launch counts.     */
int ls_profile_enable(ls_handle h, int on);
int ls_profile_read(ls_handle h, double* ms_per_phase, int64_t* launches_per_phase, int nphase);

/* ---- test hooks ----------------------------------------------------------------------- */
/* batched forward DFT (natural order out) / round trip of `nlines` lines of length N through
 * the line-FFT engine; device-side unit test of fft_engine.cuh.                           */
int ls_test_fft_lines(int64_t N, int64_t nlines, const ls_cdouble* in_host, ls_cdouble* out_host,
                      int inverse_roundtrip);

/* measured device peaks used as roofline denominators by bench.py: FP64 FMA TFLOP/s, FP64 add/mul lane-instructions
 * per second (in 1e12), and the read+write GB/s of a plain 1 GiB copy kernel                                     */
int ls_test_device_peaks(double* dfma_tflops, double* dadd_tinst, double* copy_gbs);

#ifdef __cplusplus
}
#endif
#endif /* LS_CUDA_H */
