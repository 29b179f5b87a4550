// 2-D Lippmann-Schwinger operator  y = b + omega^2 * G (nu .* b)   on one B200.
// Stands behind struct FastM and its `*` / mul! / fastconvolution / FFTconvolution methods
// (reference FastConvolution.jl:11-154).  Three launches per apply:
//   P1  k_fwd_pruned  columns (x, contiguous):  b, nu      -> A  [ne x m]   (slot order in x)
//   P2  k_mid_swap    rows (y): A, Green spectrum          -> C  [m x ne]   (k_mid_fused with LS_FLAG_PAD4)
//   P3  k_inv_pruned  columns (x): C, b                    -> y
// Padding.  The reference pads 4x per dimension (Greengard_Vico) because the truncated-kernel spectrum has
// to be *built* on the 4n grid; the apply itself only ever touches the spatial kernel g = ifft2(GFFT) at the
// lags (-n, n) x (-m, m) (input supported on [0,n), output cropped to [0,n)).  At create time the handle
// therefore computes g on the device (pruned inverse transforms of the given GFFT), wraps those lags onto a
// 2n x 2m grid and transforms back: G2 = fft2(g2).  Every apply then runs with 2x padding - the same linear
// operator to rounding (measured 1e-16 relative against the literal 4x evaluation), a quarter of the
// spectrum, half of the intermediates and about a third of the FP64 work.  LS_FLAG_PAD4 keeps the literal
// 4x evaluation (tests compare the two).
// Algorithmic HBM bytes per apply: 2x padding 24N + 64N + 64N + 64N + 32N = 248*N;
//                                  4x padding (SURVEY.md section 8(d)) 568*N.
// Zero embedding (LS_FLAG_EMBED, any n, m <= 4096, both quadratures).  The same restriction argument: an n x m apply
// only touches the lags (-n, n) x (-m, m), and those are a subset of the lags (-n', n') x (-m', m') of the power-of-two
// grid n' = max(64, nextpow2(n)).  The handle extracts exactly those lags from the reference's spectrum (op2d_embed.cu),
// wraps them onto 2n' x 2m' and runs the n' x m' compact apply with masked P1 / P3 kernels: inputs past (n, m) read as
// zero, outputs past (n, m) are not written.
#include "ls_common.cuh"
#include "op2d_base.cuh"
#include "line_kernels.cuh"
#include "gv_spectrum2d.cuh"
#include <cudaTypedefs.h>
#include <algorithm>

using namespace ls;
using namespace lsk;

namespace {

// x-slot interleave of the P2 -> P3 intermediate C: P3's strided reads then cover 64-byte runs.  Measured at 2048^2 on
// B200: P2 + P3 = 0.326 / 0.313 / 0.304 / 0.31 ms for 1 / 2 / 4 / 8 interleaved slots.
constexpr int CW_SHIFT = 2;
constexpr long CW = 1L << CW_SHIFT;

// columns per multi-column apply (ls_op_apply_batch) of the 2x-padded routes.  Measured on B200 (1000 W,
// profiles/r5_apply_batch.log, ms per column at K = 1 / 4): 201^2 embedded 0.033 / 0.0093, 2048^2 0.317 / 0.288,
// 4096^2 1.498 / 1.449; 8 columns (two chunks) are no faster per column than 4.
constexpr int BATCH_COLS = 4;

struct Op2D : Op2DBase {
    int nr = 4;               // padding factor actually used by the applies (4: literal, 2: compact)
    long pn = 0, pm = 0;      // padded sizes nr*n, nr*m
    double* d_nu = nullptr;
    cd* d_G = nullptr;        // [sx][ry][slot_y] on the pn x pm grid, normalisation folded in
    cd* d_TABn = nullptr; cd* d_TABm = nullptr;   // engine tables (fft_engine.cuh EngTab)
    cd* d_A = nullptr;        // pn x m
    cd* d_C = nullptr;        // P2 output: slot sx of column j at C[(sx/CW)*(CW*m) + CW*j + sx%CW]
    bool embed = false;       // LS_FLAG_EMBED: lines of ln x lm points carry the n x m grid (ln = n, lm = m otherwise)
    long ln = 0, lm = 0;
    CUtensorMap tmA, tmC;     // 2x padding: P2's line loads from A and stores into C (encode_line_maps)
    int cols = 1;             // columns of A and C (ls_op_apply_batch widens them on first use), pn*lm elements apart
    int apply_dev(const cd* b, cd* y, int mode) override;
    int batch_cols() const override { return nr == 2 ? BATCH_COLS : 1; }
    size_t batch_bytes(int ncol) const override { return ncol > cols ? 2 * (size_t)ncol * pn * lm * sizeof(cd) : 0; }
    int batch_reserve(int ncol) override;
    int apply_cols_dev(const cd* const* b, cd* const* y, int ncol, int mode) override;
    void info(int* route, int64_t* n_line, int64_t* m_line, int* padding) const override {
        *route = embed ? 2 : 0; *n_line = ln; *m_line = lm; *padding = nr;
    }
};

__global__ void k_scale(cd* a, long n, double s) {
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        cd v = a[i];
        a[i] = make_double2(v.x * s, v.y * s);
    }
}

// Gd[(sx*4 + ry)*m + sy] = GFFT[(4 fx[sx%n] + sx/n + ne/2) % ne, (4 fy[sy] + ry + me/2) % me] / (ne*me)
__global__ void k_permute_g2d(const cd* __restrict__ gin, cd* __restrict__ gout,
                              const int* __restrict__ fx, const int* __restrict__ fy,
                              long n, long m, long ne, long me, double scale) {
    long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    long total = ne * me;
    if (idx >= total) return;
    long sy = idx % m;
    long ry = (idx / m) % 4;
    long sx = idx / (4 * m);
    long kx = 4L * fx[sx % n] + sx / n;
    long ky = 4L * fy[sy] + ry;
    long ix = (kx + ne / 2) % ne, iy = (ky + me / 2) % me;
    cd v = gin[ix + ne * iy];
    gout[idx] = make_double2(v.x * scale, v.y * scale);
}

// same layout as k_permute_g2d, values evaluated on the device (Gtruncated2D, Functions.jl:40-42) instead of gathered
__global__ void k_fill_g2d(cd* __restrict__ gout, const int* __restrict__ fx, const int* __restrict__ fy,
                           long n, long m, long ne, long me, double scale, Gv2dParams p) {
    long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    long total = ne * me;
    if (idx >= total) return;
    long sy = idx % m;
    long ry = (idx / m) % 4;
    long sx = idx / (4 * m);
    long kx = 4L * fx[sx % n] + sx / n;
    long ky = 4L * fy[sy] + ry;
    long ix = (kx + ne / 2) % ne, iy = (ky + me / 2) % me;
    cd v = gtrunc2d_eval(p, ix, iy, ne, me);
    gout[idx] = make_double2(v.x * scale, v.y * scale);
}
// the centred ne x me array exactly as the reference holds it (general-size path)
__global__ void k_fill_g2d_centred(cd* __restrict__ gout, long ne, long me, Gv2dParams p) {
    long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= ne * me) return;
    gout[idx] = gtrunc2d_eval(p, idx % ne, idx / ne, ne, me);
}

#define LS_DISPATCH_E(N_, CALL)                                                    \
    switch (N_) {                                                                  \
        case 64:   e = CALL(64); break;                                            \
        case 128:  e = CALL(128); break;                                           \
        case 256:  e = CALL(256); break;                                           \
        case 512:  e = CALL(512); break;                                           \
        case 1024: e = CALL(1024); break;                                          \
        case 2048: e = CALL(2048); break;                                          \
        case 4096: e = CALL(4096); break;                                          \
        default: e = cudaErrorInvalidValue;                                        \
    }

// The pointer lists of the three passes for columns b[c] -> y[c], c < ncol: P1 b -> A, P3 C (and b) -> y.  Column c of A
// and C starts c*pn*lm elements in.
void pass_cols(const Op2D* op, const cd* const* b, cd* const* y, int ncol, bool full, ColPtrs& p1, ColPtrs& p3) {
    p1 = ColPtrs{}; p3 = ColPtrs{};
    const long cs = op->pn * op->lm;
    for (int c = 0; c < ncol; ++c) {
        p1.in[c] = b[c]; p1.out[c] = op->d_A + c * cs;
        p3.in[c] = op->d_C + c * cs; p3.b[c] = full ? b[c] : nullptr; p3.out[c] = y[c];
    }
}

int apply_device(Op2D* op, const cd* const* b, cd* const* y, int ncol, int mode) {
    cudaError_t e = cudaSuccess;
    cudaStream_t s = op->stream;
    const long n = op->n, m = op->m, pn = op->pn;
    const bool full = (mode == LS_APPLY_FASTCONVOLUTION);
    const double* nu = full ? op->d_nu : nullptr;   // Q2: GV FFTconvolution has no nu
    ColPtrs p1, p3;
    pass_cols(op, b, y, ncol, full, p1, p3);
    // P1: columns (x, contiguous): point i of column j at b[i + n*j] -> slot sx at A[sx + pn*j]
    {
        LineAddr la{1L << 40, n, 0, 1, pn, 0, 1};
        la.nr = op->nr;
        op->phase_begin(0);
#define P1(N) launch_fwd_cols<N, false>(s, m, p1, ncol, nu, op->d_TABn, la)
        LS_DISPATCH_E(n, P1);
        op->phase_end(); op->launches++;
        LS_CUDA_TRY(e);
    }
    // P2: rows (y): line = x slot sx, point j at A[sx + pn*j]; output: CW adjacent x-slots interleaved,
    //     C[(sx/CW)*(CW*m) + CW*j + sx%CW].  2x padding: the swap kernel (no accumulator registers, see line_kernels.cuh)
    {
        LineAddr la{CW, 1, CW, pn, 1, CW * m, CW};
        la.nr = op->nr;
        op->phase_begin(1);
#define P2S(N) launch_mid_swap<N, CW_SHIFT>(s, pn, op->tmA, op->tmC, op->d_C, op->d_G, op->d_TABm, ncol, pn * m)
#define P2F(N) launch_mid<N, false>(s, pn, op->d_A, op->d_C, op->d_G, op->d_TABm, la)
        if (op->nr == 2) { LS_DISPATCH_E(m, P2S); } else { LS_DISPATCH_E(m, P2F); }
        op->phase_end(); op->launches++;
        LS_CUDA_TRY(e);
    }
    // P3: columns (x) + combine: line = column j; slot sx at C[(sx/CW)*(CW*m) + CW*j + sx%CW]: adjacent lanes read
    //     adjacent slots.  The next slot block and b are staged in shared memory while the current block is transformed
    //     (2048^2 on B200: 0.131 -> 0.077 ms together with the 4-slot interleave of C)
    {
        LineAddr la{1L << 40, CW, 0, 1, n, 0, 1};
        la.split_shift = CW_SHIFT; la.split_stride = CW * m;
        la.nr = op->nr;
        op->phase_begin(2);
#define P3(N) launch_inv_cols<N, false, true>(s, m, p3, ncol, op->d_TABn, full ? op->omega * op->omega : 1.0, la)
        LS_DISPATCH_E(n, P3);
        op->phase_end(); op->launches++;
        LS_CUDA_TRY(e);
    }
    return LS_OK;
}

// Zero-embedded apply: the three launches of apply_device at 2x padding on the ln x lm grid.  P1 reads the n x m input
// (column stride n) with points >= n and lines >= m as zeros and covers ceil(m / LPC) CTAs; columns [m, lm) of A that
// P2 reads stay zero from create time.  P3 writes points < n of lines < m only.  Greengard_Vico FFTconvolution has no
// nu (Q2); the trapezoidal rule applies it in both modes (FastConvolution.jl:122 vs :141).
int apply_embedded(Op2D* op, const cd* const* b, cd* const* y, int ncol, int mode) {
    cudaError_t e = cudaSuccess;
    cudaStream_t s = op->stream;
    const long n = op->n, m = op->m, ln = op->ln, lm = op->lm, pn = op->pn;
    const bool full = (mode == LS_APPLY_FASTCONVOLUTION);
    const double* nu = (full || op->quadrule == LS_QUAD_TRAPEZOIDAL) ? op->d_nu : nullptr;
    ColPtrs p1, p3;
    pass_cols(op, b, y, ncol, full, p1, p3);
    {
        LineAddr la{1L << 40, n, 0, 1, pn, 0, 1};
        la.nr = 2;
        la.mask_pts = (int16_t)n; la.mask_lines = (int)m;
        op->phase_begin(0);
#define E1(N) launch_fwd_cols<N, false, true>(s, m, p1, ncol, nu, op->d_TABn, la)
        LS_DISPATCH_E(ln, E1);
        op->phase_end(); op->launches++;
        LS_CUDA_TRY(e);
    }
    {
        op->phase_begin(1);
#define E2(N) launch_mid_swap<N, CW_SHIFT>(s, pn, op->tmA, op->tmC, op->d_C, op->d_G, op->d_TABm, ncol, pn * lm)
        LS_DISPATCH_E(lm, E2);
        op->phase_end(); op->launches++;
        LS_CUDA_TRY(e);
    }
    {
        LineAddr la{1L << 40, CW, 0, 1, n, 0, 1};
        la.split_shift = CW_SHIFT; la.split_stride = CW * lm;
        la.nr = 2;
        la.mask_pts = (int16_t)n; la.mask_lines = (int)m;
        op->phase_begin(2);
#define E3(N) launch_inv_cols<N, false, true, true>(s, m, p3, ncol, op->d_TABn, full ? op->omega * op->omega : 1.0, la)
        LS_DISPATCH_E(ln, E3);
        op->phase_end(); op->launches++;
        LS_CUDA_TRY(e);
    }
    return LS_OK;
}

}  // namespace

int Op2D::apply_dev(const cd* b, cd* y, int mode) {
    return embed ? apply_embedded(this, &b, &y, 1, mode) : apply_device(this, &b, &y, 1, mode);
}

int Op2D::apply_cols_dev(const cd* const* b, cd* const* y, int ncol, int mode) {
    if (nr != 2) return HandleBase::apply_cols_dev(b, y, ncol, mode);     // LS_FLAG_PAD4: column by column
    LS_REQUIRE(ncol >= 1 && ncol <= cols, LS_ERR_INVALID, "2-D batched apply: %d columns, %d reserved", ncol, cols);
    return embed ? apply_embedded(this, b, y, ncol, mode) : apply_device(this, b, y, ncol, mode);
}

namespace {

// The 2x-padded P2 (k_mid_swap) moves its lines by tensor copies.  As FLOAT64 arrays with re, im innermost, line sx of
// column c of A is the box {2, BOX, 1} at (2 sx, j0, c) of the 3-D view {2 pn, lm, cols}, and line sx of column c of C
// the box {2, BOX, 1, 1} at (2 (sx % CW), j0, sx / CW, c) of the 4-D view {2 CW, lm, pn / CW, cols}, i.e.
// C[c*pn*lm + (sx/CW)*(CW*lm) + CW*j + sx%CW].
// BOX = min(lm, 256), the largest box side.  cuTensorMapEncodeTiled is reached through the runtime's driver entry point,
// so the library does not link against libcuda.
int encode_line_maps(Op2D* op) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
    LS_CUDA_TRY(cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &fn, 12000, cudaEnableDefault, &q));
    LS_REQUIRE(q == cudaDriverEntryPointSuccess && fn, LS_ERR_CUDA, "the driver has no cuTensorMapEncodeTiled");
    const auto encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
    const cuuint64_t pn = (cuuint64_t)op->pn, lm = (cuuint64_t)op->lm;
    const cuuint64_t cols = (cuuint64_t)op->cols;
    const cuuint32_t box = (cuuint32_t)std::min<long>(op->lm, 256), unit[4] = {1, 1, 1, 1};
    const cuuint64_t dimA[3] = {2 * pn, lm, cols}, strideA[2] = {pn * sizeof(cd), pn * lm * sizeof(cd)};
    const cuuint32_t boxA[3] = {2, box, 1};
    const cuuint64_t dimC[4] = {2 * CW, lm, pn / CW, cols};
    const cuuint64_t strideC[3] = {CW * sizeof(cd), CW * lm * sizeof(cd), pn * lm * sizeof(cd)};
    const cuuint32_t boxC[4] = {2, box, 1, 1};
    CUresult r = encode(&op->tmA, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, op->d_A, dimA, strideA, boxA, unit,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    const char* which = "A";
    if (r == CUDA_SUCCESS) {
        which = "C";
        r = encode(&op->tmC, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 4, op->d_C, dimC, strideC, boxC, unit,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    }
    if (r != CUDA_SUCCESS) {
        const char* msg = nullptr;
        void* es = nullptr;
        if (cudaGetDriverEntryPointByVersion("cuGetErrorString", &es, 6000, cudaEnableDefault, &q) == cudaSuccess && es)
            reinterpret_cast<PFN_cuGetErrorString_v6000>(es)(r, &msg);
        set_error("cuTensorMapEncodeTiled (P2 line map of %s, pn=%ld, lm=%ld) failed: %s (CUresult %d)", which,
                  (long)pn, (long)lm, msg ? msg : "no message", (int)r);
        return LS_ERR_CUDA;
    }
    return LS_OK;
}

}  // namespace

// A and C for ncol columns: new arrays, zeroed (the embedded route reads columns [m, lm) of A, which P1 never writes),
// the old ones freed once the stream has drained, the line maps encoded again.  The caller checked the free memory.
int Op2D::batch_reserve(int ncol) {
    if (ncol <= cols) return LS_OK;
    const size_t bytes = (size_t)ncol * pn * lm * sizeof(cd);
    cd *a = nullptr, *c = nullptr;
    int rc;
    if ((rc = dmalloc((void**)&a, bytes))) return rc;
    if ((rc = dmalloc((void**)&c, bytes))) { dfree(a); return rc; }
    LS_CUDA_TRY(cudaMemsetAsync(a, 0, bytes, stream));
    LS_CUDA_TRY(cudaStreamSynchronize(stream));
    dfree(d_A); dfree(d_C);
    d_A = a; d_C = c; cols = ncol;
    return encode_line_maps(this);
}

namespace {

// G2 = fft2(g2) / (2n 2m) in the slot order of the nr = 2 kernels (n, m: the line lengths, powers of two).
// g2[jx2 + 2n*jy2]: the spatial kernel with its lags wrapped onto the 2n x 2m grid (negative lags at the end).
// Takes ownership of g2 (freed here); on return op->d_G = G2 and op->nr = 2.
int lag_spectrum(Op2D* op, cd* g2, long n, long m) {
    cudaStream_t s = op->stream;
    cudaError_t e = cudaSuccess;
    cd *t2 = nullptr, *G2 = nullptr;
    int rc;
    if ((rc = op->dmalloc((void**)&t2, (size_t)(2 * n) * (2 * m) * sizeof(cd)))) return rc;
    if ((rc = op->dmalloc((void**)&G2, (size_t)(2 * n) * (2 * m) * sizeof(cd)))) return rc;
    {   // (3) forward along x on the full 2n-point lines: T2[sx2 + 2n*jy2]
        LineAddr la{1L << 40, 2 * n, 0, 1, 2 * n, 0, 1};
        la.nr = 2; la.full2 = 1;
#define S3(N) launch_fwd<N, false>(s, 2 * m, g2, nullptr, t2, op->d_TABn, la)
        LS_DISPATCH_E(n, S3);
        LS_CUDA_TRY(e);
    }
    {   // (4) forward along y: G2[sx2*2m + (ry*m + sy)]
        LineAddr la{1L << 40, 1, 0, 2 * n, 2 * m, 0, 1};
        la.nr = 2; la.full2 = 1;
#define S4(N) launch_fwd<N, false>(s, 2 * n, t2, nullptr, G2, op->d_TABm, la)
        LS_DISPATCH_E(m, S4);
        LS_CUDA_TRY(e);
    }
    k_scale<<<148 * 8, 256, 0, s>>>(G2, (2 * n) * (2 * m), 1.0 / ((double)(2 * n) * (double)(2 * m)));
    LS_CUDA_TRY(cudaStreamSynchronize(s));
    op->dfree(g2);
    op->dfree(t2);
    op->d_G = G2;
    op->nr = 2;
    return LS_OK;
}

// Compact (2x) spectrum from the reference's 4x one.  g4s: [sx4][ry][sy] slot order on the 4n x 4m grid,
// already scaled by 1/(ne me).  On return op->d_G holds G2 = fft2(g wrapped onto 2n x 2m) in the slot order
// of the nr = 2 kernels, scaled by 1/(2n 2m).
int compact_spectrum(Op2D* op, cd* g4s) {
    const long n = op->n, m = op->m;
    cudaStream_t s = op->stream;
    cudaError_t e = cudaSuccess;
    cd *t1 = nullptr, *g2 = nullptr;
    int rc;
    if ((rc = op->dmalloc((void**)&t1, (size_t)(4 * n) * (2 * m) * sizeof(cd)))) return rc;
    // (1) inverse along y, keep lags [0, m) and [-m, 0): T1[sx4*2m + jy2]
    for (int c = 0; c <= 3; c += 3) {
        LineAddr la{1L << 40, 4 * m, 0, 1, 2 * m, 0, 1};
        la.nr = 4; la.cblock = c;
        cd* outp = t1 + (c ? m : 0);
#define S1(N) launch_inv<N, false>(s, 4 * n, g4s, nullptr, outp, op->d_TABm, 1.0, la)
        LS_DISPATCH_E(m, S1);
        LS_CUDA_TRY(e);
    }
    LS_CUDA_TRY(cudaStreamSynchronize(s));
    op->dfree(g4s);
    if ((rc = op->dmalloc((void**)&g2, (size_t)(2 * n) * (2 * m) * sizeof(cd)))) return rc;
    // (2) inverse along x: g2[jx2 + 2n*jy2]
    for (int c = 0; c <= 3; c += 3) {
        LineAddr la{1L << 40, 1, 0, 2 * m, 2 * n, 0, 1};
        la.nr = 4; la.cblock = c;
        cd* outp = g2 + (c ? n : 0);
#define S2(N) launch_inv<N, false>(s, 2 * m, t1, nullptr, outp, op->d_TABn, 1.0, la)
        LS_DISPATCH_E(n, S2);
        LS_CUDA_TRY(e);
    }
    LS_CUDA_TRY(cudaStreamSynchronize(s));
    op->dfree(t1);
    return lag_spectrum(op, g2, n, m);    // (3), (4) and the 1/(2n 2m) scale
}

// LS_FLAG_EMBED: any n, m <= 4096, both quadratures.  gfft: host spectrum, or nullptr for the Greengard_Vico
// spectrum generated on the device from (L, Lp).
int create_embedded(ls_handle* out, long n, long m, long ne, long me, const double* nu, const ls_cdouble* gfft,
                    double omega, int quadrule, double L, double Lp) {
    Op2D* op = new Op2D();
    int rc = op->init_base(KIND_OP2D);
    if (rc) { delete op; return rc; }
    op->n = n; op->m = m; op->ne = ne; op->me = me; op->omega = omega; op->quadrule = quadrule;
    op->embed = true;
    op->ln = embed_len(n); op->lm = embed_len(m);
    const long ln = op->ln, lm = op->lm;
    const size_t N = (size_t)n * m, NE = (size_t)ne * me;
#define TRY(x) do { rc = (x); if (rc) { delete op; return rc; } } while (0)
    TRY(op->dupload((void**)&op->d_nu, nu, N * sizeof(double)));
    {
        auto Tn = engine_table((int)ln), Tm = engine_table((int)lm);
        TRY(op->dupload((void**)&op->d_TABn, Tn.data(), Tn.size() * sizeof(cd)));
        TRY(op->dupload((void**)&op->d_TABm, Tm.data(), Tm.size() * sizeof(cd)));
    }
    {
        // the centred spectrum as the reference holds it, then its lags (-n, n) x (-m, m) wrapped onto 2ln x 2lm
        cd* d_gin = nullptr;
        cd* g2 = nullptr;
        if (gfft) {
            TRY(op->dupload((void**)&d_gin, gfft, NE * sizeof(cd)));
        } else {
            TRY(op->dmalloc((void**)&d_gin, NE * sizeof(cd)));
            k_fill_g2d_centred<<<(unsigned)((NE + 255) / 256), 256, 0, op->stream>>>(d_gin, ne, me, gv2d_params(L, Lp, omega));
            cudaError_t e = cudaGetLastError();
            if (e != cudaSuccess) { set_error("spectrum generation failed: %s", cudaGetErrorString(e)); delete op; return LS_ERR_CUDA; }
        }
        TRY(op->dmalloc((void**)&g2, (size_t)(2 * ln) * (2 * lm) * sizeof(cd)));
        TRY(embed_lag_grid(op, d_gin, n, m, ne, me, quadrule == LS_QUAD_TRAPEZOIDAL, g2, 2 * ln, 2 * lm));
        op->dfree(d_gin);
        TRY(lag_spectrum(op, g2, ln, lm));
    }
    op->pn = 2 * ln; op->pm = 2 * lm;
    TRY(op->dmalloc((void**)&op->d_A, (size_t)op->pn * lm * sizeof(cd)));
    TRY(op->dmalloc((void**)&op->d_C, (size_t)op->pn * lm * sizeof(cd)));
    TRY(encode_line_maps(op));
    {   // columns [m, lm) of A are read by P2 and never written by P1
        cudaError_t e = cudaMemsetAsync(op->d_A, 0, (size_t)op->pn * lm * sizeof(cd), op->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(op->stream);
        if (e != cudaSuccess) { set_error("embedded set-up failed: %s", cudaGetErrorString(e)); delete op; return LS_ERR_CUDA; }
    }
    TRY(op->dmalloc((void**)&op->d_b, N * sizeof(cd)));
    TRY(op->dmalloc((void**)&op->d_y, N * sizeof(cd)));
#undef TRY
    *out = reinterpret_cast<ls_handle>(op);
    return LS_OK;
}

}  // namespace

extern "C" {

static int op2d_create_impl(ls_handle* out, int64_t n, int64_t m, int64_t ne, int64_t me,
                            const double* nu, const ls_cdouble* gfft, double omega, int quadrule, int flags,
                            double L, double Lp);

int ls_op2d_create(ls_handle* out, int64_t n, int64_t m, int64_t ne, int64_t me,
                   const double* nu, const ls_cdouble* gfft, double omega, int quadrule, int flags) {
    LS_REQUIRE(out && nu && gfft, LS_ERR_INVALID, "ls_op2d_create: null pointer");
    return op2d_create_impl(out, n, m, ne, me, nu, gfft, omega, quadrule, flags, 0.0, 0.0);
}

int ls_op2d_create_gv(ls_handle* out, int64_t n, int64_t m, const double* nu, double omega, double L, double Lp, int flags) {
    LS_REQUIRE(out && nu, LS_ERR_INVALID, "ls_op2d_create_gv: null pointer");
    LS_REQUIRE(L > 0 && Lp > 0 && omega > 0, LS_ERR_INVALID, "ls_op2d_create_gv: L, Lp and k must be positive");
    return op2d_create_impl(out, n, m, 4 * n, 4 * m, nu, nullptr, omega, LS_QUAD_GREENGARD_VICO, flags, L, Lp);
}

static int op2d_create_impl(ls_handle* out, int64_t n, int64_t m, int64_t ne, int64_t me,
                            const double* nu, const ls_cdouble* gfft, double omega, int quadrule, int flags,
                            double L, double Lp) {
    LS_REQUIRE(n > 0 && m > 0 && ne > 0 && me > 0, LS_ERR_INVALID, "ls_op2d_create: non-positive size");
    LS_REQUIRE(quadrule == LS_QUAD_TRAPEZOIDAL || quadrule == LS_QUAD_GREENGARD_VICO, LS_ERR_INVALID,
               "ls_op2d_create: unknown quadRule %d", quadrule);
    if (flags & LS_FLAG_EMBED) {
        // every refusal before any CUDA call
        LS_REQUIRE(!(flags & LS_FLAG_FORCE_GENERIC), LS_ERR_INVALID,
                   "ls_op2d_create: LS_FLAG_EMBED and LS_FLAG_FORCE_GENERIC select different routes");
        LS_REQUIRE(!(flags & LS_FLAG_PAD4), LS_ERR_UNSUPPORTED,
                   "ls_op2d_create: the zero-embedded route runs with 2x padding only (no literal 4x evaluation)");
        if (quadrule == LS_QUAD_TRAPEZOIDAL)
            LS_REQUIRE(ne == 2 * n - 1 && me == 2 * m - 1, LS_ERR_INVALID,
                       "ls_op2d_create: trapezoidal needs ne = 2n-1, me = 2m-1 (FastConvolution.jl:183)");
        else
            LS_REQUIRE(ne == 4 * n && me == 4 * m, LS_ERR_INVALID,
                       "ls_op2d_create: Greengard_Vico needs ne = 4n, me = 4m (FastConvolution.jl:201)");
        LS_REQUIRE(n <= 4096 && m <= 4096, LS_ERR_UNSUPPORTED,
                   "ls_op2d_create: n=%ld, m=%ld: the zero-embedded route serves n, m <= 4096", (long)n, (long)m);
        return create_embedded(out, n, m, ne, me, nu, gfft, omega, quadrule, L, Lp);
    }
    if (quadrule == LS_QUAD_TRAPEZOIDAL) {
        LS_REQUIRE(ne == 2 * n - 1 && me == 2 * m - 1, LS_ERR_INVALID,
                   "ls_op2d_create: trapezoidal needs ne = 2n-1, me = 2m-1 (FastConvolution.jl:183)");
        return create_op2d_generic(out, n, m, ne, me, nu, gfft, omega, quadrule);
    }
    LS_REQUIRE(ne == 4 * n && me == 4 * m, LS_ERR_INVALID,
               "ls_op2d_create: Greengard_Vico needs ne = 4n, me = 4m (FastConvolution.jl:201)");
    if (!(fft_size_supported(n) && fft_size_supported(m)) || (flags & LS_FLAG_FORCE_GENERIC)) {
        if (gfft) return create_op2d_generic(out, n, m, ne, me, nu, gfft, omega, quadrule);
        // general-size path with the spectrum generated on the device: the centred array as the reference holds it
        LS_REQUIRE(ne + n - 1 <= 4096 && me + m - 1 <= 4096, LS_ERR_UNSUPPORTED,
                   "ls_op2d_create_gv: n=%ld, m=%ld: the general-size GPU path serves 5n - 1 <= 4096", (long)n, (long)m);
        cd* d_g = nullptr;
        LS_CUDA_TRY(cudaMalloc((void**)&d_g, (size_t)ne * me * sizeof(cd)));
        const Gv2dParams gp = gv2d_params(L, Lp, omega);
        k_fill_g2d_centred<<<(unsigned)(((size_t)ne * me + 255) / 256), 256>>>(d_g, ne, me, gp);
        cudaError_t ge = cudaDeviceSynchronize();
        int grc = ge == cudaSuccess ? create_op2d_generic(out, n, m, ne, me, nu, nullptr, omega, quadrule, d_g) : LS_ERR_CUDA;
        if (ge != cudaSuccess) set_error("spectrum generation failed: %s", cudaGetErrorString(ge));
        cudaFree(d_g);
        return grc;
    }

    Op2D* op = new Op2D();
    int rc = op->init_base(KIND_OP2D);
    if (rc) { delete op; return rc; }
    op->n = n; op->m = m; op->ne = ne; op->me = me; op->omega = omega; op->quadrule = quadrule;
    op->ln = n; op->lm = m;
    const size_t N = (size_t)n * m, NE = (size_t)ne * me;
#define TRY(x) do { rc = (x); if (rc) { delete op; return rc; } } while (0)
    TRY(op->dupload((void**)&op->d_nu, nu, N * sizeof(double)));
    {
        auto Tn = engine_table((int)n), Tm = engine_table((int)m);
        TRY(op->dupload((void**)&op->d_TABn, Tn.data(), Tn.size() * sizeof(cd)));
        TRY(op->dupload((void**)&op->d_TABm, Tm.data(), Tm.size() * sizeof(cd)));
    }
    {
        // one-time permutation of the spectrum into [x slot][ry][y slot] order, ifftshift folded in
        auto fx = slot_freq((int)n), fy = slot_freq((int)m);
        int *d_fx = nullptr, *d_fy = nullptr;
        cd* d_gin = nullptr;
        TRY(op->dupload((void**)&d_fx, fx.data(), fx.size() * sizeof(int)));
        TRY(op->dupload((void**)&d_fy, fy.data(), fy.size() * sizeof(int)));
        TRY(op->dmalloc((void**)&op->d_G, NE * sizeof(cd)));
        const int th = 256;
        if (gfft) {
            TRY(op->dupload((void**)&d_gin, gfft, NE * sizeof(cd)));
            k_permute_g2d<<<(unsigned)((NE + th - 1) / th), th, 0, op->stream>>>(
                d_gin, op->d_G, d_fx, d_fy, n, m, ne, me, 1.0 / ((double)ne * (double)me));
        } else {
            // Gtruncated2D evaluated straight into the kernel layout: no host Bessel evaluation, no 16 ne me byte upload
            k_fill_g2d<<<(unsigned)((NE + th - 1) / th), th, 0, op->stream>>>(
                op->d_G, d_fx, d_fy, n, m, ne, me, 1.0 / ((double)ne * (double)me), gv2d_params(L, Lp, omega));
        }
        cudaError_t e = cudaStreamSynchronize(op->stream);
        if (e != cudaSuccess) { set_error("spectrum set-up failed: %s", cudaGetErrorString(e)); delete op; return LS_ERR_CUDA; }
        if (d_gin) op->dfree(d_gin);
        op->dfree(d_fx); op->dfree(d_fy);
    }
    op->nr = 4;
    if (!(flags & LS_FLAG_PAD4)) {
        cd* g4s = op->d_G;
        op->d_G = nullptr;
        TRY(compact_spectrum(op, g4s));
    }
    op->pn = op->nr * n; op->pm = op->nr * m;
    TRY(op->dmalloc((void**)&op->d_A, (size_t)op->pn * m * sizeof(cd)));
    TRY(op->dmalloc((void**)&op->d_C, (size_t)op->pn * m * sizeof(cd)));
    if (op->nr == 2) TRY(encode_line_maps(op));
    TRY(op->dmalloc((void**)&op->d_b, N * sizeof(cd)));
    TRY(op->dmalloc((void**)&op->d_y, N * sizeof(cd)));
#undef TRY
    *out = reinterpret_cast<ls_handle>(op);
    return LS_OK;
}

int ls_op2d_apply(ls_handle h, const ls_cdouble* b, ls_cdouble* y, int mode, int memloc) {
    LS_REQUIRE(h && b && y, LS_ERR_INVALID, "ls_op2d_apply: null argument");
    Op2DBase* op = reinterpret_cast<Op2DBase*>(h);
    LS_REQUIRE(op->kind == KIND_OP2D, LS_ERR_INVALID, "ls_op2d_apply: not a 2-D operator handle");
    LS_REQUIRE(mode == LS_APPLY_FASTCONVOLUTION || mode == LS_APPLY_FFTCONVOLUTION, LS_ERR_INVALID,
               "ls_op2d_apply: unknown mode %d", mode);
    if (mode == LS_APPLY_FFTCONVOLUTION)
        LS_REQUIRE(op->n == op->m, LS_ERR_INVALID,
                   "FFTconvolution pads (ne,ne) and crops (n,n): square grids only (FastConvolution.jl:139-151)");
    LS_CUDA_TRY(cudaSetDevice(op->device));
    const size_t bytes = (size_t)op->n * op->m * sizeof(cd);
    if (memloc == LS_MEM_DEVICE) {
        return op->apply_dev(reinterpret_cast<const cd*>(b), reinterpret_cast<cd*>(y), mode);
    }
    LS_REQUIRE(memloc == LS_MEM_HOST, LS_ERR_INVALID, "ls_op2d_apply: unknown memloc %d", memloc);
    LS_CUDA_TRY(cudaMemcpyAsync(op->d_b, b, bytes, cudaMemcpyHostToDevice, op->stream));
    int rc = op->apply_dev(op->d_b, op->d_y, mode);
    if (rc) return rc;
    LS_CUDA_TRY(cudaMemcpyAsync(y, op->d_y, bytes, cudaMemcpyDeviceToHost, op->stream));
    LS_CUDA_TRY(cudaStreamSynchronize(op->stream));
    return LS_OK;
}

int ls_op2d_info(ls_handle h, int* route, int64_t* n_line, int64_t* m_line, int* padding_factor) {
    LS_REQUIRE(h, LS_ERR_INVALID, "ls_op2d_info: null handle");
    Op2DBase* op = reinterpret_cast<Op2DBase*>(h);
    LS_REQUIRE(op->kind == KIND_OP2D, LS_ERR_INVALID, "ls_op2d_info: not a 2-D operator handle");
    int r = 0, pf = 0;
    int64_t nl = 0, ml = 0;
    op->info(&r, &nl, &ml, &pf);
    if (route) *route = r;
    if (n_line) *n_line = nl;
    if (m_line) *m_line = ml;
    if (padding_factor) *padding_factor = pf;
    return LS_OK;
}

}  // extern "C"
