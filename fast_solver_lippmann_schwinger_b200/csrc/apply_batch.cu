// Several right-hand sides through one operator apply: ls_op_apply_batch and ls_op_batch_cols.
// The 2x-padded power-of-two routes (2-D route 0 and 2, single-GPU 3-D route 0 and 2) run a chunk of columns per launch
// of each pass (op2d.cu, op3d.cu: Op2D / Op3D::apply_cols_dev); every other operator handle serves the batch column by
// column through its single apply.  Either way every column has the bits of ls_op2d_apply / ls_op3d_apply of it.
#include "ls_common.cuh"
#include "op2d_base.cuh"
#include <algorithm>

using namespace ls;

extern "C" {

int ls_op_batch_cols(ls_handle h, int* cols) {
    LS_REQUIRE(h && cols, LS_ERR_INVALID, "ls_op_batch_cols: null argument");
    HandleBase* op = reinterpret_cast<HandleBase*>(h);
    LS_REQUIRE(op->kind == KIND_OP2D || op->kind == KIND_OP3D, LS_ERR_INVALID, "ls_op_batch_cols: not an operator handle");
    *cols = op->batch_cols();
    return LS_OK;
}

// Refusals before any CUDA call: arguments, then the device memory the work arrays of the chunk width still need.
int ls_op_apply_batch(ls_handle h, const ls_cdouble* b, int64_t ldb, ls_cdouble* y, int64_t ldy, int nrhs, int mode, int memloc) {
    const char* fn = "ls_op_apply_batch";
    LS_REQUIRE(nrhs >= 1, LS_ERR_INVALID, "%s: nrhs = %d, at least one right-hand side needed", fn, nrhs);
    LS_REQUIRE(h && b && y, LS_ERR_INVALID, "%s: null argument", fn);
    HandleBase* op = reinterpret_cast<HandleBase*>(h);
    LS_REQUIRE(op->kind == KIND_OP2D || op->kind == KIND_OP3D, LS_ERR_INVALID, "%s: not an operator handle", fn);
    LS_REQUIRE(op->dist_size() == 1, LS_ERR_UNSUPPORTED, "%s: a sharded operator (ls_op3d_create_dist) applies one column at a time", fn);
    LS_REQUIRE(mode == LS_APPLY_FASTCONVOLUTION || mode == LS_APPLY_FFTCONVOLUTION, LS_ERR_INVALID, "%s: unknown mode %d", fn, mode);
    if (op->kind == KIND_OP2D && mode == LS_APPLY_FFTCONVOLUTION) {
        const Op2DBase* o2 = static_cast<const Op2DBase*>(op);
        LS_REQUIRE(o2->n == o2->m, LS_ERR_INVALID,
                   "FFTconvolution pads (ne,ne) and crops (n,n): square grids only (FastConvolution.jl:139-151)");
    }
    LS_REQUIRE(memloc == LS_MEM_HOST || memloc == LS_MEM_DEVICE, LS_ERR_INVALID, "%s: unknown memloc %d", fn, memloc);
    const int64_t N = op->op_size();
    LS_REQUIRE(ldb >= N && ldy >= N, LS_ERR_INVALID, "%s: leading dimensions ldb = %ld, ldy = %ld must be >= N = %ld", fn,
               (long)ldb, (long)ldy, (long)N);
    {
        // y may alias b only column for column (same start, same leading dimension)
        const char* b0 = reinterpret_cast<const char*>(b);
        const char* y0 = reinterpret_cast<const char*>(y);
        const char* b1 = b0 + ((size_t)ldb * (nrhs - 1) + N) * sizeof(cd);
        const char* y1 = y0 + ((size_t)ldy * (nrhs - 1) + N) * sizeof(cd);
        const bool overlap = b0 < y1 && y0 < b1;
        LS_REQUIRE(!overlap || (b0 == y0 && ldb == ldy), LS_ERR_INVALID,
                   "%s: y overlaps b other than in place (y == b needs ldy == ldb; ldb = %ld, ldy = %ld)", fn, (long)ldb, (long)ldy);
    }
    const bool host = memloc == LS_MEM_HOST;
    const int w = std::min(nrhs, op->batch_cols());
    const size_t vb = (size_t)N * sizeof(cd);
    const size_t stage = host ? 2 * vb * (size_t)w : 0;
    LS_CUDA_TRY(cudaSetDevice(op->device));
    const size_t need = op->batch_bytes(w) + (op->bstage_bytes < stage ? stage : 0);
    if (need > 0) {
        size_t free_b = 0, total_b = 0;
        LS_CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
        LS_REQUIRE(need <= free_b, LS_ERR_NOMEM,
                   "%s: work arrays for %d columns at a time need %zu bytes of device memory; %zu of %zu bytes are free",
                   fn, w, need, free_b, total_b);
    }
    int rc;
    if ((rc = op->batch_reserve(w))) return rc;
    if (host && op->bstage_bytes < stage) {
        if (op->d_bstage) op->dfree(op->d_bstage);
        op->d_bstage = nullptr; op->bstage_bytes = 0;
        if ((rc = op->dmalloc((void**)&op->d_bstage, stage))) return rc;
        op->bstage_bytes = stage;
    }
    std::vector<const cd*> bp((size_t)w);
    std::vector<cd*> yp((size_t)w);
    if (!host) {
        for (int j0 = 0; j0 < nrhs; j0 += w) {
            const int k = std::min(w, nrhs - j0);
            for (int c = 0; c < k; ++c) {
                bp[c] = reinterpret_cast<const cd*>(b) + (size_t)(j0 + c) * ldb;
                yp[c] = reinterpret_cast<cd*>(y) + (size_t)(j0 + c) * ldy;
            }
            if ((rc = op->apply_cols_dev(bp.data(), yp.data(), k, mode))) return rc;
        }
        return LS_OK;
    }
    // host pointers: chunks of w columns through the staging buffer (b columns, then y columns)
    cd* sb = op->d_bstage;
    cd* sy = op->d_bstage + (size_t)w * N;
    for (int c = 0; c < w; ++c) { bp[c] = sb + (size_t)c * N; yp[c] = sy + (size_t)c * N; }
    const cd* hb = reinterpret_cast<const cd*>(b);
    cd* hy = reinterpret_cast<cd*>(y);
    for (int j0 = 0; j0 < nrhs; j0 += w) {
        const int k = std::min(w, nrhs - j0);
        LS_CUDA_TRY(cudaMemcpy2DAsync(sb, vb, hb + (size_t)j0 * ldb, (size_t)ldb * sizeof(cd), vb, (size_t)k,
                                      cudaMemcpyHostToDevice, op->stream));
        if ((rc = op->apply_cols_dev(bp.data(), yp.data(), k, mode))) return rc;
        LS_CUDA_TRY(cudaMemcpy2DAsync(hy + (size_t)j0 * ldy, (size_t)ldy * sizeof(cd), sy, vb, vb, (size_t)k,
                                      cudaMemcpyDeviceToHost, op->stream));
        LS_CUDA_TRY(cudaStreamSynchronize(op->stream));
    }
    return LS_OK;
}

}  // extern "C"
