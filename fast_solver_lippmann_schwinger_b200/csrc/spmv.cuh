// Sparse-matrix handle shared by spmv.cu and krylov.cu (the GMRES driver applies As on its own stream).
#pragma once
#include "ls_common.cuh"

namespace ls {

enum { SPM_FORMAT_CSR = 0, SPM_FORMAT_STENCIL = 1 };

struct SpM : HandleBase {
    long nrows = 0, ncols = 0, nnz = 0;
    int format = SPM_FORMAT_CSR;
    // CSR
    int lanes_per_row = 8;
    int* d_rowptr = nullptr;
    int* d_col = nullptr;
    cd* d_val = nullptr;
    // stencil classes: class id per row + per-class (offset, value) lists
    int ncls = 0, nent = 0;
    unsigned char* d_cls = nullptr;
    int* d_cls_ptr = nullptr;
    int* d_cls_off = nullptr;
    cd* d_cls_val = nullptr;
    cd* d_x = nullptr; cd* d_y = nullptr;   // staging for host-pointer calls
    // row slab of a matrix sharded like the 3-D operator (ls_spm_create_dist): columns are stored relative to the
    // window [row0 - halo, row0 + nrows + halo); every mv gathers the two halo pieces of x from the z-neighbours
    // (grouped ncclSend/ncclRecv on the operator's communicator, borrowed) into d_xext = [halo | local x | halo].
    long halo = 0;
    int rank = 0, P = 1;
    ncclComm_t comm = nullptr;
    cd* d_xext = nullptr;
    long x_len() const { return halo > 0 ? nrows : ncols; }      // length of the caller's x
    // y <- alpha*A*x + beta*y on device pointers, enqueued on stream s
    int mv_dev(cd alpha, const cd* x, cd beta, cd* y, cudaStream_t s);
};

// Device-resident factorisation of the sparsified system matrix Msp (msp.cu): what `MspInv \\ .` of
// preconditioner.jl:138,159 becomes when the whole preconditioned GMRES loop stays on the GPU.
constexpr uint32_t KIND_MSP = 0x4c534d53;
struct MspBase : HandleBase {
    long n = 0;
    int launches_per_solve = 0;
    // out <- Msp^-1 rhs on device pointers (out may alias rhs), enqueued on stream s
    virtual int solve_dev(const cd* rhs, cd* out, cudaStream_t s) = 0;
    // the same for nrhs column-major columns (leading dimensions ldr / ldx; out may alias rhs when ldx == ldr).
    // batch_bytes: device memory a batch of nrhs columns still has to allocate (work arrays kept per chunk width, with
    // `subsets` also those of every smaller column count, with `host` the staging of host-pointer calls); batch_reserve
    // allocates it.  solve_batch_dev needs batch_reserve first.
    virtual size_t batch_bytes(int nrhs, bool host, bool subsets) const = 0;
    virtual int batch_reserve(int nrhs, bool host, bool subsets) = 0;
    virtual int solve_batch_dev(const cd* rhs, long ldr, cd* out, long ldx, int nrhs, cudaStream_t s) = 0;
};

}  // namespace ls
