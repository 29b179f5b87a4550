// Shared host-side helpers for libls_cuda.so (error reporting, handle header, tables).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdarg>
#include <cmath>
#include <string>
#include <vector>
#include "../../include/ls_cuda.h"
#include "fft_engine.cuh"
#include <nccl.h>

namespace ls {

using lsfft::cd;

void set_error(const char* fmt, ...);

#define LS_CUDA_TRY(expr)                                                                    \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            ls::set_error("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__,               \
                          cudaGetErrorString(_e));                                           \
            return LS_ERR_CUDA;                                                              \
        }                                                                                    \
    } while (0)

#define LS_REQUIRE(cond, code, ...)                                                          \
    do {                                                                                     \
        if (!(cond)) {                                                                       \
            ls::set_error(__VA_ARGS__);                                                      \
            return (code);                                                                   \
        }                                                                                    \
    } while (0)

enum HandleKind : uint32_t { KIND_OP2D = 0x4c533244, KIND_OP3D = 0x4c533344, KIND_SPM = 0x4c53534d,
                             KIND_VEC = 0x4c535643 };

struct HandleBase {
    uint32_t kind = 0;
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    int64_t launches = 0;
    cd* stage_b = nullptr; cd* stage_y = nullptr;   // device staging for host-pointer applies (lazily allocated)
    std::vector<void*> dev_allocs;    // everything cudaMalloc'ed by the handle
    std::vector<void*> host_allocs;   // pinned staging

    virtual int64_t op_size() const { return -1; }
    // operator handles: y = M*b (mode 0) / FFTconvolution (mode 1) on device pointers, on `stream`
    virtual int apply_dev(const cd* b, cd* y, int mode) {
        (void)b; (void)y; (void)mode;
        set_error("handle is not an operator");
        return LS_ERR_INVALID;
    }

    // Several columns per apply (ls_op_apply_batch, ls_gmres_batch).  batch_cols: the chunk width of one multi-column
    // apply (1: the handle serves a batch column by column through apply_dev); batch_bytes: device bytes still to
    // allocate before a chunk of ncol columns can run; batch_reserve: allocates them; apply_cols_dev: ncol <= the
    // reserved width columns b[c] -> y[c], each with the bits of apply_dev of that column.
    virtual int batch_cols() const { return 1; }
    virtual size_t batch_bytes(int ncol) const { (void)ncol; return 0; }
    virtual int batch_reserve(int ncol) { (void)ncol; return LS_OK; }
    virtual int apply_cols_dev(const cd* const* b, cd* const* y, int ncol, int mode) {
        for (int c = 0; c < ncol; ++c) {
            int rc = apply_dev(b[c], y[c], mode);
            if (rc) return rc;
        }
        return LS_OK;
    }
    // count columns in chunks of batch_cols(); the chunk width must be reserved
    int apply_list_dev(const cd* const* b, cd* const* y, int count, int mode) {
        const int w = batch_cols();
        for (int j = 0; j < count; j += w) {
            int rc = apply_cols_dev(b + j, y + j, count - j < w ? count - j : w, mode);
            if (rc) return rc;
        }
        return LS_OK;
    }
    cd* d_bstage = nullptr; size_t bstage_bytes = 0;   // ls_op_apply_batch with host pointers: one chunk of b and y

    // sharded operators expose their communicator so that Krylov reductions can all-reduce on it
    virtual ncclComm_t nccl_comm() const { return nullptr; }
    virtual int dist_rank() const { return 0; }
    virtual int dist_size() const { return 1; }

    // optional per-phase CUDA-event profiling (bench roofline of the dominant kernel)
    bool profiling = false;
    struct PhaseEv { int phase; cudaEvent_t a, b; };
    std::vector<PhaseEv> phase_events;
    void phase_begin(int phase, cudaStream_t on = nullptr) {
        if (!profiling) return;
        PhaseEv pe; pe.phase = phase;
        cudaEventCreate(&pe.a); cudaEventCreate(&pe.b);
        cudaEventRecord(pe.a, on ? on : stream);
        phase_events.push_back(pe);
    }
    void phase_end(cudaStream_t on = nullptr) {
        if (!profiling) return;
        cudaEventRecord(phase_events.back().b, on ? on : stream);
    }

    int init_base(uint32_t k) {
        kind = k;
        LS_CUDA_TRY(cudaGetDevice(&device));
        LS_CUDA_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        LS_CUDA_TRY(cudaEventCreate(&ev0));
        LS_CUDA_TRY(cudaEventCreate(&ev1));
        return LS_OK;
    }
    int dmalloc(void** p, size_t bytes) {
        cudaError_t e = cudaMalloc(p, bytes);
        if (e == cudaErrorMemoryAllocation) {
            cudaGetLastError();
            set_error("out of device memory allocating %zu bytes", bytes);
            return LS_ERR_NOMEM;
        }
        LS_CUDA_TRY(e);
        dev_allocs.push_back(*p);
        return LS_OK;
    }
    int dupload(void** p, const void* host, size_t bytes) {
        int rc = dmalloc(p, bytes);
        if (rc) return rc;
        LS_CUDA_TRY(cudaMemcpyAsync(*p, host, bytes, cudaMemcpyHostToDevice, stream));
        LS_CUDA_TRY(cudaStreamSynchronize(stream));
        return LS_OK;
    }
    void dfree(void* p) {
        if (!p) return;
        for (size_t i = 0; i < dev_allocs.size(); ++i)
            if (dev_allocs[i] == p) { dev_allocs.erase(dev_allocs.begin() + i); break; }
        cudaFree(p);
    }
    virtual ~HandleBase() {
        if (stream) cudaStreamSynchronize(stream);
        for (auto& pe : phase_events) { cudaEventDestroy(pe.a); cudaEventDestroy(pe.b); }
        for (void* p : dev_allocs) cudaFree(p);
        for (void* p : host_allocs) cudaFreeHost(p);
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (stream) cudaStreamDestroy(stream);
    }
};

inline bool fft_size_supported(long n) {
    return n == 64 || n == 128 || n == 256 || n == 512 || n == 1024 || n == 2048 || n == 4096;
}

// line length of the zero-embedded routes (LS_FLAG_EMBED): nextpow2(n), at least 64 (the smallest engine size)
inline long embed_len(long n) {
    long p = 64;
    while (p < n) p *= 2;
    return p;
}

// slot -> frequency map of the forward engine for size N (mirrors Stage<>::addr logic)
std::vector<int> slot_freq(int N);
// exp(-2 pi i k / N), k < count, evaluated in long double
std::vector<cd> twiddle_table(long N, long count);
// modulation table: mod[(r-1)*N + j] = exp(-2 pi i r j / (4N)), r = 1..3
std::vector<cd> modulation_table(long N);

// per-size engine table (fft_engine.cuh EngTab): q_t, s_t, stage-1 twiddles
std::vector<cd> engine_table(int N);

int upload(void** dptr, const void* host, size_t bytes, cudaStream_t s);

}  // namespace ls
