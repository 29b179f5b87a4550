// 3-D Lippmann-Schwinger operator  y = b + omega^2 * G (nu .* b)  on one B200 (slab-ready layout).
// Stands behind struct FastM3D, its `*` and FFTconvolution (reference FastConvolution3D.jl:7-63).
// Five launches per apply (pruned zero padding in every dimension, see line_kernels.cuh; padding
// factor nr = 2 by default - the compact spectrum built at create time - or 4 with LS_FLAG_PAD4;
// pn = nr*n etc.):
//   P1 k_fwd_pruned<n,A>  x lines (contiguous)   b,nu [n m l]      -> A1 [pn m l]
//   P2 k_fwd_pruned<m,B>  y lines (8 x-slots/warp quarter)  A1     -> A2 [pn pm l]
//   P3 k_mid_fused <l,B>  z lines, fused spectrum multiply, in place on A2 (reads G [pn pm pl])
//   P4 k_inv_pruned<m,B>  y lines                 A2               -> C1 [pn m l]   (reuses A1)
//   P5 k_inv_pruned<n,A>  x lines + combine       C1, b            -> y
// HBM bytes per apply: 568*N with nr = 2 (spectrum 128*N), 2360*N with nr = 4 (SURVEY.md section 8(d)).
//
// Multi-GPU (one process per GPU, P = 2/4/8 ranks): the grid is split into z slabs (l/P planes per
// rank, a contiguous range of the vector).  P1 runs on the local planes and writes its output
// already grouped by destination rank; one NCCL all-to-all re-slabs the (most pruned) pn x m x l
// array along the x-slot axis; P2-P4 run on the rank's pn/P x-slots against its slab of the
// spectrum; a second all-to-all brings the result back to z slabs for P5.  Neither exchange needs
// a pack or unpack pass: both sides read/write the exchange buffers in place (slot_off()).
// All-to-all volume per rank and direction: 16*nr*N*(P-1)/P^2 bytes.
//
// Zero embedding (LS_FLAG_EMBED, any n = m, l <= 512, one GPU or sharded): the same five launches on the lines of the
// power-of-two grid n' = max(64, nextpow2(n)), l' likewise, with the kernel's lags (-n, n)^2 x (-l, l) extracted at
// create time (op3d_embed.cu).  The arrays keep the real extents wherever a pass does not transform along them
// (A1: 2n' x m x l, A2: 2n' x 2m' x l'), so the exchanges move 2n' x m x l.  Masked passes:
//   P1 reads n of n' points; P2 reads m of m' points and writes zero lines for the planes l..l'-1, which P3 (in
//   place, all l' points) would otherwise take from the previous apply; P4 writes m points of planes < l; P5 writes
//   n points and stages b with stride n.
#include "ls_common.cuh"
#include "line_kernels.cuh"
#include "dist.cuh"
#include "gv_spectrum.cuh"
#include <cerrno>
#include <chrono>
#include <climits>

using namespace ls;
using namespace lsk;

namespace {

// columns per multi-column apply (ls_op_apply_batch) of the single-GPU 2x-padded routes.  Measured on B200 (1000 W,
// profiles/r5_apply_batch.log, ms per column at K = 1 / 4): 48^3 embedded 0.045 / 0.028, 64^3 0.048 / 0.032, 256^3
// 2.03 / 1.94; at 512^3 20.1 / 19.9 lies inside the run-to-run spread (19.3 - 20.3) while the three extra columns
// would hold 38 GB of work arrays, so grids with 512-point lines go column by column.
constexpr int BATCH_COLS3 = 4;

struct Op3D : HandleBase {
    long n = 0, m = 0, l = 0, ne = 0, me = 0, le = 0;
    // LS_FLAG_EMBED: lines of ln x lm x ll points carry the n x m x l grid (ln = n, lm = m, ll = l otherwise)
    bool embed = false;
    long ln = 0, lm = 0, ll = 0;
    int nr = 4;                        // padding factor used by the applies (4: literal, 2: compact - see op2d.cu)
    long pn = 0, pm = 0, pl = 0;       // padded sizes nr*ln, nr*lm, nr*ll
    int P = 1, rank = 0;
    long nel = 0, lloc = 0;            // x-slots (pn/P) / z-planes (l/P) owned by this rank
    ncclComm_t comm = nullptr;
    double omega = 0;
    double* d_nu = nullptr;            // local z slab
    cd* d_G = nullptr;                 // [unit = (sxl + nel*sy)/8][rz][slot_z][8]  scaled by 1/(ne me le)
    cd *d_TABn = nullptr, *d_TABm = nullptr, *d_TABl = nullptr;
    // x-slot chunks: the rank's nel x-slots are handled as Cx chunks of nelc; the exchange buffers and the
    // spectrum are chunk-major, so that chunk c's transposes (on cstream) overlap chunk c+-1's P2-P4.
    int Cx = 1;
    long nelc = 0;
    cd* d_A1 = nullptr;                // P1 output / P5 input: [chunk][dest rank][nelc][m][lloc]
    cd* d_A1T = nullptr;               // re-slabbed: [chunk][nelc x m x l]  (P > 1 only)
    cd* d_A2 = nullptr;                // nelc x pm x l (one chunk, reused)
    cd* d_b = nullptr; cd* d_y = nullptr;
    cudaStream_t cstream = nullptr;    // high-priority stream of the exchanges (P > 1)
    // Copy-engine exchange (default for P > 1): both exchange buffers are exported with cudaIpcGetMemHandle, and a
    // transpose is P-1 cudaMemcpyAsync pushes of contiguous blocks straight into the peers' receive buffers (DMA
    // engines over NVLink: no SM, no staging) closed by a one-element all-reduce, after which every push into this
    // rank's buffer has landed.  LS_OP3D_XCHG=nccl keeps the grouped ncclSend/ncclRecv all-to-all (same bits).
    bool ce_exchange = false;
    std::vector<cd*> peerA1, peerA1T;  // rank q's d_A1 / d_A1T mapped into this process (own entries: the local pointers)
    double* d_bar = nullptr;
    // Completion signalling without a collective (default, LS_OP3D_SYNC=barrier keeps the all-reduce): after its pushes
    // a rank stores the exchange's sequence number into flags[dir][rank] of every peer (one small kernel, system-scope
    // stores over NVLink); the receiver's wait kernel spins until all P entries of flags[dir] have reached it.
    bool flag_sync = true;
    unsigned* d_flags = nullptr;             // [2][P] on this rank
    std::vector<unsigned*> peerFlags;        // rank q's d_flags mapped here
    unsigned** d_peerFlags = nullptr;        // the same table on the device
    unsigned seq[2] = {0, 0};                // exchanges issued so far per direction
    cudaEvent_t evP1 = nullptr, evDone = nullptr;
    std::vector<cudaEvent_t> evIn, evOut;
    int64_t op_size() const override { return n * m * lloc; }
    int apply_dev(const cd* b, cd* y, int mode) override;
    // ls_op_apply_batch: A1 and A2 hold `cols` columns, a1cs / a2cs elements apart (single GPU, 2x padding)
    int cols = 1;
    long a1cs() const { return pn * m * lloc; }
    long a2cs() const { return nelc * pm * ll; }
    int batch_cols() const override { return (P == 1 && nr == 2 && ln < 512 && ll < 512) ? BATCH_COLS3 : 1; }
    size_t batch_bytes(int ncol) const override { return ncol > cols ? (size_t)ncol * (a1cs() + a2cs()) * sizeof(cd) : 0; }
    int batch_reserve(int ncol) override;
    int apply_cols_dev(const cd* const* b, cd* const* y, int ncol, int mode) override;
    ncclComm_t nccl_comm() const override { return comm; }
    int dist_rank() const override { return rank; }
    int dist_size() const override { return P; }
    ~Op3D() override {
        if (stream) cudaStreamSynchronize(stream);
        if (cstream) cudaStreamSynchronize(cstream);
        for (int q = 0; q < (int)peerA1.size(); ++q) {
            if (q == rank) continue;
            if (peerA1[q]) cudaIpcCloseMemHandle(peerA1[q]);
            if (peerA1T[q]) cudaIpcCloseMemHandle(peerA1T[q]);
            if (q < (int)peerFlags.size() && peerFlags[q]) cudaIpcCloseMemHandle(peerFlags[q]);
        }
        if (comm) ncclCommDestroy(comm);
        for (auto ev : evIn) cudaEventDestroy(ev);
        for (auto ev : evOut) cudaEventDestroy(ev);
        if (evP1) cudaEventDestroy(evP1);
        if (evDone) cudaEventDestroy(evDone);
        if (cstream) cudaStreamDestroy(cstream);
    }
};

inline int lines_b(long N) { return N == 512 ? lines_b512 : 8; }      // LinesB<N> of the mode-B kernels (fft_engine.cuh)

struct GenParams {
    int lb = 8;         // x-adjacent z lines interleaved per spectrum unit
    long n, m, l, ne, me, le;
    long nel, sx0;      // x-slot slab of this rank
    double dk;          // 2 pi / Lp
    double L, k;        // truncation radius, wave number
    double eLk_re, eLk_im;
    double scale;
};

__device__ __forceinline__ cd gtrunc3d(double s, const GenParams& p) {
    return gtrunc3d_eval(s, p.L, p.k, p.eLk_re, p.eLk_im);
}

// fills the device spectrum in its final layout, either by gathering from the reference-ordered
// array `gin` (ne x me x le, centred) or by evaluating the Greengard-Vico formula.
__global__ void k_fill_g3d(const cd* __restrict__ gin, cd* __restrict__ gout, const int* __restrict__ fx,
                           const int* __restrict__ fy, const int* __restrict__ fz, GenParams p) {
    const long total = p.nel * p.me * p.le;
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const long lam = idx % p.lb;
        long q = idx / p.lb;
        const long sz = q % p.l; q /= p.l;
        const long rz = q & 3;
        const long unit = q >> 2;
        const long Lidx = unit * p.lb + lam;
        const long sx = p.sx0 + Lidx % p.nel, sy = Lidx / p.nel;
        const long kx = 4L * fx[sx % p.n] + sx / p.n;
        const long ky = 4L * fy[sy % p.m] + sy / p.m;
        const long kz = 4L * fz[sz] + rz;
        const long ix = (kx + p.ne / 2) % p.ne, iy = (ky + p.me / 2) % p.me, iz = (kz + p.le / 2) % p.le;
        cd v;
        if (gin != nullptr) {
            v = gin[ix + p.ne * (iy + p.me * iz)];
        } else {
            v = gtrunc3d(gv_radius(p.dk, ix, iy, iz, p.ne, p.me, p.le), p);
        }
        gout[idx] = make_double2(v.x * p.scale, v.y * p.scale);
    }
}

#define LS3_DISPATCH(N_, CALL)                                          \
    switch (N_) {                                                       \
        case 64:  e = CALL(64); break;                                  \
        case 128: e = CALL(128); break;                                 \
        case 256: e = CALL(256); break;                                 \
        case 512: e = CALL(512); break;                                 \
        default: set_error("unsupported 3-D size %ld", (long)(N_)); return LS_ERR_UNSUPPORTED; \
    }

// all-to-all of equal contiguous blocks (grouped ncclSend/ncclRecv over NVLink)
int all_to_all(Op3D* op, const cd* send, cd* recv, long blk_elems, cudaStream_t on = nullptr) {
    if (!on) on = op->stream;
    ncclResult_t r = ncclGroupStart();
    for (int q = 0; q < op->P && r == ncclSuccess; ++q) {
        r = ncclSend(send + (long)q * blk_elems, (size_t)blk_elems * 2, ncclDouble, q, op->comm, on);
        if (r == ncclSuccess)
            r = ncclRecv(recv + (long)q * blk_elems, (size_t)blk_elems * 2, ncclDouble, q, op->comm, on);
    }
    ncclResult_t r2 = ncclGroupEnd();
    if (r == ncclSuccess) r = r2;
    if (r != ncclSuccess) {
        set_error("NCCL all-to-all failed: %s", ncclGetErrorString(r));
        return LS_ERR_NCCL;
    }
    return LS_OK;
}

// The same all-to-all on the copy engines: block q of `send` goes to block `rank` of rank q's buffer `peer[q]`
// (offset `off` = chunk base in both); step s pushes to rank (rank + s) % P, so every rank receives from exactly one
// source per step.  The closing all-reduce is the completion barrier: a rank leaves it only after every rank has
// entered it, i.e. after every push (stream-ordered before the sender's all-reduce) has completed.
__global__ void k_xchg_signal(unsigned* const* peer_flags, int P, int slot, unsigned seq) {
    const int q = threadIdx.x;
    if (q < P) {
        __threadfence_system();
        *reinterpret_cast<volatile unsigned*>(peer_flags[q] + slot) = seq;
    }
}
__global__ void k_xchg_wait(const unsigned* flags, int P, unsigned seq) {
    const int q = threadIdx.x;
    if (q < P) {
        const volatile unsigned* f = flags + q;
        const long long t0 = clock64();
        while ((int)(*f - seq) < 0) {
            if (clock64() - t0 > 20000000000LL) __trap();      // ~10 s: a peer died - fail instead of hanging the GPU
        }
    }
    __threadfence_system();
}

int exchange_ce(Op3D* op, const cd* send, const std::vector<cd*>& peer, long off, long blk_elems, cudaStream_t on, int dir) {
    const size_t bytes = (size_t)blk_elems * sizeof(cd);
    for (int st = 0; st < op->P; ++st) {
        const int q = (op->rank + st) % op->P;
        LS_CUDA_TRY(cudaMemcpyAsync(peer[q] + off + (long)op->rank * blk_elems, send + off + (long)q * blk_elems, bytes,
                                    cudaMemcpyDeviceToDevice, on));
    }
    if (op->flag_sync) {
        const unsigned sq = ++op->seq[dir];
        k_xchg_signal<<<1, 32, 0, on>>>(op->d_peerFlags, op->P, dir * op->P + op->rank, sq);
        k_xchg_wait<<<1, 32, 0, on>>>(op->d_flags + dir * op->P, op->P, sq);
        LS_CUDA_TRY(cudaPeekAtLastError());
        return LS_OK;
    }
    ncclResult_t r = ncclAllReduce(op->d_bar, op->d_bar, 1, ncclDouble, ncclSum, op->comm, on);
    if (r != ncclSuccess) { set_error("exchange barrier failed: %s", ncclGetErrorString(r)); return LS_ERR_NCCL; }
    return LS_OK;
}

// maps the peers' exchange buffers into this process (all ranks of one box; handles travel by ncclAllGather)
int setup_ce_exchange(Op3D* op) {
    const int P = op->P;
    struct Pair { cudaIpcMemHandle_t a1, a1t, fl; };
    static_assert(sizeof(Pair) == 192, "three 64-byte IPC handles");
    Pair mine;
    {
        // an allocation of its own (2 MiB: never packed with other small buffers), since the IPC handle maps whole allocations
        int rc0 = op->dmalloc((void**)&op->d_flags, (size_t)2 << 20);
        if (rc0) return rc0;
        LS_CUDA_TRY(cudaMemset(op->d_flags, 0, (size_t)2 << 20));
    }
    LS_CUDA_TRY(cudaIpcGetMemHandle(&mine.a1, op->d_A1));
    LS_CUDA_TRY(cudaIpcGetMemHandle(&mine.a1t, op->d_A1T));
    LS_CUDA_TRY(cudaIpcGetMemHandle(&mine.fl, op->d_flags));
    char *d_send = nullptr, *d_recv = nullptr;
    int rc;
    if ((rc = op->dmalloc((void**)&d_send, sizeof(Pair)))) return rc;
    if ((rc = op->dmalloc((void**)&d_recv, sizeof(Pair) * P))) return rc;
    if ((rc = op->dmalloc((void**)&op->d_bar, sizeof(double)))) return rc;
    LS_CUDA_TRY(cudaMemsetAsync(op->d_bar, 0, sizeof(double), op->stream));
    LS_CUDA_TRY(cudaMemcpyAsync(d_send, &mine, sizeof(Pair), cudaMemcpyHostToDevice, op->stream));
    ncclResult_t r = ncclAllGather(d_send, d_recv, sizeof(Pair), ncclChar, op->comm, op->stream);
    if (r != ncclSuccess) { set_error("IPC handle all-gather failed: %s", ncclGetErrorString(r)); return LS_ERR_NCCL; }
    std::vector<Pair> all((size_t)P);
    LS_CUDA_TRY(cudaMemcpyAsync(all.data(), d_recv, sizeof(Pair) * P, cudaMemcpyDeviceToHost, op->stream));
    LS_CUDA_TRY(cudaStreamSynchronize(op->stream));
    op->dfree(d_send); op->dfree(d_recv);
    op->peerA1.assign((size_t)P, nullptr);
    op->peerA1T.assign((size_t)P, nullptr);
    op->peerA1[op->rank] = op->d_A1;
    op->peerA1T[op->rank] = op->d_A1T;
    op->peerFlags.assign((size_t)P, nullptr);
    op->peerFlags[op->rank] = op->d_flags;
    for (int q = 0; q < P; ++q) {
        if (q == op->rank) continue;
        void *p1 = nullptr, *p2 = nullptr, *p3 = nullptr;
        LS_CUDA_TRY(cudaIpcOpenMemHandle(&p1, all[q].a1, cudaIpcMemLazyEnablePeerAccess));
        op->peerA1[q] = (cd*)p1;
        LS_CUDA_TRY(cudaIpcOpenMemHandle(&p2, all[q].a1t, cudaIpcMemLazyEnablePeerAccess));
        op->peerA1T[q] = (cd*)p2;
        LS_CUDA_TRY(cudaIpcOpenMemHandle(&p3, all[q].fl, cudaIpcMemLazyEnablePeerAccess));
        op->peerFlags[q] = (unsigned*)p3;
    }
    if ((rc = op->dupload((void**)&op->d_peerFlags, op->peerFlags.data(), (size_t)P * sizeof(unsigned*)))) return rc;
    { const char* sv = getenv("LS_OP3D_SYNC"); op->flag_sync = !(sv && strcmp(sv, "barrier") == 0); }
    op->ce_exchange = true;
    return LS_OK;
}

// b[c] -> y[c], c < ncol (ncol = 1 unless single GPU): column c of A1 / A2 starts c*a1cs / c*a2cs elements in
int apply_device3(Op3D* op, const cd* const* b, cd* const* y, int ncol, int mode) {
    cudaError_t e = cudaSuccess;
    cudaStream_t s = op->stream, sc = op->cstream;
    const long n = op->n, m = op->m, l = op->l, me = op->pm, nel = op->nel, lloc = op->lloc, nelc = op->nelc;
    const long ln = op->ln, lm = op->lm, ll = op->ll;
    const bool embed = op->embed;
    const int nr = op->nr, Cx = op->Cx, P = op->P;
    const bool full = (mode == LS_APPLY_FASTCONVOLUTION);
    const long blk = nelc * m * lloc;                // elements exchanged with each peer per chunk
    const long cstride = (long)P * blk;              // one chunk of the exchange buffers (= nelc*m*l)
    int shc = 0, shr = 0;
    while ((1L << shc) < nelc) ++shc;
    while ((1L << shr) < nel) ++shr;
    const long a1cs = op->a1cs(), a2cs = op->a2cs();
    // P1: x lines (j, p_loc): in b[n*line + i]; slot sx -> rank q = sx/nel, chunk c = (sx%nel)/nelc:
    //     A1[c*cstride + q*blk + nelc*line + sx%nelc]
    //     embed: m*lloc need not fill the last CTA; its surplus lines wrap (ldim0) onto lines 0.. and write the same bits
    //     there (zeros would race with the real lines, and past the block they would land in the next one)
    {
        LineAddr la{1L << 40, n, 0, 1, nelc, 0, 1};
        la.split_shift = shc; la.split_stride = cstride; la.split2_shift = shr; la.split2_stride = blk; la.nr = nr;
        if (embed) { la.ldim0 = m * lloc; la.mask_pts = (int16_t)n; la.mask_lines = INT_MAX; }
        ColPtrs cp{};
        for (int c = 0; c < ncol; ++c) { cp.in[c] = b[c]; cp.out[c] = op->d_A1 + c * a1cs; }
        op->phase_begin(0);
#define C1(N) (embed ? launch_fwd_cols<N, false, true>(s, m * lloc, cp, ncol, full ? op->d_nu : nullptr, op->d_TABn, la) \
                     : launch_fwd_cols<N, false>(s, m * lloc, cp, ncol, full ? op->d_nu : nullptr, op->d_TABn, la))
        LS3_DISPATCH(ln, C1);
        op->phase_end(); op->launches++;
        LS_CUDA_TRY(e);
    }
    if (P > 1) {      // inbound transposes, chunk by chunk, on the exchange stream
        LS_CUDA_TRY(cudaEventRecord(op->evP1, s));
        LS_CUDA_TRY(cudaStreamWaitEvent(sc, op->evP1, 0));
        for (int c = 0; c < Cx; ++c) {
            op->phase_begin(5, sc);
            int rc = op->ce_exchange ? exchange_ce(op, op->d_A1, op->peerA1T, c * cstride, blk, sc, 0)
                                     : all_to_all(op, op->d_A1 + c * cstride, op->d_A1T + c * cstride, blk, sc);
            op->phase_end(sc);
            if (rc) return rc;
            LS_CUDA_TRY(cudaEventRecord(op->evIn[c], sc));
        }
    }
    for (int c = 0; c < Cx; ++c) {
        const cd* a1t = (P > 1 ? op->d_A1T : op->d_A1) + c * cstride;     // chunk c re-slabbed: nelc x m x l
        cd* c1t = (P > 1 ? op->d_A1T : op->d_A1) + c * cstride;
        const cd* Gc = op->d_G + (long)c * nelc * me * op->pl;
        if (P > 1) LS_CUDA_TRY(cudaStreamWaitEvent(s, op->evIn[c], 0));
        // P2: y lines (sxc, p): in A1T[sxc + nelc*m*p + nelc*j]; out A2[sxc + nelc*me*p + nelc*sy]
        //     embed: the plane index p is the slowest part of the line index, so the lines of planes l..l'-1 are the
        //     lines >= nelc*l: they are written as zeros
        {
            LineAddr la{nelc, 1, nelc * m, nelc, 1, nelc * me, nelc};
            la.nr = nr;
            if (embed) { la.mask_pts = (int16_t)m; la.mask_lines = (int)(nelc * l); }
            ColPtrs cp{};
            for (int c = 0; c < ncol; ++c) { cp.in[c] = a1t + c * a1cs; cp.out[c] = op->d_A2 + c * a2cs; }
#define C2(N) (embed ? launch_fwd_cols<N, true, true>(s, nelc * ll, cp, ncol, nullptr, op->d_TABm, la) \
                     : launch_fwd_cols<N, true>(s, nelc * l, cp, ncol, nullptr, op->d_TABm, la))
            op->phase_begin(1);
            LS3_DISPATCH(lm, C2);
            op->phase_end(); op->launches++;
            LS_CUDA_TRY(e);
        }
        // P3: z lines L = sxc + nelc*sy: point p at A2[L + nelc*me*p], in place
        {
            LineAddr la{1L << 40, 1, 0, nelc * me, 1, 0, nelc * me};
            la.nr = nr;
            op->phase_begin(2);
#define C3(N) launch_mid<N, true>(s, nelc * me, op->d_A2, op->d_A2, Gc, op->d_TABl, la, ncol, a2cs)
            LS3_DISPATCH(ll, C3);
            op->phase_end(); op->launches++;
            LS_CUDA_TRY(e);
        }
        // P4: inverse y lines (sxc, p): slots at A2[sxc + nelc*me*p + nelc*sy]; out C1T[sxc + nelc*m*p + nelc*j].
        //     P4 and P5 stage their next slot block (and b) in shared memory by cp.async (256^3: 1.94 -> 1.80 ms)
        //     embed: planes < l only (the surplus lines of the last CTA read planes >= l and are not written)
        {
            LineAddr la{nelc, 1, nelc * me, nelc, 1, nelc * m, nelc};
            la.nr = nr;
            if (embed) { la.mask_pts = (int16_t)m; la.mask_lines = (int)(nelc * l); }
            ColPtrs cp{};
            for (int c = 0; c < ncol; ++c) { cp.in[c] = op->d_A2 + c * a2cs; cp.out[c] = c1t + c * a1cs; }
            op->phase_begin(3);
#define C4(N) (embed ? launch_inv_cols<N, true, true, true>(s, nelc * l, cp, ncol, op->d_TABm, 1.0, la) \
                     : launch_inv_cols<N, true, true>(s, nelc * l, cp, ncol, op->d_TABm, 1.0, la))
            LS3_DISPATCH(lm, C4);
            op->phase_end(); op->launches++;
            LS_CUDA_TRY(e);
        }
        if (P > 1) {  // outbound transpose of this chunk (queued behind the inbound ones on the exchange stream)
            LS_CUDA_TRY(cudaEventRecord(op->evOut[c], s));
            LS_CUDA_TRY(cudaStreamWaitEvent(sc, op->evOut[c], 0));
            op->phase_begin(6, sc);
            int rc = op->ce_exchange ? exchange_ce(op, op->d_A1T, op->peerA1, c * cstride, blk, sc, 1)
                                     : all_to_all(op, op->d_A1T + c * cstride, op->d_A1 + c * cstride, blk, sc);
            op->phase_end(sc);
            if (rc) return rc;
        }
    }
    if (P > 1) {
        LS_CUDA_TRY(cudaEventRecord(op->evDone, sc));
        LS_CUDA_TRY(cudaStreamWaitEvent(s, op->evDone, 0));
    }
    // P5: inverse x lines + combine (staged like P4); slot sx of line (j, p_loc) addressed as in P1
    //     embed: the surplus lines of the last CTA wrap like P1's (their reads stay inside A1) and are not written
    {
        LineAddr la{1L << 40, nelc, 0, 1, n, 0, 1};
        la.split_shift = shc; la.split_stride = cstride; la.split2_shift = shr; la.split2_stride = blk; la.nr = nr;
        if (embed) { la.ldim0 = m * lloc; la.mask_pts = (int16_t)n; la.mask_lines = (int)(m * lloc); }
        ColPtrs cp{};
        for (int c = 0; c < ncol; ++c) { cp.in[c] = op->d_A1 + c * a1cs; cp.b[c] = full ? b[c] : nullptr; cp.out[c] = y[c]; }
        op->phase_begin(4);
#define C5(N) (embed ? launch_inv_cols<N, false, true, true>(s, m * lloc, cp, ncol, op->d_TABn, full ? op->omega * op->omega : 1.0, la) \
                     : launch_inv_cols<N, false, true>(s, m * lloc, cp, ncol, op->d_TABn, full ? op->omega * op->omega : 1.0, la))
        LS3_DISPATCH(ln, C5);
        op->phase_end(); op->launches++;
        LS_CUDA_TRY(e);
    }
    return LS_OK;
}

// chunk-major order of the spectrum units: unit (i, sy) of chunk c, i = x-slot group inside the chunk
__global__ void k_permute_units(const cd* __restrict__ src, cd* __restrict__ dst, long ug, long ugc, long pm, long unit_elems) {
    // ug = nel/8 x-slot groups per slab row, ugc = nelc/8 per chunk row
    const long nunits = ug * pm;
    for (long ud = blockIdx.x; ud < nunits; ud += gridDim.x) {
        const long c = ud / (ugc * pm), r = ud % (ugc * pm);
        const long i = r % ugc, sy = r / ugc;
        const long us = c * ugc + i + ug * sy;
        const cd* sp = src + us * unit_elems;
        cd* dp = dst + ud * unit_elems;
        for (long k = threadIdx.x; k < unit_elems; k += blockDim.x) dp[k] = sp[k];
    }
}

__global__ void k_scale3(cd* a, long n, double s) {
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        cd v = a[i];
        a[i] = make_double2(v.x * s, v.y * s);
    }
}

int lag_spectrum3d(Op3D* op, cd* g2, long n, long m, long l);

// Compact (2x) spectrum, 3-D version of compact_spectrum() in op2d.cu: the kernel g = ifftn(GFFT) is only
// needed at the lags (-n,n) x (-m,m) x (-l,l).  Rank r owns the x-slot slab [r*4n/P, (r+1)*4n/P) of the 4x
// spectrum (17 GB at 256^3, 137 GB at 512^3 in total), generated / gathered in chunks; each chunk goes through
// the pruned inverse z and y passes at once (those lines are complete inside a chunk).  The inverse x pass needs
// all x slots: one all-to-all re-slabs along z (P > 1).  The 2n x 2m x 2l kernel is transformed back with
// unpadded forward passes (x and y on z slabs, a second all-to-all, then z on x-slot slabs).
// On return op->d_G holds this rank's slab of G2 in the z-pass chunk layout of the nr = 2 kernels, scaled by 1/(8 n m l).
int compact_spectrum3d(Op3D* op, const cd* d_gin, const int* d_fx, const int* d_fy, const int* d_fz, GenParams p) {
    const long n = op->n, m = op->m, l = op->l;
    const int P = op->P, rank = op->rank;
    cudaStream_t s = op->stream;
    cudaError_t e = cudaSuccess;
    int rc;
    const long nel4 = 4 * n / P;            // 4x x-slots of this rank
    const long nel2 = 2 * n / P;            // 2x x-slots of this rank (final slab)
    const long lz2 = 2 * l / P;             // 2x z planes of this rank (intermediate slab)
    LS_REQUIRE(nel2 % 8 == 0 && lz2 >= 1 && (2 * l) % P == 0, LS_ERR_UNSUPPORTED,
               "compact padding needs 2n/P to be a multiple of 8 and 2l divisible by P");
    // set-up chunks: the 4x slab is generated and pruned C x-slot chunks at a time, so that no more than ~20 GB of it
    // is resident at once.  LS_OP3D_SETUP_CHUNKS forces C (a power of two that leaves each chunk >= 16 x-slots).
    int C = 1;
    if (const char* cv = getenv("LS_OP3D_SETUP_CHUNKS")) {
        C = atoi(cv);
        LS_REQUIRE(C >= 1 && (C & (C - 1)) == 0 && nel4 / (2 * C) >= 8, LS_ERR_INVALID,
                   "LS_OP3D_SETUP_CHUNKS=%s: needs a power of two C with 4n/P/C >= 16 x-slots per chunk (4n/P = %ld)", cv, nel4);
    } else {
        while ((double)(64.0 * n * m * l * 16.0) / P / C > 20e9 && nel4 / (2 * C) >= 8) C *= 2;
    }
    const long nelc = nel4 / C;
    cd *g4c = nullptr, *t1c = nullptr, *T2 = nullptr, *R = nullptr, *g2 = nullptr;
    const size_t slab4 = (size_t)nel4 * (2 * m) * (2 * l);          // elements of T2 (this rank)
    const size_t slab2 = (size_t)(2 * n) * (2 * m) * lz2;           // elements of g2 / X (this rank) == nel2*2m*2l
    if ((rc = op->dmalloc((void**)&T2, slab4 * sizeof(cd)))) return rc;
    if ((rc = op->dmalloc((void**)&g4c, (size_t)nelc * (4 * m) * (4 * l) * sizeof(cd)))) return rc;
    if ((rc = op->dmalloc((void**)&t1c, (size_t)nelc * (4 * m) * (2 * l) * sizeof(cd)))) return rc;
    for (int c = 0; c < C; ++c) {
        p.nel = nelc; p.sx0 = (long)rank * nel4 + c * nelc;
        p.lb = 8;                            // set-up buffer: units of 8 lines, read below through explicit strides
        k_fill_g3d<<<148 * 16, 256, 0, s>>>(d_gin, g4c, d_fx, d_fy, d_fz, p);
        for (int cb = 0; cb <= 3; cb += 3) {     // (1) inverse z on the chunk: t1c[L + nelc*4m*jz2], L = sxl + nelc*sy4
            LineAddr la{8, 1, 32 * l, 8, 1, 8, nelc * 4 * m};
            la.nr = 4; la.cblock = cb;
            cd* outp = t1c + (cb ? l * (nelc * 4 * m) : 0);
#define Z1(N) launch_inv<N, true>(s, nelc * 4 * m, g4c, nullptr, outp, op->d_TABl, 1.0, la)
            LS3_DISPATCH(l, Z1);
            LS_CUDA_TRY(e);
        }
        for (int cb = 0; cb <= 3; cb += 3) {     // (2) inverse y: T2[sxl + nel4*(jy2 + 2m*jz2)], sxl within the rank's slab
            LineAddr la{nelc, 1, nelc * 4 * m, nelc, 1, nel4 * 2 * m, nel4};
            la.nr = 4; la.cblock = cb;
            cd* outp = T2 + c * nelc + (cb ? m * nel4 : 0);
#define Y1(N) launch_inv<N, true>(s, nelc * 2 * l, t1c, nullptr, outp, op->d_TABm, 1.0, la)
            LS3_DISPATCH(m, Y1);
            LS_CUDA_TRY(e);
        }
    }
    LS_CUDA_TRY(cudaStreamSynchronize(s));
    op->dfree(g4c);
    op->dfree(t1c);
    // re-slab along z: block q = planes jz2 in [q*lz2, (q+1)*lz2), contiguous in T2; received blocks are ordered by source rank
    const long blkA = nel4 * 2 * m * lz2;
    if (P > 1) {
        if ((rc = op->dmalloc((void**)&R, slab4 * sizeof(cd)))) return rc;
        if ((rc = all_to_all(op, T2, R, blkA))) return rc;
        LS_CUDA_TRY(cudaStreamSynchronize(s));
        op->dfree(T2);
    } else {
        R = T2;
    }
    if ((rc = op->dmalloc((void**)&g2, slab2 * sizeof(cd)))) return rc;
    int sh4 = 0;
    while ((1L << sh4) < nel4) ++sh4;
    for (int cb = 0; cb <= 3; cb += 3) {         // (3) inverse x, lines (jy2, jz2_loc): slot sx4 at R[(sx4/nel4)*blkA + nel4*line + sx4%nel4]
        LineAddr la{1L << 40, nel4, 0, 1, 2 * n, 0, 1};
        la.nr = 4; la.cblock = cb; la.split_shift = sh4; la.split_stride = blkA;
        cd* outp = g2 + (cb ? n : 0);
#define X1(N) launch_inv<N, false>(s, 2 * m * lz2, R, nullptr, outp, op->d_TABn, 1.0, la)
        LS3_DISPATCH(n, X1);
        LS_CUDA_TRY(e);
    }
    LS_CUDA_TRY(cudaStreamSynchronize(s));
    op->dfree(R);
    return lag_spectrum3d(op, g2, n, m, l);     // (4) - (6), the 1/(8 n m l) scale and the chunk-major order
}

// G2 = fftn(g2) / (2n 2m 2l) in the z-pass chunk layout of the nr = 2 kernels (n, m, l: the line lengths, powers of
// two).  g2: this rank's z slab (planes [rank*2l/P, (rank+1)*2l/P)) of the spatial kernel with its lags wrapped onto
// the 2n x 2m x 2l grid, g2[jx2 + 2n*(jy2 + 2m*jz2_loc)].  Takes ownership of g2; on return op->d_G = G2, op->nr = 2.
int lag_spectrum3d(Op3D* op, cd* g2, long n, long m, long l) {
    const int P = op->P;
    cudaStream_t s = op->stream;
    cudaError_t e = cudaSuccess;
    int rc;
    const long nel2 = 2 * n / P;            // 2x x-slots of this rank (final slab)
    const long lz2 = 2 * l / P;             // 2x z planes of this rank (intermediate slab)
    const size_t slab2 = (size_t)(2 * n) * (2 * m) * lz2;           // elements of g2 / X (this rank) == nel2*2m*2l
    const long LBl = lines_b(l);             // lines per unit of the final (2x) spectrum = what the fused z pass reads
    cd *Y = nullptr, *X = nullptr, *Z = nullptr, *G2 = nullptr;
    if ((rc = op->dmalloc((void**)&X, slab2 * sizeof(cd)))) return rc;
    {   // (4) forward x on the unpadded 2n-point lines: X[sx2 + 2n*line]
        LineAddr la{1L << 40, 2 * n, 0, 1, 2 * n, 0, 1};
        la.nr = 2; la.full2 = 1;
#define X2(N) launch_fwd<N, false>(s, 2 * m * lz2, g2, nullptr, X, op->d_TABn, la)
        LS3_DISPATCH(n, X2);
        LS_CUDA_TRY(e);
    }
    // (5) forward y, lines (sx2, jz2_loc), written grouped by destination rank q = sx2 / nel2:
    //     Y[q*blkB + sxl2 + nel2*(sy2 + 2m*jz2_loc)]   (g2 is reused as Y)
    const long blkB = nel2 * 2 * m * lz2;
    Y = g2;
    for (int q = 0; q < P; ++q) {
        LineAddr la{nel2, 1, 2 * n * 2 * m, 2 * n, 1, nel2 * 2 * m, nel2};
        la.nr = 2; la.full2 = 1;
        const cd* inp = X + q * nel2;
        cd* outp = Y + q * blkB;
#define Y2(N) launch_fwd<N, true>(s, nel2 * lz2, inp, nullptr, outp, op->d_TABm, la)
        LS3_DISPATCH(m, Y2);
        LS_CUDA_TRY(e);
    }
    if (P > 1) {       // re-slab along x: received blocks ordered by source rank = ordered by z plane
        Z = X;
        if ((rc = all_to_all(op, Y, Z, blkB))) return rc;
        LS_CUDA_TRY(cudaStreamSynchronize(s));
        G2 = Y;
    } else {
        Z = Y;
        G2 = X;
    }
    {   // (6) forward z, lines L = sxl2 + nel2*sy2: Z[L + nel2*2m*jz2] -> G2[((L/LB)*2 + rz)*LB*l + sz*LB + L%LB]
        LineAddr la{LBl, 1, LBl, nel2 * 2 * m, 1, 2 * LBl * l, LBl};
        la.nr = 2; la.full2 = 1;
#define Z2(N) launch_fwd<N, true>(s, nel2 * 2 * m, Z, nullptr, G2, op->d_TABl, la)
        LS3_DISPATCH(l, Z2);
        LS_CUDA_TRY(e);
    }
    k_scale3<<<148 * 8, 256, 0, s>>>(G2, (long)slab2, 1.0 / (8.0 * (double)n * (double)m * (double)l));
    if (op->Cx > 1) {   // chunk-major unit order (Z is free by now and has the same size)
        k_permute_units<<<148 * 16, 256, 0, s>>>(G2, Z, nel2 / LBl, nel2 / op->Cx / LBl, 2 * m, 2 * LBl * l);
        std::swap(G2, Z);
    }
    LS_CUDA_TRY(cudaStreamSynchronize(s));
    op->dfree(Z == G2 ? nullptr : Z);
    op->d_G = G2;
    op->nr = 2;
    return LS_OK;
}

int create3d(ls_handle* out, int64_t n, int64_t m, int64_t l, int64_t ne, int64_t me, int64_t le,
             const double* nu, const ls_cdouble* gfft, double omega, double L, double Lp,
             int rank, int nranks, const void* nccl_id, int flags) {
    LS_REQUIRE(out && nu, LS_ERR_INVALID, "ls_op3d_create: null pointer");
    LS_REQUIRE(n > 0 && m > 0 && l > 0, LS_ERR_INVALID, "ls_op3d_create: non-positive size");
    LS_REQUIRE(ne == 4 * n && me == 4 * m && le == 4 * l, LS_ERR_INVALID,
               "ls_op3d_create: Greengard_Vico needs ne = 4n, me = 4m, le = 4l (FastConvolution3D.jl:100)");
    LS_REQUIRE(n == m, LS_ERR_INVALID,
               "ls_op3d_create: FFTconvolution pads (ne, ne, le): n must equal m (FastConvolution3D.jl:48)");
    const bool embed = (flags & LS_FLAG_EMBED) != 0;
    long embed_slots = 0;              // x-slots per chunk of the lag extraction; 0: by size (embed_lag_grid3d)
    if (embed) {
        // every refusal before any CUDA or NCCL call
        LS_REQUIRE(!(flags & LS_FLAG_FORCE_GENERIC), LS_ERR_INVALID,
                   "ls_op3d_create: LS_FLAG_EMBED and LS_FLAG_FORCE_GENERIC select different routes");
        LS_REQUIRE(!(flags & LS_FLAG_PAD4), LS_ERR_UNSUPPORTED,
                   "ls_op3d_create: the zero-embedded route runs with 2x padding only (no literal 4x evaluation)");
        LS_REQUIRE(n <= 512 && l <= 512, LS_ERR_UNSUPPORTED,
                   "ls_op3d_create: n=%ld, l=%ld: the zero-embedded route serves n, l <= 512", (long)n, (long)l);
        // LS_OP3D_EMBED_CHUNK_SLOTS forces the chunk width (a value at or above the rank's 4n/P x-slots: one chunk)
        if (const char* cv = getenv("LS_OP3D_EMBED_CHUNK_SLOTS")) {
            char* end = nullptr;
            errno = 0;
            embed_slots = strtol(cv, &end, 10);
            LS_REQUIRE(end != cv && *end == '\0' && errno == 0 && embed_slots > 0, LS_ERR_INVALID,
                       "LS_OP3D_EMBED_CHUNK_SLOTS=%s: needs a positive integer (x-slots per lag-extraction chunk)", cv);
        }
    }
    auto ok3 = [](long v) { return v == 64 || v == 128 || v == 256 || v == 512; };
    if (!embed && !(ok3(n) && ok3(m) && ok3(l))) {
        LS_REQUIRE(nranks == 1, LS_ERR_UNSUPPORTED,
                   "ls_op3d_create_dist: n=%ld m=%ld l=%ld - the sharded path serves powers of two in [64, 512]", (long)n, (long)m, (long)l);
        LS_REQUIRE(gfft != nullptr || (L > 0 && Lp > 0), LS_ERR_INVALID,
                   "ls_op3d_create: pass GFFT or the Greengard-Vico parameters L, Lp to generate it on the device");
        return create_op3d_generic(out, n, m, l, ne, me, le, nu, gfft, omega, L, Lp);     // any size: Bluestein lines
    }
    LS_REQUIRE(gfft != nullptr || (L > 0 && Lp > 0), LS_ERR_INVALID,
               "ls_op3d_create: pass GFFT or the Greengard-Vico parameters L, Lp to generate it on the device");
    LS_REQUIRE(nranks == 1 || nranks == 2 || nranks == 4 || nranks == 8, LS_ERR_INVALID,
               "ls_op3d_create_dist: nranks must be 1, 2, 4 or 8");
    LS_REQUIRE(rank >= 0 && rank < nranks, LS_ERR_INVALID, "ls_op3d_create_dist: rank out of range");
    LS_REQUIRE(nranks == 1 || nccl_id != nullptr, LS_ERR_INVALID, "ls_op3d_create_dist: null NCCL id");
    LS_REQUIRE(nranks == 1 || gfft == nullptr, LS_ERR_UNSUPPORTED,
               "ls_op3d_create_dist: the sharded operator generates its spectrum slab on the device (pass NULL, L, Lp)");
    LS_REQUIRE(!embed || l % nranks == 0, LS_ERR_UNSUPPORTED,
               "ls_op3d_create_dist: l=%ld over %d ranks: the z planes must divide evenly between the ranks", (long)l, nranks);

    Op3D* op = new Op3D();
    int rc = op->init_base(KIND_OP3D);
    if (rc) { delete op; return rc; }
    op->n = n; op->m = m; op->l = l; op->ne = ne; op->me = me; op->le = le; op->omega = omega;
    op->P = nranks; op->rank = rank; op->nel = ne / nranks; op->lloc = l / nranks;
    op->embed = embed;
    op->ln = embed ? embed_len(n) : n; op->lm = embed ? embed_len(m) : m; op->ll = embed ? embed_len(l) : l;
    const long ln = op->ln, lm = op->lm, ll = op->ll;
    if (nranks > 1) {
        ncclUniqueId id;
        memcpy(&id, nccl_id, sizeof(id));
        ncclResult_t r = ncclCommInitRank(&op->comm, nranks, id, rank);
        if (r != ncclSuccess) {
            set_error("ncclCommInitRank failed: %s", ncclGetErrorString(r));
            op->comm = nullptr;
            delete op;
            return LS_ERR_NCCL;
        }
    }
    const bool compact = !(flags & LS_FLAG_PAD4);
    {   // x-slot chunks (pipelined transposes).  Default: chunks of >= 16 MB per peer, at most 4 (measured on 8 GPUs:
        // 512^3 4.70 -> 4.05 ms with 4 chunks of 17 MB; 256^3 with 8 MB per peer is fastest unchunked).
        // LS_OP3D_CHUNKS overrides; chunks keep >= 8 x-slots.
        const long nelf = (compact ? 2 : 4) * ln / nranks;
        const char* ev = getenv("LS_OP3D_CHUNKS");
        int cx = 1;
        if (ev) cx = atoi(ev);
        else if (nranks > 1) {
            const double peer_mb = 16.0 * (double)nelf * (double)m * (double)(l / nranks) / 1048576.0;
            cx = peer_mb >= 64.0 ? 4 : peer_mb >= 32.0 ? 2 : 1;
        }
        if (cx < 1) cx = 1;
        while (cx & (cx - 1)) cx &= cx - 1;
        while (cx > 1 && nelf / cx < 8) cx /= 2;
        op->Cx = cx;
    }
    long nel = op->nel;
    const long lloc = op->lloc;
    const size_t Nloc = (size_t)n * m * lloc, NEloc = (size_t)nel * me * le;
#define TRY(x) do { rc = (x); if (rc) { delete op; return rc; } } while (0)
    TRY(op->dupload((void**)&op->d_nu, nu, Nloc * sizeof(double)));
    {
        auto Tn = engine_table((int)ln), Tm = engine_table((int)lm), Tl = engine_table((int)ll);
        TRY(op->dupload((void**)&op->d_TABn, Tn.data(), Tn.size() * sizeof(cd)));
        TRY(op->dupload((void**)&op->d_TABm, Tm.data(), Tm.size() * sizeof(cd)));
        TRY(op->dupload((void**)&op->d_TABl, Tl.data(), Tl.size() * sizeof(cd)));
    }
    if (embed) {
        // the kernel's lags on this rank's z slab of the 2n' x 2m' x 2l' grid, then the compact path's final passes
        cd *d_gin = nullptr, *g2 = nullptr;
        if (gfft) TRY(op->dupload((void**)&d_gin, gfft, (size_t)ne * me * le * sizeof(cd)));
        TRY(op->dmalloc((void**)&g2, (size_t)(2 * ln) * (2 * lm) * (2 * ll / nranks) * sizeof(cd)));
        const auto t0 = std::chrono::steady_clock::now();
        TRY(embed_lag_grid3d(op, d_gin, n, l, omega, L, Lp, rank, nranks, op->comm, g2, 2 * ln, 2 * ll, embed_slots));
        const auto t1 = std::chrono::steady_clock::now();
        if (d_gin) op->dfree(d_gin);
        TRY(lag_spectrum3d(op, g2, ln, lm, ll));
        if (getenv("LS_DEBUG")) {    // scripts/probe3d_embed.py reads this line
            const double tl = std::chrono::duration<double>(t1 - t0).count();
            const double ts = std::chrono::duration<double>(std::chrono::steady_clock::now() - t1).count();
            const double lx = 2.0 * n - 1, lz = 2.0 * l - 1;     // the three contractions of this rank's x-slots
            const double flop = 8.0 * ((double)ne / nranks) * ((double)me * le * lz + (double)me * lx * lz + lx * lx * lz);
            fprintf(stderr, "[ls_cuda] rank %d: embedded create: lag extraction %.3f s (%.3e flop), spectrum %.3f s\n",
                    rank, tl, flop, ts);
        }
    } else {
        auto fx = slot_freq((int)n), fy = slot_freq((int)m), fz = slot_freq((int)l);
        int *d_fx = nullptr, *d_fy = nullptr, *d_fz = nullptr;
        cd* d_gin = nullptr;
        TRY(op->dupload((void**)&d_fx, fx.data(), fx.size() * sizeof(int)));
        TRY(op->dupload((void**)&d_fy, fy.data(), fy.size() * sizeof(int)));
        TRY(op->dupload((void**)&d_fz, fz.data(), fz.size() * sizeof(int)));
        if (gfft) TRY(op->dupload((void**)&d_gin, gfft, (size_t)ne * me * le * sizeof(cd)));
        if (!compact) TRY(op->dmalloc((void**)&op->d_G, NEloc * sizeof(cd)));
        GenParams p;
        p.n = n; p.m = m; p.l = l; p.ne = ne; p.me = me; p.le = le;
        p.nel = nel; p.sx0 = (long)rank * nel;
        p.dk = gfft ? 0.0 : 2.0 * 3.141592653589793 / Lp;
        p.L = L; p.k = omega;
        p.eLk_re = cos(L * omega); p.eLk_im = sin(L * omega);
        p.scale = 1.0 / ((double)ne * (double)me * (double)le);
        if (compact) TRY(compact_spectrum3d(op, d_gin, d_fx, d_fy, d_fz, p));
        else {
            const long nc4 = nel / op->Cx;       // chunk-major spectrum: chunk c holds the x-slots [c*nc4, (c+1)*nc4) of the slab
            p.lb = lines_b(l);
            for (int c = 0; c < op->Cx; ++c) {
                p.nel = nc4; p.sx0 = (long)rank * nel + c * nc4;
                k_fill_g3d<<<148 * 16, 256, 0, op->stream>>>(d_gin, op->d_G + (size_t)c * nc4 * me * le, d_fx, d_fy, d_fz, p);
            }
        }
        cudaError_t e = cudaStreamSynchronize(op->stream);
        if (e != cudaSuccess) { set_error("spectrum setup failed: %s", cudaGetErrorString(e)); delete op; return LS_ERR_CUDA; }
        if (d_gin) op->dfree(d_gin);
        op->dfree(d_fx); op->dfree(d_fy); op->dfree(d_fz);
    }
    op->pn = op->nr * ln; op->pm = op->nr * lm; op->pl = op->nr * ll;
    op->nel = nel = op->pn / nranks;
    op->nelc = nel / op->Cx;
    TRY(op->dmalloc((void**)&op->d_A1, (size_t)op->pn * m * lloc * sizeof(cd)));
    if (nranks > 1) TRY(op->dmalloc((void**)&op->d_A1T, (size_t)nel * m * l * sizeof(cd)));
    TRY(op->dmalloc((void**)&op->d_A2, (size_t)op->nelc * op->pm * ll * sizeof(cd)));
    if (nranks > 1) {
        int lo = 0, hi = 0;
        cudaError_t ce = cudaDeviceGetStreamPriorityRange(&lo, &hi);
        const char* pv = getenv("LS_OP3D_COMM_PRIO");          // 1 (default): exchange stream at the highest priority, so its
        const bool high = pv ? atoi(pv) != 0 : true;           // copy kernels get SM slots as soon as line-kernel CTAs retire
        if (ce == cudaSuccess) ce = cudaStreamCreateWithPriority(&op->cstream, cudaStreamNonBlocking, high ? hi : lo);
        if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&op->evP1, cudaEventDisableTiming);
        if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&op->evDone, cudaEventDisableTiming);
        for (int c = 0; c < 2 * op->Cx && ce == cudaSuccess; ++c) {
            cudaEvent_t ev = nullptr;
            ce = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
            if (ce == cudaSuccess) (c < op->Cx ? op->evIn : op->evOut).push_back(ev);
        }
        if (ce != cudaSuccess) { set_error("exchange stream setup failed: %s", cudaGetErrorString(ce)); delete op; return LS_ERR_CUDA; }
        // Route of the two transposes.  LS_OP3D_XCHG = ce | nccl forces one; default: copy engines when a transpose sends at
        // least LS_OP3D_CE_MIN_MB (12) MB per peer, NCCL's concurrent channels below that (measured on 8 GPUs at 256^3,
        // 8.4 MB per peer: seven serial pushes + completion 0.66 ms against 0.59 ms; at 67 MB per peer 3.71 against 3.86 ms)
        const char* xv = getenv("LS_OP3D_XCHG");
        const char* mv = getenv("LS_OP3D_CE_MIN_MB");
        const double min_mb = mv ? atof(mv) : 12.0;
        const double peer_mb = 16.0 * (double)nel * (double)m * (double)lloc / 1048576.0;
        const bool want_ce = xv ? strcmp(xv, "nccl") != 0 : peer_mb >= min_mb;
        if (want_ce) {
            // every rank must take the same route: agree (min over ranks) after the attempt
            const int ok = setup_ce_exchange(op) == LS_OK ? 1 : 0;
            cudaGetLastError();
            int* d_ok = nullptr;
            TRY(op->dmalloc((void**)&d_ok, sizeof(int)));
            ce = cudaMemcpyAsync(d_ok, &ok, sizeof(int), cudaMemcpyHostToDevice, op->stream);
            ncclResult_t nr = ncclAllReduce(d_ok, d_ok, 1, ncclInt, ncclMin, op->comm, op->stream);
            int all_ok = 0;
            if (ce == cudaSuccess && nr == ncclSuccess) ce = cudaMemcpyAsync(&all_ok, d_ok, sizeof(int), cudaMemcpyDeviceToHost, op->stream);
            if (ce == cudaSuccess) ce = cudaStreamSynchronize(op->stream);
            if (ce != cudaSuccess || nr != ncclSuccess) { set_error("exchange route agreement failed"); delete op; return LS_ERR_NCCL; }
            op->dfree(d_ok);
            op->ce_exchange = all_ok == 1;
            if (!op->ce_exchange && getenv("LS_DEBUG")) fprintf(stderr, "[ls_cuda] rank %d: IPC exchange unavailable (%s), using the NCCL all-to-all\n", rank, ls_last_error());
        }
    }
#undef TRY
    *out = reinterpret_cast<ls_handle>(op);
    return LS_OK;
}

}  // namespace

int Op3D::apply_dev(const cd* b, cd* y, int mode) { return apply_device3(this, &b, &y, 1, mode); }

int Op3D::apply_cols_dev(const cd* const* b, cd* const* y, int ncol, int mode) {
    if (P != 1 || nr != 2) return HandleBase::apply_cols_dev(b, y, ncol, mode);     // column by column
    LS_REQUIRE(ncol >= 1 && ncol <= cols, LS_ERR_INVALID, "3-D batched apply: %d columns, %d reserved", ncol, cols);
    return apply_device3(this, b, y, ncol, mode);
}

// A1 and A2 for ncol columns: new arrays, the old ones freed once the stream has drained.  Every pass writes what the
// next one reads (the embedded P2 writes the zero planes P3 transforms), so the new arrays need no initialisation.
// The caller checked the free memory.
int Op3D::batch_reserve(int ncol) {
    if (ncol <= cols) return LS_OK;
    cd *a1 = nullptr, *a2 = nullptr;
    int rc;
    if ((rc = dmalloc((void**)&a1, (size_t)ncol * a1cs() * sizeof(cd)))) return rc;
    if ((rc = dmalloc((void**)&a2, (size_t)ncol * a2cs() * sizeof(cd)))) { dfree(a1); return rc; }
    LS_CUDA_TRY(cudaStreamSynchronize(stream));
    dfree(d_A1); dfree(d_A2);
    d_A1 = a1; d_A2 = a2; cols = ncol;
    return LS_OK;
}

extern "C" {

int ls_op3d_create(ls_handle* out, int64_t n, int64_t m, int64_t l, int64_t ne, int64_t me, int64_t le,
                   const double* nu, const ls_cdouble* gfft, double omega, double L, double Lp, int flags) {
    return create3d(out, n, m, l, ne, me, le, nu, gfft, omega, L, Lp, 0, 1, nullptr, flags);
}

int ls_op3d_create_dist(ls_handle* out, int64_t n, int64_t m, int64_t l, const double* nu_slab, double omega,
                        double L, double Lp, int rank, int nranks, const void* nccl_unique_id, int flags) {
    return create3d(out, n, m, l, 4 * n, 4 * m, 4 * l, nu_slab, nullptr, omega, L, Lp, rank, nranks, nccl_unique_id, flags);
}

int ls_nccl_unique_id(void* out128) {
    LS_REQUIRE(out128, LS_ERR_INVALID, "ls_nccl_unique_id: null pointer");
    ncclUniqueId id;
    ncclResult_t r = ncclGetUniqueId(&id);
    if (r != ncclSuccess) { set_error("ncclGetUniqueId failed: %s", ncclGetErrorString(r)); return LS_ERR_NCCL; }
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    memcpy(out128, &id, sizeof(id));
    return LS_OK;
}

int ls_op3d_info(ls_handle h, int* padding_factor, int* x_slot_chunks, int* exchange) {
    LS_REQUIRE(h, LS_ERR_INVALID, "ls_op3d_info: null handle");
    HandleBase* base = reinterpret_cast<HandleBase*>(h);
    LS_REQUIRE(base->kind == KIND_OP3D, LS_ERR_INVALID, "ls_op3d_info: not a 3-D operator handle");
    Op3D* op = dynamic_cast<Op3D*>(base);
    if (padding_factor) *padding_factor = op ? op->nr : 4;
    if (x_slot_chunks) *x_slot_chunks = op ? op->Cx : 1;
    if (exchange) *exchange = (op && op->P > 1) ? (op->ce_exchange ? 2 : 1) : 0;
    return LS_OK;
}

int ls_op3d_lines(ls_handle h, int* route, int64_t* n_line, int64_t* m_line, int64_t* l_line) {
    LS_REQUIRE(h, LS_ERR_INVALID, "ls_op3d_lines: null handle");
    HandleBase* base = reinterpret_cast<HandleBase*>(h);
    LS_REQUIRE(base->kind == KIND_OP3D, LS_ERR_INVALID, "ls_op3d_lines: not a 3-D operator handle");
    int r = 1;
    int64_t a = 0, b = 0, c = 0;
    if (const Op3D* op = dynamic_cast<const Op3D*>(base)) {
        r = op->embed ? 2 : 0; a = op->ln; b = op->lm; c = op->ll;
    } else {
        op3d_generic_lines(base, &a, &b, &c);
    }
    if (route) *route = r;
    if (n_line) *n_line = a;
    if (m_line) *m_line = b;
    if (l_line) *l_line = c;
    return LS_OK;
}

int ls_op3d_apply(ls_handle h, const ls_cdouble* b, ls_cdouble* y, int mode, int memloc) {
    LS_REQUIRE(h && b && y, LS_ERR_INVALID, "ls_op3d_apply: null argument");
    HandleBase* op = reinterpret_cast<HandleBase*>(h);      // power-of-two (Op3D) or general-size operator
    LS_REQUIRE(op->kind == KIND_OP3D, LS_ERR_INVALID, "ls_op3d_apply: not a 3-D operator handle");
    LS_REQUIRE(mode == LS_APPLY_FASTCONVOLUTION || mode == LS_APPLY_FFTCONVOLUTION, LS_ERR_INVALID,
               "ls_op3d_apply: unknown mode %d", mode);
    LS_CUDA_TRY(cudaSetDevice(op->device));
    const size_t bytes = (size_t)op->op_size() * sizeof(cd);
    if (memloc == LS_MEM_DEVICE)
        return op->apply_dev(reinterpret_cast<const cd*>(b), reinterpret_cast<cd*>(y), mode);
    LS_REQUIRE(memloc == LS_MEM_HOST, LS_ERR_INVALID, "ls_op3d_apply: unknown memloc %d", memloc);
    if (!op->stage_b) {
        int rc;
        if ((rc = op->dmalloc((void**)&op->stage_b, bytes))) return rc;
        if ((rc = op->dmalloc((void**)&op->stage_y, bytes))) return rc;
    }
    LS_CUDA_TRY(cudaMemcpyAsync(op->stage_b, b, bytes, cudaMemcpyHostToDevice, op->stream));
    int rc = op->apply_dev(op->stage_b, op->stage_y, mode);
    if (rc) return rc;
    LS_CUDA_TRY(cudaMemcpyAsync(y, op->stage_y, bytes, cudaMemcpyDeviceToHost, op->stream));
    LS_CUDA_TRY(cudaStreamSynchronize(op->stream));
    return LS_OK;
}

}  // extern "C"
