// CPU execution of the multi-column Msp sweep (csrc/msp_gemv.cuh, k_msp_gemv2_cols) next to the single-vector one
// (msp_gemv_emu.cu, included): the same __host__ __device__ phase functions, run CTA by CTA and thread by thread, the
// warp-shuffle reduction replaced by the same xor tree on an array.  Test infrastructure only
// (tests/test_msp_gemv_cols_emulation.py builds it with nvcc as a host library); nothing in the product links it.
#include "msp_gemv_emu.cu"

template <int LANES, int UNR, bool XS, int NRHS>
static void emu_run_cols(const Gemv2& a, const Cols& cs, const LaunchGeo& L) {
    std::vector<cd> xs(L.smem * NRHS / sizeof(cd) + 1);
    const size_t per = (size_t)NRHS * UNR;
    std::vector<double> SR(256 * per), SI(256 * per), TR(256 * per), TI(256 * per);
    std::vector<ThreadMap> maps(256);
    for (unsigned bid = 0; bid < L.grid; ++bid) {
        if (XS)
            for (unsigned tid = 0; tid < 256; ++tid) stage_x_cols<NRHS>(a, cs, L.g, bid, tid, xs.data());
        for (unsigned tid = 0; tid < 256; ++tid) {
            maps[tid] = map_thread<LANES, UNR>(a, L.g, bid, tid);
            double sr[NRHS][UNR], si[NRHS][UNR];
            accumulate_cols<LANES, UNR, XS, NRHS>(a, cs, L.g, maps[tid], xs.data(), sr, si);
            for (int j = 0; j < NRHS; ++j)
                for (int u = 0; u < UNR; ++u) { SR[tid * per + j * UNR + u] = sr[j][u]; SI[tid * per + j * UNR + u] = si[j][u]; }
        }
        for (int o = LANES / 2; o > 0; o >>= 1) {
            for (unsigned tid = 0; tid < 256; ++tid)
                for (size_t q = 0; q < per; ++q) {
                    TR[tid * per + q] = SR[tid * per + q] + SR[(tid ^ o) * per + q];
                    TI[tid * per + q] = SI[tid * per + q] + SI[(tid ^ o) * per + q];
                }
            SR.swap(TR); SI.swap(TI);
        }
        for (unsigned tid = 0; tid < 256; ++tid) {
            double sr[NRHS][UNR], si[NRHS][UNR];
            for (int j = 0; j < NRHS; ++j)
                for (int u = 0; u < UNR; ++u) { sr[j][u] = SR[tid * per + j * UNR + u]; si[j][u] = SI[tid * per + j * UNR + u]; }
            store_rows_cols<LANES, UNR, NRHS>(a, cs, maps[tid], sr, si);
        }
    }
}

typedef void (*emu_cols_fn)(const Gemv2&, const Cols&, const LaunchGeo&);
#define EMUC_U(L, U, R) { emu_run_cols<L, U, false, R>, emu_run_cols<L, U, true, R> }
#define EMUC_L(L, R) { EMUC_U(L, 1, R), EMUC_U(L, 2, R), EMUC_U(L, 4, R), EMUC_U(L, 8, R) }
#define EMUC_R(R) { EMUC_L(1, R), EMUC_L(2, R), EMUC_L(4, R), EMUC_L(8, R), EMUC_L(16, R), EMUC_L(32, R) }
static emu_cols_fn emu_cols_table[4][6][4][2] = { EMUC_R(1), EMUC_R(2), EMUC_R(4), EMUC_R(8) };

extern "C" {

// nrhs in {1, 2, 4, 8}; returns the grid size used, or -1
int emu_msp_gemv2_cols(const Gemv2* a, const Cols* cs, int nrhs, int lanes_log2, int unr_log2, int xs, long* smem_out) {
    const int rl = nrhs == 1 ? 0 : nrhs == 2 ? 1 : nrhs == 4 ? 2 : nrhs == 8 ? 3 : -1;
    if (rl < 0 || lanes_log2 < 0 || lanes_log2 > 5 || unr_log2 < 0 || unr_log2 > 3) return -1;
    Choice ch{lanes_log2, unr_log2, xs ? 1 : 0};
    const LaunchGeo L = launch_geo(a->rows_p, a->cols_p, a->nodes, ch);
    if (smem_out) *smem_out = (long)L.smem * nrhs;
    emu_cols_table[rl][lanes_log2][unr_log2][xs ? 1 : 0](*a, *cs, L);
    return (int)L.grid;
}

// lsmsp::cols_choice: out3 = lanes_log2, unr_log2, xs
void emu_cols_choice(int lanes_log2, int unr_log2, int xs, int nrhs, int rows_p, int cols_p, int nodes, int xmode, long limit,
                     int* out3) {
    const Choice ch = cols_choice(Choice{lanes_log2, unr_log2, xs}, nrhs, rows_p, cols_p, nodes, xmode, (size_t)limit);
    out3[0] = ch.lanes_log2; out3[1] = ch.unr_log2; out3[2] = ch.xs;
}

int emu_sizeof_cols() { return (int)sizeof(Cols); }

}  // extern "C"
