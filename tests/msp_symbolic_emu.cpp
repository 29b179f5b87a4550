// CPU access to the symbolic analysis of the device Msp factorisation (csrc/msp_symbolic.h): the very code msp.cu
// runs before it touches the device - boxes, own and ring lists, entry routing, child / parent maps and the byte count
// of the memory check.  Test infrastructure only (tests/test_msp_symbolic.py builds it as a host library); nothing in
// the product links it.
#include "../fast_solver_lippmann_schwinger_b200/csrc/msp_symbolic.h"

using lsmsp::Symbolic;

extern "C" {

// analysed dissection of the n x m x l grid (with its lists and maps if `lists`), or null (message in *err)
void* sym_create(int n, int m, int l, int leafmax, int lists, char* err, int cap) {
    Symbolic* S = new Symbolic();
    int rc = S->analyse(n, m, l, leafmax);
    if (rc == LS_OK && lists) rc = S->lists();
    if (rc == LS_OK && lists) rc = S->maps();
    if (rc != LS_OK) {
        snprintf(err, cap, "%s", S->err.c_str());
        delete S;
        return nullptr;
    }
    return S;
}

void sym_destroy(void* h) { delete static_cast<Symbolic*>(h); }

int sym_depth(void* h) { return static_cast<Symbolic*>(h)->D; }

// count, Sp, Bp, leaf, axis of depth d
void sym_level(void* h, int d, int* out5) {
    const lsmsp::LevelShape& L = static_cast<Symbolic*>(h)->lev[d];
    out5[0] = L.count; out5[1] = L.Sp; out5[2] = L.Bp; out5[3] = L.leaf ? 1 : 0; out5[4] = L.axis;
}

void sym_box(void* h, int d, int t, int* out6) {
    const lsmsp::Box& b = static_cast<Symbolic*>(h)->boxes[d][t];
    out6[0] = b.i0; out6[1] = b.i1; out6[2] = b.j0; out6[3] = b.j1; out6[4] = b.p0; out6[5] = b.p1;
}

// which: 0 Sidx, 1 Bidx, 2 pmap, 3 cmap, 4 ns, 5 nb, 6 own_node, 7 own_loc; copies at most cap values, returns the length
long sym_ints(void* h, int which, int d, int* out, long cap) {
    Symbolic* S = static_cast<Symbolic*>(h);
    const std::vector<int>* v = nullptr;
    std::vector<int> tmp;
    switch (which) {
        case 0: v = &S->Sidx[d]; break;
        case 1: v = &S->Bidx[d]; break;
        case 2: v = &S->pmap[d]; break;
        case 3: v = &S->cmap[d]; break;
        case 4: v = &S->lev[d].ns; break;
        case 5: v = &S->lev[d].nb; break;
        case 6: v = &S->own_node; break;
        case 7: v = &S->own_loc; break;
        default: return -1;
    }
    const long len = (long)v->size();
    for (long i = 0; i < len && i < cap; ++i) out[i] = (*v)[i];
    return len;
}

void sym_own_depth(void* h, unsigned char* out) {
    const Symbolic* S = static_cast<Symbolic*>(h);
    for (size_t i = 0; i < S->own_depth.size(); ++i) out[i] = S->own_depth[i];
}

int sym_ring_index(void* h, int d, int t, int i, int j, int p) {
    const Symbolic* S = static_cast<Symbolic*>(h);
    return S->ring_index(S->boxes[d][t], i, j, p);
}

// routes a 1-based CSC pattern; returns the status code (message in *err)
int sym_route(void* h, const int64_t* colptr, const int64_t* rowval, char* err, int cap) {
    Symbolic* S = static_cast<Symbolic*>(h);
    S->err.clear();
    const int rc = S->route(colptr, rowval);
    snprintf(err, cap, "%s", S->err.c_str());
    return rc;
}

long sym_entries(void* h, int d, long* dest, int* src, long cap) {
    const Symbolic* S = static_cast<Symbolic*>(h);
    const long len = (long)S->edest[d].size();
    for (long i = 0; i < len && i < cap; ++i) { dest[i] = S->edest[d][i]; src[i] = S->esrc[d][i]; }
    return len;
}

unsigned long long sym_need_bytes(void* h, long long nnz, int tight) {
    return (unsigned long long)static_cast<Symbolic*>(h)->need_bytes(nnz, tight != 0);
}

}  // extern "C"
