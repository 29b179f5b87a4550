// Host-side symbolic analysis of the nested-dissection factorisation of Msp (msp.cu), for 2-D and 3-D grids.
//
// The n x m x l grid (unknown i + n*(j + m*p), x fastest; l = 1 is the 2-D case) is bisected recursively: at every
// depth each box is split at its midpoint by a separator one cell thick, perpendicular to the axis with the largest
// extent over the depth's boxes (ties: x, then y, then z), until no box is wider than `leafmax` cells in any axis.
// A node's own unknowns S are its separator plane (or the whole box at the leaf depth); its ring B is the shell of
// thickness one around the box, clipped to the grid.  A 27-point stencil couples only cells at most one apart in
// every coordinate, so a plane separates and every entry of the matrix lands in exactly one front.  Own lists and
// shells are enumerated in lexicographic order (x fastest, then y, then z); with l = 1 this is the 2-D order.
//
// No CUDA in this file: tests/msp_symbolic_emu.cpp compiles the same code on the CPU (tests/test_msp_symbolic.py).
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <cstdio>
#include <string>
#include <vector>
#include "../../include/ls_cuda.h"

namespace lsmsp {

struct Box { int i0, i1, j0, j1, p0, p1; };      // region [i0, i1) x [j0, j1) x [p0, p1)

struct LevelShape {                               // all 2^d nodes of one depth
    int count = 0, Sp = 0, Bp = 0;                // padded sizes of S and B
    bool leaf = false;
    int axis = 0;                                 // split axis of this depth (0: x, 1: y, 2: z), internal levels
    std::vector<int> ns, nb;                      // actual sizes of every node's S and B
};

struct Symbolic {
    int n = 0, m = 0, l = 0;
    int D = 0;
    std::string fn = "ls_msp_factor";             // prefix of the error messages
    std::string err;
    std::vector<std::vector<Box>> boxes;          // per depth
    std::vector<LevelShape> lev;
    // filled by lists()
    std::vector<unsigned char> own_depth;
    std::vector<int> own_node, own_loc;
    std::vector<std::vector<int>> Sidx, Bidx;     // [count][Sp], [count][max(Bp, 1)]: global unknown, -1 = padding
    // filled by maps(): cmap[d+1][child][k] = position of the child's k-th ring unknown in the parent's [S; B]
    // numbering; pmap[d][parent][side][p] = k with cmap == p, or -1
    std::vector<std::vector<int>> cmap, pmap;
    // filled by route(): flat destination of every entry in the batch of column-major fronts of its depth, and its
    // position in nzval
    std::vector<std::vector<long>> edest;
    std::vector<std::vector<int>> esrc;

    long N() const { return (long)n * m * l; }

    int fail(int code, const char* fmt, long a = 0, long b = 0, long c = 0) {
        char buf[320];
        snprintf(buf, sizeof buf, fmt, a, b, c);
        err = fn + ": " + buf;
        return code;
    }

    // inclusive bounds of the shell around b, clipped to the grid
    void shell(const Box& b, int& ia, int& ib, int& ja, int& jb, int& pa, int& pb) const {
        ia = std::max(b.i0 - 1, 0); ib = std::min(b.i1, n - 1);
        ja = std::max(b.j0 - 1, 0); jb = std::min(b.j1, m - 1);
        pa = std::max(b.p0 - 1, 0); pb = std::min(b.p1, l - 1);
    }
    long ring_size(const Box& b) const {
        int ia, ib, ja, jb, pa, pb;
        shell(b, ia, ib, ja, jb, pa, pb);
        return (long)(ib - ia + 1) * (jb - ja + 1) * (pb - pa + 1) - (long)(b.i1 - b.i0) * (b.j1 - b.j0) * (b.p1 - b.p0);
    }
    long own_size(const Box& b, bool leaf, int ax) const {
        const long w = b.i1 - b.i0, h = b.j1 - b.j0, t = b.p1 - b.p0;
        if (leaf) return w * h * t;
        return ax == 0 ? h * t : (ax == 1 ? w * t : w * h);
    }
    // position of (i, j, p) in the ring around b, -1 if it is not on the ring
    int ring_index(const Box& b, int i, int j, int p) const {
        int ia, ib, ja, jb, pa, pb;
        shell(b, ia, ib, ja, jb, pa, pb);
        if (i < ia || i > ib || j < ja || j > jb || p < pa || p > pb) return -1;
        const bool ini = i >= b.i0 && i < b.i1, inj = j >= b.j0 && j < b.j1, inp = p >= b.p0 && p < b.p1;
        if (ini && inj && inp) return -1;
        const long W = ib - ia + 1, H = jb - ja + 1, w = b.i1 - b.i0, h = b.j1 - b.j0;
        const long inner_planes = std::max(0, std::min(p, b.p1) - b.p0);          // planes before p that hold the box
        long pos = (long)(p - pa) * W * H - inner_planes * w * h;
        if (!inp) return (int)(pos + (long)(j - ja) * W + (i - ia));
        const long inner_rows = std::max(0, std::min(j, b.j1) - b.j0);
        pos += (long)(j - ja) * W - inner_rows * w;
        if (!inj) return (int)(pos + (i - ia));
        return (int)(pos + (i < b.i0 ? i - ia : i - ia - w));
    }
    void ring_list(const Box& b, std::vector<int>& out) const {
        out.clear();
        int ia, ib, ja, jb, pa, pb;
        shell(b, ia, ib, ja, jb, pa, pb);
        for (int p = pa; p <= pb; ++p)
            for (int j = ja; j <= jb; ++j) {
                const bool inner = p >= b.p0 && p < b.p1 && j >= b.j0 && j < b.j1;
                for (int i = ia; i <= ib; ++i) {
                    if (inner && i == b.i0) { i = b.i1 - 1; continue; }
                    out.push_back(i + n * (j + m * p));
                }
            }
    }
    // own unknowns of a node: the separator plane (internal) or the whole box (leaf)
    void own_list(const Box& b, bool leaf, int ax, std::vector<int>& out) const {
        out.clear();
        Box r = b;
        if (!leaf) {
            if (ax == 0) { r.i0 = b.i0 + (b.i1 - b.i0) / 2; r.i1 = r.i0 + 1; }
            else if (ax == 1) { r.j0 = b.j0 + (b.j1 - b.j0) / 2; r.j1 = r.j0 + 1; }
            else { r.p0 = b.p0 + (b.p1 - b.p0) / 2; r.p1 = r.p0 + 1; }
        }
        for (int p = r.p0; p < r.p1; ++p)
            for (int j = r.j0; j < r.j1; ++j)
                for (int i = r.i0; i < r.i1; ++i) out.push_back(i + n * (j + m * p));
    }

    // boxes and per-depth sizes; no per-unknown work (cheap even for grids that are refused afterwards)
    int analyse(int n_, int m_, int l_, int leafmax) {
        n = n_; m = m_; l = l_;
        boxes.clear();
        boxes.push_back({Box{0, n, 0, m, 0, l}});
        std::vector<int> axis;
        for (;;) {
            const auto& cur = boxes.back();
            int mw = 0, mh = 0, md = 0;
            for (const Box& b : cur) { mw = std::max(mw, b.i1 - b.i0); mh = std::max(mh, b.j1 - b.j0); md = std::max(md, b.p1 - b.p0); }
            if (std::max(mw, std::max(mh, md)) <= leafmax) break;
            const int ax = (mw >= mh && mw >= md) ? 0 : (mh >= md ? 1 : 2);
            axis.push_back(ax);
            std::vector<Box> next;
            next.reserve(cur.size() * 2);
            for (const Box& b : cur) {
                Box lo = b, hi = b;
                if (ax == 0) { const int mid = b.i0 + (b.i1 - b.i0) / 2; lo.i1 = mid; hi.i0 = mid + 1; }
                else if (ax == 1) { const int mid = b.j0 + (b.j1 - b.j0) / 2; lo.j1 = mid; hi.j0 = mid + 1; }
                else { const int mid = b.p0 + (b.p1 - b.p0) / 2; lo.p1 = mid; hi.p0 = mid + 1; }
                next.push_back(lo);
                next.push_back(hi);
            }
            boxes.push_back(std::move(next));
        }
        D = (int)boxes.size() - 1;
        if (D > 254) return fail(LS_ERR_UNSUPPORTED, "dissection deeper than 254 levels");
        lev.assign((size_t)D + 1, LevelShape());
        for (int d = 0; d <= D; ++d) {
            LevelShape& L = lev[d];
            const auto& bx = boxes[d];
            L.count = (int)bx.size();
            L.leaf = (d == D);
            L.axis = L.leaf ? 0 : axis[d];
            L.ns.resize(bx.size()); L.nb.resize(bx.size());
            long Sp = 0, Bp = 0;
            for (size_t t = 0; t < bx.size(); ++t) {
                const Box& b = bx[t];
                if (!(b.i1 > b.i0 && b.j1 > b.j0 && b.p1 > b.p0))
                    return fail(LS_ERR_UNSUPPORTED, "empty region in the dissection of a %ld x %ld x %ld grid", n, m, l);
                const long s = own_size(b, L.leaf, L.axis), r = ring_size(b);
                L.ns[t] = (int)s; L.nb[t] = (int)r;
                Sp = std::max(Sp, s); Bp = std::max(Bp, r);
            }
            L.Sp = (int)Sp; L.Bp = (int)Bp;
        }
        return LS_OK;
    }

    // Device bytes the factorisation needs at its peak: the index maps, packed factor blocks and solve vectors of every
    // depth (kept), plus the largest per-depth transient (the depth's dense fronts, its children's fronts, the inverse
    // and Y work arrays, pivots, child map), plus the matrix values and the entry routing of one depth, plus four
    // N-vectors (tuning and host-pointer staging).  `tight`: solver 2's packed blocks, else identity-padded batches.
    size_t need_bytes(int64_t nnz, bool tight) const {
        const size_t z = 16;                      // complex double
        size_t keep = 0, peak = 0;
        for (int d = 0; d <= D; ++d) {
            const LevelShape& L = lev[d];
            const size_t cnt = L.count, Sp = L.Sp, Bp = L.Bp, Fp = Sp + Bp;
            size_t totS = cnt * Sp * Sp, totB = cnt * Sp * Bp;
            keep += cnt * Sp * 4 + cnt * std::max<size_t>(Bp, 1) * 4 + (d < D ? cnt * 2 * Fp * 4 : 0);
            if (tight) {
                totS = 0; totB = 0;
                for (size_t t = 0; t < cnt; ++t) { totS += (size_t)L.ns[t] * L.ns[t]; totB += (size_t)L.ns[t] * L.nb[t]; }
                keep += cnt * (4 + 4 + 8 + 8);
            }
            keep += (std::max<size_t>(totS, 1) + 2 * std::max<size_t>(totB, 1)) * z;
            keep += (cnt * Fp + cnt * Sp + std::max<size_t>(cnt * Bp, 1)) * z;
            size_t tr = cnt * Fp * Fp * z + cnt * Sp * Sp * z + std::max<size_t>(cnt * Sp * Bp, 1) * z
                        + 2 * cnt * 8 + cnt * Sp * 4 + cnt * 2 * 4;
            if (d < D) {
                const LevelShape& C = lev[d + 1];
                const size_t Fc = (size_t)C.Sp + C.Bp;
                tr += (size_t)C.count * Fc * Fc * z + (size_t)C.count * std::max<size_t>(C.Bp, 1) * 4;
            }
            peak = std::max(peak, tr);
        }
        const size_t nz = (size_t)std::max<int64_t>(nnz, 1);
        return keep + peak + nz * z + (size_t)std::max<int64_t>(nnz, 0) * 12 + 4 * (size_t)N() * z;
    }

    // owners and per-node lists
    int lists() {
        const long NN = N();
        own_depth.assign((size_t)NN, 255);
        own_node.assign((size_t)NN, -1);
        own_loc.assign((size_t)NN, -1);
        Sidx.assign((size_t)D + 1, {});
        Bidx.assign((size_t)D + 1, {});
        std::vector<int> tmp;
        for (int d = 0; d <= D; ++d) {
            const LevelShape& L = lev[d];
            const size_t Sp = L.Sp, Bp = L.Bp;
            Sidx[d].assign((size_t)L.count * Sp, -1);
            Bidx[d].assign((size_t)L.count * std::max<size_t>(Bp, 1), -1);
            for (int t = 0; t < L.count; ++t) {
                own_list(boxes[d][t], L.leaf, L.axis, tmp);
                for (size_t q = 0; q < tmp.size(); ++q) {
                    const int g = tmp[q];
                    Sidx[d][(size_t)t * Sp + q] = g;
                    own_depth[g] = (unsigned char)d; own_node[g] = t; own_loc[g] = (int)q;
                }
                ring_list(boxes[d][t], tmp);
                for (size_t q = 0; q < tmp.size(); ++q) Bidx[d][(size_t)t * Bp + q] = tmp[q];
            }
        }
        for (long g = 0; g < NN; ++g)
            if (own_node[g] < 0) return fail(LS_ERR_CUDA, "internal error, unknown %ld has no owner", g);
        return LS_OK;
    }

    // route every matrix entry (1-based CSC) to the front that assembles it; refuses entries outside the 27-point
    // pattern (9-point when l = 1), duplicate (row, col) entries and rows out of range
    int route(const int64_t* colptr, const int64_t* rowval) {
        const long NN = N();
        edest.assign((size_t)D + 1, {});
        esrc.assign((size_t)D + 1, {});
        std::vector<int> seen((size_t)NN, -1);         // column that last held row r
        const int pts = l > 1 ? 27 : 9;
        for (long c = 0; c < NN; ++c) {
            if (colptr[c + 1] < colptr[c]) return fail(LS_ERR_INVALID, "colptr decreases at column %ld", c + 1);
            const int ic = (int)(c % n), jc = (int)((c / n) % m), pc = (int)(c / ((long)n * m));
            for (int64_t q = colptr[c] - 1; q < colptr[c + 1] - 1; ++q) {
                const long r = rowval[q] - 1;
                if (r < 0 || r >= NN) return fail(LS_ERR_INVALID, "row index %ld out of range in column %ld", r + 1, c + 1);
                if (seen[r] == (int)c) return fail(LS_ERR_INVALID, "duplicate entry (%ld, %ld)", r + 1, c + 1);
                seen[r] = (int)c;
                const int ir = (int)(r % n), jr = (int)((r / n) % m), pr = (int)(r / ((long)n * m));
                if (std::abs(ir - ic) > 1 || std::abs(jr - jc) > 1 || std::abs(pr - pc) > 1)
                    return fail(LS_ERR_UNSUPPORTED, "entry (%ld, %ld) couples unknowns further apart than the %ld-point stencil",
                                r + 1, c + 1, pts);
                const int dr = own_depth[r], dc = own_depth[c];
                int d, t, lr, lc;
                if (dr == dc) {
                    if (own_node[r] != own_node[c])
                        return fail(LS_ERR_CUDA, "internal error, entry (%ld, %ld) joins two nodes of one depth", r + 1, c + 1);
                    d = dr; t = own_node[r]; lr = own_loc[r]; lc = own_loc[c];
                } else if (dr > dc) {
                    d = dr; t = own_node[r]; lr = own_loc[r];
                    const int k = ring_index(boxes[d][t], ic, jc, pc);
                    if (k < 0) return fail(LS_ERR_CUDA, "internal error, entry (%ld, %ld) outside its front", r + 1, c + 1);
                    lc = lev[d].Sp + k;
                } else {
                    d = dc; t = own_node[c]; lc = own_loc[c];
                    const int k = ring_index(boxes[d][t], ir, jr, pr);
                    if (k < 0) return fail(LS_ERR_CUDA, "internal error, entry (%ld, %ld) outside its front", r + 1, c + 1);
                    lr = lev[d].Sp + k;
                }
                const long Fp = lev[d].Sp + lev[d].Bp;
                edest[d].push_back((long)t * Fp * Fp + lr + (long)lc * Fp);
                esrc[d].push_back((int)q);
            }
        }
        return LS_OK;
    }

    // child -> parent maps
    int maps() {
        cmap.assign((size_t)D + 1, {});
        pmap.assign((size_t)D + 1, {});
        for (int d = 0; d < D; ++d) {
            const LevelShape& L = lev[d];
            const LevelShape& Lc = lev[d + 1];
            const int Fp = L.Sp + L.Bp;
            pmap[d].assign((size_t)L.count * 2 * Fp, -1);
            cmap[d + 1].assign((size_t)Lc.count * std::max(Lc.Bp, 1), -1);
            for (int t = 0; t < L.count; ++t)
                for (int side = 0; side < 2; ++side) {
                    const int c = 2 * t + side;
                    for (int k = 0; k < Lc.Bp; ++k) {
                        const int g = Bidx[d + 1][(size_t)c * Lc.Bp + k];
                        if (g < 0) continue;
                        int p;
                        if (own_depth[g] == d && own_node[g] == t) p = own_loc[g];
                        else {
                            const int q = ring_index(boxes[d][t], g % n, (g / n) % m, g / (n * m));
                            if (q < 0) return fail(LS_ERR_CUDA, "internal error, child ring unknown %ld outside the parent front", g);
                            p = L.Sp + q;
                        }
                        cmap[d + 1][(size_t)c * Lc.Bp + k] = p;
                        pmap[d][((size_t)t * 2 + side) * Fp + p] = k;
                    }
                }
        }
        return LS_OK;
    }
};

}  // namespace lsmsp
