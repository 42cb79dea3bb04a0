// vi_ccl.cuh -- run-based connected-component labelling of a bit-packed mask
// inside one CTA.  A "run" is a maximal horizontal span of set pixels; runs are
// numbered 1..R in raster order (node 0 is the virtual "outside the crop" node
// used by the hole fill).  Union-find over runs:
//   A  link every run to the first overlapping run of the row above,
//   B  pointer jumping,
//   C  lock-free unions for every further overlap (and with node 0 for runs
//      that touch the crop border when `border` is set),
//   D  pointer jumping.
// After build, parent[i] is the smallest run id of i's component -- the run that
// holds the component's first pixel in raster order, so ranking roots by id gives
// the raster-canonical label order (SURVEY A.7).
//
// Used five times per unit: background 4-connected hole fill (segmentation.py:
// 27-72 and the hole filling implied by drawContours(FILLED), indexing_ui.py:1554),
// largest 8-connected component (indexing_ui.py:2240-2248, :1505-1510) and the
// per-component contour-area filter (indexing_ui.py:1540-1558).
#pragma once
#include "vi_device.cuh"

namespace vi {

// Three words, not seven pointers: the arrays are derived from the base on use, so a workspace choice is one
// select and nothing of it has to be held across phases.
struct CclWs {
    unsigned char* base;
    int cap;
    int rf;               // bytes of the row_first table
    __device__ __forceinline__ int* row_first() const { return reinterpret_cast<int*>(base); }            // [h+2] first run id of each row; [h] = R+1
    __device__ __forceinline__ int* parent() const { return reinterpret_cast<int*>(base + rf); }          // [cap+1]
    __device__ __forceinline__ unsigned* acc0() const { return reinterpret_cast<unsigned*>(base + rf + (cap + 1) * 4); }   // per-root accumulator
    __device__ __forceinline__ unsigned* acc1() const { return reinterpret_cast<unsigned*>(base + rf + (cap + 1) * 8); }   // per-root accumulator
    __device__ __forceinline__ unsigned short* xs() const { return reinterpret_cast<unsigned short*>(base + rf + (cap + 1) * 12); }
    __device__ __forceinline__ unsigned short* xe() const { return reinterpret_cast<unsigned short*>(base + rf + (cap + 1) * 14); }
    __device__ __forceinline__ unsigned short* yy() const { return reinterpret_cast<unsigned short*>(base + rf + (cap + 1) * 16); }
};

// A table of `cap` runs at `base` takes ccl_ws_bytes(cap, h) (vi_device.cuh); `rf` = ccl_rowfirst_bytes(h).
__device__ inline CclWs ccl_ws_carve(unsigned char* base, int cap, int rf) {
    CclWs ws;
    ws.base = base; ws.cap = cap; ws.rf = rf;
    return ws;
}

__device__ __forceinline__ int uf_find(const volatile int* parent, int x) {
    int p = parent[x];
    while (p != x) { x = p; p = parent[x]; }
    return x;
}

__device__ inline void uf_unite(int* parent, int a, int b) {
    while (true) {
        a = uf_find(parent, a);
        b = uf_find(parent, b);
        if (a == b) return;
        if (a < b) { int t = a; a = b; b = t; }
        int old = atomicCAS(&parent[a], a, b);
        if (old == a) return;
    }
}

__device__ inline void ccl_jump(int* parent, int R) {
    // pointer jumping until every node points at its root
    while (true) {
        int changed = 0;
        for (int i = 1 + threadIdx.x; i <= R; i += kThreads) {
            const int p = parent[i];
            VI_CHECK(p >= 0 && p <= R, CHK_UF_PARENT);
            int q = parent[p];
            q = parent[q];
            q = parent[q];
            q = parent[q];
            if (q != p) { parent[i] = q; changed = 1; }
        }
        if (!cta_sync_or(changed)) break;
    }
}

// Start / end bit masks of the runs inside word c of row y.
__device__ __forceinline__ void run_edges(const unsigned* M, const Geom& g, int y, int c, unsigned& starts, unsigned& ends) {
    unsigned m = M[y * g.wpr + c];
    unsigned prev = c > 0 ? M[y * g.wpr + c - 1] : 0u;
    unsigned next = c < g.wpr - 1 ? M[y * g.wpr + c + 1] : 0u;
    starts = m & ~((m << 1) | (prev >> 31));
    ends = m & ~((m >> 1) | (next << 31));
}

// Builds runs + components of mask M.  ws_s (shared) is used when the runs fit,
// else ws_g (global scratch).  Returns R (run count) and the workspace used.
template <class PT>
VI_PHASE int ccl_build(Cta& cs, const unsigned* M, const Geom& g, bool conn8, bool border,
                       const CclWs& ws_s, const CclWs& ws_g, CclWs& ws, PT* pt) {
    const int per = (g.nwords + kThreads - 1) / kThreads;
    const int i0 = threadIdx.x * per;
    const int i1 = min(i0 + per, g.nwords);
    unsigned ns = 0, ne = 0;
    for (int i = i0; i < i1; ++i) {
        int y, c; word_rc(g, i, y, c);
        unsigned s, e;
        run_edges(M, g, y, c, s, e);
        ns += __popc(s);
        ne += __popc(e);
    }
    unsigned os = ns, oe = ne, R, Re;
    cta_excl_scan2(cs, os, oe, R, Re);
    if (pt) pt->acc(23);
    ws = ((int)R <= ws_s.cap) ? ws_s : ws_g;
    VI_CHECK((int)R <= ws.cap && R == Re, CHK_RUN_CAP);            // every start has its end; the global table holds any mask
    for (int i = i0; i < i1; ++i) {
        int y, c; word_rc(g, i, y, c);
        unsigned s, e;
        run_edges(M, g, y, c, s, e);
        if (c == 0) ws.row_first()[y] = (int)os + 1;
        while (s) {
            int b = __ffs(s) - 1; s &= s - 1;
            ++os;
            VI_CHECK(os >= 1 && os <= R, CHK_RUN_INDEX);
            ws.xs()[os] = (unsigned short)(c * 32 + b);
            ws.yy()[os] = (unsigned short)y;
        }
        while (e) {
            int b = __ffs(e) - 1; e &= e - 1;
            ++oe;
            VI_CHECK(oe >= 1 && oe <= R, CHK_RUN_INDEX);
            ws.xe()[oe] = (unsigned short)(c * 32 + b);
        }
    }
    if (threadIdx.x == 0) { ws.row_first()[g.h] = (int)R + 1; ws.parent()[0] = 0; ws.acc0()[0] = 0; ws.acc1()[0] = 0; }
    cta_sync();
    if (pt) pt->acc(24);
    const int c8 = conn8 ? 1 : 0;
    if (threadIdx.x == 0) cs.s->flag = 0;
    // Fast path: a stack of single runs, one per consecutive row, each touching the one above -- a solid blob, what
    // a filled plate mask is -- is one component by inspection: every run points at run 1 and the union-find is skipped.
    if (!border) {
        int ok = 1;
        for (int i = 2 + threadIdx.x; i <= (int)R; i += kThreads) {
            const int y = ws.yy()[i], xs = ws.xs()[i], xe = ws.xe()[i];
            ok &= (y == (int)ws.yy()[i - 1] + 1) && (xs <= (int)ws.xe()[i - 1] + c8) && (xe >= (int)ws.xs()[i - 1] - c8);
        }
        if (!cta_sync_or(!ok) && R > 0) {
            for (int i = 1 + threadIdx.x; i <= (int)R; i += kThreads) { ws.parent()[i] = 1; ws.acc0()[i] = 0; ws.acc1()[i] = 0; }
            if (threadIdx.x == 0) cs.s->flag = 1;             // one component: ccl_largest sums it directly
            cta_sync();
            if (pt) pt->acc(25);
            return (int)R;
        }
    }
    // Fast path of the hole fill: when every background run touches the crop border itself there is no hole (what the
    // background of a sparse defect mask, or of a plate without bright inclusions, looks like): all runs join node 0.
    if (border) {
        int inner = 0;
        for (int i = 1 + threadIdx.x; i <= (int)R; i += kThreads) {
            const int y = ws.yy()[i];
            inner |= !(y == 0 || y == g.h - 1 || ws.xs()[i] == 0 || (int)ws.xe()[i] == g.w - 1);
        }
        if (!cta_sync_or(inner)) {
            for (int i = 1 + threadIdx.x; i <= (int)R; i += kThreads) { ws.parent()[i] = 0; ws.acc0()[i] = 0; ws.acc1()[i] = 0; }
            cta_sync();
            if (pt) pt->acc(25);
            return (int)R;
        }
    }
    // A: primary link = first overlapping run of the row above
    for (int i = 1 + threadIdx.x; i <= (int)R; i += kThreads) {
        int y = ws.yy()[i];
        int link = i;
        if (y > 0) {
            int j0 = ws.row_first()[y - 1], j1 = ws.row_first()[y];
            int xs = ws.xs()[i], xe = ws.xe()[i];
            int lo = j0, hi = j1;            // first j with xe[j] >= xs - c8
            while (lo < hi) {
                int mid = (lo + hi) >> 1;
                if ((int)ws.xe()[mid] < xs - c8) lo = mid + 1; else hi = mid;
            }
            if (lo < j1 && (int)ws.xs()[lo] <= xe + c8) link = lo;
            VI_CHECK(j0 >= 1 && j0 <= j1 && j1 <= i, CHK_ROW_TABLE);
        }
        ws.parent()[i] = link;
        ws.acc0()[i] = 0;
        ws.acc1()[i] = 0;
    }
    cta_sync();
    if (pt) pt->acc(25);
    ccl_jump(ws.parent(), (int)R);
    if (pt) pt->acc(26);
    // C: remaining overlaps and the border link
    for (int i = 1 + threadIdx.x; i <= (int)R; i += kThreads) {
        int y = ws.yy()[i];
        int xs = ws.xs()[i], xe = ws.xe()[i];
        if (y > 0) {
            int j0 = ws.row_first()[y - 1], j1 = ws.row_first()[y];
            int lo = j0, hi = j1;
            while (lo < hi) {
                int mid = (lo + hi) >> 1;
                if ((int)ws.xe()[mid] < xs - c8) lo = mid + 1; else hi = mid;
            }
            for (int j = lo + 1; j < j1 && (int)ws.xs()[j] <= xe + c8; ++j) uf_unite(ws.parent(), i, j);
        }
        if (border && (y == 0 || y == g.h - 1 || xs == 0 || xe == g.w - 1)) uf_unite(ws.parent(), i, 0);
    }
    cta_sync();
    if (pt) pt->acc(27);
    ccl_jump(ws.parent(), (int)R);
    if (pt) pt->acc(28);
    return (int)R;
}

// Row scan: the shortcut in front of the labelling passes.  One thread per row finds the row's first / last set pixel
// and its pixel count (one run <=> count == last - first + 1).
//   any_multi : some row holds more than one run.  If none does, every background run touches the left or right crop
//               border, so the mask has no holes (the hole fill is the identity).
//   solid     : no such row, the occupied rows are consecutive and each run touches the one above (8-connectivity):
//               the mask is ONE component -- what a filled plate mask and its erosion are -- and area / coordinate
//               sums come straight from the row table.  No run table, no union-find, no paint.
// `info` : h words of scratch.
struct RowScan { bool any_multi, solid; unsigned area; unsigned long long sx, sy; };

VI_PHASE RowScan mask_row_scan(Cta& cs, const unsigned* M, const Geom& g, unsigned* info) {
    RowScan r;
    r.any_multi = false; r.solid = false; r.area = 0; r.sx = 0; r.sy = 0;
    unsigned long long area = 0, sx = 0, sy = 0;
    int multi = 0;
    for (int y = threadIdx.x; y < g.h; y += kThreads) {
        const unsigned* row = M + y * g.wpr;
        int xs = -1, xe = 0;
        unsigned n = 0;
        for (int c = 0; c < g.wpr; ++c) {
            const unsigned m = row[c];
            if (m) {
                if (xs < 0) xs = c * 32 + __ffs(m) - 1;
                xe = c * 32 + 31 - __clz(m);
                n += __popc(m);
            }
        }
        info[y] = n ? ((unsigned)xs | ((unsigned)xe << 16)) : 0xffffffffu;
        if (n) {
            multi |= (int)n != xe - xs + 1;
            area += n; sx += (unsigned long long)(xs + xe) * n / 2; sy += (unsigned long long)y * n;
        }
    }
    r.any_multi = cta_sync_or(multi) != 0;          // the barrier also publishes `info`
    if (r.any_multi) return r;
    unsigned long long firsts = 0, bad = 0;
    for (int y = threadIdx.x; y < g.h; y += kThreads) {
        const unsigned me = info[y];
        if (me == 0xffffffffu) continue;
        const unsigned up = y > 0 ? info[y - 1] : 0xffffffffu;
        if (up == 0xffffffffu) { ++firsts; continue; }
        const int xs = (int)(me & 0xffffu), xe = (int)(me >> 16), pxs = (int)(up & 0xffffu), pxe = (int)(up >> 16);
        if (!(xs <= pxe + 1 && xe >= pxs - 1)) bad = 1;
    }
    // coordinate sums stay below 2^48 (w, h < 2^16, area < 2^32): the two flag counts ride in the top 16 bits
    unsigned a32 = (unsigned)area;
    unsigned long long vx = sx | (firsts << 48), vy = sy | (bad << 48);
    cta_sum3(cs, a32, vx, vy);
    r.area = a32;
    r.solid = (vx >> 48) == 1u && (vy >> 48) == 0u;
    r.sx = vx & 0xffffffffffffull; r.sy = vy & 0xffffffffffffull;
    return r;
}

// The same for a mask that flood_border_background has just filled straight from its seeding round (return value 2):
// then every row but the first and the last is empty or the single run from its first to its last foreground pixel --
// the extents `info` already holds from the scan before the fill -- so no word is read again (the two edge rows, which
// the fill leaves as they are, are counted once more to see whether they are single runs).  One barrier.
VI_PHASE RowScan mask_row_rescan_filled(Cta& cs, const unsigned* M, const Geom& g, const unsigned* info) {
    RowScan r;
    r.any_multi = false;
    unsigned long long area = 0, sx = 0, sy = 0, firsts = 0, bad = 0;
    for (int y = threadIdx.x; y < g.h; y += kThreads) {
        const unsigned me = info[y];
        if (me == 0xffffffffu) continue;
        const int xs = (int)(me & 0xffffu), xe = (int)(me >> 16);
        const unsigned n = (unsigned)(xe - xs + 1);
        if (y == 0 || y == g.h - 1) {
            unsigned cnt = 0;
            for (int c = 0; c < g.wpr; ++c) cnt += __popc(M[y * g.wpr + c]);
            if (cnt != n) bad = 1;                                 // an edge row with several runs: not one solid blob
        }
        area += n; sx += (unsigned long long)(xs + xe) * n / 2; sy += (unsigned long long)y * n;
        const unsigned up = y > 0 ? info[y - 1] : 0xffffffffu;
        if (up == 0xffffffffu) { ++firsts; continue; }
        const int pxs = (int)(up & 0xffffu), pxe = (int)(up >> 16);
        if (!(xs <= pxe + 1 && xe >= pxs - 1)) bad = 1;
    }
    unsigned a32 = (unsigned)area;
    unsigned long long vx = sx | (firsts << 48), vy = sy | (bad << 48);
    cta_sum3(cs, a32, vx, vy);
    r.area = a32;
    r.solid = (vx >> 48) == 1u && (vy >> 48) == 0u;
    r.sx = vx & 0xffffffffffffull; r.sy = vy & 0xffffffffffffull;
    return r;
}

// Hole fill without labelling.  The background that is 4-connected to the crop border is grown directly on the bit
// rows: one thread owns one row and, per round, seeds it with what is already reached in the row itself and in the
// rows above and below, then extends every seed to the ends of its background run (an addition ripples a carry
// through a run of ones: left to right on the words, right to left on their bit reversals).  A round crosses any
// number of pixels horizontally and one row vertically; round 0 seeds the runs that touch the row's ends and the
// whole first / last row.  Reads of neighbour rows may see a round's old or new words -- both are subsets of the true
// reachable set, so the iteration is monotone and its fixed point is exact.  A plate with inclusions converges at
// once; if `kFloodRounds` do not suffice (spirals, long vertical channels) the caller labels the background instead.
//   M: the mask (foreground);  R: scratch, receives the reached background;  returns non-zero when converged (2: by the
//   seeding round alone), and then M | holes == ~R & row mask.
constexpr int kFloodRounds = 5;

VI_PHASE int flood_border_background(const unsigned* M, unsigned* R, const Geom& g) {
    const unsigned lastbit = 1u << ((g.w - 1) & 31);
    // Round 0, seeds only: the first and last row reach all of their background; every other row the background run
    // at its left end and the one at its right end (what the carry trick below would make of two end seeds): the words
    // up to the first foreground pixel from either side, a handful of word steps per row instead of two passes over all.
    for (int y = threadIdx.x; y < g.h; y += kThreads) {
        const unsigned* mrow = M + y * g.wpr;
        unsigned* rrow = R + y * g.wpr;
        if (y == 0 || y == g.h - 1) {
            for (int c = 0; c < g.wpr; ++c) rrow[c] = ~mrow[c] & row_mask_of(g, c);
            continue;
        }
        int c = 0;
        for (; c < g.wpr; ++c) {                                 // from the left
            const unsigned full = row_mask_of(g, c), b = ~mrow[c] & full;
            if (b == full) { rrow[c] = b; continue; }
            const int n = __ffs(~b) - 1;                          // background pixels before the first foreground one (or the row's end)
            rrow[c] = n ? (0xffffffffu >> (32 - n)) : 0u;
            break;
        }
        if (c >= g.wpr) continue;                                // no foreground in this row: all reached
        const int cl = c;
        int cr = g.wpr - 1;
        for (; cr > cl; --cr) {                                  // from the right, down to the word the left run stopped in
            const unsigned full = row_mask_of(g, cr), b = ~mrow[cr] & full;
            if (b == full) { rrow[cr] = b; continue; }
            const int top = 31 - __clz(full);                     // the row's last pixel in this word
            const int n = __clz(~b << (31 - top));                // background pixels after the last foreground one
            rrow[cr] = n ? (full & ~(0xffffffffu >> (31 - top + n))) & full : 0u;
            break;
        }
        if (cr == cl) {                                          // both runs end in the same word
            const unsigned full = row_mask_of(g, cl), b = ~mrow[cl] & full;
            const int top = 31 - __clz(full);
            const int n = __clz(~b << (31 - top));
            rrow[cl] |= n ? (full & ~(0xffffffffu >> (31 - top + n))) & full : 0u;
        } else {
            for (int k = cl + 1; k < cr; ++k) rrow[k] = 0u;      // between the two runs: not reached yet
        }
    }
    for (int round = 0; round <= kFloodRounds; ++round) {
        int changed = 0;
        if (round > 0)
        for (int y = threadIdx.x; y < g.h; y += kThreads) {
            const unsigned* mrow = M + y * g.wpr;
            unsigned* rrow = R + y * g.wpr;
            const unsigned* up = R + max(y - 1, 0) * g.wpr;
            const unsigned* dn = R + min(y + 1, g.h - 1) * g.wpr;
            const bool edge_row = y == 0 || y == g.h - 1;
            // left to right: seeds and their extension towards higher x
            unsigned carry = 0, diff = 0;
            for (int c = 0; c < g.wpr; ++c) {
                const unsigned b = ~mrow[c] & row_mask_of(g, c);
                unsigned s;
                if (round == 0) s = edge_row ? b : ((c == 0 ? 1u : 0u) | (c == g.wpr - 1 ? lastbit : 0u));
                else s = rrow[c] | up[c] | dn[c];
                s = (s | carry) & b;
                const unsigned sum = b + s;
                carry = sum < b ? 1u : 0u;                     // the run reaches bit 31: it goes on in the next word
                const unsigned v = ((sum ^ b) & b) | s;
                if (round != 0) diff |= v ^ rrow[c];
                rrow[c] = v;
            }
            // right to left: extension towards lower x
            carry = 0;
            for (int c = g.wpr - 1; c >= 0; --c) {
                const unsigned b = __brev(~mrow[c] & row_mask_of(g, c));
                const unsigned old = rrow[c];
                const unsigned s = (__brev(old) | carry) & b;
                const unsigned sum = b + s;
                carry = sum < b ? 1u : 0u;
                const unsigned v = old | __brev((sum ^ b) & b);
                diff |= v ^ old;
                rrow[c] = v;
            }
            changed |= diff != 0u;
        }
        if (round == 0) {
            // The seeds' rows usually reach everything at once (a plate in a bright field: every background row
            // runs in from the border).  Checked word-parallel instead of by a second serial round: converged iff
            // no unreached background pixel has a reached 4-neighbour.
            cta_sync();
            int grow = 0;
            for (int i = threadIdx.x; i < g.nwords; i += kThreads) {
                int y, c; word_rc(g, i, y, c);
                const unsigned r = R[i];
                const unsigned unre = ~M[i] & row_mask_of(g, c) & ~r;
                if (unre) {
                    const unsigned lw = c > 0 ? R[i - 1] : 0u, rw = c < g.wpr - 1 ? R[i + 1] : 0u;
                    const unsigned up = y > 0 ? R[i - g.wpr] : 0u, dn = y < g.h - 1 ? R[i + g.wpr] : 0u;
                    const unsigned nb = (r << 1) | (lw >> 31) | (r >> 1) | (rw << 31) | up | dn;
                    grow |= (unre & nb) != 0u;
                }
            }
            if (!cta_sync_or(grow)) return 2;                    // settled by the seeds alone
        } else if (!cta_sync_or(changed)) return 1;
    }
    return 0;
}

// Warp-aggregated per-root accumulation: lanes whose root equals the first valid
// lane's root are reduced with REDUX and added once; the rest add individually.
__device__ __forceinline__ void agg_add(unsigned* acc, bool valid, int root, unsigned val) {
    unsigned vm = __ballot_sync(kFull, valid);
    if (vm == 0) return;
    int lead = __shfl_sync(kFull, root, __ffs(vm) - 1);
    bool same = valid && root == lead;
    unsigned sum = __reduce_add_sync(kFull, same ? val : 0u);
    if (lane_id() == 0 && sum) atomicAdd(&acc[lead], sum);
    if (valid && !same && val) atomicAdd(&acc[root], val);
}

__device__ __forceinline__ void agg_min(unsigned* acc, bool valid, int root, unsigned val) {
    unsigned vm = __ballot_sync(kFull, valid);
    if (vm == 0) return;
    int lead = __shfl_sync(kFull, root, __ffs(vm) - 1);
    bool same = valid && root == lead;
    unsigned mn = __reduce_min_sync(kFull, same ? val : 0xffffffffu);
    if (lane_id() == 0 && mn != 0xffffffffu) atomicMin(&acc[lead], mn);
    if (valid && !same) atomicMin(&acc[root], val);
}

// dst[word] = OR of the spans of all runs of that row whose root satisfies pred,
// optionally OR-ed with `base` (may be null).  Word-parallel, no atomics.
template <class Pred>
VI_PHASE void ccl_paint(unsigned* dst, const unsigned* base, const Geom& g, const CclWs& ws, Pred pred) {
    for (int i = threadIdx.x; i < g.nwords; i += kThreads) {
        int y, c; word_rc(g, i, y, c);
        int x0 = c * 32, x1 = x0 + 31;
        int j0 = ws.row_first()[y], j1 = ws.row_first()[y + 1];
        VI_CHECK(j0 >= 1 && j0 <= j1 && j1 <= ws.cap + 1, CHK_PAINT_RUN);
        int lo = j0, hi = j1;                 // first run with xe >= x0
        while (lo < hi) {
            int mid = (lo + hi) >> 1;
            if ((int)ws.xe()[mid] < x0) lo = mid + 1; else hi = mid;
        }
        unsigned bits = 0;
        for (int j = lo; j < j1; ++j) {
            int xs = ws.xs()[j];
            if (xs > x1) break;
            if (pred(ws.parent()[j])) {
                int xe = ws.xe()[j];
                bits |= bit_range(max(xs, x0) - x0, min(xe, x1) - x0);
            }
        }
        dst[i] = base ? (base[i] | bits) : bits;
    }
}

// The first kc kept components of a labelling (after ccl_build and the per-root acc0 of the area filter), in raster
// order of their first pixel, into out[0..kc).  acc1[root] = 1 + slot (an exclusive count of kept roots in increasing
// run id, which is raster order); ccl_build left acc1 zero on every run, and 0 marks a root without a slot, so the
// count stops at the kc-th kept root.  tab: kc accumulators (tab_cap of them fit).  Every thread reaches every barrier.
template <class Keep>
VI_PHASE void ccl_blob_table(Cta& cs, const CclWs& ws, int R, Keep keep, int kc, int tab_cap, BlobAcc* tab,
                             vi_defect_blob* __restrict__ out) {
    unsigned carry = 0;
    for (int base = 0; base < R && (int)carry < kc; base += kThreads) {
        const int i = base + threadIdx.x + 1;
        const bool kept = i <= R && ws.parent()[i] == i && keep(i);
        unsigned a = kept ? 1u : 0u, b = 0, ta, tb;
        cta_excl_scan2(cs, a, b, ta, tb);
        const unsigned s = carry + a;
        if (kept && (int)s < kc) {
            VI_CHECK((int)s < tab_cap, CHK_BLOB_SLOT);
            ws.acc1()[i] = s + 1;
            BlobAcc e;
            e.sx = 0; e.sy = 0; e.area = 0; e.xmin = 0xffffffffu; e.xmax = 0; e.ymin = ws.yy()[i]; e.ymax = 0; e.area2 = ws.acc0()[i];
            tab[s] = e;
        }
        carry += ta;
    }
    cta_sync();
    for (int i = 1 + threadIdx.x; i <= R; i += kThreads) {
        const unsigned s = ws.acc1()[ws.parent()[i]] - 1u;        // (no slot: 0xffffffff)
        if (s < (unsigned)kc) {
            VI_CHECK((int)s < tab_cap, CHK_BLOB_SLOT);
            const unsigned xs = ws.xs()[i], xe = ws.xe()[i], y = ws.yy()[i], len = xe - xs + 1;
            BlobAcc& e = tab[s];
            atomicAdd(&e.area, len);
            atomicMin(&e.xmin, xs);
            atomicMax(&e.xmax, xe);
            atomicMax(&e.ymax, y);
            atomicAdd(&e.sx, (unsigned long long)(xs + xe) * len / 2);
            atomicAdd(&e.sy, (unsigned long long)y * len);
        }
    }
    cta_sync();
    for (int j = threadIdx.x; j < kc; j += kThreads) {
        const BlobAcc e = tab[j];
        vi_defect_blob o;
        o.x = (int)e.xmin; o.y = (int)e.ymin; o.w = (int)(e.xmax - e.xmin + 1); o.h = (int)(e.ymax - e.ymin + 1);
        o.area = (int)e.area; o.area2 = (int)e.area2;
        o.cx = __ddiv_rn((double)e.sx, (double)e.area);              // the record's centroid convention
        o.cy = __ddiv_rn((double)e.sy, (double)e.area);
        out[j] = o;
    }
}

// rows 0..h-1 need row_first for every row, including rows without runs.
// ccl_build writes row_first[y] only from the thread that owns word (y,0), which
// exists for every row, so the table is always complete.

// Largest component (max area; ties -> smallest 2x2-block key, i.e. OpenCV's label
// order, SURVEY A.7).  Returns the root id (0 if there is no run) and its area /
// coordinate sums through the out-params.  Uses acc0 = area, acc1 = min block key.
VI_PHASE int ccl_largest(Cta& cs, const Geom& g, const CclWs& ws, int R,
                                  unsigned& area, unsigned long long& sum_x, unsigned long long& sum_y) {
    area = 0; sum_x = 0; sum_y = 0;
    if (R == 0) return 0;
    if (cs.s->flag) {                                  // ccl_build found a single solid component (root = run 1)
        unsigned long long a = 0, sx = 0, sy = 0;
        for (int i = 1 + threadIdx.x; i <= R; i += kThreads) {
            const unsigned long long xs = ws.xs()[i], xe = ws.xe()[i], len = xe - xs + 1;
            a += len; sx += (xs + xe) * len / 2; sy += (unsigned long long)ws.yy()[i] * len;
        }
        unsigned a32 = (unsigned)a;
        cta_sum3(cs, a32, sx, sy);
        area = a32; sum_x = sx; sum_y = sy;
        return 1;
    }
    const int Rpad = (R + kThreads - 1) / kThreads * kThreads;
    for (int base = 0; base < Rpad; base += kThreads) {
        int i = base + threadIdx.x + 1;
        bool valid = i <= R;
        int root = valid ? ws.parent()[i] : 0;
        unsigned len = valid ? (unsigned)(ws.xe()[i] - ws.xs()[i] + 1) : 0u;
        agg_add(ws.acc0(), valid, root, len);
    }
    cta_sync();
    unsigned long long best = 0;
    for (int i = 1 + threadIdx.x; i <= R; i += kThreads)
        if (ws.parent()[i] == i) {
            unsigned long long a = ws.acc0()[i];
            best = a > best ? a : best;
        }
    unsigned amax = (unsigned)cta_max_u64(cs, best);
    // min block key among the components of maximal area
    const int w2 = (g.w + 1) / 2;
    for (int i = 1 + threadIdx.x; i <= R; i += kThreads) ws.acc1()[i] = 0xffffffffu;
    cta_sync();
    for (int base = 0; base < Rpad; base += kThreads) {
        int i = base + threadIdx.x + 1;
        bool valid = i <= R;
        int root = valid ? ws.parent()[i] : 0;
        valid = valid && ws.acc0()[root] == amax;
        unsigned key = valid ? (unsigned)((ws.yy()[i] >> 1) * w2 + (ws.xs()[i] >> 1)) : 0xffffffffu;
        agg_min(ws.acc1(), valid, root, key);
    }
    cta_sync();
    unsigned long long sel = 0;   // pick (min key) -> encode as max of (~key, root)
    for (int i = 1 + threadIdx.x; i <= R; i += kThreads)
        if (ws.parent()[i] == i && ws.acc0()[i] == amax) {
            unsigned long long v = ((unsigned long long)(0xffffffffu - ws.acc1()[i]) << 32) | (unsigned)i;
            sel = v > sel ? v : sel;
        }
    sel = cta_max_u64(cs, sel);
    int broot = (int)(sel & 0xffffffffu);
    unsigned long long sx = 0, sy = 0;
    for (int i = 1 + threadIdx.x; i <= R; i += kThreads)
        if (ws.parent()[i] == broot) {
            unsigned long long xs = ws.xs()[i], xe = ws.xe()[i];
            unsigned long long len = xe - xs + 1;
            sx += (xs + xe) * len / 2;
            sy += (unsigned long long)ws.yy()[i] * len;
        }
    unsigned long long v2[2] = {sx, sy};
    cta_sum_n<2>(cs, v2);
    sum_x = v2[0]; sum_y = v2[1];
    area = amax;
    return broot;
}

}  // namespace vi
