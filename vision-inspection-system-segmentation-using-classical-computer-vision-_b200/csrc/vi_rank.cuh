// vi_rank.cuh -- P11: |gray - median21(gray)| > thr inside the ROI, without ever
// forming the median (cv2.medianBlur(gray, 21) + absdiff + threshold,
// indexing_ui.py:1522-1527; BORDER_REPLICATE, SURVEY A.9).
//
//   med >  g+thr   <=>  #(window <= g+thr)   <= 220
//   med <= g-thr-1 <=>  #(window <= g-thr-1) >= 221          (441-pixel window)
//
// 1. Three unit-wide levels v_0 <= v_1 <= v_2 around the median of the class the ROI
//    lives in (the dark class: the seg mask is an inverse threshold).
//    C_k(p) = #(window(p) <= v_k) is a 21x21 box sum of per-pixel indicators, kept
//    for the three levels at once in one word of three 10-bit fields (441 < 1024).
// 2. C_k is evaluated exactly only on a lattice: one point per 3x3 cell (its
//    centre).  Moving the window by one pixel swaps one 21-pixel row or column, so
//    |C_k(p) - C_k(q)| <= 21 * L1(p, q) <= 42 inside a cell.  Hence for every pixel
//    of the cell   C_k >= 221 if C_k(centre) >= 263   and   C_k <= 220 if
//    C_k(centre) <= 178,   which brackets the median of every pixel of the cell:
//    LO < med <= HI with LO, HI taken from the level list (or -1 / 255).
// 3. Four byte thresholds per cell decide a pixel: defect for sure (g <= LO-thr or
//    g >= HI+thr+1), clean for sure (HI-thr <= g <= LO+thr+1), else "ambiguous".
//    A cell whose 9 pixels' min and max are both in the clean range is finished
//    (nearly every cell of the plate is).  The others are "dirty": one bit per cell
//    and the cell's bracket code go to a plane in the CTA's L2 scratch; once the ROI
//    exists, the dirty cells that touch it (a ring a few pixels wide along the plate
//    edge, and the defects) are classified per pixel, and ambiguous ROI pixels get an
//    exact rank count at their own two pivots.  Cells of the bright field are dirty by
//    construction (no level brackets their median) and are dropped by the ROI test,
//    six cells (one task of the C pass) at a time.
//    Exact for any level set and any image
//    (oracle/restate.py: residual_mask_lattice is the numpy twin).
//
// Box sums are separable and every stage below is one straight-line pass over the
// whole unit (the workspace sits in the region of the masks, which are not live yet):
//   M   one thread per cell: gray min / max of its 9 pixels -- needs no level, so it
//       runs on 15 warps while warp 0 derives the levels from the histogram.
//   V   one thread per column (whole cells per warp) walks down the rows in 3-row
//       blocks: B(b) = sum of the packed level indicators of the block
//       (field-parallel arithmetic, no table), S(j) = sum of blocks j-3..j+3 (the
//       21-row window of lattice row j) kept by a ring of block sums in registers,
//       and the cell's three columns are added by two shuffles: one store per cell.
//       Columns start 9 left of the crop and end 9 right of it (clamped = replicated
//       border), so a row of cell sums carries three virtual cells either side.
//   C   one thread per (lattice row, 6 consecutive cells): window = 7 cell sums,
//       slid along the group; two field-parallel compares give the bracket, a
//       16-entry table the four byte thresholds, the cell min / max decide clean or
//       dirty; one word per task (6 codes, 6 dirty bits) goes to the plane.
#pragma once
#include "vi_pipeline.cuh"

namespace vi {

static_assert(kLevels == 3, "one word of three 10-bit fields");

struct RankWs {
    unsigned* cs;        // [rows8][P] window-row sums per cell slot (slot = cell + kVPad; the last slot of a row is a dummy)
    unsigned short* cmm; // [nly][cpitch] cell gray min | max << 8
    unsigned* table;     // [16] thresholds U1 | U2 << 8 | U3 << 16 | U4 << 24 by code = n179 * 4 + n263
    unsigned* plane;     // [ntasks] per C task: 6 codes (4 bits each) | 6 dirty bits << 24, in the CTA's global scratch
    unsigned* exact;     // [exact_cap] ambiguous pixels (y << 16 | x), global scratch; more are counted inline
    int exact_cap;
    int* counters;       // shared: [0] dirty cells in the ROI, [1] ambiguous pixels (the first exact_cap of them are listed)
    int P, cpitch, nlx, nly, ngrp, nrb;
    int plane_cap;       // words the plane holds (CHECKED builds)
};

constexpr int kExactWarpMax = 192;       // more ambiguous pixels than this: one thread per pixel instead of one warp

// The cell pass runs before the ROI exists (next to the Otsu scan), the per-pixel pass after it: the plane and the
// list outlive the shared workspace, so they sit in the CTA's global scratch (L2-resident) and the counters in static
// shared memory.
// `lists`: the plane of `plane_words` words, then kExactCap ambiguous pixels (vi_device.cuh: rank_scratch_bytes).
__device__ inline RankWs rank_ws_carve(unsigned char* base, const Geom& g, unsigned char* lists, int plane_words, int* counters) {
    RankWs r;
    r.nlx = rank_nlx(g.w); r.nly = (g.h + kCell - 1) / kCell;
    r.ngrp = rank_ngrp(g.w); r.nrb = (r.nly + 15) >> 4;
    r.P = rank_P(g.w); r.cpitch = rank_cpitch(g.w);
    r.cs = reinterpret_cast<unsigned*>(base) + r.P; base += (((r.nly + 7) & ~7) + 1) * r.P * 4;      // row -1 takes the V pass's first (empty) deferred store
    r.cmm = reinterpret_cast<unsigned short*>(base); base += r.nly * r.cpitch * 2;
    r.table = reinterpret_cast<unsigned*>(base);
    r.counters = counters;
    r.plane = reinterpret_cast<unsigned*>(lists);
    r.plane_cap = plane_words;
    r.exact = r.plane + r.plane_cap;
    r.exact_cap = kExactCap;
    return r;
}

// The four byte thresholds of a bracket code (n179 levels with C >= 179, n263 with C >= 263 at the cell centre).
__device__ __forceinline__ unsigned rank_code_thresholds(const int* lv, int thr, int code) {
    const int n179 = code >> 2, n263 = code & 3;
    const int lo_idx = kLevels - n179;        // levels 0..lo_idx-1 surely have C <= 220: med >  LO
    const int hi_idx = kLevels - n263;        // level hi_idx surely has C >= 221:        med <= HI
    const int LO = lo_idx > 0 ? lv[lo_idx - 1] : -1;
    const int HI = hi_idx < kLevels ? lv[hi_idx] : 255;
    const int U1 = min(max(LO - thr + 1, 0), 255);     // defect if g <  U1
    const int U4 = min(HI + thr, 255);                 // defect if g >  U4
    const int U2 = max(HI - thr, 0);                   // clean needs g >= U2
    const int U3 = min(LO + thr + 1, 255);             // clean needs g <= U3
    return (unsigned)U1 | ((unsigned)U2 << 8) | ((unsigned)U3 << 16) | ((unsigned)U4 << 24);
}

// Warp 0 only (the caller synchronises): the threshold table by bracket code, the list counters.
__device__ inline void rank_tables(const int* lv, int thr, RankWs w) {
    const int lane = lane_id();
    if (lane < 16) w.table[lane] = rank_code_thresholds(lv, thr, lane);
    if (lane < 4) w.counters[lane] = 0;
}

// Exact decision for one pixel: #(window <= g+thr) <= 220 or #(window <= g-thr-1) >= 221.
// (cold: the overflow path of the ambiguous-pixel list and units the lattice does not cover.  Kept out of line and
// rolled: inlined into the nine pixels of a dirty cell it was a quarter of the kernel's instructions)
__device__ __noinline__ bool rank_exact_pixel_thread(const uint8_t* gray, int gp, int w, int h, int thr, int x, int y) {
    const int gv = gray[y * gp + x];
    const int pa = gv + thr, pb = gv - thr - 1;
    int ca = 0, cb = 0;
#pragma unroll 1
    for (int dy = -10; dy <= 10; ++dy) {
        const uint8_t* row = gray + min(max(y + dy, 0), h - 1) * gp;
#pragma unroll 3
        for (int dx = -10; dx <= 10; ++dx) {
            const int v = row[min(max(x + dx, 0), w - 1)];
            ca += v <= pa;
            cb += v <= pb;
        }
    }
    return ca <= 220 || cb >= 221;
}

// Per-pixel classification of one dirty cell (one thread): defect-for-sure pixels of
// the ROI go straight into CAND, ambiguous ones onto the exact list.
__device__ inline void rank_dirty_cell(const uint8_t* gray, const Geom& g, int thr, const unsigned* ROI, unsigned* CAND,
                                       RankWs& w, int ci, int cj, unsigned cw) {
    const unsigned u1 = cw & 255u, u2 = (cw >> 8) & 255u, u3 = (cw >> 16) & 255u, u4 = cw >> 24;
    // most dirty cells (plate edges, bright field) lie outside the ROI: three ROI bits per row decide that first
    const int x0 = ci * kCell, c0 = x0 >> 5, sh = x0 & 31;
    unsigned roi3[kCell];
    unsigned any = 0;
#pragma unroll
    for (int rr = 0; rr < kCell; ++rr) {
        const int y = min(cj * kCell + rr, g.h - 1);
        const unsigned* row = ROI + y * g.wpr;
        unsigned b = row[c0] >> sh;
        if (sh > 29 && c0 + 1 < g.wpr) b |= row[c0 + 1] << (32 - sh);
        roi3[rr] = (cj * kCell + rr < g.h) ? (b & 7u) : 0u;          // bits past the crop edge are 0 in every mask
        any |= roi3[rr];
    }
    if (!any) return;
    // Ambiguous pixels, by the test that is still open (bit rr * 3 + cc): A "more than 220 of the window lie above
    // g + thr" can only hold below the clean range (g < U2), B "at least 221 lie at or below g - thr - 1" only above it
    // (g > U3) -- one list entry per open test, so the exact pass counts against ONE pivot per entry.
    unsigned ambA = 0, ambB = 0;
#pragma unroll
    for (int rr = 0; rr < kCell; ++rr) {
        const int y = cj * kCell + rr;
        if (y >= g.h) break;
#pragma unroll
        for (int cc = 0; cc < kCell; ++cc) {
            const int x = ci * kCell + cc;
            if (x >= g.w) break;
            if (!((roi3[rr] >> cc) & 1u)) continue;
            const unsigned gv = gray[y * g.gp + x];
            if (gv < u1 || gv > u4) atomicOr(&CAND[y * g.wpr + (x >> 5)], 1u << (x & 31));
            else {
                if (gv < u2) ambA |= 1u << (rr * kCell + cc);
                if (gv > u3) ambB |= 1u << (rr * kCell + cc);
            }
        }
    }
    if (!(ambA | ambB)) return;
    int k = atomicAdd(&w.counters[1], __popc(ambA) + __popc(ambB));      // one reservation per cell (a noisy unit lists thousands)
#pragma unroll 1
    for (int t = 0; t < 2; ++t) {
        unsigned amb = t ? ambB : ambA;
        while (amb) {
            const int b = __ffs(amb) - 1; amb &= amb - 1;
            const int rr = b / kCell, cc = b - rr * kCell;
            const int y = cj * kCell + rr, x = ci * kCell + cc;
            VI_CHECK(k >= 0 && y < g.h && x < g.w && x < 0x8000, CHK_EXACT_LIST);
            if (k < w.exact_cap) w.exact[k] = ((unsigned)y << 16) | ((unsigned)t << 15) | (unsigned)x;
            else if (rank_exact_pixel_thread(gray, g.gp, g.w, g.h, thr, x, y)) atomicOr(&CAND[y * g.wpr + (x >> 5)], 1u << (x & 31));
            ++k;
        }
    }
}

// (cold: a dirty cell found when the shared list is full)
__device__ __noinline__ void rank_dirty_cell_cold(const uint8_t* gray, Geom g, int thr, const unsigned* ROI, unsigned* CAND, RankWs w,
                                                  int ci, int cj, unsigned cw) {
    rank_dirty_cell(gray, g, thr, ROI, CAND, w, ci, cj, cw);
}

// M: gray min / max of every cell, four cells (12 pixels = three gray words) per thread and step: the three rows are
// reduced field-parallel on (even bytes, odd bytes) halves, then each cell's three columns.  Rows past the crop repeat
// the last row; words past the crop's last word repeat it (their bytes past the crop edge hold in-crop pixels or stale
// ones: a superset can only turn a clean cell dirty, never the reverse, and dirty cells are classified per pixel).
// Runs on the warps first_warp .. end_warp-1.
// Lattice rows [j_begin, j_end).
VI_PHASE void rank_cmm(const uint8_t* gray, const Geom& g, const RankWs& w, int first_warp, int end_warp, int j_begin, int j_end) {
    const int nth = (end_warp - first_warp) * 32;
    const int t0 = (int)threadIdx.x - first_warp * 32;
    if (t0 < 0 || t0 >= nth || j_end <= j_begin) return;
    const int hm1 = g.h - 1, wq = g.gp >> 2, nqm1 = ((g.w + 3) >> 2) - 1;
    const int nquad = (w.nlx + 3) >> 2;
    const int ntask = nquad * (j_end - j_begin);
    const unsigned mq = magic_of((unsigned)nquad);
    const unsigned* gw = reinterpret_cast<const unsigned*>(gray);
    for (int e = t0; e < ntask; e += nth) {
        const int jr = (int)magic_div((unsigned)e, (unsigned)nquad, mq), q = e - jr * nquad, j = j_begin + jr;
        const int k0 = min(3 * q, nqm1), k1 = min(3 * q + 1, nqm1), k2 = min(3 * q + 2, nqm1);
        const unsigned* r0 = gw + (kCell * j) * wq;
        const unsigned* r1 = gw + min(kCell * j + 1, hm1) * wq;
        const unsigned* r2 = gw + min(kCell * j + 2, hm1) * wq;
        const unsigned a0 = r0[k0], a1 = r0[k1], a2 = r0[k2], b0 = r1[k0], b1 = r1[k1], b2 = r1[k2], c0 = r2[k0], c1 = r2[k1], c2 = r2[k2];
        constexpr unsigned F = 0x00FF00FFu;
        // per word k: (bytes 0, 2) and (bytes 1, 3) of the column-wise min / max over the three rows
        const unsigned en0 = __vimin3_u16x2(a0 & F, b0 & F, c0 & F), on0 = __vimin3_u16x2((a0 >> 8) & F, (b0 >> 8) & F, (c0 >> 8) & F);
        const unsigned en1 = __vimin3_u16x2(a1 & F, b1 & F, c1 & F), on1 = __vimin3_u16x2((a1 >> 8) & F, (b1 >> 8) & F, (c1 >> 8) & F);
        const unsigned en2 = __vimin3_u16x2(a2 & F, b2 & F, c2 & F), on2 = __vimin3_u16x2((a2 >> 8) & F, (b2 >> 8) & F, (c2 >> 8) & F);
        const unsigned ex0 = __vimax3_u16x2(a0 & F, b0 & F, c0 & F), ox0 = __vimax3_u16x2((a0 >> 8) & F, (b0 >> 8) & F, (c0 >> 8) & F);
        const unsigned ex1 = __vimax3_u16x2(a1 & F, b1 & F, c1 & F), ox1 = __vimax3_u16x2((a1 >> 8) & F, (b1 >> 8) & F, (c1 >> 8) & F);
        const unsigned ex2 = __vimax3_u16x2(a2 & F, b2 & F, c2 & F), ox2 = __vimax3_u16x2((a2 >> 8) & F, (b2 >> 8) & F, (c2 >> 8) & F);
        // cells: bytes (0,1,2) (3,4,5) (6,7,8) (9,10,11) of the 12; byte 4k -> e*k low, 4k+1 -> o*k low, 4k+2 -> e*k high, 4k+3 -> o*k high
        const unsigned mn0 = __vimin3_u16x2(en0, on0, en0 >> 16) & 0xFFu, mx0 = __vimax3_u16x2(ex0, ox0, ex0 >> 16) & 0xFFu;
        const unsigned mn1 = __vimin3_u16x2(on0 >> 16, en1, on1) & 0xFFu, mx1 = __vimax3_u16x2(ox0 >> 16, ex1, ox1) & 0xFFu;
        const unsigned mn2 = __vimin3_u16x2(en1 >> 16, on1 >> 16, en2) & 0xFFu, mx2 = __vimax3_u16x2(ex1 >> 16, ox1 >> 16, ex2) & 0xFFu;
        const unsigned mn3 = __vimin3_u16x2(on2, en2 >> 16, on2 >> 16) & 0xFFu, mx3 = __vimax3_u16x2(ox2, ex2 >> 16, ox2 >> 16) & 0xFFu;
        unsigned* o = reinterpret_cast<unsigned*>(w.cmm + j * w.cpitch + 4 * q);           // cpitch is even: word aligned
        o[0] = mn0 | (mx0 << 8) | (mn1 << 16) | (mx1 << 24);
        o[1] = mn2 | (mx2 << 8) | (mn3 << 16) | (mx3 << 24);
    }
}

// Level indicators without a table (table loads with data-dependent addresses were bank-conflict bound):
// with R = 1 | 1<<10 | 1<<20 and T = sum_k (lv_k + 512) << 10k, field k of T - q*R is lv_k + 512 - q in
// [257, 766], so its bit 9 is (q <= lv_k).  The three pixels' bits are added by a full adder on whole words.
constexpr unsigned kRep = 0x00100401u;
constexpr unsigned kBit9 = 0x20080200u;

__device__ __forceinline__ unsigned ind3(unsigned T, unsigned q0, unsigned q1, unsigned q2) {
    const unsigned a = T - q0 * kRep, b = T - q1 * kRep, c = T - q2 * kRep;
    const unsigned lo = (a ^ b ^ c) & kBit9, hi = ((a & b) | (c & (a | b))) & kBit9;
    return (lo + 2 * hi) >> 9;
}

// V pass, one thread per (cell slot, segment of lattice rows).  A thread owns the three columns of its cell and walks
// down in 3-row blocks: nine gray bytes per block, their level indicators counted per field by three full adders and
// two additions, the sliding 7-block sum kept by a ring of block sums (registers: the loop is unrolled by 8 so every
// ring index is static), one store per block.  No cross-lane traffic: the shared-memory pipe takes about one
// instruction per two cycles and was this pass's bound with one thread per column (three byte loads, two shuffles
// and a store per column and block; now ten instructions per cell and block instead of eighteen).  Segments of rows
// put enough warps on a unit; each warms its ring up with the six blocks above its first row.
struct VState {
    unsigned S;
    unsigned r[8];
    unsigned q[9];             // gray of the next block (3 rows x 3 columns), loaded one block ahead
};

__device__ __forceinline__ unsigned ind9(unsigned T, const unsigned* q) {
    return ind3(T, q[0], q[1], q[2]) + ind3(T, q[3], q[4], q[5]) + ind3(T, q[6], q[7], q[8]);
}

// Eight lattice rows j0 .. j0+7 <-> blocks b = j0+3 .. j0+10 (sequence n = b+3, ring slot n & 7).
template <bool CLAMP>
__device__ __forceinline__ void v_oct(VState& st, unsigned T, const uint8_t* c0, const uint8_t* c1, const uint8_t* c2, int gp, int hm1,
                                      int j0, unsigned* csp, int P) {
    int rn = kCell * (j0 + 4);                                     // first row of block j0+4 (the first load of this call)
    const uint8_t* p0 = c0 + rn * gp;
    const uint8_t* p1 = c1 + rn * gp;
    const uint8_t* p2 = c2 + rn * gp;
#pragma unroll
    for (int u = 0; u < 8; ++u) {
        const unsigned B = ind9(T, st.q);                           // block b = j0+3+u
        if (CLAMP) {
            const int o0 = min(rn, hm1) * gp, o1 = min(rn + 1, hm1) * gp, o2 = min(rn + 2, hm1) * gp;
            st.q[0] = c0[o0]; st.q[1] = c0[o1]; st.q[2] = c0[o2];
            st.q[3] = c1[o0]; st.q[4] = c1[o1]; st.q[5] = c1[o2];
            st.q[6] = c2[o0]; st.q[7] = c2[o1]; st.q[8] = c2[o2];
            rn += kCell;
        } else {
            st.q[0] = p0[0]; st.q[1] = p0[gp]; st.q[2] = p0[2 * gp];
            st.q[3] = p1[0]; st.q[4] = p1[gp]; st.q[5] = p1[2 * gp];
            st.q[6] = p2[0]; st.q[7] = p2[gp]; st.q[8] = p2[2 * gp];
            p0 += kCell * gp; p1 += kCell * gp; p2 += kCell * gp;
        }
        const int slot = (6 + u) & 7, old = (7 + u) & 7;
        st.S += B - st.r[old];
        st.r[slot] = B;
        *csp = st.S;                                                // lanes past the last slot write the dummy slot
        csp += P;
    }
}

// C: one task = kGrp consecutive cells of one lattice row.  The window of cell i is the seven cells i-3 .. i+3 = slots
// i .. i+6 of the row; a thread forms the first window and slides it over the group.  Every load is independent of the
// others; threads of a half-warp hold 16 consecutive rows (odd row pitch: distinct banks).
__device__ __forceinline__ unsigned rank_group_cells(const RankWs& w, int j, int gi, unsigned u2p, unsigned u3p) {
    const unsigned* row = w.cs + j * w.P + kGrp * gi;
    const unsigned short* cm = w.cmm + j * w.cpitch + kGrp * gi;
    unsigned c[kGrp + 6];
#pragma unroll
    for (int k = 0; k < kGrp + 6; ++k) c[k] = row[k];
    unsigned mmv[kGrp];
#pragma unroll
    for (int m = 0; m < kGrp; ++m) mmv[m] = cm[m];
    unsigned C = 0;
#pragma unroll
    for (int k = 0; k < 7; ++k) C += c[k];
    unsigned word = 0;
#pragma unroll
    for (int m = 0; m < kGrp; ++m) {
        const int n263 = __popc((C + kGe263) & kFlag), n179 = __popc((C + kGe179) & kFlag);
        const unsigned code = (unsigned)(n179 * 4 + n263);
        // the clean range [U2, U3]: U2 follows HI (n263), U3 follows LO (n179) -- a byte pick each, no table load
        const unsigned U2 = __byte_perm(u2p, 0u, 0x4440u | (unsigned)n263), U3 = __byte_perm(u3p, 0u, 0x4440u | (unsigned)n179);
        const unsigned mn = mmv[m] & 255u, mx = mmv[m] >> 8;
        const bool dirty = kGrp * gi + m < w.nlx && (mn < U2 || mx > U3);
        word |= (code << (4 * m)) | ((dirty ? 1u : 0u) << (24 + m));
        if (m + 1 < kGrp) C += c[m + 7] - c[m];
    }
    return word;
}

// Tasks of the V pass: 32 cell slots x one segment of lattice rows per warp.  Segments (up to four) are chosen so that
// the tasks fit the warps that are free for them, leaving the Otsu warp out when possible.
struct VPlan { int nchunk, nseg, seg_rows, ntask; };
__device__ __forceinline__ VPlan rank_vplan(const Geom& g) {
    VPlan v;
    const int nslot = rank_nlx(g.w) + 2 * kVPad, nly = (g.h + kCell - 1) / kCell;
    v.nchunk = (nslot + 31) >> 5;
    v.nseg = max(1, min(min(4, (kWarps - 1) / v.nchunk), (nly + 7) >> 3));
    v.seg_rows = (((nly + v.nseg - 1) / v.nseg) + 7) & ~7;
    v.nseg = (nly + v.seg_rows - 1) / v.seg_rows;
    v.ntask = v.nchunk * v.nseg;
    return v;
}
// The warp kOtsuWarp gets no task of the V pass: it can run the exact Otsu scan beside the whole stage.
__device__ __forceinline__ bool rank_otsu_aside(const Geom& g) { return rank_vplan(g).ntask <= kOtsuWarp; }

// The warps that get no task of the V pass (and do not run the Otsu scan) take the last lattice rows of the cell
// min / max pass during it: [rank_cmm_split, nly); the caller runs the rows before the split next to the level selection.
__device__ __forceinline__ int rank_v_warps(const Geom& g) { return min(kWarps, rank_vplan(g).ntask); }
__device__ __forceinline__ int rank_cmm_split(const Geom& g, bool oside) {
    const int nly = (g.h + kCell - 1) / kCell;
    const int idle = (oside ? kWarps - 1 : kWarps) - rank_v_warps(g);
    if (idle <= 0) return nly;
    return nly * 42 / (42 + 8 * idle);           // 14 warps for about 3 k cycles before, `idle` warps for about 8 k during the V pass
}

// Part 1 (needs only the gray crop and the levels; the caller has run rank_cmm): window counts on the lattice, the
// plane of dirty cells.  `oside`: the warp kOtsuWarp is busy with the exact Otsu scan (started by the caller) and
// joins at the final barrier only; else it runs the scan here after its columns.  *otsu_t holds the threshold on return.
template <class PT>
VI_PHASE void rank_cells(const uint8_t* gray, const Geom& g, RankWs w, const int* lv, const unsigned* hist, int npix,
                         double* ows, volatile const int* olast, int* otsu_t, bool oside, PT& pt) {
    const int lane = lane_id(), warp = warp_id();
    const int nly = w.nly, nlx = w.nlx;
    const int hm1 = g.h - 1, wm1 = g.w - 1;
    const int nslot = nlx + 2 * kVPad;                           // cell slots of a row: 3 virtual, the cells, 3 virtual
    const VPlan vp = rank_vplan(g);
    const bool owarp = warp == kOtsuWarp;
    if (!(oside && owarp)) {
        {
            const int vw = rank_v_warps(g);
            rank_cmm(gray, g, w, vw, oside ? kWarps - 1 : kWarps, rank_cmm_split(g, oside), nly);      // idle in the V pass: the rest of the cell min / max
        }
        const unsigned T = (unsigned)(lv[0] + 512) | ((unsigned)(lv[1] + 512) << 10) | ((unsigned)(lv[2] + 512) << 20);
        int P = w.P, gp = g.gp;
        asm volatile("" : "+r"(P), "+r"(gp));                    // opaque strides (else re-derived from the unit width per store)
        for (int task = warp; task < vp.ntask; task += kWarps) {
            const int seg = task / vp.nchunk, chunk = task - seg * vp.nchunk;
            const int j0 = seg * vp.seg_rows, j1 = min(j0 + vp.seg_rows, nly);
            const int slot = chunk * 32 + lane;
            const int x0 = kCell * (slot - kVPad);               // may lie left / right of the crop: replicated border
            const uint8_t* c0 = gray + min(max(x0, 0), wm1);
            const uint8_t* c1 = gray + min(max(x0 + 1, 0), wm1);
            const uint8_t* c2 = gray + min(max(x0 + 2, 0), wm1);
            unsigned* csp = w.cs + j0 * P + (slot < nslot ? slot : P - 1);
            VI_CHECK(nslot <= P - 1 && j1 <= ((nly + 7) & ~7), CHK_LATTICE_SLOT);
            VState st;
            {
                // warm-up: blocks b = j0-3 .. j0+2 (rows above the crop replicate row 0), then the gray of block j0+3
                st.S = 0;
                st.r[6] = st.r[7] = 0;
#pragma unroll
                for (int bb = 0; bb < 6; ++bb) {
                    const int r0 = kCell * (j0 - 3 + bb);
                    const int o0 = min(max(r0, 0), hm1) * gp, o1 = min(max(r0 + 1, 0), hm1) * gp, o2 = min(max(r0 + 2, 0), hm1) * gp;
                    unsigned q[9] = {c0[o0], c0[o1], c0[o2], c1[o0], c1[o1], c1[o2], c2[o0], c2[o1], c2[o2]};
                    const unsigned B = ind9(T, q);
                    st.S += B;
                    st.r[bb] = B;
                }
                const int r0 = kCell * (j0 + 3);
                const int o0 = min(r0, hm1) * gp, o1 = min(r0 + 1, hm1) * gp, o2 = min(r0 + 2, hm1) * gp;
                st.q[0] = c0[o0]; st.q[1] = c0[o1]; st.q[2] = c0[o2];
                st.q[3] = c1[o0]; st.q[4] = c1[o1]; st.q[5] = c1[o2];
                st.q[6] = c2[o0]; st.q[7] = c2[o1]; st.q[8] = c2[o2];
            }
            for (int j = j0; j < j1; j += 8) {
                if (kCell * (j + 11) + 2 <= hm1) v_oct<false>(st, T, c0, c1, c2, gp, hm1, j, csp, P);
                else v_oct<true>(st, T, c0, c1, c2, gp, hm1, j, csp, P);
                csp += 8 * P;
            }
        }
        if (owarp) {                                             // (not aside: the scan follows this warp's columns)
            const int t = otsu_scan(hist, npix, ows, olast, pt);
            if (lane == 0) *otsu_t = t;
        }
        if (oside) workers_sync(kThreads - 32); else cta_sync();
        pt.acc(20);
        // ---- C: one thread per (lattice row, group of kGrp cells); half-warps over 16 consecutive rows ------------
        {
            const int nhw = w.nrb * w.ngrp;
            const unsigned mr = magic_of((unsigned)w.nrb);
            const int nhalf = (oside ? kThreads - 32 : kThreads) / 16;
            unsigned u2p = 0, u3p = 0;                                // U2 by n263, U3 by n179, four bytes each
#pragma unroll
            for (int k = 0; k < 4; ++k) { u2p |= ((w.table[k] >> 8) & 255u) << (8 * k); u3p |= ((w.table[4 * k] >> 16) & 255u) << (8 * k); }
#pragma unroll 2
            for (int hb = (int)(threadIdx.x >> 4); hb < nhw; hb += nhalf) {
                const int gi = (int)magic_div((unsigned)hb, (unsigned)w.nrb, mr), rb = hb - gi * w.nrb;
                const int j = rb * 16 + (int)(threadIdx.x & 15);
                unsigned word = 0;
                if (j < nly) word = rank_group_cells(w, j, gi, u2p, u3p);
                VI_CHECK(hb * 16 + 15 < w.plane_cap, CHK_DIRTY_LIST);
                w.plane[hb * 16 + (threadIdx.x & 15)] = word;
            }
        }
        pt.acc(21);
    }
    cta_sync();
}

// Part 2 (needs the ROI): CAND (zeroed by the caller) receives every ROI pixel with |g - med| > thr.
// Returns the number of pixels that needed an exact rank count.
template <class PT>
VI_PHASE int rank_finish(const uint8_t* gray, const Geom& g, RankWs w, const int* lv, int thr, const unsigned* ROI, unsigned* CAND,
                         unsigned* clist, int ccap, unsigned* elist, int ecap, PT& pt) {
    const int tid = threadIdx.x, lane = lane_id(), warp = warp_id();
    const int hm1 = g.h - 1, wm1 = g.w - 1;
    w.exact = elist; w.exact_cap = ecap;                      // the ambiguous-pixel list sits in shared memory too
    pt.acc(35);
    // ---- dirty cells that touch the ROI: listed (they cluster along the plate edge: whole tasks of them), then
    // classified per pixel one cell per thread.  `clist` / `ccap`: a list in shared memory; what does not fit is
    // classified on the spot.
    {
        const int ntask = w.nrb * w.ngrp * 16;
        const unsigned mr = magic_of((unsigned)w.nrb);
        for (int t0 = 0; t0 < ntask; t0 += 4 * kThreads) {
            unsigned wd[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) { const int t = t0 + q * kThreads + tid; wd[q] = t < ntask ? w.plane[t] : 0u; }      // four loads in flight
            if (ON_PROF(pt)) { if ((wd[0] | wd[1] | wd[2] | wd[3]) == 0x12345678u) wd[0] ^= 1u; pt.acc(44); }
#pragma unroll 1
            for (int q = 0; q < 4; ++q) {                             // rolled (the words rotate through wd[0]): cold, branchy code
                const unsigned word = wd[0];
                wd[0] = wd[1]; wd[1] = wd[2]; wd[2] = wd[3];
                unsigned d = word >> 24;
                if (!d) continue;
                const int t = t0 + q * kThreads + tid;
                const int hb = t >> 4;
                const int gi = (int)magic_div((unsigned)hb, (unsigned)w.nrb, mr), rb = hb - gi * w.nrb;
                const int j = rb * 16 + (t & 15);
                // ROI bits of the 18-pixel strip of the task's cells, three rows OR-ed, then one bit per cell
                const int x0 = kCell * kGrp * gi, c0 = x0 >> 5, sh = x0 & 31;
                const int c1 = min(c0 + 1, g.wpr - 1);
                const unsigned keep1 = c0 + 1 < g.wpr ? 0xffffffffu : 0u;
                unsigned b = 0;
#pragma unroll
                for (int rr = 0; rr < kCell; ++rr) {
                    const unsigned* row = ROI + min(kCell * j + rr, hm1) * g.wpr;      // (a row past the crop repeats the last: its cells' pixels are re-tested one by one)
                    b |= __funnelshift_r(row[c0], row[c1] & keep1, sh);
                }
                b |= (b >> 1) | (b >> 2);                                   // bit 3k: any pixel of cell k
                const unsigned cells = (b & 1u) | ((b >> 2) & 2u) | ((b >> 4) & 4u) | ((b >> 6) & 8u) | ((b >> 8) & 16u) | ((b >> 10) & 32u);
                d &= cells;
                if (!d) continue;
                const int nc = __popc(d);
                int k = atomicAdd(&w.counters[0], nc);
                while (d) {
                    const int m = __ffs(d) - 1; d &= d - 1;
                    const unsigned code = (word >> (4 * m)) & 15u;
                    if (k < ccap) clist[k] = ((unsigned)j << 16) | ((unsigned)(kGrp * gi + m) << 4) | code;
                    else rank_dirty_cell_cold(gray, g, thr, ROI, CAND, w, kGrp * gi + m, j, rank_code_thresholds(lv, thr, (int)code));
                    ++k;
                }
            }
        }
        pt.acc(45);
        cta_sync();
        pt.acc(36);
        const int nlist = min(w.counters[0], ccap);
        for (int k = tid; k < nlist; k += kThreads) {
            const unsigned e = clist[k];
            rank_dirty_cell(gray, g, thr, ROI, CAND, w, (int)((e >> 4) & 0xfffu), (int)(e >> 16), rank_code_thresholds(lv, thr, (int)(e & 15u)));
        }
    }
    cta_sync();
    pt.acc(22);
    // ---- ambiguous pixels: exact rank counts ------------------------------------------------
    // Few of them (the usual case): one warp per pixel, 14 window pixels per lane.  Many (low thresholds, small
    // units whose windows mostly straddle the plate edge): one thread per pixel walks its own window -- a quarter
    // of the warp-instructions per pixel once the warps are full; the list is in cell order, so the lanes of a
    // warp read neighbouring windows.
    const int ne = min(w.counters[1], w.exact_cap);
    if (ne > kExactWarpMax) {
        const int gp = g.gp;
        for (int k2 = tid; k2 < ne; k2 += kThreads) {
            const unsigned ent = w.exact[k2];
            const int y = (int)(ent >> 16), x = (int)(ent & 0x7fffu);
            const bool tb = (ent >> 15) & 1u;                        // which test: B counts against g - thr - 1, A against g + thr
            const int gv = gray[y * gp + x];
            const int pv = tb ? gv - thr - 1 : gv + thr;
            int cnt = 0;
            if (x >= 10 && x + 10 <= wm1 && y >= 10 && y + 10 <= hm1) {
                // window inside the crop: six aligned words per row (the crop pitch is a multiple of 4, so the byte
                // phase o is the same on every row), bytes compared four at a time; the per-byte "greater" flags are
                // summed as byte counters (at most 126 per lane) and the count is 441 minus their total.
                const int a0 = (y - 10) * gp + (x - 10);
                const int o = a0 & 3;
                const unsigned* wp = reinterpret_cast<const unsigned*>(gray + (a0 - o));
                const unsigned fm = 0x01010101u << (8 * o), lm = 0x01010101u >> (8 * (3 - o));      // first / last word bytes
                const SwarPivot qv = swar_pivot(pv);
                unsigned gsum = 0;
                const int wpitch = gp >> 2;
                for (int dy = 0; dy < 21; ++dy) {
#pragma unroll
                    for (int k = 0; k < 6; ++k) {
                        const unsigned W = wp[k];
                        const unsigned m = k == 0 ? fm : (k == 5 ? lm : 0x01010101u);
                        gsum += swar_gt(W, qv) & m;
                    }
                    wp += wpitch;
                }
                const unsigned sa = (gsum & 0x00ff00ffu) + ((gsum >> 8) & 0x00ff00ffu);
                cnt = 441 - (int)((sa & 0xffffu) + (sa >> 16));        // (the four lanes can add up to 441: no byte-wide total)
            } else {
                // window clipped to the crop; the replicated border rows / columns enter as weights of the edge ones
                const int xa = max(x - 10, 0), xb = min(x + 10, wm1), ya = max(y - 10, 0), yb = min(y + 10, hm1);
                const int nl = xa - (x - 10), nr = (x + 10) - xb, mt = ya - (y - 10), mb = (y + 10) - yb;
                for (int r = ya; r <= yb; ++r) {
                    const uint8_t* row = gray + r * gp;
                    const int e0 = row[0], e1 = row[wm1];
                    int ra = nl * (e0 <= pv) + nr * (e1 <= pv);
                    for (int c = xa; c <= xb; ++c) ra += (int)row[c] <= pv;
                    const int wr = 1 + (r == 0 ? mt : 0) + (r == hm1 ? mb : 0);
                    cnt += wr * ra;
                }
            }
            if (tb ? cnt >= 221 : cnt <= 220) atomicOr(&CAND[y * g.wpr + (x >> 5)], 1u << (x & 31));
        }
    } else
    {
        // lane's 14 window positions e = lane + 32k -> (dy, dx) = (e / 21, e % 21), as offsets from the window's corner
        int off[14];
        int dyx[14];
        const int gp = g.gp;
#pragma unroll
        for (int k = 0; k < 14; ++k) {
            const int e = lane + 32 * k;
            const int dy = (e * 3121) >> 16, dx = e - dy * 21;         // e / 21 for e < 448
            off[k] = dy * gp + dx;
            dyx[k] = (dy << 8) | dx;
        }
        const bool tail = lane + 32 * 13 < 441;                         // the 14th position exists for lanes 0..24
        for (int k2 = warp; k2 < ne; k2 += kWarps) {
            const unsigned ent = w.exact[k2];
            const int y = (int)(ent >> 16), x = (int)(ent & 0x7fffu);
            const bool tb = (ent >> 15) & 1u;                        // which test (see rank_dirty_cell)
            const int gv = gray[y * gp + x];
            const int pv = tb ? gv - thr - 1 : gv + thr;
            unsigned cnt = 0;
            if (x >= 10 && x + 10 <= wm1 && y >= 10 && y + 10 <= hm1) {  // the window lies inside the crop (uniform over the warp)
                const uint8_t* corner = gray + (y - 10) * gp + (x - 10);
                int vals[14];
#pragma unroll
                for (int k = 0; k < 13; ++k) vals[k] = corner[off[k]];
                vals[13] = tail ? (int)corner[off[13]] : 256;
#pragma unroll
                for (int k = 0; k < 14; ++k) cnt += vals[k] <= pv;
            } else {
#pragma unroll
                for (int k = 0; k < 14; ++k) {
                    const int dy = dyx[k] >> 8, dx = dyx[k] & 255;
                    const int yy = min(max(y + dy - 10, 0), hm1), xx = min(max(x + dx - 10, 0), wm1);
                    const int v = (k < 13 || tail) ? (int)gray[yy * gp + xx] : 256;
                    cnt += v <= pv;
                }
            }
            cnt = __reduce_add_sync(kFull, cnt);
            if (lane == 0 && (tb ? cnt >= 221 : cnt <= 220)) atomicOr(&CAND[y * g.wpr + (x >> 5)], 1u << (x & 31));
        }
    }
    cta_sync();
    return w.counters[1];          // every ambiguous pixel, listed or not (the counters are next written after the next unit's histogram: barriers in between)
}

}  // namespace vi
