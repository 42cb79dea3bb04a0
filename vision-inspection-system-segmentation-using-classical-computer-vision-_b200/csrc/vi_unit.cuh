// vi_unit.cuh -- process_unit(): one CTA runs every stage of one unit with the
// crop and all masks resident in shared memory, and the persistent kernel that
// strides units over the grid.
#pragma once
#include <cmath>
#include "vi_pipeline.cuh"
#include "vi_rank.cuh"
#include "vi_canny.cuh"

namespace vi {

// Canonical (raster-order) label of every root: 1 + number of roots with a smaller
// run id.  Stored in acc1[root]; returns the number of components.
VI_PHASE int ccl_rank_roots(Cta& cs, const CclWs& ws, int R) {
    unsigned carry = 0;
    for (int base = 0; base < R; base += kThreads) {
        int i = base + threadIdx.x + 1;
        unsigned isroot = (i <= R && ws.parent()[i] == i) ? 1u : 0u;
        unsigned a = isroot, b = 0, ta, tb;
        cta_excl_scan2(cs, a, b, ta, tb);
        if (isroot) ws.acc1()[i] = carry + a + 1;
        carry += ta;
    }
    cta_sync();
    return (int)carry;
}

// int32 labels, unit-packed [h][w]: 0 background, else acc1[root].
VI_PHASE void store_labels(const Geom& g, const CclWs& ws, int32_t* __restrict__ dst) {
    for (int i = threadIdx.x; i < g.nwords; i += kThreads) {
        int y, c; word_rc(g, i, y, c);
        int x0 = c * 32, x1 = min(x0 + 31, g.w - 1);
        int j = ws.row_first()[y], j1 = ws.row_first()[y + 1];
        while (j < j1 && (int)ws.xe()[j] < x0) ++j;
        for (int x = x0; x <= x1; ++x) {
            while (j < j1 && (int)ws.xe()[j] < x) ++j;
            int lab = 0;
            if (j < j1 && (int)ws.xs()[j] <= x) lab = (int)ws.acc1()[ws.parent()[j]];
            dst[(long long)y * g.w + x] = lab;
        }
    }
}

VI_PHASE void zero_bytes(uint8_t* __restrict__ dst, int n) {
    const int head = min(n, (int)((16 - (reinterpret_cast<uintptr_t>(dst) & 15)) & 15));
    for (int e = threadIdx.x; e < head; e += kThreads) dst[e] = 0;
    const int n16 = (n - head) >> 4;
    uint4* d16 = reinterpret_cast<uint4*>(dst + head);
    for (int e = threadIdx.x; e < n16; e += kThreads) d16[e] = make_uint4(0u, 0u, 0u, 0u);
    for (int e = head + (n16 << 4) + threadIdx.x; e < n; e += kThreads) dst[e] = 0;
}

// P14 for a sparse mask (the defect mask: a few blobs in a field of zeros): 128-bit zero fill of the whole unit, then only
// the 4-pixel groups that hold a set pixel are written.  Needs w % 4 == 0 and a 4-byte aligned destination (else the
// dense store runs).
VI_PHASE void store_mask_bytes_sparse(const unsigned* M, const Geom& g, uint8_t* __restrict__ dst) {
    if ((g.w & 3) != 0 || (reinterpret_cast<uintptr_t>(dst) & 3) != 0) { store_mask_bytes(M, g, dst); return; }
    zero_bytes(dst, g.w * g.h);
    cta_sync();                                              // the fill is ordered before the set groups below
    const int qpr = g.w >> 2;
    unsigned* d32 = reinterpret_cast<unsigned*>(dst);
    for (int i = threadIdx.x; i < g.nwords; i += kThreads) {
        unsigned m = M[i];
        if (m == 0) continue;
        int y, c; word_rc(g, i, y, c);
        unsigned* row = d32 + y * qpr + c * 8;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const unsigned nib = (m >> (4 * k)) & 0xFu;
            if (nib) row[k] = ((nib * 0x00204081u) & 0x01010101u) * 0xFFu;
        }
    }
}

// Packed-bit mask out: rows of wpr 32-bit words; inside every byte the first pixel is the most significant bit (the bit
// order of a 1-bit PNG scanline and of numpy.unpackbits).  The kernel's own words hold pixel x at bit x & 31.
VI_PHASE void store_mask_words(const unsigned* M, const Geom& g, uint32_t* __restrict__ dst) {
    for (int i = threadIdx.x; i < g.nwords; i += kThreads) dst[i] = __byte_perm(__brev(M[i]), 0u, 0x0123u);
}

VI_PHASE void zero_words(uint32_t* __restrict__ dst, int n) {
    for (int i = threadIdx.x; i < n; i += kThreads) dst[i] = 0u;
}

// L2 prefetch of a unit's crop rows (issued for the CTA's next unit while this one computes).
VI_PHASE void prefetch_crop_l2(const KArgs& a, int uid) {
    const int img = uid / a.n_units, unit = uid - img * a.n_units;
    const int4 rc = a.rects[unit];
    const uint8_t* base = a.frames + (long long)img * a.image_stride + (long long)rc.y * a.row_pitch + rc.x;
    const int lines = (rc.z + 127 + 127) >> 7;                       // 128-byte lines a row can touch
    for (int i = threadIdx.x; i < rc.w * lines; i += kThreads) {
        const int y = i / lines, l = i - y * lines;
        const uint8_t* p = base + (long long)y * a.row_pitch + l * 128;
        asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
    }
}

// Warp 0 only (the caller synchronises).
__device__ inline void select_levels(UnitShared& sh, int npix, int thr, int t, bool bright) {
    // Three levels around the median of one Otsu class of the (blurred) histogram: the dark class (the seg mask is an
    // inverse threshold, so the ROI lives there), or the bright one when a caller-supplied mask does (detect_defects).
    // Any level set is exact; these make the cell brackets decide nearly every pixel of the ROI.
    {
        const int lane = lane_id();
        unsigned c[8], tot = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) { tot += sh.hist[lane * 8 + k]; c[k] = tot; }      // inclusive within the lane
        unsigned inc = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { unsigned x = __shfl_up_sync(kFull, inc, o); if (lane >= o) inc += x; }
        const unsigned base = inc - tot;
        // cumulative count at t (dark class size)
        const unsigned at_t = __shfl_sync(kFull, base, t >> 3);
        unsigned ct = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) { unsigned v = __shfl_sync(kFull, c[k], t >> 3); if (k == (t & 7)) ct = v; }
        const unsigned nd = at_t + ct, nb = (unsigned)npix - nd;
        const unsigned ncls = bright ? nb : nd;
        const unsigned tgt = bright ? nd + (nb + 1) / 2 : (nd + 1) / 2;
        // first bin whose cumulative count reaches the target
        unsigned f = 0xffffu;
#pragma unroll
        for (int k = 7; k >= 0; --k) {
            const unsigned cum = base + c[k];
            if (ncls && cum >= tgt) f = lane * 8 + k;
        }
        f = __reduce_min_sync(kFull, f);
        if (lane == 0) {
            const int cm = ncls ? (int)f : t;
            int s = 1;
            const int lim = thr / 3 > 1 ? thr / 3 : 1;
            while (s * 2 <= lim && s < 16) s *= 2;
            sh.levels[0] = min(254, max(0, cm - s)); sh.levels[1] = min(254, max(0, cm)); sh.levels[2] = min(254, max(0, cm + s));
        }
    }
    __syncwarp();
}

// Area and coordinate sums of a bit mask (segmentation.mask_stats, segmentation.py:103-111: the caller divides).
__device__ inline void mask_sums(Cta& cs, const unsigned* M, const Geom& g, long long* out3) {
    unsigned long long n = 0, sx = 0, sy = 0;
    for (int i = threadIdx.x; i < g.nwords; i += kThreads) {
        int y, c; word_rc(g, i, y, c);
        const unsigned m = M[i];
        const unsigned pc = __popc(m);
        const unsigned pos = __popc(m & 0xAAAAAAAAu) + 2 * __popc(m & 0xCCCCCCCCu) + 4 * __popc(m & 0xF0F0F0F0u) +
                             8 * __popc(m & 0xFF00FF00u) + 16 * __popc(m & 0xFFFF0000u);
        n += pc; sx += (unsigned long long)pc * (c * 32) + pos; sy += (unsigned long long)pc * y;
    }
    unsigned n32 = (unsigned)n;
    cta_sum3(cs, n32, sx, sy);
    if (threadIdx.x == 0) { out3[0] = (long long)n32; out3[1] = (long long)sx; out3[2] = (long long)sy; }
}

__device__ inline void write_record(const KArgs& a, int uid, int img, int unit, int otsu_t, unsigned seg_area,
                                    unsigned roi_area, unsigned defect_area, int n_kept, int status, int dx, int dy,
                                    double cx, double cy, int n_amb, int n_runs) {
    if (threadIdx.x == 0 && a.rec) {
        vi_unit_record r;
        r.image = img * a.image_mul + a.image_base; r.unit = unit; r.otsu_t = otsu_t; r.seg_area = (int)seg_area; r.roi_area = (int)roi_area;
        r.defect_area = (int)defect_area; r.n_kept = n_kept; r.status = status; r.dx = dx; r.dy = dy;
        r.cx = cx; r.cy = cy; r.n_ambiguous = n_amb; r.n_runs = n_runs;
        a.rec[uid] = r;
    }
    // Multi-GPU: the verdict table is gathered by the kernel itself -- the record goes straight into every rank's table
    // over NVLink (plain stores to peer-mapped memory; they are posted, nothing waits on them), so no collective runs
    // between steps.  One lane per peer.
    if (threadIdx.x < a.n_peers && a.rec) {
        vi_unit_record r;
        r.image = img * a.image_mul + a.image_base; r.unit = unit; r.otsu_t = otsu_t; r.seg_area = (int)seg_area; r.roi_area = (int)roi_area;
        r.defect_area = (int)defect_area; r.n_kept = n_kept; r.status = status; r.dx = dx; r.dy = dy;
        r.cx = cx; r.cy = cy; r.n_ambiguous = n_amb; r.n_runs = n_runs;
        a.peer_rec[threadIdx.x][(long long)r.image * a.n_units + unit] = r;
    }
}

// segmentation.fill_internal_holes on the bit mask M, in place (T: scratch mask).  The flood settles the usual masks in
// two rounds; what it cannot settle in kFloodRounds is labelled (background runs, 4-connectivity, united with the
// virtual outside node when they touch the border).  Returns the run count of the labelling pass (0: flood).
template <class PT>
VI_PHASE int fill_holes(Cta& cta, unsigned* M, unsigned* T, const Geom& g, const CclWs& ws_s, const CclWs& ws_g, CclWs& ws, PT* pt, int* how = nullptr) {
    const int fl = flood_border_background(M, T, g);
    if (how) *how = fl;
    if (fl) {
        for (int i = threadIdx.x; i < g.nwords; i += kThreads)
            M[i] = ~T[i] & row_mask_of(g, i - (int)magic_div((unsigned)i, (unsigned)g.wpr, g.mwpr) * g.wpr);
        cta_sync();
        return 0;
    }
    for (int i = threadIdx.x; i < g.nwords; i += kThreads)
        T[i] = ~M[i] & row_mask_of(g, i - (int)magic_div((unsigned)i, (unsigned)g.wpr, g.mwpr) * g.wpr);
    cta_sync();
    const int R = ccl_build(cta, T, g, false, true, ws_s, ws_g, ws, pt);
    ccl_paint(M, M, g, ws, [](int root) { return root != 0; });
    cta_sync();
    return R;
}

// SPEC: the instantiation for the reference's default configuration (full path, Otsu, 3x3 blur, 3x3 cross, threshold
// method, lattice rank stage, 16-byte aligned frames, no optional outputs): everything that is a run-time choice in
// the general kernel is a constant here, so the non-default branches are not even in the code (a third of the
// instructions, less pressure on the instruction cache and on registers).  The host picks it (vi_api.cu: launch_units).
// SPEC && SEG: the same configuration in the segmentation-only mode (vi_segment_batch): no detector, and the seg_stats
// and packed seg-bit outputs stay run-time pointers (the mask export needs them).  The mask is carried in MB / MC from
// the first close pass on, so that the next unit's crop can be gathered into gray and MA from there.
// GMEM: the instantiation for units beyond one SM's shared memory -- `smem` is then the CTA's arena in global memory
// (same layout, vi_device.cuh: unit_layout) and `hist_smem` the shared-memory home of the histogram copies.
template <bool PROF, bool SPEC, bool GMEM, bool SEG>
__device__ __forceinline__ void process_unit(const KArgs& a, int uid, unsigned char* smem, unsigned char* hist_smem, UnitShared& sh, Cta& cta) {
    const int tid = threadIdx.x;
    const int img = uid / a.n_units, unit = uid - img * a.n_units;
    const int4 rc = a.rects[unit];
    const Geom g = make_geom(rc.z, rc.w);
    const UnitLayout& L = a.layout;
    const int npix = g.w * g.h;
    const int mode = SPEC ? (SEG ? (int)MODE_SEG_ONLY : (int)MODE_FULL) : a.mode;
    const int cfg_blur_k = SPEC ? 3 : a.blur_k;
    const int cfg_se_k = SPEC ? 3 : a.se_k;
    const int cfg_seg_method = SPEC ? 0 : a.p.seg_method;
    const int cfg_defect_method = SPEC ? 0 : a.p.defect_method;
    long long* const cfg_seg_stats = SPEC && !SEG ? nullptr : a.seg_stats;
    uint32_t* const cfg_seg_bits = SPEC && !SEG ? nullptr : a.seg_bits;
    uint32_t* const cfg_def_bits = SPEC ? nullptr : a.def_bits;

    uint8_t* gray = smem;
    unsigned* MA = reinterpret_cast<unsigned*>(smem + L.gray_bytes + 0 * L.mask_bytes);
    unsigned* MB = reinterpret_cast<unsigned*>(smem + L.gray_bytes + 1 * L.mask_bytes);
    unsigned* MC = reinterpret_cast<unsigned*>(smem + L.gray_bytes + 2 * L.mask_bytes);
    unsigned* MD = reinterpret_cast<unsigned*>(smem + L.gray_bytes + 3 * L.mask_bytes);
    unsigned* ME = reinterpret_cast<unsigned*>(smem + L.gray_bytes + 4 * L.mask_bytes);
    unsigned* CAND = MC;                 // candidate mask of the median stage (ME when it could be zeroed early)
    unsigned char* WS = smem + L.ws_off;

    unsigned char* gs = a.scratch + (long long)blockIdx.x * L.scratch_bytes;
    unsigned short* g_hp = reinterpret_cast<unsigned short*>(gs);
    uint8_t* g_blur = gs + L.blur_off;
    const CclWs ws_s = ccl_ws_carve(WS, L.run_cap, L.run_rf);
    const CclWs ws_g = ccl_ws_carve(gs + L.runs_off, L.runs_cap, L.run_rf);
    CclWs ws;

    const long long moff = (long long)img * a.unit_px + a.unit_off[unit];
    uint8_t* seg_out = a.seg_out ? a.seg_out + moff : nullptr;
    uint8_t* def_out = a.def_out ? a.def_out + moff : nullptr;
    int32_t* lab_out = (!SPEC && a.labels_out) ? a.labels_out + moff : nullptr;
    const uint8_t* aux = (!SPEC && a.aux_mask) ? a.aux_mask + moff : nullptr;
    long long* stats = (!SPEC && a.stats_out) ? a.stats_out + (long long)uid * 8 : nullptr;
    // packed-bit outputs: derived on use (nothing of them is held across phases)
    auto bits_at = [&a, img, unit](uint32_t* base) { return base + ((long long)img * a.unit_words + a.unit_woff[unit]); };

    PhaseTimerT<PROF> pt;
    pt.start(&sh.pt, a.prof ? a.prof + (long long)uid * kProfSlots : nullptr);
    const bool need_gray = mode == MODE_FULL || mode == MODE_SEG_ONLY || mode == MODE_DETECT;
    const bool need_seg = mode == MODE_FULL || mode == MODE_SEG_ONLY;
    int otsu_t = 0, dx = 0, dy = 0, n_runs_max = 0;
    bool lattice = false;
    double cx = __longlong_as_double(0x7ff8000000000000ll), cy = cx;
    unsigned seg_area = 0;

    if (need_gray) {
        const uint8_t* src = a.frames + (long long)img * a.image_stride + (long long)rc.y * a.row_pitch + rc.x;
        if (SPEC && cta.gpending) {
            // the rows were fetched by the bulk-copy engine while the previous unit finished (gather_issue below)
            if (warp_id() == 0) mbar_wait(&sh.gather_mbar, cta.gpar);      // one warp polls; the barrier hands its acquire on to the rest
            cta_sync();
            pt.acc(32);
            if (a.tma_ok) gather_finish_tma(a, src, a.row_pitch, g, gray);
            else gather_finish(src, a.row_pitch, g, gray);
            cta.gpar ^= 1u; cta.gpending = 0;
        } else if (SPEC || ((a.row_pitch & 15) == 0 && (reinterpret_cast<uintptr_t>(a.frames) & 15) == 0 && (a.image_stride & 15) == 0))
            load_gray16(src, a.row_pitch, g, gray);
        else
            load_gray(src, a.row_pitch, g, gray);
        if (!(SPEC && a.tma_ok) && uid + (int)gridDim.x < a.n_images * a.n_units) prefetch_crop_l2(a, uid + (int)gridDim.x);
        cta_sync();
        pt.tick();   // 0 gather
        // ---- P1: blur + histogram ------------------------------------------------
        int src_mode = (mode == MODE_DETECT || cfg_blur_k == 0) ? 0 : (cfg_blur_k == 3 ? 1 : 2);
        const bool adaptive = need_seg && cfg_seg_method == 1;
        if (adaptive) {
            // the adaptive mean reads the blurred crop from global scratch whatever the blur size
            if (cfg_blur_k == 0) {
                for (int e = tid; e < npix; e += kThreads) { const int y = e / g.w; g_blur[e] = gray[y * g.gp + (e - y * g.w)]; }
                cta_sync();
            } else {
                blur_general(gray, g, cfg_blur_k, a.taps, g_hp, g_blur);
            }
            src_mode = 2;
        } else if (src_mode == 2) {
            blur_general(gray, g, cfg_blur_k, a.taps, g_hp, g_blur);
        }
        unsigned* hist_base = GMEM ? reinterpret_cast<unsigned*>(hist_smem) : MA;
        {
            uint4* h4 = reinterpret_cast<uint4*>(hist_base);                  // 128-bit stores: the copies are 16-byte aligned
            for (int i = tid; i < L.n_hist * (kHistWords / 4); i += kThreads) h4[i] = make_uint4(0u, 0u, 0u, 0u);
        }
        if (tid < 256) sh.hist[tid] = 0;
        if (tid == 0) sh.otsu_last = -1;              // "no bound yet" for the exact Otsu scan (vi_pipeline.cuh: otsu_scan)
        cta_sync();
        pt.acc(30);
        if (SPEC || (src_mode == 1 && hist_round_fits(L.n_hist))) {
            // default path: one histogram round on min(16, n_hist) warps
            blur3_hist(gray, g, hist_base + warp_id() * kHistWords, min(L.n_hist, kWarps));
            cta_sync();
            pt.acc(31);
            hist_collect(hist_base, min(L.n_hist, kWarps), sh.hist, false);
            cta_sync();
        } else {
            for (int r0 = 0; r0 < kWarps; r0 += L.n_hist) {
                unsigned* hw = hist_base + (warp_id() - r0) * kHistWords;
                if (src_mode == 0) blur_pass<0, true>(gray, g_blur, g, hw, sh.hist, r0, L.n_hist, nullptr, 0);
                else if (src_mode == 1) blur_pass<1, true>(gray, g_blur, g, hw, sh.hist, r0, L.n_hist, nullptr, 0);
                else blur_pass<2, true>(gray, g_blur, g, hw, sh.hist, r0, L.n_hist, nullptr, 0);
                cta_sync();
                hist_collect(hist_base, min(L.n_hist, kWarps - r0), sh.hist, true);
                cta_sync();
            }
        }
        pt.tick();   // 1 blur + histogram
        // ---- P2: Otsu.  The exact scan is a serial recurrence in doubles: one warp runs it while the others walk the
        // columns of the median stage's cell pass, which needs no mask and only approximate levels (an approximate
        // threshold splits the histogram into its classes).  The stage's lattice is not live before the threshold
        // (the first mask, outside it, holds a caller-supplied mask in MODE_DETECT).
        double* ows = reinterpret_cast<double*>(smem + L.otsu_off);
        lattice = (SPEC && !SEG) || ((mode == MODE_FULL || mode == MODE_DETECT) && cfg_defect_method == 0 && lattice_fits(g.w, g.h, L));
        RankWs rw = rank_ws_carve(smem + L.lattice_off, g, gs + L.rank_off, L.rank_words, sh.rank_cnt);
        const bool vote = !SPEC && mode == MODE_DETECT && lattice;
        if (vote) { load_mask_bits(aux, g, MA); }       // the caller's mask decides which class the levels bracket
        // the exact Otsu scan starts now on its own warp when that warp owns no column of the cell pass
        const bool oside = lattice && !vote && rank_otsu_aside(g);
        if (warp_id() == 0) {                       // one warp, no barriers in between: approximate threshold, levels, tables
            int last;
            const int ta = otsu_approx_warp(sh.hist, npix, last);
            if (lane_id() == 0) { sh.t_apx = ta; *const_cast<volatile int*>(&sh.otsu_last) = last; }
            pt.acc(33);
            if (lattice && !vote) {
                select_levels(sh, npix, a.p.threshold, ta, false);
                rank_tables(sh.levels, a.p.threshold, rw);
            }
            pt.acc(34);
        } else if (oside && warp_id() == kOtsuWarp) {
            long long c0 = pt.stamp();
            const int t = otsu_scan(sh.hist, npix, ows, &sh.otsu_last, pt);      // (warp 0 publishes the bound meanwhile)
            pt.lap(37, c0);
            if (lane_id() == 0) sh.otsu_t = t;
        } else if (lattice) {
            rank_cmm(gray, g, rw, 1, oside ? kWarps - 1 : kWarps, 0, rank_cmm_split(g, oside));     // the cells' gray min / max need no level: meanwhile
        }
        if (vote) {
            // one sample per mask word: is the mask's class the dark one or the bright one?
            cta_sync();
            const int ta = sh.t_apx;
            unsigned long long v = 0;
            for (int i = tid; i < g.nwords; i += kThreads) {
                const unsigned m = MA[i];
                if (m) {
                    int y, c; word_rc(g, i, y, c);
                    const int x = c * 32 + __ffs(m) - 1;
                    v += 1ull + ((int)gray[y * g.gp + x] <= ta ? (1ull << 32) : 0ull);
                }
            }
            v = cta_sum_u64(cta, v);
            const bool bright = 2 * (v >> 32) < (v & 0xffffffffull);
            if (warp_id() == 0) {
                select_levels(sh, npix, a.p.threshold, ta, bright);
                rank_tables(sh.levels, a.p.threshold, rw);
            }
        }
        if (oside) { if (warp_id() != kOtsuWarp) workers_sync(kThreads - 32); } else cta_sync();
        if (lattice) {
            pt.tick();   // 2 approximate threshold, levels, tables
            rank_cells(gray, g, rw, sh.levels, sh.hist, npix, ows, &sh.otsu_last, &sh.otsu_t, oside, pt);
        } else {
            if (warp_id() == kOtsuWarp) {
                const int t = otsu_scan(sh.hist, npix, ows, &sh.otsu_last, pt);
                if (lane_id() == 0) sh.otsu_t = t;
            }
            cta_sync();
            pt.tick();
        }
        otsu_t = sh.otsu_t;
        pt.tick();   // 3 cell pass with the exact Otsu scan inside

        if (need_seg) {
            // ---- P3: inverse threshold ------------------------------------------
            if (adaptive)
                adaptive_threshold(g_blur, g, a.adapt_bs, a.ataps, a.p.adapt_C, reinterpret_cast<float*>(gs + L.f32_off), MA);
            else if (src_mode == 0) blur_pass<0, false>(gray, g_blur, g, nullptr, nullptr, 0, kWarps, MA, otsu_t);
            else if (src_mode == 1) {
                // (blurring again with the SWAR loop and comparing was measured: 25.7 k cycles against 17.5 k for this)
                threshold_gray(gray, g, MB, otsu_t, sh.misc);
                cta_sync();
                pt.acc(29);
                threshold_band(gray, g, MB, MA, MC, otsu_t, reinterpret_cast<unsigned*>(smem + L.band_off), L.band_cap, sh.misc, pt);
            }
            else blur_pass<2, false>(gray, g_blur, g, nullptr, nullptr, 0, kWarps, MA, otsu_t);
            cta_sync();
            pt.tick();   // 4 threshold
            if (lattice && mode == MODE_FULL && cfg_defect_method == 0) {
                // the median stage's candidate mask collects bits with atomics: it is zeroed here, where a barrier
                // follows anyway (ME is free from the threshold's list until the contour filter)
                for (int i = tid; i < g.nwords; i += kThreads) ME[i] = 0;
                CAND = ME;
            }
            // ---- P4: close, open --------------------------------------------------
            unsigned* S = MA;                                // the seg mask from here on
            if (SPEC && SEG) {
                cross3_pass<false>(MA, MB, g); cta_sync();
                // gray and MA are dead: the next unit's crop goes into the staging area over them meanwhile
                const int nuid = uid + (int)gridDim.x;
                if (nuid < a.n_images * a.n_units)
                    cta.gpending = (a.tma_ok ? gather_issue_tma(a, nuid, smem, L.stage_bytes, &sh.gather_mbar)
                                             : gather_issue(a, nuid, smem, L.stage_bytes, &sh.gather_mbar)) ? 1 : 0;
                cross3_pass<true>(MB, MC, g); cta_sync();
                cross3_pass<true>(MC, MB, g); cta_sync();
                cross3_pass<false>(MB, MC, g); cta_sync();
                S = MC;
            } else if (cfg_se_k == 3) {
                cross3_pass<false>(MA, MB, g); cta_sync();
                cross3_pass<true>(MB, MA, g); cta_sync();
                cross3_pass<true>(MA, MB, g); cta_sync();
                cross3_pass<false>(MB, MA, g); cta_sync();
            } else if (cfg_se_k > 0) {
                se_pass<false>(MA, MB, g, cfg_se_k, a.se_lo, a.se_hi); cta_sync();
                se_pass<true>(MB, MA, g, cfg_se_k, a.se_lo, a.se_hi); cta_sync();
                se_pass<true>(MA, MB, g, cfg_se_k, a.se_lo, a.se_hi); cta_sync();
                se_pass<false>(MB, MA, g, cfg_se_k, a.se_lo, a.se_hi); cta_sync();
            }
            pt.tick();   // 5 close/open
            // ---- P5: hole fill ----------------------------------------------------
            unsigned* rowinfo = reinterpret_cast<unsigned*>(ws_s.row_first());
            RowScan rs = mask_row_scan(cta, S, g, rowinfo);
            if (rs.any_multi) {                              // a row with several runs: the background may have holes
                int how = 0;
                n_runs_max = max(n_runs_max, fill_holes(cta, S, MB, g, ws_s, ws_g, ws, &pt, &how));
                rs = how == 2 ? mask_row_rescan_filled(cta, S, g, rowinfo) : mask_row_scan(cta, S, g, rowinfo);
            }
            pt.tick();   // 6 hole fill
            {
                // ---- P6: largest 8-component centroid, shift ---------------------
                unsigned area; unsigned long long sx, sy;
                int broot = 1;
                if (rs.solid) { area = rs.area; sx = rs.sx; sy = rs.sy; }
                else {
                    const int R = ccl_build(cta, S, g, true, false, ws_s, ws_g, ws, &pt);
                    n_runs_max = max(n_runs_max, R);
                    broot = ccl_largest(cta, g, ws, R, area, sx, sy);
                }
                if (broot != 0 && area > 0) {
                    cx = __ddiv_rn((double)sx, (double)area);
                    cy = __ddiv_rn((double)sy, (double)area);
                    if (!a.is_reference && a.refc) {
                        double c0x = a.refc[2 * unit], c0y = a.refc[2 * unit + 1];
                        if (c0x == c0x && c0y == c0y) {
                            dx = __double2int_rn(__dsub_rn(cx, c0x));
                            dy = __double2int_rn(__dsub_rn(cy, c0y));
                        }
                    }
                }
                cta_sync();
                pt.tick();   // 7 centroid labelling
                // ---- P7: exclusions ------------------------------------------------
                if (a.n_excl > 0) { apply_exclusions(S, g, a.excl, a.n_excl, dx, dy); cta_sync(); }
            }
            // ---- P8: seg mask out -------------------------------------------------
            if (rs.solid && a.n_excl == 0) seg_area = rs.area;      // one solid blob, untouched since the row scan: its area is the mask's
            else seg_area = cta_popcount(cta, S, g);
            if (cfg_seg_stats) mask_sums(cta, S, g, cfg_seg_stats + (long long)uid * 3);     // CSV export's mask_stats, optional
            if (seg_out) store_mask_bytes(S, g, seg_out);
            if (cfg_seg_bits) store_mask_words(S, g, bits_at(cfg_seg_bits));
            pt.tick();   // 8 exclusions + seg mask out
            if (mode == MODE_SEG_ONLY) {
                write_record(a, uid, img, unit, otsu_t, seg_area, 0, 0, 0, VI_STATUS_SEGMENTED, dx, dy, cx, cy, 0, n_runs_max);
                return;
            }
        }
    }

    if (mode == MODE_FILL || mode == MODE_STATS || mode == MODE_ERODE || mode == MODE_LABEL || (mode == MODE_DETECT && !lattice)) {
        load_mask_bits(aux, g, MA);
        cta_sync();
    }
    if (mode == MODE_FILL) {
        fill_holes(cta, MA, MB, g, ws_s, ws_g, ws, &pt);
        store_mask_bytes(MA, g, seg_out);
        return;
    }
    if (mode == MODE_STATS) {
        mask_sums(cta, MA, g, stats);
        return;
    }
    if (mode == MODE_ERODE) {
        unsigned* X = MA;
        if (a.erode_r > 0) X = erode_square_bits(MA, MB, MC, g, a.erode_r);
        store_mask_bytes(X, g, seg_out);
        return;
    }
    if (mode == MODE_LABEL) {
        int R = ccl_build(cta, MA, g, true, false, ws_s, ws_g, ws, &pt);
        unsigned area; unsigned long long sx, sy;
        int broot = ccl_largest(cta, g, ws, R, area, sx, sy);
        int nlab = ccl_rank_roots(cta, ws, R);
        if (lab_out) store_labels(g, ws, lab_out);
        if (tid == 0) {
            stats[0] = nlab; stats[1] = broot ? (long long)ws.acc1()[broot] : 0; stats[2] = area;
            stats[3] = (long long)sx; stats[4] = (long long)sy; stats[5] = R;
        }
        return;
    }
    if (mode == MODE_DETECT) seg_area = cta_popcount(cta, MA, g);

    // =========================== detector ======================================
    // ---- P9: square erosion ---------------------------------------------------
    unsigned* X = MA;
    if (a.p.erode_px > 0) X = erode_square_bits(MA, MB, MC, g, a.p.erode_px);
    pt.tick();   // 9 erosion
    // ---- P10: largest 8-component = ROI ---------------------------------------
    unsigned roi_area = 0;
    {
        RowScan rs;
        rs.solid = false;
        if (!lab_out) rs = mask_row_scan(cta, X, g, reinterpret_cast<unsigned*>(ws_s.row_first()));
        if (rs.solid) {                                      // one solid blob: it is the ROI
            roi_area = rs.area;
            for (int i = tid; i < g.nwords; i += kThreads) MD[i] = X[i];
        } else {
            const int R = ccl_build(cta, X, g, true, false, ws_s, ws_g, ws, &pt);
            n_runs_max = max(n_runs_max, R);
            unsigned long long rsx, rsy;
            const int broot = ccl_largest(cta, g, ws, R, roi_area, rsx, rsy);
            if (lab_out) {
                ccl_rank_roots(cta, ws, R);
                store_labels(g, ws, lab_out);
            }
            if (broot == 0 || roi_area == 0) {
                if (def_out) zero_bytes(def_out, npix);
                if (cfg_def_bits) zero_words(bits_at(cfg_def_bits), g.nwords);
                write_record(a, uid, img, unit, otsu_t, seg_area, 0, 0, 0, VI_STATUS_ROI_EMPTY, dx, dy, cx, cy, 0, n_runs_max);
                return;
            }
            ccl_paint(MD, nullptr, g, ws, [broot](int root) { return root == broot; });
        }
    }
    cta_sync();
    pt.tick();   // 10 ROI labelling
    const int thr = a.p.threshold;
    int n_amb = 0;
    int any_resid = 0;
    int R = 0;
    if (cfg_defect_method == 1) {
        // ---- P11': Canny edges inside the ROI (indexing_ui.py:1536-1539) ----------------
        canny_candidates(gray, g, a.canny_low, a.canny_high, MA, MB);
        cta_sync();
        R = canny_hysteresis(cta, MA, MB, MC, g, ws_s, ws_g, ws);
        n_runs_max = max(n_runs_max, R);
        for (int i = tid; i < g.nwords; i += kThreads) { const unsigned v = MC[i] & MD[i]; MB[i] = v; any_resid |= (v != 0); }
        any_resid = cta_sync_or(any_resid);
        for (int k = 0; k < 2; ++k) pt.tick();   // 11, 12 (the residual path's slots)
    } else {
    // ---- P11: median residual (second part: the dirty cells against the ROI) ------------
    if (CAND == MC) {
        for (int i = tid; i < g.nwords; i += kThreads) MC[i] = 0;
        cta_sync();
    }
    if (SPEC || lattice) {
        RankWs rw = rank_ws_carve(smem + L.lattice_off, g, gs + L.rank_off, L.rank_words, sh.rank_cnt);
        // lists of the stage in the (free) labelling workspace: dirty cells of the ROI, ambiguous pixels
        n_amb = rank_finish(gray, g, rw, sh.levels, thr, MD, CAND, reinterpret_cast<unsigned*>(WS), L.dirty_cap,
                            reinterpret_cast<unsigned*>(WS) + L.dirty_cap, L.exact_cap, pt);
        if (SPEC) {
            // the staging area is dead from here on: start the next unit's row copies into it
            const int nuid = uid + (int)gridDim.x;
            if (nuid < a.n_images * a.n_units)
                cta.gpending = (a.tma_ok ? gather_issue_tma(a, nuid, smem, L.stage_bytes, &sh.gather_mbar)
                                         : gather_issue(a, nuid, smem, L.stage_bytes, &sh.gather_mbar)) ? 1 : 0;
        }
    } else {
        // units wider than the column-per-thread pass: exact rank count for every ROI pixel
        for (int i = tid; i < g.nwords; i += kThreads) {
            unsigned q = MD[i], add = 0;
            int y, c; word_rc(g, i, y, c);
            while (q) {
                const int bpos = __ffs(q) - 1; q &= q - 1;
                if (rank_exact_pixel_thread(gray, g.gp, g.w, g.h, thr, c * 32 + bpos, y)) add |= 1u << bpos;
            }
            MC[i] = add;
        }
        cta_sync();
        n_amb = (int)roi_area;
    }
    pt.tick();   // 11 dirty cells + exact counts
    // ---- P12: open with the 3x3 cross -----------------------------------------
    // (MD, the ROI, is free again; MA may already be receiving the next unit's rows)
    cross3_pass<true>(CAND, MD, g); cta_sync();
    cross3_pass<false>(MD, MB, g);
    for (int i = tid; i < g.nwords; i += kThreads) any_resid |= (MD[i] != 0);       // erosion result non-empty <=> opening non-empty
    any_resid = cta_sync_or(any_resid);
    pt.tick();   // 12 open
    }
    if (!any_resid) {
        // nothing survives the opening: the detector returns None (indexing_ui.py:1559-1560)
        if (def_out) zero_bytes(def_out, npix);
        if (cfg_def_bits) zero_words(bits_at(cfg_def_bits), g.nwords);
        write_record(a, uid, img, unit, otsu_t, seg_area, roi_area, 0, 0, VI_STATUS_OK, dx, dy, cx, cy, n_amb, n_runs_max);
        return;
    }
    // ---- P13: hole fill + per-component contour area filter ---------------------
    n_runs_max = max(n_runs_max, fill_holes(cta, MB, MC, g, ws_s, ws_g, ws, &pt));
    pt.tick();   // 13 defect hole fill
    R = ccl_build(cta, MB, g, true, false, ws_s, ws_g, ws, &pt);
    n_runs_max = max(n_runs_max, R);
    {
        const int Rpad = (R + kThreads - 1) / kThreads * kThreads;
        for (int base = 0; base < Rpad; base += kThreads) {
            int i = base + tid + 1;
            bool valid = i <= R;
            int root = valid ? ws.parent()[i] : 0;
            unsigned a2 = valid ? run_quad_area2(MB, g, ws.yy()[i], ws.xs()[i], ws.xe()[i]) : 0u;
            agg_add(ws.acc0(), valid, root, a2);
        }
    }
    cta_sync();
    const long long min_area = a.p.min_area;
    long long max_area = (long long)__double2ll_rz(__dmul_rn((double)roi_area, a.p.max_area_frac));
    if (max_area < min_area) max_area = min_area;
    const unsigned* acc0 = ws.acc0();
    auto keep = [acc0, min_area, max_area](int root) {
        long long a2 = acc0[root];
        return a2 >= 2 * min_area && a2 <= 2 * max_area;
    };
    unsigned long long kept = 0;
    for (int i = 1 + tid; i <= R; i += kThreads)
        if (ws.parent()[i] == i && keep(i)) ++kept;
    const int n_kept = (int)cta_sum_u64(cta, kept);
    ccl_paint(ME, nullptr, g, ws, keep);
    cta_sync();
    if (a.blobs && n_kept > 0) {
        // the kept components as a table (vi_set_defect_blob_output): a run-time pointer, in every instantiation
        const int kc = min(n_kept, a.blob_k);
        const bool in_masks = kc <= L.blob_cap;
        BlobAcc* tab = reinterpret_cast<BlobAcc*>(in_masks ? smem + L.blob_off : gs + L.blob_tail_off);
        ccl_blob_table(cta, ws, R, keep, kc, in_masks ? L.blob_cap : a.blob_k, tab, a.blobs + (long long)uid * a.blob_k);
    }
    pt.tick();   // 14 component area filter (+ blob table)
    // ---- P14: verdict ---------------------------------------------------------
    const unsigned defect_area = cta_popcount(cta, ME, g);
    if (def_out) store_mask_bytes_sparse(ME, g, def_out);
    if (cfg_def_bits) store_mask_words(ME, g, bits_at(cfg_def_bits));
    const int status = (n_kept > 0 && (long long)defect_area >= min_area) ? VI_STATUS_NG : VI_STATUS_OK;
    write_record(a, uid, img, unit, otsu_t, seg_area, roi_area, n_kept > 0 ? defect_area : 0u, n_kept, status, dx, dy,
                 cx, cy, n_amb, n_runs_max);
    pt.tick();   // 15 defect mask out + record
}

template <bool PROF, bool SPEC, bool GMEM, bool SEG>
__device__ __forceinline__ void unit_kernel_body(const KArgs& a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];      // (128: destination alignment of the tensor copies)
    __shared__ UnitShared sh_raw;
    // The two shared-memory bases are made opaque once: ptxas otherwise re-derives them (S2UR SR_CgaCtaId + a chain
    // of uniform ops) next to nearly every access instead of holding them, also inside the serial Otsu recurrence.
    unsigned char* smem = smem_raw;
    UnitShared* shp = &sh_raw;
    asm volatile("" : "+l"(smem), "+l"(shp));
    __builtin_assume(__isShared(smem));
    __builtin_assume(__isShared(shp));
    UnitShared& sh = *shp;
    const int n_total = a.n_images * a.n_units;
    Cta cta;
    cta.s = &sh.cs; cta.par = 0u; cta.gpar = 0u; cta.gpending = 0;
    if (SPEC) {
        if (threadIdx.x == 0) mbar_init(&sh.gather_mbar, 1u);
        cta_sync();
    }
    unsigned char* base = GMEM ? a.arena + (long long)blockIdx.x * a.layout.arena_bytes : smem;
    if (SPEC && a.tma_ok && (int)blockIdx.x < n_total)           // the first unit's crop arrives the same way as the later ones
        cta.gpending = gather_issue_tma(a, blockIdx.x, smem, a.layout.stage_bytes, &sh.gather_mbar) ? 1 : 0;
    for (int uid = blockIdx.x; uid < n_total; uid += gridDim.x) {
        process_unit<PROF, SPEC, GMEM, SEG>(a, uid, base, smem, sh, cta);
        cta_sync();
    }
}

template <bool PROF, bool SPEC, bool GMEM>
__global__ void __launch_bounds__(kThreads, 1) vi_unit_kernel(const __grid_constant__ KArgs a) {
    unit_kernel_body<PROF, SPEC, GMEM, false>(a);
}

// The default configuration in the segmentation-only mode (process_unit: SPEC && SEG).
template <bool PROF>
__global__ void __launch_bounds__(kThreads, 1) vi_seg_kernel(const __grid_constant__ KArgs a) {
    unit_kernel_body<PROF, true, false, true>(a);
}

}  // namespace vi
