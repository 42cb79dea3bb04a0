// vi_device.cuh -- device-side building blocks of the fused per-unit inspection
// kernel (sm_100a).  One CTA owns one unit at a time; the unit's gray crop and
// all of its masks (bit-packed, 32 px per word) live in shared memory from the
// crop gather to the verdict, so HBM sees 1 B/px in and 2 B/px out.
//
// Reference semantics: SURVEY.md Appendix A; every stage cites the reference
// call site it reproduces (paths under the reference tree).
#pragma once
#include <algorithm>
#include <cstdint>
#include <type_traits>
#include <cuda.h>              // CUtensorMap (type only: the encoder is looked up through the runtime, no libcuda link)
#include <cuda_runtime.h>
#include "../../include/vi_b200.h"

namespace vi {

// Self-checks (the pool's compute-sanitizer is closed): a build with -DVI_CHECKED=1 (libvi_b200_checked.so,
// vi_b200/_build.py) asserts the bounds of every list and table that has a capacity -- the uncertain-pixel list of the
// threshold band, the run tables and the choice between the shared and the global one, union-find parents, the
// dirty-cell and ambiguous-pixel lists and the lattice rows of the median stage, the byte counters of the histogram --
// and records the first failure in a device word that vi_debug_check_word returns (0 = none).  The production build
// compiles them away.  tests/test_gpu_parity.py::test_checked_build_over_adversarial_inputs runs it.
#ifdef VI_CHECKED
__device__ unsigned g_vi_check_word = 0;
#define VI_CHECK(cond, code)                                                          \
    do {                                                                              \
        if (!(cond)) atomicCAS(&::vi::g_vi_check_word, 0u, (unsigned)(code));         \
    } while (0)
#else
#define VI_CHECK(cond, code) do { } while (0)
#endif
enum CheckCode : unsigned {
    CHK_BAND_LIST = 1, CHK_RUN_INDEX = 2, CHK_RUN_CAP = 3, CHK_UF_PARENT = 4, CHK_DIRTY_LIST = 5, CHK_EXACT_LIST = 6,
    CHK_LATTICE_SLOT = 7, CHK_HIST_COUNTER = 8, CHK_ROW_TABLE = 9, CHK_PAINT_RUN = 10, CHK_GATHER_STAGE = 11,
    CHK_BLOB_SLOT = 12,
};

// Pipeline phases.  (Compiling them as __noinline__ functions of their own was measured: reference
// arguments then live in local memory and the labelling phases ran 2-3x slower.)
#define VI_PHASE __device__ inline

constexpr int kThreads = 512;       // worker threads: every phase loop strides by this
constexpr int kWarps = kThreads / 32;
constexpr int kOtsuWarp = kWarps - 1;   // this warp advances the exact Otsu recurrence while others walk columns (vi_rank.cuh)
constexpr int kHistWords = 2048;   // per-warp lane-private histogram: [64 bin-quads][32 lanes] u32, 4 x 8-bit counters
constexpr int kHistBytes = kHistWords * 4;
constexpr int kMaxPeers = 8;       // GPUs of one NVSwitch domain that exchange record tables
constexpr int kMaxTaps = 33;
constexpr int kMaxSE = 33;
constexpr int kMaxAdapt = 201;      // widest adaptive-threshold block (the reference's widget range, indexing_ui.py:805)
constexpr int kLevels = 3;         // rank-count levels of the median stage (one word of three 10-bit fields)
constexpr int kNumMasks = 5;
constexpr unsigned kFull = 0xffffffffu;

enum Mode : int {
    MODE_FULL = 0,      // segmentation + detector + verdict (the hot path)
    MODE_SEG_ONLY = 1,  // segmentation.segment_cell
    MODE_FILL = 2,      // segmentation.fill_internal_holes on aux mask
    MODE_STATS = 3,     // segmentation.mask_stats on aux mask
    MODE_ERODE = 4,     // cv2.erode(mask, None, iterations=r) on aux mask
    MODE_LABEL = 5,     // connectedComponentsWithStats(8) on aux mask
    MODE_DETECT = 6,    // _detect_defects_on_pix with aux mask as the seg mask
};

struct Geom {
    int w, h;
    int wpr;            // mask words per row
    int gp;             // gray pitch in bytes (multiple of 4, odd word count)
    int nwords;         // h * wpr
    unsigned lastmask;  // valid bits of the last word of a row
    unsigned mwpr;      // floor(2^32 / wpr) + 1: i / wpr == __umulhi(i, mwpr) for i < 2^32 / wpr
};

// n / d for n < 2^32 / d through a precomputed m = floor(2^32 / d) + 1 (d > 1).
__host__ __device__ inline unsigned magic_of(unsigned d) { return d > 1 ? 0xFFFFFFFFu / d + 1u : 0u; }
__device__ __forceinline__ unsigned magic_div(unsigned n, unsigned d, unsigned m) { return d > 1 ? __umulhi(n, m) : n; }

__host__ __device__ inline int gray_pitch(int w) {
    int words = (w + 3) / 4;
    if ((words & 1) == 0) words += 1;   // odd pitch in words: row-strided access hits distinct banks
    return words * 4;
}

__host__ __device__ inline Geom make_geom(int w, int h) {
    Geom g;
    g.w = w; g.h = h;
    g.wpr = (w + 31) / 32;
    g.gp = gray_pitch(w);
    g.nwords = h * g.wpr;
    int rem = w & 31;
    g.lastmask = rem ? ((1u << rem) - 1u) : 0xffffffffu;
    g.mwpr = magic_of((unsigned)g.wpr);
    return g;
}

// Geometry of the median stage's lattice workspace (vi_rank.cuh), here because the unit layout below sizes it.
constexpr int kCell = 3;
constexpr int kColsPerWarp = 30;         // V pass: 10 whole cells per warp
constexpr int kVPad = 3;                 // virtual cells either side of a lattice row (the window is 7 cells wide)
constexpr int kGrp = 6;                  // cells per task of the C pass
constexpr unsigned kFlag = 0x20080200u;  // bit 9 of each 10-bit field
constexpr unsigned kGe263 = 249u | (249u << 10) | (249u << 20);   // field + 249 >= 512  <=>  field >= 263
constexpr unsigned kGe179 = 333u | (333u << 10) | (333u << 20);   // field + 333 >= 512  <=>  field >= 179
__host__ __device__ inline int rank_nlx(int w) { return (w + kCell - 1) / kCell; }
__host__ __device__ inline int rank_ngrp(int w) { return (rank_nlx(w) + kGrp - 1) / kGrp; }
// Row pitch of cs in words: every slot a C task can read (kGrp * ngrp + 6) and the V pass's dummy slot; odd, so the
// rows that the lanes of a half-warp hold land on distinct banks.
__host__ __device__ inline int rank_P(int w) { return ((rank_nlx(w) + 2 * kVPad > kGrp * rank_ngrp(w) + 6 ? rank_nlx(w) + 2 * kVPad : kGrp * rank_ngrp(w) + 6) + 1) | 1; }
// cmm pitch: every cell a C task can read, half of it odd (same bank argument for 16-bit entries).
__host__ __device__ inline int rank_cpitch(int w) {
    const int a = kGrp * rank_ngrp(w), b = 4 * ((rank_nlx(w) + 3) / 4);          // cells a C task reads / quads the min-max pass writes
    return 2 * (((a > b ? a : b) + 1) / 2 | 1);
}
__host__ __device__ inline long long rank_ws_bytes(int w, int h) {
    const long long nly = (h + kCell - 1) / kCell;
    return ((((nly + 7) & ~7ll) + 1) * rank_P(w) * 4 + nly * rank_cpitch(w) * 2 + 64 + 15) & ~15ll;      // (+1: the row before row 0)
}

__host__ __device__ inline int align16(int v) { return (v + 15) & ~15; }
__host__ __device__ inline long long align256(long long v) { return (v + 255) & ~255ll; }

// Sizes the unit layout below is built from, defined here and used by the phases that own the regions.
constexpr int kOtsuWsBytes = 3 * 256 * (int)sizeof(double) + 64;     // exact Otsu scan arrays (vi_pipeline.cuh: otsu_scan)
constexpr int kRunBytes = 18;                       // one run of a run table (vi_ccl.cuh: CclWs): parent, 2 accumulators, xs, xe, y
__host__ __device__ inline int ccl_rowfirst_bytes(int h) { return align16((h + 2) * 4); }
__host__ __device__ inline long long ccl_ws_bytes(long long cap, int h) { return ccl_rowfirst_bytes(h) + (cap + 1) * kRunBytes + 64; }
__host__ __device__ inline int ccl_ws_cap(long long bytes, int h) { return (int)((bytes - ccl_rowfirst_bytes(h) - 64) / kRunBytes - 1); }
// Rank plane of the median stage's cell pass (vi_rank.cuh: RankWs::plane) and its list of ambiguous pixels, in scratch.
constexpr int kExactCap = 4096;
__host__ __device__ inline long long rank_plane_words(int wmax, int hmax) { return (long long)rank_ngrp(wmax) * ((((hmax + kCell - 1) / kCell) + 15) & ~15); }
__host__ __device__ inline long long rank_scratch_bytes(int wmax, int hmax) { return rank_plane_words(wmax, hmax) * 4 + kExactCap * 4; }
constexpr int kDirtyListCap = 4096, kExactListCap = 16384;     // rank_finish's lists in the labelling workspace hold at most these
// Accumulator of one kept component of the defect-blob table (vi_ccl.cuh: ccl_blob_table): pixel area, bounding box
// and coordinate sums over its runs; ymin is the root run's row, area2 the area filter's acc0.
struct BlobAcc {
    unsigned long long sx, sy;
    unsigned area, xmin, xmax, ymin, ymax, area2;
};
static_assert(sizeof(BlobAcc) == 40, "BlobAcc layout");

// The largest unit of a grid: its width and height, and the largest crop (gray pitch x height) and bit mask over the
// units (a ragged grid's widest and tallest units need not be the same one).
struct UnitExtent {
    int wmax, hmax, gray_need, mask_words;
    __host__ void add(int w, int h) {
        const Geom g = make_geom(w, h);
        wmax = std::max(wmax, w); hmax = std::max(hmax, h);
        gray_need = std::max(gray_need, g.gp * h); mask_words = std::max(mask_words, g.nwords);
    }
};

// Memory layout of one CTA of vi_unit_kernel, computed on the host per launch (unit_layout) and only read by the kernel.
//
// Dynamic shared memory -- in the arena kernel (GMEM) the CTA's arena in global memory, offsets the same -- holds the
// gray crop, five bit-packed masks MA..ME and a workspace:
//
//   [ gray | MA | MB | MC | MD | ME | workspace ..................... Otsu ]
//
// Phases reuse regions that are dead at the time.  Alias table -- region: the phases that own it; what it overlaps:
//   hist      blur + histogram (P1), shared-memory kernel only (the arena kernel keeps all 16 copies in shared memory
//             and the rest in the arena): n_hist copies from MA on;  MA..ME, workspace and what lies in them
//   lattice   the median stage's cell pass (P2, with the Otsu scan; the pass leaves its results in the scratch plane);
//             MB..ME, workspace up to the Otsu arrays, and the lists and tables below that live there later
//   otsu      the exact Otsu scan (P2);  workspace, run table, dirty / exact lists
//   band      the inverse threshold's uncertain pixels (P3);  MD, ME, lattice, blob table
//   runs      labelling (P5 hole fill to P14);  workspace, lattice, Otsu arrays, dirty / exact lists
//   dirty     dirty cells of the ROI (P11, rank_finish), exact = ambiguous pixels after them;  workspace, lattice,
//             Otsu arrays, run table (the ROI's labelling is done, the defects' has not started)
//   blob      kept-component accumulators (P14);  MC, MD (dead after the area filter), lattice, band; when they do
//             not fit, the scratch blob tail
//   stage     the next unit's crop gather, from rank_finish (P11) on (shared-memory kernel);  gray, MA (the ROI pass
//             is done with both)
//   stage, segmentation kernel: from the first close pass on (P4: the passes alternate MB / MC after reading MA,
//             and the hole fill, centroid, exclusions and stores work on MC);  gray, MA
// Per-CTA scratch in global memory (scratch_bytes apart, L2-resident), no aliases:
//   [ u16 hsum | u8 blurred (rows of whole words) | run-table overflow | rank plane + exact list | f32 plane | blobs ]
struct UnitLayout {
    int gray_bytes;             // gray crop at 0
    int mask_bytes;             // mask k (MA..ME) at gray_bytes + k * mask_bytes; 16-byte multiple
    int ws_off, ws_bytes;       // workspace after the masks
    int otsu_off;               // the last kOtsuWsBytes of the workspace
    int stage_bytes;            // staging area of the crop gather at 0 (128-byte aligned: the dynamic base is)
    int lattice_off;            // the median stage's lattice, from MB on
    int n_hist;                 // lane-private histogram copies that fit (1..16), from MA on (shared-memory kernel)
    int run_rf;                 // row_first bytes of both run tables
    int run_cap;                // runs of the table in the workspace
    int band_off, band_cap;     // inverse threshold's uncertain-pixel list, in words
    int dirty_cap, exact_cap;   // rank_finish's lists: dirty cells at ws_off, ambiguous pixels after them (words)
    int blob_off, blob_cap;     // kept-component accumulators in the masks
    int total;                  // dynamic shared memory bytes
    int arena;                  // units beyond one SM's shared memory: the arena kernel
    long long lattice_bytes;    // room for the lattice from lattice_off up to the Otsu arrays (lattice_fits)
    long long arena_bytes;      // per-CTA arena (arena kernel)
    // scratch, after the u16 horizontal sums at 0: blurred crop, run-table overflow (runs_cap runs), rank plane
    // (rank_words) and kExactCap ambiguous pixels, float plane of the adaptive mean, blobs that do not fit the masks
    long long blur_off, runs_off;
    int runs_cap;
    long long rank_off;
    int rank_words;
    long long f32_off, blob_tail_off, scratch_bytes;
};

// The median stage's lattice of a w x h unit fits the layout.
__host__ __device__ inline bool lattice_fits(int w, int h, const UnitLayout& L) { return rank_ws_bytes(w, h) <= L.lattice_bytes; }
// Enough histogram copies for one round of blur3_hist.
__host__ __device__ inline bool hist_round_fits(int n_hist) { return n_hist >= kWarps / 2; }

// Bounds of a unit: 255 * pixels must fit 32 bits (histogram moments), and the index arithmetic of the phases
// (magic_div: n * d < 2^32) holds for w <= 4096, h <= 8192.  A whole 4096x3000 frame is a legal unit.  The pixel bound
// is a bound per unit (vi_api.cu: set_grid_state): a ragged grid's largest width and largest height, which size the
// layout and the per-CTA scratch, may come from different units and multiply to more than 2^24.
constexpr long long kMaxUnitPixels = 1ll << 24;
constexpr int kMaxUnitW = 4096, kMaxUnitH = 8192;

// The layout for units up to `e`, the device's opt-in shared memory and the kernel's static shared memory (CTA
// histogram, scan scratch, scalars), and the call's options: the adaptive mean's float plane, `blob_k` kept components.
// Shared memory when everything fits one SM (the histogram copies take what is left, the run table what they leave
// past the masks), else the arena in global memory with all 16 histogram copies in shared memory.  False: beyond the
// bound of a unit.
__host__ inline bool unit_layout(const UnitExtent& e, int smem_optin, int smem_static, bool f32_plane, int blob_k, UnitLayout* out) {
    UnitLayout L{};
    L.gray_bytes = align16(e.gray_need);
    L.mask_bytes = align16(e.mask_words * 4);
    const int masks = kNumMasks * L.mask_bytes;
    const int avail = smem_optin - smem_static - L.gray_bytes;
    int ws = align16(std::max<long long>(kOtsuWsBytes, ccl_ws_bytes(2048, e.hmax)));
    if (avail >= masks + ws && avail >= kHistBytes) {
        L.n_hist = std::min(avail / kHistBytes, kWarps);
        const int r_bytes = std::max(L.n_hist * kHistBytes, masks + ws);
        if (r_bytes - masks > ws) ws = (r_bytes - masks) & ~15;
        L.total = L.gray_bytes + r_bytes;
    } else {
        if (e.wmax > kMaxUnitW || e.hmax > kMaxUnitH) return false;
        // the median stage's lattice at wmax x hmax spans the masks after the first and this workspace
        const long long lat = rank_ws_bytes(e.wmax, e.hmax) + kOtsuWsBytes - (long long)(kNumMasks - 1) * L.mask_bytes;
        const long long w = std::max(lat, ccl_ws_bytes(8192, e.hmax));
        if (w > 0x7fff0000ll) return false;
        ws = align16((int)w);
        L.n_hist = kWarps; L.total = kWarps * kHistBytes;
        L.arena = 1; L.arena_bytes = align256((long long)L.gray_bytes + masks + ws);
    }
    L.ws_off = L.gray_bytes + masks; L.ws_bytes = ws;
    L.otsu_off = L.ws_off + ws - kOtsuWsBytes;
    L.stage_bytes = L.lattice_off = L.gray_bytes + L.mask_bytes;
    L.lattice_bytes = (long long)L.otsu_off - L.lattice_off;
    L.run_rf = ccl_rowfirst_bytes(e.hmax); L.run_cap = std::min(ccl_ws_cap(ws, e.hmax), 65534);
    L.band_off = L.gray_bytes + 3 * L.mask_bytes; L.band_cap = 2 * (L.mask_bytes / 4);
    L.dirty_cap = std::min(ws >> 4, kDirtyListCap); L.exact_cap = std::min((ws >> 2) - L.dirty_cap, kExactListCap);
    L.blob_off = L.gray_bytes + 2 * L.mask_bytes; L.blob_cap = 2 * L.mask_bytes / (int)sizeof(BlobAcc);
    const long long px = (long long)e.wmax * e.hmax;
    L.blur_off = (px * 2 + 15) & ~15ll;
    L.runs_off = L.blur_off + (((long long)((e.wmax + 3) & ~3) * e.hmax + 15) & ~15ll);     // blurred rows: whole words
    L.runs_cap = e.hmax * (e.wmax / 2 + 1);
    L.rank_off = align256(L.runs_off + ccl_ws_bytes(L.runs_cap, e.hmax) + 256);
    L.rank_words = (int)rank_plane_words(e.wmax, e.hmax);
    L.f32_off = L.rank_off + align256(rank_scratch_bytes(e.wmax, e.hmax));
    L.blob_tail_off = L.f32_off + (f32_plane ? align256(px * 4) : 0);
    L.scratch_bytes = L.blob_tail_off + align256((long long)blob_k * sizeof(BlobAcc));
    *out = L;
    return true;
}

struct KArgs {
    const uint8_t* frames;
    int n_images, W, H;
    long long row_pitch, image_stride;
    const int4* rects;
    int n_units;
    const long long* unit_off;      // [n_units+1]
    long long unit_px;
    const vi_excl* excl;
    int n_excl;
    const double* refc;             // [n_units][2] or null
    int is_reference;
    vi_params p;
    int blur_k;                     // 0 skip, 3 fast path, else general (odd)
    int taps[kMaxTaps];             // 8.8 fixed-point Gaussian taps for the general path
    int se_k;                       // 0 skip, 3 = cross fast path, else general
    int canny_low, canny_high;      // cv2.Canny thresholds max(1, thr/2), max(2, thr) (indexing_ui.py:1537)
    int adapt_bs;                   // adaptive threshold block size (odd, >= 3); used when p.seg_method == 1
    float ataps[kMaxAdapt];         // float32 Gaussian taps of the adaptive mean (cv2.getGaussianKernel(bs, 0, CV_32F))
    signed char se_lo[kMaxSE], se_hi[kMaxSE];   // per SE row: x-offset span [lo,hi] relative to the anchor (lo>hi: empty)
    uint8_t* seg_out;
    uint8_t* def_out;
    int32_t* labels_out;
    vi_unit_record* rec;
    const uint8_t* aux_mask;        // compat modes: input mask, packed like the outputs
    long long* stats_out;           // compat modes: [n_total][4]
    int mode;
    int erode_r;                    // MODE_ERODE radius
    uint8_t* scratch;               // per-CTA global scratch, layout.scratch_bytes apart
    long long* seg_stats;           // optional: [n_total][3] area, sum x, sum y of the final seg mask (CSV export), or null
    uint32_t* seg_bits;             // optional packed-bit masks (1 bit per pixel, rows of wpr words, PNG bit order), or null
    uint32_t* def_bits;
    const long long* unit_woff;     // [n_units+1] word offsets of the packed-bit masks inside one image's block
    long long unit_words;
    int image_base;                 // records carry image = img * image_mul + image_base (chunked host-buffer call: base;
    int image_mul;                  //  a rank's shard of a multi-GPU job: global index = rank + k * world)
    vi_unit_record* peer_rec[kMaxPeers];   // record tables of all ranks (own included), peer-mapped: the record of global
    int n_peers;                    //  image g, unit u is stored at [g * n_units + u] of every one of them, or 0
    uint8_t* arena;                 // GMEM kernel: per-CTA global arena (layout.arena_bytes apart) holding what shared
                                    //  memory holds otherwise (gray crop, masks, workspace)
    long long* prof;                // diagnostics: [n_total][kProfSlots] per-phase cycle counts, or null
    vi_defect_blob* blobs;          // optional: [n_total][blob_k] kept defect components (vi_set_defect_blob_output), or null
    int blob_k;
    UnitLayout layout;
    // Asynchronous crop gather through the tensor-memory accelerator (vi_pipeline.cuh: gather_issue_tma): the frames as
    // a 3-D uint8 tensor (x, y, image); one box = tma_bw x tma_bh pixels, a crop = tma_ncb x tma_nrb boxes that land as
    // tma_ncb dense tiles of row pitch tma_bw (tma_tile_bytes apart) in the staging area.
    int tma_ok;
    int tma_bw, tma_bh, tma_ncb, tma_nrb, tma_tile_bytes;
    alignas(64) CUtensorMap tmap;
};

// ---------------------------------------------------------------------------
// CTA-wide primitives
// ---------------------------------------------------------------------------
struct CtaScratch {
    // two buffers, used alternately: a collective writes its partials, passes ONE barrier and every warp reduces the
    // kWarps partials on its own; the next collective uses the other buffer, so no trailing barrier is needed (a warp
    // can only reach the call after next by passing the next call's barrier, i.e. after everybody's reads of this one).
    // Kept small: every byte of static shared memory comes out of the histogram copies (unit_layout).
    unsigned long long wl[2][2][kWarps];
    unsigned w32[2][kWarps];
    int flag;
};

// Thread-local handle of the CTA collectives: the shared scratch and the buffer parity (uniform over the CTA because
// every thread runs the same sequence of collectives).
struct Cta {
    CtaScratch* s;
    unsigned par;
    // asynchronous crop gather (vi_pipeline.cuh: gather_issue / gather_finish): phase parity of its mbarrier and whether
    // the next unit's rows are in flight (uniform over the CTA)
    unsigned gpar;
    int gpending;
};

// Diagnostics: per-phase SM cycle counts of one unit (thread 0, after the barrier
// that ends the phase), written only when KArgs::prof is set.
constexpr int kProfSlots = 48;
#define ON_PROF(pt) (std::remove_reference_t<decltype(pt)>::kOn)
struct PtState { long long* out; long long t; int k; int pad; };      // lives in shared memory: no registers held across phases
// ON = false compiles every hook away (the production kernel); ON = true is the diagnostics kernel that
// vi_debug_set_profile selects.
template <bool ON>
struct PhaseTimerT {
    static constexpr bool kOn = ON;
    PtState* s;
    __device__ __forceinline__ void start(PtState* st, long long* o) {
        if (!ON) return;
        s = st;
        if (threadIdx.x == 0) { s->out = o; s->k = 0; if (o) s->t = clock64(); }
    }
    __device__ __forceinline__ void tick() {
        if (!ON) return;
        if (threadIdx.x == 0 && s->out) {
            const long long n = clock64();
            const int k = s->k;
            if (k < kProfSlots) atomicAdd(reinterpret_cast<unsigned long long*>(s->out + k), (unsigned long long)(n - s->t));      // (a reduction: nothing waits for it)
            s->k = k + 1; s->t = n;
        }
    }
    // stamps for a warp other than thread 0's (lane 0 of it records): c = stamp(); ...; c = lap(slot, c);
    __device__ __forceinline__ long long stamp() { return ON ? clock64() : 0ll; }
    __device__ __forceinline__ long long lap(int slot, long long c0) {
        if (!ON) return 0ll;
        const long long n = clock64();
        if ((threadIdx.x & 31) == 0 && s->out) atomicAdd(reinterpret_cast<unsigned long long*>(s->out + slot), (unsigned long long)(n - c0));
        return n;
    }
    __device__ __forceinline__ void count(int slot, int v) { if (ON && (threadIdx.x & 31) == 0 && s->out) atomicAdd(reinterpret_cast<unsigned long long*>(s->out + slot), (unsigned long long)v); }
    // sub-phase accounting: add the time since the last tick/acc to `slot` without consuming a phase slot
    __device__ __forceinline__ void acc(int slot) {
        if (!ON) return;
        if (threadIdx.x == 0 && s->out) { const long long n = clock64(); atomicAdd(reinterpret_cast<unsigned long long*>(s->out + slot), (unsigned long long)(n - s->t)); s->t = n; }
    }
};


__device__ __forceinline__ void cta_sync() { __syncthreads(); }
__device__ __forceinline__ int cta_sync_or(int pred) { return __syncthreads_or(pred); }
// Barrier of the first `nthreads` threads only (named barrier 1): phases that one warp sits out.
__device__ __forceinline__ void workers_sync(int nthreads) { asm volatile("bar.sync 1, %0;" ::"r"(nthreads) : "memory"); }

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ int warp_id() { return threadIdx.x >> 5; }

// Exclusive scan of (a, b) over the CTA's threads; totals returned through ta/tb.  One barrier.
__device__ inline void cta_excl_scan2(Cta& c, unsigned& a, unsigned& b, unsigned& ta, unsigned& tb) {
    const int lane = lane_id(), warp = warp_id();
    const unsigned p = c.par; c.par ^= 1u;
    unsigned ia = a, ib = b;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        unsigned xa = __shfl_up_sync(kFull, ia, o);
        unsigned xb = __shfl_up_sync(kFull, ib, o);
        if (lane >= o) { ia += xa; ib += xb; }
    }
    if (lane == 31) c.s->wl[p][0][warp] = (unsigned long long)ia | ((unsigned long long)ib << 32);
    cta_sync();
    const unsigned long long pv = lane < kWarps ? c.s->wl[p][0][lane] : 0ull;
    const unsigned va = (unsigned)pv, vb = (unsigned)(pv >> 32);
    unsigned sa = va, sb = vb;
#pragma unroll
    for (int o = 1; o < kWarps; o <<= 1) {
        unsigned xa = __shfl_up_sync(kFull, sa, o);
        unsigned xb = __shfl_up_sync(kFull, sb, o);
        if (lane >= o) { sa += xa; sb += xb; }
    }
    ta = __shfl_sync(kFull, sa, kWarps - 1);
    tb = __shfl_sync(kFull, sb, kWarps - 1);
    a = ia - a + __shfl_sync(kFull, sa - va, warp);
    b = ib - b + __shfl_sync(kFull, sb - vb, warp);
}

// Sums over the CTA, one barrier for all of them: v[0], v[1] 64-bit; cta_sum3 adds a 32-bit value in front.
template <int N>
__device__ __forceinline__ void cta_sum_n(Cta& c, unsigned long long (&v)[N]) {
    static_assert(N >= 1 && N <= 2, "cta_sum_n: 1..2 values");
    const int lane = lane_id(), warp = warp_id();
    const unsigned p = c.par; c.par ^= 1u;
#pragma unroll
    for (int k = 0; k < N; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_down_sync(kFull, v[k], o);
        if (lane == 0) c.s->wl[p][k][warp] = v[k];
    }
    cta_sync();
#pragma unroll
    for (int k = 0; k < N; ++k) {
        unsigned long long t = lane < kWarps ? c.s->wl[p][k][lane] : 0ull;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(kFull, t, o);
        v[k] = t;
    }
}

__device__ __forceinline__ void cta_sum3(Cta& c, unsigned& a, unsigned long long& b, unsigned long long& d) {
    const int lane = lane_id(), warp = warp_id();
    const unsigned p = c.par; c.par ^= 1u;
    a = __reduce_add_sync(kFull, a);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { b += __shfl_down_sync(kFull, b, o); d += __shfl_down_sync(kFull, d, o); }
    if (lane == 0) { c.s->w32[p][warp] = a; c.s->wl[p][0][warp] = b; c.s->wl[p][1][warp] = d; }
    cta_sync();
    unsigned ta = lane < kWarps ? c.s->w32[p][lane] : 0u;
    unsigned long long tb = lane < kWarps ? c.s->wl[p][0][lane] : 0ull, td = lane < kWarps ? c.s->wl[p][1][lane] : 0ull;
    a = __reduce_add_sync(kFull, ta);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { tb += __shfl_xor_sync(kFull, tb, o); td += __shfl_xor_sync(kFull, td, o); }
    b = tb; d = td;
}

__device__ inline unsigned long long cta_sum_u64(Cta& c, unsigned long long v) {
    unsigned long long a[1] = {v};
    cta_sum_n<1>(c, a);
    return a[0];
}

__device__ inline unsigned long long cta_max_u64(Cta& c, unsigned long long v) {
    const int lane = lane_id(), warp = warp_id();
    const unsigned p = c.par; c.par ^= 1u;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long x = __shfl_down_sync(kFull, v, o);
        v = x > v ? x : v;
    }
    if (lane == 0) c.s->wl[p][0][warp] = v;
    cta_sync();
    unsigned long long t = lane < kWarps ? c.s->wl[p][0][lane] : 0ull;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long x = __shfl_xor_sync(kFull, t, o);
        t = x > t ? x : t;
    }
    return t;
}

// ---------------------------------------------------------------------------
// Bit-packed mask rows.  Bit x&31 of word x>>5 is pixel x; bits >= w of the last
// word of a row are always 0.
// ---------------------------------------------------------------------------
// (row, word) of mask word index i
__device__ __forceinline__ void word_rc(const Geom& g, int i, int& y, int& c) {
    y = (int)magic_div((unsigned)i, (unsigned)g.wpr, g.mwpr);
    c = i - y * g.wpr;
}

__device__ __forceinline__ unsigned row_mask_of(const Geom& g, int c) { return c == g.wpr - 1 ? g.lastmask : 0xffffffffu; }

// Word c of row y; rows outside [0,h) and words outside [0,wpr) read as `fill`
// (0 or ~0); with fill = ~0 the padding bits of the last word read as 1 too.
__device__ __forceinline__ unsigned mword(const unsigned* M, const Geom& g, int y, int c, unsigned fill) {
    if ((unsigned)y >= (unsigned)g.h || (unsigned)c >= (unsigned)g.wpr) return fill;
    unsigned v = M[y * g.wpr + c];
    if (c == g.wpr - 1) v |= fill & ~g.lastmask;
    return v;
}

// Word c of row y shifted so that bit x takes the value of pixel x+dx
// (dx may be negative); pixels outside [0,w) read as `fill`.
__device__ __forceinline__ unsigned mword_shift(const unsigned* M, const Geom& g, int y, int c, int dx, unsigned fill) {
    if (dx == 0) return mword(M, g, y, c, fill);
    int bit0 = c * 32 + dx;                 // pixel index that lands on bit 0
    int c0 = bit0 >> 5;                     // floor division (arithmetic shift)
    int s = bit0 & 31;
    unsigned lo = mword(M, g, y, c0, fill);
    if (s == 0) return lo;
    unsigned hi = mword(M, g, y, c0 + 1, fill);
    return __funnelshift_r(lo, hi, s);
}

// Bits [a, b] (inclusive, 0 <= a <= b <= 31).
__device__ __forceinline__ unsigned bit_range(int a, int b) {
    unsigned hi = (b >= 31) ? 0xffffffffu : ((1u << (b + 1)) - 1u);
    return hi & ~((1u << a) - 1u);
}

// One pass of a 3x3-cross erosion (out-of-crop = 1) or dilation (out-of-crop = 0):
// cv2.getStructuringElement(MORPH_ELLIPSE,(3,3)) is the cross (SURVEY A.5).
template <bool ERODE>
VI_PHASE void cross3_pass(const unsigned* src, unsigned* dst, const Geom& g) {
    const unsigned fill = ERODE ? 0xffffffffu : 0u;
    const unsigned pad = fill & ~g.lastmask;             // padding bits of a row's last word read as `fill`
    for (int i = threadIdx.x; i < g.nwords; i += kThreads) {
        int y, c; word_rc(g, i, y, c);
        const bool last = c == g.wpr - 1;
        const unsigned m = src[i] | (last ? pad : 0u);
        const unsigned lw = c > 0 ? src[i - 1] : fill;
        const unsigned rw = last ? fill : (src[i + 1] | (c + 1 == g.wpr - 1 ? pad : 0u));
        const unsigned u = y > 0 ? src[i - g.wpr] : fill;
        const unsigned dn = y < g.h - 1 ? src[i + g.wpr] : fill;
        const unsigned l = (m << 1) | (lw >> 31), r = (m >> 1) | (rw << 31);
        const unsigned o = ERODE ? (m & l & r & u & dn) : (m | l | r | u | dn);
        dst[i] = o & (last ? g.lastmask : 0xffffffffu);
    }
}

// General structuring element given as per-row x-offset spans (the ellipse of
// segmentation.py:93).  erode: AND over offsets, outside = 1; dilate: OR over the
// same (un-reflected) offsets, outside = 0 (SURVEY A.5).
template <bool ERODE>
VI_PHASE void se_pass(const unsigned* src, unsigned* dst, const Geom& g, int k,
                               const signed char* lo, const signed char* hi) {
    const unsigned fill = ERODE ? 0xffffffffu : 0u;
    const int a = k / 2;
    for (int i = threadIdx.x; i < g.nwords; i += kThreads) {
        int y, c; word_rc(g, i, y, c);
        unsigned o = fill;
        for (int j = 0; j < k; ++j) {
            int ys = y + j - a;
            if (lo[j] > hi[j]) continue;
            if ((unsigned)ys >= (unsigned)g.h) continue;   // out-of-crop rows never constrain either op
            for (int dx = lo[j]; dx <= hi[j]; ++dx) {
                unsigned v = mword_shift(src, g, ys, c, dx, fill);
                o = ERODE ? (o & v) : (o | v);
            }
        }
        dst[i] = o & row_mask_of(g, c);
    }
}

// Replicate-clamped variants: pixels / rows outside the crop read as the nearest
// edge pixel / row.
__device__ __forceinline__ unsigned mword_shift_rep(const unsigned* M, const Geom& g, int y, int c, int dx) {
    unsigned edge = dx < 0 ? (M[y * g.wpr] & 1u) : ((M[y * g.wpr + g.wpr - 1] >> ((g.w - 1) & 31)) & 1u);
    return mword_shift(M, g, y, c, dx, edge ? 0xffffffffu : 0u);
}

// Centred square erosion by radius r with out-of-crop = 1
// (cv2.erode(seg_bin, None, iterations=r), indexing_ui.py:1497; SURVEY A.5).
// Window doubling on 32-px words: with W_a[x] = AND of the in-crop pixels of
// [x-a, x+a], W_{a+b}[x] = W_a[clamp(x-b)] & W_a[clamp(x+b)] for b <= a (clamping the
// position keeps every term inside the target window), so any radius takes
// ceil(log2 r)+1 passes per axis.  Ping-pongs between bufA and bufB; returns the
// buffer that holds the result.  `src` must not be bufA or bufB's partner in use.
constexpr int kErodeDirectMax = 10;     // radii up to this take one direct pass per axis

// Vertical AND over the rows y-R .. y+R (clamped: the edge row replicated) for a segment of eight rows of one word
// column: the 8 + 2R rows are read once and the windows are built by doubling in registers
// (spans 1, 2, 4, .. then one overlapped pair), about 7 ANDs and 2.5 loads per output word at R = 6 instead of 12 + 12.
template <int R>
__device__ __forceinline__ void erode_rows_seg(const unsigned* cur, unsigned* nxt, const Geom& g) {
    constexpr int S = 8, N = S + 2 * R, W = 2 * R + 1;
    constexpr int PW = W >= 16 ? 16 : (W >= 8 ? 8 : (W >= 4 ? 4 : 2));      // largest power of two <= W (W >= 3)
    const int nseg = (g.h + S - 1) / S;
    const int ntask = nseg * g.wpr;
    const int hm1 = g.h - 1;
    for (int t = threadIdx.x; t < ntask; t += kThreads) {
        int sg, c; word_rc(g, t, sg, c);
        const int y0 = sg * S;
        unsigned a[N];
        if (y0 - R >= 0 && y0 + S - 1 + R <= hm1) {
            const unsigned* p = cur + (y0 - R) * g.wpr + c;
#pragma unroll
            for (int k = 0; k < N; ++k) { a[k] = *p; p += g.wpr; }
        } else {
#pragma unroll
            for (int k = 0; k < N; ++k) a[k] = cur[min(max(y0 - R + k, 0), hm1) * g.wpr + c];
        }
        // a[i] = AND of rows i .. i + span - 1
#pragma unroll
        for (int i = 0; i + 2 <= N; ++i) a[i] &= a[i + 1];
        if (PW >= 4) {
#pragma unroll
            for (int i = 0; i + 4 <= N; ++i) a[i] &= a[i + 2];
        }
        if (PW >= 8) {
#pragma unroll
            for (int i = 0; i + 8 <= N; ++i) a[i] &= a[i + 4];
        }
        if (PW >= 16) {
#pragma unroll
            for (int i = 0; i + 16 <= N; ++i) a[i] &= a[i + 8];
        }
        unsigned* o = nxt + y0 * g.wpr + c;
#pragma unroll
        for (int i = 0; i < S; ++i) {
            if (y0 + i <= hm1) *o = a[i] & a[i + W - PW];
            o += g.wpr;
        }
    }
}

VI_PHASE unsigned* erode_square_bits(const unsigned* src, unsigned* bufA, unsigned* bufB, const Geom& g, int r) {
    const unsigned* cur = src;
    unsigned* nxt = (src == bufA) ? bufB : bufA;
    if (r <= kErodeDirectMax) {
        // horizontal: AND of the 2r+1 shifts, built from the three neighbouring words (edge pixel replicated)
        for (int i = threadIdx.x; i < g.nwords; i += kThreads) {
            int y, c; word_rc(g, i, y, c);
            const unsigned* row = cur + y * g.wpr;
            const unsigned fl = (row[0] & 1u) ? 0xffffffffu : 0u;
            const unsigned fr = ((row[g.wpr - 1] >> ((g.w - 1) & 31)) & 1u) ? 0xffffffffu : 0u;
            const unsigned padr = fr & ~g.lastmask;
            const unsigned C = row[c] | (c == g.wpr - 1 ? padr : 0u);
            const unsigned L = c > 0 ? row[c - 1] : fl;
            const unsigned R = c < g.wpr - 1 ? (row[c + 1] | (c + 1 == g.wpr - 1 ? padr : 0u)) : fr;
            unsigned v = C;
            for (int d = 1; d <= r; ++d) v &= __funnelshift_r(C, R, d) & __funnelshift_l(L, C, d);
            nxt[i] = v & row_mask_of(g, c);
        }
        cta_sync();
        cur = nxt;
        nxt = (cur == bufA) ? bufB : bufA;
        // vertical: AND of the 2r+1 rows (edge row replicated), eight rows of one word column per thread
        switch (r) {
            case 1: erode_rows_seg<1>(cur, nxt, g); break;
            case 2: erode_rows_seg<2>(cur, nxt, g); break;
            case 3: erode_rows_seg<3>(cur, nxt, g); break;
            case 4: erode_rows_seg<4>(cur, nxt, g); break;
            case 5: erode_rows_seg<5>(cur, nxt, g); break;
            case 6: erode_rows_seg<6>(cur, nxt, g); break;
            case 7: erode_rows_seg<7>(cur, nxt, g); break;
            case 8: erode_rows_seg<8>(cur, nxt, g); break;
            case 9: erode_rows_seg<9>(cur, nxt, g); break;
            default: erode_rows_seg<10>(cur, nxt, g); break;
        }
        cta_sync();
        return nxt;
    }
    int a = 0;
    while (a < r) {                                    // horizontal
        int b = (a == 0) ? 1 : ((2 * a <= r) ? a : (r - a));
        for (int i = threadIdx.x; i < g.nwords; i += kThreads) {
            int y, c; word_rc(g, i, y, c);
            unsigned v = mword_shift_rep(cur, g, y, c, -b) & mword_shift_rep(cur, g, y, c, +b);
            if (a == 0) v &= cur[i];
            nxt[i] = v & row_mask_of(g, c);
        }
        cta_sync();
        a += b;
        cur = nxt;
        nxt = (cur == bufA) ? bufB : bufA;
    }
    a = 0;
    while (a < r) {                                    // vertical
        int b = (a == 0) ? 1 : ((2 * a <= r) ? a : (r - a));
        for (int i = threadIdx.x; i < g.nwords; i += kThreads) {
            int y, c; word_rc(g, i, y, c);
            unsigned v = cur[max(y - b, 0) * g.wpr + c] & cur[min(y + b, g.h - 1) * g.wpr + c];
            if (a == 0) v &= cur[i];
            nxt[i] = v;
        }
        cta_sync();
        a += b;
        cur = nxt;
        nxt = (cur == bufA) ? bufB : bufA;
    }
    return const_cast<unsigned*>(cur);
}

// Four bytes against one pivot p at a time: flag (bit 0 of each byte) = byte > p.  K and sel encode p once per
// pixel: p < 0 -> every byte is greater; p >= 255 -> none; else the low seven bits are compared by an add that
// carries into bit 7 and the high bit decides the rest.
struct SwarPivot { unsigned K, sel; };
__device__ __forceinline__ SwarPivot swar_pivot(int p) {
    SwarPivot q;
    if (p < 0) { q.K = 0x80808080u; q.sel = 0xffffffffu; }
    else {
        const int pc = min(p, 255);
        q.K = (unsigned)(0x7f - (pc & 127)) * 0x01010101u;
        q.sel = pc < 128 ? 0xffffffffu : 0u;
    }
    return q;
}
__device__ __forceinline__ unsigned swar_gt7(unsigned W, const SwarPivot& q) {      // flags at bit 7 of each byte
    const unsigned t = (W & 0x7f7f7f7fu) + q.K;              // bit 7: low seven bits > (p & 127)
    return ((t & W) | ((t | W) & q.sel)) & 0x80808080u;       // p >= 128: high bit and low bits greater; p < 128: either
}
__device__ __forceinline__ unsigned swar_gt(unsigned W, const SwarPivot& q) { return swar_gt7(W, q) >> 7; }
// The four bit-7 flags of a word as a nibble (bit k = byte k): one multiply lines them up at bits 28..31.
__device__ __forceinline__ unsigned swar_nibble(unsigned f7) { return (f7 * 0x00204081u) >> 28; }

__device__ inline unsigned cta_popcount(Cta& cs, const unsigned* M, const Geom& g) {
    unsigned long long n = 0;
    for (int i = threadIdx.x; i < g.nwords; i += kThreads) n += __popc(M[i]);
    return (unsigned)cta_sum_u64(cs, n);
}

}  // namespace vi
