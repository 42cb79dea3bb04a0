// vi_api.cu -- C ABI (include/vi_b200.h) over the fused inspection kernel.
// Host side: context, parameter normalisation (the reference's widget rules),
// launch, the pipelined host-buffer batch call and the per-unit compat calls.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

#include "vi_unit.cuh"
#include "vi_ingest.cuh"

using namespace vi;

static thread_local std::string g_err;

static int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) return fail(VI_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_));  \
    } while (0)

// Sets the context's device for the duration of an entry point and restores the caller's current device.
struct DeviceGuard {
    int prev = -1;
    bool ok = true, changed = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) { ok = cudaSetDevice(dev) == cudaSuccess; changed = ok; }
    }
    ~DeviceGuard() { if (prev >= 0 && changed) cudaSetDevice(prev); }
};
#define VI_DEVICE(c)                                                                               \
    DeviceGuard dg_((c)->device);                                                                  \
    if (!dg_.ok) return fail(VI_ERR_CUDA, "cudaSetDevice(%d) failed", (c)->device)

struct DevBuf {
    void* p = nullptr;
    size_t n = 0;
    int ensure(size_t bytes) {
        if (bytes <= n) return VI_OK;
        if (p) cudaFree(p);
        p = nullptr; n = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) return fail(VI_ERR_CUDA, "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e));
        n = bytes;
        return VI_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
};

constexpr int kHostSlots = 3;      // chunks in flight in the host-buffer batch call (upload / kernel / download overlap)

struct GridState {
    std::vector<int4> rects;
    std::vector<long long> off;     // n+1
    long long unit_px = 0;
    UnitExtent ext{};               // the largest unit: sizes the kernel's layout (unit_layout)
    std::vector<long long> woff;    // n+1: packed-bit mask offsets in 32-bit words
    long long unit_words = 0;
    DevBuf d_rects, d_off, d_woff;
};

struct vi_ctx {
    int device = 0;
    int sm_count = 0;
    int smem_optin = 0;
    int smem_static = 0;
    GridState grid;                 // user grid
    GridState one;                  // single-rect grid of the compat calls
    std::vector<vi_excl> excl;
    DevBuf d_excl;
    DevBuf d_refc;
    bool has_refc = false;
    int is_reference = 0;
    DevBuf scratch;
    DevBuf arena;
    // compat / host-batch staging
    DevBuf st_in, st_aux, st_out, st_out2, st_rec, st_stats, st_lab;
    DevBuf hb_frames[kHostSlots], hb_seg[kHostSlots], hb_def[kHostSlots], hb_rec[kHostSlots], hb_blob[kHostSlots];
    cudaStream_t streams[kHostSlots] = {};
    int smem_set = 0;
    long long* prof = nullptr;
    long long* seg_stats = nullptr;
    uint32_t* seg_bits = nullptr;   // optional packed-bit outputs of vi_inspect_batch (vi_set_packed_mask_output)
    uint32_t* def_bits = nullptr;
    vi_defect_blob* blobs = nullptr;   // optional kept-component table of vi_inspect_batch (vi_set_defect_blob_output)
    int blob_k = 0;
    // Ordering: the context's tables and per-CTA scratch are shared by every call.  `busy` is recorded after each
    // asynchronous launch on a caller's stream; every later entry point waits on it (streams: cudaStreamWaitEvent,
    // host-side table updates: cudaEventSynchronize) before it touches them.
    cudaEvent_t busy = nullptr;
    bool busy_set = false;
    // multi-GPU record exchange (vi_set_record_peers)
    vi_unit_record* peer_rec[kMaxPeers] = {};
    int n_peers = 0, image_mul = 1, image_add = 0;
};

static int wait_busy_host(vi_ctx* c) {
    if (c->busy_set) {
        cudaError_t e = cudaEventSynchronize(c->busy);
        if (e != cudaSuccess) return fail(VI_ERR_CUDA, "cudaEventSynchronize: %s", cudaGetErrorString(e));
        c->busy_set = false;
    }
    return VI_OK;
}

static int wait_busy_stream(vi_ctx* c, cudaStream_t st) {
    if (c->busy_set) {
        cudaError_t e = cudaStreamWaitEvent(st, c->busy, 0);
        if (e != cudaSuccess) return fail(VI_ERR_CUDA, "cudaStreamWaitEvent: %s", cudaGetErrorString(e));
    }
    return VI_OK;
}

static int mark_busy(vi_ctx* c, cudaStream_t st) {
    cudaError_t e = cudaEventRecord(c->busy, st);
    if (e != cudaSuccess) return fail(VI_ERR_CUDA, "cudaEventRecord: %s", cudaGetErrorString(e));
    c->busy_set = true;
    return VI_OK;
}

extern "C" const char* vi_last_error(void) { return g_err.c_str(); }
extern "C" int vi_version(void) { return 100; }

extern "C" void vi_params_default(vi_params* p) {
    if (!p) return;
    p->seg_method = 0; p->gaussian_blur = 3; p->morph_kernel = 3; p->adapt_block = 51; p->adapt_C = 10;
    p->defect_method = 0; p->threshold = 24; p->min_area = 20; p->erode_px = 6; p->median_ksize = 21;
    p->max_area_frac = 0.98;
}

extern "C" int vi_ctx_create(int device, vi_ctx** out) {
    if (!out) return fail(VI_ERR_ARG, "vi_ctx_create: out is null");
    int n = 0;
    CU(cudaGetDeviceCount(&n));
    if (device < 0 || device >= n) return fail(VI_ERR_ARG, "vi_ctx_create: device %d of %d", device, n);
    DeviceGuard dg(device);
    if (!dg.ok) return fail(VI_ERR_CUDA, "cudaSetDevice(%d) failed", device);
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    vi_ctx* c = new vi_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->smem_optin = (int)prop.sharedMemPerBlockOptin;
    cudaFuncAttributes fa;
    CU(cudaFuncGetAttributes(&fa, vi_unit_kernel<false, false, false>));
    c->smem_static = ((int)fa.sharedSizeBytes + 127) & ~127;       // the dynamic part starts 128-byte aligned (tensor copies land there)
    for (auto& s : c->streams) {
        cudaError_t e = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
        if (e != cudaSuccess) { delete c; return fail(VI_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e)); }
    }
    {
        cudaError_t e = cudaEventCreateWithFlags(&c->busy, cudaEventDisableTiming);
        if (e != cudaSuccess) { vi_ctx_destroy(c); return fail(VI_ERR_CUDA, "cudaEventCreate: %s", cudaGetErrorString(e)); }
    }
    *out = c;
    return VI_OK;
}

extern "C" void vi_ctx_destroy(vi_ctx* c) {
    if (!c) return;
    DeviceGuard dg(c->device);
    cudaDeviceSynchronize();
    if (c->busy) cudaEventDestroy(c->busy);
    for (GridState* g : {&c->grid, &c->one}) { g->d_rects.release(); g->d_off.release(); g->d_woff.release(); }
    for (DevBuf* b : {&c->d_excl, &c->d_refc, &c->scratch, &c->arena, &c->st_in, &c->st_aux, &c->st_out, &c->st_out2, &c->st_rec,
                      &c->st_stats, &c->st_lab})
        b->release();
    for (int i = 0; i < kHostSlots; ++i) {
        c->hb_frames[i].release(); c->hb_seg[i].release(); c->hb_def[i].release(); c->hb_rec[i].release(); c->hb_blob[i].release();
        if (c->streams[i]) cudaStreamDestroy(c->streams[i]);
    }
    delete c;
}

// Table uploads come from pageable host memory: cudaMemcpy may return while the DMA to the device is still in
// flight, and the kernels run on non-blocking streams that the legacy stream does not order against -- so the
// upload is either issued on the stream that launches next (`st`) or followed by a device synchronise.
static int set_grid_state(vi_ctx* c, GridState& gs, const int32_t* r, int n, cudaStream_t st = nullptr) {
    if (!r || n <= 0) return fail(VI_ERR_ARG, "grid: need at least one rect");
    gs.rects.resize(n);
    gs.off.assign(n + 1, 0);
    gs.woff.assign(n + 1, 0);
    gs.ext = UnitExtent{};
    for (int i = 0; i < n; ++i) {
        int x = r[4 * i], y = r[4 * i + 1], w = r[4 * i + 2], h = r[4 * i + 3];
        if (w <= 0 || h <= 0 || x < 0 || y < 0) return fail(VI_ERR_ARG, "grid: rect %d = (%d,%d,%d,%d) is invalid", i, x, y, w, h);
        if (w > kMaxUnitW || h > kMaxUnitH || (long long)w * h > kMaxUnitPixels)
            return fail(VI_ERR_TOO_LARGE, "grid: rect %d is %dx%d: beyond the bound of a unit (%d wide, %d high, %lld pixels)", i, w, h,
                        kMaxUnitW, kMaxUnitH, kMaxUnitPixels);
        gs.rects[i] = make_int4(x, y, w, h);
        gs.off[i + 1] = gs.off[i] + (long long)w * h;
        gs.woff[i + 1] = gs.woff[i] + (long long)((w + 31) / 32) * h;
        gs.ext.add(w, h);
    }
    gs.unit_px = gs.off[n];
    gs.unit_words = gs.woff[n];
    // Units larger than one SM's shared memory take the arena kernel.  The pixel bound holds per unit (checked above);
    // a ragged grid's wmax x hmax may exceed it (a 4096 x 200 strip next to a 200 x 8000 column), and everything sized
    // from wmax x hmax is 64-bit or within int range up to 4096 x 8192.
    UnitLayout layout;
    if (!unit_layout(gs.ext, c->smem_optin, c->smem_static, false, 0, &layout))
        return fail(VI_ERR_TOO_LARGE, "grid: units up to %d x %d exceed the bound of a unit (%d wide, %d high)",
                    gs.ext.wmax, gs.ext.hmax, kMaxUnitW, kMaxUnitH);
    int rc;
    if ((rc = gs.d_rects.ensure(sizeof(int4) * n))) return rc;
    if ((rc = gs.d_off.ensure(sizeof(long long) * (n + 1)))) return rc;
    if ((rc = gs.d_woff.ensure(sizeof(long long) * (n + 1)))) return rc;
    if (st) {
        CU(cudaMemcpyAsync(gs.d_rects.p, gs.rects.data(), sizeof(int4) * n, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(gs.d_off.p, gs.off.data(), sizeof(long long) * (n + 1), cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(gs.d_woff.p, gs.woff.data(), sizeof(long long) * (n + 1), cudaMemcpyHostToDevice, st));
    } else {
        CU(cudaMemcpy(gs.d_rects.p, gs.rects.data(), sizeof(int4) * n, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(gs.d_off.p, gs.off.data(), sizeof(long long) * (n + 1), cudaMemcpyHostToDevice));
        CU(cudaMemcpy(gs.d_woff.p, gs.woff.data(), sizeof(long long) * (n + 1), cudaMemcpyHostToDevice));
        CU(cudaDeviceSynchronize());
    }
    return VI_OK;
}

extern "C" int vi_set_grid(vi_ctx* c, const int32_t* rects, int n) {
    if (!c) return fail(VI_ERR_ARG, "ctx is null");
    VI_DEVICE(c);
    int rcw;
    if ((rcw = wait_busy_host(c))) return rcw;             // an in-flight batch may still be reading the tables
    c->has_refc = false;     // grid changed: reference centroids no longer valid (indexing_ui.py:2196-2200)
    return set_grid_state(c, c->grid, rects, n);
}

extern "C" int vi_set_exclusions(vi_ctx* c, const vi_excl* e, int n) {
    if (!c) return fail(VI_ERR_ARG, "ctx is null");
    if (n < 0 || (n > 0 && !e)) return fail(VI_ERR_ARG, "exclusions: bad arguments");
    if (n > 4096) return fail(VI_ERR_ARG, "exclusions: %d is too many", n);
    VI_DEVICE(c);
    int rcw;
    if ((rcw = wait_busy_host(c))) return rcw;
    c->excl.assign(e, e + n);
    if (n) {
        int rc;
        if ((rc = c->d_excl.ensure(sizeof(vi_excl) * n))) return rc;
        CU(cudaMemcpy(c->d_excl.p, e, sizeof(vi_excl) * n, cudaMemcpyHostToDevice));
        CU(cudaDeviceSynchronize());
    }
    return VI_OK;
}

extern "C" int vi_set_ref_centroids(vi_ctx* c, const double* cxcy, int n_units, int is_reference) {
    if (!c) return fail(VI_ERR_ARG, "ctx is null");
    VI_DEVICE(c);
    int rcw;
    if ((rcw = wait_busy_host(c))) return rcw;
    c->is_reference = is_reference ? 1 : 0;
    if (!cxcy) { c->has_refc = false; return VI_OK; }
    if (n_units != (int)c->grid.rects.size()) return fail(VI_ERR_ARG, "ref centroids: %d entries for %zu units", n_units, c->grid.rects.size());
    int rc;
    if ((rc = c->d_refc.ensure(sizeof(double) * 2 * n_units))) return rc;
    CU(cudaMemcpy(c->d_refc.p, cxcy, sizeof(double) * 2 * n_units, cudaMemcpyHostToDevice));
    CU(cudaDeviceSynchronize());
    c->has_refc = true;
    return VI_OK;
}

// Diagnostics: div_y / div_with_y against the IEEE divide on pseudo-random operand pairs drawn like
// the Otsu recurrence's (numerator in [0, 256), divisor in (2^-24, 1]), plus divisors with
// long runs of one bits in the significand.
__global__ void fastdiv_check_kernel(unsigned long long seed, long long per_thread, unsigned long long* bad) {
    unsigned long long s = seed + 0x9E3779B97F4A7C15ull * (blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x + 1);
    unsigned long long nbad = 0;
    for (long long i = 0; i < per_thread; ++i) {
        s ^= s << 13; s ^= s >> 7; s ^= s << 17;
        unsigned long long m1 = s & 0x000fffffffffffffull;
        s ^= s << 13; s ^= s >> 7; s ^= s << 17;
        unsigned long long m2 = s & 0x000fffffffffffffull;
        const int kind = (int)((s >> 52) & 7);
        if (kind == 0) m2 |= 0x000fffffffff0000ull;                 // significand close to all ones
        if (kind == 1) m2 = 0x000fffffffffffffull - (m2 & 0xff);
        if (kind == 2) m1 &= 0x000ff00000000000ull;                 // short numerators (small integers / sums)
        const int eb = 1023 - (int)((s >> 56) % 24);                // divisor in (2^-24, 1]
        const int en = 1023 + 7 - (int)((s >> 60) % 12);            // numerator in [2^-4, 256)
        const double b = __longlong_as_double(((long long)eb << 52) | (long long)m2);
        const double n = __longlong_as_double(((long long)en << 52) | (long long)m1);
        const double q = vi::div_with_y(n, b, vi::div_y(b)), ref = __ddiv_rn(n, b);
        if (__double_as_longlong(q) != __double_as_longlong(ref)) ++nbad;
    }
    if (nbad) atomicAdd(bad, nbad);
}

extern "C" int vi_debug_fastdiv_check(vi_ctx* c, long long n_samples, unsigned long long seed, long long* mismatches) {
    if (!c || !mismatches) return fail(VI_ERR_ARG, "vi_debug_fastdiv_check: null");
    VI_DEVICE(c);
    unsigned long long* d_bad = nullptr;
    CU(cudaMalloc(&d_bad, 8));
    CU(cudaMemset(d_bad, 0, 8));
    const int blocks = 4 * c->sm_count, threads = 256;
    long long per = (n_samples + (long long)blocks * threads - 1) / ((long long)blocks * threads);
    fastdiv_check_kernel<<<blocks, threads>>>(seed, per, d_bad);
    unsigned long long h = 0;
    cudaError_t e = cudaMemcpy(&h, d_bad, 8, cudaMemcpyDeviceToHost);
    cudaFree(d_bad);
    if (e != cudaSuccess) return fail(VI_ERR_CUDA, "fastdiv check: %s", cudaGetErrorString(e));
    *mismatches = (long long)h;
    return VI_OK;
}

// Diagnostics: the device Otsu of arbitrary histograms, one 2-warp CTA each.  Warp 0 runs otsu_approx_warp and
// publishes the bound before the barrier, so otsu_scan on warp 1 always finds it (the inspection kernel runs the two
// concurrently).  out[3b .. 3b+2] = t, t_apx, last; -1 for a histogram whose npix is outside 1..2^24 or not its sum.
__global__ void otsu_debug_kernel(const uint32_t* hists, const int* npix, int* out, unsigned* bad) {
    __shared__ unsigned hist[256];
    __shared__ __align__(16) double ws[vi::kOtsuWsBytes / 8];
    __shared__ int last_s, tapx_s, ok_s;
    const long long b = blockIdx.x;
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = hists[b * 256 + i];
    __syncthreads();
    const int N = npix[b];
    if (threadIdx.x < 32) {
        unsigned long long s = 0;
        for (int i = threadIdx.x; i < 256; i += 32) s += hist[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(vi::kFull, s, o);
        if (threadIdx.x == 0) { ok_s = N >= 1 && N <= (1 << 24) && s == (unsigned long long)N; last_s = -1; }
    }
    __syncthreads();
    if (!ok_s) {
        if (threadIdx.x == 0) { out[3 * b] = out[3 * b + 1] = out[3 * b + 2] = -1; atomicAdd(bad, 1u); }
        return;
    }
    vi::PhaseTimerT<false> pt;
    if (threadIdx.x < 32) {
        int last;
        const int ta = vi::otsu_approx_warp(hist, N, last);
        if (threadIdx.x == 0) { tapx_s = ta; last_s = last; }
    }
    __syncthreads();
    if (threadIdx.x >= 32) {
        const int t = vi::otsu_scan(hist, N, ws, &last_s, pt);
        if (threadIdx.x == 32) { out[3 * b] = t; out[3 * b + 1] = tapx_s; out[3 * b + 2] = last_s; }
    }
}

extern "C" int vi_debug_otsu(vi_ctx* c, const uint32_t* d_hists, const int* d_npix, int n, int* d_out) {
    if (!c || n < 0 || (n > 0 && (!d_hists || !d_npix || !d_out))) return fail(VI_ERR_ARG, "vi_debug_otsu: null or n < 0");
    if (n == 0) return VI_OK;
    VI_DEVICE(c);
    unsigned* d_bad = nullptr;
    CU(cudaMalloc(&d_bad, 4));
    CU(cudaMemset(d_bad, 0, 4));
    otsu_debug_kernel<<<n, 64>>>(d_hists, d_npix, d_out, d_bad);
    unsigned h = 0;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpy(&h, d_bad, 4, cudaMemcpyDeviceToHost);
    cudaFree(d_bad);
    if (e != cudaSuccess) return fail(VI_ERR_CUDA, "vi_debug_otsu: %s", cudaGetErrorString(e));
    if (h) return fail(VI_ERR_ARG, "vi_debug_otsu: %u histograms whose npix is outside 1..2^24 or differs from their sum", h);
    return VI_OK;
}

// Diagnostics: the median residual stage on its own, one CTA running the device functions of the inspection kernel in
// its order (vi_unit.cuh, P2 and P11): the crop's histogram and otsu_approx_warp on warp 0 next to the cell min / max
// (the exact Otsu scan aside on kOtsuWarp when the V pass leaves it free), rank_cells, rank_finish.  The workspace is a
// global arena as in the GMEM kernel; the crop is copied to the kernel's row pitch with `pad` in the bytes past w.
// out[0] = ambiguous-pixel list entries (counters[1]), out[1] = dirty cells that touch the ROI (counters[0]), out[2] = otsu_t.
__global__ void __launch_bounds__(kThreads) rank_debug_kernel(const uint8_t* src, const uint8_t* roi, Geom g, int3 lev, int thr,
                                                              int ccap, int ecap, int pad, uint8_t* gray, unsigned* ROI,
                                                              unsigned char* ws, unsigned char* lists, unsigned* clist,
                                                              unsigned* elist, unsigned* CAND, int* out) {
    __shared__ unsigned hist[256];
    __shared__ __align__(16) double ows[kOtsuWsBytes / 8];
    __shared__ int lv[kLevels], counters[4], otsu_last, otsu_t;
    const int tid = threadIdx.x, npix = g.w * g.h;
    for (int i = tid; i < g.h * g.gp; i += kThreads) {
        const int y = i / g.gp, x = i - y * g.gp;
        gray[i] = x < g.w ? src[y * g.w + x] : (uint8_t)pad;
    }
    for (int i = tid; i < g.nwords; i += kThreads) CAND[i] = 0;
    if (tid < 256) hist[tid] = 0;
    if (tid == 0) { lv[0] = lev.x; lv[1] = lev.y; lv[2] = lev.z; otsu_last = -1; }
    load_mask_bits(roi, g, ROI);
    cta_sync();
    for (int i = tid; i < npix; i += kThreads) atomicAdd(&hist[src[i]], 1u);
    cta_sync();
    RankWs rw = rank_ws_carve(ws, g, lists, (int)rank_plane_words(g.w, g.h), counters);
    const bool oside = rank_otsu_aside(g);
    PhaseTimerT<false> pt;
    if (warp_id() == 0) {
        int last;
        otsu_approx_warp(hist, npix, last);
        if (lane_id() == 0) *const_cast<volatile int*>(&otsu_last) = last;
        rank_tables(lv, thr, rw);
    } else if (oside && warp_id() == kOtsuWarp) {
        const int t = otsu_scan(hist, npix, ows, &otsu_last, pt);
        if (lane_id() == 0) otsu_t = t;
    } else {
        rank_cmm(gray, g, rw, 1, oside ? kWarps - 1 : kWarps, 0, rank_cmm_split(g, oside));
    }
    if (oside) { if (warp_id() != kOtsuWarp) workers_sync(kThreads - 32); } else cta_sync();
    rank_cells(gray, g, rw, lv, hist, npix, ows, &otsu_last, &otsu_t, oside, pt);
    rank_finish(gray, g, rw, lv, thr, ROI, CAND, clist, ccap, elist, ecap, pt);
    if (tid == 0) { out[0] = counters[1]; out[1] = counters[0]; out[2] = otsu_t; }
}

extern "C" int vi_debug_rank_residual(vi_ctx* c, const uint8_t* d_gray, const uint8_t* d_roi, int w, int h, const int* levels,
                                      int thr, int ccap, int ecap, int pad, uint32_t* d_cand, int* counts) {
    if (!c || !d_gray || !d_roi || !levels || !d_cand || !counts) return fail(VI_ERR_ARG, "vi_debug_rank_residual: null");
    if (w < 1 || h < 1 || w > kMaxUnitW || h > kMaxUnitH || (long long)w * h > kMaxUnitPixels)
        return fail(VI_ERR_ARG, "vi_debug_rank_residual: %dx%d is outside the unit bound", w, h);
    if (levels[0] < 0 || levels[0] > levels[1] || levels[1] > levels[2] || levels[2] > 255)
        return fail(VI_ERR_ARG, "vi_debug_rank_residual: levels must be sorted and in 0..255");
    if (thr < 0 || thr > 255 || pad < 0 || pad > 255) return fail(VI_ERR_ARG, "vi_debug_rank_residual: thr and pad must be in 0..255");
    if (ccap < 0 || ccap > kDirtyListCap || ecap < 0 || ecap > kExactListCap)
        return fail(VI_ERR_ARG, "vi_debug_rank_residual: ccap in 0..%d, ecap in 0..%d", kDirtyListCap, kExactListCap);
    VI_DEVICE(c);
    const Geom g = make_geom(w, h);
    const long long gray_b = ((long long)g.gp * h + 255) & ~255ll, roi_b = ((long long)g.nwords * 4 + 255) & ~255ll;
    const long long ws_b = (rank_ws_bytes(w, h) + 255) & ~255ll, plane_b = (rank_plane_words(w, h) * 4 + 255) & ~255ll;
    const long long total = gray_b + roi_b + ws_b + plane_b + 4ll * (kDirtyListCap + kExactListCap) + 16;
    unsigned char* d = nullptr;
    CU(cudaMalloc(&d, total));
    unsigned char* p = d;
    uint8_t* gray = p; p += gray_b;
    unsigned* roi = reinterpret_cast<unsigned*>(p); p += roi_b;
    unsigned char* ws = p; p += ws_b;
    unsigned char* lists = p; p += plane_b;
    unsigned* clist = reinterpret_cast<unsigned*>(p); p += 4ll * kDirtyListCap;
    unsigned* elist = reinterpret_cast<unsigned*>(p); p += 4ll * kExactListCap;
    int* d_out = reinterpret_cast<int*>(p);
    rank_debug_kernel<<<1, kThreads>>>(d_gray, d_roi, g, make_int3(levels[0], levels[1], levels[2]), thr, ccap, ecap, pad, gray, roi,
                                       ws, lists, clist, elist, d_cand, d_out);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpy(counts, d_out, 3 * sizeof(int), cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (e != cudaSuccess) return fail(VI_ERR_CUDA, "vi_debug_rank_residual: %s", cudaGetErrorString(e));
    return VI_OK;
}

extern "C" int vi_debug_check_word(vi_ctx* c, uint32_t* out) {
    if (!c || !out) return fail(VI_ERR_ARG, "vi_debug_check_word: null");
#ifdef VI_CHECKED
    VI_DEVICE(c);
    CU(cudaDeviceSynchronize());
    unsigned w = 0;
    CU(cudaMemcpyFromSymbol(&w, vi::g_vi_check_word, sizeof w));
    *out = w;
    return VI_OK;
#else
    *out = 0;
    return fail(VI_ERR_UNSUPPORTED, "vi_debug_check_word: this library was built without VI_CHECKED");
#endif
}

extern "C" int vi_debug_set_profile(vi_ctx* c, long long* d_cycles) {
    if (!c) return fail(VI_ERR_ARG, "ctx is null");
    c->prof = d_cycles;
    return VI_OK;
}

extern "C" int vi_set_seg_stats_output(vi_ctx* c, int64_t* d_stats) {
    if (!c) return fail(VI_ERR_ARG, "ctx is null");
    c->seg_stats = (long long*)d_stats;
    return VI_OK;
}

extern "C" int vi_set_defect_blob_output(vi_ctx* c, vi_defect_blob* d_blobs, int max_per_unit) {
    if (!c) return fail(VI_ERR_ARG, "ctx is null");
    if (d_blobs && (max_per_unit < 1 || max_per_unit > VI_MAX_BLOBS_PER_UNIT))
        return fail(VI_ERR_ARG, "vi_set_defect_blob_output: %d blobs per unit (1..%d)", max_per_unit, VI_MAX_BLOBS_PER_UNIT);
    c->blobs = d_blobs;
    c->blob_k = d_blobs ? max_per_unit : 0;
    return VI_OK;
}

// Merged [y0, y1) row intervals of the frame that some unit of the grid covers: the rows the host-buffer call uploads.
static std::vector<std::pair<int, int>> covered_rows(const GridState& gs) {
    std::vector<std::pair<int, int>> iv, rows;
    for (const int4& r : gs.rects) iv.emplace_back(r.y, r.y + r.w);
    std::sort(iv.begin(), iv.end());
    for (const auto& p : iv) {
        if (!rows.empty() && p.first <= rows.back().second) rows.back().second = std::max(rows.back().second, p.second);
        else rows.push_back(p);
    }
    return rows;
}

extern "C" int64_t vi_host_upload_bytes(vi_ctx* c, int n_images, int64_t row_pitch) {
    if (!c || row_pitch <= 0) return 0;
    long long rows = 0;
    for (const auto& iv : covered_rows(c->grid)) rows += iv.second - iv.first;
    return (int64_t)rows * row_pitch * n_images;
}

// ---------------------------------------------------------------------------
// multi-GPU: per-unit record tables in peer-mapped memory (CUDA IPC over NVLink / NVSwitch)
// ---------------------------------------------------------------------------
extern "C" int vi_peer_table_create(vi_ctx* c, int64_t n_records, void** d_table, uint8_t* handle64) {
    if (!c || !d_table || !handle64 || n_records <= 0) return fail(VI_ERR_ARG, "vi_peer_table_create: bad arguments");
    VI_DEVICE(c);
    void* p = nullptr;
    CU(cudaMalloc(&p, sizeof(vi_unit_record) * (size_t)n_records));          // a whole allocation: IPC handles name allocations
    CU(cudaMemset(p, 0, sizeof(vi_unit_record) * (size_t)n_records));
    CU(cudaDeviceSynchronize());
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); return fail(VI_ERR_CUDA, "cudaIpcGetMemHandle: %s", cudaGetErrorString(e)); }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    memcpy(handle64, &h, 64);
    *d_table = p;
    return VI_OK;
}

extern "C" int vi_peer_table_open(vi_ctx* c, const uint8_t* handle64, void** d_peer) {
    if (!c || !handle64 || !d_peer) return fail(VI_ERR_ARG, "vi_peer_table_open: bad arguments");
    VI_DEVICE(c);
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    CU(cudaIpcOpenMemHandle(d_peer, h, cudaIpcMemLazyEnablePeerAccess));
    return VI_OK;
}

extern "C" int vi_peer_table_close(vi_ctx* c, void* d_peer) {
    if (!c || !d_peer) return fail(VI_ERR_ARG, "vi_peer_table_close: bad arguments");
    VI_DEVICE(c);
    CU(cudaIpcCloseMemHandle(d_peer));
    return VI_OK;
}

extern "C" int vi_peer_table_destroy(vi_ctx* c, void* d_table) {
    if (!c || !d_table) return fail(VI_ERR_ARG, "vi_peer_table_destroy: bad arguments");
    VI_DEVICE(c);
    CU(cudaDeviceSynchronize());
    CU(cudaFree(d_table));
    return VI_OK;
}

extern "C" int vi_peer_table_read(vi_ctx* c, const void* d_table, int64_t n_records, vi_unit_record* h_out) {
    if (!c || !d_table || !h_out || n_records <= 0) return fail(VI_ERR_ARG, "vi_peer_table_read: bad arguments");
    VI_DEVICE(c);
    CU(cudaMemcpy(h_out, d_table, sizeof(vi_unit_record) * (size_t)n_records, cudaMemcpyDeviceToHost));
    return VI_OK;
}

extern "C" int vi_set_record_peers(vi_ctx* c, void* const* d_tables, int n, int image_mul, int image_add) {
    if (!c) return fail(VI_ERR_ARG, "ctx is null");
    if (n < 0 || n > kMaxPeers || (n > 0 && !d_tables)) return fail(VI_ERR_ARG, "vi_set_record_peers: %d tables (at most %d)", n, kMaxPeers);
    if (n > 0 && (image_mul <= 0 || image_add < 0)) return fail(VI_ERR_ARG, "vi_set_record_peers: image index map %d * k + %d", image_mul, image_add);
    for (int i = 0; i < kMaxPeers; ++i) c->peer_rec[i] = i < n ? (vi_unit_record*)d_tables[i] : nullptr;
    c->n_peers = n;
    c->image_mul = n > 0 ? image_mul : 1;
    c->image_add = n > 0 ? image_add : 0;
    return VI_OK;
}

extern "C" int vi_set_packed_mask_output(vi_ctx* c, uint32_t* d_seg_bits, uint32_t* d_def_bits) {
    if (!c) return fail(VI_ERR_ARG, "ctx is null");
    c->seg_bits = d_seg_bits; c->def_bits = d_def_bits;
    return VI_OK;
}

extern "C" int64_t vi_packed_mask_bytes(vi_ctx* c) { return c ? c->grid.unit_words * 4 : 0; }

extern "C" int vi_packed_mask_offsets(vi_ctx* c, int64_t* out) {
    if (!c || !out) return fail(VI_ERR_ARG, "vi_packed_mask_offsets: null");
    for (size_t i = 0; i < c->grid.woff.size(); ++i) out[i] = c->grid.woff[i] * 4;
    return VI_OK;
}

extern "C" int64_t vi_unit_pixels(vi_ctx* c) { return c ? c->grid.unit_px : 0; }

extern "C" int vi_unit_offsets(vi_ctx* c, int64_t* out) {
    if (!c || !out) return fail(VI_ERR_ARG, "vi_unit_offsets: null");
    for (size_t i = 0; i < c->grid.off.size(); ++i) out[i] = c->grid.off[i];
    return VI_OK;
}

// ---------------------------------------------------------------------------
// parameter normalisation -- the reference's rules, on the host
// ---------------------------------------------------------------------------
static void gaussian_taps_q8(int k, int* q) {
    // OpenCV's 8.8 fixed-point kernel for uint8 GaussianBlur(k, sigma=0) (SURVEY A.2)
    static const double small3[] = {0.25, 0.5, 0.25};
    static const double small5[] = {0.0625, 0.25, 0.375, 0.25, 0.0625};
    static const double small7[] = {0.03125, 0.109375, 0.21875, 0.28125, 0.21875, 0.109375, 0.03125};
    std::vector<double> kern(k);
    if (k == 1) kern[0] = 1.0;
    else if (k == 3) std::copy(small3, small3 + 3, kern.begin());
    else if (k == 5) std::copy(small5, small5 + 5, kern.begin());
    else if (k == 7) std::copy(small7, small7 + 7, kern.begin());
    else {
        double sigma = ((k - 1) * 0.5 - 1) * 0.3 + 0.8;
        double s2 = -0.5 / (sigma * sigma);
        double tot = 0;
        for (int i = 0; i < k; ++i) { double x = i - (k - 1) * 0.5; kern[i] = std::exp(s2 * x * x); tot += kern[i]; }
        double inv = 1.0 / tot;
        for (int i = 0; i < k; ++i) kern[i] *= inv;
    }
    double err = 0;
    int acc = 0;
    for (int i = 0; i < k / 2; ++i) {
        double adj = kern[i] * 256.0 + err;
        int v = (int)std::nearbyint(adj);      // cvRound: half to even
        err = adj - v;
        q[i] = q[k - 1 - i] = v;
        acc += v;
    }
    q[k / 2] = 256 - 2 * acc;
}

// cv2.getGaussianKernel(bs, 0, CV_32F): the float32 taps of adaptiveThreshold's Gaussian mean
// (hard-coded tables up to 9 taps in OpenCV 4.13, else exp(-x^2 / 2 sigma^2) normalised in double).
static void gaussian_taps_f32(int k, float* out) {
    static const double s3[] = {0.25, 0.5, 0.25};
    static const double s5[] = {0.0625, 0.25, 0.375, 0.25, 0.0625};
    static const double s7[] = {0.03125, 0.109375, 0.21875, 0.28125, 0.21875, 0.109375, 0.03125};
    static const double s9[] = {4.0 / 256, 13.0 / 256, 30.0 / 256, 51.0 / 256, 60.0 / 256, 51.0 / 256, 30.0 / 256, 13.0 / 256, 4.0 / 256};
    const double* small = k == 3 ? s3 : k == 5 ? s5 : k == 7 ? s7 : k == 9 ? s9 : nullptr;
    if (k == 1) { out[0] = 1.0f; return; }
    if (small) { for (int i = 0; i < k; ++i) out[i] = (float)small[i]; return; }
    std::vector<double> kern(k);
    const double sigma = ((k - 1) * 0.5 - 1) * 0.3 + 0.8;
    const double s2 = -0.5 / (sigma * sigma);
    double tot = 0;
    for (int i = 0; i < k; ++i) { const double x = i - (k - 1) * 0.5; kern[i] = std::exp(s2 * x * x); tot += kern[i]; }
    const double inv = 1.0 / tot;
    for (int i = 0; i < k; ++i) out[i] = (float)(kern[i] * inv);
}

extern "C" int vi_debug_adaptive_taps(int block_size, float* out) {
    if (!out || block_size < 1 || block_size > kMaxAdapt || block_size % 2 == 0) return fail(VI_ERR_ARG, "vi_debug_adaptive_taps: block size %d", block_size);
    gaussian_taps_f32(block_size, out);
    return VI_OK;
}

static void ellipse_spans(int k, signed char* lo, signed char* hi) {
    // cv2.getStructuringElement(MORPH_ELLIPSE,(k,k)) as per-row offset spans (SURVEY A.5)
    int r = k / 2, c = k / 2;
    double inv_r2 = r ? 1.0 / ((double)r * r) : 0.0;
    for (int i = 0; i < k; ++i) {
        int dy = i - r;
        int j1 = 0, j2 = 0;
        if (std::abs(dy) <= r) {
            int dx = (int)std::nearbyint(c * std::sqrt((r * r - dy * dy) * inv_r2));
            j1 = std::max(c - dx, 0);
            j2 = std::min(c + dx + 1, k);
        }
        lo[i] = (signed char)(j1 - c);
        hi[i] = (signed char)(j2 - 1 - c);
    }
}

static int fill_params(KArgs& a, const vi_params* p) {
    if (!p) return fail(VI_ERR_ARG, "params is null");
    a.p = *p;
    if (p->seg_method != 0 && p->seg_method != 1) return fail(VI_ERR_ARG, "seg_method %d (0 otsu, 1 adaptive)", p->seg_method);
    a.adapt_bs = 0;
    if (p->seg_method == 1) {
        const int bs = std::max(3, p->adapt_block | 1);                                                     // segmentation.py:84
        if (bs > kMaxAdapt) return fail(VI_ERR_ARG, "adapt_block %d: block wider than %d", p->adapt_block, kMaxAdapt);
        a.adapt_bs = bs;
        gaussian_taps_f32(bs, a.ataps);
    }
    if (p->defect_method != 0 && p->defect_method != 1) return fail(VI_ERR_ARG, "defect_method %d (0 threshold, 1 canny)", p->defect_method);
    if (p->median_ksize != 21) return fail(VI_ERR_UNSUPPORTED, "median_ksize must be 21 (indexing_ui.py:1522)");
    if (p->threshold < 0 || p->threshold > 255) return fail(VI_ERR_ARG, "threshold %d outside 0..255", p->threshold);
    if (p->erode_px < 0 || p->min_area < 0) return fail(VI_ERR_ARG, "erode_px / min_area must be >= 0");
    a.canny_low = std::max(1, p->threshold / 2);                                                          // indexing_ui.py:1537
    a.canny_high = std::max(2, p->threshold);
    if (a.canny_low > a.canny_high) std::swap(a.canny_low, a.canny_high);
    int k = 0;
    if (p->gaussian_blur > 0) k = (p->gaussian_blur % 2 == 1) ? p->gaussian_blur : p->gaussian_blur + 1;   // segmentation.py:79
    if (k == 1) k = 0;                                     // a 1x1 Gaussian is the identity
    if (k > kMaxTaps) return fail(VI_ERR_ARG, "gaussian_blur %d: kernel wider than %d", p->gaussian_blur, kMaxTaps);
    a.blur_k = k;
    memset(a.taps, 0, sizeof a.taps);
    if (k >= 3) gaussian_taps_q8(k, a.taps);
    int mk = p->morph_kernel > 0 ? std::max(1, p->morph_kernel) : 0;                                   // segmentation.py:91-92
    if (mk == 1) mk = 0;                                   // a 1x1 element is the identity
    if (mk > kMaxSE) return fail(VI_ERR_ARG, "morph_kernel %d: element wider than %d", p->morph_kernel, kMaxSE);
    a.se_k = mk;
    memset(a.se_lo, 0, sizeof a.se_lo);
    memset(a.se_hi, 0, sizeof a.se_hi);
    if (mk > 0 && mk != 3) ellipse_spans(mk, a.se_lo, a.se_hi);
    return VI_OK;
}

// The frames as a tensor map for the kernel's asynchronous crop gather (vi_pipeline.cuh: gather_issue_tma).  The
// encoder is a driver entry point; it is looked up through the runtime so the library keeps linking against cudart
// only.  Returns false (a.tma_ok = 0: the kernel falls back to one bulk copy per crop row) when anything does not fit.
typedef CUresult (*PFN_tmap_encode)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static PFN_tmap_encode tmap_encoder() {
    static PFN_tmap_encode fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (PFN_tmap_encode)p;
        else
            cudaGetLastError();
    }
    return fn;
}

static bool make_frame_tensor(KArgs& a, const GridState& gs) {
    a.tma_ok = 0;
    PFN_tmap_encode enc = tmap_encoder();
    if (!enc) return false;
    // the aligned span of a crop: up to 15 bytes of phase in front; tiles of equal width (a multiple of 16) and whole
    // boxes of rows (a multiple of 8 high: every box starts 128-byte aligned); the fewest column boxes that fit the staging area
    const int w16 = (gs.ext.wmax + 15 + 15) & ~15;
    const int nrb = (gs.ext.hmax + 255) / 256;
    const int bh = (((gs.ext.hmax + nrb - 1) / nrb) + 7) & ~7;
    if (bh > 256) return false;
    int ncb = 0, bw = 0, tile_bytes = 0;
    for (int n = (w16 + 255) / 256; n <= 4; ++n) {
        const int b = (((w16 + n - 1) / n) + 15) & ~15;
        const int t = (b * bh * nrb + 127) & ~127;
        if (b <= 256 && (long long)n * t <= a.layout.stage_bytes) { ncb = n; bw = b; tile_bytes = t; break; }
    }
    if (!ncb) return false;
    if ((a.row_pitch & 15) || (a.n_images > 1 && (a.image_stride & 15)) || (reinterpret_cast<uintptr_t>(a.frames) & 15)) return false;
    const long long istride = a.n_images > 1 ? a.image_stride : a.row_pitch * (long long)a.H;
    cuuint64_t gdim[3] = {(cuuint64_t)a.W, (cuuint64_t)a.H, (cuuint64_t)a.n_images};
    cuuint64_t gstr[2] = {(cuuint64_t)a.row_pitch, (cuuint64_t)istride};
    cuuint32_t box[3] = {(cuuint32_t)bw, (cuuint32_t)bh, 1u};
    cuuint32_t estr[3] = {1u, 1u, 1u};
    if (enc(&a.tmap, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<uint8_t*>(a.frames), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
        return false;
    a.tma_bw = bw; a.tma_bh = bh; a.tma_ncb = ncb; a.tma_nrb = nrb; a.tma_tile_bytes = tile_bytes;
    a.tma_ok = 1;
    return true;
}

constexpr long long kScratchBudget = 24ll << 30;            // per-CTA scratch + arenas of the large-unit path stay below this

// `slot` selects a private copy of the per-CTA scratch so launches on the internal
// streams never share it.
static int launch_units(vi_ctx* c, KArgs& a, const GridState& gs, cudaStream_t stream, int slot = 0) {
    const long long n_total = (long long)a.n_images * a.n_units;
    if (n_total <= 0) return VI_OK;
    if (n_total > 0x7fffffffll) return fail(VI_ERR_ARG, "too many units in one call");
    int rc;
    UnitLayout& L = a.layout;
    unit_layout(gs.ext, c->smem_optin, c->smem_static, a.p.seg_method == 1, a.blobs ? a.blob_k : 0, &L);   // (checked by set_grid_state)
    const long long stride = L.scratch_bytes, astride = L.arena_bytes;
    // CTAs per slot: one per SM; fewer when the units are so large that their scratch would not fit the budget
    int bps = c->sm_count;
    if ((stride + astride) * kHostSlots * bps > kScratchBudget)
        bps = (int)std::max<long long>(1, kScratchBudget / ((stride + astride) * kHostSlots));
    const int nblocks = (int)std::min<long long>(n_total, bps);
    if ((rc = c->scratch.ensure((size_t)stride * kHostSlots * bps))) return rc;
    if (L.arena && (rc = c->arena.ensure((size_t)astride * kHostSlots * bps))) return rc;
    a.scratch = (uint8_t*)c->scratch.p + (size_t)slot * bps * stride;
    a.arena = L.arena ? (uint8_t*)c->arena.p + (size_t)slot * bps * astride : nullptr;
    if (c->smem_set < L.total) {
        const int lim = c->smem_optin - c->smem_static;
        CU(cudaFuncSetAttribute(vi_unit_kernel<false, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
        CU(cudaFuncSetAttribute(vi_unit_kernel<false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
#ifndef VI_CHECKED
        CU(cudaFuncSetAttribute(vi_unit_kernel<true, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
        CU(cudaFuncSetAttribute(vi_seg_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
#endif
        CU(cudaFuncSetAttribute(vi_seg_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
        CU(cudaFuncSetAttribute(vi_unit_kernel<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
        c->smem_set = lim;
    }
    if (L.total > c->smem_set) return fail(VI_ERR_TOO_LARGE, "shared-memory plan %d > %d", L.total, c->smem_set);
    if (L.arena) {
        // units beyond one SM's shared memory (DESIGN.md section 2): same phases over the CTA's global arena
        a.prof = nullptr;
        vi_unit_kernel<false, false, true><<<nblocks, kThreads, L.total, stream>>>(a);
        CU(cudaGetLastError());
        return VI_OK;
    }
    // The default configuration has its own instantiations (vi_unit.cuh: SPEC), one per batch mode.
    const bool aligned = (a.row_pitch & 15) == 0 && (reinterpret_cast<uintptr_t>(a.frames) & 15) == 0 && (a.image_stride & 15) == 0;
    bool spec = a.mode == MODE_FULL && a.blur_k == 3 && a.se_k == 3 && a.p.seg_method == 0 && a.p.defect_method == 0 &&
                !a.labels_out && !a.seg_stats && !a.seg_bits && !a.def_bits && !a.aux_mask && !a.stats_out && aligned &&
                lattice_fits(gs.ext.wmax, gs.ext.hmax, L) && hist_round_fits(L.n_hist);
    const bool seg = a.mode == MODE_SEG_ONLY && a.blur_k == 3 && a.se_k == 3 && a.p.seg_method == 0 && !a.labels_out &&
                     !a.def_bits && !a.aux_mask && !a.stats_out && aligned && hist_round_fits(L.n_hist);
    if (spec || seg) make_frame_tensor(a, gs);
#ifndef VI_CHECKED
    if (a.prof && spec) vi_unit_kernel<true, true, false><<<nblocks, kThreads, L.total, stream>>>(a);   // diagnostics build: phase timers
    else if (a.prof && seg) vi_seg_kernel<true><<<nblocks, kThreads, L.total, stream>>>(a);
    else
#endif
    if (spec) vi_unit_kernel<false, true, false><<<nblocks, kThreads, L.total, stream>>>(a);
    else if (seg) vi_seg_kernel<false><<<nblocks, kThreads, L.total, stream>>>(a);
    else { a.prof = nullptr; vi_unit_kernel<false, false, false><<<nblocks, kThreads, L.total, stream>>>(a); }
    CU(cudaGetLastError());
    return VI_OK;
}

static int check_frames(const GridState& gs, int n_images, int W, int H, int64_t row_pitch, int64_t image_stride) {
    if (n_images <= 0 || W <= 0 || H <= 0) return fail(VI_ERR_ARG, "frames: n_images=%d W=%d H=%d", n_images, W, H);
    if (row_pitch < W || (n_images > 1 && image_stride < row_pitch * (int64_t)H))
        return fail(VI_ERR_ARG, "frames: pitch/stride smaller than the image");
    for (size_t i = 0; i < gs.rects.size(); ++i) {
        const int4& r = gs.rects[i];
        // the reference pads (QImage.copy) or clips (QPixmap.copy) out-of-frame rects, inconsistently; reject them
        if (r.x + r.z > W || r.y + r.w > H) return fail(VI_ERR_ARG, "grid: rect %zu (%d,%d,%d,%d) leaves the %dx%d frame", i, r.x, r.y, r.z, r.w, W, H);
    }
    return VI_OK;
}

static void base_args(vi_ctx* c, KArgs& a, const GridState& gs) {
    memset(&a, 0, sizeof a);
    a.rects = (const int4*)gs.d_rects.p;
    a.n_units = (int)gs.rects.size();
    a.unit_off = (const long long*)gs.d_off.p;
    a.unit_px = gs.unit_px;
    a.unit_woff = (const long long*)gs.d_woff.p;
    a.unit_words = gs.unit_words;
    a.image_mul = 1;
}

// What a batch over the user grid launches with besides its outputs: the frames, the context's tables (exclusions,
// reference centroids) and its phase-profile buffer.
static void batch_args(vi_ctx* c, KArgs& a, const uint8_t* frames, int n_images, int W, int H, int64_t row_pitch,
                       int64_t image_stride) {
    a.frames = frames; a.n_images = n_images; a.W = W; a.H = H; a.row_pitch = row_pitch; a.image_stride = image_stride;
    a.excl = (const vi_excl*)c->d_excl.p; a.n_excl = (int)c->excl.size();
    a.refc = c->has_refc ? (const double*)c->d_refc.p : nullptr;
    a.is_reference = c->is_reference;
    a.mode = MODE_FULL;
    a.prof = c->prof;
}

// The device-buffer batch call in `mode`: MODE_FULL (vi_inspect_batch) or MODE_SEG_ONLY (vi_segment_batch, which
// takes no defect, label or blob outputs).
static int device_batch(vi_ctx* c, int mode, const char* name, const uint8_t* d_frames, int n_images, int W, int H,
                        int64_t row_pitch, int64_t image_stride, const vi_params* params, uint8_t* d_seg, uint8_t* d_def,
                        int32_t* d_labels, vi_unit_record* d_rec, void* stream) {
    if (!c) return fail(VI_ERR_ARG, "ctx is null");
    if (c->grid.rects.empty()) return fail(VI_ERR_ARG, "%s: no grid set", name);
    if (!d_frames || !d_rec) return fail(VI_ERR_ARG, "%s: frames / records pointer is null", name);
    if (n_images == 1 && image_stride < row_pitch * (int64_t)H) image_stride = row_pitch * (int64_t)H;
    VI_DEVICE(c);
    int rc;
    if ((rc = check_frames(c->grid, n_images, W, H, row_pitch, image_stride))) return rc;
    KArgs a;
    base_args(c, a, c->grid);
    if ((rc = fill_params(a, params))) return rc;
    batch_args(c, a, d_frames, n_images, W, H, row_pitch, image_stride);
    a.mode = mode;
    a.seg_out = d_seg; a.rec = d_rec;
    a.seg_stats = c->seg_stats;
    a.seg_bits = c->seg_bits;
    if (mode == MODE_FULL) {
        a.def_out = d_def; a.labels_out = d_labels; a.def_bits = c->def_bits;
        a.blobs = c->blobs; a.blob_k = c->blob_k;
    }
    a.n_peers = c->n_peers; a.image_mul = c->image_mul; a.image_base = c->image_add;
    for (int i = 0; i < c->n_peers; ++i) a.peer_rec[i] = c->peer_rec[i];
    if ((rc = wait_busy_stream(c, (cudaStream_t)stream))) return rc;     // an earlier batch on another stream shares the scratch
    if ((rc = launch_units(c, a, c->grid, (cudaStream_t)stream))) return rc;
    return mark_busy(c, (cudaStream_t)stream);
}

extern "C" int vi_inspect_batch(vi_ctx* c, const uint8_t* d_frames, int n_images, int W, int H, int64_t row_pitch,
                                int64_t image_stride, const vi_params* params, uint8_t* d_seg, uint8_t* d_def,
                                int32_t* d_labels, vi_unit_record* d_rec, void* stream) {
    return device_batch(c, MODE_FULL, "vi_inspect_batch", d_frames, n_images, W, H, row_pitch, image_stride, params, d_seg,
                        d_def, d_labels, d_rec, stream);
}

extern "C" int vi_segment_batch(vi_ctx* c, const uint8_t* d_frames, int n_images, int W, int H, int64_t row_pitch,
                                int64_t image_stride, const vi_params* params, uint8_t* d_seg, vi_unit_record* d_rec,
                                void* stream) {
    return device_batch(c, MODE_SEG_ONLY, "vi_segment_batch", d_frames, n_images, W, H, row_pitch, image_stride, params,
                        d_seg, nullptr, nullptr, d_rec, stream);
}

// Host-buffer batch call.  mask_format: VI_MASKS_BYTES (0/255 bytes, what the reference's pixmaps hold),
// VI_MASKS_PACKED (1 bit per pixel, rows of 32-bit words, PNG bit order) or VI_MASKS_NONE (records only: all that
// run_inspection needs, indexing_ui.py:1686-1706).  mode: MODE_FULL, or MODE_SEG_ONLY (vi_segment_batch_host: no
// defect masks, no blob table).
static int host_batch(vi_ctx* c, int mode, const uint8_t* h_frames, int n_images, int W, int H, int64_t row_pitch,
                      int64_t image_stride, const vi_params* params, int mask_format, void* h_seg, void* h_def,
                      vi_unit_record* h_rec, vi_defect_blob* h_blobs = nullptr, int blob_k = 0) {
    const char* name = mode == MODE_SEG_ONLY ? "vi_segment_batch_host" : "vi_inspect_batch_host";
    if (!c) return fail(VI_ERR_ARG, "ctx is null");
    if (c->grid.rects.empty()) return fail(VI_ERR_ARG, "%s: no grid set", name);
    if (!h_frames || !h_rec) return fail(VI_ERR_ARG, "%s: frames / records pointer is null", name);
    if (mask_format < VI_MASKS_BYTES || mask_format > VI_MASKS_NONE) return fail(VI_ERR_ARG, "mask_format %d", mask_format);
    if (h_blobs && (blob_k < 1 || blob_k > VI_MAX_BLOBS_PER_UNIT))
        return fail(VI_ERR_ARG, "vi_inspect_batch_host_blobs: %d blobs per unit (1..%d)", blob_k, VI_MAX_BLOBS_PER_UNIT);
    VI_DEVICE(c);
    int rc;
    if (n_images == 1 && image_stride < row_pitch * (int64_t)H) image_stride = row_pitch * (int64_t)H;   // one frame: the stride is moot
    if ((rc = check_frames(c->grid, n_images, W, H, row_pitch, image_stride))) return rc;
    if ((rc = wait_busy_host(c))) return rc;
    KArgs a0;
    base_args(c, a0, c->grid);
    if ((rc = fill_params(a0, params))) return rc;                     // validated before anything is in flight
    const int n_units = (int)c->grid.rects.size();
    const long long upx = c->grid.unit_px;
    const long long ubytes = mask_format == VI_MASKS_BYTES ? upx : mask_format == VI_MASKS_PACKED ? c->grid.unit_words * 4 : 0;
    if (mask_format == VI_MASKS_NONE) { h_seg = nullptr; h_def = nullptr; }
    if (mode == MODE_SEG_ONLY) { h_def = nullptr; h_blobs = nullptr; }
    // Chunks of about two units per SM, kHostSlots of them in flight: the call is bound by the host link (frames up,
    // masks down), so all that matters is that the copy engines never idle.  VI_HOST_CHUNK overrides (images per chunk).
    int chunk = std::max(1, (2 * c->sm_count + n_units - 1) / n_units);
    if (const char* e = getenv("VI_HOST_CHUNK")) { int v = atoi(e); if (v > 0) chunk = v; }
    chunk = std::min(chunk, n_images);
    const size_t frame_bytes = (size_t)image_stride;
    for (int b = 0; b < kHostSlots; ++b) {
        if ((rc = c->hb_frames[b].ensure(frame_bytes * chunk))) return rc;
        if (h_seg && (rc = c->hb_seg[b].ensure((size_t)ubytes * chunk))) return rc;
        if (h_def && (rc = c->hb_def[b].ensure((size_t)ubytes * chunk))) return rc;
        if ((rc = c->hb_rec[b].ensure(sizeof(vi_unit_record) * (size_t)n_units * chunk))) return rc;
        if (h_blobs && (rc = c->hb_blob[b].ensure(sizeof(vi_defect_blob) * (size_t)n_units * chunk * blob_k))) return rc;
    }
    // Upload: one strided copy per covered row interval into the slot's staging buffer (the copy engine moves whole
    // frame rows at the link rate).
    const std::vector<std::pair<int, int>> rows = covered_rows(c->grid);
    auto run_chunks = [&]() -> int {
        int slot = 0;
        for (int i0 = 0; i0 < n_images; i0 += chunk, slot = (slot + 1) % kHostSlots) {
            const int n = std::min(chunk, n_images - i0);
            cudaStream_t st = c->streams[slot];
            // the slot's previous chunk (kHostSlots iterations ago) is ordered before this one on the same stream
            for (const auto& iv : rows) {
                const size_t off = (size_t)iv.first * row_pitch, bytes = (size_t)(iv.second - iv.first) * row_pitch;
                CU(cudaMemcpy2DAsync((uint8_t*)c->hb_frames[slot].p + off, frame_bytes, h_frames + (size_t)i0 * image_stride + off,
                                     (size_t)image_stride, bytes, n, cudaMemcpyHostToDevice, st));
            }
            KArgs a = a0;
            batch_args(c, a, (const uint8_t*)c->hb_frames[slot].p, n, W, H, row_pitch, image_stride);
            a.mode = mode;
            a.image_base = i0;
            if (mask_format == VI_MASKS_BYTES) {
                a.seg_out = h_seg ? (uint8_t*)c->hb_seg[slot].p : nullptr; a.def_out = h_def ? (uint8_t*)c->hb_def[slot].p : nullptr;
            } else if (mask_format == VI_MASKS_PACKED) {
                a.seg_bits = h_seg ? (uint32_t*)c->hb_seg[slot].p : nullptr; a.def_bits = h_def ? (uint32_t*)c->hb_def[slot].p : nullptr;
            }
            a.rec = (vi_unit_record*)c->hb_rec[slot].p;
            if (h_blobs) { a.blobs = (vi_defect_blob*)c->hb_blob[slot].p; a.blob_k = blob_k; }
            int r2;
            if ((r2 = launch_units(c, a, c->grid, st, slot))) return r2;
            if (h_seg) CU(cudaMemcpyAsync((uint8_t*)h_seg + (size_t)i0 * ubytes, c->hb_seg[slot].p, (size_t)ubytes * n, cudaMemcpyDeviceToHost, st));
            if (h_def) CU(cudaMemcpyAsync((uint8_t*)h_def + (size_t)i0 * ubytes, c->hb_def[slot].p, (size_t)ubytes * n, cudaMemcpyDeviceToHost, st));
            CU(cudaMemcpyAsync(h_rec + (size_t)i0 * n_units, c->hb_rec[slot].p, sizeof(vi_unit_record) * (size_t)n_units * n,
                               cudaMemcpyDeviceToHost, st));
            // the whole slot table: entries past min(n_kept, blob_k) are unspecified
            if (h_blobs)
                CU(cudaMemcpyAsync(h_blobs + (size_t)i0 * n_units * blob_k, c->hb_blob[slot].p,
                                   sizeof(vi_defect_blob) * (size_t)n_units * n * blob_k, cudaMemcpyDeviceToHost, st));
        }
        return VI_OK;
    };
    rc = run_chunks();
    // also on failure: nothing may still be writing into the caller's buffers when this returns
    for (int b = 0; b < kHostSlots; ++b) {
        cudaError_t e = cudaStreamSynchronize(c->streams[b]);
        if (e != cudaSuccess && rc == VI_OK) rc = fail(VI_ERR_CUDA, "cudaStreamSynchronize: %s", cudaGetErrorString(e));
    }
    return rc;
}

extern "C" int vi_inspect_batch_host(vi_ctx* c, const uint8_t* h_frames, int n_images, int W, int H, int64_t row_pitch,
                                     int64_t image_stride, const vi_params* params, uint8_t* h_seg, uint8_t* h_def,
                                     vi_unit_record* h_rec) {
    return host_batch(c, MODE_FULL, h_frames, n_images, W, H, row_pitch, image_stride, params, VI_MASKS_BYTES, h_seg, h_def, h_rec);
}

extern "C" int vi_inspect_batch_host_fmt(vi_ctx* c, const uint8_t* h_frames, int n_images, int W, int H, int64_t row_pitch,
                                         int64_t image_stride, const vi_params* params, int mask_format, void* h_seg,
                                         void* h_def, vi_unit_record* h_rec) {
    return host_batch(c, MODE_FULL, h_frames, n_images, W, H, row_pitch, image_stride, params, mask_format, h_seg, h_def, h_rec);
}

extern "C" int vi_inspect_batch_host_blobs(vi_ctx* c, const uint8_t* h_frames, int n_images, int W, int H, int64_t row_pitch,
                                           int64_t image_stride, const vi_params* params, int mask_format, void* h_seg,
                                           void* h_def, vi_unit_record* h_rec, vi_defect_blob* h_blobs, int max_per_unit) {
    return host_batch(c, MODE_FULL, h_frames, n_images, W, H, row_pitch, image_stride, params, mask_format, h_seg, h_def, h_rec,
                      h_blobs, max_per_unit);
}

extern "C" int vi_segment_batch_host(vi_ctx* c, const uint8_t* h_frames, int n_images, int W, int H, int64_t row_pitch,
                                     int64_t image_stride, const vi_params* params, int mask_format, void* h_seg,
                                     vi_unit_record* h_rec) {
    return host_batch(c, MODE_SEG_ONLY, h_frames, n_images, W, H, row_pitch, image_stride, params, mask_format, h_seg, nullptr,
                      h_rec);
}

// ---------------------------------------------------------------------------
// compat entry points: one unit = the whole (h, w) array, host pointers
// ---------------------------------------------------------------------------
static int compat_run(vi_ctx* c, int mode, const uint8_t* gray, const uint8_t* aux, int h, int w, const vi_params* params,
                      int erode_r, uint8_t* out_seg, uint8_t* out_def, int32_t* out_lab, vi_unit_record* out_rec,
                      long long* out_stats /*[8]*/) {
    if (!c) return fail(VI_ERR_ARG, "ctx is null");
    if (h <= 0 || w <= 0) return fail(VI_ERR_ARG, "array is %dx%d", h, w);
    VI_DEVICE(c);
    int32_t rect[4] = {0, 0, w, h};
    int rc;
    if ((rc = wait_busy_host(c))) return rc;
    cudaStream_t st = c->streams[0];
    if ((rc = set_grid_state(c, c->one, rect, 1, st))) return rc;
    const size_t px = (size_t)w * h;
    KArgs a;
    base_args(c, a, c->one);
    vi_params dflt;
    vi_params_default(&dflt);
    if ((rc = fill_params(a, params ? params : &dflt))) return rc;
    if ((rc = c->st_in.ensure(px + 16)) || (rc = c->st_aux.ensure(px + 16)) || (rc = c->st_out.ensure(px + 16)) ||
        (rc = c->st_out2.ensure(px + 16)) || (rc = c->st_rec.ensure(sizeof(vi_unit_record))) ||
        (rc = c->st_stats.ensure(64)) || (rc = c->st_lab.ensure(px * 4 + 16)))
        return rc;
    if (gray) CU(cudaMemcpyAsync(c->st_in.p, gray, px, cudaMemcpyHostToDevice, st));
    if (aux) CU(cudaMemcpyAsync(c->st_aux.p, aux, px, cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(c->st_rec.p, 0, sizeof(vi_unit_record), st));
    CU(cudaMemsetAsync(c->st_stats.p, 0, 64, st));
    a.frames = (const uint8_t*)c->st_in.p; a.n_images = 1; a.W = w; a.H = h; a.row_pitch = w; a.image_stride = (long long)px;
    a.aux_mask = (const uint8_t*)c->st_aux.p;
    a.seg_out = (uint8_t*)c->st_out.p; a.def_out = (uint8_t*)c->st_out2.p;
    a.labels_out = out_lab ? (int32_t*)c->st_lab.p : nullptr;
    a.rec = (vi_unit_record*)c->st_rec.p;
    a.stats_out = (long long*)c->st_stats.p;
    a.mode = mode;
    a.erode_r = erode_r;
    if ((rc = launch_units(c, a, c->one, st))) return rc;
    if (out_seg) CU(cudaMemcpyAsync(out_seg, c->st_out.p, px, cudaMemcpyDeviceToHost, st));
    if (out_def) CU(cudaMemcpyAsync(out_def, c->st_out2.p, px, cudaMemcpyDeviceToHost, st));
    if (out_lab) CU(cudaMemcpyAsync(out_lab, c->st_lab.p, px * 4, cudaMemcpyDeviceToHost, st));
    if (out_rec) CU(cudaMemcpyAsync(out_rec, c->st_rec.p, sizeof(vi_unit_record), cudaMemcpyDeviceToHost, st));
    if (out_stats) CU(cudaMemcpyAsync(out_stats, c->st_stats.p, 64, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return VI_OK;
}

extern "C" int vi_segment_cell(vi_ctx* c, const uint8_t* gray, int h, int w, const vi_params* params, uint8_t* out_mask,
                               int32_t* out_otsu_t) {
    if (!gray || !out_mask) return fail(VI_ERR_ARG, "vi_segment_cell: null pointer");
    vi_unit_record rec;
    int rc = compat_run(c, MODE_SEG_ONLY, gray, nullptr, h, w, params, 0, out_mask, nullptr, nullptr, &rec, nullptr);
    if (rc == VI_OK && out_otsu_t) *out_otsu_t = rec.otsu_t;
    return rc;
}

extern "C" int vi_fill_internal_holes(vi_ctx* c, const uint8_t* mask, int h, int w, uint8_t* out_mask) {
    if (!mask || !out_mask) return fail(VI_ERR_ARG, "vi_fill_internal_holes: null pointer");
    return compat_run(c, MODE_FILL, nullptr, mask, h, w, nullptr, 0, out_mask, nullptr, nullptr, nullptr, nullptr);
}

extern "C" int vi_mask_stats(vi_ctx* c, const uint8_t* mask, int h, int w, int64_t* area, int64_t* sum_x, int64_t* sum_y) {
    if (!mask) return fail(VI_ERR_ARG, "vi_mask_stats: null pointer");
    long long st[8];
    int rc = compat_run(c, MODE_STATS, nullptr, mask, h, w, nullptr, 0, nullptr, nullptr, nullptr, nullptr, st);
    if (rc) return rc;
    if (area) *area = st[0];
    if (sum_x) *sum_x = st[1];
    if (sum_y) *sum_y = st[2];
    return VI_OK;
}

extern "C" int vi_erode_square(vi_ctx* c, const uint8_t* mask, int h, int w, int r, uint8_t* out_mask) {
    if (!mask || !out_mask) return fail(VI_ERR_ARG, "vi_erode_square: null pointer");
    if (r < 0) return fail(VI_ERR_ARG, "vi_erode_square: r = %d", r);
    return compat_run(c, MODE_ERODE, nullptr, mask, h, w, nullptr, r, out_mask, nullptr, nullptr, nullptr, nullptr);
}

extern "C" int vi_label_components(vi_ctx* c, const uint8_t* mask, int h, int w, int32_t* out_labels, int32_t* n_labels,
                                   int32_t* best_label, int64_t* best_area, int64_t* best_sum_x, int64_t* best_sum_y) {
    if (!mask) return fail(VI_ERR_ARG, "vi_label_components: null pointer");
    long long st[8];
    int rc = compat_run(c, MODE_LABEL, nullptr, mask, h, w, nullptr, 0, nullptr, nullptr, out_labels, nullptr, st);
    if (rc) return rc;
    if (n_labels) *n_labels = (int32_t)st[0];
    if (best_label) *best_label = (int32_t)st[1];
    if (best_area) *best_area = st[2];
    if (best_sum_x) *best_sum_x = st[3];
    if (best_sum_y) *best_sum_y = st[4];
    return VI_OK;
}

extern "C" int vi_detect_defects(vi_ctx* c, const uint8_t* gray, const uint8_t* seg_mask, int h, int w,
                                 const vi_params* params, uint8_t* out_mask, int32_t* found, vi_unit_record* out_rec) {
    if (!gray || !seg_mask || !out_mask) return fail(VI_ERR_ARG, "vi_detect_defects: null pointer");
    vi_unit_record rec;
    int rc = compat_run(c, MODE_DETECT, gray, seg_mask, h, w, params, 0, nullptr, out_mask, nullptr, &rec, nullptr);
    if (rc) return rc;
    if (found) *found = rec.n_kept > 0 ? 1 : 0;
    if (out_rec) *out_rec = rec;
    return VI_OK;
}

// ---------------------------------------------------------------------------
// frame ingest (device pointers, asynchronous on `stream`)
// ---------------------------------------------------------------------------
static int ingest_common(vi_ctx* c, int fmt, const void* d_src, int n_images, int W, int H, int64_t src_pitch,
                         int64_t src_stride, uint8_t* d_dst, int64_t dst_pitch, int64_t dst_stride, void* stream) {
    if (!c) return fail(VI_ERR_ARG, "ctx is null");
    if (!d_src || !d_dst) return fail(VI_ERR_ARG, "ingest: null pointer");
    const int bpp = fmt == 0 ? 4 : 2;
    if (n_images <= 0 || W <= 0 || H <= 0) return fail(VI_ERR_ARG, "ingest: n_images=%d W=%d H=%d", n_images, W, H);
    if (src_pitch < (int64_t)W * bpp || dst_pitch < W) return fail(VI_ERR_ARG, "ingest: pitch smaller than a row");
    if (n_images > 1 && (src_stride < src_pitch * H || dst_stride < dst_pitch * H)) return fail(VI_ERR_ARG, "ingest: stride smaller than an image");
    VI_DEVICE(c);
    cudaStream_t st = (cudaStream_t)stream;
    const uint8_t* src = (const uint8_t*)d_src;
    const bool aligned = ((uintptr_t)src % 16 == 0) && ((uintptr_t)d_dst % 16 == 0) && src_pitch % 16 == 0 && src_stride % 16 == 0 &&
                         dst_pitch % 16 == 0 && dst_stride % 16 == 0 && W % 16 == 0;
    const int blocks = c->sm_count * 8;                 // 8 CTAs of 256 threads per SM: a full complement of warps
    if (aligned) {
        const long long n_items = (long long)n_images * H * (W / 16);
        if (fmt == 0) ingest_argb32_v16<<<blocks, kIngestThreads, 0, st>>>(src, src_pitch, src_stride, d_dst, dst_pitch, dst_stride, W, H, n_items);
        else ingest_gray16_v16<<<blocks, kIngestThreads, 0, st>>>(src, src_pitch, src_stride, d_dst, dst_pitch, dst_stride, W, H, n_items);
    } else {
        const long long n_px = (long long)n_images * H * W;
        if (fmt == 0) ingest_argb32_scalar<<<blocks, kIngestThreads, 0, st>>>(src, src_pitch, src_stride, d_dst, dst_pitch, dst_stride, W, H, n_px);
        else ingest_gray16_scalar<<<blocks, kIngestThreads, 0, st>>>(src, src_pitch, src_stride, d_dst, dst_pitch, dst_stride, W, H, n_px);
    }
    CU(cudaGetLastError());
    return VI_OK;
}

extern "C" int vi_ingest_argb32(vi_ctx* c, const uint8_t* d_bgra, int n_images, int W, int H, int64_t src_pitch,
                                int64_t src_stride, uint8_t* d_gray, int64_t dst_pitch, int64_t dst_stride, void* stream) {
    return ingest_common(c, 0, d_bgra, n_images, W, H, src_pitch, src_stride, d_gray, dst_pitch, dst_stride, stream);
}

extern "C" int vi_ingest_gray16(vi_ctx* c, const uint16_t* d_gray16, int n_images, int W, int H, int64_t src_pitch,
                                int64_t src_stride, uint8_t* d_gray, int64_t dst_pitch, int64_t dst_stride, void* stream) {
    return ingest_common(c, 1, d_gray16, n_images, W, H, src_pitch, src_stride, d_gray, dst_pitch, dst_stride, stream);
}
