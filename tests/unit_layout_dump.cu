// Host-only driver of tests/test_unit_layout.py: prints vi::unit_layout for the grids given as arguments, one JSON
// object per line.  An argument is "smem_optin,smem_static,f32_plane,blob_k:WxH[,WxH...]" (the units of one grid).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include "vi_device.cuh"
using namespace vi;

static void region(const char* name, const char* space, long long off, long long bytes, bool& first) {
    printf("%s[\"%s\",\"%s\",%lld,%lld]", first ? "" : ",", name, space, off, bytes);
    first = false;
}

int main(int argc, char** argv) {
    for (int i = 1; i < argc; ++i) {
        int optin, fixed, f32, blob_k, n = 0;
        if (sscanf(argv[i], "%d,%d,%d,%d:%n", &optin, &fixed, &f32, &blob_k, &n) != 4 || !n) return 2;
        UnitExtent e{};
        for (const char* p = argv[i] + n; *p;) {
            int w, h, k = 0;
            if (sscanf(p, "%dx%d%n", &w, &h, &k) != 2) return 2;
            e.add(w, h);
            p += k;
            if (*p == ',') ++p;
        }
        UnitLayout L;
        if (!unit_layout(e, optin, fixed, f32 != 0, blob_k, &L)) { printf("{\"ok\":false}\n"); continue; }
        printf("{\"ok\":true,\"wmax\":%d,\"hmax\":%d,\"gray\":%d,\"mask\":%d,\"ws_off\":%d,\"ws\":%d,\"otsu_off\":%d,"
               "\"stage\":%d,\"lattice_off\":%d,\"lattice_bytes\":%lld,\"n_hist\":%d,\"run_rf\":%d,"
               "\"run_cap\":%d,\"band_off\":%d,\"band_cap\":%d,\"dirty_cap\":%d,\"exact_cap\":%d,\"blob_off\":%d,"
               "\"blob_cap\":%d,\"total\":%d,\"arena\":%d,\"arena_bytes\":%lld,\"blur_off\":%lld,\"runs_off\":%lld,"
               "\"runs_cap\":%d,\"rank_off\":%lld,\"rank_words\":%d,\"f32_off\":%lld,\"blob_tail_off\":%lld,"
               "\"scratch_bytes\":%lld,\"lattice_fits_max\":%d,\"regions\":[",
               e.wmax, e.hmax, L.gray_bytes, L.mask_bytes, L.ws_off, L.ws_bytes, L.otsu_off, L.stage_bytes,
               L.lattice_off, L.lattice_bytes, L.n_hist, L.run_rf, L.run_cap, L.band_off, L.band_cap,
               L.dirty_cap, L.exact_cap, L.blob_off, L.blob_cap, L.total, L.arena, L.arena_bytes, L.blur_off,
               L.runs_off, L.runs_cap, L.rank_off, L.rank_words, L.f32_off, L.blob_tail_off, L.scratch_bytes,
               (int)lattice_fits(e.wmax, e.hmax, L));
        // every region the kernel addresses, in "unit" space (shared memory or the arena) or "scratch" space
        bool first = true;
        static const char* kMask[kNumMasks] = {"MA", "MB", "MC", "MD", "ME"};
        region("gray", "unit", 0, L.gray_bytes, first);
        for (int k = 0; k < kNumMasks; ++k) region(kMask[k], "unit", L.gray_bytes + (long long)k * L.mask_bytes, L.mask_bytes, first);
        region("ws", "unit", L.ws_off, L.ws_bytes, first);
        if (!L.arena) region("hist", "unit", L.gray_bytes, (long long)L.n_hist * kHistBytes, first);
        if (!L.arena) region("stage", "unit", 0, L.stage_bytes, first);
        region("lattice", "unit", L.lattice_off, L.lattice_bytes, first);
        region("otsu", "unit", L.otsu_off, kOtsuWsBytes, first);
        region("band", "unit", L.band_off, 4ll * L.band_cap, first);
        region("runs", "unit", L.ws_off, ccl_ws_bytes(L.run_cap, e.hmax), first);
        region("dirty", "unit", L.ws_off, 4ll * L.dirty_cap, first);
        region("exact", "unit", L.ws_off + 4ll * L.dirty_cap, 4ll * L.exact_cap, first);
        region("blob", "unit", L.blob_off, (long long)L.blob_cap * (long long)sizeof(BlobAcc), first);
        const long long px = (long long)e.wmax * e.hmax;
        region("hsum", "scratch", 0, 2 * px, first);
        region("blurred", "scratch", L.blur_off, (long long)((e.wmax + 3) & ~3) * e.hmax, first);
        region("runs_g", "scratch", L.runs_off, ccl_ws_bytes(L.runs_cap, e.hmax), first);
        region("rank", "scratch", L.rank_off, rank_scratch_bytes(e.wmax, e.hmax), first);
        region("f32", "scratch", L.f32_off, f32 ? 4 * px : 0, first);
        region("blob_tail", "scratch", L.blob_tail_off, (long long)blob_k * (long long)sizeof(BlobAcc), first);
        printf("]}\n");
    }
    return 0;
}
