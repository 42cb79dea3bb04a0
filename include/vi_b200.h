/*
 * vi_b200.h -- C ABI of the B200 batch-inspection path.
 *
 * The reference (hazernest/Vision-Inspection-system-Segmentation-using-
 * classical-computer-vision-) has no FFI layer: its seam is the Python module
 * API of segmentation.py plus the compute body of one UI method.  Each entry
 * point below cites the reference interface it replaces (file:line under the
 * reference tree).  The Python host side (vi_b200.segmentation / vi_b200.api)
 * binds these with ctypes; INTEGRATION.md shows the stub.
 *
 * Conventions: C linkage, plain pointers and sizes, no C++ / torch types.
 * Every function returns 0 on success or a negative VI_ERR_* code;
 * vi_last_error() returns a thread-local message for the last failure.
 * There is no CPU fallback: every compute entry point runs CUDA kernels on the
 * context's device and fails with VI_ERR_CUDA if it cannot.
 *
 * Threading: one vi_ctx per host thread and device.  vi_inspect_batch and
 * vi_segment_batch are asynchronous with respect to `stream`; all *_host /
 * compat entry points block until their results are in the caller's host buffers.
 *
 * Ordering: a context's tables (grid, exclusions, reference centroids) and its
 * per-SM scratch are shared by all of its calls.  The library orders them
 * itself: every entry point waits (on the device for a stream launch, on the host
 * for a table update or a blocking call) for the last asynchronous
 * vi_inspect_batch / vi_segment_batch of the same context before touching them, whatever stream that
 * batch ran on.  Output buffers of an asynchronous batch stay the caller's to
 * synchronise.  Every entry point leaves the caller's current CUDA device as it
 * found it.
 */
#ifndef VI_B200_H
#define VI_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VI_OK 0
#define VI_ERR_ARG (-1)         /* bad argument (null pointer, rect outside frame, bad size) */
#define VI_ERR_CUDA (-2)        /* CUDA runtime / launch failure                              */
#define VI_ERR_UNSUPPORTED (-3) /* a value the reference itself never uses (e.g. median_ksize != 21) */
#define VI_ERR_TOO_LARGE (-4)   /* unit larger than the documented bound (DESIGN.md section 2)  */

/* vi_unit_record.status */
#define VI_STATUS_OK 0        /* detector returned None or area < min_area (indexing_ui.py:1687, :1699) */
#define VI_STATUS_NG 1        /* defect area >= min_area (indexing_ui.py:1618, :1699)                   */
#define VI_STATUS_ROI_EMPTY 2 /* ROI empty after erosion -> detector returns None (:1514-1516)          */
#define VI_STATUS_SEGMENTED 3 /* segmented only (vi_segment_batch): no detector ran, no verdict          */

typedef struct vi_ctx vi_ctx;

/* Exclusion in base-unit-local pixels (indexing_ui.py:1811, :1816):
 * shape 0 = rect (a,b,c,d) = (x,y,w,h); shape 1 = circle (a,b,c) = (cx,cy,r). */
typedef struct vi_excl {
    int32_t shape, a, b, c, d;
} vi_excl;

/* The reference's widget values (indexing_ui.py:799-806, 870-875, 1522, 1548). */
typedef struct vi_params {
    int32_t seg_method;    /* 0 otsu (default; unknown strings fall back to it, segmentation.py:87-89), 1 adaptive */
    int32_t gaussian_blur; /* 3;  0 skips, even k -> k+1 (segmentation.py:78-79)          */
    int32_t morph_kernel;  /* 3;  0 skips (segmentation.py:91)                            */
    int32_t adapt_block;   /* 51  */
    int32_t adapt_C;       /* 10  */
    int32_t defect_method; /* 0 threshold (default), 1 canny                              */
    int32_t threshold;     /* 24  */
    int32_t min_area;      /* 20  */
    int32_t erode_px;      /* 6   */
    int32_t median_ksize;  /* 21 (hard-coded in the reference, indexing_ui.py:1522)       */
    double max_area_frac;  /* 0.98 (indexing_ui.py:1548)                                  */
} vi_params;

/* One record per (image, unit), 64 bytes. */
typedef struct vi_unit_record {
    int32_t image;       /* image index in the batch                                      */
    int32_t unit;        /* position in the grid list (the reference's loop index)       */
    int32_t otsu_t;      /* Otsu threshold of the blurred crop (segmentation.py:82)      */
    int32_t seg_area;    /* #(seg mask > 0) after exclusions (indexing_ui.py:1491)       */
    int32_t roi_area;    /* after erosion + largest 8-CC (indexing_ui.py:1545)           */
    int32_t defect_area; /* mask_stats(defect)['area'] (indexing_ui.py:1615, :1697)      */
    int32_t n_kept;      /* contours that passed the area filter (indexing_ui.py:1551)   */
    int32_t status;      /* VI_STATUS_*                                                   */
    int32_t dx, dy;      /* centroid shift applied to exclusions (indexing_ui.py:2310)   */
    double cx, cy;       /* pre-exclusion largest-8CC centroid, NaN if none (:2285,:2296) */
    int32_t n_ambiguous; /* diagnostics: ROI pixels that needed an exact rank count      */
    int32_t n_runs;      /* diagnostics: max run count seen by the labelling passes      */
} vi_unit_record;

const char* vi_last_error(void);
int vi_version(void);

void vi_params_default(vi_params* p);

int vi_ctx_create(int device, vi_ctx** out);
void vi_ctx_destroy(vi_ctx* ctx);

/* Grid rectangles, image-space (x,y,w,h) in list order: the `boxes` of grid
 * JSON v2 (indexing_ui.py:2739-2742, :2881-2889) / update_grid_preview (:2184-2191). */
int vi_set_grid(vi_ctx* ctx, const int32_t* rects_xywh, int n_units);
/* `exclusions` of grid JSON v2 (indexing_ui.py:2316-2338). n = 0 clears. */
int vi_set_exclusions(vi_ctx* ctx, const vi_excl* excl, int n);
/* exclusion_alignment.ref_centroids (indexing_ui.py:2856-2871): [n_units][2]
 * doubles (cx,cy), NaN = absent.  is_reference != 0 means the batch IS the
 * reference image (indexing_ui.py:2259): shifts are 0.  NULL clears. */
int vi_set_ref_centroids(vi_ctx* ctx, const double* cxcy, int n_units, int is_reference);

/* Sum of w*h over the grid, and the prefix sums (n_units+1 entries) that locate
 * each unit's packed mask inside one image's mask block. */
int64_t vi_unit_pixels(vi_ctx* ctx);
int vi_unit_offsets(vi_ctx* ctx, int64_t* out_offsets);

/* The hot path: run_segmentation_all (indexing_ui.py:2268-2338) followed by
 * run_inspection (indexing_ui.py:1669-1702) for every unit of every image.
 * d_frames: device, uint8 mono, image i at d_frames + i*image_stride, rows
 * row_pitch bytes apart.  Outputs (device): masks packed per unit in grid order,
 * image-major, values 0/255 (mask of image i, unit u starts at
 * i*vi_unit_pixels + offsets[u]); d_labels (optional, may be NULL): int32
 * raster-canonical 8-connected labels of the eroded ROI source (the labelling at
 * indexing_ui.py:1505), same packing; d_records: [n_images*n_units].
 * Asynchronous on `stream` (a cudaStream_t). */
int vi_inspect_batch(vi_ctx* ctx, const uint8_t* d_frames, int n_images, int W, int H,
                     int64_t row_pitch, int64_t image_stride, const vi_params* params,
                     uint8_t* d_seg_masks, uint8_t* d_defect_masks, int32_t* d_labels_or_null,
                     vi_unit_record* d_records, void* stream);

/* Optional extra output of subsequent vi_inspect_batch calls: per (image, unit) the area, sum of x and sum of y of
 * the final segmentation mask (after exclusions) -- what segmentation.mask_stats returns for the exported
 * mask_%04d.png in export_masks_and_csv (indexing_ui.py:2716-2722; the caller divides in double, as numpy's mean
 * does).  d_stats: device, int64 [n_images*n_units][3]; NULL switches it off. */
int vi_set_seg_stats_output(vi_ctx* ctx, int64_t* d_stats);

/* One kept defect component: an external contour of the opened residual that passed the area filter
 * (indexing_ui.py:1551-1558).  Unit-local coordinates, like the masks and vi_unit_record.cx / cy.  40 bytes. */
typedef struct vi_defect_blob {
    int32_t x, y, w, h;   /* bounding box = cv2.boundingRect(contour)                                        */
    int32_t area;         /* pixels of the filled contour (drawContours FILLED): its share of defect_area     */
    int32_t area2;        /* 2 * cv2.contourArea(contour), exact                                              */
    double cx, cy;        /* mean x, mean y of those pixels (mask_stats of the filled contour)                */
} vi_defect_blob;

#define VI_MAX_BLOBS_PER_UNIT 1024

/* Optional output of subsequent vi_inspect_batch calls, the table of kept defect components.  d_blobs: device,
 * [n_images*n_units][max_per_unit].  Slot j of (image, unit) holds the j-th kept component in raster order of its
 * first pixel, for j < min(n_kept, max_per_unit); later slots are not written.  vi_unit_record.n_kept stays the total.
 * Units whose ROI is empty or whose residual does not survive the opening write none (n_kept is 0 there).
 * max_per_unit outside 1..VI_MAX_BLOBS_PER_UNIT is VI_ERR_ARG; NULL switches the table off. */
int vi_set_defect_blob_output(vi_ctx* ctx, vi_defect_blob* d_blobs, int max_per_unit);

/* Same, from and to HOST buffers: works through the batch in chunks on internal
 * streams so that upload, compute and download overlap; blocks until done.  Pinned
 * and pageable frames take the same path: the frame rows that some unit covers are
 * copied to a device staging buffer.  h_seg_masks / h_defect_masks may be NULL to
 * skip that download.  This is the end-to-end call bench.py times as `e2e`. */
int vi_inspect_batch_host(vi_ctx* ctx, const uint8_t* h_frames, int n_images, int W, int H,
                          int64_t row_pitch, int64_t image_stride, const vi_params* params,
                          uint8_t* h_seg_masks, uint8_t* h_defect_masks, vi_unit_record* h_records);

/* mask_format of vi_inspect_batch_host_fmt */
#define VI_MASKS_BYTES 0  /* 0/255 bytes, vi_unit_pixels per image: what ROLE_BASE+1 / +2 pixmaps hold (indexing_ui.py:2355, :1608) */
#define VI_MASKS_PACKED 1 /* 1 bit per pixel, rows of ceil(w/32) 32-bit words, first pixel = most significant bit of its
                           * byte: the scanline layout of a 1-bit PNG (export_masks_and_csv, indexing_ui.py:2703-2730) and of
                           * numpy.unpackbits; vi_packed_mask_bytes per image, unit u at vi_packed_mask_offsets[u]          */
#define VI_MASKS_NONE 2   /* records only -- all run_inspection keeps (indexing_ui.py:1686-1706); mask pointers ignored   */

/* vi_inspect_batch_host with a choice of mask format (VI_MASKS_BYTES = vi_inspect_batch_host itself). */
int vi_inspect_batch_host_fmt(vi_ctx* ctx, const uint8_t* h_frames, int n_images, int W, int H,
                              int64_t row_pitch, int64_t image_stride, const vi_params* params,
                              int mask_format, void* h_seg_masks, void* h_defect_masks,
                              vi_unit_record* h_records);

/* vi_inspect_batch_host_fmt plus the kept-component table (vi_set_defect_blob_output) into a host buffer
 * h_blobs [n_images*n_units][max_per_unit]; h_blobs NULL: none.  Here the slots past min(n_kept, max_per_unit)
 * are unspecified (whole device tables are downloaded beside the records). */
int vi_inspect_batch_host_blobs(vi_ctx* ctx, const uint8_t* h_frames, int n_images, int W, int H,
                                int64_t row_pitch, int64_t image_stride, const vi_params* params,
                                int mask_format, void* h_seg_masks, void* h_defect_masks,
                                vi_unit_record* h_records, vi_defect_blob* h_blobs, int max_per_unit);

/* Segmentation only: run_segmentation_all (indexing_ui.py:2203-2368) for every unit of every image, without the
 * defect detector -- what an image switch, an exclusion edit, the reference image's centroids
 * (exclusion_alignment.ref_centroids, :2214-2233) and the mask / CSV export (:2703-2730) need.  Arguments, argument
 * errors, frames, grid, exclusions, reference centroids, seg-mask packing and the peer record tables are those of
 * vi_inspect_batch; so are the vi_set_seg_stats_output and vi_set_packed_mask_output seg outputs.  Records: otsu_t,
 * seg_area, dx, dy, cx, cy and n_runs as vi_inspect_batch gives them; roi_area, defect_area, n_kept and n_ambiguous
 * are 0; status is VI_STATUS_SEGMENTED.  The defect bits, the blob table and labels are never written.
 * Asynchronous on `stream`. */
int vi_segment_batch(vi_ctx* ctx, const uint8_t* d_frames, int n_images, int W, int H, int64_t row_pitch,
                     int64_t image_stride, const vi_params* params, uint8_t* d_seg_masks, vi_unit_record* d_records,
                     void* stream);
/* vi_segment_batch from and to HOST buffers, as vi_inspect_batch_host_fmt does it (chunks on internal streams, the
 * covered rows uploaded, VI_MASKS_* formats; h_seg_masks may be NULL).  Blocks until done. */
int vi_segment_batch_host(vi_ctx* ctx, const uint8_t* h_frames, int n_images, int W, int H, int64_t row_pitch,
                          int64_t image_stride, const vi_params* params, int mask_format, void* h_seg_masks,
                          vi_unit_record* h_records);

/* Packed-bit masks (VI_MASKS_PACKED layout) as an optional extra output of subsequent vi_inspect_batch calls:
 * device pointers, vi_packed_mask_bytes per image; NULL switches one off. */
int vi_set_packed_mask_output(vi_ctx* ctx, uint32_t* d_seg_bits, uint32_t* d_defect_bits);
int64_t vi_packed_mask_bytes(vi_ctx* ctx);
int vi_packed_mask_offsets(vi_ctx* ctx, int64_t* out_byte_offsets /* n_units + 1 */);

/* ---- multi-GPU: the per-unit verdict table (SURVEY 8e) ------------------------------------------------
 * One process per GPU; images are sharded round robin (rank r owns global images r, r + world, ...).  The only
 * exchange of the path is the table of 64-byte records.  It is fused into the kernel: every rank allocates a table
 * for ALL global images (vi_peer_table_create: cudaMalloc + a CUDA IPC handle), the ranks swap handles through
 * their launcher (torch.distributed in vi_b200.dist), map each other's tables (vi_peer_table_open) and hand the list
 * to vi_set_record_peers.  From then on vi_inspect_batch stores every record -- with the global image index
 * image_mul * k + image_add for local image k -- at [image * n_units + unit] of every table over NVLink, next to
 * d_records; no collective runs on the data path.  A table is complete once all ranks' batches have finished
 * (their streams synchronised and a barrier passed).  n = 0 switches the exchange off. */
int vi_peer_table_create(vi_ctx* ctx, int64_t n_records, void** d_table, uint8_t* handle64 /* 64 bytes out */);
int vi_peer_table_open(vi_ctx* ctx, const uint8_t* handle64, void** d_peer_table);
int vi_peer_table_close(vi_ctx* ctx, void* d_peer_table);
int vi_peer_table_destroy(vi_ctx* ctx, void* d_table);
int vi_peer_table_read(vi_ctx* ctx, const void* d_table, int64_t n_records, vi_unit_record* h_out);   /* blocking download */
int vi_set_record_peers(vi_ctx* ctx, void* const* d_tables, int n, int image_mul, int image_add);

/* Bytes vi_inspect_batch_host moves host -> device for n_images frames of the given row_pitch: only the frame rows
 * that some unit covers are copied (one strided copy per merged row interval).  0 when row_pitch <= 0. */
int64_t vi_host_upload_bytes(vi_ctx* ctx, int n_images, int64_t row_pitch);

/* ---- frame ingest (device pointers, asynchronous on `stream`) ---------------- */

/* segmentation.qimage_to_gray_array (segmentation.py:15-23) on the device: QImage ARGB32 frames (bytes B,G,R,A)
 * to the mono uint8 frames vi_inspect_batch takes.  The reference reverses the colour channels before
 * cv2.cvtColor(BGR2GRAY), so gray = (R*3735 + G*19235 + B*9798 + 16384) >> 15; identity on R=G=B.
 * Pitches and strides in bytes.  HBM streaming: 4 B read + 1 B written per pixel. */
int vi_ingest_argb32(vi_ctx* ctx, const uint8_t* d_bgra, int n_images, int W, int H, int64_t src_pitch,
                     int64_t src_stride, uint8_t* d_gray, int64_t dst_pitch, int64_t dst_stride, void* stream);
/* ImageWidget.load_image's 16-bit rule (indexing_ui.py:153-155), (arr / 256).astype(uint8), on the device:
 * little-endian uint16 frames to mono uint8 frames.  2 B read + 1 B written per pixel. */
int vi_ingest_gray16(vi_ctx* ctx, const uint16_t* d_gray16, int n_images, int W, int H, int64_t src_pitch,
                     int64_t src_stride, uint8_t* d_gray, int64_t dst_pitch, int64_t dst_stride, void* stream);

/* ---- per-unit compat entry points (host pointers, synchronous) ------------ */

/* segmentation.segment_cell (segmentation.py:75-100): gray [h][w] -> mask 0/255. */
int vi_segment_cell(vi_ctx* ctx, const uint8_t* gray, int h, int w, const vi_params* params,
                    uint8_t* out_mask, int32_t* out_otsu_t);
/* segmentation.fill_internal_holes (segmentation.py:27-72). */
int vi_fill_internal_holes(vi_ctx* ctx, const uint8_t* mask, int h, int w, uint8_t* out_mask);
/* segmentation.mask_stats (segmentation.py:103-111): area, sum of x, sum of y of
 * mask>0 (the caller divides in double, as numpy's mean does). */
int vi_mask_stats(vi_ctx* ctx, const uint8_t* mask, int h, int w, int64_t* area, int64_t* sum_x,
                  int64_t* sum_y);
/* cv2.erode(mask, None, iterations=r) on a binarised mask (indexing_ui.py:1497). */
int vi_erode_square(vi_ctx* ctx, const uint8_t* mask, int h, int w, int r, uint8_t* out_mask);
/* cv2.connectedComponentsWithStats(conn=8) + argmax area (indexing_ui.py:1505-1510,
 * :2240-2248): labels in raster-canonical order (may be NULL), the chosen
 * component's canonical label, area and coordinate sums. n_labels excludes 0. */
int vi_label_components(vi_ctx* ctx, const uint8_t* mask, int h, int w, int32_t* out_labels,
                        int32_t* n_labels, int32_t* best_label, int64_t* best_area,
                        int64_t* best_sum_x, int64_t* best_sum_y);
/* MainWindow._detect_defects_on_pix (indexing_ui.py:1471-1572) minus Qt:
 * *found = 0 means the reference returns None (out_mask is then all zero). */
int vi_detect_defects(vi_ctx* ctx, const uint8_t* gray, const uint8_t* seg_mask, int h, int w,
                      const vi_params* params, uint8_t* out_mask, int32_t* found,
                      vi_unit_record* out_record_or_null);

/* ---- diagnostics -------------------------------------------------------------- */
/* Per-phase SM cycle counts of every unit of subsequent vi_inspect_batch calls:
 * d_cycles is device memory, [n_images*n_units][40] int64 (NULL switches it off). */
int vi_debug_set_profile(vi_ctx* ctx, long long* d_cycles);
/* Self-checked build (libvi_b200_checked.so, -DVI_CHECKED=1): the first bounds check that failed in any kernel since the
 * library was loaded (0 = none; codes: vi_device.cuh CheckCode).  The production library returns VI_ERR_UNSUPPORTED. */
int vi_debug_check_word(vi_ctx* ctx, uint32_t* out_code);
/* Compares the reciprocal-based division of the Otsu recurrence with the IEEE divide on
 * n_samples pseudo-random operand pairs; *mismatches must come back 0. */
int vi_debug_fastdiv_check(vi_ctx* ctx, long long n_samples, unsigned long long seed, long long* mismatches);
/* The device Otsu threshold of n histograms (device memory: d_hists [n][256], d_npix [n] = each one's pixel count,
 * 1..2^24): d_out [n][3] = t (the exact scan, cv2.threshold's OTSU value), t_apx (the float32 arg max) and last (the
 * bound the scan stops at).  VI_ERR_ARG (and -1 in that row) when an npix is out of range or not its histogram's sum. */
int vi_debug_otsu(vi_ctx* ctx, const uint32_t* d_hists, const int* d_npix, int n, int* d_out);
/* The median residual stage alone (|gray - medianBlur(gray, 21)| > thr inside the ROI), one CTA running the inspection
 * kernel's device functions on caller-chosen levels (host int[3], sorted, 0..255) instead of its own.  Device memory:
 * d_gray [h][w] and d_roi [h][w] (non-zero = inside), w x h inside the unit bound; d_cand receives the raw candidate
 * mask, h rows of (w + 31) / 32 words, bit x & 31 of word x >> 5 (padding bits 0).  thr and pad (the byte written past w
 * in each row of the kernel's crop copy) in 0..255; ccap in 0..4096 and ecap in 0..16384 cap the dirty-cell and the
 * ambiguous-pixel lists (the rest take the inline overflow paths).  Host counts[3] = ambiguous-pixel list entries (one
 * per open test), dirty cells that touch the ROI, the exact Otsu threshold of the crop's histogram. */
int vi_debug_rank_residual(vi_ctx* ctx, const uint8_t* d_gray, const uint8_t* d_roi, int w, int h, const int* levels, int thr,
                           int ccap, int ecap, int pad, uint32_t* d_cand, int* counts);

/* Host only: the float32 taps of the adaptive threshold's Gaussian mean for an odd block size
 * (cv2.getGaussianKernel(bs, 0, CV_32F) as cv2.adaptiveThreshold uses it, segmentation.py:85). */
int vi_debug_adaptive_taps(int block_size, float* out_taps);

#ifdef __cplusplus
}
#endif
#endif /* VI_B200_H */
