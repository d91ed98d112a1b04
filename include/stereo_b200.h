/*
 * stereo_b200.h -- C ABI of libstereo_b200.so, the B200 (sm_100a) replacement for
 * everything nvcc compiles in chrg127/stereomatching: src/stereo.cu,
 * src/stereo-ghost.cu, src/image.cu and src/util.cu.
 *
 * The reference has no plugin / FFI seam: each CUDA program is a monolith whose
 * main() calls file-local functions (SURVEY.md 8b).  The seam cut here is therefore
 * "every device-side thing main()/algorithm() do", one entry point per call site.
 * Each declaration cites the reference lines it stands in for (paths relative to the
 * reference checkout).
 *
 * Conventions
 *   - plain C types only; a context is an opaque pointer; no torch / C++ types.
 *   - every function returns SM_OK (0) or a negative sm_status; the message of the
 *     last failure on the calling thread is sm_last_error().  The library never
 *     calls exit() -- the reference's print-and-exit policy (util.h:49-58,
 *     helper_cuda.h:890-905) stays in the host driver (host/driver.c).
 *   - one context = one device + one stream + one frame geometry.  Contexts are
 *     independent; a single context must not be used from two threads at once.
 *     (The reference is not re-entrant at all: file-scope matches[]/scores[] and
 *     __device__ pointer tables, stereo.cu:98,157.)
 *   - images are row-major, IDX(x,y,w) = y*w + x (util.h:23), no ghost padding at
 *     the ABI: the ghost cells of stereo-ghost.cu are an internal matter of the
 *     GHOST variant and are never visible to the caller.
 *   - all work is queued on the context's stream; sm_download*, sm_elapsed_ms and
 *     sm_synchronize wait for it.
 */
#ifndef STEREO_B200_H_INCLUDED
#define STEREO_B200_H_INCLUDED

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sm_ctx sm_ctx;

typedef enum sm_status {
    SM_OK = 0,
    SM_ERR_ARG = -1,        /* bad argument (sizes, ranges, NULL) */
    SM_ERR_CUDA = -2,       /* a CUDA runtime call or kernel failed */
    SM_ERR_STATE = -3,      /* call order: e.g. sm_match_wta before any edges exist */
    SM_ERR_DEGENERATE = -4, /* draw_contour_map: (max-min)/lines == 0; the reference
                               divides by zero here (stereo.c:265-272, SURVEY 3.4) */
    SM_ERR_NOMEM = -5
} sm_status;

/* Border semantics.  WRAP = stereo.c / stereo.cu (toroidal idx(), util.h:42-47).
 * GHOST = stereo-ghost.c / stereo-ghost.cu (zero ghost cells around edge and match
 * images, 128.0 around the brightness, ghost.h, stereo-ghost.c:93-97,286-287,384-385). */
typedef enum sm_variant { SM_WRAP = 0, SM_GHOST = 1 } sm_variant;

/* Which array sm_download() fetches.  One per write_gpu_image()/write_matches()/
 * write_scores() call site of algorithm() (stereo.cu:311-331). */
typedef enum sm_plane {
    SM_EDGES1 = 0,    /* u8  first_edges   (stereo.cu:313) */
    SM_EDGES2 = 1,    /* u8  second_edges  (stereo.cu:314) */
    SM_MATCH = 2,     /* u8  matches[i]    (stereo.cu:108-114), needs shift i */
    SM_SCORE_ALL = 3, /* i32 box sum of matches[i] before masking ("score_all-i", stereo.cu:201-203) */
    SM_SCORE = 4,     /* i32 scores[i]     (stereo.cu:167-173), needs shift i */
    SM_BEST = 5,      /* i32 buf after find_highest_scoring_shifts ("score_best-0", stereo.cu:324) */
    SM_WEB = 6,       /* i32 web           ("web-1", stereo.cu:325) */
    SM_WEB_FILLED = 7,/* i32 web after fill_web_holes ("web-2", stereo.cu:330) */
    SM_OUTPUT = 8     /* u8  contour bitmap ("output-0", stereo.cu:332) */
} sm_plane;

/* Hot-path kernel selection (sm_set_kernel). */
typedef enum sm_kernel {
    SM_KERNEL_AUTO = 0,
    SM_KERNEL_DIRECT = 1,  /* one thread per pixel, popcount of the window rows (simple, slow) */
    SM_KERNEL_BITSLICE = 2 /* bit-sliced running box sums, 32 shifts per word (the fast path) */
} sm_kernel;

/* Context options (sm_set_option): what used to be environment hooks. */
typedef enum sm_option {
    SM_OPT_EDGES_FP64 = 1, /* 1: always run the FP64 edge detector (the reference's arithmetic, stereo.cu:83-92),
                              even for 8-bit uploads; 0 (default): the integer table path for 8-bit images */
    SM_OPT_PIPE_GROUP = 2, /* pairs per stage of the sm_run_batch pipeline; 0 (default): chosen by frame size.
                              Only before the first sm_run_batch of the context */
    SM_OPT_ROW_RUNS = 3    /* row runs per 32-column strip of a one-pair launch of the bit-sliced kernel;
                              0 (default): the kernel's cost model */
} sm_option;

/* What sm_get_info reports about the launch configuration of the bit-sliced kernel on this context. */
typedef enum sm_info {
    SM_INFO_WARPS_PER_SM = 1,     /* resident warps per SM of the kernel instantiation this geometry uses */
    SM_INFO_PAIRS_PER_LAUNCH = 2, /* pairs the batch entries put into one launch (0 before the first batch call) */
    SM_INFO_TMEM_COLUMNS = 3,     /* tensor-memory columns one CTA allocates for the vertical-window ring */
    SM_INFO_EDGE_THRESHOLDS = 4,  /* 1: the edge detector's current decision table is exactly a threshold table
                                     (symmetric and monotone, checked bit by bit on the device) and the fast
                                     detector uses it; 0: it falls back to the bit table; -1: no table built yet */
    SM_INFO_KERNEL_SHAPE = 5,     /* the kernel the most recent hot-path launch on this context ran, as an
                                     sm_shape code (0 before any launch).  A batch call launches once per group of
                                     pairs: the code is that of its last group */
    SM_INFO_ROW_RUNS = 6          /* row runs per strip of that launch (its grid.y, after rounding the runs to whole
                                     blocks of rows); 0 before any launch and for the direct kernel */
} sm_info;

/* SM_INFO_KERNEL_SHAPE codes.  A bit-sliced launch reports SM_SHAPE_BITSLICE | half | the flags of its
 * instantiation, the direct kernel SM_SHAPE_DIRECT. */
typedef enum sm_shape {
    SM_SHAPE_HALF = 0xF,        /* mask: window half, square_width / 2 (0..15) */
    SM_SHAPE_TWO_WORDS = 0x10,  /* two 32-bit words per lane (64 shifts per pass, or two pixels with C2) */
    SM_SHAPE_SEG8 = 0x20,       /* 8-pixel walker segments (8-row blocks); 16-pixel segments otherwise */
    SM_SHAPE_C2 = 0x40,         /* column pairs: the two words of a lane are two pixels, 32 shifts or fewer */
    SM_SHAPE_HP = 0x80,         /* half-word pairs: each word serves two pixels, 16 shifts or fewer */
    SM_SHAPE_MULTI = 0x100,     /* more than 64 shifts: successive 64-shift chunks merged in place */
    SM_SHAPE_BITSLICE = 0x200,  /* set in every bit-sliced code */
    SM_SHAPE_DIRECT = 0x400     /* the direct kernel (SM_KERNEL_DIRECT) */
} sm_shape;

/* ---- library-level -------------------------------------------------------- */

/* Message of the last failure on this thread ("" if none). */
const char *sm_last_error(void);
/* ABI version: (major << 16) | minor.  The 16-bit result entries (sm_match_wta_dev_batch16, sm_run_batch16,
 * sm_multi_run_batch16, sm_bands_run16, sm_download_web_u16), the search-range creators (sm_create_range,
 * sm_create_band_range, sm_multi_create_range, sm_bands_create_range) and the runner-up entries
 * (sm_match_wta_dev_batch_ru16, sm_run_batch_ru16, sm_multi_run_batch_ru16, sm_bands_run_ru16) and the sub-pixel
 * entries (sm_match_wta_dev_batch_sub16, sm_run_batch_sub16, sm_multi_run_batch_sub16, sm_bands_run_sub16) are
 * additions to 1.3 that leave every other entry as it was; clients detect them by symbol. */
int sm_version(void);
/* Number of CUDA devices visible, or a negative sm_status. */
int sm_device_count(void);

/* Pinned host staging memory (the reference uses pageable malloc + cudaMemcpy,
 * util.h:131-136; pinned memory lets sm_upload_* run asynchronously). */
int sm_host_alloc(void **ptr, size_t bytes);
int sm_host_free(void *ptr);

/* ---- context -------------------------------------------------------------- */

/* Replaces the device allocations at the top of algorithm() (stereo.cu:299-306;
 * stereo-ghost.cu:299-307) and allocate_matches/allocate_scores (stereo.cu:100-106,
 * 159-165).  num_shifts is the reference's compile-time NUM_SHIFTS (stereo.cu:6),
 * here a run-time value in [1, 512]; square_width in [0, 63] (the window is
 * (2*(square_width/2)+1)^2, stereo.cu:144-146: 0 is the 1x1 window, as in the reference) and <= width, height
 * (stereo.cu:395-398). */
int sm_create(sm_ctx **ctx, int device, int width, int height, int num_shifts,
              int square_width, int variant);

/* A context that owns only output rows [row0, row1) of a frame_height-row frame:
 * the row-band shard of SURVEY.md 8(e).  Uploads and downloads still take / give
 * whole-frame host arrays; only rows [row0 - half - 1, row1 + half + 1) (taken
 * mod frame_height for WRAP) are copied in, and only rows [row0,row1) are written
 * by sm_download*.  sm_create(...) == sm_create_band(..., 0, height). */
int sm_create_band(sm_ctx **ctx, int device, int width, int frame_height, int row0, int row1,
                   int num_shifts, int square_width, int variant);

/* Contexts that search the shifts [min_shift, min_shift + num_shifts) instead of [0, num_shifts): the disparity range
 * of a rig whose scene lies at min_shift or more (OpenCV's minDisparity + numDisparities).  match_s(x, y) compares the
 * first image at x with the second at x + s (WRAP: mod width, whatever the multiple; GHOST: 0 where x + s >= width);
 * box sums and the centre mask are unchanged; best = max(0, max_s score_s) and web = 1 + the highest s whose score
 * equals best, so a pixel whose scores are all zero gets web = min_shift + num_shifts, and web >= 1 + min_shift
 * everywhere (sm_fill_web_holes stays the identity).  The debug planes of sm_download take the real shift s, which must
 * lie in the range; SM_EDGES1/2 stay the whole, unshifted edge maps.  Limits: min_shift >= 0 and
 * min_shift + num_shifts <= 65535 (the 16-bit web stays exact); the u8 web (sm_download_web_u8, web_u8 of the batch
 * entries) needs min_shift + num_shifts <= 255.  The work is that of num_shifts shifts at any min_shift.  min_shift == 0 is the
 * reference's range: sm_create(...) == sm_create_range(..., 0, num_shifts, ...), and likewise for the band, multi and
 * bands creators.  All argument checks come before any device call. */
int sm_create_range(sm_ctx **ctx, int device, int width, int height, int min_shift, int num_shifts,
                    int square_width, int variant);
int sm_create_band_range(sm_ctx **ctx, int device, int width, int frame_height, int row0, int row1, int min_shift,
                         int num_shifts, int square_width, int variant);

/* Replaces the cudaFree block at the end of algorithm() (stereo.cu:339-346). */
int sm_destroy(sm_ctx *ctx);

/* Use an existing cudaStream_t (passed as void*) instead of the context's own. */
int sm_set_stream(sm_ctx *ctx, void *cuda_stream);
int sm_set_kernel(sm_ctx *ctx, int kernel);
int sm_set_option(sm_ctx *ctx, int option, int value);
/* A non-negative value, or a negative sm_status. */
int sm_get_info(sm_ctx *ctx, int what);
int sm_synchronize(sm_ctx *ctx);

/* ---- step 0: upload ------------------------------------------------------- */

/* Replaces MAKE_GPU_COPY(double, first.data, w*h) x2 (stereo.cu:402-403) and
 * ghost_add_gpu_double's per-row cudaMemcpy (stereo-ghost.cu:403-404, ghost.h:78-90).
 * sm_upload_f64 takes the reference's Image.data layout (double = u8/256.0,
 * image.c:9-15); sm_upload_u8 takes the 8-bit pixels themselves (1 B/pixel instead
 * of 8 B/pixel over PCIe) and is exactly equivalent for images that came from
 * read_image(). */
int sm_upload_f64(sm_ctx *ctx, const double *first, const double *second);
int sm_upload_u8(sm_ctx *ctx, const uint8_t *first, const uint8_t *second);

/* ---- step 1: edges (SURVEY 8f n1) ------------------------------------------ */

/* Replaces the two find_all_edges<<<>>> launches (stereo.cu:311-312 -> :83-92;
 * stereo-ghost.cu:84-93).  FP64, same operation order as stereo.c:16-28. */
int sm_edges(sm_ctx *ctx, double threshold);

/* Hot-path-only entry: supply first_edges / second_edges (u8, 0 or 1) from the host. */
int sm_set_edges(sm_ctx *ctx, const uint8_t *first_edges, const uint8_t *second_edges);

/* ---- step 2: THE HOT PATH --------------------------------------------------- */

/* Replaces fillup_matches<<<>>> (stereo.cu:316 -> :127-137), fillup_scores()
 * (stereo.cu:319 -> :194-207: 30 x {cudaMemset, addup_pixels_in_square<<<>>> :142-155,
 * record_score<<<>>> :185-192}), the cudaMemset of buf (stereo.cu:321) and
 * find_highest_scoring_shifts<<<>>> (stereo.cu:322 -> :211-225); the ghost twins are
 * stereo-ghost.cu:128-137,146-159,189-197,212-226.  Leaves `best` (the reference's
 * buf) and `web` on the device; neither matches[] nor scores[] is materialised. */
int sm_match_wta(sm_ctx *ctx);

/* Same, on caller-owned DEVICE memory (all four pointers are device pointers on the
 * context's device; edges u8 0/1, width*height; outputs i32 width*height).  For
 * callers that keep frames resident (bench.py uses torch tensors here). */
int sm_match_wta_dev(sm_ctx *ctx, const uint8_t *d_first_edges, const uint8_t *d_second_edges,
                     int32_t *d_best, int32_t *d_web);

/* The same for n_pairs resident pairs in one call: pair k's edge maps are at
 * d_*_edges + k*edge_stride (elements), its outputs at d_best/d_web + k*out_stride.
 * All inputs must be ready in stream order when the call is made.  Inside, a second
 * stream runs the bit-plane pack of pair k+1.. while the main kernel of pair k runs, so
 * per pair only the main kernel's time shows (whole-pair batches, SURVEY 8e/config 4).
 * Results are complete in stream order on the context's stream. */
int sm_match_wta_dev_batch(sm_ctx *ctx, int n_pairs, const uint8_t *d_first_edges,
                           const uint8_t *d_second_edges, size_t edge_stride, int32_t *d_best,
                           int32_t *d_web, size_t out_stride);

/* The same with 16-bit results, stored by the hot kernel itself (2 B per pixel and array instead of 4): web is in
 * 1..num_shifts <= 512 and best at most (2*(square_width/2)+1)^2 <= 3969, so both are exact.  d_best may be NULL:
 * then of the caller's memory only d_web is written (best goes to a scratch array of the context's).  Checks, streams, pairs per launch, the kernel chosen (SM_INFO_KERNEL_SHAPE) and
 * sm_elapsed_ms / sm_last_launches are those of sm_match_wta_dev_batch; n_pairs == 1 is the one-pair launch of
 * sm_match_wta. */
int sm_match_wta_dev_batch16(sm_ctx *ctx, int n_pairs, const uint8_t *d_first_edges, const uint8_t *d_second_edges,
                             size_t edge_stride, uint16_t *d_best, uint16_t *d_web, size_t out_stride);

/* The same, and each pixel's RUNNER-UP score, computed by the hot kernel's own winner-take-all: the second-largest
 * value of the multiset of the pixel's masked scores over the context's shifts, i.e. the maximum over every shift
 * but the one web names.  runner_up <= best everywhere; runner_up == best exactly where two or more shifts tie for
 * best (pixels whose scores are all 0 included, for num_shifts >= 2); 0 with num_shifts == 1.  It does not depend
 * on min_shift or on the tie rule, and web / best are those of sm_match_wta_dev_batch16.  The shifts next to the
 * winner are NOT excluded: past 64 shifts the kernel merges 64-shift chunks in place, and (best, runner_up) of two
 * chunks merge exactly while a runner-up outside an exclusion radius does not.  A uniqueness filter in the manner
 * of OpenCV's uniquenessRatio u keeps best >= T && 100 * runner_up < (100 - u) * best.  d_runner_up (not NULL)
 * takes pair k at k * out_stride, like d_web; 2 B per pixel. */
int sm_match_wta_dev_batch_ru16(sm_ctx *ctx, int n_pairs, const uint8_t *d_first_edges,
                                const uint8_t *d_second_edges, size_t edge_stride, uint16_t *d_best, uint16_t *d_web,
                                uint16_t *d_runner_up, size_t out_stride);

/* The same (best / web exactly those of sm_match_wta_dev_batch16), and each pixel's web in SIXTEENTHS of a shift,
 * interpolated by the hot kernel from the scores next to the winner (the fixed-point format of OpenCV's block
 * matchers, 4 fractional bits).  With the context's range [m, m + D), s(t) the masked score at shift t (the value
 * the winner-take-all maximises: the box sum where the centre matched, else 0) and w = web - 1 the winning shift:
 *   - w == m or w == m + D - 1 (no neighbour inside the range; also D == 1 and pixels whose scores are all 0):
 *     frac = 0;
 *   - else s- = s(w - 1), s+ = s(w + 1), den = 2 * best - s- - s+ (>= 1: ties go to the highest shift) and
 *     frac = min(7, floor((16 * (s+ - s-) + den) / (2 * den))), the vertex of the parabola through the three scores
 *     in sixteenths, rounded half up, in [-8, 7];
 *   - web_sub = 16 * web + frac.  So web_sub / 16 is a refined web and web_sub / 16 - 1 the disparity in pixels;
 *     (web_sub + 8) >> 4 == web and web_sub >= 16 * (m + 1) - 8 > 0 everywhere.
 * Integer arithmetic on exact counts: bit-exact.  Needs m + D <= 4095 (web_sub fits 16 bits), else SM_ERR_ARG
 * before any device call.  d_web_sub (not NULL) takes pair k at k * out_stride, like d_web; 2 B per pixel.  d_best
 * may be NULL. */
int sm_match_wta_dev_batch_sub16(sm_ctx *ctx, int n_pairs, const uint8_t *d_first_edges,
                                 const uint8_t *d_second_edges, size_t edge_stride, uint16_t *d_best, uint16_t *d_web,
                                 uint16_t *d_web_sub, size_t out_stride);

/* Device time of the last sm_match_wta* call on this context, CUDA events on the
 * context's stream (the reference brackets the whole algorithm() with
 * CLOCK_MONOTONIC instead, stereo.cu:308,334-335).  Waits for the call to finish. */
int sm_elapsed_ms(sm_ctx *ctx, float *ms);
/* Number of kernels the last sm_match_wta* call launched. */
int sm_last_launches(sm_ctx *ctx);

/* Per-kernel timing of many hot-path calls without synchronising in between: after
 * sm_profile_begin(ctx, max_calls) every sm_match_wta* call records its own event
 * triple (before pack, between pack and the main kernel, after) on the context's
 * stream; sm_profile_read waits for the stream and returns the number of calls
 * recorded and the summed device time of the pack kernel and of the main kernel.
 * bench.py's roofline figure comes from here.  sm_profile_begin(ctx, 0) switches it
 * off. */
int sm_profile_begin(sm_ctx *ctx, int max_calls);
int sm_profile_read(sm_ctx *ctx, int *n_calls, double *pack_ms_total, double *main_ms_total);

/* ---- step 3 (SURVEY 8f n3) --------------------------------------------------- */

/* Replaces the D2D copy + fill_web_holes() (stereo.cu:328-329 -> :247-259, kernel
 * :235-245). */
int sm_fill_web_holes(sm_ctx *ctx, int times);
/* Step 3 on a caller-supplied web (host array, i32, may contain 0 = "hole"): the entry for
 * using fill_web_holes / draw_contour_map on their own (the web sm_match_wta produces never
 * has holes, so for it sm_fill_web_holes is the identity and launches nothing). */
int sm_set_web(sm_ctx *ctx, const int32_t *web);

/* Replaces draw_contour_map() (stereo.cu:331 -> :276-285, kernel :261-274) and the
 * array_max_gpu/array_min_gpu reductions (util.cu:15-45).  web_min / web_max may be
 * NULL.  Returns SM_ERR_DEGENERATE when (max-min)/lines == 0. */
int sm_draw_contour_map(sm_ctx *ctx, int lines, int32_t *web_min, int32_t *web_max);

/* ---- download ---------------------------------------------------------------- */

/* Replaces write_gpu_image()'s make_host_copy (image.cu:15-23, util.h:138-143):
 * copies one array to host memory (u8 or i32 per sm_plane, width*height elements;
 * a band context writes only its rows [row0,row1) of the frame-sized array).
 * SM_MATCH / SM_SCORE_ALL / SM_SCORE planes are computed on demand for `shift`. */
int sm_download(sm_ctx *ctx, int which, int shift, void *host);

/* web as u8 (valid when min_shift + num_shifts <= 255): a quarter of the D2H bytes. */
int sm_download_web_u8(sm_ctx *ctx, uint8_t *host);
/* web as u16 (any num_shifts): half the D2H bytes. */
int sm_download_web_u16(sm_ctx *ctx, uint16_t *host);

/* ---- whole pairs, batched (SURVEY 8e, config 4; 8f n4) ------------------------ */

/* Runs n_pairs independent stereo pairs through upload -> edges -> hot path ->
 * download on ONE context/device as a three-stage pipeline over groups of pairs
 * (H2D of group g+1 | batched edges + hot path of group g | D2H of group g-1, three
 * streams, three rotating device buffer sets; returns when everything has landed in
 * web_out).  first/second: n_pairs frames of width*height u8,
 * back to back (pinned memory recommended).  web_out: n_pairs frames of i32 (or u8
 * when web_u8 != 0); best_out may be NULL.  Multi-GPU callers shard pairs over one
 * context per device (pair k -> device k mod n), no cross-device traffic. */
int sm_run_batch(sm_ctx *ctx, int n_pairs, const uint8_t *first, const uint8_t *second,
                 double threshold, void *web_out, int web_u8, int32_t *best_out);
/* The same with 16-bit web and best for any num_shifts: the hot kernel writes them directly (no int32 array, no
 * narrowing launch) and each comes back as one copy per group at 2 B per pixel.  best_out may be NULL. */
int sm_run_batch16(sm_ctx *ctx, int n_pairs, const uint8_t *first, const uint8_t *second, double threshold,
                   uint16_t *web_out, uint16_t *best_out);
/* The same and the runner-up scores (see sm_match_wta_dev_batch_ru16) into runner_up_out (not NULL): n_pairs
 * frames of u16, one more copy per group. */
int sm_run_batch_ru16(sm_ctx *ctx, int n_pairs, const uint8_t *first, const uint8_t *second, double threshold,
                      uint16_t *web_out, uint16_t *best_out, uint16_t *runner_up_out);
/* The same and web_sub (see sm_match_wta_dev_batch_sub16) into web_sub_out (not NULL): n_pairs frames of u16, one
 * more copy per group.  min_shift + num_shifts <= 4095. */
int sm_run_batch_sub16(sm_ctx *ctx, int n_pairs, const uint8_t *first, const uint8_t *second, double threshold,
                       uint16_t *web_out, uint16_t *best_out, uint16_t *web_sub_out);

/* The same over several GPUs of one box (SURVEY 8e, BASELINE config 4: whole pairs sharded across the
 * GPUs, inputs scattered from the host, no cross-device traffic): one context and one host thread per
 * entry of devices[] (an id may repeat); slot d runs pairs [n*d/N, n*(d+1)/N) through sm_run_batch. */
typedef struct sm_multi sm_multi;
int sm_multi_create(sm_multi **out, const int *devices, int n_devices, int width, int height,
                    int num_shifts, int square_width, int variant);
/* The same with the search range [min_shift, min_shift + num_shifts) (see sm_create_range). */
int sm_multi_create_range(sm_multi **out, const int *devices, int n_devices, int width, int height, int min_shift,
                          int num_shifts, int square_width, int variant);
int sm_multi_run_batch(sm_multi *m, int n_pairs, const uint8_t *first, const uint8_t *second,
                       double threshold, void *web_out, int web_u8, int32_t *best_out);
/* The same through sm_run_batch16 (best_out may be NULL). */
int sm_multi_run_batch16(sm_multi *m, int n_pairs, const uint8_t *first, const uint8_t *second, double threshold,
                         uint16_t *web_out, uint16_t *best_out);
/* The same through sm_run_batch_ru16 (runner_up_out not NULL). */
int sm_multi_run_batch_ru16(sm_multi *m, int n_pairs, const uint8_t *first, const uint8_t *second, double threshold,
                            uint16_t *web_out, uint16_t *best_out, uint16_t *runner_up_out);
/* The same through sm_run_batch_sub16 (web_sub_out not NULL). */
int sm_multi_run_batch_sub16(sm_multi *m, int n_pairs, const uint8_t *first, const uint8_t *second, double threshold,
                             uint16_t *web_out, uint16_t *best_out, uint16_t *web_sub_out);
int sm_multi_device_count(const sm_multi *m);
int sm_multi_destroy(sm_multi *m);

/* ONE pair as row bands over several GPUs of one box (SURVEY 8e, BASELINE config 3): slot g owns output rows
 * sm_band_rows(height, N, g), uploads them plus half + 1 halo rows per side, and writes only its own rows of the
 * caller's frame-sized web_out / best_out (best_out may be NULL).  One band context (sm_create_band) and one host
 * thread per entry of devices[]; no exchange between GPUs. */
typedef struct sm_bands sm_bands;
int sm_bands_create(sm_bands **out, const int *devices, int n_devices, int width, int height,
                    int num_shifts, int square_width, int variant);
/* The same with the search range [min_shift, min_shift + num_shifts) (see sm_create_range). */
int sm_bands_create_range(sm_bands **out, const int *devices, int n_devices, int width, int height, int min_shift,
                          int num_shifts, int square_width, int variant);
int sm_bands_run(sm_bands *b, const uint8_t *first, const uint8_t *second, double threshold,
                 int32_t *web_out, int32_t *best_out);
/* The same with 16-bit web / best (best_out may be NULL): each band's hot kernel writes its rows as u16 and only
 * those rows are copied back. */
int sm_bands_run16(sm_bands *b, const uint8_t *first, const uint8_t *second, double threshold,
                   uint16_t *web_out, uint16_t *best_out);
/* The same and the runner-up scores (see sm_match_wta_dev_batch_ru16): each band writes its own rows of the
 * frame-sized runner_up_out (not NULL). */
int sm_bands_run_ru16(sm_bands *b, const uint8_t *first, const uint8_t *second, double threshold,
                      uint16_t *web_out, uint16_t *best_out, uint16_t *runner_up_out);
/* The same and web_sub (see sm_match_wta_dev_batch_sub16): each band writes its own rows of the frame-sized
 * web_sub_out (not NULL). */
int sm_bands_run_sub16(sm_bands *b, const uint8_t *first, const uint8_t *second, double threshold,
                       uint16_t *web_out, uint16_t *best_out, uint16_t *web_sub_out);
int sm_bands_destroy(sm_bands *b);

/* ---- geometry helpers (host-side, no GPU) --------------------------------------- */

/* Splits frame rows [0,height) into n_bands contiguous bands; band b = [*row0,*row1). */
int sm_band_rows(int height, int n_bands, int band, int *row0, int *row1);

#ifdef __cplusplus
}
#endif

#endif /* STEREO_B200_H_INCLUDED */
