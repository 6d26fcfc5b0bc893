/*
 * frogmatch_debug.h -- test hooks of libfrogmatch.so.  NOT part of the drop-in boundary: these
 * exist so tests/ can check each device stage (sort + class table, FP16 operand packing, the
 * tcgen05 score tile, gate bands, candidate capture, the reject pass's per-row bounds, compaction) against
 * numpy in isolation.
 */
#ifndef FROGMATCH_DEBUG_H_
#define FROGMATCH_DEBUG_H_

#include "frogmatch.h"

#ifdef __cplusplus
extern "C" {
#endif

/*
 * Device-side view of an uploaded image.  Any output pointer may be NULL.
 *   class_lap[8], class_begin[9]; perm[n], scale_sorted[n];
 *   rowop / colop: n_pad x 64 FP16 bit patterns, de-swizzled to plain row-major
 *   (n_pad = n rounded up to 256).
 */
int fm_debug_image(fm_ctx* ctx, uint32_t img, uint32_t* flags, uint32_t* n_classes, float* class_lap,
                   uint32_t* class_begin, float* max_norm2, uint32_t* perm, float* scale_sorted,
                   uint16_t* rowop, uint16_t* colop);

/*
 * Squared-norm statistics of an uploaded image's descriptors (FP32), as the certified bounds use them:
 * min_norm2 / max_norm2 over its keypoints (min_norm2 is NaN for an image without keypoints) and max_delta2, the
 * largest squared norm of the FP16 rounding residual.  Any output pointer may be NULL.
 */
int fm_debug_image_norms(fm_ctx* ctx, uint32_t img, float* min_norm2, float* max_norm2, float* max_delta2);

/*
 * Run the band kernel and ONE unit (256 sorted rows starting at row_block * 256 of image
 * `second` against the band of image `first`) of the tensor-core scoring kernel in dump mode.
 *   t_out    : 256 x ld floats, t_out[r * ld + col] = raw score of (unit row r, sorted column col);
 *              columns of tiles the unit did not visit stay NaN.  ld >= n_pad(first).
 *   bands_out: min(256, rows left) x 2 uint32 (lo, hi) sorted-column interval per unit row
 *   cand_t / cand_col: rows x 8 captured candidates (unsorted, -inf padded; slot 0 = +inf marks an
 *              overflowed list), columns are sorted positions in image `first`
 */
int fm_debug_score_unit(fm_ctx* ctx, uint32_t first_img, uint32_t second_img, uint32_t row_block, float* t_out,
                        uint32_t ld, uint32_t* bands_out, float* cand_t, uint32_t* cand_col);

/*
 * The wide tensor-core path (descriptor lengths d != 48, d <= 4096): run the band kernel and ONE unit (128 sorted rows
 * starting at row_block * 128 of image `second` against the band of image `first`) of the wide scoring kernel in dump
 * mode.  Any output pointer may be NULL.
 *   t_out    : 128 x ld floats, t_out[r * ld + col] = t~ = fp16(a).fp16(b) - |b|^2/2 of (unit row r, sorted column col)
 *              for every column the unit's MMAs computed (the steps it visited, trimmed to its band union in
 *              16-column pieces); NaN elsewhere.  ld >= n_pad(first).
 *   bands_out: min(128, rows left) x 2 uint32 (lo, hi) sorted-column interval per unit row
 *   cand_t / cand_col: rows x 8, the row's 8 largest gated scores, descending (-inf padded); columns are sorted
 *              positions in image `first`, bit 31 of slot 0 set when the row had more than 8 gated columns
 *   eps_out  : the task's certified bound on |t~ - t_ref|;  k_pad_out: K_pad = d rounded up to 64
 * Returns FM_ERR_INVALID for d = 48 or d > 4096.
 */
int fm_debug_wide_unit(fm_ctx* ctx, uint32_t first_img, uint32_t second_img, uint32_t row_block, float* t_out,
                       uint32_t ld, uint32_t* bands_out, float* cand_t, uint32_t* cand_col, float* eps_out,
                       uint32_t* k_pad_out);

/*
 * What the reject pass of two-phase scoring computed for one task of the most recent fm_match, which must have run
 * with the option "reject_dump" set.  Task p is pair p; with FM_FLAG_SYM pair p is tasks 2p and 2p + 1.  Rows are
 * the sorted positions of the task's row image (image `second`, or `first` for task 2p + 1), n_rows of them.  Any
 * output pointer may be NULL.
 *   args       : n_rows x 4 floats, the arguments of the row's certified rejection test -- a1 (>= the best score),
 *                a2 (<= the second best score), the row's |a|^2 and the task's eps -- or 4 NaNs for a row whose
 *                gate band is empty
 *   rowstat    : n_rows bytes, 1 = rejected
 *   bands      : n_rows x 2 uint32 (lo, hi) interval of gated-in sorted columns
 *   survivors  : sorted positions of the rows that survived, ascending (room for n_rows); *n_survivors of them
 * Returns FM_ERR_INVALID for a task that did not go through the reject pass (exact-flagged, or the call scored in
 * a single pass) and for an n_rows that is not the task's row count.
 */
int fm_debug_reject_rows(fm_ctx* ctx, uint32_t task, uint32_t n_rows, float* args, uint8_t* rowstat, uint32_t* bands,
                         uint32_t* survivors, uint32_t* n_survivors);

/*
 * Run ONE batch's compaction (the last device stage of fm_match: accepted rows -> dense per-pair lists) on
 * caller-given data, through the launch routine fm_match uses, with the context's own scratch and look-back state
 * (status words and launch epoch counter), so hook calls and fm_match calls share them as production calls do.
 *   rowres[n_rows]   matched column per row, or 0xFFFFFFFF (no match)
 *   rowdist[n_rows]  squared distance per row, or NULL for a compaction without distances
 *   chunks[n_chunks * 4]  the 16-byte chunk records {row_abs, n_rows | swap << 31, row_local, pair} in output order
 *                    (n_rows <= 4096; rows of rowres that no chunk covers are ignored)
 *   path             FM_COMPACT_AUTO (fm_match's choice), FM_COMPACT_ONE (one launch, <= 1536 chunks),
 *                    FM_COMPACT_THREE (count / scan / scatter, version set by the "compact_v" option) or
 *                    FM_COMPACT_LOOKALL (one launch in which every chunk looks back all the way to chunk 0)
 *   base             matches written before this batch (the running total on entry)
 *   out_pairs[out_slots * 2], out_dist[out_slots] (out_dist required with rowdist): in/out -- uploaded first, so
 *                    slots outside [base, base + matches) come back as the caller left them unless a kernel wrote there
 *   pair_counts[n_pairs]  in/out: each chunk's matches are added to its pair's count
 *   total_out        running total after the call (may be NULL)
 *   status_out[1536] the one-pass look-back status words after the call (may be NULL)
 *   epoch_inout      in/out launch epoch counter of the context (may be NULL); the next one-launch call uses
 *                    *epoch_inout % (2^30 - 2) + 1
 * Returns FM_ERR_INVALID, before any launch, for a chunk of more than 4096 rows, one reaching past n_rows or naming a
 * pair >= n_pairs, no chunks, a one-launch path with more than 1536 chunks, or base + matches > out_slots.
 */
#define FM_COMPACT_AUTO 0
#define FM_COMPACT_ONE 1
#define FM_COMPACT_THREE 2
#define FM_COMPACT_LOOKALL 3
int fm_debug_compact(fm_ctx* ctx, const uint32_t* rowres, const float* rowdist, uint32_t n_rows, const uint32_t* chunks,
                     uint32_t n_chunks, int path, uint64_t base, uint32_t* out_pairs, float* out_dist, uint64_t out_slots,
                     uint32_t* pair_counts, uint32_t n_pairs, uint64_t* total_out, uint64_t* status_out,
                     uint32_t* epoch_inout);

/*
 * Experiment switches for kernel studies (process-wide; the defaults are the production configuration):
 *   "probe"     1 | 2   timing-attribution builds of the scoring kernel -- results are GARBAGE
 *   "variant"   n       experiment builds of the scoring kernel -- results stay exact
 *   "pre_tiles" n       look-ahead depth of the scoring kernel (-1 = built-in default)
 *   "two_phase" -1|0|1  two-phase scoring (reject pass + capture pass): library's choice / never / whenever applicable
 *                       -- results are exact either way
 *   "surv_cap"  n       survivor units the capture pass may use per batch (-1 = built-in); a small value forces the
 *                       overflow route (surplus survivors go to the exact row kernel)
 *   "compact_v" 3|2|1   version of the three-launch compaction (batches of more than 1536 chunks) -- results stay exact
 *   "reject_dump" 0|1   two-phase scoring: keep what the reject pass computed for fm_debug_reject_rows (a dump build
 *                       of the reject kernel and a synchronisation per batch) -- results stay exact
 *   "group_repeat" 0|1  fm_group_create accepts a device more than once, one context per entry, so that the whole group
 *                       path (sharding, gather, ordering) runs on one GPU -- results stay exact
 * Returns FM_ERR_INVALID for an unknown name.  Nothing reads environment variables.
 */
int fm_debug_set_option(const char* name, int value);

#ifdef __cplusplus
}
#endif
#endif /* FROGMATCH_DEBUG_H_ */
