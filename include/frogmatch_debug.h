/*
 * frogmatch_debug.h -- test hooks of libfrogmatch.so.  NOT part of the drop-in boundary: these
 * exist so tests/ can check each device stage (sort + class table, FP16 operand packing, the
 * tcgen05 score tile, gate bands, candidate capture) against numpy in isolation.
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
 * Experiment switches for kernel studies (process-wide; the defaults are the production configuration):
 *   "probe"     1 | 2   timing-attribution builds of the scoring kernel -- results are GARBAGE
 *   "variant"   n       experiment builds of the scoring kernel -- results stay exact
 *   "pre_tiles" n       look-ahead depth of the scoring kernel (-1 = built-in default)
 *   "two_phase" -1|0|1  two-phase scoring (reject pass + capture pass): library's choice / never / whenever applicable
 *                       -- results are exact either way
 *   "surv_cap"  n       survivor units the capture pass may use per batch (-1 = built-in); a small value forces the
 *                       overflow route (surplus survivors go to the exact row kernel)
 * Returns FM_ERR_INVALID for an unknown name.  Nothing reads environment variables.
 */
int fm_debug_set_option(const char* name, int value);

#ifdef __cplusplus
}
#endif
#endif /* FROGMATCH_DEBUG_H_ */
