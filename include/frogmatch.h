/*
 * frogmatch.h -- C ABI of libfrogmatch.so, the B200 (sm_100a) keypoint matcher.
 *
 * This is the drop-in boundary for the hot path of valette/FROG's `bin/match`
 * (reference: match/match.cpp).  The reference has no in-process plugin API for this path -- its
 * boundary is the `match` executable and the files on either side (SURVEY.md 8b) -- so this ABI
 * is cut at the seam the reference's own main() has: one call per group of image pairs where the
 * reference calls ComputeMatches() once per image pair (match.cpp:638-652).
 *
 * Conventions: plain C, plain pointers and sizes.  Every function returns FM_OK (0) or a negative
 * fm_status and never throws.  Input pointers are borrowed for the duration of the call; results
 * are owned by the library until fm_result_free().  A context is bound to ONE CUDA device and
 * must be used from one host thread at a time; multi-GPU callers either create one context per device
 * (one per thread or one per process/rank) and shard image pairs between them -- image pairs are
 * independent (match.cpp:638-652), so no data-path collective is needed -- or use one fm_group (below),
 * which does that in-process and gathers the lists on one GPU.
 *
 * There is NO CPU fallback: without a CUDA device fm_create() fails with FM_ERR_CUDA.
 */
#ifndef FROGMATCH_H_
#define FROGMATCH_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct fm_ctx fm_ctx;
typedef struct fm_result fm_result;

typedef enum fm_status {
  FM_OK = 0,
  FM_ERR_INVALID = -1, /* bad argument (null pointer, unknown image, D mismatch, ...) */
  FM_ERR_CUDA = -2,    /* CUDA runtime error; text in fm_last_error() */
  FM_ERR_NOMEM = -3,   /* host or device allocation failed */
  FM_ERR_UNSUPPORTED = -4 /* option the reference has but this build rejects (e.g. -d > 1.8e19) */
} fm_status;

/* fm_match flags */
#define FM_FLAG_SYM 1u          /* also run the reverse direction and append it: -sym, match.cpp:643-646 */
#define FM_FLAG_FORCE_EXACT 2u  /* score every pair with the exact FP32 brute-force kernel only */
#define FM_FLAG_DEVICE_ONLY 4u  /* leave the compacted lists in device memory (fm_result_fetch() copies later) */
#define FM_FLAG_MATCH_ALL 16u    /* the reference's -all mode, bug-compatible (match.cpp:295-300): every gated-in column under
                                 * `dist` emits a pair naming the running nearest column that was NOT under it; dist2second is
                                 * ignored; lists can hold up to N_first * N_second pairs.  Exact FP32 kernels only. */
#define FM_FLAG_DISTANCES 32u    /* also keep, per emitted match, the squared distance d1 the decision was taken on -- the
                                 * value the reference's norm() returns for that pair (match.cpp:243-251, :293).  pairs.bin
                                 * carries no distances; this is the side output the parity checks compare.  Ignored with
                                 * FM_FLAG_MATCH_ALL. */
#define FM_FLAG_ASYNC 8u        /* return as soon as the work is queued on the context's stream; fm_result_wait()
                                 * completes the result.  Several results may be in flight on one context.  (Images
                                 * uploaded since the previous fm_match are prepared first, and the call waits for
                                 * that; FM_FLAG_MATCH_ALL sizes its lists on the host and is synchronous.) */
#define FM_FLAG_ROW_TABLE 64u   /* also keep, in device memory owned by the result, one fm_row per outer-loop row of the
                                 * call (below), so that fm_result_select() can re-decide the call at other thresholds
                                 * without scoring again.  The lists at the call's own thresholds are unchanged.  Costs
                                 * 12 bytes of device memory per row -- sum of N_second (+ N_first with FM_FLAG_SYM)
                                 * over the pairs: 200 images x 20 000 keypoints, all ordered pairs, is 3.98e8 rows =
                                 * 4.8 GB -- and scoring time: no row may be rejected from its approximate scores alone,
                                 * because that test takes the thresholds, so the call scores in one pass and evaluates
                                 * the exact distances of every row with a gated-in column.  FM_ERR_NOMEM (context
                                 * still usable) when the table does not fit; FM_ERR_INVALID with FM_FLAG_MATCH_ALL. */

/* One row of a row table (FM_FLAG_ROW_TABLE): the three values ComputeMatches' accept test reads (match.cpp:262-321),
 * none of which depends on -d or -d2.  d1 and d2 are the exact nearest and second-nearest squared distances over the
 * gated-in columns (FLT_MAX where the reference leaves them at FLT_MAX); nearest is the original index of the nearest
 * column (the lowest one on ties), 0xFFFFFFFF when no column got below FLT_MAX -- in particular when none passes the
 * gates.  The row is accepted at (dist, dist2second) iff
 *   nearest != 0xFFFFFFFF && (sqrtf(d1 / d2) < dist2second || d2 == FLT_MAX) && sqrtf(d1) < dist. */
typedef struct fm_row {
  float d1;
  float d2;
  uint32_t nearest;
} fm_row;

/* ---- context --------------------------------------------------------------------------------- */

/* Number of CUDA devices this process can see (0 and FM_ERR_CUDA when there is none). */
int fm_device_count(int* n);
/* Create a context on CUDA device `device`.  Replaces: process start-up of bin/match. */
int fm_create(int device, fm_ctx** out);
/* Destroy a context.  Every fm_result it produced must have been freed first (a result returns its buffers to its
 * context in fm_result_free). */
void fm_destroy(fm_ctx* ctx);
/* Text of the most recent error on this context (or, with ctx == NULL, of the last failed
 * fm_create on this thread).  Never NULL. */
const char* fm_last_error(const fm_ctx* ctx);
/* Run all of this context's work on the caller's CUDA stream (a cudaStream_t) instead of the
 * context's own; lets a host framework time or order the work with its own events. */
int fm_set_stream(fm_ctx* ctx, void* cuda_stream);
/* Block until everything queued on the context's stream has finished. */
int fm_synchronize(fm_ctx* ctx);

/* ---- keypoint upload ------------------------------------------------------------------------- */

/*
 * Upload image `img`'s keypoints (post-prune order = the ids pairs.bin carries, match.cpp:711-723)
 * and build its device-resident tensors.  Replaces: the AoS `Points` vector the readers build
 * (match.cpp:39-48, 51-92, 137-208).
 *   desc  : n x d floats, row-major (Point::desc)
 *   scale : n floats (Point::scale)          lap : n floats (Point::laplacianSign)
 * Host memory (pageable or pinned) or DEVICE memory of the context's GPU -- e.g. keypoints that reached this GPU over
 * NVLink from the rank that read them; the direction is inferred from the pointers.  Copies are queued on the
 * context's stream, so pinned and device buffers must stay valid until the next fm_synchronize() / fm_match() on
 * this context (pageable buffers may be reused as soon as the call returns).  Re-uploading an index replaces the image.  All images of one
 * context must share d (match.cpp:575 prints one descriptor size for the group).  d = 48 (SURF3D) runs on the
 * tensor-core path; any other d (surf3d -type 1/2: 24 r^3 or 8 r^3 values) on the exact FP32 kernels.
 */
int fm_upload_image(fm_ctx* ctx, uint32_t img, const float* desc, const float* scale, const float* lap,
                    uint32_t n, uint32_t d);
/* Drop all images (device memory is kept for reuse). */
int fm_clear_images(fm_ctx* ctx);
int fm_image_points(const fm_ctx* ctx, uint32_t img, uint32_t* n);

/* ---- matching -------------------------------------------------------------------------------- */

/*
 * Match `n_pairs` image pairs.  For pair p this computes exactly what
 *   ComputeMatches(*allPoints[pair_first[p]], *allPoints[pair_second[p]], dist, dist2second, ...)
 * returns (match.cpp:255-336, called at :642): for every keypoint of image `second`, the nearest
 * and second-nearest keypoints of image `first` among those passing the Laplacian-sign and
 * scale-ratio gates, accepted iff (sqrt(d1/d2) < dist2second || only one candidate) &&
 * sqrt(d1) < dist.  Result p is the list of (first_idx, second_idx) uint32 pairs ordered by
 * second_idx; with FM_FLAG_SYM the reverse-direction list (ordered by first_idx) is appended.
 * Results are in submission order.  The accepted set is bit-identical to the reference's.
 */
int fm_match(fm_ctx* ctx, const uint32_t* pair_first, const uint32_t* pair_second, size_t n_pairs,
             float dist, float dist2second, uint32_t flags, fm_result** out);

/* Complete a result of an FM_FLAG_ASYNC call: block until its kernels have finished, read the
 * per-pair counts and (unless FM_FLAG_DEVICE_ONLY) copy the lists to pinned host memory.  A no-op
 * for results of synchronous calls.  The device views below are valid (in stream order) without it. */
int fm_result_wait(fm_result* r);

size_t fm_result_num_pairs(const fm_result* r);
/* Total matches over all pairs (device-only results included).  Counts and totals are valid once
 * fm_match returned, or, for FM_FLAG_ASYNC calls, once fm_result_wait() returned (0 before). */
uint64_t fm_result_total(const fm_result* r);
/* Number of matches of pair p (MatchVect::size(), match.cpp:734). */
uint32_t fm_result_count(const fm_result* r, size_t p);
/* Host pointer to pair p's matches: 2 * count uint32, (first, second) interleaved -- the bytes
 * match.cpp:738 writes.  NULL until fetched when FM_FLAG_DEVICE_ONLY was used. */
const uint32_t* fm_result_pairs(const fm_result* r, size_t p);
/* With FM_FLAG_DISTANCES: host pointer to pair p's `count` squared distances, in list order.  NULL otherwise, or
 * until fetched. */
const float* fm_result_distances(const fm_result* r, size_t p);
/* Copy a device-only result to (pinned) host memory. */
int fm_result_fetch(fm_result* r);
/* Device views, for callers that gather match lists GPU-to-GPU (NCCL) before the host copy:
 * counts = n_pairs uint32; pairs = 2 * total uint32, pair p's list starting at the exclusive
 * prefix sum of counts. */
const uint32_t* fm_result_device_counts(const fm_result* r);
const uint32_t* fm_result_device_pairs(const fm_result* r);
/* Free a result.  A result with a row table waits for the work queued on its context's stream (fm_result_select calls
 * on it included) before it releases the table. */
void fm_result_free(fm_result* r);

/* ---- re-deciding a call at other thresholds (FM_FLAG_ROW_TABLE) ---------------------------------------------------- */

/*
 * A new, independent result holding exactly the lists (and, with FM_FLAG_DISTANCES, distances) fm_match would return
 * at (dist, dist2second) for the pairs and -sym choice of the call that produced `r`, in the same submission order --
 * computed from r's row table (one pass over the table, then the same compaction fm_match runs), without scoring.
 * `r` must hold a row table: a result of fm_match or fm_group_match with FM_FLAG_ROW_TABLE.  flags: any of
 * FM_FLAG_DISTANCES, FM_FLAG_DEVICE_ONLY and FM_FLAG_ASYNC, with fm_match's meaning.  The work is queued on r's
 * context stream(s) behind r's own work; r may be freed as soon as this returns.  The new result has no row table;
 * fm_result_stats and fm_links_build (with the pair arrays of r's call) take it.  FM_ERR_INVALID for other flags, a
 * result without a table or NaN thresholds; FM_ERR_UNSUPPORTED for dist >= 1.8e19, as fm_match.
 */
int fm_result_select(const fm_result* r, float dist, float dist2second, uint32_t flags, fm_result** out);
/* The row table of r on its device: pair p's rows start at fm_result_row_offset(r, p) -- N_second rows in the original
 * keypoint order of image `second`, then, with FM_FLAG_SYM, the reverse direction's N_first rows.  Valid in stream order
 * (synchronise, or wait for the result, before reading it from another stream).  NULL without a table, and for a result
 * of a group of several devices, whose table is split over the members (fm_result_rows_copy reads it). */
const fm_row* fm_result_rows_device(const fm_result* r);
/* First row of pair p in the table, in submission order over the whole call (also for group results); p == n_pairs gives
 * the number of rows.  UINT64_MAX without a table or for p > n_pairs. */
uint64_t fm_result_row_offset(const fm_result* r, size_t p);
/* Copy pair p's rows (fm_result_row_offset(r, p + 1) - fm_result_row_offset(r, p) of them) to host memory `dst`; waits
 * for the work that writes them. */
int fm_result_rows_copy(fm_result* r, size_t p, fm_row* dst);

/* ---- consumer hand-off ------------------------------------------------------------------------ */

/*
 * Build, on the device, the adjacency `bin/frog` builds when it reads pairs.bin -- ImageGroup::readPairs,
 * registration/imageGroup.cxx:1386-1411: for every entry (p1, p2) of the block of images (image1, image2),
 * {image2, p2} is appended to image1's point p1 and {image1, p1} to image2's point p2 (Point::links,
 * registration/point.h:11-28) -- from the match lists of a finished fm_match, so that a consumer in the same
 * process never reads the file back.  Every point's links come out in the reference's push_back order (blocks in
 * file order, entries in list order), which its statistics depend on.
 *   pair_first / pair_second : the arrays fm_match was called with (n_pairs = fm_result_num_pairs)
 *   block_order              : the order in which the pair blocks appear in pairs.bin (match.cpp:727-742: row-major
 *                              over (first, second)); NULL = submission order
 * The result must be complete (fm_match without FM_FLAG_ASYNC, or fm_result_wait); FM_FLAG_MATCH_ALL results
 * are not supported.  Points are numbered image after image in image-index order over the context's images.
 */
typedef struct fm_links fm_links;
int fm_links_build(fm_result* r, const uint32_t* pair_first, const uint32_t* pair_second, const uint32_t* block_order,
                   fm_links** out);
/* Half-links in all = 2 x matches. */
uint64_t fm_links_total(const fm_links* l);
/* Copy offsets and links to pinned host memory (the device views are valid right after fm_links_build). */
int fm_links_fetch(fm_links* l);
/* Host, after fm_links_fetch: image `img`'s n_points + 1 offsets into fm_links_data (point p's links are entries
 * [off[p], off[p+1])); NULL for an image the context does not hold. */
const uint64_t* fm_links_offsets(const fm_links* l, uint32_t img, uint32_t* n_points);
/* Host, after fm_links_fetch: 2 x total uint32, (image, point) per link. */
const uint32_t* fm_links_data(const fm_links* l);
/* Device views: total_points + 1 offsets (points numbered image after image), and the (image, point) pairs. */
const uint64_t* fm_links_device_offsets(const fm_links* l);
const uint32_t* fm_links_device_data(const fm_links* l);
/* CUDA-event time of the build (count, scan, scatter, per-point ordering), milliseconds. */
float fm_links_build_ms(const fm_links* l);
void fm_links_free(fm_links* l);

/* ---- instrumentation ------------------------------------------------------------------------- */

typedef struct fm_stats {
  uint64_t descriptor_pairs;  /* sum over tasks of N_first * N_second (match.cpp:262-267 trip count) */
  uint64_t scored_pairs;      /* descriptor pairs the scoring kernel actually evaluated */
  uint64_t rows;              /* outer-loop rows processed */
  uint64_t rows_exact;        /* rows (re)done by the exact brute-force kernel */
  uint64_t candidates;        /* candidates rescored in exact FP32 */
  uint64_t kernel_launches;   /* kernels launched by the last fm_match */
  uint64_t score_launches;    /* of which: scoring-kernel launches */
  float ms_total;             /* CUDA-event time of the last fm_match, first launch to lists compacted */
  float ms_score;             /* ... of which the scoring kernel(s) */
  float ms_rescore;           /* ... exact rescoring / decision */
  float ms_exact;             /* ... exact brute-force kernel */
  float ms_compact;           /* ... stream compaction */
  float ms_prep;              /* CUDA-event time of all uploads' prep kernels since the last clear */
  uint64_t rows_rejected_early; /* rows proven unacceptable from their approximate scores (no exact distance evaluated) */
  uint64_t two_phase_batches;   /* batches scored in two phases (reject pass, then capture pass for the surviving rows' warps) */
} fm_stats;

/* Statistics of the most recent fm_match on this context (synchronises the stream). */
int fm_get_stats(fm_ctx* ctx, fm_stats* out);
/* Statistics of the call that produced `r` (waits for it; ms_prep is not attributed to a call: 0).  For a result of
 * fm_group_match the counters are summed over the members' calls and each ms_* field is the maximum over members. */
int fm_result_stats(fm_result* r, fm_stats* out);

/* ---- device groups: one library handle over several GPUs --------------------------------------------------------- */

/*
 * A group is one fm_ctx per device, used as one: every member holds every image, fm_group_match splits the pairs over
 * the members and gathers their lists over NVLink into one result on the LEAD device (devices[0]), in submission
 * order.  Like a context, a group is used from one host thread at a time.
 */
typedef struct fm_group fm_group;
/* Create a group over `n` distinct devices; devices[0] is the lead.  Enables peer access between every ordered pair of
 * members that supports it (process state, left enabled by fm_group_destroy); every member must be able to access the
 * lead.  FM_ERR_INVALID for a repeated or out-of-range device, FM_ERR_UNSUPPORTED when a member cannot access the lead
 * as a peer, FM_ERR_CUDA without a device; the text is in fm_group_last_error(NULL).  A group of one device behaves
 * exactly like fm_create(devices[0]). */
int fm_group_create(const int* devices, int n, fm_group** out);
/* Destroy a group.  Every fm_result it produced must have been freed first. */
void fm_group_destroy(fm_group* g);
/* Text of the most recent error on this group (NULL: of the last failed fm_group_create on this thread).  Never NULL. */
const char* fm_group_last_error(const fm_group* g);
/* Block until every member's queued work has finished. */
int fm_group_synchronize(fm_group* g);
int fm_group_clear_images(fm_group* g);
/* fm_upload_image on every member (same arguments and checks).  The image is copied once to its owner: member img % n
 * for a host image, the member on the image's GPU for device memory (the lead when it cannot access the owner as a
 * peer, or for device memory outside the group).  Every other member then copies, GPU to GPU, the device copy of a
 * member it can access as a peer: the owner's, otherwise the lead's.  So a host image crosses PCIe once.  Pinned and
 * device buffers must stay valid until the next fm_group_synchronize / fm_group_match. */
int fm_group_upload_image(fm_group* g, uint32_t img, const float* desc, const float* scale, const float* lap, uint32_t n,
                          uint32_t d);
/* fm_match over the group, with the same arguments and flags.  Pairs are split longest-first by N_first * N_second;
 * each member matches its share; the lists (and distances) are then stored into the lead's memory at their
 * submission-order offsets, all in stream order.  The result is an ordinary fm_result of the lead (every fm_result_*
 * call and fm_links_build take it; link image indices are the lead's, which are all of them), byte-identical to what
 * one context returns for the same call.  Its device views are on the lead.  Members run their shares with
 * FM_FLAG_ASYNC, so a group never probes the first batch of a synchronous call to switch to two-phase scoring within
 * that call (see fm_match): the first call at dist2second < 1 runs single-pass where one context might not, and later
 * calls use each member's rejection rate of its previous call.  Results are exact either way.  The -all row limit
 * applies to the whole call, as for one context.  With FM_FLAG_ROW_TABLE each member keeps the table of its share;
 * fm_result_select on the result selects on every member and gathers the lists on the lead the same way, and
 * fm_result_row_offset / fm_result_rows_copy address the rows in submission order over the whole call. */
int fm_group_match(fm_group* g, const uint32_t* pair_first, const uint32_t* pair_second, size_t n_pairs, float dist,
                   float dist2second, uint32_t flags, fm_result** out);

/* Library/build description, e.g. "frogmatch 0.1 sm_100a". */
const char* fm_version(void);

#ifdef __cplusplus
}
#endif
#endif /* FROGMATCH_H_ */
