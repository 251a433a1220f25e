/*
 * icpb -- batched 2-D point-to-point ICP scan matching on B200 (sm_100a): C ABI.
 *
 * This is the drop-in boundary for the reference's ICP path.  The reference has no FFI: the
 * path is the module-level Python functions of src/icp.py, fanned out over scan pairs by
 * joblib.  Each entry point below names the reference interface it replaces
 * (paths relative to the reference tree).  INTEGRATION.md shows the ctypes binding a
 * reference maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success, a non-zero status otherwise (a cudaError_t value,
 *     or one of the ICPB_E* codes); nothing throws across the ABI; icpb_last_error() returns
 *     a per-thread message for the last failure.
 *   - scans are (m_i, 2) float64 rows in one concatenated table with int64 CSR offsets -- the
 *     arrays the reference's dataloader returns (src/dataloader.py:47-55,110-112), before the
 *     callers append the homogeneous column of ones (scripts/main.py:242-243).
 *   - a transform is the top 2x3 of the reference's 3x3 SE(2) matrix, row-major, float64:
 *     [r00 r01 tx r10 r11 ty]; the bottom row is always [0 0 1] (src/icp.py:41-44,67).
 *   - pairs[b] = (source scan id, target scan id): the source is moved onto the target, the
 *     reference's icp(pc1=source, pc2=target) (src/icp.py:72-76).
 *   - pointers named d_* are device pointers on the handle's device, h_* host pointers.
 */
#ifndef ICPB_H
#define ICPB_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ICPB_ABI_VERSION 2

#define ICPB_EINVAL   10001   /* bad argument (null pointer, empty scan, negative size ...)   */
#define ICPB_ETOOLONG 10002   /* a scan beyond the kernel's 32-bit layout offsets (~100 M points);
                                 scans that do not fit shared memory run on the large-scan variant */
#define ICPB_ENOSCANS 10003   /* run called before a scan table was set                       */

/* Input magnitudes.  The alignment kernel pads target arrays with points at (1e15, 1e15) and filters
 * in fp32; within these bounds every moved source point stays below 6e13 in every pass, so a real
 * target is always far nearer than any padding point (squared distances <= 7e27 against >= 1.7e30)
 * and no fp32 square overflows (DESIGN.md section 4 has the arithmetic).  The results are exact for
 * every input within them:
 *   - scan coordinates:                      |x|, |y| <= ICPB_MAX_COORD;
 *   - the linear part of an initial guess:   |r00|, |r01|, |r10|, |r11| <= ICPB_MAX_GUESS_LINEAR
 *     (any affine map: shear, reflection, rank-deficient and zero linear parts included);
 *   - the translation of an initial guess:   |tx|, |ty| <= ICPB_MAX_GUESS_SHIFT.
 * A coordinate or guess outside them (NaN and inf included) is rejected with ICPB_EINVAL where the
 * library reads the values on the host: scans by icpb_align_host_scans (and the list form of
 * icpb_align_host_accept) while packing, guesses by the icpb_align_host* calls before anything runs.
 * The Python layer checks every entry point.  Entry points that take device buffers, and the packed
 * tables of the host calls, take the caller's word for it. */
#define ICPB_MAX_COORD        1e10
#define ICPB_MAX_GUESS_LINEAR 1e3
#define ICPB_MAX_GUESS_SHIFT  1e12
/* The smallest nonzero cell size of the submap voxel filter (icpb_set_submaps_voxel): with
 * |x| <= ICPB_MAX_COORD it keeps |x / voxel| <= 1e16, so every cell coordinate is exact in int64. */
#define ICPB_MIN_VOXEL        1e-6

/* Occupancy grid (icpb_occupancy_grid_*).  The Bresenham walk runs in 64-bit integers on cell
 * coordinates; with every |cell coordinate| <= ICPB_MAX_GRID_CELL = 2^60 a beam spans
 * M = max(|dx|, |dy|) <= 2^61 cells, the walk's error term stays within 1.5 M and `2 * error` within
 * 3 * 2^61 < 2^63, so the walk visits exactly the reference's cells (DESIGN.md section 4).  The update
 * checks this on the host before anything runs, from the poses and the grid origin alone (a global
 * beam end lies within sqrt(2) * ICPB_MAX_COORD of its pose):
 *     (max |pose x|, |pose y| + max(|min_x|, |min_y|) + sqrt(2) * ICPB_MAX_COORD) / cell_width <= 2^60
 * With coordinates of 1e10 m this rejects only cell widths below about 1.2e-8 m.  Non-finite poses,
 * min_x, min_y, min_width, min_height and cell widths are rejected by both calls, and so is a grid of
 * more than ICPB_MAX_GRID_CELLS cells: icpb_occupancy_grid_bounds reports it before a caller
 * allocates one. */
#define ICPB_MAX_GRID_CELL  1152921504606846976.0   /* 2^60 */
#define ICPB_MAX_GRID_CELLS 1073741824LL            /* 2^30: height * width */

/* Loop-closure candidates (icpb_proximity_*).  Pose coordinates |x|, |y| <= ICPB_MAX_POSE_COORD keep
 * every squared distance below 8e24, far from overflow, so every row with a candidate range finds its
 * nearest pose.  Both calls reject with ICPB_EINVAL: a pose outside the bound (NaN and inf included),
 * a `travelled` array that is not finite and non-decreasing (the row start is a binary search in it),
 * and a NaN min_dist_along_path. */
#define ICPB_MAX_POSE_COORD 1e12

/* icpb_params.flags: sweep every target for every source point (the reference's brute force,
 * src/icp.py:10-19) instead of skipping target chunks that provably cannot hold a nearest
 * neighbour.  Results are identical either way; the flag exists to measure the FP32-pipe
 * roofline of the unpruned sweep. */
#define ICPB_FLAG_EXHAUSTIVE 1

typedef struct icpb_ctx *icpb_handle;

/* Keyword arguments of the reference's icp() (src/icp.py:72) plus batch bookkeeping. */
typedef struct icpb_params {
    double  epsilon;          /* stop when error < epsilon               (src/icp.py:86)      */
    double  stopping_thresh;  /* stop when |last_err - err| < this       (src/icp.py:91-95)   */
    int32_t max_iters;        /* stop when iteration > max_iters: up to max_iters+2 passes (:88) */
    int32_t rotation_only;    /* zero the translation every pass         (src/icp.py:60-61,65-66) */
    int32_t hist_cap;         /* transforms recorded per problem in hist (0 = none)           */
    int32_t corr_stride;      /* int32 slots per problem in corr (0 = none); >= longest source */
    int32_t pair_mode;        /* 0: explicit pairs array; 1: all pairs i<j of n_scans, source=j,
                                 target=i (the argument order of src/loop_closure_detection.py:31-34),
                                 decoded on the device from a linear index                    */
    int32_t flags;            /* ICPB_FLAG_* bits                                             */
    /* pair_mode 1 and sharding: problem b of this call is global index
       k = k_first + (b / k_block) * k_stride + (b % k_block); with pair_mode 0 and pairs given
       for this shard only, leave k_first = 0, k_block = B, k_stride = 0.                      */
    int64_t k_first, k_block, k_stride;
} icpb_params;

/* Fills the reference's icp() defaults: epsilon 0.01, max_iters 100, stopping_thresh 1e-4,
 * rotation_only 0 (src/icp.py:72); no history, no correspondences, explicit pairs. */
void icpb_default_params(icpb_params *p);

int icpb_abi_version(void);

/* Per-process, per-device state: the staged scan table, the work-queue counter, scratch
 * buffers for the host-pointer entry point.  Replaces "a loky worker process"
 * (scripts/main.py:240, src/loop_closure_detection.py:134). */
int icpb_create(int device, icpb_handle *out);
int icpb_destroy(icpb_handle h);

/* Scan table = the reference's `lidar_points` list (src/dataloader.py:110-112), concatenated.
 * icpb_upload_scans copies host arrays into device memory owned by the handle;
 * icpb_set_scans_device borrows device arrays the caller keeps alive (call it again after changing
 * their contents: the first launch on a resident table derives per-scan staging data from it, once).
 * offsets has n_scans + 1 entries, offsets[0] = 0. */
int icpb_upload_scans(icpb_handle h, const double *h_xy, const int64_t *h_offsets, int64_t n_scans);
int icpb_set_scans_device(icpb_handle h, const double *d_xy, const int64_t *d_offsets,
                          int64_t n_scans, int64_t longest_scan);

/*
 * Submaps: scans of the resident table merged on the device into new scans appended to it -- the target of
 * scan-to-submap matching (a revisiting scan aligned onto scan i together with its neighbours, placed by the
 * current poses, instead of onto scan i alone).  The base table is the one last set by icpb_upload_scans,
 * icpb_set_scans_device or an icpb_align_host* call, with n_base scans.
 *   h_submap_off  n_submaps + 1 offsets into h_members: [0] = 0, strictly increasing (every submap has a member)
 *   h_members     base scan ids in [0, n_base); a scan may be a member of several submaps, and more than once of one
 *   h_member_T    one 2x3 transform per member (6 doubles, the usual row layout): it maps the member's points into
 *                 the submap's frame
 * Submap m becomes scan n_base + m of the resident table: its members' points in member order, each mapped as
 *     x' = (T00*x + T01*y) + T02        y' = (T10*x + T11*y) + T12
 * with every product and sum rounded to nearest on its own (no FMA contraction; numpy's element-wise * and +
 * give the same bits), so a submap can be restated on the host and every alignment against it checked bit for
 * bit.  Every entry point that reads the resident table sees the submaps (icpb_run_host, icpb_run_device*,
 * icpb_run_multistart_host, pair_mode 1 over the whole table), and icpb_scan_count reports n_base + n_submaps.
 * A call replaces the submaps of the previous call; n_submaps = 0 goes back to the base table alone.  A call
 * that sets a new table drops the submaps.
 * Memory: the table with its submaps is one table in memory the handle owns.  A borrowed base
 * (icpb_set_scans_device) is copied there, and from then on the handle no longer reads the caller's buffers
 * (they are never written); call icpb_set_scans_device again after changing them.  A table whose longest
 * submap does not fit shared memory gets no staging images: its short pairs stage per pair, like those of
 * any table holding scans beyond shared memory.
 * Rejected before anything is written, leaving the resident table (submaps included) as it was:
 *   ICPB_ENOSCANS  no table is set;
 *   ICPB_EINVAL    null pointers, a negative count, bad offsets, a member id outside the base table (a submap
 *                  id included), a transform outside the guess bounds (ICPB_MAX_GUESS_LINEAR / _SHIFT, NaN
 *                  included), and any merged coordinate beyond ICPB_MAX_COORD -- scans and transforms within
 *                  their bounds can still merge to coordinates of ~2e13; the device tests every merged point in
 *                  a pass of its own before the table is written;
 *   ICPB_ETOOLONG  a submap beyond the alignment kernel's 32-bit layout offsets (~100 M points).
 * Synchronous.  Like icpb_upload_scans, it must not overlap an asynchronous icpb_run_device* on the same handle.
 */
int icpb_set_submaps(icpb_handle h, const int32_t *h_members, const int64_t *h_submap_off,
                     const double *h_member_T, int64_t n_submaps);

/*
 * icpb_set_submaps with a voxel filter: each submap is merged exactly as above (the same formula and the same
 * check), then thinned to the first point of every grid cell.  In the submap's own frame the merged point
 * (x', y') lies in cell (cx, cy) = ((int64) floor(x' / voxel), (int64) floor(y' / voxel)), the division
 * correctly rounded (numpy's np.floor(x / v).astype(np.int64) gives the same bits).  A point is kept iff no
 * earlier point of the same submap, in merged order (member order, then point order within a member), lies in
 * the same cell; kept points keep their coordinates bit for bit and their merged order.  Cells are per submap.
 * No averaging: a kept point is a real merged point, so a filtered submap can be restated on the host and every
 * alignment against it checked bit for bit.
 *   voxel         0 (no filter: exactly icpb_set_submaps, which is this call with voxel = 0 and
 *                 h_submap_len = NULL), or a finite cell size >= ICPB_MIN_VOXEL
 *   h_submap_len  NULL, or n_submaps outputs: each submap's length in the table (its kept count), on success
 * icpb_scan_count, the offsets, the longest scan, the staging images and the split by scan length all follow
 * the kept counts: a filtered submap that fits shared memory runs on the shared-memory kernel.
 * Rejected before anything is written, on top of the rejections of icpb_set_submaps: a voxel that is NaN,
 * +-inf, negative, or in (0, ICPB_MIN_VOXEL) (ICPB_EINVAL).  ICPB_ETOOLONG is judged on the merged length,
 * before the filter: a submap beyond ~100 M merged points is refused even if the filter would shrink it.
 * The resident table is written only once the whole filtered result is known.  Device memory: the handle's
 * scratch grows to about 16 B (merged points) + 8-16 B (hash) + 8 B (flags and scan) per merged point.
 * Synchronous; must not overlap an asynchronous icpb_run_device* on the same handle.
 */
int icpb_set_submaps_voxel(icpb_handle h, const int32_t *h_members, const int64_t *h_submap_off,
                           const double *h_member_T, int64_t n_submaps, double voxel,
                           int64_t *h_submap_len /* n_submaps outputs, may be NULL */);

/* The points of resident scans [first, first + count), submaps included, in table order, into h_xy
 * (2 doubles per point; the caller sizes it from the offsets).  ICPB_ENOSCANS without a table; ICPB_EINVAL
 * for a null h_xy or a range outside the table.  Synchronous; like icpb_upload_scans, it must not overlap an
 * asynchronous icpb_run_device* on the same handle. */
int icpb_read_scans(icpb_handle h, int64_t first, int64_t count, double *h_xy);

/*
 * B independent icp() calls (src/icp.py:72-97) in one launch -- replaces the joblib fan-out
 * `Parallel(...)(delayed(icp.icp)(...) for ...)` of scripts/main.py:240-247,
 * src/loop_closure_detection.py:134-142 and src/pose_graph_optimization.py:60-68.
 *   d_pairs   B x 2 int32 (pair_mode 0) or NULL (pair_mode 1)
 *   d_init    B x 6 float64 initial transforms (icp()'s init_transform) or NULL for identity
 *   d_T       B x 6 float64   transforms[-1] of each call
 *   d_err     B     float64   the returned error (SSE under transforms[-2], src/icp.py:68)
 *   d_passes  B     int32     len(transforms) - 1
 *   d_hist    B x hist_cap x 6 float64 or NULL: transforms[1:], rows past the pass count untouched
 *   d_corr    B x corr_stride int32 or NULL: the last pass's correspondences (icp_iteration's
 *             second return value, src/icp.py:63,69)
 * Asynchronous on `stream` (a cudaStream_t, NULL = default stream).
 */
int icpb_run_device(icpb_handle h, const int32_t *d_pairs, const double *d_init, int64_t B,
                    const icpb_params *p, double *d_T, double *d_err, int32_t *d_passes,
                    double *d_hist, int32_t *d_corr, void *stream);

/*
 * Multi-GPU: icpb_run_device with the gather of the constraint records fused into the kernel.
 * d_peer_ptrs is a device array of n_peers pointers: the gather buffer of every rank
 * ((total pairs, 8) float64 rows [T(6), error, passes]) as mapped into THIS process (CUDA peer /
 * symmetric memory).  Each finished pair stores its record into every buffer at row
 * row0 + pair id, over NVLink, instead of a separate all-gather after the kernel.  The caller
 * orders the launch before a cross-rank barrier.  Replaces the result gather of the reference's
 * fan-out, `zip(*parallel(...))` (scripts/main.py:241), across ranks.
 */
int icpb_run_device_gather(icpb_handle h, const int32_t *d_pairs, const double *d_init, int64_t B,
                           const icpb_params *p, double *d_T, double *d_err, int32_t *d_passes,
                           const uint64_t *d_peer_ptrs, int32_t n_peers, int64_t row0, void *stream);

/*
 * What the alignment kernel does with a finished pair besides writing d_T / d_err / d_passes: the
 * exchange step of the multi-GPU path and the acceptance test of the loop-closure callers, as kernel
 * epilogues.  All pointers are device pointers; zero-initialise the struct and fill what is wanted.
 *
 * Fused all-gather (d_peer_ptrs != NULL): the pair's 64-byte record [T(6), error, passes] (8 float64)
 *   is stored into EVERY rank's gather buffer -- d_peer_ptrs is a device array of n_peers addresses,
 *   each rank's (total pairs, 8) float64 buffer as mapped into this process (CUDA peer / symmetric
 *   memory) -- at row  row0 + (b / row_block) * row_stride + b % row_block  for local problem b
 *   (row_block <= 0: rows row0 .. row0 + B - 1).  With row0 = rank * block, row_block = block,
 *   row_stride = world * block this is the interleaved-block partition of the problem index space
 *   (SURVEY.md section 8e), so every rank ends up with all records in global problem order and no
 *   collective runs after the kernel; the caller orders the launch before a cross-rank barrier.
 *   Replaces the result gather of the reference's fan-out, `zip(*parallel(...))`
 *   (scripts/main.py:241), across ranks.
 *
 * Acceptance + compaction (d_accept_rec or d_accept_peer_ptrs != NULL): pairs whose error is below
 *   accept_thresh -- the reference's `if error < err_thresh: add_constraint(...)`
 *   (src/loop_closure_detection.py:35-39, 155-159) -- append [T(6), error, tag] with the int64 tag
 *   (row << 16) | min(passes, 65535) stored in the 8th slot's bits, in completion order, so only
 *   accepted constraints cross PCIe / NVLink.  Single GPU: into d_accept_rec (accept_cap rows), the
 *   number of rows into *d_accept_count when the launch completes.  Multi-GPU: into region `rank`
 *   (rows rank * accept_cap ...) of every peer's buffer d_accept_peer_ptrs[r], the count into slot
 *   `rank` of every peer's int64 array d_accept_count_peer_ptrs[r].  A count above accept_cap is
 *   reported negated (the buffer then holds the first accept_cap rows).  The consumer restores the
 *   reference's order by sorting on the row in the tag.
 */
typedef struct icpb_epilogue {
    const uint64_t *d_peer_ptrs;
    int32_t  n_peers;
    int32_t  rank;
    int64_t  row0, row_block, row_stride;
    double   accept_thresh;
    double  *d_accept_rec;
    int64_t *d_accept_count;
    const uint64_t *d_accept_peer_ptrs;
    const uint64_t *d_accept_count_peer_ptrs;
    int64_t  accept_cap;
} icpb_epilogue;

/* icpb_run_device with epilogues (ep may be NULL); no history / correspondences. */
int icpb_run_device_ex(icpb_handle h, const int32_t *d_pairs, const double *d_init, int64_t B,
                       const icpb_params *p, double *d_T, double *d_err, int32_t *d_passes,
                       const icpb_epilogue *ep, void *stream);

/* Same with host buffers: copies the inputs to the device, runs, copies the results back and
 * synchronises.  This is the call a reference-side binding makes. */
int icpb_run_host(icpb_handle h, const int32_t *h_pairs, const double *h_init, int64_t B,
                  const icpb_params *p, double *h_T, double *h_err, int32_t *h_passes,
                  double *h_hist, int32_t *h_corr);

/*
 * Multi-start alignment on the resident scan table: every pair is aligned from K shared start transforms
 * and the start with the smallest error is returned -- the standard remedy for loop closures whose
 * relative heading is unknown (a corridor driven the other way, an image match between scans taken
 * facing different directions), where a single guess converges to the wrong minimum.
 *   h_pairs   B x 2 int32 (source, target) scan ids, as icpb_run_host
 *   h_init    B x 6 float64 per-pair guesses init[p], or NULL for the identity
 *   h_starts  K x 6 float64 start transforms S[k] (2x3 rows like every guess), 1 <= K <= 2^22
 * Problem (p, k) is exactly icp(scan[src_p], scan[dst_p], G[p,k], epsilon, max_iters, stopping_thresh,
 * rotation_only) with G = init[p] . S[k]: the start acts in the source frame first, so a heading start
 * turns the source scan about its own sensor origin and keeps the translation of init.  G is evaluated
 * in float64, every product and sum rounded to nearest on its own (no FMA contraction), left to right:
 *     G00 = I00*S00 + I01*S10     G01 = I00*S01 + I01*S11     G02 = (I00*S02 + I01*S12) + I02
 *     G10 = I10*S00 + I11*S10     G11 = I10*S01 + I11*S11     G12 = (I10*S02 + I11*S12) + I12
 * (numpy's element-wise * and + give the same bits), so every problem gives the bits icpb_run_host gives
 * for the expanded pair list (pair p repeated K times, guesses G[p, 0..K-1]).  rotation_only zeroes the
 * translation of G, as icp() does with its guess.
 * Outputs per pair: the winning start's h_T (B x 6), h_err and h_passes, and h_start[p] = the smallest k
 * with the smallest error (strict < over ascending k: np.argmin's rule, errors being finite within the
 * bounds above).  Optional (NULL = not wanted): h_err_all (B x K float64) and h_passes_all (B x K int32),
 * the results of every start, for callers that judge how ambiguous a match is.
 * Rejected with ICPB_EINVAL before anything runs (the table stays usable): K outside 1 .. 2^22, null
 * starts, a pair index out of range, hist_cap or corr_stride > 0 (for the winner's history rerun
 * icpb_run_host on the winning guesses: each problem is deterministic, so the results are the same),
 * pair_mode != 0, and any composed guess G outside the guess bounds (!(|v| <= bound), NaN included) --
 * guesses and starts can each be within them while their product is not.
 * The pairs run in slices of floor(2^22 / K) pairs, one alignment launch per slice (two when the table
 * holds scans beyond shared memory and the slice is split by scan length), and a pair's K starts are
 * next to each other in the queue.  Synchronous, like icpb_run_host.
 */
int icpb_run_multistart_host(icpb_handle h, const int32_t *h_pairs, const double *h_init, int64_t B,
                             const double *h_starts, int32_t K, const icpb_params *p,
                             double *h_T, double *h_err, int32_t *h_passes, int32_t *h_start,
                             double *h_err_all, int32_t *h_passes_all);

/* icpb_upload_scans + icpb_run_host in one call with the upload overlapped with the kernels: the
 * scan table is copied in segments and every pair is launched as soon as both of its scans have
 * arrived.  Explicit pairs only, no history / correspondences.  This is what the Python
 * `icp_batch(scans, pairs, ...)` calls: the replacement of the whole
 * `Parallel(...)(delayed(icp.icp)(np.c_[scan_i, 1], np.c_[scan_j, 1], ...) ...)` expression
 * (scripts/main.py:240-247), argument pickling included. */
int icpb_align_host(icpb_handle h, const double *h_xy, const int64_t *h_offsets, int64_t n_scans,
                    const int32_t *h_pairs, const double *h_init, int64_t B, const icpb_params *p,
                    double *h_T, double *h_err, int32_t *h_passes);

/* How icpb_align_host cuts the scan table into upload pieces (pure host logic, no CUDA call; exposed
 * for tests): piece k covers scans [piece_end[k-1], piece_end[k]); piece_end has room for 64 entries;
 * pieces_wanted = 0 picks ~4 MB pieces, at most 16.  Every piece ends on an even point offset (a
 * 32-byte sector of the fp64 table), so no cached sector can mix landed and pending bytes. */
int icpb_plan_upload(const int64_t *h_offsets, int64_t n_scans, int32_t pieces_wanted,
                     int64_t *piece_end, int32_t *n_pieces);

/* The same with the transforms in the caller's own layout: init_ld / T_ld = 9 reads and writes the
 * reference's full 3x3 row-major matrices (what scripts/main.py:244 passes and src/icp.py:97
 * returns; the bottom row is checked to be [0, 0, 1] on the way in and written on the way out),
 * 6 the packed top two rows.  Initial guesses beyond the bounds above (non-finite ones included) are
 * rejected (ICPB_EINVAL). */
int icpb_align_host_ld(icpb_handle h, const double *h_xy, const int64_t *h_offsets, int64_t n_scans,
                       const int32_t *h_pairs, const double *h_init, int32_t init_ld, int64_t B,
                       const icpb_params *p, double *h_T, int32_t T_ld, double *h_err, int32_t *h_passes);

/* icpb_align_host_ld with epilogues: on a multi-GPU run the records go from the kernel straight into
 * every rank's gather buffer while this rank's own results still come back to h_T / h_err / h_passes. */
int icpb_align_host_ex(icpb_handle h, const double *h_xy, const int64_t *h_offsets, int64_t n_scans,
                       const int32_t *h_pairs, const double *h_init, int32_t init_ld, int64_t B,
                       const icpb_params *p, double *h_T, int32_t T_ld, double *h_err, int32_t *h_passes,
                       const icpb_epilogue *ep);

/* The same with the scans exactly as the reference holds them: `lidar_points`, a list of n_scans
 * separate (m_i, 2) float64 C-ordered arrays in ordinary pageable memory (src/dataloader.py:110-112,
 * the arguments of scripts/main.py:242-243).  scan_xy[s] points at scan s, scan_len[s] = m_i.  A few
 * host threads copy the scans into a pinned staging table piece by piece (checking that every
 * coordinate is within ICPB_MAX_COORD on the way: ICPB_EINVAL) while earlier pieces are already on their way to the device and
 * the kernel is aligning the pairs whose scans have landed. */
int icpb_align_host_scans(icpb_handle h, const double *const *scan_xy, const int64_t *scan_len, int64_t n_scans,
                          const int32_t *h_pairs, const double *h_init, int32_t init_ld, int64_t B,
                          const icpb_params *p, double *h_T, int32_t T_ld, double *h_err, int32_t *h_passes,
                          const icpb_epilogue *ep);

/* Upload + align + acceptance test, for the loop-closure callers: the reference aligns every candidate
 * and keeps those with `error < err_thresh` (src/loop_closure_detection.py:35-39 with err_thresh 110,
 * :155-159 with icp_err_thresh 30).  Here the test and the compaction run in the kernel epilogue, and
 * only the accepted constraints come back: h_rows[q] = index into h_pairs (ascending, i.e. the callers'
 * own order), h_T / h_err / h_passes row q its result; *n_accepted their number (<= capacity, else
 * ICPB_EINVAL with the true count stored).  Scans either packed (h_xy, h_offsets) or as a list
 * (scan_xy, scan_len); the other pair of pointers NULL. */
int icpb_align_host_accept(icpb_handle h, const double *h_xy, const int64_t *h_offsets,
                           const double *const *scan_xy, const int64_t *scan_len, int64_t n_scans,
                           const int32_t *h_pairs, const double *h_init, int32_t init_ld, int64_t B,
                           const icpb_params *p, double accept_thresh, int64_t capacity, int64_t *n_accepted,
                           int64_t *h_rows, double *h_T, int32_t T_ld, double *h_err, int32_t *h_passes);

/* One pair given directly as two (n, 2) float64 host arrays: the reference's
 * icp(pc1, pc2, init_transform, epsilon, max_iters, stopping_thresh, rotation_only)
 * (src/icp.py:72) and, with epsilon = +inf (one pass), icp_iteration() (src/icp.py:55-69). */
int icpb_icp_pair_host(icpb_handle h, const double *h_src_xy, int64_t n_src,
                       const double *h_dst_xy, int64_t n_dst, const double *h_init6,
                       const icpb_params *p, double *h_T6, double *h_err, int32_t *h_passes,
                       double *h_hist, int32_t *h_corr);

/* Rigid fit of n matched pairs a[i] -> b[i] ((n, 2) float64 host arrays) and their sum of squared
 * differences: the reference's get_transform(pc1, pc2) (src/icp.py:22-46) and get_error(pc1, pc2)
 * (src/icp.py:49-52), which assume pc1[i] corresponds to pc2[i]. */
int icpb_fit_pairs_host(icpb_handle h, const double *h_a_xy, const double *h_b_xy, int64_t n,
                        double *h_T6, double *h_err);

/*
 * Loop-closure candidate generation: the front half of detect_proximity
 * (src/loop_closure_detection.py:12-25) without the S x S cdist matrix.  h_xy is the (n, 2)
 * position part of pose_graph.poses, h_travelled the reference's dist_traveled array (:13-14:
 * cumulative sum of consecutive distances, first entry 0).  For every pose i, start =
 * searchsorted(travelled, travelled[i] + min_dist_along_path, "right") (:18); h_closest[i] is
 * start + argmin(dist[i, start:]) (:21) if that distance is <= max_dist (:22), else -1 (also
 * when start is past the end, where the reference stops, :19-20).  Inputs are checked against
 * ICPB_MAX_POSE_COORD and the rules beside it before anything runs.
 */
int icpb_proximity_closest(icpb_handle h, const double *h_xy, const double *h_travelled, int64_t n,
                           double min_dist_along_path, double max_dist, int32_t *h_closest, double *h_dist);

/* The generalisation BASELINE config 3 names: EVERY pair (i, j), j >= start(i), within max_dist,
 * as (source = j, target = i) rows (the argument order of :31-34), ordered by i then j.  Call with
 * capacity 0 to get the count in *n_pairs, then again with a buffer of that many rows. */
int icpb_proximity_pairs(icpb_handle h, const double *h_xy, const double *h_travelled, int64_t n,
                         double min_dist_along_path, double max_dist, int64_t capacity,
                         int32_t *h_pairs, int64_t *n_pairs);

/* Chain composition of the odometry fan-out's results (scripts/main.py:249-256): poses_out has
 * n + 1 rows (x, y, theta); row 0 is pose0, row i + 1 = mat_to_pose(pose_to_mat(row i) @ T_i).
 * Pure host function (no handle): a serial dependency chain. */
int icpb_compose_chain(const double *pose0, const double *T6, int64_t n, double *poses_out);

/* The same prefix product as a parallel scan on the device (SE(2) composition is associative; the
 * result differs from the step-by-step loop by rounding only, ~1e-12 at 5,000 steps).
 * icpb_compose_chain_device: d_T6 (n x 6) and d_poses_out ((n + 1) x 3) are device arrays -- d_T6 can be
 * the d_T output of icpb_run_device, so the transforms never visit the host; asynchronous on `stream`.
 * icpb_compose_chain_gpu: host arrays in and out through the same kernel.  Measured against the host
 * loop in DESIGN.md; the Python callers use whichever is faster for the chain at hand. */
int icpb_compose_chain_device(icpb_handle h, const double *pose0, const double *d_T6, int64_t n,
                              double *d_poses_out, void *stream);
int icpb_compose_chain_gpu(icpb_handle h, const double *pose0, const double *h_T6, int64_t n, double *h_poses_out);

/*
 * Pose-graph relaxation, the consumer of the path's constraints (SURVEY.md section 8f-3): n_steps
 * passes of the reference's pose_graph_optimization_step_sgd(pose_graph, learning_rate,
 * loop_closure_uncertainty) (src/pose_graph_optimization.py:7-49), pass k with
 * h_learning_rates[k] (scripts/main.py:325-326 uses 1/(k+1)).
 *   h_poses    n x 3 float64 (x, y, theta) = pose_graph.poses, updated in place
 *   h_edges    n_edges x 2 int32 (a, b) in the order `pose_graph.graph.edges(data="object")`
 *              yields them (the optimiser is order dependent); edges with |a - b| == 1 are ignored
 *              exactly as the reference ignores them (:14-16), edges with b <= a move nothing
 *   h_edge_T6  n_edges x 6 float64: the top two rows of every edge's 3x3 transform (bottom row
 *              [0 0 1], as add_constraint receives it from the ICP path, src/pose_graph.py:38-40)
 * Results agree with the reference to rounding (closed-form 3x3 inverses, prefix sums; the goldens
 * of the unmodified reference are met to 1e-12).  Any number of poses: the sequential part of a pass
 * works on 80-byte per-edge records, not on the poses (csrc/icpb_sgd.cuh).
 */
int icpb_pose_graph_sgd(icpb_handle h, double *h_poses, int64_t n, const int32_t *h_edges,
                        const double *h_edge_T6, int64_t n_edges, const double *h_learning_rates,
                        int32_t n_steps, double loop_closure_uncertainty);

/*
 * Occupancy grid from the optimised poses and the scans (SURVEY.md section 8f-4):
 * produce_occupancy_grid(poses, lidar_points, cell_width, min_width, min_height, kHitOdds, kMissOdds)
 * and update_occupancy_grid(...) (src/produce_occupancy_grid.py:11-80).  Pose i belongs to scan i
 * of the handle's scan table (icpb_upload_scans); n <= number of scans.
 *
 * icpb_occupancy_grid_bounds: the grid origin and size of :27-51 (bounding box of all beam end
 *   points in the global frame, half a cell of margin, optional minimum size).
 * icpb_occupancy_grid_update: the double loop over beams of :54-56 / :76-78 -- a Bresenham walk per
 *   beam (:96-131), "miss" on every crossed cell, "hit" on the last -- applied to h_grid
 *   (height x width int8, row 0 at min_y, C order), in place.  Bit-identical to the reference's
 *   sequential loops, including its int8 wrap-around at :109 and :128 (see csrc/icpb_grid.cuh).
 *   kHitOdds and kMissOdds must be integers in 1..127.
 * Both calls check their inputs against ICPB_MAX_GRID_CELL / ICPB_MAX_GRID_CELLS (above) and return
 * ICPB_EINVAL before anything runs; a rejected update leaves h_grid untouched.
 */
int icpb_occupancy_grid_bounds(icpb_handle h, const double *h_poses, int64_t n, double cell_width,
                               double min_width, double min_height, double *min_x, double *min_y,
                               int64_t *height, int64_t *width);
int icpb_occupancy_grid_update(icpb_handle h, const double *h_poses, int64_t n, int8_t *h_grid,
                               int64_t height, int64_t width, double min_x, double min_y,
                               double cell_width, int32_t k_hit, int32_t k_miss);

/* Launch geometry and resource use of the alignment kernel for the current scan table
 * (reported by bench.py next to the roofline numbers). */
typedef struct icpb_kernel_info {
    int32_t threads_per_cta, ctas_per_sm, sm_count, grid;
    int32_t regs_per_thread, smem_bytes, points_per_thread, variant;
} icpb_kernel_info;
int icpb_get_kernel_info(icpb_handle h, int64_t B, icpb_kernel_info *out);

/* Tuning and test hooks, per handle (nothing is read from the environment).  Keys: "threads" (CTA
 * width cap, multiple of 32), "cluster" (force a cluster size: 0/1 never, 2/4/8), "segments" (upload
 * pieces), "pack_threads" (host threads of icpb_align_host_scans, default min(8, cpus)),
 * "drop_counter" (tests: never advance the arrival counter), "large" (1: every pair on the
 * large-scan variant, arrays in device scratch instead of shared memory -- same results; 0 / -1: only
 * pairs whose scans do not fit shared memory).  0 / -1 restore the default.
 *
 * Scans of any length: a pair whose longer scan does not fit one CTA's shared memory runs on the
 * large-scan variant of the kernel.  Where the host sees the pairs (icpb_run_host, icpb_align_host*,
 * icpb_icp_pair_host) a batch is split: the pairs that fit run on the shared-memory kernel, the others
 * on the large variant; icpb_run_device* and pair_mode 1 send the whole batch to the large variant
 * when the table's longest scan does not fit.  Both variants give the same bits. */
int icpb_set_tuning(icpb_handle h, const char *key, int64_t value);

/* Number of alignment-kernel launches made through this handle (bench.py's gpu_launches). */
int64_t icpb_launch_count(icpb_handle h);

/* Scans of the table resident on the handle's device (submaps included), 0 when there is none (never set,
 * or an icpb_align_host* or icpb_set_submaps call failed part-way and left the buffer half written). */
int64_t icpb_scan_count(icpb_handle h);

/* Optional instrumentation: while enabled, launches add the point-pair distance evaluations
 * they actually execute (after pruning) to a device counter; icpb_read_work synchronises the
 * device and returns it.  Enabling resets the counter. */
int icpb_count_work(icpb_handle h, int enable);
int icpb_read_work(icpb_handle h, uint64_t *executed_pde);

const char *icpb_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* ICPB_H */
