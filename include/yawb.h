/*
 * yawb -- C ABI of the B200 pair-counting engine for yet_another_wizz.
 *
 * The reference (jlvdb/yet_another_wizz v3.1.1, pure Python) has no FFI; the
 * drop-in boundary is the set of Python seams listed in SURVEY.md section 8b.
 * Each entry point below names the reference interface it replaces (paths are
 * relative to the reference checkout, `/root/reference/`).  The Python host
 * (`yet_another_wizz_b200/_lib.py`) binds these with ctypes; INTEGRATION.md
 * shows the stub a maintainer of the reference would add.
 *
 * Conventions
 *   - plain pointers and sizes only; the caller owns every host buffer, the
 *     library owns every device buffer;
 *   - every function returns 0 on success, non-zero on failure with a message
 *     available from yawb_last_error() (thread local);
 *   - any number of contexts per process, on the same or on different devices
 *     (library version >= 103); every entry point selects the device of the
 *     context it is given, and contexts share no state, so each context may be
 *     driven by its own host thread.  A context is not re-entrant: one thread
 *     at a time per context and its catalogs.  All work of a context is issued
 *     on CUDA streams owned by the context;
 *   - there is no CPU fallback: without a CUDA device yawb_create() fails.
 */
#ifndef YAWB_H
#define YAWB_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct yawb_ctx yawb_ctx;
typedef struct yawb_cat yawb_cat;

/* flags for yawb_count() */
#define YAWB_FLAG_EXACT_BRUTEFORCE 1u /* FP64 all-pairs kernel, no pruning (validation / cross-check) */
#define YAWB_FLAG_OUT_DEVICE 2u       /* out_f64 / out_i64 are device pointers (e.g. torch tensors)  */
/* Labelled second catalogs (library version >= 101): the per-row ids of a binned second catalog are sample labels
 * 0..L-1 (L = its n_bins; an unbinned second catalog has L = 1), not z-bins.  A row with label l is paired with
 * every z-bin of the first catalog, as a row of an unbinned catalog is, and its counts go to output block l: each
 * (first, second) catalog combination writes [L][n_pairs][n_bins][n_edges-1], so the caller's arrays (host or
 * YAWB_FLAG_OUT_DEVICE) are L times longer.  Block l equals yawb_count(cat1, U_l) for an unbinned upload U_l of
 * exactly the rows with label l (integer counts bit for bit).  Rows with a label outside [0, L) are dropped (255 in
 * yawb_upload_catalog_u8).  This is how the tomographic bins of an unknown sample are counted in one pass.  Not
 * supported with YAWB_FLAG_EXACT_BRUTEFORCE.  Unknown flag bits are rejected. */
#define YAWB_FLAG_SECOND_LABELS 4u

/* roles for yawb_build_index() */
#define YAWB_ROLE_FIRST 1  /* catalog used as first argument of yawb_count(): sky-cell index        */
#define YAWB_ROLE_SECOND 2 /* catalog used as second argument: Hilbert-ordered register tiles        */

typedef struct {
    double kernel_ms;          /* device time of planner + pair-count kernel, CUDA events on the ctx stream */
    double index_ms;           /* device time of index builds triggered by this call (0 if prebuilt)      */
    uint64_t pair_tests;       /* pair tests executed (after sky-cell / tile pruning)                     */
    uint64_t pair_tests_naive; /* sum over requested patch pairs and z-bins of n1 * n2 (n2: all labels)   */
    uint64_t rechecks;         /* tests re-evaluated in exact FP64                                        */
    uint64_t work_items;       /* work items written by the planner (tile x linked patch, non-empty)      */
    uint64_t launches;         /* kernels launched by this call                                           */
    double plan_ms;            /* part of kernel_ms spent in the planner (k_plan); the rest is the count kernel */
} yawb_stats;

/* Thread-local description of the last failure. */
const char *yawb_last_error(void);

/* Create / destroy an engine context on CUDA device `device`.
 * Replaces the reference's worker farm set-up, src/yaw/utils/parallel.py:318-343
 * (a fresh multiprocessing.Pool per iter_unordered call). */
int yawb_create(int device, yawb_ctx **out);
int yawb_destroy(yawb_ctx *ctx);

/* Upload one patch-partitioned catalog into HBM (once) and compute per-patch
 * frames, bounding spheres and sums of weights.
 *
 * Replaces Catalog.build_trees / BinnedTrees.build / build_trees /
 * AngularTree.__init__ (src/yaw/catalog/catalog.py:1406-1460,
 * src/yaw/catalog/trees.py:365-429, 215-246): instead of one pickled cKDTree
 * per patch and z-bin the points are kept resident, sorted by
 * (patch, z-bin, sky cell).
 *
 *   xyz        n x 3 float64, exactly AngularCoordinates.to_3d() of the rows
 *              (src/yaw/coordinates.py:134-147), rows grouped by patch
 *   w          n float64 weights or NULL (unweighted: sum_weights = count,
 *              trees.py:225-227; counts are then integers)
 *   zbin       n int32 z-bin index np.digitize(z, edges, right=closed=="right") - 1
 *              (trees.py:408-414); rows with zbin outside [0, n_bins) are
 *              dropped.  NULL = unbinned catalog (one "tree" per patch that is
 *              paired with every z-bin of the first catalog, trees.py:600-601)
 *   patch_off  n_patch + 1 row offsets (patch ids are 0..n_patch-1,
 *              src/yaw/correlation/measurements.py:358-364)
 *   n_bins     number of z-bins (ignored when zbin == NULL)
 *
 * The call is asynchronous: it only allocates and enqueues the host-to-device copies on a dedicated copy
 * stream (which never carries a kernel, so copies of later catalogs proceed while pair counts of earlier
 * ones occupy the GPU); the per-patch reductions run when the catalog is first used.  The host buffers
 * must stay valid until the first call that uses the catalog (or yawb_sync) has returned.  Enqueue every
 * catalog first and count in arrival order to overlap PCIe with the counts.
 */
int yawb_upload_catalog(yawb_ctx *ctx, const double *xyz, const double *w, const int32_t *zbin,
                        const int64_t *patch_off, int n_patch, int n_bins, yawb_cat **out);
/* Same with byte-sized z-bin ids (n_bins <= 254; any id >= n_bins, e.g. 255, marks a dropped row): the ids
 * are 5 % of the bytes of a z-binned catalog as int32, 1.3 % as bytes. */
int yawb_upload_catalog_u8(yawb_ctx *ctx, const double *xyz, const double *w, const uint8_t *zbin,
                           const int64_t *patch_off, int n_patch, int n_bins, yawb_cat **out);
/* Same with the raw redshifts: the rows are assigned to z-bins ON THE DEVICE, with the arithmetic of
 * np.digitize(z, edges, right = closed_right) - 1 (src/yaw/catalog/trees.py:408-414, Binning edges of
 * src/yaw/binning.py): bin b holds edges[b] < z <= edges[b + 1] (closed_right) or edges[b] <= z < edges[b + 1];
 * rows outside the binning (and NaN) are dropped.  Comparisons only, so the ids are identical to numpy's.
 *   z       n redshifts;   edges   n_bins + 1 strictly increasing doubles (copied by the call) */
int yawb_upload_catalog_z(yawb_ctx *ctx, const double *xyz, const double *w, const double *z, const double *edges,
                          int closed_right, const int64_t *patch_off, int n_patch, int n_bins, yawb_cat **out);
/* Binned labels (library version >= 102): declares the ids of a catalog uploaded with yawb_upload_catalog or
 * yawb_upload_catalog_u8 to be  id = label * B + zbin  with L = n_labels labels and B = n_bins / L z-bins, e.g. the
 * tomographic bins of a sample, each z-binned.  Rejects unbinned catalogs, yawb_upload_catalog_z catalogs,
 * n_labels < 1 and an n_bins that L does not divide.  Indexes and yawb_sum_weights ([n_bins][n_patch] =
 * [L][B][n_patch]) do not depend on it.  yawb_count then takes r2_edges as [B][n_edges] and writes
 * [L][n_pairs][B][n_edges-1] (block l = label l, as with YAWB_FLAG_SECOND_LABELS), under two rules:
 *   (a) cat1 and cat2 both labelled, with the same L and B (cat1 == cat2 included): the rows (l, z) of cat2 are
 *       counted against the rows (l, z) of cat1 -- per label, the z-binned count of its own two catalogs;
 *   (b) cat1 binned with B z-bins and no labels, cat2 labelled: the rows (l, z) of cat2 against the rows z of cat1.
 *       Pair counts are symmetric (d2 and w1 * w2 are the same doubles either way round), so a labelled sample
 *       against shared randoms is counted with the randoms as cat1 and the pair lists swapped.
 * Rejected with a message (the context stays usable): a labelled cat1 with an unlabelled cat2 (swap the roles),
 * different L or B, YAWB_FLAG_EXACT_BRUTEFORCE, YAWB_FLAG_SECOND_LABELS, and labelled catalogs in yawb_count2 /
 * yawb_count4. */
int yawb_catalog_set_labels(yawb_cat *cat, int n_labels);

/* Partial upload (library version >= 103): the rows of the patches with keep[p] != 0 only, taken from the full host
 * arrays (xyz, w, zbin / zbin8 / z and patch_off describe the whole catalog, as for the uploads above; at most one of
 * zbin, zbin8 and z with edges / closed_right).  Patch ids keep their numbers and an unkept patch is an empty patch:
 * for a kept patch the sums of weights, frames and indexes are those of a full upload (up to the order of FP64
 * sums), for an unkept one the sums are 0.  Each run of consecutive kept patches travels straight from the caller's
 * arrays, as one copy per array; no host-side gather.  This is how one device of several holds only the patches it
 * counts and their neighbours. */
int yawb_upload_catalog_patches(yawb_ctx *ctx, const double *xyz, const double *w, const int32_t *zbin,
                                const uint8_t *zbin8, const double *z, const double *edges, int closed_right,
                                const int64_t *patch_off, int n_patch, int n_bins, const uint8_t *keep, yawb_cat **out);

/* Second-role row mask (library version >= 103): mask holds one byte per uploaded row (for a partial upload: the rows
 * of the kept patches, in patch order); a row with mask 0 is left out of the second-role index (tiles, Hilbert order,
 * tile spheres) as a row outside the z-binning is.  NULL clears the mask.  The first-role index, yawb_sum_weights,
 * yawb_patch_metadata and yawb_catalog_info keep every row.  Setting or clearing the mask drops a built second-role
 * index (first-role and fused indexes stay).  Synchronous.
 * Contract: for masks m and !m on two uploads A_m, A_!m of the same rows (and A_full without a mask),
 *     count(c1, A_m) + count(c1, A_!m) == count(c1, A_full)
 * bit for bit for integer counts and to 1e-12 for weighted sums, for every count path, for labelled and binned-label
 * catalogs, in yawb_count / yawb_count2 / yawb_count4, and for auto counts (the masked upload as the second catalog,
 * the same or a full upload as the first).  The mask carries the caller's choice of rows: equal sort keys have no
 * defined order and frames are FP64 atomic sums, so no rule stated in the index's own order would split the rows
 * alike on two devices. */
int yawb_catalog_set_second_rows(yawb_cat *cat, const uint8_t *mask);
int yawb_free_catalog(yawb_cat *cat);

/* Build (or rebuild) the device-side index for a role ahead of time; otherwise
 * yawb_count() builds it on first use.  Device time is returned in *ms. */
int yawb_build_index(yawb_cat *cat, int role, double *ms);
int yawb_drop_index(yawb_cat *cat);

/* Number of rows kept (zbin in range) and device bytes held by the catalog. */
int yawb_catalog_info(const yawb_cat *cat, int64_t *n_rows, int64_t *device_bytes);

/* Sum of weights per z-bin and patch, out[n_bins][n_patch] (n_bins = 1 for an
 * unbinned catalog): AngularTree.sum_weights collected by process_patch_pair,
 * src/yaw/correlation/measurements.py:123-124, trees.py:225-234. */
int yawb_sum_weights(const yawb_cat *cat, double *out);

/* Jackknife by subtraction on the device: the sum over all patch pairs and its leave-one-patch-out samples,
 *     total[b] = sum_k v[k][b],   samples[p][b] = total[b] - sum_{k : i_k == p or j_k == p} v[k][b]
 * -- SampledPatchSum of src/yaw/correlation/paircounts.py:113-141 (total - row_p - column_p + diagonal_p) written
 * on the list of linked patch pairs instead of the dense (n_patch x n_patch) array.
 *   values[n_pairs][n_bins]  per-pair, per-z-bin counts or products of sums of weights (host)
 *   total[n_bins], samples[n_patch][n_bins]   (host)
 * Integer-valued inputs give exact results (sums of integers below 2^53 do not depend on the order); others
 * agree with numpy's einsum to rounding. */
int yawb_jackknife(yawb_ctx *ctx, const double *values, const int32_t *pair_i, const int32_t *pair_j, int n_pairs,
                   int n_patch, int n_bins, double *total, double *samples);

/* Patch meta data computed on the device from the uploaded rows (all rows of the patch, whatever their z-bin):
 * the quantities of Metadata.compute, src/yaw/catalog/patch.py:104-147.
 *   center_xyz[n_patch][3]  normalised mean direction (the reference converts it to RA / Dec)
 *   radius_chord[n_patch]   largest chord distance of a row from the centre, rounded up by 1e-12 relative
 *                           (the reference's radius is the angle 2 asin(chord / 2))
 *   num_records[n_patch]    rows of the patch
 * Any pointer may be NULL.  The sums run in a different order than numpy's, so centres agree to ~1e-15, not
 * bit for bit; the reference-exact meta data of this package's Catalog stays on the host. */
int yawb_patch_metadata(const yawb_cat *cat, double *center_xyz, double *radius_chord, int64_t *num_records);

/* Count pairs for a list of linked patch pairs.
 *
 * Replaces the body of PatchLinkage.count_pairs -> process_patch_pair ->
 * AngularTree.count -> scipy cKDTree.count_neighbors
 * (src/yaw/correlation/measurements.py:307-367, 88-128;
 *  src/yaw/catalog/trees.py:303-362, scipy call :348-353).
 *
 * For pair k = (pair_i[k], pair_j[k]) and z-bin b of cat1, every point a of
 * cat1 (patch pair_i[k], bin b) is tested against every point c of cat2
 * (patch pair_j[k]; bin b if cat2 is binned, all rows otherwise):
 *
 *     d2 = (dx*dx + dy*dy) + dz*dz          IEEE double, no FMA (scipy's order)
 *     sub-bin s (0-based) iff r2[b][s] < d2 <= r2[b][s+1]
 *
 *   r2_edges  [n_bins][n_edges] squared chord thresholds, already
 *             pow(2 sin(theta/2), 2.0) of get_ang_bins() (trees.py:84-117, :350)
 *   out_i64   [n_pairs][n_bins][n_edges-1] number of pairs (may be NULL)
 *   out_f64   [n_pairs][n_bins][n_edges-1] sum of w1*w2 (may be NULL; equals the
 *             integer count when both catalogs are unweighted)
 *
 * The host applies the r-weights / scale sums (trees.py:358-362), the 0.5 on
 * auto diagonals (measurements.py:362-363) and the scatter into PatchedCounts.
 * Results are bit-exact for integer counts; weighted sums are accumulated in
 * FP64 (order differs from the tree walk: ~1e-15 relative).
 */
int yawb_count(yawb_ctx *ctx, yawb_cat *cat1, yawb_cat *cat2, const int32_t *pair_i,
               const int32_t *pair_j, int n_pairs, const double *r2_edges, int n_edges,
               uint32_t flags, double *out_f64, int64_t *out_i64, yawb_stats *stats);

/* Two first catalogs against the same second catalog in ONE pass: results identical to
 *     yawb_count(ctx, cat1a, cat2, ...) -> out_*_a   and   yawb_count(ctx, cat1b, cat2, ...) -> out_*_b.
 *
 * This is how crosscorrelate's DD + RD (reference sample and its randoms against the unknown sample) and
 * DR + RR (the same two against the unknown sample's randoms) are counted,
 * src/yaw/correlation/measurements.py:623-626: both first catalogs share the patches, the z-binning and the
 * thresholds, so their rows are indexed together (one fused sky-cell index, cached until either catalog is
 * dropped or freed) and every register tile of the second catalog is loaded, rotated and matched against the
 * sky cells once instead of twice.  cat1a and cat1b need the same n_patch / n_bins; YAWB_FLAG_EXACT_BRUTEFORCE
 * is not supported here.  stats cover both counts. */
int yawb_count2(yawb_ctx *ctx, yawb_cat *cat1a, yawb_cat *cat1b, yawb_cat *cat2, const int32_t *pair_i,
                const int32_t *pair_j, int n_pairs, const double *r2_edges, int n_edges, uint32_t flags,
                double *out_f64_a, int64_t *out_i64_a, double *out_f64_b, int64_t *out_i64_b, yawb_stats *stats);

/* The four counts of a cross-correlation in ONE launch: two first catalogs (fused index, as in yawb_count2)
 * against TWO second catalogs.  Results identical to
 *     yawb_count(ctx, cat1a, cat2a) -> out[0]    yawb_count(ctx, cat1b, cat2a) -> out[1]
 *     yawb_count(ctx, cat1a, cat2b) -> out[2]    yawb_count(ctx, cat1b, cat2b) -> out[3]
 * i.e. DD, RD, DR, RR of src/yaw/correlation/measurements.py:623-626 for (cat1a, cat1b, cat2a, cat2b) =
 * (reference, its randoms, unknown, its randoms).  The planner lists the work items of both second catalogs for
 * one persistent kernel, so a small job (a GPU's share of a multi-GPU run) pays the ramp-up and the tail of a
 * launch, the host synchronisation and the result transfer once instead of twice.  cat2a and cat2b need the same
 * n_patch / n_bins; with YAWB_FLAG_SECOND_LABELS only the same n_patch, and each output has the L of its own second
 * catalog (a labelled unknown sample and a shared unlabelled random catalog in one launch).
 * out_f64 / out_i64: tables of four pointers each, any of which may be NULL.
 * YAWB_FLAG_EXACT_BRUTEFORCE is not supported.  stats cover all four counts. */
int yawb_count4(yawb_ctx *ctx, yawb_cat *cat1a, yawb_cat *cat1b, yawb_cat *cat2a, yawb_cat *cat2b, const int32_t *pair_i,
                const int32_t *pair_j, int n_pairs, const double *r2_edges, int n_edges, uint32_t flags,
                double *const out_f64[4], int64_t *const out_i64[4], yawb_stats *stats);

/* Pinned host memory helpers so callers can stage inputs for async copies. */
int yawb_host_alloc(void **ptr, uint64_t bytes);
int yawb_host_free(void *ptr);

/* Block until all work of the context has finished. */
int yawb_sync(yawb_ctx *ctx);

/* Device-side stopwatch on the context's stream (CUDA events), for benchmarks: everything the
 * context enqueues between start and stop is covered.  stop waits for the stream. */
int yawb_timer_start(yawb_ctx *ctx);
int yawb_timer_stop(yawb_ctx *ctx, double *ms);

/* Nearest patch centre of every row, the catalog-creation step that precedes the hot path (SURVEY.md
 * section 8f, rank 2).  Replaces `assign_patch_centers` (src/yaw/catalog/catalog.py:229-249), i.e.
 * scipy.cluster.vq.vq(xyz, centers): squared Euclidean distance summed x -> y -> z in double without FMA,
 * first minimum wins.  xyz: n x 3 and centers_xyz: n_centers x 3 float64 on the host, out_ids: n int32 on
 * the host.  Synchronous. */
int yawb_assign_patches(yawb_ctx *ctx, const double *xyz, int64_t n, const double *centers_xyz, int n_centers,
                        int32_t *out_ids);

/* Spherical k-means for patch centres (replaces treecorr's k-means behind create_patch_centers,
 * src/yaw/catalog/catalog.py:183-226).  Contract: DESIGN.md §4.4.  xyz n x 3, w n or NULL, host memory;
 * centers_xyz k x 3 out; labels n out or NULL; *n_iter, *converged out.  Synchronous.
 *
 * Deterministic and exact: every sum is an int64 sum of fixed-point coordinates q = rint(x 2^32) (weighted:
 * q = rint((w x) 2^(32 - e)), e = frexp(max w)), and the centre of a sum s is s / sqrt((sx sx + sy sy) + sz sz)
 * in correctly rounded double arithmetic.  Initial centres: bisection of the unweighted rows (split the
 * min(c, k - c) most populated splittable cells along their widest q axis at the mean, q_axis * count > sum q_axis
 * goes to the high child with id c + rank).  Lloyd iterations: C_i = centre(rows of L_(i-1)), an empty cluster
 * (s = 0) moved, in ascending order, to the row farthest from its own centre in C_(i-1) (squared vq distance,
 * ties to the lowest row, rows taken before skipped), L_i = vq(rows, C_i); stop when L_i == L_(i-1)
 * (*converged = 1) or after max_iter iterations (*n_iter = iterations run; max_iter = 0 returns the initial
 * centres and their assignment).  labels == vq(xyz, centers) always.
 * Requirements: 1 <= k <= 4096, k <= n < 2^30, max_iter >= 0, rows finite with |coordinate| <= 1, weights finite,
 * >= 0, largest weight >= 2^-992; at least k distinct fixed-point positions. */
int yawb_kmeans(yawb_ctx *ctx, const double *xyz, const double *w, int64_t n, int k, int max_iter,
                double *centers_xyz, int32_t *labels, int *n_iter, int *converged);

/* Device memory (library version >= 104).
 *
 * yawb_catalog_footprint: host arithmetic only, no device access.  An upper bound on the device bytes one catalog of
 * n_rows rows in n_patch patches and n_bins z-bins (1: unbinned; labelled: labels x z-bins) holds: `what` is an OR of
 * the YAWB_FOOT_* flags below, naming the columns that travel and the indexes to cover.  Every block the upload, its
 * per-patch frames and sums, the second-role row mask and the index builds request is summed -- scratch freed
 * again included -- each rounded as the context's allocator rounds it, so yawb_memory_stats' `peak` of a context
 * that starts empty stays at or below the bound.  The first-role sky-cell grid is bounded from the row counts alone
 * (4 (n_rows + n_patch n_bins) / 5.5 + 10241 n_patch n_bins cells, at most 2^30), the tile table by
 * n_rows / 256 + n_patch n_bins tiles.  Not covered: the rare re-cut of oversized tiles of a second-role index
 * (tiles whose bounding sphere is more than three times the expected one are cut into pieces of 32 rows).
 * YAWB_FOOT_NO_UPLOAD with one index flag bounds an index over rows uploaded by other catalogs: the fused first-role
 * index of yawb_count2 / yawb_count4 (n_rows = rows of both first catalogs) or the union second-role index of
 * yawb_count4 (rows of both second catalogs).
 *
 * yawb_count_footprint: the workspace of one yawb_count / yawb_count2 / yawb_count4 call on a device with `sms`
 * SMs (the SM count sizes the work-item lists; yawb_device_sms); host arithmetic only: the table of pair lists and thresholds, the work-item lists of the
 * planner, and the output counts (and sums if `weighted`) of n_blocks x n_pairs x n_bins x (n_edges - 1) entries,
 * where n_blocks = (first catalogs) x (labels of the second catalogs, 1 each without labels).  n_items: the planner's
 * (patch pair, tile) combinations, i.e. the sum over the pair list of the tiles of the second patch, at most
 * rows / 256 + n_bins per patch.  The bound does not decrease with n_items, so an overestimate of n_items gives
 * an upper bound, also across the count at which the planner switches to the longer lists of a small job.
 * Not covered: the repeat of a count whose work-item lists overflowed (the
 * lists are then sized exactly).
 *
 * yawb_memory_stats: `held` = bytes the context's allocator holds (blocks in use and blocks parked for reuse), `peak`
 * = the high-water mark of `held` since the context was created or since yawb_memory_reset_peak, `device_free` =
 * free bytes of the device (cudaMemGetInfo).  Any pointer may be NULL.
 * yawb_memory_parked: the bytes of the blocks the allocator holds parked for reuse (part of `held`; they go back to
 * the driver when a cudaMalloc fails).
 * yawb_memory_release: parked blocks go back to the driver (blocks in use stay). */
#define YAWB_FOOT_WEIGHTED 1u   /* weights travel                                     */
#define YAWB_FOOT_BINNED 2u     /* int32 z-bin ids (yawb_upload_catalog)              */
#define YAWB_FOOT_U8 4u         /* byte z-bin ids (yawb_upload_catalog_u8)            */
#define YAWB_FOOT_Z 8u          /* raw redshifts binned on the device (yawb_upload_catalog_z) */
#define YAWB_FOOT_LABELLED 16u  /* binned labels (yawb_catalog_set_labels): ids as YAWB_FOOT_BINNED / _U8 */
#define YAWB_FOOT_MASK 32u      /* a second-role row mask (yawb_catalog_set_second_rows) */
#define YAWB_FOOT_FIRST 64u     /* the first-role index                               */
#define YAWB_FOOT_SECOND 128u   /* the second-role index                              */
#define YAWB_FOOT_NO_UPLOAD 256u /* leave out the upload: an index over other catalogs' rows */
int yawb_catalog_footprint(int64_t n_rows, int n_patch, int n_bins, uint32_t what, int64_t *bytes);
int yawb_count_footprint(int sms, int64_t n_items, int n_pairs, int n_bins, int n_edges, int n_blocks, int weighted,
                         int64_t *bytes);
int yawb_memory_stats(yawb_ctx *ctx, int64_t *held, int64_t *peak, int64_t *device_free);
int yawb_memory_parked(yawb_ctx *ctx, int64_t *parked);
int yawb_memory_reset_peak(yawb_ctx *ctx);
int yawb_memory_release(yawb_ctx *ctx);

/* Library version and number of SMs of the context's device. */
int yawb_version(void);
int yawb_device_sms(const yawb_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* YAWB_H */
