// Internal declarations shared by the translation units of libyawb.so.
// Nothing here is part of the C ABI (see include/yawb.h).
#pragma once

#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <vector>

#include <nvtx3/nvToolsExt.h>

#include "yawb.h"

// NVTX range over a scope (header-only NVTX 3: a no-op unless a profiler is attached)
struct YawbRange {
    explicit YawbRange(const char *name) { nvtxRangePushA(name); }
    ~YawbRange() { nvtxRangePop(); }
    YawbRange(const YawbRange &) = delete;
    YawbRange &operator=(const YawbRange &) = delete;
};

void yawb_set_error(const char *fmt, ...);

#define YAWB_CUDA(call)                                                                        \
    do {                                                                                       \
        cudaError_t err__ = (call);                                                            \
        if (err__ != cudaSuccess) {                                                            \
            yawb_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call,                       \
                           cudaGetErrorString(err__));                                         \
            return 1;                                                                          \
        }                                                                                      \
    } while (0)

#define YAWB_REQUIRE(cond, ...)                                                                \
    do {                                                                                       \
        if (!(cond)) {                                                                         \
            yawb_set_error(__VA_ARGS__);                                                       \
            return 2;                                                                          \
        }                                                                                      \
    } while (0)

// Squared distance of scipy.cluster.vq.vq for fewer than 5 features: differences centre - row, squares summed
// x -> y -> z, every operation rounded on its own (no FMA).  Shared by patch assignment and k-means.
__device__ __forceinline__ double yawb_vq_d2(double cx, double cy, double cz, double x, double y, double z) {
    const double dx = __dsub_rn(cx, x), dy = __dsub_rn(cy, y), dz = __dsub_rn(cz, z);
    return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

// ---- geometry of one patch: orthonormal frame at the mean direction --------------------
struct PatchFrame {
    double c[3];   // unit vector of the patch centre (mean direction)
    double e1[3];  // tangent basis; (u, v, t) = ((P-c).e1, (P-c).e2, (P-c).c)
    double e2[3];
    double radius;                    // max chord distance of a patch point from c
    double umin, umax, vmin, vmax;    // bounding box of the patch in (u, v)
    double norm_dev;                  // max | |P|^2 - 1 | over the rows: how far they are from the unit sphere (rounded up)
};

// ---- sky-cell grid of one patch (first-role index); identical for every z-bin ------------
// The rows of the index are stored as fixed-point records in the frame of their patch:
//   k = rint((coordinate - origin) * qscale),  origin = (u0, v0, t0),  qscale = 2^m
// with m chosen per patch so that every k fits 31 bits.  A coordinate is recovered to within
// 0.5001 / qscale (a few 1e-11 for a 5-degree patch: finer than the float rounding of a tile-local
// vector), and the exact doubles stay available for the FP64 recheck.
struct SGrid {
    double u0, v0;         // cell (iu, iv) covers u0 + iu / inv_cu ..., v0 + iv / inv_cv ...
    double inv_cu, inv_cv; // cells are narrower along u, the direction of the contiguous runs (kCellAspect)
    int gu, gv;            // cells per row / number of rows
    long long cell_base;   // global cell id of (bin 0, iv 0, iu 0); bin stride = gu * gv
    double t0;             // origin of the third coordinate (t = (P - c).c <= 0)
    double qscale, qinv;   // 2^m and 2^-m
};

// One row of a first-role index: fixed-point (u, v, t) in the frame of its patch; `aux` = position of
// the row in the sorted arrays (bits 0..30) | catalog of a fused index (bit 31).
struct __align__(16) SRec {
    int ku, kv, kt;
    unsigned aux;
};

// Bounding box of a register tile in the frame of its OWN patch (second-role index): lo / hi of (u, v, t).
struct TileBox {
    double lo[3], hi[3];
};

// One work item of a pair count, written by the planner: a register tile of the second catalog against
// the z-bins [b_lo, b_hi) of one linked patch of the first catalog.  `box` is the tile's bounding box in
// the frame of that patch (hull of the rotated corners of the own-frame box, so it contains every row).
struct __align__(16) Item {
    int pair;              // index into the pair list (result row)
    int p1;                // patch of the first catalog
    int start;             // first row of the tile in the Hilbert-sorted arrays
    int count;             // rows of the tile (<= YAWB_TILE)
    int b_lo, b_hi;        // z-bins of the first catalog covered by this item
    int row_lo, row_hi;    // cell rows of the query covered, relative to its first row (whole query: 0, INT_MAX);
                           // a restriction only occurs on items of a single z-bin
    int src;               // second-role index of a joint launch (CountArgs::r2, 0 or 1): where the tile's rows live
    int blk;               // output block of the item's counts: second catalog, then label (YAWB_FLAG_SECOND_LABELS);
                           // a union tile's counts go to block 0 + (catalog of the row)
    int b_off;             // first-catalog id of z-bin 0 of the item's label (label * B when both catalogs carry
                           // binned labels, else 0): the cell rows of z-bin b are those of id b + b_off
    int pad;
    double lo[3], hi[3];
};
static_assert(sizeof(Item) == 96, "Item is copied as six 16-byte pieces");

// ---- register tile of the second-role catalog -------------------------------------------
struct Tile {
    int start;   // first row in the Hilbert-sorted arrays
    int count;   // <= YAWB_TILE
    int patch;
    int bin;     // z-bin of the tile, or -1 for an unbinned catalog
    float cx, cy, cz;  // bounding sphere (centre rounded to float, radius rounded up)
    float rad;
};

// ---- per z-bin thresholds prepared on the host for one yawb_count() call -----------------
struct BinPar {
    double lo, hi;  // r2[b][0], r2[b][n_edges-1]
    double rmax;    // sqrt(hi) * (1 + 1e-9) + 1e-14: chord search radius
    float mid, h;   // (lo + hi) / 2, (hi - lo) / 2 rounded to float
    int empty;      // 1 if the bin cannot hold pairs (hi <= lo)
    int pad;
};

constexpr int YAWB_RPL = 8;               // second-role points per lane
constexpr int YAWB_TILE = 32 * YAWB_RPL;  // points per register tile (one warp)
constexpr int YAWB_LG_CELLS_PER_EDGE = 4;  // cells of the lg2(d2) lookup per edge (sub-bin paths): finer cells = fewer fix-up steps
constexpr int YAWB_RSTRIDE = 4;           // doubles per second-role row record (x, y, z, catalog): one 32-byte sector
constexpr int YAWB_MAX_EDGES = 256;

struct yawb_ctx {
    int device = 0;
    int sms = 0;
    cudaStream_t stream = nullptr;       // all kernels and result copies
    cudaStream_t copy_stream = nullptr;  // host-to-device copies of catalog uploads (overlap with kernels)
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t ev_plan = nullptr;  // between the planner and the count kernel of the last fast count
    bool ev_plan_set = false;
    cudaEvent_t ev_i0 = nullptr, ev_i1 = nullptr;  // lazy index builds inside yawb_count (second role)
    cudaEvent_t ev_f0 = nullptr, ev_f1 = nullptr;  // ... (first role)
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;  // user stopwatch
    unsigned long long *d_counters = nullptr;  // [8] work counter + statistics
    // pinned arena for the meta data of in-flight uploads (bump allocated, reset when none is pending)
    unsigned char *pin_base = nullptr;
    size_t pin_size = 0, pin_used = 0;
    int pin_live = 0;
    struct yawb_devcache *cache = nullptr;  // device blocks, recycled (yawb_alloc.cu)
    // pinned arena that small host tables pass through on their way to the device (yawb_h2d_small)
    unsigned char *res_pin = nullptr;  // page-locked landing area of a count's results (grown on demand)
    size_t res_pin_size = 0;
    unsigned char *h2d_base = nullptr;
    size_t h2d_size = 0, h2d_used = 0;
    std::vector<struct FIndex *> fused;  // first-role indexes over pairs of catalogs (yawb_count2)
    std::vector<struct RIndex *> unions;  // second-role indexes over pairs of catalogs (yawb_count4)
};

// Second-role index: rows sorted by (patch, z-bin, Hilbert index) and cut into register tiles of YAWB_TILE rows.
// Over the rows of one catalog (yawb_cat::ri), or over the union of two catalogs with the same patches and z-bins
// (the single-bin path of yawb_count4): a tile of YAWB_TILE rows of both catalogs covers about half the sky of a tile
// of one, so every query box of the count shrinks.  The catalog of a row (0 / 1) is the fourth double of its record.
struct RIndex {
    yawb_ctx *ctx = nullptr;
    const yawb_cat *a = nullptr, *b = nullptr;  // sources (b == nullptr: single catalog)
    bool built = false;
    long long n = 0;                            // rows
    const PatchFrame *d_frames = nullptr;       // frames the tile boxes live in (a's)
    double *rrow = nullptr;                     // rows in tile order, one 32-byte record (x, y, z, catalog) per row
    double *rx = nullptr, *ry = nullptr, *rz = nullptr;  // views of rrow: row j is rx[4 j], ry[4 j], rz[4 j]
    double *rw = nullptr;                       // weights (1.0 for rows of an unweighted catalog), or nullptr
    int *d_seg_off = nullptr;                   // union only: [(n_patch * n_bins) + 1] segments of the union rows
    Tile *d_tiles = nullptr;
    TileBox *d_tile_box = nullptr;  // [n_tiles] bounding boxes in the frame of the tile's own patch
    std::vector<Tile> h_tiles;      // host copy of the tile table (source of an async upload)
    std::vector<int> h_ptile_off;   // [n_patch + 1] first tile of each patch
    int *d_ptile_off = nullptr;
    int n_tiles = 0;
    int64_t device_bytes = 0;
};

struct yawb_cat {
    yawb_ctx *ctx = nullptr;
    int64_t n_in = 0;     // rows uploaded
    int64_t n = 0;        // rows kept (z-bin in range)
    int n_patch = 0;
    int n_bins = 1;       // 1 for an unbinned catalog
    int n_labels = 0;     // binned labels (yawb_catalog_set_labels): ids are label * (n_bins / n_labels) + z-bin; 0: none
    bool binned = false;
    bool weighted = false;
    int64_t device_bytes = 0;

    // uploads are asynchronous: the host-side tables below are filled by yawb_cat_finalize() on first use
    bool finalized = false;
    cudaEvent_t ev_meta = nullptr;            // recorded on the copy stream after the last host-to-device copy
    long long *d_stage_poff = nullptr;        // row offsets of the patches, until yawb_cat_finalize()
    unsigned char *d_stage_bin8 = nullptr;    // z-bin ids uploaded as bytes, widened by yawb_cat_finalize()
    double *d_stage_z = nullptr;              // raw redshifts, digitized by yawb_cat_finalize()
    std::vector<double> h_edges;              // ... against these z-bin edges
    bool closed_right = true;
    unsigned long long *hp_counts = nullptr;  // pinned staging [n_bins][n_patch]
    double *hp_sumw = nullptr;                // pinned staging [n_bins][n_patch]
    PatchFrame *hp_frames = nullptr;          // pinned staging [n_patch]
    bool staging_in_arena = false;            // staging lives in the context's pinned arena
    void *hp_block = nullptr;                 // or in its own pinned block

    // raw rows in upload order (grouped by patch)
    double *xyz = nullptr;                    // the rows as uploaded, interleaved (n x 3)
    double *x = nullptr, *y = nullptr, *z = nullptr;  // views of xyz: row i is x[3 i], y[3 i], z[3 i]
    double *w = nullptr;
    int32_t *bin = nullptr;    // nullptr if unbinned
    int32_t *patch = nullptr;

    // per patch
    std::vector<PatchFrame> h_frames;
    PatchFrame *d_frames = nullptr;
    // per (bin, patch): number of rows and sum of weights, host copies
    std::vector<long long> h_counts;   // [n_bins][n_patch]
    std::vector<long long> h_rows_per_patch;  // [n_patch] rows uploaded, whatever their z-bin
    std::vector<int64_t> h_dev_off;           // [n_patch + 1] row offsets on the device (source of an async copy)
    std::vector<double> h_sumw;        // [n_bins][n_patch]
    std::vector<int> h_seg_off;        // [(n_patch * n_bins) + 1], patch-major, bin-minor
    int *d_seg_off = nullptr;

    // first-role index: rows sorted by global sky-cell id (built on first use)
    struct FIndex *findex = nullptr;

    // rows of the second-role index (yawb_catalog_set_second_rows): a byte per uploaded row, nullptr = every row.
    // With a mask the second-role index has its own row counts and segments; everything else keeps all rows.
    unsigned char *d_second_mask = nullptr;
    std::vector<long long> h_counts2;  // [n_bins][n_patch] masked rows (with a mask only)
    std::vector<int> h_seg_off2;       // [(n_patch * n_bins) + 1] segments of the masked rows
    int *d_seg_off2 = nullptr;
    int64_t n2 = 0;                    // masked rows
    int64_t second_rows() const { return d_second_mask ? n2 : n; }
    const std::vector<int> &second_seg_off() const { return d_second_mask ? h_seg_off2 : h_seg_off; }
    const std::vector<long long> &second_counts() const { return d_second_mask ? h_counts2 : h_counts; }
    int *second_d_seg_off() const { return d_second_mask ? d_seg_off2 : d_seg_off; }

    // second-role index over this catalog alone (built on first use)
    RIndex ri;
};

// First-role ("sky-cell") index over the rows of one catalog, or over the union of two catalogs with the
// same patches and z-bins (fused counts: both are counted against a second catalog in ONE pass, the
// catalog of a row travels in bit 31 of SRec::aux).  Rows sorted by (patch, z-bin, row-major cell).
struct FIndex {
    yawb_ctx *ctx = nullptr;
    const yawb_cat *a = nullptr, *b = nullptr;  // sources (b == nullptr: single catalog)
    long long n = 0;                            // rows (z-bin in range)
    int n_patch = 0, n_bins = 1, n_types = 1;
    bool weighted = false;
    SRec *rec = nullptr;                                    // fixed-point rows in the frame of their patch
    double *sw = nullptr;                                   // weights (1.0 for rows of an unweighted catalog)
    int *cell_start = nullptr;
    long long n_cells = 0;
    std::vector<SGrid> h_sgrid;
    SGrid *d_sgrid = nullptr;
    std::vector<PatchFrame> h_frames;  // frames of the index (the larger catalog's, boxes grown over both)
    PatchFrame *d_frames = nullptr;
    int64_t device_bytes = 0;
};

// index construction (yawb_index.cu)
// A run of rows copied from the caller's arrays: rows [src, src + rows) go to device rows [dst, dst + rows).
struct RowRun {
    int64_t src, dst, rows;
};
// patch_off: row offsets of the patches ON THE DEVICE; runs: where those rows come from in the host arrays
int yawb_index_upload(yawb_ctx *ctx, yawb_cat *cat, const double *xyz, const double *w, const uint8_t *zbin8,
                      const int32_t *zbin, const double *zred, const int64_t *patch_off, const std::vector<RowRun> &runs);
// second-role row mask (nullptr clears it); drops a built second-role index
int yawb_index_set_second_rows(yawb_cat *cat, const uint8_t *mask);
void yawb_index_free_second(yawb_cat *cat);
// device memory (yawb_alloc.cu): stream-aware caching allocator on top of cudaMalloc
int yawb_dalloc(yawb_ctx *ctx, void **out, size_t bytes, cudaStream_t st);
void yawb_dfree(yawb_ctx *ctx, void *ptr, cudaStream_t st);
void yawb_dcache_destroy(yawb_ctx *ctx);
size_t yawb_dcache_bytes(const yawb_ctx *ctx);
size_t yawb_dcache_peak(const yawb_ctx *ctx);
size_t yawb_dcache_parked(const yawb_ctx *ctx);  // bytes of the parked blocks
void yawb_dcache_reset_peak(yawb_ctx *ctx);
void yawb_dcache_release(yawb_ctx *ctx);   // parked blocks back to the driver
size_t yawb_dcache_round(size_t bytes);    // the size of the block a request of `bytes` gets
// upper bounds on device bytes (yawb_index.cu / yawb_count.cu; see yawb_catalog_footprint in include/yawb.h)
int64_t yawb_index_footprint(int64_t n_rows, int n_patch, int n_bins, uint32_t what);
int64_t yawb_count_workspace(int sms, int64_t n_items, int n_pairs, int n_bins, int n_edges, int n_blocks, bool weighted);

int yawb_cat_finalize(yawb_cat *cat);
// Small host table -> device on the main stream WITHOUT the copy engine: staged in pinned memory and
// pulled over by a kernel, so it never queues behind the bulk uploads of later catalogs.
int yawb_h2d_small(yawb_ctx *ctx, void *dst, const void *src, size_t bytes);
int yawb_index_build_first(yawb_cat *cat);
// fused first-role index over (a, b); cached in the context until either catalog is dropped or freed
int yawb_findex_get_fused(yawb_ctx *ctx, yawb_cat *a, yawb_cat *b, FIndex **out, bool *built);
void yawb_findex_drop_fused(yawb_ctx *ctx, const yawb_cat *cat);
void yawb_findex_free(FIndex *fi);
int yawb_index_build_second(yawb_cat *cat);
// second-role index over the union of (a, b); cached in the context until either catalog is dropped or freed
int yawb_rindex_get_union(yawb_ctx *ctx, yawb_cat *a, yawb_cat *b, RIndex **out, bool *built);
void yawb_rindex_drop_union(yawb_ctx *ctx, const yawb_cat *cat);
void yawb_index_free(yawb_cat *cat, bool everything);

// pair counting (yawb_count.cu)
struct CountArgs {
    const FIndex *c1;    // first-role index (one catalog, or two fused)
    const yawb_cat *c2;
    const yawb_cat *c2b = nullptr;       // second second-role catalog of a joint launch (yawb_count4), or nullptr
    // where the tiles come from: c2's index and c2b's (Item::src 0 / 1), or ONE index over the union of c2 and c2b
    // (r2[1] == nullptr; the rows' catalogs split every count, Item::blk = 0)
    const RIndex *r2[2] = {nullptr, nullptr};
    const int *d_pair_i;
    const int *d_pair_j;
    const long long *d_pair_item_base;  // [n_pairs + 1] prefix of tiles of r2[0] per pair
    long long n_items;                  // (patch pair, tile) combinations = threads of the planner
    const long long *d_pair_item_base_b = nullptr;  // the same for r2[1]
    long long n_items_b = 0;
    bool labels = false;    // YAWB_FLAG_SECOND_LABELS: the z-bin ids of a binned second catalog are sample labels
    int blk_b = 1;          // first output block of c2b (= labels of c2)
    int lab_bins = 0;       // binned labels of c2: z-bins per label B (id = label * B + z-bin), 0: none
    bool lab_first = false;  // ... and the first catalog carries the same binned labels
    long long cap_heavy, cap_light;     // capacities of the two work-item lists
    int n_pairs;
    int n_bins;
    int n_edges;
    const double *d_r2;      // [n_bins][n_edges]
    const float *d_r2f;      // same, rounded to float
    const BinPar *d_binpar;  // [n_bins]
    double rmax_all;         // max search radius over non-empty z-bins
    unsigned long long *d_out_cnt;  // [n_blocks][n_types][n_pairs][n_bins][n_edges-1], blocks: second catalog, then label
    double *d_out_w;                // same or nullptr if every catalog is unweighted
    bool weighted;
    // exact all-pairs kernel only (single catalogs): the first catalog's raw (patch, bin)-sorted rows
    const yawb_cat *c1_cat;
};
int yawb_launch_count_fast(yawb_ctx *ctx, const CountArgs &a, int *launches);
int yawb_launch_count_exact(yawb_ctx *ctx, const CountArgs &a, int *launches);
