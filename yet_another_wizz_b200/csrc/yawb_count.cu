// Pair-count kernels.
//
// Replaces scipy's cKDTree.count_neighbors as called from AngularTree.count
// (reference src/yaw/catalog/trees.py:348-353) and the per-z-bin loop of
// process_patch_pair (src/yaw/correlation/measurements.py:109-124).
//
// k_plan          -- one thread per (patch pair, register tile of the second catalog): the tile's bounding box is
//   rotated into the frame of the first catalog's patch, tested against that patch's box grown by the largest
//   search radius, and the survivors are written as self-contained work items (split so that an item never
//   holds more than CCAP (z-bin, cell row) runs).
// k_count_stream  -- the production kernel (yawb_count_stream.cuh).  One warp owns a register tile of YAWB_TILE
//   second-catalog points (YAWB_RPL per lane).  For every z-bin it gathers the first-catalog rows of the linked
//   patch that fall into the tile's bounding box grown by the bin's search radius (sky-cell rows -> contiguous
//   runs -> asynchronous 16-byte copies of fixed-point rows -> per-row cull), re-expresses them relative to the
//   tile's origin, rounds ONCE to float and stages them as (-2x, -2y, -2z, |s|^2 - mid) in shared memory.  The
//   pair test is
//       u = (|r|^2 + |s|^2 - mid) - 2 r.s = d2 - mid      4 FP32 ops (FADD + 3 FFMA, packed f32x2)
//       v = sat(C - K |u|)                                 1 FP32 op; sum(v), sum(v^2): 2 FP32 ops
//   on the CUDA cores; K is set by the bound on the FP32 error of u.  Whenever sum(v) != sum(v^2) for a lane's
//   share of a few candidates, that share is re-evaluated with the reference's exact FP64 expression
//   ((dx*dx + dy*dy) + dz*dz, no FMA), so the returned integers are bit-identical to the reference's.
//   Tensor cores are not used: K = 3 is not a dense contraction.
// k_count_exact   -- all-pairs FP64 kernel without pruning (validation and cross-check).
#include <cfloat>
#include <climits>

#include "yawb_internal.cuh"

namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr float EPS32 = 5.9604645e-8f;  // 2^-24
constexpr int CHUNK = 8;                // candidates between consistency checks (power of two)
// Coordinates of the padding rows of a short tile: NaN.  u = NaN fails |u| < h, and a saturating FMA flushes NaN to +0
// (PTX: "NaN results are flushed to +0.0f"), so every form of the pair test counts such a row as decided and outside.
#define PAD_ROW __int_as_float(0x7fffffff)
constexpr int CCAP = 160;               // (z-bin, cell row) runs per item; the planner splits items to fit
constexpr int CCAP_SMALL = 24;          // the same for a small job (yawb_launch_count_fast)
constexpr int SMALL_JOB_ITEMS = 30;     // (pair, tile) combinations per warp below which a job is small

struct FastParams {
    // first-role index (one catalog, or two fused).  The exact rows of a candidate are only needed by the FP64
    // recheck (~0.15 % of the tests): they are read from the catalog's own rows (cx / cy / cz of catalog 0 or 1
    // of the index) through the row id in SRec::aux -- the index holds no sorted copy of the doubles.
    const double *cx[2], *cy[2], *cz[2];
    const double *sw;
    const SRec *rec;
    const int *cell_start;
    const SGrid *sgrid;
    const PatchFrame *sframe;
    int n_types;
    float zeta;  // max | |P|^2 - 1 | over the rows of the second catalog(s), rounded up: part of the FP32 error bound
    // second catalog (register tiles): 32-byte row records (row j = rx[4 j .. 4 j + 3], the last double its catalog) and
    // optional weights; rx2 / rw2 = second index of a joint launch (Item::src == 1, yawb_count4)
    const double *rx, *rw;
    const double *rx2, *rw2;
    int n_sec;  // second catalogs whose counts a tile splits: 2 for tiles over the union of two catalogs, else 1
    // work items written by the planner: patch-diagonal items first, then the boundary items
    const Item *items_heavy, *items_light;
    long long cap_heavy, cap_light;
    int n_pairs, n_bins, n_edges;
    const double *r2;
    const float *r2f;
    const float *lgpar;           // [n_bins][2] (scale, offset): cell = lg2(d2) * scale + offset (sub-bin paths)
    const unsigned short *lgT;    // [n_bins][lg_cells] edges strictly below the start of a cell (lower bound)
    int lg_cells;
    int acc_global;               // general sub-bin path: segment histograms go straight to global atomics
    const BinPar *binpar;
    double rmax_all;              // largest search radius over the z-bins
    unsigned long long *out_cnt;  // [n_blocks][n_types][n_pairs][n_bins][n_edges - 1] (Item::blk: second catalog, then label)
    double *out_w;
    size_t type_stride;           // n_pairs * n_bins * (n_edges - 1)
    unsigned long long *counters;  // [0] next item, [1] tests, [2] rechecks, [4] heavy items, [5] light items, [6] overflow
};

// Cell rows of the query of one z-bin: the tile box (in the frame of the patch) grown by the bin's search radius,
// on the sky-cell grid of the patch.  Shared by the planner (which sizes the items) and the kernel.
struct BinRows {
    int iv0, nrows, iu0, iu1;
};
__device__ __forceinline__ BinRows bin_rows(const SGrid &G, double ulo, double uhi, double vlo, double vhi, const BinPar &bp,
                                            int row_lo, int row_hi) {
    BinRows r{0, 0, 0, 0};
    if (bp.empty) return r;
    // query box = tile box grown by the search radius (sound: |du|, |dv|, |dt| <= chord)
    const double fu0 = floor((ulo - bp.rmax - G.u0) * G.inv_cu), fu1 = floor((uhi + bp.rmax - G.u0) * G.inv_cu);
    const double fv0 = floor((vlo - bp.rmax - G.v0) * G.inv_cv), fv1 = floor((vhi + bp.rmax - G.v0) * G.inv_cv);
    if (fu1 < 0.0 || fv1 < 0.0 || fu0 > (double)(G.gu - 1) || fv0 > (double)(G.gv - 1)) return r;
    r.iu0 = (int)fmax(fu0, 0.0);
    r.iu1 = (int)fmin(fu1, (double)(G.gu - 1));
    const int iv0 = (int)fmax(fv0, 0.0), iv1 = (int)fmin(fv1, (double)(G.gv - 1));
    const int n = iv1 - iv0 + 1;
    const int lo = min(row_lo, n), hi = min(row_hi, n);  // an item may cover part of the rows only
    r.iv0 = iv0 + lo;
    r.nrows = max(hi - lo, 0);
    return r;
}

// Exact row of a staged candidate: aux = row of its catalog | catalog bit (SRec::aux).
#define YAWB_CAND_ROW(P, aux, X, Y, Z)                                         \
    do {                                                                       \
        const int cand_t_ = (int)((unsigned)(aux) >> 31);                      \
        const int cand_i_ = (int)((unsigned)(aux) & 0x7fffffffu);              \
        const double *cand_x_ = cand_t_ ? (P).cx[1] : (P).cx[0];               \
        const double *cand_y_ = cand_t_ ? (P).cy[1] : (P).cy[0];               \
        const double *cand_z_ = cand_t_ ? (P).cz[1] : (P).cz[0];               \
        const size_t cand_o_ = 3 * (size_t)cand_i_; /* interleaved rows */     \
        X = cand_x_[cand_o_]; Y = cand_y_[cand_o_]; Z = cand_z_[cand_o_];      \
    } while (0)

// Rows (and weights) of the second catalog a tile was cut from: `tl.patch` carries Item::src inside the streaming
// kernel (0 = first, 1 = second catalog of a joint launch).
#define YAWB_TILE_ROWS(P, tl) ((tl).patch ? (P).rx2 : (P).rx)
#define YAWB_TILE_WEIGHTS(P, tl) ((tl).patch ? (P).rw2 : (P).rw)

// The reference's comparison value: products rounded separately, summed x -> y -> z.
__device__ __forceinline__ double exact_d2(double ax, double ay, double az, double bx, double by, double bz) {
    double dx = __dsub_rn(ax, bx), dy = __dsub_rn(ay, by), dz = __dsub_rn(az, bz);
    return __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
}

// number of edges strictly below d2 (np.searchsorted(r2, d2, side="left"))
__device__ __forceinline__ int edges_below(const double *__restrict__ e, int n, double d2) {
    int lo = 0, hi = n;
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if (e[mid] < d2) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ double warp_sum(double v) {
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

// One staged candidate s, in the tile frame of the item (yawb_count_stream.cuh): (-2 s_x, -2 s_y, -2 (1 + s_z),
// |s|^2 - mid), so that for a row r of the tile  r . (x, y, z) + w = |r - s|^2 - mid  (the rows are unit vectors,
// their |r|^2 equals -2 r_z in this frame).  One broadcast LDS.128; the compiler duplicates the components into
// the register pairs of the packed f32x2 instructions.
typedef float4 Cand;
constexpr int HPL = YAWB_RPL / 2;  // row pairs per lane

// ---- the paths of the streaming kernel; the host picks one per count (yawb_launch_count_fast) ---------------
enum class CountPath {
    Single,             // unweighted, one sub-bin: saturating ramp (stream_test_sat)
    SingleUnion,        // the same on tiles over the union of two second catalogs: counts split by each row's catalog
    SingleWeighted,     // weighted, one sub-bin: predicated test, weighted sums (phase2_single)
    Cumulative,         // unweighted, a few sub-bins: cumulative counts with the saturating ramp (phase2_cumul)
    Histogram,          // unweighted, many sub-bins: in-range tests classified into a histogram (phase2_multi_queue)
    HistogramWeighted,  // weighted, several sub-bins: the same with weighted sums
};
__host__ __device__ constexpr bool path_weighted(CountPath p) {
    return p == CountPath::SingleWeighted || p == CountPath::HistogramWeighted;
}
__host__ __device__ constexpr bool path_sat(CountPath p) { return p == CountPath::Single || p == CountPath::SingleUnion; }
__host__ __device__ constexpr bool path_multi(CountPath p) { return !path_sat(p) && p != CountPath::SingleWeighted; }

// ---- a warp's block of shared memory in the streaming kernel (yawb_count_stream.cuh) ----------------------
constexpr int LB = 128;   // rows per raw chunk = capacity of the staged list
constexpr int NSLOT = 4;  // items in flight per warp: consumed, produced, planned, fetched

// The staged frame of an item ("tile frame"): origin O = the point of the unit sphere in the direction of the centre of
// the tile box, axes (t1, t2, n) with n = O - (centre of the sphere).  For a row P of the tile (a unit vector)
// |P - O|^2 = -2 (P - O).n, so the squared chord to a candidate s needs no |r|^2 term:
//     |r - s|^2 - mid = (|s|^2 - mid) + r . (-2 s_x, -2 s_y, -2 (1 + s_z))        (three FMAs per test)
struct __align__(16) ItemAux {
    double R[9];        // rows t1, t2, n of the tile frame, in coordinates of the frame of p1
    double O[3];        // origin of the tile frame, in coordinates of the frame of p1
    double dq[3];       // lattice origin - O:  (row of the index) - O = (k - ko) * qinv + dq
    int ko[3];          // lattice origin: the lattice point nearest to the centre of the tile box
    int n_combo;        // runs of the item
    float qinv;         // lattice spacing (a power of two)
    float eu, ev, et;   // half extents of the tile box about the lattice origin, rounded up
    float g;            // |lattice origin - O|, rounded up
    int end;            // 1: the work list is exhausted, this slot holds no item
    int pad[2];
};
static_assert(sizeof(ItemAux) % 16 == 0, "ItemAux layout");

struct __align__(16) SegDesc {
    short ea, eb;  // entries [ea, eb) of the staged list
    short bin;     // their z-bin
    short type;    // catalog of a fused first-role index (0 / 1)
};

struct StreamSmem {
    Item *items;               // [NSLOT]
    ItemAux *aux;              // [NSLOT]
    int *bin_iv0, *bin_iu;     // [n_bins] plan: first cell row of the query, iu0 | iu1 << 16
    int *cstart;               // [n_bins + 1] prefix of cell rows per z-bin
    int2 *cs;                  // [CCAP] cell_start at the two ends of every run (lands asynchronously)
    unsigned short *csbin;     // [CCAP] z-bin of the run
    int2 *run;                 // [CCAP] run table of the item being produced: (inclusive prefix of the run lengths,
                               //        row of the index that flat position 0 would have if the run started there)
    unsigned short *cbin;      // [CCAP]
    SRec *raw;                 // [LB] raw chunk (lands asynchronously)
    unsigned short *rawbin;    // [LB]
    double *rawlw;             // [LB] weights of the raw rows (weighted paths)
    Cand *list;                // [LB] staged candidates: type 0 from the bottom, type 1 from the top
    int *lidx;                 // [LB] row of the candidate in its catalog | catalog bit (SRec::aux)
    unsigned short *lbin;      // [LB]
    double *lw;                // [LB] (weighted paths)
    SegDesc *seg;              // [n_types * n_bins]
    float4 *binrec;            // [n_bins] half extents of the query box (x, y, z) and mid
    float2 *binthr;            // [n_bins] thresholds of the pair test
    unsigned long long *acc;   // [n_sec][n_types][n_bins * nsub]
    double *accw;              // same (weighted paths)
    unsigned *hist;            // [nsub] scratch histogram of one z-bin segment (sub-bin paths)
    double *histw;             // [nsub] (HistogramWeighted)
    float *cum;                // [n_bins][CUM_EDGES] ramp offsets K (e_k - mid) + 1/2 of the item (sub-bin paths)
    unsigned *cumtot;          // [CUM_EDGES] cumulative counts of one z-bin segment
};

// ---- exact re-evaluation of one lane's share of a chunk, done by the whole warp ----------------
// Lane `src` saw a test inside the FP32 uncertainty band.  Its (YAWB_RPL x chunk) tests are
// re-evaluated with the reference's FP64 expression, two or more per lane, and summed (weighted single-bin path).
__device__ __forceinline__ void recheck_chunk(const FastParams &P, const StreamSmem &S, int e0, int e1,
                                              const Tile &tl, int lane, int src, double lo, double hi,
                                              unsigned &cnt_out, double &w_out, unsigned &n_recheck) {
    unsigned cnt = 0;
    double wsum = 0.0;
    const double *const trow = YAWB_TILE_ROWS(P, tl);
    const double *const tw = YAWB_TILE_WEIGHTS(P, tl);
    for (int t = lane; t < CHUNK * YAWB_RPL; t += 32) {
        const int e = e0 + (t & (CHUNK - 1));
        const int k = src + 32 * (t / CHUNK);
        if (e < e1 && k < tl.count) {
            const int i = S.lidx[e], j = tl.start + k;
            double cxx, cyy, czz;
            YAWB_CAND_ROW(P, i, cxx, cyy, czz);
            const double d2 = exact_d2(cxx, cyy, czz, trow[(size_t)YAWB_RSTRIDE * j], trow[(size_t)YAWB_RSTRIDE * j + 1], trow[(size_t)YAWB_RSTRIDE * j + 2]);
            if (d2 > lo && d2 <= hi) {
                cnt += 1;
                wsum += S.lw[e] * (tw ? tw[j] : 1.0);
            }
            n_recheck += 1;
        }
    }
    cnt_out = __reduce_add_sync(FULL, cnt);
    w_out = warp_sum(wsum);
}

// The same for a span [e0, e1) of at most 16 entries (the streaming kernel checks once per <= 16 candidates): lane t
// takes row t & 7 of lane `src` against candidates t >> 3, t >> 3 + 4, ...; all operands of a lane's (up to four)
// tests are requested before the first is used, so the warp pays the memory latency once (unweighted single-bin path).
// The count is returned split by the catalog of the row in the index (the fourth double of its record): pairs with
// rows of catalog 0 in the low 16 bits, with rows of catalog 1 in the high 16 bits (stream_test_sat).
__device__ __forceinline__ void recheck_span(const FastParams &P, const StreamSmem &S, int e0, int e1,
                                             const Tile &tl, int lane, int src, double lo, double hi,
                                             unsigned &cnt_out, unsigned &n_recheck) {
    static_assert(YAWB_RPL == 8, "one lane per row of the flagged lane");
    constexpr int Q = 4;  // 16 candidates x 8 rows / 32 lanes
    unsigned cnt = 0;
    const int k = src + 32 * (lane & 7);
    const bool row_ok = k < tl.count;
    const int j = tl.start + (row_ok ? k : 0);
    const double2 *const row = reinterpret_cast<const double2 *>(YAWB_TILE_ROWS(P, tl) + (size_t)YAWB_RSTRIDE * j);
    const double2 ra = row[0], rb = row[1];
    const double bx = ra.x, by = ra.y, bz = rb.x;
    const unsigned one = rb.y != 0.0 ? 0x10000u : 1u;
    double ax[Q], ay[Q], az[Q];
    bool ok[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) {
        const int e = e0 + (lane >> 3) + 4 * q;
        ok[q] = row_ok && e < e1;
        const int i = S.lidx[ok[q] ? e : e0];
        YAWB_CAND_ROW(P, i, ax[q], ay[q], az[q]);
    }
#pragma unroll
    for (int q = 0; q < Q; ++q) {
        const double d2 = exact_d2(ax[q], ay[q], az[q], bx, by, bz);
        if (ok[q]) {
            if (d2 > lo && d2 <= hi) cnt += one;
            n_recheck += 1;
        }
    }
    cnt_out = __reduce_add_sync(FULL, cnt);
}

// ---- phase 2, single sub-bin (n_edges == 2): the hot loop ----------------------------------
// One candidate against the lane's YAWB_RPL rows:  u = (rn + s.w) + rx s.x + ry s.y + rz s.z = d2 - mid.
//   unweighted: v = sat(C - K |u|) is a ramp through the uncertainty band: exactly 1 well inside the bin,
//        exactly 0 well outside, in [0.1, 0.9] wherever FP32 cannot decide (K = 0.4 / eps,
//        C = 1/2 + h K).  sum(v) and sum(v*v) are equal iff every v of the chunk was 0 or 1 (then
//        sum(v) is the exact count); an undecidable test makes them differ by >= 0.09.  With NA = HPL accumulators
//        sum(v) is kept per register pair (rows 2k, 2k+1), so that the count splits by the catalog of each row;
//   weighted (predicated): |u| < h - eps, |u| < h + eps (2 FSETP) + 2 predicated FADD, also feeds the weighted sums.
//        Two accumulator pairs (even / odd rows) halve the length of the dependent add chains.
template <int NA>
__device__ __forceinline__ void test_candidate_sat(const Cand c, const float2 (&rx)[HPL], const float2 (&ry)[HPL],
                                                   const float2 (&rz)[HPL], float ta, float tb, float2 (&acc_a)[NA],
                                                   float2 &acc_b) {
    // Blackwell packed FP32: one FFMA2 / FADD2 carries two pair tests (rows 2k and 2k+1 of the lane)
    const float2 sx = make_float2(c.x, c.x), sy = make_float2(c.y, c.y);
    const float2 sz = make_float2(c.z, c.z), sw = make_float2(c.w, c.w);
#pragma unroll
    for (int k = 0; k < HPL; ++k) {
        float2 u = __ffma2_rn(rx[k], sx, sw);
        u = __ffma2_rn(ry[k], sy, u);
        u = __ffma2_rn(rz[k], sz, u);
        float2 v;
        v.x = __saturatef(fmaf(fabsf(u.x), ta, tb));  // ta = -K, tb = C
        v.y = __saturatef(fmaf(fabsf(u.y), ta, tb));
        acc_a[k % NA] = __fadd2_rn(acc_a[k % NA], v);
        acc_b = __ffma2_rn(v, v, acc_b);
    }
}

__device__ __forceinline__ void test_candidate_w(const Cand c, double swt, const float2 (&rx)[HPL],
                                                 const float2 (&ry)[HPL], const float2 (&rz)[HPL],
                                                 float ta, float tb, float2 &acc_a,
                                                 float2 &acc_b, double (&ws)[YAWB_RPL]) {
    const float2 sx = make_float2(c.x, c.x), sy = make_float2(c.y, c.y);
    const float2 sz = make_float2(c.z, c.z), sw = make_float2(c.w, c.w);
#pragma unroll
    for (int k = 0; k < HPL; ++k) {
        float2 u = __ffma2_rn(rx[k], sx, sw);
        u = __ffma2_rn(ry[k], sy, u);
        u = __ffma2_rn(rz[k], sz, u);
        const float a0 = fabsf(u.x), a1 = fabsf(u.y);
        const bool in0 = a0 < ta, in1 = a1 < ta;  // ta = h - eps, tb = h + eps
        if (in0) acc_a.x += 1.f;
        if (in1) acc_a.y += 1.f;
        if (a0 < tb) acc_b.x += 1.f;
        if (a1 < tb) acc_b.y += 1.f;
        // ws += [in] * swt as one select on the high word of a 0.0 / 1.0 double plus one DFMA (a
        // conditional FP64 add is lowered to an add plus two selects)
        ws[2 * k] = fma(__hiloint2double(in0 ? 0x3ff00000 : 0, 0), swt, ws[2 * k]);
        ws[2 * k + 1] = fma(__hiloint2double(in1 ? 0x3ff00000 : 0, 0), swt, ws[2 * k + 1]);
    }
}

// ---- phase 2, weighted, single sub-bin: entries [ea, eb) of the list belong to one z-bin ---------------
__device__ __forceinline__ void phase2_single(const FastParams &P, const StreamSmem &S, int ea, int eb,
                                              const float2 (&rx)[HPL], const float2 (&ry)[HPL],
                                              const float2 (&rz)[HPL],
                                              float ta, float tb, const Tile &tl, int lane, double lo,
                                              double hi, unsigned &cnt_total, double &w_total,
                                              unsigned &n_recheck, const double (&rwt)[YAWB_RPL]) {
    for (int e0 = ea; e0 < eb; e0 += CHUNK) {
        const int e1 = min(e0 + CHUNK, eb);
        float2 acc_a = make_float2(0.f, 0.f), acc_b = make_float2(0.f, 0.f);
        double ws[YAWB_RPL];
#pragma unroll
        for (int r = 0; r < YAWB_RPL; ++r) ws[r] = 0.0;
        if (e1 - e0 == CHUNK) {  // common case: fully unrolled, no loop bookkeeping
#pragma unroll
            for (int k = 0; k < CHUNK; ++k)
                test_candidate_w(S.list[e0 + k], S.lw[e0 + k], rx, ry, rz, ta, tb, acc_a, acc_b, ws);
        } else {
            for (int e = e0; e < e1; ++e)
                test_candidate_w(S.list[e], S.lw[e], rx, ry, rz, ta, tb, acc_a, acc_b, ws);
        }
        const float sa = acc_a.x + acc_a.y, sb = acc_b.x + acc_b.y;
        unsigned c = (unsigned)(sa + 0.5f);
        double wsum = 0.0;
#pragma unroll
        for (int r = 0; r < YAWB_RPL; ++r) wsum += ws[r] * rwt[r];  // row weights live in registers
        unsigned flagged = __ballot_sync(FULL, sa != sb);
        while (flagged) {  // warp-uniform: some lane met the uncertainty band of an edge
            const int src = __ffs(flagged) - 1;
            flagged &= flagged - 1;
            unsigned cx = 0;
            double wx = 0.0;
            recheck_chunk(P, S, e0, e1, tl, lane, src, lo, hi, cx, wx, n_recheck);
            if (lane == src) {
                c = cx;
                wsum = wx;
            }
        }
        cnt_total += c;
        w_total += wsum;
    }
}

// ---- phase 2, a few sub-bins (multi-scale without r-weights), unweighted: cumulative counts --------
// For up to CUM_EDGES edges the sub-bin histogram is obtained without classifying anything: for every edge
// e_k the pairs with d2 <= e_k are COUNTED with the same saturating ramp as in the single-bin test,
//     v_k = sat(K (e_k - mid - u) + 1/2),     sum(v_k) == sum(v_k^2)  <=>  every test was decided,
// G edges per pass over the chunk (the distance is recomputed per pass: 2 + 2 G FP32 lane-operations per
// test and pass; G is picked so that the edges need as few, as full passes as possible), and the histogram
// is the difference of neighbouring cumulative counts.  Undecided chunks are recounted exactly per lane as in the single-bin path.
constexpr int CUM_MAX_EDGES = 8;  // n_edges up to this selects the path
constexpr int CUM_EDGES = 16;     // table stride: room for the padded last group of any group size
constexpr int CUM_CHUNK = 8;

template <int G>
__device__ __forceinline__ void recheck_cumul(const FastParams &P, const int *lidx, int e0, int e1, const Tile &tl,
                                              int lane, int src, const double *ed, int k0, int ne,
                                              unsigned (&cnt_out)[G], unsigned &n_recheck) {
    unsigned cnt[G];
#pragma unroll
    for (int g = 0; g < G; ++g) cnt[g] = 0;
    const double *const trow = YAWB_TILE_ROWS(P, tl);
    for (int t = lane; t < CUM_CHUNK * YAWB_RPL; t += 32) {
        const int e = e0 + (t & (CUM_CHUNK - 1));
        const int k = src + 32 * (t / CUM_CHUNK);
        if (e < e1 && k < tl.count) {
            const int i = lidx[e], j = tl.start + k;
            double cxx, cyy, czz;
            YAWB_CAND_ROW(P, i, cxx, cyy, czz);
            const double d2 = exact_d2(cxx, cyy, czz, trow[(size_t)YAWB_RSTRIDE * j], trow[(size_t)YAWB_RSTRIDE * j + 1], trow[(size_t)YAWB_RSTRIDE * j + 2]);
#pragma unroll
            for (int g = 0; g < G; ++g)
                if (k0 + g < ne && d2 <= ed[k0 + g]) cnt[g] += 1;
            n_recheck += 1;
        }
    }
#pragma unroll
    for (int g = 0; g < G; ++g) cnt_out[g] = __reduce_add_sync(FULL, cnt[g]);
}

// entries [ea, eb) of the list belong to z-bin b; adds the sub-bin counts of the segment to acc
template <int CUM_GROUP>
__device__ __forceinline__ void phase2_cumul_g(const FastParams &P, const StreamSmem &S, unsigned long long *acc, int ea, int eb,
                                             const float2 (&rx)[HPL], const float2 (&ry)[HPL],
                                             const float2 (&rz)[HPL], float nk,
                                             const Tile &tl, int lane, int b, unsigned &n_recheck) {
    const int ne = P.n_edges;
    const double *ed = P.r2 + (size_t)b * ne;
    for (int k0 = 0; k0 < ne; k0 += CUM_GROUP) {
        float off[CUM_GROUP];
#pragma unroll
        for (int g = 0; g < CUM_GROUP; ++g) off[g] = S.cum[b * CUM_EDGES + k0 + g];
        unsigned cnt[CUM_GROUP];
#pragma unroll
        for (int g = 0; g < CUM_GROUP; ++g) cnt[g] = 0;
        for (int e0 = ea; e0 < eb; e0 += CUM_CHUNK) {
            const int e1 = min(e0 + CUM_CHUNK, eb);
            float2 acc_a[CUM_GROUP], acc_b[CUM_GROUP];
#pragma unroll
            for (int g = 0; g < CUM_GROUP; ++g) acc_a[g] = acc_b[g] = make_float2(0.f, 0.f);
            for (int e = e0; e < e1; ++e) {
                const Cand c = S.list[e];
                const float2 sx = make_float2(c.x, c.x), sy = make_float2(c.y, c.y);
                const float2 sz = make_float2(c.z, c.z), sw = make_float2(c.w, c.w);
#pragma unroll
                for (int k = 0; k < HPL; ++k) {
                    float2 u = __ffma2_rn(rx[k], sx, sw);
                    u = __ffma2_rn(ry[k], sy, u);
                    u = __ffma2_rn(rz[k], sz, u);
#pragma unroll
                    for (int g = 0; g < CUM_GROUP; ++g) {
                        float2 v;
                        v.x = __saturatef(fmaf(u.x, nk, off[g]));  // nk = -K
                        v.y = __saturatef(fmaf(u.y, nk, off[g]));
                        acc_a[g] = __fadd2_rn(acc_a[g], v);
                        acc_b[g] = __ffma2_rn(v, v, acc_b[g]);
                    }
                }
            }
            unsigned c[CUM_GROUP];
            bool bad = false;
#pragma unroll
            for (int g = 0; g < CUM_GROUP; ++g) {
                const float sa = acc_a[g].x + acc_a[g].y, sb = acc_b[g].x + acc_b[g].y;
                c[g] = (unsigned)(sa + 0.5f);
                bad = bad || sa != sb;
            }
            unsigned flagged = __ballot_sync(FULL, bad);
            while (flagged) {  // warp-uniform: some lane met the uncertainty band of an edge
                const int src = __ffs(flagged) - 1;
                flagged &= flagged - 1;
                unsigned cx[CUM_GROUP];
                recheck_cumul<CUM_GROUP>(P, S.lidx, e0, e1, tl, lane, src, ed, k0, ne, cx, n_recheck);
                if (lane == src) {
#pragma unroll
                    for (int g = 0; g < CUM_GROUP; ++g) c[g] = cx[g];
                }
            }
#pragma unroll
            for (int g = 0; g < CUM_GROUP; ++g) cnt[g] += c[g];
        }
#pragma unroll
        for (int g = 0; g < CUM_GROUP; ++g) {
            const unsigned tot = __reduce_add_sync(FULL, cnt[g]);
            if (lane == 0) S.cumtot[k0 + g] = tot;
        }
    }
    __syncwarp();
    // pairs with r2[s] < d2 <= r2[s + 1]: difference of the cumulative counts
    if (lane < ne - 1) acc[(size_t)b * (ne - 1) + lane] += (unsigned long long)(S.cumtot[lane + 1] - S.cumtot[lane]);
    __syncwarp();
}

__device__ __forceinline__ void phase2_cumul(const FastParams &P, const StreamSmem &S, unsigned long long *acc, int ea, int eb,
                                             const float2 (&rx)[HPL], const float2 (&ry)[HPL],
                                             const float2 (&rz)[HPL], float nk,
                                             const Tile &tl, int lane, int b, unsigned &n_recheck) {
    const int ne = P.n_edges;  // measured on C4 (6 edges): one pass of 6 beats two of 3 beats three of 2
    if (ne <= 3) phase2_cumul_g<3>(P, S, acc, ea, eb, rx, ry, rz, nk, tl, lane, b, n_recheck);
    else if (ne == 5 || ne == 6) phase2_cumul_g<6>(P, S, acc, ea, eb, rx, ry, rz, nk, tl, lane, b, n_recheck);
    else phase2_cumul_g<4>(P, S, acc, ea, eb, rx, ry, rz, nk, tl, lane, b, n_recheck);
}

// ---- phase 2, several sub-bins (r-weights, multi-scale): in-range tests queued warp-wide, classified 32 at a time ----
// With ~50 sub-bins the scale range of a z-bin is a wide annulus: some 11 % of the executed tests fall inside, spread
// over most of the eight row slots of a candidate, so classifying in place, inside the test loop (round 1), walked
// through the classification code for nearly every (candidate, row slot) with one lane in seven active (ncu: 2.15e10
// warp instructions per C3w count against 3.9e9 for the single-bin kernel, a quarter of them in the edge fix-up loop;
// C3w count kernels 38.5 ms against 34.7 with the queue).  Here every in-range test is appended to a queue of the warp
// (position by ballot + popcount; entry = d2 as float and candidate << 8 | row slot << 5 | lane), and whenever 32
// entries are waiting every lane classifies one.
template <bool WEIGHTED>
__device__ __forceinline__ void classify_queued(const FastParams &P, const StreamSmem &S, float d2f, unsigned code,
                                                float eps, const Tile &tl, const float *__restrict__ ef,
                                                const double *__restrict__ ed, const unsigned short *__restrict__ lgT,
                                                float lg_scale, float lg_off, int nc, int ne, const double *trow,
                                                const double *tw, unsigned &n_recheck) {
    const int e = (int)(code >> 8), r = (int)((code >> 5) & 7u), src_lane = (int)(code & 31u);
    const int cell = min(max((int)fmaf(__log2f(d2f), lg_scale, lg_off), 0), nc - 1);
    int k = lgT[cell];
    while (k < ne && ef[k] < d2f) ++k;
    float gap = FLT_MAX;
    if (k > 0) gap = fminf(gap, d2f - ef[k - 1]);
    if (k < ne) gap = fminf(gap, ef[k] - d2f);
    const int j = tl.start + min(src_lane + 32 * r, tl.count - 1);
    if (!(gap > eps)) {
        const int i = S.lidx[e];
        double cxx, cyy, czz;
        YAWB_CAND_ROW(P, i, cxx, cyy, czz);
        const double d2 = exact_d2(cxx, cyy, czz, trow[(size_t)YAWB_RSTRIDE * j], trow[(size_t)YAWB_RSTRIDE * j + 1], trow[(size_t)YAWB_RSTRIDE * j + 2]);
        k = edges_below(ed, ne, d2);
        n_recheck += 1;
    }
    if (k >= 1 && k < ne) {
        atomicAdd(&S.hist[k - 1], 1u);
        if (WEIGHTED) atomicAdd(&S.histw[k - 1], S.lw[e] * (tw ? tw[j] : 1.0));
    }
}

template <bool WEIGHTED>
__device__ __forceinline__ void phase2_multi_queue(const FastParams &P, const StreamSmem &S, int ea, int eb,
                                                   const float2 (&rx)[HPL], const float2 (&ry)[HPL],
                                                   const float2 (&rz)[HPL],
                                                   float h_out, float eps, float mid, const Tile &tl, int lane, int b,
                                                   unsigned &n_recheck) {
    const int ne = P.n_edges;
    const float *ef = P.r2f + (size_t)b * ne;
    const double *ed = P.r2 + (size_t)b * ne;
    const int nc = P.lg_cells;
    const float lg_scale = P.lgpar[2 * b], lg_off = P.lgpar[2 * b + 1];
    const unsigned short *lgT = P.lgT + (size_t)b * nc;
    const double *const trow = YAWB_TILE_ROWS(P, tl);
    const double *const tw = YAWB_TILE_WEIGHTS(P, tl);
    // the queue lives in the (otherwise unused) ramp table of the cumulative path: 64 floats + 64 codes
    float *const qd = S.cum;
    unsigned *const qc = reinterpret_cast<unsigned *>(S.cum + 64);
    const unsigned lt = (1u << lane) - 1u;
    int qn = 0;  // entries waiting (warp-uniform)
    for (int e = ea; e < eb; ++e) {
        const Cand c = S.list[e];
        const float2 sx = make_float2(c.x, c.x), sy = make_float2(c.y, c.y);
        const float2 sz = make_float2(c.z, c.z), sw = make_float2(c.w, c.w);
        float2 u2[HPL];
#pragma unroll
        for (int k = 0; k < HPL; ++k) {
            float2 u = __ffma2_rn(rx[k], sx, sw);
            u = __ffma2_rn(ry[k], sy, u);
            u2[k] = __ffma2_rn(rz[k], sz, u);
        }
#pragma unroll
        for (int r = 0; r < YAWB_RPL; ++r) {
            const float u = (r & 1) ? u2[r >> 1].y : u2[r >> 1].x;
            const bool in = fabsf(u) < h_out;  // possibly inside [lo, hi]; padding rows are NaN: never
            const unsigned mask = __ballot_sync(FULL, in);
            if (mask) {  // warp-uniform
                if (in) {
                    const int pos = qn + __popc(mask & lt);
                    qd[pos] = u + mid;
                    qc[pos] = ((unsigned)e << 8) | ((unsigned)r << 5) | (unsigned)lane;
                }
                qn += __popc(mask);
                if (qn >= 32) {
                    __syncwarp();
                    classify_queued<WEIGHTED>(P, S, qd[lane], qc[lane], eps, tl, ef, ed, lgT, lg_scale, lg_off, nc, ne, trow, tw, n_recheck);
                    qn -= 32;
                    float td = 0.f;
                    unsigned tc = 0u;
                    if (lane < qn) { td = qd[32 + lane]; tc = qc[32 + lane]; }
                    __syncwarp();
                    if (lane < qn) { qd[lane] = td; qc[lane] = tc; }
                }
            }
        }
    }
    __syncwarp();
    if (lane < qn) classify_queued<WEIGHTED>(P, S, qd[lane], qc[lane], eps, tl, ef, ed, lgT, lg_scale, lg_off, nc, ne, trow, tw, n_recheck);
    __syncwarp();
}

// ---- planner: work items of a pair count ---------------------------------------------------------------
// One thread per (patch pair, tile of the second catalog's patch).  The tile's bounding box, known in the frame
// of its own patch, is carried into the frame of the first catalog's patch as the hull of its eight rotated
// corners (a box is convex and the map is affine, so the hull contains every row).  The item survives if that
// box, grown by the largest search radius, meets the (u, v) box of the first catalog's patch and holds at least
// one cell row of some z-bin.  Items are split so that none exceeds CCAP (z-bin, cell row) runs: by z-bin
// ranges, and a single z-bin with more rows than that by row ranges.  Items of a patch with itself (nearly
// all of the work) are listed first, the boundary items of neighbouring patches after them, so that the tail of
// the launch consists of light items.
struct PlanParams {
    const Tile *tiles;
    const TileBox *tile_box;
    const int *ptile_off;
    const PatchFrame *frames2;  // frames of the second catalog (tile boxes live in these)
    const PatchFrame *frames1;  // frames of the first-role index
    const SGrid *sgrid;
    const int *pair_i, *pair_j;
    const long long *pair_item_base;
    int n_pairs;
    long long n_flat;
    const BinPar *binpar;
    int n_bins;
    double rmax_all;
    Item *heavy, *light;
    long long cap_heavy, cap_light;
    int ccap;  // (z-bin, cell row) runs per item: CCAP, or less to cut a small job into more, shorter items
    int src;   // which second catalog of a joint launch these tiles belong to (Item::src)
    int blk;     // first output block of that catalog (Item::blk)
    int labels;  // the tiles' z-bin ids are sample labels: paired with every z-bin, counts go to block blk + label
    int lab_bins;   // binned labels: a tile's id t is (label t / lab_bins, z-bin t % lab_bins); counts go to block
                    // blk + label (0: none)
    int lab_first;  // ... and the first catalog's ids are binned labels too: the item reads id label * lab_bins + z-bin
    unsigned long long *counters;
};

template <typename Emit>
__device__ __forceinline__ void plan_walk(const SGrid &G, const BinPar *__restrict__ binpar, int b_lo, int b_hi, double ulo,
                                          double uhi, double vlo, double vhi, int ccap, Emit emit) {
    int acc = 0, seg = b_lo;
    for (int b = b_lo; b < b_hi; ++b) {
        const int r = bin_rows(G, ulo, uhi, vlo, vhi, binpar[b], 0, INT_MAX).nrows;
        if (r > ccap) {
            if (acc > 0) emit(seg, b, 0, INT_MAX);
            for (int r0 = 0; r0 < r; r0 += ccap) emit(b, b + 1, r0, min(r0 + ccap, r));
            seg = b + 1;
            acc = 0;
        } else if (acc + r > ccap) {
            emit(seg, b, 0, INT_MAX);
            seg = b;
            acc = r;
        } else {
            acc += r;
        }
    }
    if (acc > 0) emit(seg, b_hi, 0, INT_MAX);
}

__global__ void __launch_bounds__(256) k_plan(const PlanParams Q) {
    const long long f = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    int n_emit = 0;
    bool heavy = false;
    Item it{};
    SGrid G{};
    if (f < Q.n_flat) {
        int lo = 0, hi = Q.n_pairs;  // last pair with pair_item_base[k] <= f
        while (hi - lo > 1) {
            const int m = (lo + hi) >> 1;
            if (Q.pair_item_base[m] <= f) lo = m; else hi = m;
        }
        const int k = lo;
        const int p1 = Q.pair_i[k], p2 = Q.pair_j[k];
        const int t = Q.ptile_off[p2] + (int)(f - Q.pair_item_base[k]);
        const Tile tl = Q.tiles[t];
        const PatchFrame &F1 = Q.frames1[p1];
        // z-bin of the tile (-1: paired with every z-bin of the first catalog) and its label (output block)
        const int zb = Q.lab_bins ? tl.bin % Q.lab_bins : Q.labels ? -1 : tl.bin;
        const int lab = Q.lab_bins ? tl.bin / Q.lab_bins : Q.labels && tl.bin >= 0 ? tl.bin : 0;
        const double rmax = zb >= 0 ? (Q.binpar[zb].empty ? 0.0 : Q.binpar[zb].rmax) : Q.rmax_all;
        // bounding spheres first (chord distances obey the triangle inequality)
        const double dx = (double)tl.cx - F1.c[0], dy = (double)tl.cy - F1.c[1], dz = (double)tl.cz - F1.c[2];
        const double reach = F1.radius + (double)tl.rad + rmax + 1e-9;
        if (rmax > 0.0 && dx * dx + dy * dy + dz * dz <= reach * reach) {
            const PatchFrame &F2 = Q.frames2[tl.patch];
            const TileBox bx = Q.tile_box[t];
            double lo3[3] = {1e300, 1e300, 1e300}, hi3[3] = {-1e300, -1e300, -1e300};
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const double u = (c & 1) ? bx.hi[0] : bx.lo[0], v = (c & 2) ? bx.hi[1] : bx.lo[1], w = (c & 4) ? bx.hi[2] : bx.lo[2];
                // corner in world coordinates, then relative to the centre of the first catalog's patch
                const double X = F2.c[0] + u * F2.e1[0] + v * F2.e2[0] + w * F2.c[0] - F1.c[0];
                const double Y = F2.c[1] + u * F2.e1[1] + v * F2.e2[1] + w * F2.c[1] - F1.c[1];
                const double Z = F2.c[2] + u * F2.e1[2] + v * F2.e2[2] + w * F2.c[2] - F1.c[2];
                const double q[3] = {X * F1.e1[0] + Y * F1.e1[1] + Z * F1.e1[2], X * F1.e2[0] + Y * F1.e2[1] + Z * F1.e2[2],
                                     X * F1.c[0] + Y * F1.c[1] + Z * F1.c[2]};
#pragma unroll
                for (int d = 0; d < 3; ++d) {
                    lo3[d] = fmin(lo3[d], q[d]);
                    hi3[d] = fmax(hi3[d], q[d]);
                }
            }
#pragma unroll
            for (int d = 0; d < 3; ++d) {  // far more than the rounding of the two rotations
                const double pad = 1e-14 + 1e-12 * fmax(fabs(lo3[d]), fabs(hi3[d]));
                lo3[d] -= pad;
                hi3[d] += pad;
            }
            if (lo3[0] - rmax <= F1.umax && hi3[0] + rmax >= F1.umin && lo3[1] - rmax <= F1.vmax && hi3[1] + rmax >= F1.vmin) {
                G = Q.sgrid[p1];
                it.pair = k; it.p1 = p1; it.start = tl.start; it.count = tl.count; it.src = Q.src;
                it.blk = Q.blk + lab;
                it.b_off = Q.lab_first ? lab * Q.lab_bins : 0;
                it.b_lo = zb >= 0 ? zb : 0;
                it.b_hi = zb >= 0 ? zb + 1 : Q.n_bins;
#pragma unroll
                for (int d = 0; d < 3; ++d) { it.lo[d] = lo3[d]; it.hi[d] = hi3[d]; }
                heavy = p1 == p2;
                plan_walk(G, Q.binpar, it.b_lo, it.b_hi, lo3[0], hi3[0], lo3[1], hi3[1], Q.ccap, [&](int, int, int, int) { ++n_emit; });
            }
        }
    }
    // one atomic per warp and list
    int pre_h = heavy ? n_emit : 0, pre_l = heavy ? 0 : n_emit;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int vh = __shfl_up_sync(FULL, pre_h, o), vl = __shfl_up_sync(FULL, pre_l, o);
        if (lane >= o) { pre_h += vh; pre_l += vl; }
    }
    const int tot_h = __shfl_sync(FULL, pre_h, 31), tot_l = __shfl_sync(FULL, pre_l, 31);
    if (tot_h + tot_l == 0) return;
    unsigned long long base_h = 0, base_l = 0;
    if (lane == 0) {
        if (tot_h) base_h = atomicAdd(&Q.counters[4], (unsigned long long)tot_h);
        if (tot_l) base_l = atomicAdd(&Q.counters[5], (unsigned long long)tot_l);
    }
    base_h = __shfl_sync(FULL, base_h, 0);
    base_l = __shfl_sync(FULL, base_l, 0);
    if (n_emit == 0) return;
    long long pos = heavy ? (long long)base_h + pre_h - n_emit : (long long)base_l + pre_l - n_emit;
    Item *const out = heavy ? Q.heavy : Q.light;
    const long long cap = heavy ? Q.cap_heavy : Q.cap_light;
    plan_walk(G, Q.binpar, it.b_lo, it.b_hi, it.lo[0], it.hi[0], it.lo[1], it.hi[1], Q.ccap, [&](int b0, int b1, int r0, int r1) {
        if (pos < cap) {
            Item w = it;
            w.b_lo = b0; w.b_hi = b1; w.row_lo = r0; w.row_hi = r1;
            out[pos] = w;
        } else {
            Q.counters[6] = 1ull;  // list too small: the host repeats the call with the exact sizes
        }
        ++pos;
    });
}

#include "yawb_count_stream.cuh"

// ---- exact all-pairs kernel -------------------------------------------------------------------
struct ExactParams {
    const double *cx, *cy, *cz;  // rows of the first catalog as uploaded; SRec::aux of a sorted row is its row there
    const SRec *rec;
    const double *sw;
    const int *s_seg;  // [(P * B1) + 1]
    const double *rx, *ry, *rz, *rw;
    const int *r_seg;  // [(P * B2) + 1]
    int b1, b2;        // bins of cat1 / cat2 (b2 == 1 for unbinned)
    const int *pair_i, *pair_j;
    int n_pairs, n_bins, n_edges;
    const double *r2;
    unsigned long long *out_cnt;
    double *out_w;
    unsigned long long *counters;
};

constexpr int EX_THREADS = 256;

template <bool WEIGHTED>
__global__ void __launch_bounds__(EX_THREADS) k_count_exact(const ExactParams P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int ne = P.n_edges, nsub = ne - 1;
    double *edges = (double *)smem_raw;
    double *tile = edges + ne;                       // [4][EX_THREADS] x, y, z, w
    double *histw = tile + 4 * EX_THREADS;           // [nsub]
    unsigned long long *hist = (unsigned long long *)(histw + nsub);  // [nsub]

    const int k = blockIdx.x / P.n_bins, b = blockIdx.x % P.n_bins;
    const int p1 = P.pair_i[k], p2 = P.pair_j[k];
    const int a0 = P.s_seg[p1 * P.b1 + b], a1 = P.s_seg[p1 * P.b1 + b + 1];
    const int c0 = P.b2 > 1 ? P.r_seg[p2 * P.b2 + b] : P.r_seg[p2];
    const int c1 = P.b2 > 1 ? P.r_seg[p2 * P.b2 + b + 1] : P.r_seg[p2 + 1];
    if (a0 >= a1 || c0 >= c1) return;
    if ((long long)blockIdx.y * EX_THREADS >= (a1 - a0)) return;

    for (int e = threadIdx.x; e < ne; e += EX_THREADS) edges[e] = P.r2[(size_t)b * ne + e];
    for (int e = threadIdx.x; e < nsub; e += EX_THREADS) { hist[e] = 0ull; histw[e] = 0.0; }
    __syncthreads();
    const double lo = edges[0], hi = edges[nsub];
    unsigned long long tests = 0;

    for (int ia = a0 + blockIdx.y * EX_THREADS; ia < a1; ia += gridDim.y * EX_THREADS) {
        const int i = ia + threadIdx.x;
        const bool live = i < a1;
        double ax = 0, ay = 0, az = 0, aw = 1.0;
        if (live) {
            const int row = (int)(P.rec[i].aux & 0x7fffffffu);
            ax = P.cx[3 * (size_t)row]; ay = P.cy[3 * (size_t)row]; az = P.cz[3 * (size_t)row];  // interleaved rows
            if (WEIGHTED && P.sw) aw = P.sw[i];
        }
        for (int jc = c0; jc < c1; jc += EX_THREADS) {
            const int nj = min(EX_THREADS, c1 - jc);
            __syncthreads();
            if ((int)threadIdx.x < nj) {
                const int j = jc + threadIdx.x;
                tile[threadIdx.x] = P.rx[(size_t)YAWB_RSTRIDE * j];
                tile[EX_THREADS + threadIdx.x] = P.ry[(size_t)YAWB_RSTRIDE * j];
                tile[2 * EX_THREADS + threadIdx.x] = P.rz[(size_t)YAWB_RSTRIDE * j];
                tile[3 * EX_THREADS + threadIdx.x] = (WEIGHTED && P.rw) ? P.rw[j] : 1.0;
            }
            __syncthreads();
            if (live) {
                for (int jj = 0; jj < nj; ++jj) {
                    const double d2 = exact_d2(ax, ay, az, tile[jj], tile[EX_THREADS + jj], tile[2 * EX_THREADS + jj]);
                    if (d2 > lo && d2 <= hi) {
                        const int kk = nsub == 1 ? 1 : edges_below(edges, ne, d2);
                        atomicAdd(&hist[kk - 1], 1ull);
                        if (WEIGHTED) atomicAdd(&histw[kk - 1], aw * tile[3 * EX_THREADS + jj]);
                    }
                }
                tests += nj;
            }
        }
    }
    __syncthreads();
    for (int e = threadIdx.x; e < nsub; e += EX_THREADS) {
        const size_t o = ((size_t)k * P.n_bins + b) * nsub + e;
        if (hist[e]) atomicAdd(&P.out_cnt[o], hist[e]);
        if (WEIGHTED && histw[e] != 0.0) atomicAdd(&P.out_w[o], histw[e]);
    }
    for (int o = 16; o; o >>= 1) tests += __shfl_xor_sync(FULL, tests, o);
    if ((threadIdx.x & 31) == 0 && tests) atomicAdd(&P.counters[1], tests);
}

}  // namespace

// -----------------------------------------------------------------------------------------------
int yawb_launch_count_fast(yawb_ctx *ctx, const CountArgs &a, int *launches) {
    YawbRange range("yawb:plan+count");
    const FIndex *fi = a.c1;
    FastParams P{};
    P.cx[0] = fi->a->x; P.cy[0] = fi->a->y; P.cz[0] = fi->a->z;
    P.cx[1] = fi->b ? fi->b->x : fi->a->x; P.cy[1] = fi->b ? fi->b->y : fi->a->y; P.cz[1] = fi->b ? fi->b->z : fi->a->z;
    P.sw = fi->sw; P.rec = fi->rec;
    P.cell_start = fi->cell_start; P.sgrid = fi->d_sgrid; P.sframe = fi->d_frames; P.n_types = fi->n_types;
    P.rx = a.r2[0]->rx; P.rw = a.r2[0]->rw;
    P.rx2 = P.rx; P.rw2 = P.rw;
    if (a.r2[1]) { P.rx2 = a.r2[1]->rx; P.rw2 = a.r2[1]->rw; }
    P.n_sec = a.r2[0]->b ? 2 : 1;
    {
        // the pair test takes |r|^2 of a tile row from the identity for unit vectors (yawb_count_stream.cuh); rows
        // off the unit sphere by zeta widen the band of tests that are re-evaluated in FP64 (1e-15: the frames'
        // own deviation from orthonormality)
        double zeta = 0.0;
        for (const PatchFrame &f : a.c2->h_frames) zeta = std::max(zeta, f.norm_dev);
        if (a.c2b)
            for (const PatchFrame &f : a.c2b->h_frames) zeta = std::max(zeta, f.norm_dev);
        P.zeta = (float)(zeta + 1.0e-15) * 1.000001f;
    }
    P.n_pairs = a.n_pairs; P.n_bins = a.n_bins; P.n_edges = a.n_edges;
    P.r2 = a.d_r2; P.r2f = a.d_r2f; P.binpar = a.d_binpar; P.rmax_all = a.rmax_all;
    P.lg_cells = a.n_edges > 2 ? YAWB_LG_CELLS_PER_EDGE * a.n_edges : 0;
    P.lgpar = a.d_r2f + (size_t)a.n_bins * a.n_edges;
    P.lgT = reinterpret_cast<const unsigned short *>(P.lgpar + 2 * (size_t)a.n_bins);
    P.out_cnt = a.d_out_cnt; P.out_w = a.d_out_w; P.counters = ctx->d_counters;
    P.type_stride = (size_t)a.n_pairs * a.n_bins * (a.n_edges - 1);
    const long long n_items_all = a.n_items + a.n_items_b;
    if (n_items_all == 0) return 0;

    // planner: self-contained work items (patch-diagonal ones first)
    // a small job (a rank's share of a strong-scaling run) is cut into more, shorter items, so that the warps of
    // the persistent grid finish together: below SMALL_JOB_ITEMS flat (pair, tile) combinations per warp the
    // items hold at most CCAP_SMALL runs (swept on an eighth of C3: 16 / 24 / 32 / 48 / 72 / 112 runs ->
    // count kernels 1.02 / 1.01 / 1.05 / 1.10 / 1.18 / 1.17 ms); the lists grow by the same factor
    const long long warps = (long long)ctx->sms * STREAM_CTAS * STREAM_WARPS;
    const int ccap = n_items_all < SMALL_JOB_ITEMS * warps ? CCAP_SMALL : CCAP;
    const long long cap_scale = (CCAP + ccap - 1) / ccap;
    const long long cap_heavy = a.cap_heavy * cap_scale, cap_light = a.cap_light * cap_scale;
    Item *d_items = nullptr;
    if (yawb_dalloc(ctx, (void **)&d_items, (size_t)(cap_heavy + cap_light) * sizeof(Item), ctx->stream)) return 1;
    P.items_heavy = d_items;
    P.items_light = d_items + cap_heavy;
    P.cap_heavy = cap_heavy; P.cap_light = cap_light;
    for (int sc = 0; sc < 2; ++sc) {  // one planner launch per second-role index, both append to the same two lists
        const RIndex *ri = a.r2[sc];
        const long long n_flat = sc ? a.n_items_b : a.n_items;
        if (!ri || n_flat == 0) continue;
        PlanParams Q{};
        Q.tiles = ri->d_tiles; Q.tile_box = ri->d_tile_box; Q.ptile_off = ri->d_ptile_off;
        Q.frames2 = ri->d_frames; Q.frames1 = fi->d_frames; Q.sgrid = fi->d_sgrid;
        Q.pair_i = a.d_pair_i; Q.pair_j = a.d_pair_j; Q.pair_item_base = sc ? a.d_pair_item_base_b : a.d_pair_item_base;
        Q.n_pairs = a.n_pairs; Q.n_flat = n_flat; Q.binpar = a.d_binpar; Q.n_bins = a.n_bins; Q.rmax_all = a.rmax_all;
        Q.heavy = d_items; Q.light = d_items + cap_heavy; Q.cap_heavy = cap_heavy; Q.cap_light = cap_light;
        Q.counters = ctx->d_counters;
        Q.ccap = ccap;
        Q.src = sc;
        Q.blk = sc ? a.blk_b : 0;
        Q.labels = a.labels ? 1 : 0;
        Q.lab_bins = a.lab_bins;
        Q.lab_first = a.lab_first ? 1 : 0;
        k_plan<<<(unsigned)((n_flat + 255) / 256), 256, 0, ctx->stream>>>(Q);
        *launches += 1;
    }

    if (cudaEventRecord(ctx->ev_plan, ctx->stream) == cudaSuccess) ctx->ev_plan_set = true;

    const bool multi = a.n_edges > 2;
    const int nsub = a.n_edges - 1;
    // few sub-bins (multi-scale without r-weights): cumulative counts with the saturating test
    const bool cumul = multi && !a.weighted && a.n_edges <= CUM_MAX_EDGES;
    {
        // many z-bins x sub-bins: per-warp accumulators in shared memory would cost most of the occupancy, so
        // the general sub-bin path sends every segment histogram straight to global atomics instead
        const size_t acc_bytes = (size_t)fi->n_types * a.n_bins * nsub * (a.weighted ? 16 : 8);
        P.acc_global = multi && !cumul && acc_bytes > 2048;
        const size_t per_warp = stream_carve(nullptr, nullptr, a.weighted, multi, a.n_bins, nsub, fi->n_types, P.n_sec,
                                             P.acc_global);
        const size_t smem = STREAM_WARPS * per_warp;
        YAWB_REQUIRE(smem <= 227 * 1024, "too many z-bins x sub-bins for the shared-memory accumulators (%zu B)", smem);
        // persistent grid: a multiple of the SM count, warps pull items from a global counter
        const int per_sm = std::max(1, std::min(STREAM_CTAS, (int)((227 * 1024) / (smem + 1024))));
        const int ctas = ctx->sms * per_sm;
#define LAUNCH(PATH)                                                                                         \
    do {                                                                                                     \
        YAWB_CUDA(cudaFuncSetAttribute(k_count_stream<PATH>, cudaFuncAttributeMaxDynamicSharedMemorySize,    \
                                       (int)smem));                                                          \
        k_count_stream<PATH><<<ctas, STREAM_WARPS * 32, smem, ctx->stream>>>(P);                            \
    } while (0)
        if (a.weighted) {
            if (multi) LAUNCH(CountPath::HistogramWeighted); else LAUNCH(CountPath::SingleWeighted);
        } else if (cumul) {
            LAUNCH(CountPath::Cumulative);
        } else if (multi) {
            LAUNCH(CountPath::Histogram);
        } else if (P.n_sec == 2) {  // the per-chunk split by catalog costs the single-catalog launches 7 % (C3wt RR)
            LAUNCH(CountPath::SingleUnion);
        } else {
            LAUNCH(CountPath::Single);
        }
#undef LAUNCH
    }
    yawb_dfree(ctx, d_items, ctx->stream);
    YAWB_CUDA(cudaGetLastError());
    *launches += 1;
    return 0;
}

int yawb_launch_count_exact(yawb_ctx *ctx, const CountArgs &a, int *launches) {
    YawbRange range("yawb:count_exact");
    ExactParams P{};
    P.cx = a.c1_cat->x; P.cy = a.c1_cat->y; P.cz = a.c1_cat->z; P.rec = a.c1->rec;
    P.sw = a.c1->sw; P.s_seg = a.c1_cat->d_seg_off;
    P.rx = a.c2->ri.rx; P.ry = a.c2->ri.ry; P.rz = a.c2->ri.rz; P.rw = a.c2->ri.rw; P.r_seg = a.c2->second_d_seg_off();
    P.b1 = a.c1_cat->n_bins; P.b2 = a.c2->n_bins;
    P.pair_i = a.d_pair_i; P.pair_j = a.d_pair_j;
    P.n_pairs = a.n_pairs; P.n_bins = a.n_bins; P.n_edges = a.n_edges;
    P.r2 = a.d_r2; P.out_cnt = a.d_out_cnt; P.out_w = a.d_out_w; P.counters = ctx->d_counters;
    if (a.n_pairs == 0) return 0;

    // rows of the largest (patch, bin) segment of cat1 decide grid.y
    int max_seg = 0;
    for (size_t s = 0; s + 1 < a.c1_cat->h_seg_off.size(); ++s)
        max_seg = std::max(max_seg, a.c1_cat->h_seg_off[s + 1] - a.c1_cat->h_seg_off[s]);
    int gy = std::max(1, std::min(64, (max_seg + EX_THREADS - 1) / EX_THREADS));
    const int nsub = a.n_edges - 1;
    const size_t smem = (size_t)(a.n_edges + 4 * EX_THREADS + nsub) * sizeof(double) + (size_t)nsub * 8;
    dim3 grid((unsigned)(a.n_pairs * a.n_bins), (unsigned)gy);
    if (a.weighted)
        k_count_exact<true><<<grid, EX_THREADS, smem, ctx->stream>>>(P);
    else
        k_count_exact<false><<<grid, EX_THREADS, smem, ctx->stream>>>(P);
    YAWB_CUDA(cudaGetLastError());
    *launches += 1;
    return 0;
}

// Upper bound on the device bytes of one count call (yawb_count_footprint): the blocks count_impl (yawb_api.cu) and
// yawb_launch_count_fast request, rounded as the allocator rounds them.
int64_t yawb_count_workspace(int sms, int64_t n_items, int n_pairs, int n_bins, int n_edges, int n_blocks, bool weighted) {
    const size_t np = (size_t)std::max(n_pairs, 1), B = (size_t)std::max(n_bins, 1), ne = (size_t)std::max(n_edges, 2);
    const size_t lg_cells = ne > 2 ? YAWB_LG_CELLS_PER_EDGE * ne : 0;
    const size_t r2f_words = B * ne + 2 * B + (B * lg_cells + 1) / 2;
    auto up16 = [](size_t b) { return (b + 15) & ~(size_t)15; };
    const size_t tab = 2 * up16(np * sizeof(int)) + up16(2 * (np + 1) * sizeof(long long)) + up16(B * ne * sizeof(double)) +
                       up16(r2f_words * sizeof(float)) + up16(B * sizeof(BinPar));
    const size_t n_out = std::max<size_t>((size_t)std::max(n_blocks, 1) * np * B * (ne - 1), 1);
    // work-item lists: 4 per diagonal and 2 per other (pair, tile) combination plus 1024 each; a job below
    // SMALL_JOB_ITEMS items per warp gets lists CCAP / CCAP_SMALL times longer.  The launch decides from the real item
    // count, the caller knows an upper bound n of it, so the bound takes the larger of both regimes up to n: the
    // result does not decrease with n and covers every real count up to n on either side of the threshold
    const size_t items = (size_t)std::max<int64_t>(n_items, 0);
    const size_t small = (size_t)SMALL_JOB_ITEMS * std::max(sms, 1) * STREAM_CTAS * STREAM_WARPS - 1;
    const size_t scale = (CCAP + CCAP_SMALL - 1) / CCAP_SMALL;
    const size_t item_bytes = std::max(4 * items + 2048, scale * (4 * std::min(items, small) + 2048)) * sizeof(Item);
    size_t total = yawb_dcache_round(tab) + yawb_dcache_round(n_out * sizeof(unsigned long long)) +
                   yawb_dcache_round(item_bytes);
    if (weighted) total += yawb_dcache_round(n_out * sizeof(double));
    return (int64_t)total;
}
