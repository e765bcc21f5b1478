// Catalog upload and device-side index construction.
//
// Replaces the reference's tree build (src/yaw/catalog/trees.py:365-429,
// BinnedTrees.build :483-545, Catalog.build_trees catalog.py:1406-1460): instead of
// one pickled cKDTree per (patch, z-bin) the rows stay resident in HBM in two sort
// orders, each built by a counting sort (one histogram pass, one scan, one scatter pass):
//
//   first role  (cat1 of yawb_count): rows sorted by global sky-cell id
//               (patch, z-bin, row-major cell of a per-patch tangent-plane grid),
//               plus cell_start[] -- a range query is one contiguous run per cell row;
//   second role (cat2): rows sorted by (patch, z-bin, Hilbert index) and cut into
//               register tiles of YAWB_TILE compact points with a bounding sphere.
//
// Everything here is HBM-bound streaming work: coalesced SoA double arrays, one pass
// per step, grids sized from the row count.
#include <algorithm>
#include <cmath>
#include <cstring>

#include "yawb_internal.cuh"

namespace {

constexpr int kThreads = 256;
constexpr double kTargetPerCell = 5.5;  // rows per sky cell and z-bin the grid is sized for
constexpr long long kMaxCellsPerPatchBin = 1ll << 24;
constexpr long long kMaxGridCells = 1ll << 30;  // sky cells of a first-role index, all patches and z-bins
constexpr double kCellAspect = 4.0;  // cell height / cell width

inline int blocks_for(int64_t n, int per_block = kThreads) {
    return (int)std::min<int64_t>((n + per_block - 1) / per_block, 1 << 30);
}

// Catalog buffers come from the context's caching allocator (yawb_alloc.cu): building and dropping
// indexes costs no device synchronisation and no driver round trips after the first use.
template <typename T>
int dev_alloc(yawb_cat *cat, T **ptr, size_t count, cudaStream_t stream = nullptr) {
    *ptr = nullptr;
    if (count == 0) count = 1;
    if (yawb_dalloc(cat->ctx, (void **)ptr, count * sizeof(T), stream ? stream : cat->ctx->stream)) return 1;
    cat->device_bytes += (int64_t)(count * sizeof(T));
    return 0;
}

template <typename T>
void dev_free(yawb_cat *cat, T *&ptr, size_t count) {
    if (ptr) {
        yawb_dfree(cat->ctx, ptr, cat->ctx->stream);
        cat->device_bytes -= (int64_t)(std::max<size_t>(count, 1) * sizeof(T));
        ptr = nullptr;
    }
}

// scratch that lives for one call
struct Scratch {
    yawb_ctx *ctx;
    cudaStream_t st;
    std::vector<void *> ptrs;
    Scratch(yawb_ctx *c, cudaStream_t s) : ctx(c), st(s) {}
    template <typename T>
    T *get(size_t count) {
        void *p = nullptr;
        if (yawb_dalloc(ctx, &p, std::max<size_t>(count, 1) * sizeof(T), st)) return nullptr;
        ptrs.push_back(p);
        return (T *)p;
    }
    ~Scratch() {
        for (void *p : ptrs) yawb_dfree(ctx, p, st);
    }
};

// order-preserving map double -> uint64 so atomicMin/Max work on doubles
__device__ __forceinline__ unsigned long long enc_double(double v) {
    unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
// ---- upload kernels ---------------------------------------------------------------------
// The rows stay interleaved as uploaded (xyz[3 i + 0 / 1 / 2]): consecutive threads read consecutive rows, so a
// warp's three loads cover 768 contiguous bytes between them.  k_patch_ids: the patch id of every row from the row
// offsets.

// z-bin ids that travelled as bytes (a quarter of the PCIe traffic of int32): widen; ids >= n_bins stay out of range
__global__ void k_widen_bins(const unsigned char *__restrict__ b8, long long n, int *__restrict__ bin) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) bin[i] = (int)b8[i];
}

// z-bin of every row from its redshift: np.digitize(z, edges, right) - 1 (src/yaw/catalog/trees.py:408-414).
// right: bin b holds edges[b] < z <= edges[b + 1], i.e. (number of edges strictly below z) - 1; otherwise
// edges[b] <= z < edges[b + 1], i.e. (number of edges <= z) - 1.  Comparisons only: identical to numpy's ids;
// NaN compares false everywhere and lands in bin -1 (numpy: past the last bin), dropped either way.
__global__ void k_digitize(const double *__restrict__ z, long long n, const double *__restrict__ edges, int n_edges,
                           int right, int *__restrict__ bin) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double v = z[i];
    int lo = 0, hi = n_edges;  // number of edges e with e < v (right) or e <= v
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const double e = edges[mid];
        if (right ? (e < v) : (e <= v)) lo = mid + 1; else hi = mid;
    }
    bin[i] = lo - 1;
}

__global__ void k_patch_ids(const long long *__restrict__ patch_off, int n_patch, long long n, int *__restrict__ patch) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    int lo = 0, hi = n_patch;  // last p with patch_off[p] <= i
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (patch_off[mid] <= i) lo = mid; else hi = mid;
    }
    patch[i] = lo;
}

// per patch: sum of unit vectors; per (bin, patch): row count and sum of weights.
// A block owns kSumRows consecutive rows.  Rows are grouped by patch, so a block nearly always meets one patch or
// two (a boundary inside its range): the rows of its FIRST and of its LAST patch are accumulated in registers /
// shared memory and flushed with one global atomic per quantity; only rows of a third patch in between (patches
// smaller than a block) go to global memory one by one.  (Round 1 sent every row behind the boundary to global
// atomics on the same few addresses: ~2000 serialised atomics per address and boundary, 90 us per launch
// whatever the catalog size.)
constexpr int kSumRows = 4096;
constexpr int kSumBatch = 4;  // rows in flight per thread
constexpr int kSumMaxBins = 1024;

__global__ void __launch_bounds__(kThreads) k_patch_sums(
    const double *__restrict__ x, const double *__restrict__ y, const double *__restrict__ z,
    const double *__restrict__ w, const int *__restrict__ bin, const int *__restrict__ patch, long long n,
    int n_patch, int n_bins, double *__restrict__ sums /*[n_patch][3]*/, unsigned long long *__restrict__ counts,
    double *__restrict__ sumw) {
    extern __shared__ unsigned char sm_raw[];
    const bool use_smem = n_bins <= kSumMaxBins;
    const int nb = use_smem ? n_bins : 0;
    // two slots (first / last patch of the block): [2][4] sums, [2][nb] weights (if weighted), [2][nb] counts
    double *s_xyz = (double *)sm_raw;
    double *s_w = s_xyz + 8;
    unsigned *s_cnt = (unsigned *)(s_w + (w ? 2 * nb : 0));
    const long long row0 = (long long)blockIdx.x * kSumRows;
    const long long row1 = min(row0 + (long long)kSumRows, n);
    const int p_blk = patch[row0], p_end = patch[row1 - 1];
    if (threadIdx.x < 8) s_xyz[threadIdx.x] = 0.0;
    for (int b = threadIdx.x; b < 2 * nb; b += blockDim.x) {
        s_cnt[b] = 0u;
        if (w) s_w[b] = 0.0;
    }
    __syncthreads();
    double ax = 0.0, ay = 0.0, az = 0.0, bx = 0.0, by = 0.0, bz = 0.0;
    // kSumBatch rows per thread and round, every load of a round requested before the first is used
    for (int k0 = threadIdx.x; k0 < kSumRows; k0 += kSumBatch * blockDim.x) {
        int p[kSumBatch], b[kSumBatch];
        double X[kSumBatch], Y[kSumBatch], Z[kSumBatch], W[kSumBatch];
#pragma unroll
        for (int q = 0; q < kSumBatch; ++q) {
            const long long i = row0 + k0 + q * (int)blockDim.x;
            const bool ok = k0 + q * (int)blockDim.x < kSumRows && i < n;
            p[q] = ok ? patch[i] : -1;
            b[q] = ok && bin ? bin[i] : 0;
            X[q] = ok ? x[3 * i] : 0.0;
            Y[q] = ok ? y[3 * i] : 0.0;
            Z[q] = ok ? z[3 * i] : 0.0;
            W[q] = ok && w ? w[i] : 0.0;
        }
#pragma unroll
        for (int q = 0; q < kSumBatch; ++q) {
            if (p[q] < 0) continue;
            const bool in_bin = b[q] >= 0 && b[q] < n_bins;
            const int slot = p[q] == p_blk ? 0 : p[q] == p_end ? 1 : -1;
            if (slot == 0) { ax += X[q]; ay += Y[q]; az += Z[q]; }
            else if (slot == 1) { bx += X[q]; by += Y[q]; bz += Z[q]; }
            else {
                atomicAdd(&sums[3 * p[q]], X[q]);
                atomicAdd(&sums[3 * p[q] + 1], Y[q]);
                atomicAdd(&sums[3 * p[q] + 2], Z[q]);
            }
            if (in_bin) {
                if (slot >= 0 && use_smem) {
                    atomicAdd(&s_cnt[slot * nb + b[q]], 1u);
                    if (w) atomicAdd(&s_w[slot * nb + b[q]], W[q]);
                } else {
                    atomicAdd(&counts[(size_t)b[q] * n_patch + p[q]], 1ull);
                    if (w) atomicAdd(&sumw[(size_t)b[q] * n_patch + p[q]], W[q]);
                }
            }
        }
    }
    for (int o = 16; o; o >>= 1) {
        ax += __shfl_xor_sync(0xffffffffu, ax, o);
        ay += __shfl_xor_sync(0xffffffffu, ay, o);
        az += __shfl_xor_sync(0xffffffffu, az, o);
        bx += __shfl_xor_sync(0xffffffffu, bx, o);
        by += __shfl_xor_sync(0xffffffffu, by, o);
        bz += __shfl_xor_sync(0xffffffffu, bz, o);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&s_xyz[0], ax);
        atomicAdd(&s_xyz[1], ay);
        atomicAdd(&s_xyz[2], az);
        if (p_end != p_blk) {
            atomicAdd(&s_xyz[4], bx);
            atomicAdd(&s_xyz[5], by);
            atomicAdd(&s_xyz[6], bz);
        }
    }
    __syncthreads();
    if (threadIdx.x < 3) atomicAdd(&sums[3 * p_blk + threadIdx.x], s_xyz[threadIdx.x]);
    if (p_end != p_blk && threadIdx.x >= 4 && threadIdx.x < 7) atomicAdd(&sums[3 * p_end + threadIdx.x - 4], s_xyz[threadIdx.x]);
    for (int k = threadIdx.x; k < 2 * nb; k += blockDim.x) {
        const int slot = k >= nb ? 1 : 0, b = k - slot * nb;
        const int pp = slot ? p_end : p_blk;
        if (s_cnt[k]) atomicAdd(&counts[(size_t)b * n_patch + pp], (unsigned long long)s_cnt[k]);
        if (w && s_w[k] != 0.0) atomicAdd(&sumw[(size_t)b * n_patch + pp], s_w[k]);
    }
}

// frames from the per-patch sums: centre = mean direction, e1/e2 any orthonormal tangent basis
__global__ void k_make_frames(const double *__restrict__ sums, int n_patch, PatchFrame *__restrict__ frames) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_patch) return;
    PatchFrame f;
    double cx = sums[3 * p], cy = sums[3 * p + 1], cz = sums[3 * p + 2];
    double nrm = sqrt(cx * cx + cy * cy + cz * cz);
    if (!(nrm > 1e-12)) { cx = 0; cy = 0; cz = 1; nrm = 1; }  // empty or antipodally balanced patch
    f.c[0] = cx / nrm; f.c[1] = cy / nrm; f.c[2] = cz / nrm;
    double ax = 0, ay = 0, az = 1;  // helper axis least aligned with c
    if (fabs(f.c[2]) > 0.9) { ax = 1; az = 0; }
    double e1x = ay * f.c[2] - az * f.c[1], e1y = az * f.c[0] - ax * f.c[2], e1z = ax * f.c[1] - ay * f.c[0];
    double n1 = sqrt(e1x * e1x + e1y * e1y + e1z * e1z);
    f.e1[0] = e1x / n1; f.e1[1] = e1y / n1; f.e1[2] = e1z / n1;
    f.e2[0] = f.c[1] * f.e1[2] - f.c[2] * f.e1[1];
    f.e2[1] = f.c[2] * f.e1[0] - f.c[0] * f.e1[2];
    f.e2[2] = f.c[0] * f.e1[1] - f.c[1] * f.e1[0];
    f.radius = 0.0;
    f.norm_dev = 0.0;
    f.umin = f.umax = f.vmin = f.vmax = 0.0;
    frames[p] = f;
}

__device__ __forceinline__ double dec_double_dev(unsigned long long b) {
    b = (b & 0x8000000000000000ull) ? (b & 0x7fffffffffffffffull) : ~b;
    return __longlong_as_double((long long)b);
}

constexpr int kBox = 6;  // per patch: min u, max u, min v, max v, max squared chord from the centre, max | |P|^2 - 1 |

__global__ void k_init_box(unsigned long long *__restrict__ box, int n_patch) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_patch) return;
    box[kBox * p] = box[kBox * p + 2] = ~0ull;
    box[kBox * p + 1] = box[kBox * p + 3] = box[kBox * p + 4] = box[kBox * p + 5] = 0ull;
}

__global__ void k_finish_frames(const unsigned long long *__restrict__ box, int n_patch,
                                PatchFrame *__restrict__ frames) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_patch) return;
    if (box[kBox * p] == ~0ull) return;  // no rows: extents stay zero
    frames[p].umin = dec_double_dev(box[kBox * p]);
    frames[p].umax = dec_double_dev(box[kBox * p + 1]);
    frames[p].vmin = dec_double_dev(box[kBox * p + 2]);
    frames[p].vmax = dec_double_dev(box[kBox * p + 3]);
    frames[p].radius = sqrt(dec_double_dev(box[kBox * p + 4])) * (1.0 + 1e-12) + 1e-15;
    frames[p].norm_dev = dec_double_dev(box[kBox * p + 5]) * (1.0 + 1e-9) + 4.0e-16;
}

// per patch: (u, v) bounding box and max squared chord distance from the centre.  Same blocking as
// k_patch_sums: a block owns kSumRows consecutive rows and reduces the rows of its first and of its last patch in
// registers / shuffles / shared memory (six atomics per patch and block); rows of a third patch go direct.
struct BoxAcc {
    unsigned long long umin = ~0ull, umax = 0ull, vmin = ~0ull, vmax = 0ull, dmax = 0ull, nmax = 0ull;
    __device__ __forceinline__ void add(unsigned long long eu, unsigned long long ev, unsigned long long ed, unsigned long long en) {
        umin = min(umin, eu); umax = max(umax, eu);
        vmin = min(vmin, ev); vmax = max(vmax, ev);
        dmax = max(dmax, ed);
        nmax = max(nmax, en);
    }
    __device__ __forceinline__ void warp_reduce() {
        for (int o = 16; o; o >>= 1) {
            umin = min(umin, __shfl_xor_sync(0xffffffffu, umin, o));
            umax = max(umax, __shfl_xor_sync(0xffffffffu, umax, o));
            vmin = min(vmin, __shfl_xor_sync(0xffffffffu, vmin, o));
            vmax = max(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
            dmax = max(dmax, __shfl_xor_sync(0xffffffffu, dmax, o));
            nmax = max(nmax, __shfl_xor_sync(0xffffffffu, nmax, o));
        }
    }
};

__global__ void __launch_bounds__(kThreads) k_patch_bbox(const double *__restrict__ x, const double *__restrict__ y,
                                                         const double *__restrict__ z, const int *__restrict__ patch,
                                                         long long n, const PatchFrame *__restrict__ frames,
                                                         unsigned long long *__restrict__ box /*[n_patch][kBox]*/) {
    __shared__ unsigned long long s_box[2][kBox][kThreads / 32];
    const long long row0 = (long long)blockIdx.x * kSumRows;
    const long long row1 = min(row0 + (long long)kSumRows, n);
    const int p_blk = patch[row0], p_end = patch[row1 - 1];
    const PatchFrame f = frames[p_blk], f2 = frames[p_end];
    BoxAcc A, B;
    for (int k0 = threadIdx.x; k0 < kSumRows; k0 += kSumBatch * blockDim.x) {
        int pq[kSumBatch];
        double X[kSumBatch], Y[kSumBatch], Z[kSumBatch];
#pragma unroll
        for (int q = 0; q < kSumBatch; ++q) {  // all loads of the round first
            const long long i = row0 + k0 + q * (int)blockDim.x;
            const bool ok = k0 + q * (int)blockDim.x < kSumRows && i < n;
            pq[q] = ok ? patch[i] : -1;
            X[q] = ok ? x[3 * i] : 0.0;
            Y[q] = ok ? y[3 * i] : 0.0;
            Z[q] = ok ? z[3 * i] : 0.0;
        }
#pragma unroll
        for (int q = 0; q < kSumBatch; ++q) {
            const int p = pq[q];
            if (p < 0) continue;
            const PatchFrame &g = p == p_blk ? f : p == p_end ? f2 : frames[p];
            const double dx = X[q] - g.c[0], dy = Y[q] - g.c[1], dz = Z[q] - g.c[2];
            const unsigned long long eu = enc_double(dx * g.e1[0] + dy * g.e1[1] + dz * g.e1[2]);
            const unsigned long long ev = enc_double(dx * g.e2[0] + dy * g.e2[1] + dz * g.e2[2]);
            const unsigned long long ed = enc_double(dx * dx + dy * dy + dz * dz);
            // how far the row is from the unit sphere: | |P|^2 - 1 |, evaluated without cancellation as |d . (P + c)|
            // plus the deviation of the (normalised) centre itself
            const unsigned long long en =
                enc_double(fabs(dx * (X[q] + g.c[0]) + dy * (Y[q] + g.c[1]) + dz * (Z[q] + g.c[2])) +
                           fabs(g.c[0] * g.c[0] + g.c[1] * g.c[1] + g.c[2] * g.c[2] - 1.0));
            if (p == p_blk) {
                A.add(eu, ev, ed, en);
            } else if (p == p_end) {
                B.add(eu, ev, ed, en);
            } else {
                atomicMin(&box[kBox * p], eu);
                atomicMax(&box[kBox * p + 1], eu);
                atomicMin(&box[kBox * p + 2], ev);
                atomicMax(&box[kBox * p + 3], ev);
                atomicMax(&box[kBox * p + 4], ed);
                atomicMax(&box[kBox * p + 5], en);
            }
        }
    }
    A.warp_reduce();
    B.warp_reduce();
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
        s_box[0][0][w] = A.umin; s_box[0][1][w] = A.umax; s_box[0][2][w] = A.vmin; s_box[0][3][w] = A.vmax; s_box[0][4][w] = A.dmax; s_box[0][5][w] = A.nmax;
        s_box[1][0][w] = B.umin; s_box[1][1][w] = B.umax; s_box[1][2][w] = B.vmin; s_box[1][3][w] = B.vmax; s_box[1][4][w] = B.dmax; s_box[1][5][w] = B.nmax;
    }
    __syncthreads();
    if (threadIdx.x < 2 * kBox) {
        const int slot = threadIdx.x / kBox, c = threadIdx.x % kBox;
        if (slot == 1 && p_end == p_blk) return;
        unsigned long long v = s_box[slot][c][0];
        const bool is_min = c == 0 || c == 2;
        for (int k = 1; k < kThreads / 32; ++k) v = is_min ? min(v, s_box[slot][c][k]) : max(v, s_box[slot][c][k]);
        const int pp = slot ? p_end : p_blk;
        if (is_min) atomicMin(&box[kBox * pp + c], v);  // ~0 / 0 are the neutral initial values
        else atomicMax(&box[kBox * pp + c], v);
    }
}

// ---- sort keys ----------------------------------------------------------------------------

__device__ __forceinline__ void local_uv(const PatchFrame &f, double X, double Y, double Z, double &u,
                                         double &v) {
    double dx = X - f.c[0], dy = Y - f.c[1], dz = Z - f.c[2];
    u = dx * f.e1[0] + dy * f.e1[1] + dz * f.e1[2];
    v = dx * f.e2[0] + dy * f.e2[1] + dz * f.e2[2];
}

// global sky-cell id of a row of a first-role index, or -1 for a row whose z-bin is out of range
__device__ __forceinline__ long long key_first(double X, double Y, double Z, int b, int p, int n_bins,
                                               const PatchFrame *__restrict__ frames, const SGrid *__restrict__ grids) {
    if (b < 0 || b >= n_bins) return -1;
    double u, v;
    local_uv(frames[p], X, Y, Z, u, v);
    const SGrid g = grids[p];
    // clamp in double first: the product can exceed the int range for degenerate patches
    int iu = (int)fmin(fmax(floor((u - g.u0) * g.inv_cu), 0.0), (double)(g.gu - 1));
    int iv = (int)fmin(fmax(floor((v - g.v0) * g.inv_cv), 0.0), (double)(g.gv - 1));
    return g.cell_base + ((long long)b * g.gv + iv) * g.gu + iu;
}

// Hilbert index of a cell on a 65536 x 65536 grid.  Unlike the Morton (Z) curve the Hilbert curve has
// no jumps: consecutive cells are always neighbours, so every run of YAWB_TILE consecutive rows is a
// compact clump and no register tile straddles a quadrant boundary with a patch-sized bounding box.
// Only the top `levels` levels are resolved (the top 2 * levels bits of the index; the rest stays zero).
__device__ __forceinline__ unsigned hilbert16(unsigned x, unsigned y, int levels = 16) {
    unsigned d = 0;
    const unsigned stop = levels >= 16 ? 0u : (1u << (15 - levels));
    for (unsigned s = 1u << 15; s > stop; s >>= 1) {
        const unsigned rx = (x & s) ? 1u : 0u;
        const unsigned ry = (y & s) ? 1u : 0u;
        d += s * s * ((3u * rx) ^ ry);
        if (ry == 0u) {
            if (rx == 1u) {
                x = 65535u - x;
                y = 65535u - y;
            }
            const unsigned t = x;
            x = y;
            y = t;
        }
    }
    return d;
}

// Map of a patch box onto the Hilbert square(s), per patch and index build (k_hilbert_map).
// The bounding box of the patch is stretched over the Hilbert square(s): an isotropic mapping would leave part
// of the square empty, and wherever the curve leaves the populated part and re-enters elsewhere, 256
// consecutive rows straddle the gap (measured: a few tiles per patch with patch-sized boxes, each worth several
// average work items -> a 13 % straggler tail).  An elongated box (aspect >= 2, e.g. the strip of a
// patch that two ranks share) is covered by k = round(aspect) <= 8 squares side by side along its long axis:
// the curve leaves a square at the corner where it enters the next one, so the order stays continuous and
// the cells -- hence the tiles -- stay close to square instead of being stretched k : 1 (a 4 : 1 strip in one
// square: every tile trips the straggler guard and is cut into 32-row sub-tiles).  Below 2 : 1 a single
// stretched square is better (C3's 5 x 3 degree patches: 3.6 % fewer executed tests than with two squares).
// The square index takes its bits from the Hilbert resolution: a key of hbits = 2 bits below the (patch, z-bin)
// segment has room for at most 4 squares (with more, the rows of squares 4-7 would carry the key of the next segment).
struct HMap {
    double c[3], e_long[3], e_short[3];  // centre of the patch; tangent axes along the long / short side of the box
    double o_long, o_short;              // lower edge of the box along the two axes
    double s_long, s_short;              // k / long side; 65535 / short side (0 for a degenerate box)
    int k, levels;                       // squares side by side; resolved levels of the curve
};

__global__ void k_hilbert_map(const PatchFrame *__restrict__ frames, int n_patch, int hbits, HMap *__restrict__ maps) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_patch) return;
    const PatchFrame &f = frames[p];
    const double du = f.umax - f.umin, dv = f.vmax - f.vmin;
    const bool swap = dv > du;  // the long axis is the x of the curve (which runs from (0, 0) to (max, 0))
    const double lng = swap ? dv : du, sht = swap ? du : dv;
    const int k = sht > 0.0 && lng >= 2.0 * sht ? min((int)rint(lng / sht), hbits >= 3 ? 8 : 1 << hbits) : 1;
    const int kb = k > 4 ? 3 : k > 2 ? 2 : k > 1 ? 1 : 0;  // bits of the square index
    HMap m;
    for (int d = 0; d < 3; ++d) {
        m.c[d] = f.c[d];
        m.e_long[d] = swap ? f.e2[d] : f.e1[d];
        m.e_short[d] = swap ? f.e1[d] : f.e2[d];
    }
    m.o_long = swap ? f.vmin : f.umin;
    m.o_short = swap ? f.umin : f.vmin;
    m.s_long = lng > 0.0 ? (double)k / lng : 0.0;
    m.s_short = sht > 0.0 ? 65535.0 / sht : 0.0;
    m.k = k;
    m.levels = (hbits - kb) / 2;
    maps[p] = m;
}

// key = (patch * n_bins + bin) << hbits | square << (2 * levels) | top bits of the Hilbert index, or -1 for a row whose
// z-bin is out of range
__device__ __forceinline__ long long key_second(double X, double Y, double Z, int b, int p, int n_bins, int hbits,
                                                const HMap *__restrict__ maps) {
    if (b < 0 || b >= n_bins) return -1;
    const HMap &m = maps[p];
    const double dx = X - m.c[0], dy = Y - m.c[1], dz = Z - m.c[2];
    const double tl = (dx * m.e_long[0] + dy * m.e_long[1] + dz * m.e_long[2] - m.o_long) * m.s_long;
    const double ts = (dx * m.e_short[0] + dy * m.e_short[1] + dz * m.e_short[2] - m.o_short) * m.s_short;
    const int k = m.k, levels = m.levels;
    const int sq = min(max((int)tl, 0), k - 1);
    const int qx = min(max((int)((tl - sq) * 65535.0), 0), 65535);
    const int qy = min(max((int)ts, 0), 65535);
    const unsigned long long h = levels > 0 ? (unsigned long long)(hilbert16((unsigned)qx, (unsigned)qy, levels) >> (32 - 2 * levels)) : 0ull;
    return (long long)(((unsigned long long)((long long)p * n_bins + b) << hbits) | ((unsigned long long)sq << (2 * levels)) | h);
}

// ---- counting sort ------------------------------------------------------------------------------------
// The sort keys are bounded and dense (sky-cell ids, (patch, z-bin, Hilbert cell) ids: about as many keys as rows),
// so the rows are put in order by ONE histogram pass that also hands every row its rank among the rows of its
// key (the value the atomic returns), an in-place exclusive scan of the key counts, and ONE scatter pass without
// atomics: position = first slot of the key + rank.  (key, rank) of a row travel from the first pass to the second
// in an 8-byte side array, so the second pass neither walks the curve again nor waits for an atomic.  The order of
// rows with the same key is arbitrary (it has no meaning: pair counts are sums over all rows of a cell, and the
// count kernel adds weighted sums in an order that its warps settle at run time anyway).  After the scan cur[k] is
// the first slot of key k, i.e. the cell_start table of a first-role index (entry n_keys = row count).
__global__ void k_hist_first(const double *__restrict__ x, const double *__restrict__ y, const double *__restrict__ z,
                             const int *__restrict__ bin, const int *__restrict__ patch, long long n, int n_bins,
                             const PatchFrame *__restrict__ frames, const SGrid *__restrict__ grids,
                             int *__restrict__ cur, int2 *__restrict__ kr) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long key = key_first(x[3 * i], y[3 * i], z[3 * i], bin ? bin[i] : 0, patch[i], n_bins, frames, grids);
    int rank = 0;
    if (key >= 0) rank = atomicAdd(&cur[key], 1);
    kr[i] = make_int2((int)key, rank);  // -1: dropped row
}

__global__ void k_hist_second(const double *__restrict__ x, const double *__restrict__ y, const double *__restrict__ z,
                              const int *__restrict__ bin, const int *__restrict__ patch, long long n, int n_bins,
                              int hbits, const HMap *__restrict__ maps, const unsigned char *__restrict__ mask,
                              int *__restrict__ cur, int2 *__restrict__ kr) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    // a row outside the mask (yawb_catalog_set_second_rows) is dropped like a row outside the z-binning
    const long long key = mask && !mask[i] ? -1
                                           : key_second(x[3 * i], y[3 * i], z[3 * i], bin ? bin[i] : 0, patch[i], n_bins, hbits, maps);
    int rank = 0;
    if (key >= 0) rank = atomicAdd(&cur[key], 1);
    kr[i] = make_int2((int)key, rank);  // -1: dropped row
}

// in-place exclusive scan of `cur[0, n)` in ONE pass over the data (decoupled look-back): a block takes the next
// tile of kScanBlock counts from a global ticket (tiles are therefore started in order, whatever the hardware's
// block schedule), publishes the tile total, and its first warp walks back over the descriptors of the tiles
// before it -- 32 at a time -- adding totals until it meets a tile whose inclusive prefix is already known.
// A descriptor is one 64-bit word (state << 62 | value), written with a single store, so no fence is needed.
constexpr int kScanPerThread = 16;
constexpr int kScanBlock = kThreads * kScanPerThread;

__global__ void __launch_bounds__(kThreads) k_scan_lookback(int *__restrict__ cur, long long n,
                                                            unsigned long long *__restrict__ desc /*[tiles + 1]: ticket first*/) {
    constexpr unsigned long long kScanTotal = 1ull << 62, kScanPrefix = 2ull << 62, kScanValue = (1ull << 62) - 1;
    __shared__ int s_w[kThreads / 32];
    __shared__ long long s_tile;
    __shared__ long long s_prefix;
    if (threadIdx.x == 0) s_tile = (long long)atomicAdd(&desc[0], 1ull);
    __syncthreads();
    const long long tile = s_tile;
    volatile unsigned long long *const d = desc + 1;
    // A warp owns kScanPerThread rows of 32 consecutive counts (coalesced loads and stores: with 16 consecutive counts
    // per THREAD every load instruction touched 32 sectors and the kernel sat in the LSU queue); rows are scanned
    // with shuffles, the row totals carried along in a register.
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long base = tile * kScanBlock + (long long)warp * (32 * kScanPerThread) + lane;
    int v[kScanPerThread];
#pragma unroll
    for (int r = 0; r < kScanPerThread; ++r) v[r] = base + 32 * r < n ? cur[base + 32 * r] : 0;
    int excl[kScanPerThread];  // exclusive prefix of the element within the warp's 512 counts
    int carry = 0;
#pragma unroll
    for (int r = 0; r < kScanPerThread; ++r) {
        int incl = v[r];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        excl[r] = carry + incl - v[r];
        carry += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (lane == 0) s_w[warp] = carry;
    __syncthreads();
    int before = 0, block_total = 0;  // counts of the warps before this one; of the whole tile
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) {
        const int t = s_w[w];
        if (w < warp) before += t;
        block_total += t;
    }
    if (warp == 0) {
        long long prefix = 0;
        if (tile == 0) {
            if (lane == 0) d[0] = kScanPrefix | (unsigned long long)block_total;
        } else {
            if (lane == 0) d[tile] = kScanTotal | (unsigned long long)block_total;
            // Hundreds of tiles are in flight at once and none of them knows its prefix before the oldest one does, so
            // the walk is long: every lane requests kLook descriptors per round (256 tiles per round trip to L2).
            constexpr int kLook = 8;
            long long look = tile - 1;  // nearest tile not yet accounted for
            bool found = false;
            while (!found) {
                unsigned long long w[kLook];
#pragma unroll
                for (int j = 0; j < kLook; ++j) {
                    const long long idx = look - lane - 32 * j;
                    w[j] = kScanPrefix;  // before the first tile: prefix 0
                    if (idx >= 0) w[j] = d[idx];
                }
#pragma unroll
                for (int j = 0; j < kLook; ++j) {
                    if (found) continue;
                    const long long idx = look - lane - 32 * j;
                    while ((w[j] >> 62) == 0ull) w[j] = d[idx];
                    const unsigned has_prefix = __ballot_sync(0xffffffffu, (w[j] >> 62) == 2ull);
                    const int stop = has_prefix ? __ffs(has_prefix) - 1 : 32;  // nearest tile with a known prefix
                    long long part = lane <= stop ? (long long)(w[j] & kScanValue) : 0ll;
#pragma unroll
                    for (int o = 16; o; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
                    prefix += part;
                    found = has_prefix != 0u;
                }
                look -= 32 * kLook;
            }
            if (lane == 0) d[tile] = kScanPrefix | (unsigned long long)(prefix + block_total);
        }
        if (lane == 0) s_prefix = prefix;
    }
    __syncthreads();
    const int off = (int)s_prefix + before;
#pragma unroll
    for (int r = 0; r < kScanPerThread; ++r)
        if (base + 32 * r < n) cur[base + 32 * r] = off + excl[r];
}

// second-role scatter: the row goes to the next free slot of its key
__global__ void k_scatter_second(const double *__restrict__ x, const double *__restrict__ y, const double *__restrict__ z,
                                 const double *__restrict__ w, const int2 *__restrict__ kr, long long n,
                                 const int *__restrict__ cur, double tag, double *__restrict__ ox, double *__restrict__ ow) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int2 k = kr[i];
    if (k.x < 0) return;
    const double X = x[3 * i], Y = y[3 * i], Z = z[3 * i];
    const int pos = cur[k.x] + k.y;
    // one 32-byte record per row: a full sector per scattered store (three separate arrays cost three partial ones);
    // its fourth double is the row's catalog in the index (RIndex)
    double2 *const o = reinterpret_cast<double2 *>(ox + (size_t)YAWB_RSTRIDE * pos);
    o[0] = make_double2(X, Y);
    o[1] = make_double2(Z, tag);
    if (ow) ow[pos] = w ? w[i] : 1.0;  // union of a weighted and an unweighted catalog
}

// first-role scatter (rows of one catalog; called twice for a fused index): the exact row plus its fixed-point
// record in the frame of the patch (SGrid: origin and power-of-two scale)
__global__ void k_scatter_first(const double *__restrict__ x, const double *__restrict__ y, const double *__restrict__ z,
                                const double *__restrict__ w, const int *__restrict__ bin, const int *__restrict__ patch,
                                long long n, int n_bins, unsigned type_bit, const PatchFrame *__restrict__ frames,
                                const SGrid *__restrict__ grids, const int *__restrict__ cur, const int2 *__restrict__ kr,
                                double *__restrict__ ow, SRec *__restrict__ orec) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int2 k = kr[i];
    if (k.x < 0) return;
    const double X = x[3 * i], Y = y[3 * i], Z = z[3 * i];
    const int p = patch[i];
    const int pos = cur[k.x] + k.y;
    if (ow) ow[pos] = w ? w[i] : 1.0;  // fused index of a weighted and an unweighted catalog
    const PatchFrame &f = frames[p];
    const SGrid &g = grids[p];
    const double dx = X - f.c[0], dy = Y - f.c[1], dz = Z - f.c[2];
    const double u = dx * f.e1[0] + dy * f.e1[1] + dz * f.e1[2];
    const double v = dx * f.e2[0] + dy * f.e2[1] + dz * f.e2[2];
    const double t = dx * f.c[0] + dy * f.c[1] + dz * f.c[2];
    SRec r;
    r.ku = (int)fmin(fmax(rint((u - g.u0) * g.qscale), 0.0), 2147483647.0);
    r.kv = (int)fmin(fmax(rint((v - g.v0) * g.qscale), 0.0), 2147483647.0);
    r.kt = (int)fmin(fmax(rint((t - g.t0) * g.qscale), 0.0), 2147483647.0);
    r.aux = (unsigned)i | type_bit;  // the exact row stays where it was uploaded (FP64 recheck only)
    orec[pos] = r;
}

// bounding sphere of each register tile, and its bounding box in the frame of its own patch: one warp per tile
__global__ void k_tile_spheres(const double *__restrict__ x, const double *__restrict__ y,
                               const double *__restrict__ z, Tile *__restrict__ tiles, int n_tiles,
                               const PatchFrame *__restrict__ frames, TileBox *__restrict__ boxes) {
    int t = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
    int lane = threadIdx.x & 31;
    if (t >= n_tiles) return;
    Tile tl = tiles[t];
    const unsigned full = 0xffffffffu;
    const PatchFrame &f = frames[tl.patch];
    double sx = 0, sy = 0, sz = 0;
    double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
    // the lane's rows (k = lane + 32 r) are requested together and kept for the second pass
    constexpr int kRows = YAWB_TILE / 32;
    double X[kRows], Y[kRows], Z[kRows];
#pragma unroll
    for (int r = 0; r < kRows; ++r) {
        const int k = lane + 32 * r;
        const bool ok = k < tl.count;
        X[r] = Y[r] = Z[r] = 0.0;
        if (ok) {  // 32-byte row records
            const double2 *const row = reinterpret_cast<const double2 *>(x + (size_t)YAWB_RSTRIDE * (tl.start + k));
            const double2 a = row[0], b = row[1];
            X[r] = a.x; Y[r] = a.y; Z[r] = b.x;
        }
    }
#pragma unroll
    for (int r = 0; r < kRows; ++r) {
        if (lane + 32 * r >= tl.count) continue;
        sx += X[r];
        sy += Y[r];
        sz += Z[r];
        const double dx = X[r] - f.c[0], dy = Y[r] - f.c[1], dz = Z[r] - f.c[2];
        const double q[3] = {dx * f.e1[0] + dy * f.e1[1] + dz * f.e1[2], dx * f.e2[0] + dy * f.e2[1] + dz * f.e2[2],
                             dx * f.c[0] + dy * f.c[1] + dz * f.c[2]};
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            lo[d] = fmin(lo[d], q[d]);
            hi[d] = fmax(hi[d], q[d]);
        }
    }
#pragma unroll
    for (int d = 0; d < 3; ++d)
        for (int o = 16; o; o >>= 1) {
            lo[d] = fmin(lo[d], __shfl_xor_sync(full, lo[d], o));
            hi[d] = fmax(hi[d], __shfl_xor_sync(full, hi[d], o));
        }
    if (lane < 3) {  // padded by far more than the rounding of the three dot products
        const double pad = 1e-14 + 1e-12 * fmax(fabs(lo[lane]), fabs(hi[lane]));
        boxes[t].lo[lane] = lo[lane] - pad;
        boxes[t].hi[lane] = hi[lane] + pad;
    }
    for (int o = 16; o; o >>= 1) {
        sx += __shfl_xor_sync(full, sx, o);
        sy += __shfl_xor_sync(full, sy, o);
        sz += __shfl_xor_sync(full, sz, o);
    }
    double inv = 1.0 / (double)tl.count;
    float cx = (float)(sx * inv), cy = (float)(sy * inv), cz = (float)(sz * inv);
    double r2 = 0.0;  // radius about the float-rounded centre, so the stored sphere is sound
#pragma unroll
    for (int r = 0; r < kRows; ++r) {
        if (lane + 32 * r >= tl.count) continue;
        const double dx = X[r] - (double)cx, dy = Y[r] - (double)cy, dz = Z[r] - (double)cz;
        r2 = fmax(r2, dx * dx + dy * dy + dz * dz);
    }
    for (int o = 16; o; o >>= 1) r2 = fmax(r2, __shfl_xor_sync(full, r2, o));
    if (lane == 0) {
        tl.cx = cx;
        tl.cy = cy;
        tl.cz = cz;
        tl.rad = (float)(sqrt(r2) * (1.0 + 1e-6) + 1e-12);
        if ((double)tl.rad < sqrt(r2)) tl.rad = nextafterf(tl.rad, 1e30f);
        tiles[t] = tl;
    }
}

// tile table of a second-role index: tile t covers YAWB_TILE rows (the last tile of a segment fewer) of the
// (patch, z-bin) segment s with seg_tile_off[s] <= t < seg_tile_off[s + 1].  Written on the device: the host loop
// over the tiles and the 32 bytes per tile it had to send sat on the critical path of every index build.
__global__ void k_make_tiles(const int *__restrict__ seg_off, const int *__restrict__ seg_tile_off, int n_seg, int n_bins,
                             int binned, int n_tiles, Tile *__restrict__ tiles) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tiles) return;
    int lo = 0, hi = n_seg;  // last segment with seg_tile_off[s] <= t
    while (hi - lo > 1) {
        const int m = (lo + hi) >> 1;
        if (seg_tile_off[m] <= t) lo = m; else hi = m;
    }
    const int s = lo;
    Tile tl{};
    tl.start = seg_off[s] + (t - seg_tile_off[s]) * YAWB_TILE;
    tl.count = min(YAWB_TILE, seg_off[s + 1] - tl.start);
    tl.patch = s / n_bins;
    tl.bin = binned ? s % n_bins : -1;
    tiles[t] = tl;
}

__global__ void k_count_oversized(const Tile *__restrict__ tiles, int n_tiles, const float *__restrict__ thr,
                                  unsigned *__restrict__ n_big) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n_tiles && tiles[t].count > 32 && tiles[t].rad > thr[tiles[t].patch]) atomicAdd(n_big, 1u);
}

// rows per (z-bin, patch) inside the second-role mask; rows are grouped by patch, so the lanes of a warp mostly share
// a key and one lane adds for all of them
__global__ void k_second_counts(const int *__restrict__ bin, const int *__restrict__ patch, const unsigned char *__restrict__ mask,
                                long long n, int n_bins, int n_patch, unsigned long long *__restrict__ counts) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int b = bin ? bin[i] : 0;
    if (!mask[i] || b < 0 || b >= n_bins) return;
    const int key = b * n_patch + patch[i];
    const unsigned peers = __match_any_sync(__activemask(), key);
    if ((threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&counts[key], (unsigned long long)__popc(peers));
}

template <typename T>
int fi_alloc(FIndex *fi, T **ptr, size_t count) {
    *ptr = nullptr;
    if (count == 0) count = 1;
    if (yawb_dalloc(fi->ctx, (void **)ptr, count * sizeof(T), fi->ctx->stream)) return 1;
    fi->device_bytes += (int64_t)(count * sizeof(T));
    return 0;
}

int exclusive_scan_inplace(yawb_ctx *ctx, Scratch &scr, int *cur, long long n) {
    if (n <= 0) return 0;
    const int n_blocks = (int)((n + kScanBlock - 1) / kScanBlock);
    unsigned long long *desc = scr.get<unsigned long long>((size_t)n_blocks + 1);
    YAWB_REQUIRE(desc != nullptr, "out of device memory (scan scratch)");
    YAWB_CUDA(cudaMemsetAsync(desc, 0, ((size_t)n_blocks + 1) * sizeof(unsigned long long), ctx->stream));
    k_scan_lookback<<<n_blocks, kThreads, 0, ctx->stream>>>(cur, n, desc);
    return 0;
}

// first-role rows in sky-cell order by counting sort; fills cell_start (base + 1 entries)
int build_first_counting(FIndex *fi, long long base) {
    yawb_ctx *ctx = fi->ctx;
    cudaStream_t st = ctx->stream;
    const yawb_cat *a = fi->a, *b = fi->b;
    Scratch scr(ctx, st);
    int *cur = fi->cell_start;  // key counts -> (exclusive scan over base + 1 entries) -> cell_start, the last entry = rows
    const long long na = a && a->n_in > 0 ? a->n_in : 0, nb = b && b->n_in > 0 ? b->n_in : 0;
    int2 *kr = scr.get<int2>((size_t)(na + nb));
    YAWB_REQUIRE(kr != nullptr, "out of device memory (sort keys)");
    YAWB_CUDA(cudaMemsetAsync(fi->cell_start, 0, (size_t)(base + 1) * sizeof(int), st));
    for (const yawb_cat *c : {a, b})
        if (c && c->n_in > 0)
            k_hist_first<<<blocks_for(c->n_in), kThreads, 0, st>>>(c->x, c->y, c->z, c->bin, c->patch, c->n_in, fi->n_bins,
                                                                   fi->d_frames, fi->d_sgrid, cur, kr + (c == b ? na : 0));
    if (exclusive_scan_inplace(ctx, scr, cur, base + 1)) return 1;
    for (const yawb_cat *c : {a, b})
        if (c && c->n_in > 0)
            k_scatter_first<<<blocks_for(c->n_in), kThreads, 0, st>>>(c->x, c->y, c->z, c->w, c->bin, c->patch, c->n_in,
                                                                      fi->n_bins, c == b ? 0x80000000u : 0u, fi->d_frames,
                                                                      fi->d_sgrid, cur, kr + (c == b ? na : 0), fi->sw, fi->rec);
    return 0;
}

template <typename T>
int ri_alloc(RIndex *ri, T **ptr, size_t count) {
    *ptr = nullptr;
    if (count == 0) count = 1;
    if (yawb_dalloc(ri->ctx, (void **)ptr, count * sizeof(T), ri->ctx->stream)) return 1;
    ri->device_bytes += (int64_t)(count * sizeof(T));
    return 0;
}

// second-role rows of one catalog or of two (RIndex) in (patch, z-bin, Hilbert) order by counting sort; the rows of
// both catalogs share the Hilbert maps of a's patch frames (the map only orders rows: a row of b outside a's patch
// box is clamped to its edge)
int build_second_counting(RIndex *ri, int hbits, long long n_keys) {
    yawb_ctx *ctx = ri->ctx;
    cudaStream_t st = ctx->stream;
    const yawb_cat *a = ri->a, *b = ri->b;
    const long long na = a->n_in > 0 ? a->n_in : 0, nb = b && b->n_in > 0 ? b->n_in : 0;
    if (na + nb == 0) return 0;
    Scratch scr(ctx, st);
    int *cur = scr.get<int>((size_t)n_keys);
    int2 *keys = scr.get<int2>((size_t)(na + nb));  // (key, rank among the rows of the key) of every row
    HMap *maps = scr.get<HMap>((size_t)a->n_patch);
    YAWB_REQUIRE(cur && keys && maps, "out of device memory (key counts)");
    YAWB_CUDA(cudaMemsetAsync(cur, 0, (size_t)n_keys * sizeof(int), st));
    k_hilbert_map<<<(a->n_patch + 127) / 128, 128, 0, st>>>(a->d_frames, a->n_patch, hbits, maps);
    for (const yawb_cat *c : {a, b})
        if (c && c->n_in > 0)
            k_hist_second<<<blocks_for(c->n_in), kThreads, 0, st>>>(c->x, c->y, c->z, c->bin, c->patch, c->n_in, a->n_bins,
                                                                    hbits, maps, c->d_second_mask, cur,
                                                                    keys + (c == b ? na : 0));
    if (exclusive_scan_inplace(ctx, scr, cur, n_keys)) return 1;
    for (const yawb_cat *c : {a, b})
        if (c && c->n_in > 0)
            k_scatter_second<<<blocks_for(c->n_in), kThreads, 0, st>>>(c->x, c->y, c->z, c->w, keys + (c == b ? na : 0),
                                                                       c->n_in, cur, c == b ? 1.0 : 0.0, ri->rx, ri->rw);
    return 0;
}

// cells of edge c in a first-role grid of a patch box du x dv, grown by 1.5 until a z-bin has at most
// kMaxCellsPerPatchBin cells and a cell row at most 32767
void size_cells(SGrid &g, double du, double dv, double c) {
    auto dims = [&]() {
        g.inv_cv = 1.0 / c;
        g.inv_cu = kCellAspect / c;
        g.gu = std::max(1, (int)std::floor(du * g.inv_cu) + 1);
        g.gv = std::max(1, (int)std::floor(dv * g.inv_cv) + 1);
    };
    dims();
    while ((long long)g.gu * g.gv > kMaxCellsPerPatchBin || g.gu > 32767) {
        c *= 1.5;
        dims();
    }
}

}  // namespace

// -------------------------------------------------------------------------------------------
static constexpr size_t kCopyChunk = (size_t)64 << 20;

int yawb_index_upload(yawb_ctx *ctx, yawb_cat *cat, const double *xyz, const double *w, const uint8_t *zbin8,
                      const int32_t *zbin, const double *zred, const int64_t *patch_off, const std::vector<RowRun> &runs) {
    YawbRange range("yawb:upload");
    const long long n = cat->n_in;
    const int P = cat->n_patch, B = cat->n_bins;
    // Only allocations and host-to-device copies are issued here, all on the context's copy stream, which
    // never carries a kernel: the copies of later catalogs keep the bus busy while pair counts of earlier
    // ones occupy every SM (a kernel queued on the copy stream would wait for those SMs and hold the
    // copies behind it).  The per-patch reductions run on the main stream when the catalog is first used
    // (yawb_cat_finalize), which joins the copies through `ev_meta`.
    cudaStream_t st = ctx->copy_stream;
    // the rows stay interleaved, as uploaded: x / y / z are views of `xyz` with stride 3
    if (dev_alloc(cat, &cat->xyz, (size_t)n * 3, st) || dev_alloc(cat, &cat->patch, n, st)) return 1;
    cat->x = cat->xyz;
    cat->y = cat->xyz + 1;
    cat->z = cat->xyz + 2;
    if (w && dev_alloc(cat, &cat->w, n, st)) return 1;
    if ((zbin || zbin8 || zred) && dev_alloc(cat, &cat->bin, n, st)) return 1;
    if (zbin8 && dev_alloc(cat, &cat->d_stage_bin8, n, st)) return 1;
    if (zred && dev_alloc(cat, &cat->d_stage_z, n, st)) return 1;
    if (dev_alloc(cat, &cat->d_frames, P, st) || dev_alloc(cat, &cat->d_seg_off, (size_t)P * B + 1, st)) return 1;
    if (dev_alloc(cat, &cat->d_stage_poff, P + 1, st)) return 1;

    // Each run of rows (the whole catalog, or a run of consecutive kept patches of a partial upload) travels straight
    // from the caller's array.  Bulk copies go out in pieces so that other users of the copy engine never wait behind
    // a whole catalog (the small tables of a concurrent pair count avoid the engine altogether: yawb_h2d_small).
    auto h2d = [&](void *dst, const void *src, size_t row_bytes) -> cudaError_t {
        for (const RowRun &r : runs) {
            const size_t bytes = (size_t)r.rows * row_bytes;
            char *d = (char *)dst + (size_t)r.dst * row_bytes;
            const char *s = (const char *)src + (size_t)r.src * row_bytes;
            for (size_t o = 0; o < bytes; o += kCopyChunk) {
                cudaError_t e = cudaMemcpyAsync(d + o, s + o, std::min(kCopyChunk, bytes - o), cudaMemcpyHostToDevice, st);
                if (e != cudaSuccess) return e;
            }
        }
        return cudaSuccess;
    };
    if (n > 0) YAWB_CUDA(h2d(cat->xyz, xyz, 3 * sizeof(double)));
    YAWB_CUDA(cudaMemcpyAsync(cat->d_stage_poff, patch_off, (P + 1) * sizeof(long long), cudaMemcpyHostToDevice, st));
    if (w && n > 0) YAWB_CUDA(h2d(cat->w, w, sizeof(double)));
    if (zbin && n > 0) YAWB_CUDA(h2d(cat->bin, zbin, sizeof(int32_t)));
    if (zbin8 && n > 0) YAWB_CUDA(h2d(cat->d_stage_bin8, zbin8, 1));
    if (zred && n > 0) YAWB_CUDA(h2d(cat->d_stage_z, zred, sizeof(double)));
    YAWB_CUDA(cudaEventCreateWithFlags(&cat->ev_meta, cudaEventDisableTiming));
    YAWB_CUDA(cudaEventRecord(cat->ev_meta, st));
    YAWB_CUDA(cudaGetLastError());
    cat->finalized = false;
    return 0;
}

static void release_staging(yawb_cat *cat) {
    if (cat->staging_in_arena) {
        yawb_ctx *ctx = cat->ctx;
        if (--ctx->pin_live == 0) ctx->pin_used = 0;  // nothing pending: the arena starts over
        cat->staging_in_arena = false;
    }
    if (cat->hp_block) cudaFreeHost(cat->hp_block);
    cat->hp_block = nullptr;
    cat->hp_frames = nullptr;
    cat->hp_counts = nullptr;
    cat->hp_sumw = nullptr;
}

// Completion of an upload at first use: patch ids, per-patch reductions and frames on the main stream,
// their results to pinned staging, then the host-side row tables.
int yawb_cat_finalize(yawb_cat *cat) {
    if (cat->finalized) return 0;
    YawbRange range("yawb:finalize");
    if (cat->finalized) return 0;
    yawb_ctx *ctx = cat->ctx;
    cudaStream_t st = ctx->stream;
    const long long n = cat->n_in;
    const int P = cat->n_patch, B = cat->n_bins;
    YAWB_CUDA(cudaStreamWaitEvent(st, cat->ev_meta, 0));  // the copies of this catalog have landed
    {
        Scratch scr(ctx, st);
        double *d_sums = scr.get<double>((size_t)P * 3);
        double *d_sumw = scr.get<double>((size_t)B * P);
        unsigned long long *d_counts = scr.get<unsigned long long>((size_t)B * P);
        unsigned long long *d_box = scr.get<unsigned long long>((size_t)P * kBox);
        YAWB_REQUIRE(d_sums && d_sumw && d_counts && d_box, "out of device memory (upload scratch)");
        YAWB_CUDA(cudaMemsetAsync(d_sums, 0, P * 3 * sizeof(double), st));
        YAWB_CUDA(cudaMemsetAsync(d_sumw, 0, (size_t)B * P * sizeof(double), st));
        YAWB_CUDA(cudaMemsetAsync(d_counts, 0, (size_t)B * P * sizeof(unsigned long long), st));
        const int pb = (P + 127) / 128;
        if (n > 0) {
            k_patch_ids<<<blocks_for(n), kThreads, 0, st>>>(cat->d_stage_poff, P, n, cat->patch);
            if (cat->d_stage_bin8) k_widen_bins<<<blocks_for(n), kThreads, 0, st>>>(cat->d_stage_bin8, n, cat->bin);
            if (cat->d_stage_z) {
                double *d_edges = scr.get<double>(cat->h_edges.size());
                YAWB_REQUIRE(d_edges != nullptr, "out of device memory (z-bin edges)");
                if (yawb_h2d_small(ctx, d_edges, cat->h_edges.data(), cat->h_edges.size() * sizeof(double))) return 1;
                k_digitize<<<blocks_for(n), kThreads, 0, st>>>(cat->d_stage_z, n, d_edges, (int)cat->h_edges.size(),
                                                               cat->closed_right ? 1 : 0, cat->bin);
            }
            const bool use_smem = B <= kSumMaxBins;
            const size_t smem =
                8 * sizeof(double) + (use_smem ? 2 * (size_t)B * (sizeof(unsigned) + (cat->w ? sizeof(double) : 0)) : 0);
            k_patch_sums<<<blocks_for(n, kSumRows), kThreads, smem, st>>>(cat->x, cat->y, cat->z, cat->w, cat->bin,
                                                                           cat->patch, n, P, B, d_sums, d_counts, d_sumw);
        }
        k_make_frames<<<pb, 128, 0, st>>>(d_sums, P, cat->d_frames);
        k_init_box<<<pb, 128, 0, st>>>(d_box, P);
        if (n > 0)
            k_patch_bbox<<<blocks_for(n, kSumRows), kThreads, 0, st>>>(cat->x, cat->y, cat->z, cat->patch, n,
                                                                       cat->d_frames, d_box);
        k_finish_frames<<<pb, 128, 0, st>>>(d_box, P, cat->d_frames);
        dev_free(cat, cat->d_stage_poff, P + 1);
        dev_free(cat, cat->d_stage_bin8, (size_t)n);
        dev_free(cat, cat->d_stage_z, (size_t)n);

        // meta data (frames, row counts, sums of weights) through pinned staging
        const size_t b_frames = (((size_t)std::max(P, 1) * sizeof(PatchFrame)) + 63) & ~(size_t)63;
        const size_t b_counts = (((size_t)B * P * sizeof(unsigned long long)) + 63) & ~(size_t)63;
        const size_t b_sumw = (((size_t)B * P * sizeof(double)) + 63) & ~(size_t)63;
        const size_t need = b_frames + b_counts + b_sumw;
        unsigned char *blk = nullptr;
        if (ctx->pin_base && ctx->pin_used + need <= ctx->pin_size) {
            blk = ctx->pin_base + ctx->pin_used;
            ctx->pin_used += need;
            ctx->pin_live += 1;
            cat->staging_in_arena = true;
        } else {
            YAWB_CUDA(cudaHostAlloc((void **)&blk, need, cudaHostAllocDefault));
            cat->hp_block = blk;
        }
        cat->hp_frames = (PatchFrame *)blk;
        cat->hp_counts = (unsigned long long *)(blk + b_frames);
        cat->hp_sumw = (double *)(blk + b_frames + b_counts);
        YAWB_CUDA(cudaMemcpyAsync(cat->hp_frames, cat->d_frames, P * sizeof(PatchFrame), cudaMemcpyDeviceToHost, st));
        YAWB_CUDA(cudaMemcpyAsync(cat->hp_counts, d_counts, (size_t)B * P * sizeof(unsigned long long),
                                  cudaMemcpyDeviceToHost, st));
        YAWB_CUDA(cudaMemcpyAsync(cat->hp_sumw, d_sumw, (size_t)B * P * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    YAWB_CUDA(cudaStreamSynchronize(st));
    YAWB_CUDA(cudaGetLastError());
    cat->h_frames.assign(cat->hp_frames, cat->hp_frames + P);
    cat->h_sumw.assign(cat->hp_sumw, cat->hp_sumw + (size_t)B * P);
    cat->h_counts.assign((size_t)B * P, 0);
    cat->n = 0;
    for (size_t k = 0; k < cat->h_counts.size(); ++k) {
        cat->h_counts[k] = (long long)cat->hp_counts[k];
        cat->n += cat->h_counts[k];
        if (!cat->weighted) cat->h_sumw[k] = (double)cat->hp_counts[k];  // trees.py:225-227
    }
    // rows of (patch p, bin b) in both sort orders: patch-major, bin-minor
    cat->h_seg_off.assign((size_t)P * B + 1, 0);
    for (int p = 0; p < P; ++p)
        for (int b = 0; b < B; ++b)
            cat->h_seg_off[(size_t)p * B + b + 1] =
                cat->h_seg_off[(size_t)p * B + b] + (int)cat->h_counts[(size_t)b * P + p];
    if (yawb_h2d_small(cat->ctx, cat->d_seg_off, cat->h_seg_off.data(), ((size_t)P * B + 1) * sizeof(int))) return 1;
    release_staging(cat);
    cat->finalized = true;
    return 0;
}

// -------------------------------------------------------------------------------------------
// Frames of a first-role index.  One catalog: its own frames.  Two catalogs: per patch the frame of the
// catalog with more rows there; its (u, v) box and radius are then grown -- on the host, without touching the
// rows -- to contain the other catalog's patch as well: the other patch's bounding box (a box in ITS frame) is
// carried over as the hull of its eight rotated corners, its bounding sphere by the triangle inequality.
static int findex_frames(FIndex *fi) {
    yawb_ctx *ctx = fi->ctx;
    const yawb_cat *a = fi->a, *b = fi->b;
    const int P = fi->n_patch, B = fi->n_bins;
    fi->h_frames = a->h_frames;
    if (fi_alloc(fi, &fi->d_frames, P)) return 1;
    if (b) {
        for (int p = 0; p < P; ++p) {
            const long long ra = a->h_seg_off[(size_t)(p + 1) * B] - a->h_seg_off[(size_t)p * B];
            const long long rb = b->h_seg_off[(size_t)(p + 1) * B] - b->h_seg_off[(size_t)p * B];
            const bool use_b = rb >= ra && rb > 0;
            PatchFrame f = use_b ? b->h_frames[p] : a->h_frames[p];
            const PatchFrame &o = use_b ? a->h_frames[p] : b->h_frames[p];
            const long long ro = use_b ? ra : rb;
            if (ro > 0) {
                // the other patch: rows with (u, v) in its box and t in [-radius^2 / 2, 0] of ITS frame
                const double tlo = -0.5 * o.radius * o.radius * (1.0 + 1e-9) - 1e-15;
                double umin = f.umin, umax = f.umax, vmin = f.vmin, vmax = f.vmax;
                for (int c = 0; c < 8; ++c) {
                    const double u = (c & 1) ? o.umax : o.umin, v = (c & 2) ? o.vmax : o.vmin, w = (c & 4) ? 0.0 : tlo;
                    double X[3];
                    for (int d = 0; d < 3; ++d) X[d] = o.c[d] + u * o.e1[d] + v * o.e2[d] + w * o.c[d] - f.c[d];
                    const double uu = X[0] * f.e1[0] + X[1] * f.e1[1] + X[2] * f.e1[2];
                    const double vv = X[0] * f.e2[0] + X[1] * f.e2[1] + X[2] * f.e2[2];
                    umin = std::min(umin, uu); umax = std::max(umax, uu);
                    vmin = std::min(vmin, vv); vmax = std::max(vmax, vv);
                }
                const double pad = 1e-12 * (1.0 + std::max(std::fabs(umax - umin), std::fabs(vmax - vmin)));
                f.umin = umin - pad; f.umax = umax + pad; f.vmin = vmin - pad; f.vmax = vmax + pad;
                const double dc = std::sqrt((o.c[0] - f.c[0]) * (o.c[0] - f.c[0]) + (o.c[1] - f.c[1]) * (o.c[1] - f.c[1]) +
                                            (o.c[2] - f.c[2]) * (o.c[2] - f.c[2]));
                f.radius = std::max(f.radius, (dc + o.radius) * (1.0 + 1e-12) + 1e-15);
            }
            fi->h_frames[p] = f;
        }
    }
    return yawb_h2d_small(ctx, fi->d_frames, fi->h_frames.data(), P * sizeof(PatchFrame));
}

static int findex_build(yawb_ctx *ctx, yawb_cat *a, yawb_cat *b, FIndex **out) {
    YawbRange range(b ? "yawb:index_first_fused" : "yawb:index_first");
    *out = nullptr;
    if (yawb_cat_finalize(a)) return 1;
    if (b && yawb_cat_finalize(b)) return 1;
    FIndex *fi = new (std::nothrow) FIndex();
    YAWB_REQUIRE(fi != nullptr, "out of host memory");
    fi->ctx = ctx;
    fi->a = a;
    fi->b = b;
    fi->n = a->n + (b ? b->n : 0);
    fi->n_patch = a->n_patch;
    fi->n_bins = a->n_bins;
    fi->n_types = b ? 2 : 1;
    fi->weighted = a->weighted || (b && b->weighted);
    const long long n = fi->n;
    const int P = fi->n_patch, B = fi->n_bins;
    auto fail = [&]() {
        yawb_findex_free(fi);
        return 1;
    };
    if (n >= (1ll << 31) - 1024) {
        yawb_set_error("a first-role index is limited to 2^31 rows (got %lld)", n);
        return fail();
    }
    if (findex_frames(fi)) return fail();

    // grid per patch: cell edge from the mean density of one z-bin of this patch; fixed-point scale of the rows
    fi->h_sgrid.assign(P, SGrid{});
    std::vector<double> edge(P);  // cell edge of every patch before the bound on the whole grid below
    long long base = 0;
    for (int p = 0; p < P; ++p) {
        const PatchFrame &f = fi->h_frames[p];
        long long np = a->h_seg_off[(size_t)(p + 1) * B] - a->h_seg_off[(size_t)p * B];
        if (b) np += b->h_seg_off[(size_t)(p + 1) * B] - b->h_seg_off[(size_t)p * B];
        double du = std::max(f.umax - f.umin, 0.0), dv = std::max(f.vmax - f.vmin, 0.0);
        double per_bin = std::max((double)np / B, 1.0);
        double area = std::max(du * dv, 1e-30);
        // cells of height c (the spacing of the cell rows, sized for kTargetPerCell rows of one z-bin per c x c
        // square) and width c / kCellAspect: a query is one contiguous run of rows per cell row, so narrow cells
        // trim the run to the query box at no cost in the number of runs
        double c = std::sqrt(kTargetPerCell * area / per_bin);
        double span = std::max(du, dv);
        if (!(c > 0.0) || span <= 0.0) c = 1.0;
        c = std::max(c, span / 2048.0);  // bound the grid, <= 8192 x 2048 cells
        edge[p] = c;
        SGrid &g = fi->h_sgrid[p];
        g.u0 = f.umin;
        g.v0 = f.vmin;
        size_cells(g, du, dv, c);
        g.cell_base = base;
        base += (long long)B * g.gu * g.gv;
        // t = (P - c).c = -chord^2 / 2 lies in [-radius^2 / 2, 0]; one power-of-two scale for (u, v, t)
        const double tspan = 0.5 * f.radius * f.radius * (1.0 + 1e-9) + 1e-12;
        g.t0 = -tspan;
        const double extent = std::max(std::max(du, dv), tspan) * (1.0 + 1e-9) + 1e-12;
        int m = (int)std::floor(std::log2(2147483000.0 / extent));
        m = std::min(std::max(m, 0), 60);
        g.qscale = std::ldexp(1.0, m);
        g.qinv = std::ldexp(1.0, -m);
    }
    // cell_start takes one int per cell: while the grids of all patches have more than kMaxGridCells cells together,
    // the cells of every patch grow by 1.5 (the grid only prunes pair tests, the counts do not depend on it).  With
    // one cell per patch and z-bin there are P B < 2^28.
    for (double grow = 1.5; base > kMaxGridCells; grow *= 1.5) {
        base = 0;
        for (int p = 0; p < P; ++p) {
            const PatchFrame &f = fi->h_frames[p];
            SGrid &g = fi->h_sgrid[p];
            size_cells(g, std::max(f.umax - f.umin, 0.0), std::max(f.vmax - f.vmin, 0.0), edge[p] * grow);
            g.cell_base = base;
            base += (long long)B * g.gu * g.gv;
        }
    }
    fi->n_cells = base;
    if (fi_alloc(fi, &fi->d_sgrid, P)) return fail();
    if (yawb_h2d_small(ctx, fi->d_sgrid, fi->h_sgrid.data(), P * sizeof(SGrid))) return fail();
    if (fi_alloc(fi, &fi->rec, n)) return fail();
    if (fi->weighted && fi_alloc(fi, &fi->sw, n)) return fail();
    if (fi_alloc(fi, &fi->cell_start, base + 1)) return fail();
    if (build_first_counting(fi, base)) return fail();
    if (cudaGetLastError() != cudaSuccess) {
        yawb_set_error("first-role index build failed");
        return fail();
    }
    *out = fi;
    return 0;
}

void yawb_findex_free(FIndex *fi) {
    if (!fi) return;
    yawb_ctx *ctx = fi->ctx;
    for (void *p : {(void *)fi->rec, (void *)fi->sw, (void *)fi->cell_start,
                    (void *)fi->d_sgrid, (void *)fi->d_frames})
        if (p) yawb_dfree(ctx, p, ctx->stream);
    delete fi;
}

int yawb_index_build_first(yawb_cat *cat) {
    if (yawb_cat_finalize(cat)) return 1;
    if (cat->findex) return 0;
    if (findex_build(cat->ctx, cat, nullptr, &cat->findex)) return 1;
    cat->device_bytes += cat->findex->device_bytes;
    return 0;
}

int yawb_findex_get_fused(yawb_ctx *ctx, yawb_cat *a, yawb_cat *b, FIndex **out, bool *built) {
    *built = false;
    for (FIndex *fi : ctx->fused)
        if (fi->a == a && fi->b == b) {
            *out = fi;
            return 0;
        }
    if (findex_build(ctx, a, b, out)) return 1;
    ctx->fused.push_back(*out);
    *built = true;
    return 0;
}

void yawb_findex_drop_fused(yawb_ctx *ctx, const yawb_cat *cat) {
    for (size_t k = 0; k < ctx->fused.size();) {
        if (ctx->fused[k]->a == cat || ctx->fused[k]->b == cat) {
            yawb_findex_free(ctx->fused[k]);
            ctx->fused.erase(ctx->fused.begin() + k);
        } else {
            ++k;
        }
    }
}

// -------------------------------------------------------------------------------------------
static void rindex_release(RIndex *ri) {
    for (void *p : {(void *)ri->rrow, (void *)ri->rw, (void *)ri->d_seg_off, (void *)ri->d_tiles, (void *)ri->d_tile_box,
                    (void *)ri->d_ptile_off})
        if (p) yawb_dfree(ri->ctx, p, ri->ctx->stream);
    ri->rrow = ri->rx = ri->ry = ri->rz = ri->rw = nullptr;
    ri->d_seg_off = ri->d_ptile_off = nullptr;
    ri->d_tiles = nullptr;
    ri->d_tile_box = nullptr;
    ri->h_tiles.clear();
    ri->h_ptile_off.clear();
    ri->n = 0;
    ri->n_tiles = 0;
    ri->device_bytes = 0;
    ri->built = false;
}

// Second-role index over ri->a, or over the union of ri->a and ri->b (same patches and z-bins, both finalized).
static int rindex_build(RIndex *ri) {
    yawb_ctx *ctx = ri->ctx;
    cudaStream_t st = ctx->stream;
    const yawb_cat *ca = ri->a, *cb = ri->b;
    const int P = ca->n_patch, B = ca->n_bins;
    ri->d_frames = ca->d_frames;
    // (patch, z-bin) segments of the index rows: the catalog's own, or both catalogs' rows of a segment together
    std::vector<int> union_off;
    if (cb) {
        const std::vector<int> &oa = ca->second_seg_off(), &ob = cb->second_seg_off();
        union_off.resize(oa.size());
        for (size_t k = 0; k < oa.size(); ++k) union_off[k] = oa[k] + ob[k];
    }
    const std::vector<int> &seg_off = cb ? union_off : ca->second_seg_off();
    const long long n = seg_off.back();
    YAWB_REQUIRE(ca->second_rows() + (cb ? cb->second_rows() : 0) < (1ll << 31) - 1024,
                 "a second-role index is limited to 2^31 rows");
    ri->n = n;
    if (ri_alloc(ri, &ri->rrow, (size_t)n * YAWB_RSTRIDE)) return 1;
    ri->rx = ri->rrow;
    ri->ry = ri->rrow + 1;
    ri->rz = ri->rrow + 2;
    if ((ca->weighted || (cb && cb->weighted)) && ri_alloc(ri, &ri->rw, n)) return 1;
    const int *d_seg_off = ca->second_d_seg_off();
    if (cb) {
        if (ri_alloc(ri, &ri->d_seg_off, seg_off.size())) return 1;
        if (yawb_h2d_small(ctx, ri->d_seg_off, seg_off.data(), seg_off.size() * sizeof(int))) return 1;
        d_seg_off = ri->d_seg_off;
    }
    // The curve only has to order the rows down to about one row per Hilbert cell: with m rows in the largest
    // (patch, bin) segment, 2^k x 2^k >= 1.5 m cells are enough.  The counting sort takes one count per (patch, bin,
    // Hilbert cell), so the resolution is capped at about ONE key per row (the cells then hold 1-4 rows, in arbitrary
    // order; swept on C3: 4 / 1 / 0.25 / 0.06 keys per row -> index build 1.80 / 1.60 / 1.57 / 2.89 ms, count
    // kernels 6.05 / 6.07 / 6.11 / 6.31 ms).  Keys are ints: n_keys <= max(4 P B, n_in, 2^16) < 2^31.
    {
        long long m = 1;
        for (size_t sgm = 0; sgm + 1 < seg_off.size(); ++sgm)
            m = std::max<long long>(m, seg_off[sgm + 1] - seg_off[sgm]);
        int k = 4;
        while (k < 16 && (1ll << (2 * k)) < m + m / 2) ++k;
        const long long key_budget = std::max<long long>(ca->n_in + (cb ? cb->n_in : 0), 1 << 16);
        while (k > 1 && (((long long)P * B) << (2 * k)) > key_budget) --k;
        if (build_second_counting(ri, 2 * k, ((long long)P * B) << (2 * k))) return 1;
    }

    // tiles: chunks of YAWB_TILE rows inside each (patch, bin) segment; the host only needs their number per segment
    // (the table itself is written on the device, k_make_tiles) and per patch
    std::vector<Tile> &tiles = ri->h_tiles;  // filled only if tiles have to be split (straggler guard below)
    tiles.clear();
    ri->h_ptile_off.assign(P + 1, 0);
    std::vector<int> seg_tile_off((size_t)P * B + 1, 0);
    for (int p = 0; p < P; ++p) {
        ri->h_ptile_off[p] = seg_tile_off[(size_t)p * B];
        for (int b = 0; b < B; ++b) {
            const int len = seg_off[(size_t)p * B + b + 1] - seg_off[(size_t)p * B + b];
            seg_tile_off[(size_t)p * B + b + 1] = seg_tile_off[(size_t)p * B + b] + (len + YAWB_TILE - 1) / YAWB_TILE;
        }
    }
    const int n_tiles0 = seg_tile_off[(size_t)P * B];
    ri->h_ptile_off[P] = n_tiles0;

    // Straggler guard: a chunk of consecutive rows can straddle a place where the Hilbert curve leaves the
    // populated part of the patch box and re-enters elsewhere (irregular footprints, masks).  Such a tile
    // has a bounding sphere several times the typical one and would be worth many average work items.
    // Tiles whose radius exceeds 3x the radius expected from the patch's mean density (of the index rows) are cut
    // into sub-tiles of 32 rows (rare; they run the same kernel with most register rows padded).  The common
    // case costs one 4-byte read-back.
    bool table_on_device = false;
    int n_tiles_final = n_tiles0;
    if (n_tiles0 > 0) {
        Scratch scr(ctx, st);
        if (ri_alloc(ri, &ri->d_tiles, (size_t)n_tiles0)) return 1;  // becomes the final table unless tiles are split
        Tile *d_tmp = ri->d_tiles;
        float *d_thr = scr.get<float>(P);
        unsigned *d_nbig = scr.get<unsigned>(1);
        int *d_seg_tile_off = scr.get<int>((size_t)P * B + 1);
        YAWB_REQUIRE(d_thr && d_nbig && d_seg_tile_off, "out of device memory (tile table)");
        std::vector<float> thr(P, 3.0e38f);
        for (int p = 0; p < P; ++p) {
            const PatchFrame &f = ca->h_frames[p];
            const long long np = seg_off[(size_t)(p + 1) * B] - seg_off[(size_t)p * B];
            const double area = std::max(f.umax - f.umin, 0.0) * std::max(f.vmax - f.vmin, 0.0);
            if (np >= 8 * YAWB_TILE && area > 0.0)  // radius of a disc holding YAWB_TILE rows of one z-bin
                thr[p] = (float)(3.0 * std::sqrt((double)YAWB_TILE * B * area / (3.14159265358979 * (double)np)));
        }
        if (yawb_h2d_small(ctx, d_seg_tile_off, seg_tile_off.data(), seg_tile_off.size() * sizeof(int))) return 1;
        if (yawb_h2d_small(ctx, d_thr, thr.data(), P * sizeof(float))) return 1;
        YAWB_CUDA(cudaMemsetAsync(d_nbig, 0, sizeof(unsigned), st));
        k_make_tiles<<<blocks_for((long long)n_tiles0), kThreads, 0, st>>>(d_seg_off, d_seg_tile_off, P * B, B,
                                                                          ca->binned ? 1 : 0, n_tiles0, d_tmp);
        if (ri_alloc(ri, &ri->d_tile_box, (size_t)n_tiles0)) return 1;
        k_tile_spheres<<<blocks_for((long long)n_tiles0 * 32), kThreads, 0, st>>>(ri->rx, ri->ry, ri->rz, d_tmp, n_tiles0,
                                                                                 ri->d_frames, ri->d_tile_box);
        k_count_oversized<<<blocks_for((long long)n_tiles0), kThreads, 0, st>>>(d_tmp, n_tiles0, d_thr, d_nbig);
        unsigned n_big = 0;
        YAWB_CUDA(cudaMemcpyAsync(&n_big, d_nbig, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
        YAWB_CUDA(cudaStreamSynchronize(st));
        table_on_device = n_big == 0;
        if (n_big > 0) {
            tiles.resize((size_t)n_tiles0);
            YAWB_CUDA(cudaMemcpyAsync(tiles.data(), d_tmp, tiles.size() * sizeof(Tile), cudaMemcpyDeviceToHost, st));
            YAWB_CUDA(cudaStreamSynchronize(st));
            for (void **p : {(void **)&ri->d_tiles, (void **)&ri->d_tile_box}) {
                yawb_dfree(ctx, *p, st);
                *p = nullptr;
            }
            ri->device_bytes -= (int64_t)n_tiles0 * (int64_t)(sizeof(Tile) + sizeof(TileBox));
            std::vector<Tile> out;
            out.reserve(tiles.size() + 8 * (size_t)n_big);
            std::vector<int> new_off(P + 1, 0);
            for (int p = 0; p < P; ++p) {
                new_off[p] = (int)out.size();
                for (int t = ri->h_ptile_off[p]; t < ri->h_ptile_off[p + 1]; ++t) {
                    const Tile &tl = tiles[t];
                    if (tl.rad > thr[p] && tl.count > 32) {
                        for (int s0 = 0; s0 < tl.count; s0 += 32) {
                            Tile sub = tl;
                            sub.start = tl.start + s0;
                            sub.count = std::min(32, tl.count - s0);
                            out.push_back(sub);
                        }
                    } else {
                        out.push_back(tl);
                    }
                }
            }
            new_off[P] = (int)out.size();
            tiles.swap(out);
            ri->h_ptile_off = new_off;
            n_tiles_final = (int)tiles.size();
        }
    }
    ri->n_tiles = n_tiles_final;
    if (!table_on_device && ri_alloc(ri, &ri->d_tiles, (size_t)n_tiles_final)) return 1;
    if (ri_alloc(ri, &ri->d_ptile_off, P + 1)) return 1;
    if (yawb_h2d_small(ctx, ri->d_ptile_off, ri->h_ptile_off.data(), (P + 1) * sizeof(int))) return 1;
    if (!table_on_device && ri_alloc(ri, &ri->d_tile_box, tiles.size())) return 1;
    if (!table_on_device && !tiles.empty()) {  // the split tiles need their own spheres and boxes
        if (yawb_h2d_small(ctx, ri->d_tiles, tiles.data(), tiles.size() * sizeof(Tile))) return 1;
        k_tile_spheres<<<blocks_for((long long)ri->n_tiles * 32), kThreads, 0, st>>>(ri->rx, ri->ry, ri->rz, ri->d_tiles,
                                                                                     ri->n_tiles, ri->d_frames, ri->d_tile_box);
    }
    YAWB_CUDA(cudaGetLastError());
    ri->built = true;
    return 0;
}

int yawb_index_build_second(yawb_cat *cat) {
    if (yawb_cat_finalize(cat)) return 1;
    if (cat->ri.built) return 0;
    YawbRange range("yawb:index_second");
    RIndex &ri = cat->ri;
    ri.ctx = cat->ctx;
    ri.a = cat;
    ri.b = nullptr;
    if (int rc = rindex_build(&ri)) {
        rindex_release(&ri);
        return rc;
    }
    cat->device_bytes += ri.device_bytes;
    return 0;
}

void yawb_index_free_second(yawb_cat *cat) {
    cat->device_bytes -= cat->ri.device_bytes;
    if (cat->ri.ctx) rindex_release(&cat->ri);
}

int yawb_rindex_get_union(yawb_ctx *ctx, yawb_cat *a, yawb_cat *b, RIndex **out, bool *built) {
    *built = false;
    for (RIndex *ri : ctx->unions)
        if (ri->a == a && ri->b == b) {
            *out = ri;
            return 0;
        }
    if (yawb_cat_finalize(a) || yawb_cat_finalize(b)) return 1;
    YawbRange range("yawb:index_second_union");
    RIndex *ri = new (std::nothrow) RIndex();
    YAWB_REQUIRE(ri != nullptr, "out of host memory");
    ri->ctx = ctx;
    ri->a = a;
    ri->b = b;
    if (int rc = rindex_build(ri)) {
        rindex_release(ri);
        delete ri;
        return rc;
    }
    ctx->unions.push_back(ri);
    *out = ri;
    *built = true;
    return 0;
}

void yawb_rindex_drop_union(yawb_ctx *ctx, const yawb_cat *cat) {
    for (size_t k = 0; k < ctx->unions.size();) {
        RIndex *ri = ctx->unions[k];
        if (ri->a == cat || ri->b == cat) {
            rindex_release(ri);
            delete ri;
            ctx->unions.erase(ctx->unions.begin() + k);
        } else {
            ++k;
        }
    }
}

// The mask is copied to the device and its rows are counted per (z-bin, patch) right away: the second-role index
// needs those counts on the host to size its segments and tiles.
int yawb_index_set_second_rows(yawb_cat *cat, const uint8_t *mask) {
    if (yawb_cat_finalize(cat)) return 1;
    yawb_ctx *ctx = cat->ctx;
    cudaStream_t st = ctx->stream;
    const int P = cat->n_patch, B = cat->n_bins;
    YAWB_CUDA(cudaStreamSynchronize(st));  // nothing in flight still reads the second-role index
    yawb_index_free_second(cat);
    yawb_rindex_drop_union(ctx, cat);
    dev_free(cat, cat->d_second_mask, (size_t)cat->n_in);
    dev_free(cat, cat->d_seg_off2, (size_t)P * B + 1);
    cat->h_counts2.clear();
    cat->h_seg_off2.clear();
    cat->n2 = 0;
    if (!mask) return 0;
    const long long n = cat->n_in;
    unsigned char *d_mask = nullptr;
    int *d_seg = nullptr;
    std::vector<unsigned long long> counts((size_t)B * P, 0);
    {
        Scratch scr(ctx, st);
        unsigned long long *d_counts = scr.get<unsigned long long>((size_t)B * P);
        // the catalog takes the mask only once everything has worked: on failure it stays without one
        auto fail = [&]() {
            dev_free(cat, d_mask, (size_t)n);
            dev_free(cat, d_seg, (size_t)P * B + 1);
            return 1;
        };
        if (!d_counts || dev_alloc(cat, &d_mask, (size_t)n) || dev_alloc(cat, &d_seg, (size_t)P * B + 1)) {
            yawb_set_error("out of device memory (second-role mask)");
            return fail();
        }
        cudaError_t e = cudaMemsetAsync(d_counts, 0, (size_t)B * P * sizeof(unsigned long long), st);
        if (e == cudaSuccess && n > 0) {
            e = cudaMemcpyAsync(d_mask, mask, (size_t)n, cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess)
                k_second_counts<<<blocks_for(n), kThreads, 0, st>>>(cat->bin, cat->patch, d_mask, n, B, P, d_counts);
        }
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(counts.data(), d_counts, counts.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e != cudaSuccess) {
            yawb_set_error("yawb_catalog_set_second_rows: %s", cudaGetErrorString(e));
            return fail();
        }
    }
    cat->d_second_mask = d_mask;
    cat->d_seg_off2 = d_seg;
    cat->h_counts2.assign(counts.begin(), counts.end());
    cat->h_seg_off2.assign((size_t)P * B + 1, 0);
    for (int p = 0; p < P; ++p)
        for (int b = 0; b < B; ++b)
            cat->h_seg_off2[(size_t)p * B + b + 1] = cat->h_seg_off2[(size_t)p * B + b] + (int)counts[(size_t)b * P + p];
    cat->n2 = cat->h_seg_off2.back();
    return yawb_h2d_small(ctx, cat->d_seg_off2, cat->h_seg_off2.data(), cat->h_seg_off2.size() * sizeof(int));
}

void yawb_index_free(yawb_cat *cat, bool everything) {
    const size_t P = (size_t)cat->n_patch;
    if (cat->findex) {
        cat->device_bytes -= cat->findex->device_bytes;
        yawb_findex_free(cat->findex);
        cat->findex = nullptr;
    }
    yawb_findex_drop_fused(cat->ctx, cat);
    yawb_rindex_drop_union(cat->ctx, cat);
    yawb_index_free_second(cat);
    if (everything) {
        release_staging(cat);
        // a catalog that was never used may still have copies in flight: frees are ordered behind them
        if (cat->ev_meta && !cat->finalized) cudaStreamWaitEvent(cat->ctx->stream, cat->ev_meta, 0);
        if (cat->ev_meta) cudaEventDestroy(cat->ev_meta);
        cat->ev_meta = nullptr;
        const size_t ni = (size_t)cat->n_in;
        dev_free(cat, cat->d_stage_poff, P + 1);
        dev_free(cat, cat->d_stage_bin8, ni);
        dev_free(cat, cat->xyz, ni * 3);
        cat->x = cat->y = cat->z = nullptr;
        dev_free(cat, cat->w, ni);
        dev_free(cat, cat->bin, ni);
        dev_free(cat, cat->patch, ni);
        dev_free(cat, cat->d_frames, P);
        dev_free(cat, cat->d_seg_off, P * (size_t)cat->n_bins + 1);
        dev_free(cat, cat->d_second_mask, ni);
        dev_free(cat, cat->d_seg_off2, P * (size_t)cat->n_bins + 1);
    }
}

// -------------------------------------------------------------------------------------------
// Upper bound on the device bytes of one catalog (yawb_catalog_footprint): every block the upload, the second-role
// mask and the two index builds above request, scratch included, each rounded as the allocator rounds it.  Blocks
// freed along the way are counted as well, so the bound also holds for the allocator's high-water mark of a context
// that starts empty (a freed block is only handed out again for a request it was counted for, or a smaller one).
int64_t yawb_index_footprint(int64_t n_rows, int n_patch, int n_bins, uint32_t what) {
    const size_t n = (size_t)std::max<int64_t>(n_rows, 0);
    const size_t P = (size_t)std::max(n_patch, 1), B = (size_t)std::max(n_bins, 1), PB = P * B;
    const bool w = what & YAWB_FOOT_WEIGHTED;
    size_t total = 0;
    auto blk = [&](size_t count, size_t size) { total += yawb_dcache_round(std::max<size_t>(count, 1) * size); };
    if (!(what & YAWB_FOOT_NO_UPLOAD)) {
        // yawb_index_upload
        blk(3 * n, sizeof(double));
        blk(n, sizeof(int32_t));
        if (w) blk(n, sizeof(double));
        if (what & (YAWB_FOOT_BINNED | YAWB_FOOT_U8 | YAWB_FOOT_Z | YAWB_FOOT_LABELLED)) blk(n, sizeof(int32_t));
        if (what & YAWB_FOOT_U8) blk(n, 1);
        if (what & YAWB_FOOT_Z) blk(n, sizeof(double));
        blk(P, sizeof(PatchFrame));
        blk(PB + 1, sizeof(int));
        blk(P + 1, sizeof(long long));
        // yawb_cat_finalize
        blk(3 * P, sizeof(double));
        blk(PB, sizeof(double));
        blk(PB, sizeof(unsigned long long));
        blk(P * kBox, sizeof(unsigned long long));
        if (what & YAWB_FOOT_Z) blk(B + 1, sizeof(double));
        // yawb_index_set_second_rows
        if (what & YAWB_FOOT_MASK) {
            blk(PB, sizeof(unsigned long long));
            blk(n, 1);
            blk(PB + 1, sizeof(int));
        }
    }
    if (what & YAWB_FOOT_FIRST) {
        // findex_build: the grid of a (patch, z-bin) has gu x gv cells with gu <= 4 du / c + 1, gv <= dv / c + 1,
        // c^2 = kTargetPerCell du dv / max(rows / B, 1) and c >= max(du, dv) / 2048, so gu gv <= 4 max(rows / B, 1) /
        // kTargetPerCell + 4 * 2048 + 2048 + 1 (growing the cells only lowers it); at most kMaxGridCells in all
        const double cells = std::ceil(4.0 * (double)(n + PB) / kTargetPerCell) + (double)PB * (4 * 2048 + 2048 + 1);
        const size_t base = (size_t)std::min<double>(cells, (double)kMaxGridCells);
        blk(P, sizeof(PatchFrame));
        blk(P, sizeof(SGrid));
        blk(n, sizeof(SRec));
        if (w) blk(n, sizeof(double));
        blk(base + 1, sizeof(int));
        blk(n, sizeof(int2));
        blk((base + 1 + kScanBlock - 1) / kScanBlock + 1, sizeof(unsigned long long));
    }
    if (what & YAWB_FOOT_SECOND) {
        // rindex_build: tiles are chunks of YAWB_TILE rows within each (patch, z-bin) segment
        const size_t n_keys = std::max<size_t>(std::max<size_t>(n, 1 << 16), 4 * PB);
        const size_t n_tiles = n / YAWB_TILE + PB;
        blk(n * YAWB_RSTRIDE, sizeof(double));
        if (w) blk(n, sizeof(double));
        if (what & YAWB_FOOT_NO_UPLOAD) blk(PB + 1, sizeof(int));  // the segments of a union index
        blk(n_keys, sizeof(int));
        blk(n, sizeof(int2));
        blk(P, sizeof(HMap));
        blk((n_keys + kScanBlock - 1) / kScanBlock + 1, sizeof(unsigned long long));
        blk(n_tiles, sizeof(Tile));
        blk(P, sizeof(float));
        blk(1, sizeof(unsigned));
        blk(PB + 1, sizeof(int));
        blk(n_tiles, sizeof(TileBox));
        blk(P + 1, sizeof(int));
    }
    return (int64_t)total;
}
