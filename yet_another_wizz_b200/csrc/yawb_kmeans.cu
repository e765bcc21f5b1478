// Deterministic spherical k-means for patch centres: yawb_kmeans (contract in include/yawb.h, DESIGN.md §4.4).
//
// The rows stay resident for the whole call.  Every sum is an int64 sum of fixed-point coordinates, so atomics
// in any order give the same bits, and the centre of a sum and the nearest-centre search are sequences of
// correctly rounded FP64 operations: the result equals the numpy restatement in oracle/kmeans.py bit for bit.
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstring>
#include <vector>

#include "yawb_internal.cuh"

namespace {

constexpr int KM_MAX_K = 4096;
constexpr int KM_CB = 1024;        // centres per shared-memory block (24 KB), as in k_assign_patches
constexpr int KM_THREADS = 256;    // assignment kernel
constexpr int KM_RPT = 4;          // rows per thread: a centre read from shared memory serves four rows
constexpr int KM_TILE = KM_THREADS * KM_RPT;
constexpr int KM_STAT_THREADS = 512;
constexpr int KM_CELLS = 4096;     // cells per pass of the bisection reduction (4 shared sums each: 128 KB)
constexpr int KM_FIELDS = 10;      // per cell: min q (x, y, z), max q (x, y, z), sum q (x, y, z), rows
constexpr double KM_SCALE = 4294967296.0;  // 2^32
constexpr unsigned FULL = 0xffffffffu;
constexpr unsigned long long NONE = ~0ull;

struct KmSplit {
    long long cnt, sum;  // rows of the cell and its sum of q along `axis`
    int axis;            // -1: the cell is not split in this round
    int child;           // id of the high child
};

__device__ __forceinline__ long long fixq(double v, double scale) { return __double2ll_rn(__dmul_rn(v, scale)); }

__device__ __forceinline__ long long warp_sum(long long v) {
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
__device__ __forceinline__ long long warp_min(long long v) {
    for (int o = 16; o; o >>= 1) v = min(v, (long long)__shfl_xor_sync(FULL, v, o));
    return v;
}
__device__ __forceinline__ long long warp_max(long long v) {
    for (int o = 16; o; o >>= 1) v = max(v, (long long)__shfl_xor_sync(FULL, v, o));
    return v;
}
__device__ __forceinline__ unsigned long long warp_umax(unsigned long long v) {
    for (int o = 16; o; o >>= 1) v = max(v, (unsigned long long)__shfl_xor_sync(FULL, v, o));
    return v;
}
__device__ __forceinline__ unsigned long long warp_umin(unsigned long long v) {
    for (int o = 16; o; o >>= 1) v = min(v, (unsigned long long)__shfl_xor_sync(FULL, v, o));
    return v;
}
// true when every lane of the warp holds a valid row of the same label: the warp then reduces in registers and
// one lane updates shared memory (sorted input, or k = 1, would otherwise serialise on one address)
// (every lane must reach the shuffle: it is not inside the short-circuited condition)
__device__ __forceinline__ bool warp_uniform(int lab, bool valid) {
    const int lab0 = __shfl_sync(FULL, lab, 0);
    return __all_sync(FULL, valid && lab == lab0);
}

// int64 sums in shared memory from native 32-bit atomics (a 64-bit shared atomic is a compare-and-swap loop):
// the low word wraps modulo 2^32, the lane whose addition wraps it carries into the high word, and the sum is
// hi 2^32 + lo.  hi stays far below 2^31 (a block adds fewer than 2^31 values below 2^37).
__device__ __forceinline__ void sh_add64(unsigned *lo, int *hi, long long v) {
    const unsigned l = (unsigned)v;
    const unsigned old = atomicAdd(lo, l);
    const int h = (int)(v >> 32) + ((unsigned)(old + l) < old ? 1 : 0);
    if (h) atomicAdd(hi, h);
}
__device__ __forceinline__ long long sh_get64(const unsigned *lo, const int *hi) {
    return (long long)(((unsigned long long)(long long)*hi << 32) + *lo);
}

// one pass: rows that are not finite or have |coordinate| > 1, weights that are negative or not finite, and the
// largest weight (bits of a non-negative double order like the values) -> out[0..2]
__global__ void k_km_validate(const double *__restrict__ xyz, const double *__restrict__ w, long long n,
                              unsigned long long *__restrict__ out) {
    unsigned long long bad = 0, bad_w = 0, max_w = 0;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        if (!(fabs(xyz[3 * i]) <= 1.0 && fabs(xyz[3 * i + 1]) <= 1.0 && fabs(xyz[3 * i + 2]) <= 1.0)) ++bad;
        if (w) {
            const double v = w[i];
            if (!(v >= 0.0 && v <= 1.7976931348623157e308)) ++bad_w;
            else if (v > 0.0) max_w = max(max_w, (unsigned long long)__double_as_longlong(v));
        }
    }
    bad = (unsigned long long)warp_sum((long long)bad);
    bad_w = (unsigned long long)warp_sum((long long)bad_w);
    max_w = warp_umax(max_w);
    if ((threadIdx.x & 31) == 0) {
        if (bad) atomicAdd(&out[0], bad);
        if (bad_w) atomicAdd(&out[1], bad_w);
        if (max_w) atomicMax(&out[2], max_w);
    }
}

__global__ void k_km_stats_init(long long *__restrict__ s, int cells) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= cells * KM_FIELDS) return;
    const int f = t % KM_FIELDS;
    s[t] = f < 3 ? LLONG_MAX : f < 6 ? LLONG_MIN : 0;
}

// Bisection: per-cell min / max / sum of the unweighted q and row count of the cells [c0, c0 + nc).  Sums and
// counts are accumulated per block in shared memory and flushed with one global atomic per (block, non-empty
// cell, field); minima and maxima go straight to global memory (native 64-bit atomics), once per warp when the
// whole warp holds one cell.
__global__ void __launch_bounds__(KM_STAT_THREADS) k_km_cell_stats(const double *__restrict__ xyz, const int *__restrict__ lab,
                                                                   long long n, int c0, int nc, long long *__restrict__ stats) {
    extern __shared__ unsigned shs[];  // lo words [nc][4], then hi words [nc][4]: sum q (x, y, z), rows
    unsigned *lo = shs;
    int *hi = reinterpret_cast<int *>(shs + 4 * nc);
    for (int t = threadIdx.x; t < 8 * nc; t += blockDim.x) shs[t] = 0;
    __syncthreads();
    for (long long base = blockIdx.x * (long long)blockDim.x; base < n; base += (long long)gridDim.x * blockDim.x) {
        const long long i = base + threadIdx.x;
        const int l = i < n ? lab[i] - c0 : -1;
        const bool valid = l >= 0 && l < nc;
        long long q[3] = {0, 0, 0};
        if (valid)
            for (int a = 0; a < 3; ++a) q[a] = fixq(xyz[3 * i + a], KM_SCALE);
        if (warp_uniform(l, valid)) {
            long long v[9];
            for (int a = 0; a < 3; ++a) {
                v[a] = warp_min(q[a]);
                v[3 + a] = warp_max(q[a]);
                v[6 + a] = warp_sum(q[a]);
            }
            if ((threadIdx.x & 31) == 0) {
                long long *g = stats + (size_t)(c0 + l) * KM_FIELDS;
                for (int a = 0; a < 3; ++a) {
                    atomicMin(g + a, v[a]);
                    atomicMax(g + 3 + a, v[3 + a]);
                    sh_add64(lo + 4 * l + a, hi + 4 * l + a, v[6 + a]);
                }
                sh_add64(lo + 4 * l + 3, hi + 4 * l + 3, 32);
            }
        } else if (valid) {
            long long *g = stats + (size_t)(c0 + l) * KM_FIELDS;
            for (int a = 0; a < 3; ++a) {
                atomicMin(g + a, q[a]);
                atomicMax(g + 3 + a, q[a]);
                sh_add64(lo + 4 * l + a, hi + 4 * l + a, q[a]);
            }
            sh_add64(lo + 4 * l + 3, hi + 4 * l + 3, 1);
        }
    }
    __syncthreads();
    for (int t = threadIdx.x; t < 4 * nc; t += blockDim.x) {
        const long long v = sh_get64(lo + t, hi + t);
        if (v) atomicAdd((unsigned long long *)(stats + (size_t)(c0 + t / 4) * KM_FIELDS + 6 + t % 4), (unsigned long long)v);
    }
}

// Bisection: a row of a split cell moves to the high child iff q_axis * count > sum q_axis (exact in int64).
__global__ void k_km_relabel(const double *__restrict__ xyz, int *__restrict__ lab, long long n, const KmSplit *__restrict__ sp) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const KmSplit s = sp[lab[i]];
        if (s.axis >= 0 && fixq(xyz[3 * i + s.axis], KM_SCALE) * s.cnt > s.sum) lab[i] = s.child;
    }
}

// Centre of every cluster from its int64 sums (s[j * stride + 0..2]): s / sqrt((sx sx + sy sy) + sz sz), correctly
// rounded throughout.  A cluster with s = (0, 0, 0) is empty: flagged and counted when `empty` is given.
__global__ void k_km_centre(const long long *__restrict__ s, int stride, int k, double *__restrict__ c,
                            unsigned char *__restrict__ empty, unsigned long long *__restrict__ n_empty) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= k) return;
    const long long *sj = s + (size_t)j * stride;
    const double x = __ll2double_rn(sj[0]), y = __ll2double_rn(sj[1]), z = __ll2double_rn(sj[2]);
    const double norm = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)), __dmul_rn(z, z)));
    c[3 * j] = __ddiv_rn(x, norm);
    c[3 * j + 1] = __ddiv_rn(y, norm);
    c[3 * j + 2] = __ddiv_rn(z, norm);
    if (empty) {
        const bool e = sj[0] == 0 && sj[1] == 0 && sj[2] == 0;
        empty[j] = e;
        if (e) atomicAdd(n_empty, 1ull);
    }
}

// The hot path of a Lloyd iteration: nearest centre of every row (vq arithmetic), label written and changes
// counted, and the row's q added to the sums of its new cluster.  Persistent blocks keep [k][3] int64 sums in
// shared memory and flush them once; centres are staged in shared memory in blocks of KM_CB.
template <bool WEIGHTED>
__global__ void __launch_bounds__(KM_THREADS) k_km_assign(const double *__restrict__ xyz, const double *__restrict__ w,
                                                          long long n, const double *__restrict__ centers, int k,
                                                          double scale, int *__restrict__ lab, int compare,
                                                          long long *__restrict__ sums, unsigned long long *__restrict__ changed) {
    extern __shared__ double sm[];
    const int cb = min(k, KM_CB);
    double *cs = sm;                                           // [cb][3]
    unsigned *lo = reinterpret_cast<unsigned *>(sm + 3 * cb);  // [k][3] low words of the sums (sh_add64)
    int *hi = reinterpret_cast<int *>(lo + 3 * k);             // [k][3] high words
    for (int t = threadIdx.x; t < 6 * k; t += blockDim.x) lo[t] = 0;
    const bool resident = k <= KM_CB;  // every centre fits: staged once
    if (resident)
        for (int t = threadIdx.x; t < 3 * k; t += blockDim.x) cs[t] = centers[t];
    __syncthreads();
    unsigned n_changed = 0;
    const long long n_tiles = (n + KM_TILE - 1) / KM_TILE;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long base = tile * KM_TILE + threadIdx.x;
        double x[KM_RPT], y[KM_RPT], z[KM_RPT], best[KM_RPT];
        int arg[KM_RPT];
#pragma unroll
        for (int r = 0; r < KM_RPT; ++r) {
            const long long i = base + (long long)r * KM_THREADS;
            x[r] = y[r] = z[r] = 0.0;
            if (i < n) {
                x[r] = xyz[3 * i];
                y[r] = xyz[3 * i + 1];
                z[r] = xyz[3 * i + 2];
            }
            best[r] = __longlong_as_double(0x7ff0000000000000ll);  // +inf
            arg[r] = 0;
        }
        for (int c0 = 0; c0 < k; c0 += KM_CB) {
            const int nc = min(KM_CB, k - c0);
            if (!resident) {
                __syncthreads();
                for (int t = threadIdx.x; t < 3 * nc; t += blockDim.x) cs[t] = centers[3 * (size_t)c0 + t];
                __syncthreads();
            }
            for (int c = 0; c < nc; ++c) {
                const double cx = cs[3 * c], cy = cs[3 * c + 1], cz = cs[3 * c + 2];
#pragma unroll
                for (int r = 0; r < KM_RPT; ++r) {
                    const double d = yawb_vq_d2(cx, cy, cz, x[r], y[r], z[r]);
                    if (d < best[r]) {
                        best[r] = d;
                        arg[r] = c0 + c;
                    }
                }
            }
        }
#pragma unroll
        for (int r = 0; r < KM_RPT; ++r) {
            const long long i = base + (long long)r * KM_THREADS;
            const bool valid = i < n;
            long long qx = 0, qy = 0, qz = 0;
            if (valid) {
                if (compare && lab[i] != arg[r]) ++n_changed;
                lab[i] = arg[r];
                if (WEIGHTED) {
                    const double wi = w[i];
                    qx = fixq(__dmul_rn(wi, x[r]), scale);
                    qy = fixq(__dmul_rn(wi, y[r]), scale);
                    qz = fixq(__dmul_rn(wi, z[r]), scale);
                } else {
                    qx = fixq(x[r], scale);
                    qy = fixq(y[r], scale);
                    qz = fixq(z[r], scale);
                }
            }
            if (warp_uniform(arg[r], valid)) {
                qx = warp_sum(qx);
                qy = warp_sum(qy);
                qz = warp_sum(qz);
                if ((threadIdx.x & 31) == 0) {
                    const int a = 3 * arg[r];
                    sh_add64(lo + a, hi + a, qx);
                    sh_add64(lo + a + 1, hi + a + 1, qy);
                    sh_add64(lo + a + 2, hi + a + 2, qz);
                }
            } else if (valid) {
                const int a = 3 * arg[r];
                sh_add64(lo + a, hi + a, qx);
                sh_add64(lo + a + 1, hi + a + 1, qy);
                sh_add64(lo + a + 2, hi + a + 2, qz);
            }
        }
    }
    __syncthreads();
    for (int t = threadIdx.x; t < 3 * k; t += blockDim.x) {
        const long long v = sh_get64(lo + t, hi + t);
        if (v) atomicAdd((unsigned long long *)&sums[t], (unsigned long long)v);
    }
    n_changed = __reduce_add_sync(FULL, n_changed);
    if ((threadIdx.x & 31) == 0 && n_changed) atomicAdd(changed, (unsigned long long)n_changed);
}

// Relocation of an empty cluster: the row with the largest key (squared distance to its own centre in the
// previous centres, -row index) among the rows below the key taken last (st[2], st[3]; st[3] == NONE: none yet).
// Pass 0 finds the largest distance (st[0]), pass 1 the lowest row at that distance (st[1]).
__global__ void k_km_far(const double *__restrict__ xyz, const int *__restrict__ lab, long long n,
                         const double *__restrict__ prev, int pass, unsigned long long *__restrict__ st) {
    const unsigned long long pd = st[2], pr = st[3], dmax = st[0];
    unsigned long long v = pass == 0 ? 0ull : NONE;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const double *c = prev + 3 * (size_t)lab[i];
        const unsigned long long d =
            (unsigned long long)__double_as_longlong(yawb_vq_d2(c[0], c[1], c[2], xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]));
        if (!(pr == NONE || d < pd || (d == pd && (unsigned long long)i > pr))) continue;
        if (pass == 0) v = max(v, d);
        else if (d == dmax) v = min(v, (unsigned long long)i);
    }
    if (pass == 0) {
        v = warp_umax(v);
        if ((threadIdx.x & 31) == 0 && v) atomicMax(&st[0], v);
    } else {
        v = warp_umin(v);
        if ((threadIdx.x & 31) == 0 && v != NONE) atomicMin(&st[1], v);
    }
}

__global__ void k_km_take(const double *__restrict__ xyz, int j, double *__restrict__ next, unsigned long long *__restrict__ st) {
    const unsigned long long r = st[1];
    for (int a = 0; a < 3; ++a) next[3 * j + a] = xyz[3 * r + a];
    st[2] = st[0];
    st[3] = r;
    st[0] = 0;
    st[1] = NONE;
}

struct KmBufs {
    double *xyz = nullptr, *w = nullptr, *c = nullptr;  // c: two sets of k centres (current, next)
    int *lab = nullptr;
    long long *s = nullptr;                // [k][KM_FIELDS] cell statistics, then [k][3] cluster sums
    unsigned long long *ctr = nullptr;     // [0] changed labels, [1] empty clusters, [4..7] relocation state
    KmSplit *split = nullptr;
    unsigned char *empty = nullptr;
};

int kmeans_run(yawb_ctx *ctx, const KmBufs &b, const double *xyz, const double *w, long long n, int k, int max_iter,
               double *centers_xyz, int32_t *labels, int *n_iter, int *converged) {
    cudaStream_t st = ctx->stream;
    const int stride_grid = std::max(ctx->sms, 1) * 8;
    YAWB_CUDA(cudaMemcpyAsync(b.xyz, xyz, (size_t)n * 3 * sizeof(double), cudaMemcpyHostToDevice, st));
    if (w) YAWB_CUDA(cudaMemcpyAsync(b.w, w, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, st));

    // inputs are checked on the device, in one pass
    unsigned long long h[4] = {0, 0, 0, 0};
    YAWB_CUDA(cudaMemsetAsync(b.ctr, 0, 8 * sizeof(unsigned long long), st));
    k_km_validate<<<stride_grid, 256, 0, st>>>(b.xyz, b.w, n, b.ctr);
    YAWB_CUDA(cudaGetLastError());
    YAWB_CUDA(cudaMemcpyAsync(h, b.ctr, 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    YAWB_CUDA(cudaStreamSynchronize(st));
    YAWB_REQUIRE(h[0] == 0, "yawb_kmeans: %llu rows are not finite or have a coordinate outside [-1, 1]", h[0]);
    double scale = KM_SCALE;
    if (w) {
        YAWB_REQUIRE(h[1] == 0, "yawb_kmeans: %llu weights are negative or not finite", h[1]);
        YAWB_REQUIRE(h[2] != 0, "yawb_kmeans: the weights must have a positive sum");
        double max_w;
        std::memcpy(&max_w, &h[2], sizeof(double));
        int e = 0;
        std::frexp(max_w, &e);
        YAWB_REQUIRE(e >= -991, "yawb_kmeans: the largest weight (%g) is below 2^-992", max_w);
        scale = std::ldexp(1.0, 32 - e);  // |w x| < 2^e, so |q| <= 2^32
    }

    // initial centres: deterministic bisection of the unweighted rows
    YAWB_CUDA(cudaMemsetAsync(b.lab, 0, (size_t)n * sizeof(int), st));
    int stat_blocks = 0;
    const size_t stat_smem_max = (size_t)KM_CELLS * 8 * sizeof(unsigned);
    YAWB_CUDA(cudaFuncSetAttribute(k_km_cell_stats, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)stat_smem_max));
    auto cell_stats = [&](int cells) -> int {
        k_km_stats_init<<<(cells * KM_FIELDS + 255) / 256, 256, 0, st>>>(b.s, cells);
        for (int c0 = 0; c0 < cells; c0 += KM_CELLS) {
            const int nc = std::min(KM_CELLS, cells - c0);
            const size_t smem = (size_t)nc * 8 * sizeof(unsigned);
            YAWB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&stat_blocks, k_km_cell_stats, KM_STAT_THREADS, smem));
            const long long want = (n + KM_STAT_THREADS - 1) / KM_STAT_THREADS;
            const int blocks = (int)std::min<long long>(want, (long long)std::max(stat_blocks, 1) * ctx->sms);
            k_km_cell_stats<<<blocks, KM_STAT_THREADS, smem, st>>>(b.xyz, b.lab, n, c0, nc, b.s);
        }
        YAWB_CUDA(cudaGetLastError());
        return 0;
    };
    std::vector<long long> hs((size_t)k * KM_FIELDS);
    std::vector<KmSplit> sp(k);
    std::vector<int> cand;
    for (int c = 1; c < k;) {
        if (cell_stats(c)) return 1;
        YAWB_CUDA(cudaMemcpyAsync(hs.data(), b.s, (size_t)c * KM_FIELDS * sizeof(long long), cudaMemcpyDeviceToHost, st));
        YAWB_CUDA(cudaStreamSynchronize(st));
        cand.clear();
        for (int j = 0; j < c; ++j) {
            const long long *f = &hs[(size_t)j * KM_FIELDS];
            sp[j].axis = -1;
            if (f[3] > f[0] || f[4] > f[1] || f[5] > f[2]) cand.push_back(j);
        }
        YAWB_REQUIRE(!cand.empty(), "yawb_kmeans: fewer distinct positions than patches (%d requested, %d found)", k, c);
        // the min(c, k - c) splittable cells with the most rows (ties: lower id), split in ascending id order
        const size_t m = std::min<size_t>(cand.size(), (size_t)std::min(c, k - c));
        std::stable_sort(cand.begin(), cand.end(),
                         [&](int a, int b2) { return hs[(size_t)a * KM_FIELDS + 9] > hs[(size_t)b2 * KM_FIELDS + 9]; });
        cand.resize(m);
        std::sort(cand.begin(), cand.end());
        for (size_t r = 0; r < m; ++r) {
            const int j = cand[r];
            const long long *f = &hs[(size_t)j * KM_FIELDS];
            int axis = 0;  // largest extent; ties: x, then y, then z
            for (int a = 1; a < 3; ++a)
                if (f[3 + a] - f[a] > f[3 + axis] - f[axis]) axis = a;
            sp[j] = KmSplit{f[9], f[6 + axis], axis, c + (int)r};
        }
        YAWB_CUDA(cudaMemcpyAsync(b.split, sp.data(), (size_t)c * sizeof(KmSplit), cudaMemcpyHostToDevice, st));
        k_km_relabel<<<stride_grid, 256, 0, st>>>(b.xyz, b.lab, n, b.split);
        YAWB_CUDA(cudaGetLastError());
        YAWB_CUDA(cudaStreamSynchronize(st));  // `sp` is rewritten by the next round
        c += (int)m;
    }
    if (cell_stats(k)) return 1;
    double *cset[2] = {b.c, b.c + 3 * (size_t)k};
    k_km_centre<<<(k + 127) / 128, 128, 0, st>>>(b.s + 6, KM_FIELDS, k, cset[0], nullptr, nullptr);

    // Lloyd iterations
    const size_t cb = std::min(k, KM_CB);
    const size_t smem = (3 * cb + 3 * (size_t)k) * sizeof(double);
    auto kern = w ? k_km_assign<true> : k_km_assign<false>;
    YAWB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    YAWB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, KM_THREADS, smem));
    const int assign_blocks = (int)std::min<long long>((n + KM_TILE - 1) / KM_TILE, (long long)std::max(occ, 1) * ctx->sms);
    auto assign = [&](const double *c, int compare) -> int {
        YAWB_CUDA(cudaMemsetAsync(b.s, 0, (size_t)k * 3 * sizeof(long long), st));
        YAWB_CUDA(cudaMemsetAsync(b.ctr, 0, 2 * sizeof(unsigned long long), st));
        kern<<<assign_blocks, KM_THREADS, smem, st>>>(b.xyz, b.w, n, c, k, scale, b.lab, compare, b.s, b.ctr);
        YAWB_CUDA(cudaGetLastError());
        return 0;
    };
    if (assign(cset[0], 0)) return 1;
    int cur = 0, it = 0;
    bool conv = false;
    std::vector<unsigned char> empty;
    for (;;) {
        const bool more = it < max_iter;
        if (more) k_km_centre<<<(k + 127) / 128, 128, 0, st>>>(b.s, 3, k, cset[cur ^ 1], b.empty, b.ctr + 1);
        YAWB_CUDA(cudaMemcpyAsync(h, b.ctr, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        YAWB_CUDA(cudaStreamSynchronize(st));
        if (it > 0 && h[0] == 0) {
            conv = true;
            break;
        }
        if (!more) break;
        if (h[1]) {  // rare: relocate the empty clusters in ascending order
            empty.resize(k);
            YAWB_CUDA(cudaMemcpyAsync(empty.data(), b.empty, k, cudaMemcpyDeviceToHost, st));
            const unsigned long long init[4] = {0, NONE, 0, NONE};
            YAWB_CUDA(cudaMemcpyAsync(b.ctr + 4, init, sizeof(init), cudaMemcpyHostToDevice, st));
            YAWB_CUDA(cudaStreamSynchronize(st));
            for (int j = 0; j < k; ++j) {
                if (!empty[j]) continue;
                for (int pass = 0; pass < 2; ++pass)
                    k_km_far<<<stride_grid, 256, 0, st>>>(b.xyz, b.lab, n, cset[cur], pass, b.ctr + 4);
                k_km_take<<<1, 1, 0, st>>>(b.xyz, j, cset[cur ^ 1], b.ctr + 4);
            }
            YAWB_CUDA(cudaGetLastError());
        }
        if (assign(cset[cur ^ 1], 1)) return 1;
        cur ^= 1;
        ++it;
    }
    YAWB_CUDA(cudaMemcpyAsync(centers_xyz, cset[cur], (size_t)k * 3 * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (labels) YAWB_CUDA(cudaMemcpyAsync(labels, b.lab, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, st));
    YAWB_CUDA(cudaStreamSynchronize(st));
    YAWB_CUDA(cudaGetLastError());
    *n_iter = it;
    *converged = conv ? 1 : 0;
    return 0;
}

}  // namespace

extern "C" int yawb_kmeans(yawb_ctx *ctx, const double *xyz, const double *w, int64_t n, int k, int max_iter,
                           double *centers_xyz, int32_t *labels, int *n_iter, int *converged) {
    YAWB_REQUIRE(ctx != nullptr, "yawb_kmeans: ctx is NULL");
    YAWB_REQUIRE(xyz && centers_xyz && n_iter && converged, "yawb_kmeans: NULL argument");
    YAWB_REQUIRE(k >= 1 && k <= KM_MAX_K, "yawb_kmeans: k must be in 1..%d (got %d)", KM_MAX_K, k);
    YAWB_REQUIRE(n >= k, "yawb_kmeans: more patches (%d) than rows (%lld)", k, (long long)n);
    YAWB_REQUIRE(n < (1ll << 30), "yawb_kmeans: at most 2^30 - 1 rows (got %lld)", (long long)n);
    YAWB_REQUIRE(max_iter >= 0, "yawb_kmeans: max_iter must be >= 0 (got %d)", max_iter);
    YAWB_CUDA(cudaSetDevice(ctx->device));
    YawbRange range("yawb_kmeans");
    cudaStream_t st = ctx->stream;
    KmBufs b;
    int rc = 1;
    if (!yawb_dalloc(ctx, (void **)&b.xyz, (size_t)n * 3 * sizeof(double), st) &&
        !(w && yawb_dalloc(ctx, (void **)&b.w, (size_t)n * sizeof(double), st)) &&
        !yawb_dalloc(ctx, (void **)&b.c, (size_t)k * 6 * sizeof(double), st) &&
        !yawb_dalloc(ctx, (void **)&b.lab, (size_t)n * sizeof(int), st) &&
        !yawb_dalloc(ctx, (void **)&b.s, (size_t)k * KM_FIELDS * sizeof(long long), st) &&
        !yawb_dalloc(ctx, (void **)&b.ctr, 8 * sizeof(unsigned long long), st) &&
        !yawb_dalloc(ctx, (void **)&b.split, (size_t)k * sizeof(KmSplit), st) &&
        !yawb_dalloc(ctx, (void **)&b.empty, (size_t)k, st))
        rc = kmeans_run(ctx, b, xyz, w, n, k, max_iter, centers_xyz, labels, n_iter, converged);
    cudaStreamSynchronize(st);  // nothing of a failed call may still use the buffers or the caller's arrays
    for (void *p : {(void *)b.xyz, (void *)b.w, (void *)b.c, (void *)b.lab, (void *)b.s, (void *)b.ctr,
                    (void *)b.split, (void *)b.empty})
        if (p) yawb_dfree(ctx, p, st);
    return rc;
}
