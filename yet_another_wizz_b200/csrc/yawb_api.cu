// C ABI of libyawb.so (see include/yawb.h for the contract of every entry point).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>

#include <cstdlib>

#include "yawb_internal.cuh"

namespace {
thread_local char g_err[1024] = "";

__global__ void k_u64_to_f64(const unsigned long long *__restrict__ in, double *__restrict__ out, long long n) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) out[i] = (double)in[i];
}
}  // namespace

void yawb_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

// 16 bytes per thread from mapped pinned host memory to device memory
__global__ void k_pull_host(uint4 *__restrict__ dst, const uint4 *__restrict__ src, size_t n16) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = src[i];
}

int yawb_h2d_small(yawb_ctx *ctx, void *dst, const void *src, size_t bytes) {
    if (bytes == 0) return 0;
    cudaStream_t st = ctx->stream;
    const size_t padded = (bytes + 15) & ~(size_t)15;
    // device buffers come from the caching allocator (256-byte aligned, sizes rounded up to 512 B), so
    // writing the padding is safe; tables too large for the arena take the ordinary copy path
    if (!ctx->h2d_base || padded > ctx->h2d_size / 2 || ((uintptr_t)dst & 15)) {
        YAWB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
        return 0;
    }
    if (ctx->h2d_used + padded > ctx->h2d_size) {  // arena full: everything staged so far must have been pulled
        YAWB_CUDA(cudaStreamSynchronize(st));
        ctx->h2d_used = 0;
    }
    unsigned char *stage = ctx->h2d_base + ctx->h2d_used;
    ctx->h2d_used += padded;
    memcpy(stage, src, bytes);
    const size_t n16 = padded / 16;
    const int blocks = (int)std::min<size_t>((n16 + 255) / 256, 296);
    k_pull_host<<<blocks, 256, 0, st>>>((uint4 *)dst, (const uint4 *)stage, n16);
    YAWB_CUDA(cudaGetLastError());
    return 0;
}

// nearest centre in xyz: the arithmetic of scipy.cluster.vq.vq for fewer than 5 features (differences
// code - obs, squares summed in order, strict "<" so the first minimum wins), centres staged in shared
// memory in blocks
__global__ void k_assign_patches(const double *__restrict__ xyz, long long n, const double *__restrict__ centers,
                                 int n_centers, int *__restrict__ out) {
    extern __shared__ double cs[];  // [block of centres][3]
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    double x = 0.0, y = 0.0, z = 0.0;
    if (i < n) {
        x = xyz[3 * i];
        y = xyz[3 * i + 1];
        z = xyz[3 * i + 2];
    }
    double best = 1.0e308 * 10.0;  // +inf
    int arg = 0;
    constexpr int CB = 1024;
    for (int c0 = 0; c0 < n_centers; c0 += CB) {
        const int nc = min(CB, n_centers - c0);
        __syncthreads();
        for (int k = threadIdx.x; k < 3 * nc; k += blockDim.x) cs[k] = centers[3 * (size_t)c0 + k];
        __syncthreads();
        for (int c = 0; c < nc; ++c) {
            const double d = yawb_vq_d2(cs[3 * c], cs[3 * c + 1], cs[3 * c + 2], x, y, z);
            if (d < best) {
                best = d;
                arg = c0 + c;
            }
        }
    }
    if (i < n) out[i] = arg;
}

// one thread per (pair, bin): the value joins the total and the "removed with patch p" sums of both patches
__global__ void k_jackknife(const double *__restrict__ v, const int *__restrict__ pi, const int *__restrict__ pj,
                            int n_pairs, int n_bins, double *__restrict__ total, double *__restrict__ removed) {
    const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (t >= (long long)n_pairs * n_bins) return;
    const int k = (int)(t / n_bins), b = (int)(t % n_bins);
    const double x = v[t];
    if (x == 0.0) return;
    atomicAdd(&total[b], x);
    const int i = pi[k], j = pj[k];
    atomicAdd(&removed[(size_t)i * n_bins + b], x);
    if (j != i) atomicAdd(&removed[(size_t)j * n_bins + b], x);
}
__global__ void k_jackknife_finish(const double *__restrict__ total, int n_patch, int n_bins, double *__restrict__ samples) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_patch * n_bins) return;
    samples[t] = total[t % n_bins] - samples[t];
}

extern "C" {

int yawb_assign_patches(yawb_ctx *ctx, const double *xyz, int64_t n, const double *centers_xyz, int n_centers,
                        int32_t *out_ids) {
    YAWB_REQUIRE(ctx != nullptr, "yawb_assign_patches: ctx is NULL");
    YAWB_REQUIRE(n >= 0 && (n == 0 || (xyz && out_ids)), "yawb_assign_patches: NULL rows");
    YAWB_REQUIRE(n_centers >= 1 && centers_xyz, "yawb_assign_patches: at least one centre is required");
    if (n == 0) return 0;
    YAWB_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int64_t chunk = 1 << 24;  // rows per pass: bounded device footprint for any catalog size
    double *d_xyz = nullptr, *d_c = nullptr;
    int *d_out = nullptr;
    if (yawb_dalloc(ctx, (void **)&d_xyz, (size_t)std::min(n, chunk) * 3 * sizeof(double), st) ||
        yawb_dalloc(ctx, (void **)&d_c, (size_t)n_centers * 3 * sizeof(double), st) ||
        yawb_dalloc(ctx, (void **)&d_out, (size_t)std::min(n, chunk) * sizeof(int), st)) {
        yawb_dfree(ctx, d_xyz, st); yawb_dfree(ctx, d_c, st); yawb_dfree(ctx, d_out, st);
        return 1;
    }
    cudaError_t e = cudaMemcpyAsync(d_c, centers_xyz, (size_t)n_centers * 3 * sizeof(double), cudaMemcpyHostToDevice, st);
    for (int64_t o = 0; o < n && e == cudaSuccess; o += chunk) {
        const int64_t m = std::min(chunk, n - o);
        e = cudaMemcpyAsync(d_xyz, xyz + 3 * o, (size_t)m * 3 * sizeof(double), cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) break;
        k_assign_patches<<<(unsigned)((m + 255) / 256), 256, 3 * 1024 * sizeof(double), st>>>(d_xyz, m, d_c, n_centers, d_out);
        e = cudaMemcpyAsync(out_ids + o, d_out, (size_t)m * sizeof(int), cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    }
    if (e == cudaSuccess) e = cudaGetLastError();
    yawb_dfree(ctx, d_xyz, st); yawb_dfree(ctx, d_c, st); yawb_dfree(ctx, d_out, st);
    if (e != cudaSuccess) {
        yawb_set_error("yawb_assign_patches: %s", cudaGetErrorString(e));
        return 1;
    }
    return 0;
}

const char *yawb_last_error(void) { return g_err; }

int yawb_version(void) { return 104; }

int yawb_create(int device, yawb_ctx **out) {
    YAWB_REQUIRE(out != nullptr, "yawb_create: out is NULL");
    *out = nullptr;
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev == 0) {
        yawb_set_error("yawb_create: no CUDA device available (%s); this engine has no CPU fallback",
                       cudaGetErrorString(e));
        return 3;
    }
    YAWB_REQUIRE(device >= 0 && device < n_dev, "yawb_create: device %d out of range (0..%d)", device, n_dev - 1);
    YAWB_CUDA(cudaSetDevice(device));
    yawb_ctx *ctx = new (std::nothrow) yawb_ctx();
    YAWB_REQUIRE(ctx != nullptr, "out of host memory");
    ctx->device = device;
    cudaDeviceProp prop;
    YAWB_CUDA(cudaGetDeviceProperties(&prop, device));
    ctx->sms = prop.multiProcessorCount;
    YAWB_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    YAWB_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));

    YAWB_CUDA(cudaEventCreate(&ctx->ev0));
    YAWB_CUDA(cudaEventCreate(&ctx->ev1));
    YAWB_CUDA(cudaEventCreate(&ctx->ev_plan));
    YAWB_CUDA(cudaEventCreate(&ctx->ev_i0));
    YAWB_CUDA(cudaEventCreate(&ctx->ev_i1));
    YAWB_CUDA(cudaEventCreate(&ctx->ev_f0));
    YAWB_CUDA(cudaEventCreate(&ctx->ev_f1));
    YAWB_CUDA(cudaEventCreate(&ctx->ev_t0));
    YAWB_CUDA(cudaEventCreate(&ctx->ev_t1));
    YAWB_CUDA(cudaMalloc(&ctx->d_counters, 8 * sizeof(unsigned long long)));
    ctx->pin_size = 8u << 20;
    YAWB_CUDA(cudaHostAlloc((void **)&ctx->pin_base, ctx->pin_size, cudaHostAllocDefault));
    ctx->h2d_size = 32u << 20;
    YAWB_CUDA(cudaHostAlloc((void **)&ctx->h2d_base, ctx->h2d_size, cudaHostAllocMapped));
    *out = ctx;
    return 0;
}

int yawb_destroy(yawb_ctx *ctx) {
    if (!ctx) return 0;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->copy_stream);
    cudaStreamSynchronize(ctx->stream);
    cudaFree(ctx->d_counters);
    if (ctx->pin_base) cudaFreeHost(ctx->pin_base);
    if (ctx->h2d_base) cudaFreeHost(ctx->h2d_base);
    if (ctx->res_pin) cudaFreeHost(ctx->res_pin);
    cudaStreamDestroy(ctx->copy_stream);
    yawb_dcache_destroy(ctx);
    cudaEventDestroy(ctx->ev0);
    cudaEventDestroy(ctx->ev1);
    if (ctx->ev_plan) cudaEventDestroy(ctx->ev_plan);
    cudaEventDestroy(ctx->ev_i0);
    cudaEventDestroy(ctx->ev_i1);
    cudaEventDestroy(ctx->ev_f0);
    cudaEventDestroy(ctx->ev_f1);
    cudaEventDestroy(ctx->ev_t0);
    cudaEventDestroy(ctx->ev_t1);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
    return 0;
}

int yawb_device_sms(const yawb_ctx *ctx) { return ctx ? ctx->sms : 0; }

int yawb_catalog_footprint(int64_t n_rows, int n_patch, int n_bins, uint32_t what, int64_t *bytes) {
    YAWB_REQUIRE(bytes != nullptr, "yawb_catalog_footprint: bytes is NULL");
    YAWB_REQUIRE(n_rows >= 0 && n_patch >= 1 && n_bins >= 1, "yawb_catalog_footprint: n_rows >= 0, n_patch >= 1 and "
                 "n_bins >= 1 required (got %lld, %d, %d)", (long long)n_rows, n_patch, n_bins);
    YAWB_REQUIRE(what < 2 * YAWB_FOOT_NO_UPLOAD, "yawb_catalog_footprint: unknown flag bits 0x%x", what);
    *bytes = yawb_index_footprint(n_rows, n_patch, n_bins, what);
    return 0;
}

int yawb_count_footprint(int sms, int64_t n_items, int n_pairs, int n_bins, int n_edges, int n_blocks, int weighted,
                         int64_t *bytes) {
    YAWB_REQUIRE(bytes != nullptr, "yawb_count_footprint: bytes is NULL");
    YAWB_REQUIRE(sms >= 1 && n_items >= 0 && n_pairs >= 0 && n_bins >= 1 && n_edges >= 2 && n_blocks >= 1,
                 "yawb_count_footprint: invalid sizes");
    *bytes = yawb_count_workspace(sms, n_items, n_pairs, n_bins, n_edges, n_blocks, weighted != 0);
    return 0;
}

int yawb_memory_stats(yawb_ctx *ctx, int64_t *held, int64_t *peak, int64_t *device_free) {
    YAWB_REQUIRE(ctx != nullptr, "yawb_memory_stats: ctx is NULL");
    if (held) *held = (int64_t)yawb_dcache_bytes(ctx);
    if (peak) *peak = (int64_t)yawb_dcache_peak(ctx);
    if (device_free) {
        YAWB_CUDA(cudaSetDevice(ctx->device));
        size_t free_b = 0, total_b = 0;
        YAWB_CUDA(cudaMemGetInfo(&free_b, &total_b));
        *device_free = (int64_t)free_b;
    }
    return 0;
}

int yawb_memory_parked(yawb_ctx *ctx, int64_t *parked) {
    YAWB_REQUIRE(ctx != nullptr && parked != nullptr, "yawb_memory_parked: ctx or parked is NULL");
    *parked = (int64_t)yawb_dcache_parked(ctx);
    return 0;
}

int yawb_memory_reset_peak(yawb_ctx *ctx) {
    YAWB_REQUIRE(ctx != nullptr, "yawb_memory_reset_peak: ctx is NULL");
    yawb_dcache_reset_peak(ctx);
    return 0;
}

int yawb_memory_release(yawb_ctx *ctx) {
    YAWB_REQUIRE(ctx != nullptr, "yawb_memory_release: ctx is NULL");
    YAWB_CUDA(cudaSetDevice(ctx->device));
    yawb_dcache_release(ctx);
    return 0;
}

int yawb_sync(yawb_ctx *ctx) {
    YAWB_REQUIRE(ctx != nullptr, "yawb_sync: ctx is NULL");
    YAWB_CUDA(cudaSetDevice(ctx->device));
    YAWB_CUDA(cudaStreamSynchronize(ctx->copy_stream));
    YAWB_CUDA(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int yawb_timer_start(yawb_ctx *ctx) {
    YAWB_REQUIRE(ctx != nullptr, "yawb_timer_start: ctx is NULL");
    YAWB_CUDA(cudaSetDevice(ctx->device));
    YAWB_CUDA(cudaEventRecord(ctx->ev_t0, ctx->stream));
    return 0;
}

int yawb_timer_stop(yawb_ctx *ctx, double *ms) {
    YAWB_REQUIRE(ctx && ms, "yawb_timer_stop: NULL argument");
    YAWB_CUDA(cudaSetDevice(ctx->device));
    YAWB_CUDA(cudaEventRecord(ctx->ev_t1, ctx->stream));
    YAWB_CUDA(cudaEventSynchronize(ctx->ev_t1));
    float t = 0.f;
    YAWB_CUDA(cudaEventElapsedTime(&t, ctx->ev_t0, ctx->ev_t1));
    *ms = (double)t;
    return 0;
}

int yawb_host_alloc(void **ptr, uint64_t bytes) {
    YAWB_REQUIRE(ptr != nullptr, "yawb_host_alloc: ptr is NULL");
    YAWB_CUDA(cudaHostAlloc(ptr, std::max<uint64_t>(bytes, 1), cudaHostAllocDefault));
    return 0;
}

int yawb_host_free(void *ptr) {
    if (ptr) YAWB_CUDA(cudaFreeHost(ptr));
    return 0;
}

// keep: NULL (every patch) or one byte per patch; the rows of the kept patches travel, an unkept patch is empty
static int upload_common(yawb_ctx *ctx, const double *xyz, const double *w, const int32_t *zbin, const uint8_t *zbin8,
                         const double *zred, const double *edges, int closed_right, const int64_t *patch_off,
                         int n_patch, int n_bins, const uint8_t *keep, yawb_cat **out) {
    YAWB_REQUIRE(ctx && out && patch_off, "yawb_upload_catalog: NULL argument");
    *out = nullptr;
    YAWB_REQUIRE(n_patch >= 1 && n_patch <= 65535, "n_patch must be in 1..65535 (got %d)", n_patch);
    const bool binned = zbin != nullptr || zbin8 != nullptr || zred != nullptr;
    if (!binned) n_bins = 1;
    YAWB_REQUIRE(n_bins >= 1 && n_bins <= 4096, "n_bins must be in 1..4096 (got %d)", n_bins);
    YAWB_REQUIRE(!zbin8 || n_bins <= 254, "byte-sized z-bin ids need n_bins <= 254 (got %d)", n_bins);
    YAWB_REQUIRE(patch_off[0] == 0, "patch_off[0] must be 0");
    for (int p = 0; p < n_patch; ++p)
        YAWB_REQUIRE(patch_off[p + 1] >= patch_off[p], "patch_off must be non-decreasing");
    // rows on the device: the kept patches one after the other, each run of consecutive kept patches one copy
    std::vector<int64_t> dev_off(n_patch + 1, 0);
    std::vector<RowRun> runs;
    for (int p = 0; p < n_patch; ++p) {
        const int64_t rows = keep && !keep[p] ? 0 : patch_off[p + 1] - patch_off[p];
        dev_off[p + 1] = dev_off[p] + rows;
        if (rows == 0) continue;
        if (!runs.empty() && runs.back().src + runs.back().rows == patch_off[p])
            runs.back().rows += rows;
        else
            runs.push_back({patch_off[p], dev_off[p], rows});
    }
    const int64_t n = dev_off[n_patch];
    YAWB_REQUIRE(n < (1ll << 31) - 1024, "catalogs are limited to 2^31 rows (got %lld)", (long long)n);
    YAWB_REQUIRE(n == 0 || xyz != nullptr, "xyz is NULL");
    YAWB_CUDA(cudaSetDevice(ctx->device));

    yawb_cat *cat = new (std::nothrow) yawb_cat();
    YAWB_REQUIRE(cat != nullptr, "out of host memory");
    cat->ctx = ctx;
    cat->n_in = n;
    cat->n_patch = n_patch;
    cat->n_bins = n_bins;
    cat->binned = binned;
    cat->weighted = w != nullptr;
    cat->h_rows_per_patch.resize(n_patch);
    for (int p = 0; p < n_patch; ++p) cat->h_rows_per_patch[p] = dev_off[p + 1] - dev_off[p];
    if (zred) {
        cat->h_edges.assign(edges, edges + n_bins + 1);
        cat->closed_right = closed_right != 0;
    }
    cat->h_dev_off.swap(dev_off);  // the device copies its row offsets from here, asynchronously
    if (yawb_index_upload(ctx, cat, xyz, w, zbin8, zbin, zred, cat->h_dev_off.data(), runs)) {
        yawb_index_free(cat, true);
        delete cat;
        return 1;
    }
    *out = cat;
    return 0;
}

int yawb_upload_catalog(yawb_ctx *ctx, const double *xyz, const double *w, const int32_t *zbin,
                        const int64_t *patch_off, int n_patch, int n_bins, yawb_cat **out) {
    return upload_common(ctx, xyz, w, zbin, nullptr, nullptr, nullptr, 1, patch_off, n_patch, n_bins, nullptr, out);
}

int yawb_upload_catalog_u8(yawb_ctx *ctx, const double *xyz, const double *w, const uint8_t *zbin,
                           const int64_t *patch_off, int n_patch, int n_bins, yawb_cat **out) {
    return upload_common(ctx, xyz, w, nullptr, zbin, nullptr, nullptr, 1, patch_off, n_patch, n_bins, nullptr, out);
}

static int check_edges(const double *edges, int n_bins) {
    YAWB_REQUIRE(n_bins >= 1, "yawb_upload_catalog_z: n_bins must be >= 1 (got %d)", n_bins);
    for (int b = 0; b < n_bins; ++b)
        YAWB_REQUIRE(edges[b] < edges[b + 1], "yawb_upload_catalog_z: z-bin edges must increase (edge %d)", b);
    return 0;
}

int yawb_upload_catalog_z(yawb_ctx *ctx, const double *xyz, const double *w, const double *z, const double *edges,
                          int closed_right, const int64_t *patch_off, int n_patch, int n_bins, yawb_cat **out) {
    YAWB_REQUIRE(z && edges, "yawb_upload_catalog_z: redshifts or edges are NULL");
    if (int rc = check_edges(edges, n_bins)) return rc;
    return upload_common(ctx, xyz, w, nullptr, nullptr, z, edges, closed_right, patch_off, n_patch, n_bins, nullptr, out);
}

int yawb_upload_catalog_patches(yawb_ctx *ctx, const double *xyz, const double *w, const int32_t *zbin,
                                const uint8_t *zbin8, const double *z, const double *edges, int closed_right,
                                const int64_t *patch_off, int n_patch, int n_bins, const uint8_t *keep, yawb_cat **out) {
    YAWB_REQUIRE(keep != nullptr, "yawb_upload_catalog_patches: keep is NULL");
    YAWB_REQUIRE((zbin != nullptr) + (zbin8 != nullptr) + (z != nullptr) <= 1,
                 "yawb_upload_catalog_patches: pass at most one of zbin, zbin8 and z");
    if (z) {
        YAWB_REQUIRE(edges != nullptr, "yawb_upload_catalog_patches: z-bin edges are NULL");
        if (int rc = check_edges(edges, n_bins)) return rc;
    }
    return upload_common(ctx, xyz, w, zbin, zbin8, z, edges, closed_right, patch_off, n_patch, n_bins, keep, out);
}

int yawb_catalog_set_second_rows(yawb_cat *cat, const uint8_t *mask) {
    YAWB_REQUIRE(cat != nullptr, "yawb_catalog_set_second_rows: cat is NULL");
    YAWB_CUDA(cudaSetDevice(cat->ctx->device));
    return yawb_index_set_second_rows(cat, mask);
}

int yawb_catalog_set_labels(yawb_cat *cat, int n_labels) {
    YAWB_REQUIRE(cat != nullptr, "yawb_catalog_set_labels: cat is NULL");
    YAWB_REQUIRE(cat->binned, "yawb_catalog_set_labels: the catalog has no z-bin ids");
    YAWB_REQUIRE(cat->h_edges.empty(), "yawb_catalog_set_labels: a catalog binned on the device (yawb_upload_catalog_z) "
                                       "holds z-bins, not binned labels");
    YAWB_REQUIRE(n_labels >= 1 && cat->n_bins % n_labels == 0,
                 "yawb_catalog_set_labels: n_labels must be >= 1 and divide n_bins = %d (got %d)", cat->n_bins, n_labels);
    cat->n_labels = n_labels;
    return 0;
}

int yawb_free_catalog(yawb_cat *cat) {
    if (!cat) return 0;
    cudaSetDevice(cat->ctx->device);
    cudaStreamSynchronize(cat->ctx->copy_stream);
    cudaStreamSynchronize(cat->ctx->stream);
    yawb_index_free(cat, true);
    delete cat;
    return 0;
}

int yawb_build_index(yawb_cat *cat, int role, double *ms) {
    YAWB_REQUIRE(cat != nullptr, "yawb_build_index: cat is NULL");
    YAWB_REQUIRE(role == YAWB_ROLE_FIRST || role == YAWB_ROLE_SECOND, "unknown role %d", role);
    yawb_ctx *ctx = cat->ctx;
    YAWB_CUDA(cudaSetDevice(ctx->device));
    YAWB_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
    int rc = role == YAWB_ROLE_FIRST ? yawb_index_build_first(cat) : yawb_index_build_second(cat);
    if (rc) return rc;
    YAWB_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
    YAWB_CUDA(cudaEventSynchronize(ctx->ev1));
    float t = 0.f;
    YAWB_CUDA(cudaEventElapsedTime(&t, ctx->ev0, ctx->ev1));
    if (ms) *ms = (double)t;
    return 0;
}

int yawb_drop_index(yawb_cat *cat) {
    YAWB_REQUIRE(cat != nullptr, "yawb_drop_index: cat is NULL");
    YAWB_CUDA(cudaSetDevice(cat->ctx->device));
    if (yawb_cat_finalize(cat)) return 1;
    YAWB_CUDA(cudaStreamSynchronize(cat->ctx->stream));
    yawb_index_free(cat, false);
    return 0;
}

int yawb_catalog_info(const yawb_cat *cat, int64_t *n_rows, int64_t *device_bytes) {
    YAWB_REQUIRE(cat != nullptr, "yawb_catalog_info: cat is NULL");
    YAWB_CUDA(cudaSetDevice(cat->ctx->device));
    if (yawb_cat_finalize(const_cast<yawb_cat *>(cat))) return 1;
    if (n_rows) *n_rows = cat->n;
    if (device_bytes) *device_bytes = cat->device_bytes;
    return 0;
}

int yawb_sum_weights(const yawb_cat *cat, double *out) {
    YAWB_REQUIRE(cat && out, "yawb_sum_weights: NULL argument");
    YAWB_CUDA(cudaSetDevice(cat->ctx->device));
    if (yawb_cat_finalize(const_cast<yawb_cat *>(cat))) return 1;
    std::memcpy(out, cat->h_sumw.data(), cat->h_sumw.size() * sizeof(double));
    return 0;
}

int yawb_jackknife(yawb_ctx *ctx, const double *values, const int32_t *pair_i, const int32_t *pair_j, int n_pairs,
                   int n_patch, int n_bins, double *total, double *samples) {
    YAWB_REQUIRE(ctx && total && samples, "yawb_jackknife: NULL argument");
    YAWB_REQUIRE(n_pairs >= 0 && n_patch >= 1 && n_bins >= 1, "yawb_jackknife: bad sizes");
    YAWB_REQUIRE(n_pairs == 0 || (values && pair_i && pair_j), "yawb_jackknife: NULL input");
    for (int k = 0; k < n_pairs; ++k)
        YAWB_REQUIRE(pair_i[k] >= 0 && pair_i[k] < n_patch && pair_j[k] >= 0 && pair_j[k] < n_patch,
                     "yawb_jackknife: patch pair %d out of range", k);
    YAWB_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const size_t nv = (size_t)n_pairs * n_bins, ns = (size_t)n_patch * n_bins;
    double *d_v = nullptr, *d_out = nullptr;  // d_out = [total | samples]
    int *d_p = nullptr;
    auto cleanup = [&]() {
        for (void *p : {(void *)d_v, (void *)d_out, (void *)d_p})
            if (p) yawb_dfree(ctx, p, st);
    };
    if (yawb_dalloc(ctx, (void **)&d_v, std::max<size_t>(nv, 1) * sizeof(double), st) ||
        yawb_dalloc(ctx, (void **)&d_out, (n_bins + ns) * sizeof(double), st) ||
        yawb_dalloc(ctx, (void **)&d_p, std::max<size_t>(2 * (size_t)n_pairs, 1) * sizeof(int), st)) {
        cleanup();
        return 1;
    }
    cudaError_t e = cudaMemsetAsync(d_out, 0, (n_bins + ns) * sizeof(double), st);
    if (e == cudaSuccess && n_pairs > 0) {
        e = cudaMemcpyAsync(d_v, values, nv * sizeof(double), cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_p, pair_i, n_pairs * sizeof(int), cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_p + n_pairs, pair_j, n_pairs * sizeof(int), cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess)
            k_jackknife<<<(unsigned)((nv + 255) / 256), 256, 0, st>>>(d_v, d_p, d_p + n_pairs, n_pairs, n_bins, d_out, d_out + n_bins);
    }
    if (e == cudaSuccess) {
        k_jackknife_finish<<<(unsigned)((ns + 255) / 256), 256, 0, st>>>(d_out, n_patch, n_bins, d_out + n_bins);
        e = cudaMemcpyAsync(total, d_out, n_bins * sizeof(double), cudaMemcpyDeviceToHost, st);
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(samples, d_out + n_bins, ns * sizeof(double), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaGetLastError();
    cleanup();
    if (e != cudaSuccess) {
        yawb_set_error("yawb_jackknife: %s", cudaGetErrorString(e));
        return 1;
    }
    return 0;
}

int yawb_patch_metadata(const yawb_cat *cat, double *center_xyz, double *radius_chord, int64_t *num_records) {
    YAWB_REQUIRE(cat != nullptr, "yawb_patch_metadata: NULL catalog");
    YAWB_CUDA(cudaSetDevice(cat->ctx->device));
    if (yawb_cat_finalize(const_cast<yawb_cat *>(cat))) return 1;
    for (int p = 0; p < cat->n_patch; ++p) {
        const PatchFrame &f = cat->h_frames[p];
        if (center_xyz)
            for (int d = 0; d < 3; ++d) center_xyz[3 * p + d] = f.c[d];
        if (radius_chord) radius_chord[p] = f.radius;
        if (num_records) num_records[p] = cat->h_rows_per_patch[p];
    }
    return 0;
}

// Shared body of yawb_count (one first catalog) and yawb_count2 (two first catalogs counted against the same
// second catalog in one pass over a fused first-role index).
static int count_impl(yawb_ctx *ctx, yawb_cat *cat1, yawb_cat *cat1b, yawb_cat *cat2, yawb_cat *cat2b, const int32_t *pair_i,
                      const int32_t *pair_j, int n_pairs, const double *r2_edges, int n_edges, uint32_t flags,
                      double *const out_f64[4], int64_t *const out_i64[4], yawb_stats *stats) {
    YAWB_REQUIRE(ctx && cat1 && cat2, "yawb_count: NULL context or catalog");
    YAWB_REQUIRE(cat1->ctx == ctx && cat2->ctx == ctx && (!cat1b || cat1b->ctx == ctx), "catalogs belong to a different context");
    YAWB_REQUIRE(n_pairs >= 0, "n_pairs < 0");
    YAWB_REQUIRE(n_edges >= 2 && n_edges <= YAWB_MAX_EDGES, "n_edges must be in 2..%d (got %d)", YAWB_MAX_EDGES, n_edges);
    YAWB_REQUIRE(r2_edges != nullptr, "r2_edges is NULL");
    YAWB_REQUIRE((flags & ~(uint32_t)(YAWB_FLAG_EXACT_BRUTEFORCE | YAWB_FLAG_OUT_DEVICE | YAWB_FLAG_SECOND_LABELS)) == 0,
                 "unknown flag bits 0x%x (library version %d)", flags, yawb_version());
    const bool labels = (flags & YAWB_FLAG_SECOND_LABELS) != 0;
    YAWB_REQUIRE(!(labels && (flags & YAWB_FLAG_EXACT_BRUTEFORCE)),
                 "YAWB_FLAG_SECOND_LABELS is not supported by the exact cross-check (YAWB_FLAG_EXACT_BRUTEFORCE)");
    YAWB_REQUIRE(cat1->n_patch == cat2->n_patch, "catalogs have different numbers of patches (%d vs %d)",
                 cat1->n_patch, cat2->n_patch);
    // binned labels (yawb_catalog_set_labels): (a) both catalogs labelled alike, row (l, z) of cat2 meets (l, z) of
    // cat1; (b) cat1 binned without labels, (l, z) meets z.  Counts of label l go to output block l.
    const int L1 = cat1->n_labels, L2 = cat2->n_labels;
    if (L1 || L2 || (cat1b && cat1b->n_labels) || (cat2b && cat2b->n_labels)) {
        YAWB_REQUIRE(!cat1b && !cat2b, "catalogs with binned labels are not supported by yawb_count2 / yawb_count4");
        YAWB_REQUIRE(!labels, "catalogs with binned labels cannot be combined with YAWB_FLAG_SECOND_LABELS");
        YAWB_REQUIRE(!(flags & YAWB_FLAG_EXACT_BRUTEFORCE),
                     "catalogs with binned labels are not supported by the exact cross-check (YAWB_FLAG_EXACT_BRUTEFORCE)");
        YAWB_REQUIRE(L2, "a first catalog with binned labels needs a second catalog with the same labels; "
                         "swap the roles (pair counts are symmetric)");
        YAWB_REQUIRE(cat1->binned, "a second catalog with binned labels needs a binned first catalog");
        if (L1)
            YAWB_REQUIRE(L1 == L2 && cat1->n_bins == cat2->n_bins,
                         "catalogs with binned labels differ (%d labels x %d z-bins vs %d x %d)", L1, cat1->n_bins / L1, L2,
                         cat2->n_bins / L2);
        else
            YAWB_REQUIRE(cat1->n_bins == cat2->n_bins / L2, "z-bin counts differ (%d vs %d per label)", cat1->n_bins,
                         cat2->n_bins / L2);
    } else if (!labels) {
        YAWB_REQUIRE(!(cat2->binned && !cat1->binned), "a binned second catalog needs a binned first catalog");
        YAWB_REQUIRE(!cat2->binned || cat2->n_bins == cat1->n_bins, "z-bin counts differ (%d vs %d)", cat1->n_bins,
                     cat2->n_bins);
    }
    if (cat1b) {
        YAWB_REQUIRE(cat1b != cat1, "yawb_count2: the two first catalogs must differ");
        YAWB_REQUIRE(cat1b->n_patch == cat1->n_patch && cat1b->n_bins == cat1->n_bins && cat1b->binned == cat1->binned,
                     "yawb_count2: the two first catalogs need the same patches and z-bins");
        YAWB_REQUIRE(!(flags & YAWB_FLAG_EXACT_BRUTEFORCE), "yawb_count2: the exact cross-check counts one catalog at a time");
    }
    if (cat2b) {
        YAWB_REQUIRE(cat1b != nullptr, "yawb_count4 needs two first-role catalogs");
        YAWB_REQUIRE(cat2b != cat2 && cat2b->ctx == ctx, "yawb_count4: the two second catalogs must differ and belong to the context");
        YAWB_REQUIRE(cat2b->n_patch == cat2->n_patch, "yawb_count4: the two second catalogs need the same patches");
        YAWB_REQUIRE(labels || (cat2b->n_bins == cat2->n_bins && cat2b->binned == cat2->binned),
                     "yawb_count4: the two second catalogs need the same z-bins");
    }
    YAWB_REQUIRE(n_pairs == 0 || (pair_i && pair_j), "pair lists are NULL");
    const int n_types = cat1b ? 2 : 1;
    const int n_src = cat2b ? 2 : 1;  // second catalogs of the launch
    // output blocks per second catalog: its labels (binned labels, or YAWB_FLAG_SECOND_LABELS on a binned catalog), else one
    const int n_lab[2] = {L2 ? L2 : labels && cat2->binned ? cat2->n_bins : 1,
                          labels && cat2b && cat2b->binned ? cat2b->n_bins : 1};
    const int n_blocks = n_lab[0] + (cat2b ? n_lab[1] : 0);
    // B: z-bins of the thresholds and of every output block
    const int B = L2 ? cat2->n_bins / L2 : cat1->n_bins, P = cat1->n_patch, nsub = n_edges - 1;
    for (int k = 0; k < n_pairs; ++k)
        YAWB_REQUIRE(pair_i[k] >= 0 && pair_i[k] < P && pair_j[k] >= 0 && pair_j[k] < P,
                     "patch pair %d = (%d, %d) out of range", k, pair_i[k], pair_j[k]);
    for (int b = 0; b < B; ++b)
        for (int e = 0; e + 1 < n_edges; ++e)
            YAWB_REQUIRE(r2_edges[(size_t)b * n_edges + e] <= r2_edges[(size_t)b * n_edges + e + 1] &&
                             r2_edges[(size_t)b * n_edges + e] >= 0.0,
                         "r2_edges of z-bin %d are not sorted / non-negative", b);
    YAWB_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    yawb_stats s{};
    // Indexes are built lazily.  The first catalog is completed and indexed BEFORE the host waits for the
    // copies of the second one: with asynchronous uploads that work overlaps with the transfer.  Timed with
    // events that are only read after the final synchronisation of this call (waiting for copies excluded).
    if (yawb_cat_finalize(cat1)) return 1;
    if (cat1b && yawb_cat_finalize(cat1b)) return 1;
    float t_idx = 0.f;
    FIndex *fi = nullptr;
    bool first_built = false;
    {
        const bool need = cat1b ? true : cat1->findex == nullptr;
        if (need) YAWB_CUDA(cudaEventRecord(ctx->ev_f0, st));
        if (cat1b) {
            if (yawb_findex_get_fused(ctx, cat1, cat1b, &fi, &first_built)) return 1;
        } else {
            if (yawb_index_build_first(cat1)) return 1;
            fi = cat1->findex;
            first_built = need;
        }
        if (first_built) YAWB_CUDA(cudaEventRecord(ctx->ev_f1, st));  // read after the final synchronisation
    }
    if (yawb_cat_finalize(cat2)) return 1;
    if (cat2b && yawb_cat_finalize(cat2b)) return 1;
    const bool weighted = fi->weighted || cat2->weighted || (cat2b && cat2b->weighted);
    // The single-bin path of the count kernel (unweighted, one sub-bin) takes the tiles of a joint launch from ONE
    // index over the union of both second catalogs: a tile of YAWB_TILE rows covers half the sky, so every query box
    // shrinks (C3 on a B200: 1.89e10 -> 1.30e10 executed pair tests, count kernels 5.74 -> 4.71 ms).  The other paths keep per-catalog tiles: their per-pair
    // accumulators would not fit in the registers a split by catalog needs.
    const bool use_union = cat2b && !labels && !weighted && n_edges == 2 && !(flags & YAWB_FLAG_EXACT_BRUTEFORCE);
    const RIndex *tix[2] = {nullptr, nullptr};  // where the tiles come from (CountArgs::r2)
    bool second_built = false;
    {
        YAWB_CUDA(cudaEventRecord(ctx->ev_i0, st));
        if (use_union) {
            RIndex *u = nullptr;
            if (yawb_rindex_get_union(ctx, cat2, cat2b, &u, &second_built)) return 1;
            tix[0] = u;
        } else {
            second_built = !cat2->ri.built || (cat2b && !cat2b->ri.built);
            if (yawb_index_build_second(cat2)) return 1;
            if (cat2b && yawb_index_build_second(cat2b)) return 1;
            tix[0] = &cat2->ri;
            tix[1] = cat2b ? &cat2b->ri : nullptr;
        }
        if (second_built) YAWB_CUDA(cudaEventRecord(ctx->ev_i1, st));  // read after the final synchronisation
    }
    const int n_tix = tix[1] ? 2 : 1;
    const size_t n_out1 = (size_t)n_pairs * B * nsub;  // one (first catalog, output block) combination's results
    const size_t n_out = n_out1 * n_types * n_blocks;  // [second catalog, label][first catalog][pair][bin][sub-bin]

    // host-side preparation of thresholds and the item table
    std::vector<BinPar> binpar(B);
    // float copy of the edges, followed (sub-bin paths only) by the arithmetic bin lookup of every z-bin:
    // (scale, offset) with cell = lg2(d2) * scale + offset, and a table [n_cells] of the number of edges
    // strictly below the start of each cell (a lower bound of the answer that the kernel fixes up)
    const int lg_cells = n_edges > 2 ? YAWB_LG_CELLS_PER_EDGE * n_edges : 0;
    const size_t r2f_words = (size_t)B * n_edges + 2 * (size_t)B + ((size_t)B * lg_cells + 1) / 2;
    std::vector<float> r2f(r2f_words, 0.f);
    for (int b = 0; b < B; ++b) {
        const double lo = r2_edges[(size_t)b * n_edges], hi = r2_edges[(size_t)b * n_edges + nsub];
        BinPar &bp = binpar[b];
        bp.lo = lo;
        bp.hi = hi;
        bp.rmax = std::sqrt(hi) * (1.0 + 1e-9) + 1e-14;
        bp.mid = (float)(0.5 * (lo + hi));
        bp.h = (float)(0.5 * (hi - lo));
        bp.empty = !(hi > lo);
        bp.pad = 0;
        for (int e = 0; e < n_edges; ++e) r2f[(size_t)b * n_edges + e] = (float)r2_edges[(size_t)b * n_edges + e];
        if (lg_cells) {
            const double *ed = r2_edges + (size_t)b * n_edges;
            double first = hi;  // smallest positive edge
            for (int e = n_edges - 1; e >= 0; --e)
                if (ed[e] > 0.0) first = ed[e];
            const double L0 = first > 0.0 ? std::log2(first) : 0.0, L1 = hi > 0.0 ? std::log2(hi) : 0.0;
            const double scale = L1 > L0 ? (double)lg_cells / (L1 - L0) : 0.0;
            float *par = r2f.data() + (size_t)B * n_edges + 2 * (size_t)b;
            par[0] = (float)scale;
            // bias towards the lower cell (the table is a lower bound): twice the error of lg2.approx (2^-22
            // relative) and of the float arithmetic on a value of this size, plus a margin
            const double lmax = std::max(std::fabs(L0), std::fabs(L1)) + 1.0;
            const double bias = 1.0e-3 + 2.0 * scale * lmax * 6.0e-7;
            par[1] = (float)(-L0 * scale - bias);
            unsigned short *T = reinterpret_cast<unsigned short *>(r2f.data() + (size_t)B * n_edges + 2 * (size_t)B) +
                                (size_t)b * lg_cells;
            for (int c = 0; c < lg_cells; ++c) {
                const double start = scale > 0.0 ? std::exp2(L0 + (double)c / scale) * (1.0 - 1.0e-6) : 0.0;
                int below = 0;
                while (below < n_edges && ed[below] < start) ++below;
                if (c == 0) below = 0;  // everything at or below the first positive edge starts from scratch
                T[c] = (unsigned short)below;
            }
        }
    }
    double rmax_all = 0.0;
    for (int b = 0; b < B; ++b)
        if (!binpar[b].empty) rmax_all = std::max(rmax_all, binpar[b].rmax);
    // per second-role index: prefix of tiles per pair ((patch pair, tile) combinations = threads of the planner)
    std::vector<long long> item_base((size_t)n_tix * (n_pairs + 1), 0);
    long long flat_diag = 0, n_items_all = 0;
    for (int sc = 0; sc < n_tix; ++sc) {
        long long *base = item_base.data() + (size_t)sc * (n_pairs + 1);
        for (int k = 0; k < n_pairs; ++k) {
            const int q = pair_j[k];
            const long long nt = tix[sc]->h_ptile_off[q + 1] - tix[sc]->h_ptile_off[q];
            base[k + 1] = base[k] + nt;
            if (pair_i[k] == q) flat_diag += nt;
        }
        n_items_all += base[n_pairs];
    }
    for (int sc = 0; sc < n_src; ++sc) {
        const yawb_cat *c2 = sc ? cat2b : cat2;
        for (int k = 0; k < n_pairs; ++k) {
            const int p = pair_i[k], q = pair_j[k];
            if (L2) {  // binned labels: (l, z) of the second catalog against (l, z) or z of the first
                for (int l = 0; l < L2; ++l)
                    for (int b = 0; b < B; ++b)
                        s.pair_tests_naive += (uint64_t)(cat1->h_counts[((size_t)(L1 ? l * B : 0) + b) * P + p] *
                                                         c2->second_counts()[((size_t)l * B + b) * P + q]);
                continue;
            }
            long long n2_all = 0;  // a labelled catalog pairs the rows of every label with each z-bin
            const std::vector<long long> &cnt2 = c2->second_counts();
            for (int l = 0; l < c2->n_bins; ++l) n2_all += cnt2[(size_t)l * P + q];
            for (int b = 0; b < B; ++b) {
                long long n1 = cat1->h_counts[(size_t)b * P + p];
                if (cat1b) n1 += cat1b->h_counts[(size_t)b * P + p];
                const long long n2 = c2->binned && !labels ? cnt2[(size_t)b * P + q] : n2_all;
                s.pair_tests_naive += (uint64_t)(n1 * n2);
            }
        }
    }

    // the six small tables of a count travel as ONE block (one allocation, one pull kernel): pair lists,
    // item offsets, edges (double and float + bin lookup), per-bin parameters -- each 16-byte aligned
    const size_t np1 = std::max(n_pairs, 1);
    auto up16 = [](size_t b) { return (b + 15) & ~(size_t)15; };
    const size_t o_pi = 0, o_pj = o_pi + up16(np1 * sizeof(int)), o_base = o_pj + up16(np1 * sizeof(int)),
                 o_r2 = o_base + up16((size_t)n_tix * (np1 + 1) * sizeof(long long)),
                 o_r2f = o_r2 + up16((size_t)B * n_edges * sizeof(double)), o_bp = o_r2f + up16(r2f_words * sizeof(float)),
                 tab_bytes = o_bp + up16(B * sizeof(BinPar));
    std::vector<unsigned char> tab(tab_bytes, 0);
    if (n_pairs) {
        memcpy(tab.data() + o_pi, pair_i, n_pairs * sizeof(int));
        memcpy(tab.data() + o_pj, pair_j, n_pairs * sizeof(int));
    }
    memcpy(tab.data() + o_base, item_base.data(), (size_t)n_tix * (n_pairs + 1) * sizeof(long long));
    memcpy(tab.data() + o_r2, r2_edges, (size_t)B * n_edges * sizeof(double));
    memcpy(tab.data() + o_r2f, r2f.data(), r2f_words * sizeof(float));
    memcpy(tab.data() + o_bp, binpar.data(), B * sizeof(BinPar));

    unsigned char *d_tab = nullptr;
    double *d_w = nullptr;
    unsigned long long *d_cnt = nullptr;
    auto cleanup = [&]() {
        for (void *p : {(void *)d_tab, (void *)d_cnt, (void *)d_w})
            if (p) yawb_dfree(ctx, p, st);
    };
#define TRY(call)                                                                        \
    do {                                                                                 \
        cudaError_t err__ = (call);                                                      \
        if (err__ != cudaSuccess) {                                                      \
            yawb_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(err__)); \
            cleanup();                                                                   \
            return 1;                                                                    \
        }                                                                                \
    } while (0)
#define DALLOC(ptr, bytes)                                           \
    do {                                                             \
        if (yawb_dalloc(ctx, (void **)&(ptr), (bytes), st)) {        \
            cleanup();                                               \
            return 1;                                                \
        }                                                            \
    } while (0)
    DALLOC(d_tab, tab_bytes);
    DALLOC(d_cnt, std::max<size_t>(n_out, 1) * sizeof(unsigned long long));
    if (weighted) DALLOC(d_w, std::max<size_t>(n_out, 1) * sizeof(double));
    if (yawb_h2d_small(ctx, d_tab, tab.data(), tab_bytes)) {
        cleanup();
        return 1;
    }
    int *d_pi = (int *)(d_tab + o_pi), *d_pj = (int *)(d_tab + o_pj);
    long long *d_base = (long long *)(d_tab + o_base);
    double *d_r2 = (double *)(d_tab + o_r2);
    float *d_r2f = (float *)(d_tab + o_r2f);
    BinPar *d_bp = (BinPar *)(d_tab + o_bp);

    CountArgs a{};
    a.c1 = fi; a.c1_cat = cat1; a.c2 = cat2; a.c2b = cat2b;
    a.r2[0] = tix[0]; a.r2[1] = tix[1];
    a.d_pair_i = d_pi; a.d_pair_j = d_pj; a.d_pair_item_base = d_base;
    a.d_pair_item_base_b = tix[1] ? d_base + (n_pairs + 1) : nullptr;
    a.n_items = item_base[n_pairs];
    a.n_items_b = tix[1] ? item_base[(size_t)(n_pairs + 1) + n_pairs] : 0;
    a.labels = labels;
    a.blk_b = n_lab[0];
    a.lab_bins = L2 ? B : 0;
    a.lab_first = L1 > 0;
    // work-item lists: a patch with itself needs an item per tile (a few more where items are split), of the
    // tiles of neighbouring patches only the boundary strip survives; if a list turns out too small the
    // count is repeated with the exact sizes
    a.cap_heavy = 4 * flat_diag + 1024;
    a.cap_light = 2 * (n_items_all - flat_diag) + 1024;
    a.n_pairs = n_pairs; a.n_bins = B; a.n_edges = n_edges;
    a.d_r2 = d_r2; a.d_r2f = d_r2f; a.d_binpar = d_bp; a.rmax_all = rmax_all;
    a.d_out_cnt = d_cnt; a.d_out_w = d_w; a.weighted = weighted;

    int launches = 0;
    unsigned long long h_counters[8] = {0};
    const bool to_device = (flags & YAWB_FLAG_OUT_DEVICE) != 0;
    // caller array t = (second catalog s, first catalog) holds [label][pair][bin][sub-bin]; on the device, block
    // (s, label) of first catalog t % n_types sits at this multiple of n_out1
    auto out_block = [&](int t, int l) -> size_t {
        return (size_t)((t / n_types ? n_lab[0] : 0) + l) * n_types + (size_t)(t % n_types);
    };
    // Host results land in page-locked memory of the context first (counters, counts, sums: one copy each, truly
    // asynchronous) and are handed to the caller's -- usually pageable -- arrays after the one synchronisation of
    // the call; a cudaMemcpyAsync into pageable memory is staged by the driver, one blocking round trip per array.
    // Unweighted sums are the counts as doubles: converted on the host.
    unsigned char *pin = nullptr;
    const size_t pin_cnt = 64, pin_w = pin_cnt + std::max<size_t>(n_out, 1) * sizeof(unsigned long long);
    if (!to_device) {
        const size_t need = pin_w + (weighted ? std::max<size_t>(n_out, 1) * sizeof(double) : 0);
        if (ctx->res_pin_size < need) {
            if (ctx->res_pin) cudaFreeHost(ctx->res_pin);
            ctx->res_pin = nullptr;
            ctx->res_pin_size = 0;
            TRY(cudaHostAlloc((void **)&ctx->res_pin, need + need / 2, cudaHostAllocDefault));
            ctx->res_pin_size = need + need / 2;
        }
        pin = ctx->res_pin;
    }
    for (int attempt = 0;; ++attempt) {
        TRY(cudaMemsetAsync(d_cnt, 0, std::max<size_t>(n_out, 1) * sizeof(unsigned long long), st));
        if (weighted) TRY(cudaMemsetAsync(d_w, 0, std::max<size_t>(n_out, 1) * sizeof(double), st));
        TRY(cudaMemsetAsync(ctx->d_counters, 0, 8 * sizeof(unsigned long long), st));
        ctx->ev_plan_set = false;
        TRY(cudaEventRecord(ctx->ev0, st));
        int rc = (flags & YAWB_FLAG_EXACT_BRUTEFORCE) ? yawb_launch_count_exact(ctx, a, &launches)
                                                      : yawb_launch_count_fast(ctx, a, &launches);
        if (rc) { cleanup(); return rc; }
        TRY(cudaEventRecord(ctx->ev1, st));
        // the results travel right behind the counters (ONE synchronisation per call); should a work-item list have
        // been too small -- the host only learns that now -- the count is repeated with the exact sizes
        if (to_device) {
            TRY(cudaMemcpyAsync(h_counters, ctx->d_counters, sizeof(h_counters), cudaMemcpyDeviceToHost, st));
            for (int t = 0; t < n_types * n_src && n_out1; ++t)
                for (int l = 0; l < n_lab[t / n_types]; ++l) {
                    const size_t src = out_block(t, l) * n_out1, dst = (size_t)l * n_out1;
                    if (out_i64[t]) TRY(cudaMemcpyAsync(out_i64[t] + dst, d_cnt + src, n_out1 * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
                    if (out_f64[t]) {
                        if (weighted) {
                            TRY(cudaMemcpyAsync(out_f64[t] + dst, d_w + src, n_out1 * sizeof(double), cudaMemcpyDeviceToDevice, st));
                        } else {
                            k_u64_to_f64<<<(unsigned)((n_out1 + 255) / 256), 256, 0, st>>>(d_cnt + src, out_f64[t] + dst, (long long)n_out1);
                            launches += 1;
                        }
                    }
                }
            TRY(cudaStreamSynchronize(st));
        } else {
            TRY(cudaMemcpyAsync(pin, ctx->d_counters, sizeof(h_counters), cudaMemcpyDeviceToHost, st));
            if (n_out) TRY(cudaMemcpyAsync(pin + pin_cnt, d_cnt, n_out * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
            if (n_out && weighted) TRY(cudaMemcpyAsync(pin + pin_w, d_w, n_out * sizeof(double), cudaMemcpyDeviceToHost, st));
            TRY(cudaStreamSynchronize(st));
            memcpy(h_counters, pin, sizeof(h_counters));
        }
        if (!h_counters[6]) break;
        if (attempt > 0) {
            yawb_set_error("work-item lists overflowed twice (%llu + %llu items)", h_counters[4], h_counters[5]);
            cleanup();
            return 2;
        }
        a.cap_heavy = (long long)h_counters[4] + 1024;
        a.cap_light = (long long)h_counters[5] + 1024;
    }
    if (!to_device) {
        const unsigned long long *h_cnt = reinterpret_cast<const unsigned long long *>(pin + pin_cnt);
        const double *h_w = reinterpret_cast<const double *>(pin + pin_w);
        for (int t = 0; t < n_types * n_src && n_out1; ++t)
            for (int l = 0; l < n_lab[t / n_types]; ++l) {
                const size_t src = out_block(t, l) * n_out1, dst = (size_t)l * n_out1;
                if (out_i64[t]) memcpy(out_i64[t] + dst, h_cnt + src, n_out1 * sizeof(int64_t));
                if (out_f64[t]) {
                    if (weighted) {
                        memcpy(out_f64[t] + dst, h_w + src, n_out1 * sizeof(double));
                    } else {
                        for (size_t k = 0; k < n_out1; ++k) out_f64[t][dst + k] = (double)h_cnt[src + k];
                    }
                }
            }
    }
    TRY(cudaGetLastError());
    float t_k = 0.f;
    TRY(cudaEventElapsedTime(&t_k, ctx->ev0, ctx->ev1));
    float t_plan = 0.f;
    if (ctx->ev_plan_set) TRY(cudaEventElapsedTime(&t_plan, ctx->ev0, ctx->ev_plan));
    if (second_built) {
        float t = 0.f;
        TRY(cudaEventElapsedTime(&t, ctx->ev_i0, ctx->ev_i1));
        t_idx += t;
    }
    if (first_built) {
        float t = 0.f;
        TRY(cudaEventElapsedTime(&t, ctx->ev_f0, ctx->ev_f1));
        t_idx += t;
    }
    s.index_ms = t_idx;
#undef TRY
#undef DALLOC
    cleanup();
    s.kernel_ms = t_k;
    s.plan_ms = t_plan;
    s.pair_tests = h_counters[1];
    s.rechecks = h_counters[2];
    s.work_items = (flags & YAWB_FLAG_EXACT_BRUTEFORCE) ? (uint64_t)n_pairs * B : h_counters[4] + h_counters[5];
    s.launches = (uint64_t)launches;
    if (stats) *stats = s;
    return 0;
}

int yawb_count(yawb_ctx *ctx, yawb_cat *cat1, yawb_cat *cat2, const int32_t *pair_i, const int32_t *pair_j,
               int n_pairs, const double *r2_edges, int n_edges, uint32_t flags, double *out_f64,
               int64_t *out_i64, yawb_stats *stats) {
    double *const of[4] = {out_f64, nullptr, nullptr, nullptr};
    int64_t *const oi[4] = {out_i64, nullptr, nullptr, nullptr};
    return count_impl(ctx, cat1, nullptr, cat2, nullptr, pair_i, pair_j, n_pairs, r2_edges, n_edges, flags, of, oi, stats);
}

int yawb_count2(yawb_ctx *ctx, yawb_cat *cat1a, yawb_cat *cat1b, yawb_cat *cat2, const int32_t *pair_i,
                const int32_t *pair_j, int n_pairs, const double *r2_edges, int n_edges, uint32_t flags,
                double *out_f64_a, int64_t *out_i64_a, double *out_f64_b, int64_t *out_i64_b, yawb_stats *stats) {
    YAWB_REQUIRE(cat1b != nullptr, "yawb_count2: the second first-role catalog is NULL");
    double *const of[4] = {out_f64_a, out_f64_b, nullptr, nullptr};
    int64_t *const oi[4] = {out_i64_a, out_i64_b, nullptr, nullptr};
    return count_impl(ctx, cat1a, cat1b, cat2, nullptr, pair_i, pair_j, n_pairs, r2_edges, n_edges, flags, of, oi, stats);
}

int yawb_count4(yawb_ctx *ctx, yawb_cat *cat1a, yawb_cat *cat1b, yawb_cat *cat2a, yawb_cat *cat2b, const int32_t *pair_i,
                const int32_t *pair_j, int n_pairs, const double *r2_edges, int n_edges, uint32_t flags,
                double *const out_f64[4], int64_t *const out_i64[4], yawb_stats *stats) {
    YAWB_REQUIRE(cat1b != nullptr && cat2b != nullptr, "yawb_count4: a catalog is NULL");
    YAWB_REQUIRE(out_f64 != nullptr && out_i64 != nullptr, "yawb_count4: the output pointer tables are NULL (their entries may be)");
    return count_impl(ctx, cat1a, cat1b, cat2a, cat2b, pair_i, pair_j, n_pairs, r2_edges, n_edges, flags, out_f64, out_i64, stats);
}

}  // extern "C"
