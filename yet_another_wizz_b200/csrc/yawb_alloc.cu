// Device memory for catalogs, indexes and per-call scratch: a small caching allocator on top of cudaMalloc.
//
// Why not cudaMallocAsync: growing the stream-ordered pool costs ~100-270 ms per GB on this driver (B200,
// 580.x: 40 x 100 MB first use 376 ms, one 8 GB block 2.2 s), against ~5 ms per GB for cudaMalloc.  That
// made the first pair count of a process 0.5 s (C3) to several seconds (1e8-row catalogs) slower than a
// warm one, and mixed block sizes kept the pool growing between steps.  Here a block is cudaMalloc'ed
// once and then recycled:
//   * free(ptr, stream) records an event on `stream` and parks the block in a size-ordered free list;
//   * alloc(bytes, stream) takes the smallest parked block of at least that size (and at most 25 % + 1 MB
//     larger) that is safe to touch: parked by the same stream (stream order) or with a completed event.
//     It never makes a stream wait for another stream; if nothing fits it calls cudaMalloc, and when the
//     device is full it returns every parked block to the driver and tries once more.
// One context is used by one host thread at a time (include/yawb.h), so there is no locking.
#include <algorithm>
#include <map>
#include <unordered_map>

#include "yawb_internal.cuh"

struct DevBlock {
    void *ptr;
    size_t size;
    cudaStream_t stream;  // stream of the last free
    cudaEvent_t ev;       // recorded on `stream` at the last free
};

struct yawb_devcache {
    std::multimap<size_t, DevBlock> parked;
    std::unordered_map<void *, DevBlock> live;
    size_t bytes_total = 0;  // every block cudaMalloc'ed and not yet returned, parked ones included
    size_t bytes_peak = 0;   // high-water mark of bytes_total since the last yawb_dcache_reset_peak
};

static size_t round_size(size_t bytes) {
    if (bytes < 512) return 512;
    if (bytes < (1u << 20)) return (bytes + 511) & ~(size_t)511;
    return (bytes + (1u << 20) - 1) & ~(size_t)((1u << 20) - 1);
}

static void release_parked(yawb_devcache *c) {
    for (auto &kv : c->parked) {
        cudaEventSynchronize(kv.second.ev);
        cudaFree(kv.second.ptr);
        cudaEventDestroy(kv.second.ev);
        c->bytes_total -= kv.second.size;
    }
    c->parked.clear();
}

int yawb_dalloc(yawb_ctx *ctx, void **out, size_t bytes, cudaStream_t st) {
    *out = nullptr;
    if (!ctx->cache) ctx->cache = new yawb_devcache();
    yawb_devcache *c = ctx->cache;
    const size_t size = round_size(bytes);
    const size_t limit = size + size / 4 + (1u << 20);
    for (auto it = c->parked.lower_bound(size); it != c->parked.end() && it->first <= limit; ++it) {
        DevBlock &b = it->second;
        bool usable = b.stream == st;
        if (!usable) {
            usable = cudaEventQuery(b.ev) == cudaSuccess;
            if (!usable) cudaGetLastError();  // cudaEventQuery leaves cudaErrorNotReady behind: clear it right away
        }
        if (usable) {
            DevBlock blk = b;
            c->parked.erase(it);
            c->live.emplace(blk.ptr, blk);
            *out = blk.ptr;
            return 0;
        }
    }
    DevBlock blk{nullptr, size, st, nullptr};
    cudaError_t e = cudaMalloc(&blk.ptr, size);
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        release_parked(c);
        e = cudaMalloc(&blk.ptr, size);
    }
    if (e != cudaSuccess) {
        yawb_set_error("out of device memory: %zu bytes requested, %zu bytes held (%s)", size, c->bytes_total,
                       cudaGetErrorString(e));
        cudaGetLastError();
        return 1;
    }
    YAWB_CUDA(cudaEventCreateWithFlags(&blk.ev, cudaEventDisableTiming));
    c->bytes_total += size;
    c->bytes_peak = std::max(c->bytes_peak, c->bytes_total);
    c->live.emplace(blk.ptr, blk);
    *out = blk.ptr;
    return 0;
}

void yawb_dfree(yawb_ctx *ctx, void *ptr, cudaStream_t st) {
    if (!ptr || !ctx->cache) return;
    yawb_devcache *c = ctx->cache;
    auto it = c->live.find(ptr);
    if (it == c->live.end()) return;  // not ours
    DevBlock blk = it->second;
    c->live.erase(it);
    blk.stream = st;
    cudaEventRecord(blk.ev, st);
    c->parked.emplace(blk.size, blk);
}

void yawb_dcache_destroy(yawb_ctx *ctx) {
    yawb_devcache *c = ctx->cache;
    if (!c) return;
    release_parked(c);
    for (auto &kv : c->live) {
        cudaFree(kv.second.ptr);
        cudaEventDestroy(kv.second.ev);
    }
    delete c;
    ctx->cache = nullptr;
}

size_t yawb_dcache_bytes(const yawb_ctx *ctx) { return ctx->cache ? ctx->cache->bytes_total : 0; }

size_t yawb_dcache_parked(const yawb_ctx *ctx) {
    size_t n = 0;
    if (ctx->cache)
        for (const auto &kv : ctx->cache->parked) n += kv.second.size;
    return n;
}

size_t yawb_dcache_peak(const yawb_ctx *ctx) { return ctx->cache ? ctx->cache->bytes_peak : 0; }

void yawb_dcache_reset_peak(yawb_ctx *ctx) {
    if (ctx->cache) ctx->cache->bytes_peak = ctx->cache->bytes_total;
}

void yawb_dcache_release(yawb_ctx *ctx) {
    if (ctx->cache) release_parked(ctx->cache);
}

size_t yawb_dcache_round(size_t bytes) { return round_size(bytes); }
