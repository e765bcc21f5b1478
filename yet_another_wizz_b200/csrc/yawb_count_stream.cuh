// The production pair-count kernel k_count_stream (included by yawb_count.cu after the shared device
// functions and the layout of a warp's shared memory, StreamSmem): a software-pipelined stream of work items per warp.
//
// A work item (written by the planner k_plan) is a register tile of the second catalog against some z-bins of
// one linked patch of the first catalog, with the tile's bounding box already expressed in the frame of that
// patch.  Every warp owns a block of shared memory and runs, per "tick", three things whose memory latencies
// are all hidden behind the pair tests of the previous tick (asynchronous copies, cp.async):
//
//   convert   the raw chunk that has landed (<= LB fixed-point rows of the first catalog, 16 bytes each) is
//             re-expressed relative to the tile's origin, rounded ONCE to float, culled against the z-bin's
//             query box and staged as the broadcast operands of the packed FP32 pair test;
//   produce   the next raw chunk is requested: one 16-byte asynchronous copy per candidate row, addressed
//             through the run table of the item (one contiguous run of rows per (z-bin, cell row)).  When an
//             item is exhausted the run table of the next one is built from cell boundaries that were
//             requested one tick earlier, the cell boundaries of the item after that are requested, the record
//             of the one after that is copied, and the index of a fourth is taken from the global counter;
//   test      the staged list against the 8 rows per lane of the tile, one pass per z-bin segment.
//
// Nothing in the loop waits for a load it issued in the same tick, so a handful of warps per scheduler keep
// the FP32 pipe busy (16 warps per SM at 128 registers per thread; measured against 12 warps at 160 registers and
// chunks of 192 rows: C3 count kernels 6.37 -> 6.16 ms).
#pragma once

constexpr int STREAM_WARPS = 4;  // warps per CTA
constexpr int STREAM_CTAS = 4;   // CTAs per SM the kernel is compiled for (128 registers)

__host__ __device__ inline size_t up16(size_t b) { return (b + 15) & ~(size_t)15; }

// Walks the layout of a warp's block (StreamSmem); with `base == nullptr` only the size is of interest.
__host__ __device__ inline size_t stream_carve(StreamSmem *S, unsigned char *base, bool weighted, bool multi, int n_bins,
                                               int nsub, int n_types, int n_sec, bool acc_global) {
    size_t o = 0;
    auto take = [&](size_t bytes) {
        unsigned char *p = base + o;
        o += up16(bytes);
        return p;
    };
    const size_t nacc = acc_global ? 0 : (size_t)n_sec * n_types * n_bins * nsub;
    unsigned char *p;
    p = take(NSLOT * sizeof(Item)); if (S) S->items = (Item *)p;
    p = take(NSLOT * sizeof(ItemAux)); if (S) S->aux = (ItemAux *)p;
    p = take(n_bins * sizeof(int)); if (S) S->bin_iv0 = (int *)p;
    p = take(n_bins * sizeof(int)); if (S) S->bin_iu = (int *)p;
    p = take((n_bins + 1) * sizeof(int)); if (S) S->cstart = (int *)p;
    p = take(CCAP * sizeof(int2)); if (S) S->cs = (int2 *)p;
    p = take(CCAP * sizeof(unsigned short)); if (S) S->csbin = (unsigned short *)p;
    p = take(CCAP * sizeof(int2)); if (S) S->run = (int2 *)p;
    p = take(CCAP * sizeof(unsigned short)); if (S) S->cbin = (unsigned short *)p;
    p = take(LB * sizeof(SRec)); if (S) S->raw = (SRec *)p;
    p = take(LB * sizeof(unsigned short)); if (S) S->rawbin = (unsigned short *)p;
    p = take(weighted ? LB * sizeof(double) : 0); if (S) S->rawlw = weighted ? (double *)p : nullptr;
    p = take(LB * sizeof(Cand)); if (S) S->list = (Cand *)p;
    p = take(LB * sizeof(int)); if (S) S->lidx = (int *)p;
    p = take(LB * sizeof(unsigned short)); if (S) S->lbin = (unsigned short *)p;
    p = take(weighted ? LB * sizeof(double) : 0); if (S) S->lw = weighted ? (double *)p : nullptr;
    p = take((size_t)n_types * n_bins * sizeof(SegDesc)); if (S) S->seg = (SegDesc *)p;
    p = take(n_bins * sizeof(float4)); if (S) S->binrec = (float4 *)p;
    p = take(n_bins * sizeof(float2)); if (S) S->binthr = (float2 *)p;
    p = take(nacc * sizeof(unsigned long long)); if (S) S->acc = (unsigned long long *)p;
    p = take(weighted ? nacc * sizeof(double) : 0); if (S) S->accw = weighted ? (double *)p : nullptr;
    p = take(multi ? nsub * sizeof(unsigned) : 0); if (S) S->hist = multi ? (unsigned *)p : nullptr;
    p = take(multi && weighted ? nsub * sizeof(double) : 0); if (S) S->histw = (multi && weighted) ? (double *)p : nullptr;
    // (at least 128 words: the general sub-bin path keeps its queue of in-range tests here, phase2_multi_queue)
    p = take(multi ? ((size_t)n_bins * CUM_EDGES > 128 ? (size_t)n_bins * CUM_EDGES : 128) * sizeof(float) : 0); if (S) S->cum = multi ? (float *)p : nullptr;
    p = take(multi ? CUM_EDGES * sizeof(unsigned) : 0); if (S) S->cumtot = multi ? (unsigned *)p : nullptr;
    return o;
}

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem));
}
__device__ __forceinline__ void cp_async8(void *smem, const void *gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem));
}
__device__ __forceinline__ void cp_async4(void *smem, const void *gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

__device__ __forceinline__ const Item *item_ptr(const FastParams &P, long long idx, long long n_heavy) {
    return idx < n_heavy ? P.items_heavy + idx : P.items_light + (idx - n_heavy);
}

// ---- fetch: the record of work item `idx` into a slot (asynchronous), or the end marker -------------------
__device__ __forceinline__ void stream_fetch(const FastParams &P, const StreamSmem &S, int slot, long long idx,
                                             long long n_heavy, long long n_live, int lane) {
    if (idx >= n_live) {
        if (lane == 0) S.aux[slot].end = 1;
        return;
    }
    if (lane == 0) S.aux[slot].end = 0;
    if (lane < (int)(sizeof(Item) / 16))
        cp_async16(reinterpret_cast<uint4 *>(&S.items[slot]) + lane, reinterpret_cast<const uint4 *>(item_ptr(P, idx, n_heavy)) + lane);
}

// ---- plan: cell rows of the query per z-bin, then request the cell boundaries of every run ----------------
__device__ __forceinline__ void stream_plan(const FastParams &P, const StreamSmem &S, int slot, int lane) {
    ItemAux &ax = S.aux[slot];
    if (ax.end) return;
    const Item &it = S.items[slot];
    const SGrid G = P.sgrid[it.p1];
    const double ulo = it.lo[0], uhi = it.hi[0], vlo = it.lo[1], vhi = it.hi[1];
    int carry = 0;
    for (int b0 = it.b_lo; b0 < it.b_hi; b0 += 32) {
        const int b = b0 + lane;
        int nrows = 0;
        if (b < it.b_hi) {
            const BinPar bp = P.binpar[b];
            const BinRows r = bin_rows(G, ulo, uhi, vlo, vhi, bp, it.row_lo, it.row_hi);
            nrows = r.nrows;
            S.bin_iv0[b] = r.iv0;
            S.bin_iu[b] = r.iu0 | (r.iu1 << 16);
        }
        int incl = nrows;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += v;
        }
        if (b < it.b_hi) S.cstart[b + 1] = carry + incl;
        carry += __shfl_sync(FULL, incl, 31);
    }
    const int n_combo = min(carry, CCAP);  // the planner's split guarantees carry <= CCAP
    if (lane == 0) {
        S.cstart[it.b_lo] = 0;
        // origin of the staged frame: the lattice point nearest to the centre of the tile box (clamped to the
        // lattice of the patch, so that differences of lattice coordinates never overflow 32 bits)
        const double c[3] = {0.5 * (it.lo[0] + it.hi[0]), 0.5 * (it.lo[1] + it.hi[1]), 0.5 * (it.lo[2] + it.hi[2])};
        const double org[3] = {G.u0, G.v0, G.t0};
        double o[3];
        float e[3];
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            const double k = fmin(fmax(rint((c[d] - org[d]) * G.qscale), 0.0), 2147483647.0);
            ax.ko[d] = (int)k;
            o[d] = org[d] + k * G.qinv;
            const float h = (float)fmax(it.hi[d] - o[d], o[d] - it.lo[d]);
            e[d] = h * 1.000001f + 1.0e-30f;
        }
        // tile frame: the sphere is centred at (0, 0, -1) in the frame of p1
        double n[3] = {c[0], c[1], c[2] + 1.0};
        const double nn = 1.0 / sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
        n[0] *= nn; n[1] *= nn; n[2] *= nn;
        // an axis of the frame of p1 made orthogonal to n: u inside a patch, v for a direction near the u axis
        // (search radii of tens of degrees)
        double t1[3] = {1.0 - n[0] * n[0], -n[0] * n[1], -n[0] * n[2]};
        if (fabs(n[0]) > 0.7) { t1[0] = -n[1] * n[0]; t1[1] = 1.0 - n[1] * n[1]; t1[2] = -n[1] * n[2]; }
        const double tn = 1.0 / sqrt(t1[0] * t1[0] + t1[1] * t1[1] + t1[2] * t1[2]);
        t1[0] *= tn; t1[1] *= tn; t1[2] *= tn;
        const double t2[3] = {n[1] * t1[2] - n[2] * t1[1], n[2] * t1[0] - n[0] * t1[2], n[0] * t1[1] - n[1] * t1[0]};
        double g2 = 0.0;
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            ax.R[d] = t1[d]; ax.R[3 + d] = t2[d]; ax.R[6 + d] = n[d];
            const double O = n[d] - (d == 2 ? 1.0 : 0.0);
            ax.O[d] = O;
            ax.dq[d] = o[d] - O;
            g2 += (o[d] - O) * (o[d] - O);
        }
        ax.g = (float)sqrt(g2) * 1.000001f + 1.0e-30f;
        ax.eu = e[0]; ax.ev = e[1]; ax.et = e[2];
        ax.qinv = (float)G.qinv;
        ax.n_combo = n_combo;
    }
    __syncwarp();
    const int b_lo = it.b_lo, b_hi = it.b_hi, b_off = it.b_off;
    for (int k = lane; k < n_combo; k += 32) {
        int lo = b_lo, hi = b_hi;  // last z-bin with cstart[b] <= k
        while (hi - lo > 1) {
            const int m = (lo + hi) >> 1;
            if (S.cstart[m] <= k) lo = m; else hi = m;
        }
        const int b = lo;
        const int iv = S.bin_iv0[b] + (k - S.cstart[b]);
        const int iu = S.bin_iu[b];
        // the first catalog's cells of z-bin b of the item's label (binned labels: id b + b_off); every table of
        // the warp stays indexed by the z-bin b
        const long long row = G.cell_base + ((long long)(b + b_off) * G.gv + iv) * G.gu;
        cp_async4(&S.cs[k].x, P.cell_start + row + (iu & 0xffff));
        cp_async4(&S.cs[k].y, P.cell_start + row + (iu >> 16) + 1);
        S.csbin[k] = (unsigned short)b;
    }
    // the rows of the tile: towards L2 now, into registers when the item is consumed
    const double *const rxs = it.src ? P.rx2 : P.rx;
    for (int k = lane * 4; k < it.count; k += 128)  // 32-byte row records: one 128-byte line per four rows
        prefetch_l2(rxs + (size_t)YAWB_RSTRIDE * (it.start + k));
}

// ---- run table of the item whose cell boundaries have landed; returns the number of candidate rows -------
__device__ __forceinline__ int stream_runs(const StreamSmem &S, int n_combo, int lane) {
    int running = 0;
    for (int k0 = 0; k0 < n_combo; k0 += 32) {
        const int k = k0 + lane;
        int cnt = 0, s0 = 0;
        if (k < n_combo) {
            const int2 c = S.cs[k];
            s0 = c.x;
            cnt = c.y - c.x;
        }
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += v;
        }
        if (k < n_combo) {
            S.run[k] = make_int2(running + incl, s0 - (running + incl - cnt));  // row of flat position t: .y + t
            S.cbin[k] = S.csbin[k];
        }
        running += __shfl_sync(FULL, incl, 31);
    }
    __syncwarp();
    return running;
}

// ---- request the rows [t0, t0 + cnt) of the item's flat candidate range: one lane per row ----------------
// Every lane walks the run table forwards (its flat positions grow by 32 per round, a run holds a handful of
// rows), starting from a binary search.
template <bool WEIGHTED>
__device__ __forceinline__ void stream_issue(const FastParams &P, const StreamSmem &S, int n_combo, int t0, int cnt,
                                             int lane) {
    if (cnt <= 0) return;
    int cur;
    {
        const int t = t0 + min(lane, cnt - 1);
        int lo = 0, hi = n_combo - 1;  // first run whose inclusive prefix exceeds t
        while (lo < hi) {
            const int m = (lo + hi) >> 1;
            if (S.run[m].x > t) hi = m; else lo = m + 1;
        }
        cur = lo;
    }
    int2 r = S.run[cur];
    for (int base = 0; base < cnt; base += 32) {
        const int i = base + lane;
        if (i < cnt) {
            const int t = t0 + i;
            while (t >= r.x) r = S.run[++cur];  // empty runs are skipped as well
            const int src = r.y + t;
            cp_async16(&S.raw[i], P.rec + src);
            if (WEIGHTED) {
                if (P.sw) cp_async8(&S.rawlw[i], P.sw + src);
                else S.rawlw[i] = 1.0;  // unweighted first catalog against a weighted second one
            }
            S.rawbin[i] = S.cbin[cur];
        }
    }
}

// ---- per-item tables of the consumer: half extents of the query box, FP32 error bound, thresholds --------
template <CountPath PATH>
__device__ __forceinline__ void stream_begin(const FastParams &P, const StreamSmem &S, int slot, int lane) {
    const Item &it = S.items[slot];
    const ItemAux &ax = S.aux[slot];
    const float eu = ax.eu, ev = ax.ev, et = ax.et;
    // coordinate error of a staged candidate beyond its float rounding: half a lattice step per axis
    // (0.5001 to cover the rounding of the quantisation itself), plus the roundings of the origin
    const float q = ax.qinv * 1.0001f + 1.0e-15f;
    for (int b = it.b_lo + lane; b < it.b_hi; b += 32) {
        const BinPar bp = P.binpar[b];
        if (bp.empty) continue;
        // half extents rounded up; they bound every staged vector, hence the FP32 error of u
        const float r = (float)bp.rmax * 1.000001f + q;
        const float hx = (eu + r) * 1.000001f, hy = (ev + r) * 1.000001f, hz = (et + r) * 1.000001f;
        // norm bound of every staged vector (rows of the tile, candidates inside the query box) about the origin O
        const float m1 = (sqrtf(hx * hx + hy * hy + hz * hz) + ax.g) * 1.000001f;
        const float m2 = m1 * m1;
        // |u_fp32 - (d2_ref - mid)| <= zeta + eps32 (19 M^2 + 6 mid) (DESIGN.md section 4.1: rounding of the rows 3, of
        // the candidate's operands 3, of |s|^2 - mid 1 + 1, three FMAs 12 + 3, mid/h rounding 2; zeta = how far the
        // rows are from the unit sphere), plus the lattice: a displaced candidate changes d2 by at most
        // |delta| (2 |d| + |delta|) <= 0.87 q (4 M + q) < 4 M q + q^2
        const float eps = (EPS32 * (24.0f * m2 + 8.0f * bp.mid) + 4.0f * m1 * 1.0001f * q + q * q + P.zeta) * 1.0001f;
        S.binrec[b] = make_float4(hx, hy, hz, bp.mid);
        if constexpr (PATH == CountPath::Cumulative) {
            // cumulative counts per edge: v_k = sat(K (e_k - mid - u) + 1/2); the float copy of
            // e_k - mid adds at most eps32 |e_k - mid| to the error of u
            const float K = 0.4f / (eps + 4.0f * EPS32 * (float)bp.hi);
            S.binthr[b] = make_float2(-K, 0.f);
            const int ne = P.n_edges;
            for (int k = 0; k < CUM_EDGES; ++k)
                S.cum[b * CUM_EDGES + k] =
                    k < ne ? fmaf(K, (float)(P.r2[(size_t)b * ne + k] - (double)bp.mid), 0.5f) : -1.0e30f;
        } else if constexpr (path_multi(PATH)) {  // Histogram, HistogramWeighted
            S.binthr[b] = make_float2(bp.h + eps, eps + 4.0f * EPS32 * (float)bp.hi);
        } else if constexpr (path_sat(PATH)) {
            const float K = 0.4f / eps;  // undecidable tests land in v = [0.1, 0.9]: v (1 - v) >= 0.09
            S.binthr[b] = make_float2(-K, 0.5f + bp.h * K);
        } else {  // SingleWeighted
            S.binthr[b] = make_float2(bp.h - eps, bp.h + eps);
        }
    }
}

// ---- convert the landed raw chunk into the staged list; returns (entries of type 0, entries of type 1) ----
template <bool WEIGHTED>
__device__ __forceinline__ int2 stream_convert(const StreamSmem &S, int slot, int cnt, int lane) {
    const ItemAux &ax = S.aux[slot];
    const int k0 = ax.ko[0], k1 = ax.ko[1], k2 = ax.ko[2];
    const float qinv = ax.qinv;
    const double qd = (double)qinv;
    int L0 = 0, L1 = 0;
    for (int base = 0; base < cnt; base += 32) {
        const int i = base + lane;
        bool ok = i < cnt;
        float fx = 0.f, fy = 0.f, fz = 0.f, mid = 0.f;
        int kdx = 0, kdy = 0, kdz = 0;
        unsigned aux = 0u;
        int b = 0;
        if (ok) {
            const SRec r = S.raw[i];
            b = S.rawbin[i];
            aux = r.aux;
            // exact integer differences, rounded once to float, times a power of two
            kdx = r.ku - k0; kdy = r.kv - k1; kdz = r.kt - k2;
            fx = (float)kdx * qinv;
            fy = (float)kdy * qinv;
            fz = (float)kdz * qinv;
            const float4 rec4 = S.binrec[b];
            mid = rec4.w;
            ok = fabsf(fx) <= rec4.x && fabsf(fy) <= rec4.y && fabsf(fz) <= rec4.z;
        }
        const bool second = (aux >> 31) != 0u;
        const unsigned m0 = __ballot_sync(FULL, ok && !second), m1 = __ballot_sync(FULL, ok && second);
        if (ok) {
            const unsigned below = (1u << lane) - 1u;
            const int pos = second ? LB - 1 - (L1 + __popc(m1 & below)) : L0 + __popc(m0 & below);
            // into the tile frame in double (exact lattice differences), rounded ONCE to the operands of the test
            const double qx = (double)kdx * qd + ax.dq[0], qy = (double)kdy * qd + ax.dq[1], qz = (double)kdz * qd + ax.dq[2];
            const double sx = ax.R[0] * qx + ax.R[1] * qy + ax.R[2] * qz;
            const double sy = ax.R[3] * qx + ax.R[4] * qy + ax.R[5] * qz;
            const double sz = ax.R[6] * qx + ax.R[7] * qy + ax.R[8] * qz;
            const double sn = sx * sx + sy * sy + sz * sz;
            S.list[pos] = make_float4((float)(-2.0 * sx), (float)(-2.0 * sy), (float)(-2.0 * (1.0 + sz)), (float)(sn - (double)mid));
            S.lidx[pos] = (int)aux;  // row of its catalog | catalog bit
            S.lbin[pos] = (unsigned short)b;
            if (WEIGHTED) S.lw[pos] = S.rawlw[i];
        }
        L0 += __popc(m0);
        L1 += __popc(m1);
    }
    return make_int2(L0, L1);
}

// ---- segment table: runs of equal z-bin in the two regions of the staged list; returns their number -------
__device__ __forceinline__ int stream_segments(const StreamSmem &S, int L0, int L1, int lane) {
    int n_seg = 0;
#pragma unroll
    for (int region = 0; region < 2; ++region) {
        const int lo = region ? LB - L1 : 0, hi = region ? LB : L0;
        const int first_seg = n_seg;
        for (int base = lo; base < hi; base += 32) {
            const int e = base + lane;
            const bool start = e < hi && (e == lo || S.lbin[e] != S.lbin[e - 1]);
            const unsigned ms = __ballot_sync(FULL, start);
            if (start) {
                SegDesc &d = S.seg[n_seg + __popc(ms & ((1u << lane) - 1u))];
                d.ea = (short)e;
                d.bin = (short)S.lbin[e];
                d.type = (short)region;
            }
            n_seg += __popc(ms);
        }
        __syncwarp();
        for (int s = first_seg + lane; s < n_seg; s += 32) S.seg[s].eb = s + 1 < n_seg ? S.seg[s + 1].ea : (short)hi;
    }
    __syncwarp();
    return n_seg;
}

// ---- the headline test loop: unweighted, one sub-bin, saturating ramp ----------------------------------
// Per z-bin segment: groups of four candidates fully unrolled plus a fall-through tail, the decided /
// undecided check once per <= 16 candidates, the warp total of a segment added to the accumulator while the
// next segment is already running.
// SPLIT (tiles over the union of two second catalogs): Σv is kept per register pair and the count is split by the
// catalog of each row (bit r of `tmask`: row r of the lane is a row of catalog 1) into the accumulators
// [catalog][first catalog][z-bin].  The two parts travel packed in one word, catalog 1 in the high 16 bits: a segment
// holds at most LB candidates, so a warp counts at most LB * YAWB_TILE = 32768 pairs of either catalog in it.
template <bool SPLIT>
__device__ __forceinline__ void stream_test_sat(const FastParams &P, const StreamSmem &S, int n_seg,
                                                const float2 (&rx)[HPL], const float2 (&ry)[HPL], const float2 (&rz)[HPL],
                                                unsigned tmask, const Tile &tl, int lane, unsigned &n_recheck) {
    static_assert(LB * YAWB_TILE <= 0xffff, "the packed counts of a segment fit 16 bits");
    unsigned pend_tot = 0;
    int pend_acc = -1;
    auto flush = [&]() {  // the previous segment (its REDUX is long done)
        if (!SPLIT) {
            S.acc[pend_acc] += pend_tot;
            return;
        }
        S.acc[pend_acc] += pend_tot & 0xffffu;
        S.acc[P.n_types * P.n_bins + pend_acc] += pend_tot >> 16;
    };
    for (int sg = 0; sg < n_seg; ++sg) {
        const SegDesc d = S.seg[sg];
        const float2 thr = S.binthr[d.bin];
        const float ta = thr.x, tb = thr.y;
        unsigned cnt_total = 0;
        for (int c0 = d.ea; c0 < d.eb; c0 += 16) {
            const int c1 = min(c0 + 16, (int)d.eb);
            constexpr int NA = SPLIT ? HPL : 1;
            float2 acc_a[NA], acc_b = make_float2(0.f, 0.f);
#pragma unroll
            for (int k = 0; k < NA; ++k) acc_a[k] = make_float2(0.f, 0.f);
            int e = c0;
#define YAWB_T(idx) test_candidate_sat<NA>(S.list[idx], rx, ry, rz, ta, tb, acc_a, acc_b)
            for (; e + 4 <= c1; e += 4) {
                YAWB_T(e); YAWB_T(e + 1); YAWB_T(e + 2); YAWB_T(e + 3);
            }
            switch (c1 - e) {
                case 3: YAWB_T(e + 2);
                case 2: YAWB_T(e + 1);
                case 1: YAWB_T(e);
                default: break;
            }
#undef YAWB_T
            // a decided chunk has every v at 0 or 1: the sums of v are exact integers
            float sa = 0.f, sa1 = 0.f;
#pragma unroll
            for (int k = 0; k < NA; ++k) {
                sa += acc_a[k].x + acc_a[k].y;
                if (SPLIT)
                    sa1 += ((tmask >> (2 * k)) & 1u ? acc_a[k].x : 0.f) + ((tmask >> (2 * k + 1)) & 1u ? acc_a[k].y : 0.f);
            }
            const float sb = acc_b.x + acc_b.y;
            unsigned c = (unsigned)(sa + 0.5f);
            if (SPLIT) c += 0xffffu * (unsigned)(sa1 + 0.5f);
            unsigned flagged = __ballot_sync(FULL, sa != sb);
            while (flagged) {  // warp-uniform: some lane met the uncertainty band of an edge
                const int src = __ffs(flagged) - 1;
                flagged &= flagged - 1;
                unsigned cx = 0;
                recheck_span(P, S, c0, c1, tl, lane, src, P.binpar[d.bin].lo, P.binpar[d.bin].hi, cx, n_recheck);
                if (lane == src) c = cx;
            }
            cnt_total += c;
        }
        if (lane == 0 && pend_acc >= 0) flush();
        pend_tot = __reduce_add_sync(FULL, cnt_total);
        pend_acc = d.type * P.n_bins + d.bin;
    }
    if (lane == 0 && pend_acc >= 0) flush();
}

// ---- every other path: the shared phase-2 functions, one pass per segment ------------------------------
template <CountPath PATH>
__device__ __forceinline__ void stream_test_generic(const FastParams &P, const StreamSmem &S, int n_seg,
                                                    const float2 (&rx)[HPL], const float2 (&ry)[HPL],
                                                    const float2 (&rz)[HPL], const Tile &tl,
                                                    int lane, int nsub, unsigned &n_recheck, size_t item_off,
                                                    const double (&rwt)[YAWB_RPL]) {
    constexpr bool WEIGHTED = path_weighted(PATH);
    const size_t nacc1 = (size_t)P.n_bins * nsub;  // accumulators of one type
    for (int sg = 0; sg < n_seg; ++sg) {
        const SegDesc d = S.seg[sg];
        const int ea = d.ea, eb = d.eb, b = d.bin;
        unsigned long long *const acc = S.acc ? S.acc + d.type * nacc1 : nullptr;
        double *const accw = (WEIGHTED && S.accw) ? S.accw + d.type * nacc1 : nullptr;
        const float2 thr = S.binthr[b];
        if constexpr (PATH == CountPath::Cumulative) {
            phase2_cumul(P, S, acc, ea, eb, rx, ry, rz, thr.x, tl, lane, b, n_recheck);
        } else if constexpr (path_multi(PATH)) {  // Histogram, HistogramWeighted
            for (int k = lane; k < nsub; k += 32) {
                S.hist[k] = 0u;
                if (WEIGHTED) S.histw[k] = 0.0;
            }
            __syncwarp();
            phase2_multi_queue<WEIGHTED>(P, S, ea, eb, rx, ry, rz, thr.x, thr.y, S.binrec[b].w, tl, lane, b, n_recheck);
            __syncwarp();
            if (P.acc_global) {  // straight to the result: one atomic per non-empty sub-bin of the segment
                const size_t o = item_off + (size_t)d.type * P.type_stride + (size_t)b * nsub;
                for (int k = lane; k < nsub; k += 32) {
                    if (S.hist[k]) atomicAdd(&P.out_cnt[o + k], (unsigned long long)S.hist[k]);
                    if (WEIGHTED && S.histw[k] != 0.0) atomicAdd(&P.out_w[o + k], S.histw[k]);
                }
            } else {
                for (int k = lane; k < nsub; k += 32) {
                    acc[(size_t)b * nsub + k] += S.hist[k];
                    if (WEIGHTED) accw[(size_t)b * nsub + k] += S.histw[k];
                }
            }
            __syncwarp();
        } else {  // SingleWeighted
            unsigned cnt_total = 0;
            double w_total = 0.0;
            phase2_single(P, S, ea, eb, rx, ry, rz, thr.x, thr.y, tl, lane, P.binpar[b].lo, P.binpar[b].hi, cnt_total,
                          w_total, n_recheck, rwt);
            const unsigned tot = __reduce_add_sync(FULL, cnt_total);
            const double wtot = warp_sum(w_total);
            if (lane == 0) {
                acc[b] += tot;
                accw[b] += wtot;
            }
        }
    }
}

// Results of an item (first catalog 0): its output block (second catalog of a joint launch, then label; Item::blk), its
// patch pair.  Read from the item's slot where it is needed rather than kept in registers through the tick.  The
// accumulators are flushed at the end of every item, so items of different blocks never share them.
__device__ __forceinline__ size_t item_offset(const FastParams &P, const Item &it, int nsub) {
    return (size_t)it.blk * P.n_types * P.type_stride + (size_t)it.pair * P.n_bins * nsub;
}

// ---- the kernel ----------------------------------------------------------------------------------------
template <CountPath PATH>
__global__ void __launch_bounds__(STREAM_WARPS * 32, STREAM_CTAS) k_count_stream(const FastParams P) {
    constexpr bool WEIGHTED = path_weighted(PATH), MULTI = path_multi(PATH);
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int nsub = P.n_edges - 1;
    const bool acc_global = MULTI && P.acc_global;
    const int nacc = acc_global ? 0 : P.n_sec * P.n_types * P.n_bins * nsub;  // accumulators kept in shared memory
    StreamSmem S;
    const size_t per_warp = stream_carve(nullptr, nullptr, WEIGHTED, MULTI, P.n_bins, nsub, P.n_types, P.n_sec, acc_global);
    stream_carve(&S, smem_raw + warp * per_warp, WEIGHTED, MULTI, P.n_bins, nsub, P.n_types, P.n_sec, acc_global);
    for (int k = lane; k < nacc; k += 32) {
        S.acc[k] = 0ull;
        if (WEIGHTED) S.accw[k] = 0.0;
    }
    // written by the planner (clamped: an overflowing list makes the host repeat the call)
    const long long n_heavy = min((long long)P.counters[4], P.cap_heavy);
    const long long n_live = n_heavy + min((long long)P.counters[5], P.cap_light);
    unsigned long long n_tests = 0;
    unsigned n_recheck = 0;

    // ---- prologue: two records, the plan of the first item, the index of a third ----
    long long next_idx = 0;
    bool grabbing = true;  // the global counter has not run past the end yet
    if (lane == 0) next_idx = (long long)atomicAdd(&P.counters[0], 2ull);
    next_idx = __shfl_sync(FULL, next_idx, 0);
#pragma unroll
    for (int j = 0; j < 2; ++j) stream_fetch(P, S, j, next_idx + j, n_heavy, n_live, lane);
    if (next_idx + 1 >= n_live) grabbing = false;
    cp_async_commit();
    cp_async_wait_all();
    __syncwarp();
    stream_plan(P, S, 0, lane);
    if (grabbing && lane == 0) next_idx = (long long)atomicAdd(&P.counters[0], 1ull);
    if (!grabbing) next_idx = n_live;
    cp_async_commit();

    int ip = -1;  // item of the producer (slot ip & 3)
    bool prod_done = false, prod_exhausted = true;
    int p_t0 = 0, p_ncand = 0, p_ncombo = 0;
    int raw_cnt = -1, raw_slot = 0;  // the chunk in flight: rows (-1: none), slot of its item
    bool raw_first = false, raw_last = false;

    float2 rx[HPL], ry[HPL], rz[HPL];  // rows (2k, 2k+1) of the lane share one register pair, in the tile frame
    double rwt[YAWB_RPL];                       // their weights (weighted kernels only)
    unsigned tmask = 0;                         // bit r: row r of the lane is a row of catalog 1 of the index (SingleUnion)
#pragma unroll
    for (int r = 0; r < HPL; ++r) rx[r] = ry[r] = rz[r] = make_float2(0.f, 0.f);
#pragma unroll
    for (int r = 0; r < YAWB_RPL; ++r) rwt[r] = 0.0;
    Tile tl{};

    while (true) {
        cp_async_wait_all();
        __syncwarp();
        const int c_cnt = raw_cnt, c_slot = raw_slot;
        const bool c_first = raw_first, c_last = raw_last;
        int n_seg = 0;
        if (c_cnt >= 0) {
            const Item &it = S.items[c_slot];
            double dx[YAWB_RPL], dy[YAWB_RPL], dz[YAWB_RPL];
            if (c_first) {
                // rows of the tile: loads issued now, used after the conversion of the raw chunk
                tl.start = it.start; tl.count = it.count; tl.patch = it.src; tl.bin = 0;  // patch: the tile's catalog
                const double *const rxs = it.src ? P.rx2 : P.rx, *const rws = it.src ? P.rw2 : P.rw;
                tmask = 0;
#pragma unroll
                for (int r = 0; r < YAWB_RPL; ++r) {
                    const int k = lane + 32 * r;
                    dx[r] = dy[r] = dz[r] = 0.0;
                    if (k < it.count) {
                        const int j = it.start + k;
                        const double2 *const row = reinterpret_cast<const double2 *>(rxs + (size_t)YAWB_RSTRIDE * j);
                        const double2 ra = row[0], rb = row[1];  // 32-byte row record: x, y, z, catalog
                        dx[r] = ra.x; dy[r] = ra.y; dz[r] = rb.x;
                        if (PATH == CountPath::SingleUnion && rb.y != 0.0) tmask |= 1u << r;
                        if (WEIGHTED) rwt[r] = rws ? rws[j] : 1.0;
                    }
                }
                stream_begin<PATH>(P, S, c_slot, lane);
                __syncwarp();
            }
            if (c_first) {
                const PatchFrame &F = P.sframe[it.p1];
                const ItemAux &ax = S.aux[c_slot];
                const double c0 = F.c[0], c1 = F.c[1], c2 = F.c[2];
                const double a0 = F.e1[0], a1 = F.e1[1], a2 = F.e1[2];
                const double g0 = F.e2[0], g1 = F.e2[1], g2 = F.e2[2];
#pragma unroll
                for (int r = 0; r < YAWB_RPL; ++r) {
                    const int k = lane + 32 * r;
                    float x = PAD_ROW, y = PAD_ROW, z = PAD_ROW;  // padding rows: u = NaN, every form of the test rejects it
                    if (k < it.count) {
                        const double ex = dx[r] - c0, ey = dy[r] - c1, ez = dz[r] - c2;
                        const double qx = ex * a0 + ey * a1 + ez * a2 - ax.O[0];
                        const double qy = ex * g0 + ey * g1 + ez * g2 - ax.O[1];
                        const double qz = ex * c0 + ey * c1 + ez * c2 - ax.O[2];
                        x = (float)(ax.R[0] * qx + ax.R[1] * qy + ax.R[2] * qz);
                        y = (float)(ax.R[3] * qx + ax.R[4] * qy + ax.R[5] * qz);
                        z = (float)(ax.R[6] * qx + ax.R[7] * qy + ax.R[8] * qz);
                    } else if (WEIGHTED) {
                        rwt[r] = 0.0;
                    }
                    if (r & 1) { rx[r >> 1].y = x; ry[r >> 1].y = y; rz[r >> 1].y = z; }
                    else { rx[r >> 1].x = x; ry[r >> 1].x = y; rz[r >> 1].x = z; }
                }
            }
            const int2 L = stream_convert<WEIGHTED>(S, c_slot, c_cnt, lane);
            __syncwarp();
            n_seg = stream_segments(S, L.x, L.y, lane);
            n_tests += (unsigned long long)(L.x + L.y) * (unsigned long long)it.count;
        }

        // ---- produce: request the next raw chunk; at an item boundary advance the stages behind it ----
        raw_cnt = -1;
        if (!prod_done) {
            if (prod_exhausted) {
                ++ip;
                const int slot = ip & (NSLOT - 1);
                if (S.aux[slot].end) {
                    prod_done = true;
                } else {
                    p_ncombo = S.aux[slot].n_combo;
                    p_ncand = stream_runs(S, p_ncombo, lane);
                    p_t0 = 0;
                    prod_exhausted = false;
                    stream_plan(P, S, (ip + 1) & (NSLOT - 1), lane);
                    const long long idx = __shfl_sync(FULL, next_idx, 0);
                    stream_fetch(P, S, (ip + 2) & (NSLOT - 1), idx, n_heavy, n_live, lane);
                    if (idx >= n_live) grabbing = false;
                    if (grabbing) {
                        if (lane == 0) next_idx = (long long)atomicAdd(&P.counters[0], 1ull);
                    } else {
                        next_idx = n_live;
                    }
                }
            }
            if (!prod_done) {
                const int cnt = min(LB, p_ncand - p_t0);
                stream_issue<WEIGHTED>(P, S, p_ncombo, p_t0, cnt, lane);
                raw_cnt = cnt;
                raw_slot = ip & (NSLOT - 1);
                raw_first = p_t0 == 0;
                p_t0 += cnt;
                raw_last = p_t0 >= p_ncand;
                prod_exhausted = raw_last;
            }
        }
        cp_async_commit();

        // ---- test ----
        if (c_cnt >= 0) {
            if (n_seg > 0) {
                if constexpr (path_sat(PATH))
                    stream_test_sat<PATH == CountPath::SingleUnion>(P, S, n_seg, rx, ry, rz, tmask, tl, lane, n_recheck);
                else
                    stream_test_generic<PATH>(P, S, n_seg, rx, ry, rz, tl, lane, nsub, n_recheck,
                                              item_offset(P, S.items[c_slot], nsub), rwt);
            }
            if (c_last) {  // the item is complete: its counts go to the result of its patch pair and output block
                // (accumulator group g = catalog of a union tile's row * n_types + first catalog; the output blocks of
                // the two catalogs of a union are 0 and 1)
                __syncwarp();
                const size_t nacc1 = (size_t)P.n_bins * nsub;
                const size_t item_off = item_offset(P, S.items[c_slot], nsub);
                for (int k = lane; k < nacc; k += 32) {
                    const int g = PATH == CountPath::SingleUnion ? k / (int)nacc1 : k >= (int)nacc1 ? 1 : 0;
                    const size_t o = item_off + (size_t)g * P.type_stride + (k - g * nacc1);
                    const unsigned long long c = S.acc[k];
                    if (c) {
                        atomicAdd(&P.out_cnt[o], c);
                        S.acc[k] = 0ull;
                    }
                    if (WEIGHTED) {
                        const double w = S.accw[k];
                        if (w != 0.0) {
                            atomicAdd(&P.out_w[o], w);
                            S.accw[k] = 0.0;
                        }
                    }
                }
            }
        } else if (prod_done && raw_cnt < 0) {
            break;
        }
        __syncwarp();
    }
    if (lane == 0 && n_tests) atomicAdd(&P.counters[1], n_tests);
    const unsigned rc = __reduce_add_sync(FULL, n_recheck);
    if (lane == 0 && rc) atomicAdd(&P.counters[2], (unsigned long long)rc);
}
