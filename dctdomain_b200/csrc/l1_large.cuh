// Exact L1 top-k for 992 < k <= 8192 (dctd_l1_topk_large): radix selection over the packed key instead of the heap
// scan, whose warp-private candidate buffers stop at k = 992.  Included by l1topk.cu inside its anonymous namespace,
// after the host-side scan configuration.
//
// The search orders by the key dist << 40 | position; positions make keys unique, so the k best are exactly the keys
// <= the k-th smallest one.  Here a query's keys are compressed to ck = dist << pbits | position (pbits = bits of n - 1;
// same order, T = dbits + pbits bits in all), and per query a window [lo, lo + 2^w) of ck space known to hold the k-th
// key is narrowed, kLargeBinBits bits per level, while the keys below the window are only counted:
//
//   1. l1_keyhist_kernel (histogram mode)  the TMA-staged SAD tile loop of the scan kernels (producer_loop, sad_tile,
//      load_queries, qflags tile skipping); every key inside its query's window adds 1 to bin (ck - lo) >> shift of a
//      warp-private shared-memory histogram (lanes that hit the same bin are combined with __match_any_sync), the
//      nonzero bins go to a global [nq, B] histogram at the end of the CTA.  Level 0: w = T, all queries.
//   2. l1_kresolve_kernel (one CTA per query)  the bin holding the need-th key of the window (need = min(k, n) - below):
//      below += keys in earlier bins; the query is resolved once below + count(bin) <= kLargeCand (every key up to the
//      bin's end fits the candidate list), else the bin becomes the next level's window.  A bin one key wide always
//      resolves (below < k), so there are at most ceil(T / kLargeBinBits) levels; the host launches all of them, and a
//      level no query needs costs one launch of CTAs that exit after reading the flags.  Usually one level resolves
//      everything: at d = 480 a level-0 bin is 256 distance units wide.
//   3. l1_keyhist_kernel (collect mode)  appends every key with ck <= hi (the resolved bin's end) to the query's list;
//      the count is known exactly, so the list never overflows.
//   4. l1_select_kernel  (the threshold path's selection) sorts the <= kLargeCand candidates and writes the first k.
// For n <= kLargeCand steps 1 and 2 are skipped: everything is collected.  The database is read 1 + levels times.
#pragma once

constexpr int kLargeMaxK = 8192;                  // k limit of dctd_l1_topk_large
constexpr int kLargeCand = 16384;                 // candidate slots per query: 128 KB of keys, one select CTA sorts them
constexpr int kLargeBinBits = 9;
constexpr int kLargeBins = 1 << kLargeBinBits;    // B: histogram bins per query and level
constexpr long long kLargeChunk = 2048;           // queries per chunk: ~130 KB of workspace each

struct KHistParams {
    ScanParams sp;                    // queries, database, n_groups / groups_per_split; qflags = queries still open
                                      // (null: all); collect mode: cand / cnt / cmax
    int pbits;                        // ck = dist << pbits | position
    int wbits, shift;                 // histogram mode: window [lo, lo + 2^wbits), bin = (ck - lo) >> shift
    bool collect;
    const unsigned long long *lo;     // [nq] window start (null: 0)
    const unsigned long long *hi;     // [nq] collect bound, inclusive (null: everything)
    unsigned int *hist;               // [nq, kLargeBins]
};

// one histogram per query in histogram mode; no static shared memory (large_config gives the dynamic part what the
// device allows)
template <int TQ, int kTD, int STAGES>
__global__ void __launch_bounds__((kWarps + 1) * 32, 1) l1_keyhist_kernel(const KHistParams kp) {
    const ScanParams &p = kp.sp;
    constexpr int QT = kWarps * TQ;
    extern __shared__ __align__(128) unsigned char smem[];
    const int C = chunks_of(p.d);
    const int dpad = C * 16;
    const int tile_bytes = kTD * 32 * dpad;
    unsigned long long *full = reinterpret_cast<unsigned long long *>(smem);           // [STAGES]
    unsigned long long *empty = full + STAGES;                                          // [STAGES]
    int *s_any = reinterpret_cast<int *>(empty + STAGES);                               // tile_has_flag
    unsigned char *qs = smem + 128;                                                     // [QT][dpad]
    unsigned char *st = qs + (size_t)QT * dpad;                                         // [STAGES][tile]
    unsigned int *hist = reinterpret_cast<unsigned int *>(st + (size_t)STAGES * tile_bytes);   // [QT][kLargeBins]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long q0 = (long long)blockIdx.y * QT;
    if (p.qflags && !tile_has_flag(p, q0, QT, s_any)) return;
    const long long g_begin = (long long)blockIdx.x * p.groups_per_split;
    const long long g_end = min(p.n_groups, g_begin + p.groups_per_split);
    const int n_tiles = (int)((g_end - g_begin + kTD - 1) / kTD);

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], kWarps); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    load_queries<kWarps, TQ>(p, qs, q0, dpad);
    if (!kp.collect)
        for (int i = tid; i < QT * kLargeBins; i += blockDim.x) hist[i] = 0u;
    __syncthreads();

    if (warp == kWarps) {
        if (lane == 0) producer_loop<kTD, STAGES>(p, full, empty, st, tile_bytes, C, dpad, g_begin, g_end, n_tiles);
        return;
    }

    const uint4 *qs4 = reinterpret_cast<const uint4 *>(qs) + (size_t)warp * TQ * C;
    unsigned int *whist = hist + (size_t)warp * TQ * kLargeBins;
    const unsigned long long span = kp.wbits >= 64 ? ~0ULL : (1ULL << kp.wbits);
    unsigned long long qlo[TQ], qhi[TQ];
    bool open[TQ];
#pragma unroll
    for (int a = 0; a < TQ; ++a) {
        const long long qi = q0 + warp * TQ + a;
        open[a] = qi < p.nq && (!p.qflags || p.qflags[qi]);
        qlo[a] = (kp.lo && qi < p.nq) ? kp.lo[qi] : 0ULL;
        qhi[a] = (kp.hi && qi < p.nq) ? kp.hi[qi] : ~0ULL;
    }

    for (int t = 0; t < n_tiles; ++t) {
        const int s = t % STAGES;
        mbar_wait(&full[s], (unsigned int)((t / STAGES) & 1));
        unsigned int acc[TQ][kTD];
        sad_tile<TQ, kTD>(reinterpret_cast<const uint4 *>(st + (size_t)s * tile_bytes), qs4, C, lane, acc);
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);
        const long long vbase = g_begin + (long long)t * kTD;
#pragma unroll
        for (int b = 0; b < kTD; ++b) {
            const long long id = (vbase + b) * 32 + lane;
            const bool valid = (vbase + b) < g_end && id < p.n;
#pragma unroll
            for (int a = 0; a < TQ; ++a) {
                const unsigned long long ck = ((unsigned long long)acc[a][b] << kp.pbits) | (unsigned long long)id;
                if (kp.collect) {
                    append_candidates(p, q0 + warp * TQ + a, open[a] && valid && ck <= qhi[a],
                                      ((unsigned long long)acc[a][b] << kIdBits) | (unsigned long long)id, lane);
                } else {
                    const unsigned long long rel = ck - qlo[a];
                    const bool in = open[a] && valid && rel < span;
                    if (__any_sync(0xffffffffu, in)) {
                        const unsigned int bin = in ? (unsigned int)(rel >> kp.shift) : 0xffffffffu;
                        const unsigned int peers = __match_any_sync(0xffffffffu, bin);
                        if (in && lane == __ffs(peers) - 1) atomicAdd(&whist[a * kLargeBins + bin], (unsigned int)__popc(peers));
                    }
                }
            }
        }
    }
    if (kp.collect) return;
    __syncwarp();
    for (int a = 0; a < TQ; ++a) {
        const long long qi = q0 + warp * TQ + a;
        if (!open[a]) continue;
        for (int i = lane; i < kLargeBins; i += 32) {
            const unsigned int v = whist[a * kLargeBins + i];
            if (v) atomicAdd(&kp.hist[qi * kLargeBins + i], v);
        }
    }
}

// One CTA of kLargeBins threads per query still open at `level` (level 0: every query, window [0, 2^T), below = 0).
// Reads and zeroes the query's histogram, finds the bin of the need-th key, and either resolves the query (hi = the
// bin's last ck, open = 0) or makes the bin its next window.  *levels = the most levels any query took part in.
struct KResolveParams {
    unsigned int *hist;
    unsigned long long *lo, *hi;
    unsigned int *below;
    int *open;
    unsigned int *levels;
    int level, shift;
    unsigned int want;                // min(k, n)
};

__global__ void __launch_bounds__(kLargeBins) l1_kresolve_kernel(const KResolveParams r) {
    __shared__ unsigned int wsum[kLargeBins / 32];
    const long long qi = blockIdx.x;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    if (r.level > 0 && !r.open[qi]) return;
    const unsigned long long lo = r.level > 0 ? r.lo[qi] : 0ULL;
    const unsigned int below = r.level > 0 ? r.below[qi] : 0u;
    unsigned int *h = r.hist + qi * kLargeBins;
    const unsigned int c = h[t];
    h[t] = 0u;                                      // the next level starts from zeros
    unsigned int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    for (int w = 0; w < warp; ++w) incl += wsum[w];
    const unsigned int excl = incl - c;
    const unsigned int need = r.want - below;       // rank of the k-th key among the window's keys (>= 1)
    if (excl < need && need <= incl) {              // exactly one thread
        const unsigned int nb = below + excl;
        const unsigned long long start = lo + ((unsigned long long)t << r.shift);
        if (nb + c <= (unsigned int)kLargeCand) {
            r.hi[qi] = start + ((1ULL << r.shift) - 1ULL);
            r.open[qi] = 0;
        } else {
            r.lo[qi] = start;
            r.below[qi] = nb;
            r.open[qi] = 1;
        }
        atomicMax(r.levels, (unsigned int)(r.level + 1));
    }
}

// Exact merge of sorted lists for k > 992 (the bitonic merge's shared memory holds 2k keys per warp): every element
// goes to the output slot given by its rank - its index in its own list plus the keys of every other list before it
// (smaller, or equal and in an earlier list: only padding keys repeat).  One thread per element.
template <bool PAIRS>
__global__ void __launch_bounds__(256) l1_rankmerge_kernel(const MergeParams p) {
    auto load = [&](int part, long long qi, int i) -> unsigned long long {
        const long long o = ((long long)part * p.nq + qi) * p.k + i;
        if (!PAIRS) return p.key_parts[o];
        const long long id = p.id_parts[o];
        if (id < 0) return kKeyMax;
        return ((unsigned long long)(unsigned int)p.dist_parts[o] << kIdBits) | (unsigned long long)id;
    };
    const long long total = (long long)p.parts * p.nq * p.k;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(e % p.k);
        const long long r = e / p.k;
        const long long qi = r % p.nq;
        const int part = (int)(r / p.nq);
        const unsigned long long x = load(part, qi, i);
        long long slot = i;
        for (int s = 0; s < p.parts && slot < p.k; ++s) {
            if (s == part) continue;
            int a = 0, b = p.k;                    // keys of list s that come before x
            while (a < b) {
                const int m = (a + b) >> 1;
                const unsigned long long y = load(s, qi, m);
                if (y < x || (y == x && s < part)) a = m + 1;
                else b = m;
            }
            slot += a;
        }
        if (slot >= p.k) continue;
        const long long o = qi * p.k + slot;
        if (p.key_out) p.key_out[o] = (x == kKeyMax) ? kKeyMax : x + (unsigned long long)p.id_base;
        if (p.dist) {
            if (x == kKeyMax) {
                p.dist[o] = FLT_MAX;
                p.ids[o] = -1;
            } else {
                p.dist[o] = (float)(unsigned int)(x >> kIdBits);
                p.ids[o] = (long long)(x & kIdMask) + p.id_base;
            }
        }
    }
}

int run_rank_merge(const MergeParams &mp, bool pairs, cudaStream_t stream) {
    const long long total = (long long)mp.parts * mp.nq * mp.k;
    const unsigned grid = (unsigned)std::min<long long>((total + 255) / 256, 1LL << 20);
    if (pairs) l1_rankmerge_kernel<true><<<grid, 256, 0, stream>>>(mp);
    else l1_rankmerge_kernel<false><<<grid, 256, 0, stream>>>(mp);
    DCTD_LAUNCH_CHECK();
    return DCTD_OK;
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
int bit_length(unsigned long long x) {
    int b = 0;
    while (x) { ++b; x >>= 1; }
    return b;
}

struct LargeLayout {
    long long chunk;
    size_t off_levels, off_hist, off_lo, off_hi, off_below, off_open, off_cnt, off_cand, total;
};

bool large_layout(long long nq, int d, int k, LargeLayout *l) {
    if (nq <= 0 || k < 1 || k > kLargeMaxK || d < 1 || d > 2048) return false;
    l->chunk = std::min<long long>(nq, kLargeChunk);
    const size_t q = (size_t)l->chunk;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += dctd::align_up(bytes, 256); return o; };
    l->off_levels = take(sizeof(unsigned int));
    l->off_hist = take(q * kLargeBins * sizeof(unsigned int));
    l->off_lo = take(q * 8);
    l->off_hi = take(q * 8);
    l->off_below = take(q * sizeof(unsigned int));
    l->off_open = take(q * sizeof(int));
    l->off_cnt = take(q * sizeof(int));
    l->off_cand = take(q * (size_t)kLargeCand * 8);
    l->total = off + 256;
    return true;
}

struct LargeConfig {
    int tq, td, stages;
    size_t smem_hist, smem_collect;
    long long n_qtiles, splits, groups_per_split;
};

typedef void (*KHistFn)(const KHistParams);

KHistFn keyhist_kernel(const LargeConfig &c) {
#define DCTD_KH(TD_, ST_)                                          \
    switch (c.tq) {                                                \
        case 1: return l1_keyhist_kernel<1, TD_, ST_>;             \
        case 2: return l1_keyhist_kernel<2, TD_, ST_>;             \
        case 4: return l1_keyhist_kernel<4, TD_, ST_>;             \
        default: return l1_keyhist_kernel<8, TD_, ST_>;            \
    }
    if (c.td == 1) { DCTD_KH(1, 2) }
    if (c.stages == 2) { DCTD_KH(kTDmax, 2) }
    DCTD_KH(kTDmax, kStagesMax)
#undef DCTD_KH
}

// Query tile, groups per stage and stages of l1_keyhist_kernel: the largest query tile (up to 8 per warp, fewer for
// few queries) whose histograms, queries and stages fit next to the kernel's static shared memory.  Every d <= 2048 fits.
bool large_config(const DevInfo &di, long long nq, long long n_groups, int d, LargeConfig *c) {
    const size_t dpad = (size_t)chunks_of(d) * 16;
    auto smem_of = [&](int tq, int td, int st, bool hist) {
        const size_t qt = (size_t)kWarps * tq;
        return (size_t)128 + qt * dpad + (size_t)st * td * 32 * dpad + (hist ? qt * kLargeBins * sizeof(unsigned int) : 0);
    };
    int tq = 8;
    while (tq > 1 && (long long)kWarps * (tq / 2) >= nq) tq /= 2;
    static const int shapes[3][2] = {{kTDmax, kStagesMax}, {kTDmax, 2}, {1, 2}};
    for (; tq >= 1; tq /= 2) {
        for (const auto &sh : shapes) {
            LargeConfig t{};
            t.tq = tq; t.td = sh[0]; t.stages = sh[1];
            cudaFuncAttributes attr{};
            if (cudaFuncGetAttributes(&attr, keyhist_kernel(t)) != cudaSuccess) {
                cudaGetLastError();
                attr.sharedSizeBytes = 0;     // no device: sizes only
            }
            if (attr.sharedSizeBytes + smem_of(tq, sh[0], sh[1], true) > di.smem) continue;
            *c = t;
            c->smem_hist = smem_of(tq, sh[0], sh[1], true);
            c->smem_collect = smem_of(tq, sh[0], sh[1], false);
            c->n_qtiles = (nq + (long long)kWarps * tq - 1) / ((long long)kWarps * tq);
            pick_splits(di.sms, n_groups, c->td, c->n_qtiles, 2, &c->splits, &c->groups_per_split);
            return true;
        }
    }
    return false;
}

int run_topk_large(const int8_t *d_q, int64_t nq, const void *d_packed, int64_t n, int32_t d, int32_t k, int64_t id_base,
                   float *d_dist, long long *d_ids, unsigned long long *d_keys, void *d_workspace, size_t workspace_bytes,
                   cudaStream_t stream) {
    if (nq < 0 || n < 0 || k < 1 || d < 1 || id_base < 0) return DCTD_ERR_ARG;
    if (k > kLargeMaxK || d > 2048) return DCTD_ERR_UNSUPPORTED;
    if (nq == 0) return DCTD_OK;
    if (!d_q || (d_dist == nullptr) != (d_ids == nullptr) || (!d_dist && !d_keys) || (n > 0 && !d_packed))
        return DCTD_ERR_ARG;
    if (n >= (1LL << kIdBits) || id_base + n >= (1LL << kIdBits)) return DCTD_ERR_UNSUPPORTED;
    LargeLayout l;
    if (!large_layout(nq, d, k, &l)) return DCTD_ERR_UNSUPPORTED;
    if (!d_workspace || workspace_bytes < l.total) return DCTD_ERR_WORKSPACE;
    if (((uintptr_t)d_workspace & 255) != 0 || ((uintptr_t)d_packed & 15) != 0) return DCTD_ERR_ARG;
    DevInfo di;
    dev_info(&di);
    const long long n_groups = (n + 31) / 32;
    LargeConfig cfg{};
    if (n > 0 && !large_config(di, l.chunk, n_groups, d, &cfg)) return DCTD_ERR_UNSUPPORTED;
    char *ws = (char *)d_workspace;
    unsigned int *levels = (unsigned int *)(ws + l.off_levels);
    unsigned int *hist = (unsigned int *)(ws + l.off_hist);
    unsigned long long *lo = (unsigned long long *)(ws + l.off_lo);
    unsigned long long *hi = (unsigned long long *)(ws + l.off_hi);
    unsigned int *below = (unsigned int *)(ws + l.off_below);
    int *open = (int *)(ws + l.off_open);
    int *cnt = (int *)(ws + l.off_cnt);
    unsigned long long *cand = (unsigned long long *)(ws + l.off_cand);

    const bool select_all = n <= kLargeCand;
    const int pbits = bit_length((unsigned long long)std::max<long long>(n - 1, 0));
    const int total_bits = bit_length(255ULL * (unsigned long long)d) + pbits;
    const int n_levels = select_all ? 0 : (total_bits + kLargeBinBits - 1) / kLargeBinBits;
    DCTD_CUDA_TRY(cudaMemsetAsync(levels, 0, sizeof(unsigned int), stream));
    if (n_levels > 0) DCTD_CUDA_TRY(cudaMemsetAsync(hist, 0, (size_t)l.chunk * kLargeBins * sizeof(unsigned int), stream));
    KHistFn fn = n > 0 ? keyhist_kernel(cfg) : nullptr;
    if (fn) DCTD_CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cfg.smem_hist));
    const size_t ssmem = (size_t)next_pow2((int)std::max<long long>(64, std::min<long long>(n, kLargeCand))) * 8;
    DCTD_CUDA_TRY(cudaFuncSetAttribute(l1_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ssmem));

    for (long long q0 = 0; q0 < nq; q0 += l.chunk) {
        const long long cq = std::min<long long>(l.chunk, nq - q0);
        KHistParams kp{};
        kp.sp.q = d_q + q0 * d; kp.sp.packed = (const uint4 *)d_packed; kp.sp.nq = cq; kp.sp.n = n; kp.sp.d = d; kp.sp.k = k;
        kp.sp.gstride = 1; kp.sp.n_groups = n_groups; kp.sp.groups_per_split = cfg.groups_per_split;
        kp.pbits = pbits;
        kp.hist = hist;
        const dim3 grid((unsigned)cfg.splits, (unsigned)cfg.n_qtiles);
        // 1 + 2: histogram levels
        for (int level = 0, w = total_bits; level < n_levels; ++level) {
            const int shift = std::max(w - kLargeBinBits, 0);
            kp.collect = false;
            kp.wbits = w; kp.shift = shift;
            kp.lo = level ? lo : nullptr;
            kp.sp.qflags = level ? open : nullptr;
            fn<<<grid, (kWarps + 1) * 32, cfg.smem_hist, stream>>>(kp);
            DCTD_LAUNCH_CHECK();
            KResolveParams rp{hist, lo, hi, below, open, levels, level, shift,
                              (unsigned int)std::min<long long>(k, n)};
            l1_kresolve_kernel<<<(unsigned)cq, kLargeBins, 0, stream>>>(rp);
            DCTD_LAUNCH_CHECK();
            w = shift;
        }
        // 3. collect: every key up to the resolved bound (everything when n <= kLargeCand)
        DCTD_CUDA_TRY(cudaMemsetAsync(cnt, 0, (size_t)cq * sizeof(int), stream));
        if (n > 0) {
            kp.collect = true;
            kp.lo = nullptr;
            kp.hi = n_levels ? hi : nullptr;
            kp.sp.qflags = nullptr;
            kp.sp.cand = cand; kp.sp.cnt = cnt; kp.sp.cmax = kLargeCand;
            fn<<<grid, (kWarps + 1) * 32, cfg.smem_collect, stream>>>(kp);
            DCTD_LAUNCH_CHECK();
        }
        // 4. exact selection of the k best candidates, once per output form (select_query writes one)
        SelectParams se{};
        se.cand = cand; se.cnt = cnt; se.cmax = kLargeCand; se.k = k; se.nq = cq; se.id_base = id_base;
        se.qflags = open;
        if (d_keys) {
            se.key_out = d_keys + q0 * k;
            l1_select_kernel<<<(unsigned)cq, 256, ssmem, stream>>>(se);
            DCTD_LAUNCH_CHECK();
        }
        if (d_dist) {
            se.key_out = nullptr;
            se.dist = d_dist + q0 * k;
            se.ids = d_ids + q0 * k;
            l1_select_kernel<<<(unsigned)cq, 256, ssmem, stream>>>(se);
            DCTD_LAUNCH_CHECK();
        }
    }
    return DCTD_OK;
}
