// Hits of dct-sim's database search (reference src/dct-sim.py:126-156) without the all-pairs matrices of
// l1_protein.cuh.  Included by l1topk.cu inside its anonymous namespace, after the host-side scan configuration.
//
// dct-sim ranks query protein a's hits by the similarity of the two proteins' LAST (global) fingerprints,
// s = 1 - min(last / 17000, 1): ascending by the clamped key (min(last, clamp), b).  It prints the first
// max(top', c_a) entries of that order, c_a = #{b : min(last, clamp) <= cut}.  So:
//
//   1. hits_pack_globals_kernel   database protein b's last row -> vector b of a packed set (layout of pack_kernel),
//                                 plus a flag for proteins without fingerprints (their key is (clamp, b));
//      hits_gather_queries_kernel   the same for a chunk of query proteins, row-major.
//   2. l1_hits_scan_kernel        the heap scan of l1topk.cu with ClampedKey: distances are clamped (empty proteins on
//                                 either side take the clamp) before the key is built, so its exact top-`cap` is the
//                                 first `cap` entries of dct-sim's order; the same pass counts the keys within `cut`
//                                 (exactly, whatever cap is).  Splits meet in l1_merge_kernel.
//   3. hits_output_kernel         one warp per output slot: hit count max(top', c_a), database protein, and for the
//                                 hit pair the min over all fingerprint pairs and the last-vs-last distance (the body
//                                 of pair_scores_kernel, reading the two row-major fingerprint arrays).
//
// The scan is one SAD per (query protein, database protein) pair instead of one per fingerprint pair.
#pragma once

constexpr int kHitsMaxCap = 992;               // = the heap scan's k limit (make_config)
constexpr long long kHitsMaxChunk = 1LL << 16;  // query proteins per chunk at most

struct ClampedKey {
    static constexpr bool kClamped = true;
    unsigned int clamp;                 // distances >= clamp tie at clamp (then ordered by position)
    int cut;                            // keys with clamped distance <= cut are counted
    const unsigned char *q_empty;       // [nq] 1 = query protein without fingerprints
    const unsigned char *db_empty;      // [n]  1 = database protein without fingerprints
    int *count;                         // [nq] += keys within the cut

    template <int TQ, int kTD>
    __device__ __forceinline__ void adjust(const ScanParams &p, unsigned int (&acc)[TQ][kTD], const bool (&qe)[TQ],
                                           unsigned int (&ncut)[TQ], long long vbase, long long g_end, int lane) const {
#pragma unroll
        for (int b = 0; b < kTD; ++b) {
            const long long id = real_group(p, vbase + b) * 32 + lane;
            const bool valid = (vbase + b) < g_end && id < p.n;
            const bool de = !valid || db_empty[id];
#pragma unroll
            for (int a = 0; a < TQ; ++a) {
                acc[a][b] = (qe[a] || de) ? clamp : min(acc[a][b], clamp);
                ncut[a] += (valid && (int)acc[a][b] <= cut) ? 1u : 0u;
            }
        }
    }

    template <int TQ>
    __device__ __forceinline__ void publish(unsigned int (&ncut)[TQ], long long qbase, long long nq, int lane) const {
#pragma unroll
        for (int a = 0; a < TQ; ++a) {
            unsigned int v = ncut[a];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0 && qbase + a < nq && v) atomicAdd(&count[qbase + a], (int)v);
        }
    }
};

template <int TQ, int kTD, int STAGES>
__global__ void __launch_bounds__((kWarps + 1) * 32, 1) l1_hits_scan_kernel(const ScanParams p, const ClampedKey key) {
    heap_scan<TQ, kTD, STAGES>(p, key);
}

// vector b = last row of database protein b (off[b + 1] - 1), packed as pack_kernel packs row b; empty[b] flags
// proteins without rows (their vector is padding)
__global__ void hits_pack_globals_kernel(const int8_t *__restrict__ rows, int d, const long long *__restrict__ off,
                                         long long n_prot, uint4 *__restrict__ packed, unsigned char *__restrict__ empty) {
    const int C = chunks_of(d);
    const long long total = (n_prot + 31) / 32 * 32 * C;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const long long vec = t / C;
        const int c = (int)(t % C);
        unsigned int w[4] = {0x80808080u, 0x80808080u, 0x80808080u, 0x80808080u};
        const bool has = vec < n_prot && off[vec + 1] > off[vec];
        if (has) {
            const int8_t *src = rows + (off[vec + 1] - 1) * d + c * 16;
#pragma unroll
            for (int b = 0; b < 16; ++b) {
                const int col = c * 16 + b;
                const unsigned int byte = (col < d) ? ((unsigned int)(unsigned char)src[b] ^ 0x80u) : 0x80u;
                w[b >> 2] = (w[b >> 2] & ~(0xffu << ((b & 3) * 8))) | (byte << ((b & 3) * 8));
            }
        }
        if (c == 0 && vec < n_prot) empty[vec] = has ? 0 : 1;
        packed[((vec / 32) * C + c) * 32 + (vec % 32)] = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

// q[i] = last row of query protein a0 + i (row-major [nq, d]); empty[i] flags proteins without rows (row zeroed)
__global__ void hits_gather_queries_kernel(const int8_t *__restrict__ rows, int d, const long long *__restrict__ off,
                                           long long a0, long long nq, int8_t *__restrict__ q,
                                           unsigned char *__restrict__ empty) {
    const long long total = nq * d;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const long long i = t / d;
        const int c = (int)(t % d);
        const long long e = off[a0 + i + 1];
        const bool has = e > off[a0 + i];
        q[t] = has ? rows[(e - 1) * d + c] : (int8_t)0;
        if (c == 0) empty[i] = has ? 0 : 1;
    }
}

// One warp per output slot (query i of the chunk, rank r).  count = max(top', c_a); slots r < min(count, cap) get
// the r-th key of the merged scan and the pair's (min, last) distances, the others (-1, INT32_MAX, INT32_MAX).
struct HitsOut {
    const unsigned long long *keys;     // [nq, cap] merged clamped keys of the chunk
    const int *ncut;                    // [nq] keys within the cut
    long long nq, a0;                   // chunk size, first query protein of the chunk
    int cap, top;                       // top = top' = clamp(top, 0, n_dbprot)
    const int8_t *qf, *dbf;             // row-major fingerprints
    const long long *qoff, *doff;       // device offsets
    int d;
    int *count, *hit_db, *hit_min, *hit_last;
};

template <bool VEC16>
__global__ void hits_output_kernel(const HitsOut o) {
    const int lane = threadIdx.x & 31;
    const long long w = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const long long i = w / o.cap;
    const int r = (int)(w % o.cap);
    if (i >= o.nq) return;
    const int c = max(o.top, o.ncut[i]);
    const long long a = o.a0 + i;
    if (r == 0 && lane == 0) o.count[a] = c;
    const long long slot = a * o.cap + r;
    if (r >= min(c, o.cap)) {
        if (lane == 0) { o.hit_db[slot] = -1; o.hit_min[slot] = 0x7fffffff; o.hit_last[slot] = 0x7fffffff; }
        return;
    }
    const long long b = (long long)(o.keys[i * o.cap + r] & kIdMask);
    const long long a0 = o.qoff[a], a1 = o.qoff[a + 1], b0 = o.doff[b], b1 = o.doff[b + 1];
    const int d = o.d;
    int best = 0x7fffffff, last = 0x7fffffff;
    for (long long x = a0; x < a1; ++x)
        for (long long y = b0; y < b1; ++y) {
            int s = 0;
            if (VEC16) {
                const uint4 *ra = reinterpret_cast<const uint4 *>(o.qf + x * d);
                const uint4 *rb = reinterpret_cast<const uint4 *>(o.dbf + y * d);
                unsigned int acc = 0u;
                for (int cc = lane; cc < (d >> 4); cc += 32) {
                    const uint4 u = ra[cc], v = rb[cc];
                    acc = sad4(u.x ^ 0x80808080u, v.x ^ 0x80808080u, acc);
                    acc = sad4(u.y ^ 0x80808080u, v.y ^ 0x80808080u, acc);
                    acc = sad4(u.z ^ 0x80808080u, v.z ^ 0x80808080u, acc);
                    acc = sad4(u.w ^ 0x80808080u, v.w ^ 0x80808080u, acc);
                }
                s = (int)acc;
            } else {
                for (int cc = lane; cc < d; cc += 32) s += abs((int)o.qf[x * d + cc] - (int)o.dbf[y * d + cc]);
            }
#pragma unroll
            for (int k = 16; k > 0; k >>= 1) s += __shfl_xor_sync(0xffffffffu, s, k);
            best = min(best, s);
            last = s;                   // the loops end on the last-vs-last pair
        }
    if (lane == 0) { o.hit_db[slot] = (int)b; o.hit_min[slot] = best; o.hit_last[slot] = last; }
}

typedef void (*HitsScanFn)(const ScanParams, const ClampedKey);

HitsScanFn hits_kernel(const ScanConfig &c) {
    if (c.td == kTDmax) {
        switch (c.tq) {
            case 1: return l1_hits_scan_kernel<1, kTDmax, kStagesMax>;
            case 2: return l1_hits_scan_kernel<2, kTDmax, kStagesMax>;
            case 4: return l1_hits_scan_kernel<4, kTDmax, kStagesMax>;
            default: return l1_hits_scan_kernel<8, kTDmax, kStagesMax>;
        }
    }
    switch (c.tq) {
        case 1: return l1_hits_scan_kernel<1, 1, 2>;
        case 2: return l1_hits_scan_kernel<2, 1, 2>;
        case 4: return l1_hits_scan_kernel<4, 1, 2>;
        default: return l1_hits_scan_kernel<8, 1, 2>;
    }
}

// workspace: a fixed part for the whole call, then the buffers of one chunk of `nq` query proteins
struct HitsLayout {
    ScanConfig scan;
    size_t off_packed, off_dbe, off_qoff, off_doff;                     // fixed
    size_t off_q, off_qe, off_cnt, off_parts, off_keys, off_tmp;        // per chunk
    size_t total;
};

bool hits_layout(const DevInfo &di, long long n_qprot, long long n_dbprot, int d, int cap, long long nq,
                 HitsLayout *l) {
    if (!make_config(di, nq, (n_dbprot + 31) / 32, d, cap, &l->scan)) return false;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += dctd::align_up(bytes, 256); return o; };
    l->off_packed = take((size_t)((n_dbprot + 31) / 32) * 32 * chunks_of(d) * 16);
    l->off_dbe = take((size_t)n_dbprot);
    l->off_qoff = take(((size_t)n_qprot + 1) * sizeof(long long));
    l->off_doff = take(((size_t)n_dbprot + 1) * sizeof(long long));
    const size_t list = (size_t)nq * (size_t)cap * 8;
    l->off_q = take((size_t)nq * d);
    l->off_qe = take((size_t)nq);
    l->off_cnt = take((size_t)nq * sizeof(int));
    l->off_parts = take((size_t)l->scan.splits * list);
    l->off_keys = take(list);
    l->off_tmp = take(l->scan.splits > kMergePPW ? (size_t)((l->scan.splits + kMergePPW - 1) / kMergePPW) * list : 0);
    l->total = off + 256;
    return true;
}

// the largest chunk of at most `want` query proteins whose buffers fit in `bytes` (0: not even one)
long long hits_fit(const DevInfo &di, long long n_qprot, long long n_dbprot, int d, int cap, long long want,
                   size_t bytes, HitsLayout *l) {
    long long nq = std::min(want, kHitsMaxChunk);
    while (nq > 0) {
        if (hits_layout(di, n_qprot, n_dbprot, d, cap, nq, l) && l->total <= bytes) return nq;
        nq /= 2;
    }
    return 0;
}

int run_hits(const int8_t *d_qf, const int64_t *h_qoff, long long n_qprot, const int8_t *d_dbf, const int64_t *h_doff,
             long long n_dbprot, int d, int top, int dist_clamp, int dist_cut, int cap, int *d_count, int *d_hit_db,
             int *d_hit_min, int *d_hit_last, void *d_workspace, size_t workspace_bytes, cudaStream_t stream) {
    DevInfo di;
    dev_info(&di);
    HitsLayout l;
    if (!hits_layout(di, n_qprot, n_dbprot, d, cap, 1, &l)) return DCTD_ERR_UNSUPPORTED;
    if (!d_workspace || hits_fit(di, n_qprot, n_dbprot, d, cap, n_qprot, workspace_bytes, &l) == 0)
        return DCTD_ERR_WORKSPACE;
    if (((uintptr_t)d_workspace & 255) != 0) return DCTD_ERR_ARG;
    char *ws = (char *)d_workspace;
    const long long *qoff = (const long long *)(ws + l.off_qoff), *doff = (const long long *)(ws + l.off_doff);
    uint4 *packed = (uint4 *)(ws + l.off_packed);
    unsigned char *dbe = (unsigned char *)(ws + l.off_dbe);
    DCTD_CUDA_TRY(cudaMemcpyAsync(ws + l.off_qoff, h_qoff, ((size_t)n_qprot + 1) * sizeof(long long), cudaMemcpyHostToDevice, stream));
    DCTD_CUDA_TRY(cudaMemcpyAsync(ws + l.off_doff, h_doff, ((size_t)n_dbprot + 1) * sizeof(long long), cudaMemcpyHostToDevice, stream));
    const int block = 256;
    if (n_dbprot > 0) {
        const long long total = (n_dbprot + 31) / 32 * 32 * chunks_of(d);
        const int grid = (int)std::min<long long>((total + block - 1) / block, di.sms * 16);
        hits_pack_globals_kernel<<<grid, block, 0, stream>>>(d_dbf, d, doff, n_dbprot, packed, dbe);
        DCTD_LAUNCH_CHECK();
    }
    const int top_ = (int)std::min<long long>(std::max(top, 0), n_dbprot);
    const bool vec16 = d % 16 == 0 && ((uintptr_t)d_qf & 15) == 0 && ((uintptr_t)d_dbf & 15) == 0;
    for (long long a0 = 0; a0 < n_qprot;) {
        const long long nq = hits_fit(di, n_qprot, n_dbprot, d, cap, n_qprot - a0, workspace_bytes, &l);
        if (nq == 0) return DCTD_ERR_WORKSPACE;
        int *ncut = (int *)(ws + l.off_cnt);
        unsigned long long *keys = (unsigned long long *)(ws + l.off_keys);
        DCTD_CUDA_TRY(cudaMemsetAsync(ncut, 0, (size_t)nq * sizeof(int), stream));
        if (n_dbprot > 0) {
            int8_t *q = (int8_t *)(ws + l.off_q);
            unsigned char *qe = (unsigned char *)(ws + l.off_qe);
            const int grid = (int)std::min<long long>((nq * d + block - 1) / block, di.sms * 16);
            hits_gather_queries_kernel<<<grid, block, 0, stream>>>(d_qf, d, qoff, a0, nq, q, qe);
            DCTD_LAUNCH_CHECK();
            ScanParams sp{};
            sp.q = q; sp.packed = packed; sp.nq = nq; sp.n = n_dbprot; sp.d = d; sp.k = cap; sp.gstride = 1;
            sp.parts = (unsigned long long *)(ws + l.off_parts);
            sp.cap = l.scan.cap; sp.n_groups = l.scan.n_groups; sp.groups_per_split = l.scan.groups_per_split;
            ClampedKey key{(unsigned int)dist_clamp, dist_cut, qe, dbe, ncut};
            if (l.scan.n_qtiles > 65535) return DCTD_ERR_UNSUPPORTED;
            HitsScanFn fn = hits_kernel(l.scan);
            DCTD_CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l.scan.smem));
            fn<<<dim3((unsigned)l.scan.splits, (unsigned)l.scan.n_qtiles), (kWarps + 1) * 32, l.scan.smem, stream>>>(sp, key);
            DCTD_LAUNCH_CHECK();
            const int rc = run_merge(sp.parts, l.scan.splits, nq, cap, 0, nullptr, nullptr, keys, nullptr,
                                     (unsigned long long *)(ws + l.off_tmp), stream);
            if (rc != DCTD_OK) return rc;
        }
        HitsOut o{};
        o.keys = keys; o.ncut = ncut; o.nq = nq; o.a0 = a0; o.cap = cap; o.top = top_;
        o.qf = d_qf; o.dbf = d_dbf; o.qoff = qoff; o.doff = doff; o.d = d;
        o.count = d_count; o.hit_db = d_hit_db; o.hit_min = d_hit_min; o.hit_last = d_hit_last;
        const unsigned grid = (unsigned)((nq * cap + 3) / 4);
        if (vec16) hits_output_kernel<true><<<grid, 128, 0, stream>>>(o);
        else hits_output_kernel<false><<<grid, 128, 0, stream>>>(o);
        DCTD_LAUNCH_CHECK();
        a0 += nq;
    }
    return DCTD_OK;
}
