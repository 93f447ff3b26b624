// libdctd hot path 2: exhaustive int8 L1 top-k for sm_100a.
//
// Stands in for faiss IndexFlat + METRIC_L1 `index.search(x, k)` as called by the reference
// (src/query_db.py:75-76,87; bench/cathdb/run_dct.py:51-60) on the flat index built at
// src/database.py:240-243, and for the pairwise scorer of src/dct-sim.py:12-50.
// Semantics: per query the k smallest database positions by (L1 distance, position), ascending,
// padded with (FLT_MAX, -1).
//
// Design
//   * The database lives on the device as int8 (the reference's fingerprints ARE int8; faiss
//     widens them to float32, 4x the bytes) in a packed layout: groups of 32 vectors interleaved
//     in 16-byte chunks, bytes XOR 0x80 so that an unsigned packed-byte SAD gives |a-b| for any
//     int8 pair.  A group tile is contiguous, so one TMA bulk copy (cp.async.bulk, mbarrier
//     completion) stages it in shared memory, and lane v of a warp reads vector v of the group
//     with conflict-free 16-byte shared loads.
//   * Distances: one VABSDIFF4.U8.ACC (__vsadu4) per 4 bytes per (query, vector) pair, register
//     tile of TQ queries x TD vectors per thread, queries broadcast from shared memory.
//   * Selection: 64-bit keys (dist << 40 | position) make (dist, position) order a plain integer
//     compare.  Each warp owns its queries' candidate buffers in shared memory: a candidate is
//     appended only if its key beats the query's current k-th key (warp ballot + prefix), and a
//     full buffer is re-sorted (bitonic, warp-synchronous) to tighten the threshold.
//   * The database is split over grid.x; per-split sorted lists meet in a merge kernel that also
//     converts to faiss' (float32 distance, int64 id) output.  The same merge kernel folds the
//     per-rank results of a sharded database after the NCCL all-gather.
#include <float.h>

#include <algorithm>
#include <mutex>
#include <new>
#include <vector>

#include "dctd_internal.cuh"
#include "dctd_tma.cuh"

namespace {

using namespace dctd::tma;

constexpr int kWarps = 8;            // warps per CTA of the scan kernel
constexpr int kTDmax = 2;            // database groups (of 32 vectors) per shared-memory stage (1 for wide d)
constexpr int kStagesMax = 4;        // TMA stages (2 for wide d)
constexpr int kIdBits = 40;          // key = dist << 40 | position
constexpr unsigned long long kKeyMax = ~0ULL;
constexpr unsigned long long kIdMask = (1ULL << kIdBits) - 1ULL;

__host__ __device__ inline int chunks_of(int d) { return (d + 15) / 16; }

// ------------------------------------------------------------------------------------------
// pack / unpack
// ------------------------------------------------------------------------------------------
__global__ void pack_kernel(const int8_t *__restrict__ rows, long long n, int d, long long n_offset,
                            uint4 *__restrict__ packed) {
    const int C = chunks_of(d);
    const long long v0 = n_offset / 32 * 32;                 // first vector of the first touched group
    const long long v1 = (n_offset + n + 31) / 32 * 32;      // end of the last touched group
    const long long total = (v1 - v0) * C;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const long long vec = v0 + t / C;
        const int c = (int)(t % C);
        if (vec < n_offset) continue;                        // already packed by an earlier add
        unsigned int w[4] = {0x80808080u, 0x80808080u, 0x80808080u, 0x80808080u};
        if (vec < n_offset + n) {
            const int8_t *src = rows + (vec - n_offset) * d + c * 16;
#pragma unroll
            for (int b = 0; b < 16; ++b) {
                const int col = c * 16 + b;
                const unsigned int byte = (col < d) ? ((unsigned int)(unsigned char)src[b] ^ 0x80u) : 0x80u;
                w[b >> 2] = (w[b >> 2] & ~(0xffu << ((b & 3) * 8))) | (byte << ((b & 3) * 8));
            }
        }
        const long long g = vec / 32;
        const int lane = (int)(vec % 32);
        packed[(g * C + c) * 32 + lane] = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

__global__ void unpack_kernel(const uint4 *__restrict__ packed, long long n, int d, int8_t *__restrict__ rows) {
    const int C = chunks_of(d);
    const long long total = n * C;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const long long vec = t / C;
        const int c = (int)(t % C);
        const uint4 q = packed[((vec / 32) * C + c) * 32 + (vec % 32)];
        const unsigned int w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int b = 0; b < 16; ++b) {
            const int col = c * 16 + b;
            if (col < d) rows[vec * d + col] = (int8_t)(((w[b >> 2] >> ((b & 3) * 8)) & 0xffu) ^ 0x80u);
        }
    }
}

// ------------------------------------------------------------------------------------------
// warp-synchronous bitonic sort of `cap` (power of two) keys in shared memory, ascending
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void warp_sort(unsigned long long *buf, int cap, int lane) {
    for (int k2 = 2; k2 <= cap; k2 <<= 1) {
        for (int j = k2 >> 1; j > 0; j >>= 1) {
            for (int i = lane; i < (cap >> 1); i += 32) {
                const int lo = ((i & ~(j - 1)) << 1) | (i & (j - 1));
                const int hi = lo | j;
                const bool up = (lo & k2) == 0;
                const unsigned long long a = buf[lo], b = buf[hi];
                if ((a > b) == up) { buf[lo] = b; buf[hi] = a; }
            }
            __syncwarp();
        }
    }
}

// sorts the `cnt` live keys of a candidate buffer, keeps the k best, returns the new count
__device__ __forceinline__ int warp_refine(unsigned long long *buf, int cnt, int cap, int k, int lane,
                                           unsigned long long *thr) {
    for (int i = cnt + lane; i < cap; i += 32) buf[i] = kKeyMax;
    __syncwarp();
    warp_sort(buf, cap, lane);
    const int keep = min(cnt, k);
    if (lane == 0) *thr = (keep == k) ? buf[k - 1] : kKeyMax;
    __syncwarp();
    return keep;
}

// acc + sum_i |a.byte[i] - b.byte[i]| (unsigned bytes): SASS VABSDIFF4.U8.ACC
__device__ __forceinline__ unsigned int sad4(unsigned int a, unsigned int b, unsigned int acc) {
    unsigned int r;
    asm("vabsdiff4.u32.u32.u32.add %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(acc));
    return r;
}


// bitonic merge of a bitonic sequence of `cap` keys (first half ascending, second half descending)
__device__ __forceinline__ void warp_bitonic_merge(unsigned long long *buf, int cap, int lane) {
    for (int j = cap >> 1; j > 0; j >>= 1) {
        for (int i = lane; i < (cap >> 1); i += 32) {
            const int lo = ((i & ~(j - 1)) << 1) | (i & (j - 1));
            const int hi = lo | j;
            const unsigned long long a = buf[lo], b = buf[hi];
            if (a > b) { buf[lo] = b; buf[hi] = a; }
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------
// TMA-staged, warp-specialised SAD scan shared by the two scan kernels
//   warp NW is the producer (one elected lane issues cp.async.bulk), warps 0..NW-1 compute;
//   stages are handed over with full/empty mbarriers so compute warps never meet at a CTA barrier.
// ------------------------------------------------------------------------------------------
struct ScanParams {
    const int8_t *q;            // [nq, d] row-major
    const uint4 *packed;        // packed database
    long long nq, n;
    int d, k;
    long long n_groups;         // groups visited (virtual index v; real group = v * gstride)
    long long gstride;          // 1 = every group, s = every s-th group (threshold sample)
    long long skip;             // s > 1: visit every group EXCEPT every s-th one (the sample was scored already);
                                // virtual index v -> real group v + v / (s - 1) + 1.  0 = off
    long long groups_per_split;
    const int *qflags;          // optional [nq]: only query tiles with a flagged query are processed
    // heap mode (l1_scan_kernel)
    unsigned long long *parts;  // [S, nq, k] sorted keys per database split
    int cap;
    // threshold mode (l1_thresh_scan_kernel / l1_thresh_stream_kernel)
    const unsigned int *thr_dist;         // [nq] distance bound per query: only vectors with dist <= thr_dist[q] are kept
                                          // (an upper bound of the true k-th best distance; >= 0x7fffffff = no bound)
    unsigned long long *cand;   // [nq, cmax] candidate keys
    int *cnt;                   // [nq] candidates appended (may exceed cmax: overflow)
    int cmax;
};

// real group of virtual group v (see ScanParams::gstride / skip)
__device__ __forceinline__ long long real_group(const ScanParams &p, long long v) {
    return p.skip ? v + v / (p.skip - 1) + 1 : v * p.gstride;
}

template <int NW, int TQ>
__device__ __forceinline__ void load_queries(const ScanParams &p, unsigned char *qs, long long q0, int dpad) {
    constexpr int QT = NW * TQ;
    // biased by 0x80; zero-distance padding beyond d / nq
    if ((p.d & 15) == 0 && (reinterpret_cast<unsigned long long>(p.q) & 15ULL) == 0ULL) {
        // 16 bytes per thread and step (a byte-wise loop over 128 queries x 480 bytes took a CTA 23 us)
        const int C = dpad >> 4;
        const uint4 *src = reinterpret_cast<const uint4 *>(p.q);
        uint4 *dst = reinterpret_cast<uint4 *>(qs);
        for (int i = threadIdx.x; i < QT * C; i += blockDim.x) {
            const int qi = i / C, c = i - qi * C;
            uint4 v = make_uint4(0x80808080u, 0x80808080u, 0x80808080u, 0x80808080u);
            if (q0 + qi < p.nq) {
                const uint4 r = src[(q0 + qi) * C + c];
                v = make_uint4(r.x ^ 0x80808080u, r.y ^ 0x80808080u, r.z ^ 0x80808080u, r.w ^ 0x80808080u);
            }
            dst[i] = v;
        }
        return;
    }
    for (int i = threadIdx.x; i < QT * dpad; i += blockDim.x) {
        const int qi = i / dpad, col = i % dpad;
        unsigned char b = 0x80;
        if (q0 + qi < p.nq && col < p.d) b = (unsigned char)p.q[(q0 + qi) * p.d + col] ^ 0x80;
        qs[i] = b;
    }
}

template <int kTD, int STAGES>
__device__ __forceinline__ void producer_loop(const ScanParams &p, unsigned long long *full, unsigned long long *empty,
                                              unsigned char *st, int tile_bytes, int C, int dpad,
                                              long long g_begin, long long g_end, int n_tiles) {
    for (int t = 0; t < n_tiles; ++t) {
        const int s = t % STAGES;
        if (t >= STAGES) mbar_wait_backoff(&empty[s], (unsigned int)(((t / STAGES) - 1) & 1));
        const long long v = g_begin + (long long)t * kTD;
        const int ng = (int)min((long long)kTD, g_end - v);
        const unsigned int gbytes = 32u * (unsigned int)dpad;
        mbar_expect_tx(&full[s], (unsigned int)ng * gbytes);
        const long long g0 = real_group(p, v);
        if (real_group(p, v + ng - 1) == g0 + ng - 1) {      // the tile's groups are adjacent: one copy
            bulk_g2s(st + (size_t)s * tile_bytes, p.packed + g0 * C * 32, (unsigned int)ng * gbytes, &full[s]);
        } else {
            for (int b = 0; b < ng; ++b)
                bulk_g2s(st + (size_t)s * tile_bytes + (size_t)b * gbytes, p.packed + real_group(p, v + b) * C * 32,
                         gbytes, &full[s]);
        }
    }
}

// distances of this warp's TQ queries against lane's vector of each of the kTD groups of one stage
// CT: compile-time chunk count (d = 16 CT; 30 for the reference's 480-byte fingerprints) - the chunk loop is then fully
// unrolled and every shared-memory address is base + immediate: the address increments of the rolled loop run on the
// same ALU pipe as the SADs (5 % of its slots).  CT = 0: runtime C.
template <int TQ, int kTD, int CT = 0>
__device__ __forceinline__ void sad_tile(const uint4 *st4, const uint4 *qs4, int C_, int lane,
                                         unsigned int (&acc)[TQ][kTD]) {
    const int C = CT ? CT : C_;
#pragma unroll
    for (int a = 0; a < TQ; ++a)
#pragma unroll
        for (int b = 0; b < kTD; ++b) acc[a][b] = 0u;
#pragma unroll(CT ? CT : 2)
    for (int c = 0; c < C; ++c) {
        uint4 dv[kTD], qv[TQ];
#pragma unroll
        for (int b = 0; b < kTD; ++b) dv[b] = st4[(b * C + c) * 32 + lane];
#pragma unroll
        for (int a = 0; a < TQ; ++a) qv[a] = qs4[a * C + c];
        // word-major order: TQ*kTD independent accumulators between two updates of the same one
#pragma unroll
        for (int a = 0; a < TQ; ++a)
#pragma unroll
            for (int b = 0; b < kTD; ++b) acc[a][b] = sad4(qv[a].x, dv[b].x, acc[a][b]);
#pragma unroll
        for (int a = 0; a < TQ; ++a)
#pragma unroll
            for (int b = 0; b < kTD; ++b) acc[a][b] = sad4(qv[a].y, dv[b].y, acc[a][b]);
#pragma unroll
        for (int a = 0; a < TQ; ++a)
#pragma unroll
            for (int b = 0; b < kTD; ++b) acc[a][b] = sad4(qv[a].z, dv[b].z, acc[a][b]);
#pragma unroll
        for (int a = 0; a < TQ; ++a)
#pragma unroll
            for (int b = 0; b < kTD; ++b) acc[a][b] = sad4(qv[a].w, dv[b].w, acc[a][b]);
    }
}

__device__ __forceinline__ bool tile_has_flag(const ScanParams &p, long long q0, int QT, int *s_any) {
    if (threadIdx.x == 0) *s_any = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < QT; i += blockDim.x)
        if (q0 + i < p.nq && p.qflags[q0 + i]) *s_any = 1;
    __syncthreads();
    return *s_any != 0;
}

// ------------------------------------------------------------------------------------------
// heap scan: exact top-k with warp-private candidate buffers (any database size; also computes the
// threshold sample and the fallback for queries whose candidate list overflowed)
// ------------------------------------------------------------------------------------------
// Key policy of the heap scan.  The search orders by the plain key dist << 40 | position; a policy with kClamped set
// (ClampedKey, l1_hits.cuh) rewrites each tile's distances before selection and counts the keys within a cut.
struct PlainKey {
    static constexpr bool kClamped = false;
};

template <int TQ, int kTD, int STAGES, class Key>
__device__ __forceinline__ void heap_scan(const ScanParams &p, const Key &key) {
    constexpr int QT = kWarps * TQ;
    // no static shared memory: make_config gives the dynamic part everything up to the opt-in limit (d = 833..848 leaves
    // 96 B), and even one static int takes 128 B next to the 128-B aligned dynamic array
    extern __shared__ __align__(128) unsigned char smem[];
    const int C = chunks_of(p.d);
    const int dpad = C * 16;
    const int tile_bytes = kTD * 32 * dpad;
    unsigned long long *full = reinterpret_cast<unsigned long long *>(smem);           // [STAGES]
    unsigned long long *empty = full + STAGES;                                          // [STAGES]
    int *s_any = reinterpret_cast<int *>(empty + STAGES);                               // tile_has_flag
    unsigned char *qs = smem + 128;                                                     // [QT][dpad]
    unsigned char *st = qs + (size_t)QT * dpad;                                         // [STAGES][tile]
    unsigned long long *buf = reinterpret_cast<unsigned long long *>(st + (size_t)STAGES * tile_bytes);
    unsigned long long *thr = buf + (size_t)QT * p.cap;                                 // [QT]
    int *cnt = reinterpret_cast<int *>(thr + QT);                                       // [QT]

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
    for (int i = tid; i < QT; i += blockDim.x) { thr[i] = kKeyMax; cnt[i] = 0; }
    __syncthreads();

    if (warp == kWarps) {
        if (lane == 0) producer_loop<kTD, STAGES>(p, full, empty, st, tile_bytes, C, dpad, g_begin, g_end, n_tiles);
        return;
    }

    const uint4 *qs4 = reinterpret_cast<const uint4 *>(qs) + (size_t)warp * TQ * C;
    unsigned long long *wbuf = buf + (size_t)warp * TQ * p.cap;
    unsigned long long *wthr = thr + warp * TQ;
    int *wcnt = cnt + warp * TQ;
    unsigned int tdist[TQ];      // distance part of each query's current k-th key (fast reject)
#pragma unroll
    for (int a = 0; a < TQ; ++a) tdist[a] = 0xffffffffu;
    unsigned int ncut[TQ];       // kClamped: keys within key.cut that this lane saw
    bool qempty[TQ];
    if constexpr (Key::kClamped) {
#pragma unroll
        for (int a = 0; a < TQ; ++a) {
            const long long qi = q0 + warp * TQ + a;
            ncut[a] = 0u;
            qempty[a] = qi >= p.nq || key.q_empty[qi];
        }
    }

    for (int t = 0; t < n_tiles; ++t) {
        const int s = t % STAGES;
        mbar_wait(&full[s], (unsigned int)((t / STAGES) & 1));
        unsigned int acc[TQ][kTD];
        sad_tile<TQ, kTD>(reinterpret_cast<const uint4 *>(st + (size_t)s * tile_bytes), qs4, C, lane, acc);
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);     // this warp no longer reads the stage
        if constexpr (Key::kClamped) key.template adjust<TQ, kTD>(p, acc, qempty, ncut, g_begin + (long long)t * kTD, g_end, lane);

        // ---- candidate filter (warp-private buffers: no CTA-level synchronisation) ----
        bool hit = false;
#pragma unroll
        for (int a = 0; a < TQ; ++a)
#pragma unroll
            for (int b = 0; b < kTD; ++b) hit = hit || (acc[a][b] <= tdist[a]);
        if (!__any_sync(0xffffffffu, hit)) continue;          // common case once thresholds are tight
        const long long vbase = g_begin + (long long)t * kTD;
#pragma unroll
        for (int a = 0; a < TQ; ++a) {
#pragma unroll
            for (int b = 0; b < kTD; ++b) {
                const long long id = real_group(p, vbase + b) * 32 + lane;
                const bool valid = (vbase + b) < g_end && id < p.n;
                const unsigned long long key = ((unsigned long long)acc[a][b] << kIdBits) | (unsigned long long)id;
                const bool pass = valid && key < wthr[a];
                const unsigned int vote = __ballot_sync(0xffffffffu, pass);
                if (vote) {
                    int cn = wcnt[a];
                    if (cn + 32 > p.cap) cn = warp_refine(wbuf + (size_t)a * p.cap, cn, p.cap, p.k, lane, &wthr[a]);
                    // keys that stopped passing after a refine are harmless: they sort behind the k-th key
                    if (pass) wbuf[(size_t)a * p.cap + cn + __popc(vote & ((1u << lane) - 1u))] = key;
                    __syncwarp();
                    if (lane == 0) wcnt[a] = cn + __popc(vote);
                    __syncwarp();
                }
            }
            const unsigned long long th = wthr[a];
            tdist[a] = (th == kKeyMax) ? 0xffffffffu : (unsigned int)(th >> kIdBits);
        }
    }

    // ---- final: sort each query's candidates and publish the k best keys of this split ----
    for (int a = 0; a < TQ; ++a) {
        const long long qi = q0 + warp * TQ + a;
        unsigned long long *b = wbuf + (size_t)a * p.cap;
        const int keep = warp_refine(b, wcnt[a], p.cap, p.k, lane, &wthr[a]);
        if (qi < p.nq) {
            unsigned long long *out = p.parts + ((long long)blockIdx.x * p.nq + qi) * p.k;
            for (int i = lane; i < p.k; i += 32) out[i] = (i < keep) ? b[i] : kKeyMax;
        }
    }
    if constexpr (Key::kClamped) key.template publish<TQ>(ncut, q0 + warp * TQ, p.nq, lane);
}

template <int TQ, int kTD, int STAGES>
__global__ void __launch_bounds__((kWarps + 1) * 32, 1) l1_scan_kernel(const ScanParams p) {
    heap_scan<TQ, kTD, STAGES>(p, PlainKey{});
}

// ------------------------------------------------------------------------------------------
// Thresholds for the streaming regime (nq <= 16) without a heap scan: every `red` adjacent lanes keep the
// smallest distance they have seen per query over the sampled groups (every gstride-th group, direct
// coalesced loads as in l1_thresh_stream_kernel).  Each of these M minima is the distance of a distinct real
// vector, so the k-th smallest of them is >= the true k-th best distance: a valid threshold, and with M >> k
// almost the k-th best of the sample itself.  l1_kth_kernel sorts the M <= 4096 values per query in shared
// memory and writes the threshold key.
// ------------------------------------------------------------------------------------------
constexpr int kMinSlots = 4096;      // minima per query

template <int TQ>
__global__ void __launch_bounds__(128) l1_sample_min_kernel(const ScanParams p, unsigned int *mins, int red) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int C = chunks_of(p.d);
    const int dpad = C * 16;
    unsigned char *qs = smem;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    load_queries<1, TQ>(p, qs, 0, dpad);
    __syncthreads();
    const uint4 *qs4 = reinterpret_cast<const uint4 *>(qs);
    unsigned int best[TQ];
#pragma unroll
    for (int a = 0; a < TQ; ++a) best[a] = 0xffffffffu;
    constexpr int UC = 6;
    const long long W = (long long)gridDim.x * (blockDim.x >> 5);
    const long long gw = (long long)blockIdx.x * (blockDim.x >> 5) + warp;
    for (long long v = gw; v < p.n_groups; v += W) {          // n_groups = sampled groups here
        const long long g = v * p.gstride;
        const uint4 *gp = p.packed + g * C * 32 + lane;
        unsigned int acc[TQ];
#pragma unroll
        for (int a = 0; a < TQ; ++a) acc[a] = 0u;
        for (int c0 = 0; c0 < C; c0 += UC) {
            uint4 dv[UC];
#pragma unroll
            for (int u = 0; u < UC; ++u) {
                dv[u] = make_uint4(0x80808080u, 0x80808080u, 0x80808080u, 0x80808080u);
                if (c0 + u < C) {
                    const uint4 *src = gp + (size_t)(c0 + u) * 32;
                    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                                 : "=r"(dv[u].x), "=r"(dv[u].y), "=r"(dv[u].z), "=r"(dv[u].w)
                                 : "l"(src));
                }
            }
#pragma unroll
            for (int u = 0; u < UC; ++u) {
                if (c0 + u < C) {
#pragma unroll
                    for (int a = 0; a < TQ; ++a) {
                        const uint4 qv = qs4[a * C + c0 + u];
                        unsigned int sacc = acc[a];
                        sacc = sad4(qv.x, dv[u].x, sacc);
                        sacc = sad4(qv.y, dv[u].y, sacc);
                        sacc = sad4(qv.z, dv[u].z, sacc);
                        sacc = sad4(qv.w, dv[u].w, sacc);
                        acc[a] = sacc;
                    }
                }
            }
        }
        if (g * 32 + lane < p.n) {          // the padding lanes of the last group are not vectors
#pragma unroll
            for (int a = 0; a < TQ; ++a) best[a] = min(best[a], acc[a]);
        }
    }
    // minimum over each run of `red` adjacent lanes (red = 1, 2, .., 32), one value per run
    for (int o = 1; o < red; o <<= 1) {
#pragma unroll
        for (int a = 0; a < TQ; ++a) best[a] = min(best[a], __shfl_xor_sync(0xffffffffu, best[a], o));
    }
    if ((lane & (red - 1)) == 0) {
        const long long slot = gw * (32 / red) + lane / red;
        if (slot < kMinSlots) {
#pragma unroll
            for (int a = 0; a < TQ; ++a)
                if (a < p.nq) mins[(long long)a * kMinSlots + slot] = best[a];
        }
    }
}

// one CTA per query: k-th smallest of the M minima -> thr_dist[q] (ties at the bound pass the scan)
__global__ void __launch_bounds__(256) l1_kth_kernel(const unsigned int *mins, int M, int k, unsigned int *thr_dist,
                                                     int *cnt) {
    __shared__ unsigned int v[kMinSlots];
    const long long qi = blockIdx.x;
    int P = 64;
    while (P < M) P <<= 1;
    for (int i = threadIdx.x; i < P; i += blockDim.x) v[i] = (i < M) ? mins[qi * kMinSlots + i] : 0xffffffffu;
    __syncthreads();
    for (int k2 = 2; k2 <= P; k2 <<= 1) {
        for (int j = k2 >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < (P >> 1); i += blockDim.x) {
                const int lo = ((i & ~(j - 1)) << 1) | (i & (j - 1));
                const int hi = lo | j;
                const bool up = (lo & k2) == 0;
                const unsigned int a = v[lo], b = v[hi];
                if ((a > b) == up) { v[lo] = b; v[hi] = a; }
            }
            __syncthreads();
        }
    }
    if (threadIdx.x == 0) {
        cnt[qi] = 0;                        // candidate counter of the scan that follows
        thr_dist[qi] = (k <= M) ? v[k - 1] : 0xffffffffu;
    }
}

// ------------------------------------------------------------------------------------------
// The sample's exact top-k (sorted keys, kKeyMax padding) become the first candidates of every query, so the
// threshold scan can leave the sampled groups out: a sampled vector beyond its sample's k-th key cannot be among
// the k best overall.  One warp per query; also sets the candidate counter (no memset).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) l1_seed_kernel(const unsigned long long *thr_keys, long long nq, int k,
                                                      unsigned long long *cand, int *cnt, int cmax, bool seed,
                                                      unsigned int *thr_dist) {
    const int lane = threadIdx.x & 31;
    const long long qi = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (qi >= nq) return;
    int valid = 0;
    if (seed) {
        for (int i = lane; i < k; i += 32) {
            const unsigned long long key = thr_keys[qi * k + i];
            if (key != kKeyMax) {            // keys are sorted: the valid ones are a prefix
                cand[qi * cmax + i] = key;
                ++valid;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) valid += __shfl_xor_sync(0xffffffffu, valid, o);
    }
    if (lane == 0) {
        cnt[qi] = valid;
        const unsigned long long kth = thr_keys[qi * k + k - 1];
        thr_dist[qi] = (kth == kKeyMax) ? 0xffffffffu : (unsigned int)(kth >> kIdBits);
    }
}

// ------------------------------------------------------------------------------------------
// threshold scan: every vector whose distance is <= the query's threshold (k-th best of a sample of
// the database, an upper bound of the true k-th best) is appended to the query's candidate list in
// global memory.  No per-warp selection state: the scan is SADs + one compare per pair.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void append_candidates(const ScanParams &p, long long qi, bool pass,
                                                  unsigned long long key, int lane) {
    const unsigned int vote = __ballot_sync(0xffffffffu, pass);
    if (!vote) return;
    int base = 0;
    if (lane == 0) base = atomicAdd(&p.cnt[qi], __popc(vote));
    base = __shfl_sync(0xffffffffu, base, 0);
    const int slot = base + __popc(vote & ((1u << lane) - 1u));
    if (pass && slot < p.cmax) p.cand[qi * p.cmax + slot] = key;
}

template <int NW, int TQ, int kTD, int STAGES, int CT = 0>
__global__ void __launch_bounds__((NW + 1) * 32, 1) l1_thresh_scan_kernel(const ScanParams p) {
    constexpr int QT = NW * TQ;
    extern __shared__ __align__(128) unsigned char smem[];
    const int C = chunks_of(p.d);
    const int dpad = C * 16;
    const int tile_bytes = kTD * 32 * dpad;
    unsigned long long *full = reinterpret_cast<unsigned long long *>(smem);
    unsigned long long *empty = full + STAGES;
    unsigned char *qs = smem + 128;
    unsigned char *st = qs + (size_t)QT * dpad;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long q0 = (long long)blockIdx.y * QT;
    const long long g_begin = (long long)blockIdx.x * p.groups_per_split;
    const long long g_end = min(p.n_groups, g_begin + p.groups_per_split);
    const int n_tiles = (int)((g_end - g_begin + kTD - 1) / kTD);

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], NW); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    load_queries<NW, TQ>(p, qs, q0, dpad);
    __syncthreads();

    if (warp == NW) {
        if (lane == 0) producer_loop<kTD, STAGES>(p, full, empty, st, tile_bytes, C, dpad, g_begin, g_end, n_tiles);
        return;
    }
    const uint4 *qs4 = reinterpret_cast<const uint4 *>(qs) + (size_t)warp * TQ * C;
    unsigned int tdist[TQ];
#pragma unroll
    for (int a = 0; a < TQ; ++a) {
        const long long qi = q0 + warp * TQ + a;
        tdist[a] = (qi < p.nq) ? p.thr_dist[qi] : 0u;
    }
    // real group of the tile's first virtual group, kept up without a division per tile: with `skip`, virtual group
    // v = vq * (skip - 1) + vr is real group v + vq + 1
    const long long sk1 = p.skip ? p.skip - 1 : 1;
    long long vq = p.skip ? g_begin / sk1 : 0;
    int vr = p.skip ? (int)(g_begin % sk1) : 0;
    for (int t = 0; t < n_tiles; ++t) {
        const int s = t % STAGES;
        mbar_wait(&full[s], (unsigned int)((t / STAGES) & 1));
        unsigned int acc[TQ][kTD];
        sad_tile<TQ, kTD, CT>(reinterpret_cast<const uint4 *>(st + (size_t)s * tile_bytes), qs4, C, lane, acc);
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);
        const long long vbase = g_begin + (long long)t * kTD;
        long long greal[kTD];
#pragma unroll
        for (int b = 0; b < kTD; ++b)
            greal[b] = p.skip ? (vbase + b) + vq + ((vr + b >= sk1) ? 1 : 0) + 1 : (vbase + b) * p.gstride;
        vr += kTD;
        if (p.skip && vr >= sk1) { vr -= (int)sk1; ++vq; }
        // one bit per (query, group) pair with a lane within the threshold, OR-ed over the warp in one REDUX: the
        // compares and this reduction are all the selection work of a tile unless something passes, and then only the
        // pairs that do pass are visited (these instructions share the ALU pipe with the SADs)
        unsigned int mask = 0u;
#pragma unroll
        for (int a = 0; a < TQ; ++a)
#pragma unroll
            for (int b = 0; b < kTD; ++b) mask |= (acc[a][b] <= tdist[a]) ? (1u << (a * kTD + b)) : 0u;
        const unsigned int any = __reduce_or_sync(0xffffffffu, mask);
        if (!any) continue;
#pragma unroll
        for (int a = 0; a < TQ; ++a) {
#pragma unroll
            for (int b = 0; b < kTD; ++b) {
                if (any & (1u << (a * kTD + b))) {          // warp-uniform
                    const long long qi = q0 + warp * TQ + a;
                    const long long id = greal[b] * 32 + lane;
                    const bool pass = (vbase + b) < g_end && id < p.n && qi < p.nq && acc[a][b] <= tdist[a];
                    append_candidates(p, qi, pass, ((unsigned long long)acc[a][b] << kIdBits) | (unsigned long long)id, lane);
                }
            }
        }
    }
}

// Few queries (nq <= TQ): HBM-bound streaming.  Each warp takes whole groups straight from global memory
// (lane v reads vector v: every load instruction covers 512 contiguous bytes), no shared-memory staging.
// PIPE: two batches of chunks in flight per lane (measured: +5 % for <= 4 queries, where the kernel is purely HBM-bound;
// with 8 or 16 queries the extra registers cost more occupancy than the overlap inside a warp gains)
template <int TQ, bool PIPE = (TQ <= 4)>
__global__ void __launch_bounds__(128) l1_thresh_stream_kernel(const ScanParams p) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int C = chunks_of(p.d);
    const int dpad = C * 16;
    unsigned char *qs = smem;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    load_queries<1, TQ>(p, qs, 0, dpad);
    __syncthreads();
    const uint4 *qs4 = reinterpret_cast<const uint4 *>(qs);
    unsigned int tdist[TQ];
#pragma unroll
    for (int a = 0; a < TQ; ++a) {
        tdist[a] = (a < p.nq) ? p.thr_dist[a] : 0u;
    }
    constexpr int UC = 6;      // chunks per batch; with PIPE the next batch is requested before the current one is
                               // consumed, across group boundaries too: loads and SADs overlap inside a warp
    const long long W = (long long)gridDim.x * (blockDim.x >> 5);
    const long long g_first = (long long)blockIdx.x * (blockDim.x >> 5) + warp;
    const int nb = (C + UC - 1) / UC;                         // batches per group
    auto request = [&](long long g, int c0, uint4 (&dv)[UC]) {
        const uint4 *gp = p.packed + g * C * 32 + lane;
#pragma unroll
        for (int u = 0; u < UC; ++u) {
            dv[u] = make_uint4(0x80808080u, 0x80808080u, 0x80808080u, 0x80808080u);
            if (c0 + u < C) {
                const uint4 *src = gp + (size_t)(c0 + u) * 32;
                asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                             : "=r"(dv[u].x), "=r"(dv[u].y), "=r"(dv[u].z), "=r"(dv[u].w)
                             : "l"(src));
            }
        }
    };
    uint4 cur[UC], nxt[UC];
    if (PIPE && g_first < p.n_groups) request(g_first, 0, cur);
    for (long long g = g_first; g < p.n_groups; g += W) {
        unsigned int acc[TQ];
#pragma unroll
        for (int a = 0; a < TQ; ++a) acc[a] = 0u;
        for (int bi = 0; bi < nb; ++bi) {
            const int c0 = bi * UC;
            if (PIPE) {     // next batch: of this group, or the first one of this warp's next group
                if (bi + 1 < nb) request(g, c0 + UC, nxt);
                else if (g + W < p.n_groups) request(g + W, 0, nxt);
            } else {
                request(g, c0, cur);
            }
#pragma unroll
            for (int u = 0; u < UC; ++u) {
                if (c0 + u < C) {
#pragma unroll
                    for (int a = 0; a < TQ; ++a) {
                        const uint4 qv = qs4[a * C + c0 + u];
                        unsigned int s = acc[a];
                        s = sad4(qv.x, cur[u].x, s);
                        s = sad4(qv.y, cur[u].y, s);
                        s = sad4(qv.z, cur[u].z, s);
                        s = sad4(qv.w, cur[u].w, s);
                        acc[a] = s;
                    }
                }
            }
            if (PIPE) {
#pragma unroll
                for (int u = 0; u < UC; ++u) cur[u] = nxt[u];
            }
        }
        const long long id = g * 32 + lane;
        bool hit = false;
#pragma unroll
        for (int a = 0; a < TQ; ++a) hit = hit || (acc[a] <= tdist[a]);
        if (!__any_sync(0xffffffffu, hit)) continue;
#pragma unroll
        for (int a = 0; a < TQ; ++a) {
            const bool pass = id < p.n && a < p.nq && acc[a] <= tdist[a];
            append_candidates(p, a, pass, ((unsigned long long)acc[a] << kIdBits) | (unsigned long long)id, lane);
        }
    }
}

// exact selection from a query's candidate list: CTA-wide bitonic sort of up to cmax keys in shared memory
struct SelectParams {
    const unsigned long long *cand;
    const int *cnt;
    int cmax, k;
    long long nq, id_base;
    float *dist;
    long long *ids;
    unsigned long long *key_out;   // if set: the result stays packed keys (dist << 40 | id_base + position), kKeyMax padding
    int *qflags;       // out: 1 if the query's list overflowed (its result comes from the heap scan instead)
};

// Leaves the K2 = min(P, 2^ceil(log2 k)) smallest of the P keys (P a power of two >= 64) in keys[0..K2), ascending.
// Called by `nthr` threads that `sync()` joins (a whole CTA, or the consumer warps of the fused streaming kernel).
// Only the k smallest are wanted: bitonic-sort blocks of K2 keys (alternating directions), then fold pairs of
// blocks - the element-wise minimum of an ascending and a descending block holds the K2 smallest of both as a
// bitonic sequence, log2(K2) merge steps sort it again - until one ascending block is left.  ~14 P
// compare-exchanges instead of the ~33 P of a full sort of P = 2048 keys (the step is shared-memory bound).
template <typename Sync>
__device__ __forceinline__ int select_smallest(unsigned long long *keys, int P, int k, int tid, int nthr, Sync sync) {
    int K2 = 2;
    while (K2 < k) K2 <<= 1;
    if (K2 > P) K2 = P;
    for (int k2 = 2; k2 <= K2; k2 <<= 1) {
        for (int j = k2 >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < (P >> 1); i += nthr) {
                const int lo = ((i & ~(j - 1)) << 1) | (i & (j - 1));
                const int hi = lo | j;
                const bool up = (lo & k2) == 0;
                const unsigned long long a = keys[lo], b = keys[hi];
                if ((a > b) == up) { keys[lo] = b; keys[hi] = a; }
            }
            sync();
        }
    }
    // blocks live at multiples of `span`; block c (c-th survivor) is ascending for even c, descending for odd c
    for (int span = K2; span < P; span <<= 1) {
        const int nres = P / (2 * span);                        // surviving blocks after this round
        for (int i = tid; i < nres * K2; i += nthr) {
            const int c = i / K2, t = i % K2;
            unsigned long long *A = keys + (size_t)c * 2 * span;
            const unsigned long long a = A[t], b = A[span + t];
            A[t] = a < b ? a : b;
        }
        sync();
        for (int j = K2 >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < nres * (K2 >> 1); i += nthr) {
                const int c = i / (K2 >> 1), e = i % (K2 >> 1);
                unsigned long long *A = keys + (size_t)c * 2 * span;
                const int lo = ((e & ~(j - 1)) << 1) | (e & (j - 1));
                const int hi = lo | j;
                const bool up = (c & 1) == 0;
                const unsigned long long a = A[lo], b = A[hi];
                if ((a > b) == up) { A[lo] = b; A[hi] = a; }
            }
            sync();
        }
    }
    return K2;
}

// query qi's candidate list -> its k best (faiss' output or packed keys); lists that overflowed are flagged instead
template <typename Sync>
__device__ __forceinline__ void select_query(const SelectParams &p, long long qi, unsigned long long *keys, int tid,
                                             int nthr, Sync sync) {
    const int m = __ldcg(&p.cnt[qi]);
    if (m > p.cmax) {
        if (tid == 0) p.qflags[qi] = 1;
        return;
    }
    if (tid == 0) p.qflags[qi] = 0;
    int P = 64;
    while (P < m) P <<= 1;
    for (int i = tid; i < P; i += nthr) keys[i] = (i < m) ? __ldcg(&p.cand[qi * p.cmax + i]) : kKeyMax;
    sync();
    const int K2 = select_smallest(keys, P, p.k, tid, nthr, sync);
    for (int i = tid; i < p.k; i += nthr) {
        const unsigned long long key = (i < K2) ? keys[i] : kKeyMax;
        const long long o = qi * p.k + i;
        if (p.key_out) {
            p.key_out[o] = (key == kKeyMax) ? kKeyMax : key + (unsigned long long)p.id_base;
        } else if (key == kKeyMax) {
            p.dist[o] = FLT_MAX;
            p.ids[o] = -1;
        } else {
            p.dist[o] = (float)(unsigned int)(key >> kIdBits);
            p.ids[o] = (long long)(key & kIdMask) + p.id_base;
        }
    }
}

__global__ void __launch_bounds__(256) l1_select_kernel(const SelectParams p) {
    extern __shared__ __align__(16) unsigned long long keys[];
    select_query(p, blockIdx.x, keys, threadIdx.x, blockDim.x, [] { __syncthreads(); });
}

#include "l1_stream.cuh"

// ------------------------------------------------------------------------------------------
// merge kernel: sorted lists of k keys per (part, query) -> k best.  One warp per (query, chunk of
// `ppw` parts); each further list is folded in with a bitonic MERGE (log2(cap) steps), not a sort.
// Hierarchical: grid.y chunks write intermediate key lists; the last level converts to (float32, int64).
// ------------------------------------------------------------------------------------------
struct MergeParams {
    const unsigned long long *key_parts;   // [parts, nq, k] or null
    const float *dist_parts;               // [parts, nq, k] (PAIRS input)
    const long long *id_parts;
    int parts, ppw;
    long long nq;
    int k, cap;                            // cap = power of two >= 2k
    long long id_base;
    unsigned long long *key_out;           // [grid.y, nq, k] when not the last level (or keys wanted; with dist/ids set
                                           // as well, both forms are written)
    float *dist;
    long long *ids;
    const int *qflags;                     // optional: only flagged queries are written
};

template <bool PAIRS>
__global__ void __launch_bounds__(128) l1_merge_kernel(const MergeParams p) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long *buf = reinterpret_cast<unsigned long long *>(smem) + (size_t)warp * p.cap;
    const long long qi = (long long)blockIdx.x * (blockDim.x >> 5) + warp;
    if (qi >= p.nq) return;
    if (p.qflags && !p.qflags[qi]) return;
    const int p0 = blockIdx.y * p.ppw, p1 = min(p.parts, p0 + p.ppw);
    const int hcap = p.cap >> 1;
    auto load = [&](int part, int i) -> unsigned long long {
        if (i >= p.k) return kKeyMax;
        const long long o = ((long long)part * p.nq + qi) * p.k + i;
        if (!PAIRS) return p.key_parts[o];
        const long long id = p.id_parts[o];
        if (id < 0) return kKeyMax;
        return ((unsigned long long)(unsigned int)p.dist_parts[o] << kIdBits) | (unsigned long long)id;
    };
    for (int i = lane; i < hcap; i += 32) buf[i] = load(p0, i);
    for (int s = p0 + 1; s < p1; ++s) {
        for (int i = lane; i < hcap; i += 32) buf[p.cap - 1 - i] = load(s, i);   // reversed: bitonic sequence
        __syncwarp();
        warp_bitonic_merge(buf, p.cap, lane);
    }
    __syncwarp();
    if (p.key_out) {
        unsigned long long *out = p.key_out + ((long long)blockIdx.y * p.nq + qi) * p.k;
        for (int i = lane; i < p.k; i += 32) {
            const unsigned long long key = buf[i];
            out[i] = (key == kKeyMax) ? kKeyMax : key + (unsigned long long)p.id_base;   // id_base: last level only
        }
        if (!p.dist) return;
    }
    for (int i = lane; i < p.k; i += 32) {
        const unsigned long long key = buf[i];
        const long long o = qi * p.k + i;
        if (key == kKeyMax) {
            p.dist[o] = FLT_MAX;
            p.ids[o] = -1;
        } else {
            p.dist[o] = (float)(unsigned int)(key >> kIdBits);
            p.ids[o] = (long long)(key & kIdMask) + p.id_base;
        }
    }
}

#include "l1_protein.cuh"

// ------------------------------------------------------------------------------------------
// pairwise scorer (dct-sim.py:12-50): one warp per protein pair
// ------------------------------------------------------------------------------------------
// VEC16: d is a multiple of 16 and the rows are 16-byte aligned -> lane c reads chunk c of both fingerprints as one
// uint4 and takes four packed-byte SADs (bytes biased by 0x80 so that the unsigned SAD is |a - b| for int8)
// A pair with an empty side keeps INT32_MAX in both outputs, as dctd_l1_protein_scores and dctd_l1_protein_hits report it.
template <bool VEC16>
__global__ void pair_scores_kernel(const int8_t *__restrict__ fps, int d, const long long *__restrict__ off,
                                   const int *__restrict__ pa, const int *__restrict__ pb, long long n_pairs,
                                   int *__restrict__ min_dist, int *__restrict__ last_dist) {
    const int lane = threadIdx.x & 31;
    const long long pr = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (pr >= n_pairs) return;
    const long long a0 = off[pa[pr]], a1 = off[pa[pr] + 1], b0 = off[pb[pr]], b1 = off[pb[pr] + 1];
    int best = 0x7fffffff, last = 0x7fffffff;
    for (long long i = a0; i < a1; ++i)
        for (long long j = b0; j < b1; ++j) {
            int s = 0;
            if (VEC16) {
                const uint4 *ra = reinterpret_cast<const uint4 *>(fps + i * d);
                const uint4 *rb = reinterpret_cast<const uint4 *>(fps + j * d);
                unsigned int acc = 0u;
                for (int c = lane; c < (d >> 4); c += 32) {
                    const uint4 x = ra[c], y = rb[c];
                    acc = sad4(x.x ^ 0x80808080u, y.x ^ 0x80808080u, acc);
                    acc = sad4(x.y ^ 0x80808080u, y.y ^ 0x80808080u, acc);
                    acc = sad4(x.z ^ 0x80808080u, y.z ^ 0x80808080u, acc);
                    acc = sad4(x.w ^ 0x80808080u, y.w ^ 0x80808080u, acc);
                }
                s = (int)acc;
            } else {
                for (int c = lane; c < d; c += 32) s += abs((int)fps[i * d + c] - (int)fps[j * d + c]);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            best = min(best, s);
            last = s;
        }
    if (lane == 0) {
        min_dist[pr] = best;
        last_dist[pr] = last;
    }
}

// ------------------------------------------------------------------------------------------
// bound of a sharded search: the k_local-th best distance of a sample, as int32 (see dctd_l1_bound)
// ------------------------------------------------------------------------------------------
__global__ void l1_bound_kernel(const unsigned long long *keys, long long nq, int k, int *bound) {
    const long long qi = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (qi >= nq) return;
    const unsigned long long kth = keys[qi * k + k - 1];
    bound[qi] = (kth == kKeyMax) ? 0x7fffffff : (int)(kth >> kIdBits);
}

__global__ void l1_fill_kernel(int *p, long long n, int v) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// ------------------------------------------------------------------------------------------
// host-side configuration shared by workspace_bytes and topk
// ------------------------------------------------------------------------------------------
#ifdef DCTD_TUNING
int g_l1_var = 0;
int g_l1_mode = 0;   // A/B hook of the tuning build (dctd_l1_set_mode): 2 = heap-scan thresholds in the streaming
                     // regime, 3 = the threshold scan revisits the sampled groups, 5 = rolled chunk loop
#else
constexpr int g_l1_mode = 0;
#endif

// Limits of the current device (SM count, opt-in shared memory per CTA).  Device properties never change, so the
// per-device cache below is write-once.
struct DevInfo {
    long long sms;
    size_t smem;
    bool coop;       // cooperative launches (grid-wide barriers) supported
};

bool dev_info(DevInfo *out) {
    static std::mutex mu;
    static DevInfo cache[64];
    static bool have[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) {
        out->sms = 148;                       // no device (host-only callers sizing a workspace): B200 figures
        out->smem = 227 * 1024;
        out->coop = true;
        cudaGetLastError();
        return false;
    }
    std::lock_guard<std::mutex> lock(mu);
    if (!have[dev]) {
        int sms = 0, smem = 0, coop = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev) != cudaSuccess || sms < 1) {
            out->sms = 148;
            out->smem = 227 * 1024;
            out->coop = true;
            cudaGetLastError();
            return false;
        }
        cache[dev].sms = sms;
        cache[dev].smem = (size_t)smem;
        cache[dev].coop = coop != 0;
        have[dev] = true;
    }
    *out = cache[dev];
    return true;
}

constexpr int kCmax = 8192;  // candidate slots per query (threshold path)
constexpr size_t kCmaxBytes = (size_t)kCmax * 8;
constexpr int kMergePPW = 32;

struct ScanConfig {          // heap scan (l1_scan_kernel)
    int tq, td, stages, cap;
    long long n_qtiles, n_groups, splits, groups_per_split;
    size_t smem;
};

// One CTA per SM is resident (shared memory).  The number of database splits S trades whole waves of `sms`
// CTAs against per-CTA fixed cost: time(S) ~ waves(S) * (tiles_per_split + overhead_tiles), where
// overhead_tiles is the warm-up of a CTA expressed in tiles (heap scan: candidate buffers refine often
// until the thresholds tighten, ~32 tiles' worth; threshold scan: just the query load).
void pick_splits(long long sms, long long n_groups, int td, long long n_qtiles, int overhead_tiles, long long *splits,
                 long long *groups_per_split) {
    const long long tiles = std::max<long long>(1, (n_groups + td - 1) / td);
    const long long s_max = std::max<long long>(1, std::min<long long>(1024, tiles / 4));
    long long best_s = 1;
    double best_cost = 1e300;
    for (long long sp = 1; sp <= s_max; ++sp) {
        const long long tps = (tiles + sp - 1) / sp;
        const long long real = (tiles + tps - 1) / tps;
        const long long waves = (real * n_qtiles + sms - 1) / sms;
        const double cost = (double)waves * (double)(tps + overhead_tiles);
        if (cost < best_cost * 0.995) { best_cost = cost; best_s = sp; }
        if (sp > 4 * sms && sp * n_qtiles > 16 * sms) break;
    }
    const long long tiles_per_split = (tiles + best_s - 1) / best_s;
    *groups_per_split = tiles_per_split * td;
    *splits = std::max<long long>(1, (n_groups + *groups_per_split - 1) / *groups_per_split);
}

bool make_config(const DevInfo &di, long long nq, long long n_groups, int d, int k, ScanConfig *cfg) {
    if (k < 1 || k > 992 || d < 1 || d > 2048) return false;
    int cap = 128, tq = 8;
    if (k > 96) { cap = 256; tq = 4; }
    if (k > 224) { cap = 512; tq = 2; }
    if (k > 480) { cap = 1024; tq = 1; }
    while (tq > 1 && (long long)kWarps * (tq / 2) >= nq) tq /= 2;   // few queries: smaller tiles
    const int dpad = chunks_of(d) * 16;
    int td = kTDmax, stages = kStagesMax;
    auto smem_of = [&](int tq_, int td_, int st_) {
        const size_t qt = (size_t)kWarps * tq_;
        return (size_t)128 + qt * dpad + (size_t)st_ * td_ * 32 * dpad + qt * cap * 8 + qt * 12 + 64;
    };
    if (smem_of(1, td, stages) > di.smem) { td = 1; stages = 2; }      // wide vectors
    while (tq > 1 && smem_of(tq, td, stages) > di.smem) tq /= 2;
    if (smem_of(tq, td, stages) > di.smem) return false;
    cfg->tq = tq; cfg->td = td; cfg->stages = stages; cfg->cap = cap;
    cfg->smem = smem_of(tq, td, stages);
    cfg->n_qtiles = (nq + (long long)kWarps * tq - 1) / ((long long)kWarps * tq);
    cfg->n_groups = n_groups;
    pick_splits(di.sms, n_groups, td, cfg->n_qtiles, 32, &cfg->splits, &cfg->groups_per_split);
    return true;
}

struct ThreshConfig {        // threshold scan (l1_thresh_scan_kernel / l1_thresh_stream_kernel)
    bool stream;
    int nw, tq;              // compute warps per CTA, queries per warp (stream: tq = queries per pass)
    long long n_qtiles, splits, groups_per_split;
    size_t smem;
};

struct StreamCfg {           // fused streaming kernel (l1_stream_fused_kernel)
    bool ok;
    int tq, nw, td, nh, stages, kscr_n;      // queries per pass, consumer warps, groups per turn, parts per group, ring slots
    size_t smem;
};

// ring of as many group-sized stages as fit next to the queries and the k-th scratch; the consumers hold nw * td of
// them, the rest is in flight
StreamCfg stream_cfg(const DevInfo &di, long long nq, int d) {
    StreamCfg c{};
    c.tq = nq <= 4 ? 4 : (nq <= 8 ? 8 : (nq <= 12 ? 12 : 16));
    c.nw = 7;                // d = 480: 14 group slots, every warp owns two
    c.td = 1;
    c.nh = 1;
#ifdef DCTD_TUNING
    g_l1_var = 0;
    if (g_l1_mode == 6) { c.nw = 4; c.td = 2; }
    if (g_l1_mode == 7) { c.nw = 5; c.td = 2; }
    if (g_l1_mode == 8) { c.nw = 6; c.td = 2; }
    if (g_l1_mode == 16) { c.nw = 4; c.td = 2; g_l1_var = 1; }
    if (g_l1_mode == 17) { c.nw = 5; c.td = 2; g_l1_var = 1; }
    if (g_l1_mode == 26) { c.nw = 4; c.td = 2; g_l1_var = 2; }
    if (g_l1_mode == 27) { c.nw = 5; c.td = 2; g_l1_var = 2; }
#endif
    const size_t dpad = (size_t)chunks_of(d) * 16, pbytes = 32 * dpad / c.nh;
    for (;;) {
        c.kscr_n = (int)((std::min<long long>(di.sms * c.nw, kMinSlots) + 31) / 32 * 32);   // minima per query
        const size_t fixed = kStreamHeader + (size_t)c.tq * dpad + (size_t)c.kscr_n * sizeof(unsigned int);
        const size_t avail = di.smem - 1024;          // room for the kernel's static shared memory
        if (avail <= fixed) return c;
        const long long st = std::min<long long>(kStreamMaxSlots, (long long)((avail - fixed) / pbytes));
        const long long per_round = (long long)c.nw * c.td * c.nh;
        if (st < per_round + c.td * c.nh && c.nw > 1) {                     // wide vectors: fewer consumers
            c.nw = c.nw > 4 ? 4 : c.nw / 2;
            continue;
        }
        // the ring is also the buffer of the final selection: cmax candidates + kFastSortCap compacted keys
        if (st < per_round || kCmaxBytes + (size_t)kFastSortCap * 8 > (size_t)st * pbytes) return c;
        c.stages = (int)(st >= 2 * per_round ? st / per_round * per_round : st);   // whole rounds: fixed slot owners
        c.smem = fixed + (size_t)c.stages * pbytes;
        c.ok = di.coop;
        return c;
    }
}

struct TopkPlan {
    bool thresh;
    bool bounded;            // the caller supplies the distance bounds (sharded search): no sample, no seeds
    ScanConfig full;         // heap scan of the whole database: the only scan when !thresh, else the fallback
    ScanConfig samp;         // heap scan of the sample that sets the thresholds
    long long gstride;
    ThreshConfig tc;
    StreamCfg fused;         // tc.stream: the one-launch streaming kernel, when its ring fits
    int cmax;
    size_t off_parts_full, off_parts_samp, off_tmp, off_thr, off_thrd, off_ctl, off_cnt, off_flags, off_cand, off_mins, total;
    // streaming regime: thresholds from lane minima (l1_sample_min_kernel) instead of a heap scan of the sample
    long long samp_groups;   // sampled groups
    int samp_grid, samp_red, samp_m;   // CTAs of 4 warps, lanes per minimum, minima per query
};


constexpr long long kThreshMinN = 65536;    // smaller databases: heap scan only

// does a database of n vectors take the threshold path (and therefore honour an external bound)?
bool thresh_eligible(long long n, int k, const ScanConfig &full) {
    const long long gs = std::min<long long>(32, (kCmax / 4) / std::max(1, k));
    return n >= kThreshMinN && gs >= 8 && full.td == kTDmax;
}

bool make_plan(const DevInfo &di, long long nq, long long n, int d, int k, bool bounded, TopkPlan *pl) {
    const long long n_groups = (n + 31) / 32;
    if (!make_config(di, nq, n_groups, d, k, &pl->full)) return false;
    pl->thresh = false;
    pl->bounded = false;
    pl->fused = StreamCfg{};
    pl->cmax = kCmax;
    const int dpad = chunks_of(d) * 16;
    // threshold path: large databases, moderate k (the sample must stay a small fraction of the database
    // while the expected candidate count k * gstride stays well below cmax)
    const long long gs = std::min<long long>(32, (kCmax / 4) / std::max(1, k));
    if (thresh_eligible(n, k, pl->full)) {
        pl->gstride = gs;
        const long long sg = (n_groups + gs - 1) / gs;
        ThreshConfig tc{};
        if (nq <= 16) {
            tc.stream = true;
            tc.nw = 4;
            tc.tq = nq <= 4 ? 4 : (nq <= 8 ? 8 : 16);
            tc.n_qtiles = 1;
            tc.smem = (size_t)tc.tq * dpad;
            pl->fused = stream_cfg(di, nq, d);
        } else {
            tc.stream = false;
            tc.nw = nq >= 1024 ? 16 : 8;
            tc.tq = 8;
            while (tc.tq > 4 && (long long)tc.nw * (tc.tq / 2) >= nq) tc.tq /= 2;
            const size_t qt = (size_t)tc.nw * tc.tq;
            tc.smem = 128 + qt * dpad + (size_t)kStagesMax * kTDmax * 32 * dpad + 64;
            tc.n_qtiles = (nq + (long long)qt - 1) / (long long)qt;
            // own thresholds: the sampled groups are not scanned again (their top-k seeds the candidate lists)
            pick_splits(di.sms, (bounded || g_l1_mode == 3) ? n_groups : n_groups - sg, kTDmax, tc.n_qtiles, 2, &tc.splits,
                        &tc.groups_per_split);
        }
        if (tc.smem <= di.smem && (bounded || make_config(di, nq, sg, d, k, &pl->samp))) {
            pl->tc = tc;
            pl->thresh = true;
            pl->bounded = bounded;
        }
        if (pl->thresh && tc.stream && !bounded) {
            // one warp per sampled group up to 8 CTAs of 4 warps per SM; as many minima per query as fit
            pl->samp_groups = sg;
            const long long warps = std::min<long long>(sg, di.sms * 8 * 4);
            pl->samp_grid = (int)((warps + 3) / 4);
            int red = 1;
            while ((long long)pl->samp_grid * 4 * (32 / red) > kMinSlots && red < 32) red <<= 1;
            pl->samp_red = red;
            pl->samp_m = (int)std::min<long long>((long long)pl->samp_grid * 4 * (32 / red), kMinSlots);
        }
    }
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += dctd::align_up(bytes, 256); return o; };
    const size_t list = (size_t)nq * (size_t)k * 8;
    pl->off_parts_full = take((size_t)pl->full.splits * list);
    size_t tmp_parts = pl->full.splits > kMergePPW ? (size_t)((pl->full.splits + kMergePPW - 1) / kMergePPW) : 0;
    pl->off_parts_samp = pl->off_thr = pl->off_thrd = pl->off_ctl = pl->off_cnt = pl->off_flags = pl->off_cand = pl->off_mins = 0;
    if (pl->thresh) {
        if (!pl->bounded) {
            pl->off_parts_samp = take((size_t)pl->samp.splits * list);
            if (pl->samp.splits > kMergePPW)
                tmp_parts = std::max(tmp_parts, (size_t)((pl->samp.splits + kMergePPW - 1) / kMergePPW));
            pl->off_thr = take(list);
            pl->off_thrd = take((size_t)nq * sizeof(unsigned int));
            pl->off_mins = pl->tc.stream ? take((size_t)16 * kMinSlots * sizeof(unsigned int)) : 0;
        }
        pl->off_ctl = take(256);          // grid-barrier counter + in-kernel bounds of the fused streaming kernel;
        pl->off_cnt = take((size_t)nq * sizeof(int));   // directly followed by the candidate counters (one memset)
        pl->off_flags = take((size_t)nq * sizeof(int));
        pl->off_cand = take((size_t)nq * (size_t)pl->cmax * 8);
    }
    pl->off_tmp = take(tmp_parts * list);
    pl->total = off + 256;
    return true;
}

int next_pow2(int x) {
    int p = 1;
    while (p < x) p <<= 1;
    return p;
}

typedef void (*ScanFn)(const ScanParams);

ScanFn heap_kernel(const ScanConfig &c) {
    if (c.td == kTDmax) {
        switch (c.tq) {
            case 1: return l1_scan_kernel<1, kTDmax, kStagesMax>;
            case 2: return l1_scan_kernel<2, kTDmax, kStagesMax>;
            case 4: return l1_scan_kernel<4, kTDmax, kStagesMax>;
            default: return l1_scan_kernel<8, kTDmax, kStagesMax>;
        }
    }
    switch (c.tq) {
        case 1: return l1_scan_kernel<1, 1, 2>;
        case 2: return l1_scan_kernel<2, 1, 2>;
        case 4: return l1_scan_kernel<4, 1, 2>;
        default: return l1_scan_kernel<8, 1, 2>;
    }
}

int launch_heap(const ScanConfig &c, ScanParams sp, cudaStream_t stream) {
    if (c.n_qtiles > 65535) return DCTD_ERR_UNSUPPORTED;   // caller batches queries
    sp.cap = c.cap;
    sp.n_groups = c.n_groups;
    sp.groups_per_split = c.groups_per_split;
    ScanFn fn = heap_kernel(c);
    DCTD_CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c.smem));
    fn<<<dim3((unsigned)c.splits, (unsigned)c.n_qtiles), (kWarps + 1) * 32, c.smem, stream>>>(sp);
    DCTD_LAUNCH_CHECK();
    return DCTD_OK;
}

// folds `parts` sorted key lists per query; the result goes to (dist, ids) and / or, if key_out is given, to keys
// (with id_base added to the position field)
int run_merge(const unsigned long long *keys, long long parts, long long nq, int k, long long id_base, float *dist,
              long long *ids, unsigned long long *key_out, const int *qflags, unsigned long long *tmp,
              cudaStream_t stream) {
    MergeParams mp{};
    mp.nq = nq; mp.k = k; mp.cap = next_pow2(2 * k); mp.qflags = qflags;
    const int warps = 4;
    const size_t msmem = (size_t)warps * mp.cap * 8;
    DCTD_CUDA_TRY(cudaFuncSetAttribute(l1_merge_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msmem));
    const unsigned gx = (unsigned)((nq + warps - 1) / warps);
    if (parts > kMergePPW) {
        if (parts > (long long)kMergePPW * kMergePPW) return DCTD_ERR_UNSUPPORTED;
        const long long chunks = (parts + kMergePPW - 1) / kMergePPW;
        mp.key_parts = keys; mp.parts = (int)parts; mp.ppw = kMergePPW; mp.key_out = tmp; mp.id_base = 0;
        l1_merge_kernel<false><<<dim3(gx, (unsigned)chunks), warps * 32, msmem, stream>>>(mp);
        DCTD_LAUNCH_CHECK();
        keys = tmp;
        parts = chunks;
    }
    mp.key_parts = keys; mp.parts = (int)parts; mp.ppw = (int)parts; mp.key_out = key_out; mp.id_base = id_base;
    mp.dist = dist; mp.ids = ids;
    l1_merge_kernel<false><<<dim3(gx, 1), warps * 32, msmem, stream>>>(mp);
    DCTD_LAUNCH_CHECK();
    return DCTD_OK;
}

// instantiations of the fused streaming kernel.  d = 480 (the reference's fingerprints, 30 chunks): chunk count known
// at compile time; otherwise runtime
template <int NW, int TD, int VAR = 0>
const void *stream_kernel_n(int tq, bool c480) {
#define DCTD_SK(TQ_) (c480 ? (const void *)l1_stream_fused_kernel<TQ_, NW, TD, 30, VAR> : (const void *)l1_stream_fused_kernel<TQ_, NW, TD, 0, VAR>)
    switch (tq) {
        case 4: return DCTD_SK(4);
        case 8: return DCTD_SK(8);
        case 12: return DCTD_SK(12);
        case 16: return DCTD_SK(16);
    }
#undef DCTD_SK
    return nullptr;
}

const void *stream_kernel(const StreamCfg &c, int d) {
    const bool c480 = d == 480;
    switch (c.nw * 10 + c.td) {
        case 71: return stream_kernel_n<7, 1>(c.tq, c480);
        case 41: return stream_kernel_n<4, 1>(c.tq, c480);
        case 21: return stream_kernel_n<2, 1>(c.tq, c480);
        case 11: return stream_kernel_n<1, 1>(c.tq, c480);
#ifdef DCTD_TUNING
        case 42: return g_l1_var == 1 ? stream_kernel_n<4, 2, 1>(c.tq, c480) : (g_l1_var == 2 ? stream_kernel_n<4, 2, 2>(c.tq, c480) : stream_kernel_n<4, 2>(c.tq, c480));
        case 62: return stream_kernel_n<6, 2>(c.tq, c480);
        case 52: return g_l1_var == 1 ? stream_kernel_n<5, 2, 1>(c.tq, c480) : (g_l1_var == 2 ? stream_kernel_n<5, 2, 2>(c.tq, c480) : stream_kernel_n<5, 2>(c.tq, c480));
#endif
    }
    return nullptr;
}

// The search proper.  Result as (dist, ids) and / or packed keys.  `bound` (optional, device int32 [nq]): only vectors
// with distance <= bound[q] need to be reported for query q (the caller knows that the k best over ALL shards lie within).
int run_topk(const int8_t *d_q, int64_t nq, const void *d_packed, int64_t n, int32_t d, int32_t k, int64_t id_base,
             const int32_t *d_bound, float *d_dist, long long *ids, unsigned long long *keys_out, void *d_workspace,
             size_t workspace_bytes, uint32_t flags, cudaStream_t stream) {
    if (nq < 0 || n < 0 || k < 1 || d < 1 || id_base < 0) return DCTD_ERR_ARG;
    if (nq == 0) return DCTD_OK;
    if (!d_q || (!keys_out && (!d_dist || !ids)) || (n > 0 && !d_packed)) return DCTD_ERR_ARG;
    if (n >= (1LL << kIdBits) || id_base + n >= (1LL << kIdBits)) return DCTD_ERR_UNSUPPORTED;
    DevInfo di;
    dev_info(&di);
    TopkPlan pl;
    if (!make_plan(di, nq, n, d, k, d_bound != nullptr, &pl)) return DCTD_ERR_UNSUPPORTED;
    if (!d_workspace || workspace_bytes < pl.total) return DCTD_ERR_WORKSPACE;
    if (((uintptr_t)d_workspace & 255) != 0 || ((uintptr_t)d_packed & 15) != 0) return DCTD_ERR_ARG;
    char *ws = (char *)d_workspace;
    unsigned long long *parts_full = (unsigned long long *)(ws + pl.off_parts_full);
    unsigned long long *tmp = (unsigned long long *)(ws + pl.off_tmp);

    if (n == 0) {   // empty database: every slot is padding
        DCTD_CUDA_TRY(cudaMemsetAsync(parts_full, 0xff, (size_t)nq * k * 8, stream));
        return run_merge(parts_full, 1, nq, k, id_base, d_dist, ids, keys_out, nullptr, tmp, stream);
    }
    ScanParams sp{};
    sp.q = d_q; sp.packed = (const uint4 *)d_packed; sp.nq = nq; sp.n = n; sp.d = d; sp.k = k; sp.gstride = 1;

    if (!pl.thresh || (flags & DCTD_L1_HEAP_ONLY)) {
        sp.parts = parts_full;
        int rc = launch_heap(pl.full, sp, stream);
        if (rc != DCTD_OK) return rc;
        return run_merge(parts_full, pl.full.splits, nq, k, id_base, d_dist, ids, keys_out, nullptr, tmp, stream);
    }

    // ---- threshold path ----
    int *cnt = (int *)(ws + pl.off_cnt);
    int *flagsq = (int *)(ws + pl.off_flags);
    unsigned long long *cand = (unsigned long long *)(ws + pl.off_cand);
    SelectParams se{};
    se.cand = cand; se.cnt = cnt; se.cmax = pl.cmax; se.k = k; se.nq = nq; se.id_base = id_base;
    se.dist = d_dist; se.ids = ids; se.key_out = keys_out; se.qflags = flagsq;
    const void *fused_fn = (pl.tc.stream && pl.fused.ok && g_l1_mode != 2 && g_l1_mode != 9) ? stream_kernel(pl.fused, d) : nullptr;
    if (fused_fn) {
        // ---- few queries: sample, bound, stream and selection in ONE cooperative launch (l1_stream.cuh) ----
        char *ctl = ws + pl.off_ctl;
        DCTD_CUDA_TRY(cudaMemsetAsync(ctl, 0, (pl.off_cnt - pl.off_ctl) + (size_t)nq * sizeof(int), stream));
        StreamParams P{};
        P.sp = sp;
        P.sp.gstride = pl.gstride;
        P.sp.thr_dist = pl.bounded ? (const unsigned int *)d_bound : nullptr;
        P.sp.cand = cand; P.sp.cnt = cnt; P.sp.cmax = pl.cmax;
        P.se = se;
        P.mins = pl.bounded ? nullptr : (unsigned int *)(ws + pl.off_mins);
        P.bar = (unsigned int *)ctl;
        P.thr_out = (unsigned int *)(ctl + 64);
        P.stages = pl.fused.stages;
        P.m = (int)std::min<long long>(di.sms * pl.fused.nw, kMinSlots);
        P.kscr_n = pl.fused.kscr_n;
        DCTD_CUDA_TRY(cudaFuncSetAttribute(fused_fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.fused.smem));
        void *args[] = {&P};
        DCTD_CUDA_TRY(cudaLaunchCooperativeKernel(fused_fn, dim3((unsigned)di.sms), dim3((pl.fused.nw + 1) * 32), args,
                                                  pl.fused.smem, stream));
        DCTD_LAUNCH_CHECK();
    } else {
        const unsigned int *thrd = nullptr;
        bool skip_sample = false;
        if (pl.bounded) {
            // 1'. the caller's bounds; nothing is seeded, every group is scanned
            thrd = (const unsigned int *)d_bound;
            DCTD_CUDA_TRY(cudaMemsetAsync(cnt, 0, (size_t)nq * sizeof(int), stream));
        } else {
            unsigned long long *parts_samp = (unsigned long long *)(ws + pl.off_parts_samp);
            unsigned long long *thr = (unsigned long long *)(ws + pl.off_thr);
            unsigned int *thrw = (unsigned int *)(ws + pl.off_thrd);
            thrd = thrw;
            // 1. thresholds: from lane minima over every gstride-th group (few queries), or the exact top-k of that sample
            if (pl.tc.stream && g_l1_mode != 2) {
                ScanParams s1 = sp;
                s1.gstride = pl.gstride;
                s1.n_groups = pl.samp_groups;
                unsigned int *mins = (unsigned int *)(ws + pl.off_mins);
                typedef void (*MinFn)(const ScanParams, unsigned int *, int);
                const int tq = pl.tc.tq;
                MinFn fn = tq == 4 ? l1_sample_min_kernel<4> : (tq == 8 ? l1_sample_min_kernel<8> : l1_sample_min_kernel<16>);
                // every slot below samp_m is written (lanes that saw no vector write 0xffffffff = "no bound")
                fn<<<pl.samp_grid, 128, pl.tc.smem, stream>>>(s1, mins, pl.samp_red);
                DCTD_LAUNCH_CHECK();
                l1_kth_kernel<<<(unsigned)nq, 256, 0, stream>>>(mins, pl.samp_m, k, thrw, cnt);   // also zeroes cnt
                DCTD_LAUNCH_CHECK();
            } else {
                ScanParams s1 = sp;
                s1.parts = parts_samp;
                s1.gstride = pl.gstride;
                int rc = launch_heap(pl.samp, s1, stream);
                if (rc != DCTD_OK) return rc;
                rc = run_merge(parts_samp, pl.samp.splits, nq, k, 0, nullptr, nullptr, thr, nullptr, tmp, stream);
                if (rc != DCTD_OK) return rc;
                // the sample's top-k seeds the candidate lists (then the scan can leave the sampled groups out)
                skip_sample = !pl.tc.stream && g_l1_mode != 3;
                l1_seed_kernel<<<(unsigned)((nq + 3) / 4), 128, 0, stream>>>(thr, nq, k, cand, cnt, pl.cmax, skip_sample, thrw);
                DCTD_LAUNCH_CHECK();
            }
        }
        // 2. one pass over the database: append everything within the bound
        {
            ScanParams s2 = sp;
            s2.thr_dist = thrd; s2.cand = cand; s2.cnt = cnt; s2.cmax = pl.cmax;
            s2.n_groups = (n + 31) / 32;
            const ThreshConfig &tc = pl.tc;
            if (skip_sample) {       // every group but the sampled ones
                s2.skip = pl.gstride;
                s2.n_groups -= (s2.n_groups + pl.gstride - 1) / pl.gstride;
            }
            if (tc.stream) {
                ScanFn fn = tc.tq == 4 ? l1_thresh_stream_kernel<4> : (tc.tq == 8 ? l1_thresh_stream_kernel<8> : l1_thresh_stream_kernel<16>);
                int per_sm = 0;
                DCTD_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, 128, tc.smem));
                const long long want = std::max<long long>(1, (s2.n_groups + 3) / 4);
                const int grid = (int)std::min<long long>(want, di.sms * std::max(1, per_sm));
                fn<<<grid, 128, tc.smem, stream>>>(s2);
                DCTD_LAUNCH_CHECK();
            } else {
                s2.groups_per_split = tc.groups_per_split;
                ScanFn fn;
                if (tc.nw == 16 && d == 480 && g_l1_mode != 5) fn = l1_thresh_scan_kernel<16, 8, kTDmax, kStagesMax, 30>;
                else if (tc.nw == 16) fn = l1_thresh_scan_kernel<16, 8, kTDmax, kStagesMax>;
                else if (tc.tq == 8) fn = l1_thresh_scan_kernel<8, 8, kTDmax, kStagesMax>;
                else fn = l1_thresh_scan_kernel<8, 4, kTDmax, kStagesMax>;
                if (tc.n_qtiles > 65535) return DCTD_ERR_UNSUPPORTED;
                DCTD_CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc.smem));
                fn<<<dim3((unsigned)tc.splits, (unsigned)tc.n_qtiles), (tc.nw + 1) * 32, tc.smem, stream>>>(s2);
                DCTD_LAUNCH_CHECK();
            }
        }
        // 3. exact selection per query; overflowed queries are flagged
        {
            const size_t ssmem = (size_t)pl.cmax * 8;
            DCTD_CUDA_TRY(cudaFuncSetAttribute(l1_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ssmem));
            l1_select_kernel<<<(unsigned)nq, 256, ssmem, stream>>>(se);
            DCTD_LAUNCH_CHECK();
        }
    }
    // 4. flagged queries (candidate list overflow: heavy distance ties, adversarial order, a bound that is not one)
    //    are redone by the heap scan; CTAs of unflagged query tiles exit at once, so this costs a few microseconds
    {
        ScanParams s4 = sp;
        s4.parts = parts_full;
        s4.qflags = flagsq;
        int rc = launch_heap(pl.full, s4, stream);
        if (rc != DCTD_OK) return rc;
        return run_merge(parts_full, pl.full.splits, nq, k, id_base, keys_out ? nullptr : d_dist, keys_out ? nullptr : ids,
                         keys_out, flagsq, tmp, stream);
    }
}

// sample of dctd_l1_bound: every `stride`-th group
struct BoundPlan {
    ScanConfig samp;
    long long stride;
    size_t off_parts, off_keys, off_tmp, total;
};

bool make_bound_plan(const DevInfo &di, long long nq, long long n, int d, int k_local, int stride, BoundPlan *bp) {
    const long long n_groups = (n + 31) / 32;
    bp->stride = stride > 0 ? stride : 32;
    const long long sg = (n_groups + bp->stride - 1) / bp->stride;
    if (!make_config(di, nq, sg, d, k_local, &bp->samp)) return false;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += dctd::align_up(bytes, 256); return o; };
    const size_t list = (size_t)nq * (size_t)k_local * 8;
    bp->off_parts = take((size_t)bp->samp.splits * list);
    bp->off_keys = take(list);
    bp->off_tmp = take(bp->samp.splits > kMergePPW ? (size_t)((bp->samp.splits + kMergePPW - 1) / kMergePPW) * list : 0);
    bp->total = off + 256;
    return true;
}

#include "l1_hits.cuh"
#include "l1_large.cuh"

}  // namespace

extern "C" {

#ifdef DCTD_TUNING
int dctd_l1_set_mode(int mode) { g_l1_mode = mode; return DCTD_OK; }

// phase stamps (ns, globaltimer) of CTA 0 of the last fused streaming launch that used this workspace: 8 values
int dctd_l1_stream_stamps(const void *d_workspace, int64_t nq, int64_t n, int32_t d, int32_t k, uint64_t *h_out8) {
    DevInfo di;
    dev_info(&di);
    TopkPlan pl;
    if (!make_plan(di, nq, n, d, k, false, &pl) || !pl.thresh) return DCTD_ERR_ARG;
    DCTD_CUDA_TRY(cudaMemcpy(h_out8, (const char *)d_workspace + pl.off_ctl + 128, 64, cudaMemcpyDeviceToHost));
    return DCTD_OK;
}
#endif

size_t dctd_l1_packed_bytes(int64_t n, int32_t d) {
    if (n < 0 || d < 1) return 0;
    return (size_t)((n + 31) / 32) * 32 * (size_t)chunks_of(d) * 16;
}

int dctd_l1_pack(const int8_t *d_rows, int64_t n, int32_t d, int64_t n_offset, void *d_packed, void *stream) {
    if (n < 0 || d < 1 || n_offset < 0 || (n > 0 && (!d_rows || !d_packed))) return DCTD_ERR_ARG;
    if (n == 0) return DCTD_OK;
    DevInfo di;
    dev_info(&di);
    const long long total = ((n_offset + n + 31) / 32 * 32 - n_offset / 32 * 32) * chunks_of(d);
    const int block = 256;
    const int grid = (int)std::min<long long>((total + block - 1) / block, di.sms * 16);
    pack_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(d_rows, n, d, n_offset, (uint4 *)d_packed);
    DCTD_LAUNCH_CHECK();
    return DCTD_OK;
}

int dctd_l1_unpack(const void *d_packed, int64_t n, int32_t d, int8_t *d_rows, void *stream) {
    if (n < 0 || d < 1 || (n > 0 && (!d_rows || !d_packed))) return DCTD_ERR_ARG;
    if (n == 0) return DCTD_OK;
    DevInfo di;
    dev_info(&di);
    const long long total = n * chunks_of(d);
    const int block = 256;
    const int grid = (int)std::min<long long>((total + block - 1) / block, di.sms * 16);
    unpack_kernel<<<grid, block, 0, (cudaStream_t)stream>>>((const uint4 *)d_packed, n, d, d_rows);
    DCTD_LAUNCH_CHECK();
    return DCTD_OK;
}

size_t dctd_l1_topk_workspace_bytes(int64_t nq, int64_t n, int32_t d, int32_t k) {
    DevInfo di;
    dev_info(&di);
    TopkPlan a, b;
    if (nq <= 0 || n < 0 || !make_plan(di, nq, n, d, k, false, &a) || !make_plan(di, nq, n, d, k, true, &b)) return 0;
    return std::max(a.total, b.total);
}

int dctd_l1_topk(const int8_t *d_q, int64_t nq, const void *d_packed, int64_t n, int32_t d, int32_t k,
                 int64_t id_base, float *d_dist, int64_t *d_ids, void *d_workspace, size_t workspace_bytes,
                 void *stream) {
    if (nq > 0 && (!d_dist || !d_ids)) return DCTD_ERR_ARG;
    return run_topk(d_q, nq, d_packed, n, d, k, id_base, nullptr, d_dist, (long long *)d_ids, nullptr, d_workspace,
                    workspace_bytes, 0u, (cudaStream_t)stream);
}

int dctd_l1_topk_keys(const int8_t *d_q, int64_t nq, const void *d_packed, int64_t n, int32_t d, int32_t k,
                      int64_t id_base, const int32_t *d_bound, uint64_t *d_keys, void *d_workspace,
                      size_t workspace_bytes, uint32_t flags, void *stream) {
    if (nq > 0 && !d_keys) return DCTD_ERR_ARG;
    return run_topk(d_q, nq, d_packed, n, d, k, id_base, d_bound, nullptr, nullptr, (unsigned long long *)d_keys,
                    d_workspace, workspace_bytes, flags, (cudaStream_t)stream);
}

int dctd_l1_uses_bound(int64_t nq, int64_t n, int32_t d, int32_t k) {
    DevInfo di;
    dev_info(&di);
    TopkPlan pl;
    if (nq <= 0 || n < 0 || !make_plan(di, nq, n, d, k, true, &pl)) return 0;
    return pl.thresh ? 1 : 0;
}

size_t dctd_l1_bound_workspace_bytes(int64_t nq, int64_t n, int32_t d, int32_t k_local, int32_t sample_stride) {
    DevInfo di;
    dev_info(&di);
    BoundPlan bp;
    if (nq <= 0 || n < 0 || sample_stride < 0 || !make_bound_plan(di, nq, n, d, k_local, sample_stride, &bp)) return 0;
    return bp.total;
}

int dctd_l1_bound(const int8_t *d_q, int64_t nq, const void *d_packed, int64_t n, int32_t d, int32_t k_local,
                  int32_t sample_stride, int32_t *d_bound, void *d_workspace, size_t workspace_bytes, void *stream_) {
    if (nq < 0 || n < 0 || k_local < 1 || d < 1 || sample_stride < 0) return DCTD_ERR_ARG;
    if (nq == 0) return DCTD_OK;
    if (!d_q || !d_bound || (n > 0 && !d_packed)) return DCTD_ERR_ARG;
    if (n >= (1LL << kIdBits)) return DCTD_ERR_UNSUPPORTED;
    cudaStream_t stream = (cudaStream_t)stream_;
    if (n == 0) {
        l1_fill_kernel<<<(unsigned)((nq + 255) / 256), 256, 0, stream>>>(d_bound, nq, 0x7fffffff);
        DCTD_LAUNCH_CHECK();
        return DCTD_OK;
    }
    DevInfo di;
    dev_info(&di);
    BoundPlan bp;
    if (!make_bound_plan(di, nq, n, d, k_local, sample_stride, &bp)) return DCTD_ERR_UNSUPPORTED;
    if (!d_workspace || workspace_bytes < bp.total) return DCTD_ERR_WORKSPACE;
    if (((uintptr_t)d_workspace & 255) != 0 || ((uintptr_t)d_packed & 15) != 0) return DCTD_ERR_ARG;
    char *ws = (char *)d_workspace;
    unsigned long long *parts = (unsigned long long *)(ws + bp.off_parts);
    unsigned long long *keys = (unsigned long long *)(ws + bp.off_keys);
    unsigned long long *tmp = (unsigned long long *)(ws + bp.off_tmp);
    ScanParams sp{};
    sp.q = d_q; sp.packed = (const uint4 *)d_packed; sp.nq = nq; sp.n = n; sp.d = d; sp.k = k_local;
    sp.gstride = bp.stride; sp.parts = parts;
    int rc = launch_heap(bp.samp, sp, stream);
    if (rc != DCTD_OK) return rc;
    rc = run_merge(parts, bp.samp.splits, nq, k_local, 0, nullptr, nullptr, keys, nullptr, tmp, stream);
    if (rc != DCTD_OK) return rc;
    l1_bound_kernel<<<(unsigned)((nq + 255) / 256), 256, 0, stream>>>(keys, nq, k_local, d_bound);
    DCTD_LAUNCH_CHECK();
    return DCTD_OK;
}

int dctd_l1_topk_merge(const float *d_dist_parts, const int64_t *d_ids_parts, int32_t parts, int64_t nq,
                       int32_t k, float *d_dist, int64_t *d_ids, void *stream) {
    if (parts < 1 || parts > 1024 || nq < 0 || k < 1 || k > kLargeMaxK) return DCTD_ERR_ARG;
    if (nq == 0) return DCTD_OK;
    if (!d_dist_parts || !d_ids_parts || !d_dist || !d_ids) return DCTD_ERR_ARG;
    MergeParams mp{};
    mp.dist_parts = d_dist_parts; mp.id_parts = (const long long *)d_ids_parts;
    mp.parts = parts; mp.ppw = parts; mp.nq = nq; mp.k = k; mp.cap = next_pow2(2 * k); mp.id_base = 0;
    mp.dist = d_dist; mp.ids = (long long *)d_ids;
    if (k > 992) return run_rank_merge(mp, true, (cudaStream_t)stream);
    const int warps = 4;
    const size_t msmem = (size_t)warps * mp.cap * 8;
    DCTD_CUDA_TRY(cudaFuncSetAttribute(l1_merge_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msmem));
    l1_merge_kernel<true><<<dim3((unsigned)((nq + warps - 1) / warps), 1), warps * 32, msmem, (cudaStream_t)stream>>>(mp);
    DCTD_LAUNCH_CHECK();
    return DCTD_OK;
}

int dctd_l1_keys_merge(const uint64_t *d_key_parts, int32_t parts, int64_t nq, int32_t k, float *d_dist,
                       int64_t *d_ids, uint64_t *d_keys, void *stream) {
    if (parts < 1 || parts > kMergePPW || nq < 0 || k < 1 || k > kLargeMaxK) return DCTD_ERR_ARG;
    if (nq == 0) return DCTD_OK;
    if (!d_key_parts || ((!d_dist || !d_ids) && !d_keys) || ((d_dist == nullptr) != (d_ids == nullptr))) return DCTD_ERR_ARG;
    if (k > 992) {
        MergeParams mp{};
        mp.key_parts = (const unsigned long long *)d_key_parts; mp.parts = parts; mp.nq = nq; mp.k = k;
        mp.dist = d_dist; mp.ids = (long long *)d_ids; mp.key_out = (unsigned long long *)d_keys;
        return run_rank_merge(mp, false, (cudaStream_t)stream);
    }
    return run_merge((const unsigned long long *)d_key_parts, parts, nq, k, 0, d_dist, (long long *)d_ids,
                     (unsigned long long *)d_keys, nullptr, nullptr, (cudaStream_t)stream);
}

size_t dctd_l1_topk_large_workspace_bytes(int64_t nq, int64_t n, int32_t d, int32_t k) {
    LargeLayout l;
    if (n < 0 || !large_layout(nq, d, k, &l)) return 0;
    return l.total;
}

int dctd_l1_topk_large(const int8_t *d_q, int64_t nq, const void *d_packed, int64_t n, int32_t d, int32_t k,
                       int64_t id_base, float *d_dist, int64_t *d_ids, uint64_t *d_keys, void *d_workspace,
                       size_t workspace_bytes, void *stream) {
    return run_topk_large(d_q, nq, d_packed, n, d, k, id_base, d_dist, (long long *)d_ids, (unsigned long long *)d_keys,
                          d_workspace, workspace_bytes, (cudaStream_t)stream);
}

int dctd_l1_pair_scores(const int8_t *d_fps, int32_t d, const int64_t *d_off, const int32_t *d_pair_a,
                        const int32_t *d_pair_b, int64_t n_pairs, int32_t *d_min_dist, int32_t *d_last_dist,
                        void *stream) {
    if (n_pairs < 0 || d < 1) return DCTD_ERR_ARG;
    if (n_pairs == 0) return DCTD_OK;
    if (!d_fps || !d_off || !d_pair_a || !d_pair_b || !d_min_dist || !d_last_dist) return DCTD_ERR_ARG;
    const int warps = 4;
    const unsigned grid = (unsigned)((n_pairs + warps - 1) / warps);
    if (d % 16 == 0 && ((uintptr_t)d_fps & 15) == 0)
        pair_scores_kernel<true><<<grid, warps * 32, 0, (cudaStream_t)stream>>>(
            d_fps, d, (const long long *)d_off, d_pair_a, d_pair_b, n_pairs, d_min_dist, d_last_dist);
    else
        pair_scores_kernel<false><<<grid, warps * 32, 0, (cudaStream_t)stream>>>(
            d_fps, d, (const long long *)d_off, d_pair_a, d_pair_b, n_pairs, d_min_dist, d_last_dist);
    DCTD_LAUNCH_CHECK();
    return DCTD_OK;
}

/* protein-level scores for all pairs of two sets: see dctd.h */
size_t dctd_l1_protein_scores_workspace_bytes(int64_t n_qf, int64_t n_qprot, int64_t n_dbf, int64_t n_dbprot, int32_t d) {
    if (n_qf < 0 || n_qprot < 0 || n_dbf < 0 || n_dbprot < 0 || d < 1) return 0;
    const size_t ld = (size_t)((n_dbf + 31) / 32) * 32;
    const size_t rows_all = (size_t)n_qprot * 2 + (size_t)(n_qf + 7) / 8;       // segments + last rows, upper bound
    const size_t rows_min = 128 + 128 + 16;                                     // one tile of single-fingerprint proteins
    const size_t rows = std::max(rows_min, std::min(rows_all, ((size_t)1 << 30) / std::max<size_t>(1, ld * 4)));
    size_t off = 0;
    off += dctd::align_up(rows * ld * 4, 256);
    off += dctd::align_up(((size_t)(n_qf + 7) / 8 + 64) * sizeof(int4), 256);   // slices
    off += 2 * dctd::align_up(((size_t)n_qprot + 1) * sizeof(int), 256);        // segment offsets, last rows
    off += dctd::align_up(((size_t)n_dbprot + 1) * sizeof(long long), 256);     // database offsets
    return off + 256;
}

int dctd_l1_protein_scores(const int8_t *d_qf, const int64_t *h_qoff, int64_t n_qprot, const void *d_db_packed,
                           const int64_t *h_doff, int64_t n_dbprot, int32_t d, int32_t *d_min_dist, int32_t *d_last_dist,
                           void *d_workspace, size_t workspace_bytes, void *stream_) {
    if (n_qprot < 0 || n_dbprot < 0 || d < 1) return DCTD_ERR_ARG;
    if (n_qprot == 0 || n_dbprot == 0) return DCTD_OK;
    if (!h_qoff || !h_doff || !d_min_dist || !d_last_dist || !d_workspace) return DCTD_ERR_ARG;
    const int64_t n_qf = h_qoff[n_qprot], n_dbf = h_doff[n_dbprot];
    if (h_qoff[0] != 0 || h_doff[0] != 0 || n_qf < 0 || n_dbf < 0) return DCTD_ERR_ARG;
    for (int64_t a = 0; a < n_qprot; ++a) if (h_qoff[a + 1] < h_qoff[a]) return DCTD_ERR_ARG;
    for (int64_t b = 0; b < n_dbprot; ++b) if (h_doff[b + 1] < h_doff[b]) return DCTD_ERR_ARG;
    if ((n_qf > 0 && !d_qf) || (n_dbf > 0 && !d_db_packed)) return DCTD_ERR_ARG;
    if (((uintptr_t)d_workspace & 255) != 0) return DCTD_ERR_ARG;
    cudaStream_t stream = (cudaStream_t)stream_;
    DevInfo di;
    dev_info(&di);
    constexpr int NW = 16, TQ = 8, QT = NW * TQ;
    const int dpad = chunks_of(d) * 16;
    const size_t smem = 128 + (size_t)QT * dpad + (size_t)kStagesMax * kTDmax * 32 * dpad + 64;
    if (smem > di.smem) return DCTD_ERR_UNSUPPORTED;
    const long long n_groups = (n_dbf + 31) / 32, ld = n_groups * 32;
    // workspace layout (the matrix region takes what is left after the tables)
    char *ws = (char *)d_workspace;
    size_t tables = 0;
    auto take = [&](size_t bytes) { const size_t o = tables; tables += dctd::align_up(bytes, 256); return o; };
    const size_t off_slices = take(((size_t)(n_qf + 7) / 8 + 64) * sizeof(int4));
    const size_t off_seg = take(((size_t)n_qprot + 1) * sizeof(int));
    const size_t off_last = take(((size_t)n_qprot + 1) * sizeof(int));
    const size_t off_doff = take(((size_t)n_dbprot + 1) * sizeof(long long));
    if (workspace_bytes < tables + 256) return DCTD_ERR_WORKSPACE;
    const size_t mat_bytes = (workspace_bytes - tables) / 256 * 256;
    unsigned int *mat = (unsigned int *)(ws + tables);
    const long long rows_cap = ld > 0 ? (long long)(mat_bytes / ((size_t)ld * 4)) : (1LL << 40);
    DCTD_CUDA_TRY(cudaMemcpyAsync(ws + off_doff, h_doff, ((size_t)n_dbprot + 1) * sizeof(long long), cudaMemcpyHostToDevice, stream));
    std::vector<int4> slices;
    std::vector<int> seg_off, last_row;
    try {
        int64_t a0 = 0;
        while (a0 < n_qprot) {
            // ---- the next chunk of query proteins: as many as the matrix region, the grid limits and 2^31 slots allow ----
            slices.clear(); seg_off.assign(1, 0); last_row.clear();
            const int64_t f0 = h_qoff[a0];
            int64_t a1 = a0;
            long long n_seg = 0, n_last = 0;
            while (a1 < n_qprot && a1 - a0 < 65535) {
                const int64_t s = h_qoff[a1] - f0, e = h_qoff[a1 + 1] - f0;        // slots of this protein
                const long long segs = e > s ? (e - 1) / TQ - s / TQ + 1 : 0;
                if ((n_seg + segs) + (n_last + (e > s ? 1 : 0)) > rows_cap || (e + QT - 1) / QT > 65535) break;
                n_seg += segs;
                seg_off.push_back((int)n_seg);
                last_row.push_back(e > s ? (int)n_last : -1);
                n_last += e > s ? 1 : 0;
                ++a1;
            }
            if (a1 == a0) return DCTD_ERR_WORKSPACE;         // not even one protein fits
            const int64_t nf = h_qoff[a1] - f0;
            const long long n_tiles_q = (nf + QT - 1) / QT;
            if (nf > 0 && n_dbf > 0) {
                // slice table: segment / last masks per TQ slots
                slices.assign((size_t)n_tiles_q * NW, make_int4(0, 0, 0, 0));
                long long seg = 0, lastc = 0;
                int64_t prot = a0;
                while (prot < a1 && h_qoff[prot + 1] - f0 == 0) ++prot;                  // leading empty proteins
                for (int64_t sl = 0; sl * TQ < nf; ++sl) {
                    unsigned int segend = 0, lastm = 0;
                    slices[(size_t)sl].x = (int)seg;
                    slices[(size_t)sl].y = (int)lastc;
                    for (int a = 0; a < TQ; ++a) {
                        const int64_t slot = sl * TQ + a;
                        if (slot >= nf) break;
                        while (h_qoff[prot + 1] - f0 <= slot) ++prot;                    // protein of this slot (skips empty ones)
                        const bool is_last = slot == h_qoff[prot + 1] - f0 - 1;
                        if (is_last) { lastm |= 1u << a; ++lastc; }
                        if (is_last || a == TQ - 1 || slot == nf - 1) { segend |= 1u << a; ++seg; }
                    }
                    slices[(size_t)sl].z = (int)(segend | (lastm << 8));
                }
                if (seg != n_seg || lastc != n_last) return DCTD_ERR_ARG;                // (cannot happen)
                DCTD_CUDA_TRY(cudaMemcpyAsync(ws + off_slices, slices.data(), slices.size() * sizeof(int4), cudaMemcpyHostToDevice, stream));
                ProtParams pp{};
                pp.sp.q = d_qf + f0 * d; pp.sp.nq = nf; pp.sp.packed = (const uint4 *)d_db_packed; pp.sp.n = n_dbf;
                pp.sp.d = d; pp.sp.k = 1; pp.sp.n_groups = n_groups; pp.sp.gstride = 1; pp.sp.skip = 0;
                long long splits = 1;
                pick_splits(di.sms, n_groups, kTDmax, n_tiles_q, 2, &splits, &pp.sp.groups_per_split);
                pp.slices = (const int4 *)(ws + off_slices);
                pp.mseg = mat;
                pp.mlast = mat + (size_t)n_seg * ld;
                pp.ld = ld;
                auto fn = d == 480 ? l1_protein_kernel<NW, TQ, kTDmax, kStagesMax, 30> : l1_protein_kernel<NW, TQ, kTDmax, kStagesMax, 0>;
                DCTD_CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                fn<<<dim3((unsigned)splits, (unsigned)n_tiles_q), (NW + 1) * 32, smem, stream>>>(pp);
                DCTD_LAUNCH_CHECK();
            }
            DCTD_CUDA_TRY(cudaMemcpyAsync(ws + off_seg, seg_off.data(), seg_off.size() * sizeof(int), cudaMemcpyHostToDevice, stream));
            // phase 2 (also fills INT32_MAX for proteins without fingerprints)
            // mlast rows follow protein order among the non-empty proteins: the kernel addresses row a of mlast, so
            // empty proteins are given no row by compacting through last_row
            DCTD_CUDA_TRY(cudaMemcpyAsync(ws + off_last, last_row.data(), last_row.size() * sizeof(int), cudaMemcpyHostToDevice, stream));
            l1_protein_reduce_kernel<<<dim3((unsigned)((n_dbprot + 255) / 256), (unsigned)(a1 - a0)), 256, 0, stream>>>(
                mat, mat + (size_t)n_seg * ld, ld, (const int *)(ws + off_seg), (const int *)(ws + off_last),
                (const long long *)(ws + off_doff), n_dbprot, d_min_dist + a0 * n_dbprot, d_last_dist + a0 * n_dbprot, n_dbprot);
            DCTD_LAUNCH_CHECK();
            a0 = a1;
        }
    } catch (const std::bad_alloc &) {
        return DCTD_ERR_NOMEM;
    }
    return DCTD_OK;
}

/* dct-sim database-search hits: see dctd.h */
static int hits_args(const int64_t *h_qoff, int64_t n_qprot, const int64_t *h_doff, int64_t n_dbprot, int32_t d,
                     int32_t dist_clamp, int32_t cap) {
    if (n_qprot < 0 || n_dbprot < 0 || d < 1 || cap < 1 || dist_clamp < 0 || dist_clamp >= (1 << 24)) return DCTD_ERR_ARG;
    if (!h_qoff || !h_doff || h_qoff[0] != 0 || h_doff[0] != 0) return DCTD_ERR_ARG;
    for (int64_t a = 0; a < n_qprot; ++a) if (h_qoff[a + 1] < h_qoff[a]) return DCTD_ERR_ARG;
    for (int64_t b = 0; b < n_dbprot; ++b) if (h_doff[b + 1] < h_doff[b]) return DCTD_ERR_ARG;
    if (cap > kHitsMaxCap || d > 2048 || n_dbprot >= (1LL << kIdBits)) return DCTD_ERR_UNSUPPORTED;
    return DCTD_OK;
}

size_t dctd_l1_protein_hits_workspace_bytes(int64_t n_qf, int64_t n_qprot, int64_t n_dbf, int64_t n_dbprot, int32_t d,
                                            int32_t top, int32_t cap) {
    (void)top;
    if (n_qf < 0 || n_qprot < 0 || n_dbf < 0 || n_dbprot < 0 || d < 1 || cap < 1 || cap > kHitsMaxCap) return 0;
    DevInfo di;
    dev_info(&di);
    HitsLayout l;
    if (!hits_layout(di, n_qprot, n_dbprot, d, cap, std::max<long long>(1, std::min<long long>(n_qprot, kHitsMaxChunk)), &l))
        return 0;
    return l.total;
}

int dctd_l1_protein_hits(const int8_t *d_qf, const int64_t *h_qoff, int64_t n_qprot, const int8_t *d_dbf,
                         const int64_t *h_doff, int64_t n_dbprot, int32_t d, int32_t top, int32_t dist_clamp,
                         int32_t dist_cut, int32_t cap, int32_t *d_count, int32_t *d_hit_db, int32_t *d_hit_min,
                         int32_t *d_hit_last, void *d_workspace, size_t workspace_bytes, void *stream) {
    int rc = hits_args(h_qoff, n_qprot, h_doff, n_dbprot, d, dist_clamp, cap);
    if (rc != DCTD_OK) return rc;
    if (n_qprot == 0) return DCTD_OK;
    if (!d_count || !d_hit_db || !d_hit_min || !d_hit_last) return DCTD_ERR_ARG;
    if ((h_qoff[n_qprot] > 0 && !d_qf) || (h_doff[n_dbprot] > 0 && !d_dbf)) return DCTD_ERR_ARG;
    try {
        return run_hits(d_qf, h_qoff, n_qprot, d_dbf, h_doff, n_dbprot, d, top, dist_clamp, dist_cut, cap, d_count,
                        d_hit_db, d_hit_min, d_hit_last, d_workspace, workspace_bytes, (cudaStream_t)stream);
    } catch (const std::bad_alloc &) {
        return DCTD_ERR_NOMEM;
    }
}

}  // extern "C"
