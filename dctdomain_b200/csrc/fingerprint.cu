// libdctd hot path 1: batched DCT fingerprints ("quant2D") for sm_100a.
//
// What the reference computes per (domain, layer) - src/fingerprint.py:174-201 - restated:
//   X [L, D] rows of the domain (get_doms order)                       fingerprint.py:145-171
//   Y = idct_n(dct(X along L)[:n])   -> [n, D], per column min-max     fingerprint.py:126-142, :192
//   Z = idct_m(dct(Y along D)[:m])   -> [n, m], per row min-max        fingerprint.py:193
//   out[j*m + c] = trunc(Z[j, c] * 127) as int8                        fingerprint.py:194-195
// Both min-max steps are invariant to adding a constant and to a positive scale, so the DC
// coefficient and the orthonormal scale factors drop out:
//   u_k[d] = sum_l (x[l,d] - x[0,d]) * cos(pi (2l+1) k / 2L),  k = 1..n-1      ("pass 1")
//   Y[j,d] ~ sum_k cos(pi (2j+1) k / 2n) u_k[d]
//   F[j,k] = sum_d Y'[j,d] * cos(pi (2d+1) k / 2D),             k = 1..m-1      ("pass 2")
//   Z[j,c] ~ sum_k cos(pi (2c+1) k / 2m) F[j,k]
// Pass 1 is the HBM-bound part (every embedding element is read exactly once, n-1 FMAs each);
// everything after it works on O(n*D) values per (domain, layer) and stays in shared memory.
//
// Two kernels share the planner and the C ABI in this file: the warp-specialised TMA kernel of fp_ws_kernel.cuh
// (the reference's configuration: n = 3, D = 1280 / 640, contiguous aligned rows) and the general kernel below
// (every other shape; also the A/B partner, dctd_fp_set_variant(9)).
//
// General kernel (B200: 148 SMs, persistent CTAs pulling work items from an atomic queue):
//   item = (domain, layer, row range <= 512 rows); a CTA streams the item's rows with 16-byte
//   no-allocate loads, U rows in flight per thread, float32 FMAs flushed into float64
//   accumulators every U rows; domains longer than 512 rows are split over several items whose
//   partial sums meet in the workspace, the last-arriving CTA (atomic ticket) finishing the
//   domain.  The maxlen windows of src/embedding.py:153-192 are consumed in place: rows covered
//   by two windows are loaded from both and averaged (a + b) * 0.5f exactly as embedding.py:186.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <new>
#include <vector>

#include "dctd_internal.cuh"
#include "dctd_tma.cuh"

namespace {

constexpr int kRowsPerItem = 512;  // max rows of one work item (size of the per-item basis table)
constexpr int kMaxN = 8;           // n in [2, 8]
constexpr int kMaxM = 128;         // m in [2, 128]
constexpr int kMaxThreads = 640;

struct Piece {        // a run of consecutive domain rows read from one (or two averaged) sources
    int32_t src_a, row_a;
    int32_t src_b, row_b;   // src_b < 0: single source
    int32_t nrows, l0;      // l0 = index of the first row within the concatenated domain
    int32_t g0, pad;        // g0 = protein row of the first row (basis index of a riding global fingerprint)
};
struct DomInfo {
    int32_t piece_off, n_pieces;
    int32_t L;              // rows of the concatenated domain
    int32_t nsplit;
    int32_t slab0;          // first partial-sum slab (layer-major: slab0 + layer*nsplit + split)
    int32_t counter0;       // arrival counter index base (counter0 + layer), -1: the domain is one item
    int32_t pivot;          // absolute index of the piece whose first row is the pivot
    int32_t pad1;
};
struct Item {
    int32_t dom, layer;
    int32_t r0, r1;         // domain-local row range
    int32_t split, piece_first;
    int32_t rider_dom;      // >= 0: the global domain of the same protein accumulated from these rows too
    int32_t rider_split;    // its partial-sum slot
};

struct Layout {             // thread / shared-memory layout derived from (D, n, m)
    int vec;                // 4: float4 loads, 1: scalar loads (D % 4 != 0 or misaligned rows)
    int G;                  // column groups = ceil(D / vec)
    int CT;                 // column tiles per thread
    int RL;                 // row lanes (threads sharing a column group, interleaved rows)
    int T;                  // threads per CTA
    int table_len;          // entries of the extended pass-2a cosine table: 4D + 8m
    size_t smem;            // dynamic shared memory bytes
    size_t off_t4d, off_y, off_cb, off_scr, off_tm, off_mj;
};

struct WsLayout {           // shared-memory layout of the warp-specialised kernel (fp_ws_kernel.cuh)
    int nst;                // TMA ring stages
    int DSo, DSe;           // pass-2a splits of the folded column range for odd / even coefficient pairs
    int H;                  // pass-2a coefficient pairing: a thread owns k and k + H (H = 0 mod 4)
    unsigned off_bars, off_meta, off_basis, off_desc, off_ring, off_u, off_ye, off_yo, off_f, off_tt, off_tm, off_mj;
    unsigned smem;
};

struct Params {
    const float *const *src;
    const float *table;     // extended cosine table in the workspace (fp_table_kernel)
    const Piece *pieces;
    const DomInfo *doms;
    const Item *items;
    int *counters;
    double *partials;
    long long *timing;      // [16] phase cycle counters (DCTD_FP_TIMING builds only)
    double *debug_u;        // DCTD_DEBUG_U builds: per (domain, layer, split) copy of the consumers' sums
    int8_t *out;
    int64_t ld, out_stride;
    int32_t n_src, n_items, n_layers;
    int32_t D, n, m;
    Layout lay;
    // warp-specialised kernel only
    const int32_t *wsitems; // fat item records (32 words each), same order as items
    WsLayout wl;
};

}  // namespace

struct dctd_fp_plan {
    int32_t n_layers, D, n, m, n_src, n_dom;
    std::vector<Piece> pieces;
    std::vector<DomInfo> doms;
    std::vector<Item> items;
    bool has_rider;           // some items carry their protein's global fingerprint along
    uint32_t flags;           // DCTD_FP_PLAN_* options the plan was created with
    int32_t n_counters;       // 1 (work queue) + split arrival counters
    int64_t n_slabs;          // partial-sum slabs of (n-1)*D doubles
    int64_t algo_bytes;
    // device blob layout (bytes from the workspace base)
    size_t off_pieces, off_doms, off_items, off_wsitems, off_src, off_counters, off_timing, off_table, off_partials, total;
    void *blob;               // host copy of [pieces | doms | items | 32-word item records], pinned when possible
    bool blob_pinned;
    size_t blob_bytes;        // bytes uploaded
    size_t blob_capacity;     // bytes allocated (blobs are recycled through a small cache, see blob_acquire)
    mutable cudaEvent_t uploaded;   // recorded after the last upload of the blob: the blob is not recycled before it
    mutable bool has_event;
};

namespace {

// ------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------
// packed pair of floats (sm_100 FADD2 / FMUL2 / FFMA2: two IEEE fp32 ops per instruction)
typedef unsigned long long pk2;
__device__ __forceinline__ pk2 pk(float lo, float hi) {
    pk2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpk(pk2 v, float &lo, float &hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ pk2 add2(pk2 a, pk2 b) {
    pk2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ pk2 mul2(pk2 a, pk2 b) {
    pk2 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ pk2 fma2(pk2 a, pk2 b, pk2 c) {
    pk2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}

// streaming 16-byte read (data is used exactly once: keep it out of L1), as two packed pairs
__device__ __forceinline__ void ldg_stream4(const float *p, pk2 &lo, pk2 &hi) {
    asm volatile("ld.global.nc.L1::no_allocate.v2.b64 {%0,%1}, [%2];" : "=l"(lo), "=l"(hi) : "l"(p));
}
__device__ __forceinline__ float ldg_stream1(const float *p) {
    float r;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
    return r;
}

// the K basis values of one row as (c, c) pairs (one FFMA2 covers two columns); vector shared loads when K allows.
// The table holds plain floats: shared memory is the scarce resource here (what the CTAs do not take is L1,
// and the L1 size bounds the loads in flight).
template <int K>
__device__ __forceinline__ void load_basis(const float *p, pk2 (&c)[K]) {
    if constexpr (K % 4 == 0) {
#pragma unroll
        for (int k = 0; k < K; k += 4) {
            const float4 v = *reinterpret_cast<const float4 *>(p + k);
            c[k] = pk(v.x, v.x); c[k + 1] = pk(v.y, v.y); c[k + 2] = pk(v.z, v.z); c[k + 3] = pk(v.w, v.w);
        }
    } else if constexpr (K % 2 == 0) {
#pragma unroll
        for (int k = 0; k < K; k += 2) {
            const float2 v = *reinterpret_cast<const float2 *>(p + k);
            c[k] = pk(v.x, v.x); c[k + 1] = pk(v.y, v.y);
        }
    } else {
#pragma unroll
        for (int k = 0; k < K; ++k) c[k] = pk(p[k], p[k]);
    }
}

// ---- pass 1, float4 path: rows rl, rl+RL, ... of one piece; acc[k] += (x - pivot) * c_k[row] ----
// LDC / RLC: compile-time row stride (floats) and row-lane count for the common ESM-2 widths (0 = runtime);
// with them every load of a block is base + immediate and the address arithmetic disappears.
template <int K, int U, bool DUAL, int LDC, int RLC>
__device__ __forceinline__ void stream_piece4(const float *pa, const float *pb, int64_t ld_, int nr, int rl,
                                              int RL_, const float *cb2, pk2 npiv0, pk2 npiv1,
                                              double (&acc)[K][4]) {
    const int RL = RLC ? RLC : RL_;
    const int64_t ld = LDC ? (int64_t)LDC : ld_;
    const int64_t step = (int64_t)RL * ld;
    const pk2 half = pk(0.5f, 0.5f);
    const pk2 zero = pk(0.f, 0.f);
    pa += (int64_t)rl * ld;
    if (DUAL) pb += (int64_t)rl * ld;
    const float *cbp = cb2 + rl * K;
    const int cstep = RL * K;
    int left = (nr - rl + RL - 1) / RL;      // rows this thread owns
    if (left < 0) left = 0;
    // full blocks of U rows
    for (; left >= U; left -= U) {
        pk2 x0[U], x1[U];
#pragma unroll
        for (int u = 0; u < U; ++u) ldg_stream4(pa + u * step, x0[u], x1[u]);
        if (DUAL) {
            pk2 y0[U], y1[U];
#pragma unroll
            for (int u = 0; u < U; ++u) ldg_stream4(pb + u * step, y0[u], y1[u]);
#pragma unroll
            for (int u = 0; u < U; ++u) {          // embedding.py:186: (prev + cur) / 2 in float32
                x0[u] = mul2(add2(x0[u], y0[u]), half);
                x1[u] = mul2(add2(x1[u], y1[u]), half);
            }
            pb += U * step;
        }
        pk2 a0[K], a1[K];
#pragma unroll
        for (int k = 0; k < K; ++k) { a0[k] = zero; a1[k] = zero; }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const pk2 t0 = add2(x0[u], npiv0), t1 = add2(x1[u], npiv1);
            pk2 c[K];
            load_basis<K>(cbp + u * cstep, c);
#pragma unroll
            for (int k = 0; k < K; ++k) {
                a0[k] = fma2(t0, c[k], a0[k]);
                a1[k] = fma2(t1, c[k], a1[k]);
            }
        }
#pragma unroll
        for (int k = 0; k < K; ++k) {
            float f0, f1, f2, f3;
            unpk(a0[k], f0, f1);
            unpk(a1[k], f2, f3);
            acc[k][0] += (double)f0; acc[k][1] += (double)f1;
            acc[k][2] += (double)f2; acc[k][3] += (double)f3;
        }
        pa += U * step;
        cbp += U * cstep;
    }
    // tail (< U rows): predicated loads, same arithmetic
    if (left > 0) {
        pk2 x0[U], x1[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            x0[u] = zero; x1[u] = zero;
            if (u < left) {
                ldg_stream4(pa + u * step, x0[u], x1[u]);
                if (DUAL) {
                    pk2 y0, y1;
                    ldg_stream4(pb + u * step, y0, y1);
                    x0[u] = mul2(add2(x0[u], y0), half);
                    x1[u] = mul2(add2(x1[u], y1), half);
                }
            }
        }
        pk2 a0[K], a1[K];
#pragma unroll
        for (int k = 0; k < K; ++k) { a0[k] = zero; a1[k] = zero; }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (u < left) {
                const pk2 t0 = add2(x0[u], npiv0), t1 = add2(x1[u], npiv1);
                pk2 c[K];
                load_basis<K>(cbp + u * cstep, c);
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    a0[k] = fma2(t0, c[k], a0[k]);
                    a1[k] = fma2(t1, c[k], a1[k]);
                }
            }
        }
#pragma unroll
        for (int k = 0; k < K; ++k) {
            float f0, f1, f2, f3;
            unpk(a0[k], f0, f1);
            unpk(a1[k], f2, f3);
            acc[k][0] += (double)f0; acc[k][1] += (double)f1;
            acc[k][2] += (double)f2; acc[k][3] += (double)f3;
        }
    }
}

// ---- pass 1, scalar path (D % 4 != 0 or rows not 16-byte aligned) ----
template <int K, bool DUAL>
__device__ __forceinline__ void stream_piece1(const float *pa, const float *pb, int64_t ld, int nr, int rl,
                                              int RL, const float *cb2, float piv, double (&acc)[K][4]) {
    constexpr int U = 8;
    for (int i0 = rl; i0 < nr; i0 += U * RL) {
        float x[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = i0 + u * RL;
            x[u] = 0.f;
            if (i < nr) {
                x[u] = ldg_stream1(pa + (int64_t)i * ld);
                if (DUAL) x[u] = (x[u] + ldg_stream1(pb + (int64_t)i * ld)) * 0.5f;
            }
        }
        float a32[K];
#pragma unroll
        for (int k = 0; k < K; ++k) a32[k] = 0.f;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = i0 + u * RL;
            if (i < nr) {
                const float t = x[u] - piv;
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    a32[k] = fmaf(t, cb2[i * K + k], a32[k]);
                }
            }
        }
#pragma unroll
        for (int k = 0; k < K; ++k) acc[k][0] += (double)a32[k];
    }
}

// extended cosine table for pass 2a: T[i] = cos(pi * (i mod 4D) / 2D), i < 4D + 8m
__global__ void fp_table_kernel(float *T, int D, int len) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < len; i += gridDim.x * blockDim.x)
        T[i] = (float)cospi((double)(i % (4 * D)) / (2.0 * D));
}

// Optional per-phase cycle counters (build with -DDCTD_FP_TIMING; dctd_fp_timing_read): thread 0 of every CTA
// accumulates clock64() deltas per phase into Params::timing.
#ifdef DCTD_FP_TIMING
#define TIC() long long _t0 = clock64()
#define TOC(slot)                                                         \
    do {                                                                  \
        if (threadIdx.x == 0) {                                           \
            const long long _t1 = clock64();                              \
            atomicAdd((unsigned long long *)&p.timing[slot], (unsigned long long)(_t1 - _t0)); \
            _t0 = _t1;                                                    \
        }                                                                 \
    } while (0)
#else
#define TIC() do {} while (0)
#define TOC(slot) do {} while (0)
#endif

// ------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------
// MAXT/MINB: launch bounds (registers per thread are capped at 65536 / (MAXT * MINB)).
// RIDER: items of a protein's domains also accumulate the protein's global ("1-L") fingerprint from the
// same loads (2K projections per element instead of K); the global's partial sums meet in the workspace.
template <int K, int VEC, int U, int MAXT, int MINB, int LDC = 0, int RLC = 0, bool RIDER = false>
__global__ void __launch_bounds__(MAXT, MINB) fp_kernel(const Params p) {
    constexpr int N = K + 1;
    constexpr int KS = RIDER ? 2 * K : K;      // projections accumulated while streaming
    extern __shared__ __align__(16) unsigned char smem[];
    float *TT = reinterpret_cast<float *>(smem + p.lay.off_t4d);     // cos table (extended), pass 2a
    float *Y = reinterpret_cast<float *>(smem + p.lay.off_y);        // [N][D] pass-1 result, folded
    float *cb2 = reinterpret_cast<float *>(smem + p.lay.off_cb);     // [rows][KS] basis of the item
    double *scr = reinterpret_cast<double *>(smem + p.lay.off_scr);  // u sums [KS][D], later F / Z
    double *Tm = reinterpret_cast<double *>(smem + p.lay.off_tm);    // cos(pi i / 2m), i < 4m
    double *Mj = reinterpret_cast<double *>(smem + p.lay.off_mj);    // [N][K] cos(pi (2j+1) k / 2n)
    __shared__ int s_item, s_flag, s_last, s_last_rider;
    __shared__ double s_mn[kMaxN], s_mx[kMaxN];
    __shared__ int s_bad[kMaxN];

    const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5;
    const int D = LDC ? LDC : p.D;      // specialised widths: D (= ld) is a compile-time constant
    const int m = p.m;
    const int G = p.lay.G, RL = p.lay.RL, CT = p.lay.CT;
    const int nk = m - 1;
    const int DS = max(1, T / nk);
    const int half = D / 2;

    // ---- per-CTA tables (the CTA is persistent: loaded / built once) ----
    for (int i = tid; i < p.lay.table_len; i += T) TT[i] = __ldg(p.table + i);
    for (int i = tid; i < 4 * m; i += T) Tm[i] = cospi((double)i / (2.0 * m));
    for (int i = tid; i < N * K; i += T) {
        const int j = i / K, k = i % K + 1;
        Mj[i] = cospi((double)((2 * j + 1) * k) / (2.0 * N));
    }

    const int rl = (RL > 1) ? tid / G : 0;
    const int g0 = (RL > 1) ? tid % G : tid;
    const bool lane_ok = (RL > 1) ? (rl < RL) : true;

    // Everything after pass 1 for one (domain, layer) whose u[k][d] sums sit in scr[0 .. K*D).
    auto finish = [&](int dom_index, int layer) {
        TIC();
        if (tid == 0) s_flag = 0;
        __syncthreads();
        // ---- length-n inverse + per-column min-max (fingerprint.py:138-140 on [D, n]); Y = y' - 0.5 ----
        for (int d = tid; d < D; d += T) {
            double u[K], y[N];
#pragma unroll
            for (int k = 0; k < K; ++k) u[k] = scr[k * D + d];
            double mn = INFINITY, mx = -INFINITY;
            bool bad = false;
#pragma unroll
            for (int j = 0; j < N; ++j) {
                double s = 0.0;
#pragma unroll
                for (int k = 0; k < K; ++k) s = fma(Mj[j * K + k], u[k], s);
                y[j] = s;
                bad = bad || !(s == s);
                mn = fmin(mn, s);
                mx = fmax(mx, s);
            }
            bad = bad || !(mx > mn);
            if (bad) s_flag = 1;   // constant / non-finite column: the reference yields NaN -> all 0
            const double inv = 1.0 / (mx - mn);
#pragma unroll
            for (int j = 0; j < N; ++j) Y[j * D + d] = (float)((y[j] - mn) * inv - 0.5);
        }
        __syncthreads();
        TOC(8);
        // fold: cos(pi (2(D-1-d)+1) k / 2D) = (-1)^k cos(pi (2d+1) k / 2D), so even k only need
        // e[d] = Y[d] + Y[D-1-d] (kept at index d) and odd k only o[d] = Y[d] - Y[D-1-d] (at D-1-d)
        for (int i = tid; i < N * half; i += T) {
            const int j = i / half, d = i % half;
            const float a = Y[j * D + d], b = Y[j * D + D - 1 - d];
            Y[j * D + d] = a + b;
            Y[j * D + D - 1 - d] = a - b;
        }
        __syncthreads();
        TOC(9);

        // ---- pass 2a: F[j][k] = sum_{d < D/2} (e|o)[j][d] cos(pi (2d+1) k / 2D) (+ middle column) ----
        double *Fp = scr;                                  // [DS][N][nk]
        double *Fr = scr + (size_t)DS * N * nk;            // [N][nk]
        double *Z = Fr + (size_t)N * nk;                   // [N][m]
        for (int w = tid; w < nk * DS; w += T) {
            const int k = 1 + w % nk, ds = w / nk;
            const bool odd = (k & 1) != 0;
            // split boundaries are multiples of 4 so that 16-byte shared loads stay aligned
            int d0 = (int)((int64_t)(half / 4) * ds / DS) * 4;
            int d1 = (ds == DS - 1) ? half : (int)((int64_t)(half / 4) * (ds + 1) / DS) * 4;
            int idx = (int)(((long long)(2 * d0 + 1) * k) % (4LL * D));
            const int s1 = 2 * k, s2 = 4 * k, s3 = 6 * k, s4 = 8 * k;
            double f64[N];
            float f32[N];
#pragma unroll
            for (int j = 0; j < N; ++j) { f64[j] = 0.0; f32[j] = 0.f; }
            int d = d0;
            if constexpr (VEC == 4) {
                // Four columns per step: one 16-byte shared load of e (even k, ascending from Y[j*D + d]) or
                // o (odd k, stored reversed: o[d] at Y[j*D + D-1-d], so the float4 at D-4-d holds
                // o[d+3..d]) and four table values at idx + {0,2k,4k,6k} (the table is extended by 8m entries,
                // so only idx itself wraps).  For odd k the table offsets are taken in reverse order instead of
                // reversing the vector: the loop body is the same for both parities, no divergence.
                const float *yp = odd ? (Y + D - 4 - d0) : (Y + d0);
                const int ystep = odd ? -4 : 4;
                const int o0 = odd ? s3 : 0, o1 = odd ? s2 : s1, o2 = odd ? s1 : s2, o3 = odd ? 0 : s3;
                auto step4 = [&]() {
                    const float c0 = TT[idx + o0], c1 = TT[idx + o1], c2 = TT[idx + o2], c3 = TT[idx + o3];
                    idx += s4;
                    while (idx >= 4 * D) idx -= 4 * D;
#pragma unroll
                    for (int j = 0; j < N; ++j) {
                        const float4 v = *reinterpret_cast<const float4 *>(yp + j * D);
                        f32[j] = fmaf(v.x, c0, f32[j]);
                        f32[j] = fmaf(v.y, c1, f32[j]);
                        f32[j] = fmaf(v.z, c2, f32[j]);
                        f32[j] = fmaf(v.w, c3, f32[j]);
                    }
                    yp += ystep;
                };
                const int n4 = (d1 - d0) / 4;
                int g = 0;
                for (; g + 8 <= n4; g += 8) {               // float32 chains of 32 terms, then float64
#pragma unroll
                    for (int i = 0; i < 8; ++i) step4();
#pragma unroll
                    for (int j = 0; j < N; ++j) { f64[j] += (double)f32[j]; f32[j] = 0.f; }
                }
                for (; g < n4; ++g) step4();
                d = d0 + 4 * n4;
            }
            for (; d < d1; ++d) {           // scalar path / leftovers
                const float c = TT[idx];
                idx += s1;
                if (idx >= 4 * D) idx -= 4 * D;
#pragma unroll
                for (int j = 0; j < N; ++j) {
                    const float v = odd ? Y[j * D + D - 1 - d] : Y[j * D + d];
                    f64[j] += (double)(v * c);
                }
            }
            if ((D & 1) && ds == 0 && !odd) {   // middle column of an odd D pairs with itself
                const float c = TT[(int)(((long long)D * k) % (4LL * D))];
#pragma unroll
                for (int j = 0; j < N; ++j) f64[j] += (double)(Y[j * D + half] * c);
            }
#pragma unroll
            for (int j = 0; j < N; ++j) Fp[((size_t)ds * N + j) * nk + (k - 1)] = f64[j] + (double)f32[j];
        }
        __syncthreads();
        TOC(10);
        for (int i = tid; i < N * nk; i += T) {
            double f = 0.0;
            for (int ds = 0; ds < DS; ++ds) f += Fp[(size_t)ds * N * nk + i];
            Fr[i] = f;
        }
        __syncthreads();
        TOC(11);

        // ---- pass 2b: Z[j][c] = sum_k cos(pi (2c+1) k / 2m) F[j][k] ----
        for (int w = tid; w < N * m; w += T) {
            const int j = w / m, c = w % m;
            int idx = 0;
            const int stepc = 2 * c + 1;
            const double *fr = Fr + j * nk;
            double z = 0.0;
            for (int k = 0; k < nk; ++k) {
                idx += stepc;
                if (idx >= 4 * m) idx -= 4 * m;
                z = fma(Tm[idx], fr[k], z);
            }
            Z[w] = z;
        }
        __syncthreads();
        TOC(12);

        // ---- per-row min-max (one warp per row), *127, truncating int8 cast (fingerprint.py:193-195) ----
        for (int j = warp; j < N; j += (T >> 5)) {
            double mn = INFINITY, mx = -INFINITY;
            int bad = 0;
            for (int c = lane; c < m; c += 32) {
                const double z = Z[j * m + c];
                bad |= !(z == z);
                mn = fmin(mn, z);
                mx = fmax(mx, z);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
                mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
                bad |= __shfl_xor_sync(0xffffffffu, bad, o);
            }
            if (lane == 0) { s_mn[j] = mn; s_mx[j] = mx; s_bad[j] = bad || !(mx > mn); }
        }
        __syncthreads();
        TOC(13);
        const bool layer_bad = s_flag != 0;
        int8_t *out = p.out + (int64_t)dom_index * p.out_stride + (int64_t)layer * (N * m);
        for (int w = tid; w < N * m; w += T) {
            const int j = w / m;
            int q = 0;
            if (!layer_bad && !s_bad[j]) q = (int)(((Z[w] - s_mn[j]) / (s_mx[j] - s_mn[j])) * 127.0);
            out[w] = (int8_t)q;
        }
        __syncthreads();
        TOC(14);
    };

    // publishes this item's partial sums (src[0 .. K*D) in shared memory) of a domain that is assembled
    // from several items; returns true in the CTA that arrives last, with the total in scr[0 .. K*D)
    auto meet = [&](const DomInfo &dm, int layer, int slot, const double *srcsum, int *s_result) -> bool {
        double *slab = p.partials + ((int64_t)dm.slab0 + (int64_t)layer * dm.nsplit) * (K * D);
        double *mine = slab + (int64_t)slot * (K * D);
        for (int i = tid; i < K * D; i += T) mine[i] = srcsum[i];
        __threadfence();
        __syncthreads();
        if (tid == 0) {
            const int ticket = atomicAdd(&p.counters[dm.counter0 + layer], 1);
            *s_result = (ticket == dm.nsplit - 1);
        }
        __syncthreads();
        if (!*s_result) return false;
        __threadfence();
        for (int i = tid; i < K * D; i += T) {
            double s = 0.0;
            for (int sp = 0; sp < dm.nsplit; ++sp) s += __ldcg(slab + (int64_t)sp * (K * D) + i);
            scr[i] = s;
        }
        __syncthreads();
        return true;
    };

    for (;;) {
        TIC();
        __syncthreads();
        if (tid == 0) s_item = atomicAdd(&p.counters[0], 1);
        __syncthreads();
        const int it = s_item;
        if (it >= p.n_items) break;
        TOC(0);
        const Item item = p.items[it];
        const DomInfo dom = p.doms[item.dom];
        const int L = dom.L, r0 = item.r0, r1 = item.r1;
        const bool has_rider = RIDER && item.rider_dom >= 0;

        // ---- basis of this item's rows: c_k = cos(pi (2l+1) k / 2L) by the Chebyshev recurrence
        //      c_k = 2 c_1 c_{k-1} - c_{k-2} in float64 from one cospi per row ----
        for (int r = tid; r < r1 - r0; r += T) {
            const double c1 = cospi((double)(2 * (r0 + r) + 1) / (2.0 * L));
            double ckm2 = 1.0, ckm1 = c1;
            cb2[r * KS] = (float)c1;
#pragma unroll
            for (int k = 2; k <= K; ++k) {
                const double ck = 2.0 * c1 * ckm1 - ckm2;
                cb2[r * KS + k - 1] = (float)ck;
                ckm2 = ckm1;
                ckm1 = ck;
            }
            if constexpr (RIDER) {
#pragma unroll
                for (int k = 0; k < K; ++k) cb2[r * KS + K + k] = 0.f;
            }
        }
        if constexpr (RIDER) {
            if (has_rider) {
                // second basis: the same rows at their position in the whole protein (the rider's own L)
                __syncthreads();
                const int Lg = p.doms[item.rider_dom].L;
                for (int pi = item.piece_first; pi < dom.n_pieces; ++pi) {
                    const Piece pc = p.pieces[dom.piece_off + pi];
                    if (pc.l0 >= r1) break;
                    const int a = max(pc.l0, r0), b = min(pc.l0 + pc.nrows, r1);
                    for (int l = a + tid; l < b; l += T) {
                        const int P = pc.g0 + (l - pc.l0);
                        const double c1 = cospi((double)(2 * P + 1) / (2.0 * Lg));
                        double ckm2 = 1.0, ckm1 = c1;
                        cb2[(l - r0) * KS + K] = (float)c1;
#pragma unroll
                        for (int k = 2; k <= K; ++k) {
                            const double ck = 2.0 * c1 * ckm1 - ckm2;
                            cb2[(l - r0) * KS + K + k - 1] = (float)ck;
                            ckm2 = ckm1;
                            ckm1 = ck;
                        }
                    }
                }
            }
        }
        __syncthreads();
        TOC(1);

        const float *const *src = p.src + (int64_t)item.layer * p.n_src;
        const Piece first = p.pieces[dom.pivot];
        double *rider_slab = nullptr;
        DomInfo gd{};
        if constexpr (RIDER) {
            if (has_rider) {
                gd = p.doms[item.rider_dom];
                rider_slab = p.partials + ((int64_t)gd.slab0 + (int64_t)item.layer * gd.nsplit + item.rider_split) * (K * D);
            }
        }
        for (int ct = 0; ct < CT; ++ct) {
            const int g = g0 + ct * T;
            const bool active = lane_ok && g < G;
            const int col = g * VEC;
            double acc[KS][4];
#pragma unroll
            for (int k = 0; k < KS; ++k)
#pragma unroll
                for (int v = 0; v < 4; ++v) acc[k][v] = 0.0;
            if (active) {
                // pivot: one row subtracted from every row of the domain (row 0 of the domain, or of the
                // protein when the global fingerprint rides along; the same for every item of a domain)
                const float *fa = src[first.src_a] + (int64_t)first.row_a * p.ld + col;
                const float *fb = (first.src_b >= 0) ? src[first.src_b] + (int64_t)first.row_b * p.ld + col : nullptr;
                if constexpr (VEC == 4) {
                    pk2 v0, v1;
                    ldg_stream4(fa, v0, v1);
                    if (fb) {
                        pk2 w0, w1;
                        ldg_stream4(fb, w0, w1);
                        const pk2 hf = pk(0.5f, 0.5f);
                        v0 = mul2(add2(v0, w0), hf);
                        v1 = mul2(add2(v1, w1), hf);
                    }
                    const pk2 neg = pk(-1.f, -1.f);
                    const pk2 npiv0 = mul2(v0, neg), npiv1 = mul2(v1, neg);
                    for (int pi = item.piece_first; pi < dom.n_pieces; ++pi) {
                        const Piece pc = p.pieces[dom.piece_off + pi];
                        if (pc.l0 >= r1) break;
                        const int a = max(pc.l0, r0), b = min(pc.l0 + pc.nrows, r1);
                        if (a >= b) continue;
                        const float *pa = src[pc.src_a] + (int64_t)(pc.row_a + (a - pc.l0)) * p.ld + col;
                        const float *cbp = cb2 + (a - r0) * KS;
                        if (pc.src_b < 0) {
                            stream_piece4<KS, U, false, LDC, RLC>(pa, pa, p.ld, b - a, rl, RL, cbp, npiv0, npiv1, acc);
                        } else {
                            const float *pb = src[pc.src_b] + (int64_t)(pc.row_b + (a - pc.l0)) * p.ld + col;
                            stream_piece4<KS, U, true, LDC, RLC>(pa, pb, p.ld, b - a, rl, RL, cbp, npiv0, npiv1, acc);
                        }
                    }
                } else {
                    float piv = ldg_stream1(fa);
                    if (fb) piv = (piv + ldg_stream1(fb)) * 0.5f;
                    for (int pi = item.piece_first; pi < dom.n_pieces; ++pi) {
                        const Piece pc = p.pieces[dom.piece_off + pi];
                        if (pc.l0 >= r1) break;
                        const int a = max(pc.l0, r0), b = min(pc.l0 + pc.nrows, r1);
                        if (a >= b) continue;
                        const float *pa = src[pc.src_a] + (int64_t)(pc.row_a + (a - pc.l0)) * p.ld + col;
                        const float *cbp = cb2 + (a - r0) * KS;
                        if (pc.src_b < 0) {
                            stream_piece1<KS, false>(pa, pa, p.ld, b - a, rl, RL, cbp, piv, acc);
                        } else {
                            const float *pb = src[pc.src_b] + (int64_t)(pc.row_b + (a - pc.l0)) * p.ld + col;
                            stream_piece1<KS, true>(pa, pb, p.ld, b - a, rl, RL, cbp, piv, acc);
                        }
                    }
                }
            }
            // ---- u[k][d] into shared memory, row lanes added in a fixed order ----
            if (RL == 1) {
                if (active) {
#pragma unroll
                    for (int k = 0; k < K; ++k)
#pragma unroll
                        for (int v = 0; v < VEC; ++v)
                            if (col + v < D) scr[k * D + col + v] = acc[k][v];
                    if constexpr (RIDER) {
                        if (has_rider) {       // the rider's sums go straight to its partial-sum slab
#pragma unroll
                            for (int k = 0; k < K; ++k)
#pragma unroll
                                for (int v = 0; v < VEC; ++v)
                                    if (col + v < D) rider_slab[k * D + col + v] = acc[K + k][v];
                        }
                    }
                }
            } else {
                for (int r = 0; r < RL; ++r) {
                    if (active && rl == r) {
#pragma unroll
                        for (int k = 0; k < KS; ++k)
#pragma unroll
                            for (int v = 0; v < VEC; ++v)
                                if (col + v < D) {
                                    if (r == 0) scr[k * D + col + v] = acc[k][v];
                                    else scr[k * D + col + v] += acc[k][v];
                                }
                    }
                    __syncthreads();
                }
            }
        }
        __syncthreads();
        TOC(2);

        // ---- the protein's global fingerprint riding on this item: hand its partial sums over ----
        bool rider_last = false;
        if constexpr (RIDER) {
            if (has_rider) {
                // with row lanes the rider's sums were reduced in scr[K*D .. 2*K*D) (the item's own sums in
                // scr[0 .. K*D) stay untouched); with one thread per column group they are already in the slab
                if (RL > 1)
                    for (int i = tid; i < K * D; i += T) rider_slab[i] = scr[K * D + i];
                __threadfence();
                __syncthreads();
                if (tid == 0) {
                    const int ticket = atomicAdd(&p.counters[gd.counter0 + item.layer], 1);
                    s_last_rider = (ticket == gd.nsplit - 1);
                }
                __syncthreads();
                rider_last = s_last_rider != 0;
            }
        }

        TOC(3);
        // ---- this item's own domain ----
        bool own_ready = true;
        if (dom.counter0 >= 0) own_ready = meet(dom, item.layer, item.split, scr, &s_last);
        TOC(4);
        if (own_ready) finish(item.dom, item.layer);
        TOC(5);

        if constexpr (RIDER) {
            if (rider_last) {
                double *slab = p.partials + ((int64_t)gd.slab0 + (int64_t)item.layer * gd.nsplit) * (K * D);
                __threadfence();
                for (int i = tid; i < K * D; i += T) {
                    double s = 0.0;
                    for (int sp = 0; sp < gd.nsplit; ++sp) s += __ldcg(slab + (int64_t)sp * (K * D) + i);
                    scr[i] = s;
                }
                __syncthreads();
                finish(item.rider_dom, item.layer);
            }
        }
        TOC(6);
    }
}

#include "fp_ws_kernel.cuh"

// ------------------------------------------------------------------------------------------
// host: layout, planner, launch
// ------------------------------------------------------------------------------------------
#ifdef DCTD_DEBUG_U
double *g_debug_u = nullptr;
#endif
#ifdef DCTD_TUNING
// process-global A/B switches: tuning builds only (libdctd_tuning.so, dctd_fp_set_variant).  The release library has
// no mutable global state: per-plan options travel in the flags of dctd_fp_plan_create_ex.
int g_variant = 0;
int g_ws_stages = 0; // cap on the TMA ring stages of the warp-specialised kernel (0 = as many as fit)
#else
constexpr int g_variant = 0;
constexpr int g_ws_stages = 0;
#endif

// Host blobs of the plans (pinned when a device is present) are recycled through a small cache: cudaHostAlloc /
// mmap + page faults per plan cost more than building the plan (0.7 -> 0.3 ms for 512 proteins).  This is memory
// management only: a blob carries no state from one plan to the next.
struct HostBlob { void *p; size_t bytes; bool pinned; };
std::mutex g_blob_mu;
std::vector<HostBlob> g_blobs;
size_t g_blob_cached = 0;
constexpr size_t kBlobCacheBytes = 256u << 20;
constexpr size_t kBlobCacheEntries = 16;

void blob_free(const HostBlob &b) {
    if (b.pinned) cudaFreeHost(b.p);
    else free(b.p);
}
HostBlob blob_acquire(size_t bytes) {
    {
        std::lock_guard<std::mutex> lk(g_blob_mu);
        int best = -1;
        for (int i = 0; i < (int)g_blobs.size(); ++i)
            if (g_blobs[i].bytes >= bytes && g_blobs[i].bytes <= 4 * bytes + (1u << 20) &&
                (best < 0 || g_blobs[i].bytes < g_blobs[best].bytes)) best = i;
        if (best >= 0) {
            HostBlob b = g_blobs[best];
            g_blobs.erase(g_blobs.begin() + best);
            g_blob_cached -= b.bytes;
            return b;
        }
    }
    HostBlob b{nullptr, dctd::align_up(bytes + bytes / 4, 64u << 10), false};
    if (cudaHostAlloc(&b.p, b.bytes, cudaHostAllocDefault) == cudaSuccess) {
        b.pinned = true;
    } else {
        (void)cudaGetLastError();   // no device (CPU-only planning): plain host memory
        b.p = malloc(b.bytes);
    }
    return b;
}
void blob_release(const HostBlob &b) {
    std::vector<HostBlob> drop;
    {
        std::lock_guard<std::mutex> lk(g_blob_mu);
        g_blobs.push_back(b);
        g_blob_cached += b.bytes;
        while (g_blobs.size() > kBlobCacheEntries || g_blob_cached > kBlobCacheBytes) {
            drop.push_back(g_blobs.front());
            g_blob_cached -= g_blobs.front().bytes;
            g_blobs.erase(g_blobs.begin());
        }
    }
    for (const HostBlob &d : drop) blob_free(d);
}

// Queue order of the items.  The persistent CTAs pull items from one atomic queue.  Longest first (LPT) balances the
// tail, but it also makes every CTA stream long items at the start of the launch (HBM-bound, finisher warps idle) and
// short ones at its end (finisher-bound: an item's passes 2 cost ~19 k cycles whatever its length, HBM idle).  So the
// short items - fewer rows than the finishers need to keep up, ~480 KB of input - are spread evenly, by rows, over the
// long ones, which stay in descending order; the last long items (just above the balance length) carry no short ones
// and even out the tail.
void spread_short_items(std::vector<Item> &items, int D) {
    const int balance = std::max(8, 491520 / (D * 4));
    auto len = [](const Item &a) { return a.r1 - a.r0; };
    size_t nb = 0;
    while (nb < items.size() && len(items[nb]) >= balance) ++nb;       // items are sorted longest first
    const size_t ns = items.size() - nb;
    if (nb == 0 || ns == 0) return;
    const size_t reserve = std::min<size_t>(nb / 8, 296);
    int64_t rows_big = 0;
    for (size_t i = 0; i + reserve < nb; ++i) rows_big += len(items[i]);
    std::vector<Item> out;
    out.reserve(items.size());
    size_t j = 0;
    int64_t cum = 0;
    for (size_t i = 0; i < nb; ++i) {
        out.push_back(items[i]);
        if (i + reserve >= nb) continue;
        cum += len(items[i]);
        // short item j is due once (j + 0.5) / ns of the long rows have been queued
        while (j < ns && (2 * (int64_t)j + 1) * rows_big <= 2 * cum * (int64_t)ns) out.push_back(items[nb + j++]);
        if (i + reserve + 1 == nb)
            while (j < ns) out.push_back(items[nb + j++]);
    }
    while (j < ns) out.push_back(items[nb + j++]);
    items.swap(out);
}

Layout make_layout(int D, int n, int m, bool vec4, bool rider) {
    Layout l{};
    const int K = n - 1;
    const int KS = rider ? 2 * K : K;
    l.vec = vec4 ? 4 : 1;
    l.G = (D + l.vec - 1) / l.vec;
    if (l.G <= kMaxThreads) {
        l.CT = 1;
        // one thread per column group when that still fills >= 4 warps (more, smaller CTAs per SM overlap the
        // non-streaming phases better); narrower embeddings share a CTA between several row lanes
        l.RL = (l.G >= 128 && g_variant != 5) ? 1 : std::max(1, 320 / l.G);
        l.T = (l.G * l.RL + 31) / 32 * 32;
    } else {
        l.CT = (l.G + kMaxThreads - 1) / kMaxThreads;
        l.RL = 1;
        l.T = ((l.G + l.CT - 1) / l.CT + 31) / 32 * 32;
    }
    l.T = std::max(l.T, 128);
    const int nk = m - 1;
    const int DS = std::max(1, l.T / nk);
    l.table_len = 4 * D + 8 * m;
    // Shared memory is kept small on purpose: what the CTAs of an SM do not take is L1, and the L1 size bounds
    // the loads in flight.  (Tried: letting Y alias the scratch region behind the pass-2 buffers, -9 KB; the extra
    // barrier cost more than the larger L1 gave: 5500 vs 5590 GB/s in an A/B run.)
    const size_t f_region = ((size_t)DS * n * nk + (size_t)n * nk + (size_t)n * m) * sizeof(double);
    size_t off = 0;
    l.off_t4d = off; off += dctd::align_up((size_t)l.table_len * sizeof(float), 16);
    l.off_cb = off;  off += dctd::align_up((size_t)kRowsPerItem * KS * sizeof(float), 16);
    const size_t u_bytes = (size_t)(l.RL > 1 ? KS : K) * D * sizeof(double);
    l.off_scr = off; off += dctd::align_up(std::max(u_bytes, f_region), 16);
    l.off_y = off;   off += dctd::align_up((size_t)n * D * sizeof(float), 16);
    l.off_tm = off;  off += dctd::align_up((size_t)4 * m * sizeof(double), 16);
    l.off_mj = off;  off += dctd::align_up((size_t)n * K * sizeof(double), 16);
    l.smem = off;
    return l;
}

// shared-memory layout of fp_ws_kernel<K, D, *>; nst = 0 if not even three stages fit
template <int K, int DC, bool RIDER>
WsLayout make_ws_layout(int m, int max_smem) {
    using Cfg = WsCfg<K, DC, RIDER>;
    WsLayout w{};
    const int N = K + 1, nk = m - 1;
    // pass 2a: a thread owns the coefficient pair (k, k + H), H = 0 (mod 4) so that both are of one class mod 4; the
    // D/4 folded columns are split over DSe thread groups for the even pairs and twice as many for the odd ones (an odd
    // pair costs twice as much per column): (H/2) * (DSo + DSe) units for the 256 finisher threads
    w.H = ((nk + 1) / 2 + 3) / 4 * 4;
    const int QQ = std::max(1, DC / 16);
    w.DSe = std::max(1, std::min(kWsFinThreads / (3 * (w.H / 2)), QQ / 2));
    w.DSo = std::min(2 * w.DSe, QQ);
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += dctd::align_up(bytes, 128); return (unsigned)o; };
    w.off_bars = take((2 * kWsMaxStages + 2 * kWsMaxUBufs) * sizeof(unsigned long long));
    w.off_meta = take(kWsMaxStages * sizeof(int4));
    w.off_basis = take((size_t)kWsBasisRows * Cfg::KS * sizeof(float));
    w.off_desc = take((size_t)kWsDescSlots * 32 * sizeof(int));
    w.off_u = take((size_t)Cfg::NB * K * DC * sizeof(double));
    w.off_ye = take((size_t)N * (DC / 2) * sizeof(float));
    w.off_yo = take((size_t)N * (DC / 2) * sizeof(float));
    w.off_f = take(((size_t)(w.DSo + w.DSe) * N * w.H + (size_t)N * nk + (size_t)N * m) * sizeof(double));
    w.off_tt = take((size_t)(4 * DC + 8 * m) * sizeof(float));
    w.off_tm = take((size_t)(4 * m + (4 * m >> 4) + 1) * sizeof(double));     // skewed: entry i at i + (i >> 4)
    w.off_mj = take((size_t)N * K * sizeof(double));
    w.off_ring = take(0);
    const long long room = (long long)max_smem - (long long)off - 1024;      // 1 KB for the static shared variables
    long long nst = room / Cfg::STAGE_BYTES;
    if (g_ws_stages > 0) nst = std::min<long long>(nst, g_ws_stages);
    nst = std::min<long long>(nst, kWsMaxStages);
    w.nst = nst >= 3 ? (int)nst : 0;
    if (N * ((m + 1) / 2) * 2 > kWsFinThreads || w.H < 1) w.nst = 0;      // pass 2b runs as one pass of the finisher threads
    w.smem = (unsigned)(off + (size_t)std::max(w.nst, 0) * Cfg::STAGE_BYTES);
    return w;
}

typedef void (*KernelFn)(const Params);
template <int VEC, int U, int MAXT, int MINB>
KernelFn pick_k(int K) {
    switch (K) {
        case 1: return fp_kernel<1, VEC, U, MAXT, MINB>;
        case 2: return fp_kernel<2, VEC, U, MAXT, MINB>;
        case 3: return fp_kernel<3, VEC, U, MAXT, MINB>;
        case 4: return fp_kernel<4, VEC, U, MAXT, MINB>;
        case 5: return fp_kernel<5, VEC, U, MAXT, MINB>;
        case 6: return fp_kernel<6, VEC, U, MAXT, MINB>;
        case 7: return fp_kernel<7, VEC, U, MAXT, MINB>;
    }
    return nullptr;
}

template <int VEC, int MAXT, int MINB>
KernelFn pick_rider(int K) {
    switch (K) {
        case 1: return fp_kernel<1, VEC, 8, MAXT, MINB, 0, 0, true>;
        case 2: return fp_kernel<2, VEC, 8, MAXT, MINB, 0, 0, true>;
        case 3: return fp_kernel<3, VEC, 8, MAXT, MINB, 0, 0, true>;
    }
    return nullptr;
}

// launches fp_ws_kernel<K, DC, RIDER> if its shared-memory layout fits; *launched tells
template <int K, int DC, bool RIDER>
int launch_ws(const dctd_fp_plan *plan, Params &prm, int max_smem, int n_sm, cudaStream_t stream, bool *launched) {
    using Cfg = WsCfg<K, DC, RIDER>;
    *launched = false;
    prm.wl = make_ws_layout<K, DC, RIDER>(plan->m, max_smem);
    if (prm.wl.nst == 0) return DCTD_OK;
    auto fn = fp_ws_kernel<K, DC, RIDER>;
    DCTD_CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)prm.wl.smem));
    const int grid = std::max(1, std::min(prm.n_items, n_sm));     // one persistent CTA per SM
    fn<<<grid, Cfg::T, prm.wl.smem, stream>>>(prm);
    DCTD_LAUNCH_CHECK();
    *launched = true;
    return DCTD_OK;
}

template <int DC>
int launch_ws_d(const dctd_fp_plan *plan, Params &prm, int max_smem, int n_sm, cudaStream_t stream, bool *launched) {
    return plan->has_rider ? launch_ws<2, DC, true>(plan, prm, max_smem, n_sm, stream, launched)
                           : launch_ws<2, DC, false>(plan, prm, max_smem, n_sm, stream, launched);
}

}  // namespace

extern "C" {

int dctd_fp_plan_create(const dctd_fp_geometry *geo, dctd_fp_plan **out_plan) {
    return dctd_fp_plan_create_ex(geo, 0u, out_plan);
}

int dctd_fp_plan_create_ex(const dctd_fp_geometry *geo, uint32_t flags, dctd_fp_plan **out_plan) {
    if (!geo || !out_plan) return DCTD_ERR_ARG;
    *out_plan = nullptr;
    if (flags & ~(DCTD_FP_PLAN_NO_FUSION | DCTD_FP_PLAN_GENERAL_KERNEL | DCTD_FP_PLAN_LONGEST_FIRST)) return DCTD_ERR_ARG;
    if (geo->n_layers < 1 || geo->D < 1 || geo->n < 2 || geo->n > kMaxN || geo->m < 2 ||
        geo->m > kMaxM || geo->m > geo->D || geo->n_src < 0 || geo->n_prot < 0 || geo->n_dom < 0)
        return DCTD_ERR_ARG;
    if (geo->n_dom > 0 && (!geo->dom_prot || !geo->dom_seg_off || !geo->seg_beg || !geo->seg_end ||
                           !geo->src_rows || !geo->prot_src0 || !geo->prot_nsrc))
        return DCTD_ERR_ARG;
    const int stride = geo->maxlen - geo->overlap;
    dctd_fp_plan *pl = new (std::nothrow) dctd_fp_plan();
    if (!pl) return DCTD_ERR_NOMEM;
    pl->n_layers = geo->n_layers; pl->D = geo->D; pl->n = geo->n; pl->m = geo->m;
    pl->n_src = geo->n_src; pl->n_dom = geo->n_dom;
    pl->flags = flags;
    pl->blob = nullptr; pl->blob_pinned = false; pl->blob_bytes = 0; pl->blob_capacity = 0;
    pl->has_event = false;
    pl->algo_bytes = 0;
    int rc = DCTD_OK;
    try {
        // protein lengths
        std::vector<int64_t> plen((size_t)geo->n_prot);
        for (int p = 0; p < geo->n_prot && rc == DCTD_OK; ++p) {
            const int s0 = geo->prot_src0[p], ns = geo->prot_nsrc[p];
            if (ns < 1 || s0 < 0 || (int64_t)s0 + ns > geo->n_src) { rc = DCTD_ERR_ARG; break; }
            if (ns == 1) { plen[p] = geo->src_rows[s0]; continue; }
            if (geo->overlap < 0 || stride <= 0) { rc = DCTD_ERR_ARG; break; }
            if (stride < geo->overlap) { rc = DCTD_ERR_UNSUPPORTED; break; }  // rows in > 2 windows
            for (int c = 0; c < ns - 1; ++c)
                if (geo->src_rows[s0 + c] != geo->maxlen) { rc = DCTD_ERR_ARG; break; }
            const int last = geo->src_rows[s0 + ns - 1];
            if (last <= geo->overlap || last > geo->maxlen) rc = DCTD_ERR_ARG;
            plen[p] = (int64_t)(ns - 1) * stride + last;
        }
        int32_t n_counters = 1;
        int64_t n_slabs = 0;
        pl->doms.resize((size_t)geo->n_dom);
        pl->has_rider = false;

        // rows [b, e) of protein p -> pieces (cut where the window coverage changes); l0 = domain-local index
        auto add_pieces = [&](int p, int64_t b, int64_t e, int64_t l0) {
            const int s0 = geo->prot_src0[p], ns = geo->prot_nsrc[p];
            while (b < e) {
                Piece pc{};
                int64_t run_end;
                if (ns == 1) {
                    pc.src_a = s0; pc.row_a = (int32_t)b; pc.src_b = -1; pc.row_b = 0;
                    run_end = e;
                } else {
                    int64_t c = std::min<int64_t>(b / stride, ns - 1);
                    const int64_t off = b - c * stride;
                    if (c >= 1 && off < geo->overlap) {   // covered by windows c-1 and c
                        pc.src_a = s0 + (int32_t)c - 1; pc.row_a = (int32_t)(off + stride);
                        pc.src_b = s0 + (int32_t)c;     pc.row_b = (int32_t)off;
                        run_end = std::min<int64_t>(e, c * stride + geo->overlap);
                    } else {
                        pc.src_a = s0 + (int32_t)c; pc.row_a = (int32_t)off; pc.src_b = -1; pc.row_b = 0;
                        run_end = (c < ns - 1) ? std::min<int64_t>(e, (c + 1) * stride) : e;
                    }
                }
                pc.nrows = (int32_t)(run_end - b);
                pc.l0 = (int32_t)l0;
                pc.g0 = (int32_t)b;
                pl->pieces.push_back(pc);
                l0 += pc.nrows;
                b = run_end;
            }
        };

        // rows a run of pieces reads: a row averaged from two windows is two distinct rows of input
        auto piece_rows_read = [&](int32_t off, int32_t n) {
            int64_t r = 0;
            for (int32_t i = 0; i < n; ++i) r += (int64_t)pl->pieces[off + i].nrows * (pl->pieces[off + i].src_b >= 0 ? 2 : 1);
            return r;
        };

        // ---- validation + fusion analysis: a protein whose batch holds its global domain (one segment
        //      covering every row) next to other, pairwise disjoint domains reads each row once: the other
        //      domains' items carry the global fingerprint along ("rider"), the global domain itself only
        //      streams the rows no other domain covers ----
        std::vector<int64_t> dom_len((size_t)geo->n_dom, 0);
        for (int i = 0; i < geo->n_dom && rc == DCTD_OK; ++i) {
            const int p = geo->dom_prot[i];
            if (p < 0 || p >= geo->n_prot) { rc = DCTD_ERR_ARG; break; }
            for (int j = geo->dom_seg_off[i]; j < geo->dom_seg_off[i + 1]; ++j) {
                const int64_t b = geo->seg_beg[j], e = geo->seg_end[j];
                if (b < 0 || e > plen[p] || e < b) { rc = DCTD_ERR_ARG; break; }
                dom_len[i] += e - b;
            }
            if (rc == DCTD_OK && (dom_len[i] < geo->n || dom_len[i] > (1 << 26))) rc = DCTD_ERR_ARG;  // reference: reshape fails for L < n
        }
        std::vector<int32_t> global_of((size_t)geo->n_prot, -1);   // fused proteins: index of the global domain
        // domains grouped by protein and the filler ranges of the fused proteins, both as offset + flat arrays
        std::vector<int32_t> bp_off((size_t)geo->n_prot + 1, 0), bp((size_t)geo->n_dom);
        std::vector<int32_t> fill_off((size_t)geo->n_prot + 1, 0);
        std::vector<std::pair<int64_t, int64_t>> fill;
        if (rc == DCTD_OK && !(flags & DCTD_FP_PLAN_NO_FUSION) && geo->n <= 4) {      // rider kernels are built for n <= 4 (2n - 2 projections)
            for (int i = 0; i < geo->n_dom; ++i) ++bp_off[geo->dom_prot[i] + 1];
            for (int p = 0; p < geo->n_prot; ++p) bp_off[p + 1] += bp_off[p];
            {
                std::vector<int32_t> cur(bp_off.begin(), bp_off.end() - 1);
                for (int i = 0; i < geo->n_dom; ++i) bp[cur[geo->dom_prot[i]]++] = i;
            }
            std::vector<std::pair<int64_t, int64_t>> segs;
            for (int p = 0; p < geo->n_prot; ++p) {
                fill_off[p + 1] = (int32_t)fill.size();
                const int32_t *mine = bp.data() + bp_off[p];
                const int n_mine = bp_off[p + 1] - bp_off[p];
                int gdom = -1;
                for (int t = 0; t < n_mine; ++t) {
                    const int i = mine[t], j = geo->dom_seg_off[i];
                    if (geo->dom_seg_off[i + 1] - j == 1 && geo->seg_beg[j] == 0 && geo->seg_end[j] == plen[p]) { gdom = i; break; }
                }
                if (gdom < 0 || n_mine < 2) continue;
                segs.clear();
                bool sorted = true;
                for (int t = 0; t < n_mine; ++t) {
                    const int i = mine[t];
                    if (i == gdom) continue;
                    for (int j = geo->dom_seg_off[i]; j < geo->dom_seg_off[i + 1]; ++j)
                        if (geo->seg_end[j] > geo->seg_beg[j]) {
                            if (!segs.empty() && geo->seg_beg[j] < segs.back().first) sorted = false;
                            segs.emplace_back(geo->seg_beg[j], geo->seg_end[j]);
                        }
                }
                if (!sorted) std::sort(segs.begin(), segs.end());
                bool disjoint = true;
                for (size_t t = 1; t < segs.size(); ++t)
                    if (segs[t].first < segs[t - 1].second) { disjoint = false; break; }
                if (!disjoint) continue;
                global_of[p] = gdom;
                int64_t pos = 0;
                for (auto &sg : segs) {
                    if (sg.first > pos) fill.emplace_back(pos, sg.first);
                    pos = sg.second;
                }
                if (pos < plen[p]) fill.emplace_back(pos, plen[p]);
                fill_off[p + 1] = (int32_t)fill.size();
            }
        }
        pl->pieces.reserve((geo->n_dom > 0 ? (size_t)geo->dom_seg_off[geo->n_dom] : 0) + 2 * (size_t)geo->n_prot + fill.size());
        pl->items.reserve((size_t)geo->n_layers * ((size_t)geo->n_dom + fill.size()) * 5 / 4 + 16);

        // ---- pieces, domains, items ----
        std::vector<int32_t> pivot_piece((size_t)geo->n_prot, -1);
        std::vector<int32_t> rider_next((size_t)geo->n_dom, 0);   // next free partial-sum slot of a fused global domain
        // first the fused global domains (their slot numbering starts with their own filler items)
        for (int i = 0; i < geo->n_dom && rc == DCTD_OK; ++i) {
            const int p = geo->dom_prot[i];
            const bool fused_global = global_of[p] == i;
            if (!fused_global) continue;
            DomInfo di{};
            di.piece_off = (int32_t)pl->pieces.size();
            for (int32_t t = fill_off[p]; t < fill_off[p + 1]; ++t) add_pieces(p, fill[t].first, fill[t].second, fill[t].first);
            di.n_pieces = (int32_t)pl->pieces.size() - di.piece_off;
            di.L = (int32_t)dom_len[i];
            pivot_piece[p] = (int32_t)pl->pieces.size();
            add_pieces(p, 0, 1, 0);                       // the protein's first row: pivot of all its domains
            di.pivot = pivot_piece[p];
            // contributors: filler items + every item of the other domains of the protein
            int n_fill = 0;
            for (int pi = 0; pi < di.n_pieces; ++pi)
                n_fill += (pl->pieces[di.piece_off + pi].nrows + kRowsPerItem - 1) / kRowsPerItem;
            int n_ride = 0;
            for (int32_t t = bp_off[p]; t < bp_off[p + 1]; ++t)
                if (const int o = bp[t]; o != i) n_ride += (int)((dom_len[o] + kRowsPerItem - 1) / kRowsPerItem);
            di.nsplit = n_fill + n_ride;
            di.slab0 = (int32_t)n_slabs;
            n_slabs += (int64_t)di.nsplit * geo->n_layers;
            di.counter0 = n_counters;
            n_counters += geo->n_layers;
            pl->doms[i] = di;
            rider_next[i] = n_fill;
            pl->algo_bytes += (int64_t)geo->n_layers * geo->D * 4 * piece_rows_read(di.piece_off, di.n_pieces);
            for (int layer = 0; layer < geo->n_layers; ++layer) {
                int slot = 0;
                for (int pi = 0; pi < di.n_pieces; ++pi) {
                    const Piece &pc = pl->pieces[di.piece_off + pi];
                    for (int c0 = 0; c0 < pc.nrows; c0 += kRowsPerItem) {
                        Item itm{};
                        itm.dom = i; itm.layer = layer; itm.split = slot++;
                        itm.r0 = pc.l0 + c0; itm.r1 = pc.l0 + std::min(pc.nrows, c0 + kRowsPerItem);
                        itm.piece_first = pi; itm.rider_dom = -1; itm.rider_split = 0;
                        pl->items.push_back(itm);
                    }
                }
            }
        }
        if (n_slabs > 0x7fffffff / 2) rc = DCTD_ERR_UNSUPPORTED;
        for (int i = 0; i < geo->n_dom && rc == DCTD_OK; ++i) {
            const int p = geo->dom_prot[i];
            if (global_of[p] == i) continue;
            const int gdom = global_of[p];
            DomInfo di{};
            di.piece_off = (int32_t)pl->pieces.size();
            int64_t l0 = 0;
            for (int j = geo->dom_seg_off[i]; j < geo->dom_seg_off[i + 1]; ++j) {
                add_pieces(p, geo->seg_beg[j], geo->seg_end[j], l0);
                l0 += geo->seg_end[j] - geo->seg_beg[j];
            }
            di.n_pieces = (int32_t)pl->pieces.size() - di.piece_off;
            di.L = (int32_t)l0;
            di.nsplit = (int32_t)((l0 + kRowsPerItem - 1) / kRowsPerItem);
            di.slab0 = -1; di.counter0 = -1;
            di.pivot = gdom >= 0 ? pivot_piece[p] : di.piece_off;
            if (di.nsplit > 1) {
                di.slab0 = (int32_t)n_slabs;
                n_slabs += (int64_t)di.nsplit * geo->n_layers;
                di.counter0 = n_counters;
                n_counters += geo->n_layers;
            }
            pl->doms[i] = di;
            pl->algo_bytes += (int64_t)geo->n_layers * geo->D * 4 * piece_rows_read(di.piece_off, di.n_pieces);
            const int rps = (int)((l0 + di.nsplit - 1) / di.nsplit);
            const int ride0 = gdom >= 0 ? rider_next[gdom] : 0;
            if (gdom >= 0) { rider_next[gdom] += di.nsplit; pl->has_rider = true; }
            for (int layer = 0; layer < geo->n_layers; ++layer) {
                int pf = 0;
                for (int s = 0; s < di.nsplit; ++s) {
                    Item itm{};
                    itm.dom = i; itm.layer = layer; itm.split = s;
                    itm.r0 = s * rps; itm.r1 = (int32_t)std::min<int64_t>(l0, (int64_t)(s + 1) * rps);
                    while (pf < di.n_pieces) {
                        const Piece &pc = pl->pieces[di.piece_off + pf];
                        if (pc.l0 + pc.nrows > itm.r0) break;
                        ++pf;
                    }
                    itm.piece_first = pf;
                    itm.rider_dom = gdom; itm.rider_split = gdom >= 0 ? ride0 + s : 0;
                    pl->items.push_back(itm);
                }
            }
        }
        if (rc == DCTD_OK) {
            // longest items first: the atomic work queue then behaves like LPT scheduling
            {   // stable counting sort by length (an item has at most kRowsPerItem rows)
                std::vector<int32_t> start((size_t)kRowsPerItem + 2, 0);
                auto bucket = [](const Item &it) { return kRowsPerItem - std::min(std::max(it.r1 - it.r0, 0), kRowsPerItem); };
                for (const Item &it : pl->items) ++start[bucket(it) + 1];
                for (int l = 0; l <= kRowsPerItem; ++l) start[l + 1] += start[l];
                std::vector<Item> sorted(pl->items.size());
                for (const Item &it : pl->items) sorted[start[bucket(it)]++] = it;
                pl->items.swap(sorted);
            }
            if (!(flags & DCTD_FP_PLAN_LONGEST_FIRST)) spread_short_items(pl->items, geo->D);
            pl->n_counters = n_counters;
            pl->n_slabs = n_slabs;
            size_t off = 0;
            pl->off_pieces = off; off += dctd::align_up(pl->pieces.size() * sizeof(Piece), 256);
            pl->off_doms = off;   off += dctd::align_up(pl->doms.size() * sizeof(DomInfo), 256);
            pl->off_items = off;  off += dctd::align_up(pl->items.size() * sizeof(Item), 256);
            pl->off_wsitems = off; off += dctd::align_up(pl->items.size() * 32 * sizeof(int32_t), 256);
            pl->blob_bytes = off;
            pl->off_src = off;      off += dctd::align_up((size_t)geo->n_layers * geo->n_src * sizeof(void *), 256);
            pl->off_counters = off; off += dctd::align_up((size_t)n_counters * sizeof(int), 256);
            pl->off_timing = off;   off += 256;
            pl->off_table = off;    off += dctd::align_up((size_t)(4 * geo->D + 8 * geo->m) * sizeof(float), 256);
            pl->off_partials = off; off += dctd::align_up((size_t)n_slabs * (geo->n - 1) * geo->D * sizeof(double), 256);
            pl->total = off;
            int32_t *records = nullptr;
            if (pl->blob_bytes) {
                const HostBlob hb = blob_acquire(pl->blob_bytes);
                if (!hb.p) {
                    rc = DCTD_ERR_NOMEM;
                } else {
                    char *h = (char *)hb.p;
                    pl->blob = hb.p; pl->blob_pinned = hb.pinned; pl->blob_capacity = hb.bytes;
                    if (!pl->pieces.empty()) memcpy(h + pl->off_pieces, pl->pieces.data(), pl->pieces.size() * sizeof(Piece));
                    if (!pl->doms.empty()) memcpy(h + pl->off_doms, pl->doms.data(), pl->doms.size() * sizeof(DomInfo));
                    if (!pl->items.empty()) memcpy(h + pl->off_items, pl->items.data(), pl->items.size() * sizeof(Item));
                    records = (int32_t *)(h + pl->off_wsitems);
                    memset(records, 0, pl->items.size() * 32 * sizeof(int32_t));
                }
            }
            // fat item records of the warp-specialised kernel: everything its producer / finisher warps need
            // about an item in one 128-byte read (see the word indices in fp_ws_kernel.cuh), built in place
            for (size_t t = 0; records && t < pl->items.size(); ++t) {
                const Item &itm = pl->items[t];
                const DomInfo &di = pl->doms[itm.dom];
                int32_t *w = records + t * 32;
                w[kWDom] = itm.dom; w[kWLayer] = itm.layer; w[kWR0] = itm.r0; w[kWR1] = itm.r1; w[kWL] = di.L;
                int32_t fl = 0;
                w[kWSplit] = itm.split; w[kWNsplit] = di.nsplit;
                w[kWSlabBase] = -1; w[kWCounter] = -1;
                if (di.counter0 >= 0) {
                    fl |= kWfSplit;
                    w[kWSlabBase] = di.slab0 + itm.layer * di.nsplit;
                    w[kWCounter] = di.counter0 + itm.layer;
                }
                w[kWRiderDom] = itm.rider_dom;
                w[kWLg] = 1;
                if (itm.rider_dom >= 0) {
                    const DomInfo &gd = pl->doms[itm.rider_dom];
                    fl |= kWfRider;
                    w[kWRiderSlabBase] = gd.slab0 + itm.layer * gd.nsplit;
                    w[kWRiderSlab] = w[kWRiderSlabBase] + itm.rider_split;
                    w[kWRiderNsplit] = gd.nsplit;
                    w[kWRiderCounter] = gd.counter0 + itm.layer;
                    w[kWLg] = gd.L;
                }
                const Piece &pv = pl->pieces[di.pivot];
                w[kWPivSrcA] = pv.src_a; w[kWPivRowA] = pv.row_a; w[kWPivSrcB] = pv.src_b; w[kWPivRowB] = pv.row_b;
                int n_runs = 0;
                for (int pi = itm.piece_first; pi < di.n_pieces; ++pi) {
                    const Piece &pc = pl->pieces[di.piece_off + pi];
                    if (pc.l0 >= itm.r1) break;
                    const int a = std::max(pc.l0, itm.r0), b = std::min(pc.l0 + pc.nrows, itm.r1);
                    if (a >= b) { rc = DCTD_ERR_ARG; break; }      // pieces of an item are contiguous by construction
                    if (n_runs == 0) {
                        w[kWRunSrcA] = pc.src_a; w[kWRunRowA] = pc.row_a + (a - pc.l0);
                        w[kWRunSrcB] = pc.src_b; w[kWRunRowB] = pc.row_b + (a - pc.l0);
                        w[kWRunRows] = b - a; w[kWRunL0] = a; w[kWRunG0] = pc.g0 + (a - pc.l0);
                        w[kWPieceAbs] = di.piece_off + pi;
                    }
                    ++n_runs;
                }
                w[kWNRuns] = n_runs;
                if (n_runs > 0 && w[kWRunSrcA] == pv.src_a && w[kWRunRowA] == pv.row_a && w[kWRunSrcB] == pv.src_b &&
                    (pv.src_b < 0 || w[kWRunRowB] == pv.row_b))
                    fl |= kWfPivotInline;
                w[kWFlags] = fl;
            }
        }
    } catch (const std::bad_alloc &) {
        rc = DCTD_ERR_NOMEM;
    }
    if (rc != DCTD_OK) {
        dctd_fp_plan_destroy(pl);
        return rc;
    }
    *out_plan = pl;
    return DCTD_OK;
}

void dctd_fp_plan_destroy(dctd_fp_plan *plan) {
    if (!plan) return;
    if (plan->has_event) {
        (void)cudaEventSynchronize(plan->uploaded);     // an upload of the blob may still be in flight
        (void)cudaEventDestroy(plan->uploaded);
    }
    if (plan->blob) blob_release(HostBlob{plan->blob, plan->blob_capacity, plan->blob_pinned});
    delete plan;
}

size_t dctd_fp_workspace_bytes(const dctd_fp_plan *plan) { return plan ? plan->total : 0; }
int64_t dctd_fp_algorithmic_bytes(const dctd_fp_plan *plan) { return plan ? plan->algo_bytes : 0; }
int32_t dctd_fp_num_items(const dctd_fp_plan *plan) { return plan ? (int32_t)plan->items.size() : 0; }

#ifdef DCTD_TUNING
/* tuning builds only (not in dctd.h): selects the pass-1 unroll / occupancy variant for n == 3 */
int dctd_fp_set_variant(int v) {
    if (v >= 100) { g_ws_stages = v - 100; return DCTD_OK; }   // 100 + s: cap the TMA ring at s stages (100: no cap)
    g_variant = v;
    return DCTD_OK;
}
#endif

/* DCTD_FP_TIMING builds: copies the 16 per-phase cycle counters of the last dctd_fp_execute on this
 * workspace to the host (synchronises the device) */
int dctd_fp_timing_read(const dctd_fp_plan *plan, const void *d_workspace, int64_t *h_out16) {
#if defined(DCTD_FP_TIMING) || defined(DCTD_DEBUG_U)
    if (!plan || !d_workspace || !h_out16) return DCTD_ERR_ARG;
    DCTD_CUDA_TRY(cudaDeviceSynchronize());
    DCTD_CUDA_TRY(cudaMemcpy(h_out16, (const char *)d_workspace + plan->off_timing, 256, cudaMemcpyDeviceToHost));
    return DCTD_OK;
#else
    (void)plan; (void)d_workspace; (void)h_out16;
    return DCTD_ERR_UNSUPPORTED;
#endif
}

/* introspection: copies the plan's pieces (8 int32 each) / items (8 int32 each) to host buffers */
int dctd_fp_plan_dump(const dctd_fp_plan *plan, int32_t *pieces, int64_t max_pieces, int32_t *items,
                      int64_t max_items, int64_t *n_pieces, int64_t *n_items) {
    if (!plan) return DCTD_ERR_ARG;
    if (n_pieces) *n_pieces = (int64_t)plan->pieces.size();
    if (n_items) *n_items = (int64_t)plan->items.size();
    if (pieces) memcpy(pieces, plan->pieces.data(), std::min<size_t>(max_pieces, plan->pieces.size()) * sizeof(Piece));
    if (items) memcpy(items, plan->items.data(), std::min<size_t>(max_items, plan->items.size()) * sizeof(Item));
    return DCTD_OK;
}

#ifdef DCTD_DEBUG_U
void *dctd_fp_debug_u(void) { return g_debug_u; }
#endif
/* introspection: copies the 32-word item records of the warp-specialised kernel (same order as the items) */
int dctd_fp_plan_dump_records(const dctd_fp_plan *plan, int32_t *records, int64_t max_items) {
    if (!plan || !records || max_items < 0) return DCTD_ERR_ARG;
    const size_t n = std::min<size_t>((size_t)max_items, plan->items.size());
    if (n) memcpy(records, (const char *)plan->blob + plan->off_wsitems, n * 32 * sizeof(int32_t));
    return DCTD_OK;
}

int dctd_fp_execute(const dctd_fp_plan *plan, const void *const *h_src_ptrs, int64_t ld, int8_t *d_out,
                    int64_t out_stride, void *d_workspace, size_t workspace_bytes, uint32_t flags,
                    void *stream_) {
    if (!plan || !d_workspace) return DCTD_ERR_ARG;
    if (plan->n_dom == 0) return DCTD_OK;
    if (!h_src_ptrs || !d_out || ld < plan->D || out_stride < (int64_t)plan->n_layers * plan->n * plan->m)
        return DCTD_ERR_ARG;
    if (workspace_bytes < plan->total) return DCTD_ERR_WORKSPACE;
    if (((uintptr_t)d_workspace & 255) != 0) return DCTD_ERR_ARG;
    cudaStream_t stream = (cudaStream_t)stream_;
    char *ws = (char *)d_workspace;

    // float4 path needs 16-byte aligned rows in every source
    bool vec4 = (plan->D % 4 == 0) && (ld % 4 == 0);
    const size_t nptr = (size_t)plan->n_layers * plan->n_src;
    for (size_t i = 0; i < nptr && vec4; ++i)
        if (((uintptr_t)h_src_ptrs[i] & 15) != 0) vec4 = false;

    Params prm{};
    prm.lay = make_layout(plan->D, plan->n, plan->m, vec4, plan->has_rider);
    int dev = 0, max_smem = 0, n_sm = 0;
    DCTD_CUDA_TRY(cudaGetDevice(&dev));
    DCTD_CUDA_TRY(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    DCTD_CUDA_TRY(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
    if (prm.lay.smem > (size_t)max_smem) return DCTD_ERR_UNSUPPORTED;

    if (!(flags & DCTD_FP_TABLES_RESIDENT)) {
        DCTD_CUDA_TRY(cudaMemcpyAsync(ws, plan->blob, plan->blob_bytes, cudaMemcpyHostToDevice, stream));
        if (!plan->has_event) {
            DCTD_CUDA_TRY(cudaEventCreateWithFlags(&plan->uploaded, cudaEventDisableTiming));
            plan->has_event = true;
        }
        DCTD_CUDA_TRY(cudaEventRecord(plan->uploaded, stream));
        fp_table_kernel<<<8, 256, 0, stream>>>((float *)(ws + plan->off_table), plan->D, prm.lay.table_len);
        DCTD_LAUNCH_CHECK();
    }
    DCTD_CUDA_TRY(cudaMemcpyAsync(ws + plan->off_src, h_src_ptrs, nptr * sizeof(void *), cudaMemcpyHostToDevice, stream));
    DCTD_CUDA_TRY(cudaMemsetAsync(ws + plan->off_counters, 0, (size_t)plan->n_counters * sizeof(int), stream));
#if defined(DCTD_FP_TIMING) || defined(DCTD_DEBUG_U)
    DCTD_CUDA_TRY(cudaMemsetAsync(ws + plan->off_timing, 0, 256, stream));
#endif

    prm.src = (const float *const *)(ws + plan->off_src);
    prm.table = (const float *)(ws + plan->off_table);
    prm.pieces = (const Piece *)(ws + plan->off_pieces);
    prm.doms = (const DomInfo *)(ws + plan->off_doms);
    prm.items = (const Item *)(ws + plan->off_items);
    prm.counters = (int *)(ws + plan->off_counters);
    prm.partials = (double *)(ws + plan->off_partials);
    prm.timing = (long long *)(ws + plan->off_timing);
#ifdef DCTD_DEBUG_U
    {
        static double *dbg = nullptr;
        static size_t dbg_bytes = 0;
        const size_t need = (size_t)plan->n_dom * plan->n_layers * 4 * (plan->n - 1) * plan->D * sizeof(double);
        if (need > dbg_bytes) { if (dbg) cudaFree(dbg); cudaMalloc(&dbg, need); dbg_bytes = need; }
        prm.debug_u = dbg;
        g_debug_u = dbg;
    }
#endif
    prm.out = d_out;
    prm.ld = ld;
    prm.out_stride = out_stride;
    prm.n_src = plan->n_src;
    prm.n_items = (int32_t)plan->items.size();
    prm.n_layers = plan->n_layers;
    prm.D = plan->D; prm.n = plan->n; prm.m = plan->m;

    prm.wsitems = (const int32_t *)(ws + plan->off_wsitems);

    const int K = plan->n - 1;
    // The reference's configuration (n = 3, contiguous rows) at the ESM-2 / ProtT5 widths runs on the warp-specialised
    // TMA kernel; every other shape on the general kernel below.
    if (vec4 && ld == plan->D && K == 2 && g_variant != 9 && !(plan->flags & DCTD_FP_PLAN_GENERAL_KERNEL)) {
        bool launched = false;
        int rc = DCTD_OK;
        switch (plan->D) {       // ESM-2 t33 / t30 / t12 and ProtT5.  (D = 320, ESM-2 t6: measured slower than the
                                 // general kernel - 4270 vs 4600 GB/s: at 1280 bytes per row every item is finisher-bound)
            case 1280: rc = launch_ws_d<1280>(plan, prm, max_smem, n_sm, stream, &launched); break;
            case 640: rc = launch_ws_d<640>(plan, prm, max_smem, n_sm, stream, &launched); break;
            case 1024: rc = launch_ws_d<1024>(plan, prm, max_smem, n_sm, stream, &launched); break;
            case 480: rc = launch_ws_d<480>(plan, prm, max_smem, n_sm, stream, &launched); break;
            default: break;
        }
        if (rc != DCTD_OK || launched) return rc;
    }
    KernelFn fn = nullptr;
    const bool small = prm.lay.T <= 320;
    const bool ldc = (ld == plan->D);
    if (plan->has_rider) {
        // protein-level fusion: 2K projections per element
        if (!vec4) fn = pick_rider<1, kMaxThreads, 1>(K);
        else if (K == 2 && ldc && plan->D == 1280 && prm.lay.RL == 1 && g_variant == 6) fn = fp_kernel<2, 4, 6, 320, 2, 1280, 1, true>;
        else if (K == 2 && ldc && plan->D == 1280 && prm.lay.RL == 1 && g_variant == 4) fn = fp_kernel<2, 4, 4, 320, 2, 1280, 1, true>;
        else if (K == 2 && ldc && plan->D == 1280 && prm.lay.RL == 1) fn = fp_kernel<2, 4, 8, 320, 2, 1280, 1, true>;
        else if (K == 2 && ldc && plan->D == 640 && prm.lay.RL == 1) fn = fp_kernel<2, 4, 8, 160, 3, 640, 1, true>;
        else if (small) fn = pick_rider<4, 320, 2>(K);
        else fn = pick_rider<4, kMaxThreads, 1>(K);
    } else if (!vec4) fn = pick_k<1, 8, kMaxThreads, 1>(K);
    else if (small) {
        // tuning variants of the common case n = 3 (see DESIGN.md "pass-1 occupancy")
        if (K == 2 && g_variant == 1) fn = fp_kernel<2, 4, 4, 320, 3>;
        else if (K == 2 && g_variant == 2) fn = fp_kernel<2, 4, 8, 320, 3>;
        else if (K == 2 && ldc && plan->D == 1280 && prm.lay.RL == 1) fn = fp_kernel<2, 4, 8, 320, 2, 1280, 1>;
        else if (K == 2 && ldc && plan->D == 640 && prm.lay.RL == 2) fn = fp_kernel<2, 4, 8, 320, 2, 640, 2>;
        else if (K == 2 && ldc && plan->D == 640 && prm.lay.RL == 1) fn = fp_kernel<2, 4, 8, 160, 4, 640, 1>;
        else if (K == 2 && ldc && plan->D == 1024 && prm.lay.RL == 1) fn = fp_kernel<2, 4, 8, 256, 2, 1024, 1>;
        else if (K == 2 && ldc && plan->D == 320 && prm.lay.RL == 4) fn = fp_kernel<2, 4, 8, 320, 2, 320, 4>;
        else fn = pick_k<4, 8, 320, 2>(K);
    } else if (K == 2 && ldc && plan->D == 2560 && prm.lay.RL == 1) fn = fp_kernel<2, 4, 8, kMaxThreads, 1, 2560, 1>;
    else fn = pick_k<4, 8, kMaxThreads, 1>(K);
    if (!fn) return DCTD_ERR_UNSUPPORTED;
    // the opt-in limit bounds static + dynamic shared memory: fp_kernel's static variables (176 B) can tip a layout that
    // passed the check above over it (D = 5072 at n = 3, m = 80), and cudaFuncSetAttribute would then fail
    cudaFuncAttributes fa{};
    DCTD_CUDA_TRY(cudaFuncGetAttributes(&fa, fn));
    if (prm.lay.smem + fa.sharedSizeBytes > (size_t)max_smem) return DCTD_ERR_UNSUPPORTED;
    DCTD_CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)prm.lay.smem));
    int per_sm = 0;
    DCTD_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, prm.lay.T, prm.lay.smem));
    if (per_sm < 1) return DCTD_ERR_UNSUPPORTED;
    const int grid = std::max(1, std::min(prm.n_items, n_sm * per_sm));
    fn<<<grid, prm.lay.T, prm.lay.smem, stream>>>(prm);
    DCTD_LAUNCH_CHECK();
    return DCTD_OK;
}

}  // extern "C"
