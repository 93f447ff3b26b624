// libdctd: version / error plumbing of the C ABI (include/dctd.h).
#include "dctd_internal.cuh"

#include <algorithm>
#include <atomic>
#include <cstring>
#include <thread>
#include <vector>

namespace dctd {
static thread_local cudaError_t g_last_cuda = cudaSuccess;
static thread_local int64_t g_launches = 0;
void set_cuda_error(cudaError_t e) {
    g_last_cuda = e;
    // a failed runtime call also leaves its (non-sticky) error pending in the runtime; consume it, or the launch check of
    // the next, valid call - ours or the caller's - would report it as its own
    (void)cudaGetLastError();
}
void count_launch(int n) { g_launches += n; }
}  // namespace dctd

extern "C" {

int dctd_version(void) { return DCTD_VERSION; }

const char *dctd_strerror(int code) {
    switch (code) {
        case DCTD_OK: return "ok";
        case DCTD_ERR_ARG: return "invalid argument";
        case DCTD_ERR_CUDA: return "CUDA error (see dctd_last_cuda_error_string)";
        case DCTD_ERR_WORKSPACE: return "workspace too small";
        case DCTD_ERR_UNSUPPORTED: return "configuration not supported by this kernel set";
        case DCTD_ERR_NOMEM: return "host allocation failed";
        default: return "unknown dctd error code";
    }
}

int dctd_last_cuda_error(void) { return (int)dctd::g_last_cuda; }
const char *dctd_last_cuda_error_string(void) { return cudaGetErrorString(dctd::g_last_cuda); }

/* Host -> device staging for the Python surface: n independent copies (one cudaMemcpyAsync each, in order, on
 * `stream`) of h_src[i] (nbytes[i] bytes, pinned or pageable) to d_base + d_off[i].  Saves the per-tensor
 * interpreter overhead when a batch arrives as hundreds of separate host arrays. */
int dctd_h2d_rows(const void *const *h_src, const int64_t *nbytes, int64_t n, void *d_base, const int64_t *d_off,
                  void *stream) {
    if (n < 0 || (n > 0 && (!h_src || !nbytes || !d_base || !d_off))) return DCTD_ERR_ARG;
    for (int64_t i = 0; i < n; ++i) {
        if (nbytes[i] == 0) continue;
        DCTD_CUDA_TRY(cudaMemcpyAsync((char *)d_base + d_off[i], h_src[i], (size_t)nbytes[i], cudaMemcpyHostToDevice,
                                      (cudaStream_t)stream));
    }
    return DCTD_OK;
}

/* Pageable host arrays: n_threads host threads copy slot-sized chunks of the destination range into a pinned ring, one
 * copy-engine transfer per filled slot (see dctd.h).  Chunks are handed out in ascending order; chunk c uses slot
 * c % n_slots once the transfer of chunk c - n_slots has completed (slot generation counter + event), so a worker only
 * ever waits for an EARLIER chunk, which some worker took before: no cycle. */
int dctd_h2d_rows_staged(const void *const *h_src, const int64_t *nbytes, int64_t n, void *d_base, const int64_t *d_off,
                         void *h_ring, int64_t slot_bytes, int32_t n_slots, int32_t n_threads, void *stream) {
    if (n < 0 || slot_bytes <= 0 || n_slots < 2 || n_slots > 256 || n_threads < 1 || n_threads > 64) return DCTD_ERR_ARG;
    if (n == 0) return DCTD_OK;
    if (!h_src || !nbytes || !d_base || !d_off || !h_ring) return DCTD_ERR_ARG;
    for (int64_t i = 0; i < n; ++i) {
        if (nbytes[i] < 0 || (nbytes[i] > 0 && !h_src[i])) return DCTD_ERR_ARG;
        if (i + 1 < n && d_off[i] + nbytes[i] > d_off[i + 1]) return DCTD_ERR_ARG;      // ascending, non-overlapping
    }
    const int64_t lo0 = d_off[0], hi0 = d_off[n - 1] + nbytes[n - 1];
    const int64_t nchunks = (hi0 - lo0 + slot_bytes - 1) / slot_bytes;
    if (nchunks <= 0) return DCTD_OK;
    int dev = 0;
    DCTD_CUDA_TRY(cudaGetDevice(&dev));
    std::vector<cudaEvent_t> ev((size_t)n_slots, nullptr);
    for (int s = 0; s < n_slots; ++s) {
        const cudaError_t e = cudaEventCreateWithFlags(&ev[s], cudaEventDisableTiming);
        if (e != cudaSuccess) {
            for (int t = 0; t < s; ++t) (void)cudaEventDestroy(ev[t]);
            dctd::set_cuda_error(e);
            return DCTD_ERR_CUDA;
        }
    }
    std::vector<std::atomic<int64_t>> gen((size_t)n_slots);
    for (auto &g : gen) g.store(0, std::memory_order_relaxed);
    std::atomic<int64_t> next{0};
    std::atomic<int> failed{0};
    char *const ring = static_cast<char *>(h_ring);
    char *const dbase = static_cast<char *>(d_base);
    const cudaStream_t st = (cudaStream_t)stream;
    auto worker = [&]() {
        if (cudaSetDevice(dev) != cudaSuccess) { failed.store((int)cudaGetLastError() | 0x10000); return; }
        for (;;) {
            const int64_t c = next.fetch_add(1, std::memory_order_relaxed);
            if (c >= nchunks || failed.load(std::memory_order_relaxed)) return;
            const int s = (int)(c % n_slots);
            const int64_t g = c / n_slots;
            while (gen[s].load(std::memory_order_acquire) != g) {
                if (failed.load(std::memory_order_relaxed)) return;
                std::this_thread::yield();
            }
            cudaError_t e = cudaSuccess;
            if (g > 0) e = cudaEventSynchronize(ev[s]);        // the slot's previous transfer has read it
            char *slot = ring + (size_t)s * slot_bytes;
            const int64_t lo = lo0 + c * slot_bytes, hi = std::min(lo + slot_bytes, hi0);
            if (e == cudaSuccess) {
                int64_t i = std::upper_bound(d_off, d_off + n, lo) - d_off - 1;      // last destination starting at or before lo
                if (i < 0) i = 0;
                for (; i < n && d_off[i] < hi; ++i) {
                    const int64_t a = std::max(lo, d_off[i]), b = std::min(hi, d_off[i] + nbytes[i]);
                    if (b > a) memcpy(slot + (a - lo), static_cast<const char *>(h_src[i]) + (a - d_off[i]), (size_t)(b - a));
                }
                e = cudaMemcpyAsync(dbase + lo, slot, (size_t)(hi - lo), cudaMemcpyHostToDevice, st);
            }
            if (e == cudaSuccess) e = cudaEventRecord(ev[s], st);
            if (e != cudaSuccess) failed.store((int)e | 0x10000);
            gen[s].store(g + 1, std::memory_order_release);
        }
    };
    const int nt = (int)std::min<int64_t>(n_threads, nchunks);
    std::vector<std::thread> pool;
    pool.reserve((size_t)std::max(0, nt - 1));
    for (int t = 1; t < nt; ++t) pool.emplace_back(worker);
    worker();
    for (auto &t : pool) t.join();
    cudaError_t e = cudaSuccess;
    for (int s = 0; s < n_slots; ++s) {
        if (gen[s].load() > 0 && e == cudaSuccess) e = cudaEventSynchronize(ev[s]);
        (void)cudaEventDestroy(ev[s]);
    }
    if (failed.load()) {
        dctd::set_cuda_error((cudaError_t)(failed.load() & 0xffff));
        return DCTD_ERR_CUDA;
    }
    if (e != cudaSuccess) {
        dctd::set_cuda_error(e);
        return DCTD_ERR_CUDA;
    }
    return DCTD_OK;
}

/* The same staging as a gather KERNEL for host arrays the device can read (pinned memory): the SMs pull the pieces
 * over PCIe with 16-byte loads, many pieces in flight, so the link stays busy across array boundaries (a DMA copy per
 * array leaves a gap of a few microseconds between arrays).  d_table: n descriptors in device-accessible memory
 * (pinned host memory or device memory), every src / dst / nbytes a multiple of 16. */
namespace {
__global__ void __launch_bounds__(128, 16) gather_kernel(const dctd_copy_desc *__restrict__ table, long long n) {
    for (long long e = blockIdx.x; e < n; e += gridDim.x) {
        const dctd_copy_desc dsc = table[e];
        const uint4 *src = reinterpret_cast<const uint4 *>(dsc.src);
        uint4 *dst = reinterpret_cast<uint4 *>(dsc.dst);
        const unsigned int m = (unsigned int)(dsc.nbytes / 16);        // pieces are far below 64 GB
        constexpr int U = 4;       // 64 bytes in flight per thread: with one CTA per SM still 1.2 MB, the link needs ~1 MB
        for (unsigned int i0 = threadIdx.x; i0 < m; i0 += blockDim.x * U) {
            uint4 v[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const unsigned int i = i0 + u * blockDim.x;
                if (i < m)
                    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                                 : "=r"(v[u].x), "=r"(v[u].y), "=r"(v[u].z), "=r"(v[u].w)
                                 : "l"(src + i));
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const unsigned int i = i0 + u * blockDim.x;
                if (i < m) dst[i] = v[u];
            }
        }
    }
}
}  // namespace

int dctd_h2d_gather(const dctd_copy_desc *d_table, int64_t n, void *stream) {
    if (n < 0 || (n > 0 && !d_table)) return DCTD_ERR_ARG;
    if (n == 0) return DCTD_OK;
    // The link is saturated by ~1 MB in flight (measured: 32 CTAs x 256 threads x 128 bytes reach the 51.4 GB/s that
    // 1184 CTAs reach; scripts/microbench/h2d_pull.cu), so the gather stays small enough to run NEXT TO the fingerprint
    // kernel's one CTA per SM (608 threads x 96 registers, 223 KB of shared memory): one CTA of 128 threads per SM, no
    // shared memory, and <= 32 registers - the register file is split over the four SM sub-partitions, the fingerprint
    // kernel's 19 warps leave 1024 registers in three of them, i.e. room for one warp of 32 registers each (with 48
    // registers the big kernel never got onto an SM before the whole gather launch had ended:
    // scripts/microbench/coreside.cu).  In quantize_stream the copies of batch i+1 then run beside the fingerprint
    // kernel of batch i instead of keeping it off the SMs.
    int dev = 0, n_sm = 0;
    DCTD_CUDA_TRY(cudaGetDevice(&dev));
    DCTD_CUDA_TRY(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
    const int grid = (int)(n < (int64_t)n_sm ? n : (int64_t)n_sm);
    // An SM changes its L1 / shared-memory split only when it is idle.  The fingerprint kernel needs the maximum shared
    // carveout; asking for the same split here (the loads bypass L1 anyway) lets its CTAs start on SMs that run gather
    // CTAs (same microbenchmark: with the default carveout the big kernel waits for the end of the gather launch, 30 ms;
    // with this attribute it is done 1.7 ms after the gather began).
    DCTD_CUDA_TRY(cudaFuncSetAttribute(gather_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                       (int)cudaSharedmemCarveoutMaxShared));
    gather_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(d_table, (long long)n);
    DCTD_LAUNCH_CHECK();
    return DCTD_OK;
}

/* RecCut domain strings -> segment arrays with get_doms' rules (reference src/fingerprint.py:160-171), for a whole
 * batch in one call.  See dctd.h. */
int dctd_parse_domains(const char *text, int64_t text_len, int32_t n_str, const int32_t *str_prot,
                       const int32_t *prot_len, int32_t n_prot, int32_t *dom_str, int32_t *dom_seg_off,
                       int32_t *seg_beg, int32_t *seg_end, int64_t max_segs, int32_t *n_dom_out,
                       int32_t *n_irregular_out) {
    if (n_str < 0 || text_len < 0 || max_segs < 0 || !n_dom_out || !n_irregular_out) return DCTD_ERR_ARG;
    if (n_str > 0 && (!text || !str_prot || !prot_len || !dom_str || !dom_seg_off || !seg_beg || !seg_end))
        return DCTD_ERR_ARG;
    int32_t n_dom = 0, n_irr = 0;
    int64_t n_seg = 0, pos = 0;
    if (dom_seg_off) dom_seg_off[0] = 0;
    for (int32_t i = 0; i < n_str; ++i) {
        const int32_t p = str_prot[i];
        if (p < 0 || p >= n_prot) return DCTD_ERR_ARG;
        const int64_t rows_p = prot_len[p];
        const int64_t seg0 = n_seg;
        int64_t rows = 0;
        bool regular = true, at_end = false;
        // one string: "beg-end" segments separated by ',', terminated by '\n' (or the end of the text)
        while (!at_end) {
            int64_t v[2] = {0, 0};
            for (int part = 0; part < 2 && regular; ++part) {
                int digits = 0;
                while (pos < text_len && text[pos] >= '0' && text[pos] <= '9') {
                    if (v[part] < (1LL << 40)) v[part] = v[part] * 10 + (text[pos] - '0');
                    ++pos;
                    ++digits;
                }
                if (digits == 0) regular = false;
                if (part == 0) {
                    if (pos < text_len && text[pos] == '-') ++pos;
                    else regular = false;
                }
            }
            if (regular) {
                // reference: a segment whose begin lies beyond the protein (or begin 0) takes get_doms' special paths
                if (v[0] < 1 || v[0] > rows_p) {
                    regular = false;
                } else if (n_seg >= max_segs) {
                    return DCTD_ERR_WORKSPACE;
                } else {
                    const int64_t lo = v[0] - 1, hi = v[1] < rows_p ? v[1] : rows_p;
                    seg_beg[n_seg] = (int32_t)lo;
                    seg_end[n_seg] = (int32_t)(hi > lo ? hi : lo);
                    rows += seg_end[n_seg] - seg_beg[n_seg];
                    ++n_seg;
                }
            }
            if (regular && pos < text_len && text[pos] == ',') {
                ++pos;
                continue;
            }
            if (!(pos >= text_len || text[pos] == '\n')) regular = false;      // anything else: leave it to the caller
            while (pos < text_len && text[pos] != '\n') ++pos;               // skip to the end of this string
            if (pos < text_len) ++pos;
            at_end = true;
        }
        if (!regular) {
            ++n_irr;
            n_seg = seg0;
            continue;
        }
        if (rows == 0) {          // reference: an empty embedding slice -> the domain is skipped
            n_seg = seg0;
            continue;
        }
        dom_str[n_dom] = i;
        dom_seg_off[n_dom + 1] = (int32_t)n_seg;
        ++n_dom;
    }
    *n_dom_out = n_dom;
    *n_irregular_out = n_irr;
    return DCTD_OK;
}

int64_t dctd_launch_count(int reset) {
    int64_t v = dctd::g_launches;
    if (reset) dctd::g_launches = 0;
    return v;
}

}  // extern "C"
