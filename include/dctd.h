/* dctd.h - C ABI of libdctd (B200 / sm_100a implementation of the two DCTdomain hot paths).
 *
 * The reference (mgtools/DCTdomain) is pure Python on these paths: there is no native
 * interface to replace one-for-one.  Each entry point below states the reference code it
 * stands in for (file:line under the reference tree); INTEGRATION.md shows the ctypes
 * binding a reference maintainer would add.
 *
 * Conventions
 *   - every function returns DCTD_OK (0) or a negative DCTD_ERR_* code, never throws or exits;
 *   - pointers named d_* / "device" are device pointers on the CURRENT CUDA device, pointers
 *     named h_* / "host" are host pointers; the caller owns every buffer including workspaces;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); all device work
 *     is stream-ordered on it and the functions do not synchronise unless stated;
 *   - the library keeps no global mutable state besides a thread-local "last CUDA error" and launch counter and an
 *     internal cache of host staging buffers (memory management only): options
 *     are per plan / per call (flags).  The A/B switches used while tuning (dctd_fp_set_variant, dctd_l1_set_mode) exist
 *     only in the separate tuning build (make -C dctdomain_b200/csrc tuning), not in libdctd.so.
 */
#ifndef DCTD_H
#define DCTD_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DCTD_VERSION 100

#define DCTD_OK 0
#define DCTD_ERR_ARG (-1)         /* invalid argument */
#define DCTD_ERR_CUDA (-2)        /* a CUDA call failed: see dctd_last_cuda_error() */
#define DCTD_ERR_WORKSPACE (-3)   /* workspace too small */
#define DCTD_ERR_UNSUPPORTED (-4) /* valid in the reference, not supported by this kernel set */
#define DCTD_ERR_NOMEM (-5)       /* host allocation failed */

int dctd_version(void);
const char *dctd_strerror(int code);
/* cudaError_t of the last failing CUDA call on this thread (0 if none) and its string */
int dctd_last_cuda_error(void);
const char *dctd_last_cuda_error_string(void);
/* number of kernel launches issued by this library on this thread since the last reset */
int64_t dctd_launch_count(int reset);

/* n host->device copies (one cudaMemcpyAsync each, in order, on `stream`): h_src[i] (nbytes[i] bytes, pinned or
 * pageable host memory) -> d_base + d_off[i].  Used by the Python surface to stage a batch of host embeddings
 * (the reference hands fingerprint.py numpy arrays, src/make_db.py:82) without per-array interpreter overhead. */
int dctd_h2d_rows(const void *const *h_src, const int64_t *nbytes, int64_t n, void *d_base,
                  const int64_t *d_off, void *stream);

/* The same staging for host arrays that the device can read directly (pinned memory): one gather kernel pulls all
 * pieces over PCIe instead of one DMA copy per array.  d_table: n descriptors in device-accessible memory (pinned
 * host or device memory); src, dst and nbytes of every piece must be multiples of 16. */
typedef struct dctd_copy_desc {
    const void *src; /* device-accessible source (pinned host memory) */
    void *dst;       /* device destination */
    int64_t nbytes;
} dctd_copy_desc;
int dctd_h2d_gather(const dctd_copy_desc *d_table, int64_t n, void *stream);

/* The same staging for PAGEABLE host arrays (what the reference's `.cpu().numpy()` leaves in Fingerprint.embed,
 * src/embedding.py:191): cudaMemcpyAsync from pageable memory goes through the driver's own bounce buffer on one thread
 * (~10 GB/s measured here).  This call copies with `n_threads` host threads into a caller-owned PINNED ring of `n_slots`
 * slots of `slot_bytes` and issues one copy-engine transfer per filled slot.  The destinations must be ascending and
 * non-overlapping (d_off[i] + nbytes[i] <= d_off[i+1]); the range d_off[0] .. d_off[n-1] + nbytes[n-1] is moved in
 * slot-sized chunks, so small arrays share a transfer (bytes in the gaps between destinations are overwritten with
 * unspecified values).  Returns after the last transfer has COMPLETED: the host arrays and the ring are free again;
 * the data is visible to work queued on `stream` afterwards. */
int dctd_h2d_rows_staged(const void *const *h_src, const int64_t *nbytes, int64_t n, void *d_base,
                         const int64_t *d_off, void *h_ring, int64_t slot_bytes, int32_t n_slots, int32_t n_threads,
                         void *stream);

/* =====================================================================================
 * Hot path 1: DCT fingerprints ("quant2D")
 *   replaces reference src/fingerprint.py:110-201 (scale / idct_quant / get_doms / quantize)
 *   and consumes the maxlen windows of src/embedding.py:153-192 directly (the 200-row overlap
 *   average (prev+cur)/2 is applied while the rows are loaded).
 *
 * Geometry is described once per batch by a host-side plan:
 *   sources   : n_src row-major float32 matrices [rows, D] per layer (one per protein, or one per
 *               maxlen window of a protein); all layers share the geometry;
 *   proteins  : protein p owns sources prot_src0[p] .. prot_src0[p]+prot_nsrc[p]-1; window c
 *               covers protein rows [c*stride, c*stride + rows(window c)) with stride =
 *               maxlen - overlap; rows covered by two windows are (a + b) * 0.5f;
 *   domains   : domain i belongs to protein dom_prot[i] and is the concatenation, in listed
 *               order, of its segments seg_beg[j] .. seg_end[j] (0-based, end exclusive,
 *               j in [dom_seg_off[i], dom_seg_off[i+1])), exactly the row order that
 *               get_doms (fingerprint.py:160-171) builds.
 * Output: int8 [n_dom, out_stride] with layer l's n*m bytes at column l*n*m + j*m + c
 *   (quantize's reshape(n*m) and per-layer extend, fingerprint.py:194-196).
 * ===================================================================================== */
typedef struct dctd_fp_plan dctd_fp_plan; /* opaque, host memory only */

typedef struct dctd_fp_geometry {
    int32_t n_layers;          /* embedding layers per source (reference: 2, layers 15 and 21) */
    int32_t D;                 /* embedding width (1280 for ESM-2 t33, 640 for t30); D >= m */
    int32_t n, m;              /* qdim pair applied to every layer (reference: 3, 80) */
    int32_t maxlen, overlap;   /* window length / overlap of embedding.py:163-165 (500 / 200);
                                  only used for proteins with more than one source */
    int32_t n_src;
    const int32_t *src_rows;   /* host [n_src] rows of each source */
    int32_t n_prot;
    const int32_t *prot_src0;  /* host [n_prot] */
    const int32_t *prot_nsrc;  /* host [n_prot] */
    int32_t n_dom;
    const int32_t *dom_prot;    /* host [n_dom] */
    const int32_t *dom_seg_off; /* host [n_dom+1] */
    const int32_t *seg_beg;     /* host [n_seg] 0-based first row */
    const int32_t *seg_end;     /* host [n_seg] exclusive end row (already clipped to the protein) */
} dctd_fp_geometry;

/* RecCut domain strings of a whole batch -> the segment arrays of dctd_fp_geometry, with get_doms' rules
 * (src/fingerprint.py:160-171: 1-based inclusive "beg-end" segments separated by ',', rows in listed order, an end beyond
 * the protein is clipped).  text: the n_str strings, each terminated by '\n'; str_prot[i]: protein of string i;
 * prot_len[p]: rows of protein p.  Strings with no rows are dropped (the reference skips them); domain j of the output
 * comes from string dom_str[j] and owns segments dom_seg_off[j] .. dom_seg_off[j+1]-1 (0-based begin, exclusive end).
 * Strings that need the reference's special paths - a begin beyond the protein (the segment is dropped and the next one
 * passed over, fingerprint.py:163-165), a begin < 1, anything that is not digits - are counted in *n_irregular and left
 * out: the caller handles those with its mirror of the reference code (dctdomain_b200.fingerprint.parse_domain).
 * max_segs: capacity of seg_beg / seg_end (number of ',' in text + n_str is enough).  Host only. */
int dctd_parse_domains(const char *text, int64_t text_len, int32_t n_str, const int32_t *str_prot,
                       const int32_t *prot_len, int32_t n_prot, int32_t *dom_str, int32_t *dom_seg_off,
                       int32_t *seg_beg, int32_t *seg_end, int64_t max_segs, int32_t *n_dom,
                       int32_t *n_irregular);

/* Builds the work decomposition (pieces; items of at most 512 rows in queue order: long items longest first with the
 * short ones spread evenly between them).  Host only. */
int dctd_fp_plan_create(const dctd_fp_geometry *geo, dctd_fp_plan **out_plan);
/* The same with per-plan options (0 = dctd_fp_plan_create): */
#define DCTD_FP_PLAN_NO_FUSION 1u      /* do not let a protein's global fingerprint ride on its other domains' items
                                          (every domain then reads its own rows, as the reference does) */
#define DCTD_FP_PLAN_GENERAL_KERNEL 2u /* run on the general kernel even where the warp-specialised TMA kernel applies
                                          (cross-check of the two: results agree to <= 1 LSB on a handful of bytes) */
#define DCTD_FP_PLAN_LONGEST_FIRST 4u  /* plain longest-first queue order */
int dctd_fp_plan_create_ex(const dctd_fp_geometry *geo, uint32_t flags, dctd_fp_plan **out_plan);
void dctd_fp_plan_destroy(dctd_fp_plan *plan);
/* bytes of device workspace dctd_fp_execute needs for this plan */
size_t dctd_fp_workspace_bytes(const dctd_fp_plan *plan);
/* algorithmic input bytes of the plan (roofline numerator): n_layers * D * 4 per row read - every row of every
 * domain once (rows shared with a riding global fingerprint once, rows averaged from two windows twice) */
int64_t dctd_fp_algorithmic_bytes(const dctd_fp_plan *plan);
int32_t dctd_fp_num_items(const dctd_fp_plan *plan);
/* introspection (tests): the plan's pieces and items as 8 int32 each, and the 32-word item records of the
 * warp-specialised kernel, in queue order; counts through n_pieces / n_items (either may be NULL) */
int dctd_fp_plan_dump(const dctd_fp_plan *plan, int32_t *pieces, int64_t max_pieces, int32_t *items, int64_t max_items,
                      int64_t *n_pieces, int64_t *n_items);
int dctd_fp_plan_dump_records(const dctd_fp_plan *plan, int32_t *records, int64_t max_items);

#define DCTD_FP_TABLES_RESIDENT 1u /* the plan tables were already uploaded to this workspace by an
                                      earlier dctd_fp_execute with the same plan: skip the copy */

/* h_src_ptrs: host array [n_layers * n_src] of DEVICE pointers, layer-major
 *             (h_src_ptrs[l * n_src + s] = rows of source s, layer l); row stride = ld elements.
 * d_out     : device int8 [n_dom, out_stride], out_stride >= n_layers*n*m.
 * Launches: 1 memset + (unless TABLES_RESIDENT) 1 H2D copy of the plan tables + 1 kernel.
 * Returns DCTD_ERR_UNSUPPORTED, with nothing written to d_out, when the general kernel's shared memory for (D, n, m)
 * (dynamic layout plus its static variables) exceeds the device's opt-in per-block limit, or when not one of its CTAs
 * fits on an SM.  The layout grows with D, n and m: on a B200 (232 448 B per block) at n = 3, m = 80 without fusion the
 * widest supported D is 5068, so D = 5120 (ESM-2 15B) is unsupported.  A fused protein needs a little more. */
int dctd_fp_execute(const dctd_fp_plan *plan, const void *const *h_src_ptrs, int64_t ld,
                    int8_t *d_out, int64_t out_stride, void *d_workspace, size_t workspace_bytes,
                    uint32_t flags, void *stream);

/* The two small public helpers of reference src/fingerprint.py on arbitrary float64 matrices (device
 * pointers): Fingerprint.scale (:110-123) over a whole vector, and Fingerprint.idct_quant (:126-142):
 * d_x [rows, cols] row-major -> d_out [min(num, rows), cols].  Not tuned; quantize() itself is
 * dctd_fp_execute. */
int dctd_scale_f64(const double *d_x, int64_t n, double *d_out, void *stream);
int dctd_idct_quant_f64(const double *d_x, int32_t rows, int32_t cols, int32_t num, double *d_out,
                        void *stream);

/* =====================================================================================
 * Hot path 2: exhaustive L1 top-k over int8 fingerprints
 *   replaces faiss.IndexFlat + METRIC_L1 search as called at reference src/query_db.py:75-76,87
 *   and bench/cathdb/run_dct.py:51-60 on the index built at src/database.py:240-243.
 *   Result per query: the k smallest database positions by (distance, position), ascending;
 *   unfilled slots are (FLT_MAX, -1).
 *
 * The database is kept on the device in a packed layout (groups of 32 vectors interleaved in
 * 16-byte chunks, bytes biased by 0x80) produced by dctd_l1_pack from row-major int8.
 * ===================================================================================== */
/* bytes of the packed form of n vectors of dimension d */
size_t dctd_l1_packed_bytes(int64_t n, int32_t d);
/* d_rows: device int8 [n, d] row-major  ->  d_packed (dctd_l1_packed_bytes(n, d) bytes).
 * `n_offset` vectors are assumed to be already packed in d_packed (append, as IndexFlat.add). */
int dctd_l1_pack(const int8_t *d_rows, int64_t n, int32_t d, int64_t n_offset, void *d_packed,
                 void *stream);
/* inverse of dctd_l1_pack (used by write_index / reconstruct) */
int dctd_l1_unpack(const void *d_packed, int64_t n, int32_t d, int8_t *d_rows, void *stream);

size_t dctd_l1_topk_workspace_bytes(int64_t nq, int64_t n, int32_t d, int32_t k);
/* d_q: device int8 [nq, d] row-major queries.  id_base is added to every reported position
 * (shard offset).  d_dist float32 [nq, k], d_ids int64 [nq, k]. */
int dctd_l1_topk(const int8_t *d_q, int64_t nq, const void *d_packed, int64_t n, int32_t d,
                 int32_t k, int64_t id_base, float *d_dist, int64_t *d_ids, void *d_workspace,
                 size_t workspace_bytes, void *stream);
/* ---- sharded databases (one shard per GPU / process; reference call site src/query_db.py:75-76,87 on a database too
 * large for one device).  Results travel between ranks as packed 64-bit keys: distance << 40 | global position,
 * ascending = (distance, position) order, UINT64_MAX = empty slot - 8 bytes per entry, one exchange.
 *
 *   1. dctd_l1_bound        per query an upper bound of this shard's k_local-th best distance, from a sample of the
 *                           shard (every sample_stride-th group of 32 vectors; 0 = 32).  INT32_MAX = no bound.
 *                           With g shards and k_local = ceil(k / g), the maximum over the shards of these bounds is an
 *                           upper bound of the k-th best distance over the whole database (at least k_local sampled
 *                           vectors of every shard lie within it): one MAX all-reduce of nq int32.
 *   2. dctd_l1_topk_keys    this shard's k best among the vectors with distance <= d_bound[q] (d_bound NULL: the
 *                           function finds its own bound), as keys with id_base added to the positions.
 *   3. all-gather / all-to-all of the keys, then dctd_l1_keys_merge -> faiss' (float32 distance, int64 id) result. */
#define DCTD_L1_HEAP_ONLY 1u /* flags of dctd_l1_topk_keys: skip the threshold path (exact heap scan of everything) */
size_t dctd_l1_bound_workspace_bytes(int64_t nq, int64_t n, int32_t d, int32_t k_local, int32_t sample_stride);
int dctd_l1_bound(const int8_t *d_q, int64_t nq, const void *d_packed, int64_t n, int32_t d, int32_t k_local,
                  int32_t sample_stride, int32_t *d_bound, void *d_workspace, size_t workspace_bytes, void *stream);
/* 1 if dctd_l1_topk_keys would honour an external bound for this problem size (large shard, moderate k); otherwise the
 * bound exchange can be skipped (the result is the same either way) */
int dctd_l1_uses_bound(int64_t nq, int64_t n, int32_t d, int32_t k);
/* workspace: dctd_l1_topk_workspace_bytes(nq, n, d, k) */
int dctd_l1_topk_keys(const int8_t *d_q, int64_t nq, const void *d_packed, int64_t n, int32_t d, int32_t k,
                      int64_t id_base, const int32_t *d_bound, uint64_t *d_keys, void *d_workspace,
                      size_t workspace_bytes, uint32_t flags, void *stream);
/* d_key_parts uint64 [parts, nq, k] (parts <= 32, k <= 8192), each list ascending -> the k smallest keys per query as
 * (d_dist float32 [nq, k], d_ids int64 [nq, k]) with (FLT_MAX, -1) padding and / or as keys (d_keys, may be NULL;
 * d_dist and d_ids may both be NULL when d_keys is given).  k > 992 merges by rank (no shared memory). */
int dctd_l1_keys_merge(const uint64_t *d_key_parts, int32_t parts, int64_t nq, int32_t k, float *d_dist,
                       int64_t *d_ids, uint64_t *d_keys, void *stream);

/* k-way merge of `parts` sorted lists: d_dist_parts float32 [parts, nq, k], d_ids_parts int64
 * [parts, nq, k] (each ascending by (dist, id), padded with (FLT_MAX, -1)) -> [nq, k], k <= 8192.
 * Used after the NCCL all-gather of the per-rank results of a sharded database. */
int dctd_l1_topk_merge(const float *d_dist_parts, const int64_t *d_ids_parts, int32_t parts,
                       int64_t nq, int32_t k, float *d_dist, int64_t *d_ids, void *stream);

/* ---- large k: 1 <= k <= 8192 (dctd_l1_topk / dctd_l1_topk_keys stop at k = 992).  The same result as those two -
 * faiss' (d_dist float32 [nq, k], d_ids int64 [nq, k]) with (FLT_MAX, -1) padding past n, and / or (d_keys uint64
 * [nq, k], may be NULL; d_dist and d_ids both NULL or both set) the packed keys distance << 40 | id_base + position with
 * UINT64_MAX padding - by radix selection instead of a heap: per query, histogram passes over the database narrow a
 * window of the key space to one holding the k-th key with at most 16384 keys at or below it (normally one pass), one
 * more pass collects those keys and they are sorted.  n <= 16384: one pass collects everything.
 * Queries are processed in chunks of 2048; the workspace (dctd_l1_topk_large_workspace_bytes, 0 for an unsupported k or
 * d) is ~130 KB per query of one chunk, ~270 MB from 2048 queries upwards, whatever n is.
 * DCTD_ERR_UNSUPPORTED for k > 8192 or d > 2048; arguments are checked before any CUDA call.  When the call's work has
 * completed, the first 4 bytes of the workspace hold, as uint32, the number of histogram passes the call needed: the
 * most any query took part in (0 for n <= 16384). */
size_t dctd_l1_topk_large_workspace_bytes(int64_t nq, int64_t n, int32_t d, int32_t k);
int dctd_l1_topk_large(const int8_t *d_q, int64_t nq, const void *d_packed, int64_t n, int32_t d, int32_t k,
                       int64_t id_base, float *d_dist, int64_t *d_ids, uint64_t *d_keys, void *d_workspace,
                       size_t workspace_bytes, void *stream);

/* Pairwise scorer of reference src/dct-sim.py:12-50: for pair p, the int L1 distances of every
 * fingerprint of protein a[p] against every fingerprint of protein b[p] (rows
 * [off[x], off[x+1]) of d_fps, int8 [n_fps, d] row-major): d_min_dist[p] = min over all
 * fingerprint pairs, d_last_dist[p] = distance of the last-vs-last pair; both INT32_MAX when either protein has no
 * fingerprints, as in dctd_l1_protein_scores and dctd_l1_protein_hits.  Any d >= 1.  The caller turns them
 * into similarities (1 - min(dist/17000, 1)) on the host in float64, as the reference does. */
int dctd_l1_pair_scores(const int8_t *d_fps, int32_t d, const int64_t *d_off, const int32_t *d_pair_a,
                        const int32_t *d_pair_b, int64_t n_pairs, int32_t *d_min_dist,
                        int32_t *d_last_dist, void *stream);

/* The same two scores for ALL pairs of two protein sets - dct-sim.py's db_search / all_sim loops (src/dct-sim.py:126-176) -
 * at the rate of the search kernels: every fingerprint pair is scored once by the TMA-staged SAD tile loop, minima are
 * taken per protein pair on the device, no per-pair index arrays.
 *   d_qf        device int8 [h_qoff[n_qprot], d] row-major: fingerprints of the query proteins, protein a owns rows
 *               h_qoff[a] .. h_qoff[a+1]-1 (HOST offsets, h_qoff[0] = 0)
 *   d_db_packed the other set's fingerprints in the packed layout (dctd_l1_pack), protein b owns h_doff[b] .. h_doff[b+1]-1
 *   d_min_dist, d_last_dist   device int32 [n_qprot, n_dbprot]; INT32_MAX where a protein has no fingerprints
 * The query proteins are processed in as many chunks as the workspace requires (dctd_l1_protein_scores_workspace_bytes
 * returns a size that keeps the intermediate matrices at <= 1 GB; anything from one tile of queries upwards works).
 * DCTD_ERR_UNSUPPORTED, before any launch, for vectors too wide for the shared-memory tiles: the kernel needs
 * 192 + 384 * dpad bytes (dpad = d rounded up to a multiple of 16), so on a B200 (232 448 B opt-in per block) d <= 592
 * runs and d >= 593 does not: use dctd_l1_pair_scores there. */
size_t dctd_l1_protein_scores_workspace_bytes(int64_t n_qf, int64_t n_qprot, int64_t n_dbf, int64_t n_dbprot, int32_t d);
int dctd_l1_protein_scores(const int8_t *d_qf, const int64_t *h_qoff, int64_t n_qprot, const void *d_db_packed,
                           const int64_t *h_doff, int64_t n_dbprot, int32_t d, int32_t *d_min_dist,
                           int32_t *d_last_dist, void *d_workspace, size_t workspace_bytes, void *stream);

/* The HITS of dct-sim's database search (src/dct-sim.py:126-156) without the [n_qprot, n_dbprot] matrices above: per
 * query protein a, database proteins in ascending order of the clamped key (min(last(a,b), dist_clamp), b), where
 * last(a,b) is the L1 distance of the two proteins' LAST fingerprint rows (dist_clamp when either protein has none).
 * That is dct-sim's stable descending sort on s = 1 - min(last / 17000, 1) with dist_clamp = 17000.  The hits of a are
 * the first count[a] = max(top', c_a) entries of that order, top' = min(max(top, 0), n_dbprot) and
 * c_a = #{b : min(last(a,b), dist_clamp) <= dist_cut} (dist_cut < 0: none; dist_cut >= dist_clamp: all).
 *   d_qf, d_dbf   device int8 row-major fingerprints; protein a owns rows h_qoff[a] .. h_qoff[a+1]-1 of d_qf, protein b
 *                 rows h_doff[b] .. h_doff[b+1]-1 of d_dbf (HOST offsets starting at 0)
 *   d_count       device int32 [n_qprot]: count[a], exact whatever cap is
 *   d_hit_db, d_hit_min, d_hit_last   device int32 [n_qprot, cap]: row a holds the first min(count[a], cap) hits in
 *                 order - database protein, min over all fingerprint pairs, last-vs-last distance (INT32_MAX when
 *                 either protein has no fingerprints) - and (-1, INT32_MAX, INT32_MAX) after them
 * One SAD per (query protein, database protein) pair selects the hits (heap scan of the search path with the clamped
 * key); the min is computed for the hit pairs only.  Query proteins are processed in as many chunks as the workspace
 * allows (dctd_l1_protein_hits_workspace_bytes: one chunk of up to 65536 of them).  1 <= cap <= 992;
 * DCTD_ERR_UNSUPPORTED for cap > 992 (a caller that needs longer rows reruns those queries through
 * dctd_l1_protein_scores) and for d > 2048 (up to 2048 its heap scan fits a B200's shared memory at every cap).  Arguments are checked before any CUDA call. */
size_t dctd_l1_protein_hits_workspace_bytes(int64_t n_qf, int64_t n_qprot, int64_t n_dbf, int64_t n_dbprot, int32_t d,
                                            int32_t top, int32_t cap);
int dctd_l1_protein_hits(const int8_t *d_qf, const int64_t *h_qoff, int64_t n_qprot, const int8_t *d_dbf,
                         const int64_t *h_doff, int64_t n_dbprot, int32_t d, int32_t top, int32_t dist_clamp,
                         int32_t dist_cut, int32_t cap, int32_t *d_count, int32_t *d_hit_db, int32_t *d_hit_min,
                         int32_t *d_hit_last, void *d_workspace, size_t workspace_bytes, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* DCTD_H */
