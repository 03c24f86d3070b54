/*
 * nrb200.h -- C-ABI of libnrb200.so, the B200 (sm_100a) candidate-retrieval library.
 *
 * This is the drop-in boundary below the Python `faiss`-compatible surface
 * (newsrecommend_b200/faiss.py). The reference has no FFI of its own: its hot path
 * (/root/reference/Retrieval.py) reaches native code only through the SWIG-wrapped `faiss`
 * module, so each entry point below cites the reference call site (Retrieval.py:LINE) and the
 * faiss routine it stands in for. All pointers are plain DEVICE pointers unless the name ends in
 * `_host`; sizes are element counts; `stream` is a cudaStream_t passed as void* (NULL = default
 * stream). Every function returns 0 on success and a negative code on failure, never throws,
 * and leaves a message retrievable with nrb_last_error(). There is no CPU fallback: on a
 * machine without an sm_100 GPU the compute entry points return NRB_ERR_NO_DEVICE.
 */
#ifndef NRB200_H
#define NRB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NRB_OK 0
#define NRB_ERR_INVALID -1   /* bad argument */
#define NRB_ERR_CUDA -2      /* CUDA runtime / driver error */
#define NRB_ERR_NO_DEVICE -3 /* no sm_100 device */
#define NRB_ERR_WORKSPACE -4 /* workspace too small */

#define NRB_METRIC_INNER_PRODUCT 0 /* faiss.METRIC_INNER_PRODUCT */
#define NRB_METRIC_L2 1            /* faiss.METRIC_L2 (squared L2, as Retrieval.py:16,25) */

#define NRB_PATH_AUTO 0
#define NRB_PATH_SIMT 1 /* fp32 CUDA-core kernels */
#define NRB_PATH_TC 2   /* tcgen05 3xTF32 kernels */
#define NRB_PATH_TC1 3  /* tcgen05 1xTF32 filter with a rigorous error margin + exact fp32 refine;
                           flat search only, rows that overflow the margin set fall back to TC */
#define NRB_PATH_TC16 4 /* the same filter + refine on power-of-two scaled IEEE fp16 planes (11-bit
                           significand like tf32, hence the same margin) at twice the tensor rate */

#define NRB_MAX_K 128 /* largest k / nprobe supported by the selection stage */

/* A row-major matrix in its device ("packed") form, produced by nrb_pack_rows():
 *   raw  [n, kp]  fp32 rows zero-padded from d to kp columns (kp % 32 == 0)
 *   hi   [n, kp]  tf32(raw)            (cvt.rna, low 13 mantissa bits zero)
 *   lo   [n, kp]  tf32(raw - hi)
 *   norms[n]      squared L2 norms (fp32)
 *   h16  [n, kp]  fp16(raw * s), s a power of two chosen so that |row| * s < 2^15: one s for the
 *                 whole matrix on the item side (h16_scale), one per row on the query side
 *                 (h16_row_scale); see nrb_pack_rows_h16
 * raw feeds the SIMT kernels and the exact refine, hi/lo feed the 3xTF32 tcgen05 kernels via
 * TMA, hi alone the 1xTF32 filter, h16 the fp16 filter. */
typedef struct nrb_matrix {
    const float* raw;
    const float* hi;
    const float* lo;
    const float* norms;
    int64_t n;
    int32_t d;
    int32_t kp;
    float max_norm; /* max row L2 norm (not squared) over the matrix, 0 = unknown; needed on the
                       item side by NRB_PATH_TC1 / NRB_PATH_TC16 */
    float h16_scale; /* item side: the power of two every row of h16 was multiplied by (0 = none) */
    const void* h16; /* [n, kp] IEEE fp16 = raw * scale (NRB_PATH_TC16), or NULL */
    const float* h16_row_scale; /* query side: per-row power-of-two scales f32[n] of h16, or NULL */
} nrb_matrix;

/* ---- diagnostics ------------------------------------------------------------------------ */
int nrb_version(void);
/* Copies the calling thread's last error message (NUL terminated) into buf. */
int nrb_last_error(char* buf, int buflen);
/* sm count and compute capability of the current device. */
int nrb_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* Number of kernel launches issued by this library since load (bench.py's gpu_launches). */
int64_t nrb_launch_count(void);

/* Device-side timing of the dominant (distance + selection) kernel: when enabled, every such
 * launch is bracketed by CUDA events on its stream; nrb_profile_read() synchronises, returns the
 * summed milliseconds and the launch count since the last read, and resets. */
int nrb_profile_enable(int on);
int nrb_profile_read(double* total_ms, int* n_launches);

/* ---- K0: pack ---------------------------------------------------------------------------- */
/* Replaces the numpy cast + contiguity at Retrieval.py:8,17,31 (and IndexFlatCodes::add's
 * memcpy, Retrieval.py:26): x is fp32 [n, d] with row stride ldx elements. Any of raw/hi/lo/
 * norms may be NULL. */
int nrb_pack_rows(const float* x, int64_t n, int32_t d, int64_t ldx, int32_t kp, float* raw,
                  float* hi, float* lo, float* norms, void* stream);
/* fp16 plane of NRB_PATH_TC16: h16[i, :] = fp16(x[i, :] * s_i), zero-padded to kp columns.
 * uniform_scale > 0: s_i = uniform_scale for every row (item side; the caller guarantees
 * max|row| * uniform_scale <= 65504 -- newsrecommend_b200 uses 2^(14 - floor(log2(max_norm)))).
 * uniform_scale == 0: s_i = 2^(14 - floor(log2(|x_i|))) per row (1 for a zero row), written to
 * row_scale f32[n] (query side). */
int nrb_pack_rows_h16(const float* x, int64_t n, int32_t d, int64_t ldx, int32_t kp, float uniform_scale,
                      void* h16, float* row_scale, void* stream);
/* dst[i, :] = src[idx[i], :] for rows of `width` floats (width % 4 == 0). Builds the
 * list-contiguous IVF planes (ArrayInvertedLists, Retrieval.py:23) and query groups. */
int nrb_gather_rows(const float* src, int32_t width, const int32_t* idx, int64_t n, float* dst,
                    void* stream);
/* dst[i] = src[idx[i]] for 64-bit ids (external ids in list order). */
int nrb_gather_i64(const int64_t* src, const int32_t* idx, int64_t n, int64_t* dst, void* stream);
/* faiss.normalize_L2 (fvec_renorm_L2): in place, zero rows untouched. */
int nrb_normalize_l2(float* x, int64_t n, int32_t d, int64_t ldx, void* stream);

/* ---- K2: exact top-k (IndexFlat::search -> knn_inner_product / knn_L2sqr) ------------------ */
/* Replaces IndexFlatL2/IndexFlatIP.search at Retrieval.py:21,32 and the k-means assignment
 * search inside Clustering::train (Retrieval.py:18). D f32[nq,k] best-first (IP descending,
 * L2 ascending squared distance clamped at 0), I i64[nq,k] = row index + id_base; missing
 * results are I = -1, D = -FLT_MAX (IP) / +FLT_MAX (L2). 1 <= k <= NRB_MAX_K.
 * path: NRB_PATH_AUTO picks NRB_PATH_TC16 when its preconditions hold (raw + h16 + norms planes and
 * scales on both sides, b->max_norm, kp <= 256, k <= 112), else NRB_PATH_TC1 (hi instead of h16),
 * else NRB_PATH_TC. The filter paths synchronise the stream once per call (they read back the
 * number of flagged queries); flagged queries are recomputed by NRB_PATH_TC, for which the lo
 * planes must be present or q->raw / b->hi,lo (the query rows are split on the fly). That fallback
 * takes its scratch from the stream-ordered allocator (cudaMallocAsync) and, the first time it runs
 * on a device, raises the release threshold of the device's DEFAULT memory pool so that the pool
 * keeps the memory between searches (a process-wide setting of that pool). */
size_t nrb_search_flat_workspace(int64_t nq, int64_t nb, int32_t k, int32_t kp);
int nrb_search_flat(const nrb_matrix* q, const nrb_matrix* b, int32_t metric, int32_t k,
                    int64_t id_base, float* D, int64_t* I, void* workspace,
                    size_t workspace_bytes, int32_t path, void* stream);

/* Queries that NRB_PATH_TC1 had to recompute with the 3xTF32 kernel since the library was loaded
 * (candidate slots exhausted inside the error margin, or an estimate outside its bound). */
int64_t nrb_fallback_query_count(void);

/* The work plan nrb_search_flat would use (host logic only, no device needed; 148 SMs are assumed
 * when there is no device): out10 = { query tiles, tile pairs, full pairs (one pass over the whole
 * catalog each), tail pairs, item chunks per tail pair (or per tile), item rows per chunk, units,
 * partial-result slots per query, CTAs launched, 1 if the single-CTA kernel form is used }.
 * path must be a concrete NRB_PATH_* (not AUTO). */
int nrb_plan_flat_describe(int64_t nq, int64_t nb, int32_t k, int32_t path, int32_t* out10);

/* ---- K1b: k-means centroid update (Clustering.cpp compute_centroids) ---------------------- */
/* Replaces the update step of clustering.train (Retrieval.py:18). x_raw is the packed raw
 * plane [n, kp]; assign i64[n] in [0, k). Writes centroids f32[k, d] (row stride d) as the
 * mean of the assigned rows and hassign f32[k] = counts. Empty clusters keep zeros.
 * A segmented reduction over the counting-sorted rows, balanced under list skew: every list is
 * cut into 64-row chunks, one block per chunk sums in fp64 (fixed association), one block per
 * centroid adds the chunk partials in order, rounds to fp32 and multiplies by 1.0f/count like
 * faiss. Deterministic. HBM-bound: reads n * kp * 4 bytes. */
size_t nrb_kmeans_update_workspace(int64_t n, int32_t k, int32_t kp);
int nrb_kmeans_update(const float* x_raw, int64_t n, int32_t d, int32_t kp,
                      const int64_t* assign, int32_t k, float* centroids, float* hassign,
                      void* workspace, size_t workspace_bytes, void* stream);
/* Data-parallel form of K1b (SURVEY 8e: shared coarse quantizer, one all-reduce of <= 0.65 MB per
 * Lloyd iteration; no reference analogue, the reference trains in one process at Retrieval.py:18).
 * nrb_kmeans_partial_sums: the same segmented fp64 reduction over THIS rank's rows, but it stops
 * before the division: sums f64[k, d + 1], columns 0..d-1 = sum of the assigned rows, column d =
 * their count. The ranks add their tables (ncclAllReduce, fp64) and nrb_kmeans_means turns the
 * total into centroids f32[k, d] = float(sum) * (1.0f / count) and hassign f32[k] = count -- the
 * rounding of nrb_kmeans_update. Workspace: nrb_kmeans_update_workspace. */
int nrb_kmeans_partial_sums(const float* x_raw, int64_t n, int32_t d, int32_t kp, const int64_t* assign,
                            int32_t k, double* sums, void* workspace, size_t workspace_bytes, void* stream);
int nrb_kmeans_means(const double* sums, int32_t k, int32_t d, float* centroids, float* hassign, void* stream);
/* Host-side pieces of Clustering::train that faiss also runs on the host (tiny, sequential,
 * RNG-driven): rand_perm (utils/random.cpp, std::mt19937, seed 1234 subsample / seed+1 init)
 * and split_clusters (EPS = 1/1024, rng(1234)). Return value of split = nsplit. These two
 * restate third-party faiss routines (facebookresearch/faiss, MIT licence: utils/random.cpp
 * rand_perm, Clustering.cpp split_clusters) because RNG-exact k-means needs their exact
 * arithmetic; they are not taken from /root/reference, which holds no native code. */
int nrb_rand_perm_host(int32_t* perm, int64_t n, int64_t seed);
int nrb_split_clusters_host(int32_t d, int32_t k, int64_t n, float* hassign, float* centroids);
/* split_clusters on the DEVICE (one block; std::mt19937(1234) restated in the kernel), so that
 * the training loop needs no host round trip: hassign f32[k] and centroids f32[k, d] are
 * updated in place; stats3 f64[3]: [1] = imbalance factor k * sum(size^2) / n^2 of the sizes
 * on entry, [2] = number of splits (-1: no cluster could be split); [0] is not touched. */
int nrb_split_clusters(int32_t d, int32_t k, int64_t n, float* hassign, float* centroids, double* stats3,
                       void* stream);
/* Clustering::train's iteration loop (Retrieval.py:18; IndexIVFFlat.train) as ONE call: niter x
 * { pack the centroids, exact nearest-centroid assignment of every row (K2 with k = 1: fp16 filter +
 * exact fp32 refine when x carries h16 + row scales and kp <= 256, else the 1xTF32 filter on hi,
 * else 3xTF32 on hi / lo; rows a filter flags are recomputed exactly by a device-driven kernel),
 * K1b update + objective (sum over rows of |x - c|^2 or x.c against the centroids the iteration
 * started with, exact fp32 products, fixed-order fp64 sums), device split_clusters, optional L2
 * renormalisation (spherical) }, all queued on `stream` with NO host synchronisation.
 * x: packed training rows (raw, norms, and h16 + h16_row_scale or hi [+ lo]); x->max_norm must
 * hold the largest row norm (it bounds every centroid: a mean is no longer than the longest row,
 * a split scales by at most 1 + 1/1024). centroids f32[k, d]: initial centroids in (rows of x, or
 * anything no longer than x->max_norm), final centroids out. assign i64[n] (optional): the last
 * iteration's assignment. stats f64[niter, 4] (device): objective, imbalance factor, nsplit, 0.
 * `metric` is the assigner's metric (NRB_METRIC_L2 for IndexFlatL2 / the reference's quantizer). */
size_t nrb_kmeans_train_workspace(int64_t n, int32_t k, int32_t kp);
int nrb_kmeans_train(const nrb_matrix* x, int32_t k, int32_t niter, int32_t metric, int32_t spherical,
                     float* centroids, int64_t* assign, double* stats, void* workspace, size_t workspace_bytes,
                     void* stream);

/* ---- K3: IVF lists (ArrayInvertedLists + search_preassigned / IVFFlatScanner) ------------- */
/* Stable counting sort of rows by list id. Replaces the 300 boolean masks at Retrieval.py:23
 * and IndexIVF::add_core. assign i64[n] in [0, nlist); writes offsets i32[nlist+1] and
 * order i32[n]: packed position p holds source row order[p]; within a list, source order. */
size_t nrb_ivf_build_lists_workspace(int64_t n, int32_t nlist);
int nrb_ivf_build_lists(const int64_t* assign, int64_t n, int32_t nlist, int32_t* offsets,
                        int32_t* order, void* workspace, size_t workspace_bytes, void* stream);
/* Scans, for each query, the nprobe lists named by coarse i64[nq, nprobe] (best first; -1 =
 * none) and keeps the top k by `metric`. `lists` is the list-contiguous packed matrix, ids
 * i64[lists->n] the external id of each packed row. Replaces Retrieval.py:32-34 in its
 * IndexIVFFlat form (north_star); results as nrb_search_flat. max_list_len = longest list
 * (host-known since add()). The (query, list) pairs are regrouped list-major on the device so
 * that every list is read once per 128 probing queries, not once per query.
 * path: NRB_PATH_SIMT, NRB_PATH_TC (3xTF32 scan), NRB_PATH_TC16 (fp16 filter over the lists with the
 * proven margin + exact fp32 refine; needs raw, norms, h16 + scales and, for the queries the filter
 * flags, hi / lo on both sides, lists->max_norm, kp <= 256, k <= 112) or NRB_PATH_AUTO (TC16 when
 * those preconditions hold, else TC). TC16 synchronises the stream once per call. */
size_t nrb_ivf_search_workspace(int64_t nq, int32_t nprobe, int32_t k, int32_t kp, int32_t nlist,
                                int32_t max_list_len);
int nrb_ivf_search(const nrb_matrix* q, const nrb_matrix* lists, const int32_t* offsets,
                   int32_t nlist, int32_t max_list_len, const int64_t* ids, const int64_t* coarse,
                   int32_t nprobe, int32_t metric, int32_t k, float* D, int64_t* I,
                   void* workspace, size_t workspace_bytes, int32_t path, void* stream);

/* ---- neighbours of the path (SURVEY 8f) --------------------------------------------------- */
/* Retrieval.py:33-34 batched: out[out_off[u] + j] = list_ids[list_off[user_list[u]] + j] for
 * every member j of the user's nearest list (user_list[u] < 0: nothing). out_off is the
 * exclusive prefix sum of the list lengths per user. */
int nrb_expand_lists(const int64_t* user_list, const int32_t* list_off, const int64_t* list_ids,
                     const int64_t* out_off, int64_t nu, int64_t* out, void* stream);
/* utils.py:12-17 and finialize_retrieval.py:10-11: out[u] = 1 iff target[u] occurs in row u of
 * the CSR (off i64[nrows+1], ids). */
int nrb_csr_contains(const int64_t* off, const int64_t* ids, const int64_t* target, int64_t nrows,
                     uint8_t* out, void* stream);

/* ---- K4: k-way merge of per-shard results ------------------------------------------------- */
/* Dp f32[nparts, nq, k], Ip i64[nparts, nq, k] (each best-first, -1 padded) -> global top-k.
 * Sits after the NCCL all-gather of the catalog-sharded search (north_star item 4). */
int nrb_merge_topk(const float* Dp, const int64_t* Ip, int32_t nparts, int64_t nq, int32_t k,
                   int32_t metric, float* D, int64_t* I, void* stream);

/* ---- low-latency path for tiny batches (csrc/small_batch.cu)
 * faiss's own route for nq < distance_compute_blas_threshold (20): no GEMM, every (query, item)
 * distance computed directly in fp32 (L2 as sum (q - x)^2, not via norms) and selected exactly
 * (knn_inner_product / knn_L2sqr sequential branch, SURVEY 3.2). This is the route each of the
 * 50,000 `centroid_index.search(profile, 1)` calls of Retrieval.py:30-32 takes. Here: every item
 * row is read once with 128-bit loads (a warp per row, several rows in flight, HBM-bound), the
 * scores of one query go to a scratch row and the top-k is selected exactly by radix select (in two
 * levels of 8,192-element slices for long rows); catalogs of up to
 * 8,192 rows (the centroid index) run as ONE launch with the scores in shared memory. No plan
 * kernels, no packing of the queries (xq is plain fp32 [nq, d], row stride ldq), no host
 * synchronisation. nq <= NRB_SMALL_MAX_NQ, k <= NRB_MAX_K; b needs only its raw plane. */
#define NRB_SMALL_MAX_NQ 64
size_t nrb_search_small_workspace(int64_t nq, int64_t nb, int32_t k);
int nrb_search_small(const float* xq, int64_t ldq, int32_t nq, int32_t d, const nrb_matrix* b, int32_t metric,
                     int32_t k, int64_t id_base, float* D, int64_t* I, void* workspace, size_t workspace_bytes,
                     void* stream);
/* The same with HOST query rows in and HOST results out (numpy in, numpy out; Retrieval.py:31-32):
 * the library keeps a page-locked staging buffer that is MAPPED into the device address space
 * (grow-only, per device): the kernels read the query rows from it and write D / I into it, so a
 * call is the kernel launch(es) plus one stream synchronisation, no copy calls. Synchronous. */
int nrb_search_small_host(const nrb_matrix* b, const float* xq_host, int32_t nq, int32_t d, int32_t metric, int32_t k,
                          int64_t id_base, float* D_host, int64_t* I_host, void* stream);
/* HBM-regime inverted-list scan for small batches (north_star item 3; IVFFlatScanner over
 * nprobe lists per query, Retrieval.py:32-34 in IndexIVFFlat form): block per (query, probed
 * list, 256-row chunk), a warp per row with 128-bit loads of the list-contiguous raw plane,
 * exact fp32 scores to scratch, block-per-query radix select. Algorithmic bytes = sum over
 * (query, probed list) of |list| * kp * 4. nq * nprobe <= 65,535. xq plain fp32 [nq, d]. */
size_t nrb_ivf_scan_small_workspace(int64_t nq, int32_t nprobe, int32_t max_list_len, int64_t ntotal, int32_t k);
int nrb_ivf_scan_small(const float* xq, int64_t ldq, int32_t nq, int32_t d, const nrb_matrix* lists,
                       const int32_t* offsets, int32_t nlist, int32_t max_list_len, const int64_t* ids,
                       const int64_t* coarse, int32_t nprobe, int32_t metric, int32_t k, float* D, int64_t* I,
                       void* workspace, size_t workspace_bytes, void* stream);
/* Search-time ID selectors (faiss SearchParameters::sel) on the three routes above: the same calls
 * with two more arguments, member i64 (device; nrb_id_select's output) and keep. Only the rows with
 * member[row] == keep take part; keep = 0 evaluates faiss's IDSelectorNot of the selector that
 * produced member, with no extra pass. member is indexed like the plane the kernel scans: catalog
 * rows (b) for the flat forms, packed list rows (lists, the order of ids) for the IVF scan. A warp
 * skips the row load of an unselected row, and the selection treats such rows as absent, not as low
 * scores: when fewer than k rows qualify, the result is padded exactly as for k > n (I = -1,
 * D = -FLT_MAX / +FLT_MAX).
 * Workspaces as for the unfiltered calls; nrb_search_small_host_sel stays one synchronous call and
 * runs after the kernel that wrote member when both are queued on `stream`. */
int nrb_search_small_sel(const float* xq, int64_t ldq, int32_t nq, int32_t d, const nrb_matrix* b, int32_t metric,
                         int32_t k, int64_t id_base, float* D, int64_t* I, void* workspace, size_t workspace_bytes,
                         void* stream, const int64_t* member, int64_t keep);
int nrb_search_small_host_sel(const nrb_matrix* b, const float* xq_host, int32_t nq, int32_t d, int32_t metric, int32_t k,
                              int64_t id_base, float* D_host, int64_t* I_host, void* stream, const int64_t* member,
                              int64_t keep);
int nrb_ivf_scan_small_sel(const float* xq, int64_t ldq, int32_t nq, int32_t d, const nrb_matrix* lists,
                           const int32_t* offsets, int32_t nlist, int32_t max_list_len, const int64_t* ids,
                           const int64_t* coarse, int32_t nprobe, int32_t metric, int32_t k, float* D, int64_t* I,
                           void* workspace, size_t workspace_bytes, void* stream, const int64_t* member, int64_t keep);

/* Retrieval.py:6-8 on the device (SURVEY 8f row 1): table f64[n, width] = embedding values followed by
 * the article id (news/article_table.npy) -> emb f32[n, width-1] C-contiguous, ids i64[n]. */
int nrb_split_table_f64(const double* table, int64_t n, int32_t width, float* emb, int64_t* ids, void* stream);

/* ---- external ids (faiss IndexIDMap, IndexIVF::add_with_ids / remove_ids) -------------------
 * The reference keeps the article ids in an array beside the index and translates row positions
 * by hand (Retrieval.py:7 splits article_ids off the table, Retrieval.py:23 maps rows to ids);
 * these entry points let the index carry the ids and drop rows by id.
 * nrb_id_select: faiss IDSelectorBatch / IDSelectorRange over n ids: member[i] = 1 if ids[i] is
 * selected, else 0. ids == NULL: the id of row i is i (IndexFlat without an id map). batch == NULL:
 * range, imin <= id < imax (empty when imin >= imax). Otherwise a set of nbatch ids (any int64
 * value, duplicates allowed; nbatch == 0 selects nothing), built in the workspace as an
 * open-addressing hash table (64-bit atomicCAS inserts, then one probe per id); the empty-slot
 * sentinel (-1) is tracked by a separate flag word, so a batch may contain it. member is i64 so it
 * feeds nrb_ivf_build_lists(member, n, 2, ...) directly: a stable keep / remove partition,
 * offsets[1] = rows kept. Workspace: nrb_id_select_workspace(nbatch) bytes (0 for a range). */
size_t nrb_id_select_workspace(int64_t nbatch);
int nrb_id_select(const int64_t* ids, int64_t n, const int64_t* batch, int64_t nbatch, int64_t imin,
                  int64_t imax, int64_t* member, void* workspace, size_t workspace_bytes, void* stream);
/* IndexIDMap::search's label translation, in place: I[i] = I[i] < 0 ? I[i] : id_map[I[i]]. */
int nrb_map_ids(const int64_t* id_map, int64_t* I, int64_t n, void* stream);
/* Bucket keys of a filtered IVF scan: out[i] = member[i] == keep ? key[i] : drop. With key = the
 * list of every row and drop = nlist, nrb_ivf_build_lists(out, n, nlist + 1, ...) lays out the lists
 * of the selected rows only (in the same order as the unfiltered lists) and puts the rest in bucket
 * nlist, which the scan never reads. */
int nrb_sel_keys(const int64_t* member, int64_t keep, const int64_t* key, int64_t n, int64_t drop, int64_t* out,
                 void* stream);

/* Wire format of the all-to-all by query range (the exchange step of the catalog-sharded search):
 * P[i] = (fp32 bits of D[i]) << 32 | uint32(I[i] - id_base), 0xffffffff in the low word when
 * I[i] < 0. 8 bytes per candidate, one collective instead of two. n = nq * k elements. */
int nrb_pack_topk(const float* D, const int64_t* I, int64_t id_base, int64_t n, uint64_t* P, void* stream);
/* P u64[nparts, nq, k] (each part best-first) + bases i64[nparts] (device; the id_base each part was
 * packed with) -> global top-k D f32[nq, k], I i64[nq, k]. Exact ties resolve by part order. */
int nrb_merge_topk_packed(const uint64_t* P, const int64_t* bases, int32_t nparts, int64_t nq, int32_t k,
                          int32_t metric, float* D, int64_t* I, void* stream);
/* The wire format of the id-carrying sharded indexes, whose ids are arbitrary int64 values rather
 * than offsets from a shard base: 16 bytes per candidate, still one collective per chunk.
 * P u64[n, 2]: P[t][0] = fp32 bits of D[t] << 32 | (I[t] < 0 ? 0xffffffff : 0), P[t][1] = I[t]. */
int nrb_pack_topk_ids(const float* D, const int64_t* I, int64_t n, uint64_t* P, void* stream);
/* P u64[nparts, nq, k, 2] (each part best-first) -> D f32[nq, k], I i64[nq, k]. Exact ties resolve by
 * part order, then list position, as nrb_merge_topk_packed does. */
int nrb_merge_topk_packed_ids(const uint64_t* P, int32_t nparts, int64_t nq, int32_t k, int32_t metric,
                              float* D, int64_t* I, void* stream);

/* Per-query exclusion after an over-fetched search. Row r of Din/Iin (f32/i64 [nrows, kin], best-first,
 * labels already translated) belongs to query q = qidx ? qidx[r] : r. Entries whose label is >= 0 and
 * occurs in excl_ids[excl_off[q] .. excl_off[q+1]) are dropped; the first k survivors, in order, go to
 * D[q, :], I[q, :] (f32/i64 [*, k]); the rest of the row is padding (I = -1, D = -FLT_MAX for IP,
 * +FLT_MAX for L2). 1 <= k <= kin <= 128. A warp per row; the cost is O(kin * list length / 32). */
int nrb_exclude_topk(const float* Din, const int64_t* Iin, int64_t nrows, int32_t kin, const int64_t* qidx,
                     const int64_t* excl_off, const int64_t* excl_ids, int32_t metric, int32_t k,
                     float* D, int64_t* I, void* stream);

/* Stable compaction of CSR lists: off i64[nrows+1] (off[0] = 0, off[nrows] = nids) over ids i64[nids].
 * Entry i is kept when member[i] == 1 (what nrb_id_select wrote over the list ids) and written as
 * ids[i] - shift; out_off i64[nrows+1] are the kept lists' offsets, out_ids (room for nids) their
 * entries, in the input order within each row. Deterministic. ids, member and out_ids may be NULL
 * when nids == 0; nrows == 0 writes out_off[0] = 0. The sharded indexes use it to keep the part of
 * per-query exclusion lists a shard holds, in the shard's label space.
 * Workspace: nrb_csr_compact_workspace(nrows) bytes. */
size_t nrb_csr_compact_workspace(int64_t nrows);
int nrb_csr_compact(const int64_t* off, const int64_t* ids, int64_t nrows, int64_t nids, const int64_t* member,
                    int64_t shift, int64_t* out_off, int64_t* out_ids, void* workspace, size_t workspace_bytes,
                    void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NRB200_H */
