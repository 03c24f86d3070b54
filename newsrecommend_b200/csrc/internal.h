// Internal C++ interfaces between the translation units of libnrb200.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/nrb200.h"

namespace nrb {

// One unit of selection work: rows [a_row0, a_row0 + a_rows) of the query-side matrix against
// rows [b_row0, b_row0 + b_rows) of the item-side matrix. a_rows <= 128. Unit u writes its
// partial result (best-first top-k per row, padded) to partial rows [u*128, u*128 + 128).
struct Unit {
    int a_row0;
    int a_rows;
    int b_row0;
    int b_rows;
};

constexpr int UNIT_ROWS = 128;

// ---- topk_tc.cu: tcgen05 3xTF32 distance + selection. n_units lives in device memory so that
// unit lists built on the device (IVF grouping) need no host round trip; `grid` is the host's
// launch width (<= number of SMs).
int tc_available();  // 1 when the current device is sm_100
size_t tc_scratch_bytes(int grid);
int tc_grid(int n_units_upper);
// gthr (optional): zero-initialised per-query shared bounds; row_map/row_div map query-side rows
// to queries (null = identity).
int launch_topk_tc_dev(const nrb_matrix* a, const nrb_matrix* b, const Unit* units,
                       const int* n_units_dev, int grid, int metric, int k, float* part_key,
                       int* part_idx, void* scratch, size_t scratch_bytes, unsigned* gthr,
                       const int* row_map, int row_div, cudaStream_t st);

// 1xTF32 filter + exact refine (NRB_PATH_TC1): partial rows are `pw` = k + TC1_EXTRA wide and hold
// every candidate within the error margin of the k-th; row_flags[a_row] = 1 marks rows whose
// margin set did not fit. margin_scale = 2 * eps * max|x| (the kernel multiplies by |q|).
constexpr int TC1_EXTRA = 32;      // margin slots per row when they fit (IVF scans: partial rows per (query, list)) ...
constexpr int TC1_EXTRA_FLAT = 96; // ... flat searches: as many as the 128-entry exact stage of the refine can take
constexpr int TC1_MIN_EXTRA = 16;  // ... never fewer than this (partial rows are at most 128 wide)
constexpr int TC1_MAX_PW = 128;
static inline int tc1_pw(int k, bool flat = false) {
    const int extra = flat ? TC1_EXTRA_FLAT : TC1_EXTRA;
    return k + extra <= TC1_MAX_PW ? k + extra : TC1_MAX_PW;
}
static inline int tc1_k_ok(int k) { return k + TC1_MIN_EXTRA <= TC1_MAX_PW; }
constexpr float TC1_EPS = 1.1f / 1024.f;  // both operands rounded to tf32 (2 * 2^-11) + accumulation slack
int tc1_eligible(const nrb_matrix* a, const nrb_matrix* b, int k);
// fp16 filter (NRB_PATH_TC16): same kernel and error bound (fp16 and tf32 both carry an 11-bit
// significand) on power-of-two scaled fp16 planes, at twice the tensor rate.
int tc16_eligible(const nrb_matrix* a, const nrb_matrix* b, int k);
int launch_topk_tc1_dev(const nrb_matrix* a, const nrb_matrix* b, const Unit* units,
                        const int* n_units_dev, int grid, int metric, int k, int pw, float margin_scale,
                        float* part_key, int* part_idx, int* part_cnt, int* row_flags, void* scratch,
                        size_t scratch_bytes, unsigned* gthr, const int* row_map, int row_div, int f16,
                        int single, int ivf_mode, cudaStream_t st);
// ivf_mode: 0 = flat search; 1 = IVF list scan, cold rows (two resident query tiles: units are short);
// 2 = IVF phase B, every row starts from its query's shared bound (also: no scheduled prunes, no union
// prune at the end of a unit)

// ---- topk_simt.cu: fp32 CUDA-core distance + selection over the same Unit list
size_t simt_scratch_bytes(int grid);
int simt_grid(int n_units_upper);
int launch_topk_simt_dev(const nrb_matrix* a, const nrb_matrix* b, const Unit* units,
                         const int* n_units_dev, int grid, int metric, int k, float* part_key,
                         int* part_idx, void* scratch, size_t scratch_bytes, cudaStream_t st);

// ---- kernels_misc.cu
// src[q*S + s] = partial row index (or -1). id_map (optional) translates idx -> external id;
// otherwise id = idx + id_base.
int launch_select(const float* part_key, const int* part_idx, const int* src, int S, int64_t nq,
                  int k, int metric, const int64_t* id_map, int64_t id_base, float* D, int64_t* I,
                  cudaStream_t st);
// filter paths: gathers the unsorted partial rows of every query (part_cnt entries each), cuts at
// (k-th estimate - margin), rescoring the survivors exactly in fp32 and sorting them
int launch_gather_refine(const float* part_key, const int* part_idx, const int* part_cnt, const int* src, int S,
                         int64_t nq, int k, int pw, int metric, const nrb_matrix* q, const nrb_matrix* b, float eps_xmax,
                         int64_t id_base, const int64_t* id_map, int* flags, float* D, int64_t* I, cudaStream_t st);
int launch_compact_flags(const int* flags, int64_t n, int* list, int* count, cudaStream_t st);
int launch_scatter_results(const float* Df, const int64_t* If, const int* list, int n, int k, float* D,
                           int64_t* I, cudaStream_t st);
int launch_fill_flat_units(Unit* units, int* n_units_out, int* src, int64_t nq, int64_t nb, int nqt,
                           int full_pairs, int tail_pairs, int tsplit, int chunk_rows, int wgs, cudaStream_t st);
// single-CTA plan: unit c*nqt + t = query tile t against item chunk c (no phantom units)
int launch_fill_flat_units_single(Unit* units, int* n_units_out, int* src, int64_t nq, int64_t nb, int nqt,
                                  int tsplit, int chunk_rows, int wgs, cudaStream_t st);
size_t counting_sort_ws(int64_t n, int nb);
int launch_counting_sort_i64(const int64_t* key, int64_t n, int nb, int* offsets, int* order,
                             int* pos_of, void* ws, size_t ws_bytes, cudaStream_t st);
int launch_pack_rows(const float* x, int64_t n, int d, int64_t ldx, int kp, float* raw, float* hi, float* lo,
                     float* norms, cudaStream_t st);
int launch_gather_rows(const float* src, int width, const int32_t* idx, int div, int64_t n,
                       float* dst, cudaStream_t st);
int launch_gather_scalar(const float* src, const int32_t* idx, int div, int64_t n, float* dst,
                         cudaStream_t st);

size_t kmeans_update_ws(int64_t n, int k, int kp);
// cent_in (optional, f32[k, d]): the centroids the assignment was made against -> obj_out (f64) = the
// k-means objective sum over rows of |x - c|^2 (L2) or x.c (IP), exact fp32 products, fixed-order fp64 sum
int launch_kmeans_update(const float* x_raw, int64_t n, int d, int kp, const int64_t* assign, int k, float* centroids,
                         float* hassign, void* workspace, const float* cent_in, int metric, double* obj_out,
                         cudaStream_t st, double* sums_out = nullptr);
int launch_km_split(int d, int k, int64_t n, float* hassign, float* centroids, double* stats, cudaStream_t st);

// small_batch.cu: exact fp32 recompute of the rows listed in list[0 .. *count) for k = 1 (device-driven)
constexpr int K1_FALLBACK_MAX_ROWS = 65536;  // item rows up to which flagged k = 1 rows are recomputed on the device
int launch_exact_k1_fallback(const nrb_matrix* q, const nrb_matrix* b, int metric, int64_t id_base, const int* list,
                             const int* count, float* D, int64_t* I, cudaStream_t st);

int sm_count();
// NRB_OK, or NRB_ERR_NO_DEVICE (with the message set) when there is no sm_100 device
int require_device();

}  // namespace nrb
