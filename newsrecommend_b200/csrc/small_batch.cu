// Low-latency exact search for tiny query batches, and the HBM-regime inverted-list scan.
//
// faiss takes a different route when nq < distance_compute_blas_threshold (20): no sgemm, every
// (query, item) distance is computed directly in fp32 and pushed through the heap (SURVEY 3.2;
// this is the route each of the 50,000 calls at Retrieval.py:32 takes with nq = 1). The B200 form
// of that route is a bandwidth problem, not a tensor-core problem: every catalog (or probed-list)
// row is read ONCE with 128-bit loads, a warp owns a row, all queries of the group sit in shared
// memory, and the scores go to a small scratch (nq x n floats) from which one block per query
// selects the exact top-k by radix select + a 128-entry bitonic sort. No plan kernels, no unit
// lists, no partial rows, no host synchronisation inside; two launches (one when the catalog is
// small enough for the scores to stay in shared memory: the 300-centroid search of the reference).
//
//   small_scores_kernel<QG>      flat: rows x (up to 16 queries) -> scores[q][row]
//   small_fused_kernel<QG>       flat, n <= FUSED_MAX_ROWS: scores in shared memory + selection
//   ivf_small_scores_kernel      (query, probe, row chunk) -> scores[q][prefix(q, probe) + r]
//   small_select_kernel          block per query: exact top-k of the score row
//
// Algorithmic bytes: flat n * kp * 4 per group of <= 16 queries; IVF sum over (query, probed list)
// of |list| * kp * 4 (SURVEY 8d "small nq: HBM").
//
// Search-time ID selectors (faiss SearchParameters::sel): the MASKED instantiations take a row mask
// member i64[n] (nrb_id_select's output, in the order of the plane the kernel scans) and a keep value.
// A warp reads member[row] first and skips the row load of an unselected row; its score slot gets
// absent_score(), which the masked selection sources map to the ordered key 0, below every real key
// (even -inf). Absent rows therefore sort after every selected row, and the result writers turn a
// candidate with ordered key 0 into padding (I = -1), so an unselected row never appears in a result.
#include <float.h>
#include <mutex>
#include <string.h>
#include <type_traits>

#include "common.cuh"
#include "internal.h"

namespace nrb {

constexpr int SMALL_QG = 16;             // queries that share one pass over the rows
constexpr int SMALL_THREADS = 256;       // 8 warps
constexpr int FUSED_MAX_ROWS = 8192;     // scores of one query in shared memory: 32 KB
constexpr int SELECT_MAX_K = 128;

// Sum of acc[i] over the warp for QG accumulators at once: a halving butterfly (each step keeps one
// half of the values and ships the other), QG - 1 + (5 - log2 QG) shuffles instead of 5 * QG.
// The total of acc[qi] ends up in every lane with lane / (32 / QG) == qi, returned as one float.
template <int QG>
__device__ __forceinline__ float warp_reduce_multi(float (&acc)[QG], int lane) {
    int m = QG;
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
        if (m > 1) {
            const int h = m >> 1;
            const bool up = (lane & o) != 0;
#pragma unroll
            for (int i = 0; i < QG / 2; i++) {
                if (i < h) {
                    const float keep = up ? acc[i + h] : acc[i];
                    const float send = up ? acc[i] : acc[i + h];
                    acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
                }
            }
            m = h;
        } else {
            acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], o);
        }
    }
    return acc[0];
}

// R rows (one per pointer) against QG queries held in shared memory (qs[q * kp + c]); kp % 32 == 0.
// Lane l owns columns [c*128 + 4l, c*128 + 4l + 4) of every 128-column chunk c. The loads of all R
// rows are issued before any arithmetic: R x 16 bytes in flight per lane and chunk.
// MASKED: only the rows whose bit is set in `use` are loaded (the others contribute zeros).
template <int QG, bool L2, int R, bool MASKED = false>
__device__ __forceinline__ void rows_scores(const float* const (&row)[R], const float* qs, int kp, int lane,
                                            float (&out)[R], unsigned use = ~0u) {
    float acc[R][QG];
#pragma unroll
    for (int r = 0; r < R; r++)
#pragma unroll
        for (int q = 0; q < QG; q++) acc[r][q] = 0.f;
    for (int c0 = 0; c0 < kp; c0 += 128) {
        const int col = c0 + lane * 4;
        if (col < kp) {
            float4 x[R];
#pragma unroll
            for (int r = 0; r < R; r++)
                x[r] = (!MASKED || ((use >> r) & 1u)) ? __ldg(reinterpret_cast<const float4*>(row[r] + col))
                                                      : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int q = 0; q < QG; q++) {
                const float4 y = *reinterpret_cast<const float4*>(qs + q * kp + col);
#pragma unroll
                for (int r = 0; r < R; r++) {
                    if (L2) {
                        const float a = y.x - x[r].x, b = y.y - x[r].y, c = y.z - x[r].z, d = y.w - x[r].w;
                        acc[r][q] = fmaf(a, a, acc[r][q]);
                        acc[r][q] = fmaf(b, b, acc[r][q]);
                        acc[r][q] = fmaf(c, c, acc[r][q]);
                        acc[r][q] = fmaf(d, d, acc[r][q]);
                    } else {
                        acc[r][q] = fmaf(x[r].x, y.x, acc[r][q]);
                        acc[r][q] = fmaf(x[r].y, y.y, acc[r][q]);
                        acc[r][q] = fmaf(x[r].z, y.z, acc[r][q]);
                        acc[r][q] = fmaf(x[r].w, y.w, acc[r][q]);
                    }
                }
            }
        }
    }
#pragma unroll
    for (int r = 0; r < R; r++) out[r] = warp_reduce_multi<QG>(acc[r], lane);
}

template <int QG, bool L2>
__device__ __forceinline__ float row_scores(const float* __restrict__ row, const float* qs, int kp, int lane) {
    const float* const rows[1] = {row};
    float out[1];
    rows_scores<QG, L2, 1>(rows, qs, kp, lane, out);
    return out[0];
}

// Queries [q0, q0 + QG) of xq (row stride ldq, d valid columns) into shared memory, zero padded
// to kp columns and to QG rows.
template <int QG>
__device__ __forceinline__ void stage_queries(const float* __restrict__ xq, int64_t ldq, int d, int kp, int q0, int nq,
                                              float* qs) {
    for (int t = threadIdx.x; t < QG * kp; t += blockDim.x) {
        const int q = t / kp, c = t - q * kp;
        qs[t] = (q0 + q < nq && c < d) ? xq[(int64_t)(q0 + q) * ldq + c] : 0.f;
    }
}

// Score of a row a MASKED kernel skipped: the NaN bit pattern 0xffffffff, which fp32 arithmetic never
// produces (it yields the canonical NaN 0x7fffffff). MaskedScoreSrc tests these bits before any
// arithmetic (negating a NaN leaves its sign unspecified) and returns them as the key: ordered_u32 == 0.
constexpr unsigned ABSENT_BITS = 0xffffffffu;
__device__ __forceinline__ float absent_score() { return __uint_as_float(ABSENT_BITS); }
// a sorted candidate that stands for an absent row (packed key word 0)
__device__ __forceinline__ bool absent_cand(unsigned long long c) { return (c >> 32) == 0; }

// ------------------------------------------------------------------ block-wide exact top-k
// Keys are "larger is better" (score, or -distance). Radix select over the ordered-uint image of
// the keys finds the exact k-th largest key T and how many elements equal to T belong to the
// answer; elements above T and the lowest-position elements equal to T are collected (<= k) and
// sorted by one warp (key descending, position ascending) into S.cand[0 .. kk). `src.key(i)` /
// `src.pos(i)` give the key and the reported position of element i. Histogram updates are
// aggregated per warp (match_any): the top byte of fp32 scores takes only a few distinct values.
struct SelectShared {
    unsigned hist[256];
    unsigned long long cand[SELECT_MAX_K];
    unsigned prefix, need, n_gt, n_eq, run;
    unsigned wsum[32];
};

template <typename Src>
__device__ __forceinline__ int block_select(const Src& src, int n, int k, SelectShared& S) {
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5;
    const int kk = k < n ? k : n;
    if (tid == 0) { S.prefix = 0; S.need = kk; S.n_gt = 0; S.n_eq = 0; S.run = 0; }
    if (kk < n) {
        unsigned mask = 0;
        for (int shift = 24; shift >= 0; shift -= 8) {
            for (int b = tid; b < 256; b += nt) S.hist[b] = 0;
            __syncthreads();
            const unsigned prefix = S.prefix;
            for (int base = 0; base < n; base += nt) {  // warp-uniform trip count
                const int i = base + tid;
                unsigned u = 0;
                bool in = false;
                if (i < n) {
                    u = ordered_u32(src.key(i));
                    in = (u & mask) == prefix;
                }
                const unsigned act = __ballot_sync(0xffffffffu, in);
                if (in) {
                    const unsigned bin = (u >> shift) & 255u;
                    const unsigned peers = __match_any_sync(act, bin);
                    if (lane == __ffs(peers) - 1) atomicAdd(&S.hist[bin], (unsigned)__popc(peers));
                }
            }
            __syncthreads();
            if (warp == 0) {
                // lane l owns bins [8l, 8l + 8); suffix sums from the top bin down
                unsigned h[8], sum = 0;
#pragma unroll
                for (int j = 0; j < 8; j++) { h[j] = S.hist[lane * 8 + j]; sum += h[j]; }
                unsigned suf = sum;  // inclusive suffix scan over the lanes
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const unsigned t = __shfl_down_sync(0xffffffffu, suf, o);
                    if (lane + o < 32) suf += t;
                }
                const unsigned above = suf - sum;  // elements in the bins of higher lanes
                const unsigned need = S.need;
                __syncwarp();
                if (above < need && suf >= need) {  // the k-th lies in this lane's bins
                    unsigned a = above;
                    bool found = false;
#pragma unroll
                    for (int j = 7; j >= 0; j--) {
                        if (!found && a + h[j] >= need) {
                            S.prefix = prefix | ((unsigned)(lane * 8 + j) << shift);
                            S.need = need - a;
                            found = true;
                        }
                        a += h[j];
                    }
                }
            }
            mask |= 255u << shift;
            __syncthreads();
        }
    }
    __syncthreads();
    const unsigned T = S.prefix, need_eq = S.need;
    const bool all = !(kk < n);
    // collect: everything above T (unordered) and the elements equal to T
    for (int i = tid; i < n; i += nt) {
        const float key = src.key(i);
        const unsigned u = ordered_u32(key);
        if (all || u > T) {
            const unsigned s = atomicAdd(&S.n_gt, 1u);
            S.cand[s] = pack_cand(key, src.pos(i));
        } else if (u == T) {
            const unsigned s = atomicAdd(&S.n_eq, 1u);
            if (s < need_eq) S.cand[(kk - need_eq) + s] = pack_cand(key, src.pos(i));
        }
    }
    __syncthreads();
    if (!all && S.n_eq > need_eq) {
        // more ties at T than slots: take the lowest positions, in order (block-wide ballot scan)
        for (int base = 0; base < n && S.run < need_eq; base += nt) {
            const int i = base + tid;
            const bool f = i < n && ordered_u32(src.key(i)) == T;
            const unsigned bal = __ballot_sync(0xffffffffu, f);
            if (lane == 0) S.wsum[warp] = __popc(bal);
            __syncthreads();
            unsigned before = S.run;
            for (int w = 0; w < warp; w++) before += S.wsum[w];
            const unsigned r = before + __popc(bal & ((1u << lane) - 1u));
            if (f && r < need_eq) S.cand[(kk - need_eq) + r] = pack_cand(src.key(i), src.pos(i));
            __syncthreads();
            if (tid == 0) { unsigned t = 0; for (int w = 0; w < (nt >> 5); w++) t += S.wsum[w]; S.run += t; }
            __syncthreads();
        }
    }
    if (warp == 0) {
        uint64_t c[4];
#pragma unroll
        for (int i = 0; i < 4; i++) { const int e = i * 32 + lane; c[i] = e < kk ? S.cand[e] : empty_cand(); }
        __syncwarp();
        warp_bitonic_desc<4>(c, lane);
#pragma unroll
        for (int i = 0; i < 4; i++) S.cand[i * 32 + lane] = c[i];
    }
    __syncthreads();
    return kk;
}

// score array source: key = +-value, reported position = base + i
struct ScoreSrc {
    const float* p;
    int base;
    bool l2;
    __device__ __forceinline__ float key(int i) const { const float v = p[i]; return l2 ? -v : v; }
    __device__ __forceinline__ int pos(int i) const { return base + i; }
};
// the same for the score rows of the MASKED kernels: an absent row keeps the key ABSENT_BITS
struct MaskedScoreSrc {
    const float* p;
    int base;
    bool l2;
    __device__ __forceinline__ float key(int i) const {
        const float v = p[i];
        return __float_as_uint(v) == ABSENT_BITS ? __uint_as_float(ABSENT_BITS) : (l2 ? -v : v);
    }
    __device__ __forceinline__ int pos(int i) const { return base + i; }
};
template <bool MASKED>
using ScoreSrcT = typename std::conditional<MASKED, MaskedScoreSrc, ScoreSrc>::type;
// packed-candidate source (second level of the two-level selection)
struct CandSrc {
    const unsigned long long* c;
    __device__ __forceinline__ float key(int i) const { return cand_key(c[i]); }
    __device__ __forceinline__ int pos(int i) const { return cand_idx(c[i]); }
};

// ------------------------------------------------------------------ flat
template <int QG, bool L2, int R, bool MASKED>
__global__ void __launch_bounds__(SMALL_THREADS)
small_scores_kernel(const float* __restrict__ xq, int64_t ldq, int nq, int d, const float* __restrict__ xb, int64_t nb,
                    int kp, float* __restrict__ scores, const int64_t* __restrict__ member, int64_t keep) {
    extern __shared__ __align__(16) float qs[];
    const int q0 = blockIdx.y * QG;
    stage_queries<QG>(xq, ldq, d, kp, q0, nq, qs);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (SMALL_THREADS / 32);
    constexpr int LPQ = 32 / QG;  // lanes that hold the total of one query
    const int q = lane / LPQ;
    const bool writer = (lane % LPQ) == 0 && q0 + q < nq;
    for (int64_t r = (int64_t)blockIdx.x * (SMALL_THREADS / 32) + (threadIdx.x >> 5); r < nb; r += warps * R) {
        const float* rows[R];
        unsigned use = 0;
#pragma unroll
        for (int j = 0; j < R; j++) {
            const int64_t rj = r + j * warps;
            rows[j] = xb + (rj < nb ? rj : r) * kp;
            if (MASKED && rj < nb && member[rj] == keep) use |= 1u << j;
        }
        float out[R];
        if (MASKED && use == 0) {
#pragma unroll
            for (int j = 0; j < R; j++) out[j] = 0.f;
        } else {
            rows_scores<QG, L2, R, MASKED>(rows, qs, kp, lane, out, use);
        }
#pragma unroll
        for (int j = 0; j < R; j++) {
            const int64_t rj = r + j * warps;
            if (writer && rj < nb)
                scores[(int64_t)(q0 + q) * nb + rj] = (!MASKED || ((use >> j) & 1u)) ? out[j] : absent_score();
        }
    }
}

// results of one query from the sorted candidates in S.cand (MASKED: absent rows become padding)
template <bool MASKED>
__device__ __forceinline__ void write_flat_results(const SelectShared& S, int kk, int k, bool l2, int64_t id_base,
                                                   float* __restrict__ Dq, int64_t* __restrict__ Iq) {
    for (int e = threadIdx.x; e < k; e += blockDim.x) {
        const int ps = e < kk && !(MASKED && absent_cand(S.cand[e])) ? cand_idx(S.cand[e]) : -1;
        const float key = cand_key(S.cand[e < kk ? e : 0]);
        Dq[e] = ps < 0 ? (l2 ? FLT_MAX : -FLT_MAX) : (l2 ? -key : key);
        Iq[e] = ps < 0 ? -1 : id_base + ps;
    }
}

// one level: block per query over the whole score row
template <bool MASKED>
__global__ void __launch_bounds__(1024)
small_select_kernel(const float* __restrict__ scores, int64_t ld, int n, int k, int l2, int64_t id_base,
                    float* __restrict__ D, int64_t* __restrict__ I) {
    __shared__ SelectShared S;
    const int q = blockIdx.x;
    ScoreSrcT<MASKED> src{scores + (int64_t)q * ld, 0, l2 != 0};
    const int kk = block_select(src, n, k, S);
    write_flat_results<MASKED>(S, kk, k, l2 != 0, id_base, D + (int64_t)q * k, I + (int64_t)q * k);
}

// two levels for long rows: block (b, q) selects the top-k of slice b of query q's scores into
// cands[q][b][k] (padded with empty candidates); small_select2_kernel then selects among the B*k.
template <bool MASKED>
__global__ void __launch_bounds__(1024)
small_select1_kernel(const float* __restrict__ scores, int64_t ld, int n, int k, int l2,
                     unsigned long long* __restrict__ cands) {
    __shared__ SelectShared S;
    const int q = blockIdx.y, b = blockIdx.x, B = gridDim.x;
    const int per = (n + B - 1) / B;
    const int lo = min(n, b * per), hi = min(n, lo + per);
    ScoreSrcT<MASKED> src{scores + (int64_t)q * ld + lo, lo, l2 != 0};
    const int kk = block_select(src, hi - lo, k, S);
    unsigned long long* out = cands + ((int64_t)q * B + b) * k;
    for (int e = threadIdx.x; e < k; e += blockDim.x) out[e] = e < kk ? S.cand[e] : empty_cand();
}

template <bool MASKED>
__global__ void __launch_bounds__(1024)
small_select2_kernel(const unsigned long long* __restrict__ cands, int B, int k, int l2, int64_t id_base,
                     float* __restrict__ D, int64_t* __restrict__ I) {
    __shared__ SelectShared S;
    const int q = blockIdx.x;
    CandSrc src{cands + (int64_t)q * B * k};
    const int kk = block_select(src, B * k, k, S);
    write_flat_results<MASKED>(S, kk, k, l2 != 0, id_base, D + (int64_t)q * k, I + (int64_t)q * k);
}

// n <= FUSED_MAX_ROWS: one block per query computes the scores into shared memory and selects.
template <bool L2, bool MASKED>
__global__ void __launch_bounds__(SMALL_THREADS)
small_fused_kernel(const float* __restrict__ xq, int64_t ldq, int nq, int d, const float* __restrict__ xb, int n, int kp,
                   int k, int64_t id_base, float* __restrict__ D, int64_t* __restrict__ I,
                   const int64_t* __restrict__ member, int64_t keep) {
    extern __shared__ __align__(16) float sm[];
    float* qs = sm;            // [kp]
    float* sc = sm + kp;       // [n]
    __shared__ SelectShared S;
    const int q = blockIdx.x;
    stage_queries<1>(xq, ldq, d, kp, q, nq, qs);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    constexpr int W = SMALL_THREADS / 32, R = 4;
    for (int r = threadIdx.x >> 5; r < n; r += W * R) {
        const float* rows[R];
        unsigned use = 0;
#pragma unroll
        for (int j = 0; j < R; j++) {
            rows[j] = xb + (int64_t)(r + j * W < n ? r + j * W : r) * kp;
            if (MASKED && r + j * W < n && member[r + j * W] == keep) use |= 1u << j;
        }
        float out[R];
        if (MASKED && use == 0) {
#pragma unroll
            for (int j = 0; j < R; j++) out[j] = 0.f;
        } else {
            rows_scores<1, L2, R, MASKED>(rows, qs, kp, lane, out, use);
        }
#pragma unroll
        for (int j = 0; j < R; j++)
            if (lane == 0 && r + j * W < n) sc[r + j * W] = (!MASKED || ((use >> j) & 1u)) ? out[j] : absent_score();
    }
    __syncthreads();
    ScoreSrcT<MASKED> src{sc, 0, L2};
    const int kk = block_select(src, n, k, S);
    write_flat_results<MASKED>(S, kk, k, L2, id_base, D + (int64_t)q * k, I + (int64_t)q * k);
}

// ------------------------------------------------------------------ IVF (HBM-regime list scan)
// grid = (row chunks of IVF_CHUNK, nq * nprobe). Block (c, q*nprobe + p) scans rows
// [c*IVF_CHUNK, ...) of the p-th probed list of query q; one warp per row (four rows in flight),
// 128-bit loads of the list-contiguous raw plane; scores[q*ld + prefix(q, p) + r].
constexpr int IVF_CHUNK = 256;

template <bool L2, bool MASKED>
__global__ void __launch_bounds__(SMALL_THREADS)
ivf_small_scores_kernel(const float* __restrict__ xq, int64_t ldq, int d, const float* __restrict__ xb, int kp,
                        const int* __restrict__ offsets, const int64_t* __restrict__ coarse, int nprobe,
                        float* __restrict__ scores, int64_t ld, const int64_t* __restrict__ member, int64_t keep) {
    extern __shared__ __align__(16) float qs[];
    const int q = blockIdx.y / nprobe, p = blockIdx.y - q * nprobe;
    const int64_t l = coarse[(int64_t)q * nprobe + p];
    if (l < 0) return;
    const int row0 = offsets[l], len = offsets[l + 1] - row0;
    const int c0 = blockIdx.x * IVF_CHUNK;
    if (c0 >= len) return;
    int64_t prefix = 0;
    for (int j = 0; j < p; j++) {
        const int64_t lj = coarse[(int64_t)q * nprobe + j];
        if (lj >= 0) prefix += offsets[lj + 1] - offsets[lj];
    }
    stage_queries<1>(xq, ldq, d, kp, q, q + 1, qs);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int c1 = c0 + IVF_CHUNK < len ? c0 + IVF_CHUNK : len;
    constexpr int W = SMALL_THREADS / 32, R = 4;
    for (int r = c0 + (threadIdx.x >> 5); r < c1; r += W * R) {
        const float* rows[R];
        unsigned use = 0;
#pragma unroll
        for (int j = 0; j < R; j++) {
            rows[j] = xb + (int64_t)(row0 + (r + j * W < c1 ? r + j * W : r)) * kp;
            if (MASKED && r + j * W < c1 && member[row0 + r + j * W] == keep) use |= 1u << j;
        }
        float out[R];
        if (MASKED && use == 0) {
#pragma unroll
            for (int j = 0; j < R; j++) out[j] = 0.f;
        } else {
            rows_scores<1, L2, R, MASKED>(rows, qs, kp, lane, out, use);
        }
#pragma unroll
        for (int j = 0; j < R; j++)
            if (lane == 0 && r + j * W < c1)
                scores[(int64_t)q * ld + prefix + r + j * W] = (!MASKED || ((use >> j) & 1u)) ? out[j] : absent_score();
    }
}

// segment table of one query: seg_end[p] = rows of probes 0..p, seg_row0[p] = first packed row of probe p
__device__ __forceinline__ int ivf_segments(const int* __restrict__ offsets, const int64_t* __restrict__ coarse_q, int nprobe,
                                            int* seg_end, int* seg_row0) {
    if (threadIdx.x == 0) {
        int tot = 0;
        for (int p = 0; p < nprobe; p++) {
            const int64_t l = coarse_q[p];
            const int r0 = l < 0 ? 0 : offsets[l], len = l < 0 ? 0 : offsets[l + 1] - r0;
            tot += len;
            seg_end[p] = tot;
            seg_row0[p] = r0;
        }
    }
    __syncthreads();
    return seg_end[nprobe - 1];
}

template <bool MASKED>
__device__ __forceinline__ void write_ivf_results(const SelectShared& S, int kk, int k, bool l2, const int* seg_end,
                                                  const int* seg_row0, const int64_t* __restrict__ ids,
                                                  float* __restrict__ Dq, int64_t* __restrict__ Iq) {
    for (int e = threadIdx.x; e < k; e += blockDim.x) {
        const int ps = e < kk && !(MASKED && absent_cand(S.cand[e])) ? cand_idx(S.cand[e]) : -1;
        const float key = cand_key(S.cand[e < kk ? e : 0]);
        int64_t id = -1;
        if (ps >= 0) {
            int p = 0;
            while (ps >= seg_end[p]) p++;
            id = ids[seg_row0[p] + ps - (p ? seg_end[p - 1] : 0)];
        }
        Dq[e] = ps < 0 ? (l2 ? FLT_MAX : -FLT_MAX) : (l2 ? -key : key);
        Iq[e] = id;
    }
}

// level 1: block (b, q) selects over slice b of query q's concatenated list scores
template <bool MASKED>
__global__ void __launch_bounds__(1024)
ivf_small_select1_kernel(const float* __restrict__ scores, int64_t ld, const int* __restrict__ offsets,
                         const int64_t* __restrict__ coarse, int nprobe, int k, int l2,
                         unsigned long long* __restrict__ cands) {
    __shared__ SelectShared S;
    __shared__ int seg_end[SELECT_MAX_K], seg_row0[SELECT_MAX_K];
    const int q = blockIdx.y, b = blockIdx.x, B = gridDim.x;
    const int n = ivf_segments(offsets, coarse + (int64_t)q * nprobe, nprobe, seg_end, seg_row0);
    const int per = (n + B - 1) / B;
    const int lo = min(n, b * per), hi = min(n, lo + per);
    ScoreSrcT<MASKED> src{scores + (int64_t)q * ld + lo, lo, l2 != 0};
    const int kk = block_select(src, hi - lo, k, S);
    unsigned long long* out = cands + ((int64_t)q * B + b) * k;
    for (int e = threadIdx.x; e < k; e += blockDim.x) out[e] = e < kk ? S.cand[e] : empty_cand();
}

template <bool MASKED>
__global__ void __launch_bounds__(1024)
ivf_small_select2_kernel(const unsigned long long* __restrict__ cands, int B, const int* __restrict__ offsets,
                         const int64_t* __restrict__ coarse, int nprobe, const int64_t* __restrict__ ids, int k, int l2,
                         float* __restrict__ D, int64_t* __restrict__ I) {
    __shared__ SelectShared S;
    __shared__ int seg_end[SELECT_MAX_K], seg_row0[SELECT_MAX_K];
    const int q = blockIdx.x;
    ivf_segments(offsets, coarse + (int64_t)q * nprobe, nprobe, seg_end, seg_row0);
    CandSrc src{cands + (int64_t)q * B * k};
    const int kk = block_select(src, B * k, k, S);
    write_ivf_results<MASKED>(S, kk, k, l2 != 0, seg_end, seg_row0, ids, D + (int64_t)q * k, I + (int64_t)q * k);
}

// ------------------------------------------------------------------ exact k = 1 fallback (no host round trip)
// Rows a filter path flagged (margin set overflow, heavy ties) when k = 1 and the item side is
// small (k-means assignment, IndexIVFFlat.add: rows x centroids): recomputed here exactly in fp32,
// driven by the DEVICE-side list of flagged rows, so the caller needs no synchronisation. One block
// per flagged row (grid-stride over list[0 .. *count)); ties resolve to the lowest id.
template <bool L2>
__global__ void __launch_bounds__(SMALL_THREADS)
exact_k1_fallback_kernel(const float* __restrict__ qraw, const float* __restrict__ braw, int nb, int kp,
                         const int* __restrict__ list, const int* __restrict__ count, int64_t id_base,
                         float* __restrict__ D, int64_t* __restrict__ I) {
    extern __shared__ __align__(16) float qs[];
    __shared__ unsigned long long best[SMALL_THREADS / 32];
    const int n = *count;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int e = blockIdx.x; e < n; e += gridDim.x) {
        const int q = list[e];
        for (int c = threadIdx.x; c < kp; c += blockDim.x) qs[c] = qraw[(int64_t)q * kp + c];
        __syncthreads();
        unsigned long long bw = empty_cand();
        for (int r = warp; r < nb; r += SMALL_THREADS / 32) {
            const float s = row_scores<1, L2>(braw + (int64_t)r * kp, qs, kp, lane);
            const unsigned long long c = pack_cand(L2 ? -s : s, r);
            bw = c > bw ? c : bw;
        }
        if (lane == 0) best[warp] = bw;
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned long long b = best[0];
            for (int w = 1; w < SMALL_THREADS / 32; w++) b = best[w] > b ? best[w] : b;
            const float key = cand_key(b);
            D[q] = L2 ? -key : key;
            I[q] = id_base + cand_idx(b);
        }
        __syncthreads();
    }
}

int launch_exact_k1_fallback(const nrb_matrix* q, const nrb_matrix* b, int metric, int64_t id_base, const int* list,
                             const int* count, float* D, int64_t* I, cudaStream_t st) {
    NRB_REQUIRE(q->raw && b->raw && q->kp == b->kp && b->n > 0 && b->n < (1LL << 31), "k1 fallback: raw planes required");
    const int64_t cap = q->n < 2048 ? q->n : 2048;
    const unsigned grid = (unsigned)(cap < 1 ? 1 : cap);
    const size_t sh = (size_t)q->kp * sizeof(float);
    if (metric == NRB_METRIC_L2)
        exact_k1_fallback_kernel<true><<<grid, SMALL_THREADS, sh, st>>>(q->raw, b->raw, (int)b->n, q->kp, list, count, id_base, D, I);
    else
        exact_k1_fallback_kernel<false><<<grid, SMALL_THREADS, sh, st>>>(q->raw, b->raw, (int)b->n, q->kp, list, count, id_base, D, I);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

// ------------------------------------------------------------------ host side
constexpr int SELECT_SLICE = 8192;  // elements per first-level selection block
constexpr int SELECT_MAX_B = 64;

static int select_slices(int64_t n) {
    if (n <= 2 * SELECT_SLICE) return 1;
    const int64_t b = (n + SELECT_SLICE - 1) / SELECT_SLICE;
    return (int)(b > SELECT_MAX_B ? SELECT_MAX_B : b);
}

static int small_grid_rows(int64_t nb, int rows_per_iter) {
    const int64_t per_block = (int64_t)(SMALL_THREADS / 32) * rows_per_iter * 2;  // >= 2 iterations per warp
    const int64_t want = (nb + per_block - 1) / per_block;
    const int64_t cap = (int64_t)sm_count() * 8;
    return (int)(want < 1 ? 1 : (want > cap ? cap : want));
}

struct SmallWs {
    float* scores;
    unsigned long long* cands;
    size_t total;
};
static SmallWs carve_small(void* ws, int64_t nq, int64_t ld, int B, int k) {
    char* w = (char*)ws;
    SmallWs s;
    size_t off = 0;
    s.scores = (float*)(w ? w + off : nullptr);
    off += align_up((size_t)nq * (size_t)(ld > 0 ? ld : 1) * sizeof(float), 256);
    s.cands = (unsigned long long*)(w ? w + off : nullptr);
    off += align_up((size_t)nq * B * k * sizeof(unsigned long long), 256);
    s.total = off;
    return s;
}

// member == nullptr: every row (the unmasked kernels); else the rows with member[row] == keep
template <bool L2, bool MASKED>
static int small_flat_launch(const float* xq, int64_t ldq, int nq, int d, const nrb_matrix* b, int k, int64_t id_base,
                             void* workspace, float* D, int64_t* I, const int64_t* member, int64_t keep, cudaStream_t st) {
    const int kp = b->kp;
    const int n = (int)b->n;
    if (b->n <= FUSED_MAX_ROWS) {
        const size_t sh = (size_t)(kp + n) * sizeof(float);
        small_fused_kernel<L2, MASKED><<<nq, SMALL_THREADS, sh, st>>>(xq, ldq, nq, d, b->raw, n, kp, k, id_base, D, I,
                                                                     member, keep);
        NRB_LAUNCH_CHECK();
        return NRB_OK;
    }
    const int B = select_slices(n);
    const SmallWs w = carve_small(workspace, nq, n, B, k);
    if (nq == 1) {
        small_scores_kernel<1, L2, 4, MASKED><<<dim3(small_grid_rows(n, 4), 1), SMALL_THREADS, kp * sizeof(float), st>>>(
            xq, ldq, nq, d, b->raw, b->n, kp, w.scores, member, keep);
    } else if (nq <= 4) {
        small_scores_kernel<4, L2, 4, MASKED><<<dim3(small_grid_rows(n, 4), 1), SMALL_THREADS, 4 * kp * sizeof(float), st>>>(
            xq, ldq, nq, d, b->raw, b->n, kp, w.scores, member, keep);
    } else {
        small_scores_kernel<SMALL_QG, L2, 4, MASKED><<<dim3(small_grid_rows(n, 4), (nq + SMALL_QG - 1) / SMALL_QG),
                                                       SMALL_THREADS, SMALL_QG * kp * sizeof(float), st>>>(
            xq, ldq, nq, d, b->raw, b->n, kp, w.scores, member, keep);
    }
    NRB_LAUNCH_CHECK();
    if (B == 1) {
        small_select_kernel<MASKED><<<nq, n <= 4096 ? 256 : 1024, 0, st>>>(w.scores, n, n, k, L2 ? 1 : 0, id_base, D, I);
        NRB_LAUNCH_CHECK();
    } else {
        small_select1_kernel<MASKED><<<dim3(B, nq), 1024, 0, st>>>(w.scores, n, n, k, L2 ? 1 : 0, w.cands);
        NRB_LAUNCH_CHECK();
        small_select2_kernel<MASKED><<<nq, B * k <= 2048 ? 256 : 1024, 0, st>>>(w.cands, B, k, L2 ? 1 : 0, id_base, D, I);
        NRB_LAUNCH_CHECK();
    }
    return NRB_OK;
}

static int search_small_impl(const float* xq, int64_t ldq, int32_t nq, int32_t d, const nrb_matrix* b, int32_t metric,
                             int32_t k, int64_t id_base, float* D, int64_t* I, void* workspace, size_t workspace_bytes,
                             const int64_t* member, int64_t keep, void* stream) {
    NRB_REQUIRE(b && b->raw && b->n > 0 && b->n < (1LL << 31), "search_small: the item matrix needs its raw plane (0 < n < 2^31)");
    NRB_REQUIRE(nq > 0 && nq <= NRB_SMALL_MAX_NQ && k > 0 && k <= SELECT_MAX_K && d == b->d && b->kp % 32 == 0 && b->kp <= 2048,
                "search_small: bad sizes (nq <= %d, k <= %d)", NRB_SMALL_MAX_NQ, SELECT_MAX_K);
    NRB_REQUIRE(xq && D && I && ldq >= d, "search_small: null argument");
    NRB_REQUIRE(workspace_bytes >= nrb_search_small_workspace(nq, b->n, k) && (workspace || b->n <= FUSED_MAX_ROWS),
                "search_small: workspace too small");
    if (!tc_available()) return NRB_ERR_NO_DEVICE;
    cudaStream_t st = (cudaStream_t)stream;
    if (member)
        return metric == NRB_METRIC_L2
                   ? small_flat_launch<true, true>(xq, ldq, nq, d, b, k, id_base, workspace, D, I, member, keep, st)
                   : small_flat_launch<false, true>(xq, ldq, nq, d, b, k, id_base, workspace, D, I, member, keep, st);
    return metric == NRB_METRIC_L2
               ? small_flat_launch<true, false>(xq, ldq, nq, d, b, k, id_base, workspace, D, I, nullptr, 0, st)
               : small_flat_launch<false, false>(xq, ldq, nq, d, b, k, id_base, workspace, D, I, nullptr, 0, st);
}

}  // namespace nrb

using namespace nrb;

extern "C" size_t nrb_search_small_workspace(int64_t nq, int64_t nb, int32_t k) {
    if (nb <= FUSED_MAX_ROWS) return 256;
    return carve_small(nullptr, nq, nb, select_slices(nb), k).total;
}

extern "C" int nrb_search_small(const float* xq, int64_t ldq, int32_t nq, int32_t d, const nrb_matrix* b, int32_t metric,
                                int32_t k, int64_t id_base, float* D, int64_t* I, void* workspace, size_t workspace_bytes,
                                void* stream) {
    return search_small_impl(xq, ldq, nq, d, b, metric, k, id_base, D, I, workspace, workspace_bytes, nullptr, 0, stream);
}

extern "C" int nrb_search_small_sel(const float* xq, int64_t ldq, int32_t nq, int32_t d, const nrb_matrix* b,
                                    int32_t metric, int32_t k, int64_t id_base, float* D, int64_t* I, void* workspace,
                                    size_t workspace_bytes, void* stream, const int64_t* member, int64_t keep) {
    NRB_REQUIRE(member, "search_small_sel: null member");
    return search_small_impl(xq, ldq, nq, d, b, metric, k, id_base, D, I, workspace, workspace_bytes, member, keep, stream);
}

// Host arrays in, host arrays out. The staging buffer is page-locked AND mapped into the device
// address space: the kernels read the query rows from it and write D / I into it directly
// (a few KB over PCIe inside the kernel), so a call is the kernel launch(es) and ONE stream
// synchronisation -- no copy calls at all. Staging and device scratch are cached per device
// (grow-only).
namespace {
struct SmallCache {
    void* pin = nullptr;
    void* pin_dev = nullptr;
    size_t pin_bytes = 0;
    void* dev = nullptr;
    size_t dev_bytes = 0;
};
SmallCache g_small[64];
std::mutex g_small_mu;
}  // namespace

static int search_small_host_impl(const nrb_matrix* b, const float* xq_host, int32_t nq, int32_t d, int32_t metric,
                                  int32_t k, int64_t id_base, float* D_host, int64_t* I_host, const int64_t* member,
                                  int64_t keep, void* stream) {
    NRB_REQUIRE(b && xq_host && D_host && I_host && nq > 0 && nq <= NRB_SMALL_MAX_NQ && k > 0 && k <= SELECT_MAX_K && d > 0,
                "search_small_host: bad arguments");
    int dev = 0;
    NRB_CUDA_CHECK(cudaGetDevice(&dev));
    NRB_REQUIRE(dev >= 0 && dev < 64, "search_small_host: device index out of range");
    std::lock_guard<std::mutex> lock(g_small_mu);
    SmallCache& c = g_small[dev];
    const size_t q_bytes = align_up((size_t)nq * d * sizeof(float), 256);
    const size_t i_bytes = align_up((size_t)nq * k * sizeof(int64_t), 256);
    const size_t d_bytes = align_up((size_t)nq * k * sizeof(float), 256);
    const size_t io = q_bytes + i_bytes + d_bytes;
    const size_t ws = nrb_search_small_workspace(nq, b->n, k);
    if (c.pin_bytes < io) {
        if (c.pin) cudaFreeHost(c.pin);
        c.pin = c.pin_dev = nullptr;
        c.pin_bytes = 0;
        NRB_CUDA_CHECK(cudaHostAlloc(&c.pin, io * 2, cudaHostAllocMapped));
        NRB_CUDA_CHECK(cudaHostGetDevicePointer(&c.pin_dev, c.pin, 0));
        c.pin_bytes = io * 2;
    }
    if (c.dev_bytes < ws) {
        if (c.dev) cudaFree(c.dev);
        c.dev = nullptr;
        c.dev_bytes = 0;
        NRB_CUDA_CHECK(cudaMalloc(&c.dev, ws * 2));
        c.dev_bytes = ws * 2;
    }
    cudaStream_t st = (cudaStream_t)stream;
    char* hp = (char*)c.pin;
    char* mp = (char*)c.pin_dev;
    memcpy(hp, xq_host, (size_t)nq * d * sizeof(float));
    const int rc = search_small_impl((const float*)mp, d, nq, d, b, metric, k, id_base, (float*)(mp + q_bytes + i_bytes),
                                     (int64_t*)(mp + q_bytes), c.dev, c.dev_bytes, member, keep, stream);
    if (rc != NRB_OK) return rc;
    NRB_CUDA_CHECK(cudaStreamSynchronize(st));
    memcpy(I_host, hp + q_bytes, (size_t)nq * k * sizeof(int64_t));
    memcpy(D_host, hp + q_bytes + i_bytes, (size_t)nq * k * sizeof(float));
    return NRB_OK;
}

extern "C" int nrb_search_small_host(const nrb_matrix* b, const float* xq_host, int32_t nq, int32_t d, int32_t metric,
                                     int32_t k, int64_t id_base, float* D_host, int64_t* I_host, void* stream) {
    return search_small_host_impl(b, xq_host, nq, d, metric, k, id_base, D_host, I_host, nullptr, 0, stream);
}

extern "C" int nrb_search_small_host_sel(const nrb_matrix* b, const float* xq_host, int32_t nq, int32_t d, int32_t metric,
                                         int32_t k, int64_t id_base, float* D_host, int64_t* I_host, void* stream,
                                         const int64_t* member, int64_t keep) {
    NRB_REQUIRE(member, "search_small_host_sel: null member");
    return search_small_host_impl(b, xq_host, nq, d, metric, k, id_base, D_host, I_host, member, keep, stream);
}

static int64_t ivf_small_ld(int32_t nprobe, int32_t max_list_len, int64_t ntotal) {
    int64_t ld = (int64_t)nprobe * max_list_len;
    return ld > ntotal ? ntotal : ld;
}

extern "C" size_t nrb_ivf_scan_small_workspace(int64_t nq, int32_t nprobe, int32_t max_list_len, int64_t ntotal, int32_t k) {
    const int64_t ld = ivf_small_ld(nprobe, max_list_len, ntotal);
    return carve_small(nullptr, nq, ld, select_slices(ld), k).total;
}

template <bool MASKED>
static int ivf_small_launch(const float* xq, int64_t ldq, int32_t nq, int32_t d, const nrb_matrix* lists,
                             const int32_t* offsets, int32_t max_list_len, const int64_t* ids, const int64_t* coarse,
                             int32_t nprobe, int l2, int32_t k, float* D, int64_t* I, const SmallWs& w, int64_t ld, int B,
                             const int64_t* member, int64_t keep, cudaStream_t st) {
    const dim3 grid((max_list_len + IVF_CHUNK - 1) / IVF_CHUNK, nq * nprobe);
    const size_t sh = lists->kp * sizeof(float);
    if (l2)
        ivf_small_scores_kernel<true, MASKED><<<grid, SMALL_THREADS, sh, st>>>(xq, ldq, d, lists->raw, lists->kp, offsets,
                                                                               coarse, nprobe, w.scores, ld, member, keep);
    else
        ivf_small_scores_kernel<false, MASKED><<<grid, SMALL_THREADS, sh, st>>>(xq, ldq, d, lists->raw, lists->kp, offsets,
                                                                                coarse, nprobe, w.scores, ld, member, keep);
    NRB_LAUNCH_CHECK();
    ivf_small_select1_kernel<MASKED><<<dim3(B, nq), 1024, 0, st>>>(w.scores, ld, offsets, coarse, nprobe, k, l2, w.cands);
    NRB_LAUNCH_CHECK();
    ivf_small_select2_kernel<MASKED><<<nq, B * k <= 2048 ? 256 : 1024, 0, st>>>(w.cands, B, offsets, coarse, nprobe, ids, k,
                                                                               l2, D, I);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

static int ivf_scan_small_impl(const float* xq, int64_t ldq, int32_t nq, int32_t d, const nrb_matrix* lists,
                               const int32_t* offsets, int32_t nlist, int32_t max_list_len, const int64_t* ids,
                               const int64_t* coarse, int32_t nprobe, int32_t metric, int32_t k, float* D, int64_t* I,
                               void* workspace, size_t workspace_bytes, const int64_t* member, int64_t keep,
                               void* stream) {
    NRB_REQUIRE(lists && lists->raw && lists->n > 0 && lists->n < (1LL << 31) && d == lists->d && lists->kp % 32 == 0 &&
                    lists->kp <= 2048, "ivf_scan_small: the list matrix needs its raw plane");
    NRB_REQUIRE(nq > 0 && nprobe > 0 && nprobe <= SELECT_MAX_K && nprobe <= nlist && k > 0 && k <= SELECT_MAX_K &&
                    max_list_len > 0, "ivf_scan_small: bad sizes");
    NRB_REQUIRE(xq && offsets && ids && coarse && D && I && workspace, "ivf_scan_small: null argument");
    NRB_REQUIRE(workspace_bytes >= nrb_ivf_scan_small_workspace(nq, nprobe, max_list_len, lists->n, k),
                "ivf_scan_small: workspace too small");
    NRB_REQUIRE((int64_t)nq * nprobe <= 65535, "ivf_scan_small: nq * nprobe > 65535 (use nrb_ivf_search)");
    if (!tc_available()) return NRB_ERR_NO_DEVICE;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t ld = ivf_small_ld(nprobe, max_list_len, lists->n);
    const int B = select_slices(ld);
    const SmallWs w = carve_small(workspace, nq, ld, B, k);
    const int l2 = metric == NRB_METRIC_L2 ? 1 : 0;
    if (member)
        return ivf_small_launch<true>(xq, ldq, nq, d, lists, offsets, max_list_len, ids, coarse, nprobe, l2, k, D, I, w, ld,
                                      B, member, keep, st);
    return ivf_small_launch<false>(xq, ldq, nq, d, lists, offsets, max_list_len, ids, coarse, nprobe, l2, k, D, I, w, ld, B,
                                   nullptr, 0, st);
}

extern "C" int nrb_ivf_scan_small(const float* xq, int64_t ldq, int32_t nq, int32_t d, const nrb_matrix* lists,
                                  const int32_t* offsets, int32_t nlist, int32_t max_list_len, const int64_t* ids,
                                  const int64_t* coarse, int32_t nprobe, int32_t metric, int32_t k, float* D, int64_t* I,
                                  void* workspace, size_t workspace_bytes, void* stream) {
    return ivf_scan_small_impl(xq, ldq, nq, d, lists, offsets, nlist, max_list_len, ids, coarse, nprobe, metric, k, D, I,
                               workspace, workspace_bytes, nullptr, 0, stream);
}

extern "C" int nrb_ivf_scan_small_sel(const float* xq, int64_t ldq, int32_t nq, int32_t d, const nrb_matrix* lists,
                                      const int32_t* offsets, int32_t nlist, int32_t max_list_len, const int64_t* ids,
                                      const int64_t* coarse, int32_t nprobe, int32_t metric, int32_t k, float* D, int64_t* I,
                                      void* workspace, size_t workspace_bytes, void* stream, const int64_t* member,
                                      int64_t keep) {
    NRB_REQUIRE(member, "ivf_scan_small_sel: null member");
    return ivf_scan_small_impl(xq, ldq, nq, d, lists, offsets, nlist, max_list_len, ids, coarse, nprobe, metric, k, D, I,
                               workspace, workspace_bytes, member, keep, stream);
}
