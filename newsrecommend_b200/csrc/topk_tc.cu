// K2: fused distance + selection on the 5th-generation tensor cores (NRB_PATH_TC, NRB_PATH_TC1,
// NRB_PATH_TC16).
//
// Stands in for faiss's exhaustive_inner_product_blas / exhaustive_L2sqr_blas (sgemm blocks +
// HeapBlockResultHandler) behind IndexFlat::search, i.e. Retrieval.py:21,32 and the assignment
// search inside Clustering::train (Retrieval.py:18), and for IVFFlatScanner over list units.
//
// Persistent CTAs (384 threads = three hardware warpgroups) walk a list of Units (128 query rows
// x a run of item rows). Per 128 x 256 score tile:
//   warp 0            TMA producer: operand tiles in K chunks of 128 bytes (128-byte swizzle),
//                     mbarrier ring
//   warp 1            MMA issuer: tcgen05.mma into one of two fp32 TMEM accumulators (2 x 256
//                     columns), so the MMAs of tile t+1 overlap the selection of tile t
//   warps 2-3         idle (they complete the control warpgroup, which gives its registers to
//                     the selection warpgroups with setmaxnreg)
//   warps 4-7, 8-11   two selection warpgroups; warpgroup g owns columns [128g, 128g+128) of EVERY
//                     tile: tcgen05.ld 32 rows x 128 scores into registers (one query row per
//                     thread), hand the accumulator back, then skip / append: group maxima decide
//                     per 32-column chunk whether anything beats the row's running threshold, and
//                     only then are keys appended to the row's candidate buffer. Thresholds are
//                     tightened by scheduled prunes (bisection + compaction on the union of the
//                     two warpgroups' buffers); an exact bitonic sort per row ends the unit.
// The score matrix never exists in HBM.
//
// Kernels (shared epilogue, epilogue_run):
//   topk_tc3_kernel<fp16|tf32>  filter: ONE pass over reduced-precision operand planes (scaled fp16,
//                 or the tf32 hi planes), query tile resident in shared memory, CTA pairs
//                 (cta_group::2, M = 256); keeps the best k plus everything inside a proven
//                 error margin, exact fp32 refine follows (select_refine_kernel). Default.
//   topk_tc3s_kernel            its single-CTA form (cta_group::1, M = 128) for single partial waves.
//   topk_tc2_kernel             3xTF32: per K step lo*hi, hi*lo, hi*hi into one accumulator, CTA
//                 pairs; each CTA stages its own 128 query rows and HALF of the 256-row item
//                 tile, so the item stream is read from L2 once per 256 queries. 3 x 64 KB stages.
//                 The exact path (NRB_PATH_TC) and the recompute of queries the filter flags.
#include <cuda.h>

#include <cstdlib>

#include "common.cuh"
#include "internal.h"
#include "ptx.cuh"

namespace nrb {

namespace {

constexpr int BM = 128;   // query rows per CTA tile (= TMEM lanes)
constexpr int BN = 256;   // item rows per tile (= TMEM columns per accumulator)
constexpr int KC = 32;    // fp32 elements per K chunk (128-byte swizzle span)
constexpr int A_BYTES = BM * KC * 4;        // 16 KB: 128 rows x 128 B
constexpr int BH_BYTES = (BN / 2) * KC * 4; // 16 KB: half item tile (CTA pairs)
constexpr int B_BYTES = BN * KC * 4;        // 32 KB: full item tile (single CTA)
// Warps 0-3: control warpgroup (warp 0 TMA producer, warp 1 MMA issuer, warps 2-3 idle); warps
// 4-7 and 8-11: the two selection warpgroups. Roles are aligned to hardware warpgroups so that
// setmaxnreg can move registers from the control warps to the selection warps.
constexpr int NUM_THREADS = 384;
constexpr int EPI_WARP0 = 4;
constexpr int EPI_WGS = 2;
constexpr int HALF_N = BN / EPI_WGS;  // columns of every tile handled by one warpgroup
constexpr int TMEM_COLS = 512;

constexpr int V2_STAGES = 3;
constexpr int V2_STAGE_BYTES = 2 * A_BYTES + 2 * BH_BYTES;  // 64 KB

// Exchange area of the scheduled (pairwise) prune: the two selection warps that own the same 32
// query rows -- one per warpgroup, i.e. per column half -- publish their rows' state here, split
// the rows between them, and read the new state back.
struct XchgShared {
    int cnt[EPI_WGS][BM];    // in: the row's buffered entries per warpgroup; out: entries kept
    int fresh[EPI_WGS][BM];  // in: entries appended since the row's last prune
    int done[BM];            // out: 1 if the row was pruned (0: too few new entries, left as it is)
    float thr[EPI_WGS][BM];  // in: each warpgroup's append threshold for the row
    float margin[BM];        // in: the row's error margin (filter kernels; else 0)
    float nthr[BM];          // out: new append threshold (both warpgroups)
    uint32_t lb[BM];         // out: ordered-uint lower bound of the row's k-th key (0: none yet)
    int ovf[BM];             // out: 1 if entries inside the row's margin had to be dropped (the query must be recomputed)
};

template <int STAGES>
struct TcShared {
    uint64_t full[STAGES];
    uint64_t empty[STAGES];
    uint64_t tfull[2];
    uint64_t tempty[2];
    uint32_t tmem_base;
    uint32_t pad;
    float nrm[EPI_WGS][2][HALF_N];  // [warpgroup][tile parity]: staged item norms (L2)
    XchgShared xchg;
};

constexpr size_t V2_SMEM = (size_t)V2_STAGES * V2_STAGE_BYTES + sizeof(TcShared<V2_STAGES>) + 1024;

// ---------------------------------------------------------------------------- timeline trace
// Build with -DNRB_TRACE (make trace -> libnrb200_trace.so): cluster 0's leader CTA records
// clock64() at the hand-off points of its first NRB_TRACE_TILES tiles; scripts/trace_timeline.py
// reads it back with nrb_debug_trace_read and prints where each tile's time goes.
#ifdef NRB_TRACE
constexpr int NRB_TRACE_TILES = 4096;
// [who][tile][event]: who 0 = MMA warp (0 tempty seen, 1 MMAs issued + committed),
// who 1..8 = selection warps 4..11 (0 wait start, 1 tfull seen, 2 released, 3 tile done)
__device__ long long g_trace[9][NRB_TRACE_TILES][4];
// scheduled prunes of the same warps: [who][prune #][0 publish, 1 partner arrived, 2 rows done, 3 partner done]
__device__ long long g_trace_prune[9][64][4];
__device__ int g_trace_prune_n[9];
// 1: the launch records (set per launch by the host side: NRB_TRACE_IVF_MODE=1 / 2 keeps only the
// phase A / phase B launches of an IVF scan, so that the LAST launch does not overwrite the others)
__device__ int g_trace_enable = 1;
#define NRB_TRP(who, ev)                                                                                   \
    do {                                                                                                   \
        if (blockIdx.x == 0 && (threadIdx.x & 31) == 0 && g_trace_enable && g_trace_prune_n[who] < 64)      \
            g_trace_prune[who][g_trace_prune_n[who]][ev] = clock64();                                      \
    } while (0)
#define NRB_TRP_NEXT(who)                                                                           \
    do {                                                                                            \
        if (blockIdx.x == 0 && (threadIdx.x & 31) == 0 && g_trace_enable) g_trace_prune_n[who]++; \
    } while (0)
#define NRB_TR(who, tile, ev)                                                                                      \
    do {                                                                                                           \
        if (blockIdx.x == 0 && (threadIdx.x & 31) == 0 && g_trace_enable && (tile) < (uint32_t)NRB_TRACE_TILES)      \
            g_trace[who][tile][ev] = clock64();                                                                    \
    } while (0)
#else
#define NRB_TR(who, tile, ev) \
    do {                      \
    } while (0)
#define NRB_TRP(who, ev) \
    do {                 \
    } while (0)
#define NRB_TRP_NEXT(who) \
    do {                  \
    } while (0)
#endif

// ---------------------------------------------------------------------------- epilogue
struct EpiRow {
    int cnt;
    int base;      // entries kept by the row's last prune (nothing was appended while cnt == base)
    float thr;     // append threshold: kth - margin (NEG_INF until k candidates exist)
    float cthr;    // thr in the domain the pass mask compares in (IP: thr * sc; L2: thr + |q|^2, against 2 q.x - |x|^2)
    float sc;      // accumulator = sc * (q . x): product of the operands' power-of-two fp16 scales, else 1
    float inv;     // 1 / sc (exact)
    float qn;      // squared query norm (L2 keys, margins)
    float margin;  // 0 for the 3xTF32 kernels; error margin of the 1xTF32 filter
    int flag;      // set when more than keep_max candidates fell inside the margin
    unsigned* gslot;  // the query's shared running lower bound of its k-th key (ordered uint), or null
};

struct PruneOut {
    float thr, kth;
    int kept, ovf;
};

// One row's prune behind a real call: the kernel has three call sites (in-tile overflow guard,
// scheduled prune, unit end) and two sort widths; inlining all of them multiplies the unrolled
// bitonic networks and the kernel no longer fits the instruction cache.
// Input: the row's AoS candidate buffer. Output: back into that buffer (ob == b: in place) or into a
// partial row (ok, oi) when ob is null.
__device__ __noinline__ PruneOut prune_row_call(const uint2* b, int n, int k, float margin, int keep_max, int width,
                                                uint2* ob, float* ok, int* oi, float floor_thr) {
    const int lane = threadIdx.x & 31;
    const AoSView in{const_cast<uint2*>(b)};
    const EitherView out{ob, ok, oi};
    PruneOut o;
    bool ovf;
    // the sort is sized by the entries present: a row whose threshold was hot from the start (later
    // lists of an IVF query, later chunks of a split catalog) ends its unit with a handful
    if (n == 0) {  // nothing buffered (dead row, or nothing beat an already hot threshold): padding only
        for (int e = lane; e < width; e += 32) out.store(e, NEG_INF, -1);
        __syncwarp();
        o.thr = floor_thr;
        o.kth = NEG_INF;
        o.kept = 0;
        o.ovf = 0;
        return o;
    }
    const bool inplace = ob != nullptr;  // in-place prunes must also cover the whole output width
    if (n <= 32 && !inplace)
        o.thr = warp_prune_row_v<1>(in, n, k, margin, keep_max, width, out, lane, &o.kept, &ovf, floor_thr, &o.kth);
    else if (n <= 64 && !inplace)
        o.thr = warp_prune_row_v<2>(in, n, k, margin, keep_max, width, out, lane, &o.kept, &ovf, floor_thr, &o.kth);
    else if (n <= 128 && width <= 128)
        o.thr = warp_prune_row_v<4>(in, n, k, margin, keep_max, width, out, lane, &o.kept, &ovf, floor_thr, &o.kth);
    else
        o.thr = warp_prune_row_v<CAND_CAP / 32>(in, n, k, margin, keep_max, width, out, lane, &o.kept, &ovf, floor_thr,
                                                &o.kth);
    o.ovf = ovf ? 1 : 0;
    return o;
}

// Mid-unit prune of one row, in place: the bisection/compaction fast path, and the exact sort only
// when that leaves too many entries (heavy ties, or a margin set that does not fit).
constexpr int TIGHTEN_MAX_KEEP = 160;
__device__ __noinline__ PruneOut tighten_row_call(uint2* b, int n, int k, float margin, int keep_max, float floor_thr) {
    const int lane = threadIdx.x & 31;
    PruneOut o;
    uint32_t lb;
    if (n <= 128)
        o.thr = warp_tighten_row<4>(AoSView{b}, n, k, margin, floor_thr, lane, &o.kept, &lb);
    else
        o.thr = warp_tighten_row<CAND_CAP / 32>(AoSView{b}, n, k, margin, floor_thr, lane, &o.kept, &lb);
    o.kth = from_ordered_u32(lb);
    o.ovf = 0;
    if (o.kept > TIGHTEN_MAX_KEEP) o = prune_row_call(b, o.kept, k, margin, keep_max, keep_max, b, nullptr, nullptr, o.thr);
    return o;
}

// A row whose margin set did not fit its slots is incomplete whatever happens next: its query is
// flagged and recomputed by the exact path. Stop collecting for it -- on a near-duplicate-heavy
// catalog such rows otherwise refill their buffers within a few tiles and run the exact-sort prune
// over and over (measured: 13-30x slower searches at 16-64 copies per article).
__device__ __forceinline__ void epi_abandon_row(EpiRow& st) {
    st.flag = 1;
    st.cnt = 0;
    st.base = 0;
    st.thr = __builtin_huge_valf();
    st.cthr = st.thr;
}

// Prunes the rows of the warp named by `need` (one bit per lane = row) back to (about) their best
// k (+ margin set), in place, and raises their thresholds.
template <bool L2>
__device__ __forceinline__ void epi_prune_rows(unsigned need, EpiRow& st, uint2* cb, int k, int keep_max, int lane) {
    while (need) {
        const int src = __ffs(need) - 1;
        need &= need - 1;
        const int n = __shfl_sync(0xffffffffu, st.cnt, src);
        const float mg = __shfl_sync(0xffffffffu, st.margin, src);
        const float fl = __shfl_sync(0xffffffffu, st.thr, src);  // entries were appended above it
        const PruneOut o = tighten_row_call(cb + (int64_t)src * CAND_CAP, n, k, mg, keep_max, fl);
        if (lane == src) {
            st.cnt = o.kept;
            st.base = o.kept;
            st.thr = o.thr;
            st.cthr = L2 ? o.thr + st.qn : o.thr * st.sc;
            st.flag |= o.ovf;
            if (st.gslot && o.kth > NEG_INF) atomicMax(st.gslot, ordered_u32(o.kth));
            if (o.ovf) epi_abandon_row(st);
        }
    }
}

// 32 accumulator columns of the warp's 32 rows (thread = row): `v` holds the raw TMEM words of
// columns [c0, c0 + 32) of this warpgroup's half. Keys above the row's threshold are appended to
// the row's candidate buffer.
//   * The common case is "nothing passes": instead of 32 compares, four 3-input max trees give
//     the maxima of the four 8-column groups (16 FMNMX3/FMNMX), one more the chunk maximum, and a
//     single compare + vote lets the warp skip the chunk.
//   * Otherwise only the groups in which some lane has a hit are expanded, with STATIC register
//     indices (predicated stores): a run-time index into the 32 keys would put them in local
//     memory, and with 227 KB of the SM's 256 KB configured as shared memory nearly every local
//     access is an L2 round trip on the epilogue's critical path.
template <bool L2, bool FULL>
__device__ __forceinline__ void epi_chunk(const uint32_t (&v)[32], int c0, int valid, int id0, const float* nrm,
                                          float m2inv, EpiRow& st, uint2* cb, uint2* myb, int k, int keep_max,
                                          int lane) {
    float f[32];
#pragma unroll
    for (int i = 0; i < 32; i++) {
        float x = __uint_as_float(v[i]);  // IP: stays in the accumulator's (scaled) domain
        // L2: ONE fma per element -- t = 2 q.x - |x|^2 (nrm holds -|x|^2); the row constant |q|^2 lives in
        // the threshold (cthr = thr + |q|^2) and the clamp at distance 0 is applied to appended keys only
        if (L2) x = fmaf(x, m2inv, nrm[c0 + i]);
        if (!FULL && c0 + i >= valid) x = NEG_INF;
        f[i] = x;
    }
    constexpr int GW = 8;  // columns per hit group (4 was measured slower: see DESIGN)
    constexpr int NG = 32 / GW;
    float g[NG];
#pragma unroll
    for (int j = 0; j < NG; j++) {
        const float* e = f + GW * j;
        g[j] = fmaxf(fmaxf(fmaxf(fmaxf(e[0], e[1]), e[2]), fmaxf(fmaxf(e[3], e[4]), e[5])), fmaxf(e[6], e[7]));
    }
    float cmax = g[0];
#pragma unroll
    for (int j = 1; j < NG; j++) cmax = fmaxf(cmax, g[j]);
    if (!__any_sync(0xffffffffu, cmax > st.cthr)) return;
    const float ksc = L2 ? 1.f : st.inv;  // stored keys are always unscaled
#pragma unroll
    for (int j = 0; j < NG; j++) {
        if (!__any_sync(0xffffffffu, g[j] > st.cthr)) continue;  // warp-uniform
        if (g[j] > st.cthr) {
#pragma unroll
            for (int i = 0; i < GW; i++) {
                if (f[GW * j + i] > st.cthr) {  // one 64-bit store per appended entry
                    const float key = L2 ? fminf(f[GW * j + i] - st.qn, 0.f) : f[GW * j + i] * ksc;
                    myb[st.cnt] = make_uint2(__float_as_uint(key), (uint32_t)(id0 + c0 + GW * j + i));
                    st.cnt++;
                }
            }
        }
    }
    // overflow guard (rare once the prune schedule is running): a chunk adds at most 32 entries
    const unsigned need = __ballot_sync(0xffffffffu, st.cnt > CAND_CAP - 32);
    if (need) epi_prune_rows<L2>(need, st, cb, k, keep_max, lane);
}

// The ragged last tile of a unit (fewer than 128 valid columns in this warpgroup's half), chunk
// by chunk.
//   taddr0  TMEM address of (this warp's lane quarter, first column of the warpgroup's half)
//   valid   number of valid item columns in this half
//   id0     item row index of column 0 of the half
//   nrm     item norms of the half in shared memory (L2 only)
//   cb      candidate buffers of this warp's 32 rows ((key, idx) entries); myb = this lane's row
template <bool L2>
__device__ __forceinline__ void epi_tile_ragged(uint32_t taddr0, int valid, int id0, const float* nrm, EpiRow& st,
                                                uint2* cb, uint2* myb, int k, int keep_max, int lane) {
    const float m2inv = 2.f * st.inv;  // epi_chunk: t = acc * (2 / scale) - |x|^2
#pragma unroll 1
    for (int c0 = 0; c0 < HALF_N; c0 += 32) {
        if (c0 >= valid) break;  // warp-uniform
        uint32_t v[32];
        ptx::tmem_ld_32x32b_x32(taddr0 + c0, v);
        ptx::tmem_ld_wait();
        epi_chunk<L2, false>(v, c0, valid, id0, nrm, m2inv, st, cb, myb, k, keep_max, lane);
    }
}

// Unit finished: the warp's 32 rows, best-first, into the unit's partial rows (`pw` entries
// per row: the best k plus, for the margin filter, everything within the margin of the k-th).
__device__ __forceinline__ void epi_unit_end(EpiRow& st, uint2* cb, int64_t prow0, int k, int pw, float* part_key,
                                             int* part_idx, int lane) {
    for (int src = 0; src < 32; src++) {
        const int n = __shfl_sync(0xffffffffu, st.cnt, src);
        const float mg = __shfl_sync(0xffffffffu, st.margin, src);
        const float fl = __shfl_sync(0xffffffffu, st.thr, src);
        const int64_t o = (prow0 + src) * pw;
        const PruneOut r = prune_row_call(cb + (int64_t)src * CAND_CAP, n, k, mg, pw, pw, nullptr, part_key + o, part_idx + o,
                                          fl < __builtin_huge_valf() ? fl : NEG_INF);
        if (lane == src) {
            st.flag |= r.ovf;
            if (st.gslot && r.kth > NEG_INF) atomicMax(st.gslot, ordered_u32(r.kth));
        }
    }
}

// Unit finished, filter kernels: the warp's 32 rows go to the unit's partial rows UNSORTED (`pw`
// slots per row, part_cnt[row] of them used). The refine stage gathers every partial row of a
// query, finds the k-th best estimate by bisection and rescoring the survivors exactly sorts them,
// so the per-(unit, row) sort of the plain top-k kernels would be wasted work here -- for the short
// units of an IVF scan it cost more than the unit's MMAs. The caller has already brought every
// row down to at most pw entries (final union prune) or flagged it.
__device__ __forceinline__ void epi_unit_end_unsorted(int n, const uint2* cb, int64_t prow0, int pw, float* part_key,
                                                      int* part_idx, int* part_cnt, int lane) {
    part_cnt[prow0 + lane] = n;
    // rows with more than a few entries: warp-cooperative, coalesced copies
    unsigned big = __ballot_sync(0xffffffffu, n > 4);
    while (big) {
        const int src = __ffs(big) - 1;
        big &= big - 1;
        const int nn = __shfl_sync(0xffffffffu, n, src);
        const uint2* rb = cb + (int64_t)src * CAND_CAP;
        const int64_t o = (prow0 + src) * pw;
        for (int e = lane; e < nn; e += 32) {
            const uint2 v = rb[e];
            part_key[o + e] = __uint_as_float(v.x);
            part_idx[o + e] = (int)v.y;
        }
    }
    if (n <= 4) {  // the common case of a hot row: a handful of entries, copied by the row's own lane
        const uint2* rb = cb + (int64_t)lane * CAND_CAP;
        const int64_t o = (prow0 + lane) * pw;
        for (int e = 0; e < n; e++) {
            const uint2 v = rb[e];
            part_key[o + e] = __uint_as_float(v.x);
            part_idx[o + e] = (int)v.y;
        }
    }
}

// Scheduled prune of 16 query rows by one warp, on the UNION of the two warpgroups' buffers of
// each row (xs->cnt / thr / margin were published by both warps of the lane quarter):
//   * a lower bound lb of the k-th best key of the union is found by bisection on the ordered-uint
//     keys (count(key >= lb) in [k, k + 3], or exact after 32 halvings);
//   * both buffers are compacted in place to their entries >= T = max(lb - margin, old thresholds)
//     (everything dropped is below a valid bound of the row's k-th minus the margin);
//   * T, lb and the new counts go back through xs.
// Thresholds therefore follow the k-th best of ALL the row's columns although each warpgroup
// keeps its own buffer, and the append rate per row is that of a single running top-k.
// Two rows are processed together so that their loads and reduction chains overlap. Buffers
// with more than 128 entries (possible only after heavy ties) are first brought down by the
// single-buffer prune.
constexpr int UT_SLACK = 3;
constexpr int UT_ROWS = 2;  // rows of a scheduled prune in flight together (4 was measured: flat +0 %, IVF -17 %)
// min_new > 0 (units that share running bounds with other units of the same query: IVF lists):
// a row pair is pruned only once min_new new candidates have arrived in one of its rows -- rows
// whose threshold was already hot when the unit started are left alone and the scheduled prune
// costs them nothing but the barrier (IVF scan -5 %; the flat search prunes every row anyway).
// min_new < 0 (unit end, unsorted partial output): a row pair is pruned only if one of its rows can
// still yield something -- a buffer that does not fit the partial row (more than keep_max entries),
// or at least k candidates in the union with some of them new since the row's last prune (a
// tighter bound of the k-th for the query's other units, and fewer candidates for the refine).
__device__ __noinline__ void union_tighten_rows(XchgShared* xs, uint2* cb_cta, int quad, int half, int k, int keep_max,
                                                int min_new) {
    constexpr int NB = UT_ROWS;  // rows in flight: their loads and reduction chains overlap
    const int lane = threadIdx.x & 31;
    const uint32_t lt = (1u << lane) - 1u;
#pragma unroll 1
    for (int it = 0; it < 16 / NB; it++) {
        int row[NB], nA[NB], nB[NB];
        uint2 *bA[NB], *bB[NB];  // the row's buffer in warpgroup 0 / warpgroup 1
        float floor_t[NB], mg[NB];
        int ov[NB];
        if (min_new != 0) {
            const int r0 = quad * 32 + half * 16 + NB * it;
            bool quiet = true;
#pragma unroll
            for (int b = 0; b < NB; b++) {
                const int c0 = xs->cnt[0][r0 + b], c1 = xs->cnt[1][r0 + b];
                const int fr = xs->fresh[0][r0 + b] + xs->fresh[1][r0 + b];
                if (min_new > 0)
                    quiet = quiet && (fr < min_new);
                else
                    quiet = quiet && !(c0 > keep_max || c1 > keep_max || (c0 + c1 >= k && fr > 0));
            }
            if (quiet) {
                if (lane < NB) {
                    xs->done[r0 + lane] = 0;
                    xs->ovf[r0 + lane] = 0;
                }
                continue;  // warp-uniform
            }
        }
#pragma unroll
        for (int b = 0; b < NB; b++) {
            row[b] = quad * 32 + half * 16 + NB * it + b;
            bA[b] = cb_cta + (int64_t)row[b] * CAND_CAP;
            bB[b] = bA[b] + (int64_t)BM * CAND_CAP;
            nA[b] = xs->cnt[0][row[b]];
            nB[b] = xs->cnt[1][row[b]];
            mg[b] = xs->margin[row[b]];
            floor_t[b] = fmaxf(xs->thr[0][row[b]], xs->thr[1][row[b]]);
            ov[b] = 0;
            // rare: a buffer beyond the 128-entry fast path is first pruned on its own. If that has to
            // drop entries INSIDE the margin (more than keep_max of them: a near-duplicate-heavy catalog),
            // the row is reported as overflowed: its query is recomputed by the exact path.
            if (nA[b] > 128) {
                const PruneOut o = tighten_row_call(bA[b], nA[b], k, mg[b], keep_max, floor_t[b]);
                nA[b] = o.kept;
                ov[b] |= o.ovf;
                floor_t[b] = fmaxf(floor_t[b], o.thr);
                if (nA[b] > 128) {  // still too large (ties): exact prune to the best keep_max
                    const PruneOut e = prune_row_call(bA[b], nA[b], k, mg[b], keep_max, keep_max, bA[b], nullptr, nullptr, floor_t[b]);
                    nA[b] = e.kept;
                    ov[b] |= e.ovf;
                    floor_t[b] = fmaxf(floor_t[b], e.thr);
                }
            }
            if (nB[b] > 128) {
                const PruneOut o = tighten_row_call(bB[b], nB[b], k, mg[b], keep_max, floor_t[b]);
                nB[b] = o.kept;
                ov[b] |= o.ovf;
                floor_t[b] = fmaxf(floor_t[b], o.thr);
                if (nB[b] > 128) {
                    const PruneOut e = prune_row_call(bB[b], nB[b], k, mg[b], keep_max, keep_max, bB[b], nullptr, nullptr, floor_t[b]);
                    nB[b] = e.kept;
                    ov[b] |= e.ovf;
                    floor_t[b] = fmaxf(floor_t[b], e.thr);
                }
            }
        }
        // All 32 loads are UNCONDITIONAL (entries beyond a buffer's count are inside its 256-entry
        // allocation and are masked afterwards): predicated loads were issued a few at a time, each
        // batch waiting for the previous one -- eight L2 round trips per row pair instead of one.
        float rk[NB][8];
        int id[NB][8];
#pragma unroll
        for (int b = 0; b < NB; b++) {
#pragma unroll
            for (int i = 0; i < 4; i++) {  // one 64-bit load per entry
                const int e = i * 32 + lane;
                const uint2 va = bA[b][e], vb = bB[b][e];
                rk[b][i] = __uint_as_float(va.x);
                id[b][i] = (int)va.y;
                rk[b][4 + i] = __uint_as_float(vb.x);
                id[b][4 + i] = (int)vb.y;
            }
        }
        uint32_t u[NB][8];
#pragma unroll
        for (int b = 0; b < NB; b++) {
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int e = i * 32 + lane;
                u[b][i] = e < nA[b] ? ordered_u32(rk[b][i]) : 0u;
                u[b][4 + i] = e < nB[b] ? ordered_u32(rk[b][4 + i]) : 0u;
            }
        }
        __syncwarp();
        uint32_t lo[NB], hi[NB];
        bool run[NB];
#pragma unroll
        for (int b = 0; b < NB; b++) {
            uint32_t mn = 0xffffffffu, mx = 0u;
#pragma unroll
            for (int i = 0; i < 8; i++) {
                mn = (u[b][i] != 0u && u[b][i] < mn) ? u[b][i] : mn;
                mx = u[b][i] > mx ? u[b][i] : mx;
            }
            mn = __reduce_min_sync(0xffffffffu, mn);
            mx = __reduce_max_sync(0xffffffffu, mx);
            run[b] = nA[b] + nB[b] >= k;
            lo[b] = run[b] ? mn : 0u;  // invariant while running: count(u >= lo) >= k > count(u >= hi)
            hi[b] = mx + 1u;
            run[b] = run[b] && (hi[b] - lo[b] > 1u);
        }
        bool any_run = false;
#pragma unroll
        for (int b = 0; b < NB; b++) any_run = any_run || run[b];
        while (any_run) {  // warp-uniform
            uint32_t mid[NB];
            int c[NB];
#pragma unroll
            for (int b = 0; b < NB; b++) {
                mid[b] = lo[b] + ((hi[b] - lo[b]) >> 1);
                int cc = 0;
#pragma unroll
                for (int i = 0; i < 8; i++) cc += (u[b][i] >= mid[b]) ? 1 : 0;
                c[b] = cc;
            }
#pragma unroll
            for (int b = 0; b < NB; b++) c[b] = __reduce_add_sync(0xffffffffu, c[b]);
            any_run = false;
#pragma unroll
            for (int b = 0; b < NB; b++) {
                if (run[b]) {
                    if (c[b] >= k) {
                        lo[b] = mid[b];
                        if (c[b] <= k + UT_SLACK) run[b] = false;
                    } else {
                        hi[b] = mid[b];
                    }
                    if (hi[b] - lo[b] <= 1u) run[b] = false;
                }
                any_run = any_run || run[b];
            }
        }
#pragma unroll
        for (int b = 0; b < NB; b++) {
            const float thr = fmaxf(from_ordered_u32(lo[b]) - mg[b], floor_t[b]);  // lo == 0 -> NEG_INF
            int baseA = 0, baseB = 0;
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const float ka = from_ordered_u32(u[b][i]), kb = from_ordered_u32(u[b][4 + i]);
                const bool keepa = (u[b][i] != 0u) && ka >= thr;
                const bool keepb = (u[b][4 + i] != 0u) && kb >= thr;
                const uint32_t ma = __ballot_sync(0xffffffffu, keepa), mb = __ballot_sync(0xffffffffu, keepb);
                if (keepa) bA[b][baseA + __popc(ma & lt)] = make_uint2(__float_as_uint(ka), (uint32_t)id[b][i]);
                if (keepb) bB[b][baseB + __popc(mb & lt)] = make_uint2(__float_as_uint(kb), (uint32_t)id[b][4 + i]);
                baseA += __popc(ma);
                baseB += __popc(mb);
            }
            if (lane == 0) {
                xs->cnt[0][row[b]] = baseA;
                xs->cnt[1][row[b]] = baseB;
                xs->nthr[row[b]] = thr;
                xs->lb[row[b]] = lo[b];
                xs->done[row[b]] = 1;
                xs->ovf[row[b]] = ov[b];
            }
        }
        __syncwarp();
    }
}

// One-tile units from a cold start: the coarse-quantizer search and the nearest-centroid assignment
// (every query x at most 256 centroids), and the short lists of an IVF scan. The generic path would
// append the whole tile to the candidate buffers (every key beats a threshold of -inf) and then prune
// 250 entries per row -- ~200k cycles for 16 MMAs. Here the warp keeps its 32 rows x 128 columns in
// registers, and every THREAD bisects on its own row: 16 halvings of [row min, row max], the count of
// keys >= mid summed with the partner warp's (the other 128 columns of the same rows) through shared
// memory, one 64-thread named barrier per round. lo ends as a lower bound of the row's k-th best key
// with count(>= lo) >= k; keys >= lo - margin are appended (the margin set the refine stage needs).
// Returns with st.cnt entries in the row's buffer; *lb_out = lo (unscaled key domain), NEG_INF if the
// row has fewer than k columns.
struct OneShotOut {
    int cnt;
    float lb;
};
// Behind a real call: the routine wants ~150 registers for the row's 128 keys; inlined into the
// epilogue (which ptxas allocates at the kernel's 168-register bound) the keys spilled to local
// memory. As a call, the caller's live state is saved once around it instead.
template <bool L2, bool PAIR>
__device__ __noinline__ OneShotOut single_tile_call(uint32_t taddr0, int valid, int id0, const float* nrm, float sc,
                                                    float inv, float qn, float margin, uint2* myb, int k,
                                                    XchgShared* xs, int wg, int row, int quad, uint32_t tempty_remote,
                                                    uint64_t* tempty_local) {
    const int lane = threadIdx.x & 31;
    float f[HALF_N];
    {
        uint32_t v[4][32];
        ptx::tmem_ld_32x32b_x32(taddr0, v[0]);
        ptx::tmem_ld_32x32b_x32(taddr0 + 32, v[1]);
        ptx::tmem_ld_32x32b_x32(taddr0 + 64, v[2]);
        ptx::tmem_ld_32x32b_x32(taddr0 + 96, v[3]);
        ptx::tmem_ld_wait();
        // hand the accumulator back to the MMA warp
        ptx::tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) {
            if (PAIR)
                ptx::mbar_arrive_cluster_relaxed(tempty_remote);
            else
                ptx::mbar_arrive(tempty_local);
        }
#pragma unroll
        for (int c = 0; c < 4; c++)
#pragma unroll
            for (int i = 0; i < 32; i++) f[c * 32 + i] = __uint_as_float(v[c][i]);  // IP: the accumulator's (scaled) domain
    }
    const float m2inv = -2.f * inv;
    float mn = __builtin_huge_valf(), mx = NEG_INF;
#pragma unroll
    for (int i = 0; i < HALF_N; i++) {
        float x = f[i];
        if (L2) x = -fmaxf(fmaf(x, m2inv, qn - nrm[i]), 0.f);  // nrm holds -|x|^2
        const bool ok = i < valid;
        f[i] = ok ? x : NEG_INF;
        mn = ok ? fminf(mn, x) : mn;
        mx = ok ? fmaxf(mx, x) : mx;
    }
    const int nv = valid < 0 ? 0 : (valid > HALF_N ? HALF_N : valid);
    // exchange (min, max, valid columns) with the partner warp: the same rows, the other column half
    xs->thr[wg][row] = mn;
    xs->cnt[wg][row] = nv;
    xs->fresh[wg][row] = __float_as_int(mx);
    ptx::named_bar_sync(3 + quad, 64);
    float lo = fminf(mn, xs->thr[wg ^ 1][row]);
    float hi = fmaxf(mx, __int_as_float(xs->fresh[wg ^ 1][row]));
    const int ntot = nv + xs->cnt[wg ^ 1][row];
    ptx::named_bar_sync(3 + quad, 64);
    const bool enough = ntot >= k;
    // invariant: count(>= lo) >= k. 16 rounds leave (max - min) / 65536 of slack below the k-th key. Rows
    // with fewer than k columns keep everything but still meet the partner at every barrier.
#pragma unroll 1
    for (int r = 0; r < 16; r++) {
        const float mid = lo + 0.5f * (hi - lo);
        int c = 0;
#pragma unroll
        for (int i = 0; i < HALF_N; i++) c += (f[i] >= mid) ? 1 : 0;
        int* slot = (r & 1) ? xs->fresh[wg] : xs->cnt[wg];
        const int* pslot = (r & 1) ? xs->fresh[wg ^ 1] : xs->cnt[wg ^ 1];
        slot[row] = c;
        ptx::named_bar_sync(3 + quad, 64);
        const int tot = c + pslot[row];
        if (tot >= k && mid > lo)
            lo = mid;
        else
            hi = mid;
    }
    // margin in the domain of f (IP keys carry the row's scale)
    const float cut = enough ? lo - (L2 ? margin : margin * sc) : NEG_INF;
    const float ksc = L2 ? 1.f : inv;
    int cnt = 0;
#pragma unroll
    for (int i = 0; i < HALF_N; i++) {
        if (f[i] >= cut && i < valid) {
            myb[cnt] = make_uint2(__float_as_uint(f[i] * ksc), (uint32_t)(id0 + i));
            cnt++;
        }
    }
    OneShotOut o;
    o.cnt = cnt;
    o.lb = enough ? lo * ksc : NEG_INF;
    return o;
}

template <bool L2>
__device__ __forceinline__ void epi_stage_norms(float* nrm, const float* b_norms, const Unit& un, int col_base,
                                                int valid, int64_t b_total, int etid, int wg) {
    if (L2) {
        // stage the norms of this warpgroup's 128 columns (one per thread); the warpgroup's named
        // barrier also orders reuse of the buffer
        const int64_t br = (int64_t)un.b_row0 + col_base + etid;
        nrm[etid] = (etid < valid && br < b_total) ? -b_norms[br] : 0.f;  // NEGATED: the addend of the epilogue's fma
        if (wg == 0)
            asm volatile("bar.sync 1, 128;" ::: "memory");
        else
            asm volatile("bar.sync 2, 128;" ::: "memory");
    }
}

// The selection epilogue shared by every kernel of this file. Executed by warps 2..9; warpgroup
// g = (warp-2)/4 handles the tiles whose running index (over all units of this CTA) has parity
// g, i.e. TMEM accumulator g. PAIR: units are taken in CTA pairs and the accumulator is handed
// back with a cluster-scope arrive on the leader's barrier.
struct EpiArgs {
    const Unit* units;
    int n_units, k, pw;
    float margin_scale;  // 0: plain top-k (3xTF32 kernels)
    const float *a_norms, *b_norms;
    int64_t a_total, b_total;
    float* part_key;
    int* part_idx;
    int* part_cnt;  // filter kernels: partial rows are UNSORTED, part_cnt[partial row] entries each (see epi_unit_end_unsorted)
    int* row_flags;
    uint2* cand_buf;  // candidate buffers: [CTA][warpgroup][row][CAND_CAP] (key, idx) entries
    // Shared running bounds: gthr[query] (zero-initialised ordered uints) is raised by every
    // unit of the query and read back at each tile, so units that start later (IVF lists, tail
    // chunks, the second warpgroup) begin with a hot threshold instead of re-discovering it.
    // Query of query-side row r: row_map ? row_map[r] / row_div : r.
    unsigned* gthr;
    const int* row_map;
    int row_div;
    // fp16 filter: accumulator = a_row_scale[row] * b_scale * (q . x), powers of two (null / 1: unscaled)
    const float* a_row_scale;
    float b_scale;
    // IVF phase B (every row starts from the bound its query's closest list established): units run
    // no scheduled prunes, and a unit ends without the pairwise union prune. Their rows collect what
    // beats the bound of phase A -- ~9 candidates per (query, list) pair on average, ~110 in the
    // longest lists -- and the few rows that outgrow a buffer are tightened one by one by the in-tile
    // overflow guard and at the unit's end.
    int hot;
};

// IVFX compiles in the short-unit machinery (hot rows, one-tile units): only the double-buffered
// kernel (topk_tc3d_kernel) carries it, so the flat search kernels keep their exact code.
template <bool L2, bool PAIR, bool NEED_QN, bool IVFX = false>
__device__ __forceinline__ void epilogue_run(const EpiArgs& A, uint64_t* tfull, uint64_t* tempty,
                                             float (*nrm)[2][HALF_N], XchgShared* xs, uint32_t tmem_base, int warp,
                                             int lane, uint32_t rank) {
    const int wg = (warp - EPI_WARP0) >> 2;  // warpgroup = column half of every tile
    const int quad = warp & 3;         // TMEM lane quarter this warp may read
    const int row = quad * 32 + lane;  // query row inside the tile
    const int etid = ((warp - EPI_WARP0) & 3) * 32 + lane;
    const int64_t crow0 = ((int64_t)blockIdx.x * EPI_WGS + wg) * BM + quad * 32;  // this warp's 32 buffer rows
    uint2* cb = A.cand_buf + crow0 * CAND_CAP;
    uint2* myb = cb + (int64_t)lane * CAND_CAP;
    uint32_t tempty_remote0 = 0, tempty_remote1 = 0;  // scalars: an indexed array would live in local memory
    if (PAIR) {
        tempty_remote0 = ptx::mapa_u32(&tempty[0], 0);
        tempty_remote1 = ptx::mapa_u32(&tempty[1], 0);
    }
    const int first = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int stride = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    const int count = PAIR ? (A.n_units + 1) >> 1 : A.n_units;
    const uint32_t taddr_wg = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(wg * HALF_N);
    uint32_t gt = 0;  // running tile index of this CTA (same sequence as the MMA warp)
    for (int i = first; i < count; i += stride) {
        const int u = PAIR ? 2 * i + (int)rank : i;
        const Unit un = A.units[u];
        const int ntiles = (PAIR || un.a_rows > 0) ? (un.b_rows + BN - 1) / BN : 0;
        const int64_t ar = (int64_t)un.a_row0 + row;
        const bool live = row < un.a_rows && ar < A.a_total;
        EpiRow st;
        st.cnt = 0;
        st.base = 0;
        st.thr = live ? NEG_INF : __builtin_huge_valf();
        st.cthr = st.thr;
        st.sc = (A.a_row_scale && live) ? A.a_row_scale[ar] * A.b_scale : 1.f;
        st.inv = 1.f / st.sc;
        st.qn = ((L2 || NEED_QN) && live) ? A.a_norms[ar] : 0.f;
        st.margin = NEED_QN ? A.margin_scale * sqrtf(st.qn) * (L2 ? 2.f : 1.f) : 0.f;
        st.flag = 0;
        st.gslot = nullptr;
        if (A.gthr && live) st.gslot = A.gthr + (A.row_map ? A.row_map[ar] / A.row_div : (int)ar);
        // filter kernels, one-tile unit, cold rows: per-thread bisection in registers (epi_single_tile)
        const bool hot = IVFX && A.hot;
        const bool one_shot = IVFX && NEED_QN && !hot && ntiles == 1;
        // the unit's end (below) is chosen here, ahead of the tile loop: tested after the loop, the
        // condition let the compiler reshape the whole loop around ntiles == 1 (more spills, IVF scan
        // with inner products ~2 % slower on a B200)
        const bool short_end = IVFX && NEED_QN && (hot || one_shot);
        // Cold multi-tile units (flat search: full-catalog and first-round tail units; IVF phase A): the
        // generic path appends the whole first tile (every key beats -inf: 256 entries per row, 112k
        // cycles) and then prunes 256 entries per row (58k). Their first tile takes the in-register
        // bisection of single_tile_call instead: ~k + margin-set entries per row are appended, the row's
        // threshold is known at once and the scheduled prune after tile 1 is skipped. The two warps of a
        // lane quarter must take the same path (barriers inside): they agree through shared memory on
        // whether ANY of their 32 rows already holds a bound from another unit of its query.
        bool first_shot = false;
        if (NEED_QN && !hot && ntiles > 1) {
            unsigned g0 = 0u;
            if (st.gslot) g0 = *(volatile unsigned*)st.gslot;
            if (wg == 0)
                xs->nthr[row] = g0 != 0u ? 1.f : 0.f;
            else
                xs->lb[row] = g0 != 0u ? 1u : 0u;
            ptx::named_bar_sync(3 + quad, 64);
            const bool warm = xs->nthr[row] != 0.f || xs->lb[row] != 0u;
            first_shot = !__any_sync(0xffffffffu, warm);
        }
        for (int t = 0; t < ntiles; t++, gt++) {
            const int acc = (int)(gt & 1);
            const uint32_t acc_phase = (gt >> 1) & 1;
            const int col_base = t * BN + wg * HALF_N;  // first item column of this warpgroup's half
            const int valid = un.b_rows - col_base;     // may be <= 0: nothing of this half is real
            // issued before the wait so that its latency hides behind the MMAs: what the query's
            // other units (lists, tail chunks, the other warpgroup) have established so far
            unsigned g_raw = 0;
            if (st.gslot) g_raw = *(volatile unsigned*)st.gslot;
            // two norm buffers per warpgroup: a fast warp may stage its next tile while a slow
            // one still reads the current one (the named barrier keeps them within one tile)
            float* nrm_t = nrm[wg][acc];
            epi_stage_norms<L2>(nrm_t, A.b_norms, un, col_base, valid, A.b_total, etid, wg);
            NRB_TR(warp - EPI_WARP0 + 1, gt, 0);
            ptx::mbar_wait(&tfull[acc], acc_phase);
            ptx::tcgen05_fence_after();
            NRB_TR(warp - EPI_WARP0 + 1, gt, 1);
            if (st.gslot) {
                st.thr = fmaxf(st.thr, from_ordered_u32(g_raw) - st.margin);
                st.cthr = L2 ? st.thr + st.qn : st.thr * st.sc;
            }
            const uint32_t taddr0 = taddr_wg + (uint32_t)(acc * BN);
            // hands this warp's part of the accumulator back to the MMA warp
            auto release = [&]() {
                ptx::tcgen05_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if (PAIR)
                        ptx::mbar_arrive_cluster_relaxed(acc ? tempty_remote1 : tempty_remote0);
                    else
                        ptx::mbar_arrive(&tempty[acc]);
                }
            };
            if ((IVFX && one_shot) || (first_shot && t == 0)) {
                const OneShotOut o = single_tile_call<L2, PAIR>(taddr0, valid, un.b_row0 + col_base, nrm_t, st.sc, st.inv, st.qn,
                                                              st.margin, myb, A.k, xs, wg, row, quad,
                                                              acc ? tempty_remote1 : tempty_remote0, &tempty[acc]);
                st.cnt = live ? o.cnt : 0;
                st.base = st.cnt;
                if (first_shot && live && o.lb > NEG_INF) {  // the unit goes on: appends continue above the bound
                    st.thr = fmaxf(st.thr, o.lb - st.margin);
                    st.cthr = L2 ? st.thr + st.qn : st.thr * st.sc;
                }
                NRB_TR(warp - EPI_WARP0 + 1, gt, 2);
                if (wg == 0 && st.gslot && o.lb > NEG_INF) atomicMax(st.gslot, ordered_u32(o.lb));
            } else if (valid >= HALF_N) {
                // Full tile: copy the warp's 32 x 128 scores into registers and give the accumulator
                // back BEFORE selecting. The selection time of a tile varies from warp to warp (it
                // depends on how many keys pass), and the MMA warp needs all 16 warps of the CTA
                // pair to release an accumulator: releasing after the loads instead of after the
                // selection lets the MMAs run a tile further ahead of the slowest warp.
                uint32_t v0[32], v1[32], v2[32], v3[32];
                ptx::tmem_ld_32x32b_x32(taddr0, v0);
                ptx::tmem_ld_32x32b_x32(taddr0 + 32, v1);
                ptx::tmem_ld_32x32b_x32(taddr0 + 64, v2);
                ptx::tmem_ld_32x32b_x32(taddr0 + 96, v3);
                ptx::tmem_ld_wait();
                release();
                NRB_TR(warp - EPI_WARP0 + 1, gt, 2);
                const float m2inv = 2.f * st.inv;  // epi_chunk: t = acc * (2 / scale) - |x|^2
                const int id0 = un.b_row0 + col_base;
                epi_chunk<L2, true>(v0, 0, valid, id0, nrm_t, m2inv, st, cb, myb, A.k, A.pw, lane);
                epi_chunk<L2, true>(v1, 32, valid, id0, nrm_t, m2inv, st, cb, myb, A.k, A.pw, lane);
                epi_chunk<L2, true>(v2, 64, valid, id0, nrm_t, m2inv, st, cb, myb, A.k, A.pw, lane);
                epi_chunk<L2, true>(v3, 96, valid, id0, nrm_t, m2inv, st, cb, myb, A.k, A.pw, lane);
            } else {
                if (valid > 0)
                    epi_tile_ragged<L2>(taddr0, valid, un.b_row0 + col_base, nrm_t, st, cb, myb, A.k, A.pw, lane);
                release();
            }
            // Scheduled prune: at tile counts 1, 2, 4, 8, ... every warp of the CTA pair brings its
            // rows back to (about) their best k and tightens their thresholds. A row's pass rate is
            // ~k/n after n items, so each doubling admits ~k new candidates per row; and because the 16
            // warps that share every accumulator hand-off prune in the SAME tiles, the hand-offs in
            // between never wait for one straggler. The two warps of a lane quarter (one per column
            // half) do it together on the union of their buffers: see union_tighten_rows.
            NRB_TR(warp - EPI_WARP0 + 1, gt, 3);
            const uint32_t tp = (uint32_t)t + 1u;
            // flat search: tile counts 1, 2, 4, 8, ...; IVF scan: 1, 2, 8, 32, 128, ... -- with 8-byte entries an
            // append costs less than it did and a scheduled prune the same, and the short cold units of an IVF
            // scan (a 19-tile unit spent two thirds of its cycles in four prunes) are better off with half the
            // prunes and ~25 % more appends (scan kernels 9.2 -> 8.8 ms; the flat kernel is indifferent: 8.0 / 8.3
            // vs 8.05 ms, so it keeps the schedule its buffers were sized for)
            const bool sched = (tp & (tp - 1u)) == 0u && (!IVFX || tp == 1u || ((__ffs(tp) - 1) & 1) == 1);
            if (sched && t + 1 < ntiles && !hot && !(first_shot && t == 0)) {
                xs->cnt[wg][row] = st.cnt;
                xs->fresh[wg][row] = st.cnt - st.base;
                xs->thr[wg][row] = st.thr;
                if (wg == 0) xs->margin[row] = st.margin;
                NRB_TRP(warp - EPI_WARP0 + 1, 0);
                ptx::named_bar_sync(3 + quad, 64);
                NRB_TRP(warp - EPI_WARP0 + 1, 1);
                union_tighten_rows(xs, A.cand_buf + (int64_t)blockIdx.x * EPI_WGS * BM * CAND_CAP, quad, wg, A.k, A.pw,
                                   A.row_map ? max(4, A.k >> 2) : 0);
                NRB_TRP(warp - EPI_WARP0 + 1, 2);
                ptx::named_bar_sync(3 + quad, 64);
                NRB_TRP(warp - EPI_WARP0 + 1, 3);
                NRB_TRP_NEXT(warp - EPI_WARP0 + 1);
                if (xs->done[row]) {
                    st.cnt = xs->cnt[wg][row];
                    st.base = st.cnt;
                    st.thr = xs->nthr[row];
                    st.cthr = L2 ? st.thr + st.qn : st.thr * st.sc;
                    const uint32_t lbu = xs->lb[row];
                    if (wg == 0 && st.gslot && lbu != 0u) atomicMax(st.gslot, lbu);
                    if (NEED_QN && xs->ovf[row] && live) epi_abandon_row(st);
                }
            }
        }
        if (short_end) {
            // hot units: rows hold a handful of entries; only rows over pw are tightened, each on its own
            // (no exchange with the partner warp, no barriers), then the rows leave unsorted
            const unsigned need = __ballot_sync(0xffffffffu, st.cnt > A.pw);
            if (need) epi_prune_rows<L2>(need, st, cb, A.k, A.pw, lane);
            if (st.cnt > A.pw) {
                st.flag = 1;
                st.cnt = A.pw;
            }
            epi_unit_end_unsorted(live ? st.cnt : 0, cb, ((int64_t)u * EPI_WGS + wg) * UNIT_ROWS + quad * 32, A.pw,
                                  A.part_key, A.part_idx, A.part_cnt, lane);
        } else if (NEED_QN) {
            // final union prune (rows that need one only), then the rows leave unsorted
            xs->cnt[wg][row] = st.cnt;
            xs->fresh[wg][row] = st.cnt - st.base;
            xs->thr[wg][row] = st.thr;
            if (wg == 0) xs->margin[row] = st.margin;
            ptx::named_bar_sync(3 + quad, 64);
            union_tighten_rows(xs, A.cand_buf + (int64_t)blockIdx.x * EPI_WGS * BM * CAND_CAP, quad, wg, A.k, A.pw, -1);
            ptx::named_bar_sync(3 + quad, 64);
            if (xs->done[row]) {
                st.cnt = xs->cnt[wg][row];
                const uint32_t lbu = xs->lb[row];
                if (wg == 0 && st.gslot && lbu != 0u) atomicMax(st.gslot, lbu);
                if (xs->ovf[row] && live) epi_abandon_row(st);
            }
            if (st.cnt > A.pw) {  // the margin set does not fit: the query is recomputed by the exact path
                st.flag = 1;
                st.cnt = A.pw;
            }
            epi_unit_end_unsorted(live ? st.cnt : 0, cb, ((int64_t)u * EPI_WGS + wg) * UNIT_ROWS + quad * 32, A.pw,
                                  A.part_key, A.part_idx, A.part_cnt, lane);
        } else {
            epi_unit_end(st, cb, ((int64_t)u * EPI_WGS + wg) * UNIT_ROWS + quad * 32, A.k, A.pw, A.part_key, A.part_idx, lane);
        }
        if (NEED_QN && st.flag && live) A.row_flags[A.row_map ? A.row_map[ar] / A.row_div : (int)ar] = 1;  // per QUERY
    }
}

// ---------------------------------------------------------------------------- v2: CTA pairs
// Cluster c handles unit pairs p = c, c + n_clusters, ...; CTA rank r of the pair owns unit
// 2p + r. Both units of a pair have the same item rows (the planners guarantee it).
template <bool L2>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
topk_tc2_kernel(const __grid_constant__ CUtensorMap map_ah, const __grid_constant__ CUtensorMap map_al,
                const __grid_constant__ CUtensorMap map_bh, const __grid_constant__ CUtensorMap map_bl,
                const Unit* __restrict__ units, const int* __restrict__ n_units_p, int nkc, int k,
                const float* __restrict__ a_norms, const float* __restrict__ b_norms,
                int64_t a_total, int64_t b_total, float* __restrict__ part_key,
                int* __restrict__ part_idx, float* __restrict__ cand_key_buf,
                int* __restrict__ cand_idx_buf, unsigned* __restrict__ gthr, const int* __restrict__ row_map,
                int row_div) {
    constexpr int STAGES = V2_STAGES, STAGE_BYTES = V2_STAGE_BYTES;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    TcShared<STAGES>* sh = reinterpret_cast<TcShared<STAGES>*>(smem + (size_t)STAGES * STAGE_BYTES);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = ptx::cluster_ctarank();
    const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
    const int n_pairs = (*n_units_p + 1) >> 1;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; s++) {
            ptx::mbar_init(&sh->full[s], 1);   // leader: its own arrive.expect_tx covers both CTAs' bytes
            ptx::mbar_init(&sh->empty[s], 1);  // multicast tcgen05.commit from the leader
        }
        for (int a = 0; a < 2; a++) {
            ptx::mbar_init(&sh->tfull[a], 1);   // multicast tcgen05.commit from the leader
            ptx::mbar_init(&sh->tempty[a], 16);  // leader: 8 epilogue warps of each CTA
        }
        ptx::fence_barrier_init();
        ptx::prefetch_tensormap(&map_ah);
        ptx::prefetch_tensormap(&map_al);
        ptx::prefetch_tensormap(&map_bh);
        ptx::prefetch_tensormap(&map_bl);
    }
    if (warp == 1) {
        ptx::tmem_alloc_cg2(&sh->tmem_base, TMEM_COLS);
        ptx::tmem_relinquish_cg2();
    }
    ptx::tcgen05_fence_before();
    __syncwarp();
    ptx::cluster_sync_all();
    ptx::tcgen05_fence_after();
    const uint32_t tmem_base = sh->tmem_base;
    if (warp < EPI_WARP0) ptx::setmaxnreg_dec<40>();

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer (both CTAs)
        const uint32_t full0_base = ptx::mapa_u32(&sh->full[0], 0);  // the leader's full barriers
        int stage = 0;
        uint32_t phase = 0;
        for (int p = cluster_id; p < n_pairs; p += n_clusters) {
            const Unit un = units[2 * p + rank];
            const int ntiles = (un.b_rows + BN - 1) / BN;
            for (int t = 0; t < ntiles; t++) {
                const int brow = un.b_row0 + t * BN + (int)rank * (BN / 2);  // this CTA's half of the item tile
                for (int kc = 0; kc < nkc; kc++) {
                    ptx::mbar_wait<64>(&sh->empty[stage], phase ^ 1);
                    uint8_t* st = smem + (size_t)stage * STAGE_BYTES;
                    const uint32_t fb = full0_base + (uint32_t)stage * 8;
                    if (ptx::elect_one()) {
                        if (rank == 0) ptx::mbar_arrive_expect_tx(&sh->full[stage], 2 * STAGE_BYTES);
                        ptx::tma_load_2d_cg2(st, &map_ah, fb, kc * KC, un.a_row0);
                        ptx::tma_load_2d_cg2(st + A_BYTES, &map_al, fb, kc * KC, un.a_row0);
                        ptx::tma_load_2d_cg2(st + 2 * A_BYTES, &map_bh, fb, kc * KC, brow);
                        ptx::tma_load_2d_cg2(st + 2 * A_BYTES + BH_BYTES, &map_bl, fb, kc * KC, brow);
                    }
                    __syncwarp();
                    if (++stage == STAGES) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (leader CTA only)
        if (rank == 0) {
            constexpr uint32_t idesc = ptx::umma_idesc_tf32(2 * BM, BN);
            const uint32_t lo0 = ptx::umma_desc_lo(ptx::smem_u32(smem));
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int p = cluster_id; p < n_pairs; p += n_clusters) {
                const Unit un = units[2 * p];
                const int ntiles = (un.b_rows + BN - 1) / BN;
                for (int t = 0; t < ntiles; t++) {
                    ptx::mbar_wait(&sh->tempty[acc], acc_phase ^ 1);
                    ptx::tcgen05_fence_after();
                    const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
                    for (int kc = 0; kc < nkc; kc++) {
                        ptx::mbar_wait(&sh->full[stage], phase);
                        ptx::tcgen05_fence_after();
                        const uint32_t l_ah = lo0 + (uint32_t)(stage * STAGE_BYTES) / 16;
                        const uint32_t l_al = l_ah + A_BYTES / 16, l_bh = l_ah + 2 * A_BYTES / 16,
                                       l_bl = l_ah + (2 * A_BYTES + BH_BYTES) / 16;
                        if (ptx::elect_one()) {
#pragma unroll
                            for (int ks = 0; ks < KC / 8; ks++) {
                                const uint64_t d_ah = ptx::umma_desc_join(l_ah + 2 * ks), d_al = ptx::umma_desc_join(l_al + 2 * ks);
                                const uint64_t d_bh = ptx::umma_desc_join(l_bh + 2 * ks), d_bl = ptx::umma_desc_join(l_bl + 2 * ks);
                                ptx::umma_tf32_cg2(d_tmem, d_al, d_bh, idesc, (kc | ks) != 0);
                                ptx::umma_tf32_cg2(d_tmem, d_ah, d_bl, idesc, 1);
                                ptx::umma_tf32_cg2(d_tmem, d_ah, d_bh, idesc, 1);
                            }
                            ptx::umma_commit_cg2_mc(&sh->empty[stage], 3);  // both CTAs' stage is free
                        }
                        __syncwarp();
                        if (++stage == STAGES) {
                            stage = 0;
                            phase ^= 1;
                        }
                    }
                    if (ptx::elect_one()) ptx::umma_commit_cg2_mc(&sh->tfull[acc], 3);  // both halves complete
                    __syncwarp();
                    acc ^= 1;
                    if (acc == 0) acc_phase ^= 1;
                }
            }
        }
    } else if (warp >= EPI_WARP0) {
        // ------------------------------------------------------------------ selection epilogue (both CTAs)
        ptx::setmaxnreg_inc<232>();
        EpiArgs ea{units, *n_units_p, k, k, 0.f, a_norms, b_norms, a_total, b_total, part_key, part_idx, nullptr, nullptr,
                   reinterpret_cast<uint2*>(cand_key_buf), gthr, row_map, row_div, nullptr, 1.f, 0};
        epilogue_run<L2, true, false>(ea, sh->tfull, sh->tempty, sh->nrm, &sh->xchg, tmem_base, warp, lane, rank);
    }

    ptx::tcgen05_fence_before();
    __syncwarp();
    ptx::cluster_sync_all();  // both CTAs are done with the pair's TMEM and barriers
    if (warp == 1) {
        ptx::tcgen05_fence_after();
        ptx::tmem_dealloc_cg2(tmem_base, TMEM_COLS);
    }
}


// ---------------------------------------------------------------------------- v3: 1xTF32 filter
// CTA pairs again, but ONE tf32 pass (hi planes only) and the query tile resident in shared
// memory for the whole unit (128 rows x kp <= 256 fp32 = 128 KB), so only the item half-tiles
// stream (16 KB stages, 5 deep). The scores carry a bounded error |a - s| <= eps*|q|*|x| with
// eps ~ 2^-10 (both operands rounded to tf32), so the epilogue keeps, per row, the best k AND
// every candidate within margin = 2*eps*|q|*max|x| of the k-th: that set provably contains the
// true top-k. select_refine_kernel rescoring those <= k+32 candidates exactly in fp32 gives
// the final order; rows with more candidates than slots are flagged and recomputed by the
// 3xTF32 kernel.
constexpr int V3_MAX_NKC = 8;  // tf32: kp <= 256 floats = 8 chunks of 128 bytes; fp16: 4 chunks

template <bool F16>
struct Tc3Cfg {
    static constexpr int STAGES = F16 ? 8 : 5;                          // 16 KB item half-tile stages
    static constexpr int A_TILE_BYTES = (F16 ? 4 : V3_MAX_NKC) * A_BYTES;  // resident query tile: 64 / 128 KB
};

template <int STAGES>
struct Tc3Shared {
    uint64_t full[STAGES];
    uint64_t empty[STAGES];
    uint64_t tfull[2];
    uint64_t tempty[2];
    uint64_t afull[2];
    uint64_t aempty[2];
    uint32_t tmem_base;
    uint32_t pad;
    float nrm[EPI_WGS][2][HALF_N];
    XchgShared xchg;
};
template <bool F16>
constexpr size_t v3_smem() {  // no slack: the dynamic shared memory is declared __align__(1024)
    return (size_t)Tc3Cfg<F16>::A_TILE_BYTES + (size_t)Tc3Cfg<F16>::STAGES * BH_BYTES + sizeof(Tc3Shared<Tc3Cfg<F16>::STAGES>);
}
static_assert(v3_smem<false>() <= 232448 && v3_smem<true>() <= 232448,
              "topk_tc3_kernel exceeds the 227 KB of shared memory per CTA");

// F16: the operand planes are IEEE fp16 (same 11-bit significand as tf32, so the same error
// bound) scaled by powers of two -- per row on the query side, one scale on the item side. K
// chunks are still 128-byte rows (64 halves), four K = 16 MMAs each, at twice the tf32 rate and
// half the shared-memory / L2 traffic.
//
// PAIR = false is the single-CTA form (cta_group::1, M = 128, every CTA streams whole 256-row
// item tiles in 32 KB stages): one unit per CTA instead of two per CTA pair. It exists for
// batches that are a single partial wave, where an odd number of query tiles or a phantom tile
// keeps CTA pairs from cutting the catalog finely enough to use every SM (e.g. 49 tiles x 3
// chunks = 147 units fill 147 of 148 SMs; 25 pairs can only be cut 2 ways = 50 of 74 pairs).
// A2 = two resident query tiles (fp16 CTA pairs only): the producer loads the NEXT unit's query tile
// while the current unit computes, which takes the query-tile load (and the drain of the previous
// unit's MMAs it had to wait for) off the critical path between units. It pays when units are
// short -- the (list, 256 queries) units of an IVF scan average a few item tiles -- and costs three
// item stages (5 instead of 8), so the flat search keeps the single-buffer form.
template <bool F16, bool PAIR, bool A2 = false>
struct Tc3Lay {
    static constexpr int NA = A2 ? 2 : 1;
    static constexpr int B_STAGE_BYTES = PAIR ? BH_BYTES : B_BYTES;
    static constexpr int STAGES = A2 ? 5 : (PAIR ? Tc3Cfg<F16>::STAGES : Tc3Cfg<F16>::STAGES / 2);
    static constexpr size_t SMEM = (size_t)NA * Tc3Cfg<F16>::A_TILE_BYTES + (size_t)STAGES * B_STAGE_BYTES + sizeof(Tc3Shared<STAGES>);
};
static_assert(Tc3Lay<true, false>::SMEM <= 232448, "single-CTA filter kernel exceeds the shared memory per CTA");
static_assert(Tc3Lay<true, true, true>::SMEM <= 232448, "double-buffered filter kernel exceeds the shared memory per CTA");

template <bool L2, bool F16, bool PAIR, bool A2 = false>
__device__ __forceinline__ void tc3_body(const CUtensorMap& map_ah, const CUtensorMap& map_bh,
                                         const Unit* __restrict__ units, const int* __restrict__ n_units_p, int nkc,
                                         int k, int pw, float margin_scale, const float* __restrict__ a_norms,
                                         const float* __restrict__ b_norms, int64_t a_total, int64_t b_total,
                                         float* __restrict__ part_key, int* __restrict__ part_idx,
                                         int* __restrict__ part_cnt, int* __restrict__ row_flags,
                                         float* __restrict__ cand_key_buf,
                                         int* __restrict__ cand_idx_buf, unsigned* __restrict__ gthr,
                                         const float* __restrict__ a_row_scale, float b_scale,
                                         const int* __restrict__ row_map, int row_div, int hot) {
    constexpr int STAGES = Tc3Lay<F16, PAIR, A2>::STAGES;
    constexpr int BSB = Tc3Lay<F16, PAIR, A2>::B_STAGE_BYTES;
    constexpr int NA = Tc3Lay<F16, PAIR, A2>::NA;
    constexpr int ATB = Tc3Cfg<F16>::A_TILE_BYTES;
    constexpr int KE = F16 ? 2 * KC : KC;  // elements per 128-byte K chunk
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw;  // 128-byte swizzled tiles need 1024-byte alignment
    if ((ptx::smem_u32(smem) & 1023u) != 0) __trap();
    uint8_t* smem_b = smem + (size_t)NA * ATB;
    Tc3Shared<STAGES>* sh = reinterpret_cast<Tc3Shared<STAGES>*>(smem_b + (size_t)STAGES * BSB);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = PAIR ? ptx::cluster_ctarank() : 0u;
    // work items: unit pairs for CTA pairs, units for single CTAs
    const int wid = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int nworkers = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    const int n_items = PAIR ? (*n_units_p + 1) >> 1 : *n_units_p;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; s++) {
            ptx::mbar_init(&sh->full[s], 1);
            ptx::mbar_init(&sh->empty[s], 1);
        }
        for (int a = 0; a < 2; a++) {
            ptx::mbar_init(&sh->tfull[a], 1);
            ptx::mbar_init(&sh->tempty[a], PAIR ? 16 : 8);
        }
        for (int a = 0; a < 2; a++) {
            ptx::mbar_init(&sh->afull[a], 1);
            ptx::mbar_init(&sh->aempty[a], 1);
        }
        ptx::fence_barrier_init();
        ptx::prefetch_tensormap(&map_ah);
        ptx::prefetch_tensormap(&map_bh);
    }
    if (warp == 1) {
        if (PAIR) {
            ptx::tmem_alloc_cg2(&sh->tmem_base, TMEM_COLS);
            ptx::tmem_relinquish_cg2();
        } else {
            ptx::tmem_alloc(&sh->tmem_base, TMEM_COLS);
            ptx::tmem_relinquish();
        }
    }
    ptx::tcgen05_fence_before();
    if (PAIR) {
        __syncwarp();
        ptx::cluster_sync_all();
    } else {
        __syncthreads();
    }
    ptx::tcgen05_fence_after();
    const uint32_t tmem_base = sh->tmem_base;
    if (warp < EPI_WARP0) ptx::setmaxnreg_dec<40>();  // the CTA owns 12 warps x 168 registers; 4 x 40 + 8 x 232 = 12 x 168 exactly (a larger request never succeeds)

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer (every CTA)
        const uint32_t full0_base = PAIR ? ptx::mapa_u32(&sh->full[0], 0) : 0u;
        const uint32_t afull0 = PAIR ? ptx::mapa_u32(&sh->afull[0], 0) : 0u;
        int stage = 0;
        uint32_t phase = 0;
        int uc = 0;  // units taken by this CTA: query-tile buffer uc % NA, barrier parity (uc / NA) & 1
        for (int p = wid; p < n_items; p += nworkers, uc++) {
            const Unit un = units[PAIR ? 2 * p + (int)rank : p];
            const int ntiles = (PAIR || un.a_rows > 0) ? (un.b_rows + BN - 1) / BN : 0;
            const int ab = uc % NA;
            const uint32_t a_par = (uint32_t)(uc / NA) & 1u;
            uint8_t* smem_a = smem + (size_t)ab * ATB;
            // the unit's query tile, once (A2: into the buffer the unit before last has released)
            ptx::mbar_wait<64>(&sh->aempty[ab], a_par ^ 1);
            if (ptx::elect_one()) {
                if (PAIR) {
                    if (rank == 0) ptx::mbar_arrive_expect_tx(&sh->afull[ab], 2 * nkc * A_BYTES);
                    for (int kc = 0; kc < nkc; kc++)
                        ptx::tma_load_2d_cg2(smem_a + (size_t)kc * A_BYTES, &map_ah, afull0 + (uint32_t)ab * 8, kc * KE, un.a_row0);
                } else {
                    ptx::mbar_arrive_expect_tx(&sh->afull[ab], nkc * A_BYTES);
                    for (int kc = 0; kc < nkc; kc++)
                        ptx::tma_load_2d(smem_a + (size_t)kc * A_BYTES, &map_ah, &sh->afull[ab], kc * KE, un.a_row0);
                }
            }
            __syncwarp();
            for (int t = 0; t < ntiles; t++) {
                const int brow = un.b_row0 + t * BN + (PAIR ? (int)rank * (BN / 2) : 0);
                for (int kc = 0; kc < nkc; kc++) {
                    ptx::mbar_wait<64>(&sh->empty[stage], phase ^ 1);
                    if (ptx::elect_one()) {
                        if (PAIR) {
                            if (rank == 0) ptx::mbar_arrive_expect_tx(&sh->full[stage], 2 * BSB);
                            ptx::tma_load_2d_cg2(smem_b + (size_t)stage * BSB, &map_bh, full0_base + (uint32_t)stage * 8,
                                                 kc * KE, brow);
                        } else {
                            ptx::mbar_arrive_expect_tx(&sh->full[stage], BSB);
                            ptx::tma_load_2d(smem_b + (size_t)stage * BSB, &map_bh, &sh->full[stage], kc * KE, brow);
                        }
                    }
                    __syncwarp();
                    if (++stage == STAGES) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (leader CTA of a pair)
        if (rank == 0) {
            constexpr int MM = PAIR ? 2 * BM : BM;
            constexpr uint32_t idesc = F16 ? ptx::umma_idesc_f16(MM, BN) : ptx::umma_idesc_tf32(MM, BN);
            const uint32_t la0 = ptx::umma_desc_lo(ptx::smem_u32(smem));
            const uint32_t lb0 = ptx::umma_desc_lo(ptx::smem_u32(smem_b));
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            uint32_t mma_gt = 0;  // running tile index (trace builds)
            int uc = 0;
            for (int p = wid; p < n_items; p += nworkers, uc++) {
                const Unit un = units[PAIR ? 2 * p : p];
                const int ntiles = (PAIR || un.a_rows > 0) ? (un.b_rows + BN - 1) / BN : 0;
                const int ab = uc % NA;
                const uint32_t la_u = la0 + (uint32_t)(ab * ATB) / 16;
                ptx::mbar_wait(&sh->afull[ab], (uint32_t)(uc / NA) & 1u);
                ptx::tcgen05_fence_after();
                for (int t = 0; t < ntiles; t++, mma_gt++) {
                    ptx::mbar_wait(&sh->tempty[acc], acc_phase ^ 1);
                    ptx::tcgen05_fence_after();
                    NRB_TR(0, mma_gt, 0);
                    const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
                    for (int kc = 0; kc < nkc; kc++) {
                        ptx::mbar_wait(&sh->full[stage], phase);
                        ptx::tcgen05_fence_after();
                        const uint32_t l_a = la_u + (uint32_t)(kc * A_BYTES) / 16;
                        const uint32_t l_b = lb0 + (uint32_t)(stage * BSB) / 16;
                        if (ptx::elect_one()) {
#pragma unroll
                            for (int ks = 0; ks < 4; ks++) {  // 32 bytes of K per MMA: 8 tf32 / 16 fp16
                                const uint64_t da = ptx::umma_desc_join(l_a + 2 * ks), db = ptx::umma_desc_join(l_b + 2 * ks);
                                const uint32_t accum = (kc | ks) != 0;
                                if (PAIR) {
                                    if (F16)
                                        ptx::umma_f16_cg2(d_tmem, da, db, idesc, accum);
                                    else
                                        ptx::umma_tf32_cg2(d_tmem, da, db, idesc, accum);
                                } else {
                                    if (F16)
                                        ptx::umma_f16(d_tmem, da, db, idesc, accum);
                                    else
                                        ptx::umma_tf32(d_tmem, da, db, idesc, accum);
                                }
                            }
                            if (PAIR)
                                ptx::umma_commit_cg2_mc(&sh->empty[stage], 3);
                            else
                                ptx::umma_commit(&sh->empty[stage]);
                        }
                        __syncwarp();
                        if (++stage == STAGES) {
                            stage = 0;
                            phase ^= 1;
                        }
                    }
                    if (ptx::elect_one()) {
                        if (PAIR)
                            ptx::umma_commit_cg2_mc(&sh->tfull[acc], 3);
                        else
                            ptx::umma_commit(&sh->tfull[acc]);
                    }
                    __syncwarp();
                    NRB_TR(0, mma_gt, 1);
                    acc ^= 1;
                    if (acc == 0) acc_phase ^= 1;
                }
                // query tile may be replaced once these MMAs retire
                if (ptx::elect_one()) {
                    if (PAIR)
                        ptx::umma_commit_cg2_mc(&sh->aempty[ab], 3);
                    else
                        ptx::umma_commit(&sh->aempty[ab]);
                }
                __syncwarp();
            }
        }
    } else if (warp >= EPI_WARP0) {
        // ------------------------------------------------------------------ filter epilogue (every CTA)
        ptx::setmaxnreg_inc<232>();
        EpiArgs ea{units, *n_units_p, k, pw, margin_scale, a_norms, b_norms, a_total, b_total, part_key, part_idx,
                   part_cnt, row_flags, reinterpret_cast<uint2*>(cand_key_buf), gthr, row_map, row_div, a_row_scale, b_scale, hot};
        epilogue_run<L2, PAIR, true, A2>(ea, sh->tfull, sh->tempty, sh->nrm, &sh->xchg, tmem_base, warp, lane, rank);
    }

    ptx::tcgen05_fence_before();
    if (PAIR) {
        __syncwarp();
        ptx::cluster_sync_all();
    } else {
        __syncthreads();
    }
    if (warp == 1) {
        ptx::tcgen05_fence_after();
        if (PAIR)
            ptx::tmem_dealloc_cg2(tmem_base, TMEM_COLS);
        else
            ptx::tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

#define NRB_TC3_PARAMS                                                                                              \
    const __grid_constant__ CUtensorMap map_ah, const __grid_constant__ CUtensorMap map_bh,                         \
        const Unit *__restrict__ units, const int *__restrict__ n_units_p, int nkc, int k, int pw, float margin_scale, \
        const float *__restrict__ a_norms, const float *__restrict__ b_norms, int64_t a_total, int64_t b_total,    \
        float *__restrict__ part_key, int *__restrict__ part_idx, int *__restrict__ part_cnt,                      \
        int *__restrict__ row_flags,                                                                               \
        float *__restrict__ cand_key_buf, int *__restrict__ cand_idx_buf, unsigned *__restrict__ gthr,             \
        const float *__restrict__ a_row_scale, float b_scale, const int *__restrict__ row_map, int row_div, int hot
#define NRB_TC3_ARGS                                                                                                  \
    map_ah, map_bh, units, n_units_p, nkc, k, pw, margin_scale, a_norms, b_norms, a_total, b_total, part_key, part_idx, \
        part_cnt, row_flags, cand_key_buf, cand_idx_buf, gthr, a_row_scale, b_scale, row_map, row_div, hot

template <bool L2, bool F16>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1) topk_tc3_kernel(NRB_TC3_PARAMS) {
    tc3_body<L2, F16, true>(NRB_TC3_ARGS);
}

// fp16 CTA pairs with two resident query tiles (IVF list scan: short units)
template <bool L2>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1) topk_tc3d_kernel(NRB_TC3_PARAMS) {
    tc3_body<L2, true, true, true>(NRB_TC3_ARGS);
}

// single-CTA form (fp16 planes only)
template <bool L2>
__global__ void __launch_bounds__(NUM_THREADS, 1) topk_tc3s_kernel(NRB_TC3_PARAMS) {
    tc3_body<L2, true, false>(NRB_TC3_ARGS);
}

// ---------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) != cudaSuccess ||
            qr != cudaDriverEntryPointSuccess)
            return nullptr;
        fn = (EncodeTiledFn)p;
    }
    return fn;
}

// Tensor map over a [rows, kp] fp32 plane, box = KC columns x box_rows rows, 128-byte swizzle.
int make_plane_map(CUtensorMap* m, const float* base, int64_t rows, int kp, int box_rows) {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) {
        set_error("cuTensorMapEncodeTiled not available from the driver");
        return NRB_ERR_CUDA;
    }
    cuuint64_t gdim[2] = {(cuuint64_t)kp, (cuuint64_t)(rows > 0 ? rows : 1)};
    cuuint64_t gstr[1] = {(cuuint64_t)kp * sizeof(float)};
    cuuint32_t box[2] = {(cuuint32_t)KC, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, gdim, gstr, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed: CUresult %d (rows=%lld kp=%d)", (int)r, (long long)rows, kp);
        return NRB_ERR_CUDA;
    }
    return NRB_OK;
}

// Tensor map over a [rows, kp] fp16 plane: box = 64 columns (128 bytes) x box_rows rows, 128-byte
// swizzle; a last chunk that sticks out of the row (kp % 64 != 0) is zero-filled by TMA.
int make_plane_map_h16(CUtensorMap* m, const void* base, int64_t rows, int kp, int box_rows) {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) {
        set_error("cuTensorMapEncodeTiled not available from the driver");
        return NRB_ERR_CUDA;
    }
    cuuint64_t gdim[2] = {(cuuint64_t)kp, (cuuint64_t)(rows > 0 ? rows : 1)};
    cuuint64_t gstr[1] = {(cuuint64_t)kp * 2};
    cuuint32_t box[2] = {(cuuint32_t)(2 * KC), (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, (void*)base, gdim, gstr, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled (fp16) failed: CUresult %d (rows=%lld kp=%d)", (int)r, (long long)rows, kp);
        return NRB_ERR_CUDA;
    }
    return NRB_OK;
}

}  // namespace

int tc_available() {
    // cudaGetDeviceProperties costs milliseconds: query the one attribute, once per device.
    static int cached[64] = {0};  // 0 unknown, 1 yes, -1 no
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 0;
    if (dev >= 0 && dev < 64 && cached[dev] != 0) return cached[dev] > 0;
    int major = 0;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return 0;
    if (dev >= 0 && dev < 64) cached[dev] = major == 10 ? 1 : -1;
    return major == 10 ? 1 : 0;
}

int tc_grid(int n_units) {
    int g = sm_count() & ~1;  // whole CTA pairs
    int need = (n_units + 1) & ~1;
    if (need > 0 && need < g) g = need;
    return g < 2 ? 2 : g;
}

size_t tc_scratch_bytes(int grid) {
    return (size_t)grid * EPI_WGS * BM * CAND_CAP * (sizeof(float) + sizeof(int)) + 256;
}

int launch_topk_tc_dev(const nrb_matrix* a, const nrb_matrix* b, const Unit* units,
                       const int* n_units_dev, int grid, int metric, int k, float* part_key,
                       int* part_idx, void* scratch, size_t scratch_bytes, unsigned* gthr,
                       const int* row_map, int row_div, cudaStream_t st) {
    NRB_REQUIRE(a->hi && a->lo && b->hi && b->lo, "tc: hi/lo planes required");
    NRB_REQUIRE(a->kp == b->kp && a->kp % KC == 0 && a->kp >= KC, "tc: kp mismatch / not a multiple of %d", KC);
    NRB_REQUIRE(k >= 1 && k <= NRB_MAX_K, "tc: k=%d out of range [1,%d]", k, NRB_MAX_K);
    NRB_REQUIRE(metric != NRB_METRIC_L2 || (a->norms && b->norms), "tc: norms required for L2");
    NRB_REQUIRE(grid >= 2 && grid % 2 == 0, "tc: grid must be a positive even number");
    if (scratch_bytes < tc_scratch_bytes(grid)) {
        set_error("tc: scratch too small");
        return NRB_ERR_WORKSPACE;
    }
    CUtensorMap mah, mal, mbh, mbl;
    int rc;
    if ((rc = make_plane_map(&mah, a->hi, a->n, a->kp, BM))) return rc;
    if ((rc = make_plane_map(&mal, a->lo, a->n, a->kp, BM))) return rc;
    if ((rc = make_plane_map(&mbh, b->hi, b->n, b->kp, BN / 2))) return rc;
    if ((rc = make_plane_map(&mbl, b->lo, b->n, b->kp, BN / 2))) return rc;
    float* ck = (float*)scratch;
    int* ci = (int*)((char*)scratch + (size_t)grid * EPI_WGS * BM * CAND_CAP * sizeof(float));
    const int nkc = a->kp / KC;
#define NRB_TC_LAUNCH(KERNEL, SMEM)                                                                          \
    do {                                                                                                     \
        NRB_CUDA_CHECK(cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(SMEM))); \
        KERNEL<<<grid, NUM_THREADS, SMEM, st>>>(mah, mal, mbh, mbl, units, n_units_dev, nkc, k, a->norms,     \
                                                b->norms, a->n, b->n, part_key, part_idx, ck, ci, gthr,     \
                                                row_map, row_div);                                           \
    } while (0)
    if (metric == NRB_METRIC_L2)
        NRB_TC_LAUNCH(topk_tc2_kernel<true>, V2_SMEM);
    else
        NRB_TC_LAUNCH(topk_tc2_kernel<false>, V2_SMEM);
#undef NRB_TC_LAUNCH
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

int tc1_eligible(const nrb_matrix* a, const nrb_matrix* b, int k) {
    return a->hi && b->hi && a->raw && b->raw && a->norms && b->norms && b->max_norm > 0.f &&
           a->kp == b->kp && a->kp <= V3_MAX_NKC * KC && tc1_k_ok(k);
}

int tc16_eligible(const nrb_matrix* a, const nrb_matrix* b, int k) {
    return a->h16 && a->h16_row_scale && b->h16 && b->h16_scale > 0.f && a->raw && b->raw && a->norms &&
           b->norms && b->max_norm > 0.f && a->kp == b->kp && a->kp <= V3_MAX_NKC * KC && tc1_k_ok(k);
}

int launch_topk_tc1_dev(const nrb_matrix* a, const nrb_matrix* b, const Unit* units,
                        const int* n_units_dev, int grid, int metric, int k, int pw, float margin_scale,
                        float* part_key, int* part_idx, int* part_cnt, int* row_flags, void* scratch,
                        size_t scratch_bytes, unsigned* gthr, const int* row_map, int row_div, int f16,
                        int single, int ivf_mode, cudaStream_t st) {
    const int hot = ivf_mode == 2 ? 1 : 0;  // IVF phase B: rows start from their query's shared bound
    NRB_REQUIRE(part_cnt, "tc1: part_cnt required (the filter kernels write unsorted partial rows)");
    NRB_REQUIRE(!single || f16, "tc1: the single-CTA form exists for the fp16 planes only");
    // what the KERNEL reads (the raw planes are the refine stage's business: *_eligible)
    if (f16)
        NRB_REQUIRE(a->h16 && a->h16_row_scale && b->h16 && b->h16_scale > 0.f, "tc16: scaled fp16 planes required");
    else
        NRB_REQUIRE(a->hi && b->hi, "tc1: hi planes required");
    NRB_REQUIRE(a->norms && b->norms && a->kp == b->kp && a->kp <= V3_MAX_NKC * KC && tc1_k_ok(k) && row_div >= 1,
                "tc1: norms on both sides, kp <= 256 and k <= %d required", TC1_MAX_PW - TC1_MIN_EXTRA);
    NRB_REQUIRE(a->kp % KC == 0 && pw >= k && pw <= CAND_CAP - HALF_N, "tc1: bad kp / pw");
    NRB_REQUIRE(grid >= 1 && (single || grid % 2 == 0), "tc1: grid must be positive (and even for CTA pairs)");
    if (scratch_bytes < tc_scratch_bytes(grid)) {
        set_error("tc1: scratch too small");
        return NRB_ERR_WORKSPACE;
    }
#ifdef NRB_TRACE
    {
        const char* e = getenv("NRB_TRACE_IVF_MODE");
        const int en = (!e || atoi(e) == ivf_mode) ? 1 : 0;
        NRB_CUDA_CHECK(cudaMemcpyToSymbolAsync(g_trace_enable, &en, sizeof(int), 0, cudaMemcpyHostToDevice, st));
    }
#endif
    CUtensorMap mah, mbh;
    int rc;
    if (f16) {
        if ((rc = make_plane_map_h16(&mah, a->h16, a->n, a->kp, BM))) return rc;
        if ((rc = make_plane_map_h16(&mbh, b->h16, b->n, b->kp, single ? BN : BN / 2))) return rc;
    } else {
        if ((rc = make_plane_map(&mah, a->hi, a->n, a->kp, BM))) return rc;
        if ((rc = make_plane_map(&mbh, b->hi, b->n, b->kp, BN / 2))) return rc;
    }
    float* ck = (float*)scratch;
    int* ci = (int*)((char*)scratch + (size_t)grid * EPI_WGS * BM * CAND_CAP * sizeof(float));
    const int nkc = f16 ? (a->kp + 2 * KC - 1) / (2 * KC) : a->kp / KC;
    const float* ars = f16 ? a->h16_row_scale : nullptr;
    const float bsc = f16 ? b->h16_scale : 1.f;
#define NRB_TC3_LAUNCH(L2V, F16V)                                                                                   \
    do {                                                                                                            \
        NRB_CUDA_CHECK(cudaFuncSetAttribute(topk_tc3_kernel<L2V, F16V>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                            (int)v3_smem<F16V>()));                                                 \
        topk_tc3_kernel<L2V, F16V><<<grid, NUM_THREADS, v3_smem<F16V>(), st>>>(mah, mbh, units, n_units_dev, nkc, k, pw,      \
                                                                      margin_scale, a->norms, b->norms, a->n, b->n, \
                                                                      part_key, part_idx, part_cnt, row_flags, ck, ci, gthr,  \
                                                                      ars, bsc, row_map, row_div, hot);             \
    } while (0)
    if (ivf_mode != 0 && f16 && !single) {
        // IVF list scan: short units -> two resident query tiles
        constexpr size_t SM2 = Tc3Lay<true, true, true>::SMEM;
        if (metric == NRB_METRIC_L2) {
            NRB_CUDA_CHECK(cudaFuncSetAttribute(topk_tc3d_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SM2));
            topk_tc3d_kernel<true><<<grid, NUM_THREADS, SM2, st>>>(mah, mbh, units, n_units_dev, nkc, k, pw, margin_scale,
                                                                   a->norms, b->norms, a->n, b->n, part_key, part_idx,
                                                                   part_cnt, row_flags, ck, ci, gthr, ars, bsc, row_map, row_div, hot);
        } else {
            NRB_CUDA_CHECK(cudaFuncSetAttribute(topk_tc3d_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SM2));
            topk_tc3d_kernel<false><<<grid, NUM_THREADS, SM2, st>>>(mah, mbh, units, n_units_dev, nkc, k, pw, margin_scale,
                                                                    a->norms, b->norms, a->n, b->n, part_key, part_idx,
                                                                    part_cnt, row_flags, ck, ci, gthr, ars, bsc, row_map, row_div, hot);
        }
    } else if (single) {
        constexpr size_t SM1 = Tc3Lay<true, false>::SMEM;
        if (metric == NRB_METRIC_L2) {
            NRB_CUDA_CHECK(cudaFuncSetAttribute(topk_tc3s_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SM1));
            topk_tc3s_kernel<true><<<grid, NUM_THREADS, SM1, st>>>(mah, mbh, units, n_units_dev, nkc, k, pw, margin_scale,
                                                                   a->norms, b->norms, a->n, b->n, part_key, part_idx,
                                                                   part_cnt, row_flags, ck, ci, gthr, ars, bsc, row_map, row_div, hot);
        } else {
            NRB_CUDA_CHECK(cudaFuncSetAttribute(topk_tc3s_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SM1));
            topk_tc3s_kernel<false><<<grid, NUM_THREADS, SM1, st>>>(mah, mbh, units, n_units_dev, nkc, k, pw, margin_scale,
                                                                    a->norms, b->norms, a->n, b->n, part_key, part_idx,
                                                                    part_cnt, row_flags, ck, ci, gthr, ars, bsc, row_map, row_div, hot);
        }
    } else if (metric == NRB_METRIC_L2) {
        if (f16)
            NRB_TC3_LAUNCH(true, true);
        else
            NRB_TC3_LAUNCH(true, false);
    } else {
        if (f16)
            NRB_TC3_LAUNCH(false, true);
        else
            NRB_TC3_LAUNCH(false, false);
    }
#undef NRB_TC3_LAUNCH
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

}  // namespace nrb

#ifdef NRB_TRACE
// Debug builds only (not part of include/nrb200.h): copies the timeline trace to the host.
extern "C" int nrb_debug_trace_read(void* host_buf, size_t bytes) {
    const size_t have = sizeof(long long) * 9 * nrb::NRB_TRACE_TILES * 4;
    if (bytes < have) return -1;
    if (cudaDeviceSynchronize() != cudaSuccess) return -2;
    return cudaMemcpyFromSymbol(host_buf, nrb::g_trace, have) == cudaSuccess ? 0 : -2;
}
extern "C" int nrb_debug_trace_prune_read(void* host_buf, size_t bytes, int reset) {
    const size_t have = sizeof(long long) * 9 * 64 * 4;
    if (bytes < have) return -1;
    if (cudaDeviceSynchronize() != cudaSuccess) return -2;
    if (cudaMemcpyFromSymbol(host_buf, nrb::g_trace_prune, have) != cudaSuccess) return -2;
    if (reset) {
        int z[9] = {0};
        cudaMemcpyToSymbol(nrb::g_trace_prune_n, z, sizeof(z));
    }
    return 0;
}
#endif
