// extern "C" entry points of libnrb200 (declared in include/nrb200.h) that orchestrate several
// kernels: exact flat top-k and the IVF list scan. Also error plumbing and the host-side RNG
// pieces of k-means.
#include <atomic>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <random>
#include <vector>

#include <cuda_fp16.h>

#include "common.cuh"
#include "internal.h"

namespace nrb {

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
void count_launch(int n) { g_launches += n; }

int sm_count() {
    static int cached = -1;
    if (cached < 0) {
        int dev = 0, n = 0;
        if (cudaGetDevice(&dev) == cudaSuccess &&
            cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
            cached = n;
        else
            return 148;
    }
    return cached;
}

int require_device() {
    static int n = -1;
    if (n <= 0 && (cudaGetDeviceCount(&n) != cudaSuccess || n == 0)) {
        n = 0;
        cudaGetLastError();
        set_error("no CUDA device: libnrb200 has no CPU fallback");
        return NRB_ERR_NO_DEVICE;
    }
    if (!tc_available()) {
        set_error("current device is not sm_100: libnrb200 is built for B200 (sm_100a) only");
        return NRB_ERR_NO_DEVICE;
    }
    return NRB_OK;
}

// Bump allocator over the caller's workspace.
struct Carver {
    char* base;
    size_t off = 0;
    explicit Carver(void* p) : base((char*)p) {}
    template <typename T>
    T* take(size_t count) {
        T* r = (T*)(base ? base + off : nullptr);
        off += align_up(count * sizeof(T), 256);
        return r;
    }
};

// ------------------------------------------------------------------------------ flat plan
// Query tiles (128 rows) are taken in PAIRS (the CTA-pair kernels need units 2p, 2p+1 to share
// their item rows). With P pairs and C concurrently resident CTA pairs:
//   * the first R = floor(P / C) * C pairs are FULL units: one pass over the whole catalog, so
//     the running top-k threshold warms up once (appends and prunes grow with log(items), a
//     catalog split s ways pays the warm-up s times);
//   * the remaining T = P - R pairs are TAIL units, split s ways over the item rows (s chosen
//     so that T*s fills whole waves), ordered chunk-major so that concurrent CTAs stream the
//     same item rows.
// Every query therefore has S = max(1, s) source slots per epilogue warpgroup.
struct FlatPlan {
    int nqt;         // query tiles
    int npairs;      // ceil(nqt / 2)
    int full_pairs;  // R
    int tail_pairs;  // T
    int tsplit;      // s (>= 1)
    int chunk_rows;  // item rows per tail chunk (multiple of 256)
    int n_units;     // 2 * (R + T * s)
    int wgs;         // epilogue warpgroups writing partial rows (2 for the tcgen05 kernels)
    int S;           // source slots per query = tsplit * wgs
    int grid;
    int single;      // 1: single-CTA units (fp16 filter, one partial wave): unit c*nqt + t, no phantoms
    int pw;          // partial row width of the filter paths: k + margin slots (wide rows for catalogs beyond a few tiles)
};

static FlatPlan plan_flat(int64_t nq, int64_t nb, int k, int path) {
    FlatPlan p;
    // searches over a real catalog take the widest margin set the refine stage can hold (near-duplicate
    // tolerance); the <= 4096-row searches (coarse quantizer, nearest centroid) keep the narrow rows
    p.pw = (path == NRB_PATH_TC1 || path == NRB_PATH_TC16) ? tc1_pw(k, nb > 4096) : k;
    const bool simt = path == NRB_PATH_SIMT;
    p.wgs = simt ? 1 : 2;
    p.nqt = (int)((nq + UNIT_ROWS - 1) / UNIT_ROWS);
    if (p.nqt < 1) p.nqt = 1;
    p.npairs = (p.nqt + 1) / 2;
    const int C = simt ? sm_count() : sm_count() / 2;  // units in flight: SIMT runs 2 CTAs per SM
    const int tile = 256;
    int nbt = (int)((nb + tile - 1) / tile);
    if (nbt < 1) nbt = 1;
    p.full_pairs = (p.npairs / C) * C;
    p.tail_pairs = p.npairs - p.full_pairs;
    // cost of a plan = waves x (chunk length + per-unit overhead), in catalogs per CTA pair (or CTA);
    // a unit costs about 200 tiles of MMA time on top of its item rows (query-tile load, the
    // append-heavy threshold warm-up and its prunes, 32 final sorts per warp; measured by sweeping
    // that overhead on config 1), which is what stops small batches from being cut into dozens of
    // slivers
    const double ov = 200.0 / nbt;
    int best = 1;
    if (p.tail_pairs > 0) {
        int max_split = nbt < 64 ? nbt : 64;
        double best_cost = 1e30;
        for (int s = 1; s <= max_split; s++) {
            const double waves = (double)(((int64_t)p.tail_pairs * s + C - 1) / C);
            const double cost = waves * (1.0 / s + ov);
            if (cost < best_cost * 0.97) {  // prefer fewer splits unless >3% better
                best_cost = cost;
                best = s;
            }
        }
    }
    p.single = 0;
    // One partial wave of the fp16 filter: single-CTA units (one query tile each, no phantom
    // tile, 148 slots instead of 74) can sometimes be cut one step finer than CTA pairs, e.g.
    // 49 tiles x 3 chunks = 147 units where 25 pairs stop at 2 chunks. CTA pairs halve the L2
    // traffic per unit of work, so they stay unless the single-CTA plan is clearly shorter.
    // (catalogs of one tile -- coarse quantizers -- go to the CTA-pair short-unit kernel instead)
    if (path == NRB_PATH_TC16 && p.full_pairs == 0 && p.nqt <= sm_count() && nb > 256) {
        const int C1 = sm_count();
        const int max_split = nbt < 64 ? nbt : 64;
        const double pair_cost = (double)(((int64_t)p.tail_pairs * best + C - 1) / C) * (1.0 / best + ov);
        int best1 = 1;
        double best_cost1 = 1e30;
        for (int s = 1; s <= max_split; s++) {
            const double waves = (double)(((int64_t)p.nqt * s + C1 - 1) / C1);
            const double cost = waves * (1.0 / s + ov);
            if (cost < best_cost1 * 0.97) {
                best_cost1 = cost;
                best1 = s;
            }
        }
        if (best_cost1 < 0.9 * pair_cost || getenv("NRB_FORCE_SINGLE_CTA")) {  // (the override is for tests)
            p.single = 1;
            best = best1;
        }
    }
    const int tiles_per = (nbt + best - 1) / best;
    p.chunk_rows = tiles_per * tile;
    p.tsplit = (nbt + tiles_per - 1) / tiles_per;
    p.n_units = p.single ? p.nqt * p.tsplit : 2 * (p.full_pairs + p.tail_pairs * p.tsplit);
    p.S = p.tsplit * p.wgs;
    if (p.single)
        p.grid = p.n_units < sm_count() ? p.n_units : sm_count();
    else
        p.grid = simt ? simt_grid(p.n_units) : tc_grid(p.n_units);
    return p;
}

struct FlatWs {
    Unit* units;
    int* n_units;
    int* src;
    float* part_key;
    int* part_idx;
    int* part_cnt;                        // filter paths: entries per (unsorted) partial row
    int *flags, *flag_list, *flag_count;  // filter paths only
    unsigned* gthr;                       // per-query shared bounds (tcgen05 paths)
    void* scratch;
    size_t scratch_bytes;
    size_t total;
};

static FlatWs carve_flat(void* ws, const FlatPlan& p, int64_t nq, int k, int path) {
    Carver c(ws);
    FlatWs w;
    const bool filt = path == NRB_PATH_TC1 || path == NRB_PATH_TC16;
    const int pw = p.pw;  // partial row width
    w.units = c.take<Unit>(p.n_units);
    w.n_units = c.take<int>(1);
    w.src = c.take<int>((size_t)nq * p.S);
    w.part_key = c.take<float>((size_t)p.n_units * p.wgs * UNIT_ROWS * pw);
    w.part_idx = c.take<int>((size_t)p.n_units * p.wgs * UNIT_ROWS * pw);
    w.flags = w.flag_list = w.flag_count = w.part_cnt = nullptr;
    w.gthr = path == NRB_PATH_SIMT ? nullptr : c.take<unsigned>(nq);
    if (filt) {
        w.part_cnt = c.take<int>((size_t)p.n_units * p.wgs * UNIT_ROWS);
        w.flags = c.take<int>(nq);
        w.flag_list = c.take<int>(nq);
        w.flag_count = c.take<int>(1);
    }
    w.scratch_bytes = path == NRB_PATH_SIMT ? simt_scratch_bytes(p.grid) : tc_scratch_bytes(p.grid);
    w.scratch = c.take<char>(w.scratch_bytes);
    w.total = c.off;
    return w;
}

// Optional device-side timing of the dominant kernel (bench.py's roofline leg): CUDA events on
// the launching stream around every distance+selection launch.
static bool g_profile = false;
static std::vector<std::pair<cudaEvent_t, cudaEvent_t>> g_prof_events;

struct ProfScope {
    cudaStream_t st;
    cudaEvent_t e1 = nullptr;
    explicit ProfScope(cudaStream_t s) : st(s) {
        if (!g_profile) return;
        cudaEvent_t e0;
        if (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess) {
            e1 = nullptr;
            return;
        }
        cudaEventRecord(e0, st);
        g_prof_events.emplace_back(e0, e1);
    }
    ~ProfScope() {
        if (e1) cudaEventRecord(e1, st);
    }
};

static int resolve_path(int path) { return path == NRB_PATH_SIMT ? NRB_PATH_SIMT : NRB_PATH_TC; }

// The fallback of the filter paths (a handful of flagged queries recomputed by the 3xTF32 pipeline)
// takes its scratch from the stream-ordered allocator. The device's default memory pool releases
// freed memory back to the OS at the next synchronisation (release threshold 0), so every search with
// even ONE flagged query paid ~10 ms for mapping ~100 MB again (measured: scripts/bench_robustness.py,
// 16 copies per article: 19 ms per 50,000 queries of which 9 ms kernels). Keep the pool's memory.
static void keep_pool_memory() {
    static bool done[64] = {false};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64 || done[dev]) return;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        uint64_t thr = UINT64_MAX;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    cudaGetLastError();
    done[dev] = true;
}

static std::atomic<long long> g_fallback_queries{0};

// ------------------------------------------------------------------------------ IVF grouping
// The scan runs in up to two PHASES, each with its own grouping of (query, list) pairs by list:
//   phase A: every query's closest list (coarse rank 0), cold start -- it ends with the k-th best
//            of that list in the query's shared running bound gthr[query];
//   phase B: the other nprobe - 1 lists, which start from that bound: nearly every 32-column
//            chunk is skipped by the first compare, rows end with a handful of candidates and
//            need no prune at all.
// (One pass over all nprobe lists in list order gave every (query, list) row its own cold start:
// per-unit prunes and sorts, not the tensor pipe, bounded the scan.)

// Single block: per list, the number of (query, list) pairs m_l, query tiles (padded to an even
// count so that units 2p, 2p+1 share their item rows), item-run splits and the first unit
// index; writes the unit list ordered (list, split, tile) with the lists taken LONGEST FIRST:
// persistent CTAs take units round-robin, so a descending cost order balances them, and units of
// one list stay adjacent (concurrent CTAs stream the same item rows through L2).
__global__ void ivf_plan_kernel(const int* __restrict__ p_off, const int* __restrict__ l_off, int nlist,
                                int chunk, int* __restrict__ ubase, int* __restrict__ nsl,
                                int* __restrict__ n_units_out, Unit* __restrict__ units, int max_units) {
    extern __shared__ int sh_plan[];  // cnt[nlist + 1], perm[nlist]
    int* cnt = sh_plan;
    int* perm = sh_plan + nlist + 1;
    for (int l = threadIdx.x; l < nlist; l += blockDim.x) {
        const int m = p_off[l + 1] - p_off[l];
        const int len = l_off[l + 1] - l_off[l];
        const int tiles2 = (((m + UNIT_ROWS - 1) / UNIT_ROWS) + 1) & ~1;
        const int ns = (m > 0 && len > 0) ? (len + chunk - 1) / chunk : 0;
        nsl[l] = ns;
        cnt[l] = tiles2 * ns;
        int rank = l;
        if (nlist <= 2048) {  // rank sort by list length, descending (ties: list id)
            rank = 0;
            for (int o = 0; o < nlist; o++) {
                const int lo = l_off[o + 1] - l_off[o];
                rank += (lo > len || (lo == len && o < l)) ? 1 : 0;
            }
        }
        perm[rank] = l;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int run = 0;
        for (int r = 0; r < nlist; r++) {
            const int l = perm[r];
            const int t = cnt[l];
            cnt[l] = run;
            run += t;
        }
        cnt[nlist] = run;
        *n_units_out = run < max_units ? (run & ~1) : (max_units & ~1);
    }
    __syncthreads();
    for (int l = threadIdx.x; l <= nlist; l += blockDim.x) ubase[l] = cnt[l];
    for (int l = threadIdx.x; l < nlist; l += blockDim.x) {
        const int m = p_off[l + 1] - p_off[l];
        const int len = l_off[l + 1] - l_off[l];
        const int ns = nsl[l];
        if (ns == 0) continue;
        const int tiles = (m + UNIT_ROWS - 1) / UNIT_ROWS;
        const int tiles2 = (tiles + 1) & ~1;
        int u = cnt[l];
        for (int sp = 0; sp < ns; sp++)
            for (int t = 0; t < tiles2; t++, u++) {
                if (u >= max_units) continue;
                Unit un;
                un.a_row0 = t < tiles ? p_off[l] + t * UNIT_ROWS : 0;
                un.a_rows = t < tiles ? min(UNIT_ROWS, m - t * UNIT_ROWS) : 0;
                un.b_row0 = l_off[l] + sp * chunk;
                un.b_rows = min(chunk, len - sp * chunk);
                units[u] = un;
            }
    }
}

// Pair e = q*ncols + j of a phase (list coarse[e]): src[q*S + s_off + (j*maxsplit + sp)*wgs + g] =
// partial row of the pair in split sp, warpgroup g (prow_base + local partial row), or -1.
__global__ void ivf_src_kernel(const int64_t* __restrict__ coarse, const int* __restrict__ pos_of,
                               const int* __restrict__ p_off, const int* __restrict__ ubase,
                               const int* __restrict__ nsl, int nlist, int64_t npairs, int ncols, int maxsplit,
                               int wgs, int S, int s_off, int prow_base, int* __restrict__ src) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < npairs;
         e += (int64_t)gridDim.x * blockDim.x) {
        const int pos = pos_of[e];
        const int64_t l = coarse[e];
        int ns = 0, u0 = 0, r = 0, tiles2 = 0;
        if (pos >= 0 && l >= 0 && l < nlist) {
            ns = nsl[l];
            const int i = pos - p_off[l];
            const int m = p_off[l + 1] - p_off[l];
            tiles2 = (((m + UNIT_ROWS - 1) / UNIT_ROWS) + 1) & ~1;
            u0 = ubase[l] + i / UNIT_ROWS;
            r = i % UNIT_ROWS;
        }
        const int64_t q = e / ncols;
        const int j = (int)(e - q * ncols);
        int* dst = src + q * S + s_off + (int64_t)j * maxsplit * wgs;
        // partial row of (unit u, warpgroup g, row r) = (u*wgs + g)*128 + r
        for (int sp = 0; sp < maxsplit; sp++)
            for (int g = 0; g < wgs; g++)
                dst[sp * wgs + g] = (sp < ns) ? prow_base + ((u0 + sp * tiles2) * wgs + g) * UNIT_ROWS + r : -1;
    }
}

// coarse i64[nq, nprobe] -> ca[nq] (rank 0) and cb[nq, nprobe - 1] (the rest)
__global__ void ivf_split_coarse_kernel(const int64_t* __restrict__ coarse, int64_t nq, int nprobe,
                                        int64_t* __restrict__ ca, int64_t* __restrict__ cb) {
    const int64_t total = nq * nprobe;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t q = t / nprobe;
        const int j = (int)(t - q * nprobe);
        if (j == 0)
            ca[q] = coarse[t];
        else
            cb[q * (nprobe - 1) + (j - 1)] = coarse[t];
    }
}

// item rows per unit inside one list: long runs amortise the per-unit work (sweep on config 2:
// 4,096 -> 40.4 ms, 8,192 -> 36.2, 16,384 -> 35.4, 32,768 -> 33.8); NRB_IVF_CHUNK overrides
static int ivf_chunk() {
    const char* e = getenv("NRB_IVF_CHUNK");  // read per call: tests force small runs to cover split lists
    const int v = e ? atoi(e) : 32768;
    return v >= 256 ? (v + 255) / 256 * 256 : 32768;
}

constexpr int IVF_MAX_SOURCES = 256;  // partial rows per query the sorted merge can take (select_merge_kernel<8>)

struct IvfPhase {
    int ncols;  // lists of every query handled by this phase
    int64_t npairs;
    int max_units, grid, s_off, prow_base;
};

struct IvfPlan {
    int chunk, maxsplit, wgs, S, nph;
    IvfPhase ph[2];
    int64_t total_units;
};

static IvfPlan plan_ivf(int64_t nq, int nprobe, int nlist, int max_list_len, int path) {
    IvfPlan p;
    p.wgs = path == NRB_PATH_SIMT ? 1 : 2;
    // long lists are cut into runs of `chunk` rows; the run length grows until the partial rows of a
    // query (nprobe x splits x warpgroups) fit the merge (a 10M-row catalog with one list of 70k rows
    // and nprobe 64 used to be refused)
    p.chunk = ivf_chunk();
    p.maxsplit = 1;
    for (;;) {
        p.maxsplit = (max_list_len + p.chunk - 1) / p.chunk;
        if (p.maxsplit < 1) p.maxsplit = 1;
        if ((int64_t)nprobe * p.maxsplit * p.wgs <= IVF_MAX_SOURCES || p.maxsplit == 1) break;
        p.chunk *= 2;
    }
    p.S = nprobe * p.maxsplit * p.wgs;
    // the SIMT kernels keep no shared running bounds: one phase
    p.nph = (nprobe > 1 && path != NRB_PATH_SIMT) ? 2 : 1;
    p.total_units = 0;
    for (int i = 0; i < p.nph; i++) {
        IvfPhase& f = p.ph[i];
        f.ncols = p.nph == 1 ? nprobe : (i == 0 ? 1 : nprobe - 1);
        f.npairs = nq * f.ncols;
        f.max_units = (int)((f.npairs / UNIT_ROWS + 2 * (int64_t)nlist) * p.maxsplit);
        f.grid = path == NRB_PATH_SIMT ? simt_grid(f.max_units) : tc_grid(f.max_units);
        f.s_off = i == 0 ? 0 : p.ph[0].ncols * p.maxsplit * p.wgs;
        f.prow_base = (int)(p.total_units * p.wgs * UNIT_ROWS);
        p.total_units += f.max_units;
    }
    return p;
}

struct IvfPhaseWs {
    void* cs;
    size_t cs_bytes;
    int64_t* coarse;  // this phase's columns of the coarse assignment, contiguous (two phases only)
    int *p_off, *order, *pos_of, *ubase, *nsl, *n_units;
    Unit* units;
    float *g_raw, *g_hi, *g_lo, *g_norms;
    void* g_h16;     // fp16 filter: regrouped scaled fp16 query rows ...
    float* g_scale;  // ... and their per-row scales
};

struct IvfWs {
    IvfPhaseWs ph[2];
    int* src;
    unsigned* gthr;
    float* part_key;
    int *part_idx, *part_cnt;
    int *flags, *flag_list, *flag_count;
    void* scratch;
    size_t scratch_bytes, total;
};

static IvfWs carve_ivf(void* ws, const IvfPlan& p, int nlist, int k, int kp, int path, int64_t nq) {
    Carver c(ws);
    IvfWs w;
    const bool filt = path == NRB_PATH_TC16;
    const int pw = filt ? tc1_pw(k) : k;  // partial row width
    w.gthr = path == NRB_PATH_SIMT ? nullptr : c.take<unsigned>(nq);
    w.src = c.take<int>((size_t)nq * p.S);
    int max_grid = 0;
    for (int i = 0; i < p.nph; i++) {
        const IvfPhase& f = p.ph[i];
        IvfPhaseWs& v = w.ph[i];
        v.cs_bytes = counting_sort_ws(f.npairs, nlist);
        v.cs = c.take<char>(v.cs_bytes);
        v.coarse = p.nph > 1 ? c.take<int64_t>(f.npairs) : nullptr;
        v.p_off = c.take<int>(nlist + 2);
        v.order = c.take<int>(f.npairs);
        v.pos_of = c.take<int>(f.npairs);
        v.ubase = c.take<int>(nlist + 1);
        v.nsl = c.take<int>(nlist);
        v.n_units = c.take<int>(1);
        v.units = c.take<Unit>(f.max_units);
        const size_t plane = (size_t)(f.npairs + UNIT_ROWS) * kp;
        v.g_raw = v.g_hi = v.g_lo = v.g_scale = nullptr;
        v.g_h16 = nullptr;
        if (path == NRB_PATH_SIMT) {
            v.g_raw = c.take<float>(plane);
        } else if (filt) {
            v.g_h16 = c.take<uint16_t>(plane);
            v.g_scale = c.take<float>(f.npairs + UNIT_ROWS);
        } else {
            v.g_hi = c.take<float>(plane);
            v.g_lo = c.take<float>(plane);
        }
        v.g_norms = c.take<float>(f.npairs + UNIT_ROWS);
        max_grid = f.grid > max_grid ? f.grid : max_grid;
    }
    w.flags = w.flag_list = w.flag_count = w.part_cnt = nullptr;
    if (filt) {
        w.part_cnt = c.take<int>((size_t)p.total_units * p.wgs * UNIT_ROWS);
        w.flags = c.take<int>(nq);
        w.flag_list = c.take<int>(nq);
        w.flag_count = c.take<int>(1);
    }
    w.part_key = c.take<float>((size_t)p.total_units * p.wgs * UNIT_ROWS * pw);
    w.part_idx = c.take<int>((size_t)p.total_units * p.wgs * UNIT_ROWS * pw);
    w.scratch_bytes = path == NRB_PATH_SIMT ? simt_scratch_bytes(max_grid) : tc_scratch_bytes(max_grid);
    w.scratch = c.take<char>(w.scratch_bytes);
    w.total = c.off;
    return w;
}

}  // namespace nrb

using namespace nrb;

extern "C" int nrb_version(void) { return 100; }

extern "C" int nrb_last_error(char* buf, int buflen) {
    if (!buf || buflen <= 0) return NRB_ERR_INVALID;
    strncpy(buf, g_err, buflen - 1);
    buf[buflen - 1] = 0;
    return NRB_OK;
}

extern "C" int nrb_device_info(int* sms, int* cc_major, int* cc_minor) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
        cudaGetLastError();
        set_error("no CUDA device");
        return NRB_ERR_NO_DEVICE;
    }
    int dev = 0;
    NRB_CUDA_CHECK(cudaGetDevice(&dev));
    cudaDeviceProp p;
    NRB_CUDA_CHECK(cudaGetDeviceProperties(&p, dev));
    if (sms) *sms = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    return NRB_OK;
}

extern "C" int nrb_profile_enable(int on) {
    g_profile = on != 0;
    return NRB_OK;
}

extern "C" int nrb_profile_read(double* total_ms, int* n_launches) {
    double tot = 0;
    int n = 0;
    for (auto& pr : g_prof_events) {
        float ms = 0;
        if (cudaEventSynchronize(pr.second) == cudaSuccess &&
            cudaEventElapsedTime(&ms, pr.first, pr.second) == cudaSuccess) {
            tot += ms;
            n++;
        }
        cudaEventDestroy(pr.first);
        cudaEventDestroy(pr.second);
    }
    g_prof_events.clear();
    if (total_ms) *total_ms = tot;
    if (n_launches) *n_launches = n;
    return NRB_OK;
}

extern "C" int64_t nrb_launch_count(void) { return (int64_t)g_launches.load(); }

extern "C" size_t nrb_search_flat_workspace(int64_t nq, int64_t nb, int32_t k, int32_t kp) {
    (void)kp;
    if (nq <= 0 || k <= 0 || k > NRB_MAX_K) return 256;
    // take the largest over the paths so that `path` can be chosen per call
    size_t best = 0;
    for (int path : {NRB_PATH_TC, NRB_PATH_SIMT, NRB_PATH_TC1, NRB_PATH_TC16}) {
        if ((path == NRB_PATH_TC1 || path == NRB_PATH_TC16) && !tc1_k_ok(k)) continue;
        FlatPlan p = plan_flat(nq, nb, k, path);
        size_t t = carve_flat(nullptr, p, nq, k, path).total;
        best = t > best ? t : best;
    }
    return best + 256;
}

namespace nrb {

static int search_flat_impl(const nrb_matrix* q, const nrb_matrix* b, int metric, int k, int64_t id_base,
                            float* D, int64_t* I, void* workspace, size_t workspace_bytes, int path,
                            cudaStream_t st) {
    if (path == NRB_PATH_AUTO)
        path = tc16_eligible(q, b, k) ? NRB_PATH_TC16 : tc1_eligible(q, b, k) ? NRB_PATH_TC1 : NRB_PATH_TC;
    if (path == NRB_PATH_TC1 && !tc1_eligible(q, b, k)) {
        set_error("search_flat: NRB_PATH_TC1 needs raw/hi/norms planes on both sides, max_norm on the item "
                  "side, kp <= 256 and k <= %d", TC1_MAX_PW - TC1_MIN_EXTRA);
        return NRB_ERR_INVALID;
    }
    if (path == NRB_PATH_TC16 && !tc16_eligible(q, b, k)) {
        set_error("search_flat: NRB_PATH_TC16 needs raw/h16/norms planes and h16 scales on both sides, max_norm on "
                  "the item side, kp <= 256 and k <= %d", TC1_MAX_PW - TC1_MIN_EXTRA);
        return NRB_ERR_INVALID;
    }
    const bool filt = path == NRB_PATH_TC1 || path == NRB_PATH_TC16;
    if (!filt) path = resolve_path(path);
    const FlatPlan p = plan_flat(q->n, b->n, k, path);
    const FlatWs w = carve_flat(workspace, p, q->n, k, path);
    if (!workspace || workspace_bytes < w.total) {
        set_error("search_flat: workspace %zu < %zu bytes", workspace_bytes, w.total);
        return NRB_ERR_WORKSPACE;
    }
    int rc;
    if (p.single)
        rc = launch_fill_flat_units_single(w.units, w.n_units, w.src, q->n, b->n, p.nqt, p.tsplit, p.chunk_rows, p.wgs, st);
    else
        rc = launch_fill_flat_units(w.units, w.n_units, w.src, q->n, b->n, p.nqt, p.full_pairs, p.tail_pairs, p.tsplit,
                                    p.chunk_rows, p.wgs, st);
    if (rc) return rc;
    if (w.gthr) {
        NRB_CUDA_CHECK(cudaMemsetAsync(w.gthr, 0, (size_t)q->n * sizeof(unsigned), st));
    }
    if (!filt) {
        {
            ProfScope prof(st);
            if (path == NRB_PATH_SIMT)
                rc = launch_topk_simt_dev(q, b, w.units, w.n_units, p.grid, metric, k, w.part_key, w.part_idx, w.scratch, w.scratch_bytes, st);
            else
                rc = launch_topk_tc_dev(q, b, w.units, w.n_units, p.grid, metric, k, w.part_key, w.part_idx, w.scratch,
                                        w.scratch_bytes, w.gthr, nullptr, 1, st);
        }
        if (rc) return rc;
        return launch_select(w.part_key, w.part_idx, w.src, p.S, q->n, k, metric, nullptr, id_base, D, I, st);
    }
    // ---- 1xTF32 / fp16 filter + exact refine, then the 3xTF32 kernel for whatever was flagged
    const int pw = p.pw;
    const float eps_xmax = TC1_EPS * b->max_norm;
    NRB_CUDA_CHECK(cudaMemsetAsync(w.flags, 0, (size_t)q->n * sizeof(int), st));
    {
        ProfScope prof(st);
        rc = launch_topk_tc1_dev(q, b, w.units, w.n_units, p.grid, metric, k, pw, 2.f * eps_xmax, w.part_key,
                                 w.part_idx, w.part_cnt, w.flags, w.scratch, w.scratch_bytes, w.gthr, nullptr, 1,
                                 path == NRB_PATH_TC16, p.single, (!p.single && b->n <= 256) ? 1 : 0,
                                 st);  // <= 256 items: every unit is one tile (coarse search, nearest centroid) -> the short-unit kernel
    }
    if (rc) return rc;
    if ((rc = launch_gather_refine(w.part_key, w.part_idx, w.part_cnt, w.src, p.S, q->n, k, pw, metric, q, b, eps_xmax,
                                   id_base, nullptr, w.flags, D, I, st))) return rc;
    if ((rc = launch_compact_flags(w.flags, q->n, w.flag_list, w.flag_count, st))) return rc;
    if (k == 1 && b->n <= K1_FALLBACK_MAX_ROWS) {
        // nearest-centroid assignment (k-means, IndexIVFFlat.add): flagged rows are recomputed exactly by
        // a kernel driven by the device-side list -- no host round trip, the call stays asynchronous
        return launch_exact_k1_fallback(q, b, metric, id_base, w.flag_list, w.flag_count, D, I, st);
    }
    int nflag = 0;
    NRB_CUDA_CHECK(cudaMemcpyAsync(&nflag, w.flag_count, sizeof(int), cudaMemcpyDeviceToHost, st));
    NRB_CUDA_CHECK(cudaStreamSynchronize(st));
    if (nflag == 0) return NRB_OK;
    NRB_REQUIRE(b->hi && b->lo && ((q->hi && q->lo) || q->raw),
                "search_flat: %d queries need the 3xTF32 fallback but the item hi/lo planes are missing", nflag);
    g_fallback_queries += nflag;
    const size_t plane = (size_t)nflag * q->kp * sizeof(float);
    const size_t wsb2 = nrb_search_flat_workspace(nflag, b->n, k, q->kp);
    char* tmp = nullptr;
    const size_t tmp_bytes = 3 * align_up(plane, 256) + align_up((size_t)nflag * 4, 256) +
                             align_up((size_t)nflag * k * 4, 256) + align_up((size_t)nflag * k * 8, 256) + wsb2;
    keep_pool_memory();
    NRB_CUDA_CHECK(cudaMallocAsync((void**)&tmp, tmp_bytes, st));
    Carver c(tmp);
    float* fhi = c.take<float>((size_t)nflag * q->kp);
    float* flo = c.take<float>((size_t)nflag * q->kp);
    float* fraw = c.take<float>((size_t)nflag * q->kp);
    float* fnr = c.take<float>(nflag);
    float* Df = c.take<float>((size_t)nflag * k);
    int64_t* If = c.take<int64_t>((size_t)nflag * k);
    void* ws2 = c.take<char>(wsb2);
    if (q->hi && q->lo) {
        rc = launch_gather_rows(q->hi, q->kp, w.flag_list, 1, nflag, fhi, st);
        if (!rc) rc = launch_gather_rows(q->lo, q->kp, w.flag_list, 1, nflag, flo, st);
    } else {
        // the filter paths pack queries without hi/lo planes: split the flagged raw rows here
        rc = launch_gather_rows(q->raw, q->kp, w.flag_list, 1, nflag, fraw, st);
        if (!rc) rc = launch_pack_rows(fraw, nflag, q->kp, q->kp, q->kp, nullptr, fhi, flo, nullptr, st);
    }
    if (!rc) rc = launch_gather_scalar(q->norms, w.flag_list, 1, nflag, fnr, st);
    nrb_matrix qf = *q;
    qf.raw = nullptr;
    qf.h16 = nullptr;
    qf.h16_row_scale = nullptr;
    qf.hi = fhi;
    qf.lo = flo;
    qf.norms = fnr;
    qf.n = nflag;
    if (!rc) rc = search_flat_impl(&qf, b, metric, k, id_base, Df, If, ws2, wsb2, NRB_PATH_TC, st);
    if (!rc) rc = launch_scatter_results(Df, If, w.flag_list, nflag, k, D, I, st);
    cudaFreeAsync(tmp, st);
    return rc;
}

}  // namespace nrb

extern "C" int nrb_search_flat(const nrb_matrix* q, const nrb_matrix* b, int32_t metric, int32_t k,
                               int64_t id_base, float* D, int64_t* I, void* workspace,
                               size_t workspace_bytes, int32_t path, void* stream) {
    NRB_REQUIRE(q && b && D && I, "search_flat: null argument");
    NRB_REQUIRE(metric == NRB_METRIC_INNER_PRODUCT || metric == NRB_METRIC_L2, "search_flat: bad metric %d", metric);
    NRB_REQUIRE(k >= 1 && k <= NRB_MAX_K, "search_flat: k=%d out of range [1,%d]", k, NRB_MAX_K);
    NRB_REQUIRE(q->d == b->d && q->kp == b->kp, "search_flat: dimension mismatch (%d/%d vs %d/%d)", q->d, q->kp, b->d, b->kp);
    NRB_REQUIRE(q->n >= 0 && b->n >= 0 && b->n < (1LL << 31) - 4096 && q->n < (1LL << 31), "search_flat: sizes out of range");
    NRB_REQUIRE(path >= NRB_PATH_AUTO && path <= NRB_PATH_TC16, "search_flat: bad path %d", path);
    if (q->n == 0) return NRB_OK;
    int rc = require_device();
    if (rc) return rc;
    return search_flat_impl(q, b, metric, k, id_base, D, I, workspace, workspace_bytes, path, (cudaStream_t)stream);
}

extern "C" int64_t nrb_fallback_query_count(void) { return (int64_t)g_fallback_queries.load(); }

extern "C" int nrb_plan_flat_describe(int64_t nq, int64_t nb, int32_t k, int32_t path, int32_t* out10) {
    NRB_REQUIRE(out10 && nq >= 1 && nb >= 0 && k >= 1 && k <= NRB_MAX_K, "plan_flat_describe: bad arguments");
    NRB_REQUIRE(path == NRB_PATH_SIMT || path == NRB_PATH_TC || path == NRB_PATH_TC1 || path == NRB_PATH_TC16,
                "plan_flat_describe: path must be a concrete path, not %d", path);
    const FlatPlan p = plan_flat(nq, nb, k, path);
    const int v[10] = {p.nqt, p.npairs, p.full_pairs, p.tail_pairs, p.tsplit, p.chunk_rows, p.n_units, p.S, p.grid, p.single};
    for (int i = 0; i < 10; i++) out10[i] = v[i];
    return NRB_OK;
}

extern "C" size_t nrb_ivf_search_workspace(int64_t nq, int32_t nprobe, int32_t k, int32_t kp,
                                           int32_t nlist, int32_t max_list_len) {
    if (nq <= 0 || nprobe <= 0 || k <= 0) return 256;
    size_t best = 0;
    for (int path : {NRB_PATH_TC, NRB_PATH_SIMT, NRB_PATH_TC16}) {
        if (path == NRB_PATH_TC16 && !tc1_k_ok(k)) continue;
        const IvfPlan p = plan_ivf(nq, nprobe, nlist, max_list_len, path);
        const size_t t = carve_ivf(nullptr, p, nlist, k, kp, path, nq).total;
        best = t > best ? t : best;
    }
    return best + 256;
}

namespace nrb {

// phase A (or a single-phase scan): cold rows; phase B: rows start from their query's shared bound
static inline int ivf_mode_of(int nph, int i) { return (nph > 1 && i == 1) ? 2 : 1; }

// dst[i, :] = src[list[i], :] for rows of `width` 64-bit ids (coarse assignments of flagged queries)
__global__ void gather_i64_rows_kernel(const int64_t* __restrict__ src, int width, const int* __restrict__ list,
                                       int n, int64_t* __restrict__ dst) {
    const int64_t total = (int64_t)n * width;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int i = (int)(t / width), j = (int)(t - (int64_t)i * width);
        dst[t] = src[(int64_t)list[i] * width + j];
    }
}

// path: NRB_PATH_SIMT, NRB_PATH_TC (3xTF32) or NRB_PATH_TC16 (fp16 filter + exact refine, flagged
// queries recomputed through NRB_PATH_TC).
static int ivf_search_impl(const nrb_matrix* q, const nrb_matrix* lists, const int32_t* offsets, int nlist,
                           int max_list_len, const int64_t* ids, const int64_t* coarse, int nprobe, int metric,
                           int k, float* D, int64_t* I, void* workspace, size_t workspace_bytes, int path,
                           cudaStream_t st) {
    int rc;
    const bool filt = path == NRB_PATH_TC16;
    const IvfPlan p = plan_ivf(q->n, nprobe, nlist, max_list_len, path);
    NRB_REQUIRE(filt || p.S <= IVF_MAX_SOURCES, "ivf_search: nprobe*splits = %d > %d merge sources", p.S, IVF_MAX_SOURCES);
    const IvfWs w = carve_ivf(workspace, p, nlist, k, q->kp, path, q->n);
    if (!workspace || workspace_bytes < w.total) {
        set_error("ivf_search: workspace %zu < %zu bytes", workspace_bytes, w.total);
        return NRB_ERR_WORKSPACE;
    }
    if (metric == NRB_METRIC_L2 || filt) NRB_REQUIRE(q->norms && lists->norms, "ivf_search: norms required");
    if (p.nph > 1) {
        int64_t blocks = (q->n * nprobe + 255) / 256;
        if (blocks > 148 * 16) blocks = 148 * 16;
        ivf_split_coarse_kernel<<<(unsigned)blocks, 256, 0, st>>>(coarse, q->n, nprobe, w.ph[0].coarse, w.ph[1].coarse);
        NRB_LAUNCH_CHECK();
    }
    if (path != NRB_PATH_SIMT) NRB_CUDA_CHECK(cudaMemsetAsync(w.gthr, 0, (size_t)q->n * sizeof(unsigned), st));
    if (filt) NRB_CUDA_CHECK(cudaMemsetAsync(w.flags, 0, (size_t)q->n * sizeof(int), st));
    const int pw = filt ? tc1_pw(k) : k;
    const float eps_xmax = TC1_EPS * lists->max_norm;
    nrb_matrix g[2];
    // ---- per phase: grouping, unit list, src table, regrouped query rows (all on the device)
    for (int i = 0; i < p.nph; i++) {
        const IvfPhase& f = p.ph[i];
        const IvfPhaseWs& v = w.ph[i];
        const int64_t* co = p.nph > 1 ? v.coarse : coarse;
        // 1. group (query, list) pairs by list (stable): p_off, order (position -> pair), pos_of
        NRB_CUDA_CHECK(cudaMemsetAsync(v.order, 0, (size_t)f.npairs * sizeof(int), st));
        if ((rc = launch_counting_sort_i64(co, f.npairs, nlist, v.p_off, v.order, v.pos_of, v.cs, v.cs_bytes, st))) return rc;
        // 2. units + src table
        const size_t sh = (size_t)(2 * nlist + 1) * sizeof(int);
        NRB_REQUIRE(sh <= 48 * 1024, "ivf_search: too many lists (%d)", nlist);
        ivf_plan_kernel<<<1, 512, sh, st>>>(v.p_off, offsets, nlist, p.chunk, v.ubase, v.nsl, v.n_units, v.units, f.max_units);
        NRB_LAUNCH_CHECK();
        {
            int64_t blocks = (f.npairs + 255) / 256;
            if (blocks > 148 * 16) blocks = 148 * 16;
            ivf_src_kernel<<<(unsigned)blocks, 256, 0, st>>>(co, v.pos_of, v.p_off, v.ubase, v.nsl, nlist, f.npairs, f.ncols,
                                                             p.maxsplit, p.wgs, p.S, f.s_off, f.prow_base, w.src);
            NRB_LAUNCH_CHECK();
        }
        // 3. query rows in group order: row p of the regrouped plane is pair order[p], i.e. query order[p] / ncols
        nrb_matrix& gm = g[i];
        memset(&gm, 0, sizeof(gm));
        gm.n = f.npairs;
        gm.d = q->d;
        gm.kp = q->kp;
        gm.raw = v.g_raw;
        gm.hi = v.g_hi;
        gm.lo = v.g_lo;
        if (path == NRB_PATH_SIMT) {
            NRB_REQUIRE(q->raw, "ivf_search: raw plane required");
            if ((rc = launch_gather_rows(q->raw, q->kp, v.order, f.ncols, f.npairs, v.g_raw, st))) return rc;
        } else if (filt) {
            // fp16 rows are kp/2 floats wide; their per-row scales and norms travel with them
            if ((rc = launch_gather_rows((const float*)q->h16, q->kp / 2, v.order, f.ncols, f.npairs, (float*)v.g_h16, st))) return rc;
            if ((rc = launch_gather_scalar(q->h16_row_scale, v.order, f.ncols, f.npairs, v.g_scale, st))) return rc;
            gm.h16 = v.g_h16;
            gm.h16_row_scale = v.g_scale;
        } else {
            NRB_REQUIRE(q->hi && q->lo, "ivf_search: hi/lo planes required");
            if ((rc = launch_gather_rows(q->hi, q->kp, v.order, f.ncols, f.npairs, v.g_hi, st))) return rc;
            if ((rc = launch_gather_rows(q->lo, q->kp, v.order, f.ncols, f.npairs, v.g_lo, st))) return rc;
        }
        if (metric == NRB_METRIC_L2 || filt) {
            if ((rc = launch_gather_scalar(q->norms, v.order, f.ncols, f.npairs, v.g_norms, st))) return rc;
            gm.norms = v.g_norms;
        }
    }
    // ---- 4. distance + selection over the units, phase A then phase B (which starts from A's bounds)
    for (int i = 0; i < p.nph; i++) {
        const IvfPhase& f = p.ph[i];
        const IvfPhaseWs& v = w.ph[i];
        const size_t po = (size_t)f.prow_base * pw;
        ProfScope prof(st);
        if (path == NRB_PATH_SIMT)
            rc = launch_topk_simt_dev(&g[i], lists, v.units, v.n_units, f.grid, metric, k, w.part_key + po, w.part_idx + po,
                                      w.scratch, w.scratch_bytes, st);
        else if (!filt)
            // all units of a query share one running bound
            rc = launch_topk_tc_dev(&g[i], lists, v.units, v.n_units, f.grid, metric, k, w.part_key + po, w.part_idx + po,
                                    w.scratch, w.scratch_bytes, w.gthr, v.order, f.ncols, st);
        else
            rc = launch_topk_tc1_dev(&g[i], lists, v.units, v.n_units, f.grid, metric, k, pw, 2.f * eps_xmax, w.part_key + po,
                                     w.part_idx + po, w.part_cnt + f.prow_base, w.flags, w.scratch, w.scratch_bytes, w.gthr,
                                     v.order, f.ncols, 1, 0, ivf_mode_of(p.nph, i), st);
        if (rc) return rc;
    }
    // ---- 5. per query: merge (sorted partial rows) or gather + exact refine (filter)
    if (!filt) return launch_select(w.part_key, w.part_idx, w.src, p.S, q->n, k, metric, ids, 0, D, I, st);
    if ((rc = launch_gather_refine(w.part_key, w.part_idx, w.part_cnt, w.src, p.S, q->n, k, pw, metric, q, lists, eps_xmax,
                                   0, ids, w.flags, D, I, st))) return rc;
    if ((rc = launch_compact_flags(w.flags, q->n, w.flag_list, w.flag_count, st))) return rc;
    int nflag = 0;
    NRB_CUDA_CHECK(cudaMemcpyAsync(&nflag, w.flag_count, sizeof(int), cudaMemcpyDeviceToHost, st));
    NRB_CUDA_CHECK(cudaStreamSynchronize(st));
    if (nflag == 0) return NRB_OK;
    g_fallback_queries += nflag;
    const size_t plane = (size_t)nflag * q->kp * sizeof(float);
    const size_t wsb2 = nrb_ivf_search_workspace(nflag, nprobe, k, q->kp, nlist, max_list_len);
    char* tmp = nullptr;
    const size_t tmp_bytes = 2 * align_up(plane, 256) + align_up((size_t)nflag * 4, 256) +
                             align_up((size_t)nflag * nprobe * 8, 256) + align_up((size_t)nflag * k * 4, 256) +
                             align_up((size_t)nflag * k * 8, 256) + wsb2;
    keep_pool_memory();
    NRB_CUDA_CHECK(cudaMallocAsync((void**)&tmp, tmp_bytes, st));
    Carver c(tmp);
    float* fhi = c.take<float>((size_t)nflag * q->kp);
    float* flo = c.take<float>((size_t)nflag * q->kp);
    float* fnr = c.take<float>(nflag);
    int64_t* fco = c.take<int64_t>((size_t)nflag * nprobe);
    float* Df = c.take<float>((size_t)nflag * k);
    int64_t* If = c.take<int64_t>((size_t)nflag * k);
    void* ws2 = c.take<char>(wsb2);
    rc = launch_gather_rows(q->hi, q->kp, w.flag_list, 1, nflag, fhi, st);
    if (!rc) rc = launch_gather_rows(q->lo, q->kp, w.flag_list, 1, nflag, flo, st);
    if (!rc) rc = launch_gather_scalar(q->norms, w.flag_list, 1, nflag, fnr, st);
    if (!rc) {
        gather_i64_rows_kernel<<<(unsigned)(((int64_t)nflag * nprobe + 255) / 256), 256, 0, st>>>(coarse, nprobe, w.flag_list, nflag, fco);
        count_launch();
        if (cudaGetLastError() != cudaSuccess) rc = NRB_ERR_CUDA;
    }
    nrb_matrix qf = *q;
    qf.raw = nullptr;
    qf.h16 = nullptr;
    qf.h16_row_scale = nullptr;
    qf.hi = fhi;
    qf.lo = flo;
    qf.norms = fnr;
    qf.n = nflag;
    if (!rc) rc = ivf_search_impl(&qf, lists, offsets, nlist, max_list_len, ids, fco, nprobe, metric, k, Df, If, ws2, wsb2, NRB_PATH_TC, st);
    if (!rc) rc = launch_scatter_results(Df, If, w.flag_list, nflag, k, D, I, st);
    cudaFreeAsync(tmp, st);
    return rc;
}

}  // namespace nrb

extern "C" int nrb_ivf_search(const nrb_matrix* q, const nrb_matrix* lists, const int32_t* offsets,
                              int32_t nlist, int32_t max_list_len, const int64_t* ids,
                              const int64_t* coarse, int32_t nprobe, int32_t metric, int32_t k,
                              float* D, int64_t* I, void* workspace, size_t workspace_bytes,
                              int32_t path, void* stream) {
    NRB_REQUIRE(q && lists && offsets && ids && coarse && D && I, "ivf_search: null argument");
    NRB_REQUIRE(metric == NRB_METRIC_INNER_PRODUCT || metric == NRB_METRIC_L2, "ivf_search: bad metric %d", metric);
    NRB_REQUIRE(k >= 1 && k <= NRB_MAX_K, "ivf_search: k=%d out of range [1,%d]", k, NRB_MAX_K);
    NRB_REQUIRE(nprobe >= 1 && nlist >= 1 && nlist <= 8192, "ivf_search: bad nprobe/nlist");
    NRB_REQUIRE(q->d == lists->d && q->kp == lists->kp, "ivf_search: dimension mismatch");
    NRB_REQUIRE(q->n * (int64_t)nprobe < (1LL << 31) - 4096 && lists->n < (1LL << 31) - 4096, "ivf_search: sizes out of range");
    NRB_REQUIRE(path >= NRB_PATH_AUTO && path <= NRB_PATH_TC16 && path != NRB_PATH_TC1, "ivf_search: bad path %d", path);
    if (q->n == 0) return NRB_OK;
    int rc = require_device();
    if (rc) return rc;
    // the fp16 filter needs, besides its own planes, the raw planes (exact refine) and the hi/lo
    // planes on both sides (flagged queries are recomputed by the 3xTF32 scan)
    const bool filt_ok = tc16_eligible(q, lists, k) && q->hi && q->lo && lists->hi && lists->lo;
    if (path == NRB_PATH_TC16 && !filt_ok) {
        set_error("ivf_search: NRB_PATH_TC16 needs raw/h16/hi/lo/norms planes and h16 scales on both sides, "
                  "max_norm on the list side, kp <= 256 and k <= %d", TC1_MAX_PW - TC1_MIN_EXTRA);
        return NRB_ERR_INVALID;
    }
    if (path == NRB_PATH_AUTO) path = filt_ok ? NRB_PATH_TC16 : NRB_PATH_TC;
    return ivf_search_impl(q, lists, offsets, nlist, max_list_len, ids, coarse, nprobe, metric, k, D, I, workspace,
                           workspace_bytes, path, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------ fused k-means
namespace nrb {
struct KmTrainWs {
    float *craw, *chi, *clo, *cnorms, *hassign, *dis, *cent_in;
    __half* ch16;
    int64_t* assign;
    void* upd;
    size_t upd_bytes;
    void* search;
    size_t search_bytes;
    size_t total;
};
static KmTrainWs carve_km_train(void* ws, int64_t n, int k, int d, int kp) {
    Carver c(ws);
    KmTrainWs w;
    w.craw = c.take<float>((size_t)k * kp);
    w.chi = c.take<float>((size_t)k * kp);
    w.clo = c.take<float>((size_t)k * kp);
    w.ch16 = c.take<__half>((size_t)k * kp);
    w.cnorms = c.take<float>(k);
    w.hassign = c.take<float>(k);
    w.cent_in = c.take<float>((size_t)k * d);
    w.dis = c.take<float>(n);
    w.assign = c.take<int64_t>(n);
    w.upd_bytes = kmeans_update_ws(n, k, kp);
    w.upd = c.take<char>(w.upd_bytes);
    w.search_bytes = nrb_search_flat_workspace(n, k, 1, kp);
    w.search = c.take<char>(w.search_bytes);
    w.total = c.off;
    return w;
}
}  // namespace nrb

extern "C" size_t nrb_kmeans_train_workspace(int64_t n, int32_t k, int32_t kp) {
    if (n <= 0 || k <= 0 || kp <= 0) return 256;
    return carve_km_train(nullptr, n, k, kp, kp).total + 256;
}

extern "C" int nrb_kmeans_train(const nrb_matrix* x, int32_t k, int32_t niter, int32_t metric, int32_t spherical,
                                float* centroids, int64_t* assign, double* stats, void* workspace,
                                size_t workspace_bytes, void* stream) {
    NRB_REQUIRE(x && centroids && stats && workspace, "kmeans_train: null argument");
    NRB_REQUIRE(x->raw && x->norms, "kmeans_train: the training rows need their raw plane and norms");
    NRB_REQUIRE(metric == NRB_METRIC_INNER_PRODUCT || metric == NRB_METRIC_L2, "kmeans_train: bad metric %d", metric);
    NRB_REQUIRE(k > 0 && niter >= 0 && x->n > k && x->n < (1LL << 31) && x->kp % 32 == 0 && x->kp <= 2048,
                "kmeans_train: bad sizes n=%lld k=%d", (long long)x->n, k);
    int rc = require_device();
    if (rc) return rc;
    const int64_t n = x->n;
    const int d = x->d, kp = x->kp;
    const KmTrainWs w = carve_km_train(workspace, n, k, d, kp);
    if (workspace_bytes < w.total) {
        set_error("kmeans_train: workspace %zu < %zu bytes", workspace_bytes, w.total);
        return NRB_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    // Norm bound of every centroid this loop can produce, known on the host: a mean of rows is no longer
    // than the longest row, and split_clusters scales coordinates by at most (1 + 1/1024) per split
    // (<= k splits per iteration); spherical centroids have norm 1. It sizes the filter's error margin
    // and the fp16 scale of the centroid plane, so the loop never reads a norm back.
    float bound = x->max_norm * powf(1.f + 1.f / 1024.f, (float)(k < 1024 ? k : 1024)) * 1.0001f;
    if (spherical && bound < 1.0001f) bound = 1.0001f;
    // assignment path: fp16 filter + exact refine when the rows carry their scaled fp16 plane, else the
    // 1xTF32 filter (hi plane), else 3xTF32; k = 1 makes every one of them free of host round trips
    const bool f16 = x->h16 && x->h16_row_scale && x->max_norm > 0.f && kp <= 256;
    const bool f32 = !f16 && x->hi && x->max_norm > 0.f && kp <= 256;
    NRB_REQUIRE(f16 || f32 || (x->hi && x->lo), "kmeans_train: the training rows need h16 (+ row scales), or hi, or hi + lo planes");
    const int path = f16 ? NRB_PATH_TC16 : f32 ? NRB_PATH_TC1 : NRB_PATH_TC;
    nrb_matrix cm;
    memset(&cm, 0, sizeof(cm));
    cm.raw = w.craw;
    cm.hi = w.chi;
    cm.lo = w.clo;
    cm.norms = w.cnorms;
    cm.n = k;
    cm.d = d;
    cm.kp = kp;
    cm.max_norm = bound;
    if (f16) {
        cm.h16 = w.ch16;
        cm.h16_scale = ldexpf(1.f, 14 - ilogbf(bound));
    }
    for (int it = 0; it < niter; it++) {
        double* s = stats + (size_t)it * 4;
        if ((rc = launch_pack_rows(centroids, k, d, d, kp, w.craw, w.chi, w.clo, w.cnorms, st))) return rc;
        if (f16 && (rc = nrb_pack_rows_h16(w.craw, k, d, kp, kp, cm.h16_scale, w.ch16, nullptr, stream))) return rc;
        if ((rc = search_flat_impl(x, &cm, metric, 1, 0, w.dis, w.assign, w.search, w.search_bytes, path, st))) return rc;
        NRB_CUDA_CHECK(cudaMemcpyAsync(w.cent_in, centroids, (size_t)k * d * sizeof(float), cudaMemcpyDeviceToDevice, st));
        if ((rc = launch_kmeans_update(x->raw, n, d, kp, w.assign, k, centroids, w.hassign, w.upd, w.cent_in, metric, s, st)))
            return rc;
        if ((rc = launch_km_split(d, k, n, w.hassign, centroids, s, st))) return rc;
        if (spherical && (rc = nrb_normalize_l2(centroids, k, d, d, stream))) return rc;
    }
    if (assign && niter > 0)
        NRB_CUDA_CHECK(cudaMemcpyAsync(assign, w.assign, (size_t)n * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
    return NRB_OK;
}

// The two host helpers below restate third-party faiss routines (facebookresearch/faiss, MIT licence:
// utils/random.cpp rand_perm and Clustering.cpp split_clusters) because RNG-exact k-means needs their
// exact arithmetic -- the draw order of std::mt19937, the float conversions, EPS = 1/1024. They are
// not taken from /root/reference, which contains no native code.
extern "C" int nrb_rand_perm_host(int32_t* perm, int64_t n, int64_t seed) {
    NRB_REQUIRE(perm && n >= 0, "rand_perm: bad arguments");
    std::mt19937 mt((unsigned)seed);
    for (int64_t i = 0; i < n; i++) perm[i] = (int32_t)i;
    for (int64_t i = 0; i + 1 < n; i++) {
        const int64_t i2 = i + (int64_t)(mt() % (uint32_t)(n - i));
        std::swap(perm[i], perm[i2]);
    }
    return NRB_OK;
}

extern "C" int nrb_split_clusters_host(int32_t d, int32_t k, int64_t n, float* hassign, float* centroids) {
    NRB_REQUIRE(hassign && centroids && d > 0 && k > 0 && n > k, "split_clusters: bad arguments");
    const double EPS = 1 / 1024.;
    std::mt19937 mt(1234);
    int nsplit = 0;
    for (int ci = 0; ci < k; ci++) {
        if (hassign[ci] != 0) continue;
        int cj = 0;
        for (int guard = 0;; cj = (cj + 1) % k) {
            const float p = (hassign[cj] - 1.0) / (float)(n - k);
            const float r = mt() / float(mt.max());
            if (r < p) break;
            if (++guard > 100000000) {
                set_error("split_clusters: no cluster to split");
                return NRB_ERR_INVALID;
            }
        }
        float* a = centroids + (size_t)ci * d;
        float* b = centroids + (size_t)cj * d;
        memcpy(a, b, sizeof(float) * d);
        for (int j = 0; j < d; j++) {
            if (j % 2 == 0) {
                a[j] *= 1 + EPS;
                b[j] *= 1 - EPS;
            } else {
                a[j] *= 1 - EPS;
                b[j] *= 1 + EPS;
            }
        }
        hassign[ci] = hassign[cj] / 2;
        hassign[cj] -= hassign[ci];
        nsplit++;
    }
    return nsplit;
}
