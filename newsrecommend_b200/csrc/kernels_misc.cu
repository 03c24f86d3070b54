// HBM-bound helper kernels: pack/split (K0), row gather, L2 normalise, stable counting sort by
// list (K3 layout / K1b grouping), segmented centroid update (K1b), and the final select /
// k-way merge (K4).
#include <cfloat>

#include <cuda_fp16.h>

#include "common.cuh"
#include "internal.h"

namespace nrb {

// ------------------------------------------------------------------------------------ K0 pack
// One warp per row. x[n, d] (stride ldx) -> raw/hi/lo [n, kp] and norms[n].
// Reference: replaces the numpy astype/ascontiguousarray at Retrieval.py:8,17,31.
__global__ void pack_rows_kernel(const float* __restrict__ x, int64_t n, int d, int64_t ldx,
                                 int kp, float* __restrict__ raw, float* __restrict__ hi,
                                 float* __restrict__ lo, float* __restrict__ norms) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t row = warp0; row < n; row += nwarps) {
        const float* xr = x + row * ldx;
        float acc = 0.f;
        for (int c = lane; c < kp; c += 32) {
            float v = (c < d) ? xr[c] : 0.f;
            acc = fmaf(v, v, acc);
            const int64_t o = row * kp + c;
            if (raw) raw[o] = v;
            if (hi || lo) {
                uint32_t hb, lb;
                asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb) : "f"(v));
                float h = __uint_as_float(hb);
                float l = v - h;  // exact in fp32
                asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(lb) : "f"(l));
                if (hi) hi[o] = h;
                if (lo) lo[o] = __uint_as_float(lb);
            }
        }
        if (norms) {
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
            if (lane == 0) norms[row] = acc;
        }
    }
}

// fp16 plane of the fp16 filter. One warp per row: h16[row, c] = fp16(x[row, c] * s), s a power
// of two -- `uniform` when > 0, else 2^(14 - floor(log2(|row|))) (so |row| * s is in [2^14, 2^15)
// and no element can overflow fp16), stored in row_scale[row].
__global__ void pack_rows_h16_kernel(const float* __restrict__ x, int64_t n, int d, int64_t ldx, int kp,
                                     float uniform, __half* __restrict__ h16, float* __restrict__ row_scale) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t row = warp0; row < n; row += nwarps) {
        const float* xr = x + row * ldx;
        float s = uniform;
        if (!(uniform > 0.f)) {
            float acc = 0.f;
            for (int c = lane; c < d; c += 32) acc = fmaf(xr[c], xr[c], acc);
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
            // sqrt(acc) rounded up a little so that an fp32 sum that came out low cannot push an
            // element past 2^15 * (1 + 2^-10) (far below the fp16 maximum anyway)
            const float nr = sqrtf(acc);
            int e = (nr > 0.f && nr < __builtin_huge_valf()) ? ilogbf(nr) : 14;
            e = e < -60 ? -60 : (e > 60 ? 60 : e);
            s = exp2f((float)(14 - e));
            if (lane == 0 && row_scale) row_scale[row] = s;
        }
        for (int c = lane; c < kp; c += 32) {
            const float v = (c < d) ? xr[c] * s : 0.f;
            h16[row * kp + c] = __float2half_rn(v);
        }
    }
}

// dst[i, :] = src[idx[i] / div, :], rows of `width` floats (width % 4 == 0), float4 lanes.
__global__ void gather_rows_kernel(const float4* __restrict__ src, int w4,
                                   const int32_t* __restrict__ idx, int div, int64_t n,
                                   float4* __restrict__ dst) {
    const int64_t total = n * w4;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = t / w4;
        const int c = (int)(t - i * w4);
        const int64_t s = idx[i] / div;
        dst[t] = __ldg(src + s * w4 + c);
    }
}

__global__ void gather_scalar_kernel(const float* __restrict__ src, const int32_t* __restrict__ idx,
                                     int div, int64_t n, float* __restrict__ dst) {
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n;
         t += (int64_t)gridDim.x * blockDim.x)
        dst[t] = src[idx[t] / div];
}

__global__ void gather_i64_kernel(const int64_t* __restrict__ src, const int32_t* __restrict__ idx,
                                  int64_t n, int64_t* __restrict__ dst) {
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n;
         t += (int64_t)gridDim.x * blockDim.x)
        dst[t] = src[idx[t]];
}

// faiss.normalize_L2: warp per row, in place.
__global__ void normalize_l2_kernel(float* __restrict__ x, int64_t n, int d, int64_t ldx) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t row = warp0; row < n; row += nwarps) {
        float* xr = x + row * ldx;
        float acc = 0.f;
        for (int c = lane; c < d; c += 32) acc = fmaf(xr[c], xr[c], acc);
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (acc > 0.f) {
            const float inv = 1.0f / sqrtf(acc);
            for (int c = lane; c < d; c += 32) xr[c] *= inv;
        }
    }
}

// ------------------------------------------------------------------- stable counting sort
// Sorts items 0..n by key[i] in [0, nb) (keys outside the range, e.g. -1, go to bucket nb and
// are dropped from `order`) keeping source order inside a bucket. Three kernels:
//   hist: per-chunk bucket counts; scan: bucket offsets + per-chunk bases; scatter.
constexpr int CS_CHUNK = 2048;
constexpr int CS_THREADS = 256;

template <typename KeyT>
__global__ void cs_hist_kernel(const KeyT* __restrict__ key, int64_t n, int nb,
                               int* __restrict__ chunk_hist /*[nchunks, nb+1]*/) {
    extern __shared__ int sh[];
    const int nb1 = nb + 1;
    for (int b = threadIdx.x; b < nb1; b += blockDim.x) sh[b] = 0;
    __syncthreads();
    const int64_t i0 = (int64_t)blockIdx.x * CS_CHUNK;
    for (int t = threadIdx.x; t < CS_CHUNK; t += blockDim.x) {
        const int64_t i = i0 + t;
        if (i < n) {
            int64_t kk = (int64_t)key[i];
            int b = (kk >= 0 && kk < nb) ? (int)kk : nb;
            atomicAdd(&sh[b], 1);
        }
    }
    __syncthreads();
    for (int b = threadIdx.x; b < nb1; b += blockDim.x)
        chunk_hist[(int64_t)blockIdx.x * nb1 + b] = sh[b];
}

// Single block. offsets[nb+1] (exclusive scan of bucket totals over real buckets; offsets[nb] =
// number of kept items) and chunk_hist rewritten in place to per-chunk bases.
__global__ void cs_scan_kernel(int* __restrict__ chunk_hist, int nchunks, int nb,
                               int* __restrict__ offsets) {
    extern __shared__ int tot[];  // nb + 2
    const int nb1 = nb + 1;
    for (int b = threadIdx.x; b < nb1; b += blockDim.x) {
        int s = 0;
        for (int c = 0; c < nchunks; c++) s += chunk_hist[(int64_t)c * nb1 + b];
        tot[b] = s;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int run = 0;
        for (int b = 0; b < nb1; b++) {
            int t = tot[b];
            tot[b] = run;
            run += t;
        }
        tot[nb1] = run;
    }
    __syncthreads();
    for (int b = threadIdx.x; b <= nb; b += blockDim.x) offsets[b] = tot[b];
    for (int b = threadIdx.x; b < nb1; b += blockDim.x) {
        int run = tot[b];
        for (int c = 0; c < nchunks; c++) {
            const int64_t o = (int64_t)c * nb1 + b;
            int t = chunk_hist[o];
            chunk_hist[o] = run;
            run += t;
        }
    }
}

// The same scan for long inputs (thousands of chunks: the (query, list) pairs of an IVF batch), in
// three small grids instead of one block walking every chunk twice: the chunks are cut into
// CS_GROUPS groups; (1) per-group bucket totals, (2) one block: exclusive scan over (bucket, group) +
// the bucket offsets, (3) per group: the chunks' exclusive prefixes.
constexpr int CS_GROUPS = 64;
__global__ void cs_group_tot_kernel(const int* __restrict__ chunk_hist, int nchunks, int nb1, int* __restrict__ gtot) {
    const int g = blockIdx.x, per = (nchunks + CS_GROUPS - 1) / CS_GROUPS;
    const int c0 = g * per, c1 = min(nchunks, c0 + per);
    for (int b = threadIdx.x; b < nb1; b += blockDim.x) {
        int s = 0;
        for (int c = c0; c < c1; c++) s += chunk_hist[(int64_t)c * nb1 + b];
        gtot[g * nb1 + b] = s;
    }
}
__global__ void cs_group_scan_kernel(int* __restrict__ gtot, int nb, int* __restrict__ offsets) {
    extern __shared__ int tot[];  // nb + 2
    const int nb1 = nb + 1;
    for (int b = threadIdx.x; b < nb1; b += blockDim.x) {
        int s = 0;
        for (int g = 0; g < CS_GROUPS; g++) s += gtot[g * nb1 + b];
        tot[b] = s;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int run = 0;
        for (int b = 0; b < nb1; b++) {
            int t = tot[b];
            tot[b] = run;
            run += t;
        }
        tot[nb1] = run;
    }
    __syncthreads();
    for (int b = threadIdx.x; b <= nb; b += blockDim.x) offsets[b] = tot[b];
    for (int b = threadIdx.x; b < nb1; b += blockDim.x) {
        int run = tot[b];
        for (int g = 0; g < CS_GROUPS; g++) {
            const int t = gtot[g * nb1 + b];
            gtot[g * nb1 + b] = run;
            run += t;
        }
    }
}
__global__ void cs_group_prefix_kernel(int* __restrict__ chunk_hist, int nchunks, int nb1, const int* __restrict__ gtot) {
    const int g = blockIdx.x, per = (nchunks + CS_GROUPS - 1) / CS_GROUPS;
    const int c0 = g * per, c1 = min(nchunks, c0 + per);
    for (int b = threadIdx.x; b < nb1; b += blockDim.x) {
        int run = gtot[g * nb1 + b];
        for (int c = c0; c < c1; c++) {
            const int64_t o = (int64_t)c * nb1 + b;
            const int t = chunk_hist[o];
            chunk_hist[o] = run;
            run += t;
        }
    }
}

template <typename KeyT>
__global__ void cs_scatter_kernel(const KeyT* __restrict__ key, int64_t n, int nb,
                                  const int* __restrict__ chunk_base, int* __restrict__ order,
                                  int* __restrict__ pos_of /*optional: item -> position*/) {
    extern __shared__ int run[];  // nb + 1 running positions
    const int nb1 = nb + 1;
    for (int b = threadIdx.x; b < nb1; b += blockDim.x)
        run[b] = chunk_base[(int64_t)blockIdx.x * nb1 + b];
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int64_t i0 = (int64_t)blockIdx.x * CS_CHUNK;
    for (int r0 = 0; r0 < CS_CHUNK; r0 += blockDim.x) {
        const int64_t i = i0 + r0 + threadIdx.x;
        int b = -1;
        if (i < n) {
            int64_t kk = (int64_t)key[i];
            b = (kk >= 0 && kk < nb) ? (int)kk : nb;
        }
        // rank among same-bucket lanes of this warp (lower lanes first)
        unsigned peers = __match_any_sync(0xffffffffu, b);
        const int rank = __popc(peers & ((1u << lane) - 1u));
        const int leader = __ffs(peers) - 1;
        int base = 0;
        // warps take turns so that positions follow source order
        for (int w = 0; w < nwarps; w++) {
            if (w == warp && b >= 0 && lane == leader) {
                base = run[b];
                run[b] = base + __popc(peers);
            }
            __syncthreads();
        }
        base = __shfl_sync(0xffffffffu, base, leader);
        if (b >= 0) {
            const int p = base + rank;
            if (b < nb) order[p] = (int)i;
            if (pos_of) pos_of[i] = (b < nb) ? p : -1;
        }
    }
}

// ------------------------------------------------------------------- K1b centroid update
// Segmented reduction over the counting-sorted row order, balanced under list skew: every
// centroid's run of rows is cut into chunks of KM_CHUNK rows (a chunk never crosses a centroid
// boundary), one block per chunk sums its rows in fp64 (threads = kp/4 float4 columns x `slices`
// row slices, each slice in source order, slices combined in a fixed order), and one block per
// centroid adds the chunk partials in chunk order. Every sum has a fixed association, so the
// result is deterministic and independent of the grid; a 18,000-row list is 280 blocks of work
// instead of one. mean = float(sum) * (1.0f / count)  (Clustering.cpp compute_centroids).
constexpr int KM_CHUNK = 64;

// chunk_base[c] = number of chunks of centroids < c (exclusive scan of ceil(len / KM_CHUNK));
// chunk_base[k] = total. One block.
__global__ void km_plan_kernel(const int* __restrict__ offsets, int k, int* __restrict__ chunk_base) {
    __shared__ int wsum[32];
    __shared__ int carry;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < k; base += blockDim.x) {
        const int c = base + threadIdx.x;
        const int v = c < k ? (offsets[c + 1] - offsets[c] + KM_CHUNK - 1) / KM_CHUNK : 0;
        int inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (lane == 31) wsum[warp] = inc;
        __syncthreads();
        int before = carry;
        for (int w = 0; w < warp; w++) before += wsum[w];
        if (c < k) chunk_base[c] = before + inc - v;
        __syncthreads();
        if (threadIdx.x == 0) {
            int t = 0;
            for (int w = 0; w < nw; w++) t += wsum[w];
            carry += t;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) chunk_base[k] = carry;
}

__global__ void km_partial_kernel(const float* __restrict__ x_raw, int kp, const int* __restrict__ offsets,
                                  const int* __restrict__ order, const int* __restrict__ chunk_base, int k, int slices,
                                  double* __restrict__ partial, const float* __restrict__ cent_in, int d, int l2,
                                  double* __restrict__ obj_part) {
    extern __shared__ double part[];  // [slices][kp]
    const int j = blockIdx.x;
    if (j >= chunk_base[k]) return;
    int lo = 0, hi = k;  // largest c with chunk_base[c] <= j (an empty centroid shares its base with the next one)
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (chunk_base[mid] <= j) lo = mid; else hi = mid;
    }
    const int c = lo;
    const int r0 = offsets[c] + (j - chunk_base[c]) * KM_CHUNK;
    const int r1 = min(offsets[c + 1], r0 + KM_CHUNK);
    const int w4 = kp >> 2;
    const int col4 = threadIdx.x % w4, slice = threadIdx.x / w4;
    // objective against the centroid the rows were assigned to (the one the iteration started with)
    float4 cc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (cent_in) {
        const float* cr = cent_in + (int64_t)c * d;
        const int c0 = col4 * 4;
        cc.x = c0 < d ? cr[c0] : 0.f;
        cc.y = c0 + 1 < d ? cr[c0 + 1] : 0.f;
        cc.z = c0 + 2 < d ? cr[c0 + 2] : 0.f;
        cc.w = c0 + 3 < d ? cr[c0 + 3] : 0.f;
    }
    double a0 = 0, a1 = 0, a2 = 0, a3 = 0, ob = 0;
#pragma unroll 4
    for (int r = r0 + slice; r < r1; r += slices) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(x_raw + (int64_t)order[r] * kp) + col4);
        a0 += v.x;
        a1 += v.y;
        a2 += v.z;
        a3 += v.w;
        float t;
        if (l2) {
            const float e0 = v.x - cc.x, e1 = v.y - cc.y, e2 = v.z - cc.z, e3 = v.w - cc.w;
            t = fmaf(e3, e3, fmaf(e2, e2, fmaf(e1, e1, e0 * e0)));
        } else {
            t = fmaf(v.w, cc.w, fmaf(v.z, cc.z, fmaf(v.y, cc.y, v.x * cc.x)));
        }
        ob += t;
    }
    double* p = part + (int64_t)slice * kp + col4 * 4;
    p[0] = a0;
    p[1] = a1;
    p[2] = a2;
    p[3] = a3;
    __syncthreads();
    for (int col = threadIdx.x; col < kp; col += blockDim.x) {
        double s = 0;
        for (int q = 0; q < slices; q++) s += part[(int64_t)q * kp + col];
        partial[(int64_t)j * kp + col] = s;
    }
    if (obj_part) {  // fixed-order block sum (blockDim <= 1024 = slices * kp / 4 <= the part[] capacity in doubles)
        __syncthreads();
        part[threadIdx.x] = ob;
        __syncthreads();
        if (threadIdx.x == 0) {
            double s = 0;
            for (int t = 0; t < (int)blockDim.x; t++) s += part[t];
            obj_part[j] = s;
        }
    }
}

__global__ void km_finish_kernel(const double* __restrict__ partial, const int* __restrict__ chunk_base,
                                 const int* __restrict__ offsets, int kp, int d, int k, float* __restrict__ centroids,
                                 float* __restrict__ hassign, const double* __restrict__ obj_part,
                                 double* __restrict__ obj_out, double* __restrict__ sums_out) {
    const int c = blockIdx.x;
    const int j0 = chunk_base[c], j1 = chunk_base[c + 1];
    const int cnt = offsets[c + 1] - offsets[c];
    if (threadIdx.x == 0) {
        if (sums_out) sums_out[(int64_t)c * (d + 1) + d] = (double)cnt;  // data-parallel form: [k, d + 1] sums | count
        else hassign[c] = (float)cnt;
    }
    for (int col = threadIdx.x; col < d; col += blockDim.x) {
        double s = 0;
#pragma unroll 8
        for (int j = j0; j < j1; j++) s += partial[(int64_t)j * kp + col];
        if (sums_out) sums_out[(int64_t)c * (d + 1) + col] = s;
        else centroids[(int64_t)c * d + col] = cnt > 0 ? (float)s * (1.0f / (float)cnt) : 0.f;
    }
    if (obj_out && c == 0) {  // objective = sum of the chunk objectives, fixed order
        __shared__ double red[256];
        const int total = chunk_base[k];
        double s = 0;
        for (int j = threadIdx.x; j < total; j += blockDim.x) s += obj_part[j];
        red[threadIdx.x] = s;
        __syncthreads();
        for (int o = blockDim.x >> 1; o > 0; o >>= 1) {
            if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
            __syncthreads();
        }
        if (threadIdx.x == 0) *obj_out = red[0];
    }
}

// Data-parallel k-means: centroids from the all-reduced [k, d + 1] table of fp64 sums | counts
// (nrb_kmeans_partial_sums on every rank's rows, summed over the ranks): the same rounding as
// km_finish_kernel -- float(sum) * (1.0f / count).
__global__ void km_means_kernel(const double* __restrict__ sums, int k, int d, float* __restrict__ centroids,
                                float* __restrict__ hassign) {
    const int c = blockIdx.x;
    const double* row = sums + (int64_t)c * (d + 1);
    const float cnt = (float)row[d];
    if (threadIdx.x == 0) hassign[c] = cnt;
    for (int col = threadIdx.x; col < d; col += blockDim.x)
        centroids[(int64_t)c * d + col] = cnt > 0.f ? (float)row[col] * (1.0f / cnt) : 0.f;
}

// faiss Clustering.cpp split_clusters on the device (same arithmetic as nrb_split_clusters_host
// in api.cu, which the tests compare it with): for every empty cluster ci, walk the clusters
// round-robin and pick cj with probability (size_cj - 1) / (n - k) using std::mt19937(1234)
// (restated below: MT19937 of Matsumoto & Nishimura with the standard tempering), copy cj's centroid
// to ci and perturb the pair symmetrically by +-1/1024, split the size. Thread 0 draws the
// (ci, cj) pairs in batches; the block applies each batch in order. stats[1] = imbalance factor
// k * sum(size^2) / n^2 of the assignment BEFORE the split, stats[2] = number of splits (-1 if no
// cluster could be split).
struct Mt19937Dev {
    uint32_t* s;  // 624 words of shared memory
    int idx;
    __device__ void seed(uint32_t v) {
        s[0] = v;
        for (int i = 1; i < 624; i++) s[i] = 1812433253u * (s[i - 1] ^ (s[i - 1] >> 30)) + (uint32_t)i;
        idx = 624;
    }
    __device__ uint32_t next() {
        if (idx >= 624) {
            for (int i = 0; i < 624; i++) {
                const uint32_t y = (s[i] & 0x80000000u) | (s[(i + 1) % 624] & 0x7fffffffu);
                s[i] = s[(i + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
            }
            idx = 0;
        }
        uint32_t y = s[idx++];
        y ^= y >> 11;
        y ^= (y << 7) & 0x9d2c5680u;
        y ^= (y << 15) & 0xefc60000u;
        y ^= y >> 18;
        return y;
    }
};

constexpr int KM_SPLIT_BATCH = 512;

__global__ void km_split_kernel(int d, int k, int64_t n, float* __restrict__ hassign, float* __restrict__ centroids,
                                double* __restrict__ stats) {
    __shared__ uint32_t mt_state[624];
    __shared__ int pair_ci[KM_SPLIT_BATCH], pair_cj[KM_SPLIT_BATCH];
    __shared__ int npairs, next_ci, any_empty, failed;
    __shared__ double red[1024];
    // imbalance factor + "is any cluster empty"
    double s2 = 0;
    int empty = 0;
    for (int c = threadIdx.x; c < k; c += blockDim.x) {
        const double h = hassign[c];
        s2 += h * h;
        empty |= (h == 0.0) ? 1 : 0;
    }
    red[threadIdx.x] = s2;
    if (threadIdx.x == 0) { any_empty = 0; next_ci = 0; failed = 0; }
    __syncthreads();
    if (empty) any_empty = 1;
    for (int o = blockDim.x >> 1; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        stats[1] = red[0] * (double)k / ((double)n * (double)n);
        stats[2] = 0.0;
    }
    if (!any_empty) return;
    Mt19937Dev mt{mt_state, 624};
    if (threadIdx.x == 0) mt.seed(1234u);
    const double EPS = 1 / 1024.;
    int nsplit = 0;
    int cj = 0;  // (thread 0) faiss restarts cj at 0 for every empty cluster
    for (;;) {
        if (threadIdx.x == 0) {
            int np = 0;
            int ci = next_ci;
            for (; ci < k && np < KM_SPLIT_BATCH; ci++) {
                if (hassign[ci] != 0) continue;
                long long guard = 0;
                for (cj = 0;; cj = (cj + 1) % k) {
                    const float p = (float)(((double)hassign[cj] - 1.0) / (double)(float)(n - k));
                    const float r = (float)mt.next() / 4294967296.0f;
                    if (r < p) break;
                    if (++guard > 100000000LL) { failed = 1; break; }
                }
                if (failed) break;
                pair_ci[np] = ci;
                pair_cj[np] = cj;
                np++;
                hassign[ci] = hassign[cj] / 2;
                hassign[cj] -= hassign[ci];
            }
            next_ci = ci;
            npairs = np;
        }
        __syncthreads();
        const int np = npairs;
        for (int e = 0; e < np; e++) {
            float* a = centroids + (size_t)pair_ci[e] * d;
            float* b = centroids + (size_t)pair_cj[e] * d;
            for (int j = threadIdx.x; j < d; j += blockDim.x) {
                const float v = b[j];
                if (j % 2 == 0) {
                    a[j] = (float)((double)v * (1 + EPS));
                    b[j] = (float)((double)v * (1 - EPS));
                } else {
                    a[j] = (float)((double)v * (1 - EPS));
                    b[j] = (float)((double)v * (1 + EPS));
                }
            }
            __syncthreads();
        }
        nsplit += np;
        const bool done = next_ci >= k || failed;
        __syncthreads();
        if (done) break;
    }
    if (threadIdx.x == 0) stats[2] = failed ? -1.0 : (double)nsplit;
}

// ------------------------------------------------------------------- select / merge (K4)
// Every source list (a unit's partial row, or a shard's result row) is already best-first, so
// the final top-k is a k-way merge: one warp per query, lane l owns sources l, l+32, ...;
// each round the warp takes the best head (64-bit (key, idx) max via shuffles) and the owning
// lane advances that list. Results are parked in registers (result r in lane r%32) and written
// coalesced.
struct PartSource {  // partial rows produced by the distance+selection kernels
    const float* key;
    const int* idx;
    const int* src;  // [nq, S] partial row per (query, source) or -1
    int S, k;
    __device__ __forceinline__ int row(int64_t q, int s) const { return src[q * S + s]; }
    __device__ __forceinline__ uint64_t load(int64_t, int, int prow, int pos) const {
        const int64_t o = (int64_t)prow * k + pos;
        const int i = idx[o];
        return i >= 0 ? pack_cand(key[o], i) : empty_cand();
    }
};
struct ShardSource {  // per-shard final results [G, nq, k] with 64-bit ids (K4)
    const float* Dp;
    const int64_t* Ip;
    int64_t nq;
    int S, k, metric;
    __device__ __forceinline__ int row(int64_t, int s) const { return s; }
    __device__ __forceinline__ uint64_t load(int64_t q, int s, int, int pos) const {
        const int64_t o = ((int64_t)s * nq + q) * k + pos;
        if (Ip[o] < 0) return empty_cand();
        const float d = Dp[o];
        // the idx slot carries (source, position): ties between shards resolve by shard order,
        // which is ascending id order for a row-sharded catalog
        return pack_cand(metric == NRB_METRIC_L2 ? -d : d, s * k + pos);
    }
};

// Per-shard final results on the wire (catalog-sharded search, all-to-all by query range):
// P[s, q, pos] = (fp32 bits of D) << 32 | local row index (0xffffffff = no result); the global id is
// bases[s] + local index. 8 bytes per candidate instead of 12, one collective instead of two.
struct PackedShardSource {
    const uint64_t* P;
    int64_t nq;
    int S, k, metric;
    __device__ __forceinline__ int row(int64_t, int s) const { return s; }
    __device__ __forceinline__ uint64_t load(int64_t q, int s, int, int pos) const {
        const uint64_t e = P[((int64_t)s * nq + q) * k + pos];
        if ((uint32_t)e == 0xffffffffu) return empty_cand();
        const float d = __uint_as_float((uint32_t)(e >> 32));
        return pack_cand(metric == NRB_METRIC_L2 ? -d : d, s * k + pos);  // ties: shard order = ascending id
    }
};

template <int MAXL, typename Source>
__device__ __forceinline__ void warp_kway_merge(const Source& S, int64_t q, int k, int lane,
                                                uint64_t (&res)[4]) {
    uint64_t head[MAXL];
    int prow[MAXL], pos[MAXL];
#pragma unroll
    for (int j = 0; j < MAXL; j++) {
        const int s = lane + 32 * j;
        prow[j] = s < S.S ? S.row(q, s) : -1;
        pos[j] = 0;
        head[j] = prow[j] >= 0 ? S.load(q, s, prow[j], 0) : empty_cand();
    }
#pragma unroll
    for (int i = 0; i < 4; i++) res[i] = empty_cand();
    const uint64_t EMPTY = empty_cand();
    for (int r = 0; r < k; r++) {
        uint64_t best = head[0];
#pragma unroll
        for (int j = 1; j < MAXL; j++) best = head[j] > best ? head[j] : best;
        uint64_t w = best;
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) {
            const uint64_t t = shfl_xor_u64(w, o);
            w = t > w ? t : w;
        }
        if (w == EMPTY) break;  // every list exhausted (warp-uniform)
        const unsigned owners = __ballot_sync(0xffffffffu, best == w);
        const int owner = __ffs(owners) - 1;
        if (lane == (r & 31)) {
#pragma unroll
            for (int i = 0; i < 4; i++)
                if (i == (r >> 5)) res[i] = w;
        }
        if (lane == owner) {
            bool done = false;
#pragma unroll
            for (int j = 0; j < MAXL; j++) {
                if (!done && head[j] == w) {
                    done = true;
                    pos[j]++;
                    head[j] = pos[j] < k ? S.load(q, lane + 32 * j, prow[j], pos[j]) : EMPTY;
                }
            }
        }
    }
}

template <int MAXL>
__global__ void select_merge_kernel(PartSource S, int64_t nq, int metric,
                                    const int64_t* __restrict__ id_map, int64_t id_base,
                                    float* __restrict__ D, int64_t* __restrict__ I) {
    const int lane = threadIdx.x & 31;
    const int64_t q = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (q >= nq) return;
    uint64_t res[4];
    warp_kway_merge<MAXL>(S, q, S.k, lane, res);
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int r = i * 32 + lane;
        if (r < S.k) {
            const int idx = cand_idx(res[i]);
            const float key = cand_key(res[i]);
            if (idx < 0) {
                I[q * S.k + r] = -1;
                D[q * S.k + r] = (metric == NRB_METRIC_L2) ? FLT_MAX : -FLT_MAX;
            } else {
                I[q * S.k + r] = id_map ? id_map[idx] : (int64_t)idx + id_base;
                D[q * S.k + r] = (metric == NRB_METRIC_L2) ? -key : key;
            }
        }
    }
}

template <int MAXL>
__global__ void shard_merge_kernel(ShardSource S, float* __restrict__ D, int64_t* __restrict__ I) {
    const int lane = threadIdx.x & 31;
    const int64_t q = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (q >= S.nq) return;
    uint64_t res[4];
    warp_kway_merge<MAXL>(S, q, S.k, lane, res);
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int r = i * 32 + lane;
        if (r < S.k) {
            const int e = cand_idx(res[i]);
            if (e < 0) {
                I[q * S.k + r] = -1;
                D[q * S.k + r] = (S.metric == NRB_METRIC_L2) ? FLT_MAX : -FLT_MAX;
            } else {
                const int s = e / S.k, pos = e - s * S.k;
                const int64_t o = ((int64_t)s * S.nq + q) * S.k + pos;
                I[q * S.k + r] = S.Ip[o];
                D[q * S.k + r] = S.Dp[o];
            }
        }
    }
}

template <int MAXL>
__global__ void shard_merge_packed_kernel(PackedShardSource S, const int64_t* __restrict__ bases,
                                          float* __restrict__ D, int64_t* __restrict__ I) {
    const int lane = threadIdx.x & 31;
    const int64_t q = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (q >= S.nq) return;
    uint64_t res[4];
    warp_kway_merge<MAXL>(S, q, S.k, lane, res);
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int r = i * 32 + lane;
        if (r < S.k) {
            const int e = cand_idx(res[i]);
            if (e < 0) {
                I[q * S.k + r] = -1;
                D[q * S.k + r] = (S.metric == NRB_METRIC_L2) ? FLT_MAX : -FLT_MAX;
            } else {
                const int s = e / S.k, pos = e - s * S.k;
                const uint64_t v = S.P[((int64_t)s * S.nq + q) * S.k + pos];
                I[q * S.k + r] = bases[s] + (int64_t)(uint32_t)v;
                D[q * S.k + r] = __uint_as_float((uint32_t)(v >> 32));
            }
        }
    }
}

__global__ void pack_topk_kernel(const float* __restrict__ D, const int64_t* __restrict__ I, int64_t id_base,
                                 int64_t n, uint64_t* __restrict__ P) {
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t id = I[t];
        const uint32_t lo = id < 0 ? 0xffffffffu : (uint32_t)(id - id_base);
        P[t] = ((uint64_t)__float_as_uint(D[t]) << 32) | lo;
    }
}

// Gather + exact refine of the filter paths (NRB_PATH_TC1 / NRB_PATH_TC16). The filter kernels
// leave, per (unit, warpgroup, query row), an UNSORTED partial row of part_cnt candidates
// (estimate, idx): everything the unit saw above its running threshold. One warp per query:
//   1. gather the candidates of all S partial rows of the query into shared memory (keys as
//      ordered uints), dropping what is below the running cut;
//   2. bisection on the keys gives a lower bound lb of the k-th best estimate (count(key >= lb)
//      in [k, k+3]); cut = lb - margin; the survivors (key >= cut) provably contain the true
//      top-k (|estimate - score| <= margin / 2 for every item);
//   3. exact fp32 rescoring of the survivors from the raw planes (coalesced float4 row reads +
//      warp reduction), bitonic sort by (exact key, idx), write the best k.
// When the staging buffer fills up mid-gather, step 2 runs early and raises the cut. flags[q] is
// raised when more than 128 candidates survive, the buffer overflows even after a reduction, or an
// exact score disagrees with its estimate by more than the assumed error bound; flagged queries
// are recomputed by the 3xTF32 kernel.
constexpr int GR_CAP = 512;  // staged candidates per warp
constexpr int GR_WPB = 4;    // warps (queries) per block

// lower bound of the k-th largest of su[0..n) (ordered uints, n >= k): count(su >= lb) in [k, k+3]
// or exact
__device__ __forceinline__ uint32_t warp_kth_bound(const uint32_t* su, int n, int k, int lane) {
    uint32_t mn = 0xffffffffu, mx = 0u;
    for (int e = lane; e < n; e += 32) {
        const uint32_t v = su[e];
        mn = v < mn ? v : mn;
        mx = v > mx ? v : mx;
    }
    mn = __reduce_min_sync(0xffffffffu, mn);
    mx = __reduce_max_sync(0xffffffffu, mx);
    uint32_t lo = mn, hi = mx + 1u;  // invariant: count(>= lo) >= k > count(>= hi)   (hi may wrap to 0 only for NaN payloads; keys are finite or -inf)
    if (hi == 0u) hi = 0xffffffffu;
    while (hi - lo > 1u) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        int c = 0;
        for (int e = lane; e < n; e += 32) c += (su[e] >= mid) ? 1 : 0;
        c = __reduce_add_sync(0xffffffffu, c);
        if (c >= k) {
            lo = mid;
            if (c <= k + 3) break;
        } else {
            hi = mid;
        }
    }
    return lo;
}

// keeps the entries with su >= cut_u, in place (order preserved); returns the new count
__device__ __forceinline__ int warp_compact_ge(uint32_t* su, int* si, int n, uint32_t cut_u, int lane) {
    const uint32_t lt = (1u << lane) - 1u;
    int w = 0;
    for (int base = 0; base < n; base += 32) {
        const int e = base + lane;
        const uint32_t v = e < n ? su[e] : 0u;
        const int id = e < n ? si[e] : -1;
        const bool keep = e < n && v >= cut_u;
        const uint32_t b = __ballot_sync(0xffffffffu, keep);
        __syncwarp();  // every lane has read its entry of this chunk; writes go to positions <= base + lane
        if (keep) {
            const int pos = w + __popc(b & lt);
            su[pos] = v;
            si[pos] = id;
        }
        w += __popc(b);
        __syncwarp();
    }
    return w;
}

template <bool L2>
__global__ void __launch_bounds__(GR_WPB * 32)
gather_refine_kernel(const float* __restrict__ part_key, const int* __restrict__ part_idx,
                     const int* __restrict__ part_cnt, const int* __restrict__ src, int S, int pw, int64_t nq, int k,
                     const float* __restrict__ q_raw, const float* __restrict__ q_norms,
                     const float* __restrict__ b_raw, const float* __restrict__ b_norms, int kp, float eps_xmax,
                     int64_t id_base, const int64_t* __restrict__ id_map, int* __restrict__ flags,
                     float* __restrict__ D, int64_t* __restrict__ I) {
    __shared__ uint32_t s_key[GR_WPB][GR_CAP];
    __shared__ int s_idx[GR_WPB][GR_CAP];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t q = (int64_t)blockIdx.x * GR_WPB + w;
    if (q >= nq) return;
    uint32_t* su = s_key[w];
    int* si = s_idx[w];
    const uint32_t lt = (1u << lane) - 1u;
    const float qn = q_norms[q];
    const float ebound = eps_xmax * sqrtf(qn) * (L2 ? 2.f : 1.f);
    const float margin = 2.f * ebound;
    bool bad = false;
    int fill = 0;
    uint32_t cut_u = 0u;  // entries below it are dropped (0 = below everything)
    for (int s0 = 0; s0 < S; s0 += 32) {
        const int s = s0 + lane;
        const int prow = s < S ? src[q * S + s] : -1;
        const int c = prow >= 0 ? part_cnt[prow] : 0;
        unsigned m = __ballot_sync(0xffffffffu, c > 0);
        while (m) {  // warp-uniform
            const int l = __ffs(m) - 1;
            m &= m - 1;
            const int pr = __shfl_sync(0xffffffffu, prow, l);
            const int cc = __shfl_sync(0xffffffffu, c, l);
            if (fill + cc > GR_CAP) {  // staging buffer full: raise the cut from what is there
                if (fill >= k) {
                    const uint32_t lb = warp_kth_bound(su, fill, k, lane);
                    const uint32_t nc = ordered_u32(from_ordered_u32(lb) - margin);
                    cut_u = nc > cut_u ? nc : cut_u;
                    fill = warp_compact_ge(su, si, fill, cut_u, lane);
                }
                if (fill + cc > GR_CAP) {  // still no room (a huge margin set): recompute exactly
                    bad = true;
                    break;
                }
            }
            const int64_t o = (int64_t)pr * pw;
            for (int e0 = 0; e0 < cc; e0 += 32) {
                const int e = e0 + lane;
                uint32_t v = 0u;
                int id = -1;
                if (e < cc) {
                    v = ordered_u32(part_key[o + e]);
                    id = part_idx[o + e];
                }
                const bool keep = e < cc && v >= cut_u;
                const uint32_t b = __ballot_sync(0xffffffffu, keep);
                if (keep) {
                    const int pos = fill + __popc(b & lt);
                    su[pos] = v;
                    si[pos] = id;
                }
                fill += __popc(b);
            }
            __syncwarp();
        }
        if (bad) break;
    }
    __syncwarp();
    if (fill > k) {
        const uint32_t lb = warp_kth_bound(su, fill, k, lane);
        const uint32_t nc = ordered_u32(from_ordered_u32(lb) - margin);
        cut_u = nc > cut_u ? nc : cut_u;
        fill = warp_compact_ge(su, si, fill, cut_u, lane);
    }
    int nv = fill;
    if (nv > 128) {  // more survivors than the exact stage holds
        bad = true;
        nv = 128;
    }
    // query row in registers
    const int w4 = kp >> 2;
    float4 qv[2];
#pragma unroll
    for (int j = 0; j < 2; j++) {
        const int c = lane + 32 * j;
        qv[j] = c < w4 ? __ldg(reinterpret_cast<const float4*>(q_raw + q * kp) + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    uint64_t ex[4];
#pragma unroll
    for (int i = 0; i < 4; i++) ex[i] = empty_cand();
#pragma unroll
    for (int i = 0; i < 4; i++) {
        for (int l = 0; l < 32; l++) {
            const int r = i * 32 + l;
            if (r >= nv) break;  // warp-uniform
            const int idx = si[r];
            const float approx = from_ordered_u32(su[r]);
            const float4* xr = reinterpret_cast<const float4*>(b_raw + (int64_t)idx * kp);
            float acc = 0.f;
#pragma unroll
            for (int j = 0; j < 2; j++) {
                const int c = lane + 32 * j;
                if (c < w4) {
                    const float4 xv = __ldg(xr + c);
                    acc = fmaf(qv[j].x, xv.x, acc);
                    acc = fmaf(qv[j].y, xv.y, acc);
                    acc = fmaf(qv[j].z, xv.z, acc);
                    acc = fmaf(qv[j].w, xv.w, acc);
                }
            }
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
            float key = acc;
            if (L2) key = -fmaxf(qn + b_norms[idx] - 2.f * acc, 0.f);
            if (fabsf(key - approx) > ebound) bad = true;
            if (lane == l) ex[i] = pack_cand(key, idx);
        }
    }
    warp_bitonic_desc<4>(ex, lane);
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int r = i * 32 + lane;
        if (r < k) {
            const int idx = cand_idx(ex[i]);
            const float key = cand_key(ex[i]);
            if (idx < 0) {
                I[q * k + r] = -1;
                D[q * k + r] = L2 ? FLT_MAX : -FLT_MAX;
            } else {
                I[q * k + r] = id_map ? id_map[idx] : (int64_t)idx + id_base;
                D[q * k + r] = L2 ? -key : key;
            }
        }
    }
    if (bad && lane == 0) flags[q] = 1;
}

__global__ void compact_flags_kernel(const int* __restrict__ flags, int64_t n, int* __restrict__ list,
                                     int* __restrict__ count) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        if (flags[i]) list[atomicAdd(count, 1)] = (int)i;
}

__global__ void scatter_results_kernel(const float* __restrict__ Df, const int64_t* __restrict__ If,
                                       const int* __restrict__ list, int n, int k, float* __restrict__ D,
                                       int64_t* __restrict__ I) {
    const int64_t total = (int64_t)n * k;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int i = (int)(t / k), j = (int)(t - (int64_t)i * k);
        const int64_t o = (int64_t)list[i] * k + j;
        D[o] = Df[t];
        I[o] = If[t];
    }
}

// Units + src table of the flat search (plan in api.cu: plan_flat). Pair p < full_pairs: units
// 2p, 2p+1 = query tiles 2p, 2p+1 against the whole catalog. Tail pair j, chunk c: pair index
// full_pairs + c*tail_pairs + j = query tiles 2(full_pairs + j) (+1) against item chunk c.
// A unit whose query tile does not exist (odd tile count) is a phantom with a_rows = 0.
// Partial row of (unit u, warpgroup g, row r) = (u*wgs + g)*128 + r.
__global__ void fill_flat_units_kernel(Unit* __restrict__ units, int* __restrict__ n_units_out,
                                       int* __restrict__ src, int64_t nq, int64_t nb, int nqt,
                                       int full_pairs, int tail_pairs, int tsplit, int chunk_rows, int wgs) {
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nunits = 2 * ((int64_t)full_pairs + (int64_t)tail_pairs * tsplit);
    if (tid == 0) *n_units_out = (int)nunits;
    if (tid < nunits) {
        const int pair = (int)(tid >> 1), r = (int)(tid & 1);
        int t, c;  // query tile, item chunk (-1 = whole catalog)
        if (pair < full_pairs) {
            t = 2 * pair + r;
            c = -1;
        } else {
            const int tp = pair - full_pairs;
            c = tp / tail_pairs;
            t = 2 * (full_pairs + tp % tail_pairs) + r;
        }
        Unit u;
        const int64_t ar = nq - (int64_t)t * UNIT_ROWS;
        u.a_rows = t < nqt ? (int)(ar < UNIT_ROWS ? ar : UNIT_ROWS) : 0;
        u.a_row0 = t < nqt ? t * UNIT_ROWS : 0;
        if (c < 0) {
            u.b_row0 = 0;
            u.b_rows = (int)nb;
        } else {
            u.b_row0 = c * chunk_rows;
            const int64_t br = nb - (int64_t)c * chunk_rows;
            u.b_rows = (int)(br < chunk_rows ? (br > 0 ? br : 0) : chunk_rows);
        }
        units[tid] = u;
    }
    const int S = tsplit * wgs;
    const int64_t total = nq * S;
    for (int64_t e = tid; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t q = e / S;
        const int sl = (int)(e - q * S);
        const int c = sl / wgs, g = sl - c * wgs;
        const int t = (int)(q / UNIT_ROWS), pair = t >> 1, r = t & 1;
        int64_t u = -1;
        if (pair < full_pairs) {
            if (c == 0) u = 2 * (int64_t)pair + r;
        } else {
            u = 2 * ((int64_t)full_pairs + (int64_t)c * tail_pairs + (pair - full_pairs)) + r;
        }
        src[e] = u < 0 ? -1 : (int)((u * wgs + g) * UNIT_ROWS + q % UNIT_ROWS);
    }
}

// Single-CTA plan of the flat search: unit c*nqt + t = query tile t against item chunk c.
__global__ void fill_flat_units_single_kernel(Unit* __restrict__ units, int* __restrict__ n_units_out,
                                              int* __restrict__ src, int64_t nq, int64_t nb, int nqt, int tsplit,
                                              int chunk_rows, int wgs) {
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nunits = (int64_t)nqt * tsplit;
    if (tid == 0) *n_units_out = (int)nunits;
    if (tid < nunits) {
        const int c = (int)(tid / nqt), t = (int)(tid - (int64_t)c * nqt);
        Unit u;
        const int64_t ar = nq - (int64_t)t * UNIT_ROWS;
        u.a_rows = (int)(ar < UNIT_ROWS ? ar : UNIT_ROWS);
        u.a_row0 = t * UNIT_ROWS;
        u.b_row0 = c * chunk_rows;
        const int64_t br = nb - (int64_t)c * chunk_rows;
        u.b_rows = (int)(br < chunk_rows ? (br > 0 ? br : 0) : chunk_rows);
        units[tid] = u;
    }
    const int S = tsplit * wgs;
    const int64_t total = nq * S;
    for (int64_t e = tid; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t q = e / S;
        const int sl = (int)(e - q * S);
        const int c = sl / wgs, g = sl - c * wgs;
        const int64_t u = (int64_t)c * nqt + q / UNIT_ROWS;
        src[e] = (int)((u * wgs + g) * UNIT_ROWS + q % UNIT_ROWS);
    }
}

// ------------------------------------------------------------------- host launchers
int launch_select(const float* part_key, const int* part_idx, const int* src, int S, int64_t nq,
                  int k, int metric, const int64_t* id_map, int64_t id_base, float* D, int64_t* I,
                  cudaStream_t st) {
    if (nq == 0) return NRB_OK;
    NRB_REQUIRE(S >= 1 && S <= 256 && k >= 1 && k <= 128, "select: S=%d (<=256) k=%d (<=128)", S, k);
    PartSource ps{part_key, part_idx, src, S, k};
    const int wpb = 8;
    const unsigned blocks = (unsigned)((nq + wpb - 1) / wpb);
    if (S <= 32)
        select_merge_kernel<1><<<blocks, wpb * 32, 0, st>>>(ps, nq, metric, id_map, id_base, D, I);
    else if (S <= 64)
        select_merge_kernel<2><<<blocks, wpb * 32, 0, st>>>(ps, nq, metric, id_map, id_base, D, I);
    else if (S <= 128)
        select_merge_kernel<4><<<blocks, wpb * 32, 0, st>>>(ps, nq, metric, id_map, id_base, D, I);
    else
        select_merge_kernel<8><<<blocks, wpb * 32, 0, st>>>(ps, nq, metric, id_map, id_base, D, I);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

int launch_gather_refine(const float* part_key, const int* part_idx, const int* part_cnt, const int* src, int S,
                         int64_t nq, int k, int pw, int metric, const nrb_matrix* q, const nrb_matrix* b, float eps_xmax,
                         int64_t id_base, const int64_t* id_map, int* flags, float* D, int64_t* I, cudaStream_t st) {
    if (nq == 0) return NRB_OK;
    NRB_REQUIRE(S >= 1 && pw <= 128 && k <= pw && q->kp <= 256, "gather_refine: S=%d pw=%d kp=%d", S, pw, q->kp);
    const unsigned blocks = (unsigned)((nq + GR_WPB - 1) / GR_WPB);
    if (metric == NRB_METRIC_L2)
        gather_refine_kernel<true><<<blocks, GR_WPB * 32, 0, st>>>(part_key, part_idx, part_cnt, src, S, pw, nq, k, q->raw,
                                                                    q->norms, b->raw, b->norms, q->kp, eps_xmax, id_base,
                                                                    id_map, flags, D, I);
    else
        gather_refine_kernel<false><<<blocks, GR_WPB * 32, 0, st>>>(part_key, part_idx, part_cnt, src, S, pw, nq, k, q->raw,
                                                                     q->norms, b->raw, b->norms, q->kp, eps_xmax, id_base,
                                                                     id_map, flags, D, I);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

int launch_compact_flags(const int* flags, int64_t n, int* list, int* count, cudaStream_t st) {
    NRB_CUDA_CHECK(cudaMemsetAsync(count, 0, sizeof(int), st));
    if (n == 0) return NRB_OK;
    int64_t blocks = (n + 255) / 256;
    if (blocks > 1024) blocks = 1024;
    compact_flags_kernel<<<(unsigned)blocks, 256, 0, st>>>(flags, n, list, count);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

int launch_scatter_results(const float* Df, const int64_t* If, const int* list, int n, int k, float* D,
                           int64_t* I, cudaStream_t st) {
    if (n == 0) return NRB_OK;
    int64_t blocks = ((int64_t)n * k + 255) / 256;
    if (blocks > 4096) blocks = 4096;
    scatter_results_kernel<<<(unsigned)blocks, 256, 0, st>>>(Df, If, list, n, k, D, I);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

int launch_fill_flat_units(Unit* units, int* n_units_out, int* src, int64_t nq, int64_t nb, int nqt,
                           int full_pairs, int tail_pairs, int tsplit, int chunk_rows, int wgs, cudaStream_t st) {
    const int64_t total = nq * tsplit * wgs;
    const int64_t nunits = 2 * ((int64_t)full_pairs + (int64_t)tail_pairs * tsplit);
    int64_t blocks = (total + 255) / 256;
    if (blocks > 4096) blocks = 4096;
    if (blocks < (nunits + 255) / 256) blocks = (nunits + 255) / 256;
    if (blocks < 1) blocks = 1;
    fill_flat_units_kernel<<<(unsigned)blocks, 256, 0, st>>>(units, n_units_out, src, nq, nb, nqt, full_pairs,
                                                             tail_pairs, tsplit, chunk_rows, wgs);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

int launch_fill_flat_units_single(Unit* units, int* n_units_out, int* src, int64_t nq, int64_t nb, int nqt,
                                  int tsplit, int chunk_rows, int wgs, cudaStream_t st) {
    const int64_t total = nq * tsplit * wgs;
    const int64_t nunits = (int64_t)nqt * tsplit;
    int64_t blocks = (total + 255) / 256;
    if (blocks > 4096) blocks = 4096;
    if (blocks < (nunits + 255) / 256) blocks = (nunits + 255) / 256;
    if (blocks < 1) blocks = 1;
    fill_flat_units_single_kernel<<<(unsigned)blocks, 256, 0, st>>>(units, n_units_out, src, nq, nb, nqt, tsplit,
                                                                    chunk_rows, wgs);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

size_t counting_sort_ws(int64_t n, int nb);
int launch_counting_sort_i64(const int64_t* key, int64_t n, int nb, int* offsets, int* order,
                             int* pos_of, void* ws, size_t ws_bytes, cudaStream_t st) {
    const int nchunks = (int)((n + CS_CHUNK - 1) / CS_CHUNK);
    const size_t need = counting_sort_ws(n, nb);
    if (ws_bytes < need) {
        set_error("counting sort: workspace %zu < %zu", ws_bytes, need);
        return NRB_ERR_WORKSPACE;
    }
    int* chunk_hist = (int*)ws;
    const size_t sh = (size_t)(nb + 2) * sizeof(int);
    NRB_REQUIRE(sh <= 48 * 1024, "counting sort: too many buckets (%d)", nb);
    if (nchunks > 0) {
        cs_hist_kernel<int64_t><<<nchunks, CS_THREADS, sh, st>>>(key, n, nb, chunk_hist);
        NRB_LAUNCH_CHECK();
    }
    if (nchunks > 4 * CS_GROUPS) {
        int* gtot = chunk_hist + (size_t)nchunks * (nb + 1);
        cs_group_tot_kernel<<<CS_GROUPS, 256, 0, st>>>(chunk_hist, nchunks, nb + 1, gtot);
        NRB_LAUNCH_CHECK();
        cs_group_scan_kernel<<<1, 512, sh, st>>>(gtot, nb, offsets);
        NRB_LAUNCH_CHECK();
        cs_group_prefix_kernel<<<CS_GROUPS, 256, 0, st>>>(chunk_hist, nchunks, nb + 1, gtot);
        NRB_LAUNCH_CHECK();
    } else {
        cs_scan_kernel<<<1, 512, sh, st>>>(chunk_hist, nchunks, nb, offsets);
        NRB_LAUNCH_CHECK();
    }
    if (nchunks > 0) {
        cs_scatter_kernel<int64_t><<<nchunks, CS_THREADS, sh, st>>>(key, n, nb, chunk_hist, order, pos_of);
        NRB_LAUNCH_CHECK();
    }
    return NRB_OK;
}

size_t counting_sort_ws(int64_t n, int nb) {
    const int64_t nchunks = (n + CS_CHUNK - 1) / CS_CHUNK;
    return align_up((size_t)((nchunks > 0 ? nchunks : 1) + CS_GROUPS) * (nb + 1) * sizeof(int), 256);
}

}  // namespace nrb

using namespace nrb;

extern "C" int nrb_pack_rows(const float* x, int64_t n, int32_t d, int64_t ldx, int32_t kp,
                             float* raw, float* hi, float* lo, float* norms, void* stream) {
    NRB_REQUIRE(n >= 0 && d > 0 && kp >= d && kp % 32 == 0 && ldx >= d,
                "pack_rows: bad shape n=%lld d=%d kp=%d ldx=%lld", (long long)n, d, kp, (long long)ldx);
    if (n == 0) return NRB_OK;
    int64_t blocks = (n + 7) / 8;
    if (blocks > 148 * 16) blocks = 148 * 16;
    pack_rows_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, n, d, ldx, kp, raw, hi, lo, norms);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

extern "C" int nrb_pack_rows_h16(const float* x, int64_t n, int32_t d, int64_t ldx, int32_t kp,
                                 float uniform_scale, void* h16, float* row_scale, void* stream) {
    NRB_REQUIRE(x && h16 && n >= 0 && d > 0 && kp >= d && kp % 32 == 0 && ldx >= d,
                "pack_rows_h16: bad shape n=%lld d=%d kp=%d ldx=%lld", (long long)n, d, kp, (long long)ldx);
    NRB_REQUIRE(uniform_scale > 0.f || row_scale, "pack_rows_h16: per-row scaling needs row_scale");
    if (n == 0) return NRB_OK;
    int64_t blocks = (n + 7) / 8;
    if (blocks > 148 * 16) blocks = 148 * 16;
    pack_rows_h16_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, n, d, ldx, kp, uniform_scale,
                                                                            (__half*)h16, row_scale);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

namespace nrb {
int launch_pack_rows(const float* x, int64_t n, int d, int64_t ldx, int kp, float* raw, float* hi, float* lo,
                     float* norms, cudaStream_t st) {
    return nrb_pack_rows(x, n, d, ldx, kp, raw, hi, lo, norms, (void*)st);
}
int launch_gather_rows(const float* src, int width, const int32_t* idx, int div, int64_t n,
                       float* dst, cudaStream_t st) {
    if (n == 0) return NRB_OK;
    int64_t total = n * (width / 4);
    int64_t blocks = (total + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    gather_rows_kernel<<<(unsigned)blocks, 256, 0, st>>>((const float4*)src, width / 4, idx, div, n, (float4*)dst);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}
int launch_gather_scalar(const float* src, const int32_t* idx, int div, int64_t n, float* dst,
                         cudaStream_t st) {
    if (n == 0) return NRB_OK;
    int64_t blocks = (n + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    gather_scalar_kernel<<<(unsigned)blocks, 256, 0, st>>>(src, idx, div, n, dst);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}
}  // namespace nrb

extern "C" int nrb_gather_rows(const float* src, int32_t width, const int32_t* idx, int64_t n,
                               float* dst, void* stream) {
    NRB_REQUIRE(width > 0 && width % 4 == 0 && n >= 0, "gather_rows: width %d must be a multiple of 4", width);
    return launch_gather_rows(src, width, idx, 1, n, dst, (cudaStream_t)stream);
}

extern "C" int nrb_gather_i64(const int64_t* src, const int32_t* idx, int64_t n, int64_t* dst,
                              void* stream) {
    if (n == 0) return NRB_OK;
    int64_t blocks = (n + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    gather_i64_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(src, idx, n, dst);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

extern "C" int nrb_normalize_l2(float* x, int64_t n, int32_t d, int64_t ldx, void* stream) {
    NRB_REQUIRE(n >= 0 && d > 0 && ldx >= d, "normalize_l2: bad shape");
    if (n == 0) return NRB_OK;
    int64_t blocks = (n + 7) / 8;
    if (blocks > 148 * 16) blocks = 148 * 16;
    normalize_l2_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, n, d, ldx);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

extern "C" size_t nrb_ivf_build_lists_workspace(int64_t n, int32_t nlist) {
    return counting_sort_ws(n, nlist);
}

extern "C" int nrb_ivf_build_lists(const int64_t* assign, int64_t n, int32_t nlist,
                                   int32_t* offsets, int32_t* order, void* workspace,
                                   size_t workspace_bytes, void* stream) {
    NRB_REQUIRE(n >= 0 && n < (1LL << 31) && nlist > 0, "ivf_build_lists: bad sizes");
    return launch_counting_sort_i64(assign, n, nlist, offsets, order, nullptr, workspace,
                                    workspace_bytes, (cudaStream_t)stream);
}

namespace nrb {

struct KmUpdateWs {
    void* cs;
    size_t cs_bytes;
    int *offsets, *order, *chunk_base;
    double *partial, *obj_part;
    size_t total;
};

static KmUpdateWs carve_km_update(void* ws, int64_t n, int k, int kp) {
    char* w = (char*)ws;
    size_t off = 0;
    auto take = [&](size_t bytes) { void* r = w ? w + off : nullptr; off += align_up(bytes, 256); return r; };
    KmUpdateWs u;
    u.cs_bytes = counting_sort_ws(n, k);
    u.cs = take(u.cs_bytes);
    u.offsets = (int*)take((size_t)(k + 2) * sizeof(int));
    u.order = (int*)take((size_t)(n > 0 ? n : 1) * sizeof(int));
    u.chunk_base = (int*)take((size_t)(k + 2) * sizeof(int));
    u.partial = (double*)take((size_t)(n / KM_CHUNK + k + 1) * kp * sizeof(double));
    u.obj_part = (double*)take((size_t)(n / KM_CHUNK + k + 1) * sizeof(double));
    u.total = off;
    return u;
}

size_t kmeans_update_ws(int64_t n, int k, int kp) { return carve_km_update(nullptr, n, k, kp).total; }

// centroids f32[k, d], hassign f32[k] from assign i64[n] (K1b): counting sort + plan + partial + finish
int launch_kmeans_update(const float* x_raw, int64_t n, int d, int kp, const int64_t* assign, int k, float* centroids,
                         float* hassign, void* workspace, const float* cent_in, int metric, double* obj_out,
                         cudaStream_t st, double* sums_out) {
    const KmUpdateWs u = carve_km_update(workspace, n, k, kp);
    int rc = launch_counting_sort_i64(assign, n, k, u.offsets, u.order, nullptr, u.cs, u.cs_bytes, st);
    if (rc) return rc;
    km_plan_kernel<<<1, 1024, 0, st>>>(u.offsets, k, u.chunk_base);
    NRB_LAUNCH_CHECK();
    const int w4 = kp / 4;
    int slices = 256 / w4;
    slices = slices < 1 ? 1 : (slices > 8 ? 8 : slices);
    const int threads = w4 * slices;
    NRB_REQUIRE(threads <= 1024, "kmeans_update: kp %d too large", kp);
    const size_t smem = (size_t)slices * kp * sizeof(double);
    const unsigned nchunks = (unsigned)(n / KM_CHUNK + k + 1);
    const bool obj = cent_in && obj_out;
    km_partial_kernel<<<nchunks, threads, smem, st>>>(x_raw, kp, u.offsets, u.order, u.chunk_base, k, slices, u.partial,
                                                      obj ? cent_in : nullptr, d, metric == NRB_METRIC_L2 ? 1 : 0,
                                                      obj ? u.obj_part : nullptr);
    NRB_LAUNCH_CHECK();
    km_finish_kernel<<<k, 256, 0, st>>>(u.partial, u.chunk_base, u.offsets, kp, d, k, centroids, hassign,
                                        obj ? u.obj_part : nullptr, obj ? obj_out : nullptr, sums_out);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

int launch_km_means(const double* sums, int k, int d, float* centroids, float* hassign, cudaStream_t st) {
    km_means_kernel<<<k, 256, 0, st>>>(sums, k, d, centroids, hassign);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

int launch_km_split(int d, int k, int64_t n, float* hassign, float* centroids, double* stats, cudaStream_t st) {
    km_split_kernel<<<1, 1024, 0, st>>>(d, k, n, hassign, centroids, stats);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

}  // namespace nrb

extern "C" size_t nrb_kmeans_update_workspace(int64_t n, int32_t k, int32_t kp) {
    return nrb::kmeans_update_ws(n, k, kp);
}

extern "C" int nrb_kmeans_update(const float* x_raw, int64_t n, int32_t d, int32_t kp,
                                 const int64_t* assign, int32_t k, float* centroids,
                                 float* hassign, void* workspace, size_t workspace_bytes,
                                 void* stream) {
    NRB_REQUIRE(n >= 0 && n < (1LL << 31) && k > 0 && d > 0 && kp >= d && kp % 32 == 0 && kp <= 2048,
                "kmeans_update: bad sizes n=%lld k=%d d=%d kp=%d", (long long)n, k, d, kp);
    if (workspace_bytes < nrb_kmeans_update_workspace(n, k, kp)) {
        set_error("kmeans_update: workspace too small");
        return NRB_ERR_WORKSPACE;
    }
    return nrb::launch_kmeans_update(x_raw, n, d, kp, assign, k, centroids, hassign, workspace, nullptr, 0, nullptr,
                                     (cudaStream_t)stream);
}

extern "C" int nrb_kmeans_partial_sums(const float* x_raw, int64_t n, int32_t d, int32_t kp, const int64_t* assign,
                                       int32_t k, double* sums, void* workspace, size_t workspace_bytes,
                                       void* stream) {
    NRB_REQUIRE(n >= 0 && n < (1LL << 31) && k > 0 && d > 0 && kp >= d && kp % 32 == 0 && kp <= 2048 && sums,
                "kmeans_partial_sums: bad arguments n=%lld k=%d d=%d kp=%d", (long long)n, k, d, kp);
    if (workspace_bytes < nrb_kmeans_update_workspace(n, k, kp)) {
        set_error("kmeans_partial_sums: workspace too small");
        return NRB_ERR_WORKSPACE;
    }
    return nrb::launch_kmeans_update(x_raw, n, d, kp, assign, k, nullptr, nullptr, workspace, nullptr, 0, nullptr,
                                     (cudaStream_t)stream, sums);
}

extern "C" int nrb_kmeans_means(const double* sums, int32_t k, int32_t d, float* centroids, float* hassign,
                                void* stream) {
    NRB_REQUIRE(sums && centroids && hassign && k > 0 && d > 0, "kmeans_means: bad arguments");
    return nrb::launch_km_means(sums, k, d, centroids, hassign, (cudaStream_t)stream);
}

extern "C" int nrb_split_clusters(int32_t d, int32_t k, int64_t n, float* hassign, float* centroids, double* stats3,
                                  void* stream) {
    NRB_REQUIRE(hassign && centroids && stats3 && d > 0 && k > 0 && n > k, "split_clusters: bad arguments");
    return nrb::launch_km_split(d, k, n, hassign, centroids, stats3, (cudaStream_t)stream);
}

extern "C" int nrb_merge_topk(const float* Dp, const int64_t* Ip, int32_t nparts, int64_t nq,
                              int32_t k, int32_t metric, float* D, int64_t* I, void* stream) {
    NRB_REQUIRE(nparts > 0 && nparts <= 256 && nq >= 0 && k > 0 && k <= 128, "merge_topk: bad sizes");
    NRB_REQUIRE((int64_t)nparts * k < (1LL << 31), "merge_topk: nparts*k too large");
    if (nq == 0) return NRB_OK;
    ShardSource ss{Dp, Ip, nq, nparts, k, metric};
    const int wpb = 8;
    const unsigned blocks = (unsigned)((nq + wpb - 1) / wpb);
    cudaStream_t st = (cudaStream_t)stream;
    if (nparts <= 32)
        shard_merge_kernel<1><<<blocks, wpb * 32, 0, st>>>(ss, D, I);
    else if (nparts <= 64)
        shard_merge_kernel<2><<<blocks, wpb * 32, 0, st>>>(ss, D, I);
    else if (nparts <= 128)
        shard_merge_kernel<4><<<blocks, wpb * 32, 0, st>>>(ss, D, I);
    else
        shard_merge_kernel<8><<<blocks, wpb * 32, 0, st>>>(ss, D, I);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

extern "C" int nrb_pack_topk(const float* D, const int64_t* I, int64_t id_base, int64_t n, uint64_t* P,
                             void* stream) {
    NRB_REQUIRE(n >= 0 && (n == 0 || (D && I && P)), "pack_topk: bad arguments");
    if (n == 0) return NRB_OK;
    int64_t blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    pack_topk_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(D, I, id_base, n, P);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

extern "C" int nrb_merge_topk_packed(const uint64_t* P, const int64_t* bases, int32_t nparts, int64_t nq,
                                     int32_t k, int32_t metric, float* D, int64_t* I, void* stream) {
    NRB_REQUIRE(nparts > 0 && nparts <= 256 && nq >= 0 && k > 0 && k <= 128, "merge_topk_packed: bad sizes");
    NRB_REQUIRE((int64_t)nparts * k < (1LL << 31), "merge_topk_packed: nparts*k too large");
    if (nq == 0) return NRB_OK;
    NRB_REQUIRE(P && bases && D && I, "merge_topk_packed: null argument");
    PackedShardSource ss{P, nq, nparts, k, metric};
    const int wpb = 8;
    const unsigned blocks = (unsigned)((nq + wpb - 1) / wpb);
    cudaStream_t st = (cudaStream_t)stream;
    if (nparts <= 32)
        shard_merge_packed_kernel<1><<<blocks, wpb * 32, 0, st>>>(ss, bases, D, I);
    else if (nparts <= 64)
        shard_merge_packed_kernel<2><<<blocks, wpb * 32, 0, st>>>(ss, bases, D, I);
    else if (nparts <= 128)
        shard_merge_packed_kernel<4><<<blocks, wpb * 32, 0, st>>>(ss, bases, D, I);
    else
        shard_merge_packed_kernel<8><<<blocks, wpb * 32, 0, st>>>(ss, bases, D, I);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

// ------------------------------------------------------------------- article table (SURVEY 8f row 1)
// Retrieval.py:6-8 on the device: news/article_table.npy is a float64 table whose rows are the
// embedding values followed by the article id. One pass: ids[i] = (int64) t[i, w-1],
// emb[i, :] = (float) t[i, :w-1] (C-contiguous, row stride w-1) -- the two .astype() copies and
// np.ascontiguousarray of the script as one HBM-bound kernel (reads n*w*8 bytes).
__global__ void split_table_f64_kernel(const double* __restrict__ t, int64_t n, int w, float* __restrict__ emb,
                                       int64_t* __restrict__ ids) {
    const int d = w - 1;
    const int64_t total = n * (int64_t)w;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = e / w;
        const int c = (int)(e - i * w);
        const double v = t[e];
        if (c == d)
            ids[i] = (int64_t)v;
        else
            emb[i * d + c] = (float)v;
    }
}

extern "C" int nrb_split_table_f64(const double* table, int64_t n, int32_t width, float* emb, int64_t* ids, void* stream) {
    NRB_REQUIRE(n >= 0 && width >= 2 && (n == 0 || (table && emb && ids)), "split_table_f64: bad arguments");
    if (n == 0) return NRB_OK;
    int64_t blocks = (n * width + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    split_table_f64_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(table, n, width, emb, ids);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

// ------------------------------------------------------------------- candidate lists (SURVEY 8f)
// Retrieval.py:33-34 batched: user u gets the whole inverted list of its nearest centroid.
// Warp per user: out[out_off[u] + j] = list_ids[list_off[l_u] + j].
__global__ void expand_lists_kernel(const int64_t* __restrict__ user_list, const int32_t* __restrict__ list_off,
                                    const int64_t* __restrict__ list_ids, const int64_t* __restrict__ out_off,
                                    int64_t nu, int64_t* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t u = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (u >= nu) return;
    const int64_t l = user_list[u];
    if (l < 0) return;
    const int b = list_off[l], e = list_off[l + 1];
    int64_t* dst = out + out_off[u];
    for (int j = lane; j < e - b; j += 32) dst[j] = list_ids[b + j];
}

// utils.py:12-17 / finialize_retrieval.py:10-11: is target[u] in row u of the CSR (off, ids)?
__global__ void csr_contains_kernel(const int64_t* __restrict__ off, const int64_t* __restrict__ ids,
                                    const int64_t* __restrict__ target, int64_t nrows,
                                    uint8_t* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t u = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (u >= nrows) return;
    const int64_t t = target[u];
    bool hit = false;
    for (int64_t j = off[u] + lane; j < off[u + 1]; j += 32) hit |= (ids[j] == t);
    hit = __any_sync(0xffffffffu, hit);
    if (lane == 0) out[u] = hit ? 1 : 0;
}

extern "C" int nrb_expand_lists(const int64_t* user_list, const int32_t* list_off, const int64_t* list_ids,
                                const int64_t* out_off, int64_t nu, int64_t* out, void* stream) {
    NRB_REQUIRE(nu >= 0, "expand_lists: bad size");
    if (nu == 0) return NRB_OK;
    expand_lists_kernel<<<(unsigned)((nu + 7) / 8), 256, 0, (cudaStream_t)stream>>>(user_list, list_off, list_ids,
                                                                                   out_off, nu, out);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

extern "C" int nrb_csr_contains(const int64_t* off, const int64_t* ids, const int64_t* target, int64_t nrows,
                                uint8_t* out, void* stream) {
    NRB_REQUIRE(nrows >= 0, "csr_contains: bad size");
    if (nrows == 0) return NRB_OK;
    csr_contains_kernel<<<(unsigned)((nrows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(off, ids, target, nrows, out);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

// ------------------------------------------------------------------- id selectors (faiss IDSelector*)
// Retrieval.py:7,23 keep the article ids in a second array beside the index; these two entry points
// let the index carry them (IndexIDMap, IndexIVFFlat.add_with_ids) and drop rows by id (remove_ids).
// IDSelectorBatch is an open-addressing hash table with linear probing in the workspace: a power-of-two
// capacity of at least twice the batch (load factor <= 1/2), empty slots hold ID_EMPTY, and a batch
// entry equal to ID_EMPTY sets the flag word instead of occupying a slot.
constexpr int64_t ID_EMPTY = -1;  // workspace is cleared with cudaMemsetAsync(0xff)

static int64_t id_table_cap(int64_t nbatch) {
    int64_t cap = 64;
    while (cap < 2 * nbatch) cap <<= 1;
    return cap;
}

__device__ __forceinline__ uint64_t id_hash(int64_t v) {  // splitmix64 finaliser
    uint64_t z = (uint64_t)v;
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
}

__global__ void id_insert_kernel(const int64_t* __restrict__ batch, int64_t nbatch, unsigned long long* table,
                                 uint64_t mask, int* has_empty) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nbatch; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t v = batch[i];
        if (v == ID_EMPTY) {
            *has_empty = 1;
            continue;
        }
        for (uint64_t s = id_hash(v) & mask;; s = (s + 1) & mask) {
            const unsigned long long prev = atomicCAS(table + s, (unsigned long long)ID_EMPTY, (unsigned long long)v);
            if (prev == (unsigned long long)ID_EMPTY || prev == (unsigned long long)v) break;
        }
    }
}

// member[i] = 1 if the id of row i (ids[i], or i when ids == NULL) is selected. table == NULL: range.
__global__ void id_member_kernel(const int64_t* __restrict__ ids, int64_t n, const int64_t* __restrict__ table,
                                 uint64_t mask, const int* __restrict__ has_empty, int64_t imin, int64_t imax,
                                 int64_t* __restrict__ member) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t v = ids ? ids[i] : i;
        int64_t m;
        if (!table) {
            m = imin <= v && v < imax;
        } else if (v == ID_EMPTY) {
            m = *has_empty;
        } else {
            m = 0;
            for (uint64_t s = id_hash(v) & mask;; s = (s + 1) & mask) {
                const int64_t t = table[s];
                if (t == v) { m = 1; break; }
                if (t == ID_EMPTY) break;
            }
        }
        member[i] = m;
    }
}

__global__ void map_ids_kernel(const int64_t* __restrict__ id_map, int64_t* __restrict__ I, int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t v = I[i];
        if (v >= 0) I[i] = id_map[v];
    }
}

extern "C" size_t nrb_id_select_workspace(int64_t nbatch) {
    if (nbatch <= 0) return 0;
    return 256 + (size_t)id_table_cap(nbatch) * sizeof(int64_t);
}

extern "C" int nrb_id_select(const int64_t* ids, int64_t n, const int64_t* batch, int64_t nbatch, int64_t imin,
                             int64_t imax, int64_t* member, void* workspace, size_t workspace_bytes, void* stream) {
    NRB_REQUIRE(n >= 0 && nbatch >= 0 && nbatch < (1LL << 40), "id_select: bad sizes n=%lld nbatch=%lld",
                (long long)n, (long long)nbatch);
    NRB_REQUIRE(batch || nbatch == 0, "id_select: nbatch=%lld with no batch", (long long)nbatch);
    NRB_REQUIRE(n == 0 || member, "id_select: null member");
    if (batch && nbatch == 0) {  // an empty batch selects nothing: the empty range
        batch = nullptr;
        imin = imax = 0;
    }
    const size_t need = batch ? nrb_id_select_workspace(nbatch) : 0;
    if (workspace_bytes < need || (need && !workspace)) {
        set_error("id_select: workspace %zu < %zu", workspace_bytes, need);
        return NRB_ERR_WORKSPACE;
    }
    if (n == 0) return NRB_OK;
    int rc = require_device();
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t* table = nullptr;
    const int* has_empty = nullptr;
    uint64_t mask = 0;
    if (batch) {
        const int64_t cap = id_table_cap(nbatch);
        int* flag = (int*)workspace;
        unsigned long long* tab = (unsigned long long*)((char*)workspace + 256);
        NRB_CUDA_CHECK(cudaMemsetAsync(flag, 0, sizeof(int), st));
        NRB_CUDA_CHECK(cudaMemsetAsync(tab, 0xff, (size_t)cap * sizeof(int64_t), st));
        mask = (uint64_t)cap - 1;
        int64_t blocks = (nbatch + 255) / 256;
        if (blocks > 148 * 16) blocks = 148 * 16;
        id_insert_kernel<<<(unsigned)blocks, 256, 0, st>>>(batch, nbatch, tab, mask, flag);
        NRB_LAUNCH_CHECK();
        table = (const int64_t*)tab;
        has_empty = flag;
    }
    int64_t blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    id_member_kernel<<<(unsigned)blocks, 256, 0, st>>>(ids, n, table, mask, has_empty, imin, imax, member);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}

extern "C" int nrb_map_ids(const int64_t* id_map, int64_t* I, int64_t n, void* stream) {
    NRB_REQUIRE(n >= 0 && (n == 0 || (id_map && I)), "map_ids: bad arguments");
    if (n == 0) return NRB_OK;
    int rc = require_device();
    if (rc) return rc;
    int64_t blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    map_ids_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(id_map, I, n);
    NRB_LAUNCH_CHECK();
    return NRB_OK;
}
