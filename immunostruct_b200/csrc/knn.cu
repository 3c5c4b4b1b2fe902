// Exact k-nearest-neighbour search of query rows in a bank of rows (neighbors.nearest).
//
// Contract (INTEGRATION 3, DESIGN 4.4i):
//   distance  squared Euclidean distance in fp32 with one rounding sequence per pair: acc = 0, then for d = 0 .. D-1 in
//             ascending order t = q_d - r_d, acc = fmaf(t, t, acc).  It does not depend on tiling, slicing or Q.  One
//             metric only: for cosine order pass L2-normalised rows (|a - b|^2 = 2 - 2 cos).
//   order     results ascending in the total order (distance, bank index); ties go to the smaller index.  The key of a
//             pair is (float_bits(distance) << 32) | index as uint64: for distance >= 0 the float bits order like the
//             floats, so the output is bit-identical whatever the launch configuration.
//   missing   a pair whose distance is NaN is never returned: a bank row with a NaN feature is never a neighbour and a
//             query with a NaN feature has none.  Unfilled slots (fewer than k eligible rows) hold index -1 and
//             distance +inf (the key 0x7f800000ffffffff, which sorts after every eligible pair, +inf distances included;
//             a NaN key sorts after it and so never enters a list).  exclude[q] (-1: none) is a bank row query q skips.
//
// Kernels (plain SIMT fp32, no floating-point atomics):
//   knn_partial_kernel  grid (query tiles of 64, bank slices S).  The CTA keeps its 64 queries in shared memory and
//                       walks its slice in 128-row x 32-feature chunks (the next chunk is prefetched into registers while
//                       the current one is used).  A thread owns 4 queries x 8 rows of distances in registers.  After
//                       each 128-row tile the pairs below the query's current k-th key are appended to its candidate
//                       list (shared counter: the append order does not matter, the sort is on a total order); when a
//                       list could overflow on the next tile, and at the end of the slice, one warp bitonic-sorts it and
//                       keeps the first k.  S = 1 writes the result, else the slice's sorted k keys go to the workspace.
//   knn_merge_kernel    one warp per query merges the S sorted lists, two at a time by a bitonic merge.
#include "common.cuh"

#include <stdint.h>

namespace is {

constexpr int KNN_QT = 64;                 // queries per CTA
constexpr int KNN_RT = 128;                // bank rows per tile
constexpr int KNN_DC = 32;                 // features per staged chunk
constexpr int KNN_LDR = KNN_DC + 4;        // padded row of the staged chunk: conflict-free float4 reads
constexpr int KNN_CAP = 256;               // per-query list: the running k best, then candidates
constexpr int KNN_KMAX = 64;
constexpr int KNN_DMAX = 256;
constexpr int KNN_SMAX = 65535;            // slices are gridDim.y
constexpr unsigned long long KNN_NONE = 0x7f800000ffffffffull;     // (+inf, -1)
constexpr unsigned long long KNN_PAD = ~0ull;                      // sort padding, after every real key

__device__ __forceinline__ int knn_pair_lo(int p, int stride) {   // first element of compare pair p at a power-of-2 stride
    return ((p & ~(stride - 1)) << 1) | (p & (stride - 1));
}

// ascending bitonic sort of a[0, n) by one warp, n a power of two
__device__ void knn_warp_sort(unsigned long long* a, int n, int lane) {
    for (int size = 2; size <= n; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int p = lane; p < (n >> 1); p += 32) {
                const int i = knn_pair_lo(p, stride), j = i + stride;
                const unsigned long long x = a[i], y = a[j];
                if ((x > y) == ((i & size) == 0)) { a[i] = y; a[j] = x; }
            }
            __syncwarp();
        }
}

__device__ __forceinline__ void knn_write(unsigned long long key, int64_t* index, float* distance, int64_t at) {
    const unsigned row = (unsigned)key;
    index[at] = row == 0xffffffffu ? -1 : (int64_t)row;
    distance[at] = __uint_as_float((unsigned)(key >> 32));
}

__global__ void __launch_bounds__(IS_THREADS, 1)
knn_partial_kernel(const float* __restrict__ query, const float* __restrict__ bank, const int64_t* __restrict__ exclude,
                   int Q, int R, int D, int k, int64_t rows_per_slice, int S, unsigned long long* __restrict__ ws,
                   int64_t* __restrict__ out_index, float* __restrict__ out_dist) {
    extern __shared__ __align__(16) unsigned char knn_smem[];
    const int DP = (D + KNN_DC - 1) / KNN_DC * KNN_DC;     // features padded to whole chunks with zeros: fmaf(0, 0, acc)
    const int LDQ = DP + 4;                                 // is acc exactly, so the padding changes no distance
    unsigned long long* list = reinterpret_cast<unsigned long long*>(knn_smem);     // [QT][CAP]
    unsigned long long* thresh = list + KNN_QT * KNN_CAP;                          // [QT] current k-th key
    int* cnt = reinterpret_cast<int*>(thresh + KNN_QT);                             // [QT] filled slots of list
    float* sq = reinterpret_cast<float*>(cnt + KNN_QT);                             // [QT][LDQ]
    float* sr = sq + KNN_QT * LDQ;                                                  // [RT][LDR]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tr = tid & 15, tq = tid >> 4;                 // rows tr + 16 j (j < 8), queries tq + 16 i (i < 4)
    const int q0 = blockIdx.x * KNN_QT, s = blockIdx.y;
    const int lo = (int)min((int64_t)R, s * rows_per_slice), hi = (int)min((int64_t)R, lo + rows_per_slice);

    for (int idx = tid; idx < KNN_QT * DP; idx += IS_THREADS) {
        const int q = idx / DP, d = idx - q * DP;
        sq[q * LDQ + d] = q0 + q < Q && d < D ? __ldg(query + (int64_t)(q0 + q) * D + d) : 0.0f;
    }
    for (int q = tid; q < KNN_QT; q += IS_THREADS) { thresh[q] = KNN_NONE; cnt[q] = k; }
    for (int idx = tid; idx < KNN_QT * k; idx += IS_THREADS) list[(idx / k) * KNN_CAP + idx % k] = KNN_NONE;
    int ex[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int q = q0 + tq + 16 * i;
        ex[i] = exclude != nullptr && q < Q ? (int)__ldg(exclude + q) : -1;
    }

    const int n_dc = DP / KNN_DC, n_tiles = (hi - lo + KNN_RT - 1) / KNN_RT, n_chunks = n_tiles * n_dc;
    constexpr int PER = KNN_RT * KNN_DC / IS_THREADS;      // staged floats per thread
    float pre[PER];
    auto load = [&](int c) {                                // chunk c = (tile c / n_dc, features (c % n_dc) * 32 + ..)
        const int t = c / n_dc, d0 = (c - t * n_dc) * KNN_DC;
#pragma unroll
        for (int m = 0; m < PER; ++m) {
            const int idx = tid + m * IS_THREADS, d = d0 + (idx & 31);
            const int64_t row = (int64_t)lo + t * KNN_RT + (idx >> 5);
            pre[m] = row < hi && d < D ? __ldg(bank + (int64_t)row * D + d) : 0.0f;
        }
    };
    auto store = [&]() {
#pragma unroll
        for (int m = 0; m < PER; ++m) {
            const int idx = tid + m * IS_THREADS;
            sr[(idx >> 5) * KNN_LDR + (idx & 31)] = pre[m];
        }
    };
    if (n_chunks > 0) load(0);
    float acc[4][8];
    for (int c = 0; c < n_chunks; ++c) {
        const int t = c / n_dc, dc = c - t * n_dc;
        __syncthreads();                                    // the previous chunk's readers are done
        store();
        __syncthreads();
        if (c + 1 < n_chunks) load(c + 1);                  // in flight while this chunk is used
        if (dc == 0) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;
        }
        const float* qs = sq + dc * KNN_DC;
#pragma unroll 2
        for (int d4 = 0; d4 < KNN_DC; d4 += 4) {
            float4 qv[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) qv[i] = *reinterpret_cast<const float4*>(qs + (tq + 16 * i) * LDQ + d4);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float4 rv = *reinterpret_cast<const float4*>(sr + (tr + 16 * j) * KNN_LDR + d4);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    float u = qv[i].x - rv.x;
                    acc[i][j] = fmaf(u, u, acc[i][j]);
                    u = qv[i].y - rv.y;
                    acc[i][j] = fmaf(u, u, acc[i][j]);
                    u = qv[i].z - rv.z;
                    acc[i][j] = fmaf(u, u, acc[i][j]);
                    u = qv[i].w - rv.w;
                    acc[i][j] = fmaf(u, u, acc[i][j]);
                }
            }
        }
        if (dc != n_dc - 1) continue;
        // the tile is complete: append the pairs below each query's current k-th key
        const int r0 = lo + t * KNN_RT;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int q = tq + 16 * i;
            if (q0 + q >= Q) continue;
            const unsigned long long th = thresh[q];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const unsigned row = (unsigned)r0 + tr + 16 * j;        // unsigned: a bank of up to 2^31 - 1 rows
                const unsigned long long key = ((unsigned long long)__float_as_uint(acc[i][j]) << 32) | row;
                if (row < (unsigned)hi && (int)row != ex[i] && key < th) list[q * KNN_CAP + atomicAdd(&cnt[q], 1)] = key;
            }
        }
        __syncthreads();
        // a list that could overflow on the next tile, and every list at the end of the slice: sort, keep the first k
        const bool last = t == n_tiles - 1;
        for (int q = warp; q < KNN_QT; q += IS_THREADS / 32) {
            const int n = cnt[q];
            if (n > KNN_CAP - KNN_RT || (last && n > k)) {
                int np = 2;
                while (np < n) np <<= 1;
                unsigned long long* a = list + q * KNN_CAP;
                for (int x = n + lane; x < np; x += 32) a[x] = KNN_PAD;
                __syncwarp();
                knn_warp_sort(a, np, lane);
                if (lane == 0) { cnt[q] = k; thresh[q] = a[k - 1]; }
                __syncwarp();
            }
        }
    }
    __syncthreads();
    for (int idx = tid; idx < KNN_QT * k; idx += IS_THREADS) {
        const int q = idx / k, x = idx - q * k;
        if (q0 + q >= Q) continue;
        const unsigned long long key = list[q * KNN_CAP + x];
        if (ws != nullptr) ws[((int64_t)(q0 + q) * S + s) * k + x] = key;
        else knn_write(key, out_index, out_dist, (int64_t)(q0 + q) * k + x);
    }
}

__global__ void __launch_bounds__(IS_THREADS)
knn_merge_kernel(const unsigned long long* __restrict__ ws, int Q, int S, int k, int64_t* __restrict__ out_index,
                 float* __restrict__ out_dist) {
    __shared__ unsigned long long buf[IS_THREADS / 32][2 * KNN_KMAX];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = blockIdx.x * (IS_THREADS / 32) + warp;
    if (q >= Q) return;                                     // warp-uniform; the kernel has no block barrier
    int kp = 1;
    while (kp < k) kp <<= 1;
    unsigned long long* a = buf[warp];
    const unsigned long long* src = ws + (int64_t)q * S * k;
    for (int x = lane; x < kp; x += 32) a[x] = x < k ? src[x] : KNN_PAD;
    for (int s = 1; s < S; ++s) {
        // [best ascending | list s descending] is bitonic: half-cleaners sort it, the first kp are the kp smallest
        for (int x = lane; x < kp; x += 32) a[kp + x] = kp - 1 - x < k ? src[(int64_t)s * k + kp - 1 - x] : KNN_PAD;
        __syncwarp();
        for (int stride = kp; stride > 0; stride >>= 1) {
            for (int p = lane; p < kp; p += 32) {
                const int i = knn_pair_lo(p, stride), j = i + stride;
                const unsigned long long x = a[i], y = a[j];
                if (x > y) { a[i] = y; a[j] = x; }
            }
            __syncwarp();
        }
    }
    for (int x = lane; x < k; x += 32) knn_write(a[x], out_index, out_dist, (int64_t)q * k + x);
}

size_t knn_smem_bytes(int D) {
    const int DP = (D + KNN_DC - 1) / KNN_DC * KNN_DC;
    return sizeof(unsigned long long) * (KNN_QT * KNN_CAP + KNN_QT) + sizeof(int) * KNN_QT +
           sizeof(float) * ((size_t)KNN_QT * (DP + 4) + KNN_RT * KNN_LDR);
}

}  // namespace is

using namespace is;

extern "C" {

// k nearest bank rows of every query (see the header of this file).  query [Q, D], bank [R, D] fp32 row-major;
// 1 <= k <= 64, 1 <= D <= 256, 1 <= R < 2^31; exclude [Q] int64 in [-1, R) or NULL.  slices S in
// [1, min(65535, ceil(R / 128))] (every slice holds a 128-row tile): S > 1 needs workspace [Q, S, k] uint64 and
// launches the merge kernel.
// -> index [Q, k] int64 (-1 = unfilled), distance [Q, k] fp32 (+inf = unfilled), ascending.
int is_knn(const float* query, const float* bank, const int64_t* exclude, int64_t n_query, int64_t n_bank, int dim, int k,
           int slices, unsigned long long* workspace, int64_t* index, float* distance, void* stream) {
    if (!query || !bank || !index || !distance) return IS_ERR_ARG;
    if (n_query < 1 || n_bank < 1 || dim < 1 || dim > KNN_DMAX || k < 1 || k > KNN_KMAX) return IS_ERR_ARG;
    if (n_bank > 0x7fffffffLL || n_query > 0x7fffffffLL - KNN_QT) return IS_ERR_UNSUPPORTED;
    if (slices < 1 || slices > min((int64_t)KNN_SMAX, (n_bank + KNN_RT - 1) / KNN_RT) || (slices > 1 && !workspace))
        return IS_ERR_ARG;
    const int64_t S = slices, rows = ((n_bank + S - 1) / S + KNN_RT - 1) / KNN_RT * KNN_RT;
    const size_t smem = knn_smem_bytes(dim);
    cudaError_t e = cudaFuncSetAttribute(knn_partial_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const dim3 grid((unsigned)((n_query + KNN_QT - 1) / KNN_QT), (unsigned)S);
    knn_partial_kernel<<<grid, IS_THREADS, smem, (cudaStream_t)stream>>>(
        query, bank, exclude, (int)n_query, (int)n_bank, dim, k, rows, slices, slices > 1 ? workspace : nullptr, index,
        distance);
    IS_LAUNCH_CHECK();
    if (slices > 1) {
        const int64_t warps = IS_THREADS / 32;
        knn_merge_kernel<<<(unsigned)((n_query + warps - 1) / warps), IS_THREADS, 0, (cudaStream_t)stream>>>(
            workspace, (int)n_query, slices, k, index, distance);
        IS_LAUNCH_CHECK();
    }
    return IS_OK;
}

}  // extern "C"
