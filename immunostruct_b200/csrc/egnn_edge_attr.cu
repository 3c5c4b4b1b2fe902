// Gradient of an EGNN layer with respect to its scalar edge features (edge_attr, edge_feat_size = 1).
//
// The first edge-MLP layer reads a_e through one weight column: z1[p] = P[src] + Q[dst] + r wr + a_e wa (wa = W1[:, 2F+1]),
// so  g_a[e] = sum_k gz1[p, k] wa[k]  with e = csr_eid[p].  gz1 [E, 64] (CSR order) is what the edge backward already
// writes for the node-side backward; this kernel streams it once more (256 bytes per edge, HBM-bound) and writes one
// float per edge.  csr_eid is a permutation, so every edge is written by exactly one thread: no atomics, and the sum
// over k runs in a fixed order (four products per lane, then a fixed butterfly over the 16 lanes of a row) --
// bit-reproducible.  With `accumulate` the layer's contribution is added to g_a (the stack sums its layers in a fixed
// order).  Kept a standalone kernel rather than an epilogue of the warp-specialised edge backward (DESIGN.md 4.2).
#include "common.cuh"

namespace is {

constexpr int EA_THREADS = 256, EA_UNROLL = 4;          // 16 lanes per gz1 row, 4 rows per half-warp in flight

__global__ void __launch_bounds__(EA_THREADS)
edge_attr_grad_kernel(const float* __restrict__ gz1, const int* __restrict__ csr_eid, const float* __restrict__ W1, int ldw,
                      int col, float* __restrict__ g_attr, int64_t E, int accumulate) {
    const int lane = threadIdx.x & 31, half = lane >> 4, sub = lane & 15;
    float w[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) w[j] = __ldg(W1 + (size_t)(4 * sub + j) * ldw + col);
    const int64_t warp_g = ((int64_t)blockIdx.x * EA_THREADS + threadIdx.x) >> 5;
    const int64_t stride = 2 * (((int64_t)gridDim.x * EA_THREADS) >> 5);    // rows per sweep of the grid
    // the loop bound is warp-uniform (the shuffles below need the whole warp); the row bound is per half-warp
    for (int64_t base = 2 * warp_g; base < E; base += EA_UNROLL * stride) {
        float4 v[EA_UNROLL];
        int eid[EA_UNROLL];
#pragma unroll
        for (int u = 0; u < EA_UNROLL; ++u) {
            const int64_t p = base + half + u * stride;
            v[u] = p < E ? __ldg(reinterpret_cast<const float4*>(gz1 + p * 64) + sub) : make_float4(0.f, 0.f, 0.f, 0.f);
            eid[u] = (sub == 0 && p < E) ? __ldg(csr_eid + p) : 0;
        }
#pragma unroll
        for (int u = 0; u < EA_UNROLL; ++u) {
            float s = v[u].x * w[0];
            s = fmaf(v[u].y, w[1], s);
            s = fmaf(v[u].z, w[2], s);
            s = fmaf(v[u].w, w[3], s);
            s += __shfl_xor_sync(0xffffffffu, s, 8);
            s += __shfl_xor_sync(0xffffffffu, s, 4);
            s += __shfl_xor_sync(0xffffffffu, s, 2);
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            const int64_t p = base + half + u * stride;
            if (sub == 0 && p < E) g_attr[eid[u]] = accumulate ? g_attr[eid[u]] + s : s;
        }
    }
}

}  // namespace is

using namespace is;

extern "C" {

// g_attr [E] (original edge order) (+)= gz1 [E, 64] (CSR order) . W1[:, 2F+1]; W1 = edge_mlp.0.weight [64, 2F+2]
int is_egnn_edge_attr_grad(const float* gz1, const int* csr_eid, const float* W1, int F, float* g_attr, int64_t n_edges,
                           int accumulate, void* stream) {
    if (!(F == 20 || F == 64) || n_edges < 0 || n_edges > 0x7fffffff) return IS_ERR_ARG;
    if (n_edges == 0) return IS_OK;
    if (!gz1 || !csr_eid || !W1 || !g_attr || (reinterpret_cast<uintptr_t>(gz1) & 15) != 0) return IS_ERR_ARG;
    const int64_t rows_per_cta = (EA_THREADS / 16) * EA_UNROLL;
    const int64_t need = (n_edges + rows_per_cta - 1) / rows_per_cta, cap = 4 * (int64_t)current_num_sms();     // 64 registers: four CTAs per SM
    const int grid = (int)(need < cap ? need : cap);
    edge_attr_grad_kernel<<<grid, EA_THREADS, 0, (cudaStream_t)stream>>>(gz1, csr_eid, W1, 2 * F + 2, 2 * F + 1, g_attr, n_edges,
                                                                         accumulate);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

}  // extern "C"
