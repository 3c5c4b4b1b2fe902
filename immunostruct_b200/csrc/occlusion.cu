// Structural occlusion: one pass of single-removal variants of a resident batch (immunostruct_b200/occlusion.py).
//
// Variant v of a pass is a copy of base graph b = sample[v] with one thing removed:
//   * node_b[v] == -1, residue occlusion of graph-local row a = node_a[v]: the 23 floats of row a become 0.0 (features and
//     coordinates, as pad_graph writes an absent residue) and every edge with src == a or dst == a is dropped (multi-edges
//     and a self-loop included).  The row stays, so node counts are unchanged.
//   * node_b[v] >= 0, contact occlusion of the unordered pair {a, b'} (a != b'): every edge a -> b' and b' -> a is dropped.
//     Rows are unchanged; a self-loop is not a contact and is never dropped.
// The kept edges keep their base order: the variant is exactly the graph a boolean edge mask would build.
//
// Work units are (variant, part), grid-strided over the CTAs.  Part 0 copies the graph's x23 rows to x23_out from row
// node_out[v] (row a zeroed in residue mode); part 1 writes the kept edges (graph-local endpoints and attribute) to
// src_out / dst_out / edge_attr_out from edge_out[v].  The compaction is order-preserving without atomics: warp w takes
// the contiguous slice w of the graph's edges (one CTA round is 256 edges, one per thread; a larger graph gives every
// warp several 32-edge steps), counts its kept edges with ballots, one exclusive scan over the eight warp counts in shared
// memory gives each warp its output base, and the warps then read their slices again (from L2) and write each kept edge
// at base + the popcount of the kept lanes below it.
//
// The kept count is known before anything is written.  Both parts compute it, so a variant is written whole or not at all:
// the flag (int32, set to 1, never cleared here) is raised and the variant is skipped when its count disagrees with
// edge_out[v+1] - edge_out[v], when sample is outside [0, B), node_a outside [0, n_b), node_b outside [-1, n_b) or equal
// to node_a, when node_out[v+1] - node_out[v] != n_b, or when an offset runs past n_out / e_out.  Only copies and 0.0 are
// written, so the output is bit-exact by construction.
#include "common.cuh"

namespace is {

constexpr int OC_THREADS = 256;
constexpr int OC_WARPS = OC_THREADS / 32;
constexpr int OC_CTAS_PER_SM = 4;

__device__ __forceinline__ bool oc_keep(int64_t s, int64_t d, int64_t a, int64_t b2) {
    return b2 < 0 ? (s != a && d != a) : !((s == a && d == b2) || (s == b2 && d == a));
}

// kept edges of warp `warp`'s slice [lo, hi) of the graph's edges (graph-local arrays from e0); warp-wide
__device__ __forceinline__ int64_t oc_warp_kept(const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                                                int64_t lo, int64_t hi, int64_t a, int64_t b2, int lane) {
    int64_t n = 0;
    for (int64_t i0 = lo; i0 < hi; i0 += 32) {
        const int64_t i = i0 + lane;
        const bool keep = i < hi && oc_keep(__ldg(src + i), __ldg(dst + i), a, b2);
        n += __popc(__ballot_sync(0xffffffffu, keep));
    }
    return n;
}

__global__ void __launch_bounds__(OC_THREADS, OC_CTAS_PER_SM) occlusion_expand_kernel(
        const float* __restrict__ x23, const int64_t* __restrict__ node_off, const int64_t* __restrict__ edge_off,
        const int64_t* __restrict__ src_local, const int64_t* __restrict__ dst_local, const float* __restrict__ edge_attr,
        const int64_t* __restrict__ sample, const int64_t* __restrict__ node_a, const int64_t* __restrict__ node_b,
        const int64_t* __restrict__ node_out, const int64_t* __restrict__ edge_out, int r, int B, int64_t n_out,
        int64_t e_out, float* __restrict__ x23_out, int64_t* __restrict__ src_out, int64_t* __restrict__ dst_out,
        float* __restrict__ edge_attr_out, int* __restrict__ flag) {
    __shared__ int64_t warp_base[OC_WARPS + 1];
    const int64_t units = 2 * (int64_t)r;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t u = blockIdx.x; u < units; u += gridDim.x) {
        const int v = (int)(u >> 1), part = (int)(u & 1);
        const int64_t b = __ldg(sample + v), a = __ldg(node_a + v), b2 = __ldg(node_b + v);
        if (b < 0 || b >= B) { if (part == 0 && threadIdx.x == 0) *(volatile int*)flag = 1; continue; }
        const int64_t n0 = __ldg(node_off + b), nb = __ldg(node_off + b + 1) - n0;
        const int64_t e0 = __ldg(edge_off + b), eb = __ldg(edge_off + b + 1) - e0;
        const int64_t no = __ldg(node_out + v), eo = __ldg(edge_out + v), ek = __ldg(edge_out + v + 1) - eo;
        if (a < 0 || a >= nb || b2 < -1 || b2 >= nb || b2 == a || no < 0 || __ldg(node_out + v + 1) - no != nb ||
            no + nb > n_out || eo < 0 || ek < 0 || eo + ek > e_out) {
            if (part == 0 && threadIdx.x == 0) *(volatile int*)flag = 1;
            continue;
        }
        const int64_t* src = src_local + e0;
        const int64_t* dst = dst_local + e0;
        const int64_t per = (eb + OC_WARPS - 1) / OC_WARPS;              // warp slice: [warp * per, (warp + 1) * per)
        const int64_t lo = min((int64_t)warp * per, eb), hi = min(lo + per, eb);
        const int64_t kept = oc_warp_kept(src, dst, lo, hi, a, b2, lane);
        __syncthreads();                                                 // warp_base of the previous unit is consumed
        if (lane == 0) warp_base[warp + 1] = kept;
        __syncthreads();
        if (threadIdx.x == 0) {
            warp_base[0] = 0;
            for (int w = 1; w <= OC_WARPS; ++w) warp_base[w] += warp_base[w - 1];
        }
        __syncthreads();
        if (warp_base[OC_WARPS] != ek) {                                 // CTA-uniform
            if (part == 1 && threadIdx.x == 0) *(volatile int*)flag = 1;
            continue;
        }
        if (part == 0) {
            const int64_t n = nb * 23, za = b2 < 0 ? a * 23 : n;        // residue mode: floats [23 a, 23 a + 23) are 0
            const float* xs = x23 + n0 * 23;
            float* xd = x23_out + no * 23;
            for (int64_t i = threadIdx.x; i < n; i += OC_THREADS)
                xd[i] = (uint64_t)(i - za) < 23u ? 0.0f : __ldg(xs + i);
            continue;
        }
        int64_t out = eo + warp_base[warp];
        for (int64_t i0 = lo; i0 < hi; i0 += 32) {
            const int64_t i = i0 + lane;
            int64_t s = 0, d = 0;
            bool keep = false;
            if (i < hi) {
                s = __ldg(src + i);
                d = __ldg(dst + i);
                keep = oc_keep(s, d, a, b2);
            }
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            if (keep) {
                const int64_t o = out + __popc(m & ((1u << lane) - 1u));
                src_out[o] = s;
                dst_out[o] = d;
                edge_attr_out[o] = __ldg(edge_attr + e0 + i);
            }
            out += __popc(m);
        }
    }
}

}  // namespace is

using namespace is;

extern "C" {

// grid: min(2 r, 4 x SMs) CTAs of 256 threads, each looping over (variant, part) units
int is_occlusion_expand(const float* x23, const int64_t* node_off, const int64_t* edge_off, const int64_t* src_local,
                        const int64_t* dst_local, const float* edge_attr, const int64_t* sample, const int64_t* node_a,
                        const int64_t* node_b, const int64_t* node_out, const int64_t* edge_out, int r, int n_graphs,
                        int64_t n_nodes_out, int64_t n_edges_out, float* x23_out, int64_t* src_out, int64_t* dst_out,
                        float* edge_attr_out, int* flag, void* stream) {
    if (r < 1 || n_graphs < 1 || n_nodes_out < 0 || n_edges_out < 0) return IS_ERR_ARG;
    if (!x23 || !node_off || !edge_off || !sample || !node_a || !node_b || !node_out || !edge_out || !flag ||
        (n_nodes_out > 0 && !x23_out) ||
        (n_edges_out > 0 && (!src_local || !dst_local || !edge_attr || !src_out || !dst_out || !edge_attr_out)))
        return IS_ERR_ARG;
    if ((int64_t)r > 0x3fffffff) return IS_ERR_UNSUPPORTED;
    const int64_t units = 2 * (int64_t)r, cap = (int64_t)OC_CTAS_PER_SM * current_num_sms();
    occlusion_expand_kernel<<<(unsigned)(units < cap ? units : cap), OC_THREADS, 0, (cudaStream_t)stream>>>(
        x23, node_off, edge_off, src_local, dst_local, edge_attr, sample, node_a, node_b, node_out, edge_out, r, n_graphs,
        n_nodes_out, n_edges_out, x23_out, src_out, dst_out, edge_attr_out, flag);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

}  // extern "C"
