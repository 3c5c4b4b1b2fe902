// In-silico saturation mutagenesis: one pass of single-residue mutants of a resident batch (immunostruct_b200/mutagenesis.py),
// and one pass of a variant library (any substitution list on any sample; is_variant_expand, below).
//
// A pass holds r copies of the base batch (B graphs, N nodes, sequence one-hots [B, L, V]).  Copy k carries one substitution
// (site p_k, residue-feature column c_k): in every graph b of the copy, the node row node_off[b] + node_index[b, p_k] gets
// one_hot_20(c_k) in its residue columns, and sequence row seq_index[b, p_k] of sample b gets one_hot_V(seq_columns[c_k]).
// Coordinates, edges and every other row are copied unchanged; a site absent from sample b (node_index[b, p_k] < 0) leaves
// that sample's copy unmodified.  The kernel only copies floats and writes 0.0 / 1.0, so it is bit-exact by construction.
//
// Work units are (copy, graph, part): part 0 copies the graph's x23 rows, part 1 the sample's sequence block.  Both are
// contiguous runs of floats, and the site row is a contiguous sub-run of each, so an element is patched by one unsigned
// compare -- no division per element.  The kernel is HBM-bound (one read of L2-resident base data, one write of r copies).
//
// Checks (device flag, set to 1, never cleared here): the base site rows must be exactly one-hot (x23 columns 0..19 and the
// V sequence columns), and the sequence's hot column must be seq_columns[native residue column]; an index outside its
// graph / sequence, a site or column outside the table, or a seq_columns entry outside [0, V) also raises the flag, and then
// nothing of that (copy, graph) is patched.  Plain stores of 1 from any thread: no atomics.
#include "common.cuh"

namespace is {

constexpr int MS_THREADS = 256;
constexpr int MS_CTAS_PER_SM = 6;          // 40 registers: six 256-thread CTAs per SM

struct MutSite {
    int64_t node_row;      // graph-local node row to patch, -1 = none
    int64_t seq_row;       // sequence row to patch
    int c;                 // residue-feature column of the substitution
    int seq_col;           // its sequence column
};

__device__ __forceinline__ MutSite mut_site(const int64_t* __restrict__ node_index, const int64_t* __restrict__ seq_index,
                                            const int64_t* __restrict__ seq_columns, const int* __restrict__ sites,
                                            int k, int b, int P, int64_t nb, int L, int V, bool& bad) {
    MutSite s{-1, -1, 0, 0};
    const int p = __ldg(sites + 2 * k), c = __ldg(sites + 2 * k + 1);
    if (p < 0 || p >= P || c < 0 || c >= 20) { bad = true; return s; }
    const int64_t ni = __ldg(node_index + (int64_t)b * P + p), si = __ldg(seq_index + (int64_t)b * P + p);
    if (ni < 0) return s;                                           // absent site: the copy stays unmodified
    const int64_t sc = __ldg(seq_columns + c);
    if (ni >= nb || si < 0 || si >= L || sc < 0 || sc >= V) { bad = true; return s; }
    s.node_row = ni; s.seq_row = si; s.c = c; s.seq_col = (int)sc;
    return s;
}

// warp-wide: the hot column of a sequence row of V floats if it is exactly one-hot, else -1
__device__ __forceinline__ int seq_row_hot(const float* __restrict__ srow, int V, int lane) {
    int s_ones = 0, s_nz = 0, hot = -1;
    for (int v0 = 0; v0 < V; v0 += 32) {
        const int v = v0 + lane;
        const float sv = v < V ? __ldg(srow + v) : 0.0f;
        const unsigned one = __ballot_sync(0xffffffffu, sv == 1.0f), nz = __ballot_sync(0xffffffffu, sv != 0.0f);
        if (one && hot < 0) hot = v0 + __ffs(one) - 1;
        s_ones += __popc(one);
        s_nz += __popc(nz);
    }
    return s_ones == 1 && s_nz == 1 ? hot : -1;
}

// warp-wide check of the base site rows: x23 residue columns and the sequence row exactly one-hot, and the sequence's hot
// column equal to seq_columns[native residue column]
__device__ __forceinline__ bool site_rows_bad(const float* __restrict__ xrow, const float* __restrict__ srow, int V,
                                              const int64_t* __restrict__ seq_columns, int lane) {
    const float xv = lane < 20 ? __ldg(xrow + lane) : 0.0f;
    const unsigned x_one = __ballot_sync(0xffffffffu, xv == 1.0f), x_nz = __ballot_sync(0xffffffffu, xv != 0.0f);
    const int hot = seq_row_hot(srow, V, lane);
    if (__popc(x_one) != 1 || x_nz != x_one || hot < 0) return true;
    return __ldg(seq_columns + (__ffs(x_one) - 1)) != (int64_t)hot;
}

// dst[e] = src[e] for e < n, except dst[row0 + j] = (j == hot) for j < width (row0 < 0: no patch)
__device__ __forceinline__ void copy_patch(const float* __restrict__ src, float* __restrict__ dst, int n, int row0, int width,
                                           int hot) {
    const unsigned w = row0 >= 0 ? (unsigned)width : 0u;
#pragma unroll 4
    for (int e = threadIdx.x; e < n; e += MS_THREADS) {
        float v = __ldg(src + e);
        const unsigned j = (unsigned)(e - row0);
        if (j < w) v = j == (unsigned)hot ? 1.0f : 0.0f;
        dst[e] = v;
    }
}

__global__ void __launch_bounds__(MS_THREADS, MS_CTAS_PER_SM) mutscan_expand_kernel(
        const float* __restrict__ x23, const int64_t* __restrict__ node_off, const int64_t* __restrict__ node_index,
        const float* __restrict__ seq, const int64_t* __restrict__ seq_index, const int64_t* __restrict__ seq_columns,
        const int* __restrict__ sites, int r, int B, int P, int64_t N, int L, int V,
        float* __restrict__ x23_out, float* __restrict__ seq_out, int* __restrict__ flag) {
    const int64_t units = 2 * (int64_t)r * B, LV = (int64_t)L * V;
    for (int64_t u = blockIdx.x; u < units; u += gridDim.x) {
        const int part = (int)(u & 1);
        const int kb = (int)(u >> 1), k = kb / B, b = kb - k * B;
        const int64_t n0 = __ldg(node_off + b), nb = __ldg(node_off + b + 1) - n0;
        bool bad = false;
        const MutSite s = mut_site(node_index, seq_index, seq_columns, sites, k, b, P, nb, L, V, bad);
        if (part == 0) {
            if (threadIdx.x < 32 && s.node_row >= 0 &&
                site_rows_bad(x23 + (n0 + s.node_row) * 23, seq + b * LV + s.seq_row * V, V, seq_columns, threadIdx.x))
                bad = true;
            if (bad && threadIdx.x == 0) *(volatile int*)flag = 1;
            copy_patch(x23 + n0 * 23, x23_out + ((int64_t)k * N + n0) * 23, (int)(nb * 23),
                       s.node_row >= 0 ? (int)s.node_row * 23 : -1, 20, s.c);
        } else {
            copy_patch(seq + b * LV, seq_out + ((int64_t)k * B + b) * LV, (int)LV, s.node_row >= 0 ? (int)s.seq_row * V : -1,
                       V, s.seq_col);
        }
    }
}

// ---- variant libraries: any substitution list on any sample of the batch ----------------------------------------------
//
// One pass holds r variants.  Variant v is a copy of base graph b = sample[v] (its x23 rows at node_out[v]..., its edges
// at edge_out[v]..., endpoints graph-local, and sequence sample v) with the substitutions offsets[v] .. offsets[v+1] - 1
// of the table: node row node_index[s] (graph-local, -1 = not in the graph) gets one_hot_20(residue[s]) in its residue
// columns and sequence row seq_index[s] gets one_hot_V(seq_columns[residue[s]]).
//
// Work units are (variant, part): part 0 the graph's x23 rows, part 1 its edges (src, dst, attribute), part 2 the
// sequence block.  Parts 0 and 2 go in chunks of 32 rows, one chunk per warp: every substitution whose row falls in the
// chunk is checked by the whole warp (ballots over the base rows) and, if it passes, the lane owning that row records the
// hot column; the warp then streams the chunk's rows coalesced and takes each element's patch from its row's lane by a
// shuffle.  No barrier, no atomics.  Both units that touch a substitution (x23 and sequence) run the same checks on the
// same base data, so a substitution is applied to both rows or to neither.
constexpr int VX_THREADS = 256;
constexpr int VX_WARPS = VX_THREADS / 32;
constexpr int VX_CTAS_PER_SM = 4;         // 64 registers, no spills (at six CTAs the 40-register cap spills 96 bytes)

// dst rows [0, n_rows) (n_rows <= 32) = src rows, W floats each; the row owned by lane i gets (j == hot_i) for columns
// j < width when hot_i >= 0.  Warp-wide: every lane takes part in each shuffle.
__device__ __forceinline__ void copy_chunk(const float* __restrict__ src, float* __restrict__ dst, int n_rows, int W,
                                           int width, int hot, int lane) {
    const int n = n_rows * W;
    int row = lane / W, col = lane - row * W;
#pragma unroll 4
    for (int e0 = 0; e0 < n; e0 += 32) {
        const int e = e0 + lane;
        const int h = __shfl_sync(0xffffffffu, hot, row < 32 ? row : 31);
        if (e < n) {
            float v = __ldg(src + e);
            if (h >= 0 && col < width) v = col == h ? 1.0f : 0.0f;
            dst[e] = v;
        }
        col += 32;
        while (col >= W) { col -= W; ++row; }
    }
}

__global__ void __launch_bounds__(VX_THREADS, VX_CTAS_PER_SM) variant_expand_kernel(
        const float* __restrict__ x23, const int64_t* __restrict__ node_off, const int64_t* __restrict__ edge_off,
        const int64_t* __restrict__ src_local, const int64_t* __restrict__ dst_local, const float* __restrict__ edge_attr,
        const float* __restrict__ seq, const int64_t* __restrict__ sample, const int64_t* __restrict__ offsets,
        const int64_t* __restrict__ node_index, const int64_t* __restrict__ seq_index, const int64_t* __restrict__ residue,
        const int64_t* __restrict__ seq_columns, const int64_t* __restrict__ node_out, const int64_t* __restrict__ edge_out,
        int r, int B, int64_t n_subs, int L, int V, int64_t n_out, int64_t e_out, float* __restrict__ x23_out,
        int64_t* __restrict__ src_out, int64_t* __restrict__ dst_out, float* __restrict__ edge_attr_out,
        float* __restrict__ seq_out, int* __restrict__ flag) {
    const int64_t units = 3 * (int64_t)r, LV = (int64_t)L * V;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t u = blockIdx.x; u < units; u += gridDim.x) {
        const int v = (int)(u / 3), part = (int)(u - 3 * (int64_t)v);
        const int64_t b = __ldg(sample + v);
        if (b < 0 || b >= B) { if (part == 0 && threadIdx.x == 0) *(volatile int*)flag = 1; continue; }
        const int64_t n0 = __ldg(node_off + b), nb = __ldg(node_off + b + 1) - n0;
        const int64_t e0 = __ldg(edge_off + b), eb = __ldg(edge_off + b + 1) - e0;
        const int64_t no = __ldg(node_out + v), eo = __ldg(edge_out + v);
        if (no < 0 || __ldg(node_out + v + 1) - no != nb || no + nb > n_out ||
            eo < 0 || __ldg(edge_out + v + 1) - eo != eb || eo + eb > e_out) {
            if (part == 0 && threadIdx.x == 0) *(volatile int*)flag = 1;
            continue;
        }
        if (part == 1) {
            for (int64_t i = threadIdx.x; i < eb; i += VX_THREADS) {
                src_out[eo + i] = __ldg(src_local + e0 + i);
                dst_out[eo + i] = __ldg(dst_local + e0 + i);
                edge_attr_out[eo + i] = __ldg(edge_attr + e0 + i);
            }
            continue;
        }
        int64_t s0 = __ldg(offsets + v), s1 = __ldg(offsets + v + 1);
        if (s0 < 0 || s1 < s0 || s1 > n_subs) {
            if (part == 2 && threadIdx.x == 0) *(volatile int*)flag = 1;
            s0 = s1 = 0;                                                 // copied, nothing substituted
        }
        const float* sbase = seq + b * LV;
        if (part == 2 && warp == 0) {                // index ranges, including rows that fall in no chunk of either part
            bool bad = false;
            for (int64_t s = s0 + lane; s < s1; s += 32) {
                const int64_t ni = __ldg(node_index + s), si = __ldg(seq_index + s), c = __ldg(residue + s);
                bad |= ni < -1 || ni >= nb || si < 0 || si >= L || c < 0 || c >= 20;
            }
            if (__any_sync(0xffffffffu, bad) && lane == 0) *(volatile int*)flag = 1;
        }
        const int64_t n_rows = part == 0 ? nb : L;
        const int W = part == 0 ? 23 : V;
        const float* src = part == 0 ? x23 + n0 * 23 : sbase;
        float* dst = part == 0 ? x23_out + no * 23 : seq_out + (int64_t)v * LV;
        for (int64_t c0 = (int64_t)warp * 32; c0 < n_rows; c0 += VX_WARPS * 32) {
            int hot = -1;
            for (int64_t s = s0; s < s1; ++s) {                               // warp-uniform
                const int64_t ni = __ldg(node_index + s), si = __ldg(seq_index + s), c = __ldg(residue + s);
                const int64_t row = part == 0 ? ni : si;
                if (row < c0 || row >= c0 + 32) continue;
                if (ni < -1 || ni >= nb || si < 0 || si >= L || c < 0 || c >= 20) continue;   // raised above
                const int64_t sc = __ldg(seq_columns + c);
                bool bad = sc < 0 || sc >= V;
                if (!bad) bad = ni >= 0 ? site_rows_bad(x23 + (n0 + ni) * 23, sbase + si * V, V, seq_columns, lane)
                                        : seq_row_hot(sbase + si * V, V, lane) < 0;
                if (bad) {
                    if (lane == 0) *(volatile int*)flag = 1;
                    continue;
                }
                if (lane == (int)(row - c0)) hot = part == 0 ? (int)c : (int)sc;
            }
            const int rows = (int)(n_rows - c0 < 32 ? n_rows - c0 : 32);
            copy_chunk(src + c0 * W, dst + c0 * W, rows, W, part == 0 ? 20 : V, hot, lane);
        }
    }
}

}  // namespace is

using namespace is;

extern "C" {

// grid: min(2 r B, 6 x SMs) CTAs of 256 threads, each looping over (copy, graph, part) units
int is_mutscan_expand(const float* x23, const int64_t* node_off, const int64_t* node_index, const float* seq,
                      const int64_t* seq_index, const int64_t* seq_columns, const int* sites, int r, int n_graphs, int n_sites,
                      int64_t n_nodes, int seq_len, int vocab, float* x23_out, float* seq_out, int* flag, void* stream) {
    if (r < 1 || n_graphs < 1 || n_sites < 1 || n_nodes < 0 || seq_len < 1 || vocab < 1) return IS_ERR_ARG;
    if (!x23 || !node_off || !node_index || !seq || !seq_index || !seq_columns || !sites || !x23_out || !seq_out || !flag)
        return IS_ERR_ARG;
    // element offsets inside one graph's rows / one sample's sequence are 32-bit (graphs hold at most 256 nodes)
    if ((int64_t)r * n_graphs > 0x3fffffff || (int64_t)seq_len * vocab > 0x7fffffff) return IS_ERR_UNSUPPORTED;
    const int64_t units = 2 * (int64_t)r * n_graphs, cap = (int64_t)MS_CTAS_PER_SM * current_num_sms();
    mutscan_expand_kernel<<<(unsigned)(units < cap ? units : cap), MS_THREADS, 0, (cudaStream_t)stream>>>(
        x23, node_off, node_index, seq, seq_index, seq_columns, sites, r, n_graphs, n_sites, n_nodes, seq_len, vocab, x23_out,
        seq_out, flag);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

// grid: min(3 r, 4 x SMs) CTAs of 256 threads, each looping over (variant, part) units
int is_variant_expand(const float* x23, const int64_t* node_off, const int64_t* edge_off, const int64_t* src_local,
                      const int64_t* dst_local, const float* edge_attr, const float* seq, const int64_t* sample,
                      const int64_t* offsets, const int64_t* node_index, const int64_t* seq_index, const int64_t* residue,
                      const int64_t* seq_columns, const int64_t* node_out, const int64_t* edge_out, int r, int n_graphs,
                      int64_t n_subs, int seq_len, int vocab, int64_t n_nodes_out, int64_t n_edges_out, float* x23_out,
                      int64_t* src_out, int64_t* dst_out, float* edge_attr_out, float* seq_out, int* flag, void* stream) {
    if (r < 1 || n_graphs < 1 || n_subs < 0 || seq_len < 1 || vocab < 1 || n_nodes_out < 0 || n_edges_out < 0)
        return IS_ERR_ARG;
    if (!x23 || !node_off || !edge_off || !seq || !sample || !offsets || !seq_columns || !node_out || !edge_out || !seq_out ||
        !flag || (n_subs > 0 && (!node_index || !seq_index || !residue)) ||
        (n_nodes_out > 0 && !x23_out) || (n_edges_out > 0 && (!src_local || !dst_local || !edge_attr || !src_out ||
                                                              !dst_out || !edge_attr_out)))
        return IS_ERR_ARG;
    if ((int64_t)r > 0x2aaaaaaa) return IS_ERR_UNSUPPORTED;
    const int64_t units = 3 * (int64_t)r, cap = (int64_t)VX_CTAS_PER_SM * current_num_sms();
    variant_expand_kernel<<<(unsigned)(units < cap ? units : cap), VX_THREADS, 0, (cudaStream_t)stream>>>(
        x23, node_off, edge_off, src_local, dst_local, edge_attr, seq, sample, offsets, node_index, seq_index, residue,
        seq_columns, node_out, edge_out, r, n_graphs, n_subs, seq_len, vocab, n_nodes_out, n_edges_out, x23_out, src_out,
        dst_out, edge_attr_out, seq_out, flag);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

}  // extern "C"
