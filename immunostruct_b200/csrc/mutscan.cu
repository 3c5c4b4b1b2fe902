// In-silico saturation mutagenesis: one pass of single-residue mutants of a resident batch (immunostruct_b200/mutagenesis.py).
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

// warp-wide check of the base site rows: x23 residue columns and the sequence row exactly one-hot, and the sequence's hot
// column equal to seq_columns[native residue column]
__device__ __forceinline__ bool site_rows_bad(const float* __restrict__ xrow, const float* __restrict__ srow, int V,
                                              const int64_t* __restrict__ seq_columns, int lane) {
    const float xv = lane < 20 ? __ldg(xrow + lane) : 0.0f;
    const unsigned x_one = __ballot_sync(0xffffffffu, xv == 1.0f), x_nz = __ballot_sync(0xffffffffu, xv != 0.0f);
    int s_ones = 0, s_nz = 0, hot = -1;
    for (int v0 = 0; v0 < V; v0 += 32) {
        const int v = v0 + lane;
        const float sv = v < V ? __ldg(srow + v) : 0.0f;
        const unsigned one = __ballot_sync(0xffffffffu, sv == 1.0f), nz = __ballot_sync(0xffffffffu, sv != 0.0f);
        if (one && hot < 0) hot = v0 + __ffs(one) - 1;
        s_ones += __popc(one);
        s_nz += __popc(nz);
    }
    if (__popc(x_one) != 1 || x_nz != x_one || s_ones != 1 || s_nz != 1) return true;
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

}  // extern "C"
