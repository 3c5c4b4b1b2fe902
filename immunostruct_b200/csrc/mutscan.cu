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

// ---- beam search over residue substitutions (immunostruct_b200/design.py) ----------------------------------------------
//
// Sample b's beam holds W states of its P sites (int64 [B, W, P] residue columns, -1 at absent sites), their keys
// sum_p digit(state[p]) 20^p (digit 0 at absent sites; they break ties), their Hamming distances to the native state and
// a valid flag.
// A round enumerates the slots (w, p, c) = "state w with site p set to residue c" of its first Wt states,
// k = (w P + p) 20 + c; every slot is one copy of the whole batch.  design_slot_valid is the slot rule both kernels share.
constexpr int DX_THREADS = 256;
constexpr int DX_WARPS = DX_THREADS / 32;
constexpr int DX_CTAS_PER_SM = 4;
constexpr int DS_THREADS = 256;
constexpr int DS_WARPS = DS_THREADS / 32;

__device__ __forceinline__ int64_t design_digit(int64_t s) { return s < 0 ? 0 : s; }

__device__ __forceinline__ int64_t pow20(int p) {
    int64_t v = 1;
    for (int i = 0; i < p; ++i) v *= 20;
    return v;
}

// warp-wide (Wt <= 32; every lane gets the same answer): slot (w, p, c) of one sample is valid -- its parent w is valid,
// site p is present, c is allowed there and differs from the parent's residue, the new state is within max_mut of the
// native state, and it is canonical: no valid state l < Wt equals it, and none with l < w is one substitution away from
// it (slot (l, p', c') yields the same state and comes first).  Lane l compares state l with the new state site by site:
// two beam states two substitutions apart reach a common state at two different sites, which a comparison at site p
// alone would miss.  Pointers are the sample's rows.
__device__ __forceinline__ bool design_slot_valid(const int64_t* __restrict__ st, const int64_t* __restrict__ n_mut,
                                                  const unsigned char* __restrict__ valid,
                                                  const int64_t* __restrict__ native, const unsigned char* __restrict__ allowed,
                                                  const int64_t* __restrict__ ni, int w, int p, int c, int P, int Wt,
                                                  int max_mut, int lane) {
    const int64_t* sw = st + (int64_t)w * P;
    const int64_t sp = __ldg(sw + p);
    if (!__ldg(valid + w) || __ldg(ni + p) < 0 || !__ldg(allowed + p * 20 + c) || sp == c) return false;
    const int64_t nat = __ldg(native + p);
    if (__ldg(n_mut + w) - (sp != nat) + (c != nat) > max_mut) return false;
    bool dup = false;
    if (lane < Wt && __ldg(valid + lane)) {
        const int64_t* sl = st + (int64_t)lane * P;
        int h = 0;
        for (int q = 0; q < P; ++q) h += __ldg(sl + q) != (q == p ? (int64_t)c : __ldg(sw + q));
        dup = h == 0 || (h == 1 && lane < w);
    }
    return !__any_sync(0xffffffffu, dup);
}

// One pass: copy k < r is slot slot0 + k.  Units (copy, graph, part) as in mutscan_expand_kernel; rows go in 32-row
// chunks, one per warp, as in variant_expand_kernel.  Every present site of graph b gets the parent state's residue, and
// site p the slot's residue c when the slot is valid (an invalid slot is written as its parent state).  Writing a residue
// a row already holds is a bit-exact no-op, so only the mutated rows change.
__global__ void __launch_bounds__(DX_THREADS, DX_CTAS_PER_SM) design_expand_kernel(
        const float* __restrict__ x23, const int64_t* __restrict__ node_off, const int64_t* __restrict__ node_index,
        const float* __restrict__ seq, const int64_t* __restrict__ seq_index, const int64_t* __restrict__ seq_columns,
        const int64_t* __restrict__ states, const int64_t* __restrict__ n_mut, const unsigned char* __restrict__ valid,
        const int64_t* __restrict__ native, const unsigned char* __restrict__ allowed, int slot0, int r, int B, int P, int W, int Wt, int max_mut,
        int64_t N, int L, int V, float* __restrict__ x23_out, float* __restrict__ seq_out, int* __restrict__ flag) {
    const int64_t units = 2 * (int64_t)r * B, LV = (int64_t)L * V;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t u = blockIdx.x; u < units; u += gridDim.x) {
        const int part = (int)(u & 1);
        const int kb = (int)(u >> 1), k = kb / B, b = kb - k * B;
        const int s = slot0 + k, w = s / (P * 20), p = (s - w * P * 20) / 20, c = s - (w * P + p) * 20;
        const int64_t n0 = __ldg(node_off + b), nb = __ldg(node_off + b + 1) - n0;
        const int64_t* st = states + (int64_t)b * W * P;
        const int64_t* ni = node_index + (int64_t)b * P;
        const int64_t* si = seq_index + (int64_t)b * P;
        const bool ok = design_slot_valid(st, n_mut + (int64_t)b * W, valid + (int64_t)b * W, native + (int64_t)b * P,
                                          allowed + (int64_t)b * P * 20, ni, w, p, c, P, Wt, max_mut, lane);
        const float* sbase = seq + b * LV;
        if (part == 0 && warp == 0) {
            const int64_t np = __ldg(ni + p), sq = __ldg(si + p);
            if (np >= 0 && np < nb && sq >= 0 && sq < L &&
                site_rows_bad(x23 + (n0 + np) * 23, sbase + sq * V, V, seq_columns, lane) && lane == 0)
                *(volatile int*)flag = 1;
        }
        const int64_t n_rows = part == 0 ? nb : L;
        const int Wd = part == 0 ? 23 : V;
        const float* src = part == 0 ? x23 + n0 * 23 : sbase;
        float* dst = part == 0 ? x23_out + ((int64_t)k * N + n0) * 23 : seq_out + ((int64_t)k * B + b) * LV;
        for (int64_t c0 = (int64_t)warp * 32; c0 < n_rows; c0 += DX_WARPS * 32) {
            int hot = -1;
            for (int q = 0; q < P; ++q) {                                     // warp-uniform
                const int64_t nq = __ldg(ni + q), sq = __ldg(si + q);
                if (nq < 0) continue;                                         // absent site
                const int64_t d = q == p && ok ? c : __ldg(st + (int64_t)w * P + q);
                const int64_t sc = d >= 0 && d < 20 ? __ldg(seq_columns + d) : -1;
                if (nq >= nb || sq < 0 || sq >= L || sc < 0 || sc >= V) {
                    if (lane == 0) *(volatile int*)flag = 1;
                    continue;
                }
                const int64_t row = part == 0 ? nq : sq;
                if (lane == (int)(row - c0)) hot = part == 0 ? (int)d : (int)sc;
            }
            const int rows = (int)(n_rows - c0 < 32 ? n_rows - c0 : 32);
            copy_chunk(src + c0 * Wd, dst + c0 * Wd, rows, Wd, part == 0 ? 20 : V, hot, lane);
        }
    }
}

// o1 / k1 ranks strictly before o2 / k2: the better objective, then the smaller key (keys in one pool are distinct)
__device__ __forceinline__ bool design_before(float o1, int64_t k1, float o2, int64_t k2, bool maximize) {
    return (maximize ? o1 > o2 : o1 < o2) || (o1 == o2 && k1 < k2);
}

// One CTA per sample.  The pool is the Wt carried states (with their scores) and the round's Wt P 20 slots; an entry is
// eligible when it is valid (a valid beam state, or a valid slot) and its objective fmaf(kappa, std, mean) is not NaN.
// The next beam is the first W eligible entries in design_before order, found by W block-wide arg-best passes over the
// pool in shared memory (each pass takes the best entry ranked after the previous pick): deterministic, no atomics.
__global__ void __launch_bounds__(DS_THREADS, 1) design_select_kernel(
        const int64_t* __restrict__ states, const int64_t* __restrict__ keys, const int64_t* __restrict__ n_mut,
        const unsigned char* __restrict__ valid, const float* __restrict__ logits, const float* __restrict__ mean,
        const float* __restrict__ std_, const float* __restrict__ r_logits, const float* __restrict__ r_mean,
        const float* __restrict__ r_std, const int64_t* __restrict__ native, const unsigned char* __restrict__ allowed,
        const int64_t* __restrict__ node_index, int B, int P, int W, int Wt, int K, int max_mut, float kappa, int maximize,
        int64_t* __restrict__ states_out, int64_t* __restrict__ keys_out, int64_t* __restrict__ n_mut_out,
        unsigned char* __restrict__ valid_out, float* __restrict__ logits_out, float* __restrict__ mean_out,
        float* __restrict__ std_out, float* __restrict__ obj_out, float* __restrict__ best, int64_t best_stride) {
    extern __shared__ int64_t ds_smem[];
    const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n_slots = Wt * P * 20, n_pool = Wt + n_slots;
    int64_t* pkey = ds_smem;
    float* pobj = (float*)(ds_smem + n_pool);
    __shared__ float red_o[DS_WARPS];
    __shared__ int64_t red_k[DS_WARPS];
    __shared__ int red_i[DS_WARPS];
    __shared__ int sel[32];
    const int64_t* st = states + (int64_t)b * W * P;
    const int64_t* ky = keys + (int64_t)b * W;
    const int64_t* nm = n_mut + (int64_t)b * W;
    const unsigned char* vd = valid + (int64_t)b * W;
    const int64_t* nat = native + (int64_t)b * P;
    const float nan = __int_as_float(0x7fffffff);
    for (int e = threadIdx.x; e < Wt; e += DS_THREADS) {
        pkey[e] = __ldg(ky + e);
        pobj[e] = __ldg(vd + e) ? fmaf(kappa, __ldg(std_ + (int64_t)b * W + e), __ldg(mean + (int64_t)b * W + e)) : nan;
    }
    for (int s = warp; s < n_slots; s += DS_WARPS) {                        // warp-uniform: the slot rule is warp-wide
        const int w = s / (P * 20), p = (s - w * P * 20) / 20, c = s - (w * P + p) * 20;
        const bool ok = design_slot_valid(st, nm, vd, nat, allowed + (int64_t)b * P * 20, node_index + (int64_t)b * P,
                                          w, p, c, P, Wt, max_mut, lane);
        if (lane == 0) {
            pkey[Wt + s] = __ldg(ky + w) + (c - design_digit(__ldg(st + (int64_t)w * P + p))) * pow20(p);
            pobj[Wt + s] = ok ? fmaf(kappa, __ldg(r_std + (int64_t)s * B + b), __ldg(r_mean + (int64_t)s * B + b)) : nan;
        }
    }
    __syncthreads();
    const bool mx = maximize != 0;
    float prev_o = 0.0f;
    int64_t prev_k = 0;
    int n_sel = 0;
    for (int j = 0; j < W; ++j) {
        float bo = 0.0f;
        int64_t bk = 0;
        int bi = -1;
        for (int e = threadIdx.x; e < n_pool; e += DS_THREADS) {
            const float o = pobj[e];
            if (o != o) continue;
            const int64_t k = pkey[e];
            if (j > 0 && !design_before(prev_o, prev_k, o, k, mx)) continue;
            if (bi < 0 || design_before(o, k, bo, bk, mx)) { bo = o; bk = k; bi = e; }
        }
        for (int off = 16; off > 0; off >>= 1) {
            const float oo = __shfl_down_sync(0xffffffffu, bo, off);
            const int64_t ok_ = __shfl_down_sync(0xffffffffu, bk, off);
            const int oi = __shfl_down_sync(0xffffffffu, bi, off);
            if (oi >= 0 && (bi < 0 || design_before(oo, ok_, bo, bk, mx))) { bo = oo; bk = ok_; bi = oi; }
        }
        if (lane == 0) { red_o[warp] = bo; red_k[warp] = bk; red_i[warp] = bi; }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int i = 1; i < DS_WARPS; ++i)
                if (red_i[i] >= 0 && (bi < 0 || design_before(red_o[i], red_k[i], bo, bk, mx))) {
                    bo = red_o[i]; bk = red_k[i]; bi = red_i[i];
                }
            sel[j] = bi;
            red_o[0] = bo; red_k[0] = bk; red_i[0] = bi;
        }
        __syncthreads();
        bi = red_i[0];
        prev_o = red_o[0];
        prev_k = red_k[0];
        __syncthreads();                                                      // red_* is rewritten by the next pass
        if (bi < 0) break;
        ++n_sel;
    }
    // the next beam: picks in order, then empty entries holding the native state (so a slot of theirs stays finite)
    const int64_t bo_ = (int64_t)b * W;
    for (int i = threadIdx.x; i < W * P; i += DS_THREADS) {
        const int j = i / P, q = i - j * P;
        int64_t v = __ldg(nat + q);
        if (j < n_sel) {
            const int e = sel[j];
            const int w = e < Wt ? e : (e - Wt) / (P * 20);
            v = __ldg(st + (int64_t)w * P + q);
            if (e >= Wt && q == ((e - Wt) - w * P * 20) / 20) v = (e - Wt) % 20;
        }
        states_out[bo_ * P + i] = v;
    }
    for (int i = threadIdx.x; i < W * K; i += DS_THREADS) {
        const int j = i / K, k = i - j * K;
        float v = nan;
        if (j < n_sel) {
            const int e = sel[j];
            v = e < Wt ? __ldg(logits + (bo_ + e) * K + k) : __ldg(r_logits + ((int64_t)(e - Wt) * B + b) * K + k);
        }
        logits_out[bo_ * K + i] = v;
    }
    for (int j = threadIdx.x; j < W; j += DS_THREADS) {
        int64_t key = 0, nmut = 0;
        float m = nan, sd = nan, o = nan;
        if (j < n_sel) {
            const int e = sel[j];
            key = pkey[e];
            o = pobj[e];
            if (e < Wt) {
                nmut = __ldg(nm + e);
                m = __ldg(mean + bo_ + e);
                sd = __ldg(std_ + bo_ + e);
            } else {
                const int s = e - Wt, w = s / (P * 20), p = (s - w * P * 20) / 20, c = s % 20;
                const int64_t sp = __ldg(st + (int64_t)w * P + p), na = __ldg(nat + p);
                nmut = __ldg(nm + w) - (sp != na) + (c != na);
                m = __ldg(r_mean + (int64_t)s * B + b);
                sd = __ldg(r_std + (int64_t)s * B + b);
            }
        } else {
            for (int q = 0; q < P; ++q) key += design_digit(__ldg(nat + q)) * pow20(q);
        }
        keys_out[bo_ + j] = key;
        n_mut_out[bo_ + j] = nmut;
        valid_out[bo_ + j] = j < n_sel ? 1 : 0;
        mean_out[bo_ + j] = m;
        std_out[bo_ + j] = sd;
        obj_out[bo_ + j] = o;
    }
    if (threadIdx.x == 0) best[(int64_t)b * best_stride] = n_sel > 0 ? pobj[sel[0]] : nan;
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

// grid: min(2 r B, 4 x SMs) CTAs of 256 threads, each looping over (copy, graph, part) units
int is_design_expand(const float* x23, const int64_t* node_off, const int64_t* node_index, const float* seq,
                     const int64_t* seq_index, const int64_t* seq_columns, const int64_t* states, const int64_t* n_mut,
                     const unsigned char* valid, const int64_t* native, const unsigned char* allowed, int slot0, int r, int n_graphs, int n_sites, int beam, int n_states, int max_mutations, int64_t n_nodes,
                     int seq_len, int vocab, float* x23_out, float* seq_out, int* flag, void* stream) {
    if (r < 1 || n_graphs < 1 || n_sites < 1 || n_sites > 14 || beam < 1 || beam > 32 || n_states < 1 ||
        n_states > beam || slot0 < 0 || slot0 + r > n_states * n_sites * 20 || n_nodes < 0 || seq_len < 1 || vocab < 1)
        return IS_ERR_ARG;
    if (!x23 || !node_off || !node_index || !seq || !seq_index || !seq_columns || !states || !n_mut || !valid || !native ||
        !allowed || !x23_out || !seq_out || !flag)
        return IS_ERR_ARG;
    if ((int64_t)r * n_graphs > 0x3fffffff || (int64_t)seq_len * vocab > 0x7fffffff) return IS_ERR_UNSUPPORTED;
    const int64_t units = 2 * (int64_t)r * n_graphs, cap = (int64_t)DX_CTAS_PER_SM * current_num_sms();
    design_expand_kernel<<<(unsigned)(units < cap ? units : cap), DX_THREADS, 0, (cudaStream_t)stream>>>(
        x23, node_off, node_index, seq, seq_index, seq_columns, states, n_mut, valid, native, allowed, slot0, r,
        n_graphs, n_sites, beam, n_states, max_mutations, n_nodes, seq_len, vocab, x23_out, seq_out, flag);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

// grid: one CTA of 256 threads per sample, (n_states (1 + 20 P)) x 12 bytes of dynamic shared memory (108 KB at the caps)
int is_design_select(const int64_t* states, const int64_t* keys, const int64_t* n_mut, const unsigned char* valid,
                     const float* logits, const float* prob_mean, const float* prob_std, const float* round_logits,
                     const float* round_mean, const float* round_std, const int64_t* native, const unsigned char* allowed,
                     const int64_t* node_index, int n_graphs, int n_sites, int beam, int n_states, int n_draws,
                     int max_mutations, float kappa, int maximize, int64_t* states_out, int64_t* keys_out,
                     int64_t* n_mut_out, unsigned char* valid_out, float* logits_out, float* mean_out, float* std_out,
                     float* objective_out, float* best, int64_t best_stride, void* stream) {
    if (n_graphs < 1 || n_sites < 1 || n_sites > 14 || beam < 1 || beam > 32 || n_states < 1 || n_states > beam ||
        n_draws < 1 || best_stride < 1)
        return IS_ERR_ARG;
    if (!states || !keys || !n_mut || !valid || !logits || !prob_mean || !prob_std || !round_logits || !round_mean ||
        !round_std || !native || !allowed || !node_index || !states_out || !keys_out || !n_mut_out || !valid_out ||
        !logits_out || !mean_out || !std_out || !objective_out || !best)
        return IS_ERR_ARG;
    const size_t smem = (size_t)n_states * (1 + 20 * n_sites) * (sizeof(int64_t) + sizeof(float));
    cudaError_t e = cudaFuncSetAttribute(design_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    design_select_kernel<<<(unsigned)n_graphs, DS_THREADS, smem, (cudaStream_t)stream>>>(
        states, keys, n_mut, valid, logits, prob_mean, prob_std, round_logits, round_mean, round_std, native, allowed,
        node_index, n_graphs, n_sites, beam, n_states, n_draws, max_mutations, kappa, maximize, states_out, keys_out,
        n_mut_out, valid_out, logits_out, mean_out, std_out, objective_out, best, best_stride);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

}  // extern "C"
