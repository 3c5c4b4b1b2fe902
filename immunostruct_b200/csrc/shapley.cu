// Shapley values of residues and residue groups over structural removals (immunostruct_b200/shapley.py).
//
// Players of sample b are graph-local ids 0 .. P_b - 1 held by its node rows (players[i] = -1: the row is never removed),
// P_b <= 256.  Removing a set S of players zeroes the 23 floats of every row of S and drops every edge with an endpoint
// in such a row; the kept edges keep their base order (as is_occlusion_expand).  Permutation pair u = 0 .. T/2 - 1 of
// sample b orders the players by the key v0 of Philox4x32-10 with counter (p, b, u, 2) and key (low, high 32 bits of
// seed), ties to the smaller id: rank_2u(p) = #{q : (key_q, q) < (key_p, p)}; permutation 2u + 1 is its reverse,
// rank_2u+1(p) = P_b - 1 - rank_2u(p) (antithetic pair).  Coalition (t, j) removes the players with rank_t < j.
//
// Variants of sample b start at var_off[b]: the empty coalition (every player removed, j = P_b) first, then j = 1 ..
// P_b - 1 of each permutation t ascending; 1 + T (P_b - 1) variants, none without players.  j = 0 is the base batch.
//
// is_shapley_plan: one CTA per (sample b, pair u).  The P_b keys are drawn and ranked in shared memory (O(P^2) compares),
// the two rank rows are written to ranks [B, T, Pmax] (-1 past P_b), and the kept-edge count of every chain variant of
// both permutations comes from one pass over the graph's edges: an edge is kept in coalition j iff j <= the smaller rank
// of its player endpoints (P_b for a non-player endpoint), so a histogram of that minimum per permutation, read as a
// suffix sum, gives every count.  Integer shared-memory counts only.
//
// is_shapley_expand: one pass of coalition variants, variant v = (base sample, rank row, threshold j): row i of the
// sample is removed iff players[i] >= 0 and ranks[rank_row][players[i]] < j.  Work units are (variant, part), grid-strided
// as in is_occlusion_expand: the unit's removed-row mask goes to shared memory (n_b <= 256), part 0 copies the rows with
// the removed ones zeroed, part 1 compacts the kept edges in base order without atomics (warp slices, ballots, one
// shared-memory scan of the warp counts).  Both parts check the kept count against edge_out, so a variant is written
// whole or not at all; copies and 0.0 only, bit-exact.
//
// is_shapley_reduce: one CTA per sample, one thread per player.  v_logit(t, j) = mean over the K draws of the logit and
// v_prob(t, j) = mean of sigmoid(logit), in fp64.  The player at position j - 1 of permutation t gets
// Δ = v(t, j - 1) - v(t, j); d_u = (Δ_2u + Δ_2u+1) / 2, φ = mean over u of d_u, se = sqrt(Σ_u (d_u - φ)^2 / (U (U - 1)))
// (NaN for U = 1), each accumulated over u ascending by its own thread: no atomics, independent of the pass split.
// gap = (v(base) - v(empty)) - Σ_p φ(p), summed in player order.
//
// The flag (int32, set to 1, never cleared here) reports tables that disagree with the batch: an index out of range, a
// variant count that is not 1 + T (P_b - 1), P_b > min(256, Pmax), a player id of a row past the rank row, offsets that
// disagree with the node or kept counts or run past the outputs, or a rank row that is not a permutation.
//
// Contact games (shapley.contact_shapley) use the same chains, variant order and reduction with edges as the players:
// is_shapley_edge_plan and is_shapley_edge_expand below.
#include "common.cuh"
#include "philox.cuh"

namespace is {

constexpr int SH_THREADS = 256;
constexpr int SH_WARPS = SH_THREADS / 32;
constexpr int SH_MAX = 256;                     // players per sample, and rows per graph in the expansion's mask
constexpr int SH_CTAS_PER_SM = 4;
constexpr uint32_t SH_STREAM = 2;               // counter word 3: apart from coordnoise's items 0 and 1

__device__ __forceinline__ void sh_raise(int* flag) { *(volatile int*)flag = 1; }

// The P keys of pair u of sample b (counter (p, b, u, stream)) and their ranks, ties to the smaller id; clears the two
// histograms while the keys are drawn.  Ends with rank[0 .. P) written and not yet synchronised.  tid = threadIdx.x;
// its range is restated so that the ranking loop compiles as it did written inline in shapley_plan_kernel.
__device__ __forceinline__ void sh_rank(uint32_t* key, int* rank, int (*hist)[SH_MAX + 1], int tid, int P, int b,
                                        int u, uint32_t stream, uint32_t k0, uint32_t k1) {
    __builtin_assume(tid >= 0 && tid < SH_THREADS);
    if (tid < P) key[tid] = philox4x32_10((uint32_t)tid, (uint32_t)b, (uint32_t)u, stream, k0, k1).v[0];
    for (int i = tid; i < 2 * (SH_MAX + 1); i += SH_THREADS) (&hist[0][0])[i] = 0;
    __syncthreads();
    if (tid < P) {
        const uint32_t kp = key[tid];
        int r = 0;
        for (int q = 0; q < P; ++q) {
            const uint32_t kq = key[q];
            r += kq < kp || (kq == kp && q < tid);
        }
        rank[tid] = r;
    }
}

__global__ void __launch_bounds__(SH_THREADS) shapley_plan_kernel(
        const int64_t* __restrict__ node_off, const int64_t* __restrict__ edge_off, const int64_t* __restrict__ src_local,
        const int64_t* __restrict__ dst_local, const int* __restrict__ players, const int64_t* __restrict__ player_off,
        const int64_t* __restrict__ var_off, int T, int pmax, uint32_t k0, uint32_t k1, int* __restrict__ ranks,
        int64_t* __restrict__ kept, int* __restrict__ flag) {
    __shared__ uint32_t key[SH_MAX];
    __shared__ int rank[SH_MAX];
    __shared__ int hist[2][SH_MAX + 1];
    const int b = blockIdx.x, u = blockIdx.y, tid = threadIdx.x;
    const int64_t P64 = __ldg(player_off + b + 1) - __ldg(player_off + b);
    const int64_t v0 = __ldg(var_off + b), nvar = __ldg(var_off + b + 1) - v0;
    if (P64 < 0 || P64 > SH_MAX || P64 > pmax || v0 < 0 || nvar != (P64 ? 1 + (int64_t)T * (P64 - 1) : 0)) {
        if (tid == 0) sh_raise(flag);
        return;
    }
    const int P = (int)P64;
    int* row0 = ranks + ((int64_t)b * T + 2 * u) * pmax;
    int* row1 = row0 + pmax;
    if (P == 0) {
        for (int p = tid; p < pmax; p += SH_THREADS) row0[p] = row1[p] = -1;
        return;
    }
    sh_rank(key, rank, hist, tid, P, b, u, SH_STREAM, k0, k1);
    __syncthreads();
    for (int p = tid; p < pmax; p += SH_THREADS) {
        row0[p] = p < P ? rank[p] : -1;
        row1[p] = p < P ? P - 1 - rank[p] : -1;
    }
    const int64_t n0 = __ldg(node_off + b), nb = __ldg(node_off + b + 1) - n0;
    const int64_t e0 = __ldg(edge_off + b), eb = __ldg(edge_off + b + 1) - e0;
    for (int64_t i = tid; i < eb; i += SH_THREADS) {
        const int64_t s = __ldg(src_local + e0 + i), d = __ldg(dst_local + e0 + i);
        const int ps = (uint64_t)s < (uint64_t)nb ? __ldg(players + n0 + s) : -1;
        const int pd = (uint64_t)d < (uint64_t)nb ? __ldg(players + n0 + d) : -1;
        const bool hs = (unsigned)ps < (unsigned)P, hd = (unsigned)pd < (unsigned)P;
        const int rs = hs ? rank[ps] : P, rd = hd ? rank[pd] : P;                  // P: never removed
        const int qs = hs ? P - 1 - rs : P, qd = hd ? P - 1 - rd : P;              // the reversed permutation
        atomicAdd(&hist[0][min(rs, rd)], 1);
        atomicAdd(&hist[1][min(qs, qd)], 1);
    }
    __syncthreads();
    // coalition j keeps the edges whose minimum rank is >= j: kept(j) = hist[j] + ... + hist[P]
    for (int j = 1 + tid; j < P; j += SH_THREADS) {
        int64_t s0 = 0, s1 = 0;
        for (int m = j; m <= P; ++m) { s0 += hist[0][m]; s1 += hist[1][m]; }
        kept[v0 + 1 + (int64_t)(2 * u) * (P - 1) + (j - 1)] = s0;
        kept[v0 + 1 + (int64_t)(2 * u + 1) * (P - 1) + (j - 1)] = s1;
    }
    if (u == 0 && tid == 0) kept[v0] = hist[0][P];                                 // every player removed
}

// an edge is kept unless an endpoint is a removed row of the graph
__device__ __forceinline__ bool sh_keep(int64_t s, int64_t d, int64_t nb, const unsigned char* gone) {
    return !(((uint64_t)s < (uint64_t)nb && gone[s]) || ((uint64_t)d < (uint64_t)nb && gone[d]));
}

__global__ void __launch_bounds__(SH_THREADS, SH_CTAS_PER_SM) shapley_expand_kernel(
        const float* __restrict__ x23, const int64_t* __restrict__ node_off, const int64_t* __restrict__ edge_off,
        const int64_t* __restrict__ src_local, const int64_t* __restrict__ dst_local, const float* __restrict__ edge_attr,
        const int* __restrict__ players, const int* __restrict__ ranks, const int64_t* __restrict__ sample,
        const int64_t* __restrict__ rank_row, const int64_t* __restrict__ threshold, const int64_t* __restrict__ node_out,
        const int64_t* __restrict__ edge_out, int r, int B, int64_t n_rows, int pmax, int64_t n_out, int64_t e_out,
        float* __restrict__ x23_out, int64_t* __restrict__ src_out, int64_t* __restrict__ dst_out,
        float* __restrict__ edge_attr_out, int* __restrict__ flag) {
    __shared__ int64_t warp_base[SH_WARPS + 1];
    __shared__ unsigned char gone[SH_MAX];
    const int64_t units = 2 * (int64_t)r;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t unit = blockIdx.x; unit < units; unit += gridDim.x) {
        const int v = (int)(unit >> 1), part = (int)(unit & 1);
        const int64_t b = __ldg(sample + v), row = __ldg(rank_row + v), j = __ldg(threshold + v);
        if (b < 0 || b >= B || row < 0 || row >= n_rows || j < 0 || j > pmax) {
            if (part == 0 && threadIdx.x == 0) sh_raise(flag);
            continue;
        }
        const int64_t n0 = __ldg(node_off + b), nb = __ldg(node_off + b + 1) - n0;
        const int64_t e0 = __ldg(edge_off + b), eb = __ldg(edge_off + b + 1) - e0;
        const int64_t no = __ldg(node_out + v), eo = __ldg(edge_out + v), ek = __ldg(edge_out + v + 1) - eo;
        if (nb > SH_MAX || no < 0 || __ldg(node_out + v + 1) - no != nb || no + nb > n_out || eo < 0 || ek < 0 ||
            eo + ek > e_out) {
            if (part == 0 && threadIdx.x == 0) sh_raise(flag);
            continue;
        }
        const int* rk = ranks + row * pmax;
        __syncthreads();                                                 // the previous unit's mask is consumed
        bool bad = false;
        for (int i = threadIdx.x; i < nb; i += SH_THREADS) {
            const int id = __ldg(players + n0 + i);
            bad |= id >= pmax;
            gone[i] = id >= 0 && id < pmax && __ldg(rk + id) < j;
        }
        if (__syncthreads_or(bad)) {                                     // CTA-uniform
            if (part == 0 && threadIdx.x == 0) sh_raise(flag);
            continue;
        }
        const int64_t* src = src_local + e0;
        const int64_t* dst = dst_local + e0;
        const int64_t per = (eb + SH_WARPS - 1) / SH_WARPS;              // warp slice: [warp * per, (warp + 1) * per)
        const int64_t lo = min((int64_t)warp * per, eb), hi = min(lo + per, eb);
        int64_t kept = 0;
        for (int64_t i0 = lo; i0 < hi; i0 += 32) {
            const int64_t i = i0 + lane;
            const bool keep = i < hi && sh_keep(__ldg(src + i), __ldg(dst + i), nb, gone);
            kept += __popc(__ballot_sync(0xffffffffu, keep));
        }
        if (lane == 0) warp_base[warp + 1] = kept;
        __syncthreads();
        if (threadIdx.x == 0) {
            warp_base[0] = 0;
            for (int w = 1; w <= SH_WARPS; ++w) warp_base[w] += warp_base[w - 1];
        }
        __syncthreads();
        if (warp_base[SH_WARPS] != ek) {                                 // CTA-uniform
            if (part == 1 && threadIdx.x == 0) sh_raise(flag);
            continue;
        }
        if (part == 0) {
            const int n = (int)nb * 23;
            const float* xs = x23 + n0 * 23;
            float* xd = x23_out + no * 23;
            for (int i = threadIdx.x; i < n; i += SH_THREADS) xd[i] = gone[i / 23] ? 0.0f : __ldg(xs + i);
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
                keep = sh_keep(s, d, nb, gone);
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

// ---- contact games: the players are sets of edges ------------------------------------------------------------------
//
// edge_players[e] is the graph-local player id of edge e (-1: never removed).  Removing a set of players drops their
// edges; rows, the attributes of the kept edges and their base order are unchanged.  The keys use counter word 3 =
// SH_EDGE_STREAM, so the permutations of a contact game are independent of a residue game's on the same seed.

constexpr uint32_t SH_EDGE_STREAM = 3;          // apart from coordnoise's 0 and 1 and the residue games' 2

// One CTA per (sample b, pair u), as shapley_plan_kernel: an edge of player q is kept in coalition j iff j <= rank_t(q),
// an edge without a player (or with an id outside [0, P_b)) always, so a histogram of its rank per permutation, read as
// a suffix sum, gives every kept count.
__global__ void __launch_bounds__(SH_THREADS) shapley_edge_plan_kernel(
        const int64_t* __restrict__ edge_off, const int* __restrict__ edge_players,
        const int64_t* __restrict__ player_off, const int64_t* __restrict__ var_off, int T, int pmax, uint32_t k0,
        uint32_t k1, int* __restrict__ ranks, int64_t* __restrict__ kept, int* __restrict__ flag) {
    __shared__ uint32_t key[SH_MAX];
    __shared__ int rank[SH_MAX];
    __shared__ int hist[2][SH_MAX + 1];
    const int b = blockIdx.x, u = blockIdx.y, tid = threadIdx.x;
    const int64_t P64 = __ldg(player_off + b + 1) - __ldg(player_off + b);
    const int64_t v0 = __ldg(var_off + b), nvar = __ldg(var_off + b + 1) - v0;
    if (P64 < 0 || P64 > SH_MAX || P64 > pmax || v0 < 0 || nvar != (P64 ? 1 + (int64_t)T * (P64 - 1) : 0)) {
        if (tid == 0) sh_raise(flag);
        return;
    }
    const int P = (int)P64;
    int* row0 = ranks + ((int64_t)b * T + 2 * u) * pmax;
    int* row1 = row0 + pmax;
    if (P == 0) {
        for (int p = tid; p < pmax; p += SH_THREADS) row0[p] = row1[p] = -1;
        return;
    }
    sh_rank(key, rank, hist, tid, P, b, u, SH_EDGE_STREAM, k0, k1);
    __syncthreads();
    for (int p = tid; p < pmax; p += SH_THREADS) {
        row0[p] = p < P ? rank[p] : -1;
        row1[p] = p < P ? P - 1 - rank[p] : -1;
    }
    const int64_t e0 = __ldg(edge_off + b), eb = __ldg(edge_off + b + 1) - e0;
    for (int64_t i = tid; i < eb; i += SH_THREADS) {
        const int q = __ldg(edge_players + e0 + i);
        const bool h = (unsigned)q < (unsigned)P;
        const int r = h ? rank[q] : P;                                              // P: never removed
        atomicAdd(&hist[0][r], 1);
        atomicAdd(&hist[1][h ? P - 1 - r : P], 1);                                  // the reversed permutation
    }
    __syncthreads();
    // coalition j keeps the edges whose rank is >= j: kept(j) = hist[j] + ... + hist[P]
    for (int j = 1 + tid; j < P; j += SH_THREADS) {
        int64_t s0 = 0, s1 = 0;
        for (int m = j; m <= P; ++m) { s0 += hist[0][m]; s1 += hist[1][m]; }
        kept[v0 + 1 + (int64_t)(2 * u) * (P - 1) + (j - 1)] = s0;
        kept[v0 + 1 + (int64_t)(2 * u + 1) * (P - 1) + (j - 1)] = s1;
    }
    if (u == 0 && tid == 0) kept[v0] = hist[0][P];                                 // every player removed
}

// One pass of contact coalitions, units (variant, part) grid-strided as shapley_expand_kernel.  The unit's rank row is
// staged in shared memory; an edge with id q >= 0 is dropped iff rank[q] < j.  Part 0 copies the rows verbatim, part 1
// compacts the kept edges in base order (warp slices, ballots, one scan of the warp counts); both check the kept count
// against edge_out first, so a variant is written whole or not at all.
__global__ void __launch_bounds__(SH_THREADS, SH_CTAS_PER_SM) shapley_edge_expand_kernel(
        const float* __restrict__ x23, const int64_t* __restrict__ node_off, const int64_t* __restrict__ edge_off,
        const int64_t* __restrict__ src_local, const int64_t* __restrict__ dst_local, const float* __restrict__ edge_attr,
        const int* __restrict__ edge_players, const int* __restrict__ ranks, const int64_t* __restrict__ sample,
        const int64_t* __restrict__ rank_row, const int64_t* __restrict__ threshold, const int64_t* __restrict__ node_out,
        const int64_t* __restrict__ edge_out, int r, int B, int64_t n_rows, int pmax, int64_t n_out, int64_t e_out,
        float* __restrict__ x23_out, int64_t* __restrict__ src_out, int64_t* __restrict__ dst_out,
        float* __restrict__ edge_attr_out, int* __restrict__ flag) {
    __shared__ int64_t warp_base[SH_WARPS + 1];
    __shared__ int rk[SH_MAX];
    const int64_t units = 2 * (int64_t)r;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t unit = blockIdx.x; unit < units; unit += gridDim.x) {
        const int v = (int)(unit >> 1), part = (int)(unit & 1);
        const int64_t b = __ldg(sample + v), row = __ldg(rank_row + v), j = __ldg(threshold + v);
        if (b < 0 || b >= B || row < 0 || row >= n_rows || j < 0 || j > pmax) {
            if (part == 0 && threadIdx.x == 0) sh_raise(flag);
            continue;
        }
        const int64_t n0 = __ldg(node_off + b), nb = __ldg(node_off + b + 1) - n0;
        const int64_t e0 = __ldg(edge_off + b), eb = __ldg(edge_off + b + 1) - e0;
        const int64_t no = __ldg(node_out + v), eo = __ldg(edge_out + v), ek = __ldg(edge_out + v + 1) - eo;
        if (nb < 0 || no < 0 || __ldg(node_out + v + 1) - no != nb || no + nb > n_out || eo < 0 || ek < 0 ||
            eo + ek > e_out) {
            if (part == 0 && threadIdx.x == 0) sh_raise(flag);
            continue;
        }
        __syncthreads();                                                 // the previous unit's rank row is consumed
        for (int p = threadIdx.x; p < pmax; p += SH_THREADS) rk[p] = __ldg(ranks + row * pmax + p);
        __syncthreads();
        const int* ids = edge_players + e0;
        const int64_t per = (eb + SH_WARPS - 1) / SH_WARPS;              // warp slice: [warp * per, (warp + 1) * per)
        const int64_t lo = min((int64_t)warp * per, eb), hi = min(lo + per, eb);
        int64_t kept = 0;
        bool bad = false;
        for (int64_t i0 = lo; i0 < hi; i0 += 32) {
            const int64_t i = i0 + lane;
            const int q = i < hi ? __ldg(ids + i) : -1;
            bad |= q >= pmax;
            kept += __popc(__ballot_sync(0xffffffffu, i < hi && (q < 0 || (q < pmax && rk[q] >= j))));
        }
        if (lane == 0) warp_base[warp + 1] = kept;
        if (__syncthreads_or(bad)) {                                     // CTA-uniform
            if (part == 0 && threadIdx.x == 0) sh_raise(flag);
            continue;
        }
        if (threadIdx.x == 0) {
            warp_base[0] = 0;
            for (int w = 1; w <= SH_WARPS; ++w) warp_base[w] += warp_base[w - 1];
        }
        __syncthreads();
        if (warp_base[SH_WARPS] != ek) {                                 // CTA-uniform
            if (part == 1 && threadIdx.x == 0) sh_raise(flag);
            continue;
        }
        if (part == 0) {
            const int64_t n = nb * 23;
            const float* xs = x23 + n0 * 23;
            float* xd = x23_out + no * 23;
            for (int64_t i = threadIdx.x; i < n; i += SH_THREADS) xd[i] = __ldg(xs + i);
            continue;
        }
        int64_t out = eo + warp_base[warp];
        for (int64_t i0 = lo; i0 < hi; i0 += 32) {
            const int64_t i = i0 + lane;
            const int q = i < hi ? __ldg(ids + i) : -1;
            const bool keep = i < hi && (q < 0 || rk[q] >= j);           // q < pmax: checked above
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            if (keep) {
                const int64_t o = out + __popc(m & ((1u << lane) - 1u));
                src_out[o] = __ldg(src_local + e0 + i);
                dst_out[o] = __ldg(dst_local + e0 + i);
                edge_attr_out[o] = __ldg(edge_attr + e0 + i);
            }
            out += __popc(m);
        }
    }
}

// (v_logit, v_prob) of the K draws at row `lg`, in fp64, summed over k ascending
__device__ __forceinline__ void sh_value(const float* __restrict__ lg, int K, double& vl, double& vp) {
    double sl = 0.0, sp = 0.0;
    for (int k = 0; k < K; ++k) {
        const double x = (double)__ldg(lg + k);
        sl += x;
        sp += __drcp_rn(1.0 + exp(-x));                          // = 1.0 / (1.0 + exp(-x)), correctly rounded
    }
    vl = sl / K;
    vp = sp / K;
}

__global__ void __launch_bounds__(SH_THREADS) shapley_reduce_kernel(
        const float* __restrict__ logits, const float* __restrict__ base, const int* __restrict__ ranks,
        const int64_t* __restrict__ player_off, const int64_t* __restrict__ var_off, int T, int pmax, int K,
        int64_t n_var, float* __restrict__ phi_logit, float* __restrict__ phi_prob, float* __restrict__ se_logit,
        float* __restrict__ se_prob, float* __restrict__ gap_logit, float* __restrict__ gap_prob, int* __restrict__ flag) {
    __shared__ double val[2][SH_MAX + 1];                                // v_logit, v_prob of j = 0 .. P of one permutation
    __shared__ double acc[6][SH_MAX];
    __shared__ int bad_s;
    const int b = blockIdx.x, p = threadIdx.x;
    const int64_t q0 = __ldg(player_off + b), P64 = __ldg(player_off + b + 1) - q0;
    const int64_t v0 = __ldg(var_off + b), nvar = __ldg(var_off + b + 1) - v0;
    if (P64 < 0 || P64 > SH_MAX || P64 > pmax || v0 < 0 || v0 + nvar > n_var ||
        nvar != (P64 ? 1 + (int64_t)T * (P64 - 1) : 0)) {
        if (p == 0) sh_raise(flag);
        return;
    }
    const int P = (int)P64, U = T / 2;
    if (P == 0) {                                                        // empty = base: nothing to attribute
        if (p == 0) gap_logit[b] = gap_prob[b] = 0.0f;
        return;
    }
    const int* rows = ranks + (int64_t)b * T * pmax;
    // player p's accumulators live in shared memory, not registers: the fp64 divisions of the value loop are calls
    double* dl = acc[0] + p;                                             // Δ_2u + Δ_2u+1 of the pair in progress
    double* dp = acc[1] + p;
    double* fl = acc[2] + p;                                             // Σ d_u, then φ
    double* fp = acc[3] + p;
    double* ql = acc[4] + p;                                             // Σ (d_u - φ)^2
    double* qp = acc[5] + p;
    if (p < P) *dl = *dp = *fl = *fp = *ql = *qp = 0.0;
    if (p == 0) bad_s = 0;
    // pass 0 sums d_u into φ, pass 1 sums (d_u - φ)^2; both over t ascending
    for (int pass = 0; pass < 2; ++pass) {
        for (int t = 0; t < T; ++t) {
            __syncthreads();                                             // the previous permutation's values are consumed
            for (int j = p; j <= P; j += SH_THREADS) {
                const float* lg = j == 0 ? base + (int64_t)b * K
                                : logits + (j == P ? v0 : v0 + 1 + (int64_t)t * (P - 1) + (j - 1)) * K;
                double vl, vp;
                sh_value(lg, K, vl, vp);
                val[0][j] = vl;
                val[1][j] = vp;
            }
            __syncthreads();
            if (p < P) {
                const int r = __ldg(rows + (int64_t)t * pmax + p);
                if (r < 0 || r >= P) {
                    bad_s = 1;
                    continue;
                }
                *dl += val[0][r] - val[0][r + 1];
                *dp += val[1][r] - val[1][r + 1];
                if (t & 1) {                                             // d_u of the antithetic pair u = t / 2
                    const double el = *dl * 0.5, ep = *dp * 0.5;
                    if (pass == 0) {
                        *fl += el;
                        *fp += ep;
                    } else {
                        *ql += (el - *fl) * (el - *fl);
                        *qp += (ep - *fp) * (ep - *fp);
                    }
                    *dl = *dp = 0.0;
                }
            }
        }
        if (pass == 0 && p < P) {
            *fl /= U;
            *fp /= U;
        }
    }
    __syncthreads();
    if (bad_s) {
        if (p == 0) sh_raise(flag);
        return;
    }
    if (p < P) {
        const double den = (double)U * (double)(U - 1);
        phi_logit[q0 + p] = (float)*fl;
        phi_prob[q0 + p] = (float)*fp;
        se_logit[q0 + p] = U > 1 ? (float)sqrt(*ql / den) : __int_as_float(0x7fc00000);
        se_prob[q0 + p] = U > 1 ? (float)sqrt(*qp / den) : __int_as_float(0x7fc00000);
    }
    __syncthreads();
    if (p == 0) {                                                        // val[.][0] = v(base), val[.][P] = v(empty)
        double sl = 0.0, sp = 0.0;
        for (int q = 0; q < P; ++q) { sl += acc[2][q]; sp += acc[3][q]; }
        gap_logit[b] = (float)((val[0][0] - val[0][P]) - sl);
        gap_prob[b] = (float)((val[1][0] - val[1][P]) - sp);
    }
}

}  // namespace is

using namespace is;

extern "C" {

// grid: (B, T/2) CTAs of 256 threads
int is_shapley_plan(const int64_t* node_off, const int64_t* edge_off, const int64_t* src_local, const int64_t* dst_local,
                    const int* players, const int64_t* player_off, const int64_t* var_off, int n_graphs,
                    int permutations, int max_players, uint64_t seed, int* ranks, int64_t* kept, int* flag,
                    void* stream) {
    if (n_graphs < 1 || permutations < 2 || permutations % 2 || max_players < 1 || !node_off || !edge_off ||
        !players || !player_off || !var_off || !ranks || !kept || !flag)
        return IS_ERR_ARG;
    if (permutations > 65536) return IS_ERR_UNSUPPORTED;
    shapley_plan_kernel<<<dim3((unsigned)n_graphs, (unsigned)(permutations / 2)), SH_THREADS, 0, (cudaStream_t)stream>>>(
        node_off, edge_off, src_local, dst_local, players, player_off, var_off, permutations, max_players,
        (uint32_t)seed, (uint32_t)(seed >> 32), ranks, kept, flag);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

// grid: min(2 r, 4 x SMs) CTAs of 256 threads, each looping over (variant, part) units
int is_shapley_expand(const float* x23, const int64_t* node_off, const int64_t* edge_off, const int64_t* src_local,
                      const int64_t* dst_local, const float* edge_attr, const int* players, const int* ranks,
                      const int64_t* sample, const int64_t* rank_row, const int64_t* threshold, const int64_t* node_out,
                      const int64_t* edge_out, int r, int n_graphs, int64_t n_rank_rows, int max_players,
                      int64_t n_nodes_out, int64_t n_edges_out, float* x23_out, int64_t* src_out, int64_t* dst_out,
                      float* edge_attr_out, int* flag, void* stream) {
    if (r < 1 || n_graphs < 1 || n_rank_rows < 1 || max_players < 1 || n_nodes_out < 0 || n_edges_out < 0) return IS_ERR_ARG;
    if (!x23 || !node_off || !edge_off || !players || !ranks || !sample || !rank_row || !threshold || !node_out ||
        !edge_out || !flag || (n_nodes_out > 0 && !x23_out) ||
        (n_edges_out > 0 && (!src_local || !dst_local || !edge_attr || !src_out || !dst_out || !edge_attr_out)))
        return IS_ERR_ARG;
    if ((int64_t)r > 0x3fffffff) return IS_ERR_UNSUPPORTED;
    const int64_t units = 2 * (int64_t)r, cap = (int64_t)SH_CTAS_PER_SM * current_num_sms();
    shapley_expand_kernel<<<(unsigned)(units < cap ? units : cap), SH_THREADS, 0, (cudaStream_t)stream>>>(
        x23, node_off, edge_off, src_local, dst_local, edge_attr, players, ranks, sample, rank_row, threshold, node_out,
        edge_out, r, n_graphs, n_rank_rows, max_players, n_nodes_out, n_edges_out, x23_out, src_out, dst_out,
        edge_attr_out, flag);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

// grid: (B, T/2) CTAs of 256 threads
int is_shapley_edge_plan(const int64_t* edge_off, const int* edge_players, const int64_t* player_off,
                         const int64_t* var_off, int n_graphs, int permutations, int max_players, uint64_t seed,
                         int* ranks, int64_t* kept, int* flag, void* stream) {
    if (n_graphs < 1 || permutations < 2 || permutations % 2 || max_players < 1 || !edge_off || !player_off ||
        !var_off || !ranks || !kept || !flag)
        return IS_ERR_ARG;
    if (permutations > 65536 || max_players > SH_MAX) return IS_ERR_UNSUPPORTED;
    shapley_edge_plan_kernel<<<dim3((unsigned)n_graphs, (unsigned)(permutations / 2)), SH_THREADS, 0,
                               (cudaStream_t)stream>>>(edge_off, edge_players, player_off, var_off, permutations,
                                                       max_players, (uint32_t)seed, (uint32_t)(seed >> 32), ranks,
                                                       kept, flag);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

// grid: min(2 r, 4 x SMs) CTAs of 256 threads, each looping over (variant, part) units
int is_shapley_edge_expand(const float* x23, const int64_t* node_off, const int64_t* edge_off,
                           const int64_t* src_local, const int64_t* dst_local, const float* edge_attr,
                           const int* edge_players, const int* ranks, const int64_t* sample, const int64_t* rank_row,
                           const int64_t* threshold, const int64_t* node_out, const int64_t* edge_out, int r,
                           int n_graphs, int64_t n_rank_rows, int max_players, int64_t n_nodes_out,
                           int64_t n_edges_out, float* x23_out, int64_t* src_out, int64_t* dst_out,
                           float* edge_attr_out, int* flag, void* stream) {
    if (r < 1 || n_graphs < 1 || n_rank_rows < 1 || max_players < 1 || n_nodes_out < 0 || n_edges_out < 0) return IS_ERR_ARG;
    if (!x23 || !node_off || !edge_off || !ranks || !sample || !rank_row || !threshold || !node_out || !edge_out ||
        !flag || (n_nodes_out > 0 && !x23_out) ||
        (n_edges_out > 0 && (!src_local || !dst_local || !edge_attr || !edge_players || !src_out || !dst_out ||
                             !edge_attr_out)))
        return IS_ERR_ARG;
    if ((int64_t)r > 0x3fffffff || max_players > SH_MAX) return IS_ERR_UNSUPPORTED;
    const int64_t units = 2 * (int64_t)r, cap = (int64_t)SH_CTAS_PER_SM * current_num_sms();
    shapley_edge_expand_kernel<<<(unsigned)(units < cap ? units : cap), SH_THREADS, 0, (cudaStream_t)stream>>>(
        x23, node_off, edge_off, src_local, dst_local, edge_attr, edge_players, ranks, sample, rank_row, threshold,
        node_out, edge_out, r, n_graphs, n_rank_rows, max_players, n_nodes_out, n_edges_out, x23_out, src_out, dst_out,
        edge_attr_out, flag);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

// grid: B CTAs of 256 threads, one per sample
int is_shapley_reduce(const float* logits, const float* base_logits, const int* ranks, const int64_t* player_off,
                      const int64_t* var_off, int n_graphs, int permutations, int max_players, int n_draws,
                      int64_t n_variants, float* phi_logit, float* phi_prob, float* se_logit, float* se_prob,
                      float* gap_logit, float* gap_prob, int* flag, void* stream) {
    if (n_graphs < 1 || permutations < 2 || permutations % 2 || max_players < 1 || n_draws < 1 || n_variants < 0 ||
        !base_logits || !ranks || !player_off || !var_off || !gap_logit || !gap_prob || !flag ||
        (n_variants > 0 && (!logits || !phi_logit || !phi_prob || !se_logit || !se_prob)))
        return IS_ERR_ARG;
    shapley_reduce_kernel<<<(unsigned)n_graphs, SH_THREADS, 0, (cudaStream_t)stream>>>(
        logits, base_logits, ranks, player_off, var_off, permutations, max_players, n_draws, n_variants, phi_logit,
        phi_prob, se_logit, se_prob, gap_logit, gap_prob, flag);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

}  // extern "C"
