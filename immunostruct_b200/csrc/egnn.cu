// E(n)-equivariant message-passing layer (the reference's dgl.nn.EGNNConv(in, 64, 64, edge_feat=1),
// constructed at immunostruct/models/hybrid_models.py:29-31 / :261-263 and applied at :89-90 /
// :323-324; semantics restated in SURVEY.md Appendix A.3) as fused fp32 SIMT kernels.
//
// Algebraic restructuring (exact in real arithmetic): the first edge-MLP layer acts on
// [h_src | h_dst | radial | a], so  W1 f = Ws h_src + Wd h_dst + w_r radial + w_a a + b1.
// P = h Ws^T and Q = h Wd^T + b1 are computed once per NODE (node_pre), and the edge kernel only
// gathers and adds them.  One layer = node_pre -> edge -> node_post.
//
//   edge e=(s->d) : z1 = P[s] + Q[d] + w_r r + w_a a ; t1 = silu(z1)
//                   m  = silu(W2 t1 + b2)             ; u = silu(W3 m + b3) ; c = w4 . u
//   node d        : hn = sum_e m ; x' = x + (1/max(deg,1)) sum_e c * dhat_e
//                   h' = W6 silu(W5 [h | hn] + b5) + b6
//
// Edges are processed in destination-sorted CSR order in node-aligned tiles of <= 128 edges, so
// every destination-side reduction is a plain in-tile segment sum (warp per destination node).
// The backward pass recomputes the per-edge activations inside the tile, writes the gradient
// w.r.t. z1 ([E,64], CSR order) once, and the source-side reduction is a gather through the
// precomputed CSC transpose in node_pre_bwd -- no floating-point atomics anywhere.
// Weight gradients are accumulated in registers by persistent CTAs and written as one partial
// block per CTA; is_reduce_partials sums the blocks in CTA order.
#include "common.cuh"
#include "egnn_common.cuh"

namespace is {

// =============================================================================================
// node_pre forward:  PQ[n][0:64] = Ws h[n] ,  PQ[n][64:128] = Wd h[n] + b1
// =============================================================================================
__global__ void __launch_bounds__(IS_THREADS)
node_pre_fwd_kernel(const float* __restrict__ h, int64_t ldh, int F, const float* __restrict__ W1,
                    const float* __restrict__ b1, float* __restrict__ PQ, int64_t M) {
    extern __shared__ __align__(16) float smem[];
    const int lda = F + 4;
    float* A = smem;                    // [128][F+4]
    float* Bs = A + IS_TM * lda;        // [F][64]
    float* Bd = Bs + F * 64;            // [F][64]
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    const int ldw = 2 * F + 2;
    load_w_kmajor(Bs, W1, ldw, 0, F, tid);
    load_w_kmajor(Bd, W1, ldw, F, F, tid);
    const float4 bq = *reinterpret_cast<const float4*>(b1 + 4 * tx);
    const int64_t ntiles = (M + IS_TM - 1) / IS_TM;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int64_t m0 = t * IS_TM;
        __syncthreads();
        load_rows(A, lda, h, ldh, m0, M, F, tid);
        __syncthreads();
        float acc[8][4];
        zero_acc(acc);
        gemm_128x64(acc, A, lda, Bs, F, ty, tx);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            int64_t m = m0 + ty + 16 * i;
            if (m < M) *reinterpret_cast<float4*>(PQ + m * 128 + 4 * tx) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
        }
        zero_acc(acc);
        gemm_128x64(acc, A, lda, Bd, F, ty, tx);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            int64_t m = m0 + ty + 16 * i;
            if (m < M)
                *reinterpret_cast<float4*>(PQ + m * 128 + 64 + 4 * tx) =
                    make_float4(acc[i][0] + bq.x, acc[i][1] + bq.y, acc[i][2] + bq.z, acc[i][3] + bq.w);
        }
    }
}

// =============================================================================================
// edge forward
// =============================================================================================
template <bool HAS_COORD>
__global__ void __launch_bounds__(IS_THREADS, 2)
edge_fwd_kernel(EdgeCommon p, float* __restrict__ hn, float* __restrict__ x_out) {
    extern __shared__ __align__(16) float smem[];
    float* W2t = smem;                    // [64][64] k-major
    float* W3t = W2t + 4096;
    float* vec = W3t + 4096;              // b2, b3, w4, wr, wa
    float* A1 = vec + 5 * 64;             // [128][68]
    float* A2 = A1 + IS_TM * IS_LD;       // [128][68]
    float* e_c = A2 + IS_TM * IS_LD;      // [128]
    float* e_dh = e_c + IS_TM;            // [128][3]
    __shared__ int s_tile[4];

    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15, warp = tid >> 5, lane = tid & 31;
    const int ldw1 = 2 * p.F + 2;
    load_w_kmajor(W2t, p.W2, 64, 0, 64, tid);
    if (HAS_COORD) load_w_kmajor(W3t, p.W3, 64, 0, 64, tid);
    if (tid < 64) {
        vec[tid] = p.b2[tid];
        vec[64 + tid] = HAS_COORD ? p.b3[tid] : 0.0f;
        vec[128 + tid] = HAS_COORD ? p.w4[tid] : 0.0f;
        vec[192 + tid] = p.W1[tid * ldw1 + 2 * p.F];
        vec[256 + tid] = p.W1[tid * ldw1 + 2 * p.F + 1];
    }
    const int chunk = (p.n_nodes + gridDim.x - 1) / gridDim.x;
    int n0 = blockIdx.x * chunk;
    const int nend = min(p.n_nodes, n0 + chunk);
    __syncthreads();

    while (n0 < nend) {
        select_tile(s_tile, p.indptr, n0, nend, p.status);
        __syncthreads();
        const int n1 = s_tile[1], p0 = s_tile[2], ne = s_tile[3];
        if (ne < 0) { n0 = n1; __syncthreads(); continue; }

        // ---- gather: one warp per edge, lanes over feature pairs --------------------------------
        const float2 wr = *reinterpret_cast<const float2*>(vec + 192 + 2 * lane);
        const float2 wa = *reinterpret_cast<const float2*>(vec + 256 + 2 * lane);
#pragma unroll 2
        for (int j = warp; j < IS_TM; j += IS_THREADS / 32) {
            float2 t = make_float2(0.0f, 0.0f);
            if (j < ne) {
                const int e = p0 + j;
                const int s = __ldg(p.csr_src + e), d = __ldg(p.csr_dst + e);
                const float a = __ldg(p.edge_attr + __ldg(p.csr_eid + e));
                const float dx = __ldg(p.x + s * p.ldx + 0) - __ldg(p.x + d * p.ldx + 0);
                const float dy = __ldg(p.x + s * p.ldx + 1) - __ldg(p.x + d * p.ldx + 1);
                const float dz = __ldg(p.x + s * p.ldx + 2) - __ldg(p.x + d * p.ldx + 2);
                const float r = dx * dx + dy * dy + dz * dz;
                const float2 pv = __ldg(reinterpret_cast<const float2*>(p.PQ + (size_t)s * 128) + lane);
                const float2 qv = __ldg(reinterpret_cast<const float2*>(p.PQ + (size_t)d * 128 + 64) + lane);
                t.x = silu(pv.x + qv.x + wr.x * r + wa.x * a);
                t.y = silu(pv.y + qv.y + wr.y * r + wa.y * a);
                if (HAS_COORD && lane == 0) {
                    const float inv = 1.0f / (sqrtf(r) + 1e-30f);
                    e_dh[j * 3 + 0] = dx * inv; e_dh[j * 3 + 1] = dy * inv; e_dh[j * 3 + 2] = dz * inv;
                }
            }
            *reinterpret_cast<float2*>(A1 + j * IS_LD + 2 * lane) = t;
        }
        __syncthreads();

        // ---- m = silu(t1 W2^T + b2) -------------------------------------------------------------
        float acc[8][4];
        zero_acc(acc);
        gemm_128x64(acc, A1, IS_LD, W2t, 64, ty, tx);
        {
            const float4 b = *reinterpret_cast<const float4*>(vec + 4 * tx);
#pragma unroll
            for (int i = 0; i < 8; ++i)
                *reinterpret_cast<float4*>(A2 + (ty + 16 * i) * IS_LD + 4 * tx) =
                    make_float4(silu(acc[i][0] + b.x), silu(acc[i][1] + b.y), silu(acc[i][2] + b.z), silu(acc[i][3] + b.w));
        }
        __syncthreads();

        // ---- c = w4 . silu(m W3^T + b3) ---------------------------------------------------------
        if (HAS_COORD) {
            zero_acc(acc);
            gemm_128x64(acc, A2, IS_LD, W3t, 64, ty, tx);
            const float4 b = *reinterpret_cast<const float4*>(vec + 64 + 4 * tx);
            const float4 w = *reinterpret_cast<const float4*>(vec + 128 + 4 * tx);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                float c = w.x * silu(acc[i][0] + b.x) + w.y * silu(acc[i][1] + b.y) +
                          w.z * silu(acc[i][2] + b.z) + w.w * silu(acc[i][3] + b.w);
                c = half_warp_sum(c);
                if (tx == 0) e_c[ty + 16 * i] = c;
            }
            __syncthreads();
        }

        // ---- destination-side aggregation: one warp per destination node -----------------------
        for (int node = n0 + warp; node < n1; node += IS_THREADS / 32) {
            const int jb = __ldg(p.indptr + node) - p0, je = __ldg(p.indptr + node + 1) - p0;
            float2 s = make_float2(0.0f, 0.0f);
            for (int j = jb; j < je; ++j) {
                const float2 v = *reinterpret_cast<const float2*>(A2 + j * IS_LD + 2 * lane);
                s.x += v.x; s.y += v.y;
            }
            *reinterpret_cast<float2*>(hn + (size_t)node * 64 + 2 * lane) = s;
            if (HAS_COORD && lane < 3) {
                float sx = 0.0f;
                for (int j = jb; j < je; ++j) sx += e_c[j] * e_dh[j * 3 + lane];
                const int deg = je - jb;
                x_out[(size_t)node * 3 + lane] = __ldg(p.x + node * p.ldx + lane) + sx / (float)max(deg, 1);
            }
        }
        n0 = n1;
        __syncthreads();
    }
}

// =============================================================================================
// node_post forward:  h' = W6 silu(W5 [h | hn] + b5) + b6
// =============================================================================================
__global__ void __launch_bounds__(IS_THREADS)
node_post_fwd_kernel(const float* __restrict__ h, int64_t ldh, int F, const float* __restrict__ hn,
                     const float* __restrict__ W5, const float* __restrict__ b5,
                     const float* __restrict__ W6, const float* __restrict__ b6,
                     float* __restrict__ h_out, int64_t M) {
    extern __shared__ __align__(16) float smem[];
    const int K = F + 64, lda = K + 4;
    float* A = smem;                      // [128][K+4]
    float* T = A + IS_TM * lda;           // [128][68]
    float* B5 = T + IS_TM * IS_LD;        // [K][64]
    float* B6 = B5 + K * 64;              // [64][64]
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    load_w_kmajor(B5, W5, K, 0, K, tid);
    load_w_kmajor(B6, W6, 64, 0, 64, tid);
    const float4 bb5 = *reinterpret_cast<const float4*>(b5 + 4 * tx);
    const float4 bb6 = *reinterpret_cast<const float4*>(b6 + 4 * tx);
    const int64_t ntiles = (M + IS_TM - 1) / IS_TM;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int64_t m0 = t * IS_TM;
        __syncthreads();
        load_rows(A, lda, h, ldh, m0, M, F, tid);
        load_rows(A + F, lda, hn, 64, m0, M, 64, tid);
        __syncthreads();
        float acc[8][4];
        zero_acc(acc);
        gemm_128x64(acc, A, lda, B5, K, ty, tx);
#pragma unroll
        for (int i = 0; i < 8; ++i)
            *reinterpret_cast<float4*>(T + (ty + 16 * i) * IS_LD + 4 * tx) =
                make_float4(silu(acc[i][0] + bb5.x), silu(acc[i][1] + bb5.y), silu(acc[i][2] + bb5.z), silu(acc[i][3] + bb5.w));
        __syncthreads();
        zero_acc(acc);
        gemm_128x64(acc, T, IS_LD, B6, 64, ty, tx);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            int64_t m = m0 + ty + 16 * i;
            if (m < M)
                *reinterpret_cast<float4*>(h_out + m * 64 + 4 * tx) =
                    make_float4(acc[i][0] + bb6.x, acc[i][1] + bb6.y, acc[i][2] + bb6.z, acc[i][3] + bb6.w);
        }
    }
}

// =============================================================================================
// node_post backward.  Partial block per CTA: [gW5 64*K][gb5 64][gW6 64*64][gb6 64].
// =============================================================================================
__global__ void __launch_bounds__(IS_THREADS)
node_post_bwd_kernel(const float* __restrict__ gh_out, const float* __restrict__ h, int64_t ldh, int F,
                     const float* __restrict__ hn, const float* __restrict__ W5, const float* __restrict__ b5,
                     const float* __restrict__ W6, float* __restrict__ gh_direct /* [M,F] or null */,
                     float* __restrict__ ghn, float* __restrict__ partials, int64_t M) {
    extern __shared__ __align__(16) float smem[];
    const int K = F + 64, lda = K + 4;
    float* A = smem;                      // [128][K+4]
    float* G = A + IS_TM * lda;           // [128][68]
    float* T = G + IS_TM * IS_LD;         // [128][68]
    float* WB = T + IS_TM * IS_LD;        // [128][64] weight staging
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    const float4 bb5 = *reinterpret_cast<const float4*>(b5 + 4 * tx);
    float w6[4][4], w5a[4][4], w5b[4][4];
    zero_w(w6); zero_w(w5a); zero_w(w5b);
    float b5acc[4] = {0, 0, 0, 0}, b6acc[4] = {0, 0, 0, 0};
    const int64_t ntiles = (M + IS_TM - 1) / IS_TM;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int64_t m0 = t * IS_TM;
        __syncthreads();
        load_rows(A, lda, h, ldh, m0, M, F, tid);
        load_rows(A + F, lda, hn, 64, m0, M, 64, tid);
        load_rows(G, IS_LD, gh_out, 64, m0, M, 64, tid);
        load_w_kmajor(WB, W5, K, 0, K, tid);
        __syncthreads();
        float acc[8][4], d5[8][4];
        zero_acc(acc);
        gemm_128x64(acc, A, lda, WB, K, ty, tx);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float y[4];
            silu_both(acc[i][0] + bb5.x, y[0], d5[i][0]);
            silu_both(acc[i][1] + bb5.y, y[1], d5[i][1]);
            silu_both(acc[i][2] + bb5.z, y[2], d5[i][2]);
            silu_both(acc[i][3] + bb5.w, y[3], d5[i][3]);
            *reinterpret_cast<float4*>(T + (ty + 16 * i) * IS_LD + 4 * tx) = make_float4(y[0], y[1], y[2], y[3]);
        }
        __syncthreads();
        load_w_rowmajor(WB, W6, 64, 0, 64, tid);         // dgrad operand: rows = out index
        wgrad_64x64(w6, G, IS_LD, T, IS_LD, tid);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float4 g = *reinterpret_cast<const float4*>(G + (ty + 16 * i) * IS_LD + 4 * tx);
            b6acc[0] += g.x; b6acc[1] += g.y; b6acc[2] += g.z; b6acc[3] += g.w;
        }
        __syncthreads();
        zero_acc(acc);
        gemm_128x64(acc, G, IS_LD, WB, 64, ty, tx);      // gt5 = gh' W6
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float4 g = make_float4(acc[i][0] * d5[i][0], acc[i][1] * d5[i][1], acc[i][2] * d5[i][2], acc[i][3] * d5[i][3]);
            *reinterpret_cast<float4*>(G + (ty + 16 * i) * IS_LD + 4 * tx) = g;   // gz5 (zero on padded rows)
            b5acc[0] += g.x; b5acc[1] += g.y; b5acc[2] += g.z; b5acc[3] += g.w;
        }
        // stage W5[:, F:F+64] (the hn half) for the dgrad while the wgrads run
        load_w_rowmajor(WB, W5, K, F, 64, tid);
        if (gh_direct) load_w_rowmajor(WB + 4096, W5, K, 0, F, tid);
        __syncthreads();
        wgrad_64x64(w5a, G, IS_LD, A, lda, tid);
        wgrad_64x64(w5b, G, IS_LD, A + 64, lda, tid);
        zero_acc(acc);
        gemm_128x64(acc, G, IS_LD, WB, 64, ty, tx);      // ghn = gz5 W5[:, F:]
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            int64_t m = m0 + ty + 16 * i;
            if (m < M) *reinterpret_cast<float4*>(ghn + m * 64 + 4 * tx) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
        }
        if (gh_direct) {                                  // [M, F]: columns F .. 63 of the product are zero (zero-padded W5h)
            zero_acc(acc);
            gemm_128x64(acc, G, IS_LD, WB + 4096, 64, ty, tx);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                int64_t m = m0 + ty + 16 * i;
                if (m < M && 4 * tx < F) *reinterpret_cast<float4*>(gh_direct + m * F + 4 * tx) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
            }
        }
    }
    // ---- per-CTA partials ---------------------------------------------------------------------
    float* P = partials + (size_t)blockIdx.x * (64 * K + 64 + 4096 + 64);
    store_w(P, K, 0, w5a, tid);
    store_w(P, K, 64, w5b, tid);
    store_w(P + 64 * K + 64, 64, 0, w6, tid);
    __syncthreads();
    cta_colsum_store(T, b5acc, ty, tx);
    cta_colsum_store(T + 1024, b6acc, ty, tx);
    __syncthreads();
    if (tid < 64) {
        P[64 * K + tid] = cta_colsum_read(T, tid);
        P[64 * K + 64 + 4096 + tid] = cta_colsum_read(T + 1024, tid);
    }
}

// =============================================================================================
// edge backward.  Partial block per CTA: [gW2 4096][gW3 4096][gb2 64][gb3 64][gw4 64][gwr 64][gwa 64].
// =============================================================================================
#define IS_EDGE_BWD_PARTIAL (4096 + 4096 + 5 * 64)

template <bool HAS_COORD>
__global__ void __launch_bounds__(IS_THREADS, 1)
edge_bwd_kernel(EdgeCommon p, const float* __restrict__ ghn, const float* __restrict__ gx_out /* [N,3] */,
                float* __restrict__ gz1 /* [E,64] CSR order */, float* __restrict__ gQ /* [N,64] */,
                float* __restrict__ gD /* [E,3] CSR order: grad wrt (x_src - x_dst) */,
                float* __restrict__ gxd /* [N,3]: destination-side coordinate gradient */,
                float* __restrict__ partials) {
    extern __shared__ __align__(16) float smem[];
    float* W2t = smem;                    // k-major (forward operand)
    float* W3t = W2t + 4096;
    float* W2r = W3t + 4096;              // row-major (dgrad operand)
    float* W3r = W2r + 4096;
    float* vec = W3r + 4096;              // b2, b3, w4, wr, wa
    float* A1 = vec + 5 * 64;             // t1
    float* A2 = A1 + IS_TM * IS_LD;       // m, later gz1
    float* G = A2 + IS_TM * IS_LD;        // gz3, later gz2
    float* e_f = G + IS_TM * IS_LD;       // per-edge floats, 16 arrays of 128
    float* e_dx = e_f;                    // [3][128] raw difference
    float* e_r = e_f + 3 * IS_TM;
    float* e_a = e_f + 4 * IS_TM;
    float* e_inv = e_f + 5 * IS_TM;
    float* e_c = e_f + 6 * IS_TM;
    float* e_gc = e_f + 7 * IS_TM;
    float* e_v = e_f + 8 * IS_TM;         // [3][128] gx_out[dst] / deg
    float* e_gr = e_f + 11 * IS_TM;
    float* e_gd = e_f + 12 * IS_TM;       // [3][128]
    int* e_src = reinterpret_cast<int*>(e_f + 15 * IS_TM);
    int* e_dst = e_src + IS_TM;
    __shared__ int s_tile[4];

    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15, warp = tid >> 5, lane = tid & 31;
    const int ldw1 = 2 * p.F + 2;
    load_w_kmajor(W2t, p.W2, 64, 0, 64, tid);
    load_w_rowmajor(W2r, p.W2, 64, 0, 64, tid);
    if (HAS_COORD) {
        load_w_kmajor(W3t, p.W3, 64, 0, 64, tid);
        load_w_rowmajor(W3r, p.W3, 64, 0, 64, tid);
    }
    if (tid < 64) {
        vec[tid] = p.b2[tid];
        vec[64 + tid] = HAS_COORD ? p.b3[tid] : 0.0f;
        vec[128 + tid] = HAS_COORD ? p.w4[tid] : 0.0f;
        vec[192 + tid] = p.W1[tid * ldw1 + 2 * p.F];
        vec[256 + tid] = p.W1[tid * ldw1 + 2 * p.F + 1];
    }
    float w2[4][4], w3[4][4];
    zero_w(w2); zero_w(w3);
    float gb2[4] = {0, 0, 0, 0}, gb3[4] = {0, 0, 0, 0}, gw4[4] = {0, 0, 0, 0}, gwr[4] = {0, 0, 0, 0}, gwa[4] = {0, 0, 0, 0};

    const int chunk = (p.n_nodes + gridDim.x - 1) / gridDim.x;
    int n0 = blockIdx.x * chunk;
    const int nend = min(p.n_nodes, n0 + chunk);
    __syncthreads();
    const float4 vb2 = *reinterpret_cast<const float4*>(vec + 4 * tx);
    const float4 vb3 = *reinterpret_cast<const float4*>(vec + 64 + 4 * tx);
    const float4 vw4 = *reinterpret_cast<const float4*>(vec + 128 + 4 * tx);
    const float4 vwr = *reinterpret_cast<const float4*>(vec + 192 + 4 * tx);
    const float4 vwa = *reinterpret_cast<const float4*>(vec + 256 + 4 * tx);

    while (n0 < nend) {
        select_tile(s_tile, p.indptr, n0, nend, p.status);
        __syncthreads();
        const int n1 = s_tile[1], p0 = s_tile[2], ne = s_tile[3];
        if (ne < 0) { n0 = n1; __syncthreads(); continue; }

        // ---- gather + geometry (warp per edge) --------------------------------------------------
        {
            const float2 wr = *reinterpret_cast<const float2*>(vec + 192 + 2 * lane);
            const float2 wa = *reinterpret_cast<const float2*>(vec + 256 + 2 * lane);
#pragma unroll 2
            for (int j = warp; j < IS_TM; j += IS_THREADS / 32) {
                float2 t = make_float2(0.0f, 0.0f);
                if (j < ne) {
                    const int e = p0 + j;
                    const int s = __ldg(p.csr_src + e), d = __ldg(p.csr_dst + e);
                    const float a = __ldg(p.edge_attr + __ldg(p.csr_eid + e));
                    const float dx = __ldg(p.x + s * p.ldx + 0) - __ldg(p.x + d * p.ldx + 0);
                    const float dy = __ldg(p.x + s * p.ldx + 1) - __ldg(p.x + d * p.ldx + 1);
                    const float dz = __ldg(p.x + s * p.ldx + 2) - __ldg(p.x + d * p.ldx + 2);
                    const float r = dx * dx + dy * dy + dz * dz;
                    const float2 pv = __ldg(reinterpret_cast<const float2*>(p.PQ + (size_t)s * 128) + lane);
                    const float2 qv = __ldg(reinterpret_cast<const float2*>(p.PQ + (size_t)d * 128 + 64) + lane);
                    t.x = silu(pv.x + qv.x + wr.x * r + wa.x * a);
                    t.y = silu(pv.y + qv.y + wr.y * r + wa.y * a);
                    if (lane == 0) {
                        const float inv = 1.0f / (sqrtf(r) + 1e-30f);
                        e_src[j] = s; e_dst[j] = d;
                        e_dx[j] = dx; e_dx[IS_TM + j] = dy; e_dx[2 * IS_TM + j] = dz;
                        e_r[j] = r; e_a[j] = a; e_inv[j] = inv;
                        float v0 = 0.f, v1 = 0.f, v2 = 0.f;
                        if (HAS_COORD) {
                            const int deg = __ldg(p.indptr + d + 1) - __ldg(p.indptr + d);
                            const float sc = 1.0f / (float)max(deg, 1);
                            v0 = __ldg(gx_out + (size_t)d * 3 + 0) * sc;
                            v1 = __ldg(gx_out + (size_t)d * 3 + 1) * sc;
                            v2 = __ldg(gx_out + (size_t)d * 3 + 2) * sc;
                        }
                        e_v[j] = v0; e_v[IS_TM + j] = v1; e_v[2 * IS_TM + j] = v2;
                        e_gc[j] = (v0 * dx + v1 * dy + v2 * dz) * inv;      // dL/dc = v . dhat
                    }
                } else if (lane == 0) {
                    e_src[j] = 0; e_dst[j] = 0;
                    e_dx[j] = 0.f; e_dx[IS_TM + j] = 0.f; e_dx[2 * IS_TM + j] = 0.f;
                    e_r[j] = 0.f; e_a[j] = 0.f; e_inv[j] = 0.f; e_gc[j] = 0.f;
                    e_v[j] = 0.f; e_v[IS_TM + j] = 0.f; e_v[2 * IS_TM + j] = 0.f;
                }
                *reinterpret_cast<float2*>(A1 + j * IS_LD + 2 * lane) = t;
            }
        }
        __syncthreads();

        // ---- recompute m = silu(z2), keep silu'(z2) in registers --------------------------------
        float acc[8][4], d2[8][4];
        zero_acc(acc);
        gemm_128x64(acc, A1, IS_LD, W2t, 64, ty, tx);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float y[4];
            silu_both(acc[i][0] + vb2.x, y[0], d2[i][0]);
            silu_both(acc[i][1] + vb2.y, y[1], d2[i][1]);
            silu_both(acc[i][2] + vb2.z, y[2], d2[i][2]);
            silu_both(acc[i][3] + vb2.w, y[3], d2[i][3]);
            *reinterpret_cast<float4*>(A2 + (ty + 16 * i) * IS_LD + 4 * tx) = make_float4(y[0], y[1], y[2], y[3]);
        }
        __syncthreads();

        if (HAS_COORD) {
            // ---- coord branch: z3, c, gz3 = gc * w4 * silu'(z3) ---------------------------------
            zero_acc(acc);
            gemm_128x64(acc, A2, IS_LD, W3t, 64, ty, tx);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int row = ty + 16 * i;
                const float gc = e_gc[row];
                float u[4], d3[4];
                silu_both(acc[i][0] + vb3.x, u[0], d3[0]);
                silu_both(acc[i][1] + vb3.y, u[1], d3[1]);
                silu_both(acc[i][2] + vb3.z, u[2], d3[2]);
                silu_both(acc[i][3] + vb3.w, u[3], d3[3]);
                float c = half_warp_sum(vw4.x * u[0] + vw4.y * u[1] + vw4.z * u[2] + vw4.w * u[3]);
                if (tx == 0) e_c[row] = c;
                const float4 g = make_float4(gc * vw4.x * d3[0], gc * vw4.y * d3[1], gc * vw4.z * d3[2], gc * vw4.w * d3[3]);
                *reinterpret_cast<float4*>(G + row * IS_LD + 4 * tx) = g;
                gw4[0] += gc * u[0]; gw4[1] += gc * u[1]; gw4[2] += gc * u[2]; gw4[3] += gc * u[3];
                gb3[0] += g.x; gb3[1] += g.y; gb3[2] += g.z; gb3[3] += g.w;
            }
            __syncthreads();
            wgrad_64x64(w3, G, IS_LD, A2, IS_LD, tid);           // gW3 += gz3^T m
            zero_acc(acc);
            gemm_128x64(acc, G, IS_LD, W3r, 64, ty, tx);         // gm (coord part) = gz3 W3
            __syncthreads();                                      // everyone done reading G
        } else {
            zero_acc(acc);
        }
        // ---- gm += ghn[dst] ; gz2 = gm * silu'(z2) -> G -----------------------------------------
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int row = ty + 16 * i;
            float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
            if (row < ne) {
                const float4 gh = __ldg(reinterpret_cast<const float4*>(ghn + (size_t)e_dst[row] * 64) + tx);
                g = make_float4((acc[i][0] + gh.x) * d2[i][0], (acc[i][1] + gh.y) * d2[i][1],
                                (acc[i][2] + gh.z) * d2[i][2], (acc[i][3] + gh.w) * d2[i][3]);
            }
            *reinterpret_cast<float4*>(G + row * IS_LD + 4 * tx) = g;
            gb2[0] += g.x; gb2[1] += g.y; gb2[2] += g.z; gb2[3] += g.w;
        }
        __syncthreads();
        wgrad_64x64(w2, G, IS_LD, A1, IS_LD, tid);               // gW2 += gz2^T t1
        zero_acc(acc);
        gemm_128x64(acc, G, IS_LD, W2r, 64, ty, tx);             // gt1 = gz2 W2
        // ---- gz1 = gt1 * silu'(z1)  (z1 re-gathered in the accumulator mapping) ------------------
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int row = ty + 16 * i;
            float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
            if (row < ne) {
                const float r = e_r[row], a = e_a[row];
                const float4 pv = __ldg(reinterpret_cast<const float4*>(p.PQ + (size_t)e_src[row] * 128) + tx);
                const float4 qv = __ldg(reinterpret_cast<const float4*>(p.PQ + (size_t)e_dst[row] * 128 + 64) + tx);
                g.x = acc[i][0] * dsilu(pv.x + qv.x + vwr.x * r + vwa.x * a);
                g.y = acc[i][1] * dsilu(pv.y + qv.y + vwr.y * r + vwa.y * a);
                g.z = acc[i][2] * dsilu(pv.z + qv.z + vwr.z * r + vwa.z * a);
                g.w = acc[i][3] * dsilu(pv.w + qv.w + vwr.w * r + vwa.w * a);
                *reinterpret_cast<float4*>(gz1 + (size_t)(p0 + row) * 64 + 4 * tx) = g;
                gwr[0] += g.x * r; gwr[1] += g.y * r; gwr[2] += g.z * r; gwr[3] += g.w * r;
                gwa[0] += g.x * a; gwa[1] += g.y * a; gwa[2] += g.z * a; gwa[3] += g.w * a;
            }
            // A2 (m) is no longer needed by anyone: the last reader was wgrad(w3)/gemm(W3t), both
            // behind a barrier.  Reuse it for gz1 so the destination-side sum stays on chip.
            *reinterpret_cast<float4*>(A2 + row * IS_LD + 4 * tx) = g;
            const float gr = half_warp_sum(vwr.x * g.x + vwr.y * g.y + vwr.z * g.z + vwr.w * g.w);
            if (tx == 0) e_gr[row] = gr;
        }
        __syncthreads();

        // ---- geometry backward: one thread per edge ---------------------------------------------
        if (tid < IS_TM) {
            const int j = tid;
            float g0 = 0.f, g1 = 0.f, g2 = 0.f;
            if (j < ne) {
                const float dx = e_dx[j], dy = e_dx[IS_TM + j], dz = e_dx[2 * IS_TM + j];
                const float two_gr = 2.0f * e_gr[j];
                g0 = two_gr * dx; g1 = two_gr * dy; g2 = two_gr * dz;
                if (HAS_COORD) {
                    // dhat = diff * inv, inv = 1/(rho + eps), rho = sqrt(r):
                    // g_diff = g_dhat*inv - (g_dhat . diff) * inv^2 * diff / rho
                    const float c = e_c[j], inv = e_inv[j];
                    const float h0 = c * e_v[j], h1 = c * e_v[IS_TM + j], h2 = c * e_v[2 * IS_TM + j];
                    const float rho = sqrtf(e_r[j]);
                    const float k = (h0 * dx + h1 * dy + h2 * dz) * inv * inv / rho;
                    g0 += h0 * inv - k * dx; g1 += h1 * inv - k * dy; g2 += h2 * inv - k * dz;
                }
                gD[(size_t)(p0 + j) * 3 + 0] = g0;
                gD[(size_t)(p0 + j) * 3 + 1] = g1;
                gD[(size_t)(p0 + j) * 3 + 2] = g2;
            }
            e_gd[j] = g0; e_gd[IS_TM + j] = g1; e_gd[2 * IS_TM + j] = g2;
        }
        __syncthreads();

        // ---- destination-side sums: gQ[d] = sum gz1 ; gxd[d] = -sum g_diff -----------------------
        for (int node = n0 + warp; node < n1; node += IS_THREADS / 32) {
            const int jb = __ldg(p.indptr + node) - p0, je = __ldg(p.indptr + node + 1) - p0;
            float2 s = make_float2(0.0f, 0.0f);
            for (int j = jb; j < je; ++j) {
                const float2 v = *reinterpret_cast<const float2*>(A2 + j * IS_LD + 2 * lane);
                s.x += v.x; s.y += v.y;
            }
            *reinterpret_cast<float2*>(gQ + (size_t)node * 64 + 2 * lane) = s;
            if (lane < 3) {
                float sx = 0.0f;
                for (int j = jb; j < je; ++j) sx += e_gd[lane * IS_TM + j];
                gxd[(size_t)node * 3 + lane] = -sx;
            }
        }
        n0 = n1;
        __syncthreads();
    }

    // ---- per-CTA partials -------------------------------------------------------------------------
    float* P = partials + (size_t)blockIdx.x * IS_EDGE_BWD_PARTIAL;
    store_w(P, 64, 0, w2, tid);
    store_w(P + 4096, 64, 0, w3, tid);
    float* scratch = A1;                       // 5 * 1024 floats <= 128*68
    __syncthreads();
    cta_colsum_store(scratch + 0 * 1024, gb2, ty, tx);
    cta_colsum_store(scratch + 1 * 1024, gb3, ty, tx);
    cta_colsum_store(scratch + 2 * 1024, gw4, ty, tx);
    cta_colsum_store(scratch + 3 * 1024, gwr, ty, tx);
    cta_colsum_store(scratch + 4 * 1024, gwa, ty, tx);
    __syncthreads();
    for (int idx = tid; idx < 5 * 64; idx += IS_THREADS)
        P[8192 + idx] = cta_colsum_read(scratch + (idx >> 6) * 1024, idx & 63);
}

// =============================================================================================
// node_pre backward:  gP[s] = sum over out-edges of gz1 (CSC gather);
//   gh = gh_direct + gP Ws + gQ Wd ;  gx = gx_out + gxd + sum over out-edges of gD
//   partial block per CTA: [gWs 64*F][gWd 64*F][gb1 64]
// =============================================================================================
__global__ void __launch_bounds__(IS_THREADS)
node_pre_bwd_kernel(const float* __restrict__ gz1, const float* __restrict__ gQ, const float* __restrict__ gD,
                    const float* __restrict__ gxd, const float* __restrict__ gx_out /* or null */,
                    const float* __restrict__ gh_direct /* [M,F] or null */,
                    const int* __restrict__ outptr, const int* __restrict__ csc_pos,
                    const float* __restrict__ h, int64_t ldh, int F, const float* __restrict__ W1,
                    float* __restrict__ gh /* [M,F] or null */, float* __restrict__ gx /* [M,3] or null */,
                    float* __restrict__ partials, int64_t M) {
    extern __shared__ __align__(16) float smem[];
    const int lda = F + 4;
    float* GP = smem;                      // [128][68]
    float* GQ = GP + IS_TM * IS_LD;        // [128][68]
    float* A = GQ + IS_TM * IS_LD;         // [128][F+4]   (followed by WB so that wide reads stay in bounds)
    float* WB = A + IS_TM * lda;           // [2][64][64]
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15, warp = tid >> 5, lane = tid & 31;
    const int ldw = 2 * F + 2;
    float ws[4][4], wd[4][4];
    zero_w(ws); zero_w(wd);
    float gb1[4] = {0, 0, 0, 0};
    if (gh) {
        load_w_rowmajor(WB, W1, ldw, 0, F, tid);
        load_w_rowmajor(WB + 4096, W1, ldw, F, F, tid);
    }
    const int64_t ntiles = (M + IS_TM - 1) / IS_TM;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int64_t m0 = t * IS_TM;
        __syncthreads();
        // source-side reduction through the CSC transpose: one warp per node, sixteen nodes per warp.  The loads are
        // batched (the dependent chain outptr -> csc_pos -> gz1 row used to be walked edge by edge: ~20 serial L2
        // round trips per node, 75 % of this kernel's time): lane i preloads the CSC range of the warp's i-th node,
        // the positions of up to 32 out-edges are loaded with one coalesced access and broadcast by shuffle, eight
        // gz1 rows are in flight per lane.  Summation order is unchanged (ascending CSC position): bit-identical.
        {
            constexpr int NPW = IS_TM / (IS_THREADS / 32);                 // nodes per warp (16)
            int my_qb = 0, my_qe = 0;
            if (lane < NPW) {
                const int64_t n = m0 + warp + (IS_THREADS / 32) * lane;
                if (n < M) { my_qb = __ldg(outptr + n); my_qe = __ldg(outptr + n + 1); }
            }
            for (int i = 0; i < NPW; ++i) {
                const int r = warp + (IS_THREADS / 32) * i;
                const int64_t n = m0 + r;
                const int qb = __shfl_sync(0xffffffffu, my_qb, i), qe = __shfl_sync(0xffffffffu, my_qe, i);
                float2 s = make_float2(0.f, 0.f);
                float sx = 0.0f;
                const bool want_x = gx != nullptr && lane < 3 && n < M;
                if (want_x) {
                    sx = __ldg(gxd + n * 3 + lane);
                    if (gx_out) sx += __ldg(gx_out + n * 3 + lane);
                }
                for (int q0 = qb; q0 < qe; q0 += 32) {
                    const int cnt = min(32, qe - q0);
                    const int my_pos = lane < cnt ? __ldg(csc_pos + q0 + lane) : 0;
                    for (int j0 = 0; j0 < cnt; j0 += 8) {
                        float2 v[8];
                        float d[8];
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            const int pos = __shfl_sync(0xffffffffu, my_pos, (j0 + u) & 31);
                            const bool ok = j0 + u < cnt;
                            v[u] = ok ? __ldg(reinterpret_cast<const float2*>(gz1 + (size_t)pos * 64) + lane) : make_float2(0.f, 0.f);
                            d[u] = (ok && want_x) ? __ldg(gD + (size_t)pos * 3 + lane) : 0.0f;
                        }
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            if (j0 + u < cnt) { s.x += v[u].x; s.y += v[u].y; sx += d[u]; }
                        }
                    }
                }
                if (want_x) gx[n * 3 + lane] = sx;
                *reinterpret_cast<float2*>(GP + r * IS_LD + 2 * lane) = s;
            }
        }
        load_rows(GQ, IS_LD, gQ, 64, m0, M, 64, tid);
        load_rows(A, lda, h, ldh, m0, M, F, tid);
        __syncthreads();
        wgrad_64x64(ws, GP, IS_LD, A, lda, tid);
        wgrad_64x64(wd, GQ, IS_LD, A, lda, tid);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float4 g = *reinterpret_cast<const float4*>(GQ + (ty + 16 * i) * IS_LD + 4 * tx);
            gb1[0] += g.x; gb1[1] += g.y; gb1[2] += g.z; gb1[3] += g.w;
        }
        if (gh) {
            float acc[8][4];
            zero_acc(acc);
            gemm_128x64(acc, GP, IS_LD, WB, 64, ty, tx);
            gemm_128x64(acc, GQ, IS_LD, WB + 4096, 64, ty, tx);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                int64_t m = m0 + ty + 16 * i;
                if (m < M && 4 * tx < F) {                 // [M, F] rows (F = 20: Ws / Wd zero-padded beyond column F)
                    const size_t off = (size_t)m * F + 4 * tx;
                    float4 o = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
                    if (gh_direct) {
                        const float4 g = __ldg(reinterpret_cast<const float4*>(gh_direct + off));
                        o.x += g.x; o.y += g.y; o.z += g.z; o.w += g.w;
                    }
                    *reinterpret_cast<float4*>(gh + off) = o;
                }
            }
        }
    }
    float* P = partials + (size_t)blockIdx.x * (2 * 64 * F + 64);
    store_w(P, F, 0, ws, tid);
    store_w(P + 64 * F, F, 0, wd, tid);
    __syncthreads();
    cta_colsum_store(GP, gb1, ty, tx);
    __syncthreads();
    if (tid < 64) P[2 * 64 * F + tid] = cta_colsum_read(GP, tid);
}

// out[i] = sum_b partials[b * stride + i] in ascending b (deterministic)
__global__ void reduce_partials_kernel(const float* __restrict__ partials, int nparts, int64_t stride,
                                       float* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= stride) return;
    float s = 0.0f;
#pragma unroll 8
    for (int b = 0; b < nparts; ++b) s += partials[(size_t)b * stride + i];
    out[i] = s;
}

// the three partial buffers of one EGNN layer's backward (node_post, edge, node_pre) in ONE launch: blockIdx.y = set
struct Partials3 {
    const float* partials[3];
    float* out[3];
    int nparts[3];
    int64_t stride[3];
};
__global__ void reduce_partials3_kernel(Partials3 a) {
    const int k = blockIdx.y;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = a.stride[k];
    if (i >= stride) return;
    const float* __restrict__ p = a.partials[k];
    const int n = a.nparts[k];
    float s = 0.0f;
#pragma unroll 8
    for (int b = 0; b < n; ++b) s += p[(size_t)b * stride + i];        // ascending CTA order: deterministic
    a.out[k][i] = s;
}

}  // namespace is

// =================================================================================================
// C ABI
// =================================================================================================
using namespace is;

static int num_sms() { return current_num_sms(); }

template <typename K>
static int set_smem(K kernel, size_t bytes) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    return e == cudaSuccess ? 0 : (int)e;
}

static inline int node_grid(int64_t M) {
    int64_t tiles = (M + IS_TM - 1) / IS_TM;
    int64_t g = tiles < num_sms() ? tiles : num_sms();
    return (int)(g < 1 ? 1 : g);
}
static inline int edge_grid(int64_t n_nodes, int ctas_per_sm) {
    int64_t g = (n_nodes + 31) / 32;
    int64_t cap = (int64_t)num_sms() * ctas_per_sm;
    if (g > cap) g = cap;
    return (int)(g < 1 ? 1 : g);
}

extern "C" {

int is_num_sms(void) { return num_sms(); }

// number of per-CTA partial blocks each backward kernel writes for a problem of this size
int is_egnn_node_grid(int64_t n_nodes) { return node_grid(n_nodes); }
int is_egnn_edge_bwd_grid(int64_t n_nodes) { return edge_grid(n_nodes, 1); }

int is_egnn_node_pre_fwd(const float* h, int64_t ldh, int F, const float* W1, const float* b1, float* PQ,
                         int64_t n_nodes, void* stream) {
    if (!(F == 20 || F == 64) || n_nodes <= 0) return IS_ERR_ARG;
    size_t smem = sizeof(float) * (IS_TM * (F + 4) + 2 * F * 64);
    int rc = set_smem(node_pre_fwd_kernel, smem);
    if (rc) return rc;
    // a streaming kernel (20- or 64-wide rows in, 128-wide rows out, no per-CTA partials): four CTAs per SM hide the
    // load -> barrier -> store chain of a tile that one CTA per SM (node_grid) leaves exposed
    const int64_t tiles = (n_nodes + IS_TM - 1) / IS_TM, cap = 4 * (int64_t)num_sms();
    const int grid = (int)(tiles < cap ? tiles : cap);
    node_pre_fwd_kernel<<<grid < 1 ? 1 : grid, IS_THREADS, smem, (cudaStream_t)stream>>>(h, ldh, F, W1, b1, PQ, n_nodes);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

static EdgeCommon make_common(const int* indptr, const int* csr_src, const int* csr_dst, const int* csr_eid,
                              const float* PQ, const float* x, int64_t ldx, const float* edge_attr,
                              const float* W1, int F, const float* W2, const float* b2, const float* W3,
                              const float* b3, const float* w4, int64_t n_nodes, int* status) {
    EdgeCommon c;
    c.indptr = indptr; c.csr_src = csr_src; c.csr_dst = csr_dst; c.csr_eid = csr_eid;
    c.PQ = PQ; c.x = x; c.ldx = ldx; c.edge_attr = edge_attr; c.W1 = W1; c.F = F;
    c.W2 = W2; c.b2 = b2; c.W3 = W3; c.b3 = b3; c.w4 = w4; c.n_nodes = (int)n_nodes; c.status = status;
    return c;
}

int is_egnn_edge_fwd(const int* indptr, const int* csr_src, const int* csr_dst, const int* csr_eid,
                     const float* PQ, const float* x, int64_t ldx, const float* edge_attr,
                     const float* W1, int F, const float* W2, const float* b2,
                     const float* W3, const float* b3, const float* w4, int update_coords,
                     float* hn, float* x_out, int64_t n_nodes, int* status, void* stream) {
    if (!(F == 20 || F == 64) || n_nodes <= 0 || n_nodes > 0x7fffffff) return IS_ERR_ARG;
    EdgeCommon c = make_common(indptr, csr_src, csr_dst, csr_eid, PQ, x, ldx, edge_attr, W1, F, W2, b2, W3, b3, w4, n_nodes, status);
    size_t smem = sizeof(float) * (2 * 4096 + 5 * 64 + 2 * IS_TM * IS_LD + IS_TM + 3 * IS_TM);
    int grid = edge_grid(n_nodes, 2);
    if (update_coords) {
        int rc = set_smem(edge_fwd_kernel<true>, smem);
        if (rc) return rc;
        edge_fwd_kernel<true><<<grid, IS_THREADS, smem, (cudaStream_t)stream>>>(c, hn, x_out);
    } else {
        int rc = set_smem(edge_fwd_kernel<false>, smem);
        if (rc) return rc;
        edge_fwd_kernel<false><<<grid, IS_THREADS, smem, (cudaStream_t)stream>>>(c, hn, x_out);
    }
    IS_LAUNCH_CHECK();
    return IS_OK;
}

int is_egnn_node_post_fwd(const float* h, int64_t ldh, int F, const float* hn, const float* W5, const float* b5,
                          const float* W6, const float* b6, float* h_out, int64_t n_nodes, void* stream) {
    if (!(F == 20 || F == 64) || n_nodes <= 0) return IS_ERR_ARG;
    int K = F + 64;
    size_t smem = sizeof(float) * (IS_TM * (K + 4) + IS_TM * IS_LD + K * 64 + 4096);
    int rc = set_smem(node_post_fwd_kernel, smem);
    if (rc) return rc;
    node_post_fwd_kernel<<<node_grid(n_nodes), IS_THREADS, smem, (cudaStream_t)stream>>>(h, ldh, F, hn, W5, b5, W6, b6, h_out, n_nodes);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

// partials: [is_egnn_node_grid(n_nodes)][64*(F+64) + 64 + 4096 + 64] floats
int is_egnn_node_post_bwd(const float* gh_out, const float* h, int64_t ldh, int F, const float* hn,
                          const float* W5, const float* b5, const float* W6,
                          float* gh_direct, float* ghn, float* partials, int64_t n_nodes, void* stream) {
    if (!(F == 20 || F == 64) || n_nodes <= 0) return IS_ERR_ARG;
    if ((reinterpret_cast<uintptr_t>(gh_direct) & 15) != 0) return IS_ERR_ARG;          // 128-bit stores
    int K = F + 64;
    size_t smem = sizeof(float) * (IS_TM * (K + 4) + 2 * IS_TM * IS_LD + IS_TM * 64);
    int rc = set_smem(node_post_bwd_kernel, smem);
    if (rc) return rc;
    node_post_bwd_kernel<<<node_grid(n_nodes), IS_THREADS, smem, (cudaStream_t)stream>>>(
        gh_out, h, ldh, F, hn, W5, b5, W6, gh_direct, ghn, partials, n_nodes);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

// partials: [is_egnn_edge_bwd_grid(n_nodes)][4096 + 4096 + 5*64] floats; gx_out == NULL means the layer's
// coordinate output is unused (no gradient reaches coord_mlp).
int is_egnn_edge_bwd(const int* indptr, const int* csr_src, const int* csr_dst, const int* csr_eid,
                     const float* PQ, const float* x, int64_t ldx, const float* edge_attr,
                     const float* W1, int F, const float* W2, const float* b2,
                     const float* W3, const float* b3, const float* w4,
                     const float* ghn, const float* gx_out,
                     float* gz1, float* gQ, float* gD, float* gxd, float* partials,
                     int64_t n_nodes, int* status, void* stream) {
    if (!(F == 20 || F == 64) || n_nodes <= 0 || n_nodes > 0x7fffffff) return IS_ERR_ARG;
    EdgeCommon c = make_common(indptr, csr_src, csr_dst, csr_eid, PQ, x, ldx, edge_attr, W1, F, W2, b2, W3, b3, w4, n_nodes, status);
    size_t smem = sizeof(float) * (4 * 4096 + 5 * 64 + 3 * IS_TM * IS_LD + 17 * IS_TM);
    int grid = edge_grid(n_nodes, 1);
    if (gx_out) {
        int rc = set_smem(edge_bwd_kernel<true>, smem);
        if (rc) return rc;
        edge_bwd_kernel<true><<<grid, IS_THREADS, smem, (cudaStream_t)stream>>>(c, ghn, gx_out, gz1, gQ, gD, gxd, partials);
    } else {
        int rc = set_smem(edge_bwd_kernel<false>, smem);
        if (rc) return rc;
        edge_bwd_kernel<false><<<grid, IS_THREADS, smem, (cudaStream_t)stream>>>(c, ghn, gx_out, gz1, gQ, gD, gxd, partials);
    }
    IS_LAUNCH_CHECK();
    return IS_OK;
}

// partials: [is_egnn_node_grid(n_nodes)][2*64*F + 64] floats
int is_egnn_node_pre_bwd(const float* gz1, const float* gQ, const float* gD, const float* gxd,
                         const float* gx_out, const float* gh_direct,
                         const int* outptr, const int* csc_pos, const float* h, int64_t ldh, int F,
                         const float* W1, float* gh, float* gx, float* partials, int64_t n_nodes, void* stream) {
    if (!(F == 20 || F == 64) || n_nodes <= 0) return IS_ERR_ARG;
    if (((reinterpret_cast<uintptr_t>(gh) | reinterpret_cast<uintptr_t>(gh_direct)) & 15) != 0) return IS_ERR_ARG;   // 128-bit accesses
    size_t smem = sizeof(float) * (2 * IS_TM * IS_LD + IS_TM * (F + 4) + 2 * 4096);
    int rc = set_smem(node_pre_bwd_kernel, smem);
    if (rc) return rc;
    node_pre_bwd_kernel<<<node_grid(n_nodes), IS_THREADS, smem, (cudaStream_t)stream>>>(
        gz1, gQ, gD, gxd, gx_out, gh_direct, outptr, csc_pos, h, ldh, F, W1, gh, gx, partials, n_nodes);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

int is_reduce_partials3(const float* p0, int n0, int64_t s0, float* o0, const float* p1, int n1, int64_t s1, float* o1,
                        const float* p2, int n2, int64_t s2, float* o2, void* stream) {
    if (n0 <= 0 || n1 <= 0 || n2 <= 0 || s0 <= 0 || s1 <= 0 || s2 <= 0) return IS_ERR_ARG;
    Partials3 a;
    a.partials[0] = p0; a.partials[1] = p1; a.partials[2] = p2;
    a.out[0] = o0; a.out[1] = o1; a.out[2] = o2;
    a.nparts[0] = n0; a.nparts[1] = n1; a.nparts[2] = n2;
    a.stride[0] = s0; a.stride[1] = s1; a.stride[2] = s2;
    int64_t smax = s0 > s1 ? s0 : s1;
    if (s2 > smax) smax = s2;
    dim3 grid((unsigned)((smax + 255) / 256), 3);
    reduce_partials3_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(a);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

int is_reduce_partials(const float* partials, int nparts, int64_t stride, float* out, void* stream) {
    if (nparts <= 0 || stride <= 0) return IS_ERR_ARG;
    int threads = 256;
    int64_t blocks = (stride + threads - 1) / threads;
    reduce_partials_kernel<<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(partials, nparts, stride, out);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

}  // extern "C"
