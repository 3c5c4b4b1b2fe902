// EGNN edge forward on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a.
//
// Same contract as is::edge_fwd_kernel (egnn.cu): per tile of <= 128 in-edges (node-aligned, CSR
// order)   t1 = silu(P[src] + Q[dst] + w_r r + w_a a)  ->  m = silu(t1 W2^T + b2)  ->
// c = w4 . silu(m W3^T + b3)  ->  warp per destination node:  hn = sum m,  x' = x + mean(c dhat).
// The two 128x64x64 per-tile GEMMs run as tcgen05.mma (M = 128, N = 64) with the accumulators in
// TMEM; everything else (gather, SiLU, aggregation) stays on the SIMT pipes of the same CTA:
//
//   gather (all warps)  -> A operand tile in smem (canonical K-major layout, umma.cuh)
//   MMA 1 (one thread)  -> TMEM cols [0,64)      -> epilogue 1 (all warps: tcgen05.ld, +b2, SiLU)
//                                                   writes m as the next A operand and as fp32 rows
//   MMA 2 (one thread)  -> TMEM cols [64,128)    -> meanwhile: hn aggregation from the fp32 rows
//                                                -> epilogue 2 (tcgen05.ld, +b3, SiLU, . w4)
//   coordinate aggregation (warp per destination node)
//
// Two precisions (template PREC):
//   PREC_BF16   : bf16 operands, fp32 accumulate, fast SiLU        (bf16 mode, tolerance 1e-2)
//   PREC_TF32X3 : 3xTF32 split  a = hi + lo, D = lo*Bhi + hi*Blo + hi*Bhi, accurate SiLU
//                 (fp32 parity: the self-test measures 2.6e-7 relative error for the GEMM)
// Two CTAs per SM share the tensor core: while one waits on its MMA mbarrier the other runs its
// SIMT phases.
#include "common.cuh"
#include "egnn_common.cuh"

#include "egnn_node_tc.cuh"

namespace is {

struct TileMeta {            // per-edge scalars of one tile, produced by the prefetch warps
    int src[IS_TM];
    int dst[IS_TM];
    float r[IS_TM];
    float a[IS_TM];
    float dh[IS_TM * 3];
};

__device__ __forceinline__ void load_meta(const EdgeCommon& p, TileMeta& m, int j, int p0, int ne) {
    if (j < ne) {
        const int e = p0 + j;
        const int s = __ldg(p.csr_src + e), d = __ldg(p.csr_dst + e);
        const float a = __ldg(p.edge_attr + __ldg(p.csr_eid + e));
        const float dx = __ldg(p.x + s * p.ldx + 0) - __ldg(p.x + d * p.ldx + 0);
        const float dy = __ldg(p.x + s * p.ldx + 1) - __ldg(p.x + d * p.ldx + 1);
        const float dz = __ldg(p.x + s * p.ldx + 2) - __ldg(p.x + d * p.ldx + 2);
        const float r = dx * dx + dy * dy + dz * dz;
        const float inv = 1.0f / (sqrtf(r) + 1e-30f);
        m.src[j] = s; m.dst[j] = d; m.r[j] = r; m.a[j] = a;
        m.dh[j * 3 + 0] = dx * inv; m.dh[j * 3 + 1] = dy * inv; m.dh[j * 3 + 2] = dz * inv;
    }
}

// NT threads per CTA: 256 (two CTAs per SM) for bf16, 512 (one CTA per SM, 16 warps) for 3xTF32 whose
// hi/lo operand tiles need 147 KB of shared memory.
template <int PREC, bool HAS_COORD, int NT, bool FAST>
__global__ void __launch_bounds__(NT, NT == 256 ? (PREC == PREC_BF16 ? 3 : 2) : 1)
edge_fwd_tc_kernel(EdgeCommon p, float* __restrict__ hn, float* __restrict__ x_out) {
    using C = TcCfg<PREC>;
    constexpr int NW = NT / 32;                 // warps
    constexpr int CQ = NW / 4;                  // column splits of the epilogue (TMEM lane quarter x column block)
    constexpr int CW = 64 / CQ;                 // accumulator columns per thread
    extern __shared__ __align__(128) uint8_t smem_raw[];
    uint8_t* sA = smem_raw;                                            // [NSPLIT][A_BYTES] t1, then m
    uint8_t* sW2 = sA + C::NSPLIT * C::A_BYTES;                        // [NSPLIT][W_BYTES]
    uint8_t* sW3 = sW2 + C::NSPLIT * C::W_BYTES;
    // fp32 copy of m for the hn aggregation: only the tf32 variant needs it; the bf16 variants
    // re-read the (split) bf16 operand tile, which is bank-conflict free thanks to the 144-byte LBO
    constexpr bool USE_M32 = PREC == PREC_TF32X3;
    float* M32 = reinterpret_cast<float*>(sW3 + C::NSPLIT * C::W_BYTES);   // [128][68] fp32 m
    float* vec = M32 + (USE_M32 ? IS_TM * IS_LD : 0);                  // b2, b3, w4, wr, wa
    float* e_c = vec + 5 * 64;                                         // [CQ][128] partial c per column block
    TileMeta* meta = reinterpret_cast<TileMeta*>(e_c + CQ * IS_TM);    // [2]
    __shared__ int s_tile[2][4];
    __shared__ __align__(8) uint64_t mbar[2];
    __shared__ uint32_t s_tmem;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ldw1 = 2 * p.F + 2;
    if (warp == 0) tmem_alloc(&s_tmem, 128);
    if (tid == 32) { mbar_init(&mbar[0], 1); mbar_init(&mbar[1], 1); }
    for (int idx = tid; idx < 64 * 64; idx += NT) {                    // stage W2 / W3 as B operands
        const int n = idx >> 6, k = idx & 63;
        store_weight1<PREC>(sW2, C::W_BYTES, n, k, __ldg(p.W2 + idx));
        store_weight1<PREC>(sW3, C::W_BYTES, n, k, HAS_COORD ? __ldg(p.W3 + idx) : 0.0f);
    }
    if (tid < 64) {
        vec[tid] = p.b2[tid];
        vec[64 + tid] = HAS_COORD ? p.b3[tid] : 0.0f;
        vec[128 + tid] = HAS_COORD ? p.w4[tid] : 0.0f;
        vec[192 + tid] = p.W1[tid * ldw1 + 2 * p.F];
        vec[256 + tid] = p.W1[tid * ldw1 + 2 * p.F + 1];
    }
    const int chunk = (p.n_nodes + gridDim.x - 1) / gridDim.x;
    const int nbeg = blockIdx.x * chunk;
    const int nend = min(p.n_nodes, nbeg + chunk);
    // prologue: first tile + its per-edge scalars (the last four warps are the prefetch warps)
    if (warp >= NW - 4) {
        int tn0, tn1, tp0, tne;
        next_tile(p.indptr, nbeg, nend, p.status, lane, tn0, tn1, tp0, tne);
        if (warp == NW - 4 && lane == 0) { s_tile[0][0] = tn0; s_tile[0][1] = tn1; s_tile[0][2] = tp0; s_tile[0][3] = tne; }
        load_meta(p, meta[0], (warp - (NW - 4)) * 32 + lane, tp0, tne);
    }
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = s_tmem;
    const uint32_t a_addr = smem_u32(sA), w2_addr = smem_u32(sW2), w3_addr = smem_u32(sW3);
    // epilogue mapping: TMEM lane quarter q = warp % 4 (rows 32q + lane), column block cq = warp / 4
    const int q = warp & 3, cq = warp >> 2, erow = 32 * q + lane;
    const uint32_t t_lane = tmem + ((uint32_t)(32 * q) << 16) + CW * cq;
    // gather mapping: 4 edges per warp per pass, 8 lanes per edge, 8 features per lane
    const int esub = lane >> 3, kc8 = lane & 7;
    const float4 wr0 = *reinterpret_cast<const float4*>(vec + 192 + 8 * kc8), wr1 = *reinterpret_cast<const float4*>(vec + 196 + 8 * kc8);
    const float4 wa0 = *reinterpret_cast<const float4*>(vec + 256 + 8 * kc8), wa1 = *reinterpret_cast<const float4*>(vec + 260 + 8 * kc8);
    uint32_t phase = 0;
    int cur = 0;

    while (true) {
        const int n0 = s_tile[cur][0], n1 = s_tile[cur][1], p0 = s_tile[cur][2], ne = s_tile[cur][3];
        if (n0 >= nend) break;
        const TileMeta& mt = meta[cur];

        // ---- gather -> A operand (t1): all row loads of a batch of passes are issued before any use --
        {
            constexpr int NPASS = IS_TM / (4 * NW);            // 4 (256 threads) or 2 (512 threads)
            constexpr int PB = NPASS < 2 ? NPASS : 2;          // passes per load batch (32 registers of rows)
#pragma unroll
            for (int pb = 0; pb < NPASS; pb += PB) {
                float4 pv[PB][2], qv[PB][2];
                float rr[PB], aa[PB];
#pragma unroll
                for (int u = 0; u < PB; ++u) {
                    const int j = (pb + u) * 4 * NW + warp * 4 + esub;
                    const bool valid = j < ne;
                    const int s = valid ? mt.src[j] : 0, d = valid ? mt.dst[j] : 0;
                    rr[u] = valid ? mt.r[j] : 0.0f;
                    aa[u] = valid ? mt.a[j] : 0.0f;
                    const float4* pp = reinterpret_cast<const float4*>(p.PQ + (size_t)s * 128 + 8 * kc8);
                    const float4* qp = reinterpret_cast<const float4*>(p.PQ + (size_t)d * 128 + 64 + 8 * kc8);
                    pv[u][0] = __ldg(pp); pv[u][1] = __ldg(pp + 1); qv[u][0] = __ldg(qp); qv[u][1] = __ldg(qp + 1);
                }
#pragma unroll
                for (int u = 0; u < PB; ++u) {
                    const int j = (pb + u) * 4 * NW + warp * 4 + esub;
                    const float r = rr[u], a = aa[u];
                    float v[8];
                    v[0] = act<PREC, FAST>(pv[u][0].x + qv[u][0].x + wr0.x * r + wa0.x * a);
                    v[1] = act<PREC, FAST>(pv[u][0].y + qv[u][0].y + wr0.y * r + wa0.y * a);
                    v[2] = act<PREC, FAST>(pv[u][0].z + qv[u][0].z + wr0.z * r + wa0.z * a);
                    v[3] = act<PREC, FAST>(pv[u][0].w + qv[u][0].w + wr0.w * r + wa0.w * a);
                    v[4] = act<PREC, FAST>(pv[u][1].x + qv[u][1].x + wr1.x * r + wa1.x * a);
                    v[5] = act<PREC, FAST>(pv[u][1].y + qv[u][1].y + wr1.y * r + wa1.y * a);
                    v[6] = act<PREC, FAST>(pv[u][1].z + qv[u][1].z + wr1.z * r + wa1.z * a);
                    v[7] = act<PREC, FAST>(pv[u][1].w + qv[u][1].w + wr1.w * r + wa1.w * a);
                    // rows beyond the tile's edges hold finite garbage: they are never aggregated
                    store_operand8<PREC>(sA, C::A_BYTES, j, kc8, v);
                }
            }
        }
        fence_async_smem();
        fence_before_sync();
        __syncthreads();                                                           // S1
        if (warp == 0) {              // one elected lane of the converged warp issues (bare UTCHMMA, no election loop)
            if (elect_one()) {
                fence_after_sync();
                issue_gemm<PREC>(tmem, a_addr, C::A_BYTES, w2_addr, C::W_BYTES, 64, 0);
                mma_commit(&mbar[0]);
            }
            __syncwarp();
        }
        // ---- while MMA 1 runs: walk to the next tile and prefetch its per-edge scalars ------------
        if (warp >= NW - 4) {
            int tn0, tn1, tp0, tne;
            next_tile(p.indptr, n1, nend, p.status, lane, tn0, tn1, tp0, tne);
            if (warp == NW - 4 && lane == 0) {
                s_tile[cur ^ 1][0] = tn0; s_tile[cur ^ 1][1] = tn1; s_tile[cur ^ 1][2] = tp0; s_tile[cur ^ 1][3] = tne;
            }
            load_meta(p, meta[cur ^ 1], (warp - (NW - 4)) * 32 + lane, tp0, tne);
        }
        if (tid == 0) mbar_wait(&mbar[0], phase);      // one poller; everybody else parks on the barrier
        __syncthreads();                                                           // S2
        fence_after_sync();

        // ---- epilogue 1: m = silu(acc0 + b2) -> fp32 rows (+ next A operand) ----------------------
        {
            float z[CW];
            tmem_ld<CW>(t_lane, z);
#pragma unroll
            for (int g = 0; g < CW / 8; ++g) {
                const float4 b0 = *reinterpret_cast<const float4*>(vec + CW * cq + 8 * g);
                const float4 b1 = *reinterpret_cast<const float4*>(vec + CW * cq + 8 * g + 4);
                float m8[8];
                m8[0] = act<PREC, FAST>(z[8 * g + 0] + b0.x); m8[1] = act<PREC, FAST>(z[8 * g + 1] + b0.y);
                m8[2] = act<PREC, FAST>(z[8 * g + 2] + b0.z); m8[3] = act<PREC, FAST>(z[8 * g + 3] + b0.w);
                m8[4] = act<PREC, FAST>(z[8 * g + 4] + b1.x); m8[5] = act<PREC, FAST>(z[8 * g + 5] + b1.y);
                m8[6] = act<PREC, FAST>(z[8 * g + 6] + b1.z); m8[7] = act<PREC, FAST>(z[8 * g + 7] + b1.w);
                if (USE_M32) {
                    float* dst = M32 + erow * IS_LD + CW * cq + 8 * g;
                    *reinterpret_cast<float4*>(dst) = make_float4(m8[0], m8[1], m8[2], m8[3]);
                    *reinterpret_cast<float4*>(dst + 4) = make_float4(m8[4], m8[5], m8[6], m8[7]);
                }
                if (HAS_COORD || !USE_M32) store_operand8<PREC>(sA, C::A_BYTES, erow, (CW / 8) * cq + g, m8);   // MMA 1 is done with sA
            }
        }
        fence_async_smem();
        fence_before_sync();
        __syncthreads();                                                           // S3
        if (HAS_COORD && warp == 0) {
            if (elect_one()) {
                fence_after_sync();
                issue_gemm<PREC>(tmem + 64, a_addr, C::A_BYTES, w3_addr, C::W_BYTES, 64, 0);
                mma_commit(&mbar[1]);
            }
            __syncwarp();
        }

        // ---- hn aggregation (overlaps MMA 2): one warp per destination node -----------------------
        for (int node = n0 + warp; node < n1; node += NW) {
            const int jb = __ldg(p.indptr + node) - p0, je = __ldg(p.indptr + node + 1) - p0;
            float2 s = make_float2(0.0f, 0.0f);
            for (int j = jb; j < je; ++j) {
                float2 v;
                if constexpr (USE_M32) v = *reinterpret_cast<const float2*>(M32 + j * IS_LD + 2 * lane);
                else v = load_operand2<PREC>(sA, C::A_BYTES, j, lane);
                s.x += v.x; s.y += v.y;
            }
            *reinterpret_cast<float2*>(hn + (size_t)node * 64 + 2 * lane) = s;
        }

        if (HAS_COORD) {
            // ---- epilogue 2: c = w4 . silu(acc1 + b3) (each thread: one row, CW columns) ----------
            if (tid == 0) mbar_wait(&mbar[1], phase);
            __syncthreads();                                                       // S4
            fence_after_sync();
            float z[CW];
            tmem_ld<CW>(t_lane + 64, z);
            float c = 0.0f;
#pragma unroll
            for (int g = 0; g < CW / 4; ++g) {
                const float4 b = *reinterpret_cast<const float4*>(vec + 64 + CW * cq + 4 * g);
                const float4 w = *reinterpret_cast<const float4*>(vec + 128 + CW * cq + 4 * g);
                c = fmaf(w.x, act<PREC, FAST>(z[4 * g + 0] + b.x), c);
                c = fmaf(w.y, act<PREC, FAST>(z[4 * g + 1] + b.y), c);
                c = fmaf(w.z, act<PREC, FAST>(z[4 * g + 2] + b.z), c);
                c = fmaf(w.w, act<PREC, FAST>(z[4 * g + 3] + b.w), c);
            }
            e_c[cq * IS_TM + erow] = c;
            fence_before_sync();
            __syncthreads();                                                       // S5
            for (int node = n0 + warp; node < n1; node += NW) {
                if (lane < 3) {
                    const int jb = __ldg(p.indptr + node) - p0, je = __ldg(p.indptr + node + 1) - p0;
                    float sx = 0.0f;
                    for (int j = jb; j < je; ++j) {
                        float cj = e_c[j];
#pragma unroll
                        for (int t = 1; t < CQ; ++t) cj += e_c[t * IS_TM + j];
                        sx += cj * mt.dh[j * 3 + lane];
                    }
                    const int deg = je - jb;
                    x_out[(size_t)node * 3 + lane] = __ldg(p.x + node * p.ldx + lane) + sx / (float)max(deg, 1);
                }
            }
        }
        // No barrier here when the coordinate branch ran: the next tile's gather only writes sA (both
        // MMAs of this tile have been waited for; the hn aggregation, which reads sA in the bf16
        // variants, finished before S4) and reads meta[cur ^ 1]; M32 / e_c / meta[cur] / TMEM are next
        // written after the barriers S1..S4 of the next iteration.
        if (!HAS_COORD && !USE_M32) __syncthreads();   // hn aggregation reads sA: finish before the next gather
        phase ^= 1;
        cur ^= 1;
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 128);
}

template <int PREC, int NT>
static size_t tc_smem_bytes() {
    using C = TcCfg<PREC>;
    return (size_t)C::NSPLIT * (C::A_BYTES + 2 * C::W_BYTES) +
           sizeof(float) * ((PREC == PREC_TF32X3 ? IS_TM * IS_LD : 0) + 5 * 64 + (NT / 128) * IS_TM) + 2 * sizeof(TileMeta) + 128;
}

template <int PREC, bool HAS_COORD, int NT, bool FAST>
static int launch_tc2(const EdgeCommon& c, float* hn, float* x_out, int grid, cudaStream_t st) {
    const size_t smem = tc_smem_bytes<PREC, NT>();
    cudaError_t e = cudaFuncSetAttribute(edge_fwd_tc_kernel<PREC, HAS_COORD, NT, FAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    edge_fwd_tc_kernel<PREC, HAS_COORD, NT, FAST><<<grid, NT, smem, st>>>(c, hn, x_out);
    e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

template <int PREC, bool HAS_COORD, int NT>
static int launch_tc(const EdgeCommon& c, float* hn, float* x_out, int grid, cudaStream_t st, bool fast) {
    if (PREC == PREC_BF16 || fast) return launch_tc2<PREC, HAS_COORD, NT, true>(c, hn, x_out, grid, st);
    return launch_tc2<PREC, HAS_COORD, NT, false>(c, hn, x_out, grid, st);
}

// warp-specialised asynchronous kernel (egnn_tc2.cu): bf16 / bf16x3, destination-side sums on the tensor cores
int launch_edge_fwd_ws(const EdgeCommon& c, float* hn, float* x_out, int precision, bool update_coords, bool fast,
                       cudaStream_t st);
// the same kernel with the node tail: one launch per fp16x2 inference layer
int launch_layer_fwd_fp16x2(const EdgeCommon& c, float* hn, float* x_out, bool update_coords, const NodeArgs& nd, int next_kind,
                            cudaStream_t st);

static EdgeCommon edge_common(const int* indptr, const int* csr_src, const int* csr_dst, const int* csr_eid, const float* PQ,
                              const float* x, int64_t ldx, const float* edge_attr, const float* W1, int F, const float* W2,
                              const float* b2, const float* W3, const float* b3, const float* w4, int64_t n_nodes, int* status) {
    EdgeCommon c;
    c.indptr = indptr; c.csr_src = csr_src; c.csr_dst = csr_dst; c.csr_eid = csr_eid;
    c.PQ = PQ; c.x = x; c.ldx = ldx; c.edge_attr = edge_attr; c.W1 = W1; c.F = F;
    c.W2 = W2; c.b2 = b2; c.W3 = W3; c.b3 = b3; c.w4 = w4; c.n_nodes = (int)n_nodes; c.status = status;
    return c;
}

}  // namespace is

using namespace is;

extern "C" {

// Tensor-core variant of is_egnn_edge_fwd.  precision: 0 = bf16 operands, 2 = 3xTF32, 3 = bf16x3 (both fp32-accurate).
// precision | 16 selects the lock-step first-generation kernel of this file for bf16 / bf16x3 (kept for A/B timing);
// default = the warp-specialised kernel of egnn_tc2.cu.
// fast_act: use the 5-instruction SiLU in the fp32-accurate modes (inference); 0 keeps expf (training forward).
int is_egnn_edge_fwd_tc(const int* indptr, const int* csr_src, const int* csr_dst, const int* csr_eid,
                        const float* PQ, const float* x, int64_t ldx, const float* edge_attr,
                        const float* W1, int F, const float* W2, const float* b2,
                        const float* W3, const float* b3, const float* w4, int update_coords, int precision,
                        int fast_act, float* hn, float* x_out, int64_t n_nodes, int* status, void* stream) {
    if (!(F == 20 || F == 64) || n_nodes <= 0 || n_nodes > 0x7fffffff) return IS_ERR_ARG;
    const bool legacy = (precision & 16) != 0;
    precision &= ~16;
    if (precision != PREC_BF16 && precision != PREC_TF32X3 && precision != PREC_BF16X3 && precision != PREC_FP16X2) return IS_ERR_ARG;
    if (precision == PREC_FP16X2 && legacy) return IS_ERR_ARG;          // the fp16 hi / lo split exists in the warp-specialised kernel only
    const EdgeCommon c = edge_common(indptr, csr_src, csr_dst, csr_eid, PQ, x, ldx, edge_attr, W1, F, W2, b2, W3, b3, w4, n_nodes, status);
    const int sms = current_num_sms();
    const int per_sm = precision == PREC_BF16 ? 3 : precision == PREC_BF16X3 ? 2 : 1;
    int64_t g = (n_nodes + 31) / 32;
    if (g > (int64_t)sms * per_sm) g = (int64_t)sms * per_sm;
    const int grid = (int)(g < 1 ? 1 : g);
    cudaStream_t st = (cudaStream_t)stream;
    if (((reinterpret_cast<uintptr_t>(PQ) | reinterpret_cast<uintptr_t>(hn)) & 31) != 0) return IS_ERR_ARG;   // 256-bit accesses
    if (!legacy && precision != PREC_TF32X3) return launch_edge_fwd_ws(c, hn, x_out, precision, update_coords != 0, fast_act != 0, st);
    if (precision == PREC_BF16)
        return update_coords ? launch_tc<PREC_BF16, true, 256>(c, hn, x_out, grid, st, fast_act != 0) : launch_tc<PREC_BF16, false, 256>(c, hn, x_out, grid, st, fast_act != 0);
    if (precision == PREC_BF16X3)
        return update_coords ? launch_tc<PREC_BF16X3, true, 256>(c, hn, x_out, grid, st, fast_act != 0) : launch_tc<PREC_BF16X3, false, 256>(c, hn, x_out, grid, st, fast_act != 0);
    return update_coords ? launch_tc<PREC_TF32X3, true, 512>(c, hn, x_out, grid, st, fast_act != 0) : launch_tc<PREC_TF32X3, false, 512>(c, hn, x_out, grid, st, fast_act != 0);
}

// One whole EGNN layer of the fp16x2 inference forward in one launch: is_egnn_edge_fwd_tc (precision 4) followed by
// is_egnn_node_post_pre_tc (precision 4) on the same arguments, with bit-identical results.  h / ldh / F is the layer's input
// (the node MLP reads h and the hn this launch computes); update_coords = 0 needs next_kind 2 (W1n = [Wq;Wk;Wv]) or W1n NULL,
// update_coords = 1 needs next_kind 1.
int is_egnn_layer_fwd_fp16x2(const int* indptr, const int* csr_src, const int* csr_dst, const int* csr_eid,
                             const float* PQ, const float* x, int64_t ldx, const float* edge_attr,
                             const float* W1, int F, const float* W2, const float* b2,
                             const float* W3, const float* b3, const float* w4, int update_coords, float* hn, float* x_out,
                             const float* h, int64_t ldh, const float* W5, const float* b5, const float* W6, const float* b6,
                             float* h_out, const float* W1n, const float* b1n, float* PQn, int next_kind,
                             int64_t n_nodes, int* status, void* stream) {
    if (!(F == 20 || F == 64) || n_nodes <= 0 || n_nodes > 0x7fffffff) return IS_ERR_ARG;
    if ((W1n == nullptr) != (PQn == nullptr)) return IS_ERR_ARG;
    if (next_kind != 1 && next_kind != 2) return IS_ERR_ARG;
    if (update_coords && (next_kind != 1 || x_out == nullptr)) return IS_ERR_ARG;
    if (!update_coords && next_kind == 1 && W1n != nullptr) return IS_ERR_ARG;
    if (((reinterpret_cast<uintptr_t>(PQ) | reinterpret_cast<uintptr_t>(hn) | reinterpret_cast<uintptr_t>(h_out) |
          reinterpret_cast<uintptr_t>(PQn)) & 31) != 0) return IS_ERR_ARG;          // 256-bit accesses
    const EdgeCommon c = edge_common(indptr, csr_src, csr_dst, csr_eid, PQ, x, ldx, edge_attr, W1, F, W2, b2, W3, b3, w4, n_nodes, status);
    const NodeArgs nd{h, ldh, F, hn, W5, b5, W6, b6, h_out, W1n, b1n, PQn};
    return launch_layer_fwd_fp16x2(c, hn, x_out, update_coords != 0, nd, next_kind, (cudaStream_t)stream);
}

}  // extern "C"
