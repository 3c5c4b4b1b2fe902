// EGNN edge forward on the tcgen05 tensor cores, warp-specialised and asynchronous (bf16 and bf16x3 operands), sm_100a.
//
// Same contract as is::edge_fwd_kernel (egnn.cu) / edge_fwd_tc_kernel (egnn_tc.cu, the lock-step first generation).
// What changed, each step driven by ncu source counters of the previous kernel (profiles/):
//
//   * the destination-side feature sum  hn[v] = sum_{e -> v} m[e]  is a THIRD MMA of the tile:
//         hn_tile[32 nodes, 64] = S[32, 128 edges] * m[128 edges, 64]
//     with S the tile's 0/1 segment-selector matrix (exact in bf16, built from the tile's CSR offsets with two
//     16-byte stores per thread) and m read straight from the operand tile that epilogue 1 has just written
//     for MMA 2, through a descriptor with LBO / SBO swapped and the MN-major bit set (= its transpose, no
//     second copy).  M = 64 accumulator (row r in TMEM lane 32 (r / 16) + r % 16).  In the bf16x3 mode the three
//     split terms of m are accumulated (S m3 + S m2 + S m1): hn keeps fp32 accuracy.  (35 % of the first kernel's
//     executed instructions were its two SIMT aggregation loops.)
//   * the coordinate aggregation is one thread per (node, component) instead of one warp per node;
//   * operand tiles are unpadded (LBO = 128 bytes): the gather maps a quarter-warp to 4 rows x 2 K-chunks with
//     the row half chosen by the chunk parity, so every 16-byte operand store of a warp is conflict free;
//   * MMAs are issued by ONE ELECTED LANE OF A CONVERGED WARP with compile-time descriptor offsets: ptxas then
//     emits bare UTCHMMA instructions.  Issued under `if (tid == 0)` every MMA was wrapped in an election loop
//     (~13 instructions, one issuing thread): 72 small MMAs per tile cost ~4 000 cycles of pure issue;
//   * the phases of different tiles overlap (see the third-generation comment below).
//
// Per tile (<= 128 in-edges of <= 32 consecutive destination nodes, CSR order):
//   build S, gather t1 = silu(P[src] + Q[dst] + w_r r + w_a a) -> operand tile
//   MMA 1  z2 = t1 W2^T            -> TMEM acc1
//   epilogue 1: m = silu(z2 + b2)  -> operand tile (bf16 / three bf16 terms)
//   MMA 2  z3 = m W3^T             -> TMEM acc2      (coordinate branch only)
//   MMA 3  hn = S m                -> TMEM hn        (M = 64)
//   epilogue 2: c = w4 . silu(z3 + b3);  hn rows TMEM -> global;  x' = x + mean(c dhat)
#include "common.cuh"
#include "egnn_common.cuh"

#include "egnn_node_tc.cuh"

namespace is {

namespace e2 {
constexpr uint32_t LBO = 144;                    // bytes between K-adjacent core matrices: padded by 16 bytes, so that the eight
                                                 // 16-byte stores of a quarter-warp that holds ONE row (chunks 0..7) hit 8 bank groups
constexpr uint32_t SBO = 8 * LBO;                // bytes between 8-row groups of a 64-wide bf16 tile
constexpr uint32_t A_BYTES = 16 * SBO;           // 128-row operand tile, one split term (18 KB)
constexpr uint32_t W_BYTES = 8 * 8 * umma::kLBO_W;   // 64-row weight tile, one split term (8 KB)
constexpr uint32_t S_LBO = 128;                  // selector tile: K = 128 edges = 16 chunks per node row
constexpr uint32_t S_SBO = 16 * S_LBO;
constexpr uint32_t S_BYTES = 4 * S_SBO;          // 32 node rows (8 KB); the M = 64 MMA also reads the 8 KB behind it
constexpr int MAX_TILE_NODES = 32;

// D[tmem_d] = A * W^T over the 64-wide K block (ONE thread); bf16: 4 MMAs, bf16x3: 24
template <int PREC>
__device__ __forceinline__ void issue_fwd(uint32_t tmem_d, uint32_t a_addr, uint32_t w_addr) {
    using namespace umma;
    const uint32_t idesc = make_instr_desc(TcCfg<PREC>::FMT, 128, 64);
    uint32_t acc = 0;
    // (a-term, w-term), smallest products first -- bf16x3: a3w1 a1w3 a2w2 a2w1 a1w2 a1w1; fp16x2: lo hi, hi lo, hi hi
    constexpr int NP = PREC == PREC_BF16X3 ? 6 : PREC == PREC_FP16X2 ? 3 : 1;
    const uint32_t ta[6] = {PREC == PREC_BF16X3 ? 2u : PREC == PREC_FP16X2 ? 1u : 0u, 0, PREC == PREC_BF16X3 ? 1u : 0u, 1, 0, 0};
    const uint32_t tw[6] = {0, PREC == PREC_BF16X3 ? 2u : 1u, PREC == PREC_BF16X3 ? 1u : 0u, 0, 1, 0};
#pragma unroll
    for (int t = 0; t < NP; ++t)
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
            mma_bf16(tmem_d, make_smem_desc(a_addr + ta[t] * A_BYTES + ks * 2 * LBO, LBO, SBO),
                     make_smem_desc(w_addr + tw[t] * W_BYTES + ks * 2 * kLBO_W, kLBO_W, 8 * kLBO_W), idesc, acc);
            acc = 1;
        }
}

// same product with the A operand in TENSOR MEMORY (split term t at columns tmem_a + 32 t, 8 columns per K step): the
// epilogue threads own one accumulator row each, so they can put m straight into their TMEM lane; the tensor core
// then reads only the weights from shared memory (a third of the operand bytes of the shared-memory form)
template <int PREC>
__device__ __forceinline__ void issue_fwd_ts(uint32_t tmem_d, uint32_t tmem_a, uint32_t w_addr) {
    using namespace umma;
    const uint32_t idesc = make_instr_desc(TcCfg<PREC>::FMT, 128, 64);
    uint32_t acc = 0;
    constexpr int NP = PREC == PREC_BF16X3 ? 6 : PREC == PREC_FP16X2 ? 3 : 1;
    const uint32_t ta[6] = {PREC == PREC_BF16X3 ? 2u : PREC == PREC_FP16X2 ? 1u : 0u, 0, PREC == PREC_BF16X3 ? 1u : 0u, 1, 0, 0};
    const uint32_t tw[6] = {0, PREC == PREC_BF16X3 ? 2u : 1u, PREC == PREC_BF16X3 ? 1u : 0u, 0, 1, 0};
#pragma unroll
    for (int t = 0; t < NP; ++t)
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
            mma_bf16_ts(tmem_d, tmem_a + 32 * ta[t] + 8 * ks,
                        make_smem_desc(w_addr + tw[t] * W_BYTES + ks * 2 * kLBO_W, kLBO_W, 8 * kLBO_W), idesc, acc);
            acc = 1;
        }
}

// hn tile:  D[tmem_d] (M = 64 rows = nodes) = S[64, 16 nks] * m[16 nks, 64]; m = the A tile read MN-major
template <int PREC>
__device__ __forceinline__ void issue_segsum(uint32_t tmem_d, uint32_t s_addr, uint32_t a_addr, int nks) {
    using namespace umma;
    const uint32_t idesc = make_instr_desc(TcCfg<PREC>::FMT, 64, 64, 0, 1);
    uint32_t acc = 0;
    constexpr int NS = TcCfg<PREC>::NSPLIT;
#pragma unroll
    for (int t = NS - 1; t >= 0; --t)                       // smallest term first
#pragma unroll 8
        for (int ks = 0; ks < nks; ++ks) {
            mma_bf16(tmem_d, make_smem_desc(s_addr + ks * 2 * S_LBO, S_LBO, S_SBO),
                     make_smem_desc(a_addr + t * A_BYTES + ks * 2 * SBO, SBO, LBO), idesc, acc);
            acc = 1;
        }
}
}  // namespace e2

// =====================================================================================================
// The tile pipeline, warp-specialised and asynchronous (one 704-thread CTA per SM).
//
// The lock-step kernels (egnn_tc.cu) leave the SM idle 65 % of the issue slots: every phase of a tile ends in a CTA
// barrier, the L2 gather latency, the dependent scalar prefetch chain and the MMA latencies are all exposed, and
// two CTAs per SM are not enough to cover them (ncu: barrier 3.9 + long-scoreboard 2.5 stall cycles per issue).
// Here the phases of DIFFERENT tiles overlap; mbarriers replace every CTA barrier:
//
//   warps 18-21 (scalars) walk the CSR, computes the per-edge scalars (src, r, a, dhat, local dst) of tile i+3
//   warps 8-15 (gather) build S and gather t1 of tile i+1 into operand buffer (i+1)&1
//   warps 16, 17 (MMA)  one elected lane each: MMA1(i+1) | MMA2(i), MMA3(i); commits to the mbarriers below
//   warps 0-7 (epilog)  epilogue 1 of tile i, then epilogue 2 / hn rows / coordinate sums of tile i-1
//
//   meta_full[4]  scalars -> everyone      meta_free[4]  epilog -> scalars (tile fully consumed)
//   a_full[2]     gather  -> MMA           acc1_full[2]  MMA1 commit -> epilog
//   m_full[2]     epilog  -> MMA           acc2_full[2]  MMA2 commit -> epilog
//   hn_full[2]    MMA3 commit -> epilog (hn rows) and gather (operand buffer + S free again)
// TMEM: acc1[2] | acc2[2] | hn[2], 64 columns each (512 allocated).  Shared memory: two operand buffers
// (bf16x3: 2 x 48 KB), W2 / W3 once (48 KB; no W3 without the coordinate branch), two selector tiles, four scalar stages:
// 175 KB.
//
// NODE != 0 (fp16x2 inference forward, egnn_layer_fwd): the kernel is the whole EGNN layer.  A CTA's tiles cover its node
// range [nbeg, nend) and hold every in-edge of those nodes, so when its last tile is done the CTA has the complete hn of
// exactly its own nodes -- all the node MLP and the next layer's projections need (node_chain, egnn_node_tc.cuh).  After a
// CTA barrier warps 0-15 run that chain over [nbeg, nend), in the TMEM allocation and over the operand region of the edge
// phase; its weight blocks were staged next to W2 / W3 in the prologue.  NODE = 1: P' / Q' of the next layer (or nothing
// when nd.W1n is null); NODE = 2: the fused QKV projections after the last layer.  The only dependency across the grid is
// the next layer's gather of P'[src] / Q'[dst], which is the next launch.
// =====================================================================================================
namespace e3 {
using namespace e2;
constexpr int NW_EPI = 8, NW_PROD = 8;
constexpr int W_MMA = NW_EPI + NW_PROD, W_META = W_MMA + 2;   // two MMA warps
constexpr int NW_META = 4;                       // scalar warps: one edge per lane
constexpr int NT3 = 32 * (W_META + NW_META);     // 704 threads
constexpr int NM = 4;                            // scalar stages
constexpr uint32_t TM_ACC1 = 0, TM_ACC2 = 128, TM_HN = 256;   // + 64 * buffer
constexpr uint32_t TM_MA = 384;                  // m as the A operand of MMA 2: 32 columns per split term

struct Meta3 {
    int src[IS_TM];
    float r[IS_TM];
    float a[IS_TM];
    float dh[IS_TM * 3];
    int nptr[MAX_TILE_NODES + 1];   // indptr[n0 + i] - p0
    int tile[3];                    // n0, n1, ne   (n0 >= nend: no more tiles)
    uint8_t dloc[IS_TM];            // destination node - n0
};

__device__ __forceinline__ void meta_edge(const EdgeCommon& p, Meta3& m, int j, int n0, int p0, int ne) {
    if (j < ne) {
        const int e = p0 + j;
        const int s = __ldg(p.csr_src + e), d = __ldg(p.csr_dst + e);
        const float a = __ldg(p.edge_attr + __ldg(p.csr_eid + e));
        const float dx = __ldg(p.x + s * p.ldx + 0) - __ldg(p.x + d * p.ldx + 0);
        const float dy = __ldg(p.x + s * p.ldx + 1) - __ldg(p.x + d * p.ldx + 1);
        const float dz = __ldg(p.x + s * p.ldx + 2) - __ldg(p.x + d * p.ldx + 2);
        const float r = dx * dx + dy * dy + dz * dz;
        const float inv = 1.0f / (sqrtf(r) + 1e-30f);
        m.src[j] = s; m.dloc[j] = (uint8_t)(d - n0); m.r[j] = r; m.a[j] = a;
        m.dh[j * 3 + 0] = dx * inv; m.dh[j * 3 + 1] = dy * inv; m.dh[j * 3 + 2] = dz * inv;
    }
}
}  // namespace e3

#ifndef IS_WS_WAIT_HINT_NS
#define IS_WS_WAIT_HINT_NS 2000
#endif
#define WS_WAIT(bar, parity) mbar_wait_hint(bar, parity, IS_WS_WAIT_HINT_NS)

// TSA = the A operand of MMA 2 comes from TENSOR MEMORY (is_egnn_set_ws_variant bit 0, default on): the kernel is bound by the
// L1 / shared-memory data pipe (ncu: LSU wavefronts 56 % + tensor-core operand wavefronts 43 % of the pipe's cycles), and
// every shared-memory A operand is read six times by the bf16x3 products (3 x a1, 2 x a2, 1 x a3).  Epilogue 1 therefore
// also puts the packed split terms of m into its own TMEM lanes (tcgen05.st: 96 columns, single buffered -- MMA 2 of
// tile i - 1 has completed before epilogue 1 of tile i stores: it waits for acc2_full of tile i - 1 first); the shared-memory
// copy of m stays for MMA 3, which reads it transposed as its B operand.
// The gather maps a quarter-warp to ONE row (8 lanes x 32 bytes = the row's 256 contiguous bytes of P or Q, two whole
// 128-byte lines per quarter-warp and instruction); with LBO = 144 its eight 16-byte operand stores are conflict free.
template <int PREC, bool HAS_COORD>
__host__ __device__ constexpr uint32_t ws_edge_bytes() {
    using namespace e3;
    return 2 * S_BYTES + TcCfg<PREC>::NSPLIT * (2 * A_BYTES + (HAS_COORD ? 2 : 1) * W_BYTES) + sizeof(float) * (5 * 64 + 4 * IS_TM) +
           NM * sizeof(Meta3);
}

// shared memory of the node tail: the operand buffers reuse the edge region (which they may outgrow), the weight blocks and
// biases follow it
template <int PREC, bool HAS_COORD, int NODE>
__host__ __device__ constexpr uint32_t ws_node_offset() {
    using NC = NodeCfg<PREC, NODE>;
    constexpr uint32_t e = ws_edge_bytes<PREC, HAS_COORD>();
    return NODE == 0 ? 0u : ((e > NC::A_REGION ? e : NC::A_REGION) + 127u) / 128u * 128u;
}

template <int PREC, bool HAS_COORD, int NODE>
__host__ __device__ constexpr uint32_t ws_smem_bytes() {
    using NC = NodeCfg<PREC, NODE>;
    return NODE == 0 ? ws_edge_bytes<PREC, HAS_COORD>() : ws_node_offset<PREC, HAS_COORD, NODE>() + NC::W_REGION + NC::VEC_BYTES;
}

template <int PREC, bool HAS_COORD, bool FAST, bool TSA, int NODE>
__global__ void __launch_bounds__(e3::NT3, 1)
edge_fwd_ws_kernel(EdgeCommon p, float* __restrict__ hn, float* __restrict__ x_out, NodeArgs nd) {
    using namespace e3;
    using C = TcCfg<PREC>;
    constexpr int NS = C::NSPLIT;
    constexpr int CW = 32;                      // accumulator columns per epilogue thread (two column halves)
    constexpr uint32_t ABUF = NS * A_BYTES;     // one operand buffer (all split terms)
    constexpr bool TS2 = TSA && HAS_COORD;      // MMA 2 exists and takes m from TMEM
    static_assert(NODE == 0 || (PREC == PREC_FP16X2 && FAST), "the node tail is the fp16x2 inference chain");
    static_assert(ws_smem_bytes<PREC, HAS_COORD, NODE>() <= 227 * 1024 - 1024, "shared memory (+ the static mbarriers)");
    extern __shared__ __align__(128) uint8_t smem_raw[];
    uint8_t* sS = smem_raw;                                            // [2][S_BYTES]; rows 32..63 of a tile alias what follows
    uint8_t* sA = sS + 2 * S_BYTES;                                    // [2][NS][A_BYTES] t1, then m
    uint8_t* sW2 = sA + 2 * ABUF;                                      // [NS][W_BYTES]
    uint8_t* sW3 = sW2 + NS * W_BYTES;                                 // [NS][W_BYTES] (coordinate branch only)
    float* vec = reinterpret_cast<float*>(sW3 + (HAS_COORD ? NS * W_BYTES : 0));   // b2, b3, w4, wr, wa
    float* e_c = vec + 5 * 64;                                         // [2 buffers][2 halves][128] partial c
    Meta3* meta = reinterpret_cast<Meta3*>(e_c + 4 * IS_TM);           // [NM]
    uint8_t* sNW = smem_raw + ws_node_offset<PREC, HAS_COORD, NODE>(); // node tail: [NS][NBLK][W_BYTES], then its biases
    float* nvec = reinterpret_cast<float*>(sNW + NodeCfg<PREC, NODE>::W_REGION);
    __shared__ __align__(8) uint64_t meta_full[NM], meta_free[NM], a_full[2], acc1_full[2], m_full[2], acc2_full[2], hn_full[2];
    __shared__ __align__(8) uint64_t node_bar;
    __shared__ NodeArgs s_nd;     // the tail reads its arguments from here: kept in registers across the edge phase they spill
    __shared__ uint32_t s_tmem;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ldw1 = 2 * p.F + 2;
    if (warp == 0) tmem_alloc(&s_tmem, 512);
    if (tid == 32) {
        for (int i = 0; i < NM; ++i) { mbar_init(&meta_full[i], NW_META); mbar_init(&meta_free[i], NW_EPI); }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&a_full[i], NW_PROD); mbar_init(&m_full[i], NW_EPI);
            mbar_init(&acc1_full[i], 1); mbar_init(&acc2_full[i], 1); mbar_init(&hn_full[i], 1);
        }
        if (NODE != 0) { mbar_init(&node_bar, 1); s_nd = nd; }
    }
    stage_weight_block<PREC>(sW2, W_BYTES, p.W2, 64, 0, 64, tid, NT3);                 // W2 / W3 as B operands
    if (HAS_COORD) stage_weight_block<PREC>(sW3, W_BYTES, p.W3, 64, 0, 64, tid, NT3);
    if (NODE != 0) node_stage_weights<PREC, NODE>(nd, sNW, nvec, tid, NT3);
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
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = s_tmem;

    if (warp >= W_META) {
        // ================= scalars: tile walk + per-edge geometry, up to NM - 1 tiles ahead =================
        int cursor = nbeg;
        for (int i = 0;; ++i) {
            const int s = i % NM;
            if (i >= NM) WS_WAIT(&meta_free[s], ((i / NM) - 1) & 1);
            int tn0, tn1, tp0, tne;
            next_tile(p.indptr, cursor, nend, p.status, lane, tn0, tn1, tp0, tne);
            Meta3& m = meta[s];
            const int mw = warp - W_META;                      // every scalar warp walks the CSR (same result)
            if (mw == 0 && lane == 0) { m.tile[0] = tn0; m.tile[1] = tn1; m.tile[2] = tne; }
            if (tn0 < nend) {
                meta_edge(p, m, lane + 32 * mw, tn0, tp0, tne);
                if (mw == 1 || (mw == 2 && lane == 0)) {
                    const int j = mw == 1 ? lane : MAX_TILE_NODES;
                    const int node = tn0 + j;
                    m.nptr[j] = node <= tn1 ? __ldg(p.indptr + node) - tp0 : tne;
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&meta_full[s]);
            if (tn0 >= nend) break;
            cursor = tn1;
        }
    } else if (warp == W_MMA || warp == W_MMA + 1) {
        // ================= MMA issue: warp 16 MMA1(i); warp 17 MMA2(i) + MMA3(i) -- two independent streams =========
        // Each warp walks its loop converged and one elected lane issues.  Every descriptor is a compile-time offset
        // from the shared-memory base (two unrolled copies for the two operand buffers, MMA 3 always over all eight K
        // steps: rows beyond the tile's edges are finite and meet zeros in S), so ptxas keeps them in uniform registers
        // and emits bare UTCHMMA instructions instead of a per-MMA election loop.  Two warps because a single in-order
        // stream would hold back MMA2/MMA3 of tile i-1 (which free the operand buffer for the gather of tile i+1)
        // behind the wait for the gather of tile i.
        const uint32_t s_addr = smem_u32(sS), a_addr = smem_u32(sA), w2_addr = smem_u32(sW2), w3_addr = smem_u32(sW3);
        const bool first = warp == W_MMA;
        bool done = false;
        for (int i2 = 0; !done; i2 += 2) {
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int i = i2 + u;
                const int b = u;                         // compile-time after unrolling (i2 is even)
                WS_WAIT(&meta_full[i % NM], (i / NM) & 1);
                done = meta[i % NM].tile[0] >= nend;
                if (done) break;
                if (first) {
                    WS_WAIT(&a_full[b], (i >> 1) & 1);
                    fence_after_sync();
                    if (elect_one()) {
                        issue_fwd<PREC>(tmem + TM_ACC1 + 64 * b, a_addr + b * ABUF, w2_addr);
                        mma_commit(&acc1_full[b]);
                    }
                } else {
                    WS_WAIT(&m_full[b], (i >> 1) & 1);
                    fence_after_sync();
                    if (elect_one()) {
                        if (HAS_COORD) {
                            if (TS2) issue_fwd_ts<PREC>(tmem + TM_ACC2 + 64 * b, tmem + TM_MA, w3_addr);
                            else issue_fwd<PREC>(tmem + TM_ACC2 + 64 * b, a_addr + b * ABUF, w3_addr);
                            mma_commit(&acc2_full[b]);
                        }
                        issue_segsum<PREC>(tmem + TM_HN + 64 * b, s_addr + b * S_BYTES, a_addr + b * ABUF, 8);
                        mma_commit(&hn_full[b]);
                    }
                }
                __syncwarp();
            }
        }
    } else if (warp >= NW_EPI) {
        // ================= gather: S + t1 of tile i into operand buffer i & 1 =================
        const int pw = warp - NW_EPI;
        // a quarter-warp takes ONE row: lane -> row rl = lane / 8 of a 4-row pass, K chunk kc = lane % 8 (8 features, 32 bytes)
        const int rl = lane >> 3, kc = lane & 7;
        const float4 wr0 = *reinterpret_cast<const float4*>(vec + 192 + 8 * kc), wr1 = *reinterpret_cast<const float4*>(vec + 196 + 8 * kc);
        const float4 wa0 = *reinterpret_cast<const float4*>(vec + 256 + 8 * kc), wa1 = *reinterpret_cast<const float4*>(vec + 260 + 8 * kc);
        for (int i = 0;; ++i) {
            const int b = i & 1;
            WS_WAIT(&meta_full[i % NM], (i / NM) & 1);
            const Meta3& mt = meta[i % NM];
            const int n0 = mt.tile[0], ne = mt.tile[2];
            if (n0 >= nend) break;
            uint8_t* A = sA + b * ABUF;
            const float wr[8] = {wr0.x, wr0.y, wr0.z, wr0.w, wr1.x, wr1.y, wr1.z, wr1.w};
            const float wa[8] = {wa0.x, wa0.y, wa0.z, wa0.w, wa1.x, wa1.y, wa1.z, wa1.w};
            float pv[2][8], qv[2][8];
            float rr[2], aa[2];
            auto load_rows = [&](int gi) {          // P[src] and Q[dst] of this thread's two (row, chunk) items of 8-row group pair gi
                const int g8 = 8 * (2 * pw + gi);
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int j = g8 + 4 * u + rl;
                    const bool valid = j < ne;
                    const int s = valid ? mt.src[j] : 0, d = n0 + (valid ? (int)mt.dloc[j] : 0);
                    rr[u] = valid ? mt.r[j] : 0.0f;
                    aa[u] = valid ? mt.a[j] : 0.0f;
                    ldg256(p.PQ + (size_t)s * 128 + 8 * kc, pv[u]);      // one whole 32-byte sector per lane
                    ldg256(p.PQ + (size_t)d * 128 + 64 + 8 * kc, qv[u]);
                }
            };
            auto store_rows = [&](int gi) {
                const int g8 = 8 * (2 * pw + gi);
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int j = g8 + 4 * u + rl;
                    const float r = rr[u], a = aa[u];
                    float v[8];
#pragma unroll
                    for (int i2 = 0; i2 < 8; ++i2) v[i2] = act<PREC, FAST>(pv[u][i2] + qv[u][i2] + wr[i2] * r + wa[i2] * a);
                    // rows beyond the tile's edges hold finite values: the selector has zeros there
                    store_chunk8<PREC>(A + (j >> 3) * SBO + (j & 7) * 16 + kc * LBO, A_BYTES, v);
                }
            };
            // the first round of row loads needs the scalars only, not the operand buffer: it is in flight while this warp
            // waits for MMA 2 / MMA 3 of tile i-2 to release the buffer
            load_rows(0);
            if (i >= 2) WS_WAIT(&hn_full[b], ((i >> 1) - 1) & 1);    // MMA2 / MMA3 of tile i-2 are done with the buffer
            {   // S[node][edge] = 1 for the node's in-edges (two 16-byte chunks per thread)
                const int jb = mt.nptr[lane], je = mt.nptr[lane + 1];         // rows beyond the tile: jb = je = ne
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int c = pw + 8 * u;
                    const int lo = min(max(jb - 8 * c, 0), 8), hi = min(max(je - 8 * c, 0), 8);
                    const uint32_t mask = (1u << hi) - (1u << lo);            // bits lo .. hi-1
                    constexpr uint32_t ONE = PREC == PREC_FP16X2 ? 0x3C00u : 0x3F80u;      // 1.0 in the operand format
                    uint4 w;
                    w.x = ((mask >> 0) & 1u) * ONE + ((mask >> 1) & 1u) * (ONE << 16);
                    w.y = ((mask >> 2) & 1u) * ONE + ((mask >> 3) & 1u) * (ONE << 16);
                    w.z = ((mask >> 4) & 1u) * ONE + ((mask >> 5) & 1u) * (ONE << 16);
                    w.w = ((mask >> 6) & 1u) * ONE + ((mask >> 7) & 1u) * (ONE << 16);
                    *reinterpret_cast<uint4*>(sS + b * S_BYTES + (lane >> 3) * S_SBO + c * S_LBO + (lane & 7) * 16) = w;
                }
            }
            store_rows(0);
            load_rows(1);
            store_rows(1);
            fence_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&a_full[b]);
        }
    } else {
        // ================= epilogue: epilogue 1 of tile i, then epilogue 2 / hn rows / coordinates of tile i-1 =====
        const int q = warp & 3, cq = warp >> 2, erow = 32 * q + lane;      // TMEM lane quarter, column half, tile row
        const uint32_t t_lane = tmem + ((uint32_t)(32 * q) << 16) + CW * cq;
        const uint32_t t_ma = tmem + ((uint32_t)(32 * q) << 16) + TM_MA + (CW / 2) * cq;      // 4 columns per 8-feature chunk
        for (int i = 0;; ++i) {
            const int b = i & 1;
            WS_WAIT(&meta_full[i % NM], (i / NM) & 1);
            const bool done = meta[i % NM].tile[0] >= nend;
            if (!done) {
                // ---- epilogue 1: m = silu(acc1 + b2) -> operand buffer (B of MMA 3, transposed) and TMEM (A of MMA 2) ----
                WS_WAIT(&acc1_full[b], (i >> 1) & 1);
                if (TS2 && i >= 1) WS_WAIT(&acc2_full[b ^ 1], ((i - 1) >> 1) & 1);   // MMA 2 of tile i-1 has read the TMEM copy
                fence_after_sync();
                uint8_t* A = sA + b * ABUF;
                float z[CW];
                tmem_ld<CW>(t_lane + TM_ACC1 + 64 * b, z);
#pragma unroll
                for (int g = 0; g < CW / 8; ++g) {
                    const float4 b0 = *reinterpret_cast<const float4*>(vec + CW * cq + 8 * g);
                    const float4 b1 = *reinterpret_cast<const float4*>(vec + CW * cq + 8 * g + 4);
                    float m8[8];
                    m8[0] = act<PREC, FAST>(z[8 * g + 0] + b0.x); m8[1] = act<PREC, FAST>(z[8 * g + 1] + b0.y);
                    m8[2] = act<PREC, FAST>(z[8 * g + 2] + b0.z); m8[3] = act<PREC, FAST>(z[8 * g + 3] + b0.w);
                    m8[4] = act<PREC, FAST>(z[8 * g + 4] + b1.x); m8[5] = act<PREC, FAST>(z[8 * g + 5] + b1.y);
                    m8[6] = act<PREC, FAST>(z[8 * g + 6] + b1.z); m8[7] = act<PREC, FAST>(z[8 * g + 7] + b1.w);
                    uint4 qs[3];
                    split_chunk8<PREC>(m8, qs);
                    uint8_t* dst = A + (erow >> 3) * SBO + (erow & 7) * 16 + ((CW / 8) * cq + g) * LBO;
#pragma unroll
                    for (int t = 0; t < NS; ++t) {
                        *reinterpret_cast<uint4*>(dst + t * A_BYTES) = qs[t];
                        if (TS2) tmem_st4(t_ma + 32 * t + 4 * g, qs[t].x, qs[t].y, qs[t].z, qs[t].w);
                    }
                }
                if (TS2) tmem_st_wait();
                fence_async_smem();
                fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(&m_full[b]);
            }
            if (i >= 1) {
                const int j = i - 1, bp = b ^ 1;
                const Meta3& mj = meta[j % NM];
                const int n0 = mj.tile[0], n1 = mj.tile[1];
                float* ec = e_c + bp * 2 * IS_TM;
                if (HAS_COORD) {
                    // ---- epilogue 2: c = w4 . silu(acc2 + b3) (each thread: one row, CW columns) ----
                    WS_WAIT(&acc2_full[bp], (j >> 1) & 1);
                    fence_after_sync();
                    float z[CW];
                    tmem_ld<CW>(t_lane + TM_ACC2 + 64 * bp, z);
                    float c = 0.0f;
#pragma unroll
                    for (int g = 0; g < CW / 4; ++g) {
                        const float4 bb = *reinterpret_cast<const float4*>(vec + 64 + CW * cq + 4 * g);
                        const float4 w = *reinterpret_cast<const float4*>(vec + 128 + CW * cq + 4 * g);
                        c = fmaf(w.x, act<PREC, FAST>(z[4 * g + 0] + bb.x), c);
                        c = fmaf(w.y, act<PREC, FAST>(z[4 * g + 1] + bb.y), c);
                        c = fmaf(w.z, act<PREC, FAST>(z[4 * g + 2] + bb.z), c);
                        c = fmaf(w.w, act<PREC, FAST>(z[4 * g + 3] + bb.w), c);
                    }
                    ec[cq * IS_TM + erow] = c;
                }
                // ---- hn rows: M = 64 accumulator, node row r sits in TMEM lane 32 (r / 16) + r % 16 ----
                WS_WAIT(&hn_full[bp], (j >> 1) & 1);
                fence_after_sync();
                if (q < 2) {
                    float z[CW];
                    tmem_ld<CW>(t_lane + TM_HN + 64 * bp, z);
                    const int node = n0 + 16 * q + lane;
                    if (lane < 16 && node < n1) {
#pragma unroll
                        for (int g = 0; g < CW / 8; ++g) {
                            const float o[8] = {z[8 * g], z[8 * g + 1], z[8 * g + 2], z[8 * g + 3], z[8 * g + 4], z[8 * g + 5], z[8 * g + 6], z[8 * g + 7]};
                            stg256(hn + (size_t)node * 64 + CW * cq + 8 * g, o);
                        }
                    }
                }
                if (HAS_COORD) {
                    asm volatile("bar.sync 1, %0;" ::"n"(32 * NW_EPI) : "memory");      // partial c of all 256 rows visible
                    // ---- coordinate aggregation: one thread per (node, component) ----
                    if (tid < 3 * MAX_TILE_NODES) {
                        const int nl = tid / 3, comp = tid - 3 * nl, node = n0 + nl;
                        if (node < n1) {
                            const int jb = mj.nptr[nl], je = mj.nptr[nl + 1];
                            float sx = 0.0f;
                            for (int e = jb; e < je; ++e) sx += (ec[e] + ec[IS_TM + e]) * mj.dh[e * 3 + comp];
                            x_out[(size_t)node * 3 + comp] = __ldg(p.x + node * p.ldx + comp) + sx / (float)max(je - jb, 1);
                        }
                    }
                }
                fence_before_sync();
                __syncwarp();
                if (lane == 0) mbar_arrive(&meta_free[j % NM]);
            }
            if (done) break;
        }
    }
    if (NODE != 0) {
        // every MMA of the edge phase has been observed complete through its commit mbarrier by the epilogue warps (acc2_full /
        // hn_full of the last tile) and every tcgen05.ld / st has been waited for: TMEM and the operand region are free
        constexpr int NT_NODE = 512;                 // warps 0-15: the epilogue and gather warps
        static_assert(NodeCfg<PREC, NODE>::NTILE * NodeCfg<PREC, NODE>::TCOLS <= 512, "TMEM columns");
        fence_before_sync();
        __syncthreads();
        fence_after_sync();
        if (tid < NT_NODE) {
            uint32_t phase = 0;
            node_chain<PREC, NT_NODE, FAST, NODE>(s_nd, smem_raw, sNW, nvec, tmem, &node_bar, phase, nbeg,
                                                  NodeCfg<PREC, NODE>::NTILE * IS_TM, nend, tid, 2);
        }
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

// variant bits of the warp-specialised kernel (is_egnn_set_ws_variant): bit 0 = A operand of MMA 2 from tensor memory
int g_ws_variant = 1;

template <int PREC, bool HAS_COORD, bool FAST, bool TSA, int NODE = 0>
static int launch_wsk_v(const EdgeCommon& c, float* hn, float* x_out, int grid, cudaStream_t st, const NodeArgs& nd = NodeArgs{}) {
    const size_t smem = ws_smem_bytes<PREC, HAS_COORD, NODE>();
    cudaError_t e = cudaFuncSetAttribute(edge_fwd_ws_kernel<PREC, HAS_COORD, FAST, TSA, NODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    edge_fwd_ws_kernel<PREC, HAS_COORD, FAST, TSA, NODE><<<grid, e3::NT3, smem, st>>>(c, hn, x_out, nd);
    e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

template <int PREC, bool HAS_COORD, bool FAST>
static int launch_wsk(const EdgeCommon& c, float* hn, float* x_out, int grid, cudaStream_t st) {
    if (HAS_COORD && (g_ws_variant & 1)) return launch_wsk_v<PREC, HAS_COORD, FAST, true>(c, hn, x_out, grid, st);
    return launch_wsk_v<PREC, HAS_COORD, FAST, false>(c, hn, x_out, grid, st);
}

static int ws_grid(int n_nodes) {
    const int sms = current_num_sms();
    int64_t g = ((int64_t)n_nodes + 31) / 32;
    if (g > sms) g = sms;
    return (int)(g < 1 ? 1 : g);
}

// entry used by is_egnn_edge_fwd_tc (egnn_tc.cu) for the bf16 / bf16x3 precisions: warp-specialised kernel
int launch_edge_fwd_ws(const EdgeCommon& c, float* hn, float* x_out, int precision, bool update_coords, bool fast,
                       cudaStream_t st) {
    const int grid = ws_grid(c.n_nodes);
    if (precision == PREC_BF16)
        return update_coords ? launch_wsk<PREC_BF16, true, true>(c, hn, x_out, grid, st)
                             : launch_wsk<PREC_BF16, false, true>(c, hn, x_out, grid, st);
    if (precision == PREC_FP16X2)          // inference forward only (fast SiLU)
        return update_coords ? launch_wsk<PREC_FP16X2, true, true>(c, hn, x_out, grid, st)
                             : launch_wsk<PREC_FP16X2, false, true>(c, hn, x_out, grid, st);
    if (fast)
        return update_coords ? launch_wsk<PREC_BF16X3, true, true>(c, hn, x_out, grid, st)
                             : launch_wsk<PREC_BF16X3, false, true>(c, hn, x_out, grid, st);
    return update_coords ? launch_wsk<PREC_BF16X3, true, false>(c, hn, x_out, grid, st)
                         : launch_wsk<PREC_BF16X3, false, false>(c, hn, x_out, grid, st);
}

// the whole fp16x2 inference layer in one launch (is_egnn_layer_fwd_fp16x2): edge phase with the node tail.  With the
// coordinate branch: P' / Q' of the next layer; without: the QKV projections (next_kind 2) or P' / Q' (W1n null: h' only).
// MMA 2 always takes m from tensor memory (the default variant of the two-kernel path).
int launch_layer_fwd_fp16x2(const EdgeCommon& c, float* hn, float* x_out, bool update_coords, const NodeArgs& nd, int next_kind,
                            cudaStream_t st) {
    const int grid = ws_grid(c.n_nodes);
    if (update_coords) return launch_wsk_v<PREC_FP16X2, true, true, true, 1>(c, hn, x_out, grid, st, nd);
    if (next_kind == 2) return launch_wsk_v<PREC_FP16X2, false, true, false, 2>(c, hn, x_out, grid, st, nd);
    return launch_wsk_v<PREC_FP16X2, false, true, false, 1>(c, hn, x_out, grid, st, nd);
}

}  // namespace is

// Operand buffers of the warp-specialised edge forward kernel.  A third buffer was measured on the B200 (225 vs 227 us in
// inference, slower in training and in bf16: the free-buffer wait is not on the critical path) and no longer fits next to
// the padded operand tiles: only 2 is accepted.
extern "C" int is_egnn_set_ws_buffers(int n) { return n == 2 ? IS_OK : IS_ERR_UNSUPPORTED; }

// Variant bits of the warp-specialised edge forward kernel (A/B timing): bit 0 = A operand of MMA 2 from tensor memory.
extern "C" int is_egnn_set_ws_variant(int bits) {
    if (bits < 0 || bits > 1) return IS_ERR_ARG;
    is::g_ws_variant = bits;
    return IS_OK;
}
