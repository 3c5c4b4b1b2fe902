// The node tile chain of the tensor-core node kernel (egnn_node_tc.cu), shared with the fused layer kernel of egnn_tc2.cu:
//
//   node_post(l) :  h' = W6 silu(W5 [h | hn] + b5) + b6              (reference: EGNNConv node_mlp)
//   node_pre(l+1):  P' = h' Ws'^T ,  Q' = h' Wd'^T + b1'              (first edge-MLP layer of layer l+1, split per node)
//   or, after the LAST layer (NEXT_KIND = 2):  QKV = h' [Wq; Wk; Wv]^T + [bq; bk; bv]
//
// Per group of NTILE tiles of 128 nodes, four chained tcgen05 GEMM groups run against weight blocks resident in shared memory:
//   D1 = h W5h^T + hn W5n^T  -> +b5, SiLU -> D2 = t5 W6^T -> +b6 = h' (stored) -> D3 = h' [Ws'; Wd']^T (+b1')
// The chain is run by NT threads (warps 0 .. NT/32 - 1 of the CTA) that synchronise with the named barrier `bar_id`.
#pragma once
#include "tc_common.cuh"

namespace is {

struct NodeArgs {
    const float* h;       // [M, F] rows with leading dimension ldh
    int64_t ldh;
    int F;
    const float* hn;      // [M, 64]
    const float* W5;
    const float* b5;
    const float* W6;
    const float* b6;
    float* h_out;         // [M, 64]
    const float* W1n;     // next layer edge_mlp.0.weight [64,130] | [Wq;Wk;Wv] [192,64] | null
    const float* b1n;
    float* PQn;           // [M, 128] | QKV [M, 192] | null
};

template <int PREC, int NEXT_KIND>
struct NodeCfg {
    using C = TcCfg<PREC>;
    static constexpr int NBLK = NEXT_KIND == 2 ? 6 : 5;                      // resident weight blocks
    static constexpr uint32_t ASPL = C::A_BYTES, WSPL = NBLK * C::W_BYTES;    // split-term strides
    // TWO_BUF (one- and two-term operand splits: the three-term tiles leave no room): a second A-operand buffer, so that h
    // and hn are staged together (their row loads overlap) and D1 = h W5h^T + hn W5n^T is ONE MMA group with one hand-over
    // instead of two; the epilogues then alternate between the buffers.
    static constexpr bool TWO_BUF = C::NSPLIT <= 2;
    // NTILE (fp16x2: 2) tiles of 128 nodes share every hand-over: a tile's chain is a string of fixed latencies (barriers, MMA
    // completion, the row loads' round trip) -- shortening its rows by 10 % did not change the kernel's time at all -- so two
    // tiles per round halve the rounds (800 tiles on 148 CTAs: 6 -> 3) at little extra cost per round.  Needs both tiles'
    // operand buffers (4 x 32 KB next to 96 KB of weights) and 2 x 256 TMEM columns.
    static constexpr int NTILE = (PREC == PREC_FP16X2 && NEXT_KIND == 1) ? 2 : 1;   // (the six blocks of the QKV tail leave no room)
    static constexpr uint32_t ABUF = C::NSPLIT * ASPL, ASTRIDE = (TWO_BUF ? 2 : 1) * ABUF, TCOLS = 256;
    static constexpr uint32_t A_REGION = NTILE * ASTRIDE;                    // [NTILE][1 or 2 buffers][NSPLIT][A_BYTES]
    static constexpr uint32_t W_REGION = C::NSPLIT * WSPL;                    // [NSPLIT][NBLK][W_BYTES]
    static constexpr uint32_t VEC_BYTES = 5 * 64 * sizeof(float);            // b5, b6, next bias (64: b1' for Q' | 192: bq bk bv)
};

// stage the resident weight blocks (W5h W5n W6 | Ws' Wd' - or Wq Wk Wv) into sW and the biases into vec; thread tid of nthreads
// (nthreads >= 192)
template <int PREC, int NEXT_KIND>
__device__ __forceinline__ void node_stage_weights(const NodeArgs& a, uint8_t* sW, float* vec, int tid, int nthreads) {
    using C = TcCfg<PREC>;
    constexpr uint32_t WSPL = NodeCfg<PREC, NEXT_KIND>::WSPL;
    const bool has_next = a.W1n != nullptr;
    const int K5 = a.F + 64;
    stage_weight_block<PREC>(sW + 0 * C::W_BYTES, WSPL, a.W5, K5, 0, a.F, tid, nthreads);
    stage_weight_block<PREC>(sW + 1 * C::W_BYTES, WSPL, a.W5, K5, a.F, 64, tid, nthreads);
    stage_weight_block<PREC>(sW + 2 * C::W_BYTES, WSPL, a.W6, 64, 0, 64, tid, nthreads);
    if (NEXT_KIND == 2) {
        stage_weight_block<PREC>(sW + 3 * C::W_BYTES, WSPL, a.W1n, 64, 0, 64, tid, nthreads);
        stage_weight_block<PREC>(sW + 4 * C::W_BYTES, WSPL, a.W1n + 4096, 64, 0, 64, tid, nthreads);
        stage_weight_block<PREC>(sW + 5 * C::W_BYTES, WSPL, a.W1n + 8192, 64, 0, 64, tid, nthreads);
    } else {
        stage_weight_block<PREC>(sW + 3 * C::W_BYTES, WSPL, has_next ? a.W1n : nullptr, 130, 0, 64, tid, nthreads);
        stage_weight_block<PREC>(sW + 4 * C::W_BYTES, WSPL, has_next ? a.W1n : nullptr, 130, 64, 64, tid, nthreads);
    }
    if (tid < 64) {
        vec[tid] = a.b5[tid];
        vec[64 + tid] = a.b6[tid];
    }
    if (tid < 192) vec[128 + tid] = !has_next ? 0.0f : NEXT_KIND == 2 ? a.b1n[tid] : (tid < 64 ? a.b1n[tid] : 0.0f);
}

// The chain over the row groups mg = m_first, m_first + m_step, ... < m_end (rows >= m_end are zero operands and are not
// stored).  Called by threads 0 .. NT-1 of the CTA, after the weights are staged and visible; sA = the operand buffers
// (NodeCfg::A_REGION bytes), tmem = NTILE * 256 allocated columns, mbar = an initialised mbarrier at `phase`.
template <int PREC, int NT, bool FAST, int NEXT_KIND>
__device__ __forceinline__ void node_chain(const NodeArgs& a, uint8_t* sA, const uint8_t* sW, const float* vec, uint32_t tmem,
                                           uint64_t* mbar, uint32_t& phase, int64_t m_first, int64_t m_step, int64_t m_end,
                                           int tid, int bar_id) {
    using C = TcCfg<PREC>;
    using NC = NodeCfg<PREC, NEXT_KIND>;
    constexpr int NW = NT / 32, CQ = NW / 4, CW = 64 / CQ;
    constexpr int NTILE = NC::NTILE;
    constexpr bool TWO_BUF = NC::TWO_BUF;
    constexpr uint32_t ASPL = NC::ASPL, WSPL = NC::WSPL, ASTRIDE = NC::ASTRIDE, TCOLS = NC::TCOLS;
    uint8_t* sA2 = TWO_BUF ? sA + NC::ABUF : sA;
    const int warp = tid >> 5, lane = tid & 31;
    const bool has_next = a.W1n != nullptr;
    const int64_t M = m_end;
    const uint32_t a_addr = smem_u32(sA), a2_addr = smem_u32(sA2), w_addr = smem_u32(sW);
    const int q = warp & 3, cq = warp >> 2, erow = 32 * q + lane;
    const uint32_t t_lane = tmem + ((uint32_t)(32 * q) << 16);
    const int rsub = lane >> 3, kc8 = lane & 7;
    auto sync = [&] { asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "n"(NT) : "memory"); };

    // a [128 x 64] fp32 tile (rows m0.., `ncols` valid columns, row stride ld) as the A operand: every row load of the tile is
    // issued before the first is converted, so that the tile costs one load latency, not one per pass
    constexpr int NPASS = IS_TM / (4 * NW);
    auto load_rows = [&](float (&v)[NPASS][8], const float* __restrict__ src, int64_t ld, int ncols, int64_t m0, bool l2) {
        const bool vec4 = ncols == 64 && (ld & 3) == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0;
#pragma unroll
        for (int pass = 0; pass < NPASS; ++pass) {
            const int64_t m = m0 + pass * 4 * NW + warp * 4 + rsub;
            const float* rp = src + m * ld + 8 * kc8;
            if (vec4) {
                float4 x = make_float4(0.0f, 0.0f, 0.0f, 0.0f), y = x;
                if (m < M) {
                    // hn (l2): written by this CTA earlier in the fused layer launch, so read through L2, not the read-only path
                    x = l2 ? __ldcg(reinterpret_cast<const float4*>(rp)) : __ldg(reinterpret_cast<const float4*>(rp));
                    y = l2 ? __ldcg(reinterpret_cast<const float4*>(rp) + 1) : __ldg(reinterpret_cast<const float4*>(rp) + 1);
                }
                v[pass][0] = x.x; v[pass][1] = x.y; v[pass][2] = x.z; v[pass][3] = x.w;
                v[pass][4] = y.x; v[pass][5] = y.y; v[pass][6] = y.z; v[pass][7] = y.w;
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) v[pass][i] = (m < M && 8 * kc8 + i < ncols) ? __ldg(rp + i) : 0.0f;
            }
        }
    };
    auto store_rows = [&](uint8_t* __restrict__ dstA, const float (&v)[NPASS][8]) {
#pragma unroll
        for (int pass = 0; pass < NPASS; ++pass) store_operand8<PREC>(dstA, ASPL, pass * 4 * NW + warp * 4 + rsub, kc8, v[pass]);
    };
    // publish the staged operands, let one elected lane issue `issue_fn` (MMAs of one hand-over) and wait for them
    auto run_gemms = [&](auto&& issue_fn) {
        fence_async_smem();
        fence_before_sync();
        sync();
        if (tid < 32) {               // one elected lane of the converged warp issues (bare UTCHMMA, no election loop)
            if (elect_one()) {
                fence_after_sync();
                issue_fn();
                mma_commit(mbar);
            }
            __syncwarp();
            mbar_wait(mbar, phase);
        }
        phase ^= 1;
        sync();
        fence_after_sync();
    };
    auto run_gemm = [&](uint32_t tmem_d, uint32_t a_tile, int wblock, uint32_t ncols, uint32_t accumulate) {
        run_gemms([&] { issue_gemm<PREC, !FAST>(tmem_d, a_tile, ASPL, w_addr + wblock * C::W_BYTES, WSPL, ncols, accumulate); });
    };

    for (int64_t mg = m_first; mg < m_end; mg += m_step) {
        // ---- D1 = h W5h^T + hn W5n^T ---------------------------------------------------------------
        if (TWO_BUF) {
#pragma unroll
            for (int u = 0; u < NTILE; ++u) {
                float vh[NPASS][8], vn[NPASS][8];
                load_rows(vh, a.h, a.ldh, a.F, mg + u * IS_TM, false);
                load_rows(vn, a.hn, 64, 64, mg + u * IS_TM, true);
                store_rows(sA + u * ASTRIDE, vh);
                store_rows(sA2 + u * ASTRIDE, vn);
            }
            run_gemms([&] {
#pragma unroll
                for (int u = 0; u < NTILE; ++u) {
                    issue_gemm<PREC, !FAST>(tmem + u * TCOLS, a_addr + u * ASTRIDE, ASPL, w_addr + 0 * C::W_BYTES, WSPL, 64, 0);
                    issue_gemm<PREC, !FAST>(tmem + u * TCOLS, a2_addr + u * ASTRIDE, ASPL, w_addr + 1 * C::W_BYTES, WSPL, 64, 1);
                }
            });
        } else {
            float v[NPASS][8];
            load_rows(v, a.h, a.ldh, a.F, mg, false);
            store_rows(sA, v);
            run_gemm(tmem, a_addr, 0, 64, 0);
            load_rows(v, a.hn, 64, 64, mg, true);
            store_rows(sA, v);
            run_gemm(tmem, a_addr, 1, 64, 1);
        }
        // ---- t5 = silu(D1 + b5) -> A operand ; D2 = t5 W6^T -------------------------------------------
#pragma unroll
        for (int u = 0; u < NTILE; ++u) {
            float z[CW];
            tmem_ld<CW>(t_lane + u * TCOLS + CW * cq, z);
#pragma unroll
            for (int g = 0; g < CW / 8; ++g) {
                float v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = act<PREC, FAST>(z[8 * g + i] + vec[CW * cq + 8 * g + i]);
                store_operand8<PREC>(sA + u * ASTRIDE, ASPL, erow, (CW / 8) * cq + g, v);
            }
        }
        run_gemms([&] {
#pragma unroll
            for (int u = 0; u < NTILE; ++u)
                issue_gemm<PREC, !FAST>(tmem + u * TCOLS + 64, a_addr + u * ASTRIDE, ASPL, w_addr + 2 * C::W_BYTES, WSPL, 64, 0);
        });
        // ---- h' = D2 + b6 -> global (+ A operand for the next layer's P/Q) ------------------------------
#pragma unroll
        for (int u = 0; u < NTILE; ++u) {
            float z[CW];
            tmem_ld<CW>(t_lane + u * TCOLS + 64 + CW * cq, z);
            const int64_t m = mg + u * IS_TM + erow;
#pragma unroll
            for (int g = 0; g < CW / 8; ++g) {
                float v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = z[8 * g + i] + vec[64 + CW * cq + 8 * g + i];
                if (m < M) stg256(a.h_out + m * 64 + CW * cq + 8 * g, v);
                if (has_next) store_operand8<PREC>(sA2 + u * ASTRIDE, ASPL, erow, (CW / 8) * cq + g, v);
            }
        }
        if (has_next && NEXT_KIND == 2) {
            // ---- D3 = h' [Wq; Wk; Wv]^T (N = 192: blocks 3..5), written over the dead accumulators D1 / D2 ----
            run_gemms([&] {
#pragma unroll
                for (int u = 0; u < NTILE; ++u)
                    issue_gemm<PREC, !FAST>(tmem + u * TCOLS, a2_addr + u * ASTRIDE, ASPL, w_addr + 3 * C::W_BYTES, WSPL, 192, 0);
            });
#pragma unroll
            for (int u = 0; u < NTILE; ++u) {
                const int64_t m = mg + u * IS_TM + erow;
#pragma unroll
                for (int part = 0; part < 3; ++part) {
                    float z[CW];
                    tmem_ld<CW>(t_lane + u * TCOLS + 64 * part + CW * cq, z);
                    if (m < M) {
#pragma unroll
                        for (int g = 0; g < CW / 8; ++g) {
                            const int c = 64 * part + CW * cq + 8 * g;
                            float o[8];
#pragma unroll
                            for (int i = 0; i < 8; ++i) o[i] = z[8 * g + i] + vec[128 + c + i];
                            stg256(a.PQn + m * 192 + c, o);
                        }
                    }
                }
            }
        } else if (has_next) {
            // ---- D3 = h' [Ws'; Wd']^T (N = 128: weight blocks 3 and 4 are contiguous row groups) -------
            run_gemms([&] {
#pragma unroll
                for (int u = 0; u < NTILE; ++u)
                    issue_gemm<PREC, !FAST>(tmem + u * TCOLS + 128, a2_addr + u * ASTRIDE, ASPL, w_addr + 3 * C::W_BYTES, WSPL, 128, 0);
            });
#pragma unroll
            for (int u = 0; u < NTILE; ++u) {
                const int64_t m = mg + u * IS_TM + erow;
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    float z[CW];
                    tmem_ld<CW>(t_lane + u * TCOLS + 128 + 64 * half + CW * cq, z);
                    if (m < M) {
#pragma unroll
                        for (int g = 0; g < CW / 8; ++g) {
                            const int c = CW * cq + 8 * g;
                            float o[8];
#pragma unroll
                            for (int i = 0; i < 8; ++i) o[i] = z[8 * g + i] + (half ? vec[128 + c + i] : 0.0f);
                            stg256(a.PQn + m * 128 + 64 * half + c, o);
                        }
                    }
                }
            }
        }
        fence_before_sync();      // TMEM reads of this group are ordered before the next group's MMAs
    }
}

}  // namespace is
