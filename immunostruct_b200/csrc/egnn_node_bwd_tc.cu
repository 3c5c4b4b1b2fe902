// Node-side backward of an EGNN layer on the tcgen05 tensor cores (bf16x3 split, fp32-accurate).
//
// Same contracts, outputs and per-CTA partial layouts as the SIMT kernels node_post_bwd_kernel / node_pre_bwd_kernel
// (egnn.cu), which top out at ~45 % issue utilisation: an fp32 register-tiled GEMM fed from shared memory needs
// 12 LDS.128 per 128 FFMA, i.e. it is shared-memory-bandwidth bound at two thirds of the FMA peak (ncu, round 1).
//
//   node_post backward (reference: EGNNConv.node_mlp, h' = W6 silu(W5 [h | hn] + b5) + b6), per 128-node tile:
//     z5  = h W5h^T + hn W5n^T            MMA (recompute)          t5 = silu(z5 + b5), d5 = silu'(z5 + b5)
//     gt5 = gh' W6                         MMA (B = W6 read MN-major = transposed view)
//     gW6 += gh'^T t5                      MMA, M = 64, both operands MN-major, accumulates in TMEM over the CTA's tiles
//     gz5 = gt5 * d5 ;  gb5 += colsum(gz5) ;  gb6 += colsum(gh')
//     ghn = gz5 W5n ,  gh_direct = gz5 W5h MMA (transposed views of the forward weight tiles)
//     gW5n += gz5^T hn ,  gW5h += gz5^T h  MMA, M = 64, TMEM accumulators
//   node_pre backward (P = h Ws^T, Q = h Wd^T + b1), per 128-node tile:
//     gP[s] = sum over out-edges of gz1 (CSC gather, batched loads) ;  gx = gx_out + gxd + sum over out-edges of gD
//     gh  = gh_direct + gP Ws + gQ Wd      MMA (transposed views)
//     gWs += gP^T h ,  gWd += gQ^T h       MMA, M = 64, TMEM accumulators ;  gb1 += colsum(gQ)
//
// Three 48 KB operand tiles (unpadded canonical K-major, three bf16 terms) + the weight tiles fill the shared memory,
// so the h rows of node_post are staged twice (once for the recompute, once for gW5h).  One 512-thread CTA per SM,
// lock-step phases, MMAs issued by an elected lane of warp 0.  Deterministic: fixed summation order everywhere.
#include "tc_common.cuh"

namespace is {
namespace nb {
constexpr int NT = 512, NW = NT / 32, CW = 16;          // 16 warps: TMEM lane quarter q = warp % 4, column quarter cq = warp / 4
constexpr uint32_t LBO = 128, SBO = 8 * LBO, T_BYTES = 16 * SBO;     // 128-row operand tile, one split term (16 KB)
constexpr uint32_t W_BYTES = 8 * 8 * umma::kLBO_W;                   // 64-row weight tile, one split term (8 KB)

struct Geom { uint32_t base, split, step, lbo, sbo; };  // operand view: start, split-term stride, K-step advance, LBO, SBO
__device__ __forceinline__ Geom act_k(uint32_t base) { return {base, T_BYTES, 2 * LBO, LBO, SBO}; }          // [128 rows] x K = features
__device__ __forceinline__ Geom act_t(uint32_t base) { return {base, T_BYTES, 2 * SBO, SBO, LBO}; }          // transposed: K = rows
__device__ __forceinline__ Geom wgt_k(uint32_t base) { return {base, W_BYTES, 2 * umma::kLBO_W, umma::kLBO_W, 8 * umma::kLBO_W}; }
__device__ __forceinline__ Geom wgt_t(uint32_t base) { return {base, W_BYTES, 2 * 8 * umma::kLBO_W, 8 * umma::kLBO_W, umma::kLBO_W}; }

// D (+)= A B^T in the bf16x3 split: six partial products, smallest first (ONE elected thread)
__device__ __forceinline__ void issue6(uint32_t tmem_d, const Geom& a, const Geom& b, int nks, uint32_t idesc, uint32_t accumulate) {
    using namespace umma;
    const uint32_t ta[6] = {2, 0, 1, 1, 0, 0}, tb[6] = {0, 2, 1, 0, 1, 0};
    uint32_t acc = accumulate;
#pragma unroll
    for (int t = 0; t < 6; ++t)
#pragma unroll 8
        for (int ks = 0; ks < nks; ++ks) {
            mma_bf16(tmem_d, make_smem_desc(a.base + ta[t] * a.split + ks * a.step, a.lbo, a.sbo),
                     make_smem_desc(b.base + tb[t] * b.split + ks * b.step, b.lbo, b.sbo), idesc, acc);
            acc = 1;
        }
}

// rows m0.. of a [*, ncols <= 64] fp32 matrix (row stride ld) -> this thread's two 8-wide chunks; rows >= M / columns
// >= ncols read as zero.  Staging map: warp w owns rows 8w..8w+7; a quarter-warp covers rows r4 + 4 (chunk parity ^ u)
// for two adjacent chunks (conflict-free 16-byte stores into the unpadded tile).
__device__ __forceinline__ void load2(float (&v)[2][8], const float* __restrict__ src, int64_t ld, int ncols, int64_t m0, int64_t M,
                                      int warp, int r4, int kc) {
    const bool v8 = ncols == 64 && (ld & 7) == 0 && (reinterpret_cast<uintptr_t>(src) & 31) == 0;
#pragma unroll
    for (int u = 0; u < 2; ++u) {
        const int64_t m = m0 + 8 * warp + r4 + 4 * ((kc & 1) ^ u);
#pragma unroll
        for (int i = 0; i < 8; ++i) v[u][i] = 0.0f;
        if (m < M) {
            const float* rp = src + m * ld + 8 * kc;
            if (v8) {
                ldg256(rp, v[u]);
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) v[u][i] = (8 * kc + i < ncols) ? __ldg(rp + i) : 0.0f;
            }
        }
    }
}
__device__ __forceinline__ void store2(uint8_t* __restrict__ tile, const float (&v)[2][8], int warp, int r4, int kc) {
#pragma unroll
    for (int u = 0; u < 2; ++u) {
        const int row = 8 * warp + r4 + 4 * ((kc & 1) ^ u);
        store_chunk8<PREC_BF16X3>(tile + (row >> 3) * SBO + (row & 7) * 16 + kc * LBO, T_BYTES, v[u]);
    }
}
__device__ __forceinline__ uint8_t* chunk_at(uint8_t* tile, int row, int chunk) { return tile + (row >> 3) * SBO + (row & 7) * 16 + chunk * LBO; }

// The 16 columns c0 .. c0 + 15 of one row of an [M, F] fp32 matrix, F = 20 (the layer-0 input features): 80-byte rows are
// only 16-byte aligned, so 128-bit accesses, and only the columns below F (c0 = 16 holds 16 .. 19).
__device__ __forceinline__ void load_row16_narrow(float (&v)[CW], const float* __restrict__ row, int c0, int F) {
#pragma unroll
    for (int j = 0; j < CW / 4; ++j)
        if (c0 + 4 * j < F) {
            const float4 a = __ldg(reinterpret_cast<const float4*>(row + c0 + 4 * j));
            v[4 * j] = a.x; v[4 * j + 1] = a.y; v[4 * j + 2] = a.z; v[4 * j + 3] = a.w;
        }
}
__device__ __forceinline__ void store_row16_narrow(float* __restrict__ row, const float (&v)[CW], int c0, int F) {
#pragma unroll
    for (int j = 0; j < CW / 4; ++j)
        if (c0 + 4 * j < F)
            *reinterpret_cast<float4*>(row + c0 + 4 * j) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
}

// sum over the warp's 32 rows of 16 per-lane column values; afterwards lane L holds the total of column (L >> 1) & 15
__device__ __forceinline__ float colsum16(const float (&v)[16], int lane) {
    float w8[8], w4[4], w2[2];
    const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4, b1 = lane & 2;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const float send = b4 ? v[i] : v[i + 8], keep = b4 ? v[i + 8] : v[i];
        w8[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float send = b3 ? w8[i] : w8[i + 4], keep = b3 ? w8[i + 4] : w8[i];
        w4[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const float send = b2 ? w4[i] : w4[i + 2], keep = b2 ? w4[i + 2] : w4[i];
        w2[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
    const float send = b1 ? w2[0] : w2[1], keep = b1 ? w2[1] : w2[0];
    float s = keep + __shfl_xor_sync(0xffffffffu, send, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    return s;
}
// accurate SiLU and derivative (same arithmetic as the SIMT kernels up to the approximate reciprocal, 1 ulp)
__device__ __forceinline__ void silu_both_acc(float z, float& y, float& dy) {
    float s;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(s) : "f"(1.0f + exp_comp(-z)));
    y = z * s;
    dy = s * (1.0f + z * (1.0f - s));
}
}  // namespace nb

// =====================================================================================================================
__global__ void __launch_bounds__(nb::NT, 1)
node_post_bwd_tc_kernel(const float* __restrict__ gh_out, const float* __restrict__ h, int64_t ldh, int F,
                        const float* __restrict__ hn, const float* __restrict__ W5, const float* __restrict__ b5,
                        const float* __restrict__ W6, float* __restrict__ gh_direct /* [M,F] or null */,
                        float* __restrict__ ghn, float* __restrict__ partials, int64_t M) {
    using namespace nb;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    uint8_t* sX = smem_raw;                               // [3][T_BYTES]  hn, later h (for gW5h)
    uint8_t* sT = sX + 3 * T_BYTES;                       // [3][T_BYTES]  h (recompute), then t5
    uint8_t* sG = sT + 3 * T_BYTES;                       // [3][T_BYTES]  gh', then gz5
    uint8_t* sW = sG + 3 * T_BYTES;                       // [3 blocks][3][W_BYTES]: W5h | W5n | W6 (block stride 3 * W_BYTES)
    float* vec = reinterpret_cast<float*>(sW + 9 * W_BYTES);     // b5 [64]
    float* red = vec + 64;                                // [16 warps][16]
    __shared__ __align__(8) uint64_t mbar, mbar_wg;
    __shared__ uint32_t s_tmem;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int K5 = F + 64;
    if (warp == 0) tmem_alloc(&s_tmem, 512);
    if (tid == 32) { mbar_init(&mbar, 1); mbar_init(&mbar_wg, 1); }
    stage_weight_block<PREC_BF16X3>(sW + 0 * 3 * W_BYTES, W_BYTES, W5, K5, 0, F, tid, NT);
    stage_weight_block<PREC_BF16X3>(sW + 1 * 3 * W_BYTES, W_BYTES, W5, K5, F, 64, tid, NT);
    stage_weight_block<PREC_BF16X3>(sW + 2 * 3 * W_BYTES, W_BYTES, W6, 64, 0, 64, tid, NT);
    if (tid < 64) vec[tid] = b5[tid];
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = s_tmem;
    // TMEM columns: D1 z5 [0,64) | D2 gt5 [64,128) | D3 ghn [128,192) | D4 gh_direct [192,256) | DW6 [256,320) | DW5h [320,384) | DW5n [384,448)
    const int q = warp & 3, cq = warp >> 2, erow = 32 * q + lane;
    const uint32_t t_lane = tmem + ((uint32_t)(32 * q) << 16) + CW * cq;
    const int r4 = lane & 3, kc = lane >> 2;
    const Geom gX = act_k(smem_u32(sX)), gT = act_k(smem_u32(sT)), gG = act_k(smem_u32(sG));
    const Geom gXt = act_t(smem_u32(sX)), gTt = act_t(smem_u32(sT)), gGt = act_t(smem_u32(sG));
    const Geom w5h = wgt_k(smem_u32(sW)), w5n = wgt_k(smem_u32(sW + 3 * W_BYTES));
    const Geom w5ht = wgt_t(smem_u32(sW)), w5nt = wgt_t(smem_u32(sW + 3 * W_BYTES)), w6t = wgt_t(smem_u32(sW + 6 * W_BYTES));
    const uint32_t id_fwd = umma::make_instr_desc(1u, 128, 64, 0, 0);
    const uint32_t id_dgrad = umma::make_instr_desc(1u, 128, 64, 0, 1);
    const uint32_t id_wgrad = umma::make_instr_desc(1u, 64, 64, 1, 1);
    uint32_t phase = 0, phase_wg = 0, started = 0;
    bool wg_pending = false;
    float acc_gb5 = 0.0f;                 // column (lane >> 1) & 15 of this warp's column quarter
    float gb6[8];                         // columns 8 kc .. 8 kc + 7 over this thread's staged rows
#pragma unroll
    for (int i = 0; i < 8; ++i) gb6[i] = 0.0f;

    auto publish = [&]() { fence_async_smem(); fence_before_sync(); __syncthreads(); };
    auto wait_data = [&]() { mbar_wait(&mbar, phase); phase ^= 1; fence_after_sync(); };
    auto wait_wg = [&]() { if (wg_pending) { mbar_wait(&mbar_wg, phase_wg); phase_wg ^= 1; wg_pending = false; fence_after_sync(); } };

    const int64_t ntiles = (M + IS_TM - 1) / IS_TM;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int64_t m0 = t * IS_TM;
        float v[2][8];
        wait_wg();                                     // gW5h of the previous tile still reads X and G
        // ---- z5 = h W5h^T + hn W5n^T   (h in T, hn in X: X survives for gW5n) ---------------------------------------
        load2(v, h, ldh, F, m0, M, warp, r4, kc);
        store2(sT, v, warp, r4, kc);
        load2(v, hn, 64, 64, m0, M, warp, r4, kc);
        store2(sX, v, warp, r4, kc);
        publish();
        if (warp == 0) {
            if (elect_one()) {
                fence_after_sync();
                issue6(tmem + 0, gT, w5h, 4, id_fwd, 0);
                issue6(tmem + 0, gX, w5n, 4, id_fwd, 1);
                mma_commit(&mbar);
            }
            __syncwarp();
        }
        load2(v, gh_out, 64, 64, m0, M, warp, r4, kc);      // gh' rows travel while the MMAs run
        wait_data();
        // ---- t5, d5 ; t5 -> T (h is no longer needed there) ------------------------------------------------------------
        float d5[CW];
        {
            float z[CW], y[CW];
            tmem_ld<CW>(t_lane, z);
#pragma unroll
            for (int i = 0; i < CW; ++i) silu_both_acc(z[i] + vec[CW * cq + i], y[i], d5[i]);
#pragma unroll
            for (int g = 0; g < CW / 8; ++g) {
                const float y8[8] = {y[8 * g], y[8 * g + 1], y[8 * g + 2], y[8 * g + 3], y[8 * g + 4], y[8 * g + 5], y[8 * g + 6], y[8 * g + 7]};
                store_chunk8<PREC_BF16X3>(chunk_at(sT, erow, 2 * cq + g), T_BYTES, y8);
            }
        }
        // ---- G = gh' ; gb6 += colsum(gh') ; gt5 = gh' W6 ; gW6 += gh'^T t5 -------------------------------------------
#pragma unroll
        for (int u = 0; u < 2; ++u)
#pragma unroll
            for (int i = 0; i < 8; ++i) gb6[i] += v[u][i];
        store2(sG, v, warp, r4, kc);
        publish();
        if (warp == 0) {
            if (elect_one()) {
                fence_after_sync();
                issue6(tmem + 64, gG, w6t, 4, id_dgrad, 0);
                mma_commit(&mbar);
                issue6(tmem + 256, gGt, gTt, 8, id_wgrad, started);
                mma_commit(&mbar_wg);
            }
            __syncwarp();
        }
        wg_pending = true;
        wait_data();
        // ---- gz5 = gt5 * d5 ; gb5 += colsum(gz5) ; gz5 -> G (after gW6 has finished reading G and T) -----------------
        {
            float gz[CW];
            tmem_ld<CW>(t_lane + 64, gz);
#pragma unroll
            for (int i = 0; i < CW; ++i) gz[i] *= d5[i];
            acc_gb5 += colsum16(gz, lane);
            wait_wg();
#pragma unroll
            for (int g = 0; g < CW / 8; ++g) {
                const float g8[8] = {gz[8 * g], gz[8 * g + 1], gz[8 * g + 2], gz[8 * g + 3], gz[8 * g + 4], gz[8 * g + 5], gz[8 * g + 6], gz[8 * g + 7]};
                store_chunk8<PREC_BF16X3>(chunk_at(sG, erow, 2 * cq + g), T_BYTES, g8);
            }
        }
        publish();
        // ---- ghn = gz5 W5n ; gh_direct = gz5 W5h ; gW5n += gz5^T hn ---------------------------------------------------
        if (warp == 0) {
            if (elect_one()) {
                fence_after_sync();
                issue6(tmem + 128, gG, w5nt, 4, id_dgrad, 0);
                if (gh_direct) issue6(tmem + 192, gG, w5ht, 4, id_dgrad, 0);
                mma_commit(&mbar);
                issue6(tmem + 384, gGt, gXt, 8, id_wgrad, started);
                mma_commit(&mbar_wg);
            }
            __syncwarp();
        }
        wg_pending = true;
        load2(v, h, ldh, F, m0, M, warp, r4, kc);            // h again (for gW5h), in flight under the MMAs
        wait_data();
        {
            const int64_t m = m0 + erow;
            float z[CW];
            tmem_ld<CW>(t_lane + 128, z);
            if (m < M) {
#pragma unroll
                for (int g = 0; g < CW / 8; ++g) {
                    const float o[8] = {z[8 * g], z[8 * g + 1], z[8 * g + 2], z[8 * g + 3], z[8 * g + 4], z[8 * g + 5], z[8 * g + 6], z[8 * g + 7]};
                    stg256(ghn + m * 64 + CW * cq + 8 * g, o);
                }
            }
            if (gh_direct) {
                // (F = 20: W5h was staged zero-padded beyond column F, so columns F .. 63 of the product are zero)
                tmem_ld<CW>(t_lane + 192, z);
                if (m < M && F == 64) {
#pragma unroll
                    for (int g = 0; g < CW / 8; ++g) {
                        const float o[8] = {z[8 * g], z[8 * g + 1], z[8 * g + 2], z[8 * g + 3], z[8 * g + 4], z[8 * g + 5], z[8 * g + 6], z[8 * g + 7]};
                        stg256(gh_direct + m * 64 + CW * cq + 8 * g, o);
                    }
                } else if (m < M) {
                    store_row16_narrow(gh_direct + m * F, z, CW * cq, F);
                }
            }
        }
        // ---- gW5h += gz5^T h (X is free once gW5n has read hn) ------------------------------------------------------------
        wait_wg();
        store2(sX, v, warp, r4, kc);
        publish();
        if (warp == 0) {
            if (elect_one()) {
                fence_after_sync();
                issue6(tmem + 320, gGt, gXt, 8, id_wgrad, started);
                mma_commit(&mbar_wg);
            }
            __syncwarp();
        }
        wg_pending = true;
        started = 1;
    }

    // ---- per-CTA partials: [gW5 64 x K5][gb5 64][gW6 64 x 64][gb6 64] -----------------------------------------------------
    wait_wg();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    float* P = partials + (size_t)blockIdx.x * (64 * K5 + 64 + 4096 + 64);
    {
        // M = 64 accumulators: row r lives in TMEM lane 32 (r / 16) + r % 16 -> lanes 0..15 of warp quarter q hold rows 16 q + lane
        float w[CW];
        const int o = 16 * q + lane;
        if (started) tmem_ld<CW>(t_lane + 320, w);
        if (lane < 16) {
#pragma unroll
            for (int i = 0; i < CW; ++i) {
                const int k = CW * cq + i;
                if (k < F) P[o * K5 + k] = started ? w[i] : 0.0f;
            }
        }
        if (started) tmem_ld<CW>(t_lane + 384, w);
        if (lane < 16) {
#pragma unroll
            for (int i = 0; i < CW; ++i) P[o * K5 + F + CW * cq + i] = started ? w[i] : 0.0f;
        }
        if (started) tmem_ld<CW>(t_lane + 256, w);
        if (lane < 16) {
#pragma unroll
            for (int i = 0; i < CW; ++i) P[64 * K5 + 64 + o * 64 + CW * cq + i] = started ? w[i] : 0.0f;
        }
    }
    // gb5: warps (q, cq) hold column (lane >> 1) & 15 of quarter cq
    if ((lane & 1) == 0) red[warp * 16 + (lane >> 1)] = acc_gb5;
    __syncthreads();
    if (tid < 64) {
        const int cqq = tid >> 4, col = tid & 15;
        float s = 0.0f;
#pragma unroll
        for (int qq = 0; qq < 4; ++qq) s += red[(cqq * 4 + qq) * 16 + col];
        P[64 * K5 + tid] = s;
    }
    // gb6: thread (warp, r4, kc) holds columns 8 kc .. 8 kc + 7 over its rows -> scratch [NT][8] in the (idle) X tile
    float* scr = reinterpret_cast<float*>(sX);
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; ++i) scr[tid * 8 + i] = gb6[i];
    __syncthreads();
    if (tid < 64) {
        const int kcc = tid >> 3, i = tid & 7;
        float s = 0.0f;
        for (int w = 0; w < NW; ++w)
#pragma unroll
            for (int r = 0; r < 4; ++r) s += scr[(w * 32 + kcc * 4 + r) * 8 + i];
        P[64 * K5 + 64 + 4096 + tid] = s;
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}


// =====================================================================================================================
__global__ void __launch_bounds__(nb::NT, 1)
node_pre_bwd_tc_kernel(const float* __restrict__ gz1, const float* __restrict__ gQ, const float* __restrict__ gD,
                       const float* __restrict__ gxd, const float* __restrict__ gx_out /* or null */,
                       const float* __restrict__ gh_direct /* [M,F] or null */,
                       const int* __restrict__ outptr, const int* __restrict__ csc_pos,
                       const float* __restrict__ h, int64_t ldh, int F, const float* __restrict__ W1,
                       float* __restrict__ gh /* [M,F] or null */, float* __restrict__ gx /* [M,3] or null */,
                       float* __restrict__ partials, int64_t M) {
    using namespace nb;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    uint8_t* sP = smem_raw;                               // [3][T_BYTES]  gP (source-side sums of gz1)
    uint8_t* sQ = sP + 3 * T_BYTES;                       // [3][T_BYTES]  gQ
    uint8_t* sH = sQ + 3 * T_BYTES;                       // [3][T_BYTES]  h
    uint8_t* sW = sH + 3 * T_BYTES;                       // [2 blocks][3][W_BYTES]: Ws | Wd
    float* sS = reinterpret_cast<float*>(sW + 6 * W_BYTES);   // [NW][8][64] fp32 staging of the gathered sums
    __shared__ __align__(8) uint64_t mbar, mbar_wg;
    __shared__ uint32_t s_tmem;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ldw = 2 * F + 2;
    if (warp == 0) tmem_alloc(&s_tmem, 256);
    if (tid == 32) { mbar_init(&mbar, 1); mbar_init(&mbar_wg, 1); }
    stage_weight_block<PREC_BF16X3>(sW, W_BYTES, gh ? W1 : nullptr, ldw, 0, F, tid, NT);
    stage_weight_block<PREC_BF16X3>(sW + 3 * W_BYTES, W_BYTES, gh ? W1 : nullptr, ldw, F, F, tid, NT);
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = s_tmem;
    // TMEM columns: D gh [0,64) | DWs [64,128) | DWd [128,192)
    const int q = warp & 3, cq = warp >> 2, erow = 32 * q + lane;
    const uint32_t t_lane = tmem + ((uint32_t)(32 * q) << 16) + CW * cq;
    const int r4 = lane & 3, kc = lane >> 2;
    const Geom gP = act_k(smem_u32(sP)), gQk = act_k(smem_u32(sQ));
    const Geom gPt = act_t(smem_u32(sP)), gQt = act_t(smem_u32(sQ)), gHt = act_t(smem_u32(sH));
    const Geom wst = wgt_t(smem_u32(sW)), wdt = wgt_t(smem_u32(sW + 3 * W_BYTES));
    const uint32_t id_dgrad = umma::make_instr_desc(1u, 128, 64, 0, 1);
    const uint32_t id_wgrad = umma::make_instr_desc(1u, 64, 64, 1, 1);
    uint32_t phase = 0, phase_wg = 0, started = 0;
    bool wg_pending = false;
    float gb1[8];                         // columns 8 kc .. 8 kc + 7 of gQ over this thread's staged rows
#pragma unroll
    for (int i = 0; i < 8; ++i) gb1[i] = 0.0f;

    // The head of the gather's dependent chain (CSC range of this warp's eight nodes -> first 32 CSC positions) is fetched
    // one tile ahead, under the MMAs and the epilogue of the tile before.
    int pf_ptr = 0, pf_pos = 0;
    auto prefetch_run = [&](int64_t m0n) {
        const int64_t n0 = m0n + (IS_TM / NW) * warp;
        pf_ptr = lane <= IS_TM / NW ? __ldg(outptr + (n0 + lane < M ? n0 + lane : M)) : 0;
        const int qb = __shfl_sync(0xffffffffu, pf_ptr, 0), qe = __shfl_sync(0xffffffffu, pf_ptr, IS_TM / NW);
        pf_pos = qb + lane < qe ? __ldg(csc_pos + qb + lane) : 0;
    };
    const int64_t ntiles = (M + IS_TM - 1) / IS_TM;
    prefetch_run((int64_t)blockIdx.x * IS_TM);
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int64_t m0 = t * IS_TM;
        if (wg_pending) { mbar_wait(&mbar_wg, phase_wg); phase_wg ^= 1; wg_pending = false; fence_after_sync(); }
        // ---- gQ and h rows travel while the CSC gather runs -------------------------------------------------------------
        float vq[2][8], vh[2][8];
        load2(vq, gQ, 64, 64, m0, M, warp, r4, kc);
        load2(vh, h, ldh, F, m0, M, warp, r4, kc);
        // ---- source-side reduction through the CSC transpose.  A warp owns EIGHT CONSECUTIVE nodes, so their CSC ranges
        // form one contiguous run of positions; the run is walked GB rows at a time with all GB row loads in flight and the
        // next 32 positions already fetched, and a node's sum is flushed when the walk crosses its end.  Each node's sum
        // still starts at zero and adds its rows in ascending CSC position (= the SIMT kernel's order: bit-identical). ----
        {
            constexpr int NPW = IS_TM / NW;                    // 8
            constexpr int GB = 16;                             // row loads in flight per warp
            const int r0 = NPW * warp;
            const int64_t n0 = m0 + r0;
            const bool lane_x = gx != nullptr && lane < 3;
            const float* gz_lane = gz1 + 2 * lane;
            const float* gd_lane = gD + lane;
            const int my_ptr = pf_ptr;                         // fetched under the previous tile's MMAs
            float my_gx0 = 0.0f;                               // lanes 0..23: the eight nodes' direct coordinate gradients
            if (gx != nullptr && lane < 3 * NPW && n0 * 3 + lane < M * 3) {
                my_gx0 = __ldg(gxd + n0 * 3 + lane);
                if (gx_out) my_gx0 += __ldg(gx_out + n0 * 3 + lane);
            }
            const int qbeg = __shfl_sync(0xffffffffu, my_ptr, 0), qend = __shfl_sync(0xffffffffu, my_ptr, NPW);
            int node_i = 0, q_next = __shfl_sync(0xffffffffu, my_ptr, 1);
            float2 s = make_float2(0.f, 0.f);
            float sx = __shfl_sync(0xffffffffu, my_gx0, lane % 3);
            // A finished sum goes to the warp's fp32 staging rows (lane L holds features 2L, 2L+1; the 8-float chunk index is
            // XORed with the row so that both this store and the row-per-lane read below are bank-conflict free); the operand
            // split into sP happens once per tile with all 32 lanes busy.
            float* stage = sS + warp * (NPW * 64);
            auto flush = [&]() {
                const int r = r0 + node_i;
                if (lane_x && m0 + r < M) gx[(m0 + r) * 3 + lane] = sx;
                *reinterpret_cast<float2*>(stage + node_i * 64 + (((lane >> 2) ^ node_i) & 7) * 8 + (lane & 3) * 2) = s;
                ++node_i;
                s = make_float2(0.f, 0.f);
                sx = __shfl_sync(0xffffffffu, my_gx0, (3 * node_i + lane % 3) & 31);
                q_next = __shfl_sync(0xffffffffu, my_ptr, (node_i + 1) & 31);
            };
            int pos_next = pf_pos;
            for (int c0 = qbeg; c0 < qend; c0 += 32) {
                const int my_pos = pos_next;
                if (c0 + 32 + lane < qend) pos_next = __ldg(csc_pos + c0 + 32 + lane);
                const int cnt = min(32, qend - c0);
                for (int j0 = 0; j0 < cnt; j0 += GB) {
                    float2 v[GB];
                    float d[GB];
#pragma unroll
                    for (int u = 0; u < GB; ++u) {
                        // past the end of the run the position is 0: row 0 exists (the run is not empty) and is not summed,
                        // so the GB loads issue back to back with no branch between them
                        const int pos = __shfl_sync(0xffffffffu, my_pos, (j0 + u) & 31);
                        v[u] = __ldg(reinterpret_cast<const float2*>(gz_lane + (size_t)(uint32_t)pos * 64));
                        d[u] = lane_x ? __ldg(gd_lane + (size_t)(uint32_t)pos * 3) : 0.0f;
                    }
#pragma unroll
                    for (int u = 0; u < GB; ++u) {
                        if (j0 + u < cnt) {
                            while (c0 + j0 + u >= q_next) flush();      // warp-uniform; also passes over edge-less nodes
                            s.x += v[u].x; s.y += v[u].y; sx += d[u];
                        }
                    }
                }
            }
            while (node_i < NPW) flush();
            __syncwarp();
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int row = lane & 7, cc = (lane >> 3) + 4 * u;
                const float4* sp = reinterpret_cast<const float4*>(stage + row * 64 + ((cc ^ row) & 7) * 8);
                const float4 a = sp[0], b = sp[1];
                const float c8[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
                store_chunk8<PREC_BF16X3>(chunk_at(sP, r0 + row, cc), T_BYTES, c8);
            }
            __syncwarp();
        }
#pragma unroll
        for (int u = 0; u < 2; ++u)
#pragma unroll
            for (int i = 0; i < 8; ++i) gb1[i] += vq[u][i];
        store2(sQ, vq, warp, r4, kc);
        store2(sH, vh, warp, r4, kc);
        fence_async_smem();
        fence_before_sync();
        __syncthreads();
        if (warp == 0) {
            if (elect_one()) {
                fence_after_sync();
                if (gh) {
                    issue6(tmem + 0, gP, wst, 4, id_dgrad, 0);
                    issue6(tmem + 0, gQk, wdt, 4, id_dgrad, 1);
                    mma_commit(&mbar);
                }
                issue6(tmem + 64, gPt, gHt, 8, id_wgrad, started);
                issue6(tmem + 128, gQt, gHt, 8, id_wgrad, started);
                mma_commit(&mbar_wg);
            }
            __syncwarp();
        }
        wg_pending = true;
        started = 1;
        prefetch_run((t + gridDim.x) * IS_TM);
        if (gh) {
            const int64_t m = m0 + erow;
            float g[CW];
#pragma unroll
            for (int i = 0; i < CW; ++i) g[i] = 0.0f;
            if (gh_direct && m < M) {                        // in flight under the MMAs
                if (F == 64) {
                    ldg256(gh_direct + m * 64 + CW * cq, *reinterpret_cast<float(*)[8]>(g));
                    ldg256(gh_direct + m * 64 + CW * cq + 8, *reinterpret_cast<float(*)[8]>(g + 8));
                } else {
                    load_row16_narrow(g, gh_direct + m * F, CW * cq, F);
                }
            }
            mbar_wait(&mbar, phase);
            phase ^= 1;
            fence_after_sync();
            float z[CW];
            tmem_ld<CW>(t_lane, z);
            if (m < M && F == 64) {
#pragma unroll
                for (int gg = 0; gg < CW / 8; ++gg) {
                    float o[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) o[i] = z[8 * gg + i] + g[8 * gg + i];
                    stg256(gh + m * 64 + CW * cq + 8 * gg, o);
                }
            } else if (m < M) {                              // F = 20: Ws / Wd staged zero-padded beyond column F
#pragma unroll
                for (int i = 0; i < CW; ++i) z[i] += g[i];
                store_row16_narrow(gh + m * F, z, CW * cq, F);
            }
            fence_before_sync();
        }
    }

    // ---- per-CTA partials: [gWs 64 x F][gWd 64 x F][gb1 64] ----------------------------------------------------------------
    if (wg_pending) { mbar_wait(&mbar_wg, phase_wg); fence_after_sync(); }
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    float* P = partials + (size_t)blockIdx.x * (2 * 64 * F + 64);
    {
        float w[CW];
        const int o = 16 * q + lane;                          // M = 64 accumulator: row r in TMEM lane 32 (r / 16) + r % 16
        if (started) tmem_ld<CW>(t_lane + 64, w);
        if (lane < 16) {
#pragma unroll
            for (int i = 0; i < CW; ++i) {
                const int k = CW * cq + i;
                if (k < F) P[o * F + k] = started ? w[i] : 0.0f;
            }
        }
        if (started) tmem_ld<CW>(t_lane + 128, w);
        if (lane < 16) {
#pragma unroll
            for (int i = 0; i < CW; ++i) {
                const int k = CW * cq + i;
                if (k < F) P[64 * F + o * F + k] = started ? w[i] : 0.0f;
            }
        }
    }
    float* scr = reinterpret_cast<float*>(sP);               // [NT][8]
#pragma unroll
    for (int i = 0; i < 8; ++i) scr[tid * 8 + i] = gb1[i];
    __syncthreads();
    if (tid < 64) {
        const int kcc = tid >> 3, i = tid & 7;
        float s = 0.0f;
        for (int w = 0; w < NW; ++w)
#pragma unroll
            for (int r = 0; r < 4; ++r) s += scr[(w * 32 + kcc * 4 + r) * 8 + i];
        P[2 * 64 * F + tid] = s;
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 256);
}

}  // namespace is

using namespace is;

extern "C" {

// Tensor-core variant of is_egnn_node_post_bwd (same outputs, same partial layout, grid = is_egnn_node_grid).
int is_egnn_node_post_bwd_tc(const float* gh_out, const float* h, int64_t ldh, int F, const float* hn,
                             const float* W5, const float* b5, const float* W6,
                             float* gh_direct, float* ghn, float* partials, int64_t n_nodes, void* stream) {
    if (!(F == 20 || F == 64) || n_nodes <= 0) return IS_ERR_ARG;
    if ((reinterpret_cast<uintptr_t>(ghn) & 31) != 0) return IS_ERR_ARG;                                // 256-bit stores
    if ((reinterpret_cast<uintptr_t>(gh_direct) & (F == 64 ? 31 : 15)) != 0) return IS_ERR_ARG;         // 256- / 128-bit stores
    const size_t smem = 9 * (size_t)nb::T_BYTES + 9 * (size_t)nb::W_BYTES + sizeof(float) * (64 + 16 * 16);
    cudaError_t e = cudaFuncSetAttribute(node_post_bwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const int sms = current_num_sms();
    const int64_t tiles = (n_nodes + IS_TM - 1) / IS_TM;
    const int grid = (int)(tiles < sms ? tiles : sms);
    node_post_bwd_tc_kernel<<<grid, nb::NT, smem, (cudaStream_t)stream>>>(gh_out, h, ldh, F, hn, W5, b5, W6, gh_direct, ghn, partials, n_nodes);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

// Tensor-core variant of is_egnn_node_pre_bwd (same outputs, same partial layout, grid = is_egnn_node_grid).
int is_egnn_node_pre_bwd_tc(const float* gz1, const float* gQ, const float* gD, const float* gxd, const float* gx_out,
                            const float* gh_direct, const int* outptr, const int* csc_pos, const float* h, int64_t ldh, int F,
                            const float* W1, float* gh, float* gx, float* partials, int64_t n_nodes, void* stream) {
    if (!(F == 20 || F == 64) || n_nodes <= 0) return IS_ERR_ARG;
    if (((reinterpret_cast<uintptr_t>(gh) | reinterpret_cast<uintptr_t>(gh_direct)) & (F == 64 ? 31 : 15)) != 0)
        return IS_ERR_ARG;                                                                  // 256- / 128-bit accesses
    const size_t smem = 9 * (size_t)nb::T_BYTES + 6 * (size_t)nb::W_BYTES + (size_t)IS_TM * 64 * sizeof(float);
    cudaError_t e = cudaFuncSetAttribute(node_pre_bwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const int sms = current_num_sms();
    const int64_t tiles = (n_nodes + IS_TM - 1) / IS_TM;
    const int grid = (int)(tiles < sms ? tiles : sms);
    node_pre_bwd_tc_kernel<<<grid, nb::NT, smem, (cudaStream_t)stream>>>(gz1, gQ, gD, gxd, gx_out, gh_direct, outptr, csc_pos, h, ldh, F,
                                                                        W1, gh, gx, partials, n_nodes);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

}  // extern "C"
