// Node-side half of an EGNN layer on the tensor cores, fused across the layer boundary (the tile chain: egnn_node_tc.cuh):
//
//   node_post(l) :  h' = W6 silu(W5 [h | hn] + b5) + b6
//   node_pre(l+1):  P' = h' Ws'^T ,  Q' = h' Wd'^T + b1'   or, after the LAST layer (next_kind = 2), QKV = h' [Wq; Wk; Wv]^T + b
//
// One persistent CTA per SM (two at 256 threads) walks the groups of NTILE 128-node tiles; its weight blocks stay resident
// in shared memory for the CTA's lifetime.  Used by the no-grad inference path in the precisions whose edge forward has no
// node tail (bf16, bf16x3) and by the training forward; the fp16x2 inference forward runs the same chain as the tail of the
// edge kernel (egnn_tc2.cu, egnn_layer_fwd).  PREC_BF16 (bf16 mode), PREC_FP16X2 or PREC_BF16X3 (fp32 parity; the hi/lo
// tf32 form of the five resident weight blocks would not fit in shared memory, the three-term bf16 form does: 138 KB).
#include "egnn_node_tc.cuh"

namespace is {

template <int PREC, int NT, bool FAST, int NEXT_KIND>
__global__ void __launch_bounds__(NT, NT == 256 ? 2 : 1)
node_post_pre_tc_kernel(NodeArgs a, int64_t M) {
    using NC = NodeCfg<PREC, NEXT_KIND>;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    uint8_t* sA = smem_raw;
    uint8_t* sW = sA + NC::A_REGION;
    float* vec = reinterpret_cast<float*>(sW + NC::W_REGION);
    __shared__ __align__(8) uint64_t mbar;
    __shared__ uint32_t s_tmem;
    const int tid = threadIdx.x, warp = tid >> 5;

    if (warp == 0) tmem_alloc(&s_tmem, NC::NTILE * NC::TCOLS);
    if (tid == 32) mbar_init(&mbar, 1);
    node_stage_weights<PREC, NEXT_KIND>(a, sW, vec, tid, NT);
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = s_tmem;
    uint32_t phase = 0;
    constexpr int64_t GROUP = NC::NTILE * IS_TM;
    node_chain<PREC, NT, FAST, NEXT_KIND>(a, sA, sW, vec, tmem, &mbar, phase, blockIdx.x * GROUP, gridDim.x * GROUP, M, tid, 0);
    fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, NC::NTILE * NC::TCOLS);
}

template <int PREC, int NT, bool FAST, int NEXT_KIND>
static int launch_node_tc2(const NodeArgs& a, int64_t M, cudaStream_t st) {
    using NC = NodeCfg<PREC, NEXT_KIND>;
    const size_t smem = (size_t)NC::A_REGION + NC::W_REGION + NC::VEC_BYTES + 128;
    cudaError_t e = cudaFuncSetAttribute(node_post_pre_tc_kernel<PREC, NT, FAST, NEXT_KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const int sms = current_num_sms();
    int64_t tiles = (M + NC::NTILE * IS_TM - 1) / (NC::NTILE * IS_TM);
    int64_t cap = (int64_t)sms * (NT == 256 ? 2 : 1);
    int grid = (int)(tiles < cap ? tiles : cap);
    node_post_pre_tc_kernel<PREC, NT, FAST, NEXT_KIND><<<grid < 1 ? 1 : grid, NT, smem, st>>>(a, M);
    e = cudaGetLastError();
    return e == cudaSuccess ? 0 : (int)e;
}

template <int PREC, int NT, bool FAST>
static int launch_node_tc(const NodeArgs& a, int64_t M, int next_kind, cudaStream_t st) {
    if (next_kind == 2) return launch_node_tc2<PREC, NT, FAST, 2>(a, M, st);
    return launch_node_tc2<PREC, NT, FAST, 1>(a, M, st);
}

}  // namespace is

using namespace is;

extern "C" {

// node_mlp of layer l fused with the per-node half of layer l+1's first edge-MLP layer (W1n / b1n / PQn
// may be NULL for the last layer), or -- next_kind = 2 -- with the attention projections that follow the last
// layer: W1n = [Wq; Wk; Wv] [192, 64], b1n [192], PQn = QKV [n_nodes, 192].  precision: 0 = bf16, 3 = bf16x3 (fp32-accurate); fast_act: 5-instruction
// SiLU (inference) vs accurate expf (training forward).  W1n must be the
// [64, 130] weight of a 64-wide layer.
int is_egnn_node_post_pre_tc(const float* h, int64_t ldh, int F, const float* hn, const float* W5, const float* b5,
                             const float* W6, const float* b6, float* h_out, const float* W1n, const float* b1n,
                             float* PQn, int64_t n_nodes, int precision, int fast_act, int next_kind, void* stream) {
    if (!(F == 20 || F == 64) || n_nodes <= 0) return IS_ERR_ARG;
    if ((W1n == nullptr) != (PQn == nullptr)) return IS_ERR_ARG;
    if (W1n != nullptr && next_kind != 1 && next_kind != 2) return IS_ERR_ARG;
    if (((reinterpret_cast<uintptr_t>(h_out) | reinterpret_cast<uintptr_t>(PQn)) & 31) != 0) return IS_ERR_ARG;   // 256-bit stores
    cudaStream_t st = (cudaStream_t)stream;
    const NodeArgs a{h, ldh, F, hn, W5, b5, W6, b6, h_out, W1n, b1n, PQn};
    if (precision == PREC_BF16)
        return launch_node_tc<PREC_BF16, 256, true>(a, n_nodes, next_kind, st);
    if (precision == PREC_FP16X2)          // fp16 hi / lo operand split: inference forward only
        return launch_node_tc<PREC_FP16X2, 512, true>(a, n_nodes, next_kind, st);
    if (precision == PREC_BF16X3 && fast_act)
        return launch_node_tc<PREC_BF16X3, 512, true>(a, n_nodes, next_kind, st);
    if (precision == PREC_BF16X3)
        return launch_node_tc<PREC_BF16X3, 512, false>(a, n_nodes, next_kind, st);
    return IS_ERR_ARG;
}

}  // extern "C"
