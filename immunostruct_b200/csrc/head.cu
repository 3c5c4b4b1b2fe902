// Fused small-layer kernels of the eval-mode forward (no autograd, dropout inactive).
//
// At batch 512 the head of the model is ~45 kernels of 3-16 us each (tiny cuBLAS GEMMs with their bias epilogues,
// ReLUs, exp / mul / add of the reparameterisation, concatenations): 6 % of the inference step and pure launch /
// latency overhead.  Two kernels replace them:
//
//   vae_mid_infer   property_embedding (Linear 2->32, ReLU, [Dropout], Linear 32->8, ReLU; hybrid_models.py:46-52 /
//                   280-286), mu = vae_fc21(h1), logvar = vae_fc22(h1), z = mu + eps * exp(0.5 logvar)
//                   (reparameterize, :301-304; eps comes from torch.randn_like so the RNG stream is the reference's),
//                   z_vae = [z | prop] (:339), h3 = ReLU(vae_fc3(z_vae)) (:306-307).
//   head_infer      x_gat = w_concat(pooled) (the affine map commutes with the mean pool), combined = [x_gat | z_vae]
//                   (:341), fusion attention in closed form (fusion.cu), classifier Linear(104->32) ReLU [Dropout]
//                   Linear(32->1) (:54-61, 351).
// Plain fp32 FMA arithmetic, fixed summation order.
#include "common.cuh"

#define IS_HEAD_LMAX 256
#define IS_HEAD_HMAX 8

namespace is {

// ---- vae_mid: SPB samples per CTA so that every weight row read from L2 serves SPB dot products ----------------
constexpr int VM_SPB = 2;      // 256 CTAs at batch 512: the phases below are latency chains, co-resident CTAs overlap them

// SPEC: the reference's sizes (hidden 512, latent 32, 8 property features) as compile-time constants -- the dot-product loops
// unroll completely and all their weight loads are in flight at once (the kernel is a chain of L2 latencies)
template <bool SPEC>
__global__ void __launch_bounds__(IS_THREADS)
vae_mid_infer_kernel(const float* __restrict__ h1, const float* __restrict__ prop, const float* __restrict__ eps,
                     const float* __restrict__ Wp0, const float* __restrict__ bp0, const float* __restrict__ Wp3,
                     const float* __restrict__ bp3, const float* __restrict__ W21, const float* __restrict__ b21,
                     const float* __restrict__ W22, const float* __restrict__ b22, const float* __restrict__ W3,
                     const float* __restrict__ b3, float* __restrict__ mu, float* __restrict__ logvar,
                     float* __restrict__ zv, float* __restrict__ h3, int B, int HD_, int LD_, int PD_) {
    const int HD = SPEC ? 512 : HD_, LD = SPEC ? 32 : LD_, PD = SPEC ? 8 : PD_;
    extern __shared__ __align__(16) float sm[];
    float* sh = sm;                                  // [SPB][HD]
    float* se = sh + VM_SPB * HD;                    // [SPB][32] property hidden
    float* sml = se + VM_SPB * 32;                   // [SPB][2 LD] mu | logvar
    float* sz = sml + VM_SPB * 2 * LD;               // [SPB][LD + PD]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int b0 = blockIdx.x * VM_SPB;
    const int ns = min(VM_SPB, B - b0);
    const int LZ = LD + PD;
    for (int idx = tid; idx < VM_SPB * HD; idx += IS_THREADS) {
        const int s = idx / HD;
        sh[idx] = s < ns ? __ldg(h1 + (int64_t)(b0 + s) * HD + (idx - s * HD)) : 0.0f;
    }
    if (tid < VM_SPB * 32) {
        const int s = tid >> 5, o = tid & 31;
        const float p0 = s < ns ? __ldg(prop + (b0 + s) * 2) : 0.0f, p1 = s < ns ? __ldg(prop + (b0 + s) * 2 + 1) : 0.0f;
        se[tid] = fmaxf(fmaf(__ldg(Wp0 + 2 * o + 1), p1, fmaf(__ldg(Wp0 + 2 * o), p0, __ldg(bp0 + o))), 0.0f);
    }
    __syncthreads();
    // mu | logvar: one warp per output row, lanes stride K (coalesced weight reads), SPB samples per pass
    for (int o = warp; o < 2 * LD; o += IS_THREADS / 32) {
        const float* w = o < LD ? W21 + (int64_t)o * HD : W22 + (int64_t)(o - LD) * HD;
        float acc[VM_SPB];
#pragma unroll
        for (int s = 0; s < VM_SPB; ++s) acc[s] = 0.0f;
#pragma unroll
        for (int k = lane; k < HD; k += 32) {
            const float wk = __ldg(w + k);
#pragma unroll
            for (int s = 0; s < VM_SPB; ++s) acc[s] = fmaf(wk, sh[s * HD + k], acc[s]);
        }
#pragma unroll
        for (int s = 0; s < VM_SPB; ++s) acc[s] = warp_sum(acc[s]);
        if (lane < VM_SPB) {
            float v = acc[0];
#pragma unroll
            for (int s = 1; s < VM_SPB; ++s) v = lane == s ? acc[s] : v;
            sml[lane * 2 * LD + o] = v + __ldg(o < LD ? b21 + o : b22 + (o - LD));
        }
    }
    // property embedding, second layer
    if (tid < VM_SPB * PD) {
        const int s = tid / PD, o = tid - s * PD;
        float a = __ldg(bp3 + o);
        for (int k = 0; k < 32; ++k) a = fmaf(__ldg(Wp3 + o * 32 + k), se[s * 32 + k], a);
        sz[s * LZ + LD + o] = fmaxf(a, 0.0f);
    }
    __syncthreads();
    for (int idx = tid; idx < VM_SPB * LD; idx += IS_THREADS) {
        const int s = idx / LD, o = idx - s * LD;
        if (s < ns) {
            const float m = sml[s * 2 * LD + o], lv = sml[s * 2 * LD + LD + o];
            mu[(int64_t)(b0 + s) * LD + o] = m;
            logvar[(int64_t)(b0 + s) * LD + o] = lv;
            sz[s * LZ + o] = fmaf(__ldg(eps + (int64_t)(b0 + s) * LD + o), expf(0.5f * lv), m);
        } else {
            sz[s * LZ + o] = 0.0f;
        }
    }
    __syncthreads();
    for (int idx = tid; idx < ns * LZ; idx += IS_THREADS) {
        const int s = idx / LZ;
        zv[(int64_t)(b0 + s) * LZ + (idx - s * LZ)] = sz[idx];
    }
    // h3 = relu(W3 z_vae + b3): one thread per output row (LZ = 40 weights), SPB samples
    for (int o = tid; o < HD; o += IS_THREADS) {
        float acc[VM_SPB];
        const float bo = __ldg(b3 + o);
#pragma unroll
        for (int s = 0; s < VM_SPB; ++s) acc[s] = bo;
        const float* w = W3 + (int64_t)o * LZ;
        if ((LZ & 3) == 0 && (reinterpret_cast<uintptr_t>(W3) & 15) == 0) {
            // 128-bit weight loads: a quarter of the (uncoalesced: one row per thread) load instructions, same k order
#pragma unroll
            for (int k = 0; k < LZ; k += 4) {
                const float4 w4 = __ldg(reinterpret_cast<const float4*>(w + k));
#pragma unroll
                for (int s = 0; s < VM_SPB; ++s) {
                    acc[s] = fmaf(w4.x, sz[s * LZ + k], acc[s]);
                    acc[s] = fmaf(w4.y, sz[s * LZ + k + 1], acc[s]);
                    acc[s] = fmaf(w4.z, sz[s * LZ + k + 2], acc[s]);
                    acc[s] = fmaf(w4.w, sz[s * LZ + k + 3], acc[s]);
                }
            }
        } else {
            for (int k = 0; k < LZ; ++k) {
                const float wk = __ldg(w + k);
#pragma unroll
                for (int s = 0; s < VM_SPB; ++s) acc[s] = fmaf(wk, sz[s * LZ + k], acc[s]);
            }
        }
#pragma unroll
        for (int s = 0; s < VM_SPB; ++s)
            if (s < ns) h3[(int64_t)(b0 + s) * HD + o] = fmaxf(acc[s], 0.0f);
    }
}

// ---- head: shared arithmetic of head_infer and head_mc_infer ------------------------------------------------------
// One copy of every rounding step, so that draw k of head_mc_infer is bit-identical to head_infer run on that draw.

// x_gat row o = Wc[o] . pooled + bc[o], one warp: lanes over the 64 inputs (p0 = pooled[lane], p1 = pooled[32 + lane])
__device__ __forceinline__ float head_xgat_row(const float* __restrict__ Wc, const float* __restrict__ bc, int o, float p0,
                                               float p1, int lane) {
    const float a = fmaf(__ldg(Wc + o * 64 + 32 + lane), p1, __ldg(Wc + o * 64 + lane) * p0);
    return warp_sum(a) + __ldg(bc + o);
}

// closed-form fusion attention (fusion.cu): expectation of token i under head h over the L scalars c, whose extremes are
// cmax / cmin.  Inference only: 2^(g2 c_j - m2) with ex2.approx, g2 = gamma log2 e (one FFMA + one MUFU per term; the
// rounding of g2 moves an exponent of magnitude <= ~20 by ~1e-6, an order below the 1e-5 parity bound, as in the fast SiLU
// of the inference EGNN kernels); two independent accumulator pairs
__device__ __forceinline__ float head_fusion_expect(const float* c, int L, int i, const float* __restrict__ coef, int H, int h,
                                                    float cmax, float cmin) {
    const float gamma = coef[h] * c[i] + coef[H + h];
    const float g2 = gamma * 1.4426950408889634f;
    const float m2 = gamma > 0.0f ? g2 * cmax : g2 * cmin;
    float Z0 = 0.0f, S0 = 0.0f, Z1 = 0.0f, S1 = 0.0f;
    int j = 0;
    for (; j + 1 < L; j += 2) {
        const float c0 = c[j], c1 = c[j + 1];
        float e0, e1;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(fmaf(g2, c0, -m2)));
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(fmaf(g2, c1, -m2)));
        Z0 += e0; S0 = fmaf(e0, c0, S0);
        Z1 += e1; S1 = fmaf(e1, c1, S1);
    }
    if (j < L) {
        const float c0 = c[j];
        float e0;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(fmaf(g2, c0, -m2)));
        Z0 += e0; S0 = fmaf(e0, c0, S0);
    }
    return (S0 + S1) / (Z0 + Z1);
}

// fused feature of one token from its H head expectations Eh[0..H)
__device__ __forceinline__ float head_fusion_out(const float* Eh, const float* __restrict__ coef, int H) {
    float o = coef[4 * H];
    for (int h = 0; h < H; ++h) o += coef[2 * H + h] * Eh[h] + coef[3 * H + h];
    return o;
}

// classifier hidden unit o = relu(W1[o] . f + b1[o]), one warp: lanes strided over the L features
__device__ __forceinline__ float head_hidden_row(const float* __restrict__ W1, const float* __restrict__ b1, const float* f,
                                                 int L, int o, int lane) {
    float a = 0.0f;
    for (int k = lane; k < L; k += 32) a = fmaf(__ldg(W1 + o * L + k), f[k], a);
    a = warp_sum(a);
    return fmaxf(a + __ldg(b1 + o), 0.0f);
}

// classifier output r = W2[r] . hid + b2[r], one warp (lane = hidden unit)
__device__ __forceinline__ float head_out_row(const float* __restrict__ W2, const float* __restrict__ b2, const float* hid,
                                              int r, int lane) {
    return warp_sum(__ldg(W2 + r * 32 + lane) * hid[lane]) + __ldg(b2 + r);
}

// ---- head: one CTA per sample ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(IS_THREADS)
head_infer_kernel(const float* __restrict__ pooled, const float* __restrict__ Wc, const float* __restrict__ bc,
                  const float* __restrict__ zv, int LZ, const float* __restrict__ coef, int H,
                  const float* __restrict__ W1, const float* __restrict__ b1, const float* __restrict__ W2,
                  const float* __restrict__ b2, float* __restrict__ x_gat, float* __restrict__ out, int n_out) {
    __shared__ float c[IS_HEAD_LMAX];
    __shared__ float f[IS_HEAD_LMAX];                        // fused features (after the fusion attention)
    __shared__ float Eh[IS_HEAD_LMAX * IS_HEAD_HMAX];
    __shared__ float hid[32];
    __shared__ float s_mm[2];
    __shared__ float red[2 * 8];
    const int b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int L = 64 + LZ;
    // x_gat = Wc pooled + bc (or pooled itself): warp per 8 outputs, lanes over the 64 inputs
    if (Wc != nullptr) {
        const float p0 = __ldg(pooled + (int64_t)b * 64 + lane), p1 = __ldg(pooled + (int64_t)b * 64 + 32 + lane);
        for (int o = warp; o < 64; o += IS_THREADS / 32) {
            const float a = head_xgat_row(Wc, bc, o, p0, p1, lane);
            if (lane == 0) c[o] = a;
        }
    } else if (tid < 64) {
        c[tid] = __ldg(pooled + (int64_t)b * 64 + tid);
    }
    if (tid < LZ) c[64 + tid] = __ldg(zv + (int64_t)b * LZ + tid);
    __syncthreads();
    if (tid < 64 && x_gat != nullptr) x_gat[(int64_t)b * 64 + tid] = c[tid];
    if (coef != nullptr) {
        // closed-form fusion attention over the L scalars (fusion.cu)
        float lmax = -INFINITY, lmin = INFINITY;
        for (int i = tid; i < L; i += IS_THREADS) { lmax = fmaxf(lmax, c[i]); lmin = fminf(lmin, c[i]); }
        lmax = warp_max(lmax); lmin = -warp_max(-lmin);
        if (lane == 0) { red[warp] = lmax; red[8 + warp] = lmin; }
        __syncthreads();
        if (tid == 0) {
            float a = red[0], m = red[8];
            for (int w = 1; w < 8; ++w) { a = fmaxf(a, red[w]); m = fminf(m, red[8 + w]); }
            s_mm[0] = a; s_mm[1] = m;
        }
        __syncthreads();
        const float cmax = s_mm[0], cmin = s_mm[1];
        for (int idx = tid; idx < L * H; idx += IS_THREADS) {
            const int i = idx / H, h = idx - i * H;
            Eh[idx] = head_fusion_expect(c, L, i, coef, H, h, cmax, cmin);
        }
        __syncthreads();
        for (int i = tid; i < L; i += IS_THREADS) f[i] = head_fusion_out(Eh + i * H, coef, H);
    } else {
        for (int i = tid; i < L; i += IS_THREADS) f[i] = c[i];
    }
    __syncthreads();
    // classifier: hid = relu(W1 f + b1) (32 rows, warp per 4 rows), out = W2 hid + b2 (or hid itself)
    for (int o = warp; o < 32; o += IS_THREADS / 32) {
        const float a = head_hidden_row(W1, b1, f, L, o, lane);
        if (lane == 0) hid[o] = a;
    }
    __syncthreads();
    if (W2 != nullptr) {
        if (warp < n_out) {
            const float a = head_out_row(W2, b2, hid, warp, lane);
            if (lane == 0) out[(int64_t)b * n_out + warp] = a;
        }
    } else if (tid < 32) {
        out[(int64_t)b * 32 + tid] = hid[tid];
    }
}

// ---- head over many reparameterisation draws: one CTA per (sample, chunk of MC_DRAWS draws) ----------------------
// The tokens of one item are [x_gat | z | prop] (64 + LD + PD); only z = mu + eps exp(0.5 logvar) depends on the draw.
// x_gat, mu, exp(0.5 logvar) and prop are computed once per CTA; the (draw, token, head) fusion work and the (draw, row)
// classifier rows are spread over the whole CTA.  A logit depends on (sample, eps[k]) only, never on the chunking.
constexpr int MC_DRAWS = 8;      // = warps per CTA: one warp per draw for the extremes and the output row

struct McItem {
    const float* pooled;         // [B, 64]
    const float* mu;             // [B, LD]
    const float* logvar;         // [B, LD]
    const float* zv;             // [B, LD + PD] (the PD property columns are read)
    const float* eps;            // [K, B, LD]
};

__global__ void __launch_bounds__(IS_THREADS)
head_mc_infer_kernel(McItem it0, McItem it1, int n_items, int LD, int PD, const float* __restrict__ Wc,
                     const float* __restrict__ bc, const float* __restrict__ coef, int H, const float* __restrict__ W1,
                     const float* __restrict__ b1, const float* __restrict__ W2, const float* __restrict__ b2,
                     float* __restrict__ logits, int B, int K, int n_chunks, int kc_max) {
    extern __shared__ __align__(16) float sm[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int LZ = LD + PD, LI = 64 + LZ, L = n_items * LI, LH = coef != nullptr ? L * H : 0;
    const int b = blockIdx.x / n_chunks, k0 = (blockIdx.x - b * n_chunks) * MC_DRAWS;
    const int kc = min(MC_DRAWS, K - k0);
    float* base = sm;                       // [L] draw-independent tokens (the z slots hold mu)
    float* sdev = base + L;                 // [2][LD] exp(0.5 logvar)
    float* c = sdev + 2 * LD;               // [kc_max][L] tokens of each draw
    float* f = c + kc_max * L;              // [kc_max][L] fused features
    float* hid = f + kc_max * L;            // [kc_max][32]
    float* mm = hid + kc_max * 32;          // [kc_max][2] extremes of c
    float* Eh = mm + kc_max * 2;            // [kc_max][L][H]
    for (int r = warp; r < n_items * 64; r += IS_THREADS / 32) {
        const int it = r >> 6, o = r & 63;
        const float* pooled = (it ? it1 : it0).pooled + (int64_t)b * 64;
        if (Wc != nullptr) {
            const float a = head_xgat_row(Wc, bc, o, __ldg(pooled + lane), __ldg(pooled + 32 + lane), lane);
            if (lane == 0) base[it * LI + o] = a;
        } else if (lane == 0) {
            base[it * LI + o] = __ldg(pooled + o);
        }
    }
    for (int idx = tid; idx < n_items * LZ; idx += IS_THREADS) {
        const int it = idx >= LZ, t = idx - it * LZ;
        const McItem& m = it ? it1 : it0;
        if (t < LD) {
            base[it * LI + 64 + t] = __ldg(m.mu + (int64_t)b * LD + t);
            sdev[it * LD + t] = expf(0.5f * __ldg(m.logvar + (int64_t)b * LD + t));
        } else {
            base[it * LI + 64 + t] = __ldg(m.zv + (int64_t)b * LZ + t);
        }
    }
    __syncthreads();
    // z = fmaf(eps, exp(0.5 logvar), mu): the arithmetic of vae_mid_infer_kernel
    for (int idx = tid; idx < kc * L; idx += IS_THREADS) {
        const int d = idx / L, t = idx - d * L, it = t >= LI, u = t - it * LI - 64;
        float v = base[t];
        if (u >= 0 && u < LD)
            v = fmaf(__ldg((it ? it1 : it0).eps + ((int64_t)(k0 + d) * B + b) * LD + u), sdev[it * LD + u], v);
        c[idx] = v;
    }
    __syncthreads();
    const float* feat = c;
    if (coef != nullptr) {
        if (warp < kc) {
            float lmax = -INFINITY, lmin = INFINITY;
            for (int i = lane; i < L; i += 32) { lmax = fmaxf(lmax, c[warp * L + i]); lmin = fminf(lmin, c[warp * L + i]); }
            lmax = warp_max(lmax); lmin = -warp_max(-lmin);
            if (lane == 0) { mm[2 * warp] = lmax; mm[2 * warp + 1] = lmin; }
        }
        __syncthreads();
        for (int idx = tid; idx < kc * LH; idx += IS_THREADS) {
            const int d = idx / LH, r = idx - d * LH, i = r / H, h = r - i * H;
            Eh[idx] = head_fusion_expect(c + d * L, L, i, coef, H, h, mm[2 * d], mm[2 * d + 1]);
        }
        __syncthreads();
        for (int idx = tid; idx < kc * L; idx += IS_THREADS) f[idx] = head_fusion_out(Eh + idx * H, coef, H);
        __syncthreads();
        feat = f;
    }
    for (int r = warp; r < kc * 32; r += IS_THREADS / 32) {
        const int d = r >> 5, o = r & 31;
        const float a = head_hidden_row(W1, b1, feat + d * L, L, o, lane);
        if (lane == 0) hid[r] = a;
    }
    __syncthreads();
    if (warp < kc) {
        const float a = head_out_row(W2, b2, hid + warp * 32, 0, lane);
        if (lane == 0) logits[(int64_t)b * K + k0 + warp] = a;
    }
}

// mean and population standard deviation of sigmoid(logit) over the K draws of each sample: one warp per sample, lanes
// strided over the draws, fp64, two passes, fixed butterfly order (no atomics: the result depends on the logits only)
__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__global__ void __launch_bounds__(IS_THREADS)
head_mc_stats_kernel(const float* __restrict__ logits, int B, int K, float* __restrict__ prob_mean,
                     float* __restrict__ prob_std) {
    const int b = blockIdx.x * (IS_THREADS / 32) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= B) return;
    const float* row = logits + (int64_t)b * K;
    double s = 0.0;
    for (int k = lane; k < K; k += 32) s += 1.0 / (1.0 + exp(-(double)__ldg(row + k)));
    const double mean = warp_sum_f64(s) / K;
    double v = 0.0;
    for (int k = lane; k < K; k += 32) {
        const double p = 1.0 / (1.0 + exp(-(double)__ldg(row + k))) - mean;
        v = fma(p, p, v);
    }
    const double var = warp_sum_f64(v) / K;
    if (lane == 0) {
        prob_mean[b] = (float)mean;
        prob_std[b] = (float)sqrt(var);
    }
}

}  // namespace is

using namespace is;

extern "C" {

// Eval-mode middle of the sequence branch (see the header of this file).  h1 [B,HD], prop [B,2], eps [B,LD] ->
// mu, logvar [B,LD], z_vae [B,LD+PD], h3 [B,HD].  The property MLP's hidden width is 32 (reference).
int is_vae_mid_infer(const float* h1, const float* prop, const float* eps, const float* Wp0, const float* bp0,
                     const float* Wp3, const float* bp3, const float* W21, const float* b21, const float* W22,
                     const float* b22, const float* W3, const float* b3, float* mu, float* logvar, float* z_vae,
                     float* h3, int n_samples, int hidden, int latent, int prop_dim, void* stream) {
    if (n_samples <= 0 || hidden <= 0 || latent <= 0 || prop_dim < 0 || VM_SPB * prop_dim > IS_THREADS) return IS_ERR_ARG;
    const size_t smem = sizeof(float) * (size_t)VM_SPB * (hidden + 32 + 2 * latent + latent + prop_dim);
    if (smem > 200 * 1024) return IS_ERR_UNSUPPORTED;
    const int grid = (n_samples + VM_SPB - 1) / VM_SPB;
    const bool spec = hidden == 512 && latent == 32 && prop_dim == 8;
    auto kern = spec ? vae_mid_infer_kernel<true> : vae_mid_infer_kernel<false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    kern<<<grid, IS_THREADS, smem, (cudaStream_t)stream>>>(h1, prop, eps, Wp0, bp0, Wp3, bp3, W21, b21, W22, b22, W3, b3, mu, logvar,
                                                          z_vae, h3, n_samples, hidden, latent, prop_dim);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

// Eval-mode fusion head.  pooled [B,64]; Wc / bc [64,64] / [64] or NULL (no projection); z_vae [B,LZ]; coef = the
// 4H+1 closed-form fusion coefficients or NULL (plain concatenation, v1 models); classifier W1 [32, 64+LZ], b1 [32];
// W2 [n_out,32], b2 [n_out] or NULL (then out = the 32 hidden features).  x_gat [B,64] may be NULL.
int is_head_infer(const float* pooled, const float* Wc, const float* bc, const float* z_vae, int LZ, const float* coef,
                  int n_head, const float* W1, const float* b1, const float* W2, const float* b2, int n_out,
                  float* x_gat, float* out, int n_samples, void* stream) {
    if (n_samples <= 0 || LZ < 0 || 64 + LZ > IS_HEAD_LMAX || LZ > IS_THREADS) return IS_ERR_ARG;
    if (coef != nullptr && (n_head < 1 || n_head > IS_HEAD_HMAX)) return IS_ERR_ARG;
    if (W2 != nullptr && (n_out < 1 || n_out > 8)) return IS_ERR_ARG;
    head_infer_kernel<<<n_samples, IS_THREADS, 0, (cudaStream_t)stream>>>(pooled, Wc, bc, z_vae, LZ, coef, n_head, W1, b1, W2, b2,
                                                                          x_gat, out, n_out);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

// K reparameterisation draws of the eval-mode head for B samples (see head_mc_infer_kernel): item i = (pooled_i [B,64],
// mu_i / logvar_i [B,LD], z_vae_i [B,LD+PD] (property columns), eps_i [K,B,LD]); the tokens are item-major
// [x_gat_0 | z_0 | prop_0 | x_gat_1 | ...] (L = n_items (64+LD+PD) <= IS_HEAD_LMAX); Wc / bc, coef and the classifier as
// in is_head_infer, W2 [1,32] / b2 [1] required.  -> logits [B,K] (sample-major), prob_mean / prob_std [B] (mean and
// population standard deviation of sigmoid(logit) over the draws).  Two kernels: the draws, then the statistics.
int is_head_mc_infer(const float* pooled0, const float* mu0, const float* logvar0, const float* z_vae0, const float* eps0,
                     const float* pooled1, const float* mu1, const float* logvar1, const float* z_vae1, const float* eps1,
                     int n_items, int latent, int prop_dim, const float* Wc, const float* bc, const float* coef, int n_head,
                     const float* W1, const float* b1, const float* W2, const float* b2, float* logits, float* prob_mean,
                     float* prob_std, int n_samples, int n_draws, void* stream) {
    if (n_samples <= 0 || n_draws <= 0 || latent <= 0 || prop_dim < 0 || (n_items != 1 && n_items != 2)) return IS_ERR_ARG;
    if (n_items * (64 + latent + prop_dim) > IS_HEAD_LMAX) return IS_ERR_ARG;
    if (coef != nullptr && (n_head < 1 || n_head > IS_HEAD_HMAX)) return IS_ERR_ARG;
    if ((Wc == nullptr) != (bc == nullptr) || !W1 || !b1 || !W2 || !b2 || !logits || !prob_mean || !prob_std) return IS_ERR_ARG;
    if (!pooled0 || !mu0 || !logvar0 || !z_vae0 || !eps0) return IS_ERR_ARG;
    if (n_items == 2 && (!pooled1 || !mu1 || !logvar1 || !z_vae1 || !eps1)) return IS_ERR_ARG;
    const int n_chunks = (n_draws + MC_DRAWS - 1) / MC_DRAWS, kc_max = n_draws < MC_DRAWS ? n_draws : MC_DRAWS;
    if ((int64_t)n_samples * n_chunks > 0x7fffffff) return IS_ERR_UNSUPPORTED;
    const int L = n_items * (64 + latent + prop_dim), H = coef != nullptr ? n_head : 0;
    const size_t smem = sizeof(float) * ((size_t)L + 2 * latent + (size_t)kc_max * (2 * L + 32 + 2 + L * H));
    if (smem > 227 * 1024) return IS_ERR_UNSUPPORTED;
    cudaError_t e = cudaFuncSetAttribute(head_mc_infer_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const McItem it0{pooled0, mu0, logvar0, z_vae0, eps0};
    const McItem it1 = n_items == 2 ? McItem{pooled1, mu1, logvar1, z_vae1, eps1} : it0;
    head_mc_infer_kernel<<<n_samples * n_chunks, IS_THREADS, smem, (cudaStream_t)stream>>>(
        it0, it1, n_items, latent, prop_dim, Wc, bc, coef, n_head, W1, b1, W2, b2, logits, n_samples, n_draws, n_chunks, kc_max);
    IS_LAUNCH_CHECK();
    head_mc_stats_kernel<<<(n_samples + IS_THREADS / 32 - 1) / (IS_THREADS / 32), IS_THREADS, 0, (cudaStream_t)stream>>>(
        logits, n_samples, n_draws, prob_mean, prob_std);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

}  // extern "C"
