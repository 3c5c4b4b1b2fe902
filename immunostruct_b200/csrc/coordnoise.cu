// Structural uncertainty: one pass of seeded coordinate perturbations of a resident batch (immunostruct_b200/coordnoise.py).
//
// A pass holds r copies of the base batch (B graphs, N node rows), in the layout of GraphBatch.replicate(r): copy k of
// graph b sits at node rows k N + node_off[b] ....  Copy k is structure draw m = draw0 + k.  Node row i = node_off[b] + a
// of copy k keeps its 20 residue columns and gets coordinates (x23 columns 20..22)
//     x_c + sigma_i z_c  (one fmaf, c = 0, 1, 2),
// where z = three standard normals of the counter-based stream keyed on (seed, item, m, b, a):
//   * Philox4x32-10 (Salmon, Moraes, Dror, Shaw, "Parallel random numbers: as easy as 1, 2, 3", SC 2011), counter
//     (a, b, m, item), key (low and high 32 bits of seed), one call -> four uint32 words v0..v3;
//   * u_j = (2 (v_j >> 8) + 1) 2^-25 = ((v_j >> 8) + 0.5) 2^-24 in (0, 1): one round-to-nearest conversion of an integer
//     to fp32 (exact below 2^-1) and an exact scaling;
//   * Box-Muller with the accurate library functions: z0 = sqrt(-2 log u0) cospi(2 u1), z1 = sqrt(-2 log u0) sinpi(2 u1),
//     z2 = sqrt(-2 log u2) cospi(2 u3).
// The stream depends on the key alone, so a structure does not depend on how the draws are split into passes.
// A row with sigma_i == 0 (and columns 0..19 of every row) is copied, bit-exact.
//
// Work units are (copy, graph), grid-strided over the CTAs.  Rows go in 32-row chunks, one per warp: the lane owning row
// c0 + lane computes that row's noise, then the warp streams the chunk's 23-float rows coalesced and takes each
// coordinate's sigma and z from the owning lane by shuffles.  No atomics, no barriers, no device flag: the host checks
// every argument before the launch.
#include "common.cuh"
#include "philox.cuh"

namespace is {

constexpr int CN_THREADS = 256;
constexpr int CN_WARPS = CN_THREADS / 32;
constexpr int CN_CTAS_PER_SM = 4;

__device__ __forceinline__ float cn_uniform(uint32_t v) {
    return (float)(((v >> 8) << 1) | 1u) * 0x1p-25f;
}

// three standard normals of the stream key (seed, item, m, b, a)
__device__ __forceinline__ void cn_normals(uint32_t a, uint32_t b, uint32_t m, uint32_t item, uint32_t k0, uint32_t k1,
                                           float& z0, float& z1, float& z2) {
    const Philox4 p = philox4x32_10(a, b, m, item, k0, k1);
    const float u0 = cn_uniform(p.v[0]), u1 = cn_uniform(p.v[1]), u2 = cn_uniform(p.v[2]), u3 = cn_uniform(p.v[3]);
    const float r0 = sqrtf(-2.0f * logf(u0)), r2 = sqrtf(-2.0f * logf(u2));
    float s1, c1;
    sincospif(2.0f * u1, &s1, &c1);
    z0 = r0 * c1;
    z1 = r0 * s1;
    z2 = r2 * cospif(2.0f * u3);
}

__global__ void __launch_bounds__(CN_THREADS, CN_CTAS_PER_SM) coord_noise_expand_kernel(
        const float* __restrict__ x23, const int64_t* __restrict__ node_off, const float* __restrict__ sigma, int r, int B,
        int64_t N, uint32_t k0, uint32_t k1, uint32_t item, uint32_t draw0, float* __restrict__ x23_out) {
    const int64_t units = (int64_t)r * B;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t u = blockIdx.x; u < units; u += gridDim.x) {
        const int k = (int)(u / B), b = (int)(u - (int64_t)k * B);
        const int64_t n0 = __ldg(node_off + b), nb = __ldg(node_off + b + 1) - n0;
        const float* src = x23 + n0 * 23;
        float* dst = x23_out + ((int64_t)k * N + n0) * 23;
        for (int64_t c0 = (int64_t)warp * 32; c0 < nb; c0 += CN_WARPS * 32) {
            const int64_t a = c0 + lane;
            float s = 0.0f, z0 = 0.0f, z1 = 0.0f, z2 = 0.0f;
            if (a < nb) {
                s = __ldg(sigma + n0 + a);
                if (s != 0.0f) cn_normals((uint32_t)a, (uint32_t)b, draw0 + (uint32_t)k, item, k0, k1, z0, z1, z2);
            }
            const int n = (int)(nb - c0 < 32 ? nb - c0 : 32) * 23;
            const float* cs = src + c0 * 23;
            float* cd = dst + c0 * 23;
            int row = lane / 23, col = lane - row * 23;
#pragma unroll 4
            for (int e0 = 0; e0 < n; e0 += 32) {
                const int e = e0 + lane, owner = row < 32 ? row : 31;
                const float sr = __shfl_sync(0xffffffffu, s, owner);
                const float a0 = __shfl_sync(0xffffffffu, z0, owner);
                const float a1 = __shfl_sync(0xffffffffu, z1, owner);
                const float a2 = __shfl_sync(0xffffffffu, z2, owner);
                if (e < n) {
                    float v = __ldg(cs + e);
                    if (col >= 20 && sr != 0.0f) v = fmaf(sr, col == 20 ? a0 : col == 21 ? a1 : a2, v);
                    cd[e] = v;
                }
                col += 32;
                while (col >= 23) { col -= 23; ++row; }
            }
        }
    }
}

}  // namespace is

using namespace is;

extern "C" {

// grid: min(r B, 4 x SMs) CTAs of 256 threads, each looping over (copy, graph) units
int is_coord_noise_expand(const float* x23, const int64_t* node_off, const float* sigma, int r, int n_graphs,
                          int64_t n_nodes, uint64_t seed, uint32_t item, uint32_t draw0, float* x23_out, void* stream) {
    if (r < 1 || n_graphs < 1 || n_nodes < 0 || !x23 || !node_off || !sigma || !x23_out) return IS_ERR_ARG;
    if ((uint64_t)draw0 + (uint64_t)r > 0x100000000ull) return IS_ERR_ARG;
    const int64_t units = (int64_t)r * n_graphs, cap = (int64_t)CN_CTAS_PER_SM * current_num_sms();
    if (n_nodes == 0) return IS_OK;
    coord_noise_expand_kernel<<<(unsigned)(units < cap ? units : cap), CN_THREADS, 0, (cudaStream_t)stream>>>(
        x23, node_off, sigma, r, n_graphs, n_nodes, (uint32_t)seed, (uint32_t)(seed >> 32), item, draw0, x23_out);
    IS_LAUNCH_CHECK();
    return IS_OK;
}

}  // extern "C"
