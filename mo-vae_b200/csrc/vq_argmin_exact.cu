// K4x `vq_argmin_exact`: nearest-codebook search evaluated with the reference's own formula and
// float32 roundings for every row, when (K, D) is outside the tensor-core kernel's shape or the caller asks
// for MOVAE_VQ_EXACT.  (The rows the tensor-core kernel cannot decide are re-evaluated inside that kernel with the
// same arithmetic: vq_argmin_tc.cu `recheck_row_in_kernel`.)
//
// Follows /root/reference/models/vq_vae.py:34-39:
//     dist = (sum(z^2) + sum(E^2)) - 2 * (z @ E^T)          two float32 roundings after the GEMM
//     idx  = argmin(dist)                                     first minimal index
// The three inner sums are accumulated in float64 and rounded to float32 once (the correctly
// rounded value every float32 library result is within its own accumulation error of), then
// combined with float32 add / mul / sub exactly in the reference's order.
//
// One warp per group of R rows (R = 4 when the codebook fits in shared memory): lanes own codes lane,
// lane+32, ...; the rows are staged interleaved in shared memory so that one 16-byte broadcast load
// feeds the same channel of all R rows.  The codebook is staged TRANSPOSED (Es[d][j], row stride K+1
// floats) so that a warp's 32 codes are 32 consecutive banks (a per-lane walk over global rows costs 32
// L1 wavefronts per load and ran 14x slower); each codebook element read from shared memory is used for
// R rows x 1 FMA and four codes per lane run as independent chains (the one-row version was
// shared-memory-bandwidth bound: 1300 wavefronts per row).  Two-stage evaluation: a float32 FMA pass
// over all K codes selects the candidates whose score is within a safe bound of the row minimum, only
// those are re-evaluated with float64 sums.  Inf / NaN latents or codebook entries make the bound non-finite and every
// code a candidate; as in torch.argmin the first NaN distance wins.
//
// Limits at D = 64: the staged variant (R = 4) up to K = 558, the unstaged one (R = 1, codebook read from global memory)
// up to K = 6,200; larger codebooks are MOVAE_ERR_UNSUPPORTED.
#include <math.h>

#include "common.cuh"
#include "vq_tc_common.cuh"

namespace movae {

constexpr int kExWarps = 8;
constexpr int kExThreads = kExWarps * 32;
constexpr size_t kExMaxSmem = 220 * 1024;

__device__ __forceinline__ float warp_min_f(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// shared memory: zs[kExWarps][D][R] | sc[kExWarps][R][K] | e2s[K] | (STAGE) Es[D][K+1]
template <bool STAGE, int R>
__global__ void __launch_bounds__(kExThreads)
vq_argmin_exact_kernel(const float* __restrict__ z, int64_t N, int D, int64_t HW, const float* __restrict__ E, int K,
                       const int* __restrict__ list, const unsigned int* __restrict__ list_count,
                       long long* __restrict__ idx_out) {
    extern __shared__ __align__(16) float smem_f[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t total = list ? (int64_t)(*list_count) : N;
    const int64_t n_groups = (total + R - 1) / R;
    if ((int64_t)blockIdx.x * kExWarps >= n_groups) return;   // nothing for this CTA: skip the staging
    float* zs = smem_f + (size_t)warp * D * R;
    float* sc = smem_f + (size_t)kExWarps * D * R + (size_t)warp * R * K;
    float* e2s = smem_f + (size_t)kExWarps * R * (D + K);
    float* Es = e2s + K;
    const int ldE = K + 1;
    const int64_t stride = (int64_t)gridDim.x * kExWarps;

    // ---- per-CTA: the staged codebook and |e_j|^2 (float32 chain, used by the candidate filter only) ----
    if (STAGE) {
        // transposed copy, 8 independent 16-byte loads in flight per thread (the 4-byte / one-at-a-time version made
        // this fixed cost ~20 us per CTA -- more than the re-check itself at the BASELINE sizes)
        if ((D & 3) == 0 && (reinterpret_cast<uintptr_t>(E) & 15) == 0) {
            const int n4 = K * D / 4;
            for (int i0 = threadIdx.x; i0 < n4; i0 += kExThreads * 8) {
                float4 v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int i = i0 + u * kExThreads;
                    v[u] = i < n4 ? __ldg(reinterpret_cast<const float4*>(E) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int i = i0 + u * kExThreads;
                    if (i < n4) {
                        const int e0 = i * 4, j = e0 / D, d = e0 - j * D;
                        Es[d * ldE + j] = v[u].x;
                        Es[(d + 1) * ldE + j] = v[u].y;
                        Es[(d + 2) * ldE + j] = v[u].z;
                        Es[(d + 3) * ldE + j] = v[u].w;
                    }
                }
            }
        } else {
            for (int i = threadIdx.x; i < K * D; i += kExThreads) {
                const int j = i / D, d = i - j * D;
                Es[d * ldE + j] = __ldg(E + i);
            }
        }
        __syncthreads();
    }
    for (int j = threadIdx.x; j < K; j += kExThreads) {
        float e2 = 0.f;
        for (int d = 0; d < D; ++d) {
            const float x = STAGE ? Es[d * ldE + j] : __ldg(E + (size_t)j * D + d);
            e2 = fmaf(x, x, e2);
        }
        e2s[j] = e2;
    }
    __syncthreads();
    float emax2 = 0.f;
    bool finite_e = true;
    for (int j = lane; j < K; j += 32) {
        emax2 = fmaxf(emax2, e2s[j]);
        finite_e = finite_e && e2s[j] <= 3.4028235e38f;
    }
    emax2 = -warp_min_f(-emax2);
    if (!__all_sync(0xffffffffu, finite_e)) emax2 = __uint_as_float(0x7fc00000u);   // NaN bound: every row evaluates every code
    const float emax = sqrtf(emax2);

    for (int64_t g = (int64_t)blockIdx.x * kExWarps + warp; g < n_groups; g += stride) {
        // ---- stage the R rows of this group (the last group repeats its final row) --------------------
        int64_t rows[R];
        float z2f[R];
        constexpr int kMaxPerLane = 8;                       // D <= 256 handled with loads in flight; larger D loops
        {
            const float* zp[R];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                int64_t w = g * R + r;
                w = w < total ? w : total - 1;
                rows[r] = list ? (int64_t)list[w] : w;
                const int64_t b = rows[r] / HW, hw = rows[r] - b * HW;
                zp[r] = z + (b * D) * HW + hw;
            }
            double z2p[R];
#pragma unroll
            for (int r = 0; r < R; ++r) z2p[r] = 0.0;
            for (int d0 = 0; d0 < D; d0 += 32 * kMaxPerLane) {
                float v[kMaxPerLane][R];
#pragma unroll
                for (int i = 0; i < kMaxPerLane; ++i) {
                    const int d = d0 + i * 32 + lane;
#pragma unroll
                    for (int r = 0; r < R; ++r) v[i][r] = d < D ? __ldg(zp[r] + (int64_t)d * HW) : 0.f;   // all rows' loads in flight together
                }
#pragma unroll
                for (int i = 0; i < kMaxPerLane; ++i) {
                    const int d = d0 + i * 32 + lane;
                    if (d < D) {
#pragma unroll
                        for (int r = 0; r < R; ++r) {
                            zs[d * R + r] = v[i][r];
                            z2p[r] += (double)v[i][r] * (double)v[i][r];
                        }
                    }
                }
            }
#pragma unroll
            for (int r = 0; r < R; ++r) z2f[r] = (float)warp_sum(z2p[r]);
        }
        __syncwarp();

        // ---- pass 1: float32 scores |e|^2 - 2 z.e for every code and row --------------------------------
        float best32[R];
#pragma unroll
        for (int r = 0; r < R; ++r) best32[r] = __uint_as_float(0x7f800000u);
        for (int j0 = lane; j0 < K; j0 += 128) {
            int jj[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) jj[c] = min(j0 + 32 * c, K - 1);
            float acc[4][R];
#pragma unroll
            for (int c = 0; c < 4; ++c)
#pragma unroll
                for (int r = 0; r < R; ++r) acc[c][r] = 0.f;
            if (STAGE) {
                const float* e = Es;
#pragma unroll 2
                for (int d = 0; d < D; ++d, e += ldE) {
                    float zv[R];
                    if constexpr (R == 4) {
                        const float4 q = *reinterpret_cast<const float4*>(zs + d * 4);
                        zv[0] = q.x; zv[1] = q.y; zv[2] = q.z; zv[3] = q.w;
                    } else {
#pragma unroll
                        for (int r = 0; r < R; ++r) zv[r] = zs[d * R + r];
                    }
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const float ev = e[jj[c]];
#pragma unroll
                        for (int r = 0; r < R; ++r) acc[c][r] = fmaf(ev, zv[r], acc[c][r]);
                    }
                }
            } else {
                for (int d = 0; d < D; ++d) {
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const float ev = __ldg(E + (size_t)jj[c] * D + d);
#pragma unroll
                        for (int r = 0; r < R; ++r) acc[c][r] = fmaf(ev, zs[d * R + r], acc[c][r]);
                    }
                }
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                if (j0 + 32 * c < K) {
                    const float e2 = e2s[jj[c]];
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const float s = e2 - 2.f * acc[c][r];
                        sc[r * K + jj[c]] = s;
                        best32[r] = fminf(best32[r], s);
                    }
                }
            }
        }
        __syncwarp();

        // ---- pass 2 (per row): candidates re-evaluated with float64 sums and the reference's float32 formula
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const float b32 = warp_min_f(best32[r]);
            const float znorm = sqrtf(z2f[r]);
            // float32 pass error per score <= (D+2) 2^-24 (2|z||e| + |e|^2); a code within twice that (+ the reference
            // formula's own quantum, 8 ulp of |z|^2 + |e|^2) of the minimum can be the float32-rounded argmin
            const float bound = 2.f * (float)(D + 2) * 5.9604645e-08f * (2.f * znorm * emax + emax2) +
                                8.f * 1.1920929e-07f * (z2f[r] + emax2);
            const float lim = b32 + bound;
            // inf / NaN latents or codebook rows: the limit bounds nothing and every code is evaluated
            const bool all = !(fabsf(lim) <= 3.4028235e38f);
            float bestd = __uint_as_float(0x7f800000u);
            int bestj = 0x7fffffff;
            for (int jb = 0; jb < K; jb += 32) {
                const int j = jb + lane;
                unsigned cand = __ballot_sync(0xffffffffu, j < K && (all || sc[r * K + j] <= lim));
                while (cand) {                                  // the whole warp evaluates one candidate: lanes over d
                    const int jc = jb + __ffs(cand) - 1;
                    cand &= cand - 1;
                    double dd = 0.0, ee = 0.0;
                    for (int d = lane; d < D; d += 32) {
                        const double x = (double)(STAGE ? Es[d * ldE + jc] : __ldg(E + (size_t)jc * D + d));
                        dd = fma(x, (double)zs[d * R + r], dd);
                        ee = fma(x, x, ee);
                    }
                    dd = warp_sum(dd);
                    ee = warp_sum(ee);
                    const float dist = __fsub_rn(__fadd_rn(z2f[r], (float)ee), __fmul_rn(2.f, (float)dd));
                    // candidates visited in ascending j: first minimum kept, and as in torch.argmin the first NaN beats
                    // everything
                    if (dist < bestd || (dist != dist && bestd == bestd)) { bestd = dist; bestj = jc; }
                }
            }
            // every distance inf: torch.argmin of such a row is its first element
            if (lane == 0) idx_out[rows[r]] = (long long)(bestj == 0x7fffffff ? 0 : bestj);
        }
        __syncwarp();
    }
}

// All N rows.  (The kernel can also walk a worklist -- `list` / `list_count` -- which the tensor-core search used before it
// re-checked its undecidable rows itself; kept for tools that want to re-evaluate chosen rows.)
int launch_vq_argmin_exact(const float* z, int64_t N, int D, int64_t HW, const float* E, int K, long long* idx, cudaStream_t st) {
    const int* list = nullptr;
    const unsigned int* list_count = nullptr;
    const int sms = sm_count();
    MOVAE_REQUIRE(sms > 0, MOVAE_ERR_CUDA, "CUDA device query failed (no GPU?)");
    const size_t staged = ((size_t)kExWarps * 4 * (D + K) + K + (size_t)D * (K + 1)) * sizeof(float);
    const size_t plain = ((size_t)kExWarps * 1 * (D + K) + K) * sizeof(float);
    const bool stage = staged <= kExMaxSmem && D % 1 == 0;
    MOVAE_REQUIRE(stage || plain <= kExMaxSmem, MOVAE_ERR_UNSUPPORTED, "vq_argmin: K=%d, D=%d too large for the exact kernel", K, D);
    const int R = stage ? 4 : 1;
    int64_t grid = ((N + R - 1) / R + kExWarps - 1) / kExWarps;
    const int64_t cap = stage ? (int64_t)sms : (int64_t)sms * 4;
    if (grid > cap) grid = cap;
    if (grid < 1) grid = 1;
    const int rc = stage ? allow_dynamic_smem<vq_argmin_exact_kernel<true, 4>>((int)kExMaxSmem)
                         : allow_dynamic_smem<vq_argmin_exact_kernel<false, 1>>((int)kExMaxSmem);
    if (rc != MOVAE_OK) return rc;
    if (stage)
        vq_argmin_exact_kernel<true, 4><<<(unsigned)grid, kExThreads, staged, st>>>(z, N, D, HW, E, K, list, list_count, idx);
    else
        vq_argmin_exact_kernel<false, 1><<<(unsigned)grid, kExThreads, plain, st>>>(z, N, D, HW, E, K, list, list_count, idx);
    MOVAE_CUDA_TRY(cudaGetLastError());
    return MOVAE_OK;
}

}  // namespace movae
