// VectorQuantizerEMA's codebook update (declared in include/movae_b200.h as movae_vq_ema_*).
#include "common.cuh"
#include "vq_common.cuh"

namespace movae {

// ==== VectorQuantizerEMA: exponential-moving-average codebook update ===================================================
// van den Oord et al. 2017, App. A.1, with the semantics of the `Quantize` module of rosinality/vq-vae-2-pytorch (the
// stored cluster_size is unsmoothed; the smoothing only enters the normalisation).  From the batch's indices, which were
// searched with the pre-update codebook E:
//     count_j = #{n : idx_n = j},   S_j = sum_{n : idx_n = j} z_n
//     cluster_size <- decay cluster_size + (1 - decay) count,   embed_avg <- decay embed_avg + (1 - decay) S
//     n = sum_j cluster_size_j,   E_j <- embed_avg_j / ((cluster_size_j + eps) / (n + K eps) n)
// and E_prev <- E before the update (what the backward of the straight-through output reads).  Everything after the
// statistics is float64, rounded once per stored value.
//   K = 512, D = 64: the statistics are K6b's per-CTA partials, unchanged (bit-reproducible); vq_ema_apply_kernel<true>
//     combines them with k6b_combine_partials, as vq_dE_reduce_kernel does.  Two launches, no host synchronisation.
//   Other (K, D), and a data-parallel caller that all-reduces the statistics between the two halves: float32 stats
//     [count (K) | S (K * D)].  The general stats kernel adds rows with float32 ATOMICS, so its result is NOT
//     bit-reproducible run to run (tolerance-only tests); at K = 512, D = 64 the stats come from the K6b partials.
//     The counts are float32 in that tensor: a code chosen by more than 2^24 rows of one (global) batch gets an inexact
//     count.  The fused K = 512, D = 64 update counts in integers and has no such limit.
// n needs every code's new cluster_size before any code can be normalised.  The apply kernel is a ticketed last-CTA
// finish: every CTA applies the EMA to its slice and copies E to E_prev, the last CTA to arrive sums cluster_size in a
// fixed order and normalises the whole [K, D] codebook.  A grid-wide barrier would need co-resident CTAs, and a separate
// normalisation launch would cost a third launch.  At K = 512, D = 64 (a 128 KB codebook) the whole update measured
// K6b + its reduce + a constant ~27 us at every N on a B200 (profiles/r3_vq_ema.md).  An offset independent of N points
// at this tail; that it is latency-bound (8 warps, one float4 per L2 round trip) is inferred, not profiled.  It streams K * D * 8 bytes on one SM, so it grows linearly with the codebook:
// K = 16384, D = 256 (16 MB each way) would take an estimated few hundred microseconds (not measured).
constexpr size_t kVqEmaHeaderBytes = 256;      // workspace: ticket (uint32, zero between launches) | stats | K6b partials

static size_t ema_stats_bytes(int K, int D) { return (((size_t)K + (size_t)K * D) * sizeof(float) + 15) / 16 * 16; }

size_t vq_ema_workspace_bytes(int64_t n_rows, int K, int D) {
    return kVqEmaHeaderBytes + ema_stats_bytes(K, D) + (size_t)vq_backward_parts(n_rows, K, D) * kPartFloats * sizeof(float);
}

// Split path at K = 512, D = 64: the K6b partials -> float32 stats [count | S] (what a data-parallel caller all-reduces).
__global__ void __launch_bounds__(kRdThreads)
vq_ema_partials_to_stats_kernel(const float* __restrict__ partials, int n_parts, float* __restrict__ stats) {
    const int q = threadIdx.x % kRdQuads, g = threadIdx.x / kRdQuads, quad = blockIdx.x * kRdQuads + q;
    double st[4];
    long long ct;
    k6b_combine_partials(partials, n_parts, quad, q, g, st, ct);
    if (g == 0 && quad < kBwK * kBwD / 4) {
        reinterpret_cast<float4*>(stats + kBwK)[quad] = make_float4((float)st[0], (float)st[1], (float)st[2], (float)st[3]);
        if (quad % (kBwD / 4) == 0) stats[quad * 4 / kBwD] = (float)ct;
    }
}

// General (K, D) statistics with float32 atomics into stats [count | S] (zeroed by the launcher).
__global__ void __launch_bounds__(256)
vq_ema_stats_atomic_kernel(const float* __restrict__ z, int64_t N, int D, int64_t HW, const long long* __restrict__ idx, int K,
                           float* __restrict__ stats) {
    for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (int64_t)gridDim.x * blockDim.x) {
        long long code = idx[n];
        code = code < 0 ? 0 : (code >= K ? K - 1 : code);
        const int64_t b = n / HW, hw = n - b * HW;
        const int64_t base = (b * D) * HW + hw;
        float* sp = stats + K + (size_t)code * D;
        atomicAdd(stats + code, 1.0f);
#pragma unroll 8
        for (int d = 0; d < D; ++d) atomicAdd(sp + d, ld_stream_f1(z + base + (int64_t)d * HW));
    }
}

// The EMA, then (last CTA) the normalisation.  PARTS: src = K6b partials (K = 512, D = 64; E, embed_avg, E_prev 16-byte
// aligned), one quad per group-0 thread.  Otherwise src = float32 stats [count | S], one element per thread.  vec: D % 4
// == 0 and E, embed_avg 16-byte aligned (float4 normalisation).
template <bool PARTS>
__global__ void __launch_bounds__(kRdThreads)
vq_ema_apply_kernel(const float* __restrict__ src, int n_parts, int K, int D, double decay, double eps, float* __restrict__ E,
                    float* __restrict__ cluster_size, float* __restrict__ embed_avg, float* __restrict__ E_prev,
                    unsigned int* __restrict__ ticket, int vec) {
    __shared__ double sm_n[kRdThreads];
    __shared__ int sm_last;
    const int tid = threadIdx.x;
    const double keep = decay, take = 1.0 - decay;
    const int64_t KD = (int64_t)K * D;
    if constexpr (PARTS) {
        const int q = tid % kRdQuads, g = tid / kRdQuads, quad = blockIdx.x * kRdQuads + q;
        double st[4];
        long long ct;
        k6b_combine_partials(src, n_parts, quad, q, g, st, ct);
        if (g == 0 && quad < kBwK * kBwD / 4) {
            float4 a = reinterpret_cast<const float4*>(embed_avg)[quad];
            a.x = (float)(keep * (double)a.x + take * st[0]);
            a.y = (float)(keep * (double)a.y + take * st[1]);
            a.z = (float)(keep * (double)a.z + take * st[2]);
            a.w = (float)(keep * (double)a.w + take * st[3]);
            reinterpret_cast<float4*>(embed_avg)[quad] = a;
            reinterpret_cast<float4*>(E_prev)[quad] = reinterpret_cast<const float4*>(E)[quad];
            if (quad % (kBwD / 4) == 0) {
                const int j = quad * 4 / kBwD;
                cluster_size[j] = (float)(keep * (double)cluster_size[j] + take * (double)ct);
            }
        }
    } else {
        for (int64_t i = (int64_t)blockIdx.x * kRdThreads + tid; i < KD; i += (int64_t)gridDim.x * kRdThreads) {
            embed_avg[i] = (float)(keep * (double)embed_avg[i] + take * (double)__ldg(src + K + i));
            E_prev[i] = E[i];
            if (i % D == 0) {
                const int64_t j = i / D;
                cluster_size[j] = (float)(keep * (double)cluster_size[j] + take * (double)__ldg(src + j));
            }
        }
    }
    __threadfence();                          // this CTA's cluster_size / embed_avg / E_prev stores, before its ticket
    __syncthreads();
    if (tid == 0) sm_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!sm_last) return;
    __threadfence();
    // the last CTA: n in a fixed order (strided partial sums, then a fixed tree), then E_j = embed_avg_j / smoothed_j
    double part = 0.0;
    for (int j = tid; j < K; j += kRdThreads) part += (double)__ldcg(cluster_size + j);
    sm_n[tid] = part;
    __syncthreads();
    for (int w = kRdThreads / 2; w > 0; w >>= 1) {
        if (tid < w) sm_n[tid] += sm_n[tid + w];
        __syncthreads();
    }
    const double n = sm_n[0], nk = n + (double)K * eps;
    if (vec) {
#pragma unroll 4
        for (int64_t i4 = tid; i4 < KD / 4; i4 += kRdThreads) {
            const int64_t j = i4 * 4 / D;
            const double sm = ((double)__ldcg(cluster_size + j) + eps) / nk * n;
            const float4 a = __ldcg(reinterpret_cast<const float4*>(embed_avg) + i4);
            reinterpret_cast<float4*>(E)[i4] = make_float4((float)((double)a.x / sm), (float)((double)a.y / sm),
                                                           (float)((double)a.z / sm), (float)((double)a.w / sm));
        }
    } else {
        for (int64_t i = tid; i < KD; i += kRdThreads) {
            const double sm = ((double)__ldcg(cluster_size + i / D) + eps) / nk * n;
            E[i] = (float)((double)__ldcg(embed_avg + i) / sm);
        }
    }
    if (tid == 0) *ticket = 0u;               // every other CTA has taken its ticket: the next launch starts from 0
}

static bool aligned16(const void* p) { return reinterpret_cast<uintptr_t>(p) % 16 == 0; }

// K6b's partials for K = 512, D = 64 into the workspace, after the stats region.  Needs N > 0.
static int ema_partials(const float* z, int64_t N, int64_t HW, const long long* idx, unsigned char* ws, float** partials, int* n_parts,
                        cudaStream_t st) {
    MOVAE_REQUIRE(sm_count() > 0, MOVAE_ERR_CUDA, "CUDA device query failed (no GPU?)");
    *partials = reinterpret_cast<float*>(ws + kVqEmaHeaderBytes + ema_stats_bytes(kBwK, kBwD));
    return launch_k6b_partials(z, N, HW, idx, *partials, n_parts, st);
}

int launch_vq_ema_stats(const float* z, int64_t N, int D, int64_t HW, const long long* idx, int K, float* stats, unsigned char* ws,
                        cudaStream_t st) {
    const int sms = sm_count();
    MOVAE_REQUIRE(sms > 0, MOVAE_ERR_CUDA, "CUDA device query failed (no GPU?)");
    if (K == kBwK && D == kBwD && N > 0 && aligned16(stats)) {
        float* partials = nullptr;
        int parts = 0;
        const int rc = ema_partials(z, N, HW, idx, ws, &partials, &parts, st);
        if (rc != MOVAE_OK) return rc;
        vq_ema_partials_to_stats_kernel<<<(kBwK * kBwD / 4 + kRdQuads - 1) / kRdQuads, kRdThreads, 0, st>>>(partials, parts, stats);
        MOVAE_CUDA_TRY(cudaGetLastError());
        return MOVAE_OK;
    }
    MOVAE_CUDA_TRY(cudaMemsetAsync(stats, 0, ((size_t)K + (size_t)K * D) * sizeof(float), st));
    if (N == 0) return MOVAE_OK;
    int64_t grid = (N + 255) / 256;
    if (grid > (int64_t)sms * 8) grid = (int64_t)sms * 8;
    vq_ema_stats_atomic_kernel<<<(unsigned)grid, 256, 0, st>>>(z, N, D, HW, idx, K, stats);
    MOVAE_CUDA_TRY(cudaGetLastError());
    return MOVAE_OK;
}

int launch_vq_ema_apply(const float* stats, int K, int D, double decay, double eps, float* E, float* cluster_size, float* embed_avg,
                        float* E_prev, unsigned char* ws, cudaStream_t st) {
    const int sms = sm_count();
    MOVAE_REQUIRE(sms > 0, MOVAE_ERR_CUDA, "CUDA device query failed (no GPU?)");
    const int64_t KD = (int64_t)K * D;
    int64_t grid = (KD + kRdThreads - 1) / kRdThreads;
    if (grid > (int64_t)sms * 4) grid = (int64_t)sms * 4;
    const int vec = D % 4 == 0 && aligned16(E) && aligned16(embed_avg);
    vq_ema_apply_kernel<false><<<(unsigned)grid, kRdThreads, 0, st>>>(stats, 0, K, D, decay, eps, E, cluster_size, embed_avg, E_prev,
                                                                     reinterpret_cast<unsigned int*>(ws), vec);
    MOVAE_CUDA_TRY(cudaGetLastError());
    return MOVAE_OK;
}

int launch_vq_ema_update(const float* z, int64_t N, int D, int64_t HW, const long long* idx, int K, double decay, double eps, float* E,
                         float* cluster_size, float* embed_avg, float* E_prev, unsigned char* ws, cudaStream_t st) {
    if (K == kBwK && D == kBwD && aligned16(E) && aligned16(embed_avg) && aligned16(E_prev)) {
        float* partials = nullptr;
        int parts = 0;
        const int rc = ema_partials(z, N, HW, idx, ws, &partials, &parts, st);
        if (rc != MOVAE_OK) return rc;
        vq_ema_apply_kernel<true><<<(kBwK * kBwD / 4 + kRdQuads - 1) / kRdQuads, kRdThreads, 0, st>>>(
            partials, parts, K, D, decay, eps, E, cluster_size, embed_avg, E_prev, reinterpret_cast<unsigned int*>(ws), 1);
        MOVAE_CUDA_TRY(cudaGetLastError());
        return MOVAE_OK;
    }
    float* stats = reinterpret_cast<float*>(ws + kVqEmaHeaderBytes);
    const int rc = launch_vq_ema_stats(z, N, D, HW, idx, K, stats, ws, st);
    if (rc != MOVAE_OK) return rc;
    return launch_vq_ema_apply(stats, K, D, decay, eps, E, cluster_size, embed_avg, E_prev, ws, st);
}

}  // namespace movae
