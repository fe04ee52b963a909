// K1 `gram_stream`:  G = J J^T  for a float32 row-major Jacobian J[k, P] (k <= 8 objectives).
//
// Replaces torchjd `compute_gramian` (`J @ J.T`, a cuBLAS SGEMM with M=N=k in the reference; call
// sites /root/reference/main.py:189-196 through GramianWeightedAggregator, aligned_mtl.py:39,
// mgda.py:12, nupgrad.py:37).
//
// Roofline: HBM.  Algorithmic traffic 4*k*P bytes read, k*k doubles written.  One pass:
//   * persistent grid (SMs x resident CTAs), CTA tile = 256 threads x U float4 per row, every warp
//     load instruction covers 512 contiguous bytes of one row, all k rows of a tile are in flight
//     together (k*U independent 16-byte loads per thread);
//   * k(k+1)/2 float32 FMA chains per thread, at most 64 columns long, then promoted into float64
//     registers (the reference's own float32 SGEMM is 3e-5..8e-3 off at P=2.4M..1e8, SURVEY App. C.2;
//     the parity contract is rtol 1e-5 against a float64-accumulated oracle);
//   * warp shuffle -> shared memory -> one partial per CTA -> the last CTA to finish (atomic ticket)
//     sums the partials in a fixed order: bit-reproducible for a given (k, P, grid), no float atomics.
#include "gram_device.cuh"

namespace movae {

template <int K, int U, bool VEC, int MINB>
__global__ void __launch_bounds__(kGramThreads, MINB)
gram_kernel(const float* __restrict__ J, int64_t P, int64_t ldJ, double* __restrict__ partials,
            unsigned int* __restrict__ counter, double* __restrict__ G, int accumulate) {
    constexpr int NACC = GramAcc<K>::N;
    double acc64[NACC];
#pragma unroll
    for (int a = 0; a < NACC; ++a) acc64[a] = 0.0;
    gram_stream_tiles<K, U, VEC>(J, P, ldJ, acc64);

    __shared__ double red[kGramThreads / 32][NACC];
    __shared__ double Gs[K * K];
    __shared__ int is_last;
    if (!gram_cta_partial_and_ticket<K>(acc64, partials, counter, red, &is_last)) return;
    gram_combine_partials<K>(partials, Gs);
    const int tid = threadIdx.x;
    if (tid < K * K) {
        if (accumulate) G[tid] += Gs[tid];
        else G[tid] = Gs[tid];
    }
    if (tid == 0) *counter = 0u;   // self-reset: the workspace is reusable by the next launch
}

template <int K, int U, bool VEC, int MINB>
static int launch_gram(const float* J, int64_t P, int64_t ldJ, double* G, int accumulate, void* ws, cudaStream_t st) {
    const int64_t tile_items = (int64_t)kGramThreads * U;
    unsigned int grid = 0;
    const int rc = persistent_grid<gram_kernel<K, U, VEC, MINB>>(kGramThreads, (P / (VEC ? 4 : 1) + tile_items - 1) / tile_items,
                                                                 kGramMaxBlocks, &grid);
    if (rc != MOVAE_OK) return rc;
    const GramWorkspace w(ws);
    gram_kernel<K, U, VEC, MINB><<<grid, kGramThreads, 0, st>>>(J, P, ldJ, w.partials, w.ticket, G, accumulate);
    MOVAE_CUDA_TRY(cudaGetLastError());
    return MOVAE_OK;
}

}  // namespace movae

extern "C" {

size_t movae_gram_workspace_bytes(int k) {
    if (k < 1 || k > MOVAE_MAX_K) return 0;
    return (size_t)movae::kGramHeaderBytes + (size_t)movae::kGramMaxBlocks * (k * (k + 1) / 2) * sizeof(double);
}

static int gram_entry(const float* d_J, int k, int64_t P, int64_t ldJ, double* d_G, int accumulate, void* d_ws, size_t ws_bytes,
                      void* stream) {
    using namespace movae;
    MOVAE_REQUIRE(k >= 1, MOVAE_ERR_INVALID, "gram: k must be >= 1 (got %d)", k);
    MOVAE_REQUIRE(k <= MOVAE_MAX_K, MOVAE_ERR_UNSUPPORTED, "gram: k=%d > MOVAE_MAX_K=%d", k, MOVAE_MAX_K);
    MOVAE_REQUIRE(P >= 0 && ldJ >= P, MOVAE_ERR_INVALID, "gram: need 0 <= P <= ldJ (P=%lld ldJ=%lld)", (long long)P,
                  (long long)ldJ);
    MOVAE_REQUIRE(d_G != nullptr && (d_J != nullptr || P == 0), MOVAE_ERR_INVALID, "gram: null pointer");
    MOVAE_REQUIRE(d_ws != nullptr && ws_bytes >= movae_gram_workspace_bytes(k), MOVAE_ERR_WORKSPACE,
                  "gram: workspace too small (%zu < %zu)", ws_bytes, movae_gram_workspace_bytes(k));
    MOVAE_REQUIRE(reinterpret_cast<uintptr_t>(d_ws) % 8 == 0, MOVAE_ERR_WORKSPACE, "gram: workspace must be 8-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool vec = (reinterpret_cast<uintptr_t>(d_J) % 16 == 0) && (ldJ % 4 == 0 || k == 1);
    // registers: float64 accumulators cost 2*K(K+1)/2; small k affords deeper unroll and 2+ CTAs/SM
    return dispatch_k(k, [&](auto kc) {
        constexpr int K = decltype(kc)::value;
        if (vec) {
            if constexpr (K <= 2) return launch_gram<K, 8, true, 2>(d_J, P, ldJ, d_G, accumulate, d_ws, st);
            else if constexpr (K <= 4) return launch_gram<K, 4, true, 2>(d_J, P, ldJ, d_G, accumulate, d_ws, st);
            else return launch_gram<K, 2, true, 1>(d_J, P, ldJ, d_G, accumulate, d_ws, st);
        } else {
            if constexpr (K <= 4) return launch_gram<K, 8, false, 2>(d_J, P, ldJ, d_G, accumulate, d_ws, st);
            else return launch_gram<K, 4, false, 1>(d_J, P, ldJ, d_G, accumulate, d_ws, st);
        }
    });
}

int movae_gram_f32(const float* d_J, int k, int64_t P, int64_t ldJ, double* d_G, int accumulate, void* d_ws,
                   size_t ws_bytes, void* stream) {
    return gram_entry(d_J, k, P, ldJ, d_G, accumulate, d_ws, ws_bytes, stream);
}

}  // extern "C"
