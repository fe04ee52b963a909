// K3 `recombine_writeback`:  grad (=|+=) w @ J   for float32 J[k, P], w[k] resident on the device.
//
// Replaces torchjd `WeightedAggregator.forward` (`weights @ J`, cuBLAS SGEMV in the reference) fused
// with the split / reshape / `param.grad = slice.clone()` (or `+=`) chain that follows it (call sites
// /root/reference/main.py:189-196): the parameters' .grad tensors are views of ONE flat buffer, so
// the write-back is a single streaming store of that buffer instead of one copy kernel per tensor.
//
// Roofline: HBM.  Algorithmic traffic 4*k*P read + 4*P written (+4*P read when accumulating).
// J is walked from its END backwards: K1 just streamed J front-to-back, so the last ~100 MB of it are still
// L2-resident on a 126 MB L2 and are consumed first.
#include "recombine_device.cuh"

namespace movae {

template <int K, int U, bool VEC>
__global__ void __launch_bounds__(kRecThreads)
recombine_kernel(const float* __restrict__ J, int64_t P, int64_t ldJ, const float* __restrict__ w_dev,
                 float* __restrict__ out, int accumulate) {
    recombine_tiles<K, U, VEC>(J, P, ldJ, w_dev, out, accumulate, [] {});
}

template <int K, int U, bool VEC>
static int launch_recombine(const float* J, int64_t P, int64_t ldJ, const float* w, float* out, int accumulate,
                            cudaStream_t st) {
    const int64_t tile_items = (int64_t)kRecThreads * U;
    unsigned int grid = 0;
    const int rc = persistent_grid<recombine_kernel<K, U, VEC>>(kRecThreads, (P / (VEC ? 4 : 1) + tile_items - 1) / tile_items,
                                                                INT64_MAX, &grid);
    if (rc != MOVAE_OK) return rc;
    recombine_kernel<K, U, VEC><<<grid, kRecThreads, 0, st>>>(J, P, ldJ, w, out, accumulate);
    MOVAE_CUDA_TRY(cudaGetLastError());
    return MOVAE_OK;
}

}  // namespace movae

extern "C" int movae_recombine_f32(const float* d_J, int k, int64_t P, int64_t ldJ, const float* d_w, float* d_grad,
                                   int accumulate, void* stream) {
    using namespace movae;
    MOVAE_REQUIRE(k >= 1, MOVAE_ERR_INVALID, "recombine: k must be >= 1 (got %d)", k);
    MOVAE_REQUIRE(k <= MOVAE_MAX_K, MOVAE_ERR_UNSUPPORTED, "recombine: k=%d > MOVAE_MAX_K=%d", k, MOVAE_MAX_K);
    MOVAE_REQUIRE(P >= 0 && ldJ >= P, MOVAE_ERR_INVALID, "recombine: need 0 <= P <= ldJ");
    if (P == 0) return MOVAE_OK;
    MOVAE_REQUIRE(d_J && d_w && d_grad, MOVAE_ERR_INVALID, "recombine: null pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool vec = (reinterpret_cast<uintptr_t>(d_J) % 16 == 0) && (reinterpret_cast<uintptr_t>(d_grad) % 16 == 0) &&
                     (ldJ % 4 == 0 || k == 1);
    return dispatch_k(k, [&](auto kc) {
        constexpr int K = decltype(kc)::value;
        if (vec) {
            if constexpr (K <= 4) return launch_recombine<K, 4, true>(d_J, P, ldJ, d_w, d_grad, accumulate, st);
            else return launch_recombine<K, 2, true>(d_J, P, ldJ, d_w, d_grad, accumulate, st);
        } else {
            if constexpr (K <= 4) return launch_recombine<K, 8, false>(d_J, P, ldJ, d_w, d_grad, accumulate, st);
            else return launch_recombine<K, 4, false>(d_J, P, ldJ, d_w, d_grad, accumulate, st);
        }
    });
}
