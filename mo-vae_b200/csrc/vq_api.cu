// C-ABI entry points of the VQ quantizer path (declared in include/movae_b200.h).
#include "common.cuh"
#include "vq_common.cuh"

namespace movae {

// launchers defined in vq_argmin_tc.cu / vq_argmin_exact.cu / vq_gather.cu / vq_backward.cu
int launch_vq_argmin_tc(const float* z, int64_t N, int64_t HW, const float* E, long long* idx, unsigned int* ws_words, float* dbg,
                        cudaStream_t st);
int launch_vq_argmin_exact(const float* z, int64_t N, int D, int64_t HW, const float* E, int K, long long* idx, cudaStream_t st);
int launch_vq_gather(const float* z, int64_t N, int D, int64_t HW, const float* E, int K, const long long* idx,
                     float* q_out, float* loss_out, int* usage_out, unsigned char* ws, cudaStream_t st);
int launch_vq_usage(const long long* idx, int64_t n, int K, int* usage_out, unsigned char* ws, cudaStream_t st);
int launch_vq_backward(const float* grad_out, const float* g_commit, const float* g_embed, const float* z, int64_t N, int D,
                       int64_t HW, const float* E, int K, const long long* idx, float* dz, float* dE, float* partials,
                       cudaStream_t st);
int launch_vq_pack_codes(const long long* idx, int64_t n, int K, void* out, int code_bytes, unsigned int* bitmap, cudaStream_t st);
int launch_vq_bitmap_count(const unsigned int* bitmap, int K, int* count, cudaStream_t st);
int vq_backward_parts(int64_t n_rows, int K, int D);
size_t vq_backward_part_bytes();
size_t vq_ema_workspace_bytes(int64_t n_rows, int K, int D);
int launch_vq_ema_stats(const float* z, int64_t N, int D, int64_t HW, const long long* idx, int K, float* stats, unsigned char* ws,
                        cudaStream_t st);
int launch_vq_ema_apply(const float* stats, int K, int D, double decay, double eps, float* E, float* cluster_size, float* embed_avg,
                        float* E_prev, unsigned char* ws, cudaStream_t st);
int launch_vq_ema_update(const float* z, int64_t N, int D, int64_t HW, const long long* idx, int K, double decay, double eps, float* E,
                         float* cluster_size, float* embed_avg, float* E_prev, unsigned char* ws, cudaStream_t st);

constexpr size_t kVqWsListOff = kWsListOff;
constexpr int kVqMaxK = 65536;

static int check_shape(const char* what, int64_t B, int D, int64_t HW, int K) {
    MOVAE_REQUIRE(B >= 0 && HW >= 1 && D >= 1 && K >= 1, MOVAE_ERR_INVALID, "%s: bad shape B=%lld D=%d HW=%lld K=%d", what,
                  (long long)B, D, (long long)HW, K);
    MOVAE_REQUIRE(K <= kVqMaxK, MOVAE_ERR_UNSUPPORTED, "%s: num_embeddings %d > %d", what, K, kVqMaxK);
    MOVAE_REQUIRE(B * HW < ((int64_t)1 << 31), MOVAE_ERR_UNSUPPORTED, "%s: more than 2^31 code vectors", what);
    return MOVAE_OK;
}

static int check_ema(const char* what, double decay, double eps, const float* E, const float* cs, const float* ea,
                     const float* E_prev, const void* ws, size_t ws_bytes, size_t need) {
    MOVAE_REQUIRE(decay >= 0.0 && decay < 1.0, MOVAE_ERR_INVALID, "%s: decay must be in [0, 1), got %g", what, decay);
    MOVAE_REQUIRE(eps > 0.0, MOVAE_ERR_INVALID, "%s: epsilon must be > 0, got %g", what, eps);
    MOVAE_REQUIRE(E && cs && ea && E_prev, MOVAE_ERR_INVALID, "%s: null pointer", what);
    MOVAE_REQUIRE(E != E_prev && E != ea && ea != E_prev, MOVAE_ERR_INVALID, "%s: codebook, embed_avg and the pre-update copy must not alias", what);
    MOVAE_REQUIRE(ws != nullptr && ws_bytes >= need, MOVAE_ERR_WORKSPACE, "%s: workspace too small (%zu < %zu)", what, ws_bytes, need);
    MOVAE_REQUIRE(reinterpret_cast<uintptr_t>(ws) % 16 == 0, MOVAE_ERR_WORKSPACE, "%s: workspace must be 16-byte aligned", what);
    return MOVAE_OK;
}

}  // namespace movae

extern "C" {

int movae_vq_tensor_path_supported(int K, int D) { return (K == 512 && D == 64) ? 1 : 0; }

size_t movae_vq_workspace_bytes(int64_t n_rows, int K, int D) {
    (void)D;
    if (n_rows < 0 || K < 1 || K > movae::kVqMaxK) return 0;
    return movae::kVqWsListOff;      // header + usage bitmap + K5 partial sums; nothing per row any more
}

int movae_vq_argmin_f32(const float* d_z, int64_t B, int D, int64_t HW, const float* d_E, int K, int64_t* d_idx, int mode,
                        float* d_dbg_scores, void* d_ws, size_t ws_bytes, void* stream) {
    using namespace movae;
    const int rc = check_shape("vq_argmin", B, D, HW, K);
    if (rc != MOVAE_OK) return rc;
    const int64_t N = B * HW;
    if (N == 0) return MOVAE_OK;
    MOVAE_REQUIRE(d_z && d_E && d_idx, MOVAE_ERR_INVALID, "vq_argmin: null pointer");
    MOVAE_REQUIRE(mode >= MOVAE_VQ_AUTO && mode <= MOVAE_VQ_TENSOR, MOVAE_ERR_INVALID, "vq_argmin: bad mode %d", mode);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool tensor_ok = movae_vq_tensor_path_supported(K, D) && reinterpret_cast<uintptr_t>(d_E) % 16 == 0;
    if (mode == MOVAE_VQ_TENSOR)
        MOVAE_REQUIRE(tensor_ok, MOVAE_ERR_UNSUPPORTED, "vq_argmin: the tcgen05 path needs K=512, D=64 and a 16-byte aligned codebook");
    const bool use_tensor = (mode == MOVAE_VQ_TENSOR) || (mode == MOVAE_VQ_AUTO && tensor_ok);
    long long* idx = reinterpret_cast<long long*>(d_idx);
    if (!use_tensor) {
        MOVAE_REQUIRE(d_dbg_scores == nullptr, MOVAE_ERR_INVALID, "vq_argmin: debug scores exist only on the tensor path");
        return launch_vq_argmin_exact(d_z, N, D, HW, d_E, K, idx, st);
    }
    MOVAE_REQUIRE(d_ws != nullptr && ws_bytes >= movae_vq_workspace_bytes(N, K, D), MOVAE_ERR_WORKSPACE,
                  "vq_argmin: workspace too small (%zu < %zu)", ws_bytes, movae_vq_workspace_bytes(N, K, D));
    MOVAE_REQUIRE(reinterpret_cast<uintptr_t>(d_ws) % 16 == 0, MOVAE_ERR_WORKSPACE, "vq_argmin: workspace must be 16-byte aligned");
    // ONE launch: rows the tensor path cannot decide are re-evaluated exactly inside the kernel
    return launch_vq_argmin_tc(d_z, N, HW, d_E, idx, reinterpret_cast<unsigned int*>(d_ws), d_dbg_scores, st);
}

int movae_vq_gather_f32(const float* d_z, int64_t B, int D, int64_t HW, const float* d_E, int K, const int64_t* d_idx,
                        float* d_quantized, float* d_losses, int32_t* d_usage_count, void* d_ws, size_t ws_bytes, void* stream) {
    using namespace movae;
    const int rc = check_shape("vq_gather", B, D, HW, K);
    if (rc != MOVAE_OK) return rc;
    const int64_t N = B * HW;
    MOVAE_REQUIRE(N > 0, MOVAE_ERR_INVALID, "vq_gather: empty input (the reference's mse_loss of an empty tensor is NaN)");
    MOVAE_REQUIRE(d_z && d_E && d_idx && d_quantized && d_losses, MOVAE_ERR_INVALID, "vq_gather: null pointer");
    MOVAE_REQUIRE(d_ws != nullptr && ws_bytes >= movae_vq_workspace_bytes(0, K, D), MOVAE_ERR_WORKSPACE, "vq_gather: workspace too small");
    return launch_vq_gather(d_z, N, D, HW, d_E, K, reinterpret_cast<const long long*>(d_idx), d_quantized, d_losses,
                            reinterpret_cast<int*>(d_usage_count), static_cast<unsigned char*>(d_ws), static_cast<cudaStream_t>(stream));
}

int movae_vq_forward_f32(const float* d_z, int64_t B, int D, int64_t HW, const float* d_E, int K, int64_t* d_idx,
                         float* d_quantized, float* d_losses, int32_t* d_usage_count, int mode, void* d_ws, size_t ws_bytes,
                         void* stream) {
    const int rc = movae_vq_argmin_f32(d_z, B, D, HW, d_E, K, d_idx, mode, nullptr, d_ws, ws_bytes, stream);
    if (rc != MOVAE_OK) return rc;
    return movae_vq_gather_f32(d_z, B, D, HW, d_E, K, d_idx, d_quantized, d_losses, d_usage_count, d_ws, ws_bytes, stream);
}

size_t movae_vq_backward_workspace_bytes(int64_t n_rows, int K, int D) {
    if (n_rows < 0 || K < 1 || D < 1) return 0;
    return (size_t)movae::vq_backward_parts(n_rows, K, D) * movae::vq_backward_part_bytes();
}

int movae_vq_backward_f32(const float* d_grad_quantized, const float* d_g_commit, const float* d_g_embed, const float* d_z,
                          int64_t B, int D, int64_t HW, const float* d_E, int K, const int64_t* d_idx, float* d_dz, float* d_dE,
                          void* d_ws, size_t ws_bytes, void* stream) {
    using namespace movae;
    const int rc = check_shape("vq_backward", B, D, HW, K);
    if (rc != MOVAE_OK) return rc;
    const int64_t N = B * HW;
    if (N == 0) return MOVAE_OK;
    MOVAE_REQUIRE(d_z && d_E && d_idx, MOVAE_ERR_INVALID, "vq_backward: null pointer");
    MOVAE_REQUIRE(d_dz || d_dE, MOVAE_ERR_INVALID, "vq_backward: nothing to compute (both outputs null)");
    const size_t need = movae_vq_backward_workspace_bytes(N, K, D);
    if (d_dE != nullptr && d_g_embed != nullptr && need > 0) {
        MOVAE_REQUIRE(d_ws != nullptr && ws_bytes >= need, MOVAE_ERR_WORKSPACE, "vq_backward: workspace too small (%zu < %zu)",
                      ws_bytes, need);
        MOVAE_REQUIRE(reinterpret_cast<uintptr_t>(d_ws) % 16 == 0, MOVAE_ERR_WORKSPACE, "vq_backward: workspace must be 16-byte aligned");
    }
    return launch_vq_backward(d_grad_quantized, d_g_commit, d_g_embed, d_z, N, D, HW, d_E, K,
                              reinterpret_cast<const long long*>(d_idx), d_dz, d_dE, need > 0 ? static_cast<float*>(d_ws) : nullptr,
                              static_cast<cudaStream_t>(stream));
}

size_t movae_vq_ema_workspace_bytes(int64_t n_rows, int K, int D) {
    if (n_rows < 0 || K < 1 || K > movae::kVqMaxK || D < 1) return 0;
    return movae::vq_ema_workspace_bytes(n_rows, K, D);
}

int movae_vq_ema_update_f32(const float* d_z, int64_t B, int D, int64_t HW, const int64_t* d_idx, int K, double decay, double epsilon,
                            float* d_E, float* d_cluster_size, float* d_embed_avg, float* d_E_prev, void* d_ws, size_t ws_bytes,
                            void* stream) {
    using namespace movae;
    int rc = check_shape("vq_ema_update", B, D, HW, K);
    if (rc != MOVAE_OK) return rc;
    const int64_t N = B * HW;
    rc = check_ema("vq_ema_update", decay, epsilon, d_E, d_cluster_size, d_embed_avg, d_E_prev, d_ws, ws_bytes,
                   movae_vq_ema_workspace_bytes(N, K, D));
    if (rc != MOVAE_OK) return rc;
    MOVAE_REQUIRE(N > 0, MOVAE_ERR_INVALID, "vq_ema_update: empty input (no code vector to average)");
    MOVAE_REQUIRE(d_z && d_idx, MOVAE_ERR_INVALID, "vq_ema_update: null pointer");
    return launch_vq_ema_update(d_z, N, D, HW, reinterpret_cast<const long long*>(d_idx), K, decay, epsilon, d_E, d_cluster_size,
                                d_embed_avg, d_E_prev, static_cast<unsigned char*>(d_ws), static_cast<cudaStream_t>(stream));
}

int movae_vq_ema_stats_f32(const float* d_z, int64_t B, int D, int64_t HW, const int64_t* d_idx, int K, float* d_stats, void* d_ws,
                           size_t ws_bytes, void* stream) {
    using namespace movae;
    const int rc = check_shape("vq_ema_stats", B, D, HW, K);
    if (rc != MOVAE_OK) return rc;
    const int64_t N = B * HW;
    const size_t need = movae_vq_ema_workspace_bytes(N, K, D);
    MOVAE_REQUIRE(d_stats && (N == 0 || (d_z && d_idx)), MOVAE_ERR_INVALID, "vq_ema_stats: null pointer");
    MOVAE_REQUIRE(d_ws != nullptr && ws_bytes >= need, MOVAE_ERR_WORKSPACE, "vq_ema_stats: workspace too small (%zu < %zu)", ws_bytes, need);
    MOVAE_REQUIRE(reinterpret_cast<uintptr_t>(d_ws) % 16 == 0, MOVAE_ERR_WORKSPACE, "vq_ema_stats: workspace must be 16-byte aligned");
    return launch_vq_ema_stats(d_z, N, D, HW, reinterpret_cast<const long long*>(d_idx), K, d_stats, static_cast<unsigned char*>(d_ws),
                               static_cast<cudaStream_t>(stream));
}

int movae_vq_ema_apply_f32(const float* d_stats, int K, int D, double decay, double epsilon, float* d_E, float* d_cluster_size,
                           float* d_embed_avg, float* d_E_prev, void* d_ws, size_t ws_bytes, void* stream) {
    using namespace movae;
    MOVAE_REQUIRE(K >= 1 && K <= kVqMaxK && D >= 1, MOVAE_ERR_INVALID, "vq_ema_apply: bad shape K=%d D=%d", K, D);
    const int rc = check_ema("vq_ema_apply", decay, epsilon, d_E, d_cluster_size, d_embed_avg, d_E_prev, d_ws, ws_bytes,
                             movae_vq_ema_workspace_bytes(0, K, D));
    if (rc != MOVAE_OK) return rc;
    MOVAE_REQUIRE(d_stats != nullptr, MOVAE_ERR_INVALID, "vq_ema_apply: null pointer");
    return launch_vq_ema_apply(d_stats, K, D, decay, epsilon, d_E, d_cluster_size, d_embed_avg, d_E_prev, static_cast<unsigned char*>(d_ws),
                               static_cast<cudaStream_t>(stream));
}

int movae_vq_usage(const int64_t* d_idx, int64_t n, int K, int32_t* d_count, void* d_ws, size_t ws_bytes, void* stream) {
    using namespace movae;
    MOVAE_REQUIRE(n >= 0 && K >= 1, MOVAE_ERR_INVALID, "vq_usage: bad arguments");
    MOVAE_REQUIRE(K <= kVqMaxK, MOVAE_ERR_UNSUPPORTED, "vq_usage: num_embeddings %d > %d", K, kVqMaxK);
    MOVAE_REQUIRE(d_count && (d_idx || n == 0), MOVAE_ERR_INVALID, "vq_usage: null pointer");
    MOVAE_REQUIRE(d_ws != nullptr && ws_bytes >= movae_vq_workspace_bytes(0, K, 1), MOVAE_ERR_WORKSPACE, "vq_usage: workspace too small");
    return launch_vq_usage(reinterpret_cast<const long long*>(d_idx), n, K, reinterpret_cast<int*>(d_count),
                           static_cast<unsigned char*>(d_ws), static_cast<cudaStream_t>(stream));
}

int movae_vq_pack_codes(const int64_t* d_idx, int64_t n, int K, void* d_codes, int code_bytes, uint32_t* d_bitmap, void* stream) {
    using namespace movae;
    MOVAE_REQUIRE(n >= 0 && K >= 1, MOVAE_ERR_INVALID, "vq_pack_codes: bad arguments");
    MOVAE_REQUIRE(K <= kVqMaxK, MOVAE_ERR_UNSUPPORTED, "vq_pack_codes: num_embeddings %d > %d", K, kVqMaxK);
    MOVAE_REQUIRE(code_bytes == 2 || code_bytes == 4 || code_bytes == 8, MOVAE_ERR_INVALID, "vq_pack_codes: code_bytes must be 2, 4 or 8");
    MOVAE_REQUIRE(code_bytes > 2 || K <= 32768, MOVAE_ERR_INVALID, "vq_pack_codes: %d codes do not fit a signed 16-bit code", K);
    if (n == 0) return MOVAE_OK;
    MOVAE_REQUIRE(d_idx && d_codes, MOVAE_ERR_INVALID, "vq_pack_codes: null pointer");
    return launch_vq_pack_codes(reinterpret_cast<const long long*>(d_idx), n, K, d_codes, code_bytes, d_bitmap,
                                static_cast<cudaStream_t>(stream));
}

int movae_vq_bitmap_count(const uint32_t* d_bitmap, int K, int32_t* d_count, void* stream) {
    using namespace movae;
    MOVAE_REQUIRE(K >= 1 && K <= kVqMaxK, MOVAE_ERR_INVALID, "vq_bitmap_count: bad num_embeddings %d", K);
    MOVAE_REQUIRE(d_bitmap && d_count, MOVAE_ERR_INVALID, "vq_bitmap_count: null pointer");
    return launch_vq_bitmap_count(d_bitmap, K, reinterpret_cast<int*>(d_count), static_cast<cudaStream_t>(stream));
}

}  // extern "C"
