// K5 `vq_gather_loss_ste`, the codebook-usage bitmap and the code-packing kernel of the bulk extraction path
// (K6 `vq_backward` lives in vq_backward.cu).
//
// K5 replaces, in /root/reference/models/vq_vae.py: the one-hot scatter (:43-44), the dense
// `one_hot @ E` gather GEMM (:47), both `F.mse_loss` reductions (:51-52, the same value twice), the
// straight-through add `z + (q - z)` (:55), the NHWC->NCHW permute (:57) and the `torch.unique`
// behind the usage helpers (:110-124) with ONE pass over z:
//     reads 4D B (z) + 8 B (idx) per code vector, writes 4D B (quantized, NCHW)  => HBM-bound.
//
// Thread-per-row mapping: consecutive threads own consecutive (b, h, w) positions, so every NCHW
// access is a coalesced 128-byte line per warp and channel; codebook rows are read from a padded
// shared-memory copy (stride D+1: conflict-free for arbitrary indices) when it fits.
#include <math.h>

#include "common.cuh"
#include "vq_common.cuh"

namespace movae {

constexpr int kGatherThreads = 512;
constexpr int kVqMaxPartials = 2048;


template <bool STAGE, int THREADS>
__global__ void __launch_bounds__(THREADS, 1)
vq_gather_kernel(const float* __restrict__ z, int64_t N, int D, int64_t HW, const float* __restrict__ E, int K,
                 const long long* __restrict__ idx, float* __restrict__ q_out, float* __restrict__ loss_out,
                 int* __restrict__ usage_out, unsigned char* __restrict__ ws) {
    extern __shared__ float Es[];                           // STAGE: K x (D+1)
    __shared__ unsigned int bm[kVqMaxCodes / 32];
    __shared__ double red[THREADS / 32];
    __shared__ int is_last;
    const int tid = threadIdx.x;
    const int words = (K + 31) / 32;
    unsigned int* g_bm = reinterpret_cast<unsigned int*>(ws + kWsBitmapOff);
    double* partials = reinterpret_cast<double*>(ws + kWsPartialOff);
    unsigned int* ticket = reinterpret_cast<unsigned int*>(ws + 4);

    for (int i = tid; i < words; i += THREADS) bm[i] = 0u;
    if (STAGE) {
        for (int i = tid; i < K * D; i += THREADS) {
            const int j = i / D, d = i - j * D;
            Es[j * (D + 1) + d] = __ldg(E + i);
        }
    }
    __syncthreads();

    double acc64 = 0.0;
    for (int64_t n0 = (int64_t)blockIdx.x * THREADS; n0 < N; n0 += (int64_t)gridDim.x * THREADS) {
        const int64_t n = n0 + tid;
        if (n < N) {
            long long code = idx[n];
            code = code < 0 ? 0 : (code >= K ? K - 1 : code);
            atomicOr(&bm[code >> 5], 1u << (code & 31));
            const int64_t b = n / HW, hw = n - b * HW;
            const float* zp = z + (b * D) * HW + hw;
            float* qp = q_out + (b * D) * HW + hw;
            const float* ep = STAGE ? Es + (size_t)code * (D + 1) : E + (size_t)code * D;
            float acc = 0.f;
            int d0 = 0;
            // batches of 16 channels, software-pipelined: the loads of batch i + 1 are issued before batch i is combined and
            // stored, so a thread always has 16-32 loads in flight (with one batch at a time the bytes in flight per SM swung
            // between 64 KB and 0 and the kernel sat at 0.86 of the HBM peak)
            float za[16], zb[16];
            const int n_batches = D / 16;
            if (n_batches > 0) {
#pragma unroll
                for (int i = 0; i < 16; ++i) za[i] = __ldcs(zp + (int64_t)i * HW);
            }
            for (int bt = 0; bt < n_batches; bt += 2, d0 += 32) {
                const bool has_b = bt + 1 < n_batches;
                if (has_b) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) zb[i] = __ldcs(zp + (int64_t)(d0 + 16 + i) * HW);
                }
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const float qv = STAGE ? ep[d0 + i] : __ldg(ep + d0 + i);
                    const float diff = __fsub_rn(qv, za[i]);          // (q - z) rounded to float32 like the reference
                    acc = fmaf(diff, diff, acc);
                    __stcs(qp + (int64_t)(d0 + i) * HW, __fadd_rn(za[i], diff));   // straight-through value z + (q - z)
                }
                if (!has_b) { d0 += 16; break; }
                if (bt + 2 < n_batches) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) za[i] = __ldcs(zp + (int64_t)(d0 + 32 + i) * HW);
                }
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const float qv = STAGE ? ep[d0 + 16 + i] : __ldg(ep + d0 + 16 + i);
                    const float diff = __fsub_rn(qv, zb[i]);
                    acc = fmaf(diff, diff, acc);
                    __stcs(qp + (int64_t)(d0 + 16 + i) * HW, __fadd_rn(zb[i], diff));
                }
            }
            for (; d0 < D; ++d0) {
                const float zv = __ldcs(zp + (int64_t)d0 * HW);
                const float qv = STAGE ? ep[d0] : __ldg(ep + d0);
                const float diff = __fsub_rn(qv, zv);
                acc = fmaf(diff, diff, acc);
                __stcs(qp + (int64_t)d0 * HW, __fadd_rn(zv, diff));
            }
            acc64 += (double)acc;
        }
    }

    // ---- CTA reduce + deterministic cross-CTA combine (ticket, fixed order) -------------------------
    const int warp = tid >> 5, lane = tid & 31;
    const double s = warp_sum(acc64);
    if (lane == 0) red[warp] = s;
    __syncthreads();
    if (tid == 0) {
        double t = 0.0;
        for (int w = 0; w < THREADS / 32; ++w) t += red[w];
        partials[blockIdx.x] = t;
    }
    for (int i = tid; i < words; i += THREADS)
        if (bm[i]) atomicOr(&g_bm[i], bm[i]);
    __threadfence();
    __syncthreads();
    if (tid == 0) is_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    if (warp == 0) {
        double t = 0.0;
        for (int b = lane; b < (int)gridDim.x; b += 32) t += __ldcg(&partials[b]);
        t = warp_sum(t);
        int used = 0;
        for (int i = lane; i < words; i += 32) {
            used += __popc(__ldcg(&g_bm[i]));
            g_bm[i] = 0u;                                    // leave the bitmap clean for the next call
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) used += __shfl_xor_sync(0xffffffffu, used, o);
        if (lane == 0) {
            const float loss = (float)(t / ((double)N * (double)D));
            loss_out[0] = loss;                              // commitment_loss  (vq_vae.py:51)
            loss_out[1] = loss;                              // embedding_loss   (vq_vae.py:52)
            if (usage_out) *usage_out = used;
            *ticket = 0u;
        }
    }
}

// codebook usage of an arbitrary index tensor (vq_vae.py:110-124): |unique(idx)|
__global__ void __launch_bounds__(256)
vq_usage_kernel(const long long* __restrict__ idx, int64_t n, int K, int* __restrict__ usage_out,
                unsigned char* __restrict__ ws) {
    unsigned int* g_bm = reinterpret_cast<unsigned int*>(ws + kWsBitmapOff);
    unsigned int* ticket = reinterpret_cast<unsigned int*>(ws + 8);
    __shared__ int is_last;
    const int words = (K + 31) / 32;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const long long code = idx[i];
        if (code >= 0 && code < K) atomicOr(&g_bm[code >> 5], 1u << (code & 31));
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    if (threadIdx.x < 32) {
        int used = 0;
        for (int i = threadIdx.x; i < words; i += 32) {
            used += __popc(__ldcg(&g_bm[i]));
            g_bm[i] = 0u;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) used += __shfl_xor_sync(0xffffffffu, used, o);
        if (threadIdx.x == 0) {
            *usage_out = used;
            *ticket = 0u;
        }
    }
}


int launch_vq_gather(const float* z, int64_t N, int D, int64_t HW, const float* E, int K, const long long* idx,
                     float* q_out, float* loss_out, int* usage_out, unsigned char* ws, cudaStream_t st) {
    const int sms = sm_count();
    MOVAE_REQUIRE(sms > 0, MOVAE_ERR_CUDA, "CUDA device query failed (no GPU?)");
    int64_t grid = (N + kGatherThreads - 1) / kGatherThreads;
    if (grid > sms) grid = sms;
    if (grid > kVqMaxPartials) grid = kVqMaxPartials;
    if (grid < 1) grid = 1;
    const size_t stage_bytes = (size_t)K * (D + 1) * sizeof(float);
    if (N <= kSmallN) {
        // small batches (the BASELINE model shapes): staging the codebook per CTA (~10 us) would dominate; many small
        // CTAs read the codebook rows through L1/L2 instead
        int64_t g = (N + 255) / 256;
        if (g > kVqMaxPartials) g = kVqMaxPartials;
        vq_gather_kernel<false, 256><<<(unsigned)g, 256, 0, st>>>(z, N, D, HW, E, K, idx, q_out, loss_out, usage_out, ws);
        MOVAE_CUDA_TRY(cudaGetLastError());
        return MOVAE_OK;
    }
    if (stage_bytes <= 160 * 1024) {
        const int rc = allow_dynamic_smem<vq_gather_kernel<true, kGatherThreads>>(160 * 1024);
        if (rc != MOVAE_OK) return rc;
        vq_gather_kernel<true, kGatherThreads><<<(unsigned)grid, kGatherThreads, stage_bytes, st>>>(z, N, D, HW, E, K, idx, q_out,
                                                                                                 loss_out, usage_out, ws);
    } else {
        vq_gather_kernel<false, kGatherThreads><<<(unsigned)grid, kGatherThreads, 0, st>>>(z, N, D, HW, E, K, idx, q_out, loss_out,
                                                                                        usage_out, ws);
    }
    MOVAE_CUDA_TRY(cudaGetLastError());
    return MOVAE_OK;
}

// Bulk code extraction (SURVEY 8f rank 3): narrow the int64 indices to CODE bytes for the D2H copy and OR the batch's codes
// into a caller-owned K-bit bitmap that persists ACROSS batches (replaces the host-side cat + torch.unique of main.py:261-330).
template <typename CODE>
__global__ void __launch_bounds__(256)
vq_pack_codes_kernel(const long long* __restrict__ idx, int64_t n, int K, CODE* __restrict__ out, unsigned int* __restrict__ bitmap) {
    __shared__ unsigned int bm[kVqMaxCodes / 32];
    const int words = (K + 31) / 32;
    if (bitmap != nullptr)
        for (int i = threadIdx.x; i < words; i += blockDim.x) bm[i] = 0u;
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        long long code = __ldcs(idx + i);
        code = code < 0 ? 0 : (code >= K ? K - 1 : code);
        out[i] = (CODE)code;
        if (bitmap != nullptr) atomicOr(&bm[code >> 5], 1u << (code & 31));
    }
    if (bitmap != nullptr) {
        __syncthreads();
        for (int i = threadIdx.x; i < words; i += blockDim.x)
            if (bm[i]) atomicOr(&bitmap[i], bm[i]);
    }
}

__global__ void __launch_bounds__(32)
vq_bitmap_count_kernel(const unsigned int* __restrict__ bitmap, int K, int* __restrict__ count) {
    const int words = (K + 31) / 32;
    int used = 0;
    for (int i = threadIdx.x; i < words; i += 32) {
        unsigned int w = bitmap[i];
        if (i == words - 1 && (K & 31)) w &= (1u << (K & 31)) - 1u;
        used += __popc(w);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) used += __shfl_xor_sync(0xffffffffu, used, o);
    if (threadIdx.x == 0) *count = used;
}

int launch_vq_pack_codes(const long long* idx, int64_t n, int K, void* out, int code_bytes, unsigned int* bitmap, cudaStream_t st) {
    const int sms = sm_count();
    MOVAE_REQUIRE(sms > 0, MOVAE_ERR_CUDA, "CUDA device query failed (no GPU?)");
    int64_t grid = (n + 1023) / 1024;
    if (grid > (int64_t)sms * 8) grid = (int64_t)sms * 8;
    if (grid < 1) grid = 1;
    if (code_bytes == 2) vq_pack_codes_kernel<short><<<(unsigned)grid, 256, 0, st>>>(idx, n, K, static_cast<short*>(out), bitmap);
    else if (code_bytes == 4) vq_pack_codes_kernel<int><<<(unsigned)grid, 256, 0, st>>>(idx, n, K, static_cast<int*>(out), bitmap);
    else vq_pack_codes_kernel<long long><<<(unsigned)grid, 256, 0, st>>>(idx, n, K, static_cast<long long*>(out), bitmap);
    MOVAE_CUDA_TRY(cudaGetLastError());
    return MOVAE_OK;
}

int launch_vq_bitmap_count(const unsigned int* bitmap, int K, int* count, cudaStream_t st) {
    vq_bitmap_count_kernel<<<1, 32, 0, st>>>(bitmap, K, count);
    MOVAE_CUDA_TRY(cudaGetLastError());
    return MOVAE_OK;
}

int launch_vq_usage(const long long* idx, int64_t n, int K, int* usage_out, unsigned char* ws, cudaStream_t st) {
    const int sms = sm_count();
    MOVAE_REQUIRE(sms > 0, MOVAE_ERR_CUDA, "CUDA device query failed (no GPU?)");
    int64_t grid = (n + 255) / 256;
    if (grid > (int64_t)sms * 4) grid = (int64_t)sms * 4;
    if (grid < 1) grid = 1;
    vq_usage_kernel<<<(unsigned)grid, 256, 0, st>>>(idx, n, K, usage_out, ws);
    MOVAE_CUDA_TRY(cudaGetLastError());
    return MOVAE_OK;
}

}  // namespace movae
