// Constants shared by the quantizer's streaming kernels (vq_gather.cu: K5; vq_backward.cu: K6), K6b's per-CTA partials
// (written by vq_backward.cu, read by its dE reduce and by vq_ema.cu) and the quantizer's launchers.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace movae {

constexpr int64_t kSmallN = 32768;        // at or below: no per-CTA codebook staging in K5 / K6a

// ---- layout of the quantizer workspace (movae_vq_workspace_bytes; vq_gather.cu writes it, vq_api.cu sizes it) ----
// [0]  uint  rows the LAST tensor-path search re-evaluated exactly (K4)      [4] uint ticket (K5)      [8] uint ticket (usage)
// [12] uint  running re-check count of the search in flight (K4)           [16] uint exit ticket (K4)
// [64 .. 64+8192)       usage bitmap (up to 65536 codes), all-zero between calls
// [8256 .. 8256+16384)  K5 per-CTA float64 partial sums
constexpr size_t kWsBitmapOff = 64;
constexpr size_t kWsPartialOff = 8256;
constexpr size_t kWsListOff = 24640;
constexpr int kVqMaxCodes = 65536;

// ---- K6b's per-CTA partials (K = 512, D = 64) -------------------------------------------------------------------------
// Every CTA of K6b writes kPartFloats floats: S [K, D] (the sum of the z rows that chose each code, in the CTA's fixed row
// order) then the counts [K] as int bits.  The backward's dE and VectorQuantizerEMA's statistics are both combined from
// them, in float64 and in one fixed order (k6b_combine_partials), so both are bit-reproducible.
constexpr int kBwK = 512, kBwD = 64;
constexpr size_t kPartFloats = (size_t)kBwK * kBwD + kBwK;
constexpr int kPartTileRows = 128;        // rows per K6b tile: one CTA per tile, at most 160 CTAs

// Number of per-CTA partials K6b writes for n_rows (0 = K, D outside K6b: the generic path).
inline int vq_backward_parts(int64_t n_rows, int K, int D) {
    if (K != kBwK || D != kBwD || n_rows <= 0) return 0;
    const int64_t tiles = (n_rows + kPartTileRows - 1) / kPartTileRows;
    return (int)(tiles < 160 ? tiles : 160);
}

// Fixed-order float64 combine of the partials: a block of kRdThreads threads, thread (q, g) = (tid % kRdQuads,
// tid / kRdQuads), handles output quad `quad` = S elements 4 quad .. 4 quad + 3 of one code.  Thread (q, g) sums the
// partials p = g, g + 4, g + 8, ... (16-byte loads, 4 in flight), then the four group sums are added in the order
// g = 0, 1, 2, 3 -- 16 partial loads in flight per output quad instead of 8 scalar ones per output element (the reduction
// of 148 partials was a 26 us latency chain).  Every thread of the block calls it (it holds a barrier); every thread gets
// the totals of its quad: st = S, ct = the code's count.
constexpr int kRdGroups = 4, kRdQuads = 64, kRdThreads = kRdGroups * kRdQuads;
__device__ __forceinline__ void k6b_combine_partials(const float* __restrict__ partials, int n_parts, int quad, int q, int g,
                                                     double (&st)[4], long long& ct) {
    __shared__ double sm_s[kRdGroups][kRdQuads][4];
    __shared__ long long sm_c[kRdGroups][kRdQuads];
    const int j = quad * 4 / kBwD;
    double s[4] = {0.0, 0.0, 0.0, 0.0};
    long long c = 0;
    if (quad < kBwK * kBwD / 4) {
        for (int p0 = g; p0 < n_parts; p0 += kRdGroups * 4) {
            float4 v[4];
            int cv[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int p = p0 + u * kRdGroups;
                const float* part = partials + (size_t)(p < n_parts ? p : 0) * kPartFloats;
                v[u] = p < n_parts ? __ldcs(reinterpret_cast<const float4*>(part) + quad) : make_float4(0.f, 0.f, 0.f, 0.f);
                cv[u] = p < n_parts ? __float_as_int(__ldg(part + kBwK * kBwD + j)) : 0;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                s[0] += (double)v[u].x; s[1] += (double)v[u].y; s[2] += (double)v[u].z; s[3] += (double)v[u].w;
                c += (long long)cv[u];
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) sm_s[g][q][i] = s[i];
    sm_c[g][q] = c;
    __syncthreads();
    ct = 0;
#pragma unroll
    for (int gg = 0; gg < kRdGroups; ++gg) ct += sm_c[gg][q];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        st[i] = 0.0;
#pragma unroll
        for (int gg = 0; gg < kRdGroups; ++gg) st[i] += sm_s[gg][q][i];
    }
}

// ---- launchers (vq_argmin_tc.cu, vq_argmin_exact.cu, vq_gather.cu, vq_backward.cu, vq_ema.cu) -------------------------
int launch_vq_argmin_tc(const float* z, int64_t N, int64_t HW, const float* E, long long* idx, unsigned int* ws_words, float* dbg,
                        cudaStream_t st);
int launch_vq_argmin_exact(const float* z, int64_t N, int D, int64_t HW, const float* E, int K, long long* idx, cudaStream_t st);
int launch_vq_gather(const float* z, int64_t N, int D, int64_t HW, const float* E, int K, const long long* idx,
                     float* q_out, float* loss_out, int* usage_out, unsigned char* ws, cudaStream_t st);
int launch_vq_usage(const long long* idx, int64_t n, int K, int* usage_out, unsigned char* ws, cudaStream_t st);
int launch_vq_pack_codes(const long long* idx, int64_t n, int K, void* out, int code_bytes, unsigned int* bitmap, cudaStream_t st);
int launch_vq_bitmap_count(const unsigned int* bitmap, int K, int* count, cudaStream_t st);
int launch_vq_backward(const float* grad_out, const float* g_commit, const float* g_embed, const float* z, int64_t N, int D,
                       int64_t HW, const float* E, int K, const long long* idx, float* dz, float* dE, float* partials,
                       cudaStream_t st);
// K6b alone: vq_backward_parts(N, K, D) partials into `partials`; *n_parts = CTAs launched.  Needs N > 0.
int launch_k6b_partials(const float* z, int64_t N, int64_t HW, const long long* idx, float* partials, int* n_parts, cudaStream_t st);
size_t vq_ema_workspace_bytes(int64_t n_rows, int K, int D);
int launch_vq_ema_stats(const float* z, int64_t N, int D, int64_t HW, const long long* idx, int K, float* stats, unsigned char* ws,
                        cudaStream_t st);
int launch_vq_ema_apply(const float* stats, int K, int D, double decay, double eps, float* E, float* cluster_size, float* embed_avg,
                        float* E_prev, unsigned char* ws, cudaStream_t st);
int launch_vq_ema_update(const float* z, int64_t N, int D, int64_t HW, const long long* idx, int K, double decay, double eps, float* E,
                         float* cluster_size, float* embed_avg, float* E_prev, unsigned char* ws, cudaStream_t st);

}  // namespace movae
