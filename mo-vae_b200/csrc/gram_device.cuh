// Device-side pieces of the Gramian pass, shared by K1 (`gram_kernel`, gram.cu) and phase 1 of the
// fused aggregation kernel (aggregate.cu).
//
//   * tiles of 256 threads x U float4 per row are dealt round-robin to the CTAs in whole rounds, the remainder in equal
//     slices (rr_schedule); every warp load instruction covers 512 contiguous bytes of one row, all k rows of a tile are
//     in flight together (k*U independent 16-byte loads per thread);
//   * k(k+1)/2 float32 FMA chains per thread, at most 64 columns long, then promoted into float64
//     registers (the reference's own float32 SGEMM is 3e-5..8e-3 off at P=2.4M..1e8, SURVEY App. C.2;
//     the parity contract is rtol 1e-5 against a float64-accumulated oracle);
//   * warp shuffle -> shared memory -> one partial per CTA; the partials are summed in a fixed order
//     by ONE CTA: bit-reproducible for a given (k, P, grid), no float atomics.
#pragma once
#include "common.cuh"

namespace movae {

constexpr int kGramThreads = 256;
constexpr int kGramMaxBlocks = 2048;
constexpr int kGramHeaderBytes = 256;
constexpr int kGramChain = 64;   // float32 FMA chain length (columns) between promotions to float64

// The workspace (movae_gram_workspace_bytes): a header, then one float64 partial per CTA from kGramHeaderBytes on.  Header:
// byte 0 the ticket of the Gramian pass; the fused launches (aggregate.cu) also keep their exit counter at 4, their ready
// flag at 128 and the six timestamps of their last launch at 192.
struct GramWorkspace {
    static constexpr int kTicket = 0, kExit = 4, kReady = 128, kStamps = 192;
    unsigned int* ticket;
    unsigned int* exit;
    unsigned int* ready;
    unsigned long long* stamps;
    double* partials;
    __host__ __device__ explicit GramWorkspace(void* ws) {
        unsigned char* b = static_cast<unsigned char*>(ws);
        ticket = reinterpret_cast<unsigned int*>(b + kTicket);
        exit = reinterpret_cast<unsigned int*>(b + kExit);
        ready = reinterpret_cast<unsigned int*>(b + kReady);
        stamps = reinterpret_cast<unsigned long long*>(b + kStamps);
        partials = reinterpret_cast<double*>(b + kGramHeaderBytes);
    }
};
static_assert(GramWorkspace::kStamps + 6 * 8 <= kGramHeaderBytes, "the timestamps fit the header");

// Row addressing of the tile helpers: row(i) is the first column of row i.  A flat J has its rows ldJ floats apart; the
// segmented kernel's rows are separate tensors (aggregate.cu).
struct FlatRows {
    const float* J;
    int64_t ldJ;
    __device__ __forceinline__ const float* row(int i) const { return J + i * ldJ; }
};

template <int K>
struct GramAcc {
    static constexpr int N = K * (K + 1) / 2;
};

template <int K>
__device__ __forceinline__ void gram_fma(float (&acc)[GramAcc<K>::N], const float (&x)[K]) {
    int a = 0;
#pragma unroll
    for (int i = 0; i < K; ++i)
#pragma unroll
        for (int j = i; j < K; ++j) { acc[a] = fmaf(x[i], x[j], acc[a]); ++a; }
}

// Balanced round-robin schedule of one row's n_items float4 (or float) items over g CTAs.  Whole tiles go round-robin
// (tile t to CTA t mod g), so at any moment all CTAs stream one contiguous window of every row: the DRAM page locality
// that a per-CTA contiguous span lacks (spans ran the 25 %-writes recombination pass at 0.92 of the HBM peak, round-robin
// at 0.97+).  Only whole ROUNDS of g tiles are dealt that way: what is left (< g tiles) is cut into g equal slices, one
// masked tile per CTA -- otherwise the last round keeps a fraction of the CTAs busy for a whole tile time (9 % of a
// pass at P = 1e7).  Slice boundaries are multiples of 8 items (128-byte lines).
struct RRSchedule {
    int64_t rounds;            // whole rounds: tiles b, b + g, ..., b + (rounds - 1) g are this CTA's
    int64_t rem_lo, rem_hi;    // this CTA's slice of the remainder region (may be empty)
};
__device__ __forceinline__ RRSchedule rr_schedule(int64_t n_items, int64_t tile_items, int64_t b, int64_t g) {
    RRSchedule s;
    s.rounds = (n_items / tile_items) / g;
    const int64_t r0 = s.rounds * g * tile_items;
    const int64_t m = (((n_items - r0) + g - 1) / g + 7) & ~(int64_t)7;      // <= tile_items
    s.rem_lo = r0 + b * m < n_items ? r0 + b * m : n_items;
    s.rem_hi = s.rem_lo + m < n_items ? s.rem_lo + m : n_items;
    return s;
}

// How a pass loads one of a CTA's tiles: `steps(d)` gives the loader of the step d places from the back of the CTA's
// deal (0: the remainder slice, or the last whole tile), in either pass.  K1 and K3 load every tile alike; the fused
// kernel picks an L2 eviction priority per step (aggregate.cu).
struct PlainTileIO {
    __device__ __forceinline__ float4 load(const float4* p) const { return ld_stream_f4(p); }
    __device__ __forceinline__ float load(const float* p) const { return ld_stream_f1(p); }
};
struct PlainSteps {
    __device__ __forceinline__ PlainTileIO operator()(int64_t) const { return {}; }
};

// One tile of the Gramian pass: items [t0, t0 + tile) clipped to [t0, hi).
template <int K, int U, bool VEC, class Rows, class IO = PlainTileIO>
__device__ __forceinline__ void gram_tile(const Rows& rows, int64_t t0, int64_t hi, bool full, float (&acc)[GramAcc<K>::N],
                                          IO io = {}) {
    const int64_t base = t0 + threadIdx.x;
    if constexpr (VEC) {
        float4 v[K][U];
        if (full) {
#pragma unroll
            for (int i = 0; i < K; ++i)
#pragma unroll
                for (int u = 0; u < U; ++u)
                    v[i][u] = io.load(reinterpret_cast<const float4*>(rows.row(i)) + base + u * kGramThreads);
        } else {
#pragma unroll
            for (int i = 0; i < K; ++i)
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int64_t idx = base + u * kGramThreads;
                    v[i][u] = idx < hi ? io.load(reinterpret_cast<const float4*>(rows.row(i)) + idx) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            float x[K];
#pragma unroll
            for (int i = 0; i < K; ++i) x[i] = v[i][u].x;
            gram_fma<K>(acc, x);
#pragma unroll
            for (int i = 0; i < K; ++i) x[i] = v[i][u].y;
            gram_fma<K>(acc, x);
#pragma unroll
            for (int i = 0; i < K; ++i) x[i] = v[i][u].z;
            gram_fma<K>(acc, x);
#pragma unroll
            for (int i = 0; i < K; ++i) x[i] = v[i][u].w;
            gram_fma<K>(acc, x);
        }
    } else {
        float v[K][U];
#pragma unroll
        for (int i = 0; i < K; ++i)
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int64_t idx = base + u * kGramThreads;
                v[i][u] = idx < hi ? io.load(rows.row(i) + idx) : 0.f;
            }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            float x[K];
#pragma unroll
            for (int i = 0; i < K; ++i) x[i] = v[i][u];
            gram_fma<K>(acc, x);
        }
    }
}

// Column c of the rows (a ragged tail of the float4 path) as a float32 chain of its own, promoted into acc64.
template <int K, class Rows>
__device__ __forceinline__ void gram_column(const Rows& rows, int64_t c, double (&acc64)[GramAcc<K>::N]) {
    constexpr int NACC = GramAcc<K>::N;
    float x[K];
    float acc[NACC];
#pragma unroll
    for (int a = 0; a < NACC; ++a) acc[a] = 0.f;
#pragma unroll
    for (int i = 0; i < K; ++i) x[i] = rows.row(i)[c];
    gram_fma<K>(acc, x);
#pragma unroll
    for (int a = 0; a < NACC; ++a) acc64[a] += (double)acc[a];
}

// Streams this CTA's share of J front to back (rr_schedule over gridDim.x CTAs) and adds the products into acc64.
// VEC: J base 16-byte aligned and ldJ % 4 == 0 -> float4 path; otherwise scalar path.
template <int K, int U, bool VEC, class Steps = PlainSteps>
__device__ __forceinline__ void gram_stream_tiles(const float* __restrict__ J, int64_t P, int64_t ldJ,
                                                  double (&acc64)[GramAcc<K>::N], Steps steps = {}) {
    constexpr int NACC = GramAcc<K>::N;
    constexpr int W = VEC ? 4 : 1;                       // columns per item
    constexpr int FLUSH = kGramChain / (W * U) > 0 ? kGramChain / (W * U) : 1;
    const int tid = threadIdx.x;
    const int64_t n_items = P / W;                       // float4 (or float) items per row
    constexpr int64_t tile_items = (int64_t)kGramThreads * U;
    const RRSchedule sch = rr_schedule(n_items, tile_items, blockIdx.x, gridDim.x);
    const int64_t n_steps = sch.rounds + (sch.rem_hi > sch.rem_lo ? 1 : 0);
    const FlatRows rows{J, ldJ};

    int64_t r = 0;
    while (r < sch.rounds) {
        float acc[NACC];
#pragma unroll
        for (int a = 0; a < NACC; ++a) acc[a] = 0.f;
#pragma unroll 1
        for (int f = 0; f < FLUSH && r < sch.rounds; ++f, ++r) {
            const int64_t t0 = (r * gridDim.x + blockIdx.x) * tile_items;
            gram_tile<K, U, VEC>(rows, t0, t0 + tile_items, true, acc, steps(n_steps - 1 - r));
        }
#pragma unroll
        for (int a = 0; a < NACC; ++a) acc64[a] += (double)acc[a];
    }
    if (sch.rem_hi > sch.rem_lo) {
        float acc[NACC];
#pragma unroll
        for (int a = 0; a < NACC; ++a) acc[a] = 0.f;
        gram_tile<K, U, VEC>(rows, sch.rem_lo, sch.rem_hi, false, acc, steps(0));
#pragma unroll
        for (int a = 0; a < NACC; ++a) acc64[a] += (double)acc[a];
    }

    // ragged tail of the float4 path: columns 4*(P/4) .. P-1, one thread each in CTA 0
    if (VEC && blockIdx.x == 0 && tid < (int)(P - n_items * W)) gram_column<K>(rows, n_items * W + tid, acc64);
}

// CTA reduce (shuffle within warps, fixed-order sum across the 8 warps), store this CTA's partial, take a
// ticket.  Returns true (to every thread) in the LAST CTA of the grid to arrive.  `red` is shared scratch.
template <int K>
__device__ __forceinline__ bool gram_cta_partial_and_ticket(const double (&acc64)[GramAcc<K>::N], double* __restrict__ partials,
                                                            unsigned int* __restrict__ counter,
                                                            double (*red)[GramAcc<K>::N], int* is_last_smem) {
    constexpr int NACC = GramAcc<K>::N;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
#pragma unroll
    for (int a = 0; a < NACC; ++a) {
        const double s = warp_sum(acc64[a]);
        if (lane == 0) red[warp][a] = s;
    }
    __syncthreads();
    if (tid < NACC) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < kGramThreads / 32; ++w) s += red[w][tid];
        partials[(int64_t)blockIdx.x * NACC + tid] = s;
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) *is_last_smem = (atomicAdd(counter, 1u) == gridDim.x - 1);
    __syncthreads();
    return *is_last_smem != 0;
}

// Last CTA: deterministic combine of all CTA partials into the full symmetric k x k matrix `Gs` (shared memory,
// row-major K x K).  Ends with a CTA barrier.
template <int K>
__device__ __forceinline__ void gram_combine_partials(const double* __restrict__ partials, double* __restrict__ Gs) {
    constexpr int NACC = GramAcc<K>::N;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    __threadfence();
    for (int a = warp; a < NACC; a += kGramThreads / 32) {
        // four loads in flight per lane (one dependent L2 round trip per CTA partial made this the longest piece of the
        // solve phase); the order of the additions is fixed by (lane, grid size): deterministic
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
        const int g = (int)gridDim.x;
        for (int b = lane; b < g; b += 128) {
            const double v0 = __ldcg(&partials[(int64_t)b * NACC + a]);
            const double v1 = b + 32 < g ? __ldcg(&partials[(int64_t)(b + 32) * NACC + a]) : 0.0;
            const double v2 = b + 64 < g ? __ldcg(&partials[(int64_t)(b + 64) * NACC + a]) : 0.0;
            const double v3 = b + 96 < g ? __ldcg(&partials[(int64_t)(b + 96) * NACC + a]) : 0.0;
            s0 += v0; s1 += v1; s2 += v2; s3 += v3;
        }
        double s = (s0 + s1) + (s2 + s3);
        s = warp_sum(s);
        if (lane == 0) {
            int i = 0, rem = a;          // a -> (i, j), i <= j, row-major upper triangle
            while (rem >= K - i) { rem -= K - i; ++i; }
            const int j = i + rem;
            Gs[i * K + j] = s;
            Gs[j * K + i] = s;
        }
    }
    __syncthreads();
}

}  // namespace movae
