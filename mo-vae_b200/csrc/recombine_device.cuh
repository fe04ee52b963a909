// Device-side recombination pass  out (=|+=) w @ J, shared by K3 (`recombine_kernel`, recombine.cu) and
// phase 2 of the fused aggregation kernel (aggregate.cu).
//
// Back to front: the Gramian pass streamed J front-to-back, so the last ~100 MB it touched are still L2-resident on a
// 126 MB L2 and are consumed first.  The loads of the first tile
// are issued BEFORE `ready()` is called and the weights are read after it: in the fused kernel `ready`
// waits for the solve, so the wait overlaps the first loads.
#pragma once
#include <type_traits>

#include "gram_device.cuh"

namespace movae {

constexpr int kRecThreads = 256;

template <int K, int U, bool VEC>
struct RecTile {
    using T = typename std::conditional<VEC, float4, float>::type;
    T v[K][U];
};

template <int K, int U, bool VEC, class Rows, class IO = PlainTileIO>
__device__ __forceinline__ void rec_load_tile(RecTile<K, U, VEC>& r, const Rows& rows, int64_t base, int64_t lo, int64_t hi,
                                              bool full, IO io = {}) {
#pragma unroll
    for (int i = 0; i < K; ++i)
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t idx = base + u * kRecThreads;
            if constexpr (VEC)
                r.v[i][u] = (full || (idx >= lo && idx < hi)) ? io.load(reinterpret_cast<const float4*>(rows.row(i)) + idx)
                                                    : make_float4(0.f, 0.f, 0.f, 0.f);
            else
                r.v[i][u] = (full || (idx >= lo && idx < hi)) ? io.load(rows.row(i) + idx) : 0.f;
        }
}

template <int K, int U, bool VEC>
__device__ __forceinline__ void rec_store_tile(const RecTile<K, U, VEC>& r, const float (&w)[K], float* __restrict__ out,
                                               int64_t base, int64_t lo, int64_t hi, bool full, int accumulate) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const int64_t idx = base + u * kRecThreads;
        if (!full && (idx < lo || idx >= hi)) continue;
        if constexpr (VEC) {
            float4 o;
            o.x = w[0] * r.v[0][u].x; o.y = w[0] * r.v[0][u].y; o.z = w[0] * r.v[0][u].z; o.w = w[0] * r.v[0][u].w;
#pragma unroll
            for (int i = 1; i < K; ++i) {
                o.x = fmaf(w[i], r.v[i][u].x, o.x); o.y = fmaf(w[i], r.v[i][u].y, o.y);
                o.z = fmaf(w[i], r.v[i][u].z, o.z); o.w = fmaf(w[i], r.v[i][u].w, o.w);
            }
            float4* dst = reinterpret_cast<float4*>(out) + idx;
            if (accumulate) {
                const float4 old = *dst;
                o.x += old.x; o.y += old.y; o.z += old.z; o.w += old.w;
            }
            st_stream_f4(dst, o);
        } else {
            float o = w[0] * r.v[0][u];
#pragma unroll
            for (int i = 1; i < K; ++i) o = fmaf(w[i], r.v[i][u], o);
            if (accumulate) o += out[idx];
            out[idx] = o;
        }
    }
}

// Column c of the rows (a ragged tail of the float4 path).
template <int K, class Rows>
__device__ __forceinline__ void rec_column(const Rows& rows, const float (&w)[K], float* __restrict__ out, int64_t c,
                                           int accumulate) {
    float o = w[0] * rows.row(0)[c];
#pragma unroll
    for (int q = 1; q < K; ++q) o = fmaf(w[q], rows.row(q)[c], o);
    if (accumulate) o += out[c];
    out[c] = o;
}

// The weights, read once ready() has returned: in the fused launches every CTA but the solving one waits there for their
// publication.
template <int K, class Ready>
__device__ __forceinline__ void rec_read_weights(const float* w_dev, Ready ready, float (&w)[K]) {
    ready();
#pragma unroll
    for (int q = 0; q < K; ++q) w[q] = __ldcg(w_dev + q);
}

// This CTA's share of the row (rr_schedule over gridDim.x CTAs, the same deal as the Gramian pass), BACK TO FRONT: first
// its slice of the remainder region at the end of J, then its whole tiles in descending order.  Two register tiles: the
// loads of the next tile are issued BEFORE the current one is combined and stored, so a thread never runs out of loads
// in flight.  `steps` as in gram_stream_tiles: step i here is i places from the back of the deal.
template <int K, int U, bool VEC, class Ready, class Steps = PlainSteps>
__device__ __forceinline__ void recombine_tiles(const float* __restrict__ J, int64_t P, int64_t ldJ, const float* w_dev,
                                                float* __restrict__ out, int accumulate, Ready ready, Steps steps = {}) {
    constexpr int W = VEC ? 4 : 1;
    const int tid = threadIdx.x;
    const int64_t n_items = P / W;
    constexpr int64_t tile_items = (int64_t)kRecThreads * U;
    const RRSchedule sch = rr_schedule(n_items, tile_items, blockIdx.x, gridDim.x);
    const bool has_rem = sch.rem_hi > sch.rem_lo;
    const FlatRows rows{J, ldJ};
    // step i = 0 .. n_steps - 1: (t0, lo, hi, full); step 0 is the remainder slice when there is one
    const int64_t n_steps = sch.rounds + (has_rem ? 1 : 0);
    auto t0_of = [&](int64_t i) -> int64_t {
        if (has_rem) { if (i == 0) return sch.rem_lo; --i; }
        return ((sch.rounds - 1 - i) * gridDim.x + blockIdx.x) * tile_items;
    };
    auto hi_of = [&](int64_t i, int64_t t0) -> int64_t { return (has_rem && i == 0) ? sch.rem_hi : t0 + tile_items; };
    auto full_of = [&](int64_t i) -> bool { return !(has_rem && i == 0); };

    RecTile<K, U, VEC> ra, rb;
    int64_t i = 0;
    int64_t ta = 0, tb = 0;
    if (n_steps > 0) { ta = t0_of(0); rec_load_tile<K, U, VEC>(ra, rows, ta + tid, ta, hi_of(0, ta), full_of(0), steps(0)); }
    float w[K];
    rec_read_weights<K>(w_dev, ready, w);
    while (i < n_steps) {
        const bool has_b = i + 1 < n_steps;
        if (has_b) { tb = t0_of(i + 1); rec_load_tile<K, U, VEC>(rb, rows, tb + tid, tb, hi_of(i + 1, tb), full_of(i + 1), steps(i + 1)); }
        rec_store_tile<K, U, VEC>(ra, w, out, ta + tid, ta, hi_of(i, ta), full_of(i), accumulate);
        if (!has_b) break;
        if (i + 2 < n_steps) { ta = t0_of(i + 2); rec_load_tile<K, U, VEC>(ra, rows, ta + tid, ta, hi_of(i + 2, ta), full_of(i + 2), steps(i + 2)); }
        rec_store_tile<K, U, VEC>(rb, w, out, tb + tid, tb, hi_of(i + 1, tb), full_of(i + 1), accumulate);
        i += 2;
    }
    // ragged tail of the float4 path
    if (VEC && blockIdx.x == 0 && tid < (int)(P - n_items * W)) rec_column<K>(rows, w, out, n_items * W + tid, accumulate);
}

}  // namespace movae
