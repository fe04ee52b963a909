// K4 `vq_argmin_gemm`: nearest-codebook search for K = 512 codes of dimension D = 64 as a
// tcgen05 / TMEM GEMM with a fused per-row argmin epilogue.
//
// Replaces, in /root/reference/models/vq_vae.py: the NCHW->NHWC permute (:28), the distance matrix
// `sum(z^2) + sum(E^2) - 2 z E^T` (:34-36, a cuBLAS SGEMM + 3 elementwise kernels that materialise
// dist[N,K]) and `torch.argmin` (:39).  The distance matrix never leaves the SM.
//
// Arithmetic.  The reference is true float32; tcgen05 has no float32 MMA kind.  Operands are split
// into two bfloat16 terms (x = hi + lo + O(2^-18 x)) and the product is evaluated as
// lo*hi + hi*lo + hi*hi on the tensor cores (float32 accumulation in TMEM): per-entry error of the
// score -2 z.e  <= 2^-15 |z||e|  (dropped split terms 2 * 3 * 2^-18 = 2^-15.4 worst case, plus float32
// accumulation; measured on B200: 6.8e-6 |z||e| maximum).
//
// The tensor core also BUILDS THE SORT KEY.  Three more K=16 steps per accumulator unit, whose A
// operand is a per-tile constant row and whose B operand is a per-code side table, add
//   step 13:  |e_j|^2 (3 bf16 terms)  +  C  +  8 M       C >= 2 max|z| max|e| makes the score positive,
//                                                        M = 2^m > score + C; the sum lands in [8M, 16M)
//                                                        where the float32 accumulator's ulp is 8 u (u = M 2^-23)
//   step 14:  - 7 M                                      exact: key in [M, 2M), 3 low mantissa bits zero
//   step 15:  + i3(j) u                                  exact: the 3 low mantissa bits = bits 0, 3, 4 of the column
//                                                        within its 32-column chunk (bits 1, 2 are implied by which
//                                                        of the epilogue's four min/max trackers sees the column)
// (Steps 14 and 15 cannot share one instruction: within an MMA the tensor core aligns the addends to the largest
// exponent, so i3(j) u next to -7 M is truncated away -- tried, 50% wrong indices.)
// so every accumulator entry is a positive float whose order is the order of the scores (to 8 u) and
// whose low bits say which column it is.  The epilogue is then min/max only (2.5 alu-pipe instructions
// per entry instead of 3.8 alu + 2 fma in the version that added |e|^2 and packed the index itself,
// which ran alu-pipe-bound at 47% tensor activity; profiles/r1_vq_tc.md).
//
// The epilogue keeps the two smallest keys of every row; a row whose gap is <= 1.25 M 2^-16 (tensor-path
// error 2 * 2^-15 max|z| max|e| <= M 2^-16, plus 4 rounding quanta of 8 u) goes onto a shared-memory ring
// and is re-evaluated exactly (reference formula, float32 roundings) INSIDE this kernel by two re-check
// warps (round 1 ran a second kernel over a global worklist: 16 us of fixed cost at N = 8,192, 92 us at
// N = 4.2 M).  M also exceeds 2 C + (max|z|^2 + max|e|^2) / 32 over the tile, so every other row provably has the
// same argmin as the reference formula with its float32 roundings (first minimal index).  Non-finite inputs: a
// codebook with an inf / NaN entry sends every row to the full re-check; inf / NaN latents make their tile's keys
// inf / NaN, which the epilogue's !(a - b > thr) tests count as close, so those rows are re-checked too.  The re-check
// follows torch.argmin: the first NaN distance wins.
//
// Roofline: tensor pipe.  Algorithmic work 2*K*D = 65,536 flop per code vector; executed 15/4 of that
// (three bf16 products + three key steps).  HBM traffic 4*D = 256 B read + 8 B written per code vector.
//
// CTA = 15 warps, persistent over 128-row tiles:
//   warps 0-3   epilogue group 0: codes   0..255 (TMEM columns   0..255)
//   warps 4-7   epilogue group 1: codes 256..511 (TMEM columns 256..511), merges both groups, writes idx
//   warps 8-11  producers: gather z rows from NCHW, split to bf16 hi/lo, write the swizzled A stage and the
//               tile's key constants; the loads of the NEXT tile are issued quarter by quarter while the
//               current one is converted
//   warp  12    MMA issuer (one lane) + TMEM owner
//   warps 13-14 exact re-check of the rows the epilogue could not decide (FMA pipe + shared-memory reads of the
//               resident operand image: the epilogue's alu pipe and the tensor pipe are not touched)
// TMEM (512 columns) = two 256-column accumulators, one per epilogue group; a tile is two M128 x N256
// units of 15 K-steps.  While group 0 drains unit (t, 0) the tensor core computes (t, 1), while group 1
// drains (t, 1) it computes (t+1, 0): no stall as long as draining 256 columns takes less than one
// unit's MMA time, which the min/max-only epilogue does.  (N = 128 units, tried to double-buffer each
// group, need 8 KB of operands per 64-cycle MMA = the whole 128 B/clk of shared-memory bandwidth and ran
// at ~120-137 cycles per MMA; N = 256 needs 12 KB per 128 cycles.)  The codebook (as -2E, split hi/lo)
// and the side table stay resident in shared memory for the CTA's lifetime.
#include <cuda_bf16.h>
#include <math.h>

#include "common.cuh"
#include "tc_ptx.cuh"
#include "vq_tc_common.cuh"

namespace movae {

constexpr int kTcD = 64;
constexpr int kTcK = 512;
constexpr int kTcTileM = 128;
constexpr int kTcHalfN = 256;      // codes per epilogue group
constexpr int kTcUnitN = 256;      // UMMA_N: codes per accumulator unit (= one epilogue group)
constexpr int kTcRecheckWarps = 2;
constexpr int kTcThreads = (13 + kTcRecheckWarps) * 32;

// shared-memory carve-up (bytes from a 1024-aligned base)
constexpr uint32_t kOffBhi = 0;                        // 512 rows x 128 B, 128B swizzle
constexpr uint32_t kOffBlo = 65536;
constexpr uint32_t kOffA = 131072;                     // 2 stages x (hi 16 KB + lo 16 KB), 128B swizzle
constexpr uint32_t kOffBaug = kOffA + 2 * 32768;       // 64 code groups x (2 core matrices x 128 B), no swizzle
constexpr uint32_t kOffAaug = kOffBaug + 16384;        // 2 stages x 3 steps x (2 core matrices x 128 B)
constexpr uint32_t kOffXchg = kOffAaug + 2 * 768;      // 2 slots x 128 x {key1, key2, code1 | code2 << 16, enumerate flag}
constexpr uint32_t kOffBar = kOffXchg + 2 * 128 * 16;
constexpr uint32_t kRqCap = 256;                        // re-check ring: {row (-1 = empty slot), n_candidates (0 = all 512), codes, codes}
constexpr uint32_t kOffRq = kOffBar + 256;
constexpr uint32_t kOffZs = kOffRq + kRqCap * 16;       // per re-check warp: 64 floats, the row being re-checked
constexpr uint32_t kTcSmemBytes = kOffZs + kTcRecheckWarps * 256 + 1024;    // + alignment slack
static_assert(kTcSmemBytes <= 227 * 1024, "K4 shared memory");

struct TcBarriers {
    uint64_t a_full[2], a_empty[2], acc_full[2], acc_empty[2], x_full[2], x_free[2];
    uint64_t epi_done;         // the 128 threads of epilogue group 1 arrive once, after their last tile
    uint32_t tmem_base;
    uint32_t emax2_bits;
    float pmax[2][4];          // per-producer-warp max |z|^2 of the tile being produced (double-buffered)
    uint32_t rq_tail, rq_head, rq_freed;     // re-check ring: slots allocated / claimed / released so far
};
static_assert(sizeof(TcBarriers) <= 256, "barrier block");

__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t* p) { return *reinterpret_cast<const volatile uint32_t*>(p); }
__device__ __forceinline__ int ld_volatile_i32(const int* p) { return *reinterpret_cast<const volatile int*>(p); }

// Exact re-evaluation of ONE row by ONE warp, inside the search kernel (the re-check warps).  Same arithmetic as vq_argmin_exact.cu: the reference formula fl(fl(|z|^2 + |e|^2) - 2 fl(z.e)) with the
// three sums accumulated in float64 and rounded once, first minimal index.  Candidates come from a float32 pass over
// all 512 codes that reads the RESIDENT operand image: hi(-2E) alone (bf16: relative error 2^-9 per element, so the
// candidate bound is 2 * 2^-8 |z| max|e| on top of the float32 pass's own error -- a superset of what the exact kernel
// would select; typically 2-3 codes) plus |e|^2 from the side table.  Each candidate is then evaluated by the lane that
// owns it from the float32 codebook in global memory (L2-resident).  When the bound is not finite (inf / NaN latents or
// codebook) every code is a candidate.
__device__ __noinline__ void recheck_row_in_kernel(int4 ent, const float* __restrict__ z, int64_t HW, const float* __restrict__ E,
                                                    const uint8_t* smem, float* zs, float emax, float emax2,
                                                    long long* __restrict__ idx_out, unsigned int* __restrict__ count, int lane) {
    const int n = ent.x;
    const int64_t b = n / HW, hw = n - b * HW;
    const float* zp = z + (b * kTcD) * HW + hw;
    const float za = __ldg(zp + (int64_t)lane * HW), zb = __ldg(zp + (int64_t)(lane + 32) * HW);
    __syncwarp();
    zs[lane] = za;
    zs[lane + 32] = zb;
    const float z2f = (float)warp_sum((double)za * (double)za + (double)zb * (double)zb);
    __syncwarp();
    if (lane == 0) atomicAdd(count, 1u);
    // torch.argmin's order: a NaN distance is smaller than everything (the first NaN wins), inf never wins over a finite
    // distance, and a row whose distances are all inf gets code 0
    auto key_of = [](float dist, int j) { return dist != dist ? (unsigned long long)j : pack_dist_index(dist, j); };
    if (ent.y > 0) {
        // ---- the epilogue knows every candidate (<= 4 codes, one per tracker): evaluate just those, lanes over channels ----
        const int codes[4] = {ent.z & 0xFFFF, (ent.z >> 16) & 0xFFFF, ent.w & 0xFFFF, (ent.w >> 16) & 0xFFFF};
        float e0[4], e1[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float* ep = E + (size_t)codes[i < ent.y ? i : 0] * kTcD;
            e0[i] = __ldg(ep + lane);
            e1[i] = __ldg(ep + lane + 32);
        }
        unsigned long long bestk = ~0ull;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (i < ent.y) {                               // warp-uniform
                const double dd = warp_sum(fma((double)e0[i], (double)za, (double)e1[i] * (double)zb));
                const double ee = warp_sum(fma((double)e0[i], (double)e0[i], (double)e1[i] * (double)e1[i]));
                const float dist = __fsub_rn(__fadd_rn(z2f, (float)ee), __fmul_rn(2.f, (float)dd));
                if (!(dist >= __uint_as_float(0x7f800000u))) {
                    const unsigned long long key = key_of(dist, codes[i]);
                    bestk = key < bestk ? key : bestk;
                }
            }
        }
        if (lane == 0) idx_out[n] = bestk == ~0ull ? 0ll : (long long)(unsigned int)(bestk & 0xffffffffull);
        return;
    }
    // ---- pass 1: float32 scores of this lane's 16 codes (j = lane + 32 c) from the resident image ----
    float acc[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) acc[c] = 0.f;
    const uint8_t* brow = smem + kOffBhi + (uint32_t)lane * 128u;
#pragma unroll 1
    for (int c8 = 0; c8 < 8; ++c8) {
        const float4 q0 = *reinterpret_cast<const float4*>(zs + c8 * 8), q1 = *reinterpret_cast<const float4*>(zs + c8 * 8 + 4);
        const uint32_t sw = (uint32_t)((c8 ^ (lane & 7)) << 4);
#pragma unroll
        for (int c = 0; c < 16; ++c) {
            const uint4 h = *reinterpret_cast<const uint4*>(brow + (uint32_t)c * 4096u + sw);
            float a = acc[c];
            a = fmaf(__uint_as_float(h.x << 16), q0.x, a); a = fmaf(__uint_as_float(h.x & 0xFFFF0000u), q0.y, a);
            a = fmaf(__uint_as_float(h.y << 16), q0.z, a); a = fmaf(__uint_as_float(h.y & 0xFFFF0000u), q0.w, a);
            a = fmaf(__uint_as_float(h.z << 16), q1.x, a); a = fmaf(__uint_as_float(h.z & 0xFFFF0000u), q1.y, a);
            a = fmaf(__uint_as_float(h.w << 16), q1.z, a); a = fmaf(__uint_as_float(h.w & 0xFFFF0000u), q1.w, a);
            acc[c] = a;
        }
    }
    float mn = __uint_as_float(0x7f800000u);
#pragma unroll
    for (int c = 0; c < 16; ++c) {
        const int j = lane + 32 * c;
        const uint2 t = *reinterpret_cast<const uint2*>(smem + kOffBaug + (uint32_t)(j >> 3) * 256u + (uint32_t)(j & 7) * 16u);
        const float e2 = __uint_as_float(t.x << 16) + __uint_as_float(t.x & 0xFFFF0000u) + __uint_as_float(t.y << 16);
        acc[c] += e2;                                      // score = |e|^2 - 2 z.e  (the image holds -2 E)
        mn = fminf(mn, acc[c]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    const float znorm = sqrtf(z2f);
    const float bound = 2.02f * 0.00390625f * znorm * emax +
                        2.f * (float)(kTcD + 2) * 5.9604645e-08f * (2.f * znorm * emax + emax2) + 8.f * 1.1920929e-07f * (z2f + emax2);
    // a non-finite limit (inf / NaN latents or codebook rows) bounds nothing: every code is evaluated
    const float lim = fabsf(mn + bound) <= 3.4028235e38f ? mn + bound : __uint_as_float(0x7f800000u);
    // ---- pass 2: this lane's candidates with float64 sums and the reference's float32 formula ----
    unsigned long long best = ~0ull;
    int nan_j = kTcK;                                      // first code with a NaN distance (kTcK: none)
#pragma unroll 1
    for (int c = 0; c < 16; ++c) {
        if (!(acc[c] > lim)) {
            const int j = lane + 32 * c;
            const float* ep = E + (size_t)j * kTcD;
            double dd = 0.0, ee = 0.0;
            float4 ev[kTcD / 4];
#pragma unroll
            for (int d = 0; d < kTcD / 4; ++d) ev[d] = __ldg(reinterpret_cast<const float4*>(ep) + d);   // one L2 round trip
#pragma unroll
            for (int d = 0; d < kTcD; d += 4) {
                const float4 e = ev[d / 4];
                const float4 q = *reinterpret_cast<const float4*>(zs + d);
                dd = fma((double)e.x, (double)q.x, dd); ee = fma((double)e.x, (double)e.x, ee);
                dd = fma((double)e.y, (double)q.y, dd); ee = fma((double)e.y, (double)e.y, ee);
                dd = fma((double)e.z, (double)q.z, dd); ee = fma((double)e.z, (double)e.z, ee);
                dd = fma((double)e.w, (double)q.w, dd); ee = fma((double)e.w, (double)e.w, ee);
            }
            const float dist = __fsub_rn(__fadd_rn(z2f, (float)ee), __fmul_rn(2.f, (float)dd));
            if (dist < __uint_as_float(0x7f800000u)) {     // inf never wins (index 0 if every distance is inf)
                const unsigned long long key = pack_dist_index(dist, j);
                best = key < best ? key : best;            // smallest distance, then smallest index
            }
            if (dist != dist) nan_j = min(nan_j, j);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
        best = other < best ? other : best;
        nan_j = min(nan_j, __shfl_xor_sync(0xffffffffu, nan_j, o));
    }
    if (lane == 0)
        idx_out[n] = nan_j < kTcK ? (long long)nan_j : best == ~0ull ? 0ll : (long long)(unsigned int)(best & 0xffffffffull);
}

// One attempt to take a row off the re-check ring and re-evaluate it (warp-collective).  Returns false when the ring was
// empty (or another warp won the race for the slot).
__device__ __forceinline__ bool recheck_service_one(TcBarriers* bars, int4* ring, const float* z, int64_t HW, const float* E,
                                                    const uint8_t* smem, float* zs, float emax, float emax2, long long* idx_out,
                                                    unsigned int* count, int lane) {
    int4 ent = make_int4(-1, 0, 0, 0);
    if (lane == 0) {
        const uint32_t h = ld_volatile_u32(&bars->rq_head);
        if (h != ld_volatile_u32(&bars->rq_tail) && atomicCAS(&bars->rq_head, h, h + 1u) == h) {
            int4* slot = ring + (h % kRqCap);
            while ((ent.x = ld_volatile_i32(&slot->x)) < 0) {}     // the pusher allocated the slot a moment ago: its stores are on the way
            __threadfence_block();
            ent.y = ld_volatile_i32(&slot->y);
            ent.z = ld_volatile_i32(&slot->z);
            ent.w = ld_volatile_i32(&slot->w);
            *reinterpret_cast<volatile int*>(&slot->x) = -1;
            __threadfence_block();
            atomicAdd(&bars->rq_freed, 1u);
        }
    }
    ent.x = __shfl_sync(0xffffffffu, ent.x, 0);
    if (ent.x < 0) return false;
    ent.y = __shfl_sync(0xffffffffu, ent.y, 0);
    ent.z = __shfl_sync(0xffffffffu, ent.z, 0);
    ent.w = __shfl_sync(0xffffffffu, ent.w, 0);
    recheck_row_in_kernel(ent, z, HW, E, smem, zs, emax, emax2, idx_out, count, lane);
    return true;
}


template <bool DBG>
__global__ void __launch_bounds__(kTcThreads, 1)
vq_argmin_tc_kernel(const float* __restrict__ z, int64_t N, int64_t HW, const float* __restrict__ E,
                    long long* __restrict__ idx_out, unsigned int* __restrict__ ws_words, float* __restrict__ dbg) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t raw_addr = tc::smem_u32(smem_raw);
    uint8_t* smem = smem_raw + (((raw_addr + 1023u) & ~1023u) - raw_addr);
    TcBarriers* bars = reinterpret_cast<TcBarriers*>(smem + kOffBar);
    float* xchg = reinterpret_cast<float*>(smem + kOffXchg);
    int4* ring = reinterpret_cast<int4*>(smem + kOffRq);
    // workspace words: [0] rows re-checked by the LAST search (what callers read), [3] running count of this search,
    // [4] exit ticket (the last CTA to leave publishes [3] into [0] and clears both)
    unsigned int* run_count = ws_words + 3;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t n_tiles = (N + kTcTileM - 1) / kTcTileM;

    // ---- one-time setup ---------------------------------------------------------------------------
    if (tid == 0) {
        for (int i = 0; i < 2; ++i) {
            tc::mbar_init(&bars->a_full[i], 128);
            tc::mbar_init(&bars->a_empty[i], 1);
            tc::mbar_init(&bars->acc_full[i], 1);
            tc::mbar_init(&bars->acc_empty[i], 128);
            tc::mbar_init(&bars->x_full[i], 128);
            tc::mbar_init(&bars->x_free[i], 128);
        }
        tc::mbar_init(&bars->epi_done, 128);
        bars->emax2_bits = 0u;
        bars->rq_tail = bars->rq_head = bars->rq_freed = 0u;
        tc::mbar_fence_init();
    }
    if (warp == 12) tc::tmem_alloc(&bars->tmem_base, 512);
    __syncthreads();

    // codebook -> shared memory, ONE pass with all loads of a batch in flight (the one-load-at-a-time version cost ~12 us
    // per CTA and launch -- more than the search itself at N = 8,192): thread t owns (code j = t / 8, 16-byte chunk c = t % 8).
    //   B = -2 E split into bf16 hi + lo, K-major rows of 128 B, 128B swizzle;
    //   side table (B operand of the three key steps), K-major, no swizzle: code j, K index k ->
    //     group j/8: core matrix k<8 at +0, k>=8 at +128 (all zero); row j%8 at +16*(j%8); 2 bytes per k
    //     k = 0,1,2: |e_j|^2 as three bf16 terms   k = 3,4,5: 1 (multiplies C, 8M, -7M)   k = 6: i3(j) = bits 0,3,4 of j mod 32
    //   |e_j|^2 in float64 from the 8 chunk owners of the code (three shuffle steps inside their 8-lane group).
    constexpr int kSetupBatch = 5;
    static_assert(kTcThreads % 32 == 0 && (kTcK * 8) % 32 == 0, "whole warps enter or skip a setup item together");
    for (int t0 = tid; t0 < kTcK * 8; t0 += kTcThreads * kSetupBatch) {
        float4 x0[kSetupBatch], x1[kSetupBatch];
#pragma unroll
        for (int u = 0; u < kSetupBatch; ++u) {
            const int t = t0 + u * kTcThreads;
            if (t < kTcK * 8) {
                x0[u] = __ldg(reinterpret_cast<const float4*>(E + (size_t)t * 8));
                x1[u] = __ldg(reinterpret_cast<const float4*>(E + (size_t)t * 8 + 4));
            }
        }
#pragma unroll
        for (int u = 0; u < kSetupBatch; ++u) {
            const int t = t0 + u * kTcThreads;
            if (t < kTcK * 8) {                       // warp-uniform
                const int j = t >> 3, c = t & 7;
                const float x[8] = {x0[u].x, x0[u].y, x0[u].z, x0[u].w, x1[u].x, x1[u].y, x1[u].z, x1[u].w};
                uint32_t hi[4], lo[4];
                double s = 0.0;
#pragma unroll
                for (int p = 0; p < 4; ++p) {
                    split_bf16x2(-2.f * x[2 * p], -2.f * x[2 * p + 1], hi[p], lo[p]);
                    s += (double)x[2 * p] * x[2 * p] + (double)x[2 * p + 1] * x[2 * p + 1];
                }
                const uint32_t off = (uint32_t)j * 128u + (uint32_t)((c ^ (j & 7)) << 4);
                *reinterpret_cast<uint4*>(smem + kOffBhi + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                *reinterpret_cast<uint4*>(smem + kOffBlo + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                s += __shfl_xor_sync(0xffffffffu, s, 1);
                s += __shfl_xor_sync(0xffffffffu, s, 2);
                s += __shfl_xor_sync(0xffffffffu, s, 4);
                if (c == 0) {
                    const float sf = (float)s;
                    atomicMax(&bars->emax2_bits, __float_as_uint(sf));
                    const uint32_t h = bf16_bits_rn(sf);
                    const float r1 = sf - __uint_as_float(h << 16);
                    const uint32_t m = bf16_bits_rn(r1);
                    const uint32_t l = bf16_bits_rn(r1 - __uint_as_float(m << 16));
                    const uint32_t one = 0x3F80u;
                    const uint32_t col = bf16_bits_rn((float)((j & 1) | (((j & 31) >> 3) << 1)));
                    uint8_t* row = smem + kOffBaug + (uint32_t)(j >> 3) * 256u + (uint32_t)(j & 7) * 16u;
                    *reinterpret_cast<uint4*>(row) = make_uint4(h | (m << 16), l | (one << 16), one | (one << 16), col);
                    *reinterpret_cast<uint4*>(row + 128) = make_uint4(0u, 0u, 0u, 0u);
                }
            }
        }
    }
    for (int t = tid; t < (int)kRqCap; t += kTcThreads) ring[t] = make_int4(-1, 0, 0, 0);
    // key-constant rows: zero everything once (the producers rewrite only the first 16 bytes of each row)
    for (int t = tid; t < 2 * 768 / 16; t += kTcThreads) *reinterpret_cast<uint4*>(smem + kOffAaug + t * 16) = make_uint4(0u, 0u, 0u, 0u);
    tc::fence_proxy_async_smem();
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();
    const uint32_t tmem_base = bars->tmem_base;
    const float emax2 = __uint_as_float(bars->emax2_bits) * 1.000001f;
    const float emax = sqrtf(emax2) * 1.000001f;

    if (warp >= 8 && warp < 12) {
        // ===== producers: one row of the tile per thread ==========================================
        const int r = tid - 256;
        float v[kTcD];
        const float* p_next = nullptr;                     // row pointer of the tile whose loads are in flight
        {
            const int64_t n = (int64_t)blockIdx.x * kTcTileM + r;
            if (blockIdx.x < n_tiles && n < N) {
                const int64_t b = n / HW, hw = n - b * HW;
                p_next = z + (b * kTcD) * HW + hw;
            }
#pragma unroll
            for (int d = 0; d < kTcD; ++d) v[d] = p_next ? ld_stream_f1(p_next + (int64_t)d * HW) : 0.f;
        }
        uint32_t it = 0;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
            const uint32_t s = it & 1u;
            // row of the following tile: its loads replace each quarter of v[] as soon as that quarter is converted
            const int64_t tile2 = tile + gridDim.x;
            const int64_t n2 = tile2 * kTcTileM + r;
            p_next = nullptr;
            if (tile2 < n_tiles && n2 < N) {
                const int64_t b = n2 / HW, hw = n2 - b * HW;
                p_next = z + (b * kTcD) * HW + hw;
            }
            tc::mbar_wait(&bars->a_empty[s], ((it >> 1) & 1u) ^ 1u);
            uint8_t* ahi = smem + kOffA + s * 32768u + (uint32_t)r * 128u;
            uint8_t* alo = ahi + 16384;
            float z2 = 0.f;
#pragma unroll
            for (int qd = 0; qd < 4; ++qd) {
#pragma unroll
                for (int c = 2 * qd; c < 2 * qd + 2; ++c) {
                    uint32_t hi[4], lo[4];
#pragma unroll
                    for (int p = 0; p < 4; ++p) {
                        const float a = v[c * 8 + 2 * p], b = v[c * 8 + 2 * p + 1];
                        z2 = fmaf(a, a, z2);
                        z2 = fmaf(b, b, z2);
                        split_bf16x2(a, b, hi[p], lo[p]);
                    }
                    const uint32_t off = (uint32_t)((c ^ (r & 7)) << 4);
                    *reinterpret_cast<uint4*>(ahi + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                    *reinterpret_cast<uint4*>(alo + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                }
#pragma unroll
                for (int d = 16 * qd; d < 16 * qd + 16; ++d) v[d] = p_next ? ld_stream_f1(p_next + (int64_t)d * HW) : 0.f;
            }
            // ---- the tile's key constants (identical for all 128 rows): max |z| over the tile ------------
            float zm = z2;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) zm = fmaxf(zm, __shfl_xor_sync(0xffffffffu, zm, o));
            if (lane == 0) bars->pmax[s][warp - 8] = zm;
            asm volatile("bar.sync 1, 128;" ::: "memory");                   // the four producer warps only
            if (warp == 8 && lane < 24) {
                const float z2max = fmaxf(fmaxf(bars->pmax[s][0], bars->pmax[s][1]), fmaxf(bars->pmax[s][2], bars->pmax[s][3]));
                // C >= 2 |z||e| (1 + 5e-4) rounded UP to bf16; score + C in (0, Rg) with Rg = 2 C + max|e|^2
                const float Craw = 2.001f * sqrtf(z2max * 1.00001f) * emax + 1e-30f;
                uint32_t Cb = (__float_as_uint(Craw) + 0xFFFFu) >> 16;
                const float C = __uint_as_float(Cb << 16);
                // M 2^-16 >= 2C 2^-16 (the tensor-path error) + 2^-21 (|z|^2 + |e|^2), what the reference formula's float32
                // roundings (<= 2^-22 (|z|^2 + |e|^2) per distance) can reverse, so a row decided on the tensor path gets
                // the formula's first minimum even when |z| >> |e| makes its distances round together.  max|e|^2, which the
                // key range needs anyway, covers that term unless |z|^2 > 31 max|e|^2.
                const float Rg = fmaxf(2.f * C + fmaxf(emax2, 0.03125f * (z2max + emax2)), 1e-30f) * 1.001f;
                // an inf / NaN codebook entry (atomicMax on the bits carries it into emax2) or |z|^2 overflowing float32
                // leaves no key scale: C = NaN makes every key of the tile NaN, and the epilogue sends every row to the
                // full re-check (NaN keys count as close), where the first NaN distance wins as in torch.argmin
                if (!(emax2 <= 3.4028235e38f) || !(Rg <= 3.4028235e38f)) Cb = 0x7FC0u;
                uint32_t mexp = (__float_as_uint(Rg) >> 23) + 1u;            // M = 2^m > Rg
                mexp = mexp < 40u ? 40u : mexp;                              // keep u = M 2^-23 a normal number
                const uint32_t M_hi = mexp << 7;                             // bf16 bits of M
                const uint32_t bigM = (mexp + 3u) << 7;                      // 8 M
                const uint32_t m31 = 0x8000u | ((mexp + 2u) << 7) | 0x60u;   // -7 M = -(1.11b x 2^(m+2))
                const uint32_t uu = (mexp - 23u) << 7;                       // u = M 2^-23
                (void)M_hi;
                const int step = lane >> 3, row = lane & 7;
                uint4 val;
                if (step == 0) val = make_uint4(0x3F80u | (0x3F80u << 16), 0x3F80u | (Cb << 16), bigM, 0u);   // 1, 1, 1, C, 8M
                else if (step == 1) val = make_uint4(0u, 0u, m31 << 16, 0u);                                  // k = 5: -7 M
                else val = make_uint4(0u, 0u, 0u, uu);                                                        // k = 6: u
                *reinterpret_cast<uint4*>(smem + kOffAaug + s * 768u + (uint32_t)step * 256u + (uint32_t)row * 16u) = val;
            }
            tc::fence_proxy_async_smem();
            tc::mbar_arrive(&bars->a_full[s]);
        }
    } else if (warp == 12) {
        // ===== MMA issuer ===========================================================================
        constexpr uint32_t idesc = tc::idesc_bf16_f32(kTcTileM, kTcUnitN);
        const uint32_t smem_base = tc::smem_u32(smem);
        uint32_t it = 0;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
            const uint32_t s = it & 1u;
            tc::mbar_wait(&bars->a_full[s], (it >> 1) & 1u);
            tc::tc_fence_after_sync();
#pragma unroll 1
            for (uint32_t q = 0; q < 2; ++q) {
                tc::mbar_wait(&bars->acc_empty[q], (it & 1u) ^ 1u);
                tc::tc_fence_after_sync();
                if (lane == 0) {
                    const uint32_t d_tmem = tmem_base + q * kTcUnitN;
                    const uint64_t a_hi = tc::smem_desc_kmajor_sw128(smem_base + kOffA + s * 32768u);
                    const uint64_t a_lo = tc::smem_desc_kmajor_sw128(smem_base + kOffA + s * 32768u + 16384u);
                    const uint64_t b_hi = tc::smem_desc_kmajor_sw128(smem_base + kOffBhi + q * 32768u);
                    const uint64_t b_lo = tc::smem_desc_kmajor_sw128(smem_base + kOffBlo + q * 32768u);
                    // small terms first, then the dominant hi*hi product; 16 bf16 = 32 B per K step
#pragma unroll
                    for (uint32_t k = 0; k < 4; ++k) tc::mma_bf16_ss(d_tmem, a_lo + 2 * k, b_hi + 2 * k, idesc, k > 0);
#pragma unroll
                    for (uint32_t k = 0; k < 4; ++k) tc::mma_bf16_ss(d_tmem, a_hi + 2 * k, b_lo + 2 * k, idesc, 1u);
#pragma unroll
                    for (uint32_t k = 0; k < 4; ++k) tc::mma_bf16_ss(d_tmem, a_hi + 2 * k, b_hi + 2 * k, idesc, 1u);
                    // key steps: A = the tile's constant rows (row-group stride 0: all 128 rows read the same 8),
                    // B = the side table of this unit's 256 codes (32 groups x 256 B)
                    const uint64_t b_aug = tc::smem_desc_kmajor_noswizzle(smem_base + kOffBaug + q * 8192u, 128u, 256u);
#pragma unroll
                    for (uint32_t k = 0; k < 3; ++k) {
                        const uint64_t a_aug = tc::smem_desc_kmajor_noswizzle(smem_base + kOffAaug + s * 768u + k * 256u, 128u, 0u);
                        tc::mma_bf16_ss(d_tmem, a_aug, b_aug, idesc, 1u);
                    }
                    tc::mma_commit(&bars->acc_full[q]);
                    if (q == 1) tc::mma_commit(&bars->a_empty[s]);
                }
                __syncwarp();
            }
        }
    } else if (warp > 12) {
        // ===== re-check warps: serve the ring until epilogue group 1 has finished and the ring is empty =========
        // (Letting the PRODUCER warps do this in their waits was tried first: a re-check takes longer than a stage's slack,
        // so every flagged row cost an MMA bubble -- 1.09 ms instead of 0.82 ms at N = 4.2 M.)
        float* zs_warp = reinterpret_cast<float*>(smem + kOffZs) + (warp - 13) * 64;
        for (;;) {
            // `done` is sampled BEFORE the ring is found empty: every push precedes its thread's arrival on epi_done
            const bool done = __all_sync(0xffffffffu, tc::mbar_try_wait(&bars->epi_done, 0u));
            if (!recheck_service_one(bars, ring, z, HW, E, smem, zs_warp, emax, emax2, idx_out, run_count, lane)) {
                if (done && __shfl_sync(0xffffffffu, (int)(ld_volatile_u32(&bars->rq_head) == ld_volatile_u32(&bars->rq_tail)), 0)) break;
                __nanosleep(400);
            }
        }
    } else {
        // ===== epilogue groups =====================================================================
        const int g = warp >> 2;                               // 0: codes 0..255, 1: codes 256..511
        const int r = (warp & 3) * 32 + lane;                  // tile row == TMEM lane
        const uint32_t tbase = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)g * kTcHalfN;
        const float kInf = __uint_as_float(0x7f800000u);
        uint64_t* full = &bars->acc_full[g];
        uint64_t* empty = &bars->acc_empty[g];
        uint32_t it = 0;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
            const int64_t n = tile * kTcTileM + r;
            tc::mbar_wait(full, it & 1u);
            tc::tc_fence_after_sync();
            float* dbg_row = (DBG && dbg != nullptr && n < N) ? dbg + n * kTcK + g * kTcHalfN : nullptr;
            Top2 tr[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) { tr[k].best = kInf; tr[k].second = kInf; tr[k].chunk = 0; tr[k].trk = k; }
            uint32_t va[32], vb[32];
            // 8 chunks of 32 columns, two per loop iteration; the loop is NOT unrolled: a fully unrolled
            // epilogue (30 KB of SASS) thrashed the instruction cache (44% of epilogue stall samples were
            // `no_instruction`)
            tc::tmem_ld_32x32(tbase, va);
#pragma unroll 1
            for (int c = 0; c < 8; c += 2) {
                tmem_ld_wait_for(va);
                tc::tmem_ld_32x32(tbase + (c + 1) * 32, vb);
                epi_chunk<DBG>(va, c, tr, dbg_row);
                tmem_ld_wait_for(vb);
                if (c == 6) {
                    // every column is in registers: hand the accumulator back before the last chunk is processed
                    tc::tc_fence_before_sync();
                    tc::mbar_arrive(empty);
                } else {
                    tc::tmem_ld_32x32(tbase + (c + 2) * 32, va);
                }
                epi_chunk<DBG>(vb, c + 1, tr, dbg_row);
            }

            // ---- this group's candidates: the tracker bests within the decision threshold of the group's best ----
            // (keys live in [M, 2M): threshold = tensor-path error of two scores (<= M 2^-16) + 4 quanta of 8 u (= M 2^-18).)
            // Every test is written !(a - b > thr) so that NaN / inf keys (non-finite latents) count as "close".
            const float gb = fminf(fminf(tr[0].best, tr[1].best), fminf(tr[2].best, tr[3].best));
            const float thr_g = 1.25f * __uint_as_float((__float_as_uint(gb) & 0x7F800000u) - (16u << 23));
            // best tracker (first one holding the minimum) and the best of the OTHER trackers within the threshold; all with
            // compile-time tracker indices (a runtime index would put tr[] in local memory)
            float b1 = tr[0].best;
            int ch1 = tr[0].chunk, k1 = 0;
#pragma unroll
            for (int k = 1; k < 4; ++k)
                if (tr[k].best < b1) { b1 = tr[k].best; ch1 = tr[k].chunk; k1 = k; }
            float key2 = kInf;
            int ch2 = 0, k2 = 0, n_close = 0;
            bool enumerate = false;       // some tracker holds >= 2 codes within the threshold: its second-best code is unknown
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                enumerate = enumerate || !(tr[k].second - gb > thr_g);
                if (k != k1 && !(tr[k].best - gb > thr_g)) {
                    ++n_close;
                    if (n_close == 1 || tr[k].best < key2) { key2 = tr[k].best; ch2 = tr[k].chunk; k2 = k; }
                }
            }
            enumerate = enumerate || n_close > 1;                                          // more candidates than the exchange carries
            auto code_of = [&](float key, int chunk, int k) {
                const int i3 = (int)(__float_as_uint(key) & 7u);
                return g * kTcHalfN + chunk * 32 + ((i3 >> 1) << 3) + (k << 1) + (i3 & 1);
            };
            const int code1 = code_of(b1, ch1, k1);
            const int code2 = n_close > 0 ? code_of(key2, ch2, k2) : 0;
            if (n_close == 0) key2 = kInf;
            const uint32_t slot = it & 1u;
            float* x = xchg + (slot * 128u + r) * 4u;
            if (g == 0) {
                tc::mbar_wait(&bars->x_free[slot], ((it >> 1) & 1u) ^ 1u);
                *reinterpret_cast<float4*>(x) = make_float4(gb, key2, __int_as_float(code1 | (code2 << 16)), enumerate ? 1.f : 0.f);
                tc::mbar_arrive(&bars->x_full[slot]);
            } else {
                tc::mbar_wait(&bars->x_full[slot], (it >> 1) & 1u);
                const float4 o = *reinterpret_cast<const float4*>(x);
                tc::mbar_arrive(&bars->x_free[slot]);
                if (n < N) {
                    const float best = fminf(o.x, gb);
                    const float thr = 1.25f * __uint_as_float((__float_as_uint(best) & 0x7F800000u) - (16u << 23));
                    const bool in10 = !(o.x - best > thr), in20 = !(o.y - best > thr);
                    const bool in11 = !(gb - best > thr), in21 = !(key2 - best > thr);
                    const bool full = (o.w != 0.f && in10) || (enumerate && in11);
                    const int oc = __float_as_int(o.z);
                    const int nc = (int)in10 + (int)in20 + (int)in11 + (int)in21;
                    if (!full && nc == 1) {
                        idx_out[n] = (long long)(in10 ? (oc & 0xFFFF) : code1);            // the one code within the threshold
                    } else {
                        // undecidable on the tensor path: onto the ring; a re-check warp evaluates the candidates exactly
                        // (all 512 codes when a tracker may hide one) and is the only writer of idx_out[n].  Full ring:
                        // wait for the re-check warps (they do nothing else).
                        int cz = 0, cw = 0, m = 0;
                        auto add = [&](bool in, int c) {
                            if (in) { if (m < 2) cz |= c << (16 * m); else cw |= c << (16 * (m - 2)); ++m; }
                        };
                        add(in10, oc & 0xFFFF);
                        add(in20, (oc >> 16) & 0xFFFF);
                        add(in11, code1);
                        add(in21, code2);
                        const uint32_t pos = atomicAdd(&bars->rq_tail, 1u);
                        while ((int)(pos - ld_volatile_u32(&bars->rq_freed)) >= (int)kRqCap) __nanosleep(64);
                        int4* e = ring + (pos % kRqCap);
                        *reinterpret_cast<volatile int*>(&e->y) = full ? 0 : nc;
                        *reinterpret_cast<volatile int*>(&e->z) = cz;
                        *reinterpret_cast<volatile int*>(&e->w) = cw;
                        __threadfence_block();
                        *reinterpret_cast<volatile int*>(&e->x) = (int)n;
                    }
                }
            }
        }
        if (g == 1) tc::mbar_arrive(&bars->epi_done);
    }

    // ---- teardown ---------------------------------------------------------------------------------
    tc::tc_fence_before_sync();
    __syncthreads();
    if (warp == 12) {
        tc::tc_fence_after_sync();
        tc::tmem_dealloc(tmem_base, 512);
    }
    if (tid == 0) {
        __threadfence();
        if (atomicAdd(ws_words + 4, 1u) == gridDim.x - 1) {      // last CTA out: publish this search's re-check count
            __threadfence();
            ws_words[0] = atomicExch(run_count, 0u);
            ws_words[4] = 0u;
        }
    }
}

// Host launcher (called from vq_api.cu).  `ws_words`: the head of the (zero-initialised) quantizer workspace.
int launch_vq_argmin_tc(const float* z, int64_t N, int64_t HW, const float* E, long long* idx, unsigned int* ws_words,
                        float* dbg, cudaStream_t st) {
    const int rc = dbg == nullptr ? allow_dynamic_smem<vq_argmin_tc_kernel<false>>((int)kTcSmemBytes)
                                  : allow_dynamic_smem<vq_argmin_tc_kernel<true>>((int)kTcSmemBytes);
    if (rc != MOVAE_OK) return rc;
    const int sms = sm_count();
    MOVAE_REQUIRE(sms > 0, MOVAE_ERR_CUDA, "CUDA device query failed (no GPU?)");
    const int64_t n_tiles = (N + kTcTileM - 1) / kTcTileM;
    const int64_t grid = n_tiles < sms ? n_tiles : sms;
    if (dbg)
        vq_argmin_tc_kernel<true><<<(unsigned)grid, kTcThreads, kTcSmemBytes, st>>>(z, N, HW, E, idx, ws_words, dbg);
    else
        vq_argmin_tc_kernel<false><<<(unsigned)grid, kTcThreads, kTcSmemBytes, st>>>(z, N, HW, E, idx, ws_words, nullptr);
    MOVAE_CUDA_TRY(cudaGetLastError());
    return MOVAE_OK;
}

}  // namespace movae
