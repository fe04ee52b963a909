// K6 `vq_backward`: autograd backward of /root/reference/models/vq_vae.py:47-55 (the reference's dense
// `one_hot^T @ dq` GEMM and the broadcast gradients of the two MSE losses), with upstream gradients
// d_out [B, D, H, W] (the straight-through output), g_commit and g_embed (device scalars):
//     dz     = d_out + g_commit * 2 (z - q) / (N D)
//     dE[j] += g_embed * 2 / (N D) * sum_{n : idx_n = j} (q_n - z_n)
#include <math.h>

#include <cuda.h>

#include "common.cuh"
#include "vq_common.cuh"
#include "tc_ptx.cuh"

namespace movae {

// K6 generic fallback (any K, D).  grad_out may be null (no gradient reached the quantized output);
// g_commit / g_embed are device scalars (the upstream gradients of the two loss outputs), null = 0.
// dE is accumulated with float32 global atomics: correct but atomic-bound (9 ms at N = 4.2 M in the
// first profile), only used when (K, D) is outside the segmented kernel below.
__global__ void __launch_bounds__(256)
vq_backward_atomic_kernel(const float* __restrict__ grad_out, const float* __restrict__ g_commit,
                          const float* __restrict__ g_embed, const float* __restrict__ z, int64_t N, int D, int64_t HW,
                          const float* __restrict__ E, int K, const long long* __restrict__ idx, float* __restrict__ dz,
                          float* __restrict__ dE) {
    const float scale = 2.0f / (float)((double)N * (double)D);
    const float cc = g_commit ? __ldg(g_commit) * scale : 0.f;
    const float ce = (g_embed && dE) ? __ldg(g_embed) * scale : 0.f;
    for (int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (int64_t)gridDim.x * blockDim.x) {
        long long code = idx[n];
        code = code < 0 ? 0 : (code >= K ? K - 1 : code);
        const int64_t b = n / HW, hw = n - b * HW;
        const int64_t base = (b * D) * HW + hw;
        const float* ep = E + (size_t)code * D;
        float* dep = dE ? dE + (size_t)code * D : nullptr;
#pragma unroll 8
        for (int d = 0; d < D; ++d) {
            const int64_t o = base + (int64_t)d * HW;
            const float zv = ld_stream_f1(z + o);
            const float qv = __ldg(ep + d);
            const float go = grad_out ? ld_stream_f1(grad_out + o) : 0.f;
            if (dz) __stcs(dz + o, fmaf(cc, zv - qv, go));
            if (ce != 0.f) atomicAdd(dep + d, ce * (qv - zv));
        }
    }
}

// K6 for K = 512, D = 64: no floating-point atomics, bit-reproducible.  Two kernels:
//
//  K6a `vq_backward_dz_kernel`  dz = d_out + g_commit * 2 (z - q) / (N D): thread <-> row streaming kernel with
//      the same access pattern as K5 (coalesced NCHW lines, codebook rows from a padded shared copy, 16 loads
//      in flight per thread); reads 2 * 4D + 8 B, writes 4D B per code vector.
//  K6b `vq_backward_dE_kernel`  dE[j] = g_embed * 2 / (N D) * (count_j e_j - S_j),  S_j = sum of the z rows
//      that chose code j.  The CTA keeps the WHOLE S [512, 64] (128 KB) in shared memory.  128-row z tiles arrive
//      through 4-byte cp.async (coalesced 128-byte lines per channel) into a ROW-major tile with row stride 65
//      floats, three buffers deep: both the copies (32 consecutive rows of one channel per warp) and the reads (64
//      consecutive channels of one row per warp) are bank-conflict free -- a [channel][row] tile, which is what bulk
//      (TMA) copies of NCHW runs can produce, costs a 4-way conflict on every read.  Warp w OWNS codes 32w .. 32w+31:
//      it scans the tile's codes 32 at a time (ballot) and adds each of its rows (lanes over channels) into its own
//      slice of S with plain load-add-store: single owner, fixed row order -> no atomics, bit-reproducible, no
//      indirect branch, ~12 instructions and 6 shared-memory wavefronts per row.  Every CTA then stores its S partial
//      and counts; vq_dE_reduce_kernel combines them in CTA order in float64.  Reads 4D + 8 B per code vector.
// History (profiles/r1_vq_launches.csv, profiles/r1_vq_bw.md): float atomics 9.0 ms at N = 4.2 M; fused single pass
// with a per-tile counting sort and register accumulators 1.19 ms; split + the same sort 1.0-2.3 ms; owner-warp scan
// with REGISTER accumulators selected by a warp-uniform switch (a 5-level compare-and-branch tree per row, 427
// instructions per warp and tile, 41% of the stall samples at the per-tile barrier, 4-way conflicts on the TMA-written
// [channel][row] tile) 0.63-0.69 ms = 25% of HBM peak.
constexpr int kBwRows = kPartTileRows, kBwThreads = 1024, kBwChunks = kBwRows / 32;
constexpr int kBwParts = kBwThreads / kBwRows;                 // copy roles per row: each covers kBwD / kBwParts channels
constexpr int kBwOwn = kBwK / (kBwThreads / 32);               // codes owned by one warp (16)
constexpr int kBwOwnShift = 4;
static_assert((1 << kBwOwnShift) == kBwOwn, "owner shift");
constexpr int kBwLdRow = kBwD + 1;       // row-major tile, row stride 65 floats: conflict-free copies and reads
constexpr int kBwDepth = 3;              // tile buffers: two tiles (64 KB) in flight while one is processed
constexpr size_t kBwSmemBytes = sizeof(float) * ((size_t)kBwK * kBwD + kBwDepth * (size_t)kBwRows * kBwLdRow) +
                                sizeof(unsigned short) * (kBwDepth * (size_t)kBwRows);
static_assert(kBwSmemBytes <= 227 * 1024, "K6b shared memory");
constexpr int kDzThreads = 512;

template <bool STAGE, int THREADS>
__global__ void __launch_bounds__(THREADS, 1)
vq_backward_dz_kernel(const float* __restrict__ grad_out, const float* __restrict__ g_commit, const float* __restrict__ z,
                      int64_t N, int D, int64_t HW, const float* __restrict__ E, int K, const long long* __restrict__ idx,
                      float* __restrict__ dz) {
    extern __shared__ float Es[];                           // STAGE: K x (D+1)
    const int tid = threadIdx.x;
    const float cc = g_commit ? __ldg(g_commit) * (2.0f / (float)((double)N * (double)D)) : 0.f;
    if (STAGE) {
        for (int i = tid; i < K * D; i += THREADS) {
            const int j = i / D, d = i - j * D;
            Es[j * (D + 1) + d] = __ldg(E + i);
        }
        __syncthreads();
    }
    for (int64_t n0 = (int64_t)blockIdx.x * THREADS; n0 < N; n0 += (int64_t)gridDim.x * THREADS) {
        const int64_t n = n0 + tid;
        if (n >= N) continue;
        long long code = idx[n];
        code = code < 0 ? 0 : (code >= K ? K - 1 : code);
        const int64_t b = n / HW, hw = n - b * HW;
        const int64_t base = (b * D) * HW + hw;
        const float* ep = STAGE ? Es + (size_t)code * (D + 1) : E + (size_t)code * D;
        int d0 = 0;
        // batches of 16 channels, software-pipelined like K5: the loads of batch i + 1 are issued before batch i is stored
        float za[16], ga[16], zb[16], gb[16];
        const int n_batches = D / 16;
        auto load = [&](float (&zv)[16], float (&go)[16], int dd) {
#pragma unroll
            for (int i = 0; i < 16; ++i) zv[i] = __ldcs(z + base + (int64_t)(dd + i) * HW);
            if (grad_out != nullptr) {
#pragma unroll
                for (int i = 0; i < 16; ++i) go[i] = __ldcs(grad_out + base + (int64_t)(dd + i) * HW);
            } else {
#pragma unroll
                for (int i = 0; i < 16; ++i) go[i] = 0.f;
            }
        };
        auto store = [&](const float (&zv)[16], const float (&go)[16], int dd) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const float qv = STAGE ? ep[dd + i] : __ldg(ep + dd + i);
                __stcs(dz + base + (int64_t)(dd + i) * HW, fmaf(cc, zv[i] - qv, go[i]));
            }
        };
        if (n_batches > 0) load(za, ga, 0);
        for (int bt = 0; bt < n_batches; bt += 2, d0 += 32) {
            const bool has_b = bt + 1 < n_batches;
            if (has_b) load(zb, gb, d0 + 16);
            store(za, ga, d0);
            if (!has_b) { d0 += 16; break; }
            if (bt + 2 < n_batches) load(za, ga, d0 + 32);
            store(zb, gb, d0 + 16);
        }
        for (; d0 < D; ++d0) {
            const float zv = __ldcs(z + base + (int64_t)d0 * HW);
            const float go = grad_out ? __ldcs(grad_out + base + (int64_t)d0 * HW) : 0.f;
            const float qv = STAGE ? ep[d0] : __ldg(ep + d0);
            __stcs(dz + base + (int64_t)d0 * HW, fmaf(cc, zv - qv, go));
        }
    }
}

__device__ __forceinline__ void cp_async_f32(float* smem_dst, const float* gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src)
                 : "memory");
}

__global__ void __launch_bounds__(kBwThreads, 1)
vq_backward_dE_kernel(const float* __restrict__ z, int64_t N, int64_t HW, const long long* __restrict__ idx,
                      float* __restrict__ partials) {
    extern __shared__ __align__(16) float bw_smem[];
    float* S = bw_smem;                                                    // [K][D], warp w owns rows 16w .. 16w+15
    float* zs0 = S + kBwK * kBwD;                                          // kBwDepth x [rows][65]
    unsigned short* codes0 = reinterpret_cast<unsigned short*>(zs0 + kBwDepth * kBwRows * kBwLdRow);   // kBwDepth x [rows]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    constexpr int kCh = kBwD / kBwParts;                       // channels per copy role (8)
    const int r = tid & (kBwRows - 1), part = tid / kBwRows;   // copy role: row r, channels kCh*part .. kCh*part+kCh-1
    const uint32_t hw_u = (uint32_t)HW;                        // N < 2^31 (checked by the C entry point): 32-bit index math

    for (int i = tid; i < kBwK * kBwD; i += kBwThreads) S[i] = 0.f;
    int my_count = 0;                                          // lane l < 16 of warp w counts code 16 w + l

    const int64_t n_tiles = (N + kBwRows - 1) / kBwRows;
    auto issue_tile = [&](int64_t tile, int buf) {
        float* zs = zs0 + buf * (kBwRows * kBwLdRow);
        unsigned short* codes = codes0 + buf * kBwRows;
        const int64_t n = tile * kBwRows + r;
        const bool ok = tile < n_tiles && n < N;
        if (ok) {
            const uint32_t b = (uint32_t)n / hw_u, hw = (uint32_t)n - b * hw_u;
            const float* src = z + ((int64_t)b * kBwD + part * kCh) * HW + hw;
            float* dst = zs + r * kBwLdRow + part * kCh;
#pragma unroll
            for (int d = 0; d < kCh; ++d) cp_async_f32(dst + d, src + (int64_t)d * HW);
        }
        if (part == 0) {
            unsigned short code = 0xffffu;                     // >> 4 = 4095: no warp owns it
            if (ok) {
                const long long cl = __ldg(idx + n);
                code = (unsigned short)(cl < 0 ? 0 : (cl >= kBwK ? kBwK - 1 : (int)cl));
            }
            codes[r] = code;
        }
        asm volatile("cp.async.commit_group;" ::: "memory");          // one group per tile (possibly empty)
    };

    for (int p = 0; p < kBwDepth - 1; ++p) issue_tile(blockIdx.x + (int64_t)p * gridDim.x, p);
    float* Sw = S + warp * kBwOwn * kBwD;
    uint32_t it = 0;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
        const int buf = (int)(it % kBwDepth);
        const float* zs = zs0 + buf * (kBwRows * kBwLdRow);
        const unsigned short* codes = codes0 + buf * kBwRows;
        asm volatile("cp.async.wait_group %0;" ::"n"(kBwDepth - 2) : "memory");
        __syncthreads();                                      // this tile has landed; everyone is done with the previous one
        issue_tile(tile + (int64_t)(kBwDepth - 1) * gridDim.x, (int)((it + kBwDepth - 1) % kBwDepth));   // refills the previous tile's buffer
#pragma unroll
        for (int c = 0; c < kBwChunks; ++c) {
            const int code = codes[c * 32 + lane];
            unsigned mine = __ballot_sync(0xffffffffu, (code >> kBwOwnShift) == warp);
            while (mine) {
                const int l = __ffs(mine) - 1;
                mine &= mine - 1;
                const int j = __shfl_sync(0xffffffffu, code, l) & (kBwOwn - 1);
                const float* zr = zs + (c * 32 + l) * kBwLdRow;
                float* sj = Sw + j * kBwD;
                // plain load-add-store: the warp is the only writer of its slice and the LSU keeps program order
                const float v0 = zr[lane], v1 = zr[lane + 32];
                const float s0 = sj[lane], s1 = sj[lane + 32];
                sj[lane] = s0 + v0;
                sj[lane + 32] = s1 + v1;
                my_count += (lane == j) ? 1 : 0;
            }
        }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    float* out = partials + (size_t)blockIdx.x * kPartFloats;
    for (int i = tid; i < kBwK * kBwD; i += kBwThreads) out[i] = S[i];
    if (lane < kBwOwn) out[kBwK * kBwD + warp * kBwOwn + lane] = __int_as_float(my_count);   // lane l of warp w counts code 16 w + l
}

// ---- K6b, TMA + tensor-memory variant (H*W % 32 == 0, 16-byte aligned z and idx) ------------------------------------
// The ownership scheme of vq_backward_dE_kernel (one warp is the only adder of its codes, rows in a fixed order:
// bit-reproducible, no atomics; the results are bit-identical to that kernel), re-cut around what bounded it:
//  (a) z arrives through TENSOR-MAP bulk copies (cp.async.bulk.tensor.3d -> SASS UTMALDG): z is described to the TMA
//      unit as a 3-D tensor (H*W, D, B) and ONE instruction fetches a box of 32 rows x 64 channels (8 KB, 64 runs of
//      128 bytes); a 128-row unit is four boxes plus one 1 KB bulk copy of the indices, issued by a single thread.
//      (1-D bulk copies, one per channel run, were tried first: the TMA unit spends ~70-90 cycles per copy whatever
//      its size, so 64 copies of 256-512 bytes per tile ran at 1.0 TB/s; the 4-byte LDGSTS of the kernel above cost 8
//      cycles of LSU time per 128 bytes plus ~170 instructions of address arithmetic per thread and tile.)
//  (b) the per-code sums S [512][64] live in TENSOR MEMORY, used as a 256 KB scratchpad: owner warp w keeps code j of
//      its 18-19 codes in columns 2j, 2j+1 of its own block of columns in its own lane quadrant (lane l = channels l and
//      l + 32) and does load-add-store with tcgen05.ld / tcgen05.st .32x32b.x2 (SASS LDTM / STTM) -- the address is a
//      run-time value, which registers cannot offer without a branchy switch (measured: slower).  Round 1 kept S in
//      shared memory: that left ~80 KB for the TMA ring, and throughput = bytes in flight / length of a buffer's cycle
//      (TMA latency + router + owners, ~3.3 us) capped the kernel at 3.6-3.9 TB/s.  The ring is now 6 x 33 KB.
//  (c) three ROUTER warps (every third unit each) counting-sort a unit's rows by owner warp (MATCH.ANY per 32 rows for
//      the rank, per-chunk group sizes, a warp scan over the owners) into `order`: one entry per row = (byte offset of
//      the row inside the unit's boxes before the lane swizzle) << 5 | (code - the owner's first code); rows of one owner
//      stay in row order.  An owner reads start[w] .. start[w + 1] and runs ~17 branch-free instructions per row.
//  (d) no CTA-wide barrier in the loop: full[buf] (TMA landed) -> router -> routed[buf] -> owners -> empty[buf] ->
//      producer -- a warp that owns a popular code only delays the refill of a buffer kTmDepth units away.
// The box lands as [channel][32 rows] with the 128-byte swizzle (16-byte chunk index XOR channel & 7); reads by
// lanes-over-channels are 4-way bank conflicted -- inherent to any 16-byte-granular layout of NCHW runs -- and are what
// bounds the kernel now (shared-memory wavefronts 79 %, issue slots 76 %, 5.5 TB/s: profiles/r2_k6b_tmem.md).
constexpr int kTmRows = 128, kTmChunks = kTmRows / 32, kTmDepth = 6, kTmRouters = 3, kTmConsumers = 31 - kTmRouters, kTmThreads = 1024;
constexpr int kTmOwnMax = (kBwK + kTmConsumers - 1) / kTmConsumers;                       // codes per owner warp (18 or 19)
static_assert(kTmOwnMax * 2 * ((kTmConsumers + 3) / 4) <= 512, "TMEM columns");
// A router only waits on the barriers of ITS units.  mbarrier parity waits are correct only for a waiter that sees every
// phase of a barrier, so consecutive uses of a ring buffer must belong to the same router: depth % routers == 0.  (With
// 3 routers on a ring of 4 or 8, a router that reached its next unit while the buffer's previous TMA was still in flight
// passed the parity test on a stale phase and routed garbage: intermittent hangs and illegal addresses.)
static_assert(kTmDepth % kTmRouters == 0, "every ring buffer must always be served by the same router warp");
constexpr int kTmChunkBytes = 32 * kBwD * 4;                                              // one box: 8 KB
constexpr size_t kTmUnitBytes = (size_t)kTmChunks * kTmChunkBytes;                       // 32 KB: every box stays 1024-byte aligned
constexpr size_t kTmIdxBytes = sizeof(long long) * kTmRows;                               // 1 KB per unit, in a separate ring
constexpr size_t kTmRouteBytes = sizeof(unsigned int) * (32 + kTmChunks * 32 + kTmRows);  // per unit: start [32], chunk sizes [4][32], order [128]
static_assert(kTmRouteBytes % 16 == 0, "route block alignment");
constexpr size_t kTmSmemBytes = kTmDepth * (kTmUnitBytes + kTmIdxBytes + kTmRouteBytes) + 3 * kTmDepth * sizeof(uint64_t) +
                                sizeof(int) * kBwK + 16 + 1024;
static_assert(kTmSmemBytes <= 227 * 1024, "K6b (TMA) shared memory");

__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     (uint32_t)__cvta_generic_to_shared(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"((uint32_t)__cvta_generic_to_shared(bar))
                 : "memory");
}
__device__ __forceinline__ void tma_box_3d(void* smem_dst, const CUtensorMap* tmap, int c0, int c1, int c2, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
            (uint32_t)__cvta_generic_to_shared(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(tmap)), "r"(c0), "r"(c1), "r"(c2), "r"((uint32_t)__cvta_generic_to_shared(bar))
        : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ int tm_owner(int code) { return (code * kTmConsumers) >> 9; }   // owner warp of a code: 18 or 19 codes each
__device__ __forceinline__ int tm_first(int w) { return (w * kBwK + kTmConsumers - 1) / kTmConsumers; }   // first code of owner w
// TMEM as a 256 KB scratchpad: lane l of the issuing warp reads / writes two consecutive 32-bit columns of TMEM lane
// (32 * (warp % 4) + l) -- a warp can only reach its own lane quadrant.
__device__ __forceinline__ void tmem_ld_x2(uint32_t taddr, float& a, float& b) {
    uint32_t x, y;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(x), "=r"(y) : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    a = __uint_as_float(x);
    b = __uint_as_float(y);
}
__device__ __forceinline__ void tmem_st_x2(uint32_t taddr, float a, float b) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(taddr), "r"(__float_as_uint(a)), "r"(__float_as_uint(b))
                 : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

__global__ void __launch_bounds__(kTmThreads, 1)
vq_backward_dE_tma_kernel(const __grid_constant__ CUtensorMap tmap, int64_t N, int64_t HW, const long long* __restrict__ idx,
                          float* __restrict__ partials) {
    extern __shared__ uint8_t tm_smem_raw[];
    const uint32_t raw_addr = (uint32_t)__cvta_generic_to_shared(tm_smem_raw);
    uint8_t* smem = tm_smem_raw + (((raw_addr + 1023u) & ~1023u) - raw_addr);      // swizzled boxes need 1024-byte alignment
    uint8_t* units = smem;                                                         // kTmDepth x 4 boxes
    uint8_t* idxs = units + kTmDepth * kTmUnitBytes;                               // kTmDepth x idx [128] (int64, as copied)
    uint8_t* routes = idxs + kTmDepth * kTmIdxBytes;                               // kTmDepth x { start [32], sizes [4][32], order [128] }
    uint64_t* full = reinterpret_cast<uint64_t*>(routes + kTmDepth * kTmRouteBytes);
    uint64_t* routed = full + kTmDepth;
    uint64_t* empty = routed + kTmDepth;
    int* cnt = reinterpret_cast<int*>(empty + kTmDepth);                           // rows per code (integer atomics: order-free)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(cnt + kBwK);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (tid < kBwK) cnt[tid] = 0;
    if (tid == 0) {
        for (int b = 0; b < kTmDepth; ++b) {
            tc::mbar_init(&full[b], 1);
            tc::mbar_init(&routed[b], 1);
            tc::mbar_init(&empty[b], kTmConsumers);
        }
        tc::mbar_fence_init();
    }
    if (warp == 31) tc::tmem_alloc(tmem_slot, 512);                                // the per-code sums S live in TENSOR MEMORY
    tc::tc_fence_before_sync();
    __syncthreads();
    tc::tc_fence_after_sync();
    const uint32_t tmem_base = *tmem_slot;

    const int64_t n_units = (N + kTmRows - 1) / kTmRows;
    if (warp == 31) {
        // ---- producer: one thread, five TMA instructions per unit ---------------------------------------------------
        if (lane == 0) {
            const uint32_t hw_u = (uint32_t)HW;
            uint32_t it = 0;
            for (int64_t unit = blockIdx.x; unit < n_units; unit += gridDim.x, ++it) {
                const int buf = (int)(it % kTmDepth);
                uint8_t* ub = units + buf * kTmUnitBytes;
                tc::mbar_wait(&empty[buf], ((it / kTmDepth) & 1u) ^ 1u);   // a fresh barrier passes parity 1
                const uint32_t n0 = (uint32_t)(unit * kTmRows);
                const int rows = (int)((N - n0) < kTmRows ? (N - n0) : kTmRows);      // a multiple of 32 (N % 32 == 0)
                mbar_expect_tx_(&full[buf], (uint32_t)(rows / 32) * kTmChunkBytes + (uint32_t)rows * 8u);
                for (int q = 0; q < rows / 32; ++q) {
                    const uint32_t n = n0 + 32u * q, b = n / hw_u, hw0 = n - b * hw_u;   // a box never straddles images
                    tma_box_3d(ub + q * kTmChunkBytes, &tmap, (int)hw0, 0, (int)b, &full[buf]);
                }
                bulk_g2s(idxs + buf * kTmIdxBytes, idx + n0, (uint32_t)rows * 8u, &full[buf]);
            }
        }
    } else if (warp >= kTmConsumers) {
        // ---- routers (units dealt round-robin): a warp counting-sorts a unit's rows by OWNER WARP (stable: rows of one owner stay in row order) so
        // that an owner reads one compact entry per row -- (byte offset of the row inside the unit's boxes before the lane
        // swizzle) << 5 | (code - the owner's first code) -- instead of scanning masks and code arrays; also counts the rows
        // per code ----------
        const unsigned lt_mask = (1u << lane) - 1u;
        const uint32_t row_off = (((uint32_t)lane >> 2) << 4) | (((uint32_t)lane & 3u) << 2);
        uint32_t it = 0;
        for (int64_t unit = blockIdx.x; unit < n_units; unit += gridDim.x, ++it) {
            if ((int)(it % kTmRouters) != warp - kTmConsumers) continue;
            const int buf = (int)(it % kTmDepth);
            const int* cs = reinterpret_cast<const int*>(idxs + buf * kTmIdxBytes);
            unsigned int* start = reinterpret_cast<unsigned int*>(routes + buf * kTmRouteBytes);
            unsigned int* sz = start + 32;
            unsigned int* order = sz + kTmChunks * 32;
            const int64_t n0 = unit * kTmRows;
            const int rows = (int)((N - n0) < kTmRows ? (N - n0) : kTmRows);
            tc::mbar_wait(&full[buf], (it / kTmDepth) & 1u);
            // (the owners are done with this buffer's route block: the producer refilled it only after empty[buf])
#pragma unroll
            for (int q = 0; q < kTmChunks; ++q) sz[q * 32 + lane] = 0u;
            int code[kTmChunks], owner[kTmChunks];
            unsigned rank[kTmChunks];
#pragma unroll
            for (int q = 0; q < kTmChunks; ++q) {
                const int row = q * 32 + lane;
                code[q] = 0;
                owner[q] = 31;                                           // owner 31: nobody (its slots are dummies)
                if (row < rows) {
                    int c = cs[2 * row];                                 // low word of the int64 index
                    c = c < 0 ? 0 : (c >= kBwK ? kBwK - 1 : c);
                    code[q] = c;
                    owner[q] = tm_owner(c);
                    atomicAdd(&cnt[c], 1);
                }
            }
            __syncwarp();
#pragma unroll
            for (int q = 0; q < kTmChunks; ++q) {
                const unsigned peers = __match_any_sync(0xffffffffu, owner[q]);
                rank[q] = (unsigned)__popc(peers & lt_mask);
                if (rank[q] == 0u) sz[q * 32 + owner[q]] = (unsigned)__popc(peers);      // group leader
            }
            __syncwarp();
            // lane o: rows of owner o in this unit -> exclusive scan over the owners
            unsigned tot = 0u;
#pragma unroll
            for (int q = 0; q < kTmChunks; ++q) tot += sz[q * 32 + lane];
            unsigned incl = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned y = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += y;
            }
            start[lane] = incl - tot;                                    // start[o] .. start[o + 1]: owner o's entries (o <= 30)
            __syncwarp();
#pragma unroll
            for (int q = 0; q < kTmChunks; ++q) {
                unsigned base = start[owner[q]];
#pragma unroll
                for (int p = 0; p < q; ++p) base += sz[p * 32 + owner[q]];
                if (owner[q] < kTmConsumers)
                    order[base + rank[q]] = ((((uint32_t)q << 13) | row_off) << 5) | (uint32_t)(code[q] - tm_first(owner[q]));
            }
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&routed[buf]);               // release: start and order are visible to waiters
        }
    } else {
        // ---- owner warps: warp w owns the codes c with tm_owner(c) == w; lane l adds channels l and l + 32.  The sums live in
        // TMEM: code j of the warp = columns 2 j, 2 j + 1 of the warp's block of columns in its own lane quadrant (the address
        // is a run-time value -- what registers cannot offer -- and no shared memory is spent on S, so the ring is 6 deep) ------
        const uint32_t swsh = ((uint32_t)lane & 7u) << 4;                // the 128-byte swizzle: 16-byte chunk index ^ (channel & 7)
        const uint32_t tbase = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)((warp >> 2) * 2 * kTmOwnMax);
        const int first = tm_first(warp), n_own = tm_first(warp + 1) - first;
        for (int j = 0; j < n_own; ++j) tmem_st_x2(tbase + 2u * (uint32_t)j, 0.f, 0.f);
        uint32_t it = 0;
        for (int64_t unit = blockIdx.x; unit < n_units; unit += gridDim.x, ++it) {
            const int buf = (int)(it % kTmDepth);
            const uint8_t* ubl = units + buf * kTmUnitBytes + (uint32_t)lane * 128u;   // channel `lane` (lane + 32: + 4096 B)
            const unsigned int* start = reinterpret_cast<const unsigned int*>(routes + buf * kTmRouteBytes);
            const unsigned int* order = start + 32 + kTmChunks * 32;
            const uint32_t par = (it / kTmDepth) & 1u;
            tc::mbar_wait(&routed[buf], par);
            tc::mbar_wait(&full[buf], par);                             // already complete: makes the TMA writes visible here too
            unsigned i = start[warp];
            const unsigned i_end = start[warp + 1];
            if (i < i_end) {
                // the loads of row i + 1 are issued before row i's load-add-store on TMEM (the warp is the only writer of its
                // columns; tcgen05.wait::st orders a store before the next row's load of the same column)
                uint32_t e = order[i];
                const float* zr = reinterpret_cast<const float*>(ubl + ((e >> 5) ^ swsh));
                float v0 = zr[0], v1 = zr[1024];
                for (;;) {
                    const uint32_t taddr = tbase + ((e & 31u) << 1);
                    const float c0 = v0, c1 = v1;
                    const bool more = ++i < i_end;
                    if (more) {
                        e = order[i];
                        zr = reinterpret_cast<const float*>(ubl + ((e >> 5) ^ swsh));
                        v0 = zr[0];
                        v1 = zr[1024];
                    }
                    float s0, s1;
                    tmem_ld_x2(taddr, s0, s1);
                    tmem_st_x2(taddr, s0 + c0, s1 + c1);
                    if (!more) break;
                }
            }
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&empty[buf]);
        }
        float* out_w = partials + (size_t)blockIdx.x * kPartFloats + (size_t)first * kBwD + lane;
        for (int j = 0; j < n_own; ++j) {
            float s0, s1;
            tmem_ld_x2(tbase + 2u * (uint32_t)j, s0, s1);
            out_w[j * kBwD] = s0;
            out_w[j * kBwD + 32] = s1;
        }
    }
    tc::tc_fence_before_sync();
    __syncthreads();
    if (warp == 31) {
        tc::tc_fence_after_sync();
        tc::tmem_dealloc(tmem_base, 512);
    }
    float* out = partials + (size_t)blockIdx.x * kPartFloats;
    if (tid < kBwK) out[kBwK * kBwD + tid] = __int_as_float(cnt[tid]);
}

// Tensor map of z as (H*W, D, B) float32 with boxes of 32 x 64 x 1 and the 128-byte swizzle; the driver entry point is
// resolved once through the runtime (no link against libcuda).
static int make_z_tensor_map(const float* z, int64_t B, int64_t HW, CUtensorMap* out) {
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeFn encode = nullptr;
    if (encode == nullptr) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        MOVAE_CUDA_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        MOVAE_REQUIRE(fn != nullptr && qres == cudaDriverEntryPointSuccess, MOVAE_ERR_CUDA, "CUDA driver has no cuTensorMapEncodeTiled");
        encode = reinterpret_cast<EncodeFn>(fn);
    }
    const cuuint64_t dims[3] = {(cuuint64_t)HW, (cuuint64_t)kBwD, (cuuint64_t)B};
    const cuuint64_t strides[2] = {(cuuint64_t)HW * 4u, (cuuint64_t)HW * 4u * kBwD};
    const cuuint32_t box[3] = {32u, (cuuint32_t)kBwD, 1u};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    const CUresult r = encode(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(z), dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    MOVAE_REQUIRE(r == CUDA_SUCCESS, MOVAE_ERR_CUDA, "CUDA cuTensorMapEncodeTiled failed (%d) for H*W=%lld B=%lld", (int)r,
                  (long long)HW, (long long)B);
    return MOVAE_OK;
}

// dE[j, d] += g_embed * 2 / (N D) * (count_j e[j, d] - S[j, d]), with count_j and S_j combined from K6b's partials in
// the fixed float64 order of k6b_combine_partials: bit-reproducible.
__global__ void __launch_bounds__(kRdThreads)
vq_dE_reduce_kernel(const float* __restrict__ partials, int n_parts, const float* __restrict__ g_embed,
                    const float* __restrict__ E, int64_t N, float* __restrict__ dE) {
    const int q = threadIdx.x % kRdQuads, g = threadIdx.x / kRdQuads;
    const int quad = blockIdx.x * kRdQuads + q;                 // output elements 4 quad .. 4 quad + 3 (one code: D % 4 == 0)
    double st[4];
    long long ct;
    k6b_combine_partials(partials, n_parts, quad, q, g, st, ct);
    if (g == 0 && quad < kBwK * kBwD / 4) {
        const double ce = (double)__ldg(g_embed) * (double)(2.0f / (float)((double)N * (double)kBwD));
        const float4 e = __ldg(reinterpret_cast<const float4*>(E) + quad);
        const float ev[4] = {e.x, e.y, e.z, e.w};
        float4 out = reinterpret_cast<float4*>(dE)[quad];
        float* ov = reinterpret_cast<float*>(&out);
#pragma unroll
        for (int i = 0; i < 4; ++i) ov[i] += (float)(ce * ((double)ct * (double)ev[i] - st[i]));
        reinterpret_cast<float4*>(dE)[quad] = out;
    }
}

// K6b's per-CTA partials (S [K, D] then the counts, kPartFloats each) for K = 512, D = 64: the tensor-map kernel when
// 32-row boxes never straddle images and the copies are 16-byte aligned, else the cp.async one.  *n_parts = CTAs launched.
int launch_k6b_partials(const float* z, int64_t N, int64_t HW, const long long* idx, float* partials, int* n_parts,
                        cudaStream_t st) {
    int grid = vq_backward_parts(N, kBwK, kBwD);
    if (grid > sm_count()) grid = sm_count();
    const bool tma_ok = (HW % 32 == 0) && reinterpret_cast<uintptr_t>(z) % 16 == 0 && reinterpret_cast<uintptr_t>(idx) % 16 == 0 &&
                        HW * 4 * kBwD < ((int64_t)1 << 40);
    if (tma_ok) {
        CUtensorMap tmap;
        int rc = make_z_tensor_map(z, N / HW, HW, &tmap);
        if (rc == MOVAE_OK) rc = allow_dynamic_smem<vq_backward_dE_tma_kernel>((int)kTmSmemBytes);
        if (rc != MOVAE_OK) return rc;
        vq_backward_dE_tma_kernel<<<grid, kTmThreads, kTmSmemBytes, st>>>(tmap, N, HW, idx, partials);
    } else {
        const int rc = allow_dynamic_smem<vq_backward_dE_kernel>((int)kBwSmemBytes);
        if (rc != MOVAE_OK) return rc;
        vq_backward_dE_kernel<<<grid, kBwThreads, kBwSmemBytes, st>>>(z, N, HW, idx, partials);
    }
    MOVAE_CUDA_TRY(cudaGetLastError());
    *n_parts = grid;
    return MOVAE_OK;
}

int launch_vq_backward(const float* grad_out, const float* g_commit, const float* g_embed, const float* z, int64_t N, int D,
                       int64_t HW, const float* E, int K, const long long* idx, float* dz, float* dE, float* partials,
                       cudaStream_t st) {
    const int sms = sm_count();
    MOVAE_REQUIRE(sms > 0, MOVAE_ERR_CUDA, "CUDA device query failed (no GPU?)");
    const bool want_dE = dE != nullptr && g_embed != nullptr;
    const bool quads_ok = !want_dE || (reinterpret_cast<uintptr_t>(dE) % 16 == 0 && reinterpret_cast<uintptr_t>(E) % 16 == 0);
    if (K == kBwK && D == kBwD && (partials != nullptr || !want_dE) && quads_ok) {
        if (dz != nullptr && N <= kSmallN) {
            vq_backward_dz_kernel<false, 256><<<(unsigned)((N + 255) / 256), 256, 0, st>>>(grad_out, g_commit, z, N, D, HW, E, K, idx, dz);
            MOVAE_CUDA_TRY(cudaGetLastError());
        } else if (dz != nullptr) {
            const int rc = allow_dynamic_smem<vq_backward_dz_kernel<true, kDzThreads>>(160 * 1024);
            if (rc != MOVAE_OK) return rc;
            int64_t grid = (N + kDzThreads - 1) / kDzThreads;
            if (grid > sms) grid = sms;
            vq_backward_dz_kernel<true, kDzThreads><<<(unsigned)grid, kDzThreads, (size_t)K * (D + 1) * sizeof(float), st>>>(
                grad_out, g_commit, z, N, D, HW, E, K, idx, dz);
            MOVAE_CUDA_TRY(cudaGetLastError());
        }
        if (want_dE) {
            int grid = 0;
            const int rc = launch_k6b_partials(z, N, HW, idx, partials, &grid, st);
            if (rc != MOVAE_OK) return rc;
            vq_dE_reduce_kernel<<<(K * D / 4 + kRdQuads - 1) / kRdQuads, kRdThreads, 0, st>>>(partials, grid, g_embed, E, N, dE);
            MOVAE_CUDA_TRY(cudaGetLastError());
        }
        return MOVAE_OK;
    }
    int64_t grid = (N + 255) / 256;
    if (grid > (int64_t)sms * 8) grid = (int64_t)sms * 8;
    if (grid < 1) grid = 1;
    vq_backward_atomic_kernel<<<(unsigned)grid, 256, 0, st>>>(grad_out, g_commit, g_embed, z, N, D, HW, E, K, idx, dz, dE);
    MOVAE_CUDA_TRY(cudaGetLastError());
    return MOVAE_OK;
}

}  // namespace movae
