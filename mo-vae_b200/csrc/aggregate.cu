// Fused aggregation step:  g (=|+=) w(J J^T) @ J  in ONE persistent launch per GPU.
//
// Replaces the whole chain the reference runs per training step behind `aggregator(J)` (call sites
// /root/reference/main.py:189-196): torchjd compute_gramian (`J @ J.T`), the weighting (UPGrad QPs on the host,
// utils/torchmoo/mgda.py:221-272, aligned_mtl.py:97-133, nupgrad.py:122-158, comfort.py:148-158), `weights @ J` and the
// split / `.grad` write-back -- and, across GPUs, the k x k exchange of the P-sharded path (SURVEY.md 8e).
//
// One grid of (SMs x resident CTAs) co-resident CTAs (cooperative launch), three phases:
//   1. every CTA streams its share of J (tiles dealt round-robin, front to back) into k(k+1)/2 Gramian partials
//      (gram_device.cuh) and takes a ticket;
//   2. the LAST CTA to arrive sums the partials in a fixed order, (multi-GPU) stores this rank's k x k float64 partial into
//      every peer's exchange buffer over NVLink (peer-to-peer stores + release flag), waits for the peers' flags, sums
//      the ranks' partials in RANK ORDER -- bit-identical input on every rank --, runs the small solve (solve_device.cuh)
//      and publishes w with a release store; the other CTAs have meanwhile issued the loads of their first phase-3 tile
//      and poll that flag;
//   3. every CTA walks its tiles back to front (the end of J is still in L2), FMAs with w and streams the result into
//      the flat .grad buffer (recombine_device.cuh).
// (A dedicated solver CTA that pre-runs the solve on a dummy Gramian to warm its instruction cache was tried: the solve
// phase stayed at 10.6 us for k = 3 -- it is bound by its dependent float64 divide / sqrt chains, not by instruction fetch.)
// Versus K1 -> K2 -> K3 as three launches this removes two launch gaps and a kernel ramp per step (they are 40 % of a
// step at P = 1e7) and, in the P-sharded path, the separate collective.  Nothing about a step is a host-side kernel
// argument (the exchange sequence number lives in the exchange buffer): the launch is CUDA-graph capturable.
//
// Roofline: HBM.  Algorithmic traffic 4*k*P (phase 1) + 4*k*P + 4*P (phase 3) bytes.
// Workspace: movae_gram_workspace_bytes(k), zero-filled once; header layout: GramWorkspace (gram_device.cuh).  The
// timestamps of the last launch are globaltimer ns: start, all partials in, weights published, end, partials combined,
// exchange done.
#include "recombine_device.cuh"
#include "solve_device.cuh"

namespace movae {

int fill_solve_params(int k, const movae_solve_spec* spec, SolveParams* out);          // solve.cu
int check_solve_vectors(const SolveParams& p, const float* d_vec, const float* d_aux);  // solve.cu

constexpr int kAggThreads = 256;
static_assert(kAggThreads == kGramThreads && kAggThreads == kRecThreads && kAggThreads == kSolveThreads, "one CTA shape");

struct AggArgs {
    const float* J;
    int64_t P, ldJ;
    unsigned char* ws;
    const float* vec;
    const float* aux;
    float* out;           // nullptr: weights only (phases 1 and 2)
    int accumulate;
    float* w_out;         // [k] (COMFORT: [2k], the MGDA weights second)
    double* diag_out;     // [MOVAE_DIAG_DOUBLES] or nullptr
    double* G_out;        // [k*k] summed Gramian, or nullptr
    int64_t window_gram;  // L2 hand-off (below), in steps per CTA of the Gramian pass
    int64_t window_rec;   //   and of the recombination pass
};

// ---- L2 hand-off of the tail of J from phase 1 to phase 3 ----------------------------------------------------------------
// Phase 3 walks each CTA's deal in the reverse of phase 1's order, so the last steps of phase 1 are the first of phase 3.
// The steps within `window` of the back of the deal (kL2WindowFraction of the L2 over the grid) are loaded evict_normal
// by phase 1 and evict_first by phase 3, their last use in this launch.  Every other step is loaded evict_first by
// phase 1, so that the bytes that are not reused in this launch do not push the window out of L2, and evict_normal by
// phase 3: the front of J, which it reads last, is what the next launch's phase 1 reads first.  A weights-only launch
// loads every step evict_normal, as K1 does.
constexpr double kL2WindowFraction = 0.55;

struct PolicyIO {
    uint64_t pol;
    __device__ __forceinline__ float4 load(const float4* p) const { return ld_stream_f4(p, pol); }
    __device__ __forceinline__ float load(const float* p) const { return ld_stream_f1(p, pol); }
};

template <bool LAST_USE>
struct WindowSteps {
    int64_t window;
    __device__ __forceinline__ PolicyIO operator()(int64_t d) const {
        return {(d < window) == LAST_USE ? l2_policy_evict_first() : l2_policy_evict_normal()};
    }
};

// Phase 2 of the fused launches, executed by the LAST CTA to arrive: fixed-order combine of the CTA partials, (multi-GPU) the
// k x k exchange over peer memory, the small solve, publication of w through a release store on `ready`.
template <int K>
__device__ __forceinline__ void aggregate_solve_phase(const SolveParams& sp, const P2PArgs& px, const float* vec, const float* aux,
                                                      float* w_out, double* diag_out, double* G_out, const GramWorkspace& ws,
                                                      unsigned int ready0, unsigned long long t_start) {
    __shared__ SolveSmem S;
    __shared__ double Gs[K * K];
    __shared__ unsigned long long seq_s;
    __shared__ int failed_s;
    const int tid = threadIdx.x;
    const unsigned long long t_in = global_timer_ns();
    gram_combine_partials<K>(ws.partials, Gs);
    if (tid == 0) { *ws.ticket = 0u; failed_s = 0; ws.stamps[4] = global_timer_ns(); }   // self-reset: the workspace is reusable
    if (px.world > 0) {
        XchgBuffer* own = px.peers[px.rank];
        if (tid == 0) seq_s = own->step + 1;
        __syncthreads();
        const unsigned long long seq = seq_s;
        const int par = (int)(seq & 1ull);
        if (tid < K * K) {
            const double v = Gs[tid];
            for (int r = 0; r < px.world; ++r) st_relaxed_sys_f64(&px.peers[r]->slots[par][px.rank][tid], v);   // NVLink stores
        }
        __threadfence_system();
        __syncthreads();
        if (tid < px.world) st_release_sys_u64(&px.peers[tid]->flags[par][px.rank], seq);
        if (tid == 0) own->step = seq;
        // one waiter per peer flag (round-2 first version: every summing thread polled all flags in turn, 8 dependent
        // system-scope loads at 8 ranks); the CTA barrier carries the acquired visibility over to the summing threads
        if (tid < px.world && !wait_flag_sys(&own->flags[par][tid], seq, kExchangeTimeoutNs)) failed_s = 1;
        __syncthreads();
        if (tid < K * K) {
            double g = 0.0;
            for (int r = 0; r < px.world; ++r) g += ld_relaxed_sys_f64(&own->slots[par][r][tid]);   // rank order: the same sum on every rank
            Gs[tid] = g;
        }
        __syncthreads();
    }
    if (tid == 0) ws.stamps[5] = global_timer_ns();
    if (tid < MK * MK) {
        const int i = tid / MK, j = tid % MK;
        S.G[i][j] = (i < K && j < K) ? Gs[i * K + j] : 0.0;
    }
    if (G_out && tid < K * K) G_out[tid] = Gs[tid];
    __syncthreads();
    solve_block<K>(sp, S, vec, aux, failed_s != 0, tid);
    if (tid < K) {
        w_out[tid] = S.w[tid];
        if (sp.comfort) w_out[K + tid] = S.w2[tid];
    }
    __syncthreads();
    if (tid == 0) {
        ws.stamps[0] = t_start;
        ws.stamps[1] = t_in;
        ws.stamps[2] = global_timer_ns();
        __threadfence();
        st_release_gpu_u32(ws.ready, ready0 + 1u);         // the other CTAs start their recombination pass now
    }
    solve_diagnostics(sp, S, tid);                       // nobody waits for these
    __syncthreads();
    if (tid < MOVAE_DIAG_DOUBLES && diag_out) diag_out[tid] = S.dg[tid];
}

// Prologue of the fused launches, thread 0: the ready flag's value before this launch publishes its weights, and the start
// stamp.
__device__ __forceinline__ void aggregate_prologue(const GramWorkspace& ws, unsigned int& ready0, unsigned long long& t_start) {
    if (threadIdx.x == 0) {
        ready0 = ld_acquire_gpu_u32(ws.ready);
        t_start = global_timer_ns();
    }
}

// The other CTAs' wait for the weights (thread 0 polls, the CTA follows).
__device__ __forceinline__ void aggregate_wait_ready(const unsigned int* ready, unsigned int ready0) {
    if (threadIdx.x == 0) {
        // the solving CTA is resident (cooperative launch) and its only unbounded wait -- the peers' flags -- times out by
        // itself; the bound here is a last line of defence against a hung device, not a code path
        const unsigned long long t0 = global_timer_ns();
        while (ld_acquire_gpu_u32(ready) == ready0) {
            __nanosleep(40);
            if (global_timer_ns() - t0 > 2ull * kExchangeTimeoutNs) break;
        }
    }
    __syncthreads();
}

// Epilogue of the fused launches: the last CTA to leave stamps the end of the launch (diagnostics only).
__device__ __forceinline__ void aggregate_epilogue(const GramWorkspace& ws) {
    __syncthreads();
    if (threadIdx.x == 0) {
        if (atomicAdd(ws.exit, 1u) == gridDim.x - 1) {
            ws.stamps[3] = global_timer_ns();
            *ws.exit = 0u;
        }
    }
}

template <int K, int U1, int U2, bool VEC, int MINB>
__global__ void __launch_bounds__(kAggThreads, MINB)
aggregate_kernel(AggArgs a, SolveParams sp, P2PArgs px) {
    constexpr int NACC = GramAcc<K>::N;
    const GramWorkspace ws(a.ws);
    __shared__ unsigned int ready0;
    __shared__ unsigned long long t_start;
    __shared__ double red[kGramThreads / 32][NACC];
    __shared__ int is_last;
    aggregate_prologue(ws, ready0, t_start);

    // ---- phase 1: Gramian partials ----------------------------------------------------------------------------------
    double acc64[NACC];
#pragma unroll
    for (int i = 0; i < NACC; ++i) acc64[i] = 0.0;
    gram_stream_tiles<K, U1, VEC>(a.J, a.P, a.ldJ, acc64, WindowSteps<false>{a.window_gram});
    const bool last = gram_cta_partial_and_ticket<K>(acc64, ws.partials, ws.ticket, red, &is_last);

    // ---- phase 2 (last CTA to arrive): combine, exchange, solve, publish --------------------------------------------------
    if (last) aggregate_solve_phase<K>(sp, px, a.vec, a.aux, a.w_out, a.diag_out, a.G_out, ws, ready0, t_start);
    if (a.out == nullptr) return;

    // ---- phase 3: recombine + write-back -----------------------------------------------------------------------------------
    recombine_tiles<K, U2, VEC>(
        a.J, a.P, a.ldJ, a.w_out, a.out, a.accumulate, [&] { if (!last) aggregate_wait_ready(ws.ready, ready0); },
        WindowSteps<true>{a.window_rec});
    aggregate_epilogue(ws);
}

template <int K, int U1, int U2, bool VEC, int MINB>
static int launch_aggregate(const AggArgs& a, const SolveParams& sp, const P2PArgs& px, cudaStream_t st) {
    constexpr auto kern = aggregate_kernel<K, U1, U2, VEC, MINB>;
    constexpr int W = VEC ? 4 : 1;
    static thread_local int l2_dev = -1, l2_bytes = 0;
    int dev = 0;
    MOVAE_CUDA_TRY(cudaGetDevice(&dev));
    if (l2_dev != dev) {
        MOVAE_CUDA_TRY(cudaDeviceGetAttribute(&l2_bytes, cudaDevAttrL2CacheSize, dev));
        l2_dev = dev;
    }
    const int64_t tile_items = (int64_t)kAggThreads * (U1 > U2 ? U1 : U2);
    unsigned int grid = 0;                   // every CTA must be resident: the CTAs wait for each other
    const int rc = persistent_grid<kern>(kAggThreads, (a.P / W + tile_items - 1) / tile_items, kGramMaxBlocks, &grid);
    if (rc != MOVAE_OK) return rc;
    AggArgs a_ = a;
    if (a.out != nullptr) {
        const double window = kL2WindowFraction * (double)l2_bytes / (double)grid;    // bytes per CTA
        a_.window_gram = (int64_t)(window / (double)((int64_t)K * kAggThreads * U1 * W * sizeof(float)));
        a_.window_rec = (int64_t)(window / (double)((int64_t)K * kAggThreads * U2 * W * sizeof(float)));
    } else {
        a_.window_gram = a_.window_rec = INT64_MAX;
    }
    SolveParams sp_ = sp;
    P2PArgs px_ = px;
    void* params[] = {&a_, &sp_, &px_};
    MOVAE_CUDA_TRY(cudaLaunchCooperativeKernel(reinterpret_cast<const void*>(kern), dim3(grid), dim3(kAggThreads), params, 0, st));
    return MOVAE_OK;
}

// ---- segmented Jacobian: the rows are the gradient tensors autograd produced, wherever they live -----------------------
// Replaces the flatten + `cat` of torchjd's autojac (call sites main.py:189-196) WITHOUT the copy into a flat J: segment s
// (one shared parameter tensor) has k row pointers, n[s] columns and an offset into the flat gradient buffer.  Same three
// phases as aggregate_kernel; virtual tiles of 256 x U float4 are numbered segment after segment and dealt round-robin.
struct SegArgs {
    movae_jac_segments segs;
    unsigned char* ws;
    const float* vec;
    const float* aux;
    float* out;
    int accumulate;
    float* w_out;
    double* diag_out;
    double* G_out;
};

// Row addressing of segment s (tile helpers, gram_device.cuh): its k row pointers, read from the kernel parameter.
struct SegRows {
    const float* const* rows;
    __device__ __forceinline__ const float* row(int i) const { return rows[i]; }
};

template <int K, int U, int MINB>
__global__ void __launch_bounds__(kAggThreads, MINB)
aggregate_seg_kernel(const __grid_constant__ SegArgs a, SolveParams sp, P2PArgs px) {
    constexpr int NACC = GramAcc<K>::N;
    constexpr int kTile = kAggThreads * U;                 // float4 items per tile and row
    const int tid = threadIdx.x;
    const GramWorkspace ws(a.ws);
    const int n_seg = a.segs.n_segments;

    __shared__ unsigned int ready0;
    __shared__ unsigned long long t_start;
    __shared__ double red[kGramThreads / 32][NACC];
    __shared__ int is_last;
    __shared__ int tile_start[MOVAE_MAX_SEGMENTS + 1];
    aggregate_prologue(ws, ready0, t_start);
    if (tid == 0) {
        int acc = 0;
        for (int s = 0; s < n_seg; ++s) {
            tile_start[s] = acc;
            acc += (int)(((a.segs.n[s] >> 2) + kTile - 1) / kTile);
        }
        tile_start[n_seg] = acc;
    }
    __syncthreads();
    const int n_tiles = tile_start[n_seg];
    auto segment_of = [&](int v) { int s = 0; while (v >= tile_start[s + 1]) ++s; return s; };

    // ---- phase 1: every tile is a float32 chain of its own, promoted into acc64 ----
    double acc64[NACC];
#pragma unroll
    for (int i = 0; i < NACC; ++i) acc64[i] = 0.0;
    for (int v = blockIdx.x; v < n_tiles; v += gridDim.x) {
        const int s = segment_of(v);
        float acc[NACC];
#pragma unroll
        for (int q = 0; q < NACC; ++q) acc[q] = 0.f;
        gram_tile<K, U, true>(SegRows{a.segs.rows[s]}, (int64_t)(v - tile_start[s]) * kTile, a.segs.n[s] >> 2, false, acc);
#pragma unroll
        for (int q = 0; q < NACC; ++q) acc64[q] += (double)acc[q];
    }
    // ragged tails: columns 4 * (n / 4) .. n - 1 of every segment, one thread each in CTA 0
    if (blockIdx.x == 0 && tid < 4 * n_seg) {
        const int s = tid >> 2;
        const int64_t c = (a.segs.n[s] & ~(int64_t)3) + (tid & 3);
        if (c < a.segs.n[s]) gram_column<K>(SegRows{a.segs.rows[s]}, c, acc64);
    }
    const bool last = gram_cta_partial_and_ticket<K>(acc64, ws.partials, ws.ticket, red, &is_last);

    // ---- phase 2 ----
    if (last) aggregate_solve_phase<K>(sp, px, a.vec, a.aux, a.w_out, a.diag_out, a.G_out, ws, ready0, t_start);
    if (a.out == nullptr) return;

    // ---- phase 3: the virtual tiles back to front, one register tile ----
    auto wait = [&] { if (!last) aggregate_wait_ready(ws.ready, ready0); };
    float w[K];
    bool have_w = false;
    for (int v = n_tiles - 1 - (int)blockIdx.x; v >= 0; v -= gridDim.x) {
        const int s = segment_of(v);
        const int64_t t0 = (int64_t)(v - tile_start[s]) * kTile, n_items = a.segs.n[s] >> 2;
        RecTile<K, U, true> r;
        rec_load_tile<K, U, true>(r, SegRows{a.segs.rows[s]}, t0 + tid, t0, n_items, false);
        if (!have_w) {
            rec_read_weights<K>(a.w_out, wait, w);
            have_w = true;
        }
        rec_store_tile<K, U, true>(r, w, a.out + a.segs.out_off[s], t0 + tid, t0, n_items, false, a.accumulate);
    }
    if (!have_w) rec_read_weights<K>(a.w_out, wait, w);      // a CTA without tiles still has to join the protocol
    if (blockIdx.x == 0 && tid < 4 * n_seg) {
        const int s = tid >> 2;
        const int64_t c = (a.segs.n[s] & ~(int64_t)3) + (tid & 3);
        if (c < a.segs.n[s]) rec_column<K>(SegRows{a.segs.rows[s]}, w, a.out + a.segs.out_off[s], c, a.accumulate);
    }
    aggregate_epilogue(ws);
}

template <int K, int U, int MINB>
static int launch_aggregate_seg(const SegArgs& a, const SolveParams& sp, const P2PArgs& px, cudaStream_t st) {
    constexpr auto kern = aggregate_seg_kernel<K, U, MINB>;
    int64_t n_tiles = 0;
    for (int s = 0; s < a.segs.n_segments; ++s) n_tiles += ((a.segs.n[s] >> 2) + kAggThreads * U - 1) / (kAggThreads * U);
    unsigned int grid = 0;
    const int rc = persistent_grid<kern>(kAggThreads, n_tiles, kGramMaxBlocks, &grid);
    if (rc != MOVAE_OK) return rc;
    SegArgs a_ = a;
    SolveParams sp_ = sp;
    P2PArgs px_ = px;
    void* params[] = {&a_, &sp_, &px_};
    MOVAE_CUDA_TRY(cudaLaunchCooperativeKernel(reinterpret_cast<const void*>(kern), dim3(grid), dim3(kAggThreads), params, 0, st));
    return MOVAE_OK;
}

// Validation shared by the fused entry points, in this order: the solve spec and its vectors, the entry's own arguments
// (check_args), the workspace (size, and 8-byte alignment for the float64 partials), the peer-to-peer context.
template <class CheckArgs>
static int check_fused_launch(const char* who, int k, const movae_solve_spec* spec, const float* d_vec, const float* d_aux,
                              CheckArgs check_args, const void* d_ws, size_t ws_bytes, const movae_p2p_ctx* ctx, SolveParams* sp,
                              P2PArgs* px) {
    int rc = fill_solve_params(k, spec, sp);
    if (rc == MOVAE_OK) rc = check_solve_vectors(*sp, d_vec, d_aux);
    if (rc == MOVAE_OK) rc = check_args();
    if (rc != MOVAE_OK) return rc;
    MOVAE_REQUIRE(d_ws != nullptr && ws_bytes >= movae_gram_workspace_bytes(k), MOVAE_ERR_WORKSPACE,
                  "%s: workspace too small (%zu < %zu)", who, ws_bytes, movae_gram_workspace_bytes(k));
    MOVAE_REQUIRE(reinterpret_cast<uintptr_t>(d_ws) % 8 == 0, MOVAE_ERR_WORKSPACE, "%s: workspace must be 8-byte aligned", who);
    *px = p2p_disabled();
    return ctx != nullptr ? make_p2p_args(ctx, px) : MOVAE_OK;
}

}  // namespace movae

extern "C" {

int movae_aggregate_f32(const float* d_J, int k, int64_t P, int64_t ldJ, const movae_solve_spec* spec, const float* d_vec,
                        const float* d_aux, float* d_grad, int accumulate, float* d_w, double* d_diag, double* d_G, void* d_ws,
                        size_t ws_bytes, const movae_p2p_ctx* ctx, void* stream) {
    using namespace movae;
    SolveParams sp;
    P2PArgs px;
    const int rc = check_fused_launch("aggregate", k, spec, d_vec, d_aux, [&] {
        MOVAE_REQUIRE(P >= 0 && ldJ >= P, MOVAE_ERR_INVALID, "aggregate: need 0 <= P <= ldJ (P=%lld ldJ=%lld)", (long long)P, (long long)ldJ);
        MOVAE_REQUIRE(d_w != nullptr && (d_J != nullptr || P == 0), MOVAE_ERR_INVALID, "aggregate: null pointer");
        return MOVAE_OK;
    }, d_ws, ws_bytes, ctx, &sp, &px);
    if (rc != MOVAE_OK) return rc;
    AggArgs a;
    a.J = d_J;
    a.P = P;
    a.ldJ = ldJ;
    a.ws = static_cast<unsigned char*>(d_ws);
    a.vec = d_vec;
    a.aux = d_aux;
    a.out = d_grad;
    a.accumulate = accumulate;
    a.w_out = d_w;
    a.diag_out = d_diag;
    a.G_out = d_G;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool vec = (reinterpret_cast<uintptr_t>(d_J) % 16 == 0) && (d_grad == nullptr || reinterpret_cast<uintptr_t>(d_grad) % 16 == 0) &&
                     (ldJ % 4 == 0 || k == 1);
    // registers: float64 accumulators cost 2*K(K+1)/2; small k affords deeper unroll and 2 CTAs/SM
    return dispatch_k(k, [&](auto kc) {
        constexpr int K = decltype(kc)::value;
        if (vec) {
            if constexpr (K <= 2) return launch_aggregate<K, 8, 4, true, 2>(a, sp, px, st);
            else if constexpr (K == 3) return launch_aggregate<K, 4, 4, true, 2>(a, sp, px, st);
            else if constexpr (K == 4) return launch_aggregate<K, 4, 2, true, 2>(a, sp, px, st);     // two phase-3 register tiles of U2 = 4 spill at 128 regs
            else return launch_aggregate<K, 2, 2, true, 1>(a, sp, px, st);
        } else {
            if constexpr (K <= 4) return launch_aggregate<K, 8, 8, false, 2>(a, sp, px, st);
            else return launch_aggregate<K, 4, 4, false, 1>(a, sp, px, st);
        }
    });
}

int movae_aggregate_segments_f32(const movae_jac_segments* segs, const movae_solve_spec* spec, const float* d_vec,
                                 const float* d_aux, float* d_grad, int accumulate, float* d_w, double* d_diag, double* d_G,
                                 void* d_ws, size_t ws_bytes, const movae_p2p_ctx* ctx, void* stream) {
    using namespace movae;
    MOVAE_REQUIRE(segs != nullptr, MOVAE_ERR_INVALID, "aggregate_segments: null segment table");
    const int k = segs->k;
    SolveParams sp;
    P2PArgs px;
    const int rc = check_fused_launch("aggregate_segments", k, spec, d_vec, d_aux, [&] {
        MOVAE_REQUIRE(segs->n_segments >= 1 && segs->n_segments <= MOVAE_MAX_SEGMENTS, MOVAE_ERR_UNSUPPORTED,
                      "aggregate_segments: %d segments outside 1..%d", segs->n_segments, MOVAE_MAX_SEGMENTS);
        MOVAE_REQUIRE(d_w != nullptr, MOVAE_ERR_INVALID, "aggregate_segments: null pointer");
        MOVAE_REQUIRE(d_grad == nullptr || reinterpret_cast<uintptr_t>(d_grad) % 16 == 0, MOVAE_ERR_INVALID,
                      "aggregate_segments: the gradient buffer must be 16-byte aligned");
        for (int s = 0; s < segs->n_segments; ++s) {
            MOVAE_REQUIRE(segs->n[s] >= 0 && segs->out_off[s] >= 0 && segs->out_off[s] % 4 == 0, MOVAE_ERR_INVALID,
                          "aggregate_segments: segment %d needs n >= 0 and an output offset that is a multiple of 4", s);
            for (int i = 0; i < k; ++i)
                MOVAE_REQUIRE(segs->rows[s][i] != nullptr && reinterpret_cast<uintptr_t>(segs->rows[s][i]) % 16 == 0, MOVAE_ERR_INVALID,
                              "aggregate_segments: row %d of segment %d must be a 16-byte aligned device pointer", i, s);
        }
        return MOVAE_OK;
    }, d_ws, ws_bytes, ctx, &sp, &px);
    if (rc != MOVAE_OK) return rc;
    SegArgs a;
    a.segs = *segs;
    a.ws = static_cast<unsigned char*>(d_ws);
    a.vec = d_vec;
    a.aux = d_aux;
    a.out = d_grad;
    a.accumulate = accumulate;
    a.w_out = d_w;
    a.diag_out = d_diag;
    a.G_out = d_G;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    return dispatch_k(k, [&](auto kc) {
        constexpr int K = decltype(kc)::value;
        if constexpr (K <= 3) return launch_aggregate_seg<K, 4, 2>(a, sp, px, st);
        else if constexpr (K == 4) return launch_aggregate_seg<K, 2, 2>(a, sp, px, st);
        else return launch_aggregate_seg<K, 2, 1>(a, sp, px, st);
    });
}

int movae_aggregate_timestamps(const void* d_ws, uint64_t h_stamps[6], void* stream) {
    using namespace movae;
    MOVAE_REQUIRE(d_ws != nullptr && h_stamps != nullptr, MOVAE_ERR_INVALID, "aggregate_timestamps: null pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    MOVAE_CUDA_TRY(cudaMemcpyAsync(h_stamps, static_cast<const unsigned char*>(d_ws) + GramWorkspace::kStamps, 6 * sizeof(uint64_t),
                                   cudaMemcpyDeviceToHost, st));
    MOVAE_CUDA_TRY(cudaStreamSynchronize(st));
    return MOVAE_OK;
}

}  // extern "C"
