/*
 * movae_b200 -- C ABI of the B200-native (sm_100a) implementation of MO-VAE's per-step hot path:
 * multi-objective gradient aggregation (k x P Jacobian -> k x k Gramian -> small solve -> J^T w ->
 * .grad) and the VQ nearest-codebook quantizer.
 *
 * Conventions
 *   - every pointer named d_* is DEVICE memory owned by the caller (PyTorch); the library never
 *     allocates or frees device memory, all scratch is passed in as a workspace;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing synchronises
 *     (except the *_host_* entry points, which are synchronous by contract);
 *   - return value: 0 = ok, non-zero = error (MOVAE_ERR_*); movae_last_error() returns a
 *     thread-local message that always contains the word "CUDA" for device-side failures so that the
 *     reference's `except RuntimeError` filter (main.py:197-208) keeps working when the Python
 *     mirror re-raises it.
 *
 * Reference interfaces each entry point replaces are cited as /root/reference/<file>:<line>; names
 * marked [torchjd] live in the un-vendored dependency torchjd (requirements.txt:58) and are cited
 * through their call sites.
 */
#ifndef MOVAE_B200_H
#define MOVAE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MOVAE_ABI_VERSION 2
struct movae_p2p_ctx;       /* defined below ("P-sharded aggregation") */
#define MOVAE_MAX_K 8            /* objectives per Jacobian handled by the streaming kernels */
#define MOVAE_DIAG_DOUBLES 8     /* length of the d_diag side-output of every solve */

enum {
    MOVAE_OK = 0,
    MOVAE_ERR_INVALID = 1,       /* bad argument (shape, alignment, enum value) */
    MOVAE_ERR_CUDA = 2,          /* a CUDA runtime call or launch failed */
    MOVAE_ERR_UNSUPPORTED = 3,   /* valid request this build does not cover (e.g. k > MOVAE_MAX_K) */
    MOVAE_ERR_WORKSPACE = 4      /* workspace missing / too small */
};

/* d_diag[] slots written by the solve kernels (all float64) */
enum {
    MOVAE_DIAG_SIMILARITY = 0,   /* cos(J^T w, mean_rows J) from G alone; replaces main.py:94-122 */
    MOVAE_DIAG_COUNT = 1,        /* MGDA convergence_count (mgda.py:265) */
    MOVAE_DIAG_GAMMA = 2,        /* MGDA last gamma (mgda.py:266) */
    MOVAE_DIAG_RANK = 3,         /* Aligned-MTL numerical rank (aligned_mtl.py:110); IMTL-G: eigenvalues kept by the pseudo-inverse */
    MOVAE_DIAG_STATUS = 4,       /* 0 ok; 1 = QP residual above tolerance or non-finite weights (torchjd raises ValueError);
                                  * 2 = a peer's Gramian partial never arrived (the weights are NaN then) */
    MOVAE_DIAG_RESIDUAL = 5,     /* UPGrad: worst KKT violation over the k QPs */
    MOVAE_DIAG_TRACE = 6,        /* trace(G) (float32-rounded Gramian) */
    MOVAE_DIAG_RESERVED = 7
};

enum { MOVAE_MGDA_NONE = 0, MOVAE_MGDA_L2 = 1, MOVAE_MGDA_LOSS = 2, MOVAE_MGDA_LOSS_PLUS = 3 };   /* mgda.py:9 */
enum { MOVAE_AMTL_MIN = 0, MOVAE_AMTL_MEDIAN = 1, MOVAE_AMTL_RMSE = 2 };                           /* aligned_mtl.py:121-130 */
enum { MOVAE_UPGRAD_NORM_TRACE = 0,     /* [torchjd] UPGrad: G / trace(G) (zeros if trace < norm_eps) */
       MOVAE_UPGRAD_NORM_MIN_L2 = 1,    /* NUPGrad: rows rescaled to the smallest gradient norm, nupgrad.py:129-158 */
       MOVAE_UPGRAD_NORM_L2 = 2,        /* PNUPGrad's other branch: G / (|g_i| |g_j|), pnupgrad.py:127-134 with `normalize` */
       MOVAE_UPGRAD_NORM_DRAW = 3 };    /* PNUPGrad: L2 when the device flag d_aux[0] != 0 else MIN_L2 -- the host writes its per-step
                                         * draw `torch.rand(1).item() < prob` (pnupgrad.py:129) there, so a captured launch follows it */

/* ---- library ------------------------------------------------------------------------------- */
int movae_abi_version(void);
const char* movae_last_error(void);
/* sm_count / compute capability of the current device; fails (MOVAE_ERR_CUDA) without a GPU */
int movae_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---- K1: Gramian  G = J J^T ---------------------------------------------------------------- *
 * replaces [torchjd] compute_gramian (`J @ J.T`) reached through GramianWeightedAggregator
 * (aligned_mtl.py:33,39; mgda.py:6,12; nupgrad.py:6,37; call sites main.py:189-196).
 * J: float32 row-major [k, P], row stride ldJ elements.  One streaming pass (4kP bytes), float32
 * products in short register chains promoted to float64; deterministic cross-CTA combine.
 * d_G: float64 [k*k] row-major, full symmetric.  accumulate != 0 adds into d_G (column-chunked /
 * P-sharded callers), else overwrites.  Workspace must be zero-filled once before first use. */
size_t movae_gram_workspace_bytes(int k);
int movae_gram_f32(const float* d_J, int k, int64_t P, int64_t ldJ, double* d_G, int accumulate,
                   void* d_ws, size_t ws_bytes, void* stream);

/* ---- K2: small solves  G -> w -------------------------------------------------------------- *
 * One single-CTA kernel each; no host round trip.  d_G float64 [k*k] (rounded to float32 inside,
 * because the reference's Gramian is a float32 tensor); d_w float32 [k]; d_diag float64 [8].      */
/* [torchjd] Sum / Mean weightings (main.py:1198,1223-1224): w = 1 or 1/k */
int movae_solve_constant(const double* d_G, int k, float value, float* d_w, double* d_diag, void* stream);
/* [torchjd] UPGradWeighting.forward + project_weights + qpsolvers/quadprog (main.py:1195;
 * same pipeline visible at nupgrad.py:122-126): normalize by trace (zero if < norm_eps), + reg_eps I,
 * k QPs argmin_{v >= u_i e_i} v^T G v solved exactly in float64, summed.  d_pref may be NULL (= 1/k). */
int movae_solve_upgrad(const double* d_G, int k, const float* d_pref, float norm_eps, float reg_eps,
                       float* d_w, double* d_diag, void* stream);
/* NUPGrad / PNUPGrad (utils/torchmoo/nupgrad.py:122-126, pnupgrad.py:127-134; main.py:1226-1229): the UPGrad
 * pipeline with the Gramian normalised by norm_mode (MOVAE_UPGRAD_NORM_*) instead of by its trace. */
int movae_solve_nupgrad(const double* d_G, int k, const float* d_pref, float norm_eps, float reg_eps, int norm_mode, float* d_w,
                        double* d_diag, void* stream);
/* [torchjd] DualProj (selectable as `dualproj`, main.py:1221-1222): the preference vector u (NULL = 1/k each) projected onto the
 * dual cone of the rows -- ONE QP argmin_{v >= u} v^T G v on the trace-normalised, regularised Gramian. */
int movae_solve_dualproj(const double* d_G, int k, const float* d_pref, float norm_eps, float reg_eps, float* d_w, double* d_diag,
                         void* stream);
/* MGDAWeighting.forward mgda.py:221-272 (+ normalisers :274-285, :319-367, eigen clamp :287-317).
 * d_losses may be NULL only for norm_type NONE / L2. */
int movae_solve_mgda(const double* d_G, int k, int norm_type, const float* d_losses, float epsilon,
                     int max_iters, int stable, float min_eigenvalue_eps, float* d_w, double* d_diag,
                     void* stream);
/* AlignedMTLWeighting.forward aligned_mtl.py:97-133.  d_pref may be NULL (= 1/k). */
int movae_solve_aligned_mtl(const double* d_G, int k, int scale_mode, const float* d_pref, float* d_w,
                            double* d_diag, void* stream);

/* ---- K3: recombine + write-back  grad (=|+=) w @ J ----------------------------------------- *
 * replaces [torchjd] WeightedAggregator.forward (`weights @ J`) and the split/_Reshape/Accumulate
 * chain (`param.grad = g_slice.view(shape).clone()` or `+=`), call sites main.py:189-196.
 * d_w float32 [k] stays on the device (written by K2).  d_grad float32 [P]: the flat buffer the
 * parameters' .grad tensors are views of.  accumulate: 0 assign, 1 add to existing contents. */
int movae_recombine_f32(const float* d_J, int k, int64_t P, int64_t ldJ, const float* d_w, float* d_grad,
                        int accumulate, void* stream);


/* ---- generic solve dispatch (same kernels as the four entry points above) -------------------- */
enum { MOVAE_SOLVE_CONSTANT = 0, MOVAE_SOLVE_UPGRAD = 1, MOVAE_SOLVE_MGDA = 2, MOVAE_SOLVE_ALIGNED_MTL = 3, MOVAE_SOLVE_DUALPROJ = 4,
       MOVAE_SOLVE_COMFORT = 5,     /* utils/torchmoo/comfort.py:148-158: w = c0 * w_mgda + c1 * w_upgrad, {c0, c1} = d_aux = {1 - beta, beta}
                                     * as float32 in DEVICE memory (set_epoch rewrites it; a captured launch follows the schedule);
                                     * MGDA fields + norm_eps / reg_eps of the UPGrad half; d_w receives 2k values: the blend, then w_mgda */
       MOVAE_SOLVE_PCGRAD = 6,      /* [torchjd] PCGradWeighting (selectable as `pcgrad`, main.py:1196-1220), float32: chain i starts at e_i
                                     * and, for j in the order of row i of d_aux (float32 [k*k] DEVICE table, row i = a permutation of
                                     * 0..k-1 drawn on the host, REQUIRED), subtracts its projection onto g_j when <g_j, J^T c> < 0;
                                     * w = sum of the k chains.  A row that is not a permutation: STATUS 1 and NaN weights */
       MOVAE_SOLVE_IMTLG = 7 };     /* [torchjd] IMTLGWeighting (`imtlg`): v = pinv(G) sqrt(diag G), eigenvalues |l| <= k eps32 max|l|
                                     * dropped (pinv's default tolerance; d_diag[MOVAE_DIAG_RANK] = how many were kept), w = v / sum(v),
                                     * w = 0 when |sum(v)| < 1e-12 */
typedef struct movae_solve_spec {
    int32_t kind;                /* MOVAE_SOLVE_* */
    int32_t mode;                /* MGDA: norm_type; ALIGNED_MTL: scale_mode; UPGRAD: MOVAE_UPGRAD_NORM_* */
    int32_t max_iters;           /* MGDA */
    int32_t stable;              /* MGDA */
    float value;                 /* CONSTANT: the weight (<= 0 means 1/k) */
    float norm_eps;              /* UPGRAD, DUALPROJ */
    float reg_eps;               /* UPGRAD, DUALPROJ */
    float epsilon;               /* MGDA */
    float min_eigenvalue_eps;    /* MGDA */
} movae_solve_spec;
/* d_vec: pref vector (UPGRAD / DUALPROJ / ALIGNED_MTL, may be NULL) or losses (MGDA / COMFORT loss / loss+) */
int movae_solve(const double* d_G, int k, const movae_solve_spec* spec, const float* d_vec, float* d_w,
                double* d_diag, void* stream);
/* same with the device-side auxiliary vector d_aux (COMFORT {1 - beta, beta}; UPGRAD with MOVAE_UPGRAD_NORM_DRAW {flag};
 * PCGRAD the k x k permutation table) */
int movae_solve_aux(const double* d_G, int k, const movae_solve_spec* spec, const float* d_vec, const float* d_aux, float* d_w,
                    double* d_diag, void* stream);

/* ---- fused step: K1 -> (exchange) -> K2 -> K3 in ONE persistent cooperative launch ------------------------------ *
 * replaces the whole `aggregator(J)` chain at main.py:189-196 ([torchjd] compute_gramian, the weighting, `weights @ J`,
 * split / Accumulate).  Every CTA streams its span of J into Gramian partials; the last CTA to arrive combines them,
 * (ctx != NULL) exchanges the k x k float64 partial with the peers over NVLink peer memory and sums the ranks' partials in
 * rank order, solves, and publishes w through a release flag; every CTA then streams its span again (back to front: L2
 * hits) into d_grad.  d_grad == NULL: weights only (what `aggregator.weighting(J)` returns to the hooks of
 * main.py:1248-1250).  d_w float32 [k] ([2k] for COMFORT), d_diag float64 [8] (may be NULL), d_G float64 [k*k] (may be
 * NULL) receives the (rank-summed) Gramian.  d_ws: movae_gram_workspace_bytes(k), zero-filled once, one per stream.
 * No argument changes from step to step: the launch is CUDA-graph capturable, multi-GPU exchange included. */
int movae_aggregate_f32(const float* d_J, int k, int64_t P, int64_t ldJ, const movae_solve_spec* spec, const float* d_vec,
                        const float* d_aux, float* d_grad, int accumulate, float* d_w, double* d_diag, double* d_G, void* d_ws,
                        size_t ws_bytes, const struct movae_p2p_ctx* ctx, void* stream);
/* ---- the same fused step over a SEGMENTED Jacobian: no flat J is ever built ------------------------------------- *
 * replaces the flatten + `torch.cat` of [torchjd] autojac (J construction, call sites main.py:189-196; SURVEY.md 8f
 * rank 1): segment s is one shared parameter tensor, rows[s][i] points at the gradient of objective i with respect to
 * it exactly where autograd left it (n[s] contiguous float32, 16-byte aligned; an identically zero row points at any
 * zero-filled buffer), out_off[s] (multiple of 4) is the tensor's offset in the flat gradient buffer d_grad.  The
 * struct lives in HOST memory and is passed to the kernel by value.  Everything else as movae_aggregate_f32. */
#define MOVAE_MAX_SEGMENTS 32
typedef struct movae_jac_segments {
    int32_t n_segments;                                   /* 1..MOVAE_MAX_SEGMENTS */
    int32_t k;                                            /* objectives, 1..MOVAE_MAX_K */
    int64_t n[MOVAE_MAX_SEGMENTS];
    int64_t out_off[MOVAE_MAX_SEGMENTS];
    const float* rows[MOVAE_MAX_SEGMENTS][MOVAE_MAX_K];
} movae_jac_segments;
int movae_aggregate_segments_f32(const movae_jac_segments* segs, const movae_solve_spec* spec, const float* d_vec,
                                 const float* d_aux, float* d_grad, int accumulate, float* d_w, double* d_diag, double* d_G,
                                 void* d_ws, size_t ws_bytes, const struct movae_p2p_ctx* ctx, void* stream);
/* globaltimer stamps (ns) of the LAST movae_aggregate_f32 launch on this workspace: start, all partials in, weights
 * published, end, partials combined, exchange done -- how bench.py splits one launch into its two streaming passes and
 * the solve phase into its pieces.  Synchronises `stream`. */
int movae_aggregate_timestamps(const void* d_ws, uint64_t h_stamps[6], void* stream);

/* ---- host-buffer pipeline (what a caller holding HOST Jacobians uses; bench.py `e2e`) -------- *
 * Phase 1: h_J (pinned host, [k, P], row stride h_ld) is copied to d_J ([k, P], row stride d_ld,
 * d_ld % 4 == 0) in column chunks on `copy_stream` while K1 accumulates each landed chunk into d_G on
 * `compute_stream`.  Asynchronous: returns after enqueueing.  A P-sharded caller allreduces d_G
 * (k x k float64) on compute_stream between the two phases.
 * Phase 2 (after movae_solve on compute_stream): K3 per chunk on compute_stream, each finished chunk
 * of d_grad is copied to h_grad on copy_stream; SYNCHRONOUS: returns when h_grad is complete. */
int movae_host_gram_f32(const float* h_J, int k, int64_t P, int64_t h_ld, float* d_J, int64_t d_ld, double* d_G,
                        void* d_ws, size_t ws_bytes, int64_t chunk_cols, void* compute_stream, void* copy_stream);
int movae_host_recombine_f32(const float* d_J, int k, int64_t P, int64_t d_ld, const float* d_w, float* d_grad,
                             float* h_grad, int64_t chunk_cols, void* compute_stream, void* copy_stream);
/* Phase 2 WITHOUT the final synchronisation: the device-to-host copies are left in flight on `d2h_stream` (give it a
 * stream of its own) so that the NEXT step's phase 1 (host-to-device, on its copy stream, into a second set of device
 * buffers) overlaps them -- PCIe is full duplex.  The caller synchronises `d2h_stream` (or an event recorded on it)
 * before reading h_grad. */
int movae_host_recombine_async_f32(const float* d_J, int k, int64_t P, int64_t d_ld, const float* d_w, float* d_grad,
                                   float* h_grad, int64_t chunk_cols, void* compute_stream, void* d2h_stream);

/* ==== P-sharded aggregation: k x k Gramian exchange over NVLink peer memory ==================== *
 * The multi-GPU path (one process per GPU, J split by column blocks) needs ONE exchange per step: the
 * sum of the ranks' k x k float64 Gramian partials (SURVEY.md 8e; the reference has no multi-device
 * code).  Instead of a separate NCCL all_reduce launch, movae_aggregate_f32 (ctx != NULL) stores this rank's partial
 * into every peer's exchange buffer (peer-to-peer stores + a release flag), waits for all ranks' flags and sums the
 * partials in RANK ORDER, so every rank solves on bit-identical input.  Buffers are double-buffered on the parity of a
 * sequence number that lives IN the exchange buffer and is advanced by the kernel (every rank must issue the same
 * sequence of exchanging launches).  A peer that does not show up within 20 s makes d_diag[MOVAE_DIAG_STATUS] = 2 and
 * the weights NaN.  Each rank allocates its buffer with movae_p2p_alloc (cudaMalloc + zero fill), ships the 64-byte IPC
 * handle to its peers (any transport), and opens theirs with movae_p2p_open. */
#define MOVAE_MAX_WORLD 8
typedef struct movae_p2p_ctx {
    int32_t rank, world;
    void* peers[MOVAE_MAX_WORLD];   /* peers[r]: rank r's exchange buffer as addressable from THIS device (peers[rank] = own) */
} movae_p2p_ctx;
size_t movae_p2p_exchange_bytes(void);
int movae_p2p_alloc(size_t bytes, void** d_ptr, unsigned char ipc_handle[64]);
int movae_p2p_open(const unsigned char ipc_handle[64], void** d_ptr);
int movae_p2p_close(void* d_ptr);
int movae_p2p_free(void* d_ptr);
/* device-side barrier over the exchange buffers (one tiny kernel, no host involvement, graph capturable): aligns the
 * ranks' streams to within a flag round trip.  d_status (may be NULL): 1 when a peer did not arrive within 20 s. */
int movae_p2p_barrier(const movae_p2p_ctx* ctx, int* d_status, void* stream);

/* ==== VQ quantizer (replaces /root/reference/models/vq_vae.py:11-124 `VectorQuantizer`) ========= *
 * Latents are float32 NCHW [B, D, H, W] exactly as the reference module receives them (HW = H*W);
 * a code vector ("row") n = (b, h, w) is the D channel values at one spatial position, row order
 * (b, h, w) like the reference's permute(0,2,3,1).view(-1, D) (vq_vae.py:28-31).  The codebook E is
 * `embedding.weight`, float32 row-major [K, D].  Indices are int64 like torch.argmin's.
 * All VQ entry points share one workspace (movae_vq_workspace_bytes), zero-filled ONCE before first
 * use (the kernels leave it clean); do not share a workspace between concurrent streams. */
enum { MOVAE_VQ_AUTO = 0,      /* tcgen05 path when the shape allows it, else the exact path */
       MOVAE_VQ_EXACT = 1,     /* float32 reference-formula kernel for every row (any K, D) */
       MOVAE_VQ_TENSOR = 2 };  /* tcgen05 path or MOVAE_ERR_UNSUPPORTED */
/* 1 when (K, D) is served by the tcgen05/TMEM kernel (this build: K = 512, D = 64) */
int movae_vq_tensor_path_supported(int K, int D);
size_t movae_vq_workspace_bytes(int64_t n_rows, int K, int D);

/* K4: nearest-codebook indices, vq_vae.py:28-39 (permute + distance matrix + argmin; also the
 * duplicated code at :79-93 and VQVAE.get_code_indices :410-417).  Tensor path: ONE launch -- bf16x3-split
 * tcgen05 GEMM (which also adds |e|^2 and builds the sort key) with a fused top-2 argmin epilogue; rows whose two best
 * scores are closer than the split's error bound are re-evaluated exactly INSIDE the kernel (reference formula
 * fl(fl(|z|^2+|e|^2) - 2 fl(z.e)), first minimal index).  After the call the first uint32 of the workspace holds the
 * number of rows that were re-evaluated.  d_dbg_scores (tests only, may be NULL): float32 [N, K] receiving the
 * tensor path's sort keys (score + per-tile offset, column index in the 5 low mantissa bits). */
int movae_vq_argmin_f32(const float* d_z, int64_t B, int D, int64_t HW, const float* d_E, int K, int64_t* d_idx, int mode,
                        float* d_dbg_scores, void* d_ws, size_t ws_bytes, void* stream);

/* K5: vq_vae.py:43-57 + :110-124.  d_quantized [B, D, H, W] = fl(z + fl(q - z)) (the straight-through
 * value); d_losses[0] = commitment_loss, d_losses[1] = embedding_loss (= mean((q - z)^2), float64
 * accumulation); d_usage_count (may be NULL) = number of distinct codes used. */
int movae_vq_gather_f32(const float* d_z, int64_t B, int D, int64_t HW, const float* d_E, int K, const int64_t* d_idx,
                        float* d_quantized, float* d_losses, int32_t* d_usage_count, void* d_ws, size_t ws_bytes, void* stream);

/* K4 + K5: the whole `VectorQuantizer.forward` (vq_vae.py:27-64). */
int movae_vq_forward_f32(const float* d_z, int64_t B, int D, int64_t HW, const float* d_E, int K, int64_t* d_idx,
                         float* d_quantized, float* d_losses, int32_t* d_usage_count, int mode, void* d_ws, size_t ws_bytes,
                         void* stream);

/* K6: autograd backward of vq_vae.py:47-55.  d_grad_quantized [B, D, H, W] (NULL = none),
 * d_g_commit / d_g_embed device scalars (NULL = 0).  d_dz [B, D, H, W] (NULL = skip) is assigned;
 * d_dE [K, D] (NULL = skip) is ACCUMULATED into: zero it for a fresh gradient.  K = 512, D = 64 runs
 * the owner-warp kernels (no floating-point atomics, bit-reproducible) and needs a scratch buffer of
 * movae_vq_backward_workspace_bytes() (no initialisation required, 16-byte aligned); other shapes
 * use float32 atomics and need none (the query returns 0). */
size_t movae_vq_backward_workspace_bytes(int64_t n_rows, int K, int D);
int movae_vq_backward_f32(const float* d_grad_quantized, const float* d_g_commit, const float* d_g_embed, const float* d_z,
                          int64_t B, int D, int64_t HW, const float* d_E, int K, const int64_t* d_idx, float* d_dz, float* d_dE,
                          void* d_ws, size_t ws_bytes, void* stream);

/* ---- exponential-moving-average codebook (VectorQuantizerEMA) --------------------------------- *
 * Not the reference's rule: van den Oord et al. 2017 App. A.1 with the semantics of rosinality/vq-vae-2-pytorch `Quantize`.
 * From the indices d_idx of the batch (searched with the pre-update codebook):
 *     count_j = #{n : idx_n = j},  S_j = sum_{n : idx_n = j} z_n
 *     cluster_size <- decay cluster_size + (1 - decay) count,   embed_avg <- decay embed_avg + (1 - decay) S
 *     n = sum_j cluster_size_j,   E_j <- embed_avg_j / ((cluster_size_j + epsilon) / (n + K epsilon) n)
 * E [K, D] is updated IN PLACE and d_E_prev [K, D] receives E as it was before the update.  d_cluster_size float32 [K],
 * d_embed_avg float32 [K, D].  0 <= decay < 1, epsilon > 0 (else MOVAE_ERR_INVALID).  The workspace
 * (movae_vq_ema_workspace_bytes, 16-byte aligned) is zero-filled ONCE before first use; the kernels leave it clean.
 * movae_vq_ema_update_f32: the whole update.  K = 512, D = 64 (16-byte aligned E, embed_avg, E_prev): two launches,
 * the statistics from K6b's partials, bit-reproducible; other shapes sum the rows with float32 atomics.
 * The split pair, for a caller that reduces the statistics across data-parallel replicas in between:
 * movae_vq_ema_stats_f32 writes d_stats float32 [K + K*D] = count, then S (row-major [K, D]); float32 counts are exact up
 * to 2^24 rows per code (the fused update at K = 512, D = 64 counts in integers);
 * movae_vq_ema_apply_f32 applies the EMA and the normalisation from such a d_stats. */
size_t movae_vq_ema_workspace_bytes(int64_t n_rows, int K, int D);
int movae_vq_ema_update_f32(const float* d_z, int64_t B, int D, int64_t HW, const int64_t* d_idx, int K, double decay, double epsilon,
                            float* d_E, float* d_cluster_size, float* d_embed_avg, float* d_E_prev, void* d_ws, size_t ws_bytes,
                            void* stream);
int movae_vq_ema_stats_f32(const float* d_z, int64_t B, int D, int64_t HW, const int64_t* d_idx, int K, float* d_stats, void* d_ws,
                           size_t ws_bytes, void* stream);
int movae_vq_ema_apply_f32(const float* d_stats, int K, int D, double decay, double epsilon, float* d_E, float* d_cluster_size,
                           float* d_embed_avg, float* d_E_prev, void* d_ws, size_t ws_bytes, void* stream);

/* get_codebook_usage_percentage_from_indices (vq_vae.py:110-124): *d_count = |unique(idx)|. */
int movae_vq_usage(const int64_t* d_idx, int64_t n, int K, int32_t* d_count, void* d_ws, size_t ws_bytes, void* stream);

/* ---- bulk code extraction (SURVEY.md 8f rank 3) ------------------------------------------------ *
 * utils/vq_codes_lmdb.py:58-96 calls get_code_indices per batch and ships int64 indices to the host; main.py:261-330
 * concatenates every batch's indices on the host and runs torch.unique for the codebook usage.  movae_vq_pack_codes
 * narrows the int64 indices (movae_vq_argmin_f32's output) to code_bytes = 2 (K <= 32768), 4 or 8 bytes for the D2H copy
 * and ORs the batch's codes into a caller-owned bitmap of ceil(K / 32) uint32 words that persists ACROSS batches
 * (zero it once; may be NULL); movae_vq_bitmap_count writes the number of distinct codes seen so far. */
int movae_vq_pack_codes(const int64_t* d_idx, int64_t n, int K, void* d_codes, int code_bytes, uint32_t* d_bitmap, void* stream);
int movae_vq_bitmap_count(const uint32_t* d_bitmap, int K, int32_t* d_count, void* stream);

/* ==== K7: optimizer step on the flat buffers (SURVEY.md 8f rank 4) ============================== *
 * replaces `optimizer.step()` (main.py:214) for the optimizers of main.py:1169-1176 (optim.SGD / Adam /
 * AdamW / RMSprop constructed with lr, weight_decay and, SGD only, momentum) and the `clip_grad_norm_`
 * in front of it (main.py:211-212).  d_p / d_g / d_m / d_v: float32 [n] FLAT parameter, gradient,
 * first-moment (Adam exp_avg, SGD momentum buffer) and second-moment (Adam exp_avg_sq, RMSprop
 * square_avg) buffers; buffers an optimizer does not use may be NULL.  torch.optim single-tensor
 * formulas in float32 (amsgrad/maximize/nesterov/centered off, dampening 0), bias corrections in float64.
 * d_lr (may be NULL = spec->lr): float64 learning rate read from device memory (schedulers under CUDA graphs).
 * d_gnorm_sq (may be NULL): squared global gradient norm as a device double (movae_gram_f32 with k = 1
 * over the flat gradient); with spec->max_grad_norm > 0 the gradient is scaled by
 * min(1, max_grad_norm / (sqrt(*d_gnorm_sq) + 1e-6)) on the fly (d_g itself is not modified).
 * d_state: movae_optim_state_bytes() of device memory, zero-filled once: holds the step count, which
 * the kernel advances itself (no host state: the launch is CUDA-graph capturable). */
enum { MOVAE_OPT_SGD = 0, MOVAE_OPT_ADAM = 1, MOVAE_OPT_ADAMW = 2, MOVAE_OPT_RMSPROP = 3 };
typedef struct movae_optim_spec {
    int32_t kind;                /* MOVAE_OPT_* */
    int32_t hold_step;           /* != 0: do not advance the step count (another launch of the SAME step follows) */
    /* hyper-parameters as float64, like the Python floats torch.optim derives its float32 constants from
     * (1 - beta2 is formed in float64 and THEN rounded: forming it from a float32 beta2 is 1.3e-5 off) */
    double lr;
    double beta1;                /* Adam/AdamW beta1; SGD momentum */
    double beta2;                /* Adam/AdamW beta2; RMSprop alpha */
    double eps;                  /* Adam/AdamW/RMSprop */
    double weight_decay;         /* L2 (SGD, Adam, RMSprop) or decoupled (AdamW) */
    double max_grad_norm;        /* <= 0: no clipping */
} movae_optim_spec;
size_t movae_optim_state_bytes(void);
int movae_optim_step_f32(float* d_p, const float* d_g, float* d_m, float* d_v, int64_t n, const movae_optim_spec* spec,
                         const double* d_lr, const double* d_gnorm_sq, void* d_state, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MOVAE_B200_H */
