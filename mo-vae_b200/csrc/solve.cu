// K2 `solve_small`:  k x k Gramian -> weights w[k], entirely on the device (one CTA, no host sync).
//
// Replaces, in the reference (/root/reference):
//   * UPGrad  : torchjd UPGradWeighting -> project_weights -> qpsolvers/quadprog on the HOST in
//               float64 (G.cpu().numpy(), k QP calls, back to device; main.py:1195; same pipeline
//               visible at utils/torchmoo/nupgrad.py:122-126)
//   * MGDA    : utils/torchmoo/mgda.py:221-272 -- <= 250 Frank-Wolfe iterations of ~10 tiny kernels
//               with >= 3 host syncs each (python `if c <= a`), normalisers :274-285, :319-367,
//               eigen clamp :287-317
//   * AlignedMTL: utils/torchmoo/aligned_mtl.py:97-133 -- cuSOLVER eigh on a k x k + host syncs
//   * PCGrad / IMTL-G: torchjd PCGradWeighting (a float32 loop on the CPU) / IMTLGWeighting (torch.linalg.pinv)
//   * the gradient-similarity hook main.py:94-122 (two more passes over J): here it is computed
//     from G alone, 0 extra bytes.
// Latency-bound by construction (k <= 8); excluded from GB/s, included in steps/s.
#include "solve_device.cuh"

namespace movae {

__global__ void __launch_bounds__(kSolveThreads, 1)
solve_kernel(SolveParams p, const double* __restrict__ G_in, const float* __restrict__ vec, const float* __restrict__ aux,
             float* __restrict__ w_out, double* __restrict__ diag) {
    __shared__ SolveSmem S;
    const int k = p.k;
    const int tid = threadIdx.x;
    if (tid < MK * MK) {
        const int i = tid / MK, j = tid % MK;
        S.G[i][j] = (i < k && j < k) ? G_in[i * k + j] : 0.0;
    }
    __syncthreads();
    solve_block<0>(p, S, vec, aux, false, tid);
    solve_diagnostics(p, S, tid);
    __syncthreads();
    if (tid < k) {
        w_out[tid] = S.w[tid];
        if (p.comfort) w_out[k + tid] = S.w2[tid];
    }
    if (tid < MOVAE_DIAG_DOUBLES && diag) diag[tid] = S.dg[tid];
}

int fill_solve_params(int k, const movae_solve_spec* spec, SolveParams* out) {
    MOVAE_REQUIRE(spec != nullptr, MOVAE_ERR_INVALID, "solve: null spec");
    MOVAE_REQUIRE(k >= 1, MOVAE_ERR_INVALID, "solve: k must be >= 1 (got %d)", k);
    MOVAE_REQUIRE(k <= MOVAE_MAX_K, MOVAE_ERR_UNSUPPORTED, "solve: k=%d > MOVAE_MAX_K=%d", k, MOVAE_MAX_K);
    SolveParams p{};
    p.k = k;
    switch (spec->kind) {
        case MOVAE_SOLVE_CONSTANT:
            p.kind = SOLVE_CONST;
            p.value = spec->value > 0.f ? spec->value : 1.0f / (float)k;
            break;
        case MOVAE_SOLVE_UPGRAD:
        case MOVAE_SOLVE_DUALPROJ:
            p.kind = SOLVE_UPGRAD;
            p.norm_eps = spec->norm_eps;
            p.reg_eps = spec->reg_eps;
            p.dualproj = spec->kind == MOVAE_SOLVE_DUALPROJ;
            p.upgrad_norm = p.dualproj ? MOVAE_UPGRAD_NORM_TRACE : spec->mode;
            MOVAE_REQUIRE(p.upgrad_norm >= MOVAE_UPGRAD_NORM_TRACE && p.upgrad_norm <= MOVAE_UPGRAD_NORM_DRAW, MOVAE_ERR_INVALID,
                          "upgrad: bad norm_mode %d", p.upgrad_norm);
            break;
        case MOVAE_SOLVE_MGDA:
        case MOVAE_SOLVE_COMFORT:
            p.kind = SOLVE_MGDA;
            p.comfort = spec->kind == MOVAE_SOLVE_COMFORT;
            p.norm_type = spec->mode;
            p.epsilon = spec->epsilon;
            p.max_iters = spec->max_iters;
            p.stable = spec->stable;
            p.min_eig_eps = spec->min_eigenvalue_eps;
            p.norm_eps = spec->norm_eps;
            p.reg_eps = spec->reg_eps;
            p.upgrad_norm = MOVAE_UPGRAD_NORM_TRACE;
            MOVAE_REQUIRE(p.norm_type >= MOVAE_MGDA_NONE && p.norm_type <= MOVAE_MGDA_LOSS_PLUS, MOVAE_ERR_INVALID,
                          "mgda: bad norm_type %d", p.norm_type);
            break;
        case MOVAE_SOLVE_ALIGNED_MTL:
            p.kind = SOLVE_AMTL;
            p.scale_mode = spec->mode;
            MOVAE_REQUIRE(p.scale_mode >= MOVAE_AMTL_MIN && p.scale_mode <= MOVAE_AMTL_RMSE, MOVAE_ERR_INVALID,
                          "aligned_mtl: bad scale_mode %d", p.scale_mode);
            break;
        case MOVAE_SOLVE_PCGRAD:
            p.kind = SOLVE_PCGRAD;
            break;
        case MOVAE_SOLVE_IMTLG:
            p.kind = SOLVE_IMTLG;
            break;
        default:
            set_error("solve: unknown kind %d", spec->kind);
            return MOVAE_ERR_INVALID;
    }
    *out = p;
    return MOVAE_OK;
}

int check_solve_vectors(const SolveParams& p, const float* d_vec, const float* d_aux) {
    MOVAE_REQUIRE(p.kind != SOLVE_MGDA || d_vec || p.norm_type == MOVAE_MGDA_NONE || p.norm_type == MOVAE_MGDA_L2, MOVAE_ERR_INVALID,
                  "mgda: losses must be set for norm_type 'loss'/'loss+'");
    MOVAE_REQUIRE(!p.comfort || d_aux, MOVAE_ERR_INVALID, "comfort: the blend coefficients {1 - beta, beta} must be given (d_aux)");
    MOVAE_REQUIRE(!(p.kind == SOLVE_UPGRAD && p.upgrad_norm == MOVAE_UPGRAD_NORM_DRAW) || d_aux, MOVAE_ERR_INVALID,
                  "pnupgrad: the per-step draw flag must be given (d_aux)");
    MOVAE_REQUIRE(p.kind != SOLVE_PCGRAD || d_aux, MOVAE_ERR_INVALID, "pcgrad: the k x k permutation table must be given (d_aux)");
    return MOVAE_OK;
}

static int launch_solve(const SolveParams& p, const double* G, const float* vec, const float* aux, float* w, double* diag,
                        void* stream) {
    MOVAE_REQUIRE(G && w, MOVAE_ERR_INVALID, "solve: null pointer");
    const int rc = check_solve_vectors(p, vec, aux);
    if (rc != MOVAE_OK) return rc;
    // the UPGrad QPs enumerate 2^k active sets, one per thread; every other solve runs on one or two warps (64 threads
    // load the 8 x 8 Gramian)
    const int threads = (p.kind == SOLVE_UPGRAD || p.comfort) ? kSolveThreads : 64;
    solve_kernel<<<1, threads, 0, static_cast<cudaStream_t>(stream)>>>(p, G, vec, aux, w, diag);
    MOVAE_CUDA_TRY(cudaGetLastError());
    return MOVAE_OK;
}

}  // namespace movae

extern "C" {

int movae_solve_aux(const double* d_G, int k, const movae_solve_spec* spec, const float* d_vec, const float* d_aux, float* d_w,
                    double* d_diag, void* stream) {
    movae::SolveParams p;
    const int rc = movae::fill_solve_params(k, spec, &p);
    if (rc != MOVAE_OK) return rc;
    return movae::launch_solve(p, d_G, d_vec, d_aux, d_w, d_diag, stream);
}

int movae_solve(const double* d_G, int k, const movae_solve_spec* spec, const float* d_vec, float* d_w, double* d_diag,
                void* stream) {
    return movae_solve_aux(d_G, k, spec, d_vec, nullptr, d_w, d_diag, stream);
}

static movae_solve_spec make_spec(int kind, int mode) {
    movae_solve_spec s;
    memset(&s, 0, sizeof(s));
    s.kind = kind;
    s.mode = mode;
    return s;
}

int movae_solve_constant(const double* d_G, int k, float value, float* d_w, double* d_diag, void* stream) {
    movae_solve_spec s = make_spec(MOVAE_SOLVE_CONSTANT, 0);
    s.value = value;
    return movae_solve(d_G, k, &s, nullptr, d_w, d_diag, stream);
}

int movae_solve_upgrad(const double* d_G, int k, const float* d_pref, float norm_eps, float reg_eps, float* d_w,
                       double* d_diag, void* stream) {
    return movae_solve_nupgrad(d_G, k, d_pref, norm_eps, reg_eps, MOVAE_UPGRAD_NORM_TRACE, d_w, d_diag, stream);
}

int movae_solve_nupgrad(const double* d_G, int k, const float* d_pref, float norm_eps, float reg_eps, int norm_mode, float* d_w,
                        double* d_diag, void* stream) {
    using namespace movae;
    MOVAE_REQUIRE(norm_mode >= MOVAE_UPGRAD_NORM_TRACE && norm_mode <= MOVAE_UPGRAD_NORM_L2, MOVAE_ERR_INVALID,
                  "nupgrad: bad norm_mode %d", norm_mode);
    movae_solve_spec s = make_spec(MOVAE_SOLVE_UPGRAD, norm_mode);
    s.norm_eps = norm_eps;
    s.reg_eps = reg_eps;
    return movae_solve(d_G, k, &s, d_pref, d_w, d_diag, stream);
}

int movae_solve_dualproj(const double* d_G, int k, const float* d_pref, float norm_eps, float reg_eps, float* d_w, double* d_diag,
                         void* stream) {
    movae_solve_spec s = make_spec(MOVAE_SOLVE_DUALPROJ, 0);
    s.norm_eps = norm_eps;
    s.reg_eps = reg_eps;
    return movae_solve(d_G, k, &s, d_pref, d_w, d_diag, stream);
}

int movae_solve_mgda(const double* d_G, int k, int norm_type, const float* d_losses, float epsilon, int max_iters,
                     int stable, float min_eigenvalue_eps, float* d_w, double* d_diag, void* stream) {
    movae_solve_spec s = make_spec(MOVAE_SOLVE_MGDA, norm_type);
    s.epsilon = epsilon;
    s.max_iters = max_iters;
    s.stable = stable;
    s.min_eigenvalue_eps = min_eigenvalue_eps;
    return movae_solve(d_G, k, &s, d_losses, d_w, d_diag, stream);
}

int movae_solve_aligned_mtl(const double* d_G, int k, int scale_mode, const float* d_pref, float* d_w, double* d_diag,
                            void* stream) {
    movae_solve_spec s = make_spec(MOVAE_SOLVE_ALIGNED_MTL, scale_mode);
    return movae_solve(d_G, k, &s, d_pref, d_w, d_diag, stream);
}

}  // extern "C"
