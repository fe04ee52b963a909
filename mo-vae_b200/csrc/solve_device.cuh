// Device-side small solves (k x k Gramian -> weights), callable by ONE CTA of >= 256 threads: shared by K2
// (`solve_kernel`, solve.cu) and the solve phase of the fused aggregation kernel (aggregate.cu).
#pragma once
#include <math.h>

#include <type_traits>

#include "common.cuh"

namespace movae {

constexpr int MK = MOVAE_MAX_K;
constexpr int kSolveThreads = 256;   // 2^MK active-set candidates for the UPGrad QPs
constexpr float kEps32 = 1.1920928955078125e-07f;

enum SolveKind { SOLVE_CONST = 0, SOLVE_UPGRAD = 1, SOLVE_MGDA = 2, SOLVE_AMTL = 3, SOLVE_PCGRAD = 4, SOLVE_IMTLG = 5 };

struct SolveParams {
    int kind;
    int k;
    float value;        // CONST
    float norm_eps;     // UPGRAD
    float reg_eps;      // UPGRAD
    int upgrad_norm;    // UPGRAD: MOVAE_UPGRAD_NORM_*
    int dualproj;       // UPGRAD: 1 = torchjd DualProj (ONE QP with the whole preference vector as lower bound)
    int comfort;        // MGDA: 1 = COMFORT, the MGDA weights are blended with UPGrad's (coefficients in `aux`)
    int norm_type;      // MGDA
    float epsilon;      // MGDA
    int max_iters;      // MGDA
    int stable;         // MGDA
    float min_eig_eps;  // MGDA
    int scale_mode;     // AMTL
};

// Cyclic Jacobi eigen-decomposition of a symmetric k x k matrix held in shared memory (single
// thread; k <= 8 => a few hundred rotations at most).  On exit A's diagonal holds the eigenvalues
// (unsorted) and V's columns the eigenvectors.  Only the upper triangle of the input is trusted
// (torch.linalg.eigh(UPLO="U"), aligned_mtl.py:108): it is mirrored first.
static __device__ void jacobi_eigh(double (*A)[MK], double (*V)[MK], int k) {
    for (int i = 0; i < k; ++i)
        for (int j = 0; j < k; ++j) {
            V[i][j] = (i == j) ? 1.0 : 0.0;
            if (j < i) A[i][j] = A[j][i];
        }
    for (int sweep = 0; sweep < 60; ++sweep) {
        double off = 0.0, diag = 0.0;
        for (int i = 0; i < k; ++i) {
            diag += A[i][i] * A[i][i];
            for (int j = i + 1; j < k; ++j) off += A[i][j] * A[i][j];
        }
        if (off <= 1e-34 * diag || off == 0.0) break;
        for (int p = 0; p < k - 1; ++p)
            for (int q = p + 1; q < k; ++q) {
                const double apq = A[p][q];
                if (apq == 0.0) continue;
                const double theta = (A[q][q] - A[p][p]) / (2.0 * apq);
                const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
                for (int r = 0; r < k; ++r) {   // A <- A R
                    const double arp = A[r][p], arq = A[r][q];
                    A[r][p] = c * arp - s * arq;
                    A[r][q] = s * arp + c * arq;
                }
                for (int r = 0; r < k; ++r) {   // A <- R^T A
                    const double apr = A[p][r], aqr = A[q][r];
                    A[p][r] = c * apr - s * aqr;
                    A[q][r] = s * apr + c * aqr;
                }
                A[p][q] = 0.0;
                A[q][p] = 0.0;
                for (int r = 0; r < k; ++r) {   // V <- V R
                    const double vrp = V[r][p], vrq = V[r][q];
                    V[r][p] = c * vrp - s * vrq;
                    V[r][q] = s * vrp + c * vrq;
                }
            }
    }
}

// Parallel-ordering Jacobi executed by one warp: the k (k - 1) / 2 rotations of a sweep are scheduled as a round-robin
// tournament -- n - 1 rounds (n = k rounded up to even) of n / 2 DISJOINT pairs.  Disjoint rotations commute and their
// parameters only depend on their own 2 x 2 blocks, so a round is exactly the sequential application of its rotations,
// but its column / row / eigenvector updates run as three warp-wide steps (lane = pair * 8 + index) and the float64
// divisions and square roots of the n / 2 rotation parameters run side by side: k = 8 has 7 dependent rounds per sweep
// instead of 28 dependent rotations (70 us -> ~20 us).  Same fixed point as jacobi_eigh (eigenvalues on A's diagonal,
// eigenvectors in V's columns), rounding-level differences only.
static __device__ void jacobi_eigh_warp_rr(double (*A)[MK], double (*V)[MK], int k, int lane, double (*cs)[2], int (*pq)[2]) {
    for (int e = lane; e < MK * MK; e += 32) {
        const int i = e / MK, j = e % MK;
        if (i < k && j < k) {
            V[i][j] = (i == j) ? 1.0 : 0.0;
            if (j < i) A[i][j] = A[j][i];
        }
    }
    __syncwarp();
    const int n = (k + 1) & ~1, half = n / 2;
    const int m = lane >> 3, r = lane & 7;                       // pair slot, row / column index
    for (int sweep = 0; sweep < 60; ++sweep) {
        double off = 0.0, diag = 0.0;
        for (int i = 0; i < k; ++i) {
            diag += A[i][i] * A[i][i];
            for (int j = i + 1; j < k; ++j) off += A[i][j] * A[i][j];
        }
        if (off <= 1e-34 * diag || off == 0.0) break;            // uniform: every lane read the same values
        for (int round = 0; round < n - 1; ++round) {
            __syncwarp();
            if (lane < half) {                                   // pairing of this round + rotation parameters
                int a, b;
                if (lane == 0) { a = n - 1; b = round; }
                else { a = (round + lane) % (n - 1); b = (round - lane + (n - 1)) % (n - 1); }
                int p = a < b ? a : b, q = a < b ? b : a;
                double c = 1.0, sn = 0.0;
                if (q >= k) { p = -1; q = -1; }                  // pair with the padding index of an odd k
                else {
                    const double apq = A[p][q];
                    if (apq != 0.0) {
                        // t = tan of the rotation angle, the smaller root of t^2 + 2 theta t - 1 = 0 with
                        // theta = d / (2 apq), written without forming theta: t = 2 apq / (d + sign(d) sqrt(d^2 + 4 apq^2))
                        // -- one sqrt, one division and one rsqrt instead of two sqrt and three divisions (these float64
                        // sequences are the dependent chain that makes up most of a round)
                        const double d = A[q][q] - A[p][p], b2 = 2.0 * apq;
                        const double r = sqrt(fma(d, d, b2 * b2));
                        const double t = b2 / (d >= 0.0 ? d + r : d - r);
                        c = rsqrt(fma(t, t, 1.0));
                        sn = t * c;
                    } else { p = -1; q = -1; }
                }
                pq[lane][0] = p; pq[lane][1] = q;
                cs[lane][0] = c; cs[lane][1] = sn;
            }
            __syncwarp();
            const bool on = m < half && r < k && pq[m < half ? m : 0][0] >= 0;
            const int p = on ? pq[m][0] : 0, q = on ? pq[m][1] : 0;
            const double c = on ? cs[m][0] : 1.0, sn = on ? cs[m][1] : 0.0;
            if (on) {   // A <- A R
                const double arp = A[r][p], arq = A[r][q];
                A[r][p] = c * arp - sn * arq;
                A[r][q] = sn * arp + c * arq;
            }
            __syncwarp();
            if (on) {   // A <- R^T A
                const double apr = A[p][r], aqr = A[q][r];
                A[p][r] = c * apr - sn * aqr;
                A[q][r] = sn * apr + c * aqr;
            }
            __syncwarp();
            if (on) {   // V <- V R, and the annihilated pair set exactly to zero
                if (r == 0) { A[p][q] = 0.0; A[q][p] = 0.0; }
                const double vrp = V[r][p], vrq = V[r][q];
                V[r][p] = c * vrp - sn * vrq;
                V[r][q] = sn * vrp + c * vrq;
            }
        }
        __syncwarp();
    }
    __syncwarp();
}

// ------------------------------------------------------------------------------------------------
// UPGrad: k strictly convex QPs  min 1/2 x^T H x  s.t. x >= lo_i e_i  by exhaustive active-set
// enumeration: thread s owns the active set encoded by the bits of s; the candidate with the
// smallest KKT violation is the (unique) optimum.  All float64.  The reduced system of an active set is
// embedded in a K x K system (rows / columns of the active set replaced by identity) and solved by
// Gaussian elimination without pivoting (the free block is a principal submatrix of the SPD matrix H);
// every loop bound is a template constant, so the matrix lives in registers instead of dynamically
// indexed local memory.
// ------------------------------------------------------------------------------------------------
// All k QPs of one active set at once.  The k QPs  min 1/2 x^T H x  s.t. x >= lo_i e_i  share H, and for a given active
// set the embedded K x K system matrix is the SAME for every i -- only the right-hand side changes.  So each thread
// eliminates its matrix ONCE (keeping the multipliers in the strict lower triangle) and runs k forward / backward
// substitutions: ~(1/3 K^3 + k * 2 K^2) multiply-adds instead of k * (1/3 K^3 + 2 K^2), and the k block-wide argmin
// reductions collapse into one round.  solve_i() recomputes x for the winning set of QP i from the resident factors.
template <int KT>
struct UpgradSet {
    // L D L^T factors of the embedded matrix, LOWER triangle only, packed: entry (r, c), c <= r, at r (r + 1) / 2 + c; the
    // diagonal holds D.  36 doubles for k = 8 instead of the 64 of a full LU (which, with right-hand sides and solutions,
    // spilled to local memory: the k = 8 solve took 70 us; every index below is a compile-time constant -> registers).
    double a[KT * (KT + 1) / 2];
    double inv[KT];            // 1 / D[c]: the substitutions multiply (a float64 divide is a ~40-instruction dependent chain)
    unsigned mask;

    static __device__ __forceinline__ constexpr int at(int r, int c) { return r * (r + 1) / 2 + c; }

    __device__ void factor(const double (*H)[MK], unsigned m) {
        mask = m;
#pragma unroll
        for (int r = 0; r < KT; ++r) {
            const bool ar = (m >> r) & 1u;
#pragma unroll
            for (int c = 0; c <= r; ++c) {
                const bool ac = (m >> c) & 1u;
                a[at(r, c)] = (ar || ac) ? ((r == c) ? 1.0 : 0.0) : H[r][c];
            }
        }
#pragma unroll
        for (int c = 0; c < KT; ++c) {
            inv[c] = 1.0 / a[at(c, c)];
            double l[KT];
#pragma unroll
            for (int r = c + 1; r < KT; ++r) l[r] = a[at(r, c)] * inv[c];
#pragma unroll
            for (int r = c + 1; r < KT; ++r)
#pragma unroll
                for (int cc = c + 1; cc <= r; ++cc) a[at(r, cc)] -= l[r] * a[at(cc, c)];      // a(cc, c) is still the unscaled column
#pragma unroll
            for (int r = c + 1; r < KT; ++r) a[at(r, c)] = l[r];
        }
    }

    // rhs -> x :  L y = rhs,  z = D^-1 y,  L^T x = z
    __device__ __forceinline__ void substitute(double (&rhs)[KT], double* xs) const {
#pragma unroll
        for (int r = 1; r < KT; ++r)
#pragma unroll
            for (int c = 0; c < r; ++c) rhs[r] -= a[at(r, c)] * rhs[c];
#pragma unroll
        for (int r = KT - 1; r >= 0; --r) {
            double acc = rhs[r] * inv[r];
#pragma unroll
            for (int cc = r + 1; cc < KT; ++cc) acc -= a[at(cc, r)] * xs[cc];
            xs[r] = acc;
        }
    }

    // x for QP i (lower bound lo_i on coordinate i, 0 elsewhere); returns the KKT violation of this active set
    __device__ double solve_i(const double (*H)[MK], int i, double lo_i, double* xs) const {
        const bool i_active = (mask >> i) & 1u;
        double rhs[KT];
#pragma unroll
        for (int a = 0; a < KT; ++a) {
            const bool aa = (mask >> a) & 1u;
            rhs[a] = aa ? ((a == i) ? lo_i : 0.0) : (i_active ? -H[a][i] * lo_i : 0.0);
        }
        substitute(rhs, xs);
        double viol = 0.0;
#pragma unroll
        for (int j = 0; j < KT; ++j) {
            if ((mask >> j) & 1u) {
                double g = 0.0;
#pragma unroll
                for (int c = 0; c < KT; ++c) g += H[j][c] * xs[c];
                viol = fmax(viol, -g);                                   // multiplier must be >= 0
            } else {
                viol = fmax(viol, ((j == i) ? lo_i : 0.0) - xs[j]);      // free coordinate must stay feasible
            }
        }
        return viol;
    }

    // x for the single QP  min 1/2 x^T H x  s.t. x >= lo  (every coordinate bounded: DualProj); returns the KKT violation
    __device__ double solve_vec(const double (*H)[MK], const double* lo, double* xs) const {
        double rhs[KT];
#pragma unroll
        for (int a = 0; a < KT; ++a) {
            if ((mask >> a) & 1u) {
                rhs[a] = lo[a];
            } else {
                double acc = 0.0;
#pragma unroll
                for (int b = 0; b < KT; ++b) acc -= ((mask >> b) & 1u) ? H[a][b] * lo[b] : 0.0;
                rhs[a] = acc;
            }
        }
        substitute(rhs, xs);
        double viol = 0.0;
#pragma unroll
        for (int j = 0; j < KT; ++j) {
            if ((mask >> j) & 1u) {
                double g = 0.0;
#pragma unroll
                for (int c = 0; c < KT; ++c) g += H[j][c] * xs[c];
                viol = fmax(viol, -g);
            } else {
                viol = fmax(viol, lo[j] - xs[j]);
            }
        }
        return viol;
    }
};

// Block-wide DualProj solve for k == KT (torchjd `DualProj`, selectable at main.py:1221-1222): the projection of the
// preference vector u (default 1/k each) onto the dual cone, ONE QP  argmin_{v >= u} v^T H v  over the same 2^k sets.
template <int KT>
__device__ void dualproj_all(const double (*H)[MK], const float* __restrict__ pref, float* w, double* dg, double* red_v, int* red_i,
                             double (*xbest)[MK], double* lo, double tol, int tid) {
    constexpr unsigned n_sets = 1u << KT;
    constexpr int kWarps = kSolveThreads / 32;
    UpgradSet<KT> set;
    if (tid < KT) lo[tid] = (double)(pref ? pref[tid] : __fdiv_rn(1.0f, (float)KT));
    __syncthreads();
    const bool has = (unsigned)tid < n_sets;
    double x[KT];
    double bv = 1e300;
    if (has) {
        set.factor(H, (unsigned)tid);
        bv = set.solve_vec(H, lo, x);
    }
    int bi = tid;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov < bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    if ((tid & 31) == 0) { red_v[tid >> 5] = bv; red_i[tid >> 5] = bi; }
    __syncthreads();
    if (tid == 0) {
        for (int q = 1; q < kWarps; ++q)
            if (red_v[q] < bv || (red_v[q] == bv && red_i[q] < bi)) { bv = red_v[q]; bi = red_i[q]; }
        red_v[0] = bv;
        red_i[0] = bi;
    }
    __syncthreads();
    if (has && tid == red_i[0]) {
#pragma unroll
        for (int j = 0; j < KT; ++j) xbest[0][j] = x[j];
    }
    __syncthreads();
    if (tid < KT) w[tid] = (float)xbest[0][tid];
    if (tid == 0) {
        dg[MOVAE_DIAG_RESIDUAL] = red_v[0];
        dg[MOVAE_DIAG_STATUS] = (red_v[0] <= tol) ? 0.0 : 1.0;
    }
}

// Block-wide UPGrad solve for k == KT: writes w (float32 sums of the float32-cast projections) and the worst violation.
template <int KT>
__device__ void upgrad_all(const double (*H)[MK], const float* __restrict__ pref, float* w, double* dg, double* red_v, int* red_i,
                           double (*xbest)[MK], double* lo, double tol, int tid) {
    constexpr unsigned n_sets = 1u << KT;
    constexpr int kWarps = kSolveThreads / 32;
    UpgradSet<KT> set;
    if (tid < KT) lo[tid] = (double)(pref ? pref[tid] : __fdiv_rn(1.0f, (float)KT));
    __syncthreads();
    const bool has = (unsigned)tid < n_sets;
    if (has) set.factor(H, (unsigned)tid);
    // The loop over the QPs is deliberately NOT unrolled: fully unrolled, the k = 8 kernel was ~10,000 straight-line
    // instructions per thread executed once each and ran instruction-fetch bound (ncu: 49% of the stall samples
    // `no_instruction`); rolled, the ~250-instruction body is fetched once and replayed k times.  Per-warp argmin by
    // shuffles (ties -> lowest candidate index) inside the loop, one block-level round after it.
#pragma unroll 1
    for (int i = 0; i < KT; ++i) {
        double x[KT];
        double bv = has ? set.solve_i(H, i, lo[i], x) : 1e300;
        int bi = tid;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov < bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
        }
        if ((tid & 31) == 0) { red_v[i * kWarps + (tid >> 5)] = bv; red_i[i * kWarps + (tid >> 5)] = bi; }
    }
    __syncthreads();
    if (tid < KT) {
        double bv = red_v[tid * kWarps];
        int bi = red_i[tid * kWarps];
        for (int q = 1; q < kWarps; ++q) {
            const double ov = red_v[tid * kWarps + q];
            const int oi = red_i[tid * kWarps + q];
            if (ov < bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
        }
        red_v[tid * kWarps] = bv;
        red_i[tid * kWarps] = bi;
    }
    __syncthreads();
#pragma unroll 1
    for (int i = 0; i < KT; ++i) {
        if (tid == red_i[i * kWarps]) {
            double x[KT];
            set.solve_i(H, i, lo[i], x);
#pragma unroll
            for (int j = 0; j < KT; ++j) xbest[i][j] = x[j];
        }
    }
    __syncthreads();
    if (tid < KT) {
        // W.sum(dim=0) on the float32-cast rows (torchjd casts W back to G's dtype first), rows added in order i = 0..k-1
        float acc = 0.f;
        for (int i = 0; i < KT; ++i) acc = __fadd_rn(acc, (float)xbest[i][tid]);
        w[tid] = acc;
    }
    if (tid == 0) {
        double worst = 0.0;
        for (int i = 0; i < KT; ++i) worst = fmax(worst, red_v[i * kWarps]);
        dg[MOVAE_DIAG_RESIDUAL] = worst;
        dg[MOVAE_DIAG_STATUS] = (worst <= tol) ? 0.0 : 1.0;       // NaN / inf Gramian -> status 1 (torchjd raises ValueError)
    }
}

// The same UPGrad solve for k == KT <= 5 (<= 32 active sets) run by ONE warp with shuffles only: no shared-memory round trips,
// no CTA barriers (the block-wide version above spends most of its ~7 us at k = 3 in a dozen barriers and single-thread
// sections).  Same candidates, same winner rule (smallest violation, then lowest set index), same float32 summation order
// as upgrad_all: bit-identical weights.  Call with the 32 threads of warp 0.
template <int KT>
__device__ void upgrad_all_warp(const double (*H)[MK], const float* __restrict__ pref, float* w, double* dg, double tol, int lane) {
    static_assert(KT <= 5, "one set per lane");
    constexpr unsigned n_sets = 1u << KT;
    UpgradSet<KT> set;
    const bool has = (unsigned)lane < n_sets;
    if (has) set.factor(H, (unsigned)lane);
    float acc[KT];
#pragma unroll
    for (int j = 0; j < KT; ++j) acc[j] = 0.f;
    double worst = 0.0;
#pragma unroll 1
    for (int i = 0; i < KT; ++i) {
        const double lo_i = (double)(pref ? pref[i] : __fdiv_rn(1.0f, (float)KT));
        double x[KT];
#pragma unroll
        for (int j = 0; j < KT; ++j) x[j] = 0.0;
        double bv = has ? set.solve_i(H, i, lo_i, x) : 1e300;
        int bi = lane;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov < bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
        }
        worst = fmax(worst, bv);
        // W.sum(dim=0) on the float32-cast rows (torchjd casts W back to G's dtype first), rows added in order i = 0..k-1
#pragma unroll
        for (int j = 0; j < KT; ++j) acc[j] = __fadd_rn(acc[j], (float)__shfl_sync(0xffffffffu, x[j], bi));
    }
    if (lane == 0) {
#pragma unroll
        for (int j = 0; j < KT; ++j) w[j] = acc[j];
        dg[MOVAE_DIAG_RESIDUAL] = worst;
        dg[MOVAE_DIAG_STATUS] = (worst <= tol) ? 0.0 : 1.0;       // NaN / inf Gramian -> status 1 (torchjd raises ValueError)
    }
}

// Shared-memory state of one solve (~3 KB).
struct SolveSmem {
    double G[MK][MK];     // float64 Gramian as produced by K1 (+ exchange); rows / columns >= k are zero
    float Gf[MK][MK];     // rounded once to float32: the reference's `J @ J.T` tensor
    double H[MK][MK];     // work matrix
    double V[MK][MK];
    float w[MK];          // result
    float w2[MK];         // COMFORT: the MGDA weights (what the reference's hooks see, comfort.py:131)
    double dg[MOVAE_DIAG_DOUBLES];
    double red_v[MK * (kSolveThreads / 32)];
    int red_i[MK * (kSolveThreads / 32)];
    double xbest[MK][MK];
    double rot_cs[MK / 2][2];
    int rot_pq[MK / 2][2];
    double lo[MK];
};

// normalize / regularize in float32 like the reference does on the float32 Gramian tensor, then the k (or one) QPs.
// `norm_mode` MOVAE_UPGRAD_NORM_DRAW picks L2 / MIN_L2 from the device flag aux[0] (PNUPGrad's per-step draw).
// KT > 0: k is known at compile time (the fused kernel is instantiated per k: only that QP code is generated).
template <int KT>
__device__ __noinline__ void solve_upgrad_part(const SolveParams& p, SolveSmem& S, const float* __restrict__ pref, int norm_mode,
                                               int tid) {
    const int k = p.k;
    if (norm_mode == MOVAE_UPGRAD_NORM_TRACE) {
        // torchjd `normalize` + `regularize`, one entry per thread of the first k*k (every thread forms the trace itself: k adds)
        if (tid < MK * MK) {
            const int i = tid / MK, j = tid % MK;
            float tr = 0.f;
            for (int q = 0; q < k; ++q) tr += S.Gf[q][q];
            double h = 0.0;
            if (i < k && j < k) {
                const float gn = (tr < p.norm_eps) ? 0.f : __fdiv_rn(S.Gf[i][j], tr);
                h = (double)__fadd_rn(gn, (i == j) ? p.reg_eps : 0.f);
                S.H[i][j] = h;
            }
            double hm = fabs(h);                                   // max |H| over the two warps that hold the 64 entries
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) hm = fmax(hm, __shfl_xor_sync(0xffffffffu, hm, o));
            if ((tid & 31) == 0) S.rot_cs[1 + (tid >> 5)][0] = hm;
            if (tid == 0) S.dg[MOVAE_DIAG_TRACE] = tr;
        }
        __syncthreads();
        if (tid == 0) S.rot_cs[0][0] = 1e-9 * fmax(1.0, fmax(S.rot_cs[1][0], S.rot_cs[2][0]));   // KKT tolerance relative to the scale of H
    } else
    if (tid == 0) {
        float tr = 0.f;
        for (int i = 0; i < k; ++i) tr += S.Gf[i][i];
        S.dg[MOVAE_DIAG_TRACE] = tr;
        float sc[MK];                                      // per-row scale of the two l2-based normalisations
        bool all_zero = false;
        if (norm_mode == MOVAE_UPGRAD_NORM_MIN_L2) {
            // nupgrad.py:129-158: l2 = sqrt(clamp(diag, eps)); rows with l2 > eps are scaled to the smallest such norm
            float l2[MK], mn = __uint_as_float(0x7f800000u);
            bool any = false;
            for (int i = 0; i < k; ++i) {
                l2[i] = __fsqrt_rn(fmaxf(S.Gf[i][i], p.norm_eps));
                if (l2[i] > p.norm_eps) { any = true; mn = fminf(mn, l2[i]); }
            }
            all_zero = !any;
            for (int i = 0; i < k; ++i) sc[i] = (l2[i] > p.norm_eps) ? __fdiv_rn(mn, l2[i]) : 0.f;
        } else if (norm_mode == MOVAE_UPGRAD_NORM_L2) {
            // nupgrad.py:14-24 / pnupgrad.py `normalize`: G / (|g_i| |g_j|), norms = sqrt(clamp(diag, eps))
            for (int i = 0; i < k; ++i) sc[i] = __fsqrt_rn(fmaxf(S.Gf[i][i], p.norm_eps));
        }
        double hmax = 1.0;
        for (int i = 0; i < k; ++i)
            for (int j = 0; j < k; ++j) {
                float gn;
                if (norm_mode == MOVAE_UPGRAD_NORM_MIN_L2) gn = all_zero ? 0.f : __fmul_rn(S.Gf[i][j], __fmul_rn(sc[i], sc[j]));
                else if (norm_mode == MOVAE_UPGRAD_NORM_L2) gn = __fdiv_rn(S.Gf[i][j], __fmul_rn(sc[i], sc[j]));
                else gn = (tr < p.norm_eps) ? 0.f : __fdiv_rn(S.Gf[i][j], tr);      // torchjd `normalize`: divide by the trace
                S.H[i][j] = (double)__fadd_rn(gn, (i == j) ? p.reg_eps : 0.f);
                hmax = fmax(hmax, fabs(S.H[i][j]));
            }
        S.rot_cs[0][0] = 1e-9 * hmax;      // KKT tolerance relative to the scale of H (the bounds are <= 1)
    }
    __syncthreads();
    const double tol = S.rot_cs[0][0];
    // k <= 5: warp 0 alone (shuffles only); k >= 6: the whole CTA
    auto small = [&](auto kt) {
        constexpr int K_ = decltype(kt)::value;
        if (tid < 32) upgrad_all_warp<K_>(S.H, pref, S.w, S.dg, tol, tid);
    };
    if constexpr (KT > 0) {
        if (p.dualproj) dualproj_all<KT>(S.H, pref, S.w, S.dg, S.red_v, S.red_i, S.xbest, S.lo, tol, tid);
        else if constexpr (KT <= 5) small(std::integral_constant<int, KT>{});
        else upgrad_all<KT>(S.H, pref, S.w, S.dg, S.red_v, S.red_i, S.xbest, S.lo, tol, tid);
    } else if (p.dualproj) {
        switch (k) {
            case 1: dualproj_all<1>(S.H, pref, S.w, S.dg, S.red_v, S.red_i, S.xbest, S.lo, tol, tid); break;
            case 2: dualproj_all<2>(S.H, pref, S.w, S.dg, S.red_v, S.red_i, S.xbest, S.lo, tol, tid); break;
            case 3: dualproj_all<3>(S.H, pref, S.w, S.dg, S.red_v, S.red_i, S.xbest, S.lo, tol, tid); break;
            case 4: dualproj_all<4>(S.H, pref, S.w, S.dg, S.red_v, S.red_i, S.xbest, S.lo, tol, tid); break;
            case 5: dualproj_all<5>(S.H, pref, S.w, S.dg, S.red_v, S.red_i, S.xbest, S.lo, tol, tid); break;
            case 6: dualproj_all<6>(S.H, pref, S.w, S.dg, S.red_v, S.red_i, S.xbest, S.lo, tol, tid); break;
            case 7: dualproj_all<7>(S.H, pref, S.w, S.dg, S.red_v, S.red_i, S.xbest, S.lo, tol, tid); break;
            default: dualproj_all<8>(S.H, pref, S.w, S.dg, S.red_v, S.red_i, S.xbest, S.lo, tol, tid); break;
        }
    } else {
        switch (k) {
            case 1: small(std::integral_constant<int, 1>{}); break;
            case 2: small(std::integral_constant<int, 2>{}); break;
            case 3: small(std::integral_constant<int, 3>{}); break;
            case 4: small(std::integral_constant<int, 4>{}); break;
            case 5: small(std::integral_constant<int, 5>{}); break;
            case 6: upgrad_all<6>(S.H, pref, S.w, S.dg, S.red_v, S.red_i, S.xbest, S.lo, tol, tid); break;
            case 7: upgrad_all<7>(S.H, pref, S.w, S.dg, S.red_v, S.red_i, S.xbest, S.lo, tol, tid); break;
            default: upgrad_all<8>(S.H, pref, S.w, S.dg, S.red_v, S.red_i, S.xbest, S.lo, tol, tid); break;
        }
    }
    __syncthreads();
}

// MGDA on thread 0: normalisation (float32, IEEE ops, no contraction), optional eigen clamp, Frank-Wolfe op-for-op.
static __device__ __noinline__ void solve_mgda_part(const SolveParams& p, SolveSmem& S, const float* __restrict__ losses, int tid) {
    const int k = p.k;
    if (tid == 0) {
        float s[MK];
        float (*R)[MK] = S.Gf;
        if (p.norm_type != MOVAE_MGDA_NONE) {
            for (int i = 0; i < k; ++i) {
                const float ell = (p.norm_type == MOVAE_MGDA_L2) ? 1.f : fmaxf(losses[i], 1e-20f);
                const float nrm = (p.norm_type == MOVAE_MGDA_LOSS) ? 1.f : __fsqrt_rn(fmaxf(S.Gf[i][i], 1e-20f));
                s[i] = (p.norm_type == MOVAE_MGDA_L2) ? nrm : (p.norm_type == MOVAE_MGDA_LOSS ? ell : __fmul_rn(ell, nrm));
            }
            for (int i = 0; i < k; ++i)
                for (int j = 0; j < k; ++j) R[i][j] = __fdiv_rn(S.Gf[i][j], __fmul_rn(s[i], s[j]));
        }
        if (p.stable) {   // eigen clamp, mgda.py:287-317 (float64 Jacobi on the float32 matrix)
            for (int i = 0; i < k; ++i)
                for (int j = 0; j < k; ++j) S.H[i][j] = (double)R[i][j];
            jacobi_eigh(S.H, S.V, k);
            for (int i = 0; i < k; ++i)
                for (int j = 0; j < k; ++j) {
                    double acc = 0.0;
                    for (int c = 0; c < k; ++c) acc += S.V[i][c] * fmax(S.H[c][c], (double)p.min_eig_eps) * S.V[j][c];
                    R[i][j] = (float)acc;
                }
        }
        // --- Frank-Wolfe, op-for-op in float32 (mgda.py:244-262) ---
        float alpha[MK], Ra[MK];
        for (int i = 0; i < k; ++i) alpha[i] = __fdiv_rn(1.0f, (float)k);
        float gamma = 0.f;
        int it = 0;
        for (; it < p.max_iters; ++it) {
            int t = 0;
            for (int i = 0; i < k; ++i) {
                float acc = 0.f;
                for (int j = 0; j < k; ++j) acc = fmaf(R[i][j], alpha[j], acc);
                Ra[i] = acc;
                if (acc < Ra[t]) t = i;          // first minimal index
            }
            float a = 0.f, b = 0.f;
            for (int j = 0; j < k; ++j) {
                a = fmaf(alpha[j], R[j][t], a);
                b = fmaf(alpha[j], Ra[j], b);
            }
            const float c = R[t][t];
            if (c <= a) gamma = 1.f;
            else if (b <= a) gamma = 0.f;
            else gamma = __fdiv_rn(__fsub_rn(b, a), __fsub_rn(__fadd_rn(b, c), __fmul_rn(2.f, a)));
            bool changed = false;
            const float om = __fsub_rn(1.f, gamma);
            for (int j = 0; j < k; ++j) {
                const float nv = __fadd_rn(__fmul_rn(om, alpha[j]), __fmul_rn(gamma, (j == t) ? 1.f : 0.f));
                changed |= (nv != alpha[j]);
                alpha[j] = nv;
            }
            if (gamma < p.epsilon) { ++it; break; }
            if (!changed) { it = p.max_iters; break; }   // exact fixpoint: the reference spins to max_iters with identical state
        }
        if (p.max_iters <= 0) it = 0;
        for (int i = 0; i < k; ++i) S.w[i] = alpha[i];
        S.dg[MOVAE_DIAG_COUNT] = (double)it;
        S.dg[MOVAE_DIAG_GAMMA] = (double)gamma;
    }
    __syncthreads();
}

static __device__ __noinline__ void solve_amtl_part(const SolveParams& p, SolveSmem& S, const float* __restrict__ pref, int tid) {
    const int k = p.k;
    if (tid < MK * MK) S.H[tid / MK][tid % MK] = (double)S.Gf[tid / MK][tid % MK];
    __syncthreads();
    if (tid < 32) {
        jacobi_eigh_warp_rr(S.H, S.V, k, tid, S.rot_cs, S.rot_pq);
        // every lane ranks the eigenvalues (k <= 8 values from shared memory), then the projections run lane-parallel
        double lam[MK];
        int order[MK];
        double lmax = -1e300;
        for (int i = 0; i < k; ++i) { lam[i] = S.H[i][i]; order[i] = i; lmax = fmax(lmax, lam[i]); }
        const double tol = lmax * (double)k * (double)kEps32;     // aligned_mtl.py:109
        int rank = 0;
        for (int i = 0; i < k; ++i) rank += (lam[i] > tol) ? 1 : 0;
        for (int i = 1; i < k; ++i) {                              // insertion sort, descending
            const int oi = order[i];
            int j = i - 1;
            while (j >= 0 && lam[order[j]] < lam[oi]) { order[j + 1] = order[j]; --j; }
            order[j + 1] = oi;
        }
        if (tid == 0) S.dg[MOVAE_DIAG_RANK] = (double)rank;
        double* proj = &S.rot_cs[0][0];                            // k doubles of scratch (the rotations are done)
        if (rank == 0) {
            if (tid < k) S.w[tid] = pref ? pref[tid] : __fdiv_rn(1.0f, (float)k);       // B = I
        } else {
            double scale;
            if (p.scale_mode == MOVAE_AMTL_MIN) scale = lam[order[rank - 1]];
            else if (p.scale_mode == MOVAE_AMTL_MEDIAN) scale = lam[order[rank - 1 - (rank - 1) / 2]];   // lower middle
            else { scale = 0.0; for (int r = 0; r < rank; ++r) scale += lam[order[r]]; scale /= (double)rank; }
            __syncwarp();
            if (tid < rank) {                                      // lane r: projection on eigenvector order[r]
                const int c = order[tid];
                double pr = 0.0;
                for (int i = 0; i < k; ++i) pr += S.V[i][c] * (double)(pref ? pref[i] : __fdiv_rn(1.0f, (float)k));
                proj[tid] = pr / sqrt(lam[c]);
            }
            __syncwarp();
            if (tid < k) {                                         // lane i: component i, eigenvectors in descending order
                double o = 0.0;
                for (int r = 0; r < rank; ++r) o += S.V[tid][order[r]] * proj[r];
                S.w[tid] = (float)(sqrt(scale) * o);
            }
        }
    }
    __syncthreads();
}

// PCGrad, torchjd PCGradWeighting op for op in float32: chain i starts at c = e_i and, for j in the order of row i of the
// host-drawn permutation table `perm` (float32 [k*k]), j != i, computes ip = <G_j, c> and, when ip < 0, c_j -= ip / G_jj;
// w = the k chains summed in order i = 0..k-1.  The chains are independent: lane i of warp 0 runs chain i, its c in a
// row of shared memory (the indices come from the table).  A row that is not a permutation of 0..k-1 -> STATUS 1 and NaN
// weights (check_status() raises instead of training on a corrupted draw).
static __device__ __noinline__ void solve_pcgrad_part(const SolveParams& p, SolveSmem& S, const float* __restrict__ perm, int tid) {
    const int k = p.k;
    if (tid < 32) {
        float (*C)[MK] = reinterpret_cast<float (*)[MK]>(&S.V[0][0]);     // V is unused by this solve
        bool bad = false;
        if (tid < k) {
            const float* row = perm + tid * k;
            unsigned seen = 0u;
            for (int t = 0; t < k && !bad; ++t) {
                const float v = row[t];
                bad = !(v >= 0.f && v < (float)k) || (float)(int)v != v;
                if (!bad) seen |= 1u << (int)v;
            }
            bad = bad || seen != (1u << k) - 1u;
            for (int j = 0; j < k; ++j) C[tid][j] = (j == tid) ? 1.f : 0.f;
            for (int t = 0; t < k && !bad; ++t) {
                const int j = (int)row[t];
                if (j == tid) continue;
                float ip = 0.f;
                for (int m = 0; m < k; ++m) ip = fmaf(S.Gf[j][m], C[tid][m], ip);
                if (ip < 0.f) C[tid][j] = __fsub_rn(C[tid][j], __fdiv_rn(ip, S.Gf[j][j]));
            }
        }
        bad = __any_sync(0xffffffffu, bad);
        __syncwarp();
        if (tid < k) {
            float acc = 0.f;
            for (int i = 0; i < k; ++i) acc = __fadd_rn(acc, C[i][tid]);
            S.w[tid] = bad ? __int_as_float(0x7fc00000) : acc;
        }
        if (tid == 0 && bad) S.dg[MOVAE_DIAG_STATUS] = 1.0;
    }
    __syncthreads();
}

// IMTL-G, torchjd IMTLGWeighting: v = pinv(G) d with d = sqrt(diag G) (float32), w = v / sum(v), or 0 when |sum(v)| < 1e-12.
// The pseudo-inverse of the symmetric G comes from the float64 Jacobi eigen-decomposition of the float32-rounded Gramian:
// eigenvalues with |l| <= k eps32 max|l| are dropped (torch.linalg.pinv's default tolerance -- the singular values of a
// symmetric matrix are the |l|), v = sum over the kept c of V_c (V_c . d) / l_c.  RANK = the number of kept eigenvalues.
static __device__ __noinline__ void solve_imtlg_part(const SolveParams& p, SolveSmem& S, int tid) {
    const int k = p.k;
    if (tid < MK * MK) S.H[tid / MK][tid % MK] = (double)S.Gf[tid / MK][tid % MK];
    __syncthreads();
    if (tid < 32) {
        jacobi_eigh_warp_rr(S.H, S.V, k, tid, S.rot_cs, S.rot_pq);
        double amax = 0.0;
        for (int c = 0; c < k; ++c) amax = fmax(amax, fabs(S.H[c][c]));
        const double tol = amax * (double)k * (double)kEps32;
        double* proj = &S.rot_cs[0][0];                            // k doubles of scratch (the rotations are done)
        const bool kept = tid < k && fabs(S.H[tid][tid]) > tol;
        if (tid < k) {                                             // lane c: (V_c . d) / l_c on eigenvector c
            double pr = 0.0;
            if (kept) {
                for (int i = 0; i < k; ++i) pr += S.V[i][tid] * (double)__fsqrt_rn(S.Gf[i][i]);
                pr /= S.H[tid][tid];
            }
            proj[tid] = pr;
        }
        const unsigned rank = __popc(__ballot_sync(0xffffffffu, kept));
        __syncwarp();
        if (tid < k) {                                             // lane i: component i of v
            double o = 0.0;
            for (int c = 0; c < k; ++c) o += S.V[tid][c] * proj[c];
            S.lo[tid] = o;
        }
        __syncwarp();
        if (tid < k) {
            double s = 0.0;
            for (int i = 0; i < k; ++i) s += S.lo[i];
            S.w[tid] = (fabs(s) < 1e-12) ? 0.f : (float)(S.lo[tid] / s);
        }
        if (tid == 0) S.dg[MOVAE_DIAG_RANK] = (double)rank;
    }
    __syncthreads();
}

// The whole small solve.  Precondition: S.G holds the float64 Gramian (zero outside k x k) and every thread of the
// CTA (blockDim.x >= 2^k for the UPGrad kinds, >= 64 otherwise) calls this.  `vec`: preference vector (UPGRAD /
// DUALPROJ / AMTL, may be NULL) or losses (MGDA); `aux`: COMFORT {1 - beta, beta}, PNUPGrad {1.0 = l2 branch drawn},
// PCGrad the k x k permutation table.
// `exchange_failed`: a peer's Gramian partial never arrived -> STATUS 2 and NaN weights (nothing downstream may
// silently use a partial Gramian).  Postcondition: S.w[0..k) (COMFORT: S.w2 = the MGDA weights), S.dg.
template <int KT>
__device__ __noinline__ void solve_block(const SolveParams& p, SolveSmem& S, const float* __restrict__ vec,
                                         const float* __restrict__ aux, bool exchange_failed, int tid) {
    const int k = p.k;
    if (tid < MOVAE_DIAG_DOUBLES) S.dg[tid] = 0.0;
    if (tid < MK) { S.w[tid] = 0.f; S.w2[tid] = 0.f; }
    if (tid < MK * MK) S.Gf[tid / MK][tid % MK] = (float)S.G[tid / MK][tid % MK];
    __syncthreads();

    if (p.kind == SOLVE_CONST) {
        if (tid < k) S.w[tid] = p.value;
    } else if (p.kind == SOLVE_UPGRAD) {
        int mode = p.upgrad_norm;
        if (mode == MOVAE_UPGRAD_NORM_DRAW) mode = (aux != nullptr && aux[0] != 0.f) ? MOVAE_UPGRAD_NORM_L2 : MOVAE_UPGRAD_NORM_MIN_L2;
        solve_upgrad_part<KT>(p, S, vec, mode, tid);
    } else if (p.kind == SOLVE_MGDA) {
        solve_mgda_part(p, S, vec, tid);
        if (p.comfort) {
            // comfort.py:148-158: (1 - beta) MGDA(J) + beta UPGrad(J); the recombination is linear in the weights.  The
            // MGDA normalisation overwrote Gf: restore the float32 Gramian for UPGrad (pref_vector None, trace-normalised)
            if (tid < MK) S.w2[tid] = S.w[tid];
            if (tid < MK * MK) S.Gf[tid / MK][tid % MK] = (float)S.G[tid / MK][tid % MK];
            __syncthreads();
            solve_upgrad_part<KT>(p, S, nullptr, MOVAE_UPGRAD_NORM_TRACE, tid);
            if (tid < k) S.w[tid] = __fadd_rn(__fmul_rn(aux[0], S.w2[tid]), __fmul_rn(aux[1], S.w[tid]));
        }
    } else if (p.kind == SOLVE_AMTL) {
        solve_amtl_part(p, S, vec, tid);
    } else if (p.kind == SOLVE_PCGRAD) {
        solve_pcgrad_part(p, S, aux, tid);
    } else if (p.kind == SOLVE_IMTLG) {
        solve_imtlg_part(p, S, tid);
    }
    __syncthreads();

    if (tid == 0) {
        // non-finite weights (a NaN / inf Jacobian upstream): surfaced through STATUS so that check_status() raises
        // like torchjd does when quadprog fails, instead of passing NaN gradients on silently
        bool finite = true;
        for (int i = 0; i < k; ++i) finite = finite && (fabsf(S.w[i]) <= 3.4028234e38f);
        // a non-finite Gramian must not come out as finite weights either (Aligned-MTL would count rank 0 and answer
        // 1/k; the reference's eigh propagates NaN or raises): the solved weightings answer NaN then
        bool g_finite = true;
        for (int i = 0; i < k; ++i)
            for (int j = 0; j < k; ++j) g_finite = g_finite && (fabs(S.G[i][j]) <= 1.7976931348623157e308);
        if (!g_finite && p.kind != SOLVE_CONST) {
            finite = false;
            for (int i = 0; i < k; ++i) { S.w[i] = __int_as_float(0x7fc00000); S.w2[i] = __int_as_float(0x7fc00000); }
        }
        if (!finite && S.dg[MOVAE_DIAG_STATUS] == 0.0) S.dg[MOVAE_DIAG_STATUS] = 1.0;
        if (exchange_failed) {
            S.dg[MOVAE_DIAG_STATUS] = 2.0;
            for (int i = 0; i < k; ++i) { S.w[i] = __int_as_float(0x7fc00000); S.w2[i] = __int_as_float(0x7fc00000); }
        }
    }
    __syncthreads();
}

// Diagnostics that nobody waits for (run AFTER the weights have been published): the gradient-similarity of the hook
// main.py:94-122 from G alone, and trace(G).  Thread 0; S.w / S.w2 / S.G as solve_block left them.
__device__ __forceinline__ void solve_diagnostics(const SolveParams& p, SolveSmem& S, int tid) {
    if (tid != 0) return;
    const int k = p.k;
    // cos(J^T w, J^T 1/k) = (w^T G m) / (|J^T w| |J^T m|)   (F.cosine_similarity clamps the norm product at 1e-8);
    // COMFORT: of the MGDA weights, which is what the hook registered on its weighting sees
    const float* wh = p.comfort ? S.w2 : S.w;
    double num = 0.0, ww = 0.0, mm = 0.0;
    const double m = 1.0 / (double)k;
    for (int i = 0; i < k; ++i)
        for (int j = 0; j < k; ++j) {
            num += (double)wh[i] * S.G[i][j] * m;
            ww += (double)wh[i] * S.G[i][j] * (double)wh[j];
            mm += m * S.G[i][j] * m;
        }
    S.dg[MOVAE_DIAG_SIMILARITY] = num / fmax(sqrt(fmax(ww, 0.0)) * sqrt(fmax(mm, 0.0)), 1e-8);
    if (p.kind != SOLVE_UPGRAD && !p.comfort) {
        double tr = 0.0;
        for (int i = 0; i < k; ++i) tr += (double)(float)S.G[i][i];
        S.dg[MOVAE_DIAG_TRACE] = tr;
    }
}

}  // namespace movae
