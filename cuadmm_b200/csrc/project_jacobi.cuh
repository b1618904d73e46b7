// project_jacobi.cuh — fused PSD projection of one symmetric block, svec in -> svec out.
//
// Replaces, per block, the reference chain vector_to_matrices -> cusolverDnDsyevjBatched /
// cusolverDnXsyevd -> max_dense_vector_zero -> dense_matrix_mul_diag_batch ->
// cublasDgemmStridedBatched -> matrices_to_vector  (src/solver.cu:531-647).
//
// Algorithm: shifted one-sided (Hestenes) Jacobi.  With s = ||A||_F and G = A/s + I, G is
// symmetric positive semidefinite with spectrum in [0, 2]; orthogonalising the columns of G
// by plane rotations (G <- G J) converges to G V = V (Lambda/s + I), so at convergence column j
// is g_j = sigma_j v_j, lambda_j = s (sigma_j - 1), and the eigenvectors never need to be
// accumulated:    Pi_+(A) = s * sum_{sigma_j > 1} (sigma_j - 1) / sigma_j^2 * g_j g_j^T.
// The shift removes the +lambda/-lambda ambiguity a plain one-sided Jacobi has on an indefinite
// matrix.  Only ONE n x n array lives in shared memory (n <= 168 fits the 227 KB of an SM).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace cuadmm {

// SQRT2 exactly as the reference defines it (include/cuadmm/kernels.h:173-181): the fixed point
// of the Newton iteration started at 2.0, which is 0x3FF6A09E667F3BCC = 1.414213562373095 — one ulp
// BELOW the correctly rounded sqrt(2).  SQRT2INV is 1.0/SQRT2 = 0.7071067811865476, not sqrt(0.5).
// Bit-exact svec<->smat parity with the reference needs these exact constants.
constexpr double newton_sqrt_fixed_point(double x) {
    double prev = 0.0, curr = x;
    while (curr != prev) { const double next = 0.5 * (curr + x / curr); prev = curr; curr = next; }
    return curr;
}
constexpr double kSqrt2 = newton_sqrt_fixed_point(2.0);
constexpr double kSqrt2Inv = 1.0 / kSqrt2;
static_assert(kSqrt2 == 1.414213562373095, "SQRT2 must equal the reference's Newton fixed point");
static_assert(kSqrt2Inv == 0.7071067811865476, "SQRT2INV must equal 1.0/SQRT2 of the reference");
#define CUADMM_SQRT2 (::cuadmm::kSqrt2)
#define CUADMM_SQRT2INV (::cuadmm::kSqrt2Inv)

struct BlkDesc {
    int64_t svec_off;     // first svec entry of the block
    int64_t scratch_off;  // offset into the global scratch (global-memory variant only)
    int64_t w_off;        // offset of the block's eigenvalues in the debug output
    int32_t n;            // block size
    int32_t index;        // block index in blk order
    int64_t q_off;        // offset of the block's n x n warm-start basis (shared-memory kernels only)
};

// Optional fused ADMM epilogue (src/solver.cu:652-675): with Xproj = Pi_+(Xb),
//   S   = (Xproj - X) / sig - Rd1        (dense_vector_add_dense_vector x2)
//   SmC = S - C                          (D2D copy + axpby_cusparse)
struct ProjEpilogue {
    const double* X;      // may be null => no epilogue
    const double* Rd1;
    const double* Cd;     // C as a dense svec vector
    double* S;
    double* SmC;
    const double* sig_ptr;  // device scalar sigma
};

struct ProjArgs {
    const double* Xb;
    double* Xproj;
    const BlkDesc* desc;
    int32_t nblk;           // blocks in this launch
    double threshold;       // converged when every |cos| between two columns <= threshold
    int32_t max_sweeps;
    double* eig_out;        // optional (null): eigenvalues, unsorted, at desc.w_off
    int32_t* sweeps_out;    // optional (null): sweeps used, at desc.index
    double* scratch;        // global-memory eigenvalue kernel
    const int* done_flag;   // optional device flag: kernels return at once when *done_flag != 0
    int rank_limit;         // > 0: fixed-rank projection, only the rank_limit largest eigenvalues survive the clamp
    double* Q;              // optional (null): warm-start bases, n x n column-major at desc.q_off, read AND updated
    ProjEpilogue epi;
};

// svec index -> (row r, col c) with r <= c, idx = c(c+1)/2 + r
__device__ __forceinline__ void tri_unrank(int idx, int& r, int& c) {
    int cc = (int)((sqrtf(8.0f * (float)idx + 1.0f) - 1.0f) * 0.5f);
    while ((cc + 1) * (cc + 2) / 2 <= idx) ++cc;
    while (cc * (cc + 1) / 2 > idx) --cc;
    c = cc;
    r = idx - cc * (cc + 1) / 2;
}

// round-robin (circle method) pairing: m even "players", step in [0, m-1), slot k in [0, m/2)
__device__ __forceinline__ void rr_pair(int m, int step, int k, int& a, int& b) {
    if (k == 0) { a = step; b = m - 1; return; }
    a = step + k; if (a >= m - 1) a -= (m - 1);
    b = step - k; if (b < 0) b += (m - 1);
}

template <int L>
__device__ __forceinline__ double group_sum(double v) {
#pragma unroll
    for (int o = L / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// One rotation decision from (alpha, beta, gamma) = (|gp|^2, |gq|^2, gp.gq).
// Returns true when a rotation is to be applied and fills (c, s).
__device__ __forceinline__ bool jacobi_cs(double alpha, double beta, double gamma, double& c, double& s) {
    // skip rotations below rounding level: |cos| <= 2^-53
    const double tiny2 = 1.2325951644078309e-32;  // 2^-106
    if (!(gamma * gamma > tiny2 * alpha * beta)) return false;
    double zeta = (beta - alpha) / (2.0 * gamma);
    double t = 1.0 / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
    t = zeta < 0.0 ? -t : t;
    c = rsqrt(1.0 + t * t);
    s = c * t;
    return true;
}

}  // namespace cuadmm
