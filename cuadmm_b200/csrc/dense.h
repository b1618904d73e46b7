// dense.h — dense FP64 building blocks on the device (column-major): DMMA GEMM, blocked
// Cholesky, triangular inverse.  Used by the y-solve's dense tail and the large-block projection.
#pragma once
#include "common.h"
#include "chol_host.h"

namespace cuadmm {

// C(m x n) = alpha * op(A) * op(B) + beta * C      (column-major, FP64 tensor-core mma.sync)
// shape 0: general; 1: only the 64 x 64 tiles on or below the diagonal of C are computed (symmetric updates read through
// the lower triangle); 2: op(B) is lower triangular (k x n with zeros above the diagonal): column tile n0 starts at k = n0
void dgemm(cudaStream_t st, bool transA, bool transB, int64_t m, int64_t n, int64_t k, double alpha,
           const double* A, int64_t lda, const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int shape = 0);

// in-place blocked Cholesky of the lower triangle; *d_info counts pivots <= pivot_floor[k] (treated
// as redundant directions: L_kk = +inf).
// inv_diag (n x 64, may be null) receives the inverses of the 64x64 diagonal blocks.
void potrf_lower(cudaStream_t st, int64_t n, double* A, int64_t lda, double* inv_diag, int* d_info,
                 const double* pivot_floor = nullptr);
// Linv = L^-1 for lower-triangular L (strict upper of Linv zeroed); needs inv_diag from potrf_lower
void trtri_lower(cudaStream_t st, int64_t n, const double* L, int64_t ldl, const double* inv_diag, double* Linv, int64_t ldi);

// y-solve: dense trailing block.  tail_inv = column-major L22^-1 (n_tail x n_tail), in the order of F.
void build_dense_tail(const SymCsc& Cperm, const CholFactor& F, int64_t n_lead, int64_t n_tail, DevBuf<double>& tail_inv,
                      int64_t* n_deficient = nullptr);
// flags (nt x nt row-major, nt = ceil(r / 64)): which 64 x 64 tiles of P L P^T hold a non-zero, for L column-major
// r x r on the device and ipos (device, r entries) = P's map from new to old index
void tile_occupancy(int64_t r, const double* L, const int32_t* ipos, std::vector<int>& flags);
// tiles = (I, J, dst, w) per tile: tile (I, J) of P L P^T, or of (P L P^T)^T when transpose, is copied to
// out[dst + i * w + j] (i, j < 64); entries outside the r x r matrix are written as zeros
void pack_tiles(int64_t r, const double* L, const int32_t* ipos, bool transpose, const std::vector<int64_t>& tiles, double* out);

}  // namespace cuadmm
