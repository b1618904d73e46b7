// chol_host.h — init-time host pieces of the AA^T y-solve: forming M = A A^T + eps I, a
// fill-reducing minimum-degree ordering, elimination tree, symbolic analysis and an up-looking
// numeric Cholesky.  Replaces what the reference gets from SuiteSparse CHOLMOD
// (cholmod_aat / cholmod_analyze / cholmod_factorize, include/cuadmm/cholesky_cpu.h:62-141),
// which is not vendored and not present here; written from the published algorithms
// (George-Liu quotient-graph minimum degree with Amestoy-Davis-Duff approximate degrees,
// Liu's elimination tree, up-looking row Cholesky).
#pragma once
#include <stdint.h>
#include <vector>

namespace cuadmm {

// symmetric sparse matrix, lower triangle (incl. diagonal) in CSC, row indices ascending
struct SymCsc {
    int64_t n = 0;
    std::vector<int64_t> p;   // n+1
    std::vector<int32_t> i;
    std::vector<double> x;
};

// M = A A^T + eps I from A in CSR (m x ncols); returns the lower triangle
SymCsc form_aat(int64_t m, int64_t ncols, const int32_t* rowptr, const int32_t* colind, const double* val, double eps);

// minimum-degree ordering of the graph of M (perm[k] = original index eliminated k-th)
std::vector<int32_t> min_degree_order(const SymCsc& M);

// Cholesky factor of P M P^T, lower triangular CSC, diagonal entry first in every column
struct CholFactor {
    int64_t n = 0;
    std::vector<int32_t> perm, iperm;   // perm[new] = old
    std::vector<int32_t> parent;        // elimination tree of the permuted matrix
    std::vector<int64_t> Lp;            // n+1
    std::vector<int32_t> Li;
    std::vector<double> Lx;
    int64_t n_deficient = 0;            // pivots treated as redundant constraints (L_kk = +inf)
    int64_t nnz() const { return Lp.empty() ? 0 : Lp[n]; }
};

// etree postorder of a fill-reducing permutation: returns perm' with the same fill whose elimination
// tree is postordered (children before parents, subtrees contiguous), so that columns with nested
// structure become adjacent and form supernodes.
std::vector<int32_t> postorder_perm(const SymCsc& M, const std::vector<int32_t>& perm);

// fundamental supernodes of a postordered factor: sn_ptr (size nsn+1) column ranges.  A column joins
// the previous one when it is its etree parent and has exactly one entry less; max_size caps the width.
std::vector<int64_t> find_supernodes(const CholFactor& F, int64_t max_size);

// symbolic (pattern + etree) only: fills everything but Lx
void chol_symbolic(const SymCsc& M, const std::vector<int32_t>& perm, CholFactor& F, SymCsc* permuted = nullptr);

// The y-solve's ordering: minimum degree, then the deep, narrow end of the forward solve's dependency DAG (at most
// CUADMM_YSOLVE_MAX_TAIL rows, default 10,240) moved last as the dense tail.  Fills the symbolic factor F of that
// order and the permuted matrix C; returns n_lead, the number of rows before the tail.
int64_t order_tail_last(const SymCsc& M, CholFactor& F, SymCsc& C);

// Postorder of the tail's elimination tree (F.parent restricted to rows >= n_lead): pos[i] = new index of tail
// row n_lead + i.  Descendants come before ancestors and every subtree is contiguous, so the structure of
// L22^-1 (entry (i, j) only when j is a descendant of i) stays lower triangular and gathers near the diagonal.
std::vector<int32_t> tail_postorder(const CholFactor& F, int64_t n_lead);
// numeric up-looking factorisation of rows [0, n_lead); for rows >= n_lead only the entries in
// columns < n_lead are computed (the trailing Schur complement is left to the caller).
// Pivots <= pivot_tol() * M_kk mark redundant constraints (see chol_host.cpp), they do not throw.
double pivot_tol();
void chol_numeric(const SymCsc& Mperm, CholFactor& F, int64_t n_lead);

}  // namespace cuadmm
