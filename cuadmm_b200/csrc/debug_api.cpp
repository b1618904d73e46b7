// debug_api.cpp — host-only test hooks (NOT part of include/cuadmm_b200.h): let the CPU test-suite
// exercise the init-time sparse Cholesky pipeline without a GPU.
#include "chol_host.h"
#include "common.h"
#include <algorithm>
#include <cmath>

using namespace cuadmm;

extern "C" {

// Factor P (A A^T + eps I) P^T = L L^T on the host.  Outputs: perm (m), nnz_L, and a solve of one
// right-hand side (y = M^-1 rhs) done with the host factor, so tests can check it end to end.
// n_lead_frac < 1 exercises the split factorisation: rows >= n_lead only get their leading part and
// the trailing Schur complement is factored densely on the host here.
int cuadmm_debug_chol_solve(int64_t m, int64_t ncols, const int32_t* rowptr, const int32_t* colind, const double* val,
                            double eps, double n_lead_frac, const double* rhs, double* y, int32_t* perm_out,
                            int64_t* stats /* nnz_aat, nnz_L */) {
    return guarded([&] {
        SymCsc M = form_aat(m, ncols, rowptr, colind, val, eps);
        std::vector<int32_t> perm = min_degree_order(M);
        perm = postorder_perm(M, perm);
        CholFactor F; SymCsc C;
        chol_symbolic(M, perm, F, &C);
        const int64_t n_lead = std::max<int64_t>(0, std::min<int64_t>(m, (int64_t)(n_lead_frac * (double)m)));
        chol_numeric(C, F, n_lead);
        const int64_t r = m - n_lead;
        // dense trailing block on the host: S = M22 - L21 L21^T, Cholesky
        std::vector<double> S((size_t)(r * r), 0.0);
        for (int64_t j = n_lead; j < m; ++j)
            for (int64_t p = C.p[j]; p < C.p[j + 1]; ++p) S[(C.i[p] - n_lead) + (j - n_lead) * r] = C.x[p];
        for (int64_t j = 0; j < n_lead; ++j)
            for (int64_t p = F.Lp[j] + 1; p < F.Lp[j + 1]; ++p) if (F.Li[p] >= n_lead)
                for (int64_t q = p; q < F.Lp[j + 1]; ++q)
                    S[(F.Li[q] - n_lead) + (F.Li[p] - n_lead) * r] -= F.Lx[q] * F.Lx[p];
        for (int64_t k = 0; k < r; ++k) {
            double d = S[k + k * r];
            d = (d > 1e-11) ? std::sqrt(d) : INFINITY; S[k + k * r] = d;
            for (int64_t i = k + 1; i < r; ++i) S[i + k * r] /= d;
            for (int64_t j = k + 1; j < r; ++j)
                for (int64_t i = j; i < r; ++i) S[i + j * r] -= S[i + k * r] * S[j + k * r];
        }
        // solve
        std::vector<double> z(m);
        for (int64_t k = 0; k < m; ++k) z[k] = rhs[F.perm[k]];
        for (int64_t j = 0; j < n_lead; ++j) {
            z[j] /= F.Lx[F.Lp[j]];
            for (int64_t p = F.Lp[j] + 1; p < F.Lp[j + 1]; ++p) z[F.Li[p]] -= F.Lx[p] * z[j];
        }
        for (int64_t j = 0; j < r; ++j) {
            z[n_lead + j] /= S[j + j * r];
            for (int64_t i = j + 1; i < r; ++i) z[n_lead + i] -= S[i + j * r] * z[n_lead + j];
        }
        for (int64_t j = r - 1; j >= 0; --j) {
            for (int64_t i = j + 1; i < r; ++i) z[n_lead + j] -= S[i + j * r] * z[n_lead + i];
            z[n_lead + j] /= S[j + j * r];
        }
        for (int64_t j = n_lead - 1; j >= 0; --j) {
            for (int64_t p = F.Lp[j] + 1; p < F.Lp[j + 1]; ++p) z[j] -= F.Lx[p] * z[F.Li[p]];
            z[j] /= F.Lx[F.Lp[j]];
        }
        for (int64_t k = 0; k < m; ++k) y[F.perm[k]] = z[k];
        if (perm_out) std::copy(F.perm.begin(), F.perm.end(), perm_out);
        if (stats) {
            stats[0] = M.p[m]; stats[1] = F.nnz(); stats[2] = F.n_deficient;
            // depth of the forward-solve dependency DAG, and how many rows sit in levels narrower than 8
            std::vector<int32_t> lev(m, 0);
            int32_t depth = 0;
            for (int64_t j = 0; j < m; ++j) {
                for (int64_t p = F.Lp[j] + 1; p < F.Lp[j + 1]; ++p) lev[F.Li[p]] = std::max(lev[F.Li[p]], lev[j] + 1);
                depth = std::max(depth, lev[j] + 1);
            }
            stats[3] = depth;
            std::vector<int64_t> cnt(depth + 1, 0);
            for (int64_t j = 0; j < m; ++j) cnt[lev[j]]++;
            int64_t narrow = 0;
            for (int32_t l = 0; l < depth; ++l) if (cnt[l] < 8) narrow += cnt[l];
            stats[4] = narrow;
            // supernodal depth: all columns of a fundamental supernode share one level
            std::vector<int64_t> sn = find_supernodes(F, 256);
            const int64_t nsn = (int64_t)sn.size() - 1;
            std::vector<int32_t> snof(m, 0), slev(std::max<int64_t>(nsn, 1), 0);
            for (int64_t s = 0; s < nsn; ++s) for (int64_t j = sn[s]; j < sn[s + 1]; ++j) snof[j] = (int32_t)s;
            int32_t sdepth = 0;
            for (int64_t s = 0; s < nsn; ++s) {
                for (int64_t j = sn[s]; j < sn[s + 1]; ++j)
                    for (int64_t p = F.Lp[j] + 1; p < F.Lp[j + 1]; ++p) {
                        const int32_t t = snof[F.Li[p]];
                        if (t != s) slev[t] = std::max(slev[t], slev[s] + 1);
                    }
                sdepth = std::max(sdepth, slev[s] + 1);
            }
            stats[5] = nsn; stats[6] = sdepth;
            std::vector<int64_t> scnt(sdepth + 1, 0);
            for (int64_t s = 0; s < nsn; ++s) scnt[slev[s]] += sn[s + 1] - sn[s];
            int64_t deep_rows = 0;   // rows in supernodal levels >= 48
            for (int32_t l = 48; l < sdepth; ++l) deep_rows += scnt[l];
            stats[7] = deep_rows;
        }
    });
}

// The y-solve's dense-tail relabelling, on the host: the ordering of ysolve_create (order_tail_last) and the postorder of
// the tail's elimination tree (tail_postorder).  Outputs *n_lead and, for the r = m - n_lead tail rows, parent[i] (the
// etree parent of tail row i as a tail index, -1 for a root) and pos[i] (its new index).  parent and pos hold m entries.
int cuadmm_debug_tail_order(int64_t m, int64_t ncols, const int32_t* rowptr, const int32_t* colind, const double* val,
                            double eps, int64_t* n_lead, int32_t* parent, int32_t* pos) {
    return guarded([&] {
        CUADMM_REQUIRE(rowptr && n_lead && parent && pos, "null argument");
        SymCsc M = form_aat(m, ncols, rowptr, colind, val, eps);
        CholFactor F; SymCsc C;
        *n_lead = order_tail_last(M, F, C);
        const int64_t r = m - *n_lead;
        for (int64_t i = 0; i < r; ++i) parent[i] = F.parent[*n_lead + i] >= 0 ? (int32_t)(F.parent[*n_lead + i] - *n_lead) : -1;
        const std::vector<int32_t> p = tail_postorder(F, *n_lead);
        std::copy(p.begin(), p.end(), pos);
    });
}

}  // extern "C"
