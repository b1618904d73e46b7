// chol_host.cpp — see chol_host.h.  Host-only, init-time.
#include "chol_host.h"
#include "common.h"
#include <algorithm>
#include <cmath>
#include <numeric>
#include <stdlib.h>

namespace cuadmm {

// ------------------------------------------------------------------------------------------
// M = A A^T + eps I  (lower triangle).  Row-by-row Gustavson product using the columns of A.
// ------------------------------------------------------------------------------------------
SymCsc form_aat(int64_t m, int64_t ncols, const int32_t* rowptr, const int32_t* colind, const double* val, double eps) {
    const int64_t nnz = rowptr[m];
    // CSC of A (column k -> rows that use svec entry k), rows ascending because built in row order
    std::vector<int64_t> cp(ncols + 1, 0);
    for (int64_t p = 0; p < nnz; ++p) cp[colind[p] + 1]++;
    for (int64_t k = 0; k < ncols; ++k) cp[k + 1] += cp[k];
    std::vector<int32_t> ci(nnz);
    std::vector<double> cx(nnz);
    {
        std::vector<int64_t> nx(cp.begin(), cp.end() - 1);
        for (int64_t i = 0; i < m; ++i)
            for (int p = rowptr[i]; p < rowptr[i + 1]; ++p) {
                const int64_t q = nx[colind[p]]++;
                ci[q] = (int32_t)i;
                cx[q] = val[p];
            }
    }
    SymCsc M;
    M.n = m;
    M.p.assign(m + 1, 0);
    std::vector<double> acc(m, 0.0);
    std::vector<int32_t> mark(m, -1);
    std::vector<int32_t> list;
    for (int64_t i = 0; i < m; ++i) {
        list.clear();
        mark[i] = (int32_t)i;           // diagonal always present (eps I)
        list.push_back((int32_t)i);
        acc[i] = eps;
        for (int p = rowptr[i]; p < rowptr[i + 1]; ++p) {
            const int64_t k = colind[p];
            const double aik = val[p];
            // rows j >= i of column k: binary search the first j >= i
            const int32_t* lo = std::lower_bound(ci.data() + cp[k], ci.data() + cp[k + 1], (int32_t)i);
            for (int64_t q = lo - ci.data(); q < cp[k + 1]; ++q) {
                const int32_t j = ci[q];
                if (mark[j] != (int32_t)i) { mark[j] = (int32_t)i; acc[j] = 0.0; list.push_back(j); }
                acc[j] += aik * cx[q];
            }
        }
        std::sort(list.begin(), list.end());
        for (int32_t j : list) { M.i.push_back(j); M.x.push_back(acc[j]); }
        M.p[i + 1] = (int64_t)M.i.size();
    }
    return M;
}

// ------------------------------------------------------------------------------------------
// Quotient-graph minimum degree with approximate external degrees.
// ------------------------------------------------------------------------------------------
std::vector<int32_t> min_degree_order(const SymCsc& M) {
    const int64_t n = M.n;
    std::vector<int32_t> perm(n);
    if (n == 0) return perm;
    std::vector<std::vector<int32_t>> vadj(n), eadj(n), members(n);
    {
        std::vector<int32_t> cnt(n, 0);
        for (int64_t j = 0; j < n; ++j)
            for (int64_t p = M.p[j]; p < M.p[j + 1]; ++p) if (M.i[p] != j) { cnt[j]++; cnt[M.i[p]]++; }
        for (int64_t j = 0; j < n; ++j) vadj[j].reserve(cnt[j]);
        for (int64_t j = 0; j < n; ++j)
            for (int64_t p = M.p[j]; p < M.p[j + 1]; ++p) if (M.i[p] != j) { vadj[j].push_back(M.i[p]); vadj[M.i[p]].push_back((int32_t)j); }
    }
    enum { VAR = 0, ELEM = 1, DEAD = 2 };
    std::vector<uint8_t> status(n, VAR);
    std::vector<int64_t> degree(n);
    std::vector<int32_t> head(n + 1, -1), next(n, -1), prev(n, -1);
    auto list_insert = [&](int32_t i) {
        const int64_t d = degree[i];
        next[i] = head[d]; prev[i] = -1;
        if (head[d] >= 0) prev[head[d]] = i;
        head[d] = i;
    };
    auto list_remove = [&](int32_t i) {
        const int64_t d = degree[i];
        if (prev[i] >= 0) next[prev[i]] = next[i]; else head[d] = next[i];
        if (next[i] >= 0) prev[next[i]] = prev[i];
    };
    for (int64_t i = 0; i < n; ++i) { degree[i] = (int64_t)vadj[i].size(); }
    for (int64_t i = n - 1; i >= 0; --i) list_insert((int32_t)i);   // ties: lowest index first
    std::vector<int64_t> mark(n, -1), wstamp(n, -1), w(n, 0);
    std::vector<int32_t> Lp;
    int64_t mindeg = 0;
    // Multiple elimination in rounds with a relaxed degree threshold: every round eliminates an
    // INDEPENDENT set of variables whose degree is within `slack` of the minimum.  Independent pivots
    // do not depend on each other in the triangular solves, so the depth of the solve DAG is bounded by
    // the number of rounds: on chain-like constraint graphs (moment relaxations over a time horizon)
    // this is cyclic reduction, depth O(log n), where plain minimum degree eats the chain from its
    // ends and produces depth O(n).  The GPU sweeps are latency-bound in that depth.
    std::vector<int64_t> blocked(n, -1);
    std::vector<int32_t> cands;
    int64_t k = 0, round = 0;
    auto eliminate = [&](const int32_t p) {
        list_remove(p);
        perm[k] = p;
        // ---- L_p = (A_p  U  union of L_e, e in E_p) \ {p}
        Lp.clear();
        mark[p] = k;
        for (int32_t v : vadj[p]) if (status[v] == VAR && mark[v] != k) { mark[v] = k; Lp.push_back(v); }
        for (int32_t e : eadj[p]) if (status[e] == ELEM) {
            for (int32_t v : members[e]) if (status[v] == VAR && mark[v] != k) { mark[v] = k; Lp.push_back(v); }
            status[e] = DEAD;                       // absorbed into the new element p
            std::vector<int32_t>().swap(members[e]);
        }
        status[p] = ELEM;
        std::vector<int32_t>().swap(vadj[p]);
        std::vector<int32_t>().swap(eadj[p]);
        const int64_t lp = (int64_t)Lp.size();
        // ---- pass 1: prune element lists, w[e] = |L_e \ L_p|
        for (int32_t i : Lp) {
            list_remove(i);
            auto& E = eadj[i];
            size_t o = 0;
            for (size_t t = 0; t < E.size(); ++t) {
                const int32_t e = E[t];
                if (status[e] != ELEM) continue;
                if (wstamp[e] != k) { wstamp[e] = k; w[e] = (int64_t)members[e].size(); }
                w[e] -= 1;
                E[o++] = e;
            }
            E.resize(o);
        }
        // ---- pass 2: prune variable lists, approximate degrees
        for (int32_t i : Lp) {
            auto& A = vadj[i];
            size_t o = 0;
            for (size_t t = 0; t < A.size(); ++t) {
                const int32_t v = A[t];
                if (status[v] == VAR && mark[v] != k) A[o++] = v;   // drop p, members of L_p, dead nodes
            }
            A.resize(o);
            int64_t d = (int64_t)o + (lp - 1);
            auto& E = eadj[i];
            size_t oe = 0;
            for (size_t t = 0; t < E.size(); ++t) {
                const int32_t e = E[t];
                if (status[e] != ELEM) continue;
                if (w[e] <= 0) {                     // L_e subset of L_p: aggressive absorption
                    status[e] = DEAD;
                    std::vector<int32_t>().swap(members[e]);
                    continue;
                }
                d += w[e];
                E[oe++] = e;
            }
            E.resize(oe);
            E.push_back(p);
            d = std::min<int64_t>(d, n - k - 1);
            d = std::min<int64_t>(d, degree[i] + lp - 1);
            if (d < 0) d = 0;
            degree[i] = d;
        }
        members[p] = Lp;
        for (int32_t i : Lp) {
            list_insert(i);
            blocked[i] = round;
            if (degree[i] < mindeg) mindeg = degree[i];
        }
        ++k;
    };
    const char* slack_env = getenv("CUADMM_MD_SLACK");        // relative slack in percent (default 25)
    const int64_t slack_pct = slack_env ? atoll(slack_env) : 25;
    while (k < n) {
        ++round;
        while (head[mindeg] < 0) ++mindeg;
        const int64_t limit = std::min<int64_t>(n, mindeg + std::max<int64_t>(1, mindeg * slack_pct / 100));
        cands.clear();
        for (int64_t d = mindeg; d <= limit; ++d)
            for (int32_t i = head[d]; i >= 0; i = next[i]) cands.push_back(i);
        for (int32_t p : cands) {
            if (status[p] != VAR || blocked[p] == round || degree[p] > limit) continue;
            eliminate(p);
        }
    }
    return perm;
}

// ------------------------------------------------------------------------------------------
// symbolic: permute, elimination tree (Liu, path compression), row patterns -> column structure
// ------------------------------------------------------------------------------------------
static SymCsc permute_lower(const SymCsc& M, const std::vector<int32_t>& perm, std::vector<int32_t>& iperm) {
    const int64_t n = M.n;
    iperm.assign(n, 0);
    for (int64_t k = 0; k < n; ++k) iperm[perm[k]] = (int32_t)k;
    SymCsc C;
    C.n = n;
    C.p.assign(n + 1, 0);
    const int64_t nnz = M.p[n];
    for (int64_t j = 0; j < n; ++j)
        for (int64_t p = M.p[j]; p < M.p[j + 1]; ++p) {
            const int32_t a = iperm[j], b = iperm[M.i[p]];
            C.p[std::min(a, b) + 1]++;
        }
    for (int64_t j = 0; j < n; ++j) C.p[j + 1] += C.p[j];
    C.i.resize(nnz); C.x.resize(nnz);
    std::vector<int64_t> nx(C.p.begin(), C.p.end() - 1);
    for (int64_t j = 0; j < n; ++j)
        for (int64_t p = M.p[j]; p < M.p[j + 1]; ++p) {
            const int32_t a = iperm[j], b = iperm[M.i[p]];
            const int64_t q = nx[std::min(a, b)]++;
            C.i[q] = std::max(a, b);
            C.x[q] = M.x[p];
        }
    // sort rows inside each column
    std::vector<std::pair<int32_t, double>> tmp;
    for (int64_t j = 0; j < n; ++j) {
        tmp.clear();
        for (int64_t p = C.p[j]; p < C.p[j + 1]; ++p) tmp.emplace_back(C.i[p], C.x[p]);
        std::sort(tmp.begin(), tmp.end(), [](const std::pair<int32_t, double>& a, const std::pair<int32_t, double>& b) { return a.first < b.first; });
        for (size_t t = 0; t < tmp.size(); ++t) { C.i[C.p[j] + t] = tmp[t].first; C.x[C.p[j] + t] = tmp[t].second; }
    }
    return C;
}

// rows of the lower triangle (CSR of lower == CSC of upper): for row k the columns i < k
static void lower_rows(const SymCsc& C, std::vector<int64_t>& rp, std::vector<int32_t>& rj, std::vector<double>& rx) {
    const int64_t n = C.n;
    rp.assign(n + 1, 0);
    for (int64_t j = 0; j < n; ++j)
        for (int64_t p = C.p[j]; p < C.p[j + 1]; ++p) rp[C.i[p] + 1]++;
    for (int64_t i = 0; i < n; ++i) rp[i + 1] += rp[i];
    rj.resize(rp[n]); rx.resize(rp[n]);
    std::vector<int64_t> nx(rp.begin(), rp.end() - 1);
    for (int64_t j = 0; j < n; ++j)
        for (int64_t p = C.p[j]; p < C.p[j + 1]; ++p) {
            const int64_t q = nx[C.i[p]]++;
            rj[q] = (int32_t)j;
            rx[q] = C.x[p];
        }
}

void chol_symbolic(const SymCsc& M, const std::vector<int32_t>& perm, CholFactor& F, SymCsc* permuted) {
    const int64_t n = M.n;
    F.n = n;
    F.perm = perm;
    SymCsc C = permute_lower(M, perm, F.iperm);
    std::vector<int64_t> rp; std::vector<int32_t> rj; std::vector<double> rx;
    lower_rows(C, rp, rj, rx);
    // elimination tree
    F.parent.assign(n, -1);
    std::vector<int32_t> ancestor(n, -1);
    for (int64_t k = 0; k < n; ++k) {
        for (int64_t p = rp[k]; p < rp[k + 1]; ++p) {
            int32_t i = rj[p];
            while (i != -1 && i < k) {
                const int32_t inext = ancestor[i];
                ancestor[i] = (int32_t)k;
                if (inext == -1) F.parent[i] = (int32_t)k;
                i = inext;
            }
        }
    }
    // row patterns by etree reach; count, then fill
    std::vector<int64_t> cnt(n, 1);     // diagonal
    std::vector<int32_t> flag(n, -1);
    for (int pass = 0; pass < 2; ++pass) {
        std::vector<int64_t> nx;
        if (pass == 1) {
            F.Lp.assign(n + 1, 0);
            for (int64_t j = 0; j < n; ++j) F.Lp[j + 1] = F.Lp[j] + cnt[j];
            F.Li.assign(F.Lp[n], 0);
            F.Lx.assign(F.Lp[n], 0.0);
            nx.assign(F.Lp.begin(), F.Lp.end() - 1);
            for (int64_t j = 0; j < n; ++j) F.Li[nx[j]++] = (int32_t)j;
            std::fill(flag.begin(), flag.end(), -1);
        }
        for (int64_t k = 0; k < n; ++k) {
            flag[k] = (int32_t)k;
            for (int64_t p = rp[k]; p < rp[k + 1]; ++p) {
                int32_t i = rj[p];
                while (i != -1 && i < k && flag[i] != (int32_t)k) {
                    flag[i] = (int32_t)k;
                    if (pass == 0) cnt[i]++; else F.Li[nx[i]++] = (int32_t)k;
                    i = F.parent[i];
                }
            }
        }
    }
    if (permuted) *permuted = std::move(C);
}

// post[k] = the k-th node of a postorder of the forest `parent` (-1 = root): roots and children in ascending order
static std::vector<int32_t> forest_postorder(const std::vector<int32_t>& parent) {
    const int64_t n = (int64_t)parent.size();
    // children lists (ascending), iterative DFS
    std::vector<int32_t> head(n, -1), nxt(n, -1);
    for (int64_t j = n - 1; j >= 0; --j) if (parent[j] >= 0) { nxt[j] = head[parent[j]]; head[parent[j]] = (int32_t)j; }
    std::vector<int32_t> post; post.reserve(n);
    std::vector<int32_t> stack;
    for (int64_t r = 0; r < n; ++r) {
        if (parent[r] >= 0) continue;
        stack.push_back((int32_t)r);
        while (!stack.empty()) {
            const int32_t v = stack.back();
            const int32_t c = head[v];
            if (c >= 0) { head[v] = nxt[c]; stack.push_back(c); }
            else { post.push_back(v); stack.pop_back(); }
        }
    }
    return post;
}

std::vector<int32_t> postorder_perm(const SymCsc& M, const std::vector<int32_t>& perm) {
    CholFactor F;
    chol_symbolic(M, perm, F, nullptr);
    const std::vector<int32_t> post = forest_postorder(F.parent);
    std::vector<int32_t> out(F.n);
    for (int64_t k = 0; k < F.n; ++k) out[k] = perm[post[k]];
    return out;
}

// the rows that go to the dense tail: the deep, narrow end of the forward solve's dependency DAG.  Returns the
// first level of the tail (> depth: no tail) and every row's level.
static int64_t choose_tail(const CholFactor& F, std::vector<int32_t>& level_out) {
    const int64_t n = F.n;
    std::vector<int32_t> lev(n, 0);
    for (int64_t j = 0; j < n; ++j)
        for (int64_t p = F.Lp[j] + 1; p < F.Lp[j + 1]; ++p) lev[F.Li[p]] = std::max(lev[F.Li[p]], lev[j] + 1);
    level_out = lev;
    int depth = 0;
    for (int64_t i = 0; i < n; ++i) depth = std::max(depth, lev[i] + 1);
    int64_t max_tail = 10240;
    int min_depth = 64;
    if (const char* e = getenv("CUADMM_YSOLVE_MAX_TAIL")) max_tail = atoll(e);
    if (const char* e = getenv("CUADMM_YSOLVE_MIN_DEPTH")) min_depth = atoi(e);
    if (depth <= min_depth || max_tail <= 0) return depth + 1;       // no tail
    std::vector<int64_t> cnt(depth + 1, 0);
    for (int64_t i = 0; i < n; ++i) cnt[lev[i]]++;
    // smallest cut >= min_depth/2 with count(level >= cut) <= max_tail
    int64_t above = 0;
    int cut = depth;
    for (int l = depth - 1; l >= min_depth / 2; --l) {
        if (above + cnt[l] > max_tail) break;
        above += cnt[l];
        cut = l;
    }
    if (above < 32) return depth + 1;   // a tiny tail is not worth a dense stage
    return cut;
}

int64_t order_tail_last(const SymCsc& M, CholFactor& F, SymCsc& C) {
    const int64_t m = M.n;
    std::vector<int32_t> perm0 = min_degree_order(M);
    F = CholFactor();
    chol_symbolic(M, perm0, F, nullptr);
    std::vector<int32_t> lev;
    const int64_t cut = choose_tail(F, lev);
    std::vector<int32_t> perm1; perm1.reserve(m);
    for (int64_t k = 0; k < m; ++k) if (lev[k] < cut) perm1.push_back(F.perm[k]);
    const int64_t n_lead = (int64_t)perm1.size();
    for (int64_t k = 0; k < m; ++k) if (lev[k] >= cut) perm1.push_back(F.perm[k]);
    if (n_lead < m) {
        F = CholFactor();
        chol_symbolic(M, perm1, F, &C);
    } else {
        chol_symbolic(M, perm0, F, &C);
    }
    return n_lead;
}

std::vector<int32_t> tail_postorder(const CholFactor& F, int64_t n_lead) {
    const int64_t r = F.n - n_lead;
    std::vector<int32_t> parent(r);
    for (int64_t i = 0; i < r; ++i) parent[i] = F.parent[n_lead + i] >= 0 ? (int32_t)(F.parent[n_lead + i] - n_lead) : -1;
    const std::vector<int32_t> post = forest_postorder(parent);
    std::vector<int32_t> pos(r);
    for (int64_t k = 0; k < r; ++k) pos[post[k]] = (int32_t)k;
    return pos;
}

std::vector<int64_t> find_supernodes(const CholFactor& F, int64_t max_size) {
    const int64_t n = F.n;
    std::vector<int64_t> sn;
    sn.push_back(0);
    std::vector<int32_t> nchild(n, 0);
    for (int64_t j = 0; j < n; ++j) if (F.parent[j] >= 0) nchild[F.parent[j]]++;
    for (int64_t j = 1; j < n; ++j) {
        const int64_t cprev = F.Lp[j] - F.Lp[j - 1], ccur = F.Lp[j + 1] - F.Lp[j];
        const bool join = F.parent[j - 1] == j && ccur == cprev - 1 && nchild[j] == 1 && (j - sn.back()) < max_size;
        if (!join) sn.push_back(j);
    }
    if (n > 0) sn.push_back(n);
    return sn;
}

// ------------------------------------------------------------------------------------------
// numeric up-looking Cholesky on the symbolic structure
// ------------------------------------------------------------------------------------------
// Relative pivot tolerance: a pivot d_k <= tol * M_kk marks constraint k as redundant (see below).  The default keeps
// every pivot that stands clear of the rounding noise of the factorisation (the reference keeps them all: CHOLMOD
// LDL^T of A A^T + 1e-15 I); CUADMM_PIVOT_TOL overrides it.
double pivot_tol() {
    if (const char* e = getenv("CUADMM_PIVOT_TOL")) { const double v = atof(e); if (v > 0.0 && v < 1.0) return v; }
    return 1e-11;
}

void chol_numeric(const SymCsc& C, CholFactor& F, int64_t n_lead) {
    F.n_deficient = 0;
    const double kPivotTol = pivot_tol();
    const int64_t n = F.n;
    std::vector<int64_t> rp; std::vector<int32_t> rj; std::vector<double> rx;
    lower_rows(C, rp, rj, rx);
    std::vector<double> x(n, 0.0);
    std::vector<int64_t> c(n);
    for (int64_t j = 0; j < n; ++j) c[j] = F.Lp[j] + 1;
    std::vector<int32_t> flag(n, -1), stack(n), path(n);
    for (int64_t k = 0; k < n; ++k) {
        // pattern of row k in topological order (etree reach, as in the symbolic pass)
        int64_t top = n;
        flag[k] = (int32_t)k;
        double d = 0.0, mkk = 0.0;
        for (int64_t p = rp[k]; p < rp[k + 1]; ++p) {
            int32_t i = rj[p];
            if (i == k) { d = rx[p]; mkk = rx[p]; continue; }
            x[i] = rx[p];
            int64_t len = 0;
            while (i != -1 && i < k && flag[i] != (int32_t)k) {
                path[len++] = i;
                flag[i] = (int32_t)k;
                i = F.parent[i];
            }
            while (len > 0) stack[--top] = path[--len];
        }
        for (; top < n; ++top) {
            const int32_t i = stack[top];
            if (i >= n_lead) { x[i] = 0.0; continue; }      // trailing block left to the caller
            const double lki = x[i] / F.Lx[F.Lp[i]];
            x[i] = 0.0;
            const int64_t pend = c[i];
            if (k < n_lead) {
                for (int64_t p = F.Lp[i] + 1; p < pend; ++p) x[F.Li[p]] -= F.Lx[p] * lki;
            } else {
                for (int64_t p = F.Lp[i] + 1; p < pend && F.Li[p] < n_lead; ++p) x[F.Li[p]] -= F.Lx[p] * lki;
            }
            d -= lki * lki;
            // symbolic already placed row k at slot c[i]
            F.Lx[pend] = lki;
            c[i] = pend + 1;
        }
        if (k < n_lead) {
            // Rank-deficient A A^T (redundant constraints): the reference's CHOLMOD LDL^T sails through
            // pivots of size ~eps with either sign and returns an arbitrary null-space component in y.
            // Here such a pivot is treated as a redundant constraint: L_kk = +inf, i.e. z_k = 0, which
            // leaves A^T y (all the iteration uses) unchanged and keeps y bounded.
            if (!(d > kPivotTol * std::max(mkk, 1e-300))) {
                F.Lx[F.Lp[k]] = INFINITY;
                F.n_deficient++;
            } else {
                F.Lx[F.Lp[k]] = std::sqrt(d);
            }
        } else {
            F.Lx[F.Lp[k]] = d;   // M_kk - sum_{i<n_lead} L_ki^2 : diagonal of the Schur complement
        }
    }
}

}  // namespace cuadmm
