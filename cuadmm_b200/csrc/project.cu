// project.cu — PSD projection kernels (shared-memory one-sided Jacobi) and their launcher.
// See project_jacobi.cuh for the algorithm; this file holds the kernels, the size classes
// and the svec<->smat kernels on the reference's pooled layout.
#include "plan.h"
#include <algorithm>
#include <limits>
#include <type_traits>
#include <numeric>
#include <stdlib.h>

namespace cuadmm {

// ------------------------------------------------------------------------------------------
// helpers
// ------------------------------------------------------------------------------------------
template <bool WARP>
__device__ __forceinline__ void mat_sync() {
    if (WARP) __syncwarp(); else __syncthreads();
}

// sum over the NT threads working on one matrix; every thread receives the total
template <int NT, bool WARP>
__device__ __forceinline__ double mat_sum(double v, double* red, int tid) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (WARP) return v;
    const int wid = tid >> 5;
    __syncthreads();
    if ((tid & 31) == 0) red[wid] = v;
    __syncthreads();
    double t = 0.0;
#pragma unroll 1
    for (int i = 0; i < NT / 32; ++i) t += red[i];   // same order in every thread => identical
    return t;
}

// max over the NT threads working on one matrix
template <int NT, bool WARP>
__device__ __forceinline__ double mat_max(double v, double* red, int tid) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    if (WARP) return v;
    const int wid = tid >> 5;
    __syncthreads();
    if ((tid & 31) == 0) red[wid] = v;
    __syncthreads();
    double t = 0.0;
#pragma unroll 1
    for (int i = 0; i < NT / 32; ++i) t = fmax(t, red[i]);
    return t;
}

// ------------------------------------------------------------------------------------------
// shared-memory kernel: T threads per CTA, L lanes per column pair, up to RPL rows per lane.
// WARP = true: one warp per matrix, T/32 matrices per CTA.
//
// Instruction budget per column pair is what bounds this kernel (measured: issue-bound, not
// latency-bound), so: (1) only gamma = g_p.g_q is reduced across the group, the squared column
// norms alpha/beta are tracked in shared memory by the exact update
//     alpha' = c^2 alpha - 2cs gamma + s^2 beta,  beta' = s^2 alpha + 2cs gamma + c^2 beta
// and refreshed from the data at the start of every sweep; (2) the rotation comes from two rsqrt
// and no division (jacobi_cs2); (3) L is small so one warp instruction serves 32/L pairs.
// Column stride ld == L (mod 16) makes the L-row windows of the 16/L consecutive round-robin
// columns a half-warp touches fall into disjoint banks.
// ------------------------------------------------------------------------------------------
// (16-byte sweep accesses — two rows per lane, ld == 8 mod 16 — were measured 10 % slower on B200: profiles/ncu_r02.md)
__host__ __device__ __forceinline__ int jacobi_ld(int n, int L) {
    if (L >= 16) return n | 1;
    int ld = n;
    while ((ld & 15) != (L & 15)) ++ld;
    return ld;
}
__host__ __device__ __forceinline__ size_t jacobi_per_mat(int nmax, int L) {
    // even number of doubles: every matrix of a multi-matrix CTA starts 16-byte aligned (vectorised sweeps)
    return (((size_t)jacobi_ld(nmax, L) * nmax + nmax + (nmax + 2) / 2 + 1 + 34) + 1) & ~(size_t)1;
}

// rotation from (alpha, beta, gamma) with two rsqrt: cos(2t) = |d|/h, sin(2t) = sign(d) 2gamma/h,
// d = beta - alpha, h = hypot(d, 2 gamma); c = sqrt((1+cos 2t)/2), s = sin(2t)/(2c).
// Also returns the tracked-norm updates.
__device__ __forceinline__ void jacobi_cs2(double alpha, double beta, double gamma, double& c, double& s,
                                           double& alpha_new, double& beta_new) {
    const double d = beta - alpha;
    const double g2 = gamma + gamma;
    const double rh = rsqrt(fma(d, d, g2 * g2));
    const double c2 = fabs(d) * rh;                       // cos 2theta in [0,1]
    const double s2 = (d < 0.0 ? -g2 : g2) * rh;          // sin 2theta
    const double cc = fma(0.5, c2, 0.5);                  // c^2 in [0.5,1]
    const double rc = rsqrt(cc);
    c = cc * rc;
    s = 0.5 * s2 * rc;
    const double ss = 1.0 - cc;                           // s^2
    const double x = s2 * gamma;                          // 2 c s gamma
    alpha_new = fma(cc, alpha, fma(ss, beta, -x));
    beta_new = fma(ss, alpha, fma(cc, beta, x));
}

__device__ __forceinline__ void jacobi_dmma(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// Convergence test on the STATE of the block: are all columns of G mutually orthogonal to `thr` (relative)?
// The Gram matrix G^T G is formed 8 x 8 tile by tile on the FP64 tensor cores (mma.sync.m8n8k4: n^3/2 MACs in
// n^3/512 warp instructions — about 2 % of one sweep) and every off-diagonal entry is held against the tracked squared
// norms w[].  Testing the state after a sweep, instead of the cosines met during the next one, saves a whole
// verification sweep (1 of ~3 in the warm-started regime).
// Entries below 1e-15 in absolute value (G has norm ~1) are rounding noise of null columns and never count.
template <int NT, bool WARP>
__device__ __forceinline__ bool jacobi_gram_converged(const double* G, const double* w, int n, int ld, double thr2, int tid) {
    const int lane = tid & 31;
    const int wid = WARP ? 0 : (tid >> 5);
    constexpr int NW = WARP ? 1 : NT / 32;
    const int nt = (n + 7) >> 3;
    const int kr = lane & 3, cq = lane >> 2;
    int flag = 0;
    // a warp takes row tiles P = wid, wid + NW, ... and walks the column tiles Q >= P four at a time: four independent
    // accumulator pairs per k-step hide the latency of the dependent mma chain (measured: 20 % of the kernel's stall
    // samples sat on a single-accumulator chain)
    for (int P = wid; P < nt; P += NW) {
        const int pcol = P * 8 + cq;
        const double* Gp = G + (size_t)min(pcol, n - 1) * ld;
        const bool pv = pcol < n;
        const int row = P * 8 + cq;
        const double wr = (row < n) ? w[row] : 0.0;
        for (int Q0 = P; Q0 < nt; Q0 += 4) {
            double c[4][2];
            const double* Gq[4];
            bool qv[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int qcol = (Q0 + u) * 8 + cq;
                qv[u] = (Q0 + u < nt) && qcol < n;
                Gq[u] = G + (size_t)min(qcol, n - 1) * ld;
                c[u][0] = 0.0; c[u][1] = 0.0;
            }
            for (int r0 = 0; r0 < n; r0 += 4) {
                const int r = r0 + kr;
                const bool rv = r < n;
                const double av = (pv && rv) ? Gp[r] : 0.0;
                double bv[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) bv[u] = (qv[u] && rv) ? Gq[u][r] : 0.0;
#pragma unroll
                for (int u = 0; u < 4; ++u) jacobi_dmma(c[u][0], c[u][1], av, bv[u]);
            }
            // c[u] = (G^T G)[P*8 + lane/4][(Q0+u)*8 + 2*(lane%4) + {0,1}]
            if (row < n) {
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int col0 = (Q0 + u) * 8 + 2 * kr;
                    if (Q0 + u < nt) {
                        if (col0 < n && col0 != row) { const double g2 = c[u][0] * c[u][0]; if (g2 > thr2 * wr * w[col0] && g2 > 1e-30) flag = 1; }
                        if (col0 + 1 < n && col0 + 1 != row) { const double g2 = c[u][1] * c[u][1]; if (g2 > thr2 * wr * w[col0 + 1] && g2 > 1e-30) flag = 1; }
                    }
                }
            }
        }
    }
    const int any = WARP ? __any_sync(0xffffffffu, flag) : __syncthreads_or(flag);
    return !any;
}

// resident CTAs per SM the register allocation must allow (the sweeps are throughput-bound at full batches)
constexpr int jacobi_min_ctas(int T) { return T <= 64 ? 8 : T <= 128 ? 4 : T <= 256 ? 2 : 1; }

template <int T, int L, int RPL, bool WARP>
__global__ void __launch_bounds__(T, jacobi_min_ctas(T)) proj_jacobi_kernel(ProjArgs a, int nmax) {
    extern __shared__ double smem[];
    constexpr int NT = WARP ? 32 : T;
    constexpr int NG = NT / L;
    constexpr int MPC = WARP ? T / 32 : 1;
    const int tid = WARP ? (threadIdx.x & 31) : threadIdx.x;
    const int mat_in_cta = WARP ? (threadIdx.x >> 5) : 0;
    const int bi = blockIdx.x * MPC + mat_in_cta;
    if (bi >= a.nblk) return;
    if (a.done_flag && *a.done_flag) return;

    const size_t per_mat = jacobi_per_mat(nmax, L);
    double* G = smem + per_mat * mat_in_cta;
    double* w = G + (size_t)jacobi_ld(nmax, L) * nmax;     // tracked squared norms, later rebuild weights
    int* pos = (int*)(w + nmax);
    double* red = w + nmax + (nmax + 2) / 2 + 1;

    const BlkDesc d = a.desc[bi];
    const int n = d.n;
    const int ld = jacobi_ld(n, L);
    const int ntri = n * (n + 1) / 2;
    const double* __restrict__ xin = a.Xb + d.svec_off;
    double* __restrict__ xout = a.Xproj + d.svec_off;

    // ---- svec -> smat (vector_to_matrices); max |entry| for an exact power-of-two prescale ----
    // (eight loads in flight per thread: with one block per SM — a rank's share on 8 GPUs — the stage is bound by the
    // latency of ONE block, and a loop of dependent-looking global loads was ~17 DRAM round trips of it)
    double amax = 0.0;
    for (int idx0 = tid; idx0 < ntri; idx0 += NT * 8) {
        double v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) { const int idx = idx0 + u * NT; v[u] = (idx < ntri) ? __ldg(xin + idx) : 0.0; }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int idx = idx0 + u * NT;
            if (idx < ntri) {
                int r, c;
                tri_unrank(idx, r, c);
                amax = fmax(amax, fabs(v[u]));          // fmax drops NaN; caught below through the norm
                const double v2 = (r == c) ? v[u] : v[u] * CUADMM_SQRT2INV;
                G[r + c * ld] = v2;
                G[c + r * ld] = v2;
            }
        }
    }
    amax = mat_max<NT, WARP>(amax, red, tid);
    int ex = 0;
    if (amax > 0.0 && amax < 1.7e308) frexp(amax, &ex);
    mat_sync<WARP>();
    // Frobenius norm of the 2^-ex prescaled block (no over/underflow for any finite input)
    double f2 = 0.0;
    // (r, c) of entry e = tid + k NT advanced incrementally: an integer division per entry was 8 % of the zero-sweep time
    const int e_dc = NT / n, e_dr = NT - e_dc * n;
    const int e_c0 = tid / n, e_r0 = tid - e_c0 * n;
    for (int c = e_c0, r = e_r0; c < n;) {
        const double v = ldexp(G[r + c * ld], -ex);
        G[r + c * ld] = v;
        f2 = fma(v, v, f2);
        r += e_dr; c += e_dc;
        if (r >= n) { r -= n; ++c; }
    }
    f2 = mat_sum<NT, WARP>(f2, red, tid);
    const double sp = sqrt(f2);              // ||A||_F * 2^-ex
    if (!(sp > 0.0) || !(sp < 1.7e308)) {
        // zero block: Pi_+(0) = 0; NaN/Inf input propagates NaN
        const double fill = (sp == 0.0) ? 0.0 : (sp - sp);
        for (int idx = tid; idx < ntri; idx += NT) {
            xout[idx] = fill;
            if (a.epi.X) {
                const int64_t gi = d.svec_off + idx;
                const double sig = *a.epi.sig_ptr;
                const double Sv = (fill - a.epi.X[gi]) / sig - a.epi.Rd1[gi];
                a.epi.S[gi] = Sv;
                a.epi.SmC[gi] = Sv - a.epi.Cd[gi];
            }
        }
        if (tid == 0 && a.sweeps_out) a.sweeps_out[d.index] = 0;
        if (a.eig_out) for (int j = tid; j < n; j += NT) a.eig_out[d.w_off + j] = fill;
        return;
    }
    const double inv_s = 1.0 / sp;
    // G <- A / ||A||_F + I
    for (int c = e_c0, r = e_r0; c < n;) {
        const double v = G[r + c * ld] * inv_s;
        G[r + c * ld] = (r == c) ? v + 1.0 : v;
        r += e_dr; c += e_dc;
        if (r >= n) { r -= n; ++c; }
    }
    mat_sync<WARP>();

    const int m = n + (n & 1);
    const int half = m >> 1;
    const int grp = tid / L, lane = tid % L;
    const unsigned gmask = (L == 32) ? 0xffffffffu : (((1u << L) - 1u) << ((tid & 31) / L * L));

    // ---- warm start: G <- G Q with Q the orthonormal basis the previous projection of this block
    // ended in.  G Q has the singular values and left singular vectors of G, and when the block
    // changed little since last time (successive ADMM iterates) its columns are already close to
    // orthogonal: the sweeps below converge in 2-3 passes instead of 7-9.  One group per row, the row
    // held in registers, so the product is formed in place.
    double* Qb = a.Q ? a.Q + d.q_off : nullptr;
    if (Qb) {
        // FP64 tensor cores (mma.sync.m8n8k4): every warp owns strips of 8 rows of G; the strip (8 x n) is held as A
        // fragments in registers, multiplied by the 8-column tiles of Q streamed from global memory / L2 (one 8-byte load
        // per lane feeds 256 MACs) and written back over itself — rows are independent, so the product is in place.
        constexpr int KF = (((L * RPL) > 168 ? 168 : (L * RPL)) + 3) / 4;   // k-fragments per lane for the largest n of the variant
        constexpr int NWARP = WARP ? 1 : NT / 32;
        const int wid = WARP ? 0 : (tid >> 5);
        const int l32 = tid & 31;
        const int fr = l32 >> 2, fk = l32 & 3;
        const int nk = (n + 3) >> 2;
        for (int r0 = wid * 8; r0 < n; r0 += NWARP * 8) {
            const int row = r0 + fr;
            double af[KF];
#pragma unroll
            for (int kk = 0; kk < KF; ++kk) {
                const int k = kk * 4 + fk;
                af[kk] = (kk < nk && row < n && k < n) ? G[row + k * ld] : 0.0;
            }
            __syncwarp();                                   // the whole strip is in registers before any of it is overwritten
            for (int j0 = 0; j0 < n; j0 += 16) {
                // two 8-column tiles per pass; ALL k-fragments of both tiles are requested from L2 before the first mma
                // (2 x KF loads in flight per lane) — issued one k-step at a time, every step paid an L2 round trip
                constexpr int KC = KF < 16 ? KF : 16;          // k-fragments requested per batch (register budget)
                const int col0 = j0 + fr, col1 = j0 + 8 + fr;
                const double* __restrict__ q0 = Qb + (size_t)min(col0, n - 1) * n;
                const double* __restrict__ q1 = Qb + (size_t)min(col1, n - 1) * n;
                double c00 = 0.0, c01 = 0.0, c10 = 0.0, c11 = 0.0;
#pragma unroll
                for (int kb = 0; kb < KF; kb += KC) {
                    if (kb < nk) {
                        double b0[KC], b1[KC];
#pragma unroll
                        for (int kk = 0; kk < KC; ++kk) {
                            const int k = (kb + kk) * 4 + fk;
                            const bool kv = kb + kk < nk && k < n;
                            b0[kk] = (kv && col0 < n) ? __ldg(q0 + k) : 0.0;
                            b1[kk] = (kv && col1 < n) ? __ldg(q1 + k) : 0.0;
                        }
#pragma unroll
                        for (int kk = 0; kk < KC; ++kk) {
                            if (kb + kk < KF && kb + kk < nk) {
                                jacobi_dmma(c00, c01, af[kb + kk], b0[kk]);
                                jacobi_dmma(c10, c11, af[kb + kk], b1[kk]);
                            }
                        }
                    }
                }
                if (row < n) {
                    const int cc = j0 + 2 * fk;
                    if (cc < n) G[row + cc * ld] = c00;
                    if (cc + 1 < n) G[row + (cc + 1) * ld] = c01;
                    if (cc + 8 < n) G[row + (cc + 8) * ld] = c10;
                    if (cc + 9 < n) G[row + (cc + 9) * ld] = c11;
                }
            }
        }
        mat_sync<WARP>();
    }

    // ---- Jacobi sweeps ----
    // (A "quadratic" early stop -- declare convergence after a sweep that only saw small cosines --
    // is NOT safe: inside a cluster of equal eigenvalues the rotation angle is O(1) however small the
    // cosine, and drags not-yet-visited inner products into pairs already done.  Measured: 1.6e-9
    // error on +-1 spectra.  So the loop ends when the Gram test finds every pair of the state orthogonal.)
    const double thr2 = a.threshold * a.threshold;
    const double tiny2 = 1.2325951644078309e-32;  // 2^-106: rotations below rounding level are skipped
    int sweeps = 0;
    bool converged = false;
    while (true) {
        // refresh the tracked squared norms from the data
        for (int j = grp; j < n; j += NG) {
            const double* Gj = G + j * ld;
            double al = 0.0;
            for (int r = lane; r < n; r += L) al = fma(Gj[r], Gj[r], al);
#pragma unroll
            for (int o = L / 2; o > 0; o >>= 1) al += __shfl_xor_sync(gmask, al, o);
            if (lane == 0) w[j] = al;
        }
        mat_sync<WARP>();
        if (jacobi_gram_converged<NT, WARP>(G, w, n, ld, thr2, tid)) { converged = true; break; }
        if (sweeps >= a.max_sweeps) break;
        // The row loops are unrolled and the columns of a pair live in registers, so their trip count is a compile-time
        // constant; a block smaller than its class's largest (n = 36 in the class up to 48) would issue the predicated
        // row steps of the largest one.  Four instantiations per kernel, picked by the block's own row count.
        auto run_steps = [&](auto nit_c) {
            constexpr int NIT = decltype(nit_c)::value;
            for (int step = 0; step < m - 1; ++step) {
                for (int k = grp; k < half; k += NG) {
                    int pa, pb;
                    rr_pair(m, step, k, pa, pb);
                    if (pa >= n || pb >= n) continue;  // the bye of an odd-sized block
                    const int p = min(pa, pb), q = max(pa, pb);
                    double* __restrict__ Gp = G + p * ld;
                    double* __restrict__ Gq = G + q * ld;
                    double gp[NIT], gq[NIT];
                    double ga = 0.0, gb = 0.0;
    #pragma unroll
                    for (int i = 0; i < NIT; ++i) {
                        const int r = lane + i * L;
                        if (r < n) {
                            gp[i] = Gp[r];
                            gq[i] = Gq[r];
                            if (i & 1) gb = fma(gp[i], gq[i], gb); else ga = fma(gp[i], gq[i], ga);
                        } else {
                            gp[i] = 0.0; gq[i] = 0.0;
                        }
                    }
                    ga += gb;
                    const double al = w[p], be = w[q];
    #pragma unroll
                    for (int o = L / 2; o > 0; o >>= 1) ga += __shfl_xor_sync(gmask, ga, o);
                    const double g2 = ga * ga, ab = al * be;
                    if (g2 > tiny2 * ab) {
                        double c, sn, an, bn;
                        jacobi_cs2(al, be, ga, c, sn, an, bn);
    #pragma unroll
                        for (int i = 0; i < NIT; ++i) {
                            const int r = lane + i * L;
                            if (r < n) {
                                Gp[r] = fma(c, gp[i], -sn * gq[i]);
                                Gq[r] = fma(sn, gp[i], c * gq[i]);
                            }
                        }
                        if (lane == 0) { w[p] = an; w[q] = bn; }
                    }
                }
                mat_sync<WARP>();
            }
        };
        {
            constexpr int S = RPL >= 8 ? RPL / 8 : 1;
            const int nit = (n + L - 1) / L;
            if (nit <= RPL - 3 * S) run_steps(std::integral_constant<int, RPL - 3 * S>{});
            else if (nit <= RPL - 2 * S) run_steps(std::integral_constant<int, RPL - 2 * S>{});
            else if (nit <= RPL - S) run_steps(std::integral_constant<int, RPL - S>{});
            else run_steps(std::integral_constant<int, RPL>{});
        }
        ++sweeps;
    }

    // ---- eigenvalues from the column norms; weights of the positive part ----
    const double s_true = ldexp(sp, ex);     // ||A||_F
    int q_bad = converged ? 0 : 1;
    for (int j = grp; j < n; j += NG) {
        const double* Gj = G + j * ld;
        double al = 0.0;
        for (int r = lane; r < n; r += L) al = fma(Gj[r], Gj[r], al);
#pragma unroll
        for (int o = L / 2; o > 0; o >>= 1) al += __shfl_xor_sync(gmask, al, o);
        if (Qb) {
            // next call's basis: the normalised columns.  A basis that is not orthonormal to rounding
            // would change the answer, so a block that did not converge (or has a null column) restarts
            // from the identity.
            if (!(al > 1e-24)) q_bad = 1;
            const double rs = rsqrt(al);
            double* qj = Qb + (size_t)j * n;
            for (int r = lane; r < n; r += L) qj[r] = Gj[r] * rs;
        }
        if (lane == 0) {
            const double sigma = sqrt(al);
            // sqrt of the rebuild weight: Pi_+ = s sum_j (sigma_j - 1)/sigma_j^2 g_j g_j^T
            w[j] = (sigma > 1.0) ? sqrt((sigma - 1.0) / al) : 0.0;
            if (a.eig_out) a.eig_out[d.w_off + j] = s_true * (sigma - 1.0);
        }
    }
    if (Qb) {
        const int any_bad = WARP ? __any_sync(0xffffffffu, q_bad) : __syncthreads_or(q_bad);
        if (any_bad) for (int e = tid; e < n * n; e += NT) Qb[e] = (e / n == e % n) ? 1.0 : 0.0;
    } else {
        mat_sync<WARP>();
    }
    if (a.rank_limit > 0) {
        // fixed-rank projection (max_dense_vector_zero_mask with the mask of get_eig_rank_mask, src/kernels/dense_scalar.cu:51-56,
        // src/utils/get_eig_rank_mask.cu:16-38): only the rank_limit LARGEST eigenvalues of the block may survive the clamp.
        // The rebuild weight is increasing in the eigenvalue on (0, ||A||], so ranking weights ranks eigenvalues.
        int drop = 0;
        if (tid < n && w[tid] > 0.0) {
            const double mine = w[tid];
            int rank = 0;
            for (int k = 0; k < n; ++k) { const double o = w[k]; rank += (o > mine || (o == mine && k > tid)) ? 1 : 0; }
            drop = rank >= a.rank_limit;
        }
        mat_sync<WARP>();
        if (drop) w[tid] = 0.0;
        mat_sync<WARP>();
    }
    if (tid == 0) {
        int k = 0;
        for (int j = 0; j < n; ++j) if (w[j] > 0.0) pos[k++] = j;
        pos[n] = k;
        if (a.sweeps_out) a.sweeps_out[d.index] = sweeps;
    }
    mat_sync<WARP>();
    const int kpos = pos[n];
    // h_j = sqrt(w_j) g_j for the positive columns
    for (int jj = e_c0, r = e_r0; jj < kpos;) {
        const int j = pos[jj];
        G[r + j * ld] *= w[j];
        r += e_dr; jj += e_dc;
        if (r >= n) { r -= n; ++jj; }
    }
    mat_sync<WARP>();

    // ---- rebuild + smat -> svec (matrices_to_vector), optional fused S / SmC ----
    // Pi_+ = s H H^T with H = the kpos scaled positive columns: 8 x 8 output tiles on the FP64 tensor cores
    // (mma.sync.m8n8k4: A = rows of H, B = rows of H again, read through pos[]), upper tile triangle only.  A unit of work
    // is one 8-column block and up to four 8-row blocks above it (they share the B fragment); the accumulator layout
    // (row = lane / 4, columns 2 (lane % 4) + {0, 1}) gives the svec index c (c + 1) / 2 + r directly and makes the 8
    // lanes of a column touch 64 contiguous bytes of the svec vectors.  (The scalar loop this replaces — two shared
    // loads per FMA and a triangular un-ranking per entry — was 20 % of the kernel's time at zero sweeps.)
    double sig = 1.0;
    if (a.epi.X) sig = *a.epi.sig_ptr;
    {
        constexpr int NWARP = WARP ? 1 : NT / 32;
        const int wid = WARP ? 0 : (tid >> 5);
        const int l32 = tid & 31;
        const int fr = l32 >> 2, fk = l32 & 3;
        const int T8 = (n + 7) >> 3;
        const int nkk = (kpos + 3) >> 2;
        int unit = 0;
        for (int C = 0; C < T8; ++C) {
            for (int R0 = 0; R0 <= C; R0 += 4, ++unit) {
                if (unit % NWARP != wid) continue;
                const int nR = min(4, C + 1 - R0);
                // outputs of this lane: (r_t, c_h) = (8 (R0 + t) + fr, 8 C + 2 fk + h); epilogue operands requested first
                double xv[4][2], rd[4][2], cd[4][2];
                if (a.epi.X) {
#pragma unroll
                    for (int t = 0; t < 4; ++t)
#pragma unroll
                        for (int h = 0; h < 2; ++h) {
                            const int r = 8 * (R0 + t) + fr, c = 8 * C + 2 * fk + h;
                            xv[t][h] = 0.0; rd[t][h] = 0.0; cd[t][h] = 0.0;
                            if (t < nR && r <= c && c < n) {
                                const int64_t g = d.svec_off + (int64_t)c * (c + 1) / 2 + r;
                                xv[t][h] = __ldg(a.epi.X + g); rd[t][h] = __ldg(a.epi.Rd1 + g); cd[t][h] = __ldg(a.epi.Cd + g);
                            }
                        }
                }
                double acc[4][2];
#pragma unroll
                for (int t = 0; t < 4; ++t) { acc[t][0] = 0.0; acc[t][1] = 0.0; }
                const int brow = 8 * C + fr;
                for (int kk = 0; kk < nkk; ++kk) {
                    const int k = 4 * kk + fk;
                    const bool kv = k < kpos;
                    const double* Gk = G + (kv ? pos[k] : 0) * ld;
                    const double b = (kv && brow < n) ? Gk[brow] : 0.0;
                    double av[4];
#pragma unroll
                    for (int t = 0; t < 4; ++t) {
                        const int r = 8 * (R0 + t) + fr;
                        av[t] = (kv && t < nR && r < n) ? Gk[r] : 0.0;
                    }
#pragma unroll
                    for (int t = 0; t < 4; ++t) jacobi_dmma(acc[t][0], acc[t][1], av[t], b);
                }
#pragma unroll
                for (int t = 0; t < 4; ++t)
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int r = 8 * (R0 + t) + fr, c = 8 * C + 2 * fk + h;
                        if (t < nR && r <= c && c < n) {
                            const int idx = c * (c + 1) / 2 + r;
                            const double v = acc[t][h] * s_true;
                            const double out = (r == c) ? v : v * CUADMM_SQRT2;
                            xout[idx] = out;
                            if (a.epi.X) {
                                const int64_t g = d.svec_off + idx;
                                const double Sv = (out - xv[t][h]) / sig - rd[t][h];
                                a.epi.S[g] = Sv;
                                a.epi.SmC[g] = Sv - cd[t][h];
                            }
                        }
                    }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// eigenvalues of blocks n > 168 for the debug entry cuadmm_project_psd_eig_host (their projection is the
// dense sign path's, which has none): the same shifted one-sided Jacobi with G in HBM/L2, one CTA of
// 1024 threads per block, one warp per column pair, rows streamed twice (dot, then update).
// Writes eigenvalues and sweep counts only.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) proj_jacobi_global_kernel(ProjArgs a) {
    __shared__ double red[34];
    const int tid = threadIdx.x;
    const int bi = blockIdx.x;
    if (bi >= a.nblk) return;
    if (a.done_flag && *a.done_flag) return;
    const BlkDesc d = a.desc[bi];
    const int n = d.n;
    const int64_t ld = n;
    double* G = a.scratch + d.scratch_off;          // n*n
    const double* __restrict__ xin = a.Xb + d.svec_off;

    double f2 = 0.0;
    for (int c = 0; c < n; ++c) {
        const int64_t base = (int64_t)c * (c + 1) / 2;
        for (int r = tid; r <= c; r += 1024) {
            const double v = xin[base + r];
            f2 += v * v;
            const double v2 = (r == c) ? v : v * CUADMM_SQRT2INV;
            G[r + c * ld] = v2;
            G[c + r * ld] = v2;
        }
    }
    f2 = mat_sum<1024, false>(f2, red, tid);
    const double s = sqrt(f2);
    if (!(s >= 1e-290)) {
        const double fill = (s == s) ? 0.0 : s;
        if (tid == 0 && a.sweeps_out) a.sweeps_out[d.index] = 0;
        if (a.eig_out) for (int j = tid; j < n; j += 1024) a.eig_out[d.w_off + j] = fill;
        return;
    }
    const double inv_s = 1.0 / s;
    __syncthreads();
    for (int64_t e = tid; e < (int64_t)n * n; e += 1024) {
        const int c = (int)(e / n), r = (int)(e - (int64_t)c * n);
        const double v = G[e] * inv_s;
        G[e] = (r == c) ? v + 1.0 : v;
    }
    __syncthreads();

    const int m = n + (n & 1), half = m >> 1;
    const int grp = tid >> 5, lane = tid & 31;
    const double thr2 = a.threshold * a.threshold;
    int sweeps = 0;
    while (sweeps < a.max_sweeps) {
        int big = 0;
        for (int step = 0; step < m - 1; ++step) {
            for (int k = grp; k < half; k += 32) {
                int pa, pb;
                rr_pair(m, step, k, pa, pb);
                if (pa >= n || pb >= n) continue;
                const int p = min(pa, pb), q = max(pa, pb);
                double* Gp = G + p * ld;
                double* Gq = G + q * ld;
                double al = 0.0, be = 0.0, ga = 0.0;
                for (int r = lane; r < n; r += 32) {
                    const double x = Gp[r], y = Gq[r];
                    al = fma(x, x, al); be = fma(y, y, be); ga = fma(x, y, ga);
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    al += __shfl_xor_sync(0xffffffffu, al, o);
                    be += __shfl_xor_sync(0xffffffffu, be, o);
                    ga += __shfl_xor_sync(0xffffffffu, ga, o);
                }
                if (ga * ga > thr2 * al * be) big = 1;
                double c, sn;
                if (jacobi_cs(al, be, ga, c, sn)) {
                    for (int r = lane; r < n; r += 32) {
                        const double x = Gp[r], y = Gq[r];
                        Gp[r] = c * x - sn * y;
                        Gq[r] = sn * x + c * y;
                    }
                }
            }
            __syncthreads();
        }
        ++sweeps;
        if (!__syncthreads_or(big)) break;
    }
    for (int j = grp; j < n; j += 32) {
        const double* Gj = G + j * ld;
        double al = 0.0;
        for (int r = lane; r < n; r += 32) al = fma(Gj[r], Gj[r], al);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) al += __shfl_xor_sync(0xffffffffu, al, o);
        if (lane == 0 && a.eig_out) a.eig_out[d.w_off + j] = s * (sqrt(al) - 1.0);
    }
    if (tid == 0 && a.sweeps_out) a.sweeps_out[d.index] = sweeps;
}

// ------------------------------------------------------------------------------------------
// svec <-> smat on the reference's pooled layout (one CTA per block)
// ------------------------------------------------------------------------------------------
__global__ void svec_to_smat_kernel(const double* __restrict__ svec, double* large_mat, double* small_mat,
                                    const int32_t* __restrict__ blk, const int64_t* __restrict__ svec_off,
                                    const int64_t* __restrict__ mat_off, const uint8_t* __restrict__ pool) {
    const int k = blockIdx.x;
    const int n = blk[k];
    const double* x = svec + svec_off[k];
    double* M = (pool[k] ? small_mat : large_mat) + mat_off[k];
    for (int c = blockIdx.y; c < n; c += gridDim.y) {
        const int64_t base = (int64_t)c * (c + 1) / 2;
        for (int r = threadIdx.x; r <= c; r += blockDim.x) {
            // same arithmetic as vector_to_matrices_kernel: off-diagonals * SQRT2INV, mirror copied
            const double v = (r == c) ? x[base + r] : x[base + r] * CUADMM_SQRT2INV;
            M[(int64_t)n * c + r] = v;
            M[(int64_t)n * r + c] = v;
        }
    }
}

__global__ void smat_to_svec_kernel(const double* __restrict__ large_mat, const double* __restrict__ small_mat,
                                    double* svec, const int32_t* __restrict__ blk,
                                    const int64_t* __restrict__ svec_off, const int64_t* __restrict__ mat_off,
                                    const uint8_t* __restrict__ pool) {
    const int k = blockIdx.x;
    const int n = blk[k];
    double* x = svec + svec_off[k];
    const double* M = (pool[k] ? small_mat : large_mat) + mat_off[k];
    for (int c = blockIdx.y; c < n; c += gridDim.y) {
        const int64_t base = (int64_t)c * (c + 1) / 2;
        for (int r = threadIdx.x; r <= c; r += blockDim.x) {
            const double v = M[(int64_t)n * c + r];   // map_M1: column c, row r
            x[base + r] = (r == c) ? v : v * CUADMM_SQRT2;
        }
    }
}

// ------------------------------------------------------------------------------------------
// size classes
// ------------------------------------------------------------------------------------------
// A block of n <= nmax runs on the first class that admits it, on proj_jacobi_kernel<T, L, RPL, WARP> with
// L * RPL >= nmax.  The table is the tuning sweep's result (profiles/jacobi_tuning_r01.md); retuning means
// instantiating candidate configurations again and timing them.
struct SizeClass {
    int nmax;           // largest n of the class; sizes the shared memory
    int threads;
    int L;
    int mats_per_cta;
    void (*fn)(ProjArgs, int);
};

#define CUADMM_CLASS(NMAX, T, L, RPL, WARP) {NMAX, T, L, (WARP) ? (T) / 32 : 1, proj_jacobi_kernel<T, L, RPL, WARP>}
// (a separate class for 33..48 on 12 rows per lane was 3 % faster before the sweep was instantiated per row count, and
// slower after: more distinct kernels running side by side)
static const SizeClass kSizeClasses[] = {
    CUADMM_CLASS(16, 128, 4, 4, true),
    CUADMM_CLASS(32, 64, 4, 8, false),
    CUADMM_CLASS(64, 128, 4, 16, false),
    CUADMM_CLASS(96, 192, 4, 24, false),
    CUADMM_CLASS(128, 512, 8, 16, false),
    CUADMM_CLASS(168, 352, 8, 21, false),
};
static const int kNumSizeClasses = (int)(sizeof(kSizeClasses) / sizeof(kSizeClasses[0]));
// Class::kind of the blocks above every size class in a force_global plan
static const int kGlobalKind = -1;

static size_t smem_bytes(int nmax, const SizeClass& sc) {
    return jacobi_per_mat(nmax, sc.L) * sizeof(double) * sc.mats_per_cta;
}

}  // namespace cuadmm

using namespace cuadmm;

cuadmm_plan::~cuadmm_plan() {
    if (device >= 0) {
        cudaSetDevice(device);
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (fork_event) cudaEventDestroy(fork_event);
        if (lin_stream) cudaStreamDestroy(lin_stream);
        if (lin_event) cudaEventDestroy(lin_event);
        for (auto s : side_streams) cudaStreamDestroy(s);
        for (auto e : side_events) cudaEventDestroy(e);
        if (dense) dense_part_destroy(dense);
    }
}

void cuadmm_plan::build_device() {
    const int64_t nblk = (int64_t)layout.blk.size();
    // eigenvalue offsets in blk order, over the 's' blocks (the debug entry expands them to all blocks)
    std::vector<int64_t> w_off(nblk + 1, 0);
    for (int64_t k = 0; k < nblk; ++k) w_off[k + 1] = w_off[k] + (layout.types[k] == 's' ? layout.blk[k] : 0);
    eig_len = w_off[nblk];
    // 'l' / 'u' blocks: flat chunk list of the linear-cone kernel; they take no part in the size classes below
    h_lin = linear_chunks(layout);

    // classify
    std::vector<std::vector<int64_t>> members(kNumSizeClasses + 1);
    std::vector<int64_t> dense_blocks;
    for (int64_t k = 0; k < nblk; ++k) {
        if (layout.types[k] != 's') continue;
        const int n = layout.blk[k];
        int ci = kNumSizeClasses;
        for (int c = 0; c < kNumSizeClasses; ++c) if (n <= kSizeClasses[c].nmax) { ci = c; break; }
        if (ci == kNumSizeClasses && !force_global) { dense_blocks.push_back(k); continue; }
        members[ci].push_back(k);
    }
    if (dense) { dense_part_destroy(dense); dense = nullptr; }
    if (!dense_blocks.empty()) dense = dense_part_create(device, layout.blk, layout.svec_off, dense_blocks);
    h_desc.clear(); classes.clear();
    int64_t scratch = 0, q_total = 0;
    // heaviest classes first so their launches start first
    for (int ci = kNumSizeClasses; ci >= 0; --ci) {
        auto& mem = members[ci];
        if (mem.empty()) continue;
        std::stable_sort(mem.begin(), mem.end(), [&](int64_t a, int64_t b) { return layout.blk[a] > layout.blk[b]; });
        Class cl;
        cl.kind = (ci == kNumSizeClasses) ? kGlobalKind : ci;
        cl.nmax = layout.blk[mem[0]];
        cl.count = (int32_t)mem.size();
        cl.first = (int64_t)h_desc.size();
        if (cl.kind == kGlobalKind) {
            cl.smem = 0;
            cl.grid = cl.count;
        } else {
            const SizeClass& sc = kSizeClasses[cl.kind];
            cl.smem = smem_bytes(cl.nmax, sc);
            cl.grid = (cl.count + sc.mats_per_cta - 1) / sc.mats_per_cta;
        }
        for (int64_t k : mem) {
            BlkDesc d;
            d.svec_off = layout.svec_off[k];
            d.w_off = w_off[k];
            d.n = layout.blk[k];
            d.index = (int32_t)k;
            d.scratch_off = 0;
            d.q_off = 0;
            if (cl.kind != kGlobalKind) { d.q_off = q_total; q_total += (int64_t)d.n * d.n; }
            else { d.scratch_off = scratch; scratch += (int64_t)d.n * d.n; }
            h_desc.push_back(d);
        }
        classes.push_back(cl);
    }
    if (device < 0) return;

    DeviceGuard g(device);
    d_desc.upload(h_desc);
    if (!h_lin.empty()) {
        d_lin.upload(h_lin);
        CUADMM_CUDA(cudaStreamCreateWithFlags(&lin_stream, cudaStreamNonBlocking));
        CUADMM_CUDA(cudaEventCreateWithFlags(&lin_event, cudaEventDisableTiming));
    }
    if (scratch) d_scratch.alloc(scratch);
    d_eig.alloc(std::max<int64_t>(w_off[nblk], 1));
    d_sweeps.alloc(std::max<int64_t>(nblk, 1));
    warm_start = true;
    if (const char* e = getenv("CUADMM_JACOBI_WARM")) warm_start = atoi(e) != 0;
    if (const char* e = getenv("CUADMM_JACOBI_THR")) { const double v = atof(e); if (v > 0.0 && v < 1e-3) threshold = v; }
    if (warm_start && q_total > 0) {
        d_Q.alloc(q_total);
        reset_warm_start();
    }
    d_svec_off.upload(layout.svec_off);
    d_mat_off.upload(layout.mat_off);
    d_blk.upload(layout.blk);
    d_pool.upload(layout.pool);
    CUADMM_CUDA(cudaEventCreate(&ev0));
    CUADMM_CUDA(cudaEventCreate(&ev1));
    CUADMM_CUDA(cudaEventCreateWithFlags(&fork_event, cudaEventDisableTiming));
    for (size_t i = 0; i < classes.size(); ++i) {
        cudaStream_t s; cudaEvent_t e;
        CUADMM_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        CUADMM_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        side_streams.push_back(s); side_events.push_back(e);
    }
    for (const Class& cl : classes) {
        if (cl.kind == kGlobalKind) continue;
        const SizeClass& sc = kSizeClasses[cl.kind];
        CUADMM_CUDA(cudaFuncSetAttribute((const void*)sc.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes(sc.nmax, sc)));
    }
    CUADMM_CUDA(cudaDeviceSynchronize());
}

__global__ void init_basis_kernel(const BlkDesc* __restrict__ desc, int nblk, double* Q) {
    const int b = blockIdx.x;
    if (b >= nblk) return;
    const int n = desc[b].n;
    double* q = Q + desc[b].q_off;
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) q[e] = (e / n == e % n) ? 1.0 : 0.0;
}

// all warm-start bases back to the identity (= cold Jacobi on the next projection)
void cuadmm_plan::reset_warm_start() {
    if (d_Q.n == 0) return;
    DeviceGuard g(device);
    for (const Class& cl : classes) {
        if (cl.kind == kGlobalKind) continue;
        init_basis_kernel<<<cl.count, 256>>>(d_desc.p + cl.first, cl.count, d_Q.p);
    }
    CUADMM_CUDA(cudaGetLastError());
    CUADMM_CUDA(cudaDeviceSynchronize());
}

int cuadmm_plan::project(const double* d_Xb, double* d_Xproj, cudaStream_t stream,
                         const ProjEpilogue* epi, bool want_eig) {
    if (device < 0) throw Error(CUADMM_ENODEVICE, "plan was built without a CUDA device; there is no CPU fallback");
    int launches = 0;
    // blocks on the dense path produce no eigenvalues: their debug slots read NaN
    if (want_eig) {
        CUADMM_CUDA(cudaMemsetAsync(d_eig.p, 0xFF, sizeof(double) * (size_t)d_eig.n, stream));
        CUADMM_CUDA(cudaMemsetAsync(d_sweeps.p, 0, sizeof(int32_t) * (size_t)d_sweeps.n, stream));
    }
    // fork: the dense (GEMM) part, if any, runs on the caller's stream; Jacobi classes run on side
    // streams so that small, mid and large blocks overlap (class 0 stays on the caller's stream when
    // there is no dense part)
    const bool has_dense = dense != nullptr;
    const bool has_lin = !h_lin.empty();
    // the linear-cone kernel gets its own side stream when anything else runs, else the caller's stream
    const bool lin_side = has_lin && (has_dense || !classes.empty());
    if (rank_limit > 0) {
        if (has_dense) throw Error(CUADMM_EINVAL, "fixed-rank projection is only available for blocks n <= 168 (the sign iteration of larger blocks has no eigenvalues to rank)");
    }
    if (classes.size() > 1 || (has_dense && !classes.empty()) || lin_side) CUADMM_CUDA(cudaEventRecord(fork_event, stream));
    for (size_t i = 0; i < classes.size(); ++i) {
        const Class& cl = classes[i];
        cudaStream_t st = stream;
        const bool side = has_dense || i > 0;
        if (side) {
            st = side_streams[i];
            CUADMM_CUDA(cudaStreamWaitEvent(st, fork_event, 0));
        }
        ProjArgs a;
        a.Xb = d_Xb; a.Xproj = d_Xproj;
        a.desc = d_desc.p + cl.first;
        a.nblk = cl.count;
        a.threshold = threshold;
        a.max_sweeps = max_sweeps;
        a.eig_out = want_eig ? d_eig.p : nullptr;
        a.sweeps_out = want_eig ? d_sweeps.p : nullptr;
        a.scratch = d_scratch.p;
        a.done_flag = done_flag;
        a.rank_limit = rank_limit;
        a.Q = (warm_start && cl.kind != kGlobalKind && d_Q.n > 0) ? d_Q.p : nullptr;
        if (epi) a.epi = *epi; else { a.epi.X = nullptr; a.epi.Rd1 = nullptr; a.epi.Cd = nullptr; a.epi.S = nullptr; a.epi.SmC = nullptr; a.epi.sig_ptr = nullptr; }
        if (cl.kind == kGlobalKind) {
            proj_jacobi_global_kernel<<<cl.grid, 1024, 0, st>>>(a);
        } else {
            kSizeClasses[cl.kind].fn<<<cl.grid, kSizeClasses[cl.kind].threads, cl.smem, st>>>(a, cl.nmax);
        }
        CUADMM_CUDA(cudaGetLastError());
        ++launches;
        if (side) CUADMM_CUDA(cudaEventRecord(side_events[i], st));
    }
    if (has_lin) {
        cudaStream_t st = stream;
        if (lin_side) {
            st = lin_stream;
            CUADMM_CUDA(cudaStreamWaitEvent(st, fork_event, 0));
        }
        launches += linear_project(d_lin.p, d_lin.n, d_Xb, d_Xproj, st, epi, done_flag);
        if (lin_side) CUADMM_CUDA(cudaEventRecord(lin_event, st));
    }
    if (has_dense) launches += dense_part_project(dense, d_Xb, d_Xproj, stream, epi, done_flag);
    for (size_t i = 0; i < classes.size(); ++i)
        if (has_dense || i > 0) CUADMM_CUDA(cudaStreamWaitEvent(stream, side_events[i], 0));
    if (lin_side) CUADMM_CUDA(cudaStreamWaitEvent(stream, lin_event, 0));
    return launches;
}

// ------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------
extern "C" {

int cuadmm_plan_create(const int32_t* blk, int64_t nblk, int device, cuadmm_plan** out) {
    return cuadmm_plan_create_typed(nullptr, blk, nblk, device, out);
}

int cuadmm_plan_create_typed(const char* types, const int32_t* blk, int64_t nblk, int device, cuadmm_plan** out) {
    return guarded([&] {
        CUADMM_REQUIRE(out != nullptr, "out is null");
        CUADMM_REQUIRE(blk != nullptr || nblk == 0, "blk is null");
        *out = nullptr;
        std::unique_ptr<cuadmm_plan> p(new cuadmm_plan());
        p->layout.init(blk, nblk, types);
        if (device >= 0) {
            int cnt = 0;
            cudaError_t e = cudaGetDeviceCount(&cnt);
            if (e != cudaSuccess || cnt == 0) {
                cudaGetLastError();
                throw Error(CUADMM_ENODEVICE, "no CUDA device available (pass device=-1 for a host-only plan; compute has no CPU fallback)");
            }
            CUADMM_REQUIRE(device < cnt, "device index out of range");
        }
        p->device = device;
        p->build_device();
        *out = p.release();
    });
}

void cuadmm_plan_destroy(cuadmm_plan* plan) { delete plan; }
int64_t cuadmm_plan_vec_len(const cuadmm_plan* plan) { return plan ? plan->layout.vec_len : -1; }
int64_t cuadmm_plan_nblk(const cuadmm_plan* plan) { return plan ? (int64_t)plan->layout.blk.size() : -1; }
int64_t cuadmm_plan_num_sizes(const cuadmm_plan* plan) { return plan ? (int64_t)plan->layout.sizes.size() : -1; }

int cuadmm_plan_sizes(const cuadmm_plan* plan, int32_t* sizes, int32_t* nums, int32_t* is_large) {
    return guarded([&] {
        CUADMM_REQUIRE(plan, "plan is null");
        plan->layout.require_all_psd("cuadmm_plan_sizes");
        for (size_t i = 0; i < plan->layout.sizes.size(); ++i) {
            if (sizes) sizes[i] = plan->layout.sizes[i];
            if (nums) nums[i] = plan->layout.nums[i];
            if (is_large) is_large[i] = plan->layout.large[i];
        }
    });
}

int cuadmm_plan_totals(const cuadmm_plan* plan, int64_t out[6]) {
    return guarded([&] {
        CUADMM_REQUIRE(plan && out, "null argument");
        const BlockLayout& l = plan->layout;
        l.require_all_psd("cuadmm_plan_totals");
        out[0] = l.large_mat_num; out[1] = l.sum_large_mat_size; out[2] = l.total_large_mat_size;
        out[3] = l.small_mat_num; out[4] = l.sum_small_mat_size; out[5] = l.total_small_mat_size;
    });
}

int64_t cuadmm_plan_start_indices(const cuadmm_plan* plan, int which, int64_t* out) {
    if (!plan) return -1;
    const BlockLayout& l = plan->layout;
    if (!l.all_psd()) return guarded([&] { l.require_all_psd("cuadmm_plan_start_indices"); });
    const std::vector<int64_t>* v = nullptr;
    switch (which) {
        case 0: v = &l.large_mat_start; break;
        case 1: v = &l.large_W_start; break;
        case 2: v = &l.small_mat_start; break;
        case 3: v = &l.small_W_start; break;
        default: return -1;
    }
    if (out) std::copy(v->begin(), v->end(), out);
    return (int64_t)v->size();
}

int cuadmm_plan_maps(const cuadmm_plan* plan, int32_t* map_B, int32_t* map_M1, int32_t* map_M2) {
    return guarded([&] {
        CUADMM_REQUIRE(plan && map_B && map_M1 && map_M2, "null argument");
        plan->layout.maps(map_B, map_M1, map_M2);
    });
}

int cuadmm_plan_partition(const cuadmm_plan* plan, int nparts, int32_t* owner, double* part_cost) {
    return guarded([&] {
        CUADMM_REQUIRE(plan && owner, "null argument");
        plan->layout.partition(nparts, owner, part_cost);
    });
}

int cuadmm_plan_set_rank_limit(cuadmm_plan* plan, int eig_rank) {
    return guarded([&] {
        CUADMM_REQUIRE(plan, "plan is null");
        CUADMM_REQUIRE(eig_rank >= 0, "eig_rank < 0");
        plan->rank_limit = eig_rank;
    });
}

// get_eig_rank_mask (src/utils/get_eig_rank_mask.cu:16-38): 1 on the last eig_rank positions of every block of mat_size
int cuadmm_eig_rank_mask(int32_t* mask, int64_t batch_size, int64_t mat_size, int64_t eig_rank) {
    return guarded([&] {
        CUADMM_REQUIRE(mask || batch_size * mat_size == 0, "mask is null");
        CUADMM_REQUIRE(batch_size >= 0 && mat_size >= 0 && eig_rank >= 0 && eig_rank <= mat_size, "bad sizes");
        for (int64_t i = 0; i < batch_size * mat_size; ++i) mask[i] = 0;
        for (int64_t i = 0; i < batch_size; ++i)
            for (int64_t j = 0; j < eig_rank; ++j) mask[i * mat_size + (mat_size - 1 - j)] = 1;
    });
}

int cuadmm_plan_set_warm_start(cuadmm_plan* plan, int enable) {
    return guarded([&] {
        CUADMM_REQUIRE(plan, "plan is null");
        if (plan->device < 0) return;
        plan->reset_warm_start();
        plan->warm_start = enable != 0 && plan->d_Q.n > 0;
    });
}

int cuadmm_plan_set_jacobi(cuadmm_plan* plan, double threshold, int max_sweeps) {
    return guarded([&] {
        CUADMM_REQUIRE(plan, "plan is null");
        CUADMM_REQUIRE(threshold > 0 && max_sweeps > 0, "threshold and max_sweeps must be positive");
        plan->threshold = threshold;
        plan->max_sweeps = max_sweeps;
    });
}

double cuadmm_plan_last_ms(const cuadmm_plan* plan) { return plan ? plan->last_ms : -1.0; }
int64_t cuadmm_plan_last_launches(const cuadmm_plan* plan) { return plan ? plan->last_launches : -1; }

int cuadmm_project_psd(cuadmm_plan* plan, const double* d_Xb, double* d_Xproj, void* stream) {
    return guarded([&] {
        CUADMM_REQUIRE(plan && d_Xb && d_Xproj, "null argument");
        DeviceGuard g(plan->device);
        plan->last_launches = plan->project(d_Xb, d_Xproj, (cudaStream_t)stream, nullptr, false);
    });
}

int cuadmm_project_epilogue(cuadmm_plan* plan, const double* d_Xb, double* d_Xproj, const double* d_X, const double* d_Rd1,
                            const double* d_C, double* d_S, double* d_SmC, const double* d_sig, void* stream) {
    return guarded([&] {
        CUADMM_REQUIRE(plan && d_Xb && d_Xproj && d_X && d_Rd1 && d_C && d_S && d_SmC && d_sig, "null argument");
        DeviceGuard g(plan->device);
        ProjEpilogue pe;
        pe.X = d_X; pe.Rd1 = d_Rd1; pe.Cd = d_C; pe.S = d_S; pe.SmC = d_SmC; pe.sig_ptr = d_sig;
        plan->last_launches = plan->project(d_Xb, d_Xproj, (cudaStream_t)stream, &pe, false);
    });
}

static void project_host_impl(cuadmm_plan* plan, const double* h_Xb, double* h_Xproj,
                              double* h_eig, int32_t* h_sweeps) {
    CUADMM_REQUIRE(plan && h_Xb && h_Xproj, "null argument");
    if (plan->device < 0) throw Error(CUADMM_ENODEVICE, "plan was built without a CUDA device; there is no CPU fallback");
    DeviceGuard g(plan->device);
    const int64_t L = plan->layout.vec_len;
    if (plan->d_in.n != L) { plan->d_in.alloc(L); plan->d_out.alloc(L); }
    plan->d_in.upload(h_Xb, L);
    CUADMM_CUDA(cudaEventRecord(plan->ev0, 0));
    plan->last_launches = plan->project(plan->d_in.p, plan->d_out.p, 0, nullptr, h_eig || h_sweeps);
    CUADMM_CUDA(cudaEventRecord(plan->ev1, 0));
    plan->d_out.download(h_Xproj, L);
    const BlockLayout& lay = plan->layout;
    std::vector<double> eig_s;     // typed plans: the 's' blocks' slots, expanded below
    if (h_eig) {
        if (lay.all_psd()) plan->d_eig.download(h_eig, plan->eig_len);
        else { eig_s.resize((size_t)plan->eig_len); plan->d_eig.download(eig_s.data(), plan->eig_len); }
    }
    if (h_sweeps) plan->d_sweeps.download(h_sweeps, (int64_t)plan->layout.blk.size());
    CUADMM_CUDA(cudaStreamSynchronize(0));
    if (h_eig && !lay.all_psd()) {
        // 'l' / 'u' blocks have no eigenvalues: NaN in their n slots (their sweep counts stay 0)
        int64_t o = 0, os = 0;
        for (size_t k = 0; k < lay.blk.size(); ++k) {
            const int64_t n = lay.blk[k];
            if (lay.types[k] == 's') { std::copy(eig_s.begin() + os, eig_s.begin() + os + n, h_eig + o); os += n; }
            else std::fill(h_eig + o, h_eig + o + n, std::numeric_limits<double>::quiet_NaN());
            o += n;
        }
    }
    float ms = 0.f;
    CUADMM_CUDA(cudaEventElapsedTime(&ms, plan->ev0, plan->ev1));
    plan->last_ms = ms;
    if (h_eig && plan->dense) {
        // The sign iteration of the large blocks (n > 168) yields the projection but no eigenvalues.  For this parity / debug
        // entry they come from the global-memory Jacobi kernel run on a shadow plan over those blocks (n <= 1024: beyond
        // that it is too slow to be useful and the slots stay NaN).  The solver never needs eigenvalues.
        const std::vector<int32_t>& blk = plan->layout.blk;
        std::vector<int64_t> which;
        for (size_t k = 0; k < blk.size(); ++k) if (lay.types[k] == 's' && blk[k] > 168 && blk[k] <= 1024) which.push_back((int64_t)k);
        if (!which.empty()) {
            std::vector<int32_t> sb;
            for (int64_t k : which) sb.push_back(blk[k]);
            if (!plan->eig_plan || plan->eig_plan->layout.blk != sb) {
                plan->eig_plan.reset(new cuadmm_plan());
                plan->eig_plan->layout.init(sb.data(), (int64_t)sb.size());
                plan->eig_plan->device = plan->device;
                plan->eig_plan->force_global = true;
                plan->eig_plan->build_device();
            }
            cuadmm_plan* E = plan->eig_plan.get();
            std::vector<double> xin((size_t)E->layout.vec_len), xout((size_t)E->layout.vec_len), ev((size_t)E->eig_len);
            for (size_t i = 0; i < which.size(); ++i)
                std::copy(h_Xb + plan->layout.svec_off[which[i]], h_Xb + plan->layout.svec_off[which[i] + 1], xin.begin() + E->layout.svec_off[i]);
            project_host_impl(E, xin.data(), xout.data(), ev.data(), nullptr);
            std::vector<int64_t> w_off(blk.size() + 1, 0);
            for (size_t k = 0; k < blk.size(); ++k) w_off[k + 1] = w_off[k] + blk[k];
            int64_t eo = 0;
            for (size_t i = 0; i < which.size(); ++i) {
                std::copy(ev.begin() + eo, ev.begin() + eo + sb[i], h_eig + w_off[which[i]]);
                eo += sb[i];
            }
        }
    }
    if (h_eig) {
        // ascending per block, like dsyevd / Xsyevd / syevj(sort=1)
        int64_t o = 0;
        for (size_t k = 0; k < plan->layout.blk.size(); ++k) {
            if (lay.types[k] == 's') std::sort(h_eig + o, h_eig + o + plan->layout.blk[k]);
            o += plan->layout.blk[k];
        }
    }
}

int cuadmm_project_psd_host(cuadmm_plan* plan, const double* h_Xb, double* h_Xproj) {
    return guarded([&] { project_host_impl(plan, h_Xb, h_Xproj, nullptr, nullptr); });
}

int cuadmm_project_psd_eig_host(cuadmm_plan* plan, const double* h_Xb, double* h_Xproj,
                                double* h_eigvals, int32_t* h_sweeps) {
    return guarded([&] { project_host_impl(plan, h_Xb, h_Xproj, h_eigvals, h_sweeps); });
}

int cuadmm_svec_to_smat(cuadmm_plan* plan, const double* d_svec, double* d_large_mat, double* d_small_mat, void* stream) {
    return guarded([&] {
        CUADMM_REQUIRE(plan && d_svec, "null argument");
        plan->layout.require_all_psd("cuadmm_svec_to_smat");
        if (plan->device < 0) throw Error(CUADMM_ENODEVICE, "host-only plan");
        DeviceGuard g(plan->device);
        const int nblk = (int)plan->layout.blk.size();
        if (nblk == 0) return;
        int nmax = *std::max_element(plan->layout.blk.begin(), plan->layout.blk.end());
        dim3 grid(nblk, std::min(std::max(nmax / 32, 1), 64));
        svec_to_smat_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(d_svec, d_large_mat, d_small_mat,
            plan->d_blk.p, plan->d_svec_off.p, plan->d_mat_off.p, plan->d_pool.p);
        CUADMM_CUDA(cudaGetLastError());
    });
}

int cuadmm_smat_to_svec(cuadmm_plan* plan, const double* d_large_mat, const double* d_small_mat, double* d_svec, void* stream) {
    return guarded([&] {
        CUADMM_REQUIRE(plan && d_svec, "null argument");
        plan->layout.require_all_psd("cuadmm_smat_to_svec");
        if (plan->device < 0) throw Error(CUADMM_ENODEVICE, "host-only plan");
        DeviceGuard g(plan->device);
        const int nblk = (int)plan->layout.blk.size();
        if (nblk == 0) return;
        int nmax = *std::max_element(plan->layout.blk.begin(), plan->layout.blk.end());
        dim3 grid(nblk, std::min(std::max(nmax / 32, 1), 64));
        smat_to_svec_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(d_large_mat, d_small_mat, d_svec,
            plan->d_blk.p, plan->d_svec_off.p, plan->d_mat_off.p, plan->d_pool.p);
        CUADMM_CUDA(cudaGetLastError());
    });
}

}  // extern "C"
