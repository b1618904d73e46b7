// dense.cu — dense FP64 kernels (column-major).  The GEMM runs on the FP64 tensor pipe through
// mma.sync.m8n8k4.f64 (tcgen05 has no f64 kind; DMMA via mma.sync is the FP64 tensor path on
// sm_100a), operands staged in shared memory.
#include "dense.h"
#include <stdio.h>
#include <stdlib.h>
#include <algorithm>

namespace cuadmm {

// ------------------------------------------------------------------------------------------
// GEMM: 64x64x16 CTA tile, 4 warps (2x2), each warp 32x32 = 4x4 m8n8k4 tiles
// ------------------------------------------------------------------------------------------
static constexpr int GB_M = 64, GB_N = 64, GB_K = 16, GB_PAD = 4;

__device__ __forceinline__ void dmma_m8n8k4(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

template <bool TA, bool TB>
__global__ void __launch_bounds__(128) dgemm_kernel(int64_t m, int64_t n, int64_t k, double alpha,
                                                    const double* __restrict__ A, int64_t lda,
                                                    const double* __restrict__ B, int64_t ldb,
                                                    double beta, double* C, int64_t ldc, int shape) {
    // shape 1: only the tiles on or below the diagonal are computed (symmetric rank-k updates whose consumer reads the
    // lower triangle); shape 2: op(B) is lower triangular, so output column tile n0 only needs k >= n0
    if (shape == 1 && (int64_t)blockIdx.y * GB_N > (int64_t)blockIdx.x * GB_M + (GB_M - 1)) return;
    __shared__ double As[2][GB_K][GB_M + GB_PAD];
    __shared__ double Bs[2][GB_K][GB_N + GB_PAD];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = (warp & 1) * 32, wn = (warp >> 1) * 32;
    const int64_t m0 = (int64_t)blockIdx.x * GB_M, n0 = (int64_t)blockIdx.y * GB_N;
    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }

    auto load_tiles = [&](int buf, int64_t k0) {
        // A tile: 64 (m) x 16 (k); op(A)(mm,kk) = TA ? A[kk + mm*lda] : A[mm + kk*lda]
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            const int e = tid + t * 128;
            int mm, kk;
            if (TA) { kk = e % GB_K; mm = e / GB_K; } else { mm = e % GB_M; kk = e / GB_M; }
            const int64_t gm = m0 + mm, gk = k0 + kk;
            double v = 0.0;
            if (gm < m && gk < k) v = TA ? A[gk + gm * lda] : A[gm + gk * lda];
            As[buf][kk][mm] = v;
        }
        // B tile: 16 (k) x 64 (n); op(B)(kk,nn) = TB ? B[nn + kk*ldb] : B[kk + nn*ldb]
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            const int e = tid + t * 128;
            int nn, kk;
            if (TB) { nn = e % GB_N; kk = e / GB_N; } else { kk = e % GB_K; nn = e / GB_K; }
            const int64_t gn = n0 + nn, gk = k0 + kk;
            double v = 0.0;
            if (gn < n && gk < k) v = TB ? B[gn + gk * ldb] : B[gk + gn * ldb];
            Bs[buf][kk][nn] = v;
        }
    };

    const int64_t nk = (k + GB_K - 1) / GB_K;
    const int64_t kt0 = (shape == 2) ? ((n0 / GB_K < nk) ? n0 / GB_K : nk) : 0;
    if (nk > kt0) load_tiles((int)(kt0 & 1), kt0 * GB_K);
    __syncthreads();
    for (int64_t kt = kt0; kt < nk; ++kt) {
        const int buf = (int)(kt & 1);
        if (kt + 1 < nk) load_tiles(buf ^ 1, (kt + 1) * GB_K);
#pragma unroll
        for (int kk = 0; kk < GB_K; kk += 4) {
            double a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = As[buf][kk + (lane & 3)][wm + i * 8 + (lane >> 2)];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = Bs[buf][kk + (lane & 3)][wn + j * 8 + (lane >> 2)];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) dmma_m8n8k4(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int64_t gm = m0 + wm + i * 8 + (lane >> 2);
                const int64_t gn = n0 + wn + j * 8 + (lane & 3) * 2 + h;
                if (gm < m && gn < n) {
                    double* c = C + gm + gn * ldc;
                    *c = (beta == 0.0) ? alpha * acc[i][j][h] : alpha * acc[i][j][h] + beta * (*c);
                }
            }
}

void dgemm(cudaStream_t st, bool transA, bool transB, int64_t m, int64_t n, int64_t k, double alpha,
           const double* A, int64_t lda, const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int shape) {
    if (m <= 0 || n <= 0) return;
    dim3 grid((unsigned)((m + GB_M - 1) / GB_M), (unsigned)((n + GB_N - 1) / GB_N));
    if (!transA && !transB) dgemm_kernel<false, false><<<grid, 128, 0, st>>>(m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, shape);
    else if (!transA && transB) dgemm_kernel<false, true><<<grid, 128, 0, st>>>(m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, shape);
    else if (transA && !transB) dgemm_kernel<true, false><<<grid, 128, 0, st>>>(m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, shape);
    else dgemm_kernel<true, true><<<grid, 128, 0, st>>>(m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, shape);
    CUADMM_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------
// blocked Cholesky (lower), nb = 64
// ------------------------------------------------------------------------------------------
static constexpr int NB = 64;

// factor one nb x nb diagonal block in shared memory, write L_jj back and its inverse to inv
__global__ void __launch_bounds__(256) potf2_inv_kernel(int nb, double* A, int64_t lda, double* inv, int* info, int blk_index, const double* pivot_floor) {
    extern __shared__ double potf2_smem[];
    double (*S)[NB + 1] = reinterpret_cast<double (*)[NB + 1]>(potf2_smem);
    double (*I)[NB + 1] = reinterpret_cast<double (*)[NB + 1]>(potf2_smem + NB * (NB + 1));
    __shared__ int bad;
    const int tid = threadIdx.x;
    if (tid == 0) bad = 0;
    for (int e = tid; e < nb * nb; e += 256) { const int i = e % nb, j = e / nb; S[i][j] = (i >= j) ? A[i + j * lda] : 0.0; }
    __syncthreads();
    for (int kk = 0; kk < nb; ++kk) {
        if (tid == 0) {
            const double d = S[kk][kk];
            // pivot floor: a pivot below pivot_floor[kk] marks a redundant direction (L_kk = +inf => x_k = 0)
            const double fl = pivot_floor ? pivot_floor[kk] : 0.0;
            if (!(d > fl)) { bad = 1; S[kk][kk] = INFINITY; } else S[kk][kk] = sqrt(d);
        }
        __syncthreads();
        const double dk = S[kk][kk];
        for (int i = kk + 1 + tid; i < nb; i += 256) S[i][kk] /= dk;
        __syncthreads();
        const int rem = nb - kk - 1;
        for (int e = tid; e < rem * rem; e += 256) {
            const int i = kk + 1 + e % rem, j = kk + 1 + e / rem;
            if (i >= j) S[i][j] -= S[i][kk] * S[j][kk];
        }
        __syncthreads();
    }
    // inverse by forward substitution: thread j solves L x = e_j
    if (tid < nb) {
        const int j = tid;
        for (int i = 0; i < nb; ++i) {
            double s = (i == j) ? 1.0 : 0.0;
            for (int t = j; t < i; ++t) s -= S[i][t] * I[t][j];
            I[i][j] = (i >= j) ? s / S[i][i] : 0.0;
        }
    }
    __syncthreads();
    for (int e = tid; e < nb * nb; e += 256) {
        const int i = e % nb, j = e / nb;
        if (i >= j) A[i + j * lda] = S[i][j];
        if (inv) inv[i + (int64_t)j * NB] = I[i][j];
    }
    if (tid == 0 && bad && info) atomicAdd(info, 1);
}

void potrf_lower(cudaStream_t st, int64_t n, double* A, int64_t lda, double* inv_diag, int* d_info, const double* pivot_floor) {
    DevBuf<double> tmp(std::max<int64_t>(n * NB, 1));
    DevBuf<double> inv_local;
    if (!inv_diag) { inv_local.alloc(std::max<int64_t>(n * NB, 1)); inv_diag = inv_local.p; }
    const size_t potf2_bytes = sizeof(double) * 2 * NB * (NB + 1);
    CUADMM_CUDA(cudaFuncSetAttribute((const void*)potf2_inv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)potf2_bytes));
    for (int64_t j = 0; j < n; j += NB) {
        const int nb = (int)std::min<int64_t>(NB, n - j);
        double* Ajj = A + j + j * lda;
        double* invj = inv_diag + j * NB;   // block j/NB stored as a 64-column-major tile
        potf2_inv_kernel<<<1, 256, potf2_bytes, st>>>(nb, Ajj, lda, invj, d_info, (int)(j / NB), pivot_floor ? pivot_floor + j : nullptr);
        const int64_t below = n - j - nb;
        if (below > 0) {
            double* Aij = A + (j + nb) + j * lda;
            // panel <- panel * L_jj^-T
            dgemm(st, false, true, below, nb, nb, 1.0, Aij, lda, invj, NB, 0.0, tmp.p, below);
            CUADMM_CUDA(cudaMemcpy2DAsync(Aij, sizeof(double) * lda, tmp.p, sizeof(double) * below,
                                          sizeof(double) * below, nb, cudaMemcpyDeviceToDevice, st));
            // trailing <- trailing - panel * panel^T
            double* A22 = A + (j + nb) + (j + nb) * lda;
            dgemm(st, false, true, below, below, nb, -1.0, Aij, lda, Aij, lda, 1.0, A22, lda, 1);   // lower tiles only
        }
    }
    CUADMM_CUDA(cudaGetLastError());
    CUADMM_CUDA(cudaStreamSynchronize(st));   // tmp is freed on return
}

__global__ void copy_inv_block_kernel(int nb, const double* __restrict__ inv, double* X, int64_t ldx) {
    for (int e = threadIdx.x; e < nb * nb; e += blockDim.x) {
        const int i = e % nb, j = e / nb;
        X[i + j * ldx] = inv[i + (int64_t)j * NB];
    }
}

void trtri_lower(cudaStream_t st, int64_t n, const double* L, int64_t ldl, const double* inv_diag, double* X, int64_t ldx) {
    CUADMM_CUDA(cudaMemset2DAsync(X, sizeof(double) * ldx, 0, sizeof(double) * n, n, st));
    DevBuf<double> T(std::max<int64_t>((int64_t)NB * n, 1));
    for (int64_t i = 0; i < n; i += NB) {
        const int nb = (int)std::min<int64_t>(NB, n - i);
        const double* invi = inv_diag + i * NB;
        copy_inv_block_kernel<<<1, 256, 0, st>>>(nb, invi, X + i + i * ldx, ldx);
        if (i > 0) {
            // T = L(i, 0:i) * X(0:i, 0:i) ; X(i, 0:i) = -inv_ii * T
            dgemm(st, false, false, nb, i, i, 1.0, L + i, ldl, X, ldx, 0.0, T.p, NB, 2);            // X(0:i, 0:i) is lower triangular
            dgemm(st, false, false, nb, i, nb, -1.0, invi, NB, T.p, NB, 0.0, X + i, ldx);
        }
    }
    CUADMM_CUDA(cudaGetLastError());
    CUADMM_CUDA(cudaStreamSynchronize(st));
}

// ------------------------------------------------------------------------------------------
// y-solve dense tail
// ------------------------------------------------------------------------------------------
__global__ void scatter_coo_kernel(int64_t nnz, const int32_t* __restrict__ r, const int32_t* __restrict__ c,
                                   const double* __restrict__ v, double* D, int64_t ld, int symmetric) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nnz) return;
    D[r[e] + (int64_t)c[e] * ld] = v[e];
    if (symmetric && r[e] != c[e]) D[c[e] + (int64_t)r[e] * ld] = v[e];
}

// which 64 x 64 tiles of P L P^T hold a non-zero (L column-major r x r, ipos[new] = old)
__global__ void tile_occupancy_kernel(int64_t r, int nt, const double* __restrict__ L, const int32_t* __restrict__ ipos,
                                      int* __restrict__ flags) {
    const int I = blockIdx.y, J = blockIdx.x;
    int any = 0;
    for (int e = threadIdx.x; e < 64 * 64; e += blockDim.x) {
        const int64_t i = (int64_t)I * 64 + e % 64, j = (int64_t)J * 64 + e / 64;
        if (i < r && j < r && L[ipos[i] + (int64_t)ipos[j] * r] != 0.0) any = 1;
    }
    if (__syncthreads_or(any) && threadIdx.x == 0) flags[I * nt + J] = 1;
}

void tile_occupancy(int64_t r, const double* L, const int32_t* ipos, std::vector<int>& flags) {
    cudaStream_t st = 0;
    const int nt = (int)((r + 63) / 64);
    DevBuf<int> d((int64_t)nt * nt);
    d.zero(st);
    tile_occupancy_kernel<<<dim3(nt, nt), 256, 0, st>>>(r, nt, L, ipos, d.p);
    CUADMM_CUDA(cudaGetLastError());
    flags.resize((size_t)nt * nt);
    d.download(flags.data(), (int64_t)flags.size(), st);
    CUADMM_CUDA(cudaStreamSynchronize(st));
}

// one CTA per tile: tile (I, J) of P L P^T (or of its transpose) -> out[dst + i * w + j], zeros outside the r x r matrix
__global__ void pack_tiles_kernel(int64_t r, const double* __restrict__ L, const int32_t* __restrict__ ipos, int transpose,
                                  const int64_t* __restrict__ tiles, double* __restrict__ out) {
    const int64_t* t = tiles + 4 * (int64_t)blockIdx.x;
    const int64_t I = t[0], J = t[1], dst = t[2], w = t[3];
    for (int e = threadIdx.x; e < 64 * 64; e += blockDim.x) {
        const int i = e / 64, j = e % 64;
        const int64_t a = I * 64 + i, b = J * 64 + j;
        double v = 0.0;
        if (a < r && b < r) v = transpose ? L[ipos[b] + (int64_t)ipos[a] * r] : L[ipos[a] + (int64_t)ipos[b] * r];
        out[dst + i * w + j] = v;
    }
}

void pack_tiles(int64_t r, const double* L, const int32_t* ipos, bool transpose, const std::vector<int64_t>& tiles, double* out) {
    cudaStream_t st = 0;
    const int64_t n = (int64_t)tiles.size() / 4;
    if (n == 0) return;
    DevBuf<int64_t> d;
    d.upload(tiles, st);
    pack_tiles_kernel<<<(unsigned)n, 256, 0, st>>>(r, L, ipos, transpose ? 1 : 0, d.p, out);
    CUADMM_CUDA(cudaGetLastError());
    CUADMM_CUDA(cudaStreamSynchronize(st));
}

void build_dense_tail(const SymCsc& C, const CholFactor& F, int64_t n_lead, int64_t r, DevBuf<double>& tail_inv,
                      int64_t* n_deficient) {
    cudaStream_t st = 0;
    // S <- M22 (both triangles)
    DevBuf<double> S(r * r);
    S.zero(st);
    {
        std::vector<int32_t> rr, cc; std::vector<double> vv;
        for (int64_t j = n_lead; j < n_lead + r; ++j)
            for (int64_t p = C.p[j]; p < C.p[j + 1]; ++p) { rr.push_back((int32_t)(C.i[p] - n_lead)); cc.push_back((int32_t)(j - n_lead)); vv.push_back(C.x[p]); }
        if (!vv.empty()) {
            DevBuf<int32_t> dr, dc; DevBuf<double> dv;
            dr.upload(rr, st); dc.upload(cc, st); dv.upload(vv, st);
            scatter_coo_kernel<<<(unsigned)((vv.size() + 255) / 256), 256, 0, st>>>((int64_t)vv.size(), dr.p, dc.p, dv.p, S.p, r, 1);
            CUADMM_CUDA(cudaStreamSynchronize(st));
        }
    }
    // S -= L21 L21^T, by chunks of the lead columns that reach into the tail
    {
        std::vector<int64_t> cols;
        for (int64_t j = 0; j < n_lead; ++j)
            if (F.Lp[j + 1] > F.Lp[j] + 1 && F.Li[F.Lp[j + 1] - 1] >= n_lead) cols.push_back(j);
        const int64_t budget = (int64_t)1 << 27;   // doubles per chunk (1 GiB)
        const int64_t cw = std::max<int64_t>(64, std::min<int64_t>((int64_t)cols.size(), budget / std::max<int64_t>(r, 1)));
        DevBuf<double> B(r * std::min<int64_t>(cw, std::max<int64_t>((int64_t)cols.size(), 1)));
        std::vector<int32_t> rr, cc; std::vector<double> vv;
        for (int64_t c0 = 0; c0 < (int64_t)cols.size(); c0 += cw) {
            const int64_t w = std::min<int64_t>(cw, (int64_t)cols.size() - c0);
            rr.clear(); cc.clear(); vv.clear();
            for (int64_t t = 0; t < w; ++t) {
                const int64_t j = cols[c0 + t];
                for (int64_t p = F.Lp[j + 1] - 1; p > F.Lp[j] && F.Li[p] >= n_lead; --p) {
                    rr.push_back((int32_t)(F.Li[p] - n_lead)); cc.push_back((int32_t)t); vv.push_back(F.Lx[p]);
                }
            }
            CUADMM_CUDA(cudaMemsetAsync(B.p, 0, sizeof(double) * (size_t)(r * w), st));
            DevBuf<int32_t> dr, dc; DevBuf<double> dv;
            dr.upload(rr, st); dc.upload(cc, st); dv.upload(vv, st);
            scatter_coo_kernel<<<(unsigned)((vv.size() + 255) / 256), 256, 0, st>>>((int64_t)vv.size(), dr.p, dc.p, dv.p, B.p, r, 0);
            dgemm(st, false, true, r, r, w, -1.0, B.p, r, B.p, r, 1.0, S.p, r, 1);                  // the factorisation reads the lower triangle
            CUADMM_CUDA(cudaStreamSynchronize(st));
        }
    }
    // S = L22 L22^T ; Linv = L22^-1
    DevBuf<double> inv_diag(std::max<int64_t>(r * NB, 1));
    DevBuf<int> info(1);
    info.zero(st);
    std::vector<double> h_floor(r, 0.0);
    for (int64_t j = n_lead; j < n_lead + r; ++j)
        for (int64_t p = C.p[j]; p < C.p[j + 1]; ++p) if (C.i[p] == j) h_floor[j - n_lead] = pivot_tol() * C.x[p];
    DevBuf<double> d_floor; d_floor.upload(h_floor, st);
    potrf_lower(st, r, S.p, r, inv_diag.p, info.p, d_floor.p);
    int h_info = 0;
    info.download(&h_info, 1, st);
    CUADMM_CUDA(cudaStreamSynchronize(st));
    if (n_deficient) *n_deficient = h_info;
    tail_inv.alloc(r * r);
    trtri_lower(st, r, S.p, r, inv_diag.p, tail_inv.p, r);
}

}  // namespace cuadmm
