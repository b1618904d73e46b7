// solver.cu — the sGS-ADMM iteration of the reference (SDPSolver::init / solve, src/solver.cu:27-822)
// on top of the device-resident hot path.  One iteration =
//   K1  rhsy = Rp/sig - A (S-C)                  SpMV(A)  + fused axpy            (:478-482)
//   K2  y = (A A^T)^-1 rhsy                      device triangular sweeps          (:487-500)
//   K3  Rd1 = A^T y - C ; Xb = X + sig Rd1       SpMV(At) + fused axpby/axpy       (:514-527)
//   K4  Xproj = Pi+(Xb) ; S ; SmC                fused Jacobi projection           (:531-675)
//   K5-K6 (sGS only) second rhsy / y             (:693-717)
//   K7  Rd = A^T y - C + S ; X += tau sig Rd     SpMV(At) + fused update + |Rd|^2, <C,X>   (:721-758)
//   K8  Rp = b - A X ; |normA Rp|^2 ; <b,y>      SpMV(A)  + fused reductions       (:764-777)
//   K9  residuals, sigma rule, history, stop     one tiny kernel, no host sync     (:772-810)
// The host only enqueues; it reads the state back when a log line is due (every 50/100 iterations,
// like the reference's printout) and finds out there whether the device-side stop test fired.
#include "solver.h"
#include <algorithm>
#include <chrono>
#include <cmath>
#include <string>
#include <string.h>
#include <stdlib.h>

namespace cuadmm {

void spmv_set_done_flag(cuadmm_spmv_s& A, const int* flag);

// ------------------------------------------------------------------------------------------
// small kernels
// ------------------------------------------------------------------------------------------
static constexpr int kEwThreads = 256;
static constexpr int64_t kHistRing = 4096;      // device history ring (entries per array)

// end of a grid-stride pair reduction of kEwThreads threads: warp shuffle tree, then thread 0 adds the warps in order
// and stores this CTA's pair at partial[2 * blockIdx.x]
__device__ __forceinline__ void store_cta_pair(double a0, double a1, double* partial) {
    __shared__ double red[2][kEwThreads / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { a0 += __shfl_xor_sync(0xffffffffu, a0, o); a1 += __shfl_xor_sync(0xffffffffu, a1, o); }
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = a0; red[1][threadIdx.x >> 5] = a1; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double s0 = 0.0, s1 = 0.0;
        for (int k = 0; k < kEwThreads / 32; ++k) { s0 += red[0][k]; s1 += red[1][k]; }
        partial[2 * blockIdx.x] = s0; partial[2 * blockIdx.x + 1] = s1;
    }
}

// one CTA of 256 threads: the pairwise sums of na pairs at pa and nb pairs at pb, in a fixed order
__device__ __forceinline__ void sum_pairs_256(const double* __restrict__ pa, int na, const double* __restrict__ pb, int nb,
                                              double out[4]) {
    __shared__ double sm[4][256];
    double v[4] = {};
    for (int i = threadIdx.x; i < na; i += 256) { v[0] += pa[2 * i]; v[1] += pa[2 * i + 1]; }
    for (int i = threadIdx.x; i < nb; i += 256) { v[2] += pb[2 * i]; v[3] += pb[2 * i + 1]; }
    for (int q = 0; q < 4; ++q) sm[q][threadIdx.x] = v[q];
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) for (int q = 0; q < 4; ++q) sm[q][threadIdx.x] += sm[q][threadIdx.x + o];
        __syncthreads();
    }
    for (int q = 0; q < 4; ++q) out[q] = sm[q][0];
}

// residuals and objectives (src/solver.cu:193-228, 772-790) from the sums |Rd|^2, <C, X>, |normA .* Rp|^2, <b, y>
struct Residuals { double errRp, errRd, pobj, dobj, maxfeas, relgap; };
__device__ __forceinline__ Residuals residuals(const DevState* st, const double s[4]) {
    Residuals r;
    r.errRp = st->bscale * sqrt(s[2]) / st->norm_borg;
    r.pobj = s[1] * st->objscale;
    r.errRd = st->Cscale * sqrt(s[0]) / st->norm_Corg;
    r.dobj = s[3] * st->objscale;
    r.maxfeas = fmax(r.errRp, r.errRd);
    r.relgap = fabs(r.pobj - r.dobj) / (1 + fabs(r.pobj) + fabs(r.dobj));
    return r;
}

// ADMM branch of step 4 (no second y-solve): Rd = Rd1 + S ; X += tau*sig*Rd ; partial sums
__global__ void __launch_bounds__(kEwThreads) x_update_kernel(int64_t n, const double* __restrict__ Rd1,
        const double* __restrict__ S, const double* __restrict__ Cd, double* Rd, double* X,
        const DevState* st, double* partial) {
    if (st->done) return;
    const double ts = st->tau * st->sig;
    double a0 = 0.0, a1 = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * kEwThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kEwThreads) {
        const double rd = Rd1[i] + S[i];
        Rd[i] = rd;
        const double xn = X[i] + ts * rd;
        X[i] = xn;
        a0 = fma(rd, rd, a0);
        a1 = fma(Cd[i], xn, a1);
    }
    store_cta_pair(a0, a1, partial);
}

// K9: fixed-order reduction of the per-CTA partials, then the reference's scalar logic
__global__ void __launch_bounds__(256) scalar_update_kernel(DevState* st, const double* __restrict__ part_rd, int n_rd,
        const double* __restrict__ part_rp, int n_rp, double* hist, int64_t hist_cap) {
    if (st->done) return;
    double s[4];
    sum_pairs_256(part_rd, n_rd, part_rp, n_rp, s);
    if (threadIdx.x != 0) return;
    const int iter = st->iter;
    const Residuals r = residuals(st, s);
    const double feasratio = st->ratioconst * r.errRp / r.errRd;
    if (feasratio < 1) st->prim_win += 1; else st->dual_win += 1;
    double sig = st->sig;
    if (((iter <= st->sig_update_threshold) && ((iter % st->sig_update_stage_1) == 1)) ||
        ((iter > st->sig_update_threshold) && ((iter % st->sig_update_stage_2) == 1))) {
        if (st->prim_win > 1.2 * st->dual_win) {
            st->prim_win = 0;
            sig = fmin(st->sigmax, sig * st->sigscale);
        } else if (st->dual_win > 1.2 * st->prim_win) {
            st->dual_win = 0;
            sig = fmax(st->sigmin, sig / st->sigscale);
        }
    }
    st->sig = sig;
    st->errRp = r.errRp; st->errRd = r.errRd; st->pobj = r.pobj; st->dobj = r.dobj;
    st->maxfeas = r.maxfeas; st->relgap = r.relgap; st->feasratio = feasratio;
    {
        const int64_t k = (int64_t)(iter - 1) % hist_cap;      // ring: the host drains it at every log boundary
        hist[0 * hist_cap + k] = r.pobj;  hist[1 * hist_cap + k] = r.dobj;
        hist[2 * hist_cap + k] = r.errRp; hist[3 * hist_cap + k] = r.errRd;
        hist[4 * hist_cap + k] = r.relgap; hist[5 * hist_cap + k] = sig;
        hist[6 * hist_cap + k] = st->bscale; hist[7 * hist_cap + k] = st->Cscale;
    }
    const int next = iter + 1;
    st->iter = next;
    double tau = (next < st->switch_admm) ? 1.95 : 1.618;
    if (r.errRd < st->stop_tol) tau = fmax(1.618, tau / 1.1);
    st->tau = tau;
    // stop test that the reference evaluates at the top of iteration `next`
    if (fmax(r.maxfeas, r.relgap) < st->stop_tol) { st->done = 1; st->stop_reason = 1; }
    if (next > st->max_iter) { st->done = 1; st->stop_reason = 2; }
}

// iter == switch_admm (src/solver.cu:681-690)
__global__ void switch_kernel(DevState* st) {
    if (st->done) return;
    st->sig_update_stage_2 = st->sig_update_stage_2 / 2;
    st->sigscale = st->sigscale * 1.23;
    st->sgs_KKT = fmax(st->maxfeas, st->relgap);
    st->best_KKT = st->sgs_KKT;
}

// iter > switch_admm (src/solver.cu:732-741): decide, then copy
__global__ void best_decide_kernel(DevState* st) {
    if (st->done) { st->pad_ = 0; return; }
    const double cur = fmax(st->maxfeas, st->relgap);
    if (st->best_KKT > cur) { st->best_KKT = cur; st->pad_ = 1; } else st->pad_ = 0;
}
__global__ void best_copy_kernel(const DevState* st, int64_t n, const double* __restrict__ src, double* dst) {
    if (!st->pad_) return;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) dst[i] = src[i];
}

__global__ void scale_kernel(int64_t n, double* x, double s) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) x[i] *= s;
}
// y <- y ./ normA * s   (dense_vector_div_dense_vector_mul_scalar)  or  y <- y .* normA * s
__global__ void scale_vec_kernel(int64_t n, double* y, const double* __restrict__ d, double s, int divide) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        y[i] = divide ? y[i] / d[i] * s : y[i] * d[i] * s;
}
__global__ void sub_kernel(int64_t n, const double* __restrict__ a, const double* __restrict__ b, double* out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = a[i] - b[i];
}

// K1: rhsy = Rp / sig + buf   (buf = -A (S-C), summed over the ranks when sharded)
__global__ void rhsy_kernel(int64_t m, const double* __restrict__ Rp, const double* __restrict__ buf, double* rhsy, const DevState* st) {
    if (st->done) return;
    const double sig = st->sig;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) rhsy[i] = Rp[i] / sig + buf[i];
}

// ---- update_data: new b and C on the device
// triplets -> zeroed dense vector with init's rule for repeated indices (the last triplet wins):
// pass 1 marks the last triplet of every entry (win starts at -1), pass 2 stores only that one
__global__ void triplet_mark_kernel(int32_t nnz, const int32_t* __restrict__ idx, int32_t* win) {
    for (int32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < nnz; k += gridDim.x * blockDim.x) atomicMax(win + idx[k], k);
}
__global__ void triplet_store_kernel(int32_t nnz, const int32_t* __restrict__ idx, const double* __restrict__ val,
                                     const int32_t* __restrict__ win, double* out) {
    for (int32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < nnz; k += gridDim.x * blockDim.x)
        if (win[idx[k]] == k) out[idx[k]] = val[k];
}
// per-CTA partial pair (sum x^2, sum (x ./ d)^2), the second 0 when d is null; fixed tree inside the CTA
__global__ void __launch_bounds__(kEwThreads) sumsq_kernel(int64_t n, const double* __restrict__ x, const double* __restrict__ d,
                                                           double* partial) {
    double a0 = 0.0, a1 = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * kEwThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kEwThreads) {
        const double v = x[i];
        a0 = fma(v, v, a0);
        if (d) { const double t = v / d[i]; a1 = fma(t, t, a1); }
    }
    store_cta_pair(a0, a1, partial);
}
// the scaling constants (src/solver.cu:113-191): part_b pairs (|b|^2, |b ./ normA|^2), part_c pairs (|C|^2, 0)
__global__ void __launch_bounds__(256) data_scales_kernel(DevState* st, const double* __restrict__ part_b, int n_b,
                                                          const double* __restrict__ part_c, int n_c) {
    double s[4];
    sum_pairs_256(part_b, n_b, part_c, n_c, s);
    if (threadIdx.x != 0) return;
    const double nC = sqrt(s[2]);
    st->norm_borg = 1 + sqrt(s[0]);
    st->bscale = 1 + sqrt(s[1]);
    st->norm_Corg = 1 + nC;
    st->Cscale = 1 + nC;
    st->objscale = st->bscale * st->Cscale;
}
// the initial residuals and objectives (src/solver.cu:193-228) from the partials of Rd (|Rd|^2, <C, X>) and Rp
// (|normA .* Rp|^2, <b, y>), in scalar_update_kernel's order
__global__ void __launch_bounds__(256) data_residuals_kernel(DevState* st, const double* __restrict__ part_rd, int n_rd,
                                                             const double* __restrict__ part_rp, int n_rp) {
    double s[4];
    sum_pairs_256(part_rd, n_rd, part_rp, n_rp, s);
    if (threadIdx.x != 0) return;
    const Residuals r = residuals(st, s);
    st->errRp = r.errRp; st->errRd = r.errRd; st->pobj = r.pobj; st->dobj = r.dobj;
    st->maxfeas = r.maxfeas; st->relgap = r.relgap;
}

static int ew_grid(int64_t n, int device) {
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    return (int)std::max<int64_t>(1, std::min<int64_t>((n + kEwThreads - 1) / kEwThreads, (int64_t)sms * 8));
}
}  // namespace cuadmm

using namespace cuadmm;

cuadmm_solver::~cuadmm_solver() {
    cudaSetDevice(device);
    delete A; delete At; delete ys;
    if (h_st) cudaFreeHost(h_st);
    if (ev_start) cudaEventDestroy(ev_start);
    if (ev_now) cudaEventDestroy(ev_now);
    for (auto e : prof_ev) cudaEventDestroy(e);
    if (graph_sgs) cudaGraphExecDestroy(graph_sgs);
    if (graph_admm) cudaGraphExecDestroy(graph_admm);
    if (stream) cudaStreamDestroy(stream);
}

void cuadmm_solver::init(int /*eig_stream_num_per_gpu*/, int /*cpu_eig_thread_num*/, int64_t vec_len_, int64_t con_num_,
                         const int32_t* At_col_ptrs, const int32_t* At_row_ids, const double* At_vals, int64_t At_nnz,
                         const int32_t* b_idx, const double* b_val, int64_t b_nnz,
                         const int32_t* C_idx, const double* C_val, int64_t C_nnz,
                         const int32_t* blk, int64_t mat_num, const double* X0, const double* y0, const double* S0, double sig) {
    CUADMM_REQUIRE(!initialised, "solver already initialised (one instance per problem, like SDPSolver)");
    CUADMM_REQUIRE(vec_len_ >= 0 && con_num_ >= 0 && At_nnz >= 0, "negative dimension");
    CUADMM_REQUIRE(At_col_ptrs && blk, "null argument");
    CUADMM_REQUIRE(At_col_ptrs[0] == 0 && At_col_ptrs[con_num_] == At_nnz, "At_csc_col_ptrs does not span At_nnz");
    vec_len = vec_len_; con_num = con_num_;
    check_data(b_idx, b_val, b_nnz, C_idx, C_val, C_nnz);
    int cnt = 0;
    if (cudaGetDeviceCount(&cnt) != cudaSuccess || cnt == 0) {
        cudaGetLastError();
        throw Error(CUADMM_ENODEVICE, "no CUDA device available; the solver has no CPU fallback");
    }
    // device: cuadmm_solver_set_device, else CUADMM_DEVICE, else the calling thread's current device
    if (!device_set) {
        if (const char* e = getenv("CUADMM_DEVICE")) device = atoi(e);
        else { int cur = 0; if (cudaGetDevice(&cur) == cudaSuccess) device = cur; else cudaGetLastError(); }
    }
    if (const char* e = getenv("CUADMM_NO_GRAPH")) use_graphs = atoi(e) == 0;
    CUADMM_REQUIRE(device >= 0 && device < cnt, "device index out of range");
    CUADMM_CUDA(cudaSetDevice(device));
    CUADMM_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    CUADMM_CUDA(cudaEventCreate(&ev_start));
    CUADMM_CUDA(cudaEventCreate(&ev_now));
    CUADMM_CUDA(cudaEventRecord(ev_start, stream));     // the reference starts its clock in init
    const auto t0 = std::chrono::steady_clock::now();

    // ---- block plan
    {
        // block cones (cuadmm_solver_set_block_types; none given: all 's'); only the plan looks at them
        CUADMM_REQUIRE(blk_types.empty() || (int64_t)blk_types.size() == mat_num, "block types were set for a different block count");
        BlockLayout full_layout;
        full_layout.init(blk, mat_num, blk_types.empty() ? nullptr : blk_types.data());   // checks sizes and letters
        CUADMM_REQUIRE(full_layout.vec_len == vec_len, "vec_len does not match the block sizes");
        shard.build(full_layout, world, rank);      // world == 1: everything is local
        nloc = shard.vec_len_local;
        plan.reset(new cuadmm_plan());
        plan->layout.init(shard.local_blk.data(), (int64_t)shard.local_blk.size(), shard.local_types.data());
        plan->device = device;
        plan->build_device();
        if (world > 1) {
            d_loc2glob.upload(shard.loc2glob);
        }
    }
    // ---- A: normalise the constraints (get_normA, src/solver.cu:79-80), same arithmetic
    std::vector<double> vals(At_vals, At_vals + At_nnz);
    h_normA.assign(con_num, 1.0);
    for (int64_t p = 0; p < At_nnz; ++p) CUADMM_REQUIRE(At_row_ids[p] >= 0 && At_row_ids[p] < vec_len, "At row index out of range");
    for (int64_t i = 0; i < con_num; ++i) {
        double norm = 0.0;
        for (int p = At_col_ptrs[i]; p < At_col_ptrs[i + 1]; ++p) norm += vals[p] * vals[p];
        norm = std::max(1.0, std::sqrt(norm));
        h_normA[i] = norm;
        for (int p = At_col_ptrs[i]; p < At_col_ptrs[i + 1]; ++p) vals[p] /= norm;
    }
    // A in CSR is the CSC of At as given; At in CSR by a counting-sort transpose (csr2csc in the reference)
    {
        // this rank's column slice A[:, I_g] (all of A on one GPU)
        std::vector<int32_t> l_cp, l_ri; std::vector<double> l_v;
        const int32_t* cp = At_col_ptrs; const int32_t* ri = At_row_ids; const double* vv = vals.data();
        int64_t l_nnz = At_nnz;
        if (world > 1) {
            shard.slice_csc(con_num, At_col_ptrs, At_row_ids, vals.data(), l_cp, l_ri, l_v);
            l_ri.push_back(0); l_v.push_back(0.0);   // keep data() valid when the slice is empty
            cp = l_cp.data(); ri = l_ri.data(); vv = l_v.data(); l_nnz = l_cp[con_num];
        }
        A = spmv_create(con_num, nloc, l_nnz, cp, ri, vv, device);
        std::vector<int32_t> t_rp(nloc + 1), t_ci(std::max<int64_t>(l_nnz, 1));
        std::vector<double> t_v(std::max<int64_t>(l_nnz, 1));
        if (cuadmm_csc_to_csr_host(nloc, con_num, l_nnz, cp, ri, vv, t_rp.data(), t_ci.data(), t_v.data()) != 0)
            throw Error(CUADMM_EINVAL, cuadmm_last_error());
        At = spmv_create(nloc, con_num, l_nnz, t_rp.data(), t_ci.data(), t_v.data(), device);
    }
    // ---- A A^T factorisation (src/solver.cu:91-110), eps = 1e-15
    ys = ysolve_create(con_num, vec_len, At_nnz, At_col_ptrs, At_row_ids, vals.data(), 1e-15, device);
    if (world > 1) {
        // peer arena: staging for the slice reduction, the replicated m-vectors the peers store into (asmc, Rp, y,
        // the y-solve's x and dense-tail vector) and a full-length svec vector for get_X / get_S
        CUADMM_REQUIRE(con_num < (int64_t)0xffffffffll, "sharded solver: con_num exceeds 32 bits");
        slice = (((con_num + world - 1) / world) + 1) & ~(int64_t)1;
        const int64_t mm = std::max<int64_t>(con_num, 1);
        const size_t need = sizeof(double) * (size_t)(world * slice + 4 * mm + std::max<int64_t>(ys->n_tail, 1) + std::max<int64_t>(vec_len, 1)) + 16 * 256;
        peer.reset(new PeerComm());
        peer->init(rank, world, job_id, device, need);
        const size_t o_stage = peer->alloc(sizeof(double) * world * slice);
        const size_t o_asmc = peer->alloc(sizeof(double) * mm), o_Rp = peer->alloc(sizeof(double) * mm), o_y = peer->alloc(sizeof(double) * mm);
        const size_t o_x = peer->alloc(sizeof(double) * mm), o_tmp = peer->alloc(sizeof(double) * std::max<int64_t>(ys->n_tail, 1));
        const size_t o_full = peer->alloc(sizeof(double) * std::max<int64_t>(vec_len, 1));
        stage = peer->local<double>(o_stage);
        p_stage = peer->ptrs(o_stage); p_asmc = peer->ptrs(o_asmc); p_Rp = peer->ptrs(o_Rp); p_full = peer->ptrs(o_full);
        asmc.adopt(peer->local<double>(o_asmc), mm); Rp.adopt(peer->local<double>(o_Rp), mm); y.adopt(peer->local<double>(o_y), mm);
        full_buf.adopt(peer->local<double>(o_full), std::max<int64_t>(vec_len, 1));
        ys->enable_peer(peer.get(), o_tmp, o_x);
        cta_part.alloc(2 * (int64_t)peer_reduce_grid(*peer, slice) + 2);
    }

    // ---- device vectors
    auto alloc = [&](DevBuf<double>& d, int64_t len) {
        if (d.owned || !d.p) d.alloc(std::max<int64_t>(len, 1));     // views of the peer arena are kept
    };
    alloc(X, nloc); alloc(S, nloc); alloc(y, con_num); alloc(Rp, con_num); alloc(SmC, nloc); alloc(Cd, nloc); alloc(bd, con_num);
    alloc(normA, con_num); alloc(Rd1, nloc); alloc(Rd, nloc); alloc(Xb, nloc); alloc(Xproj, nloc); alloc(rhsy, con_num); alloc(asmc, con_num);
    normA.upload(h_normA.data(), con_num, stream);
    Rd1.zero(stream); Rd.zero(stream);
    nA_blocks = spmv_grid(*A); nAt_blocks = spmv_grid(*At); nE_blocks = ew_grid(std::max(nloc, con_num), device);
    partial.alloc(2 * (int64_t)(std::max(nAt_blocks, nE_blocks) + std::max(nA_blocks, nE_blocks)) + 4);
    partial.zero(stream);
    st.alloc(1);
    CUADMM_CUDA(cudaMallocHost((void**)&h_st, sizeof(DevState)));
    const int* done_ptr = &st.p->done;
    spmv_set_done_flag(*A, done_ptr);
    spmv_set_done_flag(*At, done_ptr);
    ys->done_flag = done_ptr;
    plan->done_flag = done_ptr;

    // ---- b, C, the scaling, the start point and the initial residuals (src/solver.cu:113-228): the path of
    // update_data with the iterate kept, from X0, y0, S0 (zero where not given)
    X.zero(stream); y.zero(stream); S.zero(stream);
    set_iterate(X0, y0, S0);
    load_data(b_idx, b_val, b_nnz, C_idx, C_val, C_nnz, true, sig);
    // the staging buffers are only needed again by update_data
    upd_idx.release(); upd_win.release(); upd_val.release(); upd_part.release(); upd_zero.release(); upd_full.release();
    init_time = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    initialised = true;
}

// K1: rhsy = Rp/sig - A(S-C).  The product asmc = -A(S-C) is kept: in an sGS iteration K5 computes it for
// the NEW S, which is exactly what K1 of the next iteration needs (S does not change in between), so that
// K1 is then only the vector update — one SpMV (and, multi-GPU, one reduction over the ranks) less per sGS iteration
// than the reference's loop (src/solver.cu:478-482 recomputes it).  Multi-GPU: partial -A_g (S-C)_g, summed over ranks.
void cuadmm_solver::enqueue_k1(bool asmc_cached) {
    if (!asmc_cached) {
        if (world == 1) { SpmvEpilogue e; spmv_launch(*A, -1.0, SmC.p, 0.0, asmc.p, e, stream); ++launches; }
        else reduce_partial_A(false, SmC.p, -1.0, nullptr, 0);
    }
    rhsy_kernel<<<ew_grid(con_num, device), 256, 0, stream>>>(con_num, Rp.p, asmc.p, rhsy.p, st.p); ++launches;
}

// Steps 1 .. 5 of iteration `iter` (src/solver.cu:469-799); every kernel is a no-op once st->done
void cuadmm_solver::enqueue_iteration(int iter, int switch_admm, bool prof) {
    const double* scal = &st.p->sig;
    SpmvEpilogue e;
    // profile mode: 6 events per iteration bracket the y-solves and the projection stage
    auto mark = [&](int k) {
        if (!prof) return;
        cudaEvent_t ev;
        CUADMM_CUDA(cudaEventCreate(&ev));
        CUADMM_CUDA(cudaEventRecord(ev, stream));
        prof_ev.push_back(ev);
        prof_tag.push_back(k);
    };
    ys->prof_ev = prof ? &prof_ev : nullptr;       // the y-solve brackets its dense-tail stage (tags 20 / 21)
    ys->prof_tag = prof ? &prof_tag : nullptr;
    enqueue_k1(asmc_valid);
    // K2
    mark(0);
    ys->solve(rhsy.p, y.p, stream); launches += ys->launches_per_solve;
    mark(1);
    // K3
    e = SpmvEpilogue(); e.mode = 2; e.aux1 = Cd.p; e.aux2 = X.p; e.out2 = Xb.p; e.scal = scal;
    spmv_launch(*At, 1.0, y.p, 0.0, Rd1.p, e, stream); ++launches;
    // K4
    ProjEpilogue pe;
    pe.X = X.p; pe.Rd1 = Rd1.p; pe.Cd = Cd.p; pe.S = S.p; pe.SmC = SmC.p; pe.sig_ptr = scal;
    mark(2);
    launches += plan->project(Xb.p, Xproj.p, stream, &pe, false);
    mark(3);
    if (iter == switch_admm) {
        switch_kernel<<<1, 1, 0, stream>>>(st.p); ++launches;
        CUADMM_CUDA(cudaMemcpyAsync(X_best.p, X.p, sizeof(double) * nloc, cudaMemcpyDeviceToDevice, stream));
        CUADMM_CUDA(cudaMemcpyAsync(y_best.p, y.p, sizeof(double) * con_num, cudaMemcpyDeviceToDevice, stream));
        CUADMM_CUDA(cudaMemcpyAsync(S_best.p, S.p, sizeof(double) * nloc, cudaMemcpyDeviceToDevice, stream));
    }
    double* part_rd = partial.p;
    double* part_rp = partial.p + 2 * (int64_t)std::max(nAt_blocks, nE_blocks);
    int n_rd = 0;
    if (iter < switch_admm) {
        // K5-K7: the sGS second half-step
        mark(6);
        enqueue_k1(false);
        mark(7);
        mark(4);
        ys->solve(rhsy.p, y.p, stream); launches += ys->launches_per_solve;
        mark(5);
        e = SpmvEpilogue(); e.mode = 3; e.aux1 = Cd.p; e.aux2 = S.p; e.out2 = X.p; e.scal = scal; e.partial = part_rd;
        spmv_launch(*At, 1.0, y.p, 0.0, Rd.p, e, stream); ++launches;
        n_rd = nAt_blocks;
    } else {
        if (iter > switch_admm) {
            const int g = ew_grid(nloc, device);
            best_decide_kernel<<<1, 1, 0, stream>>>(st.p);
            best_copy_kernel<<<g, 256, 0, stream>>>(st.p, nloc, X.p, X_best.p);
            best_copy_kernel<<<g, 256, 0, stream>>>(st.p, con_num, y.p, y_best.p);
            best_copy_kernel<<<g, 256, 0, stream>>>(st.p, nloc, S.p, S_best.p);
            launches += 4;
        }
        mark(4); mark(5);
        x_update_kernel<<<nE_blocks, kEwThreads, 0, stream>>>(nloc, Rd1.p, S.p, Cd.p, Rd.p, X.p, st.p, part_rd); ++launches;
        n_rd = nE_blocks;
    }
    // K8  (multi-GPU: the two local sums of K7 ride the reduction of the partial A_g X_g)
    mark(8);
    if (world == 1) {
        e = SpmvEpilogue(); e.mode = 4; e.aux1 = bd.p; e.aux2 = normA.p; e.aux3 = y.p; e.partial = part_rp;
        spmv_launch(*A, 1.0, X.p, 0.0, Rp.p, e, stream); ++launches;
    } else {
        reduce_partial_A(true, X.p, 1.0, part_rd, n_rd);
    }
    // K9
    const ScalarPartials sp = scalar_partials(part_rd, n_rd, part_rp);
    scalar_update_kernel<<<1, 256, 0, stream>>>(st.p, sp.rd, sp.n_rd, sp.rp, sp.n_rp, hist.p, hist_cap); ++launches;
    mark(9);
    ys->prof_ev = nullptr; ys->prof_tag = nullptr;
    asmc_valid = iter < switch_admm;     // K5 ran: asmc holds -A(S-C) of the S this iteration ends with
    CUADMM_CUDA(cudaGetLastError());
}

// One iteration = one CUDA-graph launch (the kernel sequence does not depend on the iteration index
// except at iter == switch_admm, which is enqueued directly).  Launch-bound problems (ros_2000: ~15
// kernels of a few microseconds each) otherwise spend more time in the driver than on the GPU.
void cuadmm_solver::launch_iteration(int iter, int switch_admm, bool prof) {
    const bool sgs = iter < switch_admm;
    // the sGS graph is the steady-state sequence (K1 from the cached product), the ADMM graph recomputes it;
    // an iteration that starts in the other cache state is enqueued directly
    if (prof || !use_graphs || iter == switch_admm || sgs != asmc_valid) { enqueue_iteration(iter, switch_admm, prof); return; }
    cudaGraphExec_t& exec = sgs ? graph_sgs : graph_admm;
    int64_t& nl = sgs ? graph_launches_sgs : graph_launches_admm;
    if (!exec) {
        const int64_t before = launches;
        cudaGraph_t graph = nullptr;
        CUADMM_CUDA(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
        try {
            enqueue_iteration(iter, switch_admm, false);
        } catch (...) {
            cudaStreamEndCapture(stream, &graph);
            if (graph) cudaGraphDestroy(graph);
            throw;
        }
        CUADMM_CUDA(cudaStreamEndCapture(stream, &graph));
        CUADMM_CUDA(cudaGraphInstantiate(&exec, graph, 0));
        CUADMM_CUDA(cudaGraphDestroy(graph));
        nl = launches - before;
        launches = before;
    }
    CUADMM_CUDA(cudaGraphLaunch(exec, stream));
    launches += nl;
    asmc_valid = sgs;
}

// Sharded solver: sum over ranks of the partial products alpha * A[:, I_g] x_g.
//   for_rp == false:  asmc = sum                                     (K1 / K5)
//   for_rp == true :  Rp = b - sum, residual scalars for K9          (K8)
// The SpMV stores every partial row into the staging area of the rank that reduces it (mode 5), peer_reduce_kernel
// sums its slice, applies the consumer and stores the result into every rank's copy.
void cuadmm_solver::reduce_partial_A(bool for_rp, const double* x_local, double alpha, const double* part_rd, int n_rd) {
    SpmvEpilogue e;
    e.mode = 5; e.slice = (unsigned)slice; e.rank = rank;
    for (int q = 0; q < world; ++q) e.push[q] = p_stage.p[q];
    spmv_launch(*A, alpha, x_local, 0.0, stage, e, stream);
    peer_reduce_launch(*peer, for_rp ? 1 : 0, con_num, slice, stage, for_rp ? p_Rp : p_asmc, bd.p, normA.p, y.p, part_rd, n_rd,
                       cta_part.p, &st.p->done, stream);
    launches += 2;
}

// Partial sums (|Rd|^2, <C, X>) and (|normA .* Rp|^2, <b, y>) for the one-CTA consumers of K7 / K8
// (scalar_update_kernel, data_residuals_kernel): this GPU's per-CTA partials, or, sharded, the per-rank scalars of the
// peer scalar board, which every rank adds in rank order, so that the state is bit-identical on all ranks.
cuadmm_solver::ScalarPartials cuadmm_solver::scalar_partials(const double* part_rd, int n_rd, const double* part_rp) const {
    if (world == 1) return {part_rd, n_rd, part_rp, nA_blocks};
    return {peer->local<double>(peer->off_scal_rd), world, peer->local<double>(peer->off_scal_rp), world};
}

// what the reference still executes at the top of the iteration in which it breaks
// (step 1 and step 2a, src/solver.cu:478-528): y is overwritten by the next half-step.
void cuadmm_solver::enqueue_half_step() {
    enqueue_k1(asmc_valid);
    ys->solve(rhsy.p, y.p, stream); launches += ys->launches_per_solve;
}

void cuadmm_solver::run_iterations(int n_iters, bool sgs, bool profile_, double out_ms[8]) {
    CUADMM_REQUIRE(initialised && hist.n > 0, "run_iterations() needs init() and one solve() first");
    CUADMM_CUDA(cudaSetDevice(device));
    // disable the stop test, keep the reference's sigma cadence running
    CUADMM_CUDA(cudaMemcpyAsync(h_st, st.p, sizeof(DevState), cudaMemcpyDeviceToHost, stream));
    CUADMM_CUDA(cudaStreamSynchronize(stream));
    const int first = h_st->iter;
    h_st->done = 0; h_st->stop_tol = -1.0; h_st->max_iter = 0x7fffffff;
    const int sw = sgs ? 0x7fffffff : 0;
    h_st->switch_admm = sw;
    h_st->tau = sgs ? 1.95 : 1.618;
    CUADMM_CUDA(cudaMemcpyAsync(st.p, h_st, sizeof(DevState), cudaMemcpyHostToDevice, stream));
    if (!sgs && X_best.n < std::max<int64_t>(nloc, 1)) {      // same size rule as solve(); the ADMM graph bakes these pointers
        X_best.alloc(std::max<int64_t>(nloc, 1)); y_best.alloc(std::max<int64_t>(con_num, 1)); S_best.alloc(std::max<int64_t>(nloc, 1));
        if (graph_admm) { cudaGraphExecDestroy(graph_admm); graph_admm = nullptr; }
    }
    for (auto e : prof_ev) cudaEventDestroy(e);
    prof_ev.clear(); prof_tag.clear();
    cudaEvent_t e0, e1;
    CUADMM_CUDA(cudaEventCreate(&e0)); CUADMM_CUDA(cudaEventCreate(&e1));
    CUADMM_CUDA(cudaEventRecord(e0, stream));
    for (int k = 0; k < n_iters; ++k) launch_iteration(first + k, sw, profile_);
    CUADMM_CUDA(cudaEventRecord(e1, stream));
    CUADMM_CUDA(cudaStreamSynchronize(stream));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    out_ms[0] = ms;
    for (int k = 1; k < 8; ++k) out_ms[k] = 0.0;
    if (profile_) {
        // intervals between an event tagged `a` and the next one tagged `b`
        auto span = [&](int a, int b) {
            double tot = 0.0;
            for (size_t i = 0; i < prof_ev.size(); ++i) {
                if (prof_tag[i] != a) continue;
                for (size_t j = i + 1; j < prof_ev.size(); ++j)
                    if (prof_tag[j] == b) { float t = 0.f; cudaEventElapsedTime(&t, prof_ev[i], prof_ev[j]); tot += t; break; }
            }
            return tot;
        };
        out_ms[1] = span(2, 3);
        out_ms[2] = span(0, 1) + (sgs ? span(4, 5) : 0.0);
        out_ms[3] = out_ms[0] - out_ms[1] - out_ms[2];
        out_ms[4] = span(6, 7);       // K5: A (S - C) (+ reduction over ranks) + rhsy
        out_ms[5] = span(8, 9);       // K8: A X (+ reduction over ranks) + scalar update
        out_ms[6] = span(20, 21);     // dense-tail GEMVs of all y-solves
        for (auto e : prof_ev) cudaEventDestroy(e);
        prof_ev.clear(); prof_tag.clear();
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    h_st->done = 1;
    CUADMM_CUDA(cudaMemcpyAsync(&st.p->done, &h_st->done, sizeof(int), cudaMemcpyHostToDevice, stream));
    CUADMM_CUDA(cudaStreamSynchronize(stream));
    if (peer) peer->check(stream);
}

// full-length X / S on every rank, gathered by owner: every rank stores its owned ranges into every rank's
// full-length vector (peer memory)
void cuadmm_solver::gather_full(const DevBuf<double>& local, double* h_full) {
    CUADMM_REQUIRE(initialised && h_full, "solver not initialised");
    CUADMM_CUDA(cudaSetDevice(device));
    peer_scatter_full_launch(*peer, nloc, local.p, d_loc2glob.p, p_full, stream);
    full_buf.download(h_full, vec_len, stream);
    peer->check(stream);
}

static bool is_log_iter(int iter) { return (iter <= 200 && iter % 50 == 1) || (iter > 200 && iter % 100 == 1); }

void cuadmm_solver::solve(int max_iter, double stop_tol, int sig_update_threshold, int sig_update_stage_1,
                          int sig_update_stage_2, int switch_admm, double sigscale, bool if_first) {
    CUADMM_REQUIRE(initialised, "solve() before init()");
    CUADMM_REQUIRE(max_iter >= 0, "max_iter < 0");
    CUADMM_REQUIRE(sig_update_stage_1 >= 1 && sig_update_stage_2 >= 1, "sig_update_stage must be >= 1");
    CUADMM_CUDA(cudaSetDevice(device));
    const auto t0 = std::chrono::steady_clock::now();
    const int64_t n = nloc, m = con_num;
    if (X_best.n < std::max<int64_t>(n, 1)) {   // always allocated: the ADMM graph bakes these pointers
        X_best.alloc(std::max<int64_t>(n, 1)); y_best.alloc(std::max<int64_t>(m, 1)); S_best.alloc(std::max<int64_t>(n, 1));
    }
    if (hist.n == 0) {
        // history ring on the device (the reference keeps max_iter + 1 entries per array: 64 MB for main.cu's 1e6);
        // drained into host vectors whenever the loop below synchronises (every <= 100 iterations)
        hist_cap = kHistRing;
        hist.alloc(8 * hist_cap);
        // the captured graphs bake the history pointer
        if (graph_sgs) { cudaGraphExecDestroy(graph_sgs); graph_sgs = nullptr; }
        if (graph_admm) { cudaGraphExecDestroy(graph_admm); graph_admm = nullptr; }
    }
    info_iter_num = 0;
    for (auto& v : h_hist) v.clear();
    int64_t drained = 0;                 // iterations whose history entries are already on the host
    auto drain = [&](int64_t upto) {     // entries [drained, upto) of the ring -> host (stream must be idle afterwards)
        if (upto <= drained) return;
        CUADMM_REQUIRE(upto - drained <= hist_cap, "internal: history ring overrun");
        const int64_t n0 = upto - drained;
        for (int q = 0; q < 8; ++q) {
            const size_t base = h_hist[q].size();
            h_hist[q].resize(base + (size_t)n0);
            int64_t done_ = 0;
            while (done_ < n0) {
                const int64_t k = (drained + done_) % hist_cap;
                const int64_t len = std::min(n0 - done_, hist_cap - k);
                CUADMM_CUDA(cudaMemcpyAsync(h_hist[q].data() + base + done_, hist.p + q * hist_cap + k, sizeof(double) * len,
                                            cudaMemcpyDeviceToHost, stream));
                done_ += len;
            }
        }
        CUADMM_CUDA(cudaStreamSynchronize(stream));
        drained = upto;
    };
    asmc_valid = false;                  // X, y, S may have been replaced / rescaled since the last call

    // state for this call
    CUADMM_CUDA(cudaMemcpyAsync(h_st, st.p, sizeof(DevState), cudaMemcpyDeviceToHost, stream));
    CUADMM_CUDA(cudaStreamSynchronize(stream));
    if (!if_first) {
        // second call: X, y, S were replaced by unscaled values
        scale_iterate_in();
        h_st->done = 0;
        CUADMM_CUDA(cudaMemcpyAsync(st.p, h_st, sizeof(DevState), cudaMemcpyHostToDevice, stream));
        CUADMM_CUDA(cudaStreamSynchronize(stream));      // h_st is mutated below: the copy must have read it first
        if (world == 1) {
            SpmvEpilogue e; e.mode = 4; e.aux1 = bd.p; e.aux2 = normA.p; e.aux3 = y.p; e.partial = partial.p;
            spmv_launch(*A, 1.0, X.p, 0.0, Rp.p, e, stream);
            ++launches;
        } else {
            reduce_partial_A(true, X.p, 1.0, nullptr, 0);
        }
    }
    h_st->iter = 1;
    h_st->max_iter = max_iter; h_st->stop_tol = stop_tol;
    h_st->sig_update_threshold = sig_update_threshold;
    h_st->sig_update_stage_1 = sig_update_stage_1; h_st->sig_update_stage_2 = sig_update_stage_2;
    h_st->switch_admm = switch_admm; h_st->sigscale = sigscale;
    h_st->tau = (1 < switch_admm) ? 1.95 : 1.618;
    if (h_st->errRd < stop_tol) h_st->tau = std::max(1.618, h_st->tau / 1.1);
    // the reference leaves best_KKT uninitialised when switch_admm < 1 and then restores garbage;
    // here the best iterate is tracked from the first iteration in that case
    if (switch_admm < 1) h_st->best_KKT = INFINITY;
    h_st->done = 0; h_st->stop_reason = 0;
    if (std::max(h_st->maxfeas, h_st->relgap) < stop_tol) { h_st->done = 1; h_st->stop_reason = 1; }
    if (1 > max_iter) { h_st->done = 1; h_st->stop_reason = 2; }
    CUADMM_CUDA(cudaMemcpyAsync(st.p, h_st, sizeof(DevState), cudaMemcpyHostToDevice, stream));
    CUADMM_CUDA(cudaStreamSynchronize(stream));

    if (rank != 0) verbose = false;   // one log per job
    if (verbose && ys && ys->n_deficient > 0)
        printf("\n note: %lld of %lld pivots of A A^T fell below %.0e x diagonal and were treated as redundant constraints"
               "\n       (y is then only determined up to those rows; CUADMM_PIVOT_TOL changes the tolerance)\n",
               (long long)ys->n_deficient, (long long)con_num, cuadmm::pivot_tol());
    if (verbose) {
        printf("\n -------------------------------------------------------------------------------");
        printf("\n                                    cuADMM");
        printf("\n -------------------------------------------------------------------------------");
        printf("\n norm of C = %2.1e, norm of b = %2.1e\n", norm_Corg, norm_borg);
        printf("\n  it. | p infeas d infeas | primal obj.   dual obj. rel. gap |  time |   sigma | \n");
        printf(" -------------------------------------------------------------------------------\n");
    }
    int it = 1;           // next iteration to enqueue
    int stop_iter = 0;
    while (true) {
        CUADMM_CUDA(cudaMemcpyAsync(h_st, st.p, sizeof(DevState), cudaMemcpyDeviceToHost, stream));
        CUADMM_CUDA(cudaEventRecord(ev_now, stream));
        CUADMM_CUDA(cudaStreamSynchronize(stream));
        const bool done = h_st->done != 0;
        const int cur = h_st->iter;
        drain((int64_t)cur - 1);
        if (verbose && (done || is_log_iter(cur))) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, ev_start, ev_now);
            printf(" %4d | %3.2e %3.2e | %- 5.4e %- 5.4e %3.2e | %5.1f | %2.1e |\n",
                   cur - 1, h_st->errRp, h_st->errRd, h_st->pobj, h_st->dobj, h_st->relgap, ms / 1000.0, h_st->sig);
            fflush(stdout);
        }
        if (done) { stop_iter = cur; break; }
        int target = it + 1;
        while (!is_log_iter(target) && target <= max_iter) ++target;
        for (int k = it; k < target; ++k) launch_iteration(k, switch_admm, false);
        it = target;
    }
    info_iter_num = stop_iter - 1;

    // the partial iteration the reference runs before it breaks, then the best-iterate restore
    h_st->done = 0;
    CUADMM_CUDA(cudaMemcpyAsync(&st.p->done, &h_st->done, sizeof(int), cudaMemcpyHostToDevice, stream));
    enqueue_half_step();
    if (stop_iter > switch_admm && X_best.n >= std::max<int64_t>(n, 1) && (switch_admm >= 1 || stop_iter > 1)) {
        CUADMM_CUDA(cudaMemcpyAsync(X.p, X_best.p, sizeof(double) * n, cudaMemcpyDeviceToDevice, stream));
        CUADMM_CUDA(cudaMemcpyAsync(y.p, y_best.p, sizeof(double) * m, cudaMemcpyDeviceToDevice, stream));
        CUADMM_CUDA(cudaMemcpyAsync(S.p, S_best.p, sizeof(double) * n, cudaMemcpyDeviceToDevice, stream));
        CUADMM_CUDA(cudaMemcpyAsync(h_st, st.p, sizeof(DevState), cudaMemcpyDeviceToHost, stream));
        CUADMM_CUDA(cudaStreamSynchronize(stream));
        if (verbose) printf("best max KKT residual after switch  = %2.1e \n", h_st->best_KKT);
    }
    h_st->done = 1;
    CUADMM_CUDA(cudaMemcpyAsync(&st.p->done, &h_st->done, sizeof(int), cudaMemcpyHostToDevice, stream));
    unscale_iterate(bscale, Cscale);
    iterate_scaled = false;
    drain(info_iter_num);
    CUADMM_CUDA(cudaEventRecord(ev_now, stream));
    CUADMM_CUDA(cudaStreamSynchronize(stream));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ev_start, ev_now);
    total_time = ms / 1000.0;
    solve_time = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    if (peer) peer->check(stream);
    if (verbose) {
        printf("\n -------------------------------------------------------------------------------\n\n");
        printf("%s\n", h_st->stop_reason == 2 ? "Solver ended: maximum iteration reached" : "Solver ended: converged.");
        printf("\n primal infeasibility = %2.1e \n dual   infeasibility = %2.1e \n relative gap         = %2.1e",
               h_st->errRp, h_st->errRd, h_st->relgap);
        printf("\n primal objective = %- 9.8e \n dual   objective = %- 9.8e", h_st->pobj, h_st->dobj);
        printf("\n\n time per iteration = %2.4fs \n total time         = %2.1fs", total_time / std::max(stop_iter, 1), total_time);
        printf("\n -------------------------------------------------------------------------------\n\n");
        fflush(stdout);
    }
}

// b and C triplets as the caller passes them to init and update_data; every check comes before the first device
// write, so a rejected call leaves the solver as it was
void cuadmm_solver::check_data(const int32_t* b_idx, const double* b_val, int64_t b_nnz,
                               const int32_t* C_idx, const double* C_val, int64_t C_nnz) const {
    CUADMM_REQUIRE(b_nnz >= 0 && C_nnz >= 0, "negative nnz");
    CUADMM_REQUIRE((b_idx && b_val) || b_nnz == 0, "b is null");
    CUADMM_REQUIRE((C_idx && C_val) || C_nnz == 0, "C is null");
    CUADMM_REQUIRE(b_nnz + C_nnz < INT32_MAX, "b and C exceed int32 triplet indices");
    for (int64_t k = 0; k < b_nnz; ++k) CUADMM_REQUIRE(b_idx[k] >= 0 && b_idx[k] < con_num, "b index out of range");
    for (int64_t k = 0; k < C_nnz; ++k) CUADMM_REQUIRE(C_idx[k] >= 0 && C_idx[k] < vec_len, "C index out of range");
}

// Unscaled X, y, S from the caller (full-length X and S; sharded: this rank's ranges are kept); a null vector is left
// as it is.  The next solve(if_first = 0) or load_data scales them.
void cuadmm_solver::set_iterate(const double* h_X, const double* h_y, const double* h_S) {
    std::vector<double> lx, ls;
    if (world > 1) {
        if (h_X) { shard.slice_vec(h_X, lx); h_X = lx.data(); }
        if (h_S) { shard.slice_vec(h_S, ls); h_S = ls.data(); }
    }
    if (h_X) X.upload(h_X, nloc, stream);
    if (h_y) y.upload(h_y, con_num, stream);
    if (h_S) S.upload(h_S, nloc, stream);
    asmc_valid = false;
    iterate_scaled = false;
    CUADMM_CUDA(cudaStreamSynchronize(stream));      // lx, ls and the caller's buffers may be reused on return
}

// the start point into the scaled variables (src/solver.cu:385-409): y .* normA / Cscale, X / bscale, S / Cscale, S - C
void cuadmm_solver::scale_iterate_in() {
    const int gv = ew_grid(nloc, device), gm = ew_grid(con_num, device);
    scale_vec_kernel<<<gm, 256, 0, stream>>>(con_num, y.p, normA.p, 1.0 / Cscale, 0);
    scale_kernel<<<gv, 256, 0, stream>>>(nloc, X.p, 1.0 / bscale);
    scale_kernel<<<gv, 256, 0, stream>>>(nloc, S.p, 1.0 / Cscale);
    sub_kernel<<<gv, 256, 0, stream>>>(nloc, S.p, Cd.p, SmC.p);
    launches += 4;
}

// the scaled iterate back to the caller's variables with the scales it was made with (src/solver.cu:814-816)
void cuadmm_solver::unscale_iterate(double bs, double Cs) {
    const int gv = ew_grid(nloc, device), gm = ew_grid(con_num, device);
    scale_kernel<<<gv, 256, 0, stream>>>(nloc, X.p, bs);
    scale_vec_kernel<<<gm, 256, 0, stream>>>(con_num, y.p, normA.p, Cs, 1);
    scale_kernel<<<gv, 256, 0, stream>>>(nloc, S.p, Cs);
    launches += 3;
}

// New b and C for the same A and blocks: everything init derives from b and C, recomputed on the device in place.
// normA, both SpMV operators, the y-solve, the plan, the shard, the peer arena and the captured graphs are kept.
void cuadmm_solver::update_data(const int32_t* b_idx, const double* b_val, int64_t b_nnz,
                                const int32_t* C_idx, const double* C_val, int64_t C_nnz, bool keep_iterate, double sig) {
    CUADMM_REQUIRE(initialised, "update_data() before init()");
    check_data(b_idx, b_val, b_nnz, C_idx, C_val, C_nnz);
    CUADMM_CUDA(cudaSetDevice(device));
    const auto t0 = std::chrono::steady_clock::now();
    CUADMM_CUDA(cudaEventRecord(ev_start, stream));     // total_time of the next solve counts from here, as from init
    load_data(b_idx, b_val, b_nnz, C_idx, C_val, C_nnz, keep_iterate, sig);
    update_time = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
}

// Everything init derives from b and C, on the device, in the same order for init and update_data.  Order (fixed by
// the data): scatter b, C -> norms -> scales (read back: solve() scales with host copies) -> scaled b, C and the start
// point -> Rd and Rp through the SpMV epilogues -> residual state.  keep_iterate = 0 zeroes the start point; the
// scalings and the two SpMVs still run, as they do in init for a start vector that was not given: one code path.
void cuadmm_solver::load_data(const int32_t* b_idx, const double* b_val, int64_t b_nnz,
                              const int32_t* C_idx, const double* C_val, int64_t C_nnz, bool keep_iterate, double sig) {
    // this rank's C triplets at local offsets (sharded: the owned svec ranges only)
    std::vector<int32_t> lci; std::vector<double> lcv;
    const int32_t* ci = C_idx; const double* cv = C_val; int64_t cn = C_nnz;
    if (world > 1) {
        for (int64_t k = 0; k < C_nnz; ++k) {
            const int64_t l = shard.glob2loc[C_idx[k]];
            if (l >= 0) { lci.push_back((int32_t)l); lcv.push_back(C_val[k]); }
        }
        ci = lci.data(); cv = lcv.data(); cn = (int64_t)lci.size();
    }
    // staging: b, all of C, and (sharded) this rank's C
    const int64_t nt = b_nnz + C_nnz + (world > 1 ? cn : 0);
    if (upd_idx.n < std::max<int64_t>(nt, 1)) { upd_idx.alloc(std::max<int64_t>(nt, 1)); upd_val.alloc(std::max<int64_t>(nt, 1)); }
    const int64_t nwin = std::max<int64_t>(std::max(con_num, vec_len), 1);
    const int gb = ew_grid(con_num, device), gc = ew_grid(vec_len, device);
    if (upd_win.n < nwin) upd_win.alloc(nwin);
    if (upd_part.n < 2 * (int64_t)(gb + gc)) upd_part.alloc(2 * (int64_t)(gb + gc));
    if (upd_zero.n == 0) { upd_zero.alloc(2); upd_zero.zero(stream); }
    if (world > 1 && upd_full.n < std::max<int64_t>(vec_len, 1)) upd_full.alloc(std::max<int64_t>(vec_len, 1));
    auto stage_in = [&](int64_t at, const int32_t* idx, const double* val, int64_t n) {
        if (!n) return;
        CUADMM_CUDA(cudaMemcpyAsync(upd_idx.p + at, idx, sizeof(int32_t) * n, cudaMemcpyHostToDevice, stream));
        CUADMM_CUDA(cudaMemcpyAsync(upd_val.p + at, val, sizeof(double) * n, cudaMemcpyHostToDevice, stream));
    };
    stage_in(0, b_idx, b_val, b_nnz);
    stage_in(b_nnz, C_idx, C_val, C_nnz);
    if (world > 1) stage_in(b_nnz + C_nnz, ci, cv, cn);

    // scalar state as init leaves it (done = 0 also lets the SpMV and reduction kernels below run)
    const double bscale_old = bscale, Cscale_old = Cscale;
    memset(h_st, 0, sizeof(DevState));
    h_st->sig = sig; h_st->tau = 1.95;
    h_st->sigmax = 1e3; h_st->sigmin = 1e-3; h_st->ratioconst = 1e0;
    CUADMM_CUDA(cudaMemcpyAsync(st.p, h_st, sizeof(DevState), cudaMemcpyHostToDevice, stream));

    // dense b and C
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    auto scatter = [&](const int32_t* idx, const double* val, int64_t nnz, DevBuf<double>& out, int64_t len) {
        out.zero(stream);
        if (!nnz) return;
        CUADMM_CUDA(cudaMemsetAsync(upd_win.p, 0xff, sizeof(int32_t) * (size_t)len, stream));   // -1
        const int g = (int)std::min<int64_t>((nnz + 255) / 256, (int64_t)sms * 8);
        triplet_mark_kernel<<<g, 256, 0, stream>>>((int32_t)nnz, idx, upd_win.p);
        triplet_store_kernel<<<g, 256, 0, stream>>>((int32_t)nnz, idx, val, upd_win.p, out.p);
        launches += 2;
    };
    scatter(upd_idx.p, upd_val.p, b_nnz, bd, con_num);
    scatter(upd_idx.p + b_nnz, upd_val.p + b_nnz, C_nnz, world > 1 ? upd_full : Cd, vec_len);
    if (world > 1) scatter(upd_idx.p + b_nnz + C_nnz, upd_val.p + b_nnz + C_nnz, cn, Cd, nloc);

    // |b|, |b ./ normA| and |C| over the full vectors, on grids that depend on con_num and vec_len only: a sharded
    // solver reduces all of C on every rank (a scratch copy), so its scales are bit-identical to the one-GPU update's
    double* part_b = upd_part.p;
    double* part_c = upd_part.p + 2 * (int64_t)gb;
    double* part_rd = partial.p;
    double* part_rp = partial.p + 2 * (int64_t)std::max(nAt_blocks, nE_blocks);
    sumsq_kernel<<<gb, kEwThreads, 0, stream>>>(con_num, bd.p, normA.p, part_b);
    sumsq_kernel<<<gc, kEwThreads, 0, stream>>>(vec_len, world > 1 ? upd_full.p : Cd.p, nullptr, part_c);
    data_scales_kernel<<<1, 256, 0, stream>>>(st.p, part_b, gb, part_c, gc);
    launches += 2;
    ++launches;
    CUADMM_CUDA(cudaMemcpyAsync(h_st, st.p, sizeof(DevState), cudaMemcpyDeviceToHost, stream));
    CUADMM_CUDA(cudaStreamSynchronize(stream));
    bscale = h_st->bscale; Cscale = h_st->Cscale; objscale = h_st->objscale;
    norm_borg = h_st->norm_borg; norm_Corg = h_st->norm_Corg;

    // scaled b and C; the start point
    scale_vec_kernel<<<ew_grid(con_num, device), 256, 0, stream>>>(con_num, bd.p, normA.p, 1.0 / bscale, 1);
    scale_kernel<<<ew_grid(nloc, device), 256, 0, stream>>>(nloc, Cd.p, 1.0 / Cscale);
    launches += 2;
    if (!keep_iterate) {
        X.zero(stream); y.zero(stream); S.zero(stream);
        CUADMM_CUDA(cudaStreamSynchronize(stream));
        plan->reset_warm_start();   // identity bases, as a new plan has them
    } else if (iterate_scaled) {    // no solve since init / the last update: back to unscaled with the scales it was made with
        unscale_iterate(bscale_old, Cscale_old);
    }
    scale_iterate_in();

    // Rd = A^T y - C + S with |Rd|^2 and <C, X> (mode 3 with tau sig = 0 leaves X as it is), then Rp = b - A X with
    // |normA .* Rp|^2 and <b, y> (K8), then the state; sharded: summed over ranks like the iteration's K7 / K8 scalars
    SpmvEpilogue e; e.mode = 3; e.aux1 = Cd.p; e.aux2 = S.p; e.out2 = X.p; e.scal = upd_zero.p; e.partial = part_rd;
    spmv_launch(*At, 1.0, y.p, 0.0, Rd.p, e, stream); ++launches;
    if (world == 1) {
        e = SpmvEpilogue(); e.mode = 4; e.aux1 = bd.p; e.aux2 = normA.p; e.aux3 = y.p; e.partial = part_rp;
        spmv_launch(*A, 1.0, X.p, 0.0, Rp.p, e, stream); ++launches;
    } else {
        reduce_partial_A(true, X.p, 1.0, part_rd, nAt_blocks);
    }
    const ScalarPartials sp = scalar_partials(part_rd, nAt_blocks, part_rp);
    data_residuals_kernel<<<1, 256, 0, stream>>>(st.p, sp.rd, sp.n_rd, sp.rp, sp.n_rp);
    ++launches;
    CUADMM_CUDA(cudaGetLastError());
    CUADMM_CUDA(cudaMemcpyAsync(h_st, st.p, sizeof(DevState), cudaMemcpyDeviceToHost, stream));
    CUADMM_CUDA(cudaStreamSynchronize(stream));
    if (peer) peer->check(stream);
    asmc_valid = false;
    iterate_scaled = true;
    info_iter_num = 0;
    for (auto& v : h_hist) v.clear();
}

// ------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------
extern "C" {

int cuadmm_solver_create(cuadmm_solver_t** out) {
    return guarded([&] { CUADMM_REQUIRE(out, "out is null"); *out = new cuadmm_solver(); });
}
void cuadmm_solver_destroy(cuadmm_solver_t* s) { delete s; }
int cuadmm_solver_set_verbose(cuadmm_solver_t* s, int verbose) {
    return guarded([&] { CUADMM_REQUIRE(s, "solver is null"); s->verbose = verbose != 0; });
}

int cuadmm_solver_init(cuadmm_solver_t* s, int eig_stream_num_per_gpu, int cpu_eig_thread_num, int64_t vec_len, int64_t con_num,
        const int32_t* At_csc_col_ptrs, const int32_t* At_csc_row_ids, const double* At_csc_vals, int64_t At_nnz,
        const int32_t* b_indices, const double* b_vals, int64_t b_nnz,
        const int32_t* C_indices, const double* C_vals, int64_t C_nnz,
        const int32_t* blk_vals, int64_t mat_num, const double* X_vals, const double* y_vals, const double* S_vals, double sig) {
    return guarded([&] {
        CUADMM_REQUIRE(s, "solver is null");
        s->init(eig_stream_num_per_gpu, cpu_eig_thread_num, vec_len, con_num, At_csc_col_ptrs, At_csc_row_ids, At_csc_vals, At_nnz,
                b_indices, b_vals, b_nnz, C_indices, C_vals, C_nnz, blk_vals, mat_num, X_vals, y_vals, S_vals, sig);
    });
}

int cuadmm_solver_init_from_problem(cuadmm_solver_t* s, const cuadmm_problem_t* p, int eig_stream_num_per_gpu,
                                    int cpu_eig_thread_num, double sig) {
    return guarded([&] {
        CUADMM_REQUIRE(s && p, "null argument");
        const Problem& q = p->prob;
        CUADMM_REQUIRE(!s->initialised, "solver already initialised (one instance per problem, like SDPSolver)");
        s->blk_types = q.blk_types;
        s->init(eig_stream_num_per_gpu, cpu_eig_thread_num, q.vec_len, q.con_num, q.At_csc_col_ptrs.data(), q.At_csc_row_ids.data(),
                q.At_csc_vals.data(), q.At_nnz, q.b_indices.data(), q.b_vals.data(), q.b_nnz, q.C_indices.data(), q.C_vals.data(),
                q.C_nnz, q.blk_vals.data(), q.mat_num, q.X_vals.empty() ? nullptr : q.X_vals.data(),
                q.y_vals.empty() ? nullptr : q.y_vals.data(), q.S_vals.empty() ? nullptr : q.S_vals.data(), sig);
    });
}

int cuadmm_solver_solve(cuadmm_solver_t* s, int max_iter, double stop_tol, int sig_update_threshold, int sig_update_stage_1,
                        int sig_update_stage_2, int switch_admm, double sigscale, int if_first) {
    return guarded([&] {
        CUADMM_REQUIRE(s, "solver is null");
        s->solve(max_iter, stop_tol, sig_update_threshold, sig_update_stage_1, sig_update_stage_2, switch_admm, sigscale, if_first != 0);
    });
}

static void get_vec(cuadmm_solver_t* s, const DevBuf<double>& d, int64_t n, double* h) {
    CUADMM_REQUIRE(s && h, "null argument");
    CUADMM_REQUIRE(s->initialised, "solver not initialised");
    CUADMM_CUDA(cudaSetDevice(s->device));
    d.download(h, n, s->stream);
    CUADMM_CUDA(cudaStreamSynchronize(s->stream));
}
int cuadmm_solver_update_data(cuadmm_solver_t* s, const int32_t* b_idx, const double* b_vals, int64_t b_nnz,
                              const int32_t* C_idx, const double* C_vals, int64_t C_nnz, int keep_iterate, double sig) {
    return guarded([&] {
        CUADMM_REQUIRE(s, "solver is null");
        s->update_data(b_idx, b_vals, b_nnz, C_idx, C_vals, C_nnz, keep_iterate != 0, sig);
    });
}

int cuadmm_solver_get_X(cuadmm_solver_t* s, double* h) {
    return guarded([&] { if (s && s->world > 1) s->gather_full(s->X, h); else get_vec(s, s->X, s->vec_len, h); });
}
int cuadmm_solver_get_y(cuadmm_solver_t* s, double* h) { return guarded([&] { get_vec(s, s->y, s->con_num, h); }); }
int cuadmm_solver_get_S(cuadmm_solver_t* s, double* h) {
    return guarded([&] { if (s && s->world > 1) s->gather_full(s->S, h); else get_vec(s, s->S, s->vec_len, h); });
}

int cuadmm_solver_set_distributed(cuadmm_solver_t* s, int rank, int world, const char id[128]) {
    return guarded([&] {
        CUADMM_REQUIRE(s && id, "null argument");
        CUADMM_REQUIRE(!s->initialised, "set_distributed must precede init");
        CUADMM_REQUIRE(world >= 1 && rank >= 0 && rank < world, "bad rank/world");
        // a job launched for the removed NCCL transport fails here instead of running the peer transport under its name
        const char* comm = getenv("CUADMM_COMM");
        CUADMM_REQUIRE(!comm || strcmp(comm, "peer") == 0,
                       std::string("CUADMM_COMM=") + comm + ": the NCCL transport was removed; peer memory is the only transport");
        s->rank = rank; s->world = world;
        memcpy(s->job_id, id, 128);
    });
}

int cuadmm_solver_set_block_types(cuadmm_solver_t* s, const char* types, int64_t mat_num) {
    return guarded([&] {
        CUADMM_REQUIRE(s, "solver is null");
        CUADMM_REQUIRE(!s->initialised, "set_block_types must precede init");
        CUADMM_REQUIRE(mat_num >= 0, "mat_num < 0");
        if (!types) { s->blk_types.clear(); return; }
        for (int64_t k = 0; k < mat_num; ++k)
            CUADMM_REQUIRE(valid_cone(types[k]), std::string("unknown block type '") + types[k] + "' (expected 's', 'l' or 'u')");
        s->blk_types.assign(types, types + mat_num);
    });
}

int cuadmm_solver_set_device(cuadmm_solver_t* s, int device) {
    return guarded([&] {
        CUADMM_REQUIRE(s, "solver is null");
        CUADMM_REQUIRE(!s->initialised, "set_device must precede init");
        CUADMM_REQUIRE(device >= 0, "negative device index");
        s->device = device; s->device_set = true;
    });
}

int cuadmm_solver_set_XyS(cuadmm_solver_t* s, const double* h_X, const double* h_y, const double* h_S, double sig) {
    return guarded([&] {
        CUADMM_REQUIRE(s && s->initialised, "solver not initialised");
        CUADMM_CUDA(cudaSetDevice(s->device));
        s->set_iterate(h_X, h_y, h_S);
        s->h_st->sig = sig;                 // pinned mirror: stays valid until the copy below has run
        CUADMM_CUDA(cudaMemcpyAsync(&s->st.p->sig, &s->h_st->sig, sizeof(double), cudaMemcpyHostToDevice, s->stream));
        CUADMM_CUDA(cudaStreamSynchronize(s->stream));
    });
}

int64_t cuadmm_solver_iter_num(const cuadmm_solver_t* s) { return s ? s->info_iter_num : -1; }

int cuadmm_solver_history(const cuadmm_solver_t* s, int which, double* out, int64_t cap) {
    return guarded([&] {
        CUADMM_REQUIRE(s && out, "null argument");
        CUADMM_REQUIRE(which >= 0 && which < 8, "which out of range");
        const int64_t n = std::min<int64_t>(cap, s->info_iter_num);
        for (int64_t k = 0; k < n; ++k) out[k] = s->h_hist[which][(size_t)k];
    });
}

int cuadmm_solver_times(const cuadmm_solver_t* s, double out[8]) {
    return guarded([&] {
        CUADMM_REQUIRE(s && out, "null argument");
        out[0] = s->total_time; out[1] = s->init_time; out[2] = s->solve_time; out[3] = s->proj_time;
        out[4] = s->ysolve_time; out[5] = s->spmv_time; out[6] = s->update_time; out[7] = 0;
    });
}

int64_t cuadmm_solver_launches(const cuadmm_solver_t* s) { return s ? s->launches : -1; }

int cuadmm_solver_run_iterations(cuadmm_solver_t* s, int n_iters, int sgs, int profile, double out_ms[4]) {
    return guarded([&] {
        CUADMM_REQUIRE(s && out_ms && n_iters >= 0, "bad argument");
        double t[8];
        s->run_iterations(n_iters, sgs != 0, profile != 0, t);
        for (int k = 0; k < 4; ++k) out_ms[k] = t[k];
    });
}
int cuadmm_solver_run_iterations_ex(cuadmm_solver_t* s, int n_iters, int sgs, double out_ms[8]) {
    return guarded([&] {
        CUADMM_REQUIRE(s && out_ms && n_iters >= 0, "bad argument");
        s->run_iterations(n_iters, sgs != 0, true, out_ms);
    });
}

int cuadmm_solver_ysolve_stats(const cuadmm_solver_t* s, int64_t out[8]) {
    return guarded([&] {
        CUADMM_REQUIRE(s && s->ys && out, "solver not initialised");
        if (cuadmm_ysolve_stats(s->ys, out) != 0) throw Error(CUADMM_EINVAL, cuadmm_last_error());
    });
}

int cuadmm_solve_matlab_like(int eig_stream_num_per_gpu, int max_iter, double stop_tol, int64_t vec_len, int64_t con_num,
        const int64_t* At_jc, const int64_t* At_ir, const double* At_pr,
        const int64_t* b_ir, const double* b_pr, int64_t b_nnz, const int64_t* C_ir, const double* C_pr, int64_t C_nnz,
        const double* blk_vec, int64_t mat_num, const double* X0, const double* y0, const double* S0, double sig,
        int sig_update_threshold, int sig_update_stage_1, int sig_update_stage_2, int switch_admm, double sigscale,
        double* X, double* y, double* S, int64_t* iter_num, double* info, double* total_time) {
    return guarded([&] {
        CUADMM_REQUIRE(At_jc && blk_vec && X && y && S, "null argument");
        // the MEX narrows MATLAB's size_t indices to int32 (MATLAB/cuadmm_MATLAB.cu:48-51,73-88)
        const int64_t nnz = At_jc[con_num];
        CUADMM_REQUIRE(nnz <= INT32_MAX && vec_len <= INT32_MAX, "problem exceeds the int32 indices of the reference interface");
        std::vector<int32_t> cp(con_num + 1), ri(nnz), bi(b_nnz), ci(C_nnz), blk(mat_num);
        for (int64_t i = 0; i <= con_num; ++i) cp[i] = (int32_t)At_jc[i];
        for (int64_t p = 0; p < nnz; ++p) ri[p] = (int32_t)At_ir[p];
        for (int64_t k = 0; k < b_nnz; ++k) bi[k] = (int32_t)b_ir[k];
        for (int64_t k = 0; k < C_nnz; ++k) ci[k] = (int32_t)C_ir[k];
        for (int64_t k = 0; k < mat_num; ++k) blk[k] = (int32_t)blk_vec[k];
        cuadmm_solver s;
        s.init(eig_stream_num_per_gpu, 30, vec_len, con_num, cp.data(), ri.data(), At_pr, nnz, bi.data(), b_pr, b_nnz,
               ci.data(), C_pr, C_nnz, blk.data(), mat_num, X0, y0, S0, sig);
        s.solve(max_iter, stop_tol, sig_update_threshold, sig_update_stage_1, sig_update_stage_2, switch_admm, sigscale, true);
        s.X.download(X, vec_len, s.stream); s.y.download(y, con_num, s.stream); s.S.download(S, vec_len, s.stream);
        CUADMM_CUDA(cudaStreamSynchronize(s.stream));
        if (iter_num) *iter_num = s.info_iter_num;
        if (info) {
            const int64_t cap = (int64_t)max_iter + 1;
            for (int q = 0; q < 8; ++q)
                for (int64_t k = 0; k < cap; ++k)
                    info[q * cap + k] = k < s.info_iter_num ? s.h_hist[q][(size_t)k] : 0.0;
        }
        if (total_time) *total_time = s.total_time;
    });
}

}  // extern "C"
