// solver.h — sGS-ADMM driver: the reference's SDPSolver (include/cuadmm/solver.h:30-248,
// src/solver.cu) re-written around the device-resident hot path.  Host code only orchestrates:
// every scalar of the iteration (sigma, tau, residuals, win counters, stop flag, history) lives in
// device memory, so an iteration is a fixed sequence of kernel launches with no host round trip.
#pragma once
#include "common.h"
#include "plan.h"
#include "spmv.h"
#include "ysolve.h"
#include "problem.h"
#include "shard.h"
#include "peer.h"
#include "peer_kernels.h"

namespace cuadmm {

// device-resident scalar state; `sig, tau` must stay first (kernels read them as scal[0], scal[1])
struct DevState {
    double sig, tau;
    double errRp, errRd, pobj, dobj, relgap, maxfeas, feasratio;
    double bscale, Cscale, objscale, norm_borg, norm_Corg;
    double sigmax, sigmin, sigscale, stop_tol, ratioconst;
    double best_KKT, sgs_KKT;
    int prim_win, dual_win;
    int iter;            // index of the iteration about to run (1-based, as the reference's loop variable)
    int done;            // set by the scalar kernel when the stop test of the NEXT iteration fires
    int max_iter, sig_update_threshold, sig_update_stage_1, sig_update_stage_2, switch_admm;
    int stop_reason;     // 1 converged, 2 max iterations
    int pad_;
};

}  // namespace cuadmm

struct cuadmm_solver {
    int device = 0;
    bool verbose = false;
    bool initialised = false;
    int64_t vec_len = 0, con_num = 0;
    int64_t nloc = 0;                        // svec entries owned by this rank (== vec_len on one GPU)
    // multi-GPU (one process per GPU): block shard; partial products move through peer memory (kernels store into
    // the peers' arenas, peer.h)
    int rank = 0, world = 1;
    char job_id[128] = {0};                  // rendezvous key of the peer board
    cuadmm::Shard shard;
    std::vector<char> blk_types;             // block cones ('s', 'l', 'u') set before init; empty: all 's'
    bool device_set = false;                 // cuadmm_solver_set_device / CUADMM_DEVICE given
    std::unique_ptr<cuadmm::PeerComm> peer;
    int64_t slice = 0;                       // rows of an m-vector reduced by one rank (peer transport)
    double* stage = nullptr;                 // arena: world x slice staged partial rows addressed to this rank
    cuadmm::PeerPtrs p_stage, p_asmc, p_Rp, p_full;
    cuadmm::DevBuf<double> cta_part;         // per-CTA partial sums of peer_reduce_kernel
    cuadmm::DevBuf<int64_t> d_loc2glob;
    cuadmm::DevBuf<double> full_buf;         // vec_len doubles, for gathering full X / S
    void gather_full(const cuadmm::DevBuf<double>& local, double* h_full);
    void reduce_partial_A(bool for_rp, const double* x_local, double alpha, const double* part_rd, int n_rd);
    struct ScalarPartials { const double* rd; int n_rd; const double* rp; int n_rp; };
    ScalarPartials scalar_partials(const double* part_rd, int n_rd, const double* part_rp) const;
    std::unique_ptr<cuadmm_plan> plan;
    cuadmm_spmv_s* A = nullptr;    // m x vec_len (row-normalised)
    cuadmm_spmv_s* At = nullptr;   // vec_len x m
    cuadmm_ysolve_s* ys = nullptr;
    // vectors
    cuadmm::DevBuf<double> X, S, y, Rp, SmC, Rd1, Rd, Xb, Xproj, rhsy, Cd, bd, normA;
    cuadmm::DevBuf<double> X_best, y_best, S_best;
    cuadmm::DevBuf<double> partial;          // per-CTA partial sums of the fused reductions
    cuadmm::DevBuf<double> hist;             // 8 x hist_cap history ring (info_*_arr)
    int64_t hist_cap = 0;
    cuadmm::DevBuf<cuadmm::DevState> st;
    cuadmm::DevState* h_st = nullptr;        // pinned mirror
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_start = nullptr, ev_now = nullptr;
    // host copies of the scaling constants
    double bscale = 1, Cscale = 1, objscale = 1, norm_borg = 1, norm_Corg = 1;
    std::vector<double> h_normA;
    int64_t info_iter_num = 0;
    std::vector<double> h_hist[8];           // drained from the device ring while solve() runs
    double total_time = 0, init_time = 0, solve_time = 0, proj_time = 0, ysolve_time = 0, spmv_time = 0, update_time = 0;
    // update_data: X, y, S hold the scaled iterate (after init / update_data) or the unscaled one (after solve / set_XyS)
    bool iterate_scaled = true;
    cuadmm::DevBuf<int32_t> upd_idx, upd_win;   // b then C triplets on the device; last-write-wins marks per dense entry
    cuadmm::DevBuf<double> upd_val, upd_part, upd_zero;   // their values; per-CTA norm partials; (sig, tau) = (0, 0)
    cuadmm::DevBuf<double> upd_full;         // sharded: all of C, for the norm every rank takes over the full vector
    int64_t launches = 0;
    int nA_blocks = 0, nAt_blocks = 0, nE_blocks = 0;
    bool profile = false;
    std::vector<cudaEvent_t> prof_ev;
    std::vector<int> prof_tag;

    ~cuadmm_solver();
    void init(int eig_stream_num_per_gpu, int cpu_eig_thread_num, int64_t vec_len, int64_t con_num,
              const int32_t* At_col_ptrs, const int32_t* At_row_ids, const double* At_vals, int64_t At_nnz,
              const int32_t* b_idx, const double* b_val, int64_t b_nnz,
              const int32_t* C_idx, const double* C_val, int64_t C_nnz,
              const int32_t* blk, int64_t mat_num, const double* X0, const double* y0, const double* S0, double sig);
    void solve(int max_iter, double stop_tol, int sig_update_threshold, int sig_update_stage_1,
               int sig_update_stage_2, int switch_admm, double sigscale, bool if_first);
    // new b and C on the same A and blocks; every device buffer is written in place (the graphs hold the pointers)
    void update_data(const int32_t* b_idx, const double* b_val, int64_t b_nnz,
                     const int32_t* C_idx, const double* C_val, int64_t C_nnz, bool keep_iterate, double sig);
    void check_data(const int32_t* b_idx, const double* b_val, int64_t b_nnz,
                    const int32_t* C_idx, const double* C_val, int64_t C_nnz) const;
    // b, C, their scales, the scaled start point and the initial residual state, on the device (init and update_data)
    void load_data(const int32_t* b_idx, const double* b_val, int64_t b_nnz,
                   const int32_t* C_idx, const double* C_val, int64_t C_nnz, bool keep_iterate, double sig);
    void set_iterate(const double* h_X, const double* h_y, const double* h_S);
    void scale_iterate_in();
    void unscale_iterate(double bs, double Cs);
    void enqueue_k1(bool asmc_cached);
    void enqueue_iteration(int iter, int switch_admm, bool prof = false);
    void run_iterations(int n_iters, bool sgs, bool profile, double out_ms[8]);
    void enqueue_half_step();
    // whole-iteration CUDA graphs (one for the sGS iteration, one for the plain ADMM iteration)
    cudaGraphExec_t graph_sgs = nullptr, graph_admm = nullptr;
    int64_t graph_launches_sgs = 0, graph_launches_admm = 0;
    bool use_graphs = true;
    cuadmm::DevBuf<double> asmc;             // -A (S-C) (summed over the ranks when sharded), reused by the next iteration's K1
    bool asmc_valid = false;
    void launch_iteration(int iter, int switch_admm, bool prof);
};
