/*
 * cuadmm_b200.h — C ABI of the B200-native cuADMM hot path.
 *
 * The reference (ComputationalRobotics/cuADMM) has no FFI seam: its hot path is
 * inlined in SDPSolver::solve (src/solver.cu:355-822).  This header is the seam a
 * maintainer would bind instead; every entry point cites the reference interface
 * it replaces.  Conventions:
 *   - plain pointers and 64-bit sizes, no C++/torch types;
 *   - `d_` pointers are device pointers on the plan's device, `h_` pointers are host;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - every function returns 0 on success, a negative CUADMM_E* code otherwise and
 *     records a message retrievable by cuadmm_last_error() (the reference only
 *     prints CUDA errors and continues, include/cuadmm/check.h:17-56);
 *   - there is NO CPU fallback: without a CUDA device every compute entry point
 *     fails with CUADMM_ENODEVICE.
 */
#ifndef CUADMM_B200_H
#define CUADMM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CUADMM_OK          0
#define CUADMM_EINVAL     -1
#define CUADMM_ENODEVICE  -2
#define CUADMM_ECUDA      -3
#define CUADMM_ENOMEM     -4
#define CUADMM_EIO        -5
#define CUADMM_ENUMERIC   -6
#define CUADMM_ENCCL      -7

const char* cuadmm_last_error(void);
const char* cuadmm_version(void);
/* number of visible CUDA devices (0 when there is none / no driver) */
int cuadmm_device_count(void);

/* --------------------------------------------------------------------------
 * Block plan: block analysis, large/small partition, svec maps.
 * Replaces analyze_blk (src/utils/analyze_blk.cu:63-99), is_large_mat +
 * MatrixSizes::init (src/matrix_sizes.cu:14-68) and get_maps
 * (src/utils/get_maps.cu:80-134).  Pure host logic lives in the plan so it can
 * be queried without a GPU (device < 0 builds a host-only plan).
 * -------------------------------------------------------------------------- */
typedef struct cuadmm_plan cuadmm_plan;

int  cuadmm_plan_create(const int32_t* blk, int64_t nblk, int device, cuadmm_plan** out);
/* Typed blocks (SDPT3 blk.txt letters), one char per block: 's' PSD n x n (n(n+1)/2 svec entries), 'l' nonnegative
 * orthant R^n_+ (n entries, projection max(x, 0)), 'u' free R^n (n entries, projection = identity, dual slack S = 0).
 * The blocks lie contiguously in blk order in the one iterate vector.  types == NULL: every block is 's' (same plan as
 * cuadmm_plan_create).  device = -1: host-only plan. */
int  cuadmm_plan_create_typed(const char* types, const int32_t* blk, int64_t nblk, int device, cuadmm_plan** out);
void cuadmm_plan_destroy(cuadmm_plan* plan);
int64_t cuadmm_plan_vec_len(const cuadmm_plan* plan);
int64_t cuadmm_plan_nblk(const cuadmm_plan* plan);

/* Reference-layout helpers (cuadmm_plan_sizes / totals / start_indices / maps, cuadmm_svec_to_smat / smat_to_svec):
 * the pooled dense layout has no place for 'l' / 'u' blocks, so on a plan that holds any they fail with CUADMM_EINVAL
 * (cuadmm_plan_start_indices returns CUADMM_EINVAL).
 * analyze_blk: distinct sizes ascending, their counts, and the reference's
 * large(1)/small(0) classification.  Arrays must hold cuadmm_plan_num_sizes(). */
int64_t cuadmm_plan_num_sizes(const cuadmm_plan* plan);
int  cuadmm_plan_sizes(const cuadmm_plan* plan, int32_t* sizes, int32_t* nums, int32_t* is_large);
/* MatrixSizes totals: out[0..5] = large_mat_num, sum_large_mat_size, total_large_mat_size,
 * small_mat_num, sum_small_mat_size, total_small_mat_size */
int  cuadmm_plan_totals(const cuadmm_plan* plan, int64_t out[6]);
/* MatrixSizes start indices.  which: 0 large_mat_start, 1 large_W_start,
 * 2 small_mat_start, 3 small_W_start.  Returns the entry count (or writes it when out==NULL). */
int64_t cuadmm_plan_start_indices(const cuadmm_plan* plan, int which, int64_t* out);
/* get_maps: three int32 arrays of length vec_len (host), bit-exact with the reference */
int  cuadmm_plan_maps(const cuadmm_plan* plan, int32_t* map_B, int32_t* map_M1, int32_t* map_M2);

/* Eig-cost-balanced partition of the blocks onto `nparts` GPUs (replaces the
 * equal-count split of src/duo_solver.cu:266-295).  owner[k] = part of block k. */
int  cuadmm_plan_partition(const cuadmm_plan* plan, int nparts, int32_t* owner, double* part_cost);

/* --------------------------------------------------------------------------
 * svec <-> smat (vector_to_matrices / matrices_to_vector,
 * src/kernels/vec_mat_conversion.cu:11-98) on the reference's pooled layout.
 * Indices are computed from block descriptors, not from the 12 B/entry maps.
 * -------------------------------------------------------------------------- */
int cuadmm_svec_to_smat(cuadmm_plan* plan, const double* d_svec,
                        double* d_large_mat, double* d_small_mat, void* stream);
int cuadmm_smat_to_svec(cuadmm_plan* plan, const double* d_large_mat,
                        const double* d_small_mat, double* d_svec, void* stream);

/* --------------------------------------------------------------------------
 * PSD projection  Xproj = Pi_+(Xb), svec in -> svec out (typed plans: max(x, 0) on 'l' blocks, x on 'u' blocks).
 * Replaces the whole stage src/solver.cu:531-647 (vector_to_matrices, Xsyevd /
 * DsyevjBatched, max0, diag scale, gemmStridedBatched, matrices_to_vector).
 * -------------------------------------------------------------------------- */
int cuadmm_project_psd(cuadmm_plan* plan, const double* d_Xb, double* d_Xproj, void* stream);
/* same with the solver's fused epilogue (device pointers, d_sig one device scalar sigma):
 *   Xproj = Pi_K(Xb),  S = (Xproj - X) / sigma - Rd1,  SmC = S - C,
 * except on 'u' blocks, where S = 0 exactly and SmC = 0 - C (the dual cone of a free block is {0}). */
int cuadmm_project_epilogue(cuadmm_plan* plan, const double* d_Xb, double* d_Xproj, const double* d_X, const double* d_Rd1,
                            const double* d_C, double* d_S, double* d_SmC, const double* d_sig, void* stream);
/* same, host buffers (H2D + kernel + D2H inside the call) */
int cuadmm_project_psd_host(cuadmm_plan* plan, const double* h_Xb, double* h_Xproj);
/* parity/debug: also returns per-block eigenvalues ascending, concatenated in blk
 * order (length sum n_k), and the Jacobi sweep count per block (may be NULL).
 * 'l' / 'u' blocks: NaN in their n eigenvalue slots, 0 sweeps.
 * Blocks n <= 168: eigenvalues of the kernel that produced X.  168 < n <= 1024: X comes from the sign
 * iteration, which has no eigenvalues; they are computed by the global-memory Jacobi kernel on the same
 * input for this entry only.  n > 1024: NaN. */
int cuadmm_project_psd_eig_host(cuadmm_plan* plan, const double* h_Xb, double* h_Xproj,
                                double* h_eigvals, int32_t* h_sweeps);
/* device time of the last cuadmm_project_psd* call in ms (CUDA events) */
double cuadmm_plan_last_ms(const cuadmm_plan* plan);
/* number of kernel launches issued by the last projection call */
int64_t cuadmm_plan_last_launches(const cuadmm_plan* plan);
/* tuning: Jacobi convergence threshold on max |cos(g_p,g_q)| over all column pairs, tested on the state after
 * each sweep (default 1e-11: projected X within ~2e-12 relative of LAPACK's, measured), max sweeps */
int cuadmm_plan_set_jacobi(cuadmm_plan* plan, double threshold, int max_sweeps);
/* Fixed-rank projection (the reference's max_dense_vector_zero_mask + get_eig_rank_mask, src/kernels/dense_scalar.cu:51-56,
 * src/utils/get_eig_rank_mask.cu:16-38; wired but commented out in src/duo_solver.cu:843-850): with eig_rank > 0 only the
 * eig_rank largest eigenvalues of every block survive the clamp at zero.  Blocks n <= 168 only; 0 turns it off. */
int cuadmm_plan_set_rank_limit(cuadmm_plan* plan, int eig_rank);
/* get_eig_rank_mask on host arrays: mask[i * mat_size + j] = 1 for the last eig_rank positions j of every block i */
int cuadmm_eig_rank_mask(int32_t* mask, int64_t batch_size, int64_t mat_size, int64_t eig_rank);
/* Warm start (default on; env CUADMM_JACOBI_WARM=0 turns it off): the plan keeps, per block, the
 * orthonormal eigenbasis its last projection ended in and starts the next Jacobi from it, which is
 * what makes successive ADMM iterates cheap (2-3 sweeps instead of 7-9).  The result is the same
 * projection to rounding, but no longer bit-identical between two calls on the same input.
 * enable = 0: forget the bases and project from cold every time; 1: forget the bases, keep warm starting. */
int cuadmm_plan_set_warm_start(cuadmm_plan* plan, int enable);

/* --------------------------------------------------------------------------
 * Sparse constraint operators.
 * cuadmm_spmv replaces SpMV_cusparse (include/cuadmm/cusparse.h:70-83):
 *   y = alpha * A x + beta * y, CSR, f64 values, int32 column indices.
 * cuadmm_normA replaces get_normA (src/kernels/sparse_matrix_norm.cu:11-44).
 * cuadmm_csc_to_csr replaces CSC_to_CSR_cusparse (include/cuadmm/cusparse.h:35-49).
 * -------------------------------------------------------------------------- */
typedef struct cuadmm_spmv_s cuadmm_spmv_t;

int  cuadmm_spmv_create(int64_t rows, int64_t cols, int64_t nnz,
                        const int32_t* h_rowptr, const int32_t* h_colind, const double* h_val,
                        int device, cuadmm_spmv_t** out);
void cuadmm_spmv_destroy(cuadmm_spmv_t* A);
int  cuadmm_spmv(cuadmm_spmv_t* A, double alpha, const double* d_x, double beta, double* d_y, void* stream);
int  cuadmm_spmv_host(cuadmm_spmv_t* A, double alpha, const double* h_x, double beta, double* h_y);
/* host helpers (exact arithmetic of the reference: division, floor 1.0) */
int  cuadmm_normA_host(int64_t con_num, const int32_t* At_col_ptrs, double* At_vals, double* normA);
int  cuadmm_csc_to_csr_host(int64_t nrows, int64_t ncols, int64_t nnz,
                            const int32_t* col_ptrs, const int32_t* row_ids, const double* vals,
                            int32_t* row_ptrs, int32_t* col_ids, double* out_vals);

/* --------------------------------------------------------------------------
 * AA^T y-solve.  Replaces CholeskySolverCPU::{get_A,factorize,solve}
 * (include/cuadmm/cholesky_cpu.h:62-155) plus the two perform_permutation
 * launches and the PCIe round trip around it (src/solver.cu:487-500,704-717):
 *   y = (A A^T + eps I)^-1 rhs      entirely on the device.
 * A is given as the CSC arrays of At (vec_len x m) == CSR arrays of A (m x vec_len),
 * exactly what SDPSolver::init hands to get_A (src/solver.cu:91-95).
 * -------------------------------------------------------------------------- */
typedef struct cuadmm_ysolve_s cuadmm_ysolve_t;

int  cuadmm_ysolve_create(int64_t m, int64_t vec_len, int64_t nnz,
                          const int32_t* h_A_rowptr, const int32_t* h_A_colind, const double* h_A_val,
                          double eps, int device, cuadmm_ysolve_t** out);
void cuadmm_ysolve_destroy(cuadmm_ysolve_t* ys);
int  cuadmm_ysolve(cuadmm_ysolve_t* ys, const double* d_rhs, double* d_y, void* stream);
int  cuadmm_ysolve_host(cuadmm_ysolve_t* ys, const double* h_rhs, double* h_y);
/* stats: out[0]=nnz(AAt lower) out[1]=nnz(L) out[2]=levels(sparse part) out[3]=dense tail size
 * out[4]=launches per solve out[5]=algorithmic bytes per solve */
int  cuadmm_ysolve_stats(const cuadmm_ysolve_t* ys, int64_t out[8]);
/* fill-reducing permutation used (length m), CHOLMOD's L->Perm analogue */
int  cuadmm_ysolve_perm(const cuadmm_ysolve_t* ys, int32_t* perm);

/* --------------------------------------------------------------------------
 * Solver: same argument lists as SDPSolver::init (include/cuadmm/solver.h:208-223)
 * and SDPSolver::solve (solver.h:236-244).  Host arrays are copied, never mutated.
 * -------------------------------------------------------------------------- */
typedef struct cuadmm_solver cuadmm_solver_t;

int  cuadmm_solver_create(cuadmm_solver_t** out);
void cuadmm_solver_destroy(cuadmm_solver_t* s);
/* quiet != 0 suppresses the reference-format stdout log */
int  cuadmm_solver_set_verbose(cuadmm_solver_t* s, int verbose);
int  cuadmm_solver_init(cuadmm_solver_t* s,
        int eig_stream_num_per_gpu, int cpu_eig_thread_num,
        int64_t vec_len, int64_t con_num,
        const int32_t* At_csc_col_ptrs, const int32_t* At_csc_row_ids, const double* At_csc_vals, int64_t At_nnz,
        const int32_t* b_indices, const double* b_vals, int64_t b_nnz,
        const int32_t* C_indices, const double* C_vals, int64_t C_nnz,
        const int32_t* blk_vals, int64_t mat_num,
        const double* X_vals, const double* y_vals, const double* S_vals, double sig);
/* Block cones of the problem, one letter per block ('s', 'l', 'u', see cuadmm_plan_create_typed), before init like
 * set_device / set_distributed; init then checks vec_len against the typed entry counts.  NULL: every block is 's'.
 * cuadmm_solver_init_from_problem takes the types of the problem instead. */
int  cuadmm_solver_set_block_types(cuadmm_solver_t* s, const char* types, int64_t mat_num);
int  cuadmm_solver_solve(cuadmm_solver_t* s, int max_iter, double stop_tol,
        int sig_update_threshold, int sig_update_stage_1, int sig_update_stage_2,
        int switch_admm, double sigscale, int if_first);
/* results (unscaled, as SDPSolver::X/y/S after solve), copied to host */
int  cuadmm_solver_get_X(cuadmm_solver_t* s, double* h_X);
int  cuadmm_solver_get_y(cuadmm_solver_t* s, double* h_y);
int  cuadmm_solver_get_S(cuadmm_solver_t* s, double* h_S);
/* warm-restart: replace X,y,S (unscaled) before solve(..., if_first=0) (src/solver.cu:385-409) */
int  cuadmm_solver_set_XyS(cuadmm_solver_t* s, const double* h_X, const double* h_y, const double* h_S, double sig);
/* New b and C for the same A, blocks and cones (receding-horizon re-solves), keeping everything init derived from A
 * and the blocks: normA, the SpMV operators, the A A^T factorisation, the projection plan, the shard and peer arena,
 * and the captured iteration graphs.  b and C are sparse host triplets as in cuadmm_solver_init (0-based, C by typed
 * svec offset, a repeated index keeps its last value, copied and never mutated); their pattern may differ from init's.
 * Collective on a sharded solver: every rank passes the same full arrays.  Out-of-range indices return CUADMM_EINVAL
 * and leave the solver as it was.  Follow with solve(..., if_first = 1).
 *   keep_iterate = 0: the next solve behaves like a fresh init with the same A / blocks, this b, C and sig and no
 *                     X0 / y0 / S0 (the Jacobi warm-start bases are reset to the identity);
 *   keep_iterate = 1: the start point is the X, y, S the last solve returned, as if given to a fresh init as
 *                     X0 / y0 / S0 (the Jacobi bases are kept, so agreement with that init is to rounding).
 * init loads b and C through the same device path, so a cold update agrees with a fresh init bit for bit unless a
 * block takes the dense sign path (n > 168), which is not reproducible run to run.  Its wall time is
 * cuadmm_solver_times out[6]. */
int  cuadmm_solver_update_data(cuadmm_solver_t* s,
        const int32_t* b_idx, const double* b_vals, int64_t b_nnz,
        const int32_t* C_idx, const double* C_vals, int64_t C_nnz,
        int keep_iterate, double sig);
/* info_iter_num and the per-iteration history (info_*_arr, src/solver.cu:802-810).
 * which: 0 pobj 1 dobj 2 errRp 3 errRd 4 relgap 5 sig 6 bscale 7 Cscale */
int64_t cuadmm_solver_iter_num(const cuadmm_solver_t* s);
int  cuadmm_solver_history(const cuadmm_solver_t* s, int which, double* out, int64_t cap);
/* timings in seconds: out[0]=total_time (since init or the last update_data, as the reference), out[1]=init,
 * out[2]=solve loop, out[3]=projection total, out[4]=y-solve total, out[5]=spmv total,
 * out[6]=last cuadmm_solver_update_data (0 before the first) */
int  cuadmm_solver_times(const cuadmm_solver_t* s, double out[8]);
int64_t cuadmm_solver_launches(const cuadmm_solver_t* s);
/* Measurement hook: enqueue `n_iters` iterations (sGS when sgs != 0, plain ADMM otherwise) from the
 * current state with the stop test disabled, bracketed by CUDA events on the solver's stream.
 * out_ms[0] = total device ms; with profile != 0 also out_ms[1] = projection stage (src/solver.cu:531-675),
 * out_ms[2] = both y-solves (:487-500,704-717), out_ms[3] = everything else (SpMVs + scalar kernel).
 * Requires solve() to have been called once (it sets the run parameters). */
int  cuadmm_solver_run_iterations(cuadmm_solver_t* s, int n_iters, int sgs, int profile, double out_ms[4]);
/* same with the finer breakdown (always profiled): out_ms[0..3] as above, out_ms[4] = K5 (A (S-C), its reduction over
 * ranks, rhsy), out_ms[5] = K8 (A X, its reduction over ranks, scalar update), out_ms[6] = dense-tail GEMVs of all y-solves */
int  cuadmm_solver_run_iterations_ex(cuadmm_solver_t* s, int n_iters, int sgs, double out_ms[8]);
/* y-solve statistics of the solver's factorisation (see cuadmm_ysolve_stats) */
int  cuadmm_solver_ysolve_stats(const cuadmm_solver_t* s, int64_t out[8]);

/* --------------------------------------------------------------------------
 * Multi-GPU: one process per GPU of one NVSwitch box.  Blocks are sharded by eig cost (cuadmm_plan_partition);
 * every rank owns X, S, C on its svec ranges and the column slice A[:, I_g]; the only per-iteration traffic is
 * the sum over ranks of the m-vector partial products A[:, I_g] x_g (2 per iteration) and the rows of the
 * dense-tail GEMVs of the y-solve, which are split over the ranks.  Transport: peer memory (CUDA IPC
 * arenas; the SpMV / GEMV / reduction kernels store straight into the peers' buffers over NVLink and
 * synchronise with system-scope flags, csrc/peer.h).
 * Replaces SDPDuoSolver's GPU workers + cudaMemcpyPeerAsync of dense blocks
 * (src/duo_solver.cu:266-336, 487-577).  Call cuadmm_solver_set_distributed BEFORE cuadmm_solver_init,
 * with the same 128-byte id on every rank (rank 0 creates it with cuadmm_unique_id and the launcher broadcasts
 * it); init/solve then take the FULL problem on every rank, get_X/get_S return full vectors (collective calls:
 * every rank must make them).  cuadmm_solver_set_distributed returns CUADMM_EINVAL in a process whose environment
 * asks for the removed NCCL transport (INTEGRATION.md §6).
 * -------------------------------------------------------------------------- */
/* kept for compatibility with callers of the removed NCCL transport: fills the same 128 random bytes as
 * cuadmm_unique_id */
int  cuadmm_nccl_unique_id(char out[128]);
/* 128 random bytes: the job id of a sharded solver */
int  cuadmm_unique_id(char out[128]);
int  cuadmm_solver_set_distributed(cuadmm_solver_t* s, int rank, int world, const char id[128]);
/* GPU of this solver (before init).  Default: CUADMM_DEVICE if set, else the calling thread's current device
 * (cudaGetDevice), so an MPI-style launcher that did cudaSetDevice(local_rank) needs nothing else. */
int  cuadmm_solver_set_device(cuadmm_solver_t* s, int device);
/* sharding logic on its own (host only; CPU tests): */
typedef struct cuadmm_shard cuadmm_shard_t;
int  cuadmm_shard_create(const int32_t* blk, int64_t nblk, int world, int rank, cuadmm_shard_t** out);
/* typed blocks (types == NULL: all 's'); a block is never split across ranks */
int  cuadmm_shard_create_typed(const char* types, const int32_t* blk, int64_t nblk, int world, int rank, cuadmm_shard_t** out);
void cuadmm_shard_destroy(cuadmm_shard_t* s);
/* cones of the local blocks (cuadmm_shard_info out[1] chars) */
int  cuadmm_shard_local_types(const cuadmm_shard_t* s, char* local_types);
/* out[0..3] = local svec length, local block count, global svec length, world */
int  cuadmm_shard_info(const cuadmm_shard_t* s, int64_t out[4]);
int  cuadmm_shard_maps(const cuadmm_shard_t* s, int32_t* local_blk, int64_t* local_block_ids, int64_t* loc2glob, int32_t* owner);
/* At (vec_len x ncols, CSC) -> rows owned by this rank, renumbered locally; returns the local nnz */
int64_t cuadmm_shard_slice_csc(const cuadmm_shard_t* s, int64_t ncols, const int32_t* col_ptrs, const int32_t* row_ids,
                               const double* vals, int32_t* out_col_ptrs, int32_t* out_row_ids, double* out_vals);

/* MEX-shaped one-shot entry: the cuadmm_MATLAB signature
 * (MATLAB/cuadmm_MATLAB.cu:197-433) over plain arrays.  At_stack is CSC
 * (vec_len x m), b / C_stack sparse columns, blk_vec doubles, X0/y0/S0 dense.
 * Outputs X,y,S (caller-allocated) and info arrays of length max_iter+1. */
int  cuadmm_solve_matlab_like(int eig_stream_num_per_gpu, int max_iter, double stop_tol,
        int64_t vec_len, int64_t con_num,
        const int64_t* At_jc, const int64_t* At_ir, const double* At_pr,
        const int64_t* b_ir, const double* b_pr, int64_t b_nnz,
        const int64_t* C_ir, const double* C_pr, int64_t C_nnz,
        const double* blk_vec, int64_t mat_num,
        const double* X0, const double* y0, const double* S0, double sig,
        int sig_update_threshold, int sig_update_stage_1, int sig_update_stage_2,
        int switch_admm, double sigscale,
        double* X, double* y, double* S,
        int64_t* iter_num, double* info /* 8 x (max_iter+1), row-major by `which` */, double* total_time);

/* --------------------------------------------------------------------------
 * Problem I/O: Problem::from_txt (src/problem.cu:11-83, src/utils/io.cu).
 * blk.txt holds one block per line: "s <n>" (or a bare "<n>"), "l <n>" or "u <n>"; any other letter is rejected
 * with CUADMM_EIO.  vec_len is the sum of the typed entry counts.
 * -------------------------------------------------------------------------- */
typedef struct cuadmm_problem cuadmm_problem_t;
int  cuadmm_problem_from_txt(const char* prefix, int warm_start, cuadmm_problem_t** out);
void cuadmm_problem_destroy(cuadmm_problem_t* p);
/* out[0..6] = vec_len, con_num, mat_num, At_nnz, b_nnz, C_nnz, has_warm_start */
int  cuadmm_problem_dims(const cuadmm_problem_t* p, int64_t out[8]);
/* which: 0 At_csc_col_ptrs(i32) 1 At_csc_row_ids(i32) 2 At_csc_vals(f64) 3 b_indices(i32)
 * 4 b_vals(f64) 5 C_indices(i32) 6 C_vals(f64) 7 blk_vals(i32) 8 X(f64) 9 y(f64) 10 S(f64)
 * 11 block types (char, mat_num letters 's' / 'l' / 'u', not NUL-terminated) */
const void* cuadmm_problem_array(const cuadmm_problem_t* p, int which);
int  cuadmm_solver_init_from_problem(cuadmm_solver_t* s, const cuadmm_problem_t* p,
        int eig_stream_num_per_gpu, int cpu_eig_thread_num, double sig);

#ifdef __cplusplus
}
#endif
#endif /* CUADMM_B200_H */
