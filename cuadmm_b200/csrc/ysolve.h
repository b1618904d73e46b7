// ysolve.h — device-resident  y = (A A^T + eps I)^-1 rhs.
#pragma once
#include "common.h"
#include "chol_host.h"
#include "peer.h"

namespace cuadmm {

// One pull-style sparse triangular sweep: unknown u is
//   x[u] = (rhs[u] - sum_p val[p] * x[dep[p]]) * inv_diag[u]
// Forward solve with L: u = row, deps = columns < u.  Backward solve with L^T: u = column,
// deps = rows > u.  Same kernels for both (see ysolve.cu for the level/phase scheme).
struct TriSweep {
    int64_t n_unknowns = 0;       // unknowns solved by this sweep
    int64_t nnz = 0;
    DevBuf<int64_t> ptr;          // per unknown (indexed by unknown id)
    DevBuf<int32_t> dep;
    DevBuf<double> val;
    DevBuf<double> inv_diag;
    DevBuf<int32_t> slot_rows;    // 8 entries per warp-slot: 8 short rows, or 1 long row + padding (-1)
    DevBuf<int32_t> slot_info;    // level | (is_long << 30)
    DevBuf<int64_t> level_ptr;    // first slot of every level (levels+1)
    std::vector<int64_t> h_level_ptr;
    struct Phase { bool narrow; int level0, level1; };
    std::vector<Phase> phases;    // launch plan: wide levels one by one, runs of narrow levels in one CTA
    int64_t n_slots = 0;
    int levels = 0;               // levels of the top part
    // subtree part: CTA t walks levels [sub_off[t], sub_off[t+1]-1) of sub_lvl_ptr (slot offsets)
    DevBuf<int64_t> sub_off, sub_lvl_ptr;
    int64_t n_sub = 0;            // all subtrees = n_sub_pack + n_sub_warp + n_sub_cta
    int64_t n_sub_cta = 0;        // generic CTA-per-subtree kernel (not packable), indexed by sub_off
    // packed subtrees (see tri_packed_kernel / tri_packed_warp_kernel); rows of the CTA-packed ones first
    int64_t n_sub_pack = 0, n_sub_warp = 0, pk_rows = 0;
    DevBuf<unsigned char> pk_stream, pk_blobs;
    DevBuf<int64_t> pk_chunk_off, pk_blob_off, pk_row_off, pk_ext_ptr;
    DevBuf<int32_t> pk_prow_u, pk_prow_src, pk_prow_out, pk_ext_dep, pk_heavy;
    int64_t pk_n_heavy = 0;      // rows with many external entries: one warp each in pk_gather_kernel
    DevBuf<double> pk_ext_val, pk_w;
    DevBuf<long long> pk_timeline;            // debug (CUADMM_YSOLVE_TIMELINE)
    std::vector<long long> pk_timeline_meta;
    size_t pk_smem = 0;
    bool pk_has_ext = false;
    int sub_depth = 0;
    bool subtrees_first = true;
};

// side stream + events to run the two subtree kernels of a sweep concurrently
struct SweepStreams {
    cudaStream_t side = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
};

// One triangular matrix of the dense tail (L22^-1 or L22^-T, tail unknowns relabelled, see ysolve_create), stored as
// its non-empty 64 x 64 tiles only: per 64-row tile row, runs of consecutive non-empty tiles.
struct TailMatrix {
    DevBuf<double> val;           // every run as 64 rows x its full width (a multiple of 64), row-major, at toff
    DevBuf<int32_t> tptr, tcol;   // runs per tile row (CSR); [first, last) column of every run
    DevBuf<int64_t> toff;
    DevBuf<int32_t> order;        // 8-row blocks, longest rows first (one-GPU kernel)
    DevBuf<int32_t> rank_order;   // sharded solver: this rank's 8-row blocks from tail_row0, longest rows first
    std::vector<double> cost;     // per tile row: columns read (work per row)
};

}  // namespace cuadmm

struct cuadmm_ysolve_s {
    int device = -1;
    int64_t m = 0;
    int64_t n_lead = 0, n_tail = 0;
    int64_t nnz_aat = 0, nnz_L = 0, n_deficient = 0;
    cuadmm::TriSweep fwd, bwd;
    cuadmm::DevBuf<int32_t> perm;      // perm[new] = old
    cuadmm::DevBuf<double> z;          // forward result (permuted order)
    cuadmm::DevBuf<double> x;          // backward result (permuted order)
    // dense tail: inverse of the trailing Cholesky block (lower) and its transpose (upper)
    cuadmm::TailMatrix tail[2];
    cuadmm::DevBuf<double> tail_tmp;
    cuadmm::DevBuf<double> d_rhs, d_y; // staging for the host entry
    std::vector<int32_t> h_perm;
    // sharded solver (peer.h): the rows of the two dense-tail GEMVs are split over the ranks by work; every rank
    // stores its rows straight into every rank's tail_tmp / x / y (all three live in the peer arena then)
    const cuadmm::PeerComm* peer = nullptr;
    double* tail_tmp_p = nullptr;       // == tail_tmp.p, or the arena copy
    double* x_p = nullptr;              // == x.p, or the arena copy
    cuadmm::PeerPtrs peer_tmp, peer_x;
    int64_t tail_row0[2] = {0, 0}, tail_row1[2] = {0, 0};   // this rank's rows of L22^-1 / L22^-T
    void enable_peer(const cuadmm::PeerComm* pc, size_t off_tmp, size_t off_x);
    void split_tail_rows(int world, int rank);
    cuadmm::DevBuf<double> split_part;  // split-column GEMV: partial sums per (row block, split)
    cuadmm::DevBuf<unsigned int> split_count;
    const int* done_flag = nullptr;
    std::vector<cudaEvent_t>* prof_ev = nullptr;   // profiling (solver): events around the dense-tail stage, tags 20 / 21
    std::vector<int>* prof_tag = nullptr;
    cuadmm::SweepStreams streams;
    ~cuadmm_ysolve_s();
    int launches_per_solve = 0;
    int64_t alg_bytes = 0;
    void solve(const double* d_rhs, double* d_y, cudaStream_t stream);
};

namespace cuadmm {
cuadmm_ysolve_s* ysolve_create(int64_t m, int64_t vec_len, int64_t nnz, const int32_t* rowptr, const int32_t* colind,
                               const double* val, double eps, int device);
}
