// plan.h — the projection plan: host block layout + device descriptors + launch classes.
#pragma once
#include "common.h"
#include "blocks.h"
#include "project_jacobi.cuh"

namespace cuadmm { struct DensePart; }
cuadmm::DensePart* dense_part_create(int device, const std::vector<int32_t>& blk, const std::vector<int64_t>& svec_off,
                                     const std::vector<int64_t>& which);
void dense_part_destroy(cuadmm::DensePart* p);
int dense_part_project(cuadmm::DensePart* D, const double* Xb, double* Xproj, cudaStream_t st,
                       const cuadmm::ProjEpilogue* epi, const int* done_flag);

namespace cuadmm {
// one CTA of proj_linear_kernel (cones.cu): a run of 'l' or 'u' entries of at most kLinearChunk entries
struct LinChunk {
    int64_t off;      // first svec entry
    int32_t len;
    int32_t cone;     // 'l' or 'u'
};
constexpr int kLinearChunk = 4096;
// the 'l' / 'u' blocks of a layout as chunks; consecutive blocks of one cone are merged first (they are contiguous)
std::vector<LinChunk> linear_chunks(const BlockLayout& layout);
// one launch for all chunks; returns the number of kernel launches (1)
int linear_project(const LinChunk* d_chunks, int64_t nchunks, const double* Xb, double* Xproj, cudaStream_t st,
                   const ProjEpilogue* epi, const int* done_flag);
}  // namespace cuadmm

struct cuadmm_plan {
    int device = -1;
    cuadmm::BlockLayout layout;

    // launch classes: blocks grouped by size range, each class = one kernel launch
    struct Class {
        int kind;          // index into kSizeClasses (project.cu), or the global-memory eigenvalue kernel (force_global)
        int nmax;          // largest n in the class
        int32_t count;     // blocks in the class
        int64_t first;     // first descriptor (in d_desc)
        size_t smem;       // dynamic shared memory per CTA
        int grid;
    };
    std::vector<Class> classes;
    std::vector<cuadmm::BlkDesc> h_desc;       // class-major, n descending inside a class
    cuadmm::DevBuf<cuadmm::BlkDesc> d_desc;
    cuadmm::DevBuf<double> d_scratch;          // n x n per block of the global-memory eigenvalue kernel (force_global)
    cuadmm::DevBuf<double> d_eig;              // debug eigenvalue output (sum n)
    cuadmm::DevBuf<int32_t> d_sweeps;
    cuadmm::DevBuf<double> d_in, d_out;        // staging for the *_host entry points
    // pooled-layout descriptors for svec<->smat
    cuadmm::DevBuf<int64_t> d_svec_off, d_mat_off;
    cuadmm::DevBuf<int32_t> d_blk;
    cuadmm::DevBuf<uint8_t> d_pool;

    // warm start of the Jacobi kernels: per block the orthonormal basis the last projection ended in
    cuadmm::DevBuf<double> d_Q;
    bool warm_start = true;
    void reset_warm_start();
    double threshold = 1e-11;     // columns of G count as orthogonal when every |cos| <= threshold (tested on the state after each sweep)
    int max_sweeps = 40;
    bool force_global = false;    // every block above the shared-memory classes on the global-memory Jacobi kernel, which yields
                                  // eigenvalues only (the shadow plan eig_plan; never set on a plan that projects)
    std::unique_ptr<cuadmm_plan> eig_plan;   // lazily built shadow plan: eigenvalues of the blocks on the dense sign path (debug entry only)
    int rank_limit = 0;           // > 0: fixed-rank projection (cuadmm_plan_set_rank_limit)
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::vector<cudaStream_t> side_streams;    // classes run concurrently on these
    std::vector<cudaEvent_t> side_events;
    cudaEvent_t fork_event = nullptr;
    cuadmm::DensePart* dense = nullptr;        // blocks n > 168: GEMM-only sign-function path (dense_proj.cu)
    // 'l' / 'u' blocks: one proj_linear_kernel launch over these chunks (cones.cu), on its own side stream when
    // anything else runs; a plan without such blocks issues no launch and no extra event
    std::vector<cuadmm::LinChunk> h_lin;
    cuadmm::DevBuf<cuadmm::LinChunk> d_lin;
    cudaStream_t lin_stream = nullptr;
    cudaEvent_t lin_event = nullptr;
    int64_t eig_len = 0;                       // sum of n over the 's' blocks: the device eigenvalue slots
    const int* done_flag = nullptr;            // device stop flag honoured by the kernels (solver)
    double last_ms = 0.0;
    int64_t last_launches = 0;

    ~cuadmm_plan();
    void build_device();
    // core launcher; epi may be null.  Returns the number of kernel launches.
    int project(const double* d_Xb, double* d_Xproj, cudaStream_t stream,
                const cuadmm::ProjEpilogue* epi, bool want_eig);
};
