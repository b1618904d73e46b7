// shard.h — block-level sharding of an SDP across GPUs (SURVEY 8e): every rank owns a cost-balanced
// set of PSD blocks = a set of svec ranges, and holds X, S, C restricted to them plus the column slice
// A[:, I_g].  Replaces the Duo solver's equal-count split + per-iteration peer copies of dense blocks
// (src/duo_solver.cu:266-295, 517-565): here no block data ever crosses NVLink, only the m-vector
// partial products A[:, I_g] x_g are summed over the ranks.  Host-only logic (tested on CPU with gloo).
#pragma once
#include "blocks.h"
#include <vector>

namespace cuadmm {

struct Shard {
    int rank = 0, world = 1;
    std::vector<int32_t> owner;          // per global block
    std::vector<int64_t> local_blocks;   // global block ids owned by this rank, ascending
    std::vector<int32_t> local_blk;      // their sizes
    std::vector<char> local_types;       // their cones ('s', 'l', 'u'); a block is never split across ranks
    std::vector<int64_t> glob2loc;       // per global svec entry: local index or -1
    std::vector<int64_t> loc2glob;       // per local svec entry
    int64_t vec_len = 0, vec_len_local = 0;
    std::vector<double> part_cost;

    void build(const BlockLayout& layout, int world, int rank);
    // At (vec_len x m, CSC by constraint) -> rows restricted to the owned svec entries, renumbered
    void slice_csc(int64_t ncols, const int32_t* col_ptrs, const int32_t* row_ids, const double* vals,
                   std::vector<int32_t>& out_col_ptrs, std::vector<int32_t>& out_row_ids, std::vector<double>& out_vals) const;
    void slice_vec(const double* full, std::vector<double>& local) const;
};

}  // namespace cuadmm

struct cuadmm_shard { cuadmm::Shard sh; };
