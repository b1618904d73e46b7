// shard.cpp — see shard.h.
#include "shard.h"
#include "common.h"

namespace cuadmm {

void Shard::build(const BlockLayout& layout, int world_, int rank_) {
    CUADMM_REQUIRE(world_ >= 1 && rank_ >= 0 && rank_ < world_, "bad rank/world");
    rank = rank_; world = world_;
    const int64_t nblk = (int64_t)layout.blk.size();
    owner.assign(nblk, 0);
    part_cost.assign(world, 0.0);
    layout.partition(world, owner.data(), part_cost.data());
    vec_len = layout.vec_len;
    glob2loc.assign(vec_len, -1);
    local_blocks.clear(); local_blk.clear(); local_types.clear(); loc2glob.clear();
    for (int64_t k = 0; k < nblk; ++k) {
        if (owner[k] != rank) continue;
        local_blocks.push_back(k);
        local_blk.push_back(layout.blk[k]);
        local_types.push_back(layout.types[k]);
        for (int64_t e = layout.svec_off[k]; e < layout.svec_off[k + 1]; ++e) {
            glob2loc[e] = (int64_t)loc2glob.size();
            loc2glob.push_back(e);
        }
    }
    vec_len_local = (int64_t)loc2glob.size();
}

void Shard::slice_csc(int64_t ncols, const int32_t* col_ptrs, const int32_t* row_ids, const double* vals,
                      std::vector<int32_t>& ocp, std::vector<int32_t>& ori, std::vector<double>& ov) const {
    ocp.assign(ncols + 1, 0);
    ori.clear(); ov.clear();
    for (int64_t c = 0; c < ncols; ++c) {
        for (int p = col_ptrs[c]; p < col_ptrs[c + 1]; ++p) {
            const int64_t l = glob2loc[row_ids[p]];
            if (l >= 0) { ori.push_back((int32_t)l); ov.push_back(vals[p]); }
        }
        ocp[c + 1] = (int32_t)ori.size();
    }
}

void Shard::slice_vec(const double* full, std::vector<double>& local) const {
    local.resize(vec_len_local);
    for (int64_t l = 0; l < vec_len_local; ++l) local[l] = full[loc2glob[l]];
}

}  // namespace cuadmm

using namespace cuadmm;

extern "C" {

int cuadmm_shard_create(const int32_t* blk, int64_t nblk, int world, int rank, cuadmm_shard_t** out) {
    return cuadmm_shard_create_typed(nullptr, blk, nblk, world, rank, out);
}

int cuadmm_shard_create_typed(const char* types, const int32_t* blk, int64_t nblk, int world, int rank, cuadmm_shard_t** out) {
    return guarded([&] {
        CUADMM_REQUIRE(out && (blk || nblk == 0), "null argument");
        *out = nullptr;
        BlockLayout layout;
        layout.init(blk, nblk, types);
        std::unique_ptr<cuadmm_shard> s(new cuadmm_shard());
        s->sh.build(layout, world, rank);
        *out = s.release();
    });
}

void cuadmm_shard_destroy(cuadmm_shard_t* s) { delete s; }

int cuadmm_shard_info(const cuadmm_shard_t* s, int64_t out[4]) {
    return guarded([&] {
        CUADMM_REQUIRE(s && out, "null argument");
        out[0] = s->sh.vec_len_local; out[1] = (int64_t)s->sh.local_blk.size(); out[2] = s->sh.vec_len; out[3] = s->sh.world;
    });
}

int cuadmm_shard_local_types(const cuadmm_shard_t* s, char* local_types) {
    return guarded([&] {
        CUADMM_REQUIRE(s && local_types, "null argument");
        std::copy(s->sh.local_types.begin(), s->sh.local_types.end(), local_types);
    });
}

int cuadmm_shard_maps(const cuadmm_shard_t* s, int32_t* local_blk, int64_t* local_block_ids, int64_t* loc2glob, int32_t* owner) {
    return guarded([&] {
        CUADMM_REQUIRE(s, "null argument");
        const Shard& h = s->sh;
        if (local_blk) std::copy(h.local_blk.begin(), h.local_blk.end(), local_blk);
        if (local_block_ids) std::copy(h.local_blocks.begin(), h.local_blocks.end(), local_block_ids);
        if (loc2glob) std::copy(h.loc2glob.begin(), h.loc2glob.end(), loc2glob);
        if (owner) std::copy(h.owner.begin(), h.owner.end(), owner);
    });
}

int64_t cuadmm_shard_slice_csc(const cuadmm_shard_t* s, int64_t ncols, const int32_t* col_ptrs, const int32_t* row_ids,
                               const double* vals, int32_t* out_col_ptrs, int32_t* out_row_ids, double* out_vals) {
    int64_t nnz = -1;
    guarded([&] {
        CUADMM_REQUIRE(s && col_ptrs && out_col_ptrs, "null argument");
        std::vector<int32_t> cp, ri; std::vector<double> v;
        s->sh.slice_csc(ncols, col_ptrs, row_ids, vals, cp, ri, v);
        std::copy(cp.begin(), cp.end(), out_col_ptrs);
        if (out_row_ids) std::copy(ri.begin(), ri.end(), out_row_ids);
        if (out_vals) std::copy(v.begin(), v.end(), out_vals);
        nnz = (int64_t)ri.size();
    });
    return nnz;
}

}  // extern "C"
