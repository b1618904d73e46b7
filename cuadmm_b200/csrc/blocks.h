// blocks.h — host-side block analysis: the reference's analyze_blk / is_large_mat /
// MatrixSizes / get_maps restated with 64-bit offsets, plus the eig-cost partition.
#pragma once
#include <stdint.h>
#include <vector>

namespace cuadmm {

// reference: src/matrix_sizes.cu:14-19
bool is_large_mat(int mat_size, int mat_num);

// Block cones, by their blk.txt letter: 's' PSD n x n (n(n+1)/2 svec entries), 'l' the nonnegative orthant R^n_+ and
// 'u' free variables R^n (n entries each, unscaled).
bool valid_cone(char type);
int64_t block_entries(char type, int64_t n);

struct BlockLayout {
    std::vector<int32_t> blk;        // block sizes in input order
    std::vector<char> types;         // block cones in input order ('s', 'l', 'u')
    std::vector<int64_t> svec_off;   // nblk+1 prefix sums of the entry counts (n(n+1)/2 for 's', n otherwise)
    int64_t vec_len = 0;
    int64_t linear_blocks = 0;       // 'l' and 'u' blocks; the pooled layout below describes the 's' blocks only

    // analyze_blk (src/utils/analyze_blk.cu:63-99): distinct sizes ascending + counts
    std::vector<int32_t> sizes, nums;
    std::vector<uint8_t> large;      // per distinct size: reference large/small class

    // MatrixSizes (src/matrix_sizes.cu:22-68)
    int64_t large_mat_num = 0, sum_large_mat_size = 0, total_large_mat_size = 0;
    int64_t small_mat_num = 0, sum_small_mat_size = 0, total_small_mat_size = 0;
    std::vector<int32_t> large_mat_sizes, large_mat_nums, small_mat_sizes, small_mat_nums;
    std::vector<int64_t> large_mat_start, large_W_start, small_mat_start, small_W_start;

    // per block (input order): pool (0 large / 1 small), dense offset in its pool, W offset in its pool
    std::vector<uint8_t> pool;
    std::vector<int64_t> mat_off, W_off;

    // types == nullptr: every block is 's'
    void init(const int32_t* blk_vals, int64_t nblk, const char* types = nullptr);
    bool all_psd() const { return linear_blocks == 0; }
    // the pooled dense layout (sizes, totals, maps, svec<->smat) has no place for 'l' / 'u' blocks
    void require_all_psd(const char* what) const;
    // get_maps (src/utils/get_maps.cu:80-134); int32 like the reference, so it refuses layouts
    // whose dense pools overflow int32 (the reference silently wraps there).
    void maps(int32_t* map_B, int32_t* map_M1, int32_t* map_M2) const;
    // LPT greedy on cost(type, n): largest first onto the least-loaded part. Deterministic.
    void partition(int nparts, int32_t* owner, double* part_cost) const;
    static double eig_cost(int n);
    static double block_cost(char type, int n);
};

}  // namespace cuadmm
