// blocks.cpp — block analysis / pooled layout / svec maps / GPU partition (host only).
#include "blocks.h"
#include "common.h"
#include <algorithm>
#include <map>
#include <numeric>
#include <queue>

namespace cuadmm {

bool is_large_mat(int mat_size, int mat_num) {
    // reference heuristic (src/matrix_sizes.cu:14-19): single Xsyevd beats batched
    // Jacobi above 32, or when there are too few matrices of that size.
    if (mat_size > 32) return true;
    return ((double)mat_size - 17.0 > (double)mat_num * 1.4);
}

// LPT cost of one 'l' / 'u' entry in the unit of eig_cost (1e-7 us): proj_linear_kernel with the fused epilogue takes
// 0.0865 ms for 1e7 entries = 8.65e-6 us per entry (B200, 1000 W, profiles/cones_probe_r03.json)
static const double LINEAR_COST_PER_ENTRY = 86.0;

bool valid_cone(char type) { return type == 's' || type == 'l' || type == 'u'; }

int64_t block_entries(char type, int64_t n) { return type == 's' ? tri(n) : n; }

void BlockLayout::init(const int32_t* blk_vals, int64_t nblk, const char* types_in) {
    CUADMM_REQUIRE(nblk >= 0, "nblk < 0");
    blk.assign(blk_vals, blk_vals + nblk);
    if (types_in) types.assign(types_in, types_in + nblk); else types.assign(nblk, 's');
    svec_off.assign(nblk + 1, 0);
    linear_blocks = 0;
    for (int64_t k = 0; k < nblk; ++k) {
        CUADMM_REQUIRE(blk[k] >= 1, "block size must be >= 1");
        CUADMM_REQUIRE(valid_cone(types[k]), std::string("unknown block type '") + types[k] + "' (expected 's', 'l' or 'u')");
        svec_off[k + 1] = svec_off[k] + block_entries(types[k], blk[k]);
        if (types[k] != 's') ++linear_blocks;
    }
    vec_len = svec_off[nblk];

    // distinct sizes ascending with multiplicity (std::set order in the reference); 's' blocks only
    std::map<int32_t, int32_t> cnt;
    for (int64_t k = 0; k < nblk; ++k) if (types[k] == 's') cnt[blk[k]]++;
    sizes.clear(); nums.clear(); large.clear();
    for (auto& kv : cnt) {
        sizes.push_back(kv.first);
        nums.push_back(kv.second);
        large.push_back(is_large_mat(kv.first, kv.second) ? 1 : 0);
    }

    large_mat_num = sum_large_mat_size = total_large_mat_size = 0;
    small_mat_num = sum_small_mat_size = total_small_mat_size = 0;
    large_mat_sizes.clear(); large_mat_nums.clear(); small_mat_sizes.clear(); small_mat_nums.clear();
    large_mat_start.assign(1, 0); large_W_start.assign(1, 0);
    small_mat_start.assign(1, 0); small_W_start.assign(1, 0);
    std::map<int32_t, int> group_of;  // size -> index inside its pool's group list
    for (size_t i = 0; i < sizes.size(); ++i) {
        int64_t s = sizes[i], c = nums[i];
        if (large[i]) {
            large_mat_num += c; sum_large_mat_size += s * c; total_large_mat_size += c * s * s;
            group_of[sizes[i]] = (int)large_mat_sizes.size();
            large_mat_sizes.push_back(sizes[i]); large_mat_nums.push_back(nums[i]);
            large_mat_start.push_back(total_large_mat_size);
            large_W_start.push_back(sum_large_mat_size);
        } else {
            small_mat_num += c; sum_small_mat_size += s * c; total_small_mat_size += c * s * s;
            group_of[sizes[i]] = (int)small_mat_sizes.size();
            small_mat_sizes.push_back(sizes[i]); small_mat_nums.push_back(nums[i]);
            small_mat_start.push_back(total_small_mat_size);
            small_W_start.push_back(sum_small_mat_size);
        }
    }

    // per-block pooled offsets: groups ascending by size, blocks in blk order inside a group
    pool.assign(nblk, 0); mat_off.assign(nblk, 0); W_off.assign(nblk, 0);
    std::map<int32_t, int64_t> seen;
    std::map<int32_t, uint8_t> is_large_of;
    for (size_t i = 0; i < sizes.size(); ++i) is_large_of[sizes[i]] = large[i];
    for (int64_t k = 0; k < nblk; ++k) {
        if (types[k] != 's') continue;   // pool 0, offsets 0: never read
        int64_t s = blk[k];
        int64_t j = seen[blk[k]]++;
        int g = group_of[blk[k]];
        if (is_large_of[blk[k]]) {
            pool[k] = 0;
            mat_off[k] = large_mat_start[g] + j * s * s;
            W_off[k] = large_W_start[g] + j * s;
        } else {
            pool[k] = 1;
            mat_off[k] = small_mat_start[g] + j * s * s;
            W_off[k] = small_W_start[g] + j * s;
        }
    }
}

void BlockLayout::require_all_psd(const char* what) const {
    if (!all_psd())
        throw Error(CUADMM_EINVAL, std::string(what) + ": the plan holds 'l'/'u' blocks, which have no place in the "
                                   "reference's pooled dense layout (only all-'s' plans have one)");
}

void BlockLayout::maps(int32_t* map_B, int32_t* map_M1, int32_t* map_M2) const {
    require_all_psd("svec maps");
    CUADMM_REQUIRE(total_large_mat_size <= INT32_MAX && total_small_mat_size <= INT32_MAX &&
                   vec_len <= INT32_MAX,
                   "int32 svec maps requested for a layout that overflows int32 (the reference overflows here)");
    int64_t idx = 0;
    for (size_t k = 0; k < blk.size(); ++k) {
        const int64_t s = blk[k], o = mat_off[k];
        const int32_t b = pool[k];
        for (int64_t i = 0; i < s; ++i) {        // column of the upper triangle
            for (int64_t j = 0; j <= i; ++j) {   // row
                map_B[idx] = b;
                map_M1[idx] = (int32_t)(o + s * i + j);
                map_M2[idx] = (int32_t)(o + s * j + i);
                ++idx;
            }
        }
    }
}

double BlockLayout::eig_cost(int n) {
    // Calibrated on B200 (profiles/jacobi_tuning_r01.md, profiles/dense_probe_r01.json); unit = 1e-7 us,
    // only ratios matter for the LPT split.
    //   Jacobi regime (n <= 168): ~3e-6 us * n^3 per block at full-GPU batches (warm-started sweeps) + floor;
    //   dense regime: the sign iteration runs ~35 symmetric tile products; a block costs
    //   T(T+1)/2 tiles (T = ceil(n/128)) x n deep, ~0.06 us per tile per unit of depth.
    const double nn = (double)n;
    if (n <= 168) return 2.0e3 + 30.0 * nn * nn * nn;
    const double T = (double)((n + 127) / 128);
    return 6.0e5 * (0.5 * T * (T + 1.0)) * nn;
}

double BlockLayout::block_cost(char type, int n) {
    if (type == 's') return eig_cost(n);
    // 'l' / 'u': one streaming pass of the linear-cone kernel (56 B per entry with the fused epilogue) plus the floor of a
    // PSD block
    return 2.0e3 + LINEAR_COST_PER_ENTRY * (double)n;
}

void BlockLayout::partition(int nparts, int32_t* owner, double* part_cost) const {
    CUADMM_REQUIRE(nparts >= 1, "nparts < 1");
    const int64_t nblk = (int64_t)blk.size();
    std::vector<double> cost(nblk);
    for (int64_t k = 0; k < nblk; ++k) cost[k] = block_cost(types[k], blk[k]);
    std::vector<int64_t> order(nblk);
    std::iota(order.begin(), order.end(), 0);
    // (eig_cost is strictly increasing in n, so for all-'s' layouts this is the order by size)
    std::stable_sort(order.begin(), order.end(), [&](int64_t a, int64_t b) { return cost[a] > cost[b]; });
    std::vector<double> load(nparts, 0.0);
    // min-heap on (load, part index) keeps ties deterministic
    typedef std::pair<double, int> LP;
    std::priority_queue<LP, std::vector<LP>, std::greater<LP>> heap;
    for (int p = 0; p < nparts; ++p) heap.push(LP(0.0, p));
    for (int64_t t = 0; t < nblk; ++t) {
        LP top = heap.top(); heap.pop();
        int64_t k = order[t];
        owner[k] = top.second;
        top.first += cost[k];
        load[top.second] = top.first;
        heap.push(top);
    }
    if (part_cost) for (int p = 0; p < nparts; ++p) part_cost[p] = load[p];
}

}  // namespace cuadmm
