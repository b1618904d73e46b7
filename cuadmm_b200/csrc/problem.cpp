// problem.cpp — SDPT3-style TXT problem loader with the reference's file conventions
// (Problem::from_txt, src/problem.cpp... src/problem.cu:11-83; readers src/utils/io.cu:22-133,296-328;
// COO_to_CSC src/utils/io.cu:187-243).  Host-only.  Differences, all deliberate:
//   * one pass over each file with strtod/strtol instead of ifstream >> (At.txt reaches 100s of MB);
//   * `prefix` may or may not end in '/' (the reference string-concatenates and needs the slash);
//   * errors are returned (CUADMM_EIO) instead of exit(1);
//   * 64-bit counts; COO_to_CSC is a stable counting sort by (col,row) whose column pointers are
//     correct even when constraint 0 is empty (the reference's scan shifts them in that case).
#include "problem.h"
#include "blocks.h"
#include <algorithm>
#include <errno.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>

namespace cuadmm {

static bool read_file(const std::string& path, std::string& out) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) return false;
    fseek(f, 0, SEEK_END);
    long n = ftell(f);
    fseek(f, 0, SEEK_SET);
    out.resize((size_t)std::max<long>(n, 0));
    size_t got = n > 0 ? fread(&out[0], 1, (size_t)n, f) : 0;
    fclose(f);
    out.resize(got);
    return true;
}

static void require_file(const std::string& path, std::string& out) {
    if (!read_file(path, out))
        throw Error(CUADMM_EIO, "could not open file '" + path + "'. Please verify that the provided directory path is correct.");
}

// numbers separated by whitespace, like `file >> val`
static void parse_numbers(const std::string& s, std::vector<double>& out) {
    const char* p = s.c_str();
    const char* end = p + s.size();
    while (p < end) {
        char* q = nullptr;
        const double v = strtod(p, &q);
        if (q == p) break;   // ifstream >> stops at the first token that is not a number
        out.push_back(v);
        p = q;
    }
}

// blk.txt: "<letter> <int>" or "<int>" per line, other lines ignored (read_blk, io.cu:296-328); a bare "<int>" is 's'
static void parse_blk(const std::string& s, std::vector<char>& types, std::vector<int32_t>& vals) {
    size_t pos = 0;
    while (pos < s.size()) {
        size_t eol = s.find('\n', pos);
        if (eol == std::string::npos) eol = s.size();
        std::string line = s.substr(pos, eol - pos);
        pos = eol + 1;
        size_t a = 0, b = line.size();
        while (a < b && isspace((unsigned char)line[a])) ++a;
        while (b > a && isspace((unsigned char)line[b - 1])) --b;
        if (a == b) continue;
        char type = 's';
        size_t i = a;
        if (isalpha((unsigned char)line[i])) {
            type = line[i];
            ++i;
            if (i >= b || !isspace((unsigned char)line[i])) continue;   // needs whitespace after the letter
            while (i < b && isspace((unsigned char)line[i])) ++i;
        }
        size_t j = i;
        if (j < b && line[j] == '-') ++j;
        const size_t d0 = j;
        while (j < b && isdigit((unsigned char)line[j])) ++j;
        if (j == d0 || j != b) continue;   // malformed line: ignored like the reference's regexes
        types.push_back(type);
        vals.push_back((int32_t)strtol(line.c_str() + i, nullptr, 10));
    }
}

void Problem::from_txt(const std::string& prefix_in, bool warm_start) {
    std::string prefix = prefix_in;
    struct stat sb;
    if (!prefix.empty() && prefix.back() != '/' && stat(prefix.c_str(), &sb) == 0 && S_ISDIR(sb.st_mode)) prefix += '/';
    std::string buf;

    require_file(prefix + "blk.txt", buf);
    parse_blk(buf, blk_types, blk_vals);
    mat_num = (int64_t)blk_vals.size();

    if (warm_start) {
        require_file(prefix + "X.txt", buf); parse_numbers(buf, X_vals); vec_len = (int64_t)X_vals.size();
        require_file(prefix + "y.txt", buf); parse_numbers(buf, y_vals); con_num = (int64_t)y_vals.size();
        require_file(prefix + "S.txt", buf); parse_numbers(buf, S_vals);
    }
    int64_t vl = 0;
    for (int64_t i = 0; i < mat_num; ++i) {
        // 's' PSD, 'l' nonnegative orthant, 'u' free (SDPT3 letters); 'q' (second-order cones) is not supported
        if (!valid_cone(blk_types[i])) {
            throw Error(CUADMM_EIO, std::string("unknown block type '") + blk_types[i] + "' in blk.txt (expected s, l or u)");
        }
        if (blk_vals[i] < 1) throw Error(CUADMM_EIO, "non-positive block size in blk.txt");
        vl += block_entries(blk_types[i], blk_vals[i]);
    }
    if (!warm_start) {
        vec_len = vl;
        require_file(prefix + "con_num.txt", buf);
        std::vector<double> cn; parse_numbers(buf, cn);
        if (cn.empty()) throw Error(CUADMM_EIO, "con_num.txt is empty");
        con_num = (int64_t)cn[0];
    } else if (vl != vec_len) {
        throw Error(CUADMM_EIO, "the length of warmstarted X does not match the vector length.");
    }

    // At.txt: "row col val" with row = svec index, col = constraint (0-based)
    require_file(prefix + "At.txt", buf);
    std::vector<double> t; t.reserve(buf.size() / 8);
    parse_numbers(buf, t);
    At_nnz = (int64_t)(t.size() / 3);
    std::vector<int32_t> rows(At_nnz), cols(At_nnz);
    std::vector<double> vals(At_nnz);
    for (int64_t e = 0; e < At_nnz; ++e) { rows[e] = (int32_t)t[3 * e]; cols[e] = (int32_t)t[3 * e + 1]; vals[e] = t[3 * e + 2]; }
    std::vector<double>().swap(t);
    int32_t max_row = -1, max_col = -1;
    for (int64_t e = 0; e < At_nnz; ++e) {
        if (rows[e] < 0 || cols[e] < 0) throw Error(CUADMM_EIO, "negative index in At.txt");
        max_row = std::max(max_row, rows[e]); max_col = std::max(max_col, cols[e]);
    }
    if (max_row >= vec_len) throw Error(CUADMM_EIO, "At.txt has a row index beyond the svec length given by blk.txt");
    if (max_col >= con_num) throw Error(CUADMM_EIO, "At.txt has a column index beyond con_num");
    if (max_row != vec_len - 1) warnings.push_back("WARNING: the largest column index in At is different from the specified column number!");
    if (max_col != con_num - 1) warnings.push_back("WARNING: the largest row index in At is different from the SDP vector length!");
    coo_to_csc(con_num, rows, cols, vals, At_csc_col_ptrs, At_csc_row_ids, At_csc_vals);

    auto sparse_vec = [&](const std::string& name, int64_t limit, std::vector<int32_t>& idx, std::vector<double>& v) {
        require_file(prefix + name, buf);
        std::vector<double> tt; parse_numbers(buf, tt);
        const int64_t n = (int64_t)(tt.size() / 3);
        idx.resize(n); v.resize(n);
        for (int64_t e = 0; e < n; ++e) {
            idx[e] = (int32_t)tt[3 * e]; v[e] = tt[3 * e + 2];
            if (tt[3 * e + 1] != 0.0) warnings.push_back("WARNING: sparse vector data has a non-zero column index.");
            if (idx[e] < 0 || idx[e] >= limit) throw Error(CUADMM_EIO, name + " has an index out of range");
        }
    };
    sparse_vec("b.txt", con_num, b_indices, b_vals);
    sparse_vec("C.txt", vec_len, C_indices, C_vals);
    b_nnz = (int64_t)b_vals.size();
    C_nnz = (int64_t)C_vals.size();
}

void coo_to_csc(int64_t ncols, const std::vector<int32_t>& rows, const std::vector<int32_t>& cols,
                const std::vector<double>& vals, std::vector<int32_t>& col_ptrs, std::vector<int32_t>& row_ids,
                std::vector<double>& out_vals) {
    const int64_t nnz = (int64_t)vals.size();
    std::vector<int64_t> order(nnz);
    for (int64_t e = 0; e < nnz; ++e) order[e] = e;
    std::stable_sort(order.begin(), order.end(), [&](int64_t a, int64_t b) {
        if (cols[a] != cols[b]) return cols[a] < cols[b];
        return rows[a] < rows[b];
    });
    col_ptrs.assign(ncols + 1, 0);
    for (int64_t e = 0; e < nnz; ++e) col_ptrs[cols[e] + 1]++;
    for (int64_t c = 0; c < ncols; ++c) col_ptrs[c + 1] += col_ptrs[c];
    row_ids.resize(nnz); out_vals.resize(nnz);
    for (int64_t e = 0; e < nnz; ++e) { row_ids[e] = rows[order[e]]; out_vals[e] = vals[order[e]]; }
}

}  // namespace cuadmm

using namespace cuadmm;

extern "C" {

int cuadmm_problem_from_txt(const char* prefix, int warm_start, cuadmm_problem_t** out) {
    return guarded([&] {
        CUADMM_REQUIRE(prefix && out, "null argument");
        *out = nullptr;
        std::unique_ptr<cuadmm_problem> p(new cuadmm_problem());
        p->prob.from_txt(prefix, warm_start != 0);
        *out = p.release();
    });
}

void cuadmm_problem_destroy(cuadmm_problem_t* p) { delete p; }

int cuadmm_problem_dims(const cuadmm_problem_t* p, int64_t out[8]) {
    return guarded([&] {
        CUADMM_REQUIRE(p && out, "null argument");
        const Problem& q = p->prob;
        out[0] = q.vec_len; out[1] = q.con_num; out[2] = q.mat_num; out[3] = q.At_nnz; out[4] = q.b_nnz; out[5] = q.C_nnz;
        out[6] = q.X_vals.empty() ? 0 : 1; out[7] = (int64_t)q.warnings.size();
    });
}

const void* cuadmm_problem_array(const cuadmm_problem_t* p, int which) {
    if (!p) return nullptr;
    const Problem& q = p->prob;
    switch (which) {
        case 0: return q.At_csc_col_ptrs.data();
        case 1: return q.At_csc_row_ids.data();
        case 2: return q.At_csc_vals.data();
        case 3: return q.b_indices.data();
        case 4: return q.b_vals.data();
        case 5: return q.C_indices.data();
        case 6: return q.C_vals.data();
        case 7: return q.blk_vals.data();
        case 8: return q.X_vals.empty() ? nullptr : q.X_vals.data();
        case 9: return q.y_vals.empty() ? nullptr : q.y_vals.data();
        case 10: return q.S_vals.empty() ? nullptr : q.S_vals.data();
        case 11: return q.blk_types.data();
        default: return nullptr;
    }
}

}  // extern "C"
