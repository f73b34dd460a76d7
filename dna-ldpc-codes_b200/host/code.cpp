#include "code.h"

#include <algorithm>
#include <cstdio>

#include "layers.h"
#include "systematic.h"

namespace dnaldpc {

std::string build_code(int M, int N, std::vector<int64_t> &pairs, Code &c) {
    if (M <= 0 || N <= 0) return "matrix dimensions must be positive";
    c.sys = std::make_shared<SystematicCache>();
    c.layers = std::make_shared<LayersCache>();
    std::sort(pairs.begin(), pairs.end());
    pairs.erase(std::unique(pairs.begin(), pairs.end()), pairs.end());  // insert() merges duplicates (mod2sparse.cpp:521-524)
    c.M = M; c.N = N; c.E = (int)pairs.size();
    c.row_ptr.assign((size_t)M + 1, 0);
    c.col_ptr.assign((size_t)N + 1, 0);
    c.col_idx.resize(pairs.size());
    c.col_edge.resize(pairs.size());
    for (size_t e = 0; e < pairs.size(); e++) {
        int r = (int)(pairs[e] >> 32), col = (int)(pairs[e] & 0xffffffff);
        if (r < 0 || r >= M || col < 0 || col >= N) return "entry out of range";
        c.row_ptr[r + 1]++;
        c.col_ptr[col + 1]++;
        c.col_idx[e] = col;
    }
    for (int i = 0; i < M; i++) c.row_ptr[i + 1] += c.row_ptr[i];
    for (int j = 0; j < N; j++) c.col_ptr[j + 1] += c.col_ptr[j];
    std::vector<int32_t> fill(c.col_ptr.begin(), c.col_ptr.end() - 1);
    for (int e = 0; e < c.E; e++) c.col_edge[fill[c.col_idx[e]]++] = e;  // e ascending == row ascending
    c.max_row_deg = c.max_col_deg = 0;
    c.regular_rows = c.regular_cols = true;
    for (int i = 0; i < M; i++) {
        int d = c.row_ptr[i + 1] - c.row_ptr[i];
        if (d != c.row_ptr[1] - c.row_ptr[0]) c.regular_rows = false;
        c.max_row_deg = std::max(c.max_row_deg, d);
    }
    for (int j = 0; j < N; j++) {
        int d = c.col_ptr[j + 1] - c.col_ptr[j];
        if (d != c.col_ptr[1] - c.col_ptr[0]) c.regular_cols = false;
        c.max_col_deg = std::max(c.max_col_deg, d);
    }
    return "";
}

namespace {
// Four bytes low to high, two's complement, independent of host endianness (intio.cpp:35-52).
bool rd_i32(FILE *f, int32_t &v) {
    unsigned char b[4];
    if (fread(b, 1, 4, f) != 4) return false;
    v = (int32_t)((uint32_t)b[0] | ((uint32_t)b[1] << 8) | ((uint32_t)b[2] << 16) | ((uint32_t)b[3] << 24));
    return true;
}
void wr_i32(std::vector<unsigned char> &o, int32_t v) {
    uint32_t u = (uint32_t)v;
    for (int i = 0; i < 4; i++) o.push_back((unsigned char)((u >> (8 * i)) & 0xff));
}
}  // namespace

int read_pchk(const std::string &path, Code &out, std::string &err) {
    FILE *f = fopen(path.c_str(), "rb");
    if (!f) { err = "Can't open parity check file: " + path; return 2; }
    int32_t v;
    if (!rd_i32(f, v) || v != ('P' << 8) + 0x80) {
        fclose(f);
        err = "File " + path + " doesn't contain a parity check matrix";
        return 3;
    }
    int32_t M = 0, N = 0;
    bool ok = rd_i32(f, M) && M > 0 && rd_i32(f, N) && N > 0;
    std::vector<int64_t> pairs;
    int row = -1;
    bool done = false;
    while (ok && !done) {
        if (!rd_i32(f, v)) { ok = false; break; }      // EOF before the 0 terminator
        if (v == 0) done = true;
        else if (v < 0) { row = -v - 1; if (row >= M) ok = false; }
        else {
            int col = v - 1;
            if (col >= N || row == -1) ok = false;
            else pairs.push_back(((int64_t)row << 32) | (uint32_t)col);
        }
    }
    fclose(f);
    if (!ok || !done) { err = "Error reading parity check matrix from " + path; return 3; }
    std::string e = build_code(M, N, pairs, out);
    if (!e.empty()) { err = e; return 3; }
    return 0;
}

int write_pchk(const std::string &path, const Code &c, std::string &err) {
    std::vector<unsigned char> o;
    o.reserve(4 * ((size_t)c.E + c.M + 4));
    wr_i32(o, ('P' << 8) + 0x80);
    wr_i32(o, c.M);
    wr_i32(o, c.N);
    for (int i = 0; i < c.M; i++) {
        if (c.row_ptr[i] == c.row_ptr[i + 1]) continue;
        wr_i32(o, -(i + 1));
        for (int e = c.row_ptr[i]; e < c.row_ptr[i + 1]; e++) wr_i32(o, c.col_idx[e] + 1);
    }
    wr_i32(o, 0);
    FILE *f = fopen(path.c_str(), "wb");
    if (!f) { err = "Can't create " + path; return 2; }
    bool ok = fwrite(o.data(), 1, o.size(), f) == o.size();
    ok = (fclose(f) == 0) && ok;
    if (!ok) { err = "Error writing " + path; return 2; }
    return 0;
}

void check_regular(const Code &c, int &dv, int &reg_dv, int &dc, int &reg_dc) {
    // Same outcome as the reference's running-max scan: D = max degree, flag = all degrees equal.
    // (dec.cpp:154-164 compares against the running max, which equals "all equal" in aggregate.)
    dv = dc = -1; reg_dv = reg_dc = 1;
    for (int j = 0; j < c.N; j++) {
        int t = c.col_ptr[j + 1] - c.col_ptr[j];
        if (dv == -1) dv = t;
        else { if (t != dv) reg_dv = 0; if (t > dv) dv = t; }
    }
    for (int i = 0; i < c.M; i++) {
        int t = c.row_ptr[i + 1] - c.row_ptr[i];
        if (dc == -1) dc = t;
        else { if (t != dc) reg_dc = 0; if (t > dc) dc = t; }
    }
}

}  // namespace dnaldpc
