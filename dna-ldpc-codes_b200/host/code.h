// code.h - host-side parity-check matrix as flat CSR/CSC edge tables.
// Replaces the 4-way linked mod2sparse structure (mod2sparse.h:42-93) on the decode path: the only
// properties of it the decoder relies on are the traversal orders (rows by ascending column, columns by
// ascending row; mod2sparse_insert, mod2sparse.cpp:502-604), which fix the floating-point product order.
#pragma once
#include <cstdint>
#include <memory>
#include <string>
#include <vector>

namespace dnaldpc {

struct SystematicCache;
struct LayersCache;

struct Code {
    int M = 0, N = 0, E = 0;
    std::vector<int32_t> row_ptr;   // [M+1]
    std::vector<int32_t> col_idx;   // [E]   column of edge e (CSR order, ascending within a row)
    std::vector<int32_t> col_ptr;   // [N+1]
    std::vector<int32_t> col_edge;  // [E]   CSR edge ids of column j, ascending row
    int max_row_deg = 0, max_col_deg = 0;
    bool regular_rows = true, regular_cols = true;
    std::shared_ptr<SystematicCache> sys;  // systematic form (host/systematic.h), computed on first use
    std::shared_ptr<LayersCache> layers;   // row layers of the layered decoder (host/layers.h), computed on first use
};

// Build from (row, col) pairs in any order with duplicates; returns error text or "".
std::string build_code(int M, int N, std::vector<int64_t> &pairs, Code &out);
// .pchk reader (rcode.cpp:54-86, mod2sparse.cpp:381-427, intio.cpp:35-52). rc: 0 ok, 2 io, 3 format.
int read_pchk(const std::string &path, Code &out, std::string &err);
// .pchk writer (mod2sparse.cpp:338-376 + magic).
int write_pchk(const std::string &path, const Code &c, std::string &err);
// CheckRegular (dec.cpp:138-189)
void check_regular(const Code &c, int &dv, int &reg_dv, int &dc, int &reg_dc);

}  // namespace dnaldpc
