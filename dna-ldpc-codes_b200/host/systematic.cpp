// systematic.cpp - systematic form of H (definition in systematic.h) by left-looking Gauss-Jordan elimination over GF(2).
//
// The row operations are kept as an M x M bit transform T (column-major, 64-bit words), so that the reduced column of H
// at j is T * h_j: the XOR of the T columns of the (few) rows that column j of the sparse H touches. The columns are
// visited from N-1 down to 0; a reduced column with a set bit in a row that holds no pivot yet is a new parity column,
// and its other set bits are cleared from the reduced matrix by updating T. At the end the reduced rows restricted to
// the info columns (A) are read off T * H the same way. Work: one T update (M x M bits at most) per pivot, three
// M-bit XORs per other column; no dense copy of H is ever formed.
#include "systematic.h"

#include <algorithm>
#include <new>
#include <thread>

#include "../../include/dnaldpc.h"
#include "code.h"

namespace dnaldpc {

namespace {

int compute(const Code &c, Systematic &s, std::string &err) {
    const int M = c.M, N = c.N;
    if ((uint64_t)M * (uint64_t)M > kSystematicMaxBits) {
        err = "systematic form: M = " + std::to_string(M) + " rows need an M x M elimination transform of more than 2^33 bits";
        return DNALDPC_ERR_UNSUPPORTED;
    }
    const size_t W = (size_t)(M + 63) / 64;
    std::vector<int32_t> edge_row((size_t)c.E);
    for (int i = 0; i < M; i++)
        for (int e = c.row_ptr[i]; e < c.row_ptr[i + 1]; e++) edge_row[(size_t)e] = i;
    std::vector<uint64_t> T((size_t)M * W, 0);  // column k at T[k * W]
    for (int k = 0; k < M; k++) T[(size_t)k * W + k / 64] = 1ull << (k % 64);
    std::vector<uint64_t> free_rows(W, ~0ull);  // rows that hold no pivot yet
    if (M % 64) free_rows[W - 1] = (1ull << (M % 64)) - 1;
    auto reduced_column = [&](int j, uint64_t *v) {  // v = T * h_j
        std::fill(v, v + W, 0ull);
        for (int q = c.col_ptr[j]; q < c.col_ptr[j + 1]; q++) {
            const uint64_t *t = &T[(size_t)edge_row[(size_t)c.col_edge[(size_t)q]] * W];
            for (size_t w = 0; w < W; w++) v[w] ^= t[w];
        }
    };
    std::vector<int32_t> piv_row((size_t)N, -1);  // pivot row of each parity column
    std::vector<uint64_t> v(W);
    int R = 0;
    for (int j = N - 1; j >= 0 && R < M; j--) {
        if (c.col_ptr[j] == c.col_ptr[j + 1]) continue;  // an empty column is always an info column
        reduced_column(j, v.data());
        size_t w = 0;
        while (w < W && !(v[w] & free_rows[w])) w++;
        if (w == W) continue;  // dependent on the parity columns chosen so far
        const int p = (int)(w * 64) + __builtin_ctzll(v[w] & free_rows[w]);
        const uint64_t pbit = 1ull << (p % 64);
        free_rows[(size_t)p / 64] &= ~pbit;
        piv_row[(size_t)j] = p;
        R++;
        v[(size_t)p / 64] ^= pbit;  // the rows to clear: every other set bit of the reduced column
        bool any = false;
        for (size_t q = 0; q < W && !any; q++) any = v[q] != 0;
        if (!any) continue;
        for (int k = 0; k < M; k++) {  // row r ^= row p for every r in v, applied to T column by column
            uint64_t *t = &T[(size_t)k * W];
            if (t[(size_t)p / 64] & pbit)
                for (size_t q = 0; q < W; q++) t[q] ^= v[q];
        }
    }
    const int K = N - R;
    if ((uint64_t)R * (uint64_t)K > kSystematicMaxBits) {
        err = "systematic form: the dense parity part A (R = " + std::to_string(R) + " x K = " + std::to_string(K) +
              " bits) exceeds the cap of 2^33 bits";
        return DNALDPC_ERR_UNSUPPORTED;
    }
    s.R = R;
    s.K = K;
    s.kw = (K + 31) / 32;
    s.info_cols.clear();
    s.parity_cols.clear();
    s.info_cols.reserve((size_t)K);
    s.parity_cols.reserve((size_t)R);
    std::vector<int32_t> prow;
    prow.reserve((size_t)R);
    for (int j = 0; j < N; j++) {
        if (piv_row[(size_t)j] >= 0) { s.parity_cols.push_back(j); prow.push_back(piv_row[(size_t)j]); }
        else s.info_cols.push_back(j);
    }
    // A[i][t] = bit prow[i] of T * h_{info_cols[t]}, 32 info columns (one word of every row of A) at a time; the word
    // columns are shared out over threads.
    s.A.assign((size_t)R * (size_t)s.kw, 0u);
    const int nthr = (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    auto work = [&](int tid) {
        std::vector<uint64_t> vs(32 * W);
        for (int b = tid; b < s.kw; b += nthr) {
            const int t0 = b * 32, nt = std::min(32, K - t0);
            for (int u = 0; u < nt; u++) reduced_column(s.info_cols[(size_t)(t0 + u)], &vs[(size_t)u * W]);
            for (int i = 0; i < R; i++) {
                const size_t pw = (size_t)prow[(size_t)i] / 64;
                const int pb = prow[(size_t)i] % 64;
                uint32_t word = 0;
                for (int u = 0; u < nt; u++) word |= (uint32_t)((vs[(size_t)u * W + pw] >> pb) & 1) << u;
                s.A[(size_t)i * s.kw + (size_t)b] = word;
            }
        }
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < nthr; t++) pool.emplace_back(work, t);
    work(0);
    for (auto &t : pool) t.join();
    return DNALDPC_OK;
}

}  // namespace

const Systematic *systematic_form(const Code &c, int *rc, std::string *err) {
    SystematicCache &k = *c.sys;
    std::call_once(k.once, [&] {
        try {
            k.rc = compute(c, k.sys, k.err);
        } catch (const std::bad_alloc &) {
            k.rc = DNALDPC_ERR_NOMEM;
            k.err = "systematic form: out of host memory";
        }
        if (k.rc) k.sys = Systematic{};
    });
    if (k.rc) { *rc = k.rc; *err = k.err; return nullptr; }
    return &k.sys;
}

}  // namespace dnaldpc
