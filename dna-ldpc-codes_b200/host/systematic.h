// systematic.h - systematic form of a parity-check matrix over GF(2), the basis of the encoder.
//
// Definition (part of the C ABI contract, include/dnaldpc.h): scanning the columns from N-1 down to 0, column j is a
// parity column iff it is linearly independent of the parity columns already chosen (the pivot columns of the reduced
// row-echelon form of H with its column order reversed). R = rank(H) parity columns, K = N - R info columns, both lists
// ascending. Message bit t goes to info_cols[t]; parity bit i, at parity_cols[i], is XOR_t A[i][t] * m_t, where row i of
// A is the reduced row whose pivot is parity_cols[i], restricted to the info columns.
#pragma once
#include <cstdint>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

namespace dnaldpc {

struct Code;

// Size cap: the elimination keeps an M x M bit transform and the result holds R x K bits of A; each must fit in
// kSystematicMaxBits (2^33 bits = 1 GiB), otherwise the systematic form is refused with DNALDPC_ERR_UNSUPPORTED.
constexpr uint64_t kSystematicMaxBits = 1ull << 33;

struct Systematic {
    int K = 0, R = 0;
    std::vector<int32_t> info_cols, parity_cols;  // ascending
    int kw = 0;                                   // ceil(K / 32): 32-bit words of one message
    std::vector<uint32_t> A;                      // [R][kw], bit t of row i at word t / 32, bit t % 32
};

// Per-code cache: computed at most once, when first asked for, and shared by every copy of the Code.
struct SystematicCache {
    std::once_flag once;
    int rc = 0;
    std::string err;
    Systematic sys;
};

// The systematic form of `c` (cached in c.sys). Returns nullptr with *rc (a DNALDPC_* code) and *err set on failure.
const Systematic *systematic_form(const Code &c, int *rc, std::string *err);

}  // namespace dnaldpc
