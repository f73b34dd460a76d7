// layers.h - row layers of a parity-check matrix, the schedule of the layered min-sum decoder.
//
// Definition (part of the C ABI contract, include/dnaldpc.h): the rows are taken in ascending order and each goes to the
// lowest-numbered layer that holds no row sharing a column with it (first fit); a row without entries goes to layer 0.
// The checks of one layer therefore touch disjoint bits, so the order in which they are processed cannot matter.
#pragma once
#include <cstdint>
#include <mutex>
#include <vector>

namespace dnaldpc {

struct Code;

struct Layers {
    int n_layers = 0;
    std::vector<int32_t> layer_of_row;  // [M]
    std::vector<int32_t> rows;          // [M] rows grouped by layer, ascending inside a layer
    std::vector<int32_t> ptr;           // [n_layers + 1] layer l = rows[ptr[l] .. ptr[l+1])
};

// Per-code cache: computed at most once, when first asked for, and shared by every copy of the Code.
struct LayersCache {
    std::once_flag once;
    Layers layers;
};

// The row layers of `c` (cached in c.layers).
const Layers &code_layers(const Code &c);

}  // namespace dnaldpc
