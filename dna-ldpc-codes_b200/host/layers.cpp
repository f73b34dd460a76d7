#include "layers.h"

#include <algorithm>

#include "code.h"

namespace dnaldpc {

namespace {

// First fit in O(E * column degree): a column remembers the layers of the earlier rows it belongs to, and a row takes
// the smallest layer none of its columns remembers.
void compute(const Code &c, Layers &L) {
    L.layer_of_row.assign((size_t)c.M, 0);
    std::vector<std::vector<int32_t>> col_layers((size_t)c.N);
    std::vector<int32_t> taken;
    int n = c.M > 0 ? 1 : 0;
    for (int i = 0; i < c.M; i++) {
        taken.clear();
        for (int e = c.row_ptr[i]; e < c.row_ptr[i + 1]; e++) {
            const auto &cl = col_layers[(size_t)c.col_idx[e]];
            taken.insert(taken.end(), cl.begin(), cl.end());
        }
        std::sort(taken.begin(), taken.end());
        int l = 0;
        for (int32_t t : taken) {
            if (t > l) break;
            if (t == l) l++;
        }
        L.layer_of_row[(size_t)i] = l;
        n = std::max(n, l + 1);
        for (int e = c.row_ptr[i]; e < c.row_ptr[i + 1]; e++) col_layers[(size_t)c.col_idx[e]].push_back(l);
    }
    L.n_layers = n;
    L.ptr.assign((size_t)n + 1, 0);
    for (int i = 0; i < c.M; i++) L.ptr[(size_t)L.layer_of_row[(size_t)i] + 1]++;
    for (int l = 0; l < n; l++) L.ptr[(size_t)l + 1] += L.ptr[(size_t)l];
    std::vector<int32_t> fill(L.ptr.begin(), L.ptr.end() - 1);
    L.rows.resize((size_t)c.M);
    for (int i = 0; i < c.M; i++) L.rows[(size_t)fill[(size_t)L.layer_of_row[(size_t)i]]++] = i;
}

}  // namespace

const Layers &code_layers(const Code &c) {
    LayersCache &k = *c.layers;
    std::call_once(k.once, [&] { compute(c, k.layers); });
    return k.layers;
}

}  // namespace dnaldpc
