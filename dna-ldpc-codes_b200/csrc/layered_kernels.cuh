// layered_kernels.cuh - row-layered normalised min-sum (DNALDPC_FLAG_MINSUM | DNALDPC_FLAG_LAYERED) on the slot engine.
//
// Schedule (DESIGN.md §5e, include/dnaldpc.h): one iteration runs the layers of host/layers.h in ascending order; a
// check of layer l sees the posteriors the layers before it have already updated in the same iteration. The checks of
// one layer touch disjoint bits, so one launch per layer updates them all at once with no ordering between warps.
//
// Data layout (same slot groups as the flooding decoder, lane = slot):
//   q     [G][N][32] T    posterior LLR of every bit: the `lratio` array. The setup kernel writes the channel LLR there
//                         for admitted slots; the channel value is not needed once q has been initialised.
//   state [G][M][W][32] T compressed check state in the `msg` allocation: [0] alpha*min1, [1] alpha*min2, then
//                         kMetaWords 32-bit words packed into T-sized elements: word 0 = index of min1 | parity << 8
//                         (parity of the negative v), words 1.. = the sign bits of v (bit k%32 of word 1+k/32 = v_k < 0).
//                         compact_move_kernel moves M*W elements per slot, like the E messages of the flooding decoder.
//   decw  [G][N] u32      hard decisions; each check writes the words of its bits, so a bit's last write in an iteration
//                         comes from its last layer and the syndrome kernel runs unchanged.
// Every step is one IEEE operation in T and ties in the minimum change no value, so the result does not depend on the
// thread mapping: the decoder is bit-exact against a sequential C oracle (tests/layered_oracle.c).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "bp_kernels.cuh"

namespace dnaldpc {

template <typename T, int DC>
struct LayerState {
    static constexpr int kSignWords = (DC + 31) / 32;
    static constexpr int kMetaWords = 1 + kSignWords;
    static constexpr int kMetaElems = (kMetaWords * 4 + (int)sizeof(T) - 1) / (int)sizeof(T);
    static constexpr int W = 2 + kMetaElems;  // T-sized elements per check and slot
};

// Degree class the layer kernel is instantiated for (its register arrays are sized by it), and the state size it implies.
inline int layer_dc(int max_row_deg) { return max_row_deg <= 8 ? 8 : max_row_deg <= 32 ? 32 : max_row_deg <= 72 ? 72 : 128; }
template <typename T> inline int layer_state_w(int dc) {
    return dc == 8 ? LayerState<T, 8>::W : dc == 32 ? LayerState<T, 32>::W : dc == 72 ? LayerState<T, 72>::W : LayerState<T, 128>::W;
}

// 32-bit words <-> T-sized elements of the slot-interleaved state (fp64: two words per element, low word first).
__device__ __forceinline__ void meta_store(float *p, const uint32_t *w, int e) { p[0] = __uint_as_float(w[e]); }
__device__ __forceinline__ void meta_store(double *p, const uint32_t *w, int e) {
    p[0] = __hiloint2double((int)w[2 * e + 1], (int)w[2 * e]);
}
__device__ __forceinline__ void meta_load(const float *p, uint32_t *w, int e) { w[e] = __float_as_uint(p[0]); }
__device__ __forceinline__ void meta_load(const double *p, uint32_t *w, int e) {
    const double v = p[0];
    w[2 * e] = (uint32_t)__double2loint(v);
    w[2 * e + 1] = (uint32_t)__double2hiint(v);
}

template <typename T> __device__ __forceinline__ T clamp_lmax(T x) {
    const T L = (T)kLayeredLlrMax;  // bp_kernels.cuh: |q| <= 2^64
    return x < -L ? -L : (x > L ? L : x);
}

// One launch per layer. A warp is (check of the layer, group of 32 slots), a lane is a slot. KEEP: the v_k of a lane
// stay in registers between the min pass and the update pass; otherwise (fp64 rows of degree > 72, which would not fit)
// the update pass re-derives v_k = q - c2v_old with the same operation, q being untouched by the other checks of the layer.
template <typename T, int DC, bool KEEP>
__global__ void __launch_bounds__(kRowWarps * 32)
layer_pass_kernel(T *__restrict__ state, T *__restrict__ q, uint32_t *__restrict__ decw, const uint32_t *__restrict__ actw,
                  const uint32_t *__restrict__ freshw, const int32_t *__restrict__ row_ptr,
                  const int32_t *__restrict__ col_idx, const int32_t *__restrict__ rows, int nrows, int M, int N, int g0,
                  int G, T alpha) {
    using S = LayerState<T, DC>;
    constexpr int W = S::W;
    const int lane = threadIdx.x & 31;
    const long long item = (long long)blockIdx.x * kRowWarps + (threadIdx.x >> 5);
    if (item >= (long long)G * nrows) return;
    const int gl = (int)(item / nrows), r = (int)(item - (long long)gl * nrows);
    const int g = g0 + gl;
    const uint32_t act = actw[g];
    if (act == 0) return;
    const bool on = (act >> lane) & 1u;
    const bool fresh = (freshw[g] >> lane) & 1u;  // first iteration of the frame: every c2v is 0
    const int i = __ldg(rows + r);
    const int e0 = __ldg(row_ptr + i), deg = __ldg(row_ptr + i + 1) - e0;
    T *st = state + ((size_t)g * M + i) * W * kFG + lane;
    T *ql = q + (size_t)g * N * kFG + lane;

    // previous message of this check: c2v_k = (par ^ sign_k) ? -mag_k : mag_k, mag_k = k == idx ? m2 : m1
    T om1 = T(0), om2 = T(0);
    uint32_t ow[S::kMetaElems * (int)sizeof(T) / 4];
#pragma unroll
    for (int w = 0; w < S::kMetaElems * (int)sizeof(T) / 4; w++) ow[w] = 0;
    const bool old = on && !fresh;
    if (old) {
        om1 = st[0];
        om2 = st[kFG];
#pragma unroll
        for (int e = 0; e < S::kMetaElems; e++) meta_load(st + (size_t)(2 + e) * kFG, ow, e);
    }
    const int oidx = (int)(ow[0] & 0xffu);
    const uint32_t opar = (ow[0] >> 8) & 1u;
    auto old_c2v = [&](int k) -> T {
        const T mag = k == oidx ? om2 : om1;
        return (opar ^ ((ow[1 + (k >> 5)] >> (k & 31)) & 1u)) ? -mag : mag;
    };

    // pass 1: v_k = q_k - c2v_k, the two smallest |v| (first minimum wins), the index of the first and the signs
    T v[KEEP ? DC : 1];
    T m1 = T(INFINITY), m2 = T(INFINITY);
    int i1 = 0;
    uint32_t par = 0, sw[S::kSignWords];
#pragma unroll
    for (int w = 0; w < S::kSignWords; w++) sw[w] = 0;
#pragma unroll
    for (int k = 0; k < DC; k++) {
        if (k < deg) {
            const int j = __ldg(col_idx + e0 + k);
            const T qk = on ? ql[(size_t)j * kFG] : T(0);
            const T vk = qk - old_c2v(k);
            if (KEEP) v[KEEP ? k : 0] = vk;
            const T a = fabs(vk);
            const uint32_t neg = vk < T(0) ? 1u : 0u;
            sw[k >> 5] |= neg << (k & 31);
            par ^= neg;
            if (a < m1) { m2 = m1; m1 = a; i1 = k; }
            else if (a < m2) m2 = a;
        }
    }
    const T s1 = deg >= 2 ? mul_rn(alpha, m1) : T(0);  // mu of every edge but the first minimum's
    const T s2 = deg >= 2 ? mul_rn(alpha, m2) : T(0);  // mu of the first minimum's edge (0: no other edge)

    // pass 2: new c2v, q = clamp(v + c2v), decisions by ballot
    uint32_t *dw = decw + (size_t)g * N;
#pragma unroll
    for (int k = 0; k < DC; k++) {
        if (k < deg) {
            const int j = __ldg(col_idx + e0 + k);
            T vk;
            if (KEEP) vk = v[KEEP ? k : 0];
            else vk = (on ? ql[(size_t)j * kFG] : T(0)) - old_c2v(k);
            const T mag = k == i1 ? s2 : s1;
            const T c = (par ^ ((sw[k >> 5] >> (k & 31)) & 1u)) ? -mag : mag;
            const T qn = clamp_lmax(vk + c);
            if (on) ql[(size_t)j * kFG] = qn;
            const uint32_t b = __ballot_sync(0xffffffffu, !(qn > T(0)));
            if (lane == 0) dw[j] = (act == 0xffffffffu) ? b : ((b & act) | (dw[j] & ~act));
        }
    }
    if (on) {
        st[0] = s1;
        st[kFG] = s2;
        uint32_t nw[S::kMetaElems * (int)sizeof(T) / 4];
        nw[0] = (uint32_t)i1 | (par << 8);
#pragma unroll
        for (int w = 0; w < S::kSignWords; w++) nw[1 + w] = sw[w];
#pragma unroll
        for (int w = 1 + S::kSignWords; w < S::kMetaElems * (int)sizeof(T) / 4; w++) nw[w] = 0;
#pragma unroll
        for (int e = 0; e < S::kMetaElems; e++) meta_store(st + (size_t)(2 + e) * kFG, nw, e);
    }
}

}  // namespace dnaldpc
