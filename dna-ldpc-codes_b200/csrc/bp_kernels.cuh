// bp_kernels.cuh - hand-written sm_100a kernels of the flooding sum-product decoder.
//
// Data layout in HBM. The decoder owns S = 32*G "slots" (G groups of 32); a slot holds one frame from the moment it is
// admitted until its syndrome is zero (or max_iter is hit), then it is harvested and refilled with the next pending
// frame ("continuous batching": every warp lane keeps doing useful work although frames need different iteration
// counts). A warp is always "one node x the 32 slots of a group":
//   msg   [G][E][32] T     ONE in-place message per edge: holds pr (bit->check, p0/p1) before the check-node pass
//                          and lr (check->bit) after it. Edge order = CSR (row-major, ascending column), so the 72
//                          messages x 32 slots of a check are one contiguous 18 KB run.
//   lratio[G][N][32] T     channel likelihood ratios
//   decw  [G][N]  u32      hard decisions, bit f of a word = slot f of the group (warp ballot)
//   actw/donew/newfw/freshw/harvw [G] u32   slot state masks;  slot_frame/slot_iter [G*32]
// Every global access of a warp is one fully used 256 B (fp64) / 128 B (fp32) segment.
//
// Reference semantics: Iter_Belief_Propagation dec.cpp:632-694, check() check.cpp:28-47,
// Run_Belief_Propagation_Decoder dec.cpp:583-605.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "bp_math.cuh"
#include "rng.cuh"

namespace dnaldpc {

constexpr int kFG = 32;  // slots per group == warp width

template <typename T> __device__ __forceinline__ T ld_stream(const T *p) { return __ldcs(p); }
template <typename T> __device__ __forceinline__ void st_stream(T *p, T v) { __stcs(p, v); }

// ------------------------------------------------------------------------------------------------
// Check-node (row) pass, dec.cpp:644-662.  One thread = one (check i, slot f); one warp = check i of 32 slots.
//   d_k = 1 - 2/(1+pr_k);  F_0 = 1, F_{k+1} = F_k*d_k;  B_last = 1, B_{k-1} = B_k*d_k;  lr_k = (1+F_k*B_k)/(1-F_k*B_k)
// The reference evaluates d_k twice (identical values) and parks F_k in e->lr; here the d_k live in registers,
// the backward products are check-pointed every 8 edges and re-derived block by block with the same
// multiplications in the same order, so every rounded intermediate is the reference's.
// A FRESH slot (first iteration of its frame) reads pr_e = lratio[col(e)] (Init_Belief_Propagation, dec.cpp:608-629)
// instead of msg, which removes the E-sized initialisation write.
// ------------------------------------------------------------------------------------------------

// Out-of-line fallback for one (check, slot) whose inputs left the proven operand ranges. Same operations in the
// same order as the reference, with nvcc's full-range divisions; F_k is re-derived for every k (O(deg^2)) because the
// single in-place message array has no room to park it. Reached only with invalid (negative / NaN) likelihood ratios.
template <typename T>
__device__ __noinline__ void row_slow_path(T *base, const T *lr_lane, const int32_t *cols, int deg, bool fresh) {
    auto pr_at = [&](int k) -> T { return fresh ? lr_lane[(size_t)cols[k] * kFG] : base[(size_t)k * kFG]; };
    T B = T(1);
    for (int k = deg - 1; k >= 0; k--) {
        T F = T(1);
        for (int m = 0; m < k; m++) F = mul_rn(F, check_factor_slow(pr_at(m)));
        const T dk = check_factor_slow(pr_at(k));
        base[(size_t)k * kFG] = check_to_bit_slow(mul_rn(F, B));
        B = mul_rn(B, dk);
    }
}

// The arithmetic of one (check, slot): d[] holds pr_k on entry; writes lr_k to base[k*32]. One basic block.
template <typename T, int DC, bool EXACT>
__device__ __forceinline__ void row_compute(T (&d)[DC], int deg, T *base, const T *lr_lane, const int32_t *cols, bool fresh) {
    constexpr int NB = (DC + 7) / 8;
    T ck[NB];
    T B = T(1);
    bool bad = false;
#pragma unroll
    for (int k = DC - 1; k >= 0; k--) {
        T dk = (EXACT || k < deg) ? check_factor(d[k], bad) : T(1);  // padding edges: exact identity in both chains
        d[k] = dk;
        if ((k & 7) == 7 || k == DC - 1) ck[k >> 3] = B;
        B = mul_rn(B, dk);
    }
    if (bad) {  // invalid likelihood ratios (negative / NaN): redo this check with full IEEE divisions, nothing stored yet
        row_slow_path<T>(base, lr_lane, cols, deg, fresh);
        return;
    }
    T F = T(1);
#pragma unroll
    for (int b = 0; b < NB; b++) {
        const int bot = b * 8;
        const int top = (bot + 7 < DC - 1) ? bot + 7 : DC - 1;
        T Bv[8];
        Bv[top - bot] = ck[b];
#pragma unroll
        for (int k = top; k > bot; k--) Bv[k - 1 - bot] = mul_rn(Bv[k - bot], d[k]);
#pragma unroll
        for (int k = bot; k <= top; k++) {
            T t = mul_rn(F, Bv[k - bot]);
            T lr = check_to_bit(t);
            if (EXACT || k < deg) st_stream(base + (size_t)k * kFG, lr);
            F = mul_rn(F, d[k]);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Floating-point min-sum (SURVEY 8f-4): Run_MSA_Decoder_INF, dec.cpp:1216-1250, in the LLR domain (positive = bit 0).
//   check node (Check_Update_MSA_INF, dec.cpp:1398-1433): c2v_k = prod_{m != k} sign(v2c_m) * min_{m != k} |v2c_m|
//   (sign(x) = +1 when x >= 0), 0 for a check of degree 1
//   bit node (Variable_Update_MSA_INF, dec.cpp:1597-1618): v2c_k = LLR + sum_{m != k} c2v_m, added in ascending row
//   decision (Decision_MSA_INF, dec.cpp:1659-1677): L = LLR + sum_m c2v_m; bit = !(L > 0)
// Same slot layout and scheduler; `lratio` holds the channel LLR, `msg` holds v2c before / c2v after the check pass.
// ------------------------------------------------------------------------------------------------
enum Alg { ALG_BP = 0, ALG_MINSUM = 1 };

template <typename T, int DC, bool EXACT>
__device__ __forceinline__ void row_compute_minsum(T (&d)[DC], int deg, T *base) {
    // smallest and second smallest magnitude (the first of equal magnitudes counts as "the" minimum, as in the
    // reference's strict `mag_min > abs(..)` scan; equal values make the choice invisible), and the sign parity
    T m1 = T(-1), m2 = T(-1);
    int i1 = -1, neg = 0;
#pragma unroll
    for (int k = 0; k < DC; k++) {
        if (EXACT || k < deg) {
            const T a = fabs(d[k]);
            neg ^= !(d[k] >= T(0));
            if (i1 < 0 || m1 > a) { m2 = m1; m1 = a; i1 = k; }
            else if (m2 < T(0) || m2 > a) m2 = a;
        }
    }
#pragma unroll
    for (int k = 0; k < DC; k++) {
        if (EXACT || k < deg) {
            T mag = (k == i1) ? m2 : m1;
            if (mag < T(0)) mag = T(0);                       // degree-1 check: no other edge (dec.cpp:1426-1427)
            const int sneg = neg ^ (!(d[k] >= T(0)));         // parity of negative signs among the OTHER edges
            st_stream(base + (size_t)k * kFG, (sneg ? T(-1) : T(1)) * mag);
        }
    }
}

// One (check i, slot f of group g): the DC loads go straight into the registers that then hold d_k, so all of them are
// in flight at once. `mixed` (warp-uniform) = some lane of the warp starts a new frame and gathers lratio instead.
template <typename T, int DC, bool EXACT, int ALG>
__device__ __forceinline__ void row_thread(T *__restrict__ msg, const T *__restrict__ lratio,
                                           const int32_t *__restrict__ row_ptr, const int32_t *__restrict__ col_idx,
                                           int N, int E, int g, int i, int f, bool fresh, bool mixed) {
    const int e0 = EXACT ? i * DC : row_ptr[i];
    const int deg = EXACT ? DC : (row_ptr[i + 1] - e0);
    T *base = msg + ((size_t)g * E + e0) * kFG + f;
    const T *lr_lane = lratio + (size_t)g * N * kFG + f;
    T d[DC];
    if (!mixed) {
#pragma unroll
        for (int k = 0; k < DC; k++)
            if (EXACT || k < deg) d[k] = ld_stream(base + (size_t)k * kFG);
    } else {  // a slot that starts a new frame: its pr_e is the channel ratio of the edge's bit
#pragma unroll
        for (int k = 0; k < DC; k++)
            if (EXACT || k < deg) {
                const T *src = fresh ? lr_lane + (size_t)__ldg(col_idx + e0 + k) * kFG : base + (size_t)k * kFG;
                d[k] = *src;  // default cache policy: a bit's lratio is re-read by every check it belongs to
            }
    }
    if (ALG == ALG_MINSUM) row_compute_minsum<T, DC, EXACT>(d, deg, base);
    else row_compute<T, DC, EXACT>(d, deg, base, lr_lane, col_idx + e0, fresh);
}

constexpr int kRowWarps = 4;

// One warp per (check, group), lane = slot; every global access is one fully used 256 B segment.
// (Measured alternative, removed: slot-major kernels - a warp = 32 checks of ONE slot - for groups thinned out in the
// drain tail of a batch. All 32 lanes then do useful arithmetic, but every lane touches its own 32 B sector and L1
// wavefront; on B200 that was 10-20 % slower end to end than letting thin groups run through this kernel.)
template <typename T, int DC, bool EXACT, int ALG>
__global__ void __launch_bounds__(kRowWarps * 32)
row_pass_kernel(T *__restrict__ msg, const T *__restrict__ lratio, const uint32_t *__restrict__ actw,
                const uint32_t *__restrict__ freshw, const int32_t *__restrict__ row_ptr,
                const int32_t *__restrict__ col_idx, int M, int N, int E, int g0, int G) {
    const int lane = threadIdx.x & 31;
    const long long item = (long long)blockIdx.x * kRowWarps + (threadIdx.x >> 5);
    if (item >= (long long)G * M) return;
    const int gl = (int)(item / M), i = (int)(item - (long long)gl * M);
    const int g = g0 + gl;
    const uint32_t act = actw[g];
    if (!((act >> lane) & 1u)) return;            // finished / empty slots keep their messages untouched
    const uint32_t fw = freshw[g];                // warp-uniform
    row_thread<T, DC, EXACT, ALG>(msg, lratio, row_ptr, col_idx, N, E, g, i, lane, (fw >> lane) & 1u, fw != 0);
}

// ---- TMA (cp.async.bulk) + mbarrier helpers --------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// global -> shared bulk copy (SASS: UBLKCP), completion signalled on the mbarrier as transferred bytes
__device__ __forceinline__ void tma_load_1d(void *smem_dst, const void *gsrc, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// Same with an L2 evict-first policy: the message stream is read once per pass and should not push out the few lines
// that ARE reused inside a pass (the channel ratios gathered by lanes that start a frame: 8 checks per bit).
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void tma_load_1d_hint(void *smem_dst, const void *gsrc, uint32_t bytes, uint64_t *bar, uint64_t policy) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)), "l"(policy) : "memory");
}

// Arithmetic of one (check, slot) whose DC inputs sit in the lane's column of a shared-memory tile (col[k * 32]):
// pass 1, descending: d_k in place, backward products check-pointed every 8 edges; pass 2: lr_k streamed to `base`.
// EXACT = false: rows of any degree deg <= DC (irregular codes); the padding edges k >= deg are exact identities in
// both product chains and are neither read nor stored.
template <typename T, int DC, bool EXACT = true>
__device__ __forceinline__ void smem_row_compute(T *col, T *base, const T *lr_lane, const int32_t *cols, bool fresh, int deg = DC) {
    constexpr int NB = (DC + 7) / 8;
    static_assert(EXACT || DC % 8 == 0, "irregular rows: the tile is a whole number of blocks");
    T ck[NB];
    T B = T(1);
    bool bad = false;
    if (EXACT) {
#pragma unroll
        for (int k = DC - 1; k >= 0; k--) {
            const T dk = check_factor(col[k * kFG], bad);
            col[k * kFG] = dk;
            if ((k & 7) == 7 || k == DC - 1) ck[k >> 3] = B;
            B = mul_rn(B, dk);
        }
    } else {
        // Irregular rows: `deg` is the same for the whole warp, so the blocks of 8 edges that lie entirely inside the row
        // run the unpredicated code of the regular kernel behind ONE warp-uniform branch; only the row's last, partial
        // block carries per-edge predicates, and blocks of pure padding are skipped (their factors are exact ones).
        // (Per-edge predicates everywhere cost 65 instead of 41 instructions per edge, and under the power cap the
        // n=65536 code's check pass is bound by instruction issue.)
#pragma unroll
        for (int b = NB - 1; b >= 0; b--) {
            const int bot = b * 8;
            ck[b] = B;
            if (bot + 8 <= deg) {
#pragma unroll
                for (int k = bot + 7; k >= bot; k--) {
                    const T dk = check_factor(col[k * kFG], bad);
                    col[k * kFG] = dk;
                    B = mul_rn(B, dk);
                }
            } else if (bot < deg) {
#pragma unroll
                for (int k = bot + 7; k >= bot; k--) {
                    T dk = T(1);
                    if (k < deg) {
                        dk = check_factor(col[k * kFG], bad);
                        col[k * kFG] = dk;
                    }
                    B = mul_rn(B, dk);
                }
            }
        }
    }
    if (bad) {  // invalid likelihood ratios: nothing stored to msg yet, redo with full IEEE divisions
        row_slow_path<T>(base, lr_lane, cols, deg, fresh);
        return;
    }
    T F = T(1);
#pragma unroll
    for (int b = 0; b < NB; b++) {
        const int bot = b * 8;
        const int top = (bot + 7 < DC - 1) ? bot + 7 : DC - 1;
        T d[8], Bv[8];
        if (EXACT || bot + 8 <= deg) {
#pragma unroll
            for (int k = bot; k <= top; k++) d[k - bot] = col[k * kFG];
            Bv[top - bot] = ck[b];
#pragma unroll
            for (int k = top; k > bot; k--) Bv[k - 1 - bot] = mul_rn(Bv[k - bot], d[k - bot]);
#pragma unroll
            for (int k = bot; k <= top; k++) {
                const T t = mul_rn(F, Bv[k - bot]);
                st_stream(base + (size_t)k * kFG, check_to_bit(t));
                F = mul_rn(F, d[k - bot]);
            }
        } else if (bot < deg) {
#pragma unroll
            for (int k = bot; k <= top; k++) d[k - bot] = k < deg ? col[k * kFG] : T(1);
            Bv[top - bot] = ck[b];
#pragma unroll
            for (int k = top; k > bot; k--) Bv[k - 1 - bot] = mul_rn(Bv[k - bot], d[k - bot]);
#pragma unroll
            for (int k = bot; k <= top; k++) {
                const T t = mul_rn(F, Bv[k - bot]);
                if (k < deg) st_stream(base + (size_t)k * kFG, check_to_bit(t));
                F = mul_rn(F, d[k - bot]);
            }
        }
    }
}
template <typename T, int DC, bool EXACT = true>
__global__ void __launch_bounds__(kRowWarps * 32, EXACT ? 3 : 6)
row_pass_smem_kernel(T *__restrict__ msg, const T *__restrict__ lratio, const uint32_t *__restrict__ actw,
                     const uint32_t *__restrict__ freshw, const int32_t *__restrict__ row_ptr,
                     const int32_t *__restrict__ col_idx, int M, int N, int E, int g0, int G) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    T *tile = reinterpret_cast<T *>(smem_raw) + (size_t)warp * DC * kFG;
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem_raw + (size_t)kRowWarps * DC * kFG * sizeof(T)) + warp;
    const long long item = (long long)blockIdx.x * kRowWarps + warp;
    if (item >= (long long)G * M) return;
    const int gl = (int)(item / M), i = (int)(item - (long long)gl * M);
    const int g = g0 + gl;
    const uint32_t act = actw[g];
    if (act == 0) return;
    const uint32_t fw = freshw[g];
    const bool on = (act >> lane) & 1u, fresh = (fw >> lane) & 1u;
    const int e0 = EXACT ? i * DC : __ldg(row_ptr + i);
    const int deg = EXACT ? DC : (__ldg(row_ptr + i + 1) - e0);
    T *base = msg + ((size_t)g * E + e0) * kFG + lane;
    T *col = tile + lane;  // this lane's column of the tile: col[k * 32]
    const T *lr_lane = lratio + (size_t)g * N * kFG + lane;
    // Lanes that carry on with a frame take their messages from the tile: ONE bulk copy lands the check's whole
    // contiguous run (the columns of starting / idle lanes come along and are ignored or overwritten below).
    const uint32_t fresh_mask = fw & act;
    const bool streaming = (act & ~fresh_mask) != 0;  // warp-uniform
    if (streaming && lane == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
        mbar_expect_tx(bar, (uint32_t)(deg * kFG * sizeof(T)));
        tma_load_1d(tile, msg + ((size_t)g * E + e0) * kFG, (uint32_t)(deg * kFG * sizeof(T)), bar);
    }
    if (fresh_mask == 0) {
        __syncwarp();
        mbar_wait(bar, 0);
    } else {
        // Lanes that start a frame need the channel ratios of the check's bits instead (Init_Belief_Propagation): the
        // WHOLE warp gathers them, lane = (edge of a block of 32 / R edges, rank r among the starting lanes) - with the
        // usual handful of starting lanes 18 loads per lane for the 72 edges instead of one divergent load per edge.
        const int nf = __popc(fresh_mask);
        const T *lr_base = lratio + (size_t)g * N * kFG;
        if (nf <= 8) {
            constexpr int NT = (DC + 3) / 4;
            const int r = lane & 7, kq = lane >> 3;
            const bool mine = r < nf;
            const int f = mine ? (int)__fns(fresh_mask, 0, r + 1) : 0;
            // Column indices, then the ratios themselves into registers: both are in flight together with the bulk copy
            // (the registers are free here: the arithmetic's working set is not live yet). Once the bulk copy has
            // landed they overwrite the starting lanes' columns of the tile.
            int idx[NT];
#pragma unroll
            for (int t = 0; t < NT; t++) {
                const int k = t * 4 + kq;
                idx[t] = (mine && k < deg) ? __ldg(col_idx + e0 + k) : -1;
            }
            T v[NT];
#pragma unroll
            for (int t = 0; t < NT; t++) v[t] = idx[t] >= 0 ? lr_base[(size_t)idx[t] * kFG + f] : T(0);
            __syncwarp();
            if (streaming) mbar_wait(bar, 0);
#pragma unroll
            for (int t = 0; t < NT; t++) {
                const int k = t * 4 + kq;
                if (idx[t] >= 0) tile[k * kFG + f] = v[t];
            }
        } else {  // many starting lanes (the first ticks of a batch): R = 16 or 32 ranks per instruction
            const int lg = nf <= 16 ? 4 : 5, R = 1 << lg, per = 32 >> lg;
            const int r = lane & (R - 1), kq = lane >> lg;
            const bool mine = r < nf;
            const int f = mine ? (int)__fns(fresh_mask, 0, r + 1) : 0;
            __syncwarp();
            if (streaming) mbar_wait(bar, 0);
#pragma unroll 6
            for (int k0 = 0; k0 < deg; k0 += per) {
                const int k = k0 + kq;
                if (mine && k < deg)
                    asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"(smem_u32(tile + k * kFG + f)),
                                 "l"(lr_base + (size_t)__ldg(col_idx + e0 + k) * kFG + f), "n"(sizeof(T)) : "memory");
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncwarp();
    }
    if (!on) return;  // finished / empty slots keep their messages untouched
    smem_row_compute<T, DC, EXACT>(col, base, lr_lane, col_idx + e0, fresh, deg);
}

// ---- tensor memory (tcgen05) as a second on-chip tile ----------------------------------------------------
// The check pass is bound by the bytes it can keep in flight per SM: 12 shared-memory tiles of 18 KB, each either being
// filled or being worked on. The 256 KB of tensor memory per SM are idle in this kernel (no MMA anywhere), so the factors
// d_k of a check are parked THERE after pass 1 (tcgen05.st, 144 of a lane's 512 32-bit columns; three warps share a
// lane quarter) and read back block by block in pass 2 (tcgen05.ld): the shared-memory tile is free again after one
// third of the arithmetic and the bulk copy of the warp's NEXT check is in flight during the other two thirds.
__device__ __forceinline__ void tmem_alloc_512(uint32_t *smem_slot) {  // one full warp; writes the base address to smem
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_512(uint32_t taddr) {  // the allocating warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(512u) : "memory");
}
// One block of 8 edges of this lane <-> 18 consecutive 32-bit columns of the lane's tensor-memory row: the 8 factors d_k
// and the backward product check-pointed at the top of the block.
constexpr int kTmBlockCols = 18;
__device__ __forceinline__ void tmem_st_block(uint32_t taddr, const double (&d)[8], double ck) {
    uint32_t w[16];
#pragma unroll
    for (int i = 0; i < 8; i++) { w[2 * i] = (uint32_t)__double2loint(d[i]); w[2 * i + 1] = (uint32_t)__double2hiint(d[i]); }
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
                 ::"r"(taddr), "r"(w[0]),"r"(w[1]),"r"(w[2]),"r"(w[3]),"r"(w[4]),"r"(w[5]),"r"(w[6]),"r"(w[7]),"r"(w[8]),"r"(w[9]),"r"(w[10]),"r"(w[11]),"r"(w[12]),"r"(w[13]),"r"(w[14]),"r"(w[15]) : "memory");
    asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1,%2};"
                 ::"r"(taddr + 16u), "r"((uint32_t)__double2loint(ck)), "r"((uint32_t)__double2hiint(ck)) : "memory");
}
__device__ __forceinline__ void tmem_ld_block(uint32_t taddr, double (&d)[8], double &ck) {
    uint32_t w[18];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(w[0]),"=r"(w[1]),"=r"(w[2]),"=r"(w[3]),"=r"(w[4]),"=r"(w[5]),"=r"(w[6]),"=r"(w[7]),"=r"(w[8]),"=r"(w[9]),"=r"(w[10]),"=r"(w[11]),"=r"(w[12]),"=r"(w[13]),"=r"(w[14]),"=r"(w[15]) : "r"(taddr) : "memory");
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0,%1}, [%2];" : "=r"(w[16]), "=r"(w[17]) : "r"(taddr + 16u) : "memory");
    // the registers are valid after the wait: tie them to it so that no use can be scheduled ahead of it
    asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(w[0]),"+r"(w[1]),"+r"(w[2]),"+r"(w[3]),"+r"(w[4]),"+r"(w[5]),"+r"(w[6]),"+r"(w[7]),"+r"(w[8]),"+r"(w[9]),"+r"(w[10]),"+r"(w[11]),"+r"(w[12]),"+r"(w[13]),"+r"(w[14]),"+r"(w[15]),"+r"(w[16]),"+r"(w[17]) :: "memory");
#pragma unroll
    for (int i = 0; i < 8; i++) d[i] = __hiloint2double((int)w[2 * i + 1], (int)w[2 * i]);
    ck = __hiloint2double((int)w[17], (int)w[16]);
}

// position of the r-th set bit of m for r < 8 (0 when m has fewer): 8 warp-uniform steps instead of __fns's search
__device__ __forceinline__ int nth_set_bit8(uint32_t m, int r) {
    int f = 0;
#pragma unroll
    for (int q = 0; q < 8; q++) {
        if (q == r && m) f = __ffs(m) - 1;
        m &= m - 1;
    }
    return f;
}

constexpr int kTmWarps = 12;  // one CTA per SM: 12 tiles of shared memory, 3 warps per tensor-memory lane quarter

// Persistent check pass, fp64, regular rows of degree DC (multiple of 8). 12 resident warps per SM pull ITEMS (group g,
// check i; consecutive items = consecutive checks of one group, so the channel-ratio lines that the lanes starting a
// frame gather stay in L2 between the 8 checks that use a bit) from a device counter the syndrome kernel re-arms.
// Software pipeline per warp, two items deep:
//   top of item k    : claim item k+2 (atomic, result picked up at the end); slot masks and column indices of item k+1
//                      requested into registers
//   tile of k landed : the gathered ratios of the lanes that start a frame overwrite their columns
//   pass 1 of k      : d_k and the check-pointed backward products to tensor memory (the shared-memory tile is free)
//   start of k+1     : column indices to shared memory, bulk copy into the freed tile, gather of its starting lanes
//                      into registers - all in flight during
//   pass 2 of k      : factors back from tensor memory block by block, lr_k streamed to the message array.
// Both passes are loops over blocks of 8 edges, unrolled UR times (fully unrolled the kernel outgrows the instruction
// cache and spends 15 % of a refill-regime launch waiting for instructions).
template <int DC, int UR>
__global__ void __launch_bounds__(kTmWarps * 32, 1)
row_pass_tmem_kernel(double *__restrict__ msg, const double *__restrict__ lratio, const uint32_t *__restrict__ actw,
                     const uint32_t *__restrict__ freshw, const int32_t *__restrict__ col_idx, int M, int N, int E,
                     int g0, int G, unsigned int *__restrict__ job_counter, int l2_hint) {
    static_assert(DC % 8 == 0 && (DC / 8) * kTmBlockCols * (kTmWarps / 4) <= 512, "tensor-memory columns");
    constexpr uint32_t kTileBytes = DC * kFG * sizeof(double);
    constexpr int NB = DC / 8, NT = DC / 4, NI = (DC + 31) / 32;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double *tile = reinterpret_cast<double *>(smem_raw) + (size_t)warp * DC * kFG;
    unsigned char *aux = smem_raw + (size_t)kTmWarps * DC * kFG * sizeof(double);
    uint64_t *bar = reinterpret_cast<uint64_t *>(aux) + warp;
    int *sidx = reinterpret_cast<int *>(aux + kTmWarps * sizeof(uint64_t)) + warp * DC;
    uint32_t *tm_slot = reinterpret_cast<uint32_t *>(aux + kTmWarps * sizeof(uint64_t) + (size_t)kTmWarps * DC * sizeof(int));
    const double *col = tile + lane;
    const uint64_t policy = l2_evict_first_policy();
    if (warp == 0) tmem_alloc_512(tm_slot);
    if (lane == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tm_base = *tm_slot;
    // this warp's rows: lane quarter (warp % 4) - the only one its tcgen05.ld / st can reach - and a private column range
    const uint32_t taddr = tm_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)((warp >> 2) * NB * kTmBlockCols);
    const unsigned njobs = (unsigned)M * (unsigned)G;
    const int kq = lane >> 3, rk = lane & 7;
    uint32_t phase = 0;

    // starts an item: bulk copy of its messages (if any lane carries on) and ranks 0..7 of the starting lanes' gather
    auto start_item = [&](int g, int e0, uint32_t act, uint32_t fw, double (&v)[NT]) {
        const uint32_t fresh_mask = fw & act;
        if ((act & ~fresh_mask) != 0 && lane == 0) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic accesses to the tile before the bulk write
            mbar_expect_tx(bar, kTileBytes);
            if (l2_hint) tma_load_1d_hint(tile, msg + ((size_t)g * E + e0) * kFG, kTileBytes, bar, policy);
            else tma_load_1d(tile, msg + ((size_t)g * E + e0) * kFG, kTileBytes, bar);
        }
        if (fresh_mask != 0) {
            const bool mine = rk < __popc(fresh_mask);
            const int f = nth_set_bit8(fresh_mask, rk);
            const double *lr_base = lratio + (size_t)g * N * kFG;
#pragma unroll
            for (int t = 0; t < NT; t++) v[t] = mine ? lr_base[(size_t)sidx[t * 4 + kq] * kFG + f] : 0.0;
        }
    };
    auto claim_raw = [&]() -> unsigned {  // lane 0's register holds the item; nobody waits for it here
        unsigned j = 0;
        if (lane == 0) j = atomicAdd(job_counter, 1u);
        return j;
    };

    unsigned job = __shfl_sync(0xffffffffu, claim_raw(), 0);
    unsigned job_n = __shfl_sync(0xffffffffu, claim_raw(), 0);
    int g = 0, e0 = 0;
    uint32_t act = 0, fw = 0;
    double v[NT];
    if (job < njobs) {  // the first item of this warp: nothing to overlap with yet
        g = g0 + (int)(job / (unsigned)M);
        e0 = (int)(job % (unsigned)M) * DC;
        for (int k = lane; k < DC; k += 32) sidx[k] = __ldg(col_idx + e0 + k);
        __syncwarp();
        act = actw[g]; fw = freshw[g];
        if (act != 0) start_item(g, e0, act, fw, v);
    }
    while (job < njobs) {
        // look ahead: claim the item after next; masks and column indices of the next item on their way
        const unsigned raw_nn = claim_raw();
        const bool valid_n = job_n < njobs;
        const int g_n = g0 + (int)(job_n / (unsigned)M), e0_n = (int)(job_n % (unsigned)M) * DC;
        uint32_t act_n = 0, fw_n = 0;
        int idx_n[NI];
#pragma unroll
        for (int q = 0; q < NI; q++) idx_n[q] = 0;
        if (valid_n) {
            act_n = actw[g_n]; fw_n = freshw[g_n];
#pragma unroll
            for (int q = 0; q < NI; q++)
                if (lane + 32 * q < DC) idx_n[q] = __ldg(col_idx + e0_n + lane + 32 * q);
        }
        const bool on = (act >> lane) & 1u, fresh = (fw >> lane) & 1u;
        double *base = msg + ((size_t)g * E + e0) * kFG + lane;
        const double *lr_lane = lratio + (size_t)g * N * kFG + lane;
        const int32_t *cols_cur = col_idx + e0;
        bool bad = false;
        if (act != 0) {
            const uint32_t fresh_mask = fw & act;
            if ((act & ~fresh_mask) != 0) {
                mbar_wait(bar, phase);
                phase ^= 1u;
            }
            if (fresh_mask != 0) {  // the gathered ratios overwrite the starting lanes' columns of the landed tile
                const int nf = __popc(fresh_mask);
                {
                    const bool mine = rk < nf;
                    const int f = nth_set_bit8(fresh_mask, rk);
#pragma unroll
                    for (int t = 0; t < NT; t++)
                        if (mine) tile[(t * 4 + kq) * kFG + f] = v[t];
                }
                for (int r0 = 8; r0 < nf; r0 += 8) {  // more than 8 starting lanes (first ticks of a batch, kinds with short frames): further rounds, not overlapped
                    const int r = r0 + rk;
                    const bool mine = r < nf;
                    const int f = mine ? (int)__fns(fresh_mask, 0, r + 1) : 0;
                    double w[NT];
#pragma unroll
                    for (int t = 0; t < NT; t++) w[t] = mine ? lr_lane[(size_t)sidx[t * 4 + kq] * kFG + (f - lane)] : 0.0;
#pragma unroll
                    for (int t = 0; t < NT; t++)
                        if (mine) tile[(t * 4 + kq) * kFG + f] = w[t];
                }
                __syncwarp();
            }
            // pass 1, descending: d_k and the check-pointed backward products to tensor memory
            double B = 1.0;
#pragma unroll(UR)
            for (int b = NB - 1; b >= 0; b--) {
                double d8[8];
                const double ckb = B;
#pragma unroll
                for (int kk = 7; kk >= 0; kk--) {
                    const double dk = check_factor(col[(b * 8 + kk) * kFG], bad);
                    d8[kk] = dk;
                    B = mul_rn(B, dk);
                }
                tmem_st_block(taddr + (uint32_t)(b * kTmBlockCols), d8, ckb);
            }
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        }
        __syncwarp();  // every lane has read its column and the staged indices: the tile and sidx can take the next item
        // start of the next item
#pragma unroll
        for (int q = 0; q < NI; q++)
            if (lane + 32 * q < DC) sidx[lane + 32 * q] = idx_n[q];
        __syncwarp();
        if (valid_n && act_n != 0) start_item(g_n, e0_n, act_n, fw_n, v);
        // (only `on`, `fresh`, `base`, `lr_lane`, `cols_cur`, `bad` still belong to the current item from here on)
        if (on && bad) row_slow_path<double>(base, lr_lane, cols_cur, DC, fresh);  // invalid ratios: full IEEE divisions
        // pass 2, ascending: factors back from tensor memory, lr_k streamed to the message array
        if (act != 0) {
            double F = 1.0;
            const bool store = on && !bad;
#pragma unroll(UR)
            for (int b = 0; b < NB; b++) {
                double d8[8], Bv[8];
                tmem_ld_block(taddr + (uint32_t)(b * kTmBlockCols), d8, Bv[7]);
#pragma unroll
                for (int kk = 7; kk > 0; kk--) Bv[kk - 1] = mul_rn(Bv[kk], d8[kk]);
#pragma unroll
                for (int kk = 0; kk < 8; kk++) {
                    const double t = mul_rn(F, Bv[kk]);
                    const double lr = check_to_bit(t);
                    if (store) st_stream(base + (size_t)(b * 8 + kk) * kFG, lr);
                    F = mul_rn(F, d8[kk]);
                }
            }
        }
        job = job_n; g = g_n; e0 = e0_n; act = act_n; fw = fw_n;
        // pick up the claim made at the top (volatile: keeps its place behind pass 2, so the atomic's latency stays hidden)
        asm volatile("shfl.sync.idx.b32 %0, %1, 0, 31, 0xffffffff;" : "=r"(job_n) : "r"(raw_nn));
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) tmem_dealloc_512(tm_base);
}

// ------------------------------------------------------------------------------------------------
// Bit-node (column) pass, dec.cpp:667-693.  One thread = one (bit j, slot f).
//   P_0 = lratio_j, P_{k+1} = P_k*lr_k; tot = P_last (NaN -> 1); dblk_j = (tot <= 1);
//   S_last = 1, S_{k-1} = S_k*lr_k;  pr_k = P_k*S_k (NaN -> 1)
// Warp = bit j of the 32 slots of a group; the 32 hard decisions are packed with one warp ballot.
// ------------------------------------------------------------------------------------------------
constexpr int kColWarps = 8;

// Loads of one (bit, slot): edge ids, the check->bit messages and the channel ratio. Kept apart from the arithmetic so
// that the fp32 kernel can have the loads of two bits in flight before the first one's stores (which the compiler must
// otherwise keep ahead of the next bit's loads: same array).
template <typename T, int DV>
struct ColIn {
    int eid[DV];
    T lr[DV];
    T P;
    int deg;
};

template <typename T, int DV, bool EXACT>
__device__ __forceinline__ void col_load(ColIn<T, DV> &c, const T *__restrict__ gmsg, const T *__restrict__ lratio,
                                         const int32_t *__restrict__ col_ptr, const int32_t *__restrict__ col_edge, int N,
                                         int g, int j, int f, bool on) {
    const int c0 = EXACT ? j * DV : __ldg(col_ptr + j);
    c.deg = EXACT ? DV : (__ldg(col_ptr + j + 1) - c0);
#pragma unroll
    for (int k = 0; k < DV; k++) c.eid[k] = (EXACT || k < c.deg) ? __ldg(col_edge + c0 + k) : 0;
#pragma unroll
    for (int k = 0; k < DV; k++) c.lr[k] = (on && (EXACT || k < c.deg)) ? ld_stream(gmsg + (size_t)c.eid[k] * kFG) : T(1);
    c.P = on ? __ldg(lratio + ((size_t)g * N + j) * kFG + f) : T(1);
}

template <typename T, int DV, bool EXACT, int ALG>
__device__ __forceinline__ bool col_finish(const ColIn<T, DV> &c, T *__restrict__ gmsg, T *__restrict__ post, int N, int g, int j,
                                           int f, bool on) {
    const int deg = c.deg;
    const int (&eid)[DV] = c.eid;
    const T (&lr)[DV] = c.lr;
    T P = c.P;
    if (ALG == ALG_MINSUM) {  // lr[] = c2v LLRs, P = channel LLR; sums in ascending row order, own edge skipped
        const T llr = P;
#pragma unroll
        for (int k = 0; k < DV; k++) {
            if (EXACT || k < deg) {
                T sum = llr;
#pragma unroll
                for (int m = 0; m < DV; m++)
                    if (m != k && (EXACT || m < deg)) sum = sum + lr[m];
                if (on) st_stream(gmsg + (size_t)eid[k] * kFG, sum);
            }
        }
        T tot = llr;
#pragma unroll
        for (int m = 0; m < DV; m++)
            if (EXACT || m < deg) tot = tot + lr[m];
        if (post != nullptr && on) post[((size_t)g * N + j) * kFG + f] = tot;
        return !(tot > T(0));
    }
    T p[DV];
#pragma unroll
    for (int k = 0; k < DV; k++) {
        p[k] = P;
        if (EXACT || k < deg) P = mul_rn(P, lr[k]);
    }
    if (P != P) P = T(1);
    if (post != nullptr && on) post[((size_t)g * N + j) * kFG + f] = P;
    T S = T(1);
#pragma unroll
    for (int k = DV - 1; k >= 0; k--) {
        if (EXACT || k < deg) {
            T v = mul_rn(p[k], S);
            if (v != v) v = T(1);
            if (on) st_stream(gmsg + (size_t)eid[k] * kFG, v);
            S = mul_rn(S, lr[k]);
        }
    }
    return P <= T(1);
}

// BITS = bits whose loads a thread has in flight before the first one's arithmetic and stores (the stores to the message
// array keep the compiler from hoisting the next bit's loads by itself). One bit is enough for fp64 columns of weight 8
// (8 x 256-byte requests per warp); fp32 messages (128-byte requests) and low-weight columns (3 edges per bit in the
// n=65536 code) need several to keep enough bytes in flight.
template <typename T, int DV, bool EXACT, int ALG, int BITS>
__global__ void __launch_bounds__(kColWarps * 32, DV > 8 ? 1 : (BITS * DV * (int)sizeof(T) <= 64 ? 4 : (BITS * DV <= 16 ? 3 : 2)))
col_pass_kernel(T *__restrict__ msg, const T *__restrict__ lratio, uint32_t *__restrict__ decw,
                const uint32_t *__restrict__ actw, T *__restrict__ post, const int32_t *__restrict__ col_ptr,
                const int32_t *__restrict__ col_edge, int N, int E, int g0, int cols_per_warp) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = g0 + blockIdx.y;
    const uint32_t act = actw[g];
    if (act == 0) return;
    const bool on = (act >> lane) & 1u;
    const int jbeg = (blockIdx.x * kColWarps + warp) * cols_per_warp;
    const int jend = min(jbeg + cols_per_warp, N);
    T *gmsg = msg + (size_t)g * E * kFG + lane;
    auto put = [&](int j, bool bit) {
        const uint32_t w = __ballot_sync(0xffffffffu, bit);
        if (lane == 0) {
            uint32_t *dst = decw + (size_t)g * N + j;
            *dst = (act == 0xffffffffu) ? w : ((w & act) | (*dst & ~act));
        }
    };
    int j = jbeg;
    if (BITS > 1) {
        for (; j + BITS - 1 < jend; j += BITS) {
            ColIn<T, DV> in[BITS];
#pragma unroll
            for (int b = 0; b < BITS; b++) col_load<T, DV, EXACT>(in[b], gmsg, lratio, col_ptr, col_edge, N, g, j + b, lane, on);
#pragma unroll
            for (int b = 0; b < BITS; b++) put(j + b, col_finish<T, DV, EXACT, ALG>(in[b], gmsg, post, N, g, j + b, lane, on));
        }
    }
    for (; j < jend; j++) {
        ColIn<T, DV> a;
        col_load<T, DV, EXACT>(a, gmsg, lratio, col_ptr, col_edge, N, g, j, lane, on);
        put(j, col_finish<T, DV, EXACT, ALG>(a, gmsg, post, N, g, j, lane, on));
    }
}

// ------------------------------------------------------------------------------------------------
// Slot scheduler, part 1: admit pending frames into free slots (one warp per group, lane = slot).
// Frames are taken from a single device-side counter, so any number of groups / streams / passes can pull from it.
// Finished slots (donew) are handed to the harvest pass through harvw / harv_frame / harv_iter.
// ------------------------------------------------------------------------------------------------
struct SchedArrays {
    uint32_t *actw, *donew, *newfw, *freshw, *harvw, *unsatw;
    unsigned int *arrive;
    int32_t *slot_frame, *slot_iter, *harv_frame, *harv_iter;  // slot_frame / harv_frame hold the frame's queue position q
    unsigned long long *next_frame;  // next queue position to admit
    unsigned long long *avail;       // queue positions published so far: frames q < *avail have their inputs resident
    const int32_t *in_row, *out_row; // per q: row of the frame in the input / output buffers (written by publish_kernel)
    unsigned long long *iter_sum;    // += iterations of every frame that finishes (dnaldpc_stats.frame_iters)
};

// The frame queue. A batch reaches an engine as a sequence of frames q = 0, 1, 2, ... that is PUBLISHED piece by piece
// while the engine is already decoding: the producer (a copy stream that has just landed a piece of a host batch in the
// staging ring, or the decode stream itself for device-resident batches) appends the rows of the piece to in_row /
// out_row and then raises *avail. Admission (assign_kernel) takes frames below *avail only, so host->device copies,
// decoding and device->host copies of one batch overlap, several GPUs can pull pieces of one batch from a shared
// counter, and a re-decoding round can run over an arbitrary list of rows (`list`), all with the same kernels.
// One CTA; the table entries are fenced before the counter moves. Readers use ld.cg (the tables grow while kernels run).
__global__ void __launch_bounds__(1024)
publish_kernel(int32_t *__restrict__ in_row, int32_t *__restrict__ out_row, long long q0, int n,
               const int32_t *__restrict__ list_in, int row0_in, int row0_out, unsigned long long *avail) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        in_row[q0 + i] = list_in ? list_in[i] : row0_in + i;
        out_row[q0 + i] = row0_out + i;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) *((volatile unsigned long long *)avail) = (unsigned long long)(q0 + n);
}

__global__ void __launch_bounds__(256)
assign_kernel(SchedArrays s, int g0, int G, int first_round,
              unsigned int *admitted /* += frames admitted (the host schedules the next ticks from it) */,
              unsigned int *low_water /* min= smallest q still in a slot after this admission */) {
    const int lane = threadIdx.x & 31;
    const int gl = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (gl >= G) return;
    const int g = g0 + gl, slot = g * kFG + lane;
    const uint32_t act = s.actw[g], done = s.donew[g];
    if ((done >> lane) & 1u) {
        s.harv_frame[slot] = s.slot_frame[slot];
        s.harv_iter[slot] = s.slot_iter[slot];
    }
    const uint32_t free_mask = ~act;  // finished or empty slots
    const int cnt = __popc(free_mask);
    long long base = 0;
    int got = 0;
    if (lane == 0 && cnt > 0) {  // claim up to cnt of the published, not yet admitted frames
        unsigned long long cur = *((volatile unsigned long long *)s.next_frame);
        const unsigned long long av = *((volatile unsigned long long *)s.avail);
        while (cur < av) {
            const unsigned long long n = min((unsigned long long)cnt, av - cur);
            const unsigned long long old = atomicCAS(s.next_frame, cur, cur + n);
            if (old == cur) { base = (long long)cur; got = (int)n; break; }
            cur = old;
        }
    }
    base = __shfl_sync(0xffffffffu, base, 0);
    got = __shfl_sync(0xffffffffu, got, 0);
    const bool is_free = (free_mask >> lane) & 1u;
    const int rank = __popc(free_mask & ((1u << lane) - 1u));
    const bool take = is_free && rank < got;
    const uint32_t newf = __ballot_sync(0xffffffffu, take);
    if (take) { s.slot_frame[slot] = (int32_t)(base + rank); s.slot_iter[slot] = 0; }
    else if (is_free) s.slot_frame[slot] = -1;
    // everything below the smallest q that still sits in a slot has been harvested (or is being harvested by the
    // harvest kernel that follows this launch): the host retires output blocks from it
    const uint32_t inuse = act | newf;
    const unsigned mine = ((inuse >> lane) & 1u) ? (unsigned)s.slot_frame[slot] : 0xffffffffu;
    const unsigned lw = __reduce_min_sync(0xffffffffu, mine);
    if (lane == 0) {
        if (newf) atomicAdd(admitted, (unsigned)__popc(newf));
        if (lw != 0xffffffffu) atomicMin(low_water, lw);
        s.actw[g] = inuse;
        s.donew[g] = 0;
        s.newfw[g] = newf;
        s.harvw[g] = done;
        s.freshw[g] = (first_round ? 0u : s.freshw[g]) | newf;
    }
}

// ------------------------------------------------------------------------------------------------
// Syndrome + per-slot loop control (check.cpp:28-47 + dec.cpp:594-599). kSynSplit CTAs per group each XOR the
// decision words of the bits of their checks (32 slots at once) and OR-reduce with warp shuffles; the last CTA to
// arrive applies the control for the slots under consideration: syndrome zero -> done (success), iteration count ==
// max_iter -> done (failure), else the slot iterates once more. The frame's n (the value
// Run_Belief_Propagation_Decoder returns) and success flag are written by FRAME index.
// `consider_new`: only slots admitted in this round are examined (the others were examined earlier this tick).
// ------------------------------------------------------------------------------------------------
constexpr int kSynThreads = 256;
constexpr int kSynSplit = 64;  // CTAs per group; the last one to arrive applies the loop control

struct SynArgs {
    int32_t *iters_out;
    uint8_t *ok_out;
    int M, N, g0, max_iter, consider_new, fixed_iters;
    unsigned int *counter;          // [0] += slots in use (active or awaiting harvest), or NULL when a later launch of
                                    // the tick counts
    unsigned int *finished;         // += frames that finished in this launch
    unsigned int *counters_to_zero; // ring entry (kCounterWords words) re-armed for a later tick, or NULL
    int clear_fresh;                // tick without admission: no assign_kernel will reset the fresh marks
    unsigned int *row_jobs;         // job counter of the persistent check-pass kernel, re-armed for this tick's launch
};

constexpr int kCounterWords = 4;    // per tick: slots in use, frames admitted, frames finished, low-water q (armed to ~0)

// Common head: housekeeping + "nothing to examine in this group" (uniform over the CTAs of the group: the masks only
// change in the last arriver). Returns the mask of slots to examine (0 = this CTA is finished).
__device__ __forceinline__ uint32_t syn_head(const SchedArrays &s, const SynArgs &a, int g, uint32_t &act) {
    if (a.counters_to_zero && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) {
        a.counters_to_zero[0] = 0; a.counters_to_zero[1] = 0; a.counters_to_zero[2] = 0; a.counters_to_zero[3] = 0xffffffffu;
    }
    if (a.row_jobs && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) *a.row_jobs = 0;
    act = s.actw[g];
    const uint32_t consider = a.consider_new ? s.newfw[g] : act;
    if (consider == 0 && a.counter && blockIdx.x == 0 && threadIdx.x == 0) {
        const unsigned add = (unsigned)(__popc(act) + __popc(s.donew[g]));
        if (add) atomicAdd(a.counter, add);
    }
    return consider;
}

// Common tail: OR-reduce the CTA's parity words, publish them, and let the last CTA of the group to arrive apply the
// per-slot loop control (dec.cpp:594-599).
template <int THREADS>
__device__ __forceinline__ void syn_tail(const SchedArrays &s, const SynArgs &a, int g, uint32_t act, uint32_t consider, uint32_t acc) {
    acc = __reduce_or_sync(0xffffffffu, acc);
    __shared__ uint32_t s_or[THREADS / 32];
    __shared__ unsigned int s_ticket;
    if ((threadIdx.x & 31) == 0) s_or[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t part = 0;
#pragma unroll
        for (int w = 0; w < THREADS / 32; w++) part |= s_or[w];
        if (part) atomicOr(s.unsatw + g, part);
        __threadfence();
        s_ticket = atomicAdd(s.arrive + g, 1u);
    }
    __syncthreads();
    if (s_ticket != gridDim.x * gridDim.z - 1) return;
    if (threadIdx.x < 32) {  // last CTA of the group: every partial OR is visible
        __threadfence();
        const uint32_t unsat = *((volatile uint32_t *)(s.unsatw + g));
        const int f = threadIdx.x, slot = g * kFG + f;
        const bool mine = (consider >> f) & 1u;
        const int it = mine ? s.slot_iter[slot] : 0;
        const uint32_t maxed = __ballot_sync(0xffffffffu, mine && it >= a.max_iter);
        // fixed_iters (Run_Belief_Propagation_Decoder_SAVE, dec.cpp:192-223): a zero syndrome does not stop the frame
        const uint32_t done = a.fixed_iters ? (consider & maxed) : ((consider & ~unsat) | (consider & maxed));
        const uint32_t done_ok = done & ~unsat;
        const bool fin = (done >> f) & 1u;
        if (fin) {
            const int row = __ldcg(s.out_row + s.slot_frame[slot]);
            a.iters_out[row] = it;
            a.ok_out[row] = (uint8_t)((done_ok >> f) & 1u);
        } else if (mine) {
            s.slot_iter[slot] = it + 1;  // this slot runs one more iteration now
        }
        const unsigned itsum = __reduce_add_sync(0xffffffffu, fin ? (unsigned)it : 0u);
        if (f == 0) {
            if (itsum) atomicAdd(s.iter_sum, (unsigned long long)itsum);
            const uint32_t still = act & ~done;
            const uint32_t dn = s.donew[g] | done;
            s.actw[g] = still;
            s.donew[g] = dn;
            s.unsatw[g] = 0;  // re-armed
            s.arrive[g] = 0;
            if (a.clear_fresh) s.freshw[g] = 0;  // every slot admitted earlier has had its first check pass
            if (done) atomicAdd(a.finished, (unsigned)__popc(done));
            if (a.counter) {
                const unsigned add = (unsigned)(__popc(still) + __popc(dn));
                if (add) atomicAdd(a.counter, add);
            }
        }
    }
}

// Variant 1 (any N): decision words gathered from global memory (L2), gridDim.x = kSynSplit CTAs per group.
__global__ void __launch_bounds__(kSynThreads)
syndrome_update_kernel(const uint32_t *__restrict__ decw, SchedArrays s, SynArgs a, const int32_t *__restrict__ row_ptr,
                       const int32_t *__restrict__ col_idx) {
    const int g = a.g0 + blockIdx.y, M = a.M;
    uint32_t act;
    const uint32_t consider = syn_head(s, a, g, act);
    if (consider == 0) return;
    const uint32_t *dw = decw + (size_t)g * a.N;
    // 8 lanes per check: their index loads are one coalesced run and all gathers of a check are in flight at once
    // (two dependent memory latencies per check instead of one per edge); XOR-folded over the 8 lanes with shuffles.
    const int sub = threadIdx.x & 7;
    const int rows_per_cta = kSynThreads / 8;
    const int stride = gridDim.x * rows_per_cta;
    uint32_t acc = 0;
    for (int ib = blockIdx.x * rows_per_cta; ib < M; ib += stride) {  // warp-uniform trip count
        const int i = ib + (threadIdx.x >> 3);
        uint32_t p = 0;
        if (i < M) {
            const int e0 = __ldg(row_ptr + i), e1 = __ldg(row_ptr + i + 1);
#pragma unroll 4
            for (int e = e0 + sub; e < e1; e += 8) p ^= __ldg(dw + __ldg(col_idx + e));
        }
        p ^= __shfl_xor_sync(0xffffffffu, p, 1);
        p ^= __shfl_xor_sync(0xffffffffu, p, 2);
        p ^= __shfl_xor_sync(0xffffffffu, p, 4);
        acc |= p;
    }
    syn_tail<kSynThreads>(s, a, g, act, consider, acc);
}

// Variant 2 (N decision words fit in shared memory): a CTA stages the group's N decision words in shared memory with
// coalesced 16-byte loads and gathers from there. Each word is used by every check of its bit (8 for the n=18432
// code), so the L2 -> SM traffic of variant 1 (one 32 B sector per 4-byte gather, ~600 MB per launch over 128 groups)
// becomes one streamed copy of N words per CTA. gridDim.x = kSynSmemSplit CTAs per group, each taking a contiguous
// range of checks.
constexpr int kSynSmemThreads = 1024;
constexpr int kSynSmemSplit = 2;

__global__ void __launch_bounds__(kSynSmemThreads)
syndrome_update_smem_kernel(const uint32_t *__restrict__ decw, SchedArrays s, SynArgs a, const int32_t *__restrict__ row_ptr,
                            const int32_t *__restrict__ col_idx) {
    extern __shared__ __align__(16) uint32_t sdw[];
    const int g = a.g0 + blockIdx.y, M = a.M, N = a.N;
    uint32_t act;
    const uint32_t consider = syn_head(s, a, g, act);
    if (consider == 0) return;
    const uint32_t *dw = decw + (size_t)g * N;
    const int n4 = N >> 2;  // the group's words start 16-byte aligned when N % 4 == 0 (checked by the host)
    for (int q = threadIdx.x; q < n4; q += kSynSmemThreads) reinterpret_cast<uint4 *>(sdw)[q] = __ldg(reinterpret_cast<const uint4 *>(dw) + q);
    for (int j = (n4 << 2) + threadIdx.x; j < N; j += kSynSmemThreads) sdw[j] = __ldg(dw + j);
    __syncthreads();
    const int sub = threadIdx.x & 7;
    const int rows_per_iter = kSynSmemThreads / 8;
    const int per_cta = (M + gridDim.x - 1) / gridDim.x;
    const int i_beg = blockIdx.x * per_cta, i_end = min(M, i_beg + per_cta);
    uint32_t acc = 0;
    for (int ib = i_beg; ib < i_end; ib += rows_per_iter) {  // warp-uniform trip count
        const int i = ib + (threadIdx.x >> 3);
        uint32_t p = 0;
        if (i < i_end) {
            const int e0 = __ldg(row_ptr + i), e1 = __ldg(row_ptr + i + 1);
#pragma unroll 4
            for (int e = e0 + sub; e < e1; e += 8) p ^= sdw[__ldg(col_idx + e)];
        }
        p ^= __shfl_xor_sync(0xffffffffu, p, 1);
        p ^= __shfl_xor_sync(0xffffffffu, p, 2);
        p ^= __shfl_xor_sync(0xffffffffu, p, 4);
        acc |= p;
    }
    syn_tail<kSynSmemThreads>(s, a, g, act, consider, acc);
}

// Variant 3 (N decision words do not fit in shared memory, N half-words do): blockIdx.z selects 16 of the group's 32
// slots; the CTA stages those slots' bits of all N words (N x 2 bytes) and works like variant 2 on them. The words are
// read twice per group, which is nothing next to one 32-byte L2 sector per 4-byte gather of variant 1 (the n=65536 code:
// 6.3 MB per group and launch).
__global__ void __launch_bounds__(kSynSmemThreads)
syndrome_update_half_kernel(const uint32_t *__restrict__ decw, SchedArrays s, SynArgs a, const int32_t *__restrict__ row_ptr,
                            const int32_t *__restrict__ col_idx) {
    extern __shared__ __align__(16) uint16_t shw[];
    const int g = a.g0 + blockIdx.y, M = a.M, N = a.N, half = blockIdx.z;
    uint32_t act;
    const uint32_t consider = syn_head(s, a, g, act);
    if (consider == 0) return;
    const uint32_t *dw = decw + (size_t)g * N;
    const int sh = 16 * half;
    const int n4 = N >> 2;  // N % 4 == 0 (checked by the host): 16-byte loads, 8-byte stores
    for (int q = threadIdx.x; q < n4; q += kSynSmemThreads) {
        const uint4 w = __ldg(reinterpret_cast<const uint4 *>(dw) + q);
        uint2 o;
        o.x = ((w.x >> sh) & 0xffffu) | (((w.y >> sh) & 0xffffu) << 16);
        o.y = ((w.z >> sh) & 0xffffu) | (((w.w >> sh) & 0xffffu) << 16);
        reinterpret_cast<uint2 *>(shw)[q] = o;
    }
    __syncthreads();
    const int sub = threadIdx.x & 7;
    const int rows_per_iter = kSynSmemThreads / 8;
    const int per_cta = (M + gridDim.x - 1) / gridDim.x;
    const int i_beg = blockIdx.x * per_cta, i_end = min(M, i_beg + per_cta);
    uint32_t acc = 0;
    for (int ib = i_beg; ib < i_end; ib += rows_per_iter) {  // warp-uniform trip count
        const int i = ib + (threadIdx.x >> 3);
        uint32_t p = 0;
        if (i < i_end) {
            const int e0 = __ldg(row_ptr + i), e1 = __ldg(row_ptr + i + 1);
#pragma unroll 4
            for (int e = e0 + sub; e < e1; e += 8) p ^= shw[__ldg(col_idx + e)];
        }
        p ^= __shfl_xor_sync(0xffffffffu, p, 1);
        p ^= __shfl_xor_sync(0xffffffffu, p, 2);
        p ^= __shfl_xor_sync(0xffffffffu, p, 4);
        acc |= p;
    }
    syn_tail<kSynSmemThreads>(s, a, g, act, consider, acc << sh);
}

// ------------------------------------------------------------------------------------------------
// Slot scheduler, part 2: harvest finished slots and set up newly admitted ones, one 32-bit x 32-slot tile per CTA.
//  harvest : bit-transpose the ballot words back to the frame's outputs (packed bits / 0-1 chars / posterior)
//  setup   : likelihood setup ("channel options") of the admitted frames: LR from {LR, LLR, BSC bits, AWGN y, vote
//            counts} (DNA_main.cpp:1340-1345, channel.cpp:32-33,75-84, decoder.py:314), transposed through shared
//            memory into the slot-interleaved lratio array, and the initial decision lratio < 1 (dec.cpp:626).
// ------------------------------------------------------------------------------------------------
enum InKind { IN_LR_F64 = 0, IN_LLR_F64 = 1, IN_BSC_BITS = 2, IN_AWGN_F32 = 3, IN_AWGN_F64 = 4, IN_VOTE_I8 = 5 };

struct SetupArgs {
    const void *data;
    size_t frame_stride;  // bytes
    double param;         // AWGN sigma: LLR = 2*y/(sigma*sigma) like channel.cpp:32
    const double *table;  // BSC: 2 entries, VOTE: 256 entries (device)
};

struct HarvestArgs {
    uint32_t *bits;      // [F][wpf] or NULL
    uint8_t *dblk;       // [F][N] or NULL
    double *posterior;   // [F][N] or NULL
    int wpf;
};

template <int KIND> __device__ __forceinline__ double load_lr(const SetupArgs &a, long long fr, int j) {
    const char *row = (const char *)a.data + (size_t)fr * a.frame_stride;
    if (KIND == IN_LR_F64) return ((const double *)row)[j];
    if (KIND == IN_LLR_F64) return exp(a.param * ((const double *)row)[j]);  // param = LLR scale (1 unless re-decoding)
    if (KIND == IN_BSC_BITS) return a.table[(((const uint32_t *)row)[j >> 5] >> (j & 31)) & 1u];
    if (KIND == IN_AWGN_F32) return exp(2.0 * (double)((const float *)row)[j] / (a.param * a.param));
    if (KIND == IN_AWGN_F64) return exp(2.0 * ((const double *)row)[j] / (a.param * a.param));
    return a.table[(int)((const int8_t *)row)[j] + 128];
}

// channel LLR = ln(p0/p1) of a bit, for the LLR-domain decoder (min-sum). Tables hold LLRs here.
template <int KIND> __device__ __forceinline__ double load_llr(const SetupArgs &a, long long fr, int j) {
    const char *row = (const char *)a.data + (size_t)fr * a.frame_stride;
    if (KIND == IN_LR_F64) return log(((const double *)row)[j]);
    if (KIND == IN_LLR_F64) return a.param == 1.0 ? ((const double *)row)[j] : a.param * ((const double *)row)[j];
    if (KIND == IN_BSC_BITS) return a.table[(((const uint32_t *)row)[j >> 5] >> (j & 31)) & 1u];
    if (KIND == IN_AWGN_F32) return 2.0 * (double)((const float *)row)[j] / (a.param * a.param);   // channel.cpp:32
    if (KIND == IN_AWGN_F64) return 2.0 * ((const double *)row)[j] / (a.param * a.param);
    return a.table[(int)((const int8_t *)row)[j] + 128];
}

// One warp per 32-bit x 32-slot tile, no block-level synchronisation: the tiles of a group are independent, so the
// warps of a CTA (each with a private transpose buffer) overlap each other's memory latencies.
constexpr int kHsWarps = 4;         // warps per CTA
constexpr int kHsTilesPerWarp = 2;  // tiles a warp walks through

template <typename T, int KIND, int ALG>
__global__ void __launch_bounds__(kHsWarps * 32)
harvest_setup_kernel(SetupArgs a, HarvestArgs h, SchedArrays s, T *__restrict__ lratio, const T *__restrict__ post,
                     uint32_t *__restrict__ decw, int N, int g0, int tiles_per_warp) {
    const int g = g0 + blockIdx.y;
    const uint32_t hv = s.harvw[g], nf = s.newfw[g];
    if ((hv | nf) == 0) return;
    __shared__ double tiles[kHsWarps][32][33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double (*tile)[33] = tiles[warp];
    const bool is_new = (nf >> lane) & 1u, is_old = (hv >> lane) & 1u;  // lane = slot
    // rows of this slot's frames in the caller's (or the staging ring's) input / output buffers
    const int my_new = is_new ? __ldcg(s.in_row + s.slot_frame[g * kFG + lane]) : 0;
    const int my_old = is_old ? __ldcg(s.out_row + s.harv_frame[g * kFG + lane]) : 0;
    const int my_oldit = s.harv_iter[g * kFG + lane];
    const int ntiles = (N + 31) / 32;
    const int t0 = (blockIdx.x * kHsWarps + warp) * tiles_per_warp;
    for (int tile_id = t0; tile_id < min(ntiles, t0 + tiles_per_warp); tile_id++) {
        const int j0 = tile_id * 32;
        const int j = j0 + lane;                                              // lane = bit of the tile
        uint32_t word = (j < N) ? decw[(size_t)g * N + j] : 0u;               // decisions of bit j, one bit per slot
        if (hv) {
            if (h.bits) {  // 32 x 32 bit transpose by ballots: slot f ends up with the word of its frame
                uint32_t mine = 0;
                for (uint32_t m = hv; m; m &= m - 1) {
                    const int f = __ffs(m) - 1;
                    const uint32_t b = __ballot_sync(0xffffffffu, (word >> f) & 1u);
                    if (lane == f) mine = b;
                }
                if (is_old) h.bits[(size_t)my_old * h.wpf + tile_id] = mine;
            }
            if (h.dblk) {
                for (uint32_t m = hv; m; m &= m - 1) {
                    const int f = __ffs(m) - 1;
                    const int fr = __shfl_sync(0xffffffffu, my_old, f);
                    if (j < N) h.dblk[(size_t)fr * N + j] = (uint8_t)((word >> f) & 1u);
                }
            }
            if (h.posterior) {
                for (int r = 0; r < 32; r++) {  // r = bit of the tile, lane = slot
                    const int jj = j0 + r;
                    double v = 0;
                    if (jj < N && is_old) {
                        const size_t idx = ((size_t)g * N + jj) * kFG + lane;
                        v = my_oldit > 0 ? (double)post[idx] : (double)lratio[idx];
                    }
                    tile[r][lane] = v;
                }
                __syncwarp();
                for (uint32_t m = hv; m; m &= m - 1) {  // lane = bit
                    const int f = __ffs(m) - 1;
                    const int fr = __shfl_sync(0xffffffffu, my_old, f);
                    if (j < N) h.posterior[(size_t)fr * N + j] = tile[lane][f];
                }
                __syncwarp();  // the old lratio / decw values have been read: the tile may be overwritten
            }
        }
        if (nf) {
            uint32_t bsc_word = 0;
            if (KIND == IN_BSC_BITS) {  // no transpose needed: slot `lane` holds the 32 received bits of its frame's tile
                if (is_new) bsc_word = ((const uint32_t *)((const char *)a.data + (size_t)my_new * a.frame_stride))[tile_id];
            } else {
                for (uint32_t m = nf; m; m &= m - 1) {  // r = slot, lane = bit of the tile: coalesced read of the frame's row
                    const int r = __ffs(m) - 1;
                    const int fr = __shfl_sync(0xffffffffu, my_new, r);
                    double v = 1.0;
                    if (j < N) v = ALG == ALG_MINSUM ? load_llr<KIND>(a, fr, j) : load_lr<KIND>(a, fr, j);
                    tile[r][lane] = v;
                }
                __syncwarp();
            }
            uint32_t wmine = 0;
            for (int r = 0; r < 32; r++) {  // r = bit of the tile, lane = slot
                const int jj = j0 + r;
                double dv = 1.0;
                if (is_new) dv = KIND == IN_BSC_BITS ? a.table[(bsc_word >> r) & 1u] : tile[lane][r];
                const T v = ALG == ALG_MINSUM ? (T)dv : clamp_lr((T)dv);
                // initial decision: BP lratio < 1 (dec.cpp:626); min-sum !(LLR > 0) (Init_MSA_INF, dec.cpp:1311-1312)
                const uint32_t w = __ballot_sync(0xffffffffu, ALG == ALG_MINSUM ? !(v > T(0)) : (v < T(1)));
                if (lane == r) wmine = w;
                if (jj < N && is_new) lratio[((size_t)g * N + jj) * kFG + lane] = v;
            }
            if (j < N) decw[(size_t)g * N + j] = (word & ~nf) | (wmine & nf);
            __syncwarp();  // before the next tile reuses the transpose buffer
        }
    }
}

// Syndrome of the final decisions of the slots being harvested, as 0/1 chars [F][M] (the `pchk` buffer of check()).
__global__ void __launch_bounds__(256)
syndrome_bytes_kernel(const uint32_t *__restrict__ decw, SchedArrays s, const int32_t *__restrict__ row_ptr,
                      const int32_t *__restrict__ col_idx, int M, int N, int g0, uint8_t *__restrict__ out) {
    const int g = g0 + blockIdx.y;
    const uint32_t hv = s.harvw[g];
    if (hv == 0) return;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M) return;
    const uint32_t *dw = decw + (size_t)g * N;
    uint32_t p = 0;
    const int e1 = __ldg(row_ptr + i + 1);
    for (int e = __ldg(row_ptr + i); e < e1; e++) p ^= __ldg(dw + __ldg(col_idx + e));
    for (uint32_t m = hv; m; m &= m - 1) {
        const int f = __ffs(m) - 1;
        out[(size_t)__ldcg(s.out_row + s.harv_frame[g * kFG + f]) * M + i] = (uint8_t)((p >> f) & 1u);
    }
}

// ------------------------------------------------------------------------------------------------
// Slot scheduler, part 3: compaction of the drain tail. Once no frame is pending, finished slots are not refilled and
// the stragglers end up spread thinly over all groups: a warp of the check/bit pass with 3 of its 32 lanes active
// still issues every request, each for one 32 B sector. compact_plan_kernel (one warp) picks the smallest K such that
// the free slots of groups [0,K) can take every active slot of groups [K,G), pairs them by rank and moves the slot
// bookkeeping; compact_move_kernel copies the two per-slot arrays that carry state across a tick (messages and
// channel ratios; decisions and posteriors are rewritten by the next bit pass before anything reads them).
// Runs between the syndrome/loop-control kernel and the check pass. Slots awaiting harvest are neither moved nor used
// as destinations. Results are unaffected: frames are independent and outputs are written by frame index.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32)
compact_plan_kernel(SchedArrays s, int G, int32_t *__restrict__ mv_src, int32_t *__restrict__ mv_dst,
                    int32_t *__restrict__ mv_count /* [0] = number of moves, [1] = K */) {
    const int lane = threadIdx.x;
    const uint32_t lt = (1u << lane) - 1u;
    int above = 0;
    for (int g = lane; g < G; g += 32) above += __popc(s.actw[g]);
#pragma unroll
    for (int o = 16; o; o >>= 1) above += __shfl_xor_sync(0xffffffffu, above, o);
    int K = 0, free_below = 0;
    while (K < G && free_below < above) {  // warp-uniform
        const uint32_t a = s.actw[K], d = s.donew[K];
        above -= __popc(a);
        free_below += __popc(~(a | d));
        K++;
    }
    int nsrc = 0;
    for (int g = K; g < G; g++) {
        const uint32_t a = s.actw[g];
        if ((a >> lane) & 1u) mv_src[nsrc + __popc(a & lt)] = g * kFG + lane;
        nsrc += __popc(a);
    }
    int ndst = 0;
    for (int g = 0; g < K && ndst < nsrc; g++) {
        const uint32_t fr = ~(s.actw[g] | s.donew[g]);
        if ((fr >> lane) & 1u) mv_dst[ndst + __popc(fr & lt)] = g * kFG + lane;
        ndst += __popc(fr);
    }
    __threadfence_block();
    __syncwarp();
    for (int m = lane; m < nsrc; m += 32) {
        const int src = mv_src[m], dst = mv_dst[m];
        const uint32_t sb = 1u << (src & 31), db = 1u << (dst & 31);
        atomicAnd(s.actw + (src >> 5), ~sb);
        atomicOr(s.actw + (dst >> 5), db);
        if (atomicAnd(s.freshw + (src >> 5), ~sb) & sb) atomicOr(s.freshw + (dst >> 5), db);
        else atomicAnd(s.freshw + (dst >> 5), ~db);
        s.slot_frame[dst] = s.slot_frame[src];
        s.slot_iter[dst] = s.slot_iter[src];
        s.slot_frame[src] = -1;
    }
    if (lane == 0) { mv_count[0] = nsrc; mv_count[1] = K; }
}

constexpr int kMoveThreads = 256, kMoveUnroll = 8;

template <typename T>
__global__ void __launch_bounds__(kMoveThreads)
compact_move_kernel(T *__restrict__ msg, T *__restrict__ lratio, const int32_t *__restrict__ mv_src,
                    const int32_t *__restrict__ mv_dst, const int32_t *__restrict__ mv_count, int N, int E) {
    const int nmv = mv_count[0];
    for (int m = blockIdx.y; m < nmv; m += gridDim.y) {
        const int src = mv_src[m], dst = mv_dst[m];
        const T *ms = msg + (size_t)(src >> 5) * E * kFG + (src & 31);
        T *md = msg + (size_t)(dst >> 5) * E * kFG + (dst & 31);
        const T *ls = lratio + (size_t)(src >> 5) * N * kFG + (src & 31);
        T *ld = lratio + (size_t)(dst >> 5) * N * kFG + (dst & 31);
        const int base = blockIdx.x * (kMoveThreads * kMoveUnroll) + threadIdx.x;
        T v[kMoveUnroll];
#pragma unroll
        for (int u = 0; u < kMoveUnroll; u++) {
            const int x = base + u * kMoveThreads;
            v[u] = x < E ? ms[(size_t)x * kFG] : (x < E + N ? ls[(size_t)(x - E) * kFG] : T(0));
        }
#pragma unroll
        for (int u = 0; u < kMoveUnroll; u++) {
            const int x = base + u * kMoveThreads;
            if (x < E) md[(size_t)x * kFG] = v[u];
            else if (x < E + N) ld[(size_t)(x - E) * kFG] = v[u];
        }
    }
}

// Rows of the frames a re-decoding round takes (decoder.py:641-660): stable compaction of {k : ok[k] == 0}, one CTA.
__global__ void __launch_bounds__(1024)
failed_rows_kernel(const uint8_t *__restrict__ ok, const int32_t *__restrict__ prev_list, int n, int32_t *__restrict__ list_out,
                   int32_t *__restrict__ count) {
    __shared__ int warp_cnt[32];
    __shared__ int base;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    for (int k0 = 0; k0 < n; k0 += 1024) {
        const int k = k0 + threadIdx.x;
        const bool bad = k < n && ok[k] == 0;
        const uint32_t m = __ballot_sync(0xffffffffu, bad);
        if (lane == 0) warp_cnt[warp] = __popc(m);
        __syncthreads();
        int off = base;
        for (int w = 0; w < warp; w++) off += warp_cnt[w];
        if (bad) list_out[off + __popc(m & ((1u << lane) - 1u))] = prev_list ? prev_list[k] : k;
        __syncthreads();
        if (threadIdx.x == 0) { int t = 0; for (int w = 0; w < 32; w++) t += warp_cnt[w]; base += t; }
        __syncthreads();
    }
    if (threadIdx.x == 0) *count = base;
}

__global__ void init_sched_kernel(SchedArrays s, int G, unsigned int *counters, int n_counter_sets) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < G * kFG) { s.slot_frame[t] = -1; s.slot_iter[t] = 0; s.harv_frame[t] = -1; s.harv_iter[t] = 0; }
    if (t < G) { s.actw[t] = 0; s.donew[t] = 0; s.newfw[t] = 0; s.freshw[t] = 0; s.harvw[t] = 0; s.unsatw[t] = 0; s.arrive[t] = 0; }
    if (t < n_counter_sets * kCounterWords) counters[t] = (t % kCounterWords == 3) ? 0xffffffffu : 0u;
    if (t == 0) { *s.next_frame = 0; *s.avail = 0; *s.iter_sum = 0; }
}

// ------------------------------------------------------------------------------------------------
// Synthetic BSC input generator (benchmarks, csrc/sim.cu): counter RNG of rng.cuh keyed by (seed, GLOBAL frame, bit).
// Frame f is noise on codeword row (f + cw_off) % n_cw of cw_bits (cw_off = 0 for the C-ABI synth functions; the
// simulator points cw_bits at a piece of its codeword ring and picks cw_off so that frame f0 + i reads row i).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
synth_bsc_kernel(const uint32_t *__restrict__ cw_bits, int n_cw, uint64_t cw_off, uint64_t seed, long long frame0, long long F,
                 int N, int words_per_frame, uint64_t thr, uint32_t *__restrict__ out) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= F * words_per_frame) return;
    const long long fl = t / words_per_frame;
    const int w = (int)(t - fl * words_per_frame);
    const uint64_t f = (uint64_t)(frame0 + fl);
    uint32_t word = cw_bits ? cw_bits[(size_t)((f + cw_off) % (uint64_t)n_cw) * words_per_frame + w] : 0u;
    const uint64_t fkey = mix64(seed * 0x9E3779B97F4A7C15ULL + f + 0x632BE59BD9B4E019ULL);
    for (int b = 0; b < 32; b++) {
        const int j = w * 32 + b;
        if (j < N) {
            const uint64_t x = mix64(fkey ^ ((uint64_t)j * 0xD6E8FEB86659FD93ULL + 0x2545F4914F6CDD1DULL));
            if ((x >> 11) < thr) word ^= (1u << b);
        }
    }
    out[t] = word;
}

// Synthetic AWGN input (BASELINE configs[3]; channel_AWGN, channel.cpp:23-35): y = (bit ? -1 : +1) + sigma * n with
// n ~ N(0,1) by Box-Muller from the counter RNG: u1 = ((rng(seed, f, j, 4) >> 11) + 1) / 2^53 in (0, 1],
// u2 = (rng(seed, f, j, 5) >> 11) / 2^53, n = sqrt(-2 ln u1) cos(2 pi u2), all in fp64, y rounded to fp32.
// Host twin: oracle/bp_oracle.c:orc_synth_awgn (libm; agrees to the last fp32 ulp except where the fp64 values
// straddle a rounding boundary). Keyed by the GLOBAL frame index like synth_bsc_kernel.
__global__ void __launch_bounds__(256)
synth_awgn_kernel(const uint32_t *__restrict__ cw_bits, int n_cw, uint64_t cw_off, uint64_t seed, long long frame0, long long F,
                  int N, int words_per_frame, double sigma, float *__restrict__ out) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= F * N) return;
    const long long fl = t / N;
    const int j = (int)(t - fl * N);
    const uint64_t f = (uint64_t)(frame0 + fl);
    const uint32_t bit = cw_bits ? (cw_bits[(size_t)((f + cw_off) % (uint64_t)n_cw) * words_per_frame + (j >> 5)] >> (j & 31)) & 1u : 0u;
    const double u1 = ((double)(rng_u64(seed, f, (uint64_t)j, 4) >> 11) + 1.0) * (1.0 / 9007199254740992.0);
    const double u2 = (double)(rng_u64(seed, f, (uint64_t)j, 5) >> 11) * (1.0 / 9007199254740992.0);
    const double n = sqrt(-2.0 * log(u1)) * cos(6.283185307179586476925286766559 * u2);
    out[t] = (float)((bit ? -1.0 : 1.0) + sigma * n);
}

// Synthetic vote-count input (BASELINE configs[2]; the soft information ex_decoder/decoder.py:292-316 derives from
// aligned reads): reads per bit c ~ Poisson(mean) by inversion against the integer thresholds thr[k] =
// (uint64)(CDF(k) * 2^53) (kVoteMaxReads entries, computed on the host), every read wrong with probability p_err,
// k = (c - 2 * wrong) for a 0 bit and its negative for a 1 bit (count0 - count1). Integer arithmetic only, so the host
// twin (oracle/bp_oracle.c:orc_synth_vote) is exact.
constexpr int kVoteMaxReads = 64;
__global__ void __launch_bounds__(256)
synth_vote_kernel(const uint32_t *__restrict__ cw_bits, int n_cw, uint64_t cw_off, uint64_t seed, long long frame0, long long F,
                  int N, int words_per_frame, const uint64_t *__restrict__ thr, uint64_t thr_err, int8_t *__restrict__ out) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= F * N) return;
    const long long fl = t / N;
    const int j = (int)(t - fl * N);
    const uint64_t f = (uint64_t)(frame0 + fl);
    const uint32_t bit = cw_bits ? (cw_bits[(size_t)((f + cw_off) % (uint64_t)n_cw) * words_per_frame + (j >> 5)] >> (j & 31)) & 1u : 0u;
    const uint64_t u = rng_u64(seed, f, (uint64_t)j, 2) >> 11;
    int c = 0;
    while (c < kVoteMaxReads - 1 && u >= __ldg(thr + c)) c++;
    int wrong = 0;
    for (int r = 0; r < c; r++) wrong += (rng_u64(seed, f, (uint64_t)j, 3 + (uint64_t)r) >> 11) < thr_err;
    const int k = c - 2 * wrong;
    out[t] = (int8_t)(bit ? -k : k);
}

// ------------------------------------------------------------------------------------------------
// Diagnostic: inlined in-range sequences vs nvcc's full-range IEEE division, bit for bit.
// ------------------------------------------------------------------------------------------------
__global__ void math_selftest_kernel(long long n, uint64_t seed, unsigned long long *mismatch) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t r0 = rng_u64(seed, (uint64_t)i, 0, 0), r1 = rng_u64(seed, (uint64_t)i, 1, 0);
    unsigned long long bad_count = 0;
    // (1) pr >= 0 over the whole exponent range, plus +0, +inf and exact powers of two
    {
        double pr;
        const int sel = (int)(r1 & 15);
        if (sel == 0) pr = 0.0;
        else if (sel == 1) pr = __longlong_as_double(0x7FF0000000000000LL);
        else if (sel == 2) pr = __longlong_as_double((long long)((r0 >> 53) << 52));  // 2^k
        else if (sel < 10) pr = __longlong_as_double((long long)(r0 & 0x7FEFFFFFFFFFFFFFULL));  // any finite positive
        else {  // moderate ratios, the common regime: 2^[-64, 64)
            const uint64_t ex = 1023 - 64 + ((r1 >> 8) & 127);
            pr = __longlong_as_double((long long)((ex << 52) | (r0 & 0xFFFFFFFFFFFFFULL)));
        }
        bool bad = false;
        const double a = check_factor(pr, bad), b = check_factor_slow(pr);
        if (bad || __double_as_longlong(a) != __double_as_longlong(b)) bad_count++;
    }
    // (2) t in [-1, 1]: uniform, and clustered at +-1 (1 - 2^-k * m) where the quotient saturates
    {
        const uint64_t m = r0 & 0xFFFFFFFFFFFFFULL;
        const int sel = (int)((r1 >> 16) & 7);
        double t;
        if (sel == 0) t = 1.0;
        else if (sel == 1) t = -1.0;
        else if (sel == 2) t = 0.0;
        else if (sel < 5) {
            const uint64_t ex = 1023 - 1 - ((r1 >> 24) & 63);  // |t| in [2^-64, 1)
            t = __longlong_as_double((long long)((ex << 52) | m));
        } else {
            const uint64_t ex = 1023 - 1 - ((r1 >> 24) & 63);
            t = 1.0 - __longlong_as_double((long long)((ex << 52) | m));  // close to 1
            if (t > 1.0) t = 1.0;
        }
        if ((r1 >> 40) & 1) t = -t;
        const double a = check_to_bit(t), b = check_to_bit_slow(t);
        if (__double_as_longlong(a) != __double_as_longlong(b)) bad_count++;
    }
    if (bad_count) atomicAdd(mismatch, bad_count);
}

}  // namespace dnaldpc
