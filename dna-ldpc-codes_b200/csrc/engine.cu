// engine.cu - per-device slot scheduler around the kernels of bp_kernels.cuh.
#include "engine.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>

#include "bp_kernels.cuh"
#include "sw_kernels.cuh"

namespace dnaldpc {

#define CK(call)                                      \
    do {                                              \
        cudaError_t e_ = (call);                      \
        if (e_ != cudaSuccess) return fail(e_, #call); \
    } while (0)

int Engine::fail(cudaError_t e, const char *what) {
    err_ = std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what;
    return DNALDPC_ERR_CUDA;
}
int Engine::fail(const std::string &m, int rc) {
    err_ = m;
    return rc;
}

static size_t in_elem_stride(int kind, int N) {
    switch (kind) {
        case DNALDPC_IN_LR_F64: case DNALDPC_IN_LLR_F64: case DNALDPC_IN_AWGN_F64: return (size_t)N * 8;
        case DNALDPC_IN_AWGN_F32: return (size_t)N * 4;
        case DNALDPC_IN_BSC_BITS: return (size_t)((N + 31) / 32) * 4;
        case DNALDPC_IN_VOTE_I8: return (size_t)N;
    }
    return 0;
}

Engine::Engine(const Code &code, int device, int precision, int wave_frames)
    : device_(device), precision_(precision) {
    M_ = code.M; N_ = code.N; E_ = code.E;
    max_row_deg_ = code.max_row_deg; max_col_deg_ = code.max_col_deg;
    reg_rows_ = code.regular_rows; reg_cols_ = code.regular_cols;
    esz_ = precision == DNALDPC_PREC_F32 ? 4 : 8;
    if (wave_frames <= 0) wave_frames = 4096;
    wave_frames_ = (wave_frames + 31) / 32 * 32;
    if (max_row_deg_ > 128 || max_col_deg_ > 16) {
        err_ = "unsupported code: row degree > 128 or column degree > 16";
        return;
    }
    auto chk = [&](cudaError_t e, const char *w) { if (e != cudaSuccess && err_.empty()) fail(e, w); };
    chk(cudaSetDevice(device_), "cudaSetDevice");
    if (!err_.empty()) return;
    auto up = [&](int32_t **dst, const std::vector<int32_t> &v) {
        chk(cudaMalloc((void **)dst, std::max<size_t>(v.size(), 1) * sizeof(int32_t)), "cudaMalloc(H tables)");
        if (err_.empty() && !v.empty())
            chk(cudaMemcpy(*dst, v.data(), v.size() * sizeof(int32_t), cudaMemcpyHostToDevice), "cudaMemcpy(H tables)");
    };
    up(&d_row_ptr_, code.row_ptr);
    up(&d_col_idx_, code.col_idx);
    up(&d_col_ptr_, code.col_ptr);
    up(&d_col_edge_, code.col_edge);
    chk(cudaMalloc((void **)&d_table_, 256 * sizeof(double)), "cudaMalloc(table)");
    chk(cudaMalloc((void **)&d_next_, 3 * sizeof(unsigned long long)), "cudaMalloc(next)");
    chk(cudaMalloc((void **)&d_counters_, ((size_t)kRing * kCounterWords + 1) * sizeof(unsigned)), "cudaMalloc(counters)");  // + the check pass's job counter
    chk(cudaMallocHost((void **)&h_counters_, (size_t)kRing * kCounterWords * sizeof(unsigned)), "cudaMallocHost(counters)");
    chk(cudaEventCreateWithFlags(&ready_ev_, cudaEventDisableTiming), "cudaEventCreate");
    chk(cudaDeviceGetAttribute(&sm_count_, cudaDevAttrMultiProcessorCount, device_), "cudaDeviceGetAttribute");
    for (auto &e : ev_) chk(cudaEventCreateWithFlags(&e, cudaEventDisableTiming), "cudaEventCreate");
    for (auto &e : prof_ev_) chk(cudaEventCreate(&e), "cudaEventCreate");
    for (auto &e : trace_ev_) chk(cudaEventCreate(&e), "cudaEventCreate");
    chk(cudaStreamCreateWithFlags(&own_stream_, cudaStreamNonBlocking), "cudaStreamCreate");
    for (auto &s : io_stream_) chk(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking), "cudaStreamCreate");
}

Engine::~Engine() {
    cudaSetDevice(device_);
    cudaDeviceSynchronize();
    void *ptrs[] = {d_row_ptr_, d_col_idx_, d_col_ptr_, d_col_edge_, d_msg_, d_lratio_, d_post_, d_decw_, d_masks_, d_arrive_,
                    d_slot_, d_mv_, d_sw_lr_, d_edge_row_, d_next_, d_iters_, d_ok_, d_table_, d_counters_, s_in_, s_bits_, s_dblk_, s_post_, s_pchk_,
                    s_iters_, s_ok_, d_rows_, d_synth_thr_, d_list_[0], d_list_[1], d_col_row_, d_sw_sched_, s_in2_, d_sw_avail_, d_sw_lists_, d_sw_thin_, d_sw_hist_};
    for (void *p : ptrs) if (p) cudaFree(p);
    if (h_counters_) cudaFreeHost(h_counters_);
    if (h_bounce_) cudaFreeHost(h_bounce_);
    if (h_rows_) cudaFreeHost(h_rows_);
    if (h_avail_) cudaFreeHost(h_avail_);
    if (ready_ev_) cudaEventDestroy(ready_ev_);
    for (auto &e : ev_) if (e) cudaEventDestroy(e);
    for (auto &e : prof_ev_) if (e) cudaEventDestroy(e);
    for (auto &e : trace_ev_) if (e) cudaEventDestroy(e);
    for (auto &e : sw_in_ev_) if (e) cudaEventDestroy(e);
    if (own_stream_) cudaStreamDestroy(own_stream_);
    for (auto &s : io_stream_) if (s) cudaStreamDestroy(s);
}

int Engine::ensure_slots(int G, bool want_post) {
    if (G > cap_groups_) {
        void *ptrs[] = {d_msg_, d_lratio_, d_post_, d_decw_, d_masks_, d_arrive_, d_slot_, d_mv_};
        for (void *p : ptrs) if (p) cudaFree(p);
        d_msg_ = d_lratio_ = d_post_ = nullptr; d_decw_ = d_masks_ = nullptr; d_arrive_ = nullptr; d_slot_ = d_mv_ = nullptr;
        cap_groups_ = 0;
        CK(cudaMalloc(&d_msg_, std::max<size_t>((size_t)G * E_ * kFG * esz_, 16)));
        CK(cudaMalloc(&d_lratio_, (size_t)G * N_ * kFG * esz_));
        CK(cudaMalloc((void **)&d_decw_, (size_t)G * N_ * sizeof(uint32_t)));
        CK(cudaMalloc((void **)&d_masks_, (size_t)G * 6 * sizeof(uint32_t)));
        CK(cudaMalloc((void **)&d_arrive_, (size_t)G * sizeof(unsigned)));
        CK(cudaMalloc((void **)&d_slot_, (size_t)G * kFG * 4 * sizeof(int32_t)));
        CK(cudaMalloc((void **)&d_mv_, ((size_t)G * kFG * 2 + 2) * sizeof(int32_t)));
        cap_groups_ = G;
    }
    if (want_post && !d_post_) CK(cudaMalloc(&d_post_, (size_t)cap_groups_ * N_ * kFG * esz_));
    return DNALDPC_OK;
}

int Engine::ensure_frame_scratch(int64_t F) {
    if (F > cap_frames_) {
        if (d_iters_) cudaFree(d_iters_);
        if (d_ok_) cudaFree(d_ok_);
        d_iters_ = nullptr; d_ok_ = nullptr; cap_frames_ = 0;
        CK(cudaMalloc((void **)&d_iters_, (size_t)F * sizeof(int32_t)));
        CK(cudaMalloc((void **)&d_ok_, (size_t)F));
        cap_frames_ = F;
    }
    return DNALDPC_OK;
}

void Engine::fill_sched(SchedArrays &s) const {
    const size_t G = (size_t)cap_groups_;
    s.actw = d_masks_; s.donew = d_masks_ + G; s.newfw = d_masks_ + 2 * G; s.freshw = d_masks_ + 3 * G;
    s.harvw = d_masks_ + 4 * G; s.unsatw = d_masks_ + 5 * G;
    s.arrive = d_arrive_;
    const size_t S = G * kFG;
    s.slot_frame = d_slot_; s.slot_iter = d_slot_ + S; s.harv_frame = d_slot_ + 2 * S; s.harv_iter = d_slot_ + 3 * S;
    s.next_frame = d_next_;
    s.avail = d_next_ + 1;
    s.iter_sum = d_next_ + 2;
    s.in_row = d_rows_;
    s.out_row = d_rows_ + cap_rows_;
}

// ---- kernel dispatch -----------------------------------------------------------------------------

template <typename T> int Engine::launch_row(int g0, int G, cudaStream_t st) {
    T *msg = (T *)d_msg_;
    const T *lr = (const T *)d_lratio_;
    SchedArrays s;
    fill_sched(s);
    const long long items = (long long)G * M_;
    const unsigned grid = (unsigned)((items + kRowWarps - 1) / kRowWarps);
#define ROW(DC, EX)                                                                                                                       \
    do {                                                                                                                                  \
        if (minsum_) row_pass_kernel<T, DC, EX, ALG_MINSUM><<<grid, kRowWarps * 32, 0, st>>>(msg, lr, s.actw, s.freshw, d_row_ptr_, d_col_idx_, M_, N_, E_, g0, G); \
        else row_pass_kernel<T, DC, EX, ALG_BP><<<grid, kRowWarps * 32, 0, st>>>(msg, lr, s.actw, s.freshw, d_row_ptr_, d_col_idx_, M_, N_, E_, g0, G);         \
    } while (0)
    static const bool no_smem = getenv("DNALDPC_ROW_REGS") != nullptr;  // A/B switch: register-resident check kernel
    // A/B switch: the round-1 policy (smem-staged kernel only in ticks where every slot is busy and nobody is admitted)
    static const bool steady_only = getenv("DNALDPC_ROW_SMEM_STEADY_ONLY") != nullptr;
    const bool use_smem = !no_smem && (steady_ || !steady_only) && !minsum_ && sizeof(T) == 8;
    // Tensor memory as the second on-chip tile (row_pass_tmem_kernel): the default for the (.,72)-regular fp64 code.
    // A/B switches: DNALDPC_ROW_NO_TMEM=1 -> the one-item-per-warp shared-memory kernel; DNALDPC_ROW_L2HINT=0 -> bulk
    // copies without the evict-first policy.
    static const bool use_tmem = getenv("DNALDPC_ROW_NO_TMEM") == nullptr;
    static const int tm_hint = getenv("DNALDPC_ROW_L2HINT") ? atoi(getenv("DNALDPC_ROW_L2HINT")) : 1;
    if (use_smem && use_tmem && reg_rows_ && max_row_deg_ == 72) {
        // one CTA of 12 warps per SM; d_k parked in tensor memory so that the next check's bulk copy overlaps pass 2
        const size_t smem = (size_t)kTmWarps * 72 * kFG * sizeof(double) + kTmWarps * sizeof(uint64_t) + (size_t)kTmWarps * 72 * sizeof(int) + 16;
        // Blocks of 8 edges per loop trip. Same-box A/B (1.53 GHz under the power cap; steady-state step / refill-regime
        // launch): 9 (fully unrolled) 0.2387 Gbit/s / 1.86 ms, 3: 0.2367 / 1.69 ms, 1: 0.2345 / 1.73 ms - the unrolled
        // form wins while every warp runs the same streaming code and loses once the warps spread over the gather /
        // fix-up paths of groups that admit frames (instruction-cache misses), so the host picks per tick.
        static const int ur_env = getenv("DNALDPC_ROW_UNROLL") ? atoi(getenv("DNALDPC_ROW_UNROLL")) : 0;
        const int ur = ur_env ? ur_env : (steady_ ? 9 : 3);
        if (!tmem_attr_set_) {
            CK(cudaFuncSetAttribute(row_pass_tmem_kernel<72, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            CK(cudaFuncSetAttribute(row_pass_tmem_kernel<72, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            CK(cudaFuncSetAttribute(row_pass_tmem_kernel<72, 9>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            tmem_attr_set_ = true;
        }
        const unsigned pgrid = (unsigned)std::min<long long>((long long)sm_count_, (items + kTmWarps - 1) / kTmWarps);
        unsigned *jobs = d_counters_ + (size_t)kRing * kCounterWords;
#define TMROW(U) row_pass_tmem_kernel<72, U><<<pgrid, kTmWarps * 32, smem, st>>>((double *)msg, (const double *)lr, s.actw, s.freshw, d_col_idx_, M_, N_, E_, g0, G, jobs, tm_hint)
        if (ur == 9) TMROW(9);
        else if (ur == 3) TMROW(3);
        else TMROW(1);
#undef TMROW
    } else if (use_smem && reg_rows_ && max_row_deg_ == 72) {
        // the (.,72)-regular sum-product hot path: check messages staged in shared memory by TMA, 12 warps per SM
        const size_t smem = (size_t)kRowWarps * 72 * kFG * sizeof(T) + kRowWarps * sizeof(uint64_t);
        bool &attr_set = smem_attr_set_[sizeof(T) == 4];
        if (!attr_set) {  // per engine (= per device)
            CK(cudaFuncSetAttribute(row_pass_smem_kernel<T, 72>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            attr_set = true;
        }
        row_pass_smem_kernel<T, 72><<<grid, kRowWarps * 32, smem, st>>>(msg, lr, s.actw, s.freshw, d_row_ptr_, d_col_idx_, M_, N_, E_, g0, G);
    } else if (use_smem && max_row_deg_ <= 32 && max_row_deg_ > 8) {
        // irregular rows of degree <= 32 (e.g. the n=65536 column-weight-3 code): same staging, deg x 256 B bulk copies
        const size_t smem = (size_t)kRowWarps * 32 * kFG * sizeof(T) + kRowWarps * sizeof(uint64_t);
        row_pass_smem_kernel<T, 32, false><<<grid, kRowWarps * 32, smem, st>>>(msg, lr, s.actw, s.freshw, d_row_ptr_, d_col_idx_, M_, N_, E_, g0, G);
    } else if (reg_rows_ && max_row_deg_ == 72) ROW(72, true);
    else if (max_row_deg_ <= 8) ROW(8, false);
    else if (max_row_deg_ <= 32) ROW(32, false);
    else if (max_row_deg_ <= 72) ROW(72, false);
    else ROW(128, false);
#undef ROW
    stats.kernel_launches++;
    CK(cudaGetLastError());
    return DNALDPC_OK;
}

template <typename T> int Engine::launch_col(int g0, int G, bool want_post, cudaStream_t st) {
    T *msg = (T *)d_msg_;
    const T *lr = (const T *)d_lratio_;
    T *post = want_post ? (T *)d_post_ : nullptr;
    SchedArrays s;
    fill_sched(s);
    // bits a thread keeps in flight (A/B switch DNALDPC_COL_BITS): 1 for fp64 columns of weight 8, several for fp32
    // messages and for low-weight columns
    static const int bits_env = getenv("DNALDPC_COL_BITS") ? atoi(getenv("DNALDPC_COL_BITS")) : 0;
    const int bits_def = (max_col_deg_ <= 4) ? 4 : (sizeof(T) == 4 ? 2 : 1);
    const int bits = (bits_env >= 1 && bits_env <= 4) ? bits_env : bits_def;
    const int cpw = bits == 3 ? 9 : 8;  // columns per warp
    dim3 grid((unsigned)((N_ + kColWarps * cpw - 1) / (kColWarps * cpw)), (unsigned)G);
#define COLB(DV, EX, B)                                                                                                                  \
    do {                                                                                                                                 \
        if (minsum_) col_pass_kernel<T, DV, EX, ALG_MINSUM, B><<<grid, kColWarps * 32, 0, st>>>(msg, lr, d_decw_, s.actw, post, d_col_ptr_, d_col_edge_, N_, E_, g0, cpw); \
        else col_pass_kernel<T, DV, EX, ALG_BP, B><<<grid, kColWarps * 32, 0, st>>>(msg, lr, d_decw_, s.actw, post, d_col_ptr_, d_col_edge_, N_, E_, g0, cpw);         \
    } while (0)
#define COL(DV, EX)                          \
    do {                                     \
        if (bits == 4) COLB(DV, EX, 4);      \
        else if (bits == 3) COLB(DV, EX, 3); \
        else if (bits == 2) COLB(DV, EX, 2); \
        else COLB(DV, EX, 1);                \
    } while (0)
    if (reg_cols_ && max_col_deg_ == 8) COL(8, true);
    else if (reg_cols_ && max_col_deg_ == 3) COL(3, true);
    else if (max_col_deg_ <= 4) COL(4, false);
    else if (max_col_deg_ <= 8) COL(8, false);
    else COLB(16, false, 1);
#undef COL
#undef COLB
    stats.kernel_launches++;
    CK(cudaGetLastError());
    return DNALDPC_OK;
}

// check() + loop control for the slots under consideration (syndrome_update_*_kernel)
int Engine::launch_syndrome(const dnaldpc_output &out, int G, int max_iter, int consider_new, int fixed, unsigned *counter,
                            unsigned *finished, unsigned *rearm, int clear_fresh, cudaStream_t st) {
    SchedArrays s;
    fill_sched(s);
    SynArgs a;
    a.iters_out = out.iters; a.ok_out = out.is_codeword;
    a.M = M_; a.N = N_; a.g0 = 0; a.max_iter = max_iter; a.consider_new = consider_new; a.fixed_iters = fixed;
    a.counter = counter; a.finished = finished; a.counters_to_zero = rearm; a.clear_fresh = clear_fresh;
    a.row_jobs = d_counters_ + (size_t)kRing * kCounterWords;
    const size_t smem = (size_t)N_ * sizeof(uint32_t);
    static const bool no_smem = getenv("DNALDPC_SYN_GATHER") != nullptr;  // A/B switch: global-gather variant
    if (!no_smem && smem <= (size_t)kSynSmemGate && N_ % 4 == 0) {  // the group's decision words staged in shared memory
        if (!syn_attr_set_) {
            // The attribute is global per (function, device): always raise it to the fixed gate value so that decoders
            // for different codes on one GPU cannot lower each other's limit.
            CK(cudaFuncSetAttribute(syndrome_update_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSynSmemGate));
            syn_attr_set_ = true;
        }
        static const int split = getenv("DNALDPC_SYN_SPLIT") ? std::max(1, atoi(getenv("DNALDPC_SYN_SPLIT"))) : kSynSmemSplit;  // A/B switch
        syndrome_update_smem_kernel<<<dim3((unsigned)split, (unsigned)G), kSynSmemThreads, smem, st>>>(d_decw_, s, a, d_row_ptr_, d_col_idx_);
    } else if (!no_smem && (size_t)N_ * sizeof(uint16_t) <= (size_t)kSynHalfGate && N_ % 4 == 0) {  // 16 slots' bits of every word staged
        if (!syn_half_attr_set_) {
            CK(cudaFuncSetAttribute(syndrome_update_half_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSynHalfGate));
            syn_half_attr_set_ = true;
        }
        syndrome_update_half_kernel<<<dim3(kSynSmemSplit, (unsigned)G, 2), kSynSmemThreads, (size_t)N_ * sizeof(uint16_t), st>>>(d_decw_, s, a, d_row_ptr_, d_col_idx_);
    } else {
        syndrome_update_kernel<<<dim3(kSynSplit, (unsigned)G), kSynThreads, 0, st>>>(d_decw_, s, a, d_row_ptr_, d_col_idx_);
    }
    stats.kernel_launches++;
    CK(cudaGetLastError());
    return DNALDPC_OK;
}

template <typename T>
int Engine::launch_harvest_setup(const dnaldpc_input &in, const dnaldpc_output &out, int g0, int G, cudaStream_t st) {
    SetupArgs a;
    a.data = in.data;
    a.frame_stride = in.frame_stride;
    a.param = in.param;
    if (in.kind == DNALDPC_IN_LLR_F64 && in.param == 0.0) a.param = 1.0;
    a.table = d_table_;
    HarvestArgs h;
    h.bits = out.bits; h.dblk = out.dblk; h.posterior = out.posterior; h.wpf = (N_ + 31) / 32;
    SchedArrays s;
    fill_sched(s);
    if (out.pchk) {
        dim3 grid((unsigned)((M_ + 255) / 256), (unsigned)G);
        syndrome_bytes_kernel<<<grid, 256, 0, st>>>(d_decw_, s, d_row_ptr_, d_col_idx_, M_, N_, g0, out.pchk);
        stats.kernel_launches++;
    }
    static const int tpw = getenv("DNALDPC_HS_TILES") ? std::max(1, atoi(getenv("DNALDPC_HS_TILES"))) : kHsTilesPerWarp;  // A/B switch
    const int tiles_per_cta = kHsWarps * tpw;
    dim3 grid((unsigned)(((N_ + 31) / 32 + tiles_per_cta - 1) / tiles_per_cta), (unsigned)G);
    T *lr = (T *)d_lratio_;
    const T *post = (const T *)d_post_;
#define HS(K)                                                                                                   \
    do {                                                                                                        \
        if (minsum_) harvest_setup_kernel<T, K, ALG_MINSUM><<<grid, kHsWarps * 32, 0, st>>>(a, h, s, lr, post, d_decw_, N_, g0, tpw); \
        else harvest_setup_kernel<T, K, ALG_BP><<<grid, kHsWarps * 32, 0, st>>>(a, h, s, lr, post, d_decw_, N_, g0, tpw);         \
    } while (0)
    switch (in.kind) {
        case DNALDPC_IN_LR_F64: HS(IN_LR_F64); break;
        case DNALDPC_IN_LLR_F64: HS(IN_LLR_F64); break;
        case DNALDPC_IN_BSC_BITS: HS(IN_BSC_BITS); break;
        case DNALDPC_IN_AWGN_F32: HS(IN_AWGN_F32); break;
        case DNALDPC_IN_AWGN_F64: HS(IN_AWGN_F64); break;
        case DNALDPC_IN_VOTE_I8: HS(IN_VOTE_I8); break;
        default: return fail("unknown input kind", DNALDPC_ERR_ARG);
    }
#undef HS
    stats.kernel_launches++;
    CK(cudaGetLastError());
    return DNALDPC_OK;
}

// ---- one batch: every frame the source publishes flows through the slots ------------------------------

int Engine::ensure_rows(int64_t frames) {
    if (frames > cap_rows_) {
        if (d_rows_) cudaFree(d_rows_);
        if (h_rows_) cudaFreeHost(h_rows_);
        if (h_avail_) cudaFreeHost(h_avail_);
        d_rows_ = nullptr; h_rows_ = nullptr; h_avail_ = nullptr; cap_rows_ = 0;
        CK(cudaMalloc((void **)&d_rows_, (size_t)frames * 2 * sizeof(int32_t)));
        // pinned mirrors for publishing through the copy engine (publish(..., dma)); without them the kernel is used
        if (cudaMallocHost((void **)&h_rows_, (size_t)frames * 2 * sizeof(int32_t)) != cudaSuccess ||
            cudaMallocHost((void **)&h_avail_, ((size_t)frames + 1) * sizeof(unsigned long long)) != cudaSuccess) {
            cudaGetLastError();
            if (h_rows_) cudaFreeHost(h_rows_);
            h_rows_ = nullptr; h_avail_ = nullptr;
        }
        cap_rows_ = frames;
    }
    return DNALDPC_OK;
}

int Engine::set_device() {
    CK(cudaSetDevice(device_));
    return DNALDPC_OK;
}

// Called from a source's producer thread while the tick thread is inside run(): touches neither err_ nor stats.
int Engine::publish(const int32_t *list_in, int row0_in, int row0_out, int n, cudaStream_t stream, bool dma) {
    if (n <= 0) return DNALDPC_OK;
    const int64_t q0 = published_.load(std::memory_order_relaxed);
    if (q0 + n > cap_rows_) return DNALDPC_ERR_ARG;  // more frames published than the session announced
    if (dma && !list_in && h_rows_) {
        // From a copy stream: the table entries and the counter travel through the copy engine like the inputs before
        // them. A kernel here would wait for a free SM slot - the persistent check pass holds every SM's registers for
        // 1.5 ms at a time - and, the stream being in order, hold back the next piece's copy: wide inputs (fp64 ratios,
        // 147 KB per frame, 33 MB pieces) then reached the engine at 14.5 GB/s with the link idle most of the time.
        int32_t *hi = h_rows_ + q0, *ho = h_rows_ + cap_rows_ + q0;
        for (int i = 0; i < n; i++) { hi[i] = row0_in + i; ho[i] = row0_out + i; }
        h_avail_[q0 + n] = (unsigned long long)(q0 + n);  // one word per end position: never rewritten while a copy of it is pending
        if (cudaMemcpyAsync(d_rows_ + q0, hi, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, stream) != cudaSuccess ||
            cudaMemcpyAsync(d_rows_ + cap_rows_ + q0, ho, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, stream) != cudaSuccess ||
            cudaMemcpyAsync(d_next_ + 1, h_avail_ + q0 + n, sizeof(unsigned long long), cudaMemcpyHostToDevice, stream) != cudaSuccess)
            return DNALDPC_ERR_CUDA;
        published_.store(q0 + n, std::memory_order_release);
        return DNALDPC_OK;
    }
    publish_kernel<<<1, 1024, 0, stream>>>(d_rows_, d_rows_ + cap_rows_, (long long)q0, n, list_in, row0_in, row0_out, d_next_ + 1);
    if (cudaGetLastError() != cudaSuccess) return DNALDPC_ERR_CUDA;
    published_.store(q0 + n, std::memory_order_release);
    return DNALDPC_OK;
}

template <typename T>
int Engine::run(const Session &ss, FrameSource &src, cudaStream_t st) {
    const dnaldpc_input &in = ss.in;
    const int64_t Fmax = ss.max_frames;
    if (Fmax <= 0) return DNALDPC_OK;
    if (Fmax > 0x7fffffffLL) return fail("more than 2^31-1 frames in one call", DNALDPC_ERR_ARG);
    const int G = (int)std::min<int64_t>((Fmax + 31) / 32, wave_frames_ / 32);
    const long long S = (long long)G * kFG;
    const bool want_post = ss.out.posterior != nullptr;
    int rc = ensure_slots(G, want_post);
    if (rc) return rc;
    rc = ensure_rows(Fmax);
    if (rc) return rc;
    dnaldpc_output out = ss.out;
    if (!out.iters || !out.is_codeword) {  // indexed by output row: the caller's rows are below max_frames here
        rc = ensure_frame_scratch(Fmax);
        if (rc) return rc;
        if (!out.iters) out.iters = d_iters_;
        if (!out.is_codeword) out.is_codeword = d_ok_;
    }
    minsum_ = (in.flags & DNALDPC_FLAG_MINSUM) != 0;
    if (in.kind == DNALDPC_IN_BSC_BITS || in.kind == DNALDPC_IN_VOTE_I8) {
        double tab[256];
        int cnt = 256;
        bool user_table = false;
        if (in.kind == DNALDPC_IN_BSC_BITS) {
            dnaldpc_bsc_table(in.param, tab);
            cnt = 2;
            if (minsum_) { tab[0] = std::log(tab[0]); tab[1] = std::log(tab[1]); }  // received_LLR = log(received_LR), channel.cpp:78,83
        } else if (in.table) user_table = true;  // caller's table (HOST or DEVICE pointer): ratios for BP, LLRs for min-sum
        else if (minsum_) {
            const double L = std::log((1 - in.param) / in.param);
            for (int k = -128; k < 128; k++) tab[k + 128] = k * L;                   // decoder.py:314
        } else dnaldpc_vote_table(in.param, tab);
        // pageable source: copied to a driver staging buffer before the call returns. A caller's table may live on
        // either side (cudaMemcpyDefault resolves it through unified addressing).
        if (user_table) CK(cudaMemcpyAsync(d_table_, in.table, 256 * sizeof(double), cudaMemcpyDefault, st));
        else CK(cudaMemcpyAsync(d_table_, tab, cnt * sizeof(double), cudaMemcpyHostToDevice, st));
    }
    SchedArrays s;
    fill_sched(s);
    published_.store(0, std::memory_order_release);
    init_sched_kernel<<<(G * kFG + 255) / 256, 256, 0, st>>>(s, G, d_counters_, kRing);
    stats.kernel_launches++;
    CK(cudaGetLastError());
    // the queue is empty and *avail == 0 from here on in stream order; producers on other streams wait for this point
    CK(cudaEventRecord(ready_ev_, st));
    steady_ = false;
    traced_ = 0;

    // One tick = admit/harvest/check (twice) + one check-node pass + one bit-node pass over all slots.
    // (Measured alternative, removed: two halves of the groups ticking on two streams so that one half's kernel tail is
    // filled by the other's next kernel: +0.4 % with the register-resident check kernel, -3 % with the smem-staged one.)
    unsigned last_inuse = 0, last_admitted = 1, last_finished = 1;  // what the host knows (kLag ticks old)
    // Drain tail: once every frame has been admitted (the source is final and the polled `admitted` counters add up to
    // what was published) finished slots stay empty and the stragglers thin out over all groups; whenever at most
    // kCompactNum / kCompactDen (15/16, about 93 %) of the slots of the packed region are still busy they are compacted
    // into the lowest groups (compact_*_kernel) and the check / bit passes shrink to those groups.
    const bool no_compact = getenv("DNALDPC_NO_COMPACT") != nullptr;  // A/B switch, read per batch
    // threshold in per cent of the packed region (default 100 * kCompactNum / kCompactDen = 93); tests set it to
    // exercise other compaction schedules
    const long long compact_pct = getenv("DNALDPC_COMPACT_PCT") ? std::max(1, std::min(99, atoi(getenv("DNALDPC_COMPACT_PCT")))) : 100LL * kCompactNum / kCompactDen;
    long long admitted_total = 0, low_water = 0;
    bool final = false;
    bool admit_ring[kRing] = {};
    int G_rc = G;                  // groups the check / bit passes are launched over
    long long packed_cap = S;      // slots of the region the busy slots were last packed into
    const int fixed = (in.flags & DNALDPC_FLAG_FIXED_ITERS) ? 1 : 0;
    for (long long tick = 0;; tick++) {
        rc = src.pump(*this, admitted_total, low_water, &final);
        if (rc) return err_.empty() ? fail("the frame source of this batch failed", rc) : rc;
        const long long pub = published();
        // ring entry of this tick: [0] slots in use, [1] frames admitted, [2] frames finished, [3] low-water q
        unsigned *cnt = d_counters_ + kCounterWords * (tick % kRing);
        unsigned *rearm = d_counters_ + kCounterWords * ((tick + kRing / 2) % kRing);
        // Admission (assign + harvest/setup, twice) is only launched when the host has reason to expect work for it:
        // start-up, a frame finished or was admitted kLag ticks ago, or slots are idle while frames wait. In the steady
        // state of long frames a tick is just syndrome -> check pass -> bit pass; a finish is then picked up at most
        // kLag ticks late.
        const bool admit = tick < 2 + kLag || last_finished > 0 || last_admitted > 0 || (last_inuse < (unsigned)S && pub > admitted_total);
        admit_ring[tick % kRing] = admit;
        if (admit) {
            // Two admission rounds: slots that finish in round 1 (incl. frames that need no iteration at all) are
            // harvested and refilled at once, so a slot idles at most in the rare case of two finishes in a row.
            for (int round = 1; round <= 2; round++) {
                assign_kernel<<<(G + 7) / 8, 256, 0, st>>>(s, 0, G, round == 1, cnt + 1, cnt + 3);
                stats.kernel_launches++;
                rc = launch_harvest_setup<T>(in, out, 0, G, st);
                if (rc) return rc;
                rc = launch_syndrome(out, G, ss.max_iter, round == 2, fixed, round == 2 ? cnt : nullptr, cnt + 2,
                                     round == 1 ? rearm : nullptr, 0, st);
                if (rc) return rc;
            }
        } else {
            rc = launch_syndrome(out, G, ss.max_iter, 0, fixed, cnt, cnt + 2, rearm, 1, st);
            if (rc) return rc;
        }
        CK(cudaMemcpyAsync(h_counters_ + kCounterWords * (tick % kRing), cnt, kCounterWords * sizeof(unsigned), cudaMemcpyDeviceToHost, st));
        CK(cudaEventRecord(ev_[tick % kRing], st));
        if (tick >= kLag) {  // lagged poll: the host runs at most kLag ticks ahead of the device
            const long long t = tick - kLag;
            CK(cudaEventSynchronize(ev_[t % kRing]));
            const unsigned *hc = h_counters_ + kCounterWords * (t % kRing);
            last_inuse = hc[0]; last_admitted = hc[1]; last_finished = hc[2];
            admitted_total += last_admitted;
            // every q below the smallest one that was still in a slot after tick t's admission has been harvested by
            // tick t's harvest kernels, which have completed (the event above); without admission nothing was harvested
            if (admit_ring[t % kRing]) low_water = std::min<long long>(hc[3] == 0xffffffffu ? admitted_total : (long long)hc[3], admitted_total);
            if (final && admitted_total == published() && last_inuse == 0) break;  // drained: nothing active, unharvested or pending
            // steady state = every slot busy and nobody being admitted (e.g. long-running frames)
            steady_ = last_admitted == 0 && last_inuse >= (unsigned)S;
            if (!final && last_inuse == 0 && admitted_total == published()) {
                // Idle engine, starved source: do not spin empty ticks. The check / bit passes below still run: this tick's
                // admission kernels are already queued and may pick up frames published meanwhile, and a slot's fresh mark
                // is only valid until the next tick's admission.
                src.wait_for_frames();
                last_admitted = 1;  // look for frames in the next tick
            }
            if (!no_compact && !profiling && final && admitted_total == published() && packed_cap >= 2 * kFG &&
                (long long)last_inuse * 100 <= packed_cap * compact_pct) {
                // `last_inuse` is kLag ticks old and can only have shrunk since: it bounds the moves and the packed size
                int32_t *mv_src = d_mv_, *mv_dst = d_mv_ + (size_t)cap_groups_ * kFG, *mv_cnt = d_mv_ + (size_t)cap_groups_ * kFG * 2;
                compact_plan_kernel<<<1, 32, 0, st>>>(s, G, mv_src, mv_dst, mv_cnt);
                dim3 mgrid((unsigned)((E_ + N_ + kMoveThreads * kMoveUnroll - 1) / (kMoveThreads * kMoveUnroll)),
                           (unsigned)std::min<unsigned>(std::max(last_inuse, 1u), 2048u));
                compact_move_kernel<T><<<mgrid, kMoveThreads, 0, st>>>((T *)d_msg_, (T *)d_lratio_, mv_src, mv_dst, mv_cnt, N_, E_);
                stats.kernel_launches += 2;
                stats.compactions++;
                CK(cudaGetLastError());
                G_rc = (int)std::min<long long>(G, ((long long)last_inuse + kFG - 1) / kFG);
                G_rc = std::max(G_rc, 1);
                packed_cap = (long long)G_rc * kFG;
            }
        }
        const bool trace = trace_ticks_ > 0 && tick >= 8 && tick < 8 + kTrace && tick < 8 + trace_ticks_;  // in-pipeline timing, no sync
        if (trace) CK(cudaEventRecord(trace_ev_[3 * (tick - 8)], st));
        if (profiling) CK(cudaEventRecord(prof_ev_[0], st));
        rc = launch_row<T>(0, G_rc, st);
        if (rc) return rc;
        if (profiling) CK(cudaEventRecord(prof_ev_[1], st));
        if (trace) CK(cudaEventRecord(trace_ev_[3 * (tick - 8) + 1], st));
        rc = launch_col<T>(0, G_rc, want_post, st);
        if (rc) return rc;
        if (trace) { CK(cudaEventRecord(trace_ev_[3 * (tick - 8) + 2], st)); traced_ = (int)(tick - 8) + 1; }
        if (profiling) {
            CK(cudaEventRecord(prof_ev_[2], st));
            CK(cudaEventSynchronize(prof_ev_[2]));
            float a_ms = 0, b_ms = 0;
            cudaEventElapsedTime(&a_ms, prof_ev_[0], prof_ev_[1]);
            cudaEventElapsedTime(&b_ms, prof_ev_[1], prof_ev_[2]);
            stats.row_ms += a_ms;
            stats.col_ms += b_ms;
            stats.waves++;  // profiled ticks
        }
    }
    // the loop ended on a host-synchronised event that follows the last harvest: the iteration sum is final
    unsigned long long it_sum = 0;
    CK(cudaMemcpyAsync(&it_sum, d_next_ + 2, sizeof(it_sum), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    stats.frame_iters = (int64_t)it_sum;
    stats.frames = admitted_total;
    low_water = admitted_total;
    rc = src.pump(*this, admitted_total, low_water, &final);  // lets the source retire the last outputs
    return rc;
}

// In-pipeline timing of ticks 8..8+n (events recorded without any synchronisation; call after the stream has drained):
// average check-pass, bit-pass and scheduler (bit-pass end -> next check-pass start) time per tick in ms.
int Engine::trace_result(double *row_ms, double *col_ms, double *sched_ms) {
    *row_ms = *col_ms = *sched_ms = 0;
    if (traced_ < 2) return 0;
    CK(cudaSetDevice(device_));
    CK(cudaEventSynchronize(trace_ev_[3 * (traced_ - 1) + 2]));
    double r = 0, c = 0, g = 0;
    for (int t = 0; t < traced_; t++) {
        float a = 0, b = 0, d = 0;
        cudaEventElapsedTime(&a, trace_ev_[3 * t], trace_ev_[3 * t + 1]);
        cudaEventElapsedTime(&b, trace_ev_[3 * t + 1], trace_ev_[3 * t + 2]);
        if (t + 1 < traced_) cudaEventElapsedTime(&d, trace_ev_[3 * t + 2], trace_ev_[3 * (t + 1)]);
        r += a; c += b; g += d;
    }
    *row_ms = r / traced_; *col_ms = c / traced_; *sched_ms = g / (traced_ - 1);
    return traced_;
}

int Engine::run_session(const Session &ss, FrameSource &src, cudaStream_t stream) {
    if (!err_.empty() && d_row_ptr_ == nullptr) return DNALDPC_ERR_CUDA;
    err_.clear();
    if (ss.max_frames < 0 || ss.max_iter < 0) return fail("bad argument", DNALDPC_ERR_ARG);
    CK(cudaSetDevice(device_));
    stats = dnaldpc_stats{};
    cudaStream_t st = stream ? stream : own_stream_;
    return precision_ == DNALDPC_PREC_F32 ? run<float>(ss, src, st) : run<double>(ss, src, st);
}

void *Engine::stage(void **buf, size_t *cap, size_t need) {
    if (need > *cap) {
        if (*buf) cudaFree(*buf);
        *buf = nullptr; *cap = 0;
        if (cudaMalloc(buf, need) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        *cap = need;
    }
    return *buf;
}

void *Engine::pinned(size_t need) {
    if (need > c_bounce_) {
        if (h_bounce_) cudaFreeHost(h_bounce_);
        h_bounce_ = nullptr; c_bounce_ = 0;
        if (cudaMallocHost(&h_bounce_, need) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        c_bounce_ = need;
    }
    return h_bounce_;
}

// ---- sliding-window BP for spatially-coupled codes (SURVEY 8f-3) ------------------------------------

// Window ranges of every position, with the running sums of Run_SW_Decoder itself (dec.cpp:2115-2183).
// Per position: {V_Start, V_End, C_Start, C_End, V_Check_End, C_Check_End, Init_from, Init_to}.
static std::vector<int> sw_schedule(int M, int N, const dnaldpc_window &w) {
    const int L = w.L, D = w.code_type == 0 ? L + w.w - 1 : L + (w.w - 1) / 2;
    std::vector<int> s((size_t)8 * L);
    int vs = 0, ve = 0, cs = 0, ce = 0, vce = 0, cce = 0;
    for (int i = 0; i < w.w; i++) { vce += w.Mv[i]; cce += w.Mc[i]; }
    for (int i = 0; i < w.win; i++) { ve += w.Mv[i]; ce += w.Mc[i]; }
    for (int t = 0; t < L; t++) {
        int init_from = ve, init_to = ve;
        if (t == 0) init_from = 0;
        else {
            vs += w.Mv[t - 1];
            cs += w.Mc[t - 1];
            ve = (t + w.win >= L) ? N : ve + w.Mv[t + w.win - 1];
            ce = (t + w.win >= D) ? M : ce + w.Mc[t + w.win - 1];
            if (t + w.w >= L) { vce = N; cce = M; }
            else { vce += w.Mv[t + w.w - 1]; cce += w.Mc[t + w.w - 1]; }
            init_from = init_to = ve;
            if (t + w.win <= L) init_from = ve - w.Mv[t + w.win - 1];
        }
        int *r = &s[(size_t)8 * t];
        r[0] = vs; r[1] = ve; r[2] = cs; r[3] = ce; r[4] = vce; r[5] = cce; r[6] = init_from; r[7] = init_to;
    }
    return s;
}

int Engine::decode_window_host(const Code &code, const dnaldpc_window &w, const double *lratio, int64_t F, int max_iter,
                               const dnaldpc_output &out) {
    if (!err_.empty() && d_row_ptr_ == nullptr) return DNALDPC_ERR_CUDA;
    err_.clear();
    if (precision_ != DNALDPC_PREC_F64) return fail("the sliding-window decoder runs in fp64 only", DNALDPC_ERR_UNSUPPORTED);
    if (F < 0 || max_iter < 0 || (F > 0 && !lratio) || out.posterior) return fail("bad argument", DNALDPC_ERR_ARG);
    const int D = w.code_type == 0 ? w.L + w.w - 1 : w.L + (w.w - 1) / 2;
    if (w.L < 1 || w.w < 1 || w.win < 1 || !w.Mv || !w.Mc || w.win > D || w.w > D) return fail("bad window description", DNALDPC_ERR_ARG);
    const std::vector<int> sched = sw_schedule(M_, N_, w);
    for (int t = 0; t < w.L; t++) {  // the ranges index H directly in the reference; reject what would run off the matrix there
        const int *r = &sched[(size_t)8 * t];
        if (r[0] < 0 || r[1] > N_ || r[0] > r[1] || r[2] < 0 || r[3] > M_ || r[2] > r[3] || r[4] > N_ || r[5] > M_ || r[6] < 0 || r[6] > r[7])
            return fail("window ranges leave the parity-check matrix (Mv / Mc do not match the code)", DNALDPC_ERR_ARG);
    }
    if (F == 0) return DNALDPC_OK;
    CK(cudaSetDevice(device_));
    cudaStream_t st = own_stream_;
    stats = dnaldpc_stats{};
    stats.frames = F;
    const bool lockstep = getenv("DNALDPC_SW_LOCKSTEP") && atoi(getenv("DNALDPC_SW_LOCKSTEP")) != 0;  // A/B switch, see below
    // Slots of the window decoder. Most of a tick's launches are short (a few frames per group iterate on), so more
    // groups in flight fill the machine better (16 384 frames on the Z=1024 x L=24 code: 4096 slots 28.1 k frames/s, 8192
    // 30.6 k, 16 384 31.7 k): up to 4 x wave_frames when that takes at most a third of the free device memory. Decided
    // once per engine; DNALDPC_SW_SLOTS_X = 1 / 2 / 4 overrides.
    if (sw_slots_ == 0) {
        sw_slots_ = wave_frames_;
        if (!lockstep) {
            size_t free_b = 0, total_b = 0;
            CK(cudaMemGetInfo(&free_b, &total_b));
            const size_t per_slot = ((size_t)2 * E_ + N_) * sizeof(double) + (size_t)N_ / 8 + 64;
            const int want_x = getenv("DNALDPC_SW_SLOTS_X") ? atoi(getenv("DNALDPC_SW_SLOTS_X")) : 0;
            for (int x : {4, 2})
                if (want_x ? x == want_x : (size_t)wave_frames_ * x * per_slot <= free_b / 3) { sw_slots_ = wave_frames_ * x; break; }
        }
    }
    const int G = (int)std::min<int64_t>((F + 31) / 32, (lockstep ? wave_frames_ : sw_slots_) / 32);
    int rc = ensure_slots(G, false);
    if (rc) return rc;
    if (G > sw_cap_groups_) {
        if (d_sw_lr_) cudaFree(d_sw_lr_);
        d_sw_lr_ = nullptr; sw_cap_groups_ = 0;
        CK(cudaMalloc(&d_sw_lr_, std::max<size_t>((size_t)G * E_ * kFG * sizeof(double), 16)));
        sw_cap_groups_ = G;
    }
    if (!d_edge_row_) {
        std::vector<int32_t> er((size_t)std::max(E_, 1));
        for (int i = 0; i < M_; i++)
            for (int e = code.row_ptr[i]; e < code.row_ptr[i + 1]; e++) er[e] = i;
        CK(cudaMalloc((void **)&d_edge_row_, er.size() * sizeof(int32_t)));
        CK(cudaMemcpy(d_edge_row_, er.data(), er.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    }
    if (!d_col_row_) {  // check of the k-th entry of a column (same order as col_edge)
        std::vector<int32_t> cr((size_t)std::max(E_, 1));
        std::vector<int32_t> er((size_t)std::max(E_, 1));
        for (int i = 0; i < M_; i++)
            for (int e = code.row_ptr[i]; e < code.row_ptr[i + 1]; e++) er[e] = i;
        for (int k = 0; k < E_; k++) cr[k] = er[code.col_edge[k]];
        CK(cudaMalloc((void **)&d_col_row_, cr.size() * sizeof(int32_t)));
        CK(cudaMemcpy(d_col_row_, cr.data(), cr.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    }
    // A/B switch: the wave-lock-step schedule of the first version (every position runs until the slowest frame of the
    // wave has left it) instead of continuous batching by group
    if (lockstep) return sw_lockstep(w, sched, lratio, F, max_iter, out, G);
    return sw_groups(code, w, sched, lratio, F, max_iter, out, G);
}

// Continuous batching by group (sw_kernels.cuh, sw2_*): the frames of a chunk are staged in HBM (the next chunk's copy
// runs meanwhile), the groups pull them 32 at a time from a device counter, every group walks through the window
// positions at its own pace and a tick is one update of every group; the host counts harvested frames kLag ticks late.
int Engine::sw_groups(const Code &code, const dnaldpc_window &w, const std::vector<int> &sched, const double *lratio, int64_t F,
                      int max_iter, const dnaldpc_output &out, int G) {
    cudaStream_t st = own_stream_, st_in = io_stream_[0];
    const int L = w.L;
    int max_rows = 0, max_cols = 0, max_init = 0;
    for (int t = 0; t < L; t++) {
        const int *r = &sched[(size_t)8 * t];
        max_rows = std::max(max_rows, r[3] - r[2]);
        max_cols = std::max(max_cols, r[1] - r[0]);
        max_init = std::max(max_init, r[7] - r[6]);
    }
    // Does a check of some window ever touch a column Init_SW_Decoder has not reached yet? Then the zeros alloc_entry
    // left in e->pr / e->lr are operands and a group's arrays are cleared for every new set of frames; for a window
    // description that matches the code (every check's bits enter the window no later than the check) nothing a frame
    // reads was written by the group's previous frames, and the 2 x E x 256 bytes per group stay untouched.
    bool zero = false;
    {
        std::vector<int> init_at((size_t)N_, L);  // position at which a column is initialised
        for (int t = 0; t < L; t++) {
            const int *r = &sched[(size_t)8 * t];
            for (int j = r[6]; j < r[7]; j++) init_at[(size_t)j] = std::min(init_at[(size_t)j], t);
        }
        std::vector<char> seen((size_t)M_, 0);
        for (int t = 0; t < L && !zero; t++) {
            const int *r = &sched[(size_t)8 * t];
            for (int i = r[2]; i < r[3] && !zero; i++) {
                if (seen[(size_t)i]) continue;  // a check's first position decides: columns are only ever added
                seen[(size_t)i] = 1;
                for (int e = code.row_ptr[i]; e < code.row_ptr[i + 1]; e++)
                    if (init_at[(size_t)code.col_idx[e]] > t) { zero = true; break; }
            }
        }
    }
    if (getenv("DNALDPC_SW_ZERO") && atoi(getenv("DNALDPC_SW_ZERO")) != 0) zero = true;  // test switch
    const uint32_t load_flags = SW_LOAD | SW_INIT | (zero ? SW_ZERO : 0u);
    if (L > sw_cap_sched_) {
        if (d_sw_sched_) cudaFree(d_sw_sched_);
        d_sw_sched_ = nullptr; sw_cap_sched_ = 0;
        CK(cudaMalloc((void **)&d_sw_sched_, (size_t)L * 8 * sizeof(int32_t)));
        sw_cap_sched_ = L;
    }
    CK(cudaMemcpyAsync(d_sw_sched_, sched.data(), (size_t)L * 8 * sizeof(int32_t), cudaMemcpyHostToDevice, st));  // pageable: staged before the call returns
    SchedArrays sa;
    fill_sched(sa);
    SwGroups s;
    s.run = sa.actw; s.valid = sa.donew; s.flags = sa.newfw; s.unsat = sa.freshw;
    s.pos = (int32_t *)sa.harvw; s.frame0 = (int32_t *)sa.unsatw;
    s.n_pos = sa.slot_iter; s.sum = sa.harv_iter;
    s.sched = d_sw_sched_;
    s.next_frame = d_next_; s.done = d_next_ + 1;
    double *pr = (double *)d_msg_, *lr = (double *)d_sw_lr_, *lrat = (double *)d_lratio_;
    const size_t wpf = (size_t)(N_ + 31) / 32;
    // chunk of frames staged at a time: about 6 GB of input, at least the slots
    const int64_t S = (int64_t)G * kFG;
    int64_t chunk = std::max<int64_t>(S, ((int64_t)6 << 30) / ((int64_t)N_ * 8) / 32 * 32);
    if (const char *t = getenv("DNALDPC_SW_CHUNK")) chunk = std::max<int64_t>(32, atoll(t) / 32 * 32);  // test switch
    chunk = std::min<int64_t>(chunk, (F + 31) / 32 * 32);
    const bool two = F > chunk;
    void **in_buf[2] = {&s_in_, &s_in2_};
    size_t *in_cap[2] = {&c_in_, &c_in2_};
    for (int b = 0; b < (two ? 2 : 1); b++)
        if (!stage(in_buf[b], in_cap[b], (size_t)std::min<int64_t>(chunk, F) * N_ * 8)) return fail("out of device memory (input staging)", DNALDPC_ERR_NOMEM);
    if (!sw_in_ev_[0])
        for (auto &e : sw_in_ev_) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    if (!d_sw_avail_) CK(cudaMalloc((void **)&d_sw_avail_, 2 * sizeof(unsigned long long)));
    if (G > sw_cap_lists_) {
        if (d_sw_lists_) cudaFree(d_sw_lists_);
        d_sw_lists_ = nullptr; sw_cap_lists_ = 0;
        CK(cudaMalloc((void **)&d_sw_lists_, ((size_t)7 * G + 4) * sizeof(int32_t)));  // 4 lists + 4 counts, then thin_map / thin_e0 / thin_ne
        sw_cap_lists_ = G;
    }
    // straggler mode (sw2_thin_copy_kernel): side arrays with 4 slots per edge for the edges of one window's checks
    int thin_edges = 0;
    for (int t = 0; t < L; t++) thin_edges = std::max(thin_edges, code.row_ptr[sched[(size_t)8 * t + 3]] - code.row_ptr[sched[(size_t)8 * t + 2]]);
    bool thin_on = !(getenv("DNALDPC_SW_THIN") && atoi(getenv("DNALDPC_SW_THIN")) == 0) && thin_edges > 0;  // A/B switch
    if (thin_on) {
        const size_t need = (size_t)G * thin_edges * kSwThinLanes * 2 * sizeof(double);
        if (need > sw_cap_thin_) {
            if (d_sw_thin_) cudaFree(d_sw_thin_);
            d_sw_thin_ = nullptr; sw_cap_thin_ = 0;
            if (cudaMalloc(&d_sw_thin_, need) == cudaSuccess) sw_cap_thin_ = need;
            else { cudaGetLastError(); d_sw_thin_ = nullptr; thin_on = false; }  // short of memory: decode without the side arrays
        }
    }
    // A chunk is copied in pieces of about 64 MB; behind every piece the copy stream publishes how many frames of the
    // chunk are resident, and the groups only take frames that are (sw2_claim_kernel): decoding starts with the first
    // piece, and the next chunk's copy runs while this one is decoded. (Pageable host memory: the copies block the
    // calling thread, so they do not overlap the decoding; results are the same.)
    int64_t piece = std::max<int64_t>(32, ((int64_t)64 << 20) / ((int64_t)N_ * 8) / 32 * 32);
    if (const char *t = getenv("DNALDPC_SW_PIECE")) piece = std::max<int64_t>(32, atoll(t) / 32 * 32);  // test switch
    auto upload = [&](int64_t f0, int b) -> int {
        const int64_t nf = std::min<int64_t>(chunk, F - f0);
        CK(cudaMemsetAsync(d_sw_avail_ + b, 0, sizeof(unsigned long long), st_in));
        CK(cudaEventRecord(sw_in_ev_[b], st_in));  // the decoding of this chunk may start: nothing is resident yet
        for (int64_t p0 = 0; p0 < nf; p0 += piece) {
            const int64_t np = std::min<int64_t>(piece, nf - p0);
            CK(cudaMemcpyAsync((double *)*in_buf[b] + (size_t)p0 * N_, lratio + (size_t)(f0 + p0) * N_, (size_t)np * N_ * 8, cudaMemcpyHostToDevice, st_in));
            sw2_publish_kernel<<<1, 1, 0, st_in>>>(d_sw_avail_ + b, (unsigned long long)(p0 + np));
            stats.kernel_launches++;
        }
        CK(cudaGetLastError());
        return DNALDPC_OK;
    };
    int rc = upload(0, 0);
    if (rc) return rc;
    static const int packed = getenv("DNALDPC_SW_PACKED") ? atoi(getenv("DNALDPC_SW_PACKED")) : 1;  // A/B switch: 0 = a warp per node whatever the number of running frames
    long long tick = 0;
    int b = 0;
    for (int64_t f0 = 0; f0 < F; f0 += chunk, b ^= 1) {
        const int nf = (int)std::min<int64_t>(chunk, F - f0);
        const int Gc = (int)std::min<int64_t>(G, (nf + 31) / 32);
        dnaldpc_output o{};
        if (out.bits && !(o.bits = (uint32_t *)stage(&s_bits_, &c_bits_, (size_t)nf * wpf * 4))) return fail("out of device memory", DNALDPC_ERR_NOMEM);
        if (out.dblk && !(o.dblk = (uint8_t *)stage(&s_dblk_, &c_dblk_, (size_t)nf * N_))) return fail("out of device memory", DNALDPC_ERR_NOMEM);
        if (out.pchk && !(o.pchk = (uint8_t *)stage(&s_pchk_, &c_pchk_, (size_t)nf * M_))) return fail("out of device memory", DNALDPC_ERR_NOMEM);
        rc = ensure_frame_scratch(nf);
        if (rc) return rc;
        CK(cudaStreamWaitEvent(st, sw_in_ev_[b], 0));
        if (f0 + chunk < F) {  // the other buffer's last reader (the chunk before this one) has drained: see the sync below
            rc = upload(f0 + chunk, b ^ 1);
            if (rc) return rc;
        }
        const double *in = (const double *)*in_buf[b];
        s.avail = d_sw_avail_ + b;
        s.lists = d_sw_lists_;
        s.thin_map = (uint32_t *)(d_sw_lists_ + 4 * (size_t)sw_cap_lists_ + 4);
        s.thin_e0 = d_sw_lists_ + 5 * (size_t)sw_cap_lists_ + 4;
        s.thin_ne = d_sw_lists_ + 6 * (size_t)sw_cap_lists_ + 4;
        s.thin_edges = thin_edges;
        s.hist = nullptr;
        if (getenv("DNALDPC_SW_HIST")) {  // diagnostics: how many frames of a group run in an update
            if (!d_sw_hist_) CK(cudaMalloc((void **)&d_sw_hist_, 66 * sizeof(unsigned long long)));
            CK(cudaMemsetAsync(d_sw_hist_, 0, 66 * sizeof(unsigned long long), st));
            s.hist = d_sw_hist_;
        }
        s.thin_pr = thin_on ? (double *)d_sw_thin_ : nullptr;
        s.thin_lr = thin_on ? (double *)d_sw_thin_ + (size_t)G * thin_edges * kSwThinLanes : nullptr;
        CK(cudaMemsetAsync(d_next_, 0, 3 * sizeof(unsigned long long), st));
        const unsigned claim_grid = (unsigned)((Gc * kFG + 255) / 256);
        sw2_claim_kernel<<<claim_grid, 256, 0, st>>>(s, Gc, L, nf, 1, load_flags, d_iters_, d_ok_);
        stats.kernel_launches++;
        const unsigned load_x = (unsigned)((N_ + 31) / 32), head_y = (unsigned)std::min(Gc, 4);
        bool done = false;
        for (long long t0 = tick; !done; tick++) {
            sw2_list_kernel<<<1, 1024, 0, st>>>(s, Gc);
            sw2_load_kernel<<<dim3(load_x, head_y), 256, 0, st>>>(in, lrat, d_decw_, s, N_, Gc);
            if (zero) sw2_zero_kernel<<<dim3(64, head_y), 256, 0, st>>>(pr, lr, s, E_, Gc);
            if (thin_on) sw2_thin_copy_kernel<<<dim3(32, head_y), 256, 0, st>>>(pr, s, E_, Gc, 1);  // back, before Init_SW_Decoder of the new position
            if (max_init > 0) sw2_init_kernel<<<dim3((unsigned)((max_init + 7) / 8), head_y), 256, 0, st>>>(pr, lr, lrat, s, d_col_ptr_, d_col_edge_, N_, E_, Gc);
            if (thin_on) sw2_thin_copy_kernel<<<dim3(32, head_y), 256, 0, st>>>(pr, s, E_, Gc, 0);
            if (max_rows > 0) {
                const dim3 grid((unsigned)((max_rows + kSwNodesPerCta - 1) / kSwNodesPerCta), (unsigned)Gc);
                if (max_row_deg_ <= 8) sw2_row_kernel<8><<<grid, 256, 0, st>>>(pr, lr, s, d_row_ptr_, E_, packed);
                else sw2_row_kernel<0><<<grid, 256, 0, st>>>(pr, lr, s, d_row_ptr_, E_, packed);
            }
            if (max_cols > 0) {
                const dim3 grid((unsigned)((max_cols + kSwNodesPerCta - 1) / kSwNodesPerCta), (unsigned)Gc);
                if (max_col_deg_ <= 4) sw2_col_kernel<4><<<grid, 256, 0, st>>>(pr, lr, lrat, d_decw_, s, d_col_ptr_, d_col_edge_, d_col_row_, N_, E_, packed);
                else if (max_col_deg_ <= 8) sw2_col_kernel<8><<<grid, 256, 0, st>>>(pr, lr, lrat, d_decw_, s, d_col_ptr_, d_col_edge_, d_col_row_, N_, E_, packed);
                else sw2_col_kernel<0><<<grid, 256, 0, st>>>(pr, lr, lrat, d_decw_, s, d_col_ptr_, d_col_edge_, d_col_row_, N_, E_, packed);
            }
            sw2_syn_kernel<<<Gc, 256, 0, st>>>(d_decw_, s, d_row_ptr_, d_col_idx_, N_, max_iter, L);
            sw2_final_syn_kernel<<<dim3(kSwFinalSplit, (unsigned)Gc), 256, 0, st>>>(d_decw_, s, d_row_ptr_, d_col_idx_, N_, M_, o.pchk);
            if (o.bits || o.dblk) sw2_output_kernel<<<dim3((unsigned)((wpf + 7) / 8), (unsigned)Gc), 256, 0, st>>>(d_decw_, s, N_, (int)wpf, o.bits, o.dblk);
            sw2_claim_kernel<<<claim_grid, 256, 0, st>>>(s, Gc, L, nf, 0, load_flags, d_iters_, d_ok_);
            stats.kernel_launches += thin_on ? 12 : 10;
            stats.waves++;  // ticks
            unsigned *hc = h_counters_ + kCounterWords * (tick % kRing);
            CK(cudaMemcpyAsync(hc, d_next_ + 1, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
            CK(cudaEventRecord(ev_[tick % kRing], st));
            if (tick - t0 >= kLag) {
                const long long tl = tick - kLag;
                CK(cudaEventSynchronize(ev_[tl % kRing]));
                unsigned long long dn = 0;
                memcpy(&dn, h_counters_ + kCounterWords * (tl % kRing), sizeof(dn));
                done = dn >= (unsigned long long)nf;
            }
        }
        CK(cudaGetLastError());
        if (out.bits) CK(cudaMemcpyAsync(out.bits + (size_t)f0 * wpf, o.bits, (size_t)nf * wpf * 4, cudaMemcpyDeviceToHost, st));
        if (out.dblk) CK(cudaMemcpyAsync(out.dblk + (size_t)f0 * N_, o.dblk, (size_t)nf * N_, cudaMemcpyDeviceToHost, st));
        if (out.pchk) CK(cudaMemcpyAsync(out.pchk + (size_t)f0 * M_, o.pchk, (size_t)nf * M_, cudaMemcpyDeviceToHost, st));
        if (out.iters) CK(cudaMemcpyAsync(out.iters + f0, d_iters_, (size_t)nf * 4, cudaMemcpyDeviceToHost, st));
        if (out.is_codeword) CK(cudaMemcpyAsync(out.is_codeword + f0, d_ok_, (size_t)nf, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (s.hist) {
            unsigned long long h[66];
            CK(cudaMemcpy(h, d_sw_hist_, sizeof(h), cudaMemcpyDeviceToHost));
            fprintf(stderr, "sw group-updates by running frames (chunk at frame %lld):", (long long)f0);
            for (int k = 1; k <= 32; k++) fprintf(stderr, " %d:%llu", k, h[k]);
            fprintf(stderr, "\n  of which in straggler mode:");
            for (int k = 1; k <= 4; k++) fprintf(stderr, " %d:%llu", k, h[33 + k]);
            fprintf(stderr, "\n");
        }
    }
    if (out.iters) for (int64_t f = 0; f < F; f++) stats.frame_iters += out.iters[f];
    return DNALDPC_OK;
}

// The first version's schedule: the frames of a wave walk through the positions together.
int Engine::sw_lockstep(const dnaldpc_window &w, const std::vector<int> &sched, const double *lratio, int64_t F, int max_iter,
                        const dnaldpc_output &out, int G) {
    cudaStream_t st = own_stream_;
    int rc = DNALDPC_OK;
    SchedArrays s;
    fill_sched(s);
    uint32_t *runw = s.actw;
    int32_t *n_pos = s.slot_iter, *sum = s.harv_iter;
    unsigned *remaining = d_counters_;
    long long sw_upd = 0;  // updates launched so far (ring index of the progress counters)
    double *pr = (double *)d_msg_, *lr = (double *)d_sw_lr_, *lrat = (double *)d_lratio_;
    const size_t wpf = (size_t)(N_ + 31) / 32;
    const int64_t S = (int64_t)G * kFG;
    for (int64_t f0 = 0; f0 < F; f0 += S) {
        const int nf = (int)std::min<int64_t>(S, F - f0);
        const int Gw = (nf + 31) / 32;
        if (!stage(&s_in_, &c_in_, (size_t)nf * N_ * 8)) return fail("out of device memory (input staging)", DNALDPC_ERR_NOMEM);
        CK(cudaMemcpyAsync(s_in_, lratio + (size_t)f0 * N_, (size_t)nf * N_ * 8, cudaMemcpyHostToDevice, st));
        dnaldpc_output o{};
        if (out.bits && !(o.bits = (uint32_t *)stage(&s_bits_, &c_bits_, (size_t)nf * wpf * 4))) return fail("out of device memory", DNALDPC_ERR_NOMEM);
        if (out.dblk && !(o.dblk = (uint8_t *)stage(&s_dblk_, &c_dblk_, (size_t)nf * N_))) return fail("out of device memory", DNALDPC_ERR_NOMEM);
        if (out.pchk && !(o.pchk = (uint8_t *)stage(&s_pchk_, &c_pchk_, (size_t)nf * M_))) return fail("out of device memory", DNALDPC_ERR_NOMEM);
        rc = ensure_frame_scratch(nf);
        if (rc) return rc;
        sw_load_kernel<<<dim3((unsigned)((N_ + 31) / 32), (unsigned)Gw), 256, 0, st>>>((const double *)s_in_, lrat, d_decw_, N_, nf);
        CK(cudaMemsetAsync(pr, 0, (size_t)Gw * E_ * kFG * sizeof(double), st));  // alloc_entry: e->pr = e->lr = 0
        CK(cudaMemsetAsync(lr, 0, (size_t)Gw * E_ * kFG * sizeof(double), st));
        stats.kernel_launches++;
        for (int t = 0; t < w.L; t++) {
            const int *r = &sched[(size_t)8 * t];
            sw_begin_kernel<<<(Gw * kFG + 255) / 256, 256, 0, st>>>(runw, n_pos, sum, Gw, nf, t == 0);
            stats.kernel_launches++;
            if (r[7] > r[6]) {
                sw_init_kernel<<<dim3((unsigned)((r[7] - r[6] + 7) / 8), (unsigned)Gw), 256, 0, st>>>(pr, lr, lrat, d_col_ptr_, d_col_edge_, N_, E_, r[6], r[7]);
                stats.kernel_launches++;
            }
            // Every position runs at least one update, at most max_iter + 1. The host does not wait for an update's
            // "frames still running" count: it polls the count of kLag updates ago (ring of counters + events, like
            // the flooding scheduler), so the stream never drains; the updates launched after the last frame of the
            // position has finished find every group's run mask empty and return at once.
            bool done = false;
            for (int it = 0; it <= max_iter && !done; it++) {
                unsigned *rem = d_counters_ + (sw_upd % kRing);
                if (r[3] > r[2]) {
                    const long long items = (long long)Gw * (r[3] - r[2]);
                    if (max_row_deg_ <= 8) sw_row_reg_kernel<8><<<(unsigned)((items + 3) / 4), 128, 0, st>>>(pr, lr, runw, d_row_ptr_, E_, r[2], r[3], Gw);
                    else sw_row_kernel<<<(unsigned)((items + 3) / 4), 128, 0, st>>>(pr, lr, runw, d_row_ptr_, E_, r[2], r[3], Gw);
                    stats.kernel_launches++;
                }
                if (r[1] > r[0]) {
                    sw_col_kernel<<<dim3((unsigned)((r[1] - r[0] + 7) / 8), (unsigned)Gw), 256, 0, st>>>(
                        pr, lr, lrat, d_decw_, runw, d_col_ptr_, d_col_edge_, d_edge_row_, N_, E_, r[0], r[1], r[2], r[3]);
                    stats.kernel_launches++;
                }
                CK(cudaMemsetAsync(rem, 0, sizeof(unsigned), st));
                sw_syn_kernel<<<Gw, 256, 0, st>>>(d_decw_, runw, n_pos, sum, d_row_ptr_, d_col_idx_, N_, M_, r[0], r[4], r[2], r[5],
                                                  max_iter, rem, 0, w.L, nf, 0, nullptr, nullptr, nullptr);
                stats.kernel_launches++;
                CK(cudaMemcpyAsync(h_counters_ + (sw_upd % kRing), rem, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
                CK(cudaEventRecord(ev_[sw_upd % kRing], st));
                if (it >= kLag) {
                    CK(cudaEventSynchronize(ev_[(sw_upd - kLag) % kRing]));
                    done = h_counters_[(sw_upd - kLag) % kRing] == 0;
                }
                sw_upd++;
            }
        }
        sw_syn_kernel<<<Gw, 256, 0, st>>>(d_decw_, runw, n_pos, sum, d_row_ptr_, d_col_idx_, N_, M_, 0, N_, 0, M_, max_iter, remaining, 1,
                                          w.L, nf, 0, d_iters_, d_ok_, o.pchk);
        stats.kernel_launches++;
        if (o.bits || o.dblk) {
            sw_output_kernel<<<dim3((unsigned)((wpf + 255) / 256), (unsigned)nf), 256, 0, st>>>(d_decw_, N_, nf, 0, (int)wpf, o.bits, o.dblk);
            stats.kernel_launches++;
        }
        CK(cudaGetLastError());
        if (out.bits) CK(cudaMemcpyAsync(out.bits + (size_t)f0 * wpf, o.bits, (size_t)nf * wpf * 4, cudaMemcpyDeviceToHost, st));
        if (out.dblk) CK(cudaMemcpyAsync(out.dblk + (size_t)f0 * N_, o.dblk, (size_t)nf * N_, cudaMemcpyDeviceToHost, st));
        if (out.pchk) CK(cudaMemcpyAsync(out.pchk + (size_t)f0 * M_, o.pchk, (size_t)nf * M_, cudaMemcpyDeviceToHost, st));
        if (out.iters) CK(cudaMemcpyAsync(out.iters + f0, d_iters_, (size_t)nf * 4, cudaMemcpyDeviceToHost, st));
        if (out.is_codeword) CK(cudaMemcpyAsync(out.is_codeword + f0, d_ok_, (size_t)nf, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    if (out.iters) for (int64_t f = 0; f < F; f++) stats.frame_iters += out.iters[f];
    return DNALDPC_OK;
}

int Engine::synth_bsc(const uint32_t *cw_bits, int n_cw, uint64_t seed, int64_t frame0, int64_t F, double eps,
                      uint32_t *out_bits, cudaStream_t stream, uint64_t cw_off) {
    err_.clear();
    if (F < 0 || !out_bits || (cw_bits && n_cw <= 0) || !(eps >= 0.0 && eps <= 1.0)) return fail("bad argument", DNALDPC_ERR_ARG);
    CK(cudaSetDevice(device_));
    const int wpf = (N_ + 31) / 32;
    const long long total = (long long)F * wpf;
    if (total == 0) return DNALDPC_OK;
    const uint64_t thr = (uint64_t)(eps * 9007199254740992.0);
    synth_bsc_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(cw_bits, n_cw, cw_off, seed, frame0, F, N_, wpf, thr, out_bits);
    CK(cudaGetLastError());
    return DNALDPC_OK;
}

int Engine::synth_awgn(const uint32_t *cw_bits, int n_cw, uint64_t seed, int64_t frame0, int64_t F, double sigma,
                       float *out_y, cudaStream_t stream, uint64_t cw_off) {
    err_.clear();
    if (F < 0 || !out_y || (cw_bits && n_cw <= 0) || !(sigma >= 0.0)) return fail("bad argument", DNALDPC_ERR_ARG);
    CK(cudaSetDevice(device_));
    const long long total = (long long)F * N_;
    if (total == 0) return DNALDPC_OK;
    synth_awgn_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(cw_bits, n_cw, cw_off, seed, frame0, F, N_, (N_ + 31) / 32, sigma, out_y);
    CK(cudaGetLastError());
    return DNALDPC_OK;
}

// thr[k] = (uint64)(P(Poisson(mean) <= k) * 2^53), k = 0 .. kVoteMaxReads-1 (pmf by the recurrence p_k = p_{k-1} * mean / k
// from p_0 = exp(-mean), summed in ascending k): the host twin oracle/bp_oracle.c:orc_vote_thresholds does the same.
void vote_thresholds(double mean, uint64_t *thr) {
    double p = std::exp(-mean), cdf = 0;
    for (int k = 0; k < kVoteMaxReads; k++) {
        if (k > 0) p = p * mean / k;
        cdf += p;
        thr[k] = (uint64_t)(std::min(cdf, 1.0) * 9007199254740992.0);
    }
}

int Engine::synth_vote(const uint32_t *cw_bits, int n_cw, uint64_t seed, int64_t frame0, int64_t F, double mean_reads,
                       double read_err, int8_t *out_k, cudaStream_t stream, uint64_t cw_off) {
    err_.clear();
    if (F < 0 || !out_k || (cw_bits && n_cw <= 0) || !(mean_reads > 0.0 && mean_reads <= 32.0) || !(read_err >= 0.0 && read_err <= 1.0))
        return fail("bad argument (mean reads in (0, 32], read error in [0, 1])", DNALDPC_ERR_ARG);
    CK(cudaSetDevice(device_));
    const long long total = (long long)F * N_;
    if (total == 0) return DNALDPC_OK;
    uint64_t thr[kVoteMaxReads];
    vote_thresholds(mean_reads, thr);
    if (!d_synth_thr_) CK(cudaMalloc((void **)&d_synth_thr_, sizeof(thr)));
    CK(cudaMemcpyAsync(d_synth_thr_, thr, sizeof(thr), cudaMemcpyHostToDevice, stream));  // pageable: staged before the call returns
    const uint64_t thr_err = (uint64_t)(read_err * 9007199254740992.0);
    synth_vote_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(cw_bits, n_cw, cw_off, seed, frame0, F, N_, (N_ + 31) / 32, d_synth_thr_, thr_err, out_k);
    CK(cudaGetLastError());
    return DNALDPC_OK;
}

int Engine::ensure_lists(int64_t n) {
    if (n + 1 > cap_list_) {
        for (auto &p : d_list_) { if (p) cudaFree(p); p = nullptr; }
        cap_list_ = 0;
        for (auto &p : d_list_) CK(cudaMalloc((void **)&p, (size_t)(n + 1) * sizeof(int32_t)));  // [n] rows + the count
        cap_list_ = n + 1;
    }
    return DNALDPC_OK;
}

int Engine::failed_rows(const uint8_t *ok, const int32_t *prev_list, int n, int32_t *list_out, int32_t *count_dev, cudaStream_t stream) {
    failed_rows_kernel<<<1, 1024, 0, stream>>>(ok, prev_list, n, list_out, count_dev);
    CK(cudaGetLastError());
    return DNALDPC_OK;
}

int math_selftest(long long n, uint64_t seed, long long *mismatches, std::string &err) {
    unsigned long long *d = nullptr, h = 0;
    cudaError_t e = cudaMalloc((void **)&d, sizeof(h));
    if (e == cudaSuccess) e = cudaMemset(d, 0, sizeof(h));
    if (e == cudaSuccess && n > 0) {
        math_selftest_kernel<<<(unsigned)((n + 255) / 256), 256>>>(n, seed, d);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(&h, d, sizeof(h), cudaMemcpyDeviceToHost);
    if (d) cudaFree(d);
    if (e != cudaSuccess) { err = std::string("CUDA error: ") + cudaGetErrorString(e); return DNALDPC_ERR_CUDA; }
    *mismatches = (long long)h;
    return DNALDPC_OK;
}

}  // namespace dnaldpc
