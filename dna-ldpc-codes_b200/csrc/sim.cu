// sim.cu - Monte-Carlo error-rate simulation (dnaldpc_simulate): random codewords through a synthetic channel, decoded
// and counted on the GPU inside ONE engine session, so that the drain tail is paid once per run and not once per batch.
//
// Per engine a SimSource (a FrameSource) keeps two rings in HBM, in pieces of P frames:
//   input ring  [n_in pieces]:  channel values of the frames published and not yet admitted (a slot is free once every
//                               frame of its piece has been admitted);
//   output ring [n_out pieces]: sent codeword, decoded bits, iteration count, syndrome flag, raw bit errors and the
//                               per-frame record of every frame from generation until the host has its counts.
// Pieces are pulled from one shared counter (like HostBatch::next_chunk). For a piece, on the engine's io stream 0 and
// ahead of admission: sim_message_kernel -> Encoder::encode into the output ring -> the synth kernel of the channel
// (engine.cu, pointed at the ring rows) -> sim_raw_kernel -> Engine::publish through the copy engine. Once `low_water`
// has passed the piece: sim_count_kernel (one warp per frame: per-frame records + per-piece 64-bit counters), copied
// to pinned host memory behind an event. The host folds the pieces in GLOBAL piece order: when the known prefix holds
// T frame errors it stops handing out pieces, and the exact cut inside the crossing piece comes from its records.
#include "sim.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdlib>
#include <deque>
#include <map>
#include <mutex>
#include <thread>

#include "rng.cuh"

namespace dnaldpc {

namespace {

// Per-piece counters, in the order of dnaldpc_sim_result after `frames`.
enum { kIters, kFrameErr, kBitErr, kMsgFrameErr, kMsgBitErr, kDetected, kUndetected, kRawFrameErr, kRawBitErr, kCounters };
// Per-frame record: bit errors, message bit errors, raw bit errors, iterations, flags.
enum { kRecBits, kRecMsgBits, kRecRawBits, kRecIters, kRecFlags, kRecWords };
enum { kFlagFrameErr = 1, kFlagMsgFrameErr = 2, kFlagDetected = 4, kFlagUndetected = 8, kFlagRawFrameErr = 16 };
constexpr int kCountWarps = 8;

// Word w of frame f's message = low 32 bits of rng_u64(seed, f, w, 1), bits at and beyond K cleared.
__global__ void __launch_bounds__(256)
sim_message_kernel(uint64_t seed, long long f0, int n, int kw, int K, uint32_t *__restrict__ msg) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)n * kw) return;
    const long long fl = t / kw;
    const int w = (int)(t - fl * kw);
    uint32_t v = (uint32_t)rng_u64(seed, (uint64_t)(f0 + fl), (uint64_t)w, 1);
    const int rem = K - 32 * w;
    if (rem < 32) v &= rem <= 0 ? 0u : (1u << rem) - 1u;
    msg[t] = v;
}

// Raw ("without coding") bit errors of each frame: the channel's hard decision against the sent codeword. One warp per
// frame. KIND: DNALDPC_IN_BSC_BITS (received bit), DNALDPC_IN_AWGN_F32 (y < 0), DNALDPC_IN_VOTE_I8 (k < 0).
template <int KIND>
__global__ void __launch_bounds__(256)
sim_raw_kernel(const void *__restrict__ in, size_t stride, const uint32_t *__restrict__ cw, int wpf, int N, int n,
               int32_t *__restrict__ raw) {
    const int lane = threadIdx.x & 31;
    const int f = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (f >= n) return;
    const uint32_t *c = cw + (size_t)f * wpf;
    const char *row = (const char *)in + (size_t)f * stride;
    int e = 0;
    if (KIND == DNALDPC_IN_BSC_BITS) {
        const uint32_t *rx = (const uint32_t *)row;
        for (int w = lane; w < wpf; w += 32) e += __popc(rx[w] ^ c[w]);  // bits beyond N are 0 in both
    } else {
        for (int j = lane; j < N; j += 32) {
            const bool hard = KIND == DNALDPC_IN_AWGN_F32 ? ((const float *)row)[j] < 0.0f : ((const int8_t *)row)[j] < 0;
            e += hard != (bool)((c[j >> 5] >> (j & 31)) & 1u);
        }
    }
    e = __reduce_add_sync(0xffffffffu, e);
    if (lane == 0) raw[f] = e;
}

// One warp per frame: XOR of decoded and sent words, popcount over all bits and under the info-column mask, syndrome
// flag, iteration count and raw errors -> the frame's record; warp lane 0 values are reduced over the block in shared
// memory and added to the piece's 64-bit counters with one atomic per counter and block.
__global__ void __launch_bounds__(kCountWarps * 32)
sim_count_kernel(const uint32_t *__restrict__ sent, const uint32_t *__restrict__ dec, const uint32_t *__restrict__ info_mask,
                 int wpf, uint32_t last_mask, const int32_t *__restrict__ iters, const uint8_t *__restrict__ ok,
                 const int32_t *__restrict__ raw, int n, int32_t *__restrict__ rec, unsigned long long *__restrict__ cnt) {
    __shared__ unsigned long long part[kCountWarps][kCounters];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int f = blockIdx.x * kCountWarps + warp;
    unsigned long long v[kCounters];
#pragma unroll
    for (int k = 0; k < kCounters; k++) v[k] = 0;
    if (f < n) {
        int be = 0, mbe = 0;
        for (int w = lane; w < wpf; w += 32) {
            uint32_t x = sent[(size_t)f * wpf + w] ^ dec[(size_t)f * wpf + w];
            if (w == wpf - 1) x &= last_mask;
            be += __popc(x);
            mbe += __popc(x & info_mask[w]);
        }
        be = __reduce_add_sync(0xffffffffu, be);
        mbe = __reduce_add_sync(0xffffffffu, mbe);
        const int it = iters[f], rb = raw[f];
        const bool syn_ok = ok[f] != 0;
        const int flags = (be > 0 ? kFlagFrameErr : 0) | (mbe > 0 ? kFlagMsgFrameErr : 0) | (!syn_ok ? kFlagDetected : 0) |
                          (syn_ok && be > 0 ? kFlagUndetected : 0) | (rb > 0 ? kFlagRawFrameErr : 0);
        if (lane == 0) {
            int32_t *r = rec + (size_t)f * kRecWords;
            r[kRecBits] = be; r[kRecMsgBits] = mbe; r[kRecRawBits] = rb; r[kRecIters] = it; r[kRecFlags] = flags;
        }
        v[kIters] = (unsigned)it;
        v[kFrameErr] = be > 0; v[kBitErr] = (unsigned)be;
        v[kMsgFrameErr] = mbe > 0; v[kMsgBitErr] = (unsigned)mbe;
        v[kDetected] = !syn_ok; v[kUndetected] = syn_ok && be > 0;
        v[kRawFrameErr] = rb > 0; v[kRawBitErr] = (unsigned)rb;
    }
    if (lane == 0)
#pragma unroll
        for (int k = 0; k < kCounters; k++) part[warp][k] = v[k];
    __syncthreads();
    if (threadIdx.x < kCounters) {
        unsigned long long s = 0;
#pragma unroll
        for (int w = 0; w < kCountWarps; w++) s += part[w][threadIdx.x];
        if (s) atomicAdd(cnt + threadIdx.x, s);
    }
}

int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

void add_stats(dnaldpc_stats &a, const dnaldpc_stats &s) {
    a.frames += s.frames; a.frame_iters += s.frame_iters; a.kernel_launches += s.kernel_launches; a.waves += s.waves;
    a.row_ms += s.row_ms; a.col_ms += s.col_ms; a.compactions += s.compactions;
}

struct PieceResult {
    int64_t n = 0;
    int64_t cnt[kCounters] = {};
    std::vector<int32_t> rec;  // [n][kRecWords]
};

// What every engine of one simulation shares: the piece counter and the fold of the results in global piece order.
struct SimShared {
    int64_t F = 0, T = 0, P = 0, n_pieces = 0;
    std::atomic<int64_t> next_piece{0};
    std::atomic<bool> stop{false};
    std::mutex mu;
    std::map<int64_t, PieceResult> pending;  // results of pieces beyond the folded prefix
    int64_t folded = 0;                      // pieces [0, folded) are in `acc`
    bool crossed = false;
    int64_t frames = 0, acc[kCounters] = {};

    void add(int64_t piece, PieceResult &&r) {
        std::lock_guard<std::mutex> lk(mu);
        if (crossed) return;
        pending[piece] = std::move(r);
        for (auto it = pending.find(folded); it != pending.end() && !crossed; it = pending.find(folded)) {
            const PieceResult &p = it->second;
            if (T > 0 && acc[kFrameErr] + p.cnt[kFrameErr] >= T) {
                // the crossing piece: count its frames up to and including the T-th frame error
                for (int64_t i = 0; i < p.n; i++) {
                    const int32_t *q = &p.rec[(size_t)i * kRecWords];
                    const int fl = q[kRecFlags];
                    acc[kIters] += q[kRecIters];
                    acc[kFrameErr] += (fl & kFlagFrameErr) != 0; acc[kBitErr] += q[kRecBits];
                    acc[kMsgFrameErr] += (fl & kFlagMsgFrameErr) != 0; acc[kMsgBitErr] += q[kRecMsgBits];
                    acc[kDetected] += (fl & kFlagDetected) != 0; acc[kUndetected] += (fl & kFlagUndetected) != 0;
                    acc[kRawFrameErr] += (fl & kFlagRawFrameErr) != 0; acc[kRawBitErr] += q[kRecRawBits];
                    frames++;
                    if (acc[kFrameErr] >= T) break;
                }
                crossed = true;
                stop.store(true);
            } else {
                for (int k = 0; k < kCounters; k++) acc[k] += p.cnt[k];
                frames += p.n;
            }
            pending.erase(it);
            folded++;
        }
        if (crossed) pending.clear();
    }
};

struct InFlight {
    int64_t seq, piece, f0, q0;
    int n, session;
    bool counted;
};

class SimSource : public FrameSource {
  public:
    SimSource(Engine &e, Encoder &enc, const Systematic &sys, const dnaldpc_sim &s, SimShared &sh)
        : e_(e), enc_(enc), sys_(sys), s_(s), sh_(sh) {}
    ~SimSource() override {
        if (cudaSetDevice(e_.device()) != cudaSuccess) return;
        if (st_) cudaStreamSynchronize(st_);
        void *d[] = {d_msg_, d_in_, d_cw_, d_bits_, d_iters_, d_ok_, d_raw_, d_rec_, d_cnt_, d_mask_};
        for (void *p : d) if (p) cudaFree(p);
        if (h_rec_) cudaFreeHost(h_rec_);
        if (h_cnt_) cudaFreeHost(h_cnt_);
        for (cudaEvent_t ev : ev_) if (ev) cudaEventDestroy(ev);
    }
    const std::string &error() const { return err_; }

    int prepare(int64_t sess_cap) {
        if (!cu(cudaSetDevice(e_.device()), "cudaSetDevice")) return DNALDPC_ERR_CUDA;
        st_ = e_.io_stream(0);
        N_ = e_.N();
        wpf_ = (N_ + 31) / 32;
        P_ = sh_.P;
        packed_ = packed_stride(s_.channel, N_);
        sess_cap_ = sess_cap;
        // input ring: at least two waves of admissions and four pieces (generation stays pieces ahead of admission);
        // output ring: the frames admitted while a frame that runs to max_iter holds the low-water mark (§4), 2^17
        n_in_ = (int)std::max<int64_t>(4, (2 * (int64_t)e_.wave_frames() + P_ - 1) / P_);
        n_out_ = (int)std::max<int64_t>(n_in_ + 4, ((int64_t)1 << 17) / P_);
        const size_t in_f = (size_t)n_in_ * P_, out_f = (size_t)n_out_ * P_;
        auto dm = [&](void **p, size_t bytes) { return cu(cudaMalloc(p, std::max<size_t>(bytes, 4)), "cudaMalloc(simulation rings)"); };
        if (!dm((void **)&d_msg_, (size_t)P_ * std::max(sys_.kw, 1) * 4) || !dm((void **)&d_in_, in_f * packed_) ||
            !dm((void **)&d_cw_, out_f * wpf_ * 4) || !dm((void **)&d_bits_, out_f * wpf_ * 4) || !dm((void **)&d_iters_, out_f * 4) ||
            !dm((void **)&d_ok_, out_f) || !dm((void **)&d_raw_, out_f * 4) || !dm((void **)&d_rec_, out_f * kRecWords * 4) ||
            !dm((void **)&d_cnt_, (size_t)n_out_ * kCounters * 8) || !dm((void **)&d_mask_, (size_t)wpf_ * 4))
            return DNALDPC_ERR_NOMEM;
        if (!cu(cudaMallocHost((void **)&h_rec_, out_f * kRecWords * 4), "cudaMallocHost(simulation records)") ||
            !cu(cudaMallocHost((void **)&h_cnt_, (size_t)n_out_ * kCounters * 8), "cudaMallocHost(simulation counters)"))
            return DNALDPC_ERR_NOMEM;
        ev_.assign((size_t)n_out_, nullptr);
        for (auto &ev : ev_) if (!cu(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming), "cudaEventCreate")) return DNALDPC_ERR_CUDA;
        std::vector<uint32_t> mask((size_t)wpf_, 0u);
        for (int32_t j : sys_.info_cols) mask[(size_t)j / 32] |= 1u << (j % 32);
        if (!cu(cudaMemcpy(d_mask_, mask.data(), mask.size() * 4, cudaMemcpyHostToDevice), "cudaMemcpy(info mask)")) return DNALDPC_ERR_CUDA;
        in_end_.assign((size_t)n_in_, -1);
        return DNALDPC_OK;
    }

    // A new engine session: the queue restarts at q = 0.
    void begin_session(Session &ss) {
        session_++;
        sess_pub_ = 0;
        sess_final_ = false;
        waited_ready_ = false;
        std::fill(in_end_.begin(), in_end_.end(), -1);
        ss.in = dnaldpc_input{};
        ss.in.kind = s_.channel;
        ss.in.flags = s_.flags;
        ss.in.data = d_in_;
        ss.in.frame_stride = packed_;
        ss.in.param = s_.param;
        ss.out = dnaldpc_output{};
        ss.out.bits = d_bits_;
        ss.out.iters = d_iters_;
        ss.out.is_codeword = d_ok_;
        ss.max_iter = s_.max_iter;
        ss.max_frames = sess_cap_;
    }
    bool exhausted() const { return exhausted_; }

    int pump(Engine &e, int64_t admitted, int64_t low_water, bool *final) override {
        if (!collect(false)) return DNALDPC_ERR_CUDA;
        for (InFlight &p : fly_) {  // count the pieces the engine has harvested completely
            if (p.counted || p.session != session_) continue;
            if (p.q0 + p.n > low_water) break;
            if (!count(p)) return DNALDPC_ERR_CUDA;
        }
        while (!sess_final_) {
            if (sh_.stop.load() || exhausted_) { sess_final_ = true; break; }
            // every piece handed out: say so before a full queue does, so that no empty session follows
            if (sh_.next_piece.load() >= sh_.n_pieces) { exhausted_ = true; sess_final_ = true; break; }
            if (sess_pub_ + P_ > sess_cap_) { sess_final_ = true; break; }  // this session's queue is full
            const int in_slot = (int)(seq_ % n_in_);
            if (in_end_[(size_t)in_slot] > admitted) break;                 // its previous piece is not admitted yet
            if (seq_ - consumed_ >= n_out_) break;                          // output ring full until counts come back
            const int64_t c = sh_.next_piece.fetch_add(1);
            if (c >= sh_.n_pieces) { exhausted_ = true; sess_final_ = true; break; }
            const int rc = generate(e, c, in_slot);
            if (rc) return rc;
        }
        *final = sess_final_;
        return DNALDPC_OK;
    }

    void wait_for_frames() override {  // idle engine, source not final: the output ring waits for counts
        for (InFlight &p : fly_)
            if (p.counted) { cudaEventSynchronize(ev_[(size_t)(p.seq % n_out_)]); return; }
        std::this_thread::sleep_for(std::chrono::microseconds(200));
    }

    // After the last session: every piece is counted (the engine's final pump saw low_water = everything); wait for
    // the results.
    int finish() {
        if (!collect(true)) return DNALDPC_ERR_CUDA;
        if (!fly_.empty()) { err_ = "simulation pieces left uncounted"; return DNALDPC_ERR_CUDA; }
        return DNALDPC_OK;
    }
    int64_t launches = 0;

  private:
    bool cu(cudaError_t e, const char *what) {
        if (e == cudaSuccess) return true;
        if (err_.empty()) err_ = std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what;
        return false;
    }

    int generate(Engine &e, int64_t c, int in_slot) {
        const int64_t f0 = c * P_;
        const int n = (int)std::min<int64_t>(P_, sh_.F - f0);
        const int out_slot = (int)(seq_ % n_out_);
        const int K = sys_.K, kw = sys_.kw;
        if (!waited_ready_) {  // the engine's queue of this session is reset in stream order at ready_event
            if (!cu(cudaStreamWaitEvent(st_, e.ready_event(), 0), "cudaStreamWaitEvent")) return DNALDPC_ERR_CUDA;
            waited_ready_ = true;
        }
        uint32_t *cw = d_cw_ + (size_t)out_slot * P_ * wpf_;
        char *in = (char *)d_in_ + (size_t)in_slot * P_ * packed_;
        int32_t *raw = d_raw_ + (size_t)out_slot * P_;
        if (kw > 0) {
            sim_message_kernel<<<(unsigned)(((int64_t)n * kw + 255) / 256), 256, 0, st_>>>(s_.seed, (long long)f0, n, kw, K, d_msg_);
            if (!cu(cudaGetLastError(), "sim_message_kernel")) return DNALDPC_ERR_CUDA;
        }
        int rc = enc_.encode(d_msg_, n, cw, st_);
        if (rc) { err_ = enc_.error(); return rc; }
        // frame f0 + i is noise on ring row i: (f0 + i + cw_off) % n == i
        const uint64_t cw_off = (uint64_t)((n - f0 % n) % n);
        const unsigned raw_grid = (unsigned)((n + 7) / 8);
        switch (s_.channel) {
            case DNALDPC_IN_BSC_BITS:
                rc = e.synth_bsc(cw, n, s_.seed, f0, n, s_.param, (uint32_t *)in, st_, cw_off);
                if (!rc) sim_raw_kernel<DNALDPC_IN_BSC_BITS><<<raw_grid, 256, 0, st_>>>(in, packed_, cw, wpf_, N_, n, raw);
                break;
            case DNALDPC_IN_AWGN_F32:
                rc = e.synth_awgn(cw, n, s_.seed, f0, n, s_.param, (float *)in, st_, cw_off);
                if (!rc) sim_raw_kernel<DNALDPC_IN_AWGN_F32><<<raw_grid, 256, 0, st_>>>(in, packed_, cw, wpf_, N_, n, raw);
                break;
            default:
                rc = e.synth_vote(cw, n, s_.seed, f0, n, s_.mean_reads, s_.param, (int8_t *)in, st_, cw_off);
                if (!rc) sim_raw_kernel<DNALDPC_IN_VOTE_I8><<<raw_grid, 256, 0, st_>>>(in, packed_, cw, wpf_, N_, n, raw);
                break;
        }
        if (rc) { err_ = e.error(); return rc; }
        if (!cu(cudaGetLastError(), "sim_raw_kernel")) return DNALDPC_ERR_CUDA;
        // copy-engine publish: nothing queued behind the generation kernels waits for an SM slot (DESIGN §4)
        rc = e.publish(nullptr, in_slot * (int)P_, out_slot * (int)P_, n, st_, true);
        if (rc) { err_ = rc == DNALDPC_ERR_CUDA ? "CUDA error while publishing simulated frames" : "frame queue overflow"; return rc; }
        launches += (kw > 0) + 4;
        fly_.push_back(InFlight{seq_, c, f0, sess_pub_, n, session_, false});
        in_end_[(size_t)in_slot] = sess_pub_ + n;
        sess_pub_ += n;
        seq_++;
        return DNALDPC_OK;
    }

    bool count(InFlight &p) {
        const int slot = (int)(p.seq % n_out_);
        const size_t r0 = (size_t)slot * P_;
        unsigned long long *cnt = d_cnt_ + (size_t)slot * kCounters;
        if (!cu(cudaMemsetAsync(cnt, 0, kCounters * 8, st_), "cudaMemsetAsync")) return false;
        const uint32_t last_mask = N_ % 32 ? (1u << (N_ % 32)) - 1u : 0xffffffffu;
        sim_count_kernel<<<(unsigned)((p.n + kCountWarps - 1) / kCountWarps), kCountWarps * 32, 0, st_>>>(
            d_cw_ + r0 * wpf_, d_bits_ + r0 * wpf_, d_mask_, wpf_, last_mask, d_iters_ + r0, d_ok_ + r0, d_raw_ + r0, p.n,
            d_rec_ + r0 * kRecWords, cnt);
        if (!cu(cudaGetLastError(), "sim_count_kernel")) return false;
        if (!cu(cudaMemcpyAsync(h_cnt_ + (size_t)slot * kCounters, cnt, kCounters * 8, cudaMemcpyDeviceToHost, st_), "cudaMemcpyAsync(D2H)") ||
            !cu(cudaMemcpyAsync(h_rec_ + r0 * kRecWords, d_rec_ + r0 * kRecWords, (size_t)p.n * kRecWords * 4, cudaMemcpyDeviceToHost, st_), "cudaMemcpyAsync(D2H)") ||
            !cu(cudaEventRecord(ev_[(size_t)slot], st_), "cudaEventRecord"))
            return false;
        launches++;
        p.counted = true;
        return true;
    }

    // Hands the results of counted pieces to the shared fold, in this engine's piece order; `all`: wait for them.
    bool collect(bool all) {
        while (!fly_.empty() && fly_.front().counted) {
            const InFlight &p = fly_.front();
            const int slot = (int)(p.seq % n_out_);
            cudaEvent_t ev = ev_[(size_t)slot];
            if (all) { if (!cu(cudaEventSynchronize(ev), "cudaEventSynchronize")) return false; }
            else {
                const cudaError_t q = cudaEventQuery(ev);
                if (q == cudaErrorNotReady) break;
                if (!cu(q, "cudaEventQuery")) return false;
            }
            PieceResult r;
            r.n = p.n;
            std::copy(h_cnt_ + (size_t)slot * kCounters, h_cnt_ + (size_t)(slot + 1) * kCounters, r.cnt);
            const int32_t *rec = h_rec_ + (size_t)slot * P_ * kRecWords;
            r.rec.assign(rec, rec + (size_t)p.n * kRecWords);
            sh_.add(p.piece, std::move(r));
            fly_.pop_front();
            consumed_++;
        }
        return true;
    }

    Engine &e_;
    Encoder &enc_;
    const Systematic &sys_;
    const dnaldpc_sim &s_;
    SimShared &sh_;
    std::string err_;
    cudaStream_t st_ = nullptr;
    int N_ = 0, wpf_ = 0, n_in_ = 0, n_out_ = 0, session_ = 0;
    int64_t P_ = 0, sess_cap_ = 0, sess_pub_ = 0, seq_ = 0, consumed_ = 0;
    size_t packed_ = 0;
    bool sess_final_ = false, exhausted_ = false, waited_ready_ = false;
    std::vector<int64_t> in_end_;  // per input slot: session queue position after its piece (-1 = free)
    std::deque<InFlight> fly_;     // published pieces, in order, until their results reach the fold
    uint32_t *d_msg_ = nullptr, *d_cw_ = nullptr, *d_bits_ = nullptr, *d_mask_ = nullptr;
    void *d_in_ = nullptr;
    int32_t *d_iters_ = nullptr, *d_raw_ = nullptr, *d_rec_ = nullptr, *h_rec_ = nullptr;
    uint8_t *d_ok_ = nullptr;
    unsigned long long *d_cnt_ = nullptr, *h_cnt_ = nullptr;
    std::vector<cudaEvent_t> ev_;  // per output slot: its counts have reached the host
};

}  // namespace

int simulate_batch(EngineSet &eng, const std::vector<Encoder *> &encoders, const Systematic &sys, const dnaldpc_sim &s,
                   dnaldpc_sim_result &r, dnaldpc_stats &st, std::string &err) {
    st = dnaldpc_stats{};
    r = dnaldpc_sim_result{};
    SimShared sh;
    sh.F = s.max_frames;
    sh.T = s.target_frame_errors;
    int64_t P = eng[0]->wave_frames();  // a piece: about one wave of admissions
    if (const char *t = getenv("DNALDPC_SIM_PIECE")) P = std::max<int64_t>(1, atoll(t));  // test switch
    P = std::min<int64_t>(P, s.max_frames);
    sh.P = P;
    sh.n_pieces = (s.max_frames + P - 1) / P;
    const int nd = (int)std::min<int64_t>((int64_t)eng.size(), sh.n_pieces);
    // one engine session holds at most ~4 M frames (its frame queue is linear): longer runs pay one drain tail per session
    const int64_t sess_cap = std::min(round_up(s.max_frames, P), std::max<int64_t>(1, ((int64_t)1 << 22) / P) * P);
    std::vector<std::unique_ptr<SimSource>> src;
    for (int k = 0; k < nd; k++) src.emplace_back(new SimSource(*eng[(size_t)k], *encoders[(size_t)k], sys, s, sh));
    std::vector<std::string> errs((size_t)nd);
    std::vector<dnaldpc_stats> est((size_t)nd);
    std::vector<int> rcs((size_t)nd, DNALDPC_OK);
    auto run = [&](int k) {
        Engine &e = *eng[(size_t)k];
        SimSource &so = *src[(size_t)k];
        int rc = so.prepare(sess_cap);
        while (!rc) {
            Session ss;
            so.begin_session(ss);
            rc = e.run_session(ss, so, nullptr);
            if (rc) { errs[(size_t)k] = so.error().empty() ? e.error() : so.error(); break; }
            add_stats(est[(size_t)k], e.stats);
            if (so.exhausted() || sh.stop.load()) break;
        }
        if (!rc) rc = so.finish();
        if (rc) {
            sh.stop.store(true);  // the other engines wind down
            if (errs[(size_t)k].empty()) errs[(size_t)k] = so.error().empty() ? e.error() : so.error();
        }
        est[(size_t)k].kernel_launches += so.launches;
        rcs[(size_t)k] = rc;
    };
    std::vector<std::thread> th;
    for (int k = 1; k < nd; k++) th.emplace_back(run, k);
    run(0);
    for (auto &t : th) t.join();
    for (int k = 0; k < nd; k++) add_stats(st, est[(size_t)k]);
    for (int k = 0; k < nd; k++)
        if (rcs[(size_t)k]) { err = errs[(size_t)k]; return rcs[(size_t)k]; }
    if (!sh.crossed && sh.folded != sh.n_pieces) { err = "simulation ended with pieces missing from the count"; return DNALDPC_ERR_CUDA; }
    r.frames = sh.frames;
    r.iterations = sh.acc[kIters];
    r.frame_errors = sh.acc[kFrameErr]; r.bit_errors = sh.acc[kBitErr];
    r.msg_frame_errors = sh.acc[kMsgFrameErr]; r.msg_bit_errors = sh.acc[kMsgBitErr];
    r.detected = sh.acc[kDetected]; r.undetected = sh.acc[kUndetected];
    r.raw_frame_errors = sh.acc[kRawFrameErr]; r.raw_bit_errors = sh.acc[kRawBitErr];
    return DNALDPC_OK;
}

}  // namespace dnaldpc
