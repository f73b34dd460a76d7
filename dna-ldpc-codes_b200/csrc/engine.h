// engine.h - per-device decoder engine: owns the device copies of the H edge tables, the slot-interleaved message
// arrays and the host side of the slot scheduler (admit -> syndrome/loop control -> check pass -> bit pass per tick;
// early exit on zero syndrome / max_iter per frame, dec.cpp:594-599). Internal C++ interface behind include/dnaldpc.h.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/dnaldpc.h"
#include "../host/code.h"

namespace dnaldpc {

struct SchedArrays;
class Engine;

// One batch as an engine sees it: buffers the DEVICE can address (its own memory, the staging rings of a host batch, or
// a peer GPU's memory) indexed by the rows the frame queue carries, plus an upper bound of the frames it may receive.
struct Session {
    dnaldpc_input in;    // kind / flags / param / table; data + frame_stride address input row r
    dnaldpc_output out;  // output arrays addressed by output row
    int max_iter = 0;
    int64_t max_frames = 0;  // most frames this engine can be handed in this batch (sizes the slot groups and row tables)
};

// Where an engine's frames come from. pump() runs on the engine's tick thread once per tick: it may publish frames
// (Engine::publish) and retire outputs, and says when nothing more will come.
class FrameSource {
  public:
    virtual ~FrameSource() {}
    // Every queue position q < admitted has been set up in a slot (its input row may be overwritten); every q < low_water
    // has been harvested (its outputs are complete in device memory). Both are what the host knows, a few ticks old.
    // Sets *final once every frame of the batch has been published.
    virtual int pump(Engine &e, int64_t admitted, int64_t low_water, bool *final) = 0;
    // The engine is idle and the source not final: block until pump() can make progress (bounded wait).
    virtual void wait_for_frames() {}
};

class Engine {
  public:
    Engine(const Code &code, int device, int precision, int wave_frames);
    ~Engine();
    bool ok() const { return err_.empty(); }
    const std::string &error() const { return err_; }
    int device() const { return device_; }

    // Decodes every frame `src` publishes; kernels run on `stream` (NULL = the engine's own stream). Returns when the
    // queue has drained (all outputs written to device-visible memory, stream not necessarily idle).
    int run_session(const Session &ss, FrameSource &src, cudaStream_t stream);
    // Appends n frames to the queue: input rows list_in[0..n) (a DEVICE array) or row0_in.. when list_in == NULL,
    // output rows row0_out... Ordered on `stream` (the stream that made the frames' inputs resident). One producer at
    // a time.
    // dma: write the queue entries with copy-engine transfers instead of a kernel (for producers on a copy stream).
    int publish(const int32_t *list_in, int row0_in, int row0_out, int n, cudaStream_t stream, bool dma = false);
    // list_out[0..*count) = prev_list[k] (k itself when prev_list == NULL) for every k < n with ok[k] == 0, in ascending
    // k (the frames a re-decoding round takes, decoder.py:641-660). DEVICE arrays; *count_dev is a device int.
    int failed_rows(const uint8_t *ok, const int32_t *prev_list, int n, int32_t *list_out, int32_t *count_dev, cudaStream_t stream);
    int64_t published() const { return published_.load(std::memory_order_acquire); }
    cudaStream_t own_stream() const { return own_stream_; }
    cudaStream_t io_stream(int k) const { return io_stream_[k]; }  // 0: host -> device copies, 1: device -> host copies
    int wave_frames() const { return wave_frames_; }
    cudaEvent_t ready_event() const { return ready_ev_; }  // producers on other streams wait for it before publishing
    // Sliding-window BP for spatially-coupled codes (Run_SW_Decoder, dec.cpp:2092-2196); HOST pointers; blocking.
    int decode_window_host(const Code &code, const dnaldpc_window &w, const double *lratio, int64_t F, int max_iter,
                           const dnaldpc_output &out);
    // Synthetic channel outputs of frames [frame0, frame0+F) (include/dnaldpc.h); frame f is noise on codeword row
    // (f + cw_off) % n_cw (the C ABI passes 0; the simulator points the generators at rows of its codeword ring).
    int synth_bsc(const uint32_t *cw_bits, int n_cw, uint64_t seed, int64_t frame0, int64_t F, double eps,
                  uint32_t *out_bits, cudaStream_t stream, uint64_t cw_off = 0);
    int synth_awgn(const uint32_t *cw_bits, int n_cw, uint64_t seed, int64_t frame0, int64_t F, double sigma,
                   float *out_y, cudaStream_t stream, uint64_t cw_off = 0);
    int synth_vote(const uint32_t *cw_bits, int n_cw, uint64_t seed, int64_t frame0, int64_t F, double mean_reads,
                   double read_err, int8_t *out_k, cudaStream_t stream, uint64_t cw_off = 0);

    dnaldpc_stats stats{};
    bool profiling = false;
    int trace_ticks_ = 0;  // > 0: record in-pipeline events for that many ticks of the next batch (no synchronisation)
    int trace_result(double *row_ms, double *col_ms, double *sched_ms);

  private:
    template <typename T> int run(const Session &ss, FrameSource &src, cudaStream_t st);
    int sw_groups(const Code &code, const dnaldpc_window &w, const std::vector<int> &sched, const double *lratio, int64_t F,
                  int max_iter, const dnaldpc_output &out, int G);
    int sw_lockstep(const dnaldpc_window &w, const std::vector<int> &sched, const double *lratio, int64_t F, int max_iter,
                    const dnaldpc_output &out, int G);
    int ensure_rows(int64_t frames);
    template <typename T> int launch_row(int g0, int G, cudaStream_t st);
    template <typename T> int launch_col(int g0, int G, bool want_post, cudaStream_t st);
    template <typename T> int launch_harvest_setup(const dnaldpc_input &in, const dnaldpc_output &out, int g0, int G, cudaStream_t st);
    int launch_syndrome(const dnaldpc_output &out, int G, int max_iter, int consider_new, int fixed, unsigned *counter,
                        unsigned *finished, unsigned *rearm, int clear_fresh, cudaStream_t st);
    int ensure_slots(int groups, bool want_post);
    int ensure_frame_scratch(int64_t F);
    int fail(cudaError_t e, const char *what);
    int fail(const std::string &m, int rc);
    void fill_sched(SchedArrays &s) const;

    std::string err_;
    int device_ = 0, precision_ = 0, wave_frames_ = 4096, sm_count_ = 148;
    int M_ = 0, N_ = 0, E_ = 0, max_row_deg_ = 0, max_col_deg_ = 0;
    bool reg_rows_ = false, reg_cols_ = false;
    bool smem_attr_set_[2] = {false, false}, syn_attr_set_ = false, tmem_attr_set_ = false, syn_half_attr_set_ = false;
    bool steady_ = false;  // last polled tick: all slots busy, no frame admitted
    bool minsum_ = false;  // current batch runs the LLR-domain min-sum rules instead of sum-product
    size_t esz_ = 8;
    // H edge tables (device)
    int32_t *d_row_ptr_ = nullptr, *d_col_idx_ = nullptr, *d_col_ptr_ = nullptr, *d_col_edge_ = nullptr;
    // slot state (device)
    int cap_groups_ = 0;
    void *d_msg_ = nullptr, *d_lratio_ = nullptr, *d_post_ = nullptr;
    uint32_t *d_decw_ = nullptr, *d_masks_ = nullptr;  // masks: 6 words per group (act, done, newf, fresh, harv, unsat)
    unsigned int *d_arrive_ = nullptr;
    int32_t *d_slot_ = nullptr;                          // 4 ints per slot (frame, iter, harv_frame, harv_iter)
    void *d_sw_lr_ = nullptr;                            // sliding-window mode: second message array (check -> bit)
    int sw_cap_groups_ = 0;
    int sw_slots_ = 0;                                   // sliding-window mode: slots in flight (decided at the first call)
    int32_t *d_edge_row_ = nullptr;                      // sliding-window mode: check of every edge
    int32_t *d_col_row_ = nullptr;                       // sliding-window mode: check of the k-th entry of a column
    int32_t *d_sw_sched_ = nullptr;                      // sliding-window mode: window ranges per position [L][8]
    int sw_cap_sched_ = 0;
    unsigned long long *d_sw_avail_ = nullptr;           // sliding-window mode: frames resident per input buffer [2]
    int32_t *d_sw_lists_ = nullptr;                      // sliding-window mode: per-tick work lists [4][G] + 4 counts, straggler tables [3][G]
    int sw_cap_lists_ = 0;
    void *d_sw_thin_ = nullptr;                          // sliding-window mode: straggler side arrays [2][G][edges][4]
    size_t sw_cap_thin_ = 0;
    unsigned long long *d_sw_hist_ = nullptr;            // sliding-window mode: diagnostics (DNALDPC_SW_HIST)
    cudaEvent_t sw_in_ev_[2] = {nullptr, nullptr};       // sliding-window mode: a chunk's inputs have arrived
    int32_t *d_mv_ = nullptr;                            // drain-tail compaction: src[S], dst[S], {count, K}
    // compact when busy slots <= 15/16 of the packed region: a move is cheap next to the ticks it shortens (measured
    // thresholds 30 / 50 / 70 / 85 / 92 / 97 %: 16 384 frames eps 0.008 1196 / 1110 / 1084 / 1037 / 1016 / 992 ms per batch)
    static constexpr int kCompactNum = 15, kCompactDen = 16;
    // largest dynamic shared-memory size the smem-staged syndrome kernel is ever launched with (N * 4 bytes <= gate)
    static constexpr int kSynSmemGate = 96 * 1024;
    static constexpr int kSynHalfGate = 200 * 1024;  // same for the half-word variant (N * 2 bytes, one CTA per SM)
    unsigned long long *d_next_ = nullptr;               // {next_frame, avail, iter_sum}
    int32_t *d_rows_ = nullptr;                          // frame queue: in_row[cap_rows_], out_row[cap_rows_]
    int64_t cap_rows_ = 0;
    int32_t *h_rows_ = nullptr;                          // pinned mirror of d_rows_ (publish through the copy engine)
    unsigned long long *h_avail_ = nullptr;              // pinned: value of `avail` after the piece that ends at position q
    std::atomic<int64_t> published_{0};                  // frames handed to publish() in this session (host view)
    uint64_t *d_synth_thr_ = nullptr;                    // Poisson thresholds of the vote-count generator
    int32_t *d_iters_ = nullptr;                         // per-frame scratch when the caller does not want them
    uint8_t *d_ok_ = nullptr;
    int64_t cap_frames_ = 0;
    double *d_table_ = nullptr;                          // 256 doubles (BSC uses the first 2)
    // progress counters: a ring, polled kLag ticks behind the device
    static constexpr int kLag = 2, kRing = 16;
    unsigned int *d_counters_ = nullptr, *h_counters_ = nullptr;
    cudaEvent_t ev_[kRing] = {};
    cudaEvent_t ready_ev_ = nullptr;                     // recorded once a session's queue has been reset
    cudaEvent_t prof_ev_[3] = {};
    static constexpr int kTrace = 64;
    cudaEvent_t trace_ev_[3 * kTrace] = {};
    int traced_ = 0;
    cudaStream_t own_stream_ = nullptr, io_stream_[2] = {nullptr, nullptr};

  public:
    // device staging of the host-pointer paths (owned here so that it is reused across calls; managed by the sources)
    void *stage(void **buf, size_t *cap, size_t need);
    void *s_in2_ = nullptr;  // sliding-window mode: second input buffer (the next chunk's copy overlaps the decoding)
    size_t c_in2_ = 0;
    void *s_in_ = nullptr, *s_bits_ = nullptr, *s_dblk_ = nullptr, *s_post_ = nullptr, *s_pchk_ = nullptr, *s_iters_ = nullptr, *s_ok_ = nullptr;
    size_t c_in_ = 0, c_bits_ = 0, c_dblk_ = 0, c_post_ = 0, c_pchk_ = 0, c_iters_ = 0, c_ok_ = 0;
    void *h_bounce_ = nullptr;   // pinned host memory (host-side exp of LLR batches, small result read-backs)
    size_t c_bounce_ = 0;
    void *pinned(size_t need);
    int32_t *d_list_[2] = {nullptr, nullptr};  // re-decoding rounds: rows of the frames to decode (ping-pong) + a count
    int64_t cap_list_ = 0;
    int ensure_lists(int64_t n);
    int N() const { return N_; }
    int M() const { return M_; }
    int set_device();
    int fail_msg(const std::string &m, int rc) { return fail(m, rc); }
};

int math_selftest(long long n, uint64_t seed, long long *mismatches, std::string &err);

}  // namespace dnaldpc
