/* dnaldpc.h - C ABI of the B200-native LDPC belief-propagation decoder (libdnaldpc.so).
 *
 * Drop-in boundary for the `decode` hot path of sjpark0905/DNA-LDPC-codes. The reference has no
 * library/FFI boundary (one statically linked exe, global state); each entry point below cites the
 * reference interface it replaces (paths relative to LDPC_dec/ldpc/ of the reference).
 *
 * Conventions: plain pointers and sizes, no C++ / torch types; every function returns a DNALDPC_* code
 * (never calls exit(), unlike alloc.cpp:36-40 / rcode.cpp:62-80); handles are thread-compatible (one
 * thread per handle at a time); `stream` arguments are `cudaStream_t` passed as void* (NULL = default stream).
 *
 * Semantics that are part of the contract (SURVEY.md A.1, dec.cpp:583-694):
 *   lratio[j] = p0/p1; bit = 1 when the ratio is < 1 at init and <= 1 after an iteration;
 *   loop: c = weight(H*dblk); stop when n == max_iter or c == 0; else one flooding iteration; n++;
 *   fp64 mode: IEEE binary64, round-to-nearest, no FMA contraction, multiplication order = ascending
 *   column within a check and ascending row within a bit  => decoded bits / iteration counts identical
 *   to the reference, posteriors equal to the last ulp.
 */
#ifndef DNALDPC_H
#define DNALDPC_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DNALDPC_OK 0
#define DNALDPC_ERR_ARG 1      /* bad argument */
#define DNALDPC_ERR_IO 2       /* can't open file            (rcode.cpp:60-64 "Can't open parity check file") */
#define DNALDPC_ERR_FORMAT 3   /* not a .pchk / garbled body (rcode.cpp:66-78) */
#define DNALDPC_ERR_CUDA 4     /* CUDA runtime error; see dnaldpc_last_error() */
#define DNALDPC_ERR_NOMEM 5
#define DNALDPC_ERR_UNSUPPORTED 6 /* e.g. row degree > 128 or column degree > 16 */

typedef struct dnaldpc_code dnaldpc_code;       /* host-side parity-check matrix: replaces `mod2sparse *H` + globals M,N (rcode.cpp:33-38) */
typedef struct dnaldpc_decoder dnaldpc_decoder; /* device-side decoder bound to one code and one or more GPUs */

const char *dnaldpc_last_error(void);  /* thread-local message of the last failing call */
const char *dnaldpc_version(void);

/* ---- parity-check matrix --------------------------------------------------------------------- */

/* read_pchk (rcode.cpp:54-86) -> mod2sparse_read (mod2sparse.cpp:381-427) -> intio_read (intio.cpp:35-52).
 * Rows/columns end up sorted and duplicates merged exactly like mod2sparse_insert (mod2sparse.cpp:502-604). */
int dnaldpc_code_read_pchk(const char *path, dnaldpc_code **out);
/* Same from an in-memory CSR (may be unsorted, may hold duplicates). */
int dnaldpc_code_from_csr(int M, int N, int E, const int32_t *row_ptr, const int32_t *col_idx, dnaldpc_code **out);
/* mod2sparse_write (mod2sparse.cpp:338-376) preceded by the magic word intio_write(('P'<<8)+0x80). */
int dnaldpc_code_write_pchk(const dnaldpc_code *c, const char *path);
void dnaldpc_code_free(dnaldpc_code *c);
/* mod2sparse_rows / mod2sparse_cols (mod2sparse.h:117-118) and the number of entries. */
int dnaldpc_code_dims(const dnaldpc_code *c, int *M, int *N, int *E);
/* CSR (row_ptr[M+1], col_idx[E]; ascending column in each row) and CSC (col_ptr[N+1], col_edge[E]: CSR edge ids
 * of each column in ascending row) = the traversal orders of mod2sparse_first/next_in_row/_col (mod2sparse.h:102-112). */
int dnaldpc_code_export(const dnaldpc_code *c, int32_t *row_ptr, int32_t *col_idx, int32_t *col_ptr, int32_t *col_edge);
/* CheckRegular (dec.cpp:138-189): max degrees D_v, D_c and the two regularity flags. */
int dnaldpc_code_check_regular(const dnaldpc_code *c, int *dv, int *regular_dv, int *dc, int *regular_dc);

/* ---- decoder --------------------------------------------------------------------------------- */

#define DNALDPC_PREC_F64 0 /* bit-exact mode */
#define DNALDPC_PREC_F32 1 /* optional fast mode, statistical (FER) parity only */

typedef struct dnaldpc_config {
    int32_t n_devices;      /* 0 = current device only */
    int32_t devices[16];    /* CUDA ordinals; the frames of a batch are pulled by them in chunks from one shared counter */
    int32_t precision;      /* DNALDPC_PREC_* */
    int32_t wave_frames;    /* frames resident per device at once (rounded up to 32); 0 = default (4096) */
    int32_t flags;          /* reserved, 0 */
} dnaldpc_config;

int dnaldpc_decoder_create(const dnaldpc_code *c, const dnaldpc_config *cfg, dnaldpc_decoder **out);
void dnaldpc_decoder_destroy(dnaldpc_decoder *d);

/* Input kinds = the reference's "channel options" (likelihood setup; SURVEY.md §8a):                      */
#define DNALDPC_IN_LR_F64 0   /* double [F][N]  lratio = p0/p1                  (g_received_LR, DNA_main.cpp:1344)          */
#define DNALDPC_IN_LLR_F64 1  /* double [F][N]  LLR = ln(p0/p1), LR = exp(LLR)  (LDPC_Encode, DNA_main.cpp:1340-1345)       */
#define DNALDPC_IN_BSC_BITS 2 /* uint32 [F][ceil(N/32)] received hard bits, LSB first; param = p
                                 LR = (1-p)/p for a received 0, p/(1-p) for a received 1  (channel_BSC, channel.cpp:75-84)   */
#define DNALDPC_IN_AWGN_F32 3 /* float  [F][N]  received y (BPSK 0->+1, 1->-1); param = sigma
                                 LLR = 2y/sigma^2, LR = exp(LLR)                          (channel_AWGN, channel.cpp:32-33)   */
#define DNALDPC_IN_AWGN_F64 4 /* double [F][N]  same */
#define DNALDPC_IN_VOTE_I8 5  /* int8   [F][N]  k = count0 - count1 of aligned reads; param = eps
                                 LLR = k*ln((1-eps)/eps)                                  (ex_decoder/decoder.py:292-316)     */

/* exp() is outside the bit-exact boundary (device exp != glibc exp != MSVC exp in the last ulp). With this flag a
 * HOST-pointer batch of kind LLR_F64 is exponentiated on the host with libm, like the reference does. */
#define DNALDPC_FLAG_HOST_EXP 1
/* Fixed-iteration BP = Run_Belief_Propagation_Decoder_SAVE (dec.cpp:192-223): no early exit, every frame runs exactly
 * max_iter iterations; is_codeword reports the syndrome of the final decision. */
#define DNALDPC_FLAG_FIXED_ITERS 2
/* Floating-point min-sum instead of sum-product = Run_MSA_Decoder_INF (dec.cpp:1216-1250; decoder types 20-22 of the
 * reference CLI, DNA_main.cpp:1588-1594). LLR domain: `posterior` receives L = LLR + sum of check messages
 * (Decision_MSA_INF, dec.cpp:1659-1677); a user table for VOTE_I8 must hold LLRs. LR_F64 inputs are converted with the
 * device log() and AWGN / LLR / BSC / vote-count inputs are exact. */
#define DNALDPC_FLAG_MINSUM 4

typedef struct dnaldpc_input {
    int32_t kind;        /* DNALDPC_IN_* */
    int32_t flags;       /* DNALDPC_FLAG_* */
    const void *data;    /* frame-major, frame f at data + f*frame_stride bytes */
    size_t frame_stride; /* 0 = tightly packed for the kind */
    double param;        /* p | sigma | eps, per kind; LLR kinds: scale s, LR = exp(s*LLR) (0 = 1.0) */
    const double *table; /* VOTE_I8 only: optional LR table[256] indexed by (k+128), HOST or DEVICE memory; NULL = exp(k*L) by libm */
} dnaldpc_input;

typedef struct dnaldpc_output { /* any pointer may be NULL */
    uint32_t *bits;       /* [F][ceil(N/32)] decoded bits, LSB first                                                   */
    uint8_t *dblk;        /* [F][N] decoded bits as 0/1 chars          (`char *dblk`, dec.cpp:587)                     */
    int32_t *iters;       /* [F] iterations performed, 0..max_iter     (return value of Run_Belief_Propagation_Decoder) */
    uint8_t *is_codeword; /* [F] 1 when the final syndrome is zero     (`*bIsCodeword`, dec.cpp:601)                   */
    double *posterior;    /* [F][N] posterior likelihood ratio p0/p1 of the last bit-node update (dec.cpp:669-677;
                             lratio itself when no iteration ran); P(bit=1) = 1/(1+posterior)                          */
    uint8_t *pchk;        /* [F][M] syndrome of the final decision     (`char *pchk`, check.cpp:28-47)                 */
} dnaldpc_output;

/* Batched replacement of LDPC_Decode -> Run_Belief_Propagation_Decoder (DNA_main.cpp:1572-1575, dec.cpp:583-605)
 * for F independent frames; `max_iter` replaces the global of dec.h:25. HOST buffers (pinned or pageable); blocking.
 * The batch is cut into chunks that the decoder's devices pull from one shared counter (no collective: frames are
 * independent; the reference's intended split is frames over ranks, DNA_main.cpp:629-651); per device the chunks are
 * copied in, decoded and copied back concurrently (staging rings in HBM), results land by frame index. */
int dnaldpc_decode_batch(dnaldpc_decoder *d, const dnaldpc_input *in, int64_t F, int max_iter, const dnaldpc_output *out);

/* Same with DEVICE buffers resident on ONE GPU (intended for callers that keep data in HBM). The decoder's first device
 * works on `stream`; its other devices read the inputs and write the outputs in place through NVLink peer access
 * (devices without peer access to the buffers are left out), again pulling chunks from one shared counter. Blocks the
 * host until the batch has drained; outputs are complete when `stream` reaches this point. */
int dnaldpc_decode_batch_device(dnaldpc_decoder *d, const dnaldpc_input *in, int64_t F, int max_iter,
                                const dnaldpc_output *out, void *stream);

/* One-frame drop-in with the reference's exact buffer contract:
 *   int Run_Belief_Propagation_Decoder(mod2sparse *H, double *lratio, char *dblk, char *pchk, int *bIsCodeword)  (dec.h:80)
 * returns n in *iters; *is_codeword is written 0/1 (the reference leaves it untouched on failure). */
int dnaldpc_run_bp_decoder(dnaldpc_decoder *d, const double *lratio, int max_iter, char *dblk, char *pchk,
                           int *is_codeword, int *iters);

/* Re-decoding sweep of the pipeline (ex_decoder/decoder.py:594-664): round r decodes, with LR = exp(scales[r]*LLR), the
 * frames no earlier round turned into a codeword (round 0: all frames); the reference rescales the LLRs by
 * ln((1-e2)/e2)/ln((1-e)/e) for e2 = e-0.0005, e-0.001, ... and launches ldpc.exe again per failed frame per round.
 * Outputs hold each frame's result of its LAST round, rounds[f] (may be NULL) the index of that round. HOST buffers.
 * Difference from the reference, on purpose: it calls a frame failed by comparing with the TRUE codeword
 * (decoder.py:641-660), which a deployed decoder does not have; here a frame has failed when its syndrome is non-zero.
 * flags: DNALDPC_FLAG_HOST_EXP for libm exp on the host (bit-exact with the reference's exe). */
int dnaldpc_redecode_sweep(dnaldpc_decoder *d, const double *llr, int64_t F, int max_iter, const double *scales,
                           int n_scales, int flags, const dnaldpc_output *out, int32_t *rounds);
/* The same sweep for any parameterised input kind: round r decodes with in->param = params[r] (LLR kinds: the scale;
 * VOTE_I8: eps_r, i.e. LR = exp(k*ln((1-eps_r)/eps_r)) from a fresh 256-entry table per round, which is exactly what the
 * pipeline's rescaled LLR file holds; BSC_BITS: p_r; AWGN: sigma_r). HOST buffers. The inputs are uploaded ONCE (while
 * round 0 decodes) and stay in HBM; later rounds run over a device-side list of the rows whose syndrome is still
 * non-zero, so nothing but that round's results crosses PCIe again. With DNALDPC_FLAG_HOST_EXP (LLR_F64) the failed
 * frames are exponentiated on the host per round instead (libm exp, bit-exact with the reference's exe). */
int dnaldpc_redecode_sweep_ex(dnaldpc_decoder *d, const dnaldpc_input *in, int64_t F, int max_iter, const double *params,
                              int n_params, const dnaldpc_output *out, int32_t *rounds);

/* Sliding-window belief propagation for spatially-coupled (SC-LDPC) codes = Run_SW_Decoder (dec.cpp:2092-2196; decoder
 * type 60 of the reference CLI, DNA_main.cpp:1599-1602) with Init_SW_Decoder / Iter_SW_Decoder / Check_Update_SW /
 * Variable_Update_SW / Decision_SW (dec.cpp:2366-2645) and check_bound (check.cpp:49-72). The window description is the
 * reference's argument list: code_type (0: two-sided termination, SC_D = L + w - 1 positions of checks; otherwise
 * L + (w-1)/2), coupling length L, coupling width w, window size win (all in positions) and the per-position node
 * counts Mv[SC_D], Mc[SC_D] (g_SC_CODE_M / g_SC_CODE_Mc, DNA_main.cpp:440-462). Columns / rows of H are ordered by
 * position. lratio: HOST double [F][N], p0/p1. Outputs (HOST; posterior must be NULL): bits / dblk = final decisions,
 * iters = floor(sum over positions of Iter_SW_Decoder's n / L) as returned by the reference, is_codeword and pchk from
 * the closing check(). Bits no window has decided yet count as set in the bounded syndromes, as with the reference's
 * dblk buffer pre-filled with 2 (DNA_main.cpp:664-666). The position_BER diagnostic (test_BER) is not produced.
 * fp64 only. With several devices every device decodes a contiguous share of the frames (no exchange between them). */
typedef struct dnaldpc_window {
    int32_t code_type, L, w, win;
    const int32_t *Mv, *Mc;
} dnaldpc_window;
int dnaldpc_decode_window(dnaldpc_decoder *d, const dnaldpc_window *win, const double *lratio, int64_t F, int max_iter,
                          const dnaldpc_output *out);

/* ---- likelihood-setup helpers (host) ----------------------------------------------------------- */
double dnaldpc_std_dev(double ebno_db, double rate);                  /* getStd_dev, channel.cpp:9-16 */
int dnaldpc_vote_table(double eps, double *table256);                 /* table[k+128] = exp(k*ln((1-eps)/eps)) */
int dnaldpc_bsc_table(double p, double *table2);                      /* {(1-p)/p, p/(1-p)}, channel.cpp:75-84 */

/* ---- synthetic inputs on the device (benchmarks / scaling runs) --------------------------------- */
/* Received hard bits of a BSC for frames [frame0, frame0+F): bit j of frame f = codeword[(f % n_cw)][j] ^ flip,
 * flip iff (rng_u64(seed, f, j, 0) >> 11) < (uint64)(eps * 2^53)   (counter RNG specified in DESIGN.md).
 * cw_bits: DEVICE uint32 [n_cw][ceil(N/32)] or NULL for the all-zero codeword. out_bits: DEVICE uint32 [F][ceil(N/32)].
 * Keyed by the GLOBAL frame index, so any sharding over GPUs produces the same frames. */
int dnaldpc_synth_bsc_device(dnaldpc_decoder *d, const uint32_t *cw_bits, int n_cw, uint64_t seed, int64_t frame0,
                             int64_t F, double eps, uint32_t *out_bits, void *stream);

/* Received values of a BPSK/AWGN channel (BASELINE configs[3]; channel_AWGN, channel.cpp:23-35): y = (bit ? -1 : +1) +
 * sigma * n, n = sqrt(-2 ln u1) * cos(2 pi u2) with u1 = ((rng_u64(seed,f,j,4) >> 11) + 1) / 2^53, u2 =
 * (rng_u64(seed,f,j,5) >> 11) / 2^53 in fp64, rounded to float. out_y: DEVICE float [F][N]. sigma from dnaldpc_std_dev. */
int dnaldpc_synth_awgn_device(dnaldpc_decoder *d, const uint32_t *cw_bits, int n_cw, uint64_t seed, int64_t frame0,
                              int64_t F, double sigma, float *out_y, void *stream);
/* Vote counts k = count0 - count1 of aligned reads (BASELINE configs[2]; the soft information of
 * ex_decoder/decoder.py:292-316): reads per bit c ~ Poisson(mean_reads) capped at 63 (inversion of rng stream 2 against
 * integer CDF thresholds), each read wrong with probability read_err (streams 3..3+c). out_k: DEVICE int8 [F][N].
 * Integer arithmetic on the device: identical to the host twin for any sharding. mean_reads in (0, 32]. */
int dnaldpc_synth_vote_device(dnaldpc_decoder *d, const uint32_t *cw_bits, int n_cw, uint64_t seed, int64_t frame0,
                              int64_t F, double mean_reads, double read_err, int8_t *out_k, void *stream);

/* ---- systematic encoder ------------------------------------------------------------------------ */
/* Systematic form of H. Scanning the columns from N-1 down to 0, column j is a parity column iff it is linearly
 * independent over GF(2) of the parity columns already chosen (the pivot columns of the reduced row-echelon form of H
 * with its column order reversed); a column with no entries is always an info column. R = rank(H) parity columns,
 * K = N - R info columns, both lists ascending. Message bit t goes to info_cols[t]; parity bit i, at parity_cols[i], is
 * XOR_t A[i][t] m_t, where row i of A is the reduced row whose pivot is parity_cols[i], restricted to the info columns.
 * Hence encode(c[info_cols]) == c for every codeword c. Computed once per code, on first use (about a second for
 * N = 18432); DNALDPC_ERR_UNSUPPORTED when M*M or R*K exceeds 2^33 bits.
 * K receives N - rank(H); info_cols / parity_cols (capacity N each, may be NULL) receive the ascending column lists.
 * Host only, no GPU needed. */
int dnaldpc_code_systematic(const dnaldpc_code *c, int *K, int32_t *info_cols, int32_t *parity_cols);
/* msg: uint32 [F][ceil(K/32)] LSB first (bits beyond K in the last word are ignored) -> cw: uint32 [F][ceil(N/32)] (the
 * layout of dnaldpc_output.bits and of the synth functions' cw_bits; bits beyond N are written as 0). DEVICE buffers on
 * the decoder's first device, asynchronous on `stream`. Encoding runs on that one device only (no multi-GPU dispatch). */
int dnaldpc_encode_device(dnaldpc_decoder *d, const uint32_t *msg, int64_t F, uint32_t *cw, void *stream);
int dnaldpc_encode(dnaldpc_decoder *d, const uint32_t *msg, int64_t F, uint32_t *cw);        /* HOST buffers, blocking */
/* cw: uint32 [F][ceil(N/32)] -> msg: uint32 [F][ceil(K/32)], the bits at info_cols (no syndrome check; bits beyond K are
 * written as 0). */
int dnaldpc_extract_device(dnaldpc_decoder *d, const uint32_t *cw, int64_t F, uint32_t *msg, void *stream);
int dnaldpc_extract(dnaldpc_decoder *d, const uint32_t *cw, int64_t F, uint32_t *msg);       /* HOST buffers, blocking */

/* ---- Monte-Carlo error-rate simulation ---------------------------------------------------------- */
/* Random codewords through a synthetic channel, decoded and counted on the decoder's devices (Run_Simulation /
 * Print_One_Result of the reference's command line). Contract:
 *   Frames. Frame f (global index 0, 1, ...) carries the message whose 32-bit word w is the low 32 bits of
 *     rng_u64(seed, f, w, 1) (RNG stream 1 of DESIGN.md §9), bits at and beyond K cleared; its codeword is
 *     dnaldpc_encode(message); its channel values are exactly what dnaldpc_synth_{bsc,awgn,vote}_device produce for frame
 *     f given that codeword (vote counts: read_err = param, mean_reads); it is decoded as dnaldpc_decode_batch_device
 *     decodes that input kind with param and flags (vote counts with the table built from eps = param).
 *   Raw hard decision ("without coding"): BSC the received bit, AWGN y < 0, vote counts k < 0.
 *   Stopping. With T = target_frame_errors > 0 the result counts the shortest prefix of frames [0, n) that holds T frame
 *     errors, or n = max_frames if that comes first; with T = 0 exactly max_frames frames. Frames decoded past n are
 *     discarded, so every counter is a function of (code, spec) alone, whatever the piece size, wave_frames, number of
 *     GPUs or timing.
 *   Requirements. The systematic form is required: codes over its cap give DNALDPC_ERR_UNSUPPORTED (as dnaldpc_encode).
 *     DNALDPC_ERR_ARG, before any device work, for a null handle or pointer, an unknown channel or flag, p not in (0,1),
 *     sigma <= 0, mean_reads not in (0,32] (vote counts), max_iter < 0, max_frames < 1 or target_frame_errors < 0.
 *   Devices. Runs on every device of the decoder like a batch call (each device encodes its own frames with an encoder
 *     of its own); dnaldpc_get_stats reports every frame decoded, the discarded ones included. Blocking. */
typedef struct dnaldpc_sim {
    int32_t channel;   /* DNALDPC_IN_BSC_BITS (param = p), DNALDPC_IN_AWGN_F32 (param = sigma),
                          DNALDPC_IN_VOTE_I8 (param = read error probability, also the decoder's eps; mean_reads) */
    int32_t flags;     /* DNALDPC_FLAG_MINSUM, DNALDPC_FLAG_FIXED_ITERS; anything else -> DNALDPC_ERR_ARG */
    double param, mean_reads;
    uint64_t seed;
    int32_t max_iter;
    int64_t max_frames;           /* frames to simulate; the cap when target_frame_errors > 0 */
    int64_t target_frame_errors;  /* 0 = exactly max_frames */
} dnaldpc_sim;
typedef struct dnaldpc_sim_result {
    int64_t frames, iterations;                 /* frames counted; sum of their iteration counts          */
    int64_t frame_errors, bit_errors;           /* decoded != sent, over all N bits                       */
    int64_t msg_frame_errors, msg_bit_errors;   /* the same over the K info columns (the message)          */
    int64_t detected, undetected;               /* syndrome != 0 / syndrome == 0 but decoded != sent       */
    int64_t raw_frame_errors, raw_bit_errors;   /* channel hard decision != sent ("without coding")        */
} dnaldpc_sim_result;
int dnaldpc_simulate(dnaldpc_decoder *d, const dnaldpc_sim *s, dnaldpc_sim_result *r);

/* ---- statistics of the last decode call on this handle ------------------------------------------ */
typedef struct dnaldpc_stats {
    int64_t frames;
    int64_t frame_iters;     /* sum over frames of iterations performed */
    int64_t kernel_launches; /* CUDA kernels launched by the call */
    int64_t waves;
    double row_ms, col_ms;   /* device time (CUDA events) inside the check-node / bit-node kernels; 0 unless profiling enabled */
    double total_ms;
    int64_t compactions;     /* drain-tail compactions (stragglers re-packed into the lowest slot groups) */
} dnaldpc_stats;
int dnaldpc_get_stats(const dnaldpc_decoder *d, dnaldpc_stats *s);
/* 1 = bracket the row/column kernels of each iteration with CUDA events (adds host syncs; benchmarking only);
 * 2 = in-pipeline trace: events around the check pass / bit pass of ticks 8..71 of the next batch, NO synchronisation
 *     (first device only); read with dnaldpc_get_trace after the batch. 0 = off. */
int dnaldpc_set_profiling(dnaldpc_decoder *d, int on);
/* Average check-pass, bit-pass and scheduler (bit-pass end -> next check-pass start: syndrome, admission, launch gaps)
 * time per traced tick, in ms. */
int dnaldpc_get_trace(dnaldpc_decoder *d, double *row_ms, double *col_ms, double *sched_ms, int *ticks);

/* ---- diagnostics ------------------------------------------------------------------------------- */
/* Runs `n` random operands (plus the IEEE corner cases) through the inlined in-range reciprocal / division sequences
 * of the check-node kernel and through nvcc's full-range IEEE division, on the current device; *mismatches receives
 * the number of results that differ in any bit (must be 0). */
int dnaldpc_selftest_math(int64_t n, uint64_t seed, int64_t *mismatches);

#ifdef __cplusplus
}
#endif
#endif /* DNALDPC_H */
