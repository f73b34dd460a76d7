// ldpc_main.cpp - drop-in for the reference's `ldpc` command line on its belief-propagation path.
//
// Grammar (SetUp, DNA_main.cpp:300-505; pipeline instance ex_decoder/def_func.py:49):
//   ldpc <bSystematic> <decoder_type> <channel_type> <seed> <max_iter> <frame_num> [<target_frame_err> if frame_num==0]
//        <codeword_base> <soft_base> <pchk_base> <chan_param> <punctuation> <shortening> <targeting>  [extensions]
// Reads <codeword_base>.txt (true codeword), <soft_base>.txt (LLR = ln(p0/p1)) and <pchk_base>.pchk from the CWD,
// writes dec_<codeword_base>.txt, result_(...).txt and the same stdout summary as the reference
// (Set_Code :552-556, Run_Simulation :916-927, Print_One_Result :1170-1182, Print_All_Result :1048-1123).
// Decoder types 0 (BP), 20-22 (floating min-sum) and 60 (sliding-window BP for spatially-coupled codes) without
// punctuation / shortening / targeting; anything else is rejected. Type 60 takes the reference's extra block
// `<code_type> <w> <L> <WIN>` after <targeting> and reads the per-position node counts (SC_D lines of Mv, then SC_D lines
// of Mc) from <pchk_base>.txt (DNA_main.cpp:424-464). Its POSITION_BER_*.txt diagnostic is not written.
//
// Extensions (after the positional block, none of them changes the reference behaviour when absent):
//   --device N        CUDA device ordinal (default 0)
//   --fp32            optional single-precision mode (statistical parity only)
//   --list FILE       batch mode: FILE holds one "<codeword_base> <soft_base>" pair per line; all frames are decoded
//                     in ONE process / one batched GPU call; a dec_*.txt per frame, one result file for the batch
//   --timing          print a JSON line with decode time and iteration counts (total, average, per frame) on stderr
//   --gpus N          decode the frames of a --list batch on N GPUs (ordinals device .. device+N-1); the library's own
//                     dispatcher shares them out in chunks (the reference's intended split is frames over ranks,
//                     DNA_main.cpp:629-651)
//   --serve           resident worker: keeps the CUDA context and one decoder per parity-check file, and serves the
//                     command lines of clients over the Unix socket $DNALDPC_SOCKET (or --socket PATH) until
//                     `ldpc --shutdown`. A client is this same binary: when DNALDPC_SOCKET is set and a worker
//                     answers there, the command line, working directory included, is run by the worker (same files,
//                     same stdout, same exit code); otherwise it runs locally. The unmodified pipeline
//                     (ex_decoder/def_func.py:47-51, one os.system("ldpc ...") per codeword) then pays milliseconds
//                     per call instead of a CUDA context creation.
//   --layered         with decoder types 20-22: row-layered normalised min-sum (DNALDPC_FLAG_LAYERED) instead of the
//                     flooding min-sum; --scale A sets its normalisation alpha in (0, 1] (default 1)
//
// Simulation (the reference's frame_num / target_frame_err mode: random codewords through a synthetic channel):
//   ldpc --simulate <pchk_base> <channel_type> <p1[,p2,...]> <seed> <max_iter> <frame_num> [<target_frame_err> if frame_num==0]
//        [--max-frames N] [--reads R] [--decoder 0|20] [--layered [--scale A]] [--device N] [--gpus N] [--fp32] [--timing]
// runs dnaldpc_simulate once per parameter: frames carry random messages (RNG stream 1 of DESIGN.md §9) encoded with
// the systematic form, go through the channel and are decoded and counted on the GPU. Channel types: 0 = AWGN, the
// parameters are Eb/N0 in dB and sigma = getStd_dev(Eb/N0, K/N) with K = N - rank(H), the true rate of the code;
// 1 = BSC with crossover probability p; 3 = vote counts of aligned reads, p = read error probability (also the
// decoder's eps), --reads R mean reads per bit (required, in (0, 32]). 2 (BEC) and anything else are rejected.
// frame_num > 0 simulates exactly that many frames; frame_num 0 runs until <target_frame_err> frame errors, capped by
// --max-frames (default 10^9). --decoder 20 decodes with floating min-sum, --decoder 20 --layered with layered
// normalised min-sum (--scale A: alpha). Per parameter a Print_One_Result block
// (DNA_main.cpp:1170-1182) plus msg_bit_err, undetected (zero syndrome, wrong codeword) and avg_iter lines; --timing
// adds one JSON line per parameter on stderr with every counter and the wall time. Argument and file errors are
// reported before any CUDA call.
//
// Encoder (no counterpart in the reference's command line):
//   ldpc --encode <pchk_base> <msg_base> <codeword_base>   or   ldpc --encode <pchk_base> --list FILE
// reads K = N - rank(H) message bits (whitespace-separated 0/1) from <msg_base>.txt, encodes them on the GPU with the
// systematic form of include/dnaldpc.h and writes <codeword_base>.txt in the codeword-file format (N x "%d ", no
// newline) that the decode command line reads. --list FILE holds one "<msg_base> <codeword_base>" pair per line, all
// encoded in one call. --device N and --timing apply; argument and file errors are reported before any CUDA call.
#include <sys/socket.h>
#include <sys/stat.h>
#include <sys/un.h>
#include <unistd.h>

#include <cerrno>
#include <cmath>
#include <csignal>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <algorithm>
#include <chrono>
#include <atomic>
#include <map>
#include <string>
#include <thread>
#include <vector>

#include "dnaldpc.h"
#include "textio.h"

using namespace dnaldpc;

namespace {

struct Args {
    int bSystematic = 0, decoder_type = 0, channel_type = 0, seed = 0, max_iter = 0;
    long frame_num = 1;
    int target_frame_err = 0;
    std::string cw_base, soft_base, pchk_base;
    double chan_param = 0;
    int punctuation = 0, shortening = 0, targeting = 0;
    int sc_code_type = 0, sc_w = 0, sc_L = 0, sc_win = 0;  // decoder type 60 only
    int device = 0, gpus = 1;
    bool fp32 = false, timing = false, serve = false, shutdown = false, encode = false, simulate = false;
    std::string list, socket_path;
    std::string msg_base;  // --encode: <pchk_base> <msg_base> <codeword_base> (cw_base, pchk_base as for decoding)
    std::vector<std::string> sim_pos;  // --simulate: the positional arguments after the flag
    std::string max_frames, reads, decoder;  // --simulate options, checked by run_simulate
    bool layered = false;                    // --layered: DNALDPC_FLAG_LAYERED (min-sum decoders only)
    std::string scale;                       // --scale A: normalisation of the layered decoder, checked by check_layered
};

// Where a run writes: a local run uses the process's own streams, a run on behalf of a client memory streams.
struct Io {
    FILE *out = stdout, *err = stderr;
    const std::string &path(const std::string &p) const { return p; }
};

bool parse(const std::vector<std::string> &argv, Args &a, Io &io) {
    std::vector<std::string> pos;
    for (size_t i = 0; i < argv.size(); i++) {
        const std::string &s = argv[i];
        if (s == "--device" && i + 1 < argv.size()) a.device = atoi(argv[++i].c_str());
        else if (s == "--gpus" && i + 1 < argv.size()) a.gpus = atoi(argv[++i].c_str());
        else if (s == "--fp32") a.fp32 = true;
        else if (s == "--timing") a.timing = true;
        else if (s == "--serve") a.serve = true;
        else if (s == "--shutdown") a.shutdown = true;
        else if (s == "--socket" && i + 1 < argv.size()) a.socket_path = argv[++i];
        else if (s == "--list" && i + 1 < argv.size()) a.list = argv[++i];
        else if (s == "--encode") a.encode = true;
        else if (s == "--simulate") a.simulate = true;
        else if (s == "--max-frames" && i + 1 < argv.size()) a.max_frames = argv[++i];
        else if (s == "--reads" && i + 1 < argv.size()) a.reads = argv[++i];
        else if (s == "--decoder" && i + 1 < argv.size()) a.decoder = argv[++i];
        else if (s == "--layered") a.layered = true;
        else if (s == "--scale" && i + 1 < argv.size()) a.scale = argv[++i];
        else pos.push_back(s);
    }
    if (a.serve || a.shutdown) return true;
    if (a.simulate) { a.sim_pos = pos; return true; }
    if (a.encode) {
        if (pos.size() != (a.list.empty() ? 3u : 1u)) {
            fprintf(io.err, "usage: ldpc --encode <pchk_base> <msg_base> <codeword_base>  |  ldpc --encode <pchk_base> --list FILE\n");
            return false;
        }
        a.pchk_base = pos[0];
        if (a.list.empty()) { a.msg_base = pos[1]; a.cw_base = pos[2]; }
        return true;
    }
    size_t p = 0;
    bool short_of = false;
    auto next = [&]() -> const char * { if (p >= pos.size()) { short_of = true; return "0"; } return pos[p++].c_str(); };
    a.bSystematic = atoi(next());
    a.decoder_type = atoi(next());
    a.channel_type = atoi(next());
    a.seed = atoi(next());
    a.max_iter = atoi(next());
    a.frame_num = atol(next());
    if (a.frame_num == 0 && !short_of) a.target_frame_err = atoi(next());
    a.cw_base = next();
    a.soft_base = next();
    a.pchk_base = next();
    a.chan_param = atof(next());
    a.punctuation = atoi(next());
    a.shortening = atoi(next());
    a.targeting = atoi(next());
    if (a.decoder_type == 60 && !a.punctuation && !a.shortening && !a.targeting) {  // DNA_main.cpp:424-429
        a.sc_code_type = atoi(next());
        a.sc_w = atoi(next());
        a.sc_L = atoi(next());
        a.sc_win = atoi(next());
    }
    if (short_of || p != pos.size()) {
        fprintf(io.err, "\n\nargc error!\n\n");  // DNA_main.cpp:494-502
        return false;
    }
    return true;
}

bool parse_num(const std::string &s, double &v);

// --layered / --scale: the layered decoder exists for min-sum only; alpha in (0, 1]. Returns the error text or "".
std::string check_layered(const Args &a, bool minsum, double &alpha) {
    alpha = 1.0;
    if (a.layered && !minsum) return "--layered needs a min-sum decoder (decoder type 20-22, --simulate --decoder 20)";
    if (!a.scale.empty()) {
        if (!a.layered) return "--scale needs --layered";
        if (!parse_num(a.scale, alpha) || !(alpha > 0.0 && alpha <= 1.0)) return "--scale must be in (0, 1]";
    }
    return "";
}

// Decoders kept by the resident worker: one per (parity-check file, its size and modification time, precision, GPUs).
struct Cache {
    struct Entry { dnaldpc_code *code; dnaldpc_decoder *dec; };
    std::map<std::string, Entry> map;
};

// One command line, start to finish (Set_Code, LDPC_Encode, LDPC_Decode, result files). `cache` != NULL: the decoder
// comes from / goes to the worker's cache instead of being created and destroyed here.
int run(Args a, Io &io, Cache *cache) {
#define CHECK(call)                                             \
    do {                                                        \
        if ((call) != DNALDPC_OK) {                             \
            fprintf(io.err, "%s\n", dnaldpc_last_error());      \
            return 1;                                           \
        }                                                       \
    } while (0)
    // 0 = belief propagation; 20/21/22 = min-sum: with g_precision == 0 (the CLI cannot set it) all three reach the
    // floating-point Run_MSA_Decoder_INF (DNA_main.cpp:1588-1594)
    const bool minsum = a.decoder_type == 20 || a.decoder_type == 21 || a.decoder_type == 22;
    const bool window = a.decoder_type == 60;
    if (a.decoder_type != 0 && !minsum && !window) {
        fprintf(io.err, "ldpc: decoder type %d is not supported by this build (0 = belief propagation, 20-22 = floating min-sum, 60 = sliding window)\n", a.decoder_type);
        return 1;
    }
    double alpha = 1.0;
    {
        const std::string why = check_layered(a, minsum, alpha);
        if (!why.empty()) { fprintf(io.err, "ldpc: %s\n", why.c_str()); return 1; }
    }
    if (a.punctuation || a.shortening || a.targeting) {
        fprintf(io.err, "ldpc: punctuation / shortening / targeting are not supported by this build (pass 0 0 0)\n");
        return 1;
    }
    if (a.frame_num == 0) {
        fprintf(io.err, "ldpc: frame_num 0 (run until target frame errors) needs a channel simulator; not supported\n");
        return 1;
    }
    if (a.max_iter < 0) a.max_iter = 0;

    // Set_Code (DNA_main.cpp:544-609)
    const std::string pchk_file = a.pchk_base + ".pchk";
    dnaldpc_code *code = nullptr;
    dnaldpc_decoder *dec = nullptr;
    std::string cache_key;
    if (cache) {  // resident worker: one decoder per parity-check file (as long as the file does not change)
        struct stat sb;
        if (stat(io.path(pchk_file).c_str(), &sb) == 0) {
            char key[64];
            snprintf(key, sizeof(key), "|%lld|%lld.%09ld|%d|%d|%d", (long long)sb.st_size, (long long)sb.st_mtim.tv_sec, (long)sb.st_mtim.tv_nsec,
                     a.fp32 ? 1 : 0, a.device, a.gpus);
            char *rp = realpath(pchk_file.c_str(), nullptr);
            cache_key = std::string(rp ? rp : pchk_file.c_str()) + key;
            free(rp);
            auto it = cache->map.find(cache_key);
            if (it != cache->map.end()) { code = it->second.code; dec = it->second.dec; }
        }
    }
    const bool cached = dec != nullptr;
    if (!code) CHECK(dnaldpc_code_read_pchk(io.path(pchk_file).c_str(), &code));
    struct Owned {  // whatever this run created and did not hand to the cache goes away with it, on every return path
        dnaldpc_code *&code; dnaldpc_decoder *&dec; bool mine;
        ~Owned() { if (mine) { if (dec) dnaldpc_decoder_destroy(dec); if (code) dnaldpc_code_free(code); } }
    } owned{code, dec, !cached};
    int M, N, E;
    dnaldpc_code_dims(code, &M, &N, &E);
    const int K = N - M;
    fprintf(io.out, "\ng_CODE_N : %d\ng_CODE_K : %d\ng_CODE_M : %d\n\n", N, K, M);
    const double rate = 1.0 - (double)((double)M / (double)N);
    const double ebno = a.channel_type == 0 ? a.chan_param : 0.0;
    const double std_dev = dnaldpc_std_dev(ebno, rate);
    int dv, rdv, dc, rdc;
    dnaldpc_code_check_regular(code, &dv, &rdv, &dc, &rdc);  // LDPC_Set_Decoder -> CheckRegular

    // sliding window: per-position node counts from <pchk_base>.txt (SC_D values of Mv, then SC_D of Mc; DNA_main.cpp:431-462)
    std::vector<int32_t> sc_mv, sc_mc;
    if (window) {
        if (a.sc_L < 1 || a.sc_w < 1 || a.sc_win < 1) { fprintf(io.err, "ldpc: bad sliding-window parameters (w, L, WIN must be >= 1)\n"); return 1; }
        const int D = a.sc_code_type == 0 ? a.sc_L + a.sc_w - 1 : a.sc_L + (a.sc_w - 1) / 2;
        const std::string mfile = a.pchk_base + ".txt";
        FILE *f = fopen(io.path(mfile).c_str(), "r");
        if (!f) { fprintf(io.err, "Can't open node-count file: %s\n", mfile.c_str()); return 1; }
        sc_mv.assign((size_t)D, 0);
        sc_mc.assign((size_t)D, 0);
        bool ok = true;
        for (int i = 0; i < D && ok; i++) ok = fscanf(f, "%d", &sc_mv[(size_t)i]) == 1;
        for (int i = 0; i < D && ok; i++) ok = fscanf(f, "%d", &sc_mc[(size_t)i]) == 1;
        fclose(f);
        if (!ok) { fprintf(io.err, "Node-count file %s holds fewer than 2 x %d integers\n", mfile.c_str(), D); return 1; }
    }

    // frames: the positional pair, or every pair of --list
    std::vector<std::pair<std::string, std::string>> frames;
    if (a.list.empty()) frames.push_back({a.cw_base, a.soft_base});
    else {
        FILE *f = fopen(io.path(a.list).c_str(), "r");
        if (!f) { fprintf(io.err, "Can't open list file: %s\n", a.list.c_str()); return 1; }
        char c1[512], c2[512];
        while (fscanf(f, "%511s %511s", c1, c2) == 2) frames.push_back({c1, c2});
        fclose(f);
        if (frames.empty()) { fprintf(io.err, "List file %s holds no \"<codeword> <soft>\" pairs\n", a.list.c_str()); return 1; }
    }
    const size_t F = frames.size();

    time_t t_start, t_end;
    time(&t_start);

    // CUDA context creation dominates a one-process run (about a second); it runs on its own thread while the input
    // text is parsed. A one-frame run is dominated by it anyway; exposing only the requested GPU to the driver keeps it
    // from initialising every device of an 8-GPU box (the variable is only set when the caller has not set it).
    if (a.gpus < 1 || a.gpus > 16) { fprintf(io.err, "ldpc: --gpus must be between 1 and 16\n"); return 1; }
    if (!cache && a.gpus == 1 && getenv("CUDA_VISIBLE_DEVICES") == nullptr) {  // remap only when WE narrowed the view: a caller's own setting keeps its ordinals
        char dev[16];
        snprintf(dev, sizeof(dev), "%d", a.device);
        if (setenv("CUDA_VISIBLE_DEVICES", dev, 0) == 0) a.device = 0;
    }
    dnaldpc_config cfg{};
    cfg.n_devices = a.gpus;
    for (int k = 0; k < a.gpus; k++) cfg.devices[k] = a.device + k;
    cfg.precision = a.fp32 ? DNALDPC_PREC_F32 : DNALDPC_PREC_F64;
    // slots are allocated for the frames of a call (grown on demand): a resident decoder keeps the full default wave
    cfg.wave_frames = cache ? 4096 : (int)std::min<size_t>(4096, (F + 31) / 32 * 32);
    int create_rc = 0;
    std::string create_err;
    auto i0 = std::chrono::steady_clock::now();
    std::chrono::steady_clock::time_point i1 = i0;
    std::thread creator([&]() {
        if (cached) return;
        create_rc = dnaldpc_decoder_create(code, &cfg, &dec);  // includes CUDA context creation
        if (create_rc) create_err = dnaldpc_last_error();      // thread-local message: keep it before the thread ends
        i1 = std::chrono::steady_clock::now();
    });

    // LDPC_Encode (DNA_main.cpp:1319-1348): codeword + LLR text, LR = exp(LLR) with the host libm; frames in parallel
    std::vector<signed char> codewords(F * (size_t)N);
    std::vector<double> llr(F * (size_t)N), lr(F * (size_t)N);
    std::string err;
    {
        const unsigned nthr = (unsigned)std::max<size_t>(1, std::min<size_t>({F, (size_t)std::max(1u, std::thread::hardware_concurrency()), (size_t)16}));
        std::atomic<size_t> next{0};
        std::atomic<long> first_bad{-1};
        std::vector<std::string> errs(F);
        auto work = [&]() {
            for (size_t f = next++; f < F; f = next++) {
                std::vector<signed char> cw;
                std::vector<double> l;
                if (!read_codeword_txt(io.path(frames[f].first + ".txt"), N, cw, errs[f]) || !read_llr_txt(io.path(frames[f].second + ".txt"), N, l, errs[f])) {
                    long expect = -1;
                    first_bad.compare_exchange_strong(expect, (long)f);
                    continue;
                }
                memcpy(&codewords[f * (size_t)N], cw.data(), (size_t)N);
                memcpy(&llr[f * (size_t)N], l.data(), (size_t)N * sizeof(double));
                for (int j = 0; j < N; j++) lr[f * (size_t)N + j] = exp(l[(size_t)j]);
            }
        };
        std::vector<std::thread> pool;
        for (unsigned t = 1; t < nthr; t++) pool.emplace_back(work);
        work();
        for (auto &t : pool) t.join();
        if (first_bad >= 0) {
            size_t bad = 0;  // report the first frame of the list that failed, like a serial reader would
            while (errs[bad].empty()) bad++;
            creator.join();
            fprintf(io.err, "%s\n", errs[bad].c_str());
            return 1;
        }
    }
    creator.join();
    if (create_rc) { fprintf(io.err, "%s\n", create_err.c_str()); return 1; }
    if (cache && !cached && !cache_key.empty()) { cache->map[cache_key] = Cache::Entry{code, dec}; owned.mine = false; }

    std::vector<unsigned char> dblk(F * (size_t)N), okflag(F);
    std::vector<int32_t> iters(F);
    dnaldpc_input in{};
    in.kind = minsum ? DNALDPC_IN_LLR_F64 : DNALDPC_IN_LR_F64;   // min-sum works on the LLRs themselves
    in.flags = minsum ? DNALDPC_FLAG_MINSUM : 0;
    if (a.layered) in.flags |= DNALDPC_FLAG_LAYERED;
    in.data = minsum ? llr.data() : lr.data();
    CHECK(dnaldpc_set_minsum_scale(dec, alpha));  // every run: a resident decoder keeps the previous run's value
    dnaldpc_output out{};
    out.dblk = dblk.data();
    out.iters = iters.data();
    out.is_codeword = okflag.data();
    auto c0 = std::chrono::steady_clock::now();
    if (window) {  // LDPC_Decode -> Run_SW_Decoder (DNA_main.cpp:1599-1602)
        dnaldpc_window wd{};
        wd.code_type = a.sc_code_type; wd.L = a.sc_L; wd.w = a.sc_w; wd.win = a.sc_win;
        wd.Mv = sc_mv.data(); wd.Mc = sc_mc.data();
        CHECK(dnaldpc_decode_window(dec, &wd, lr.data(), (int64_t)F, a.max_iter, &out));
    } else
        CHECK(dnaldpc_decode_batch(dec, &in, (int64_t)F, a.max_iter, &out));  // LDPC_Decode -> Run_Belief_Propagation_Decoder
    auto c1 = std::chrono::steady_clock::now();

    // error counting: LDPC_Raw_Error_Check (:1711-1750, sign of the LLR) and LDPC_BIT_Check (:1675-1706)
    const int len = a.bSystematic ? K : N;
    long long bit_err[3] = {0, 0, 0}, frame_err[3] = {0, 0, 0}, total_iter = 0, n_converged = 0;
    for (size_t f = 0; f < F; f++) {
        long long raw = 0, dec_err = 0;
        for (int i = 0; i < len; i++) {
            // channel type 0 compares the sign of the soft input; types 1 / 2 look at g_recv_codeword_hard, which nothing
            // fills since the channel simulators are commented out (DNA_main.cpp:1358-1371): calloc'ed zeros, i.e.
            // "received 0" for the BSC branch and "nothing erased" for the BEC branch (:1733-1745)
            const int hard = a.channel_type == 0 ? (llr[f * (size_t)N + i] >= 0 ? 0 : 1) : 0;
            if (a.channel_type != 2) raw += (codewords[f * (size_t)N + i] != hard);
            dec_err += (codewords[f * (size_t)N + i] != (signed char)dblk[f * (size_t)N + i]);
        }
        bit_err[0] += raw; frame_err[0] += raw > 0;
        bit_err[1] += dec_err; frame_err[1] += dec_err > 0;
        bit_err[2] += dec_err; frame_err[2] += dec_err > 0;
        total_iter += iters[f];
        n_converged += okflag[f] != 0;  // zero syndrome (`*bIsCodeword`), whether or not it is the codeword that was sent
    }
    // frame_num > 1 re-reads the same files and repeats the identical decode (DNA_main.cpp:1319-1348): counters scale
    const long long reps = a.list.empty() ? a.frame_num : 1;
    const long long n_frames = (long long)F * reps;
    for (int i = 0; i < 3; i++) { bit_err[i] *= reps; frame_err[i] *= reps; }

    // dec_<codeword_base>.txt (:916-927); the file name is printed without a newline (:918)
    for (size_t f = 0; f < F; f++) {
        const std::string dec_name = "dec_" + frames[f].first + ".txt";
        if (!write_dec_txt(io.path(dec_name), &dblk[f * (size_t)N], N, err)) { fprintf(io.err, "%s\n", err.c_str()); return 1; }
        if (f + 1 == F) fprintf(io.out, "%s", dec_name.c_str());
    }
    time(&t_end);

    // Print_One_Result (:1170-1182)
    fprintf(io.out, "\n");
    if (a.channel_type == 2) fprintf(io.out, "[%d]  code : (%d,%d)\trate : %.3f\tEps : %.2f \n", 0, N, K, rate, a.chan_param);
    else fprintf(io.out, "[%d]  code : (%d,%d)\trate : %.3f\tEb/No : %.2f dB\n", 0, N, K, rate, ebno);
    fprintf(io.out, "[%d]  frame_num              : %lld\n", 0, n_frames);
    fprintf(io.out, "[%d]  bit_err                : %lld\n", 0, bit_err[2]);
    fprintf(io.out, "[%d]  frame_err              : %lld\n", 0, frame_err[2]);
    fprintf(io.out, "[%d]  without coding (bit)   : %lld\n", 0, bit_err[0]);
    fprintf(io.out, "[%d]  without coding (frame) : %lld\n\n", 0, frame_err[0]);

    // Print_All_Result (:965-1123)
    char name[1024];
    const std::string soft_file = (a.list.empty() ? a.soft_base : a.list) + (a.list.empty() ? ".txt" : "");
    if (a.channel_type == 2)
        snprintf(name, sizeof(name), "result_(%s)_%s_%d_%.3f_%d_%d_%d.txt", soft_file.c_str(), pchk_file.c_str(), a.decoder_type, a.chan_param, 0, a.max_iter, a.seed);
    else if (a.channel_type == 1)
        snprintf(name, sizeof(name), "result_(%s)_%s_%d_%.4f_%d_%d_%d.txt", soft_file.c_str(), pchk_file.c_str(), a.decoder_type, a.chan_param, 0, a.max_iter, a.seed);
    else
        snprintf(name, sizeof(name), "result_(%s)_%s_%d_%.3fdB_%d_%d_%d.txt", soft_file.c_str(), pchk_file.c_str(), a.decoder_type, ebno, 0, a.max_iter, a.seed);
    FILE *fp = fopen(io.path(name).c_str(), "w");
    if (!fp) { fprintf(io.err, "Can't create %s\n", name); return 1; }
    fprintf(fp, "code N        : %d\n", N);
    fprintf(fp, "code K        : %d\n", K);
    fprintf(fp, "code M        : %d\n", M);
    fprintf(fp, "code rate     : %.3f\n", rate);
    if (a.channel_type == 2) fprintf(fp, "Eps\t\t: %.3f \n", a.chan_param);
    else {
        fprintf(fp, "Eb/No         : %.2f dB\n", ebno);
        fprintf(fp, "g_std_dev     : %.2f\n", std_dev);
    }
    fprintf(fp, "max iteration : %d\n", a.max_iter);
    fprintf(fp, "dv            : %d\n", dv);
    fprintf(fp, "bRegular_dv   : %d\n", rdv);
    fprintf(fp, "dc            : %d\n", dc);
    fprintf(fp, "bRegular_dc   : %d\n", rdc);
    if (window) fprintf(fp, "w   : %d\n\nL   : %d\n\nW   : %d\n\n", a.sc_w, a.sc_L, a.sc_win);  // DNA_main.cpp:1069-1071
    fprintf(fp, "=============================================\n");
    fprintf(fp, "                 result\n");
    fprintf(fp, "=============================================\n");
    double d = difftime(t_end, t_start);
    const int tm_hour = (int)(d / 3600); d -= tm_hour * 3600;
    const int tm_min = (int)(d / 60); d -= tm_min * 60;
    const int tm_sec = (int)d;
    fprintf(fp, "start time      : %s", ctime(&t_start));
    fprintf(fp, "end time        : %s", ctime(&t_end));
    fprintf(fp, "simulation time : %d hours %d mins %d secs\n\n", tm_hour, tm_min, tm_sec);
    fprintf(fp, "# of processes         : %d\n", 1);
    fprintf(fp, "initial seed value     : %d\n\n", a.seed);
    for (int i = 0; i < 2; i++) fprintf(fp, "# of Frame[%2d]          :%lld\n", i, n_frames);
    fprintf(fp, "\n");
    for (int i = 0; i < 2; i++) fprintf(fp, "# of Bit Errors[%2d]     : %lld\n", i, bit_err[i]);
    fprintf(fp, "\n");
    const double denom = (double)len * (double)n_frames;
    for (int i = 0; i < 2; i++) fprintf(fp, "BER[%2d]                 : %.5e\n", i, (double)bit_err[i] / denom);
    fprintf(fp, "\n");
    fclose(fp);

    if (a.timing) {
        const double ms = std::chrono::duration<double, std::milli>(c1 - c0).count();
        const double init_ms = std::chrono::duration<double, std::milli>(i1 - i0).count();
        // per-frame iteration counts and their average (the reference reports the average, DNA_main.cpp:1022)
        fprintf(io.err, "{\"frames\": %zu, \"gpus\": %d, \"gpu_init_ms\": %.1f, \"decode_ms\": %.3f, \"total_iterations\": %lld, \"avg_iterations\": %.4f, "
                "\"converged\": %lld, \"iterations\": [", F, a.gpus, init_ms, ms, total_iter, F ? (double)total_iter / (double)F : 0.0, n_converged);
        for (size_t f = 0; f < F; f++) fprintf(io.err, "%s%d", f ? ", " : "", (int)iters[f]);
        fprintf(io.err, "]}\n");
    }
    return 0;
#undef CHECK
}

// ldpc --encode: message files -> codeword files. Everything that can fail on the host (the parity-check file, the
// systematic form, the message files) is checked before the GPU is touched.
int run_encode(Args a, Io &io, bool resident) {
    const std::string pchk_file = a.pchk_base + ".pchk";
    dnaldpc_code *code = nullptr;
    dnaldpc_decoder *dec = nullptr;
    struct Owned {
        dnaldpc_code *&code; dnaldpc_decoder *&dec;
        ~Owned() { if (dec) dnaldpc_decoder_destroy(dec); if (code) dnaldpc_code_free(code); }
    } owned{code, dec};
    if (dnaldpc_code_read_pchk(io.path(pchk_file).c_str(), &code) != DNALDPC_OK) { fprintf(io.err, "%s\n", dnaldpc_last_error()); return 1; }
    int M, N, E, K;
    dnaldpc_code_dims(code, &M, &N, &E);
    if (dnaldpc_code_systematic(code, &K, nullptr, nullptr) != DNALDPC_OK) { fprintf(io.err, "%s\n", dnaldpc_last_error()); return 1; }
    std::vector<std::pair<std::string, std::string>> frames;  // (msg_base, codeword_base)
    if (a.list.empty()) frames.push_back({a.msg_base, a.cw_base});
    else {
        FILE *f = fopen(io.path(a.list).c_str(), "r");
        if (!f) { fprintf(io.err, "Can't open list file: %s\n", a.list.c_str()); return 1; }
        char c1[512], c2[512];
        while (fscanf(f, "%511s %511s", c1, c2) == 2) frames.push_back({c1, c2});
        fclose(f);
        if (frames.empty()) { fprintf(io.err, "List file %s holds no \"<msg> <codeword>\" pairs\n", a.list.c_str()); return 1; }
    }
    const size_t F = frames.size(), kw = (size_t)(K + 31) / 32, wpf = (size_t)(N + 31) / 32;
    std::vector<uint32_t> msg(F * kw, 0u), cw(F * wpf, 0u);
    std::string err;
    for (size_t f = 0; f < F; f++) {
        std::vector<signed char> m;
        const std::string path = frames[f].first + ".txt";
        if (!read_codeword_txt(io.path(path), K, m, err)) { fprintf(io.err, "%s\n", err.c_str()); return 1; }
        for (int t = 0; t < K; t++) {
            if (m[(size_t)t] != 0 && m[(size_t)t] != 1) { fprintf(io.err, "File %s holds a value other than 0 or 1\n", path.c_str()); return 1; }
            msg[f * kw + (size_t)t / 32] |= (uint32_t)m[(size_t)t] << (t % 32);
        }
    }
    if (a.device < 0) { fprintf(io.err, "ldpc: --device must be >= 0\n"); return 1; }
    if (!resident && getenv("CUDA_VISIBLE_DEVICES") == nullptr) {  // as for decoding: initialise only the requested GPU
        char dev[16];
        snprintf(dev, sizeof(dev), "%d", a.device);
        if (setenv("CUDA_VISIBLE_DEVICES", dev, 0) == 0) a.device = 0;
    }
    dnaldpc_config cfg{};
    cfg.n_devices = 1;
    cfg.devices[0] = a.device;
    cfg.wave_frames = 32;
    auto i0 = std::chrono::steady_clock::now();
    if (dnaldpc_decoder_create(code, &cfg, &dec) != DNALDPC_OK) { fprintf(io.err, "%s\n", dnaldpc_last_error()); return 1; }
    auto c0 = std::chrono::steady_clock::now();
    if (dnaldpc_encode(dec, msg.data(), (int64_t)F, cw.data()) != DNALDPC_OK) { fprintf(io.err, "%s\n", dnaldpc_last_error()); return 1; }
    auto c1 = std::chrono::steady_clock::now();
    std::vector<unsigned char> bits((size_t)N);
    for (size_t f = 0; f < F; f++) {
        for (int j = 0; j < N; j++) bits[(size_t)j] = (unsigned char)((cw[f * wpf + (size_t)j / 32] >> (j % 32)) & 1u);
        if (!write_dec_txt(io.path(frames[f].second + ".txt"), bits.data(), N, err)) { fprintf(io.err, "%s\n", err.c_str()); return 1; }
    }
    fprintf(io.out, "encoded %zu frame(s): N = %d, K = %d, M = %d\n", F, N, K, M);
    if (a.timing)
        fprintf(io.err, "{\"frames\": %zu, \"gpu_init_ms\": %.1f, \"encode_ms\": %.3f}\n", F,
                std::chrono::duration<double, std::milli>(c0 - i0).count(), std::chrono::duration<double, std::milli>(c1 - c0).count());
    return 0;
}

// ldpc --simulate: one dnaldpc_simulate call per channel parameter.
const char kSimUsage[] =
    "usage: ldpc --simulate <pchk_base> <channel_type> <p1[,p2,...]> <seed> <max_iter> <frame_num> [<target_frame_err> if frame_num==0]\n"
    "                       [--max-frames N] [--reads R] [--decoder 0|20] [--layered [--scale A]] [--device N] [--gpus N] [--fp32] [--timing]\n"
    "  channel_type 0: AWGN, parameters Eb/N0 in dB, sigma from the true rate K/N (K = N - rank(H))\n"
    "               1: BSC, parameters crossover probabilities p\n"
    "               3: vote counts, parameters read error probabilities, --reads = mean reads per bit (required)\n";

bool parse_num(const std::string &s, double &v) {
    char *end = nullptr;
    v = strtod(s.c_str(), &end);
    return !s.empty() && end && *end == 0 && std::isfinite(v);
}
bool parse_int(const std::string &s, long long &v) {
    char *end = nullptr;
    v = strtoll(s.c_str(), &end, 10);
    return !s.empty() && end && *end == 0;
}

int run_simulate(Args a, Io &io, bool resident) {
    auto usage = [&](const char *why) {
        if (why) fprintf(io.err, "ldpc --simulate: %s\n", why);
        fputs(kSimUsage, io.err);
        return 1;
    };
    const std::vector<std::string> &p = a.sim_pos;
    if (p.size() < 6) return usage("too few arguments");
    long long chan = 0, seed = 0, max_iter = 0, frame_num = 0, target = 0, max_frames = 1000000000LL;
    if (!parse_int(p[1], chan)) return usage("channel_type is not an integer");
    if (chan == 2) { fprintf(io.err, "ldpc --simulate: channel type 2 (BEC) is not supported by this build (0 = AWGN, 1 = BSC, 3 = vote counts)\n"); return 1; }
    if (chan != 0 && chan != 1 && chan != 3) { fprintf(io.err, "ldpc --simulate: unknown channel type %lld (0 = AWGN, 1 = BSC, 3 = vote counts)\n", chan); return 1; }
    if (!parse_int(p[3], seed) || seed < 0) return usage("seed must be a non-negative integer");
    if (!parse_int(p[4], max_iter) || max_iter < 0 || max_iter > 0x7fffffff) return usage("max_iter must be a non-negative integer");
    if (!parse_int(p[5], frame_num) || frame_num < 0) return usage("frame_num must be a non-negative integer");
    if (frame_num == 0) {
        if (p.size() != 7) return usage(p.size() < 7 ? "frame_num 0 needs <target_frame_err>" : "too many arguments");
        if (!parse_int(p[6], target) || target < 1) return usage("target_frame_err must be a positive integer");
        if (!a.max_frames.empty() && (!parse_int(a.max_frames, max_frames) || max_frames < 1)) return usage("--max-frames must be a positive integer");
    } else if (p.size() != 6) return usage("too many arguments");
    std::vector<double> params;
    {
        size_t b = 0;
        for (;;) {
            const size_t e = p[2].find(',', b);
            double v = 0;
            if (!parse_num(p[2].substr(b, e == std::string::npos ? std::string::npos : e - b), v)) return usage("bad channel parameter list");
            if (chan != 0 && !(v > 0.0 && v < 1.0)) { fprintf(io.err, "ldpc --simulate: error probability %g is not in (0,1)\n", v); return 1; }
            params.push_back(v);
            if (e == std::string::npos) break;
            b = e + 1;
        }
    }
    double reads = 0;
    if (chan == 3) {
        if (a.reads.empty()) return usage("channel type 3 (vote counts) needs --reads R");
        if (!parse_num(a.reads, reads) || !(reads > 0.0 && reads <= 32.0)) return usage("--reads must be in (0, 32]");
    }
    int flags = 0;
    if (!a.decoder.empty() && a.decoder != "0") {
        if (a.decoder != "20") return usage("--decoder must be 0 (belief propagation) or 20 (floating min-sum)");
        flags = DNALDPC_FLAG_MINSUM;
    }
    double alpha = 1.0;
    {
        const std::string why = check_layered(a, flags != 0, alpha);
        if (!why.empty()) return usage(why.c_str());
    }
    if (a.layered) flags |= DNALDPC_FLAG_LAYERED;
    if (a.device < 0) return usage("--device must be >= 0");
    if (a.gpus < 1 || a.gpus > 16) return usage("--gpus must be between 1 and 16");

    const std::string pchk_file = p[0] + ".pchk";
    dnaldpc_code *code = nullptr;
    dnaldpc_decoder *dec = nullptr;
    struct Owned {
        dnaldpc_code *&code; dnaldpc_decoder *&dec;
        ~Owned() { if (dec) dnaldpc_decoder_destroy(dec); if (code) dnaldpc_code_free(code); }
    } owned{code, dec};
    if (dnaldpc_code_read_pchk(io.path(pchk_file).c_str(), &code) != DNALDPC_OK) { fprintf(io.err, "%s\n", dnaldpc_last_error()); return 1; }
    int M, N, E, K;
    dnaldpc_code_dims(code, &M, &N, &E);
    if (dnaldpc_code_systematic(code, &K, nullptr, nullptr) != DNALDPC_OK) { fprintf(io.err, "%s\n", dnaldpc_last_error()); return 1; }
    const double rate = (double)K / (double)N;

    if (!resident && a.gpus == 1 && getenv("CUDA_VISIBLE_DEVICES") == nullptr) {  // as for decoding: initialise only the requested GPU
        char dev[16];
        snprintf(dev, sizeof(dev), "%d", a.device);
        if (setenv("CUDA_VISIBLE_DEVICES", dev, 0) == 0) a.device = 0;
    }
    dnaldpc_config cfg{};
    cfg.n_devices = a.gpus;
    for (int k = 0; k < a.gpus; k++) cfg.devices[k] = a.device + k;
    cfg.precision = a.fp32 ? DNALDPC_PREC_F32 : DNALDPC_PREC_F64;
    if (dnaldpc_decoder_create(code, &cfg, &dec) != DNALDPC_OK || dnaldpc_set_minsum_scale(dec, alpha) != DNALDPC_OK) {
        fprintf(io.err, "%s\n", dnaldpc_last_error());
        return 1;
    }
    fprintf(io.out, "\ng_CODE_N : %d\ng_CODE_K : %d\ng_CODE_M : %d\n\n", N, K, M);
    for (size_t i = 0; i < params.size(); i++) {
        dnaldpc_sim sp{};
        sp.channel = chan == 0 ? DNALDPC_IN_AWGN_F32 : chan == 1 ? DNALDPC_IN_BSC_BITS : DNALDPC_IN_VOTE_I8;
        sp.flags = flags;
        sp.param = chan == 0 ? dnaldpc_std_dev(params[i], rate) : params[i];
        sp.mean_reads = reads;
        sp.seed = (uint64_t)seed;
        sp.max_iter = (int32_t)max_iter;
        sp.max_frames = frame_num > 0 ? frame_num : max_frames;
        sp.target_frame_errors = frame_num > 0 ? 0 : target;
        dnaldpc_sim_result r{};
        const auto t0 = std::chrono::steady_clock::now();
        if (dnaldpc_simulate(dec, &sp, &r) != DNALDPC_OK) { fprintf(io.err, "%s\n", dnaldpc_last_error()); return 1; }
        const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        // Print_One_Result (DNA_main.cpp:1170-1182) and the counters the reference does not have
        const int k = (int)i;
        if (chan == 0) fprintf(io.out, "[%d]  code : (%d,%d)\trate : %.3f\tEb/No : %.2f dB\n", k, N, K, rate, params[i]);
        else fprintf(io.out, "[%d]  code : (%d,%d)\trate : %.3f\tp : %.5f\n", k, N, K, rate, params[i]);
        fprintf(io.out, "[%d]  frame_num              : %lld\n", k, (long long)r.frames);
        fprintf(io.out, "[%d]  bit_err                : %lld\n", k, (long long)r.bit_errors);
        fprintf(io.out, "[%d]  frame_err              : %lld\n", k, (long long)r.frame_errors);
        fprintf(io.out, "[%d]  without coding (bit)   : %lld\n", k, (long long)r.raw_bit_errors);
        fprintf(io.out, "[%d]  without coding (frame) : %lld\n", k, (long long)r.raw_frame_errors);
        fprintf(io.out, "[%d]  msg_bit_err            : %lld\n", k, (long long)r.msg_bit_errors);
        fprintf(io.out, "[%d]  undetected             : %lld\n", k, (long long)r.undetected);
        fprintf(io.out, "[%d]  avg_iter               : %.4f\n\n", k, r.frames ? (double)r.iterations / (double)r.frames : 0.0);
        fflush(io.out);
        if (a.timing)
            fprintf(io.err, "{\"point\": %d, \"channel_type\": %lld, \"param\": %.17g, \"channel_param\": %.17g, \"frames\": %lld, "
                    "\"iterations\": %lld, \"frame_errors\": %lld, \"bit_errors\": %lld, \"msg_frame_errors\": %lld, \"msg_bit_errors\": %lld, "
                    "\"detected\": %lld, \"undetected\": %lld, \"raw_frame_errors\": %lld, \"raw_bit_errors\": %lld, \"wall_ms\": %.3f}\n",
                    k, chan, params[i], sp.param, (long long)r.frames, (long long)r.iterations, (long long)r.frame_errors,
                    (long long)r.bit_errors, (long long)r.msg_frame_errors, (long long)r.msg_bit_errors, (long long)r.detected,
                    (long long)r.undetected, (long long)r.raw_frame_errors, (long long)r.raw_bit_errors, ms);
    }
    return 0;
}

// ---- resident worker and its client ----------------------------------------------------------------------------
// Wire format (host byte order, one request per connection): u32 magic, u32 argc, argc x (u32 length, bytes), u32 length +
// bytes of the client's working directory; answer: i32 exit code, u32 length + bytes of stdout, u32 length + bytes of stderr.
constexpr uint32_t kMagic = 0x4C445043u;  // "LDPC"

bool write_all(int fd, const void *p, size_t n) {
    const char *c = (const char *)p;
    while (n) {
        const ssize_t w = write(fd, c, n);
        if (w <= 0) { if (w < 0 && errno == EINTR) continue; return false; }
        c += w; n -= (size_t)w;
    }
    return true;
}
bool read_all(int fd, void *p, size_t n) {
    char *c = (char *)p;
    while (n) {
        const ssize_t r = read(fd, c, n);
        if (r <= 0) { if (r < 0 && errno == EINTR) continue; return false; }
        c += r; n -= (size_t)r;
    }
    return true;
}
bool send_str(int fd, const std::string &s) {
    const uint32_t n = (uint32_t)s.size();
    return write_all(fd, &n, 4) && write_all(fd, s.data(), n);
}
bool recv_str(int fd, std::string &s) {
    uint32_t n = 0;
    if (!read_all(fd, &n, 4) || n > (64u << 20)) return false;
    s.resize(n);
    return n == 0 || read_all(fd, &s[0], n);
}
bool make_addr(const std::string &path, sockaddr_un &addr) {
    memset(&addr, 0, sizeof(addr));
    addr.sun_family = AF_UNIX;
    if (path.empty() || path.size() >= sizeof(addr.sun_path)) return false;
    memcpy(addr.sun_path, path.c_str(), path.size());
    return true;
}

// Client side: true when a worker took the command line (its exit code in *rc), false = run locally.
bool run_remote(const std::string &sock, const std::vector<std::string> &args, int *rc) {
    sockaddr_un addr;
    if (!make_addr(sock, addr)) return false;
    const int fd = socket(AF_UNIX, SOCK_STREAM, 0);
    if (fd < 0) return false;
    if (connect(fd, (sockaddr *)&addr, sizeof(addr)) != 0) { close(fd); return false; }
    char cwd[4096];
    if (!getcwd(cwd, sizeof(cwd))) cwd[0] = 0;
    const uint32_t argc = (uint32_t)args.size();
    bool ok = write_all(fd, &kMagic, 4) && write_all(fd, &argc, 4);
    for (const std::string &a : args) ok = ok && send_str(fd, a);
    ok = ok && send_str(fd, cwd);
    int32_t code = 1;
    std::string out, err;
    ok = ok && read_all(fd, &code, 4) && recv_str(fd, out) && recv_str(fd, err);
    close(fd);
    if (!ok) return false;  // nothing has been printed yet: the local run starts from scratch
    fwrite(out.data(), 1, out.size(), stdout);
    fwrite(err.data(), 1, err.size(), stderr);
    *rc = code;
    return true;
}

int serve(const std::string &sock) {
    sockaddr_un addr;
    if (!make_addr(sock, addr)) { fprintf(stderr, "ldpc --serve: set DNALDPC_SOCKET or pass --socket PATH (at most %zu characters)\n", sizeof(addr.sun_path) - 1); return 1; }
    signal(SIGPIPE, SIG_IGN);
    const int ls = socket(AF_UNIX, SOCK_STREAM, 0);
    if (ls < 0) { perror("socket"); return 1; }
    unlink(sock.c_str());
    if (bind(ls, (sockaddr *)&addr, sizeof(addr)) != 0 || listen(ls, 64) != 0) { perror("ldpc --serve: bind/listen"); return 1; }
    fprintf(stderr, "ldpc: serving on %s\n", sock.c_str());
    Cache cache;
    bool stop = false;
    while (!stop) {
        const int fd = accept(ls, nullptr, nullptr);
        if (fd < 0) { if (errno == EINTR) continue; break; }
        uint32_t magic = 0, argc = 0;
        std::vector<std::string> args;
        std::string cwd;
        bool ok = read_all(fd, &magic, 4) && magic == kMagic && read_all(fd, &argc, 4) && argc < 4096;
        for (uint32_t i = 0; ok && i < argc; i++) { std::string a; ok = recv_str(fd, a); args.push_back(a); }
        ok = ok && recv_str(fd, cwd);
        if (ok) {
            char *ob = nullptr, *eb = nullptr;
            size_t on = 0, en = 0;
            Io io;
            io.out = open_memstream(&ob, &on);
            io.err = open_memstream(&eb, &en);
            Args a;
            int32_t code = 1;
            // one request at a time, so the worker simply moves into the client's directory: relative file names and
            // the messages that quote them come out exactly as in a local run
            if (chdir(cwd.c_str()) != 0) fprintf(io.err, "ldpc worker: can't enter %s\n", cwd.c_str());
            else if (parse(args, a, io)) {
                if (a.shutdown) { stop = true; code = 0; }
                else if (a.serve) { fprintf(io.err, "ldpc: a worker is already serving on this socket\n"); }
                else code = a.encode ? run_encode(a, io, true) : a.simulate ? run_simulate(a, io, true) : run(a, io, &cache);
            }
            fclose(io.out);
            fclose(io.err);
            write_all(fd, &code, 4) && send_str(fd, std::string(ob, on)) && send_str(fd, std::string(eb, en));
            free(ob);
            free(eb);
        }
        close(fd);
    }
    close(ls);
    unlink(sock.c_str());
    for (auto &kv : cache.map) { dnaldpc_decoder_destroy(kv.second.dec); dnaldpc_code_free(kv.second.code); }
    return 0;
}

}  // namespace

int main(int argc, char **argv) {
    std::vector<std::string> args(argv + 1, argv + argc);
    Args a;
    Io io;
    if (!parse(args, a, io)) return 1;
    std::string sock = a.socket_path;
    if (sock.empty() && getenv("DNALDPC_SOCKET")) sock = getenv("DNALDPC_SOCKET");
    if (a.serve) return serve(sock);
    if (!sock.empty()) {  // a resident worker takes the command line when one answers
        int rc = 1;
        if (run_remote(sock, args, &rc)) return rc;
        if (a.shutdown) { fprintf(stderr, "ldpc: no worker answers on %s\n", sock.c_str()); return 1; }
    } else if (a.shutdown) { fprintf(stderr, "ldpc --shutdown: set DNALDPC_SOCKET or pass --socket PATH\n"); return 1; }
    return a.encode ? run_encode(a, io, false) : a.simulate ? run_simulate(a, io, false) : run(a, io, nullptr);
}
