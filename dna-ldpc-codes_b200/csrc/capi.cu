// capi.cu - the C ABI of include/dnaldpc.h over Code (host/code.h) and Engine (engine.h).
#include <cuda_runtime.h>

#include <cmath>
#include <cstring>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "../../include/dnaldpc.h"
#include "../host/code.h"
#include "../host/layers.h"
#include "../host/systematic.h"
#include "encoder.h"
#include "engine.h"
#include "sim.h"
#include "sources.h"

using namespace dnaldpc;

struct dnaldpc_code {
    Code c;
};
struct dnaldpc_decoder {
    Code c;
    std::vector<std::unique_ptr<Engine>> eng;
    dnaldpc_stats stats{};
    std::unique_ptr<Encoder> enc;  // on eng[0]'s device, created by the first encode / extract call
    std::vector<std::unique_ptr<Encoder>> sim_enc;  // on eng[1..]'s devices, created by the first multi-GPU simulation
};

// Every entry point leaves the calling thread's current CUDA device as it found it (the engines switch devices).
struct DeviceRestore {
    int dev = -1;
    DeviceRestore() { if (cudaGetDevice(&dev) != cudaSuccess) { dev = -1; cudaGetLastError(); } }
    ~DeviceRestore() { if (dev >= 0) cudaSetDevice(dev); }
};

static thread_local std::string g_err;
static int set_err(int rc, const std::string &m) {
    g_err = m;
    return rc;
}

extern "C" {

const char *dnaldpc_last_error(void) { return g_err.c_str(); }
const char *dnaldpc_version(void) { return "dnaldpc-b200 0.1 (sm_100a)"; }

int dnaldpc_code_read_pchk(const char *path, dnaldpc_code **out) {
    if (!path || !out) return set_err(DNALDPC_ERR_ARG, "null argument");
    std::unique_ptr<dnaldpc_code> h(new dnaldpc_code);
    std::string err;
    int rc = read_pchk(path, h->c, err);
    if (rc) return set_err(rc == 2 ? DNALDPC_ERR_IO : DNALDPC_ERR_FORMAT, err);
    *out = h.release();
    return DNALDPC_OK;
}

int dnaldpc_code_from_csr(int M, int N, int E, const int32_t *row_ptr, const int32_t *col_idx, dnaldpc_code **out) {
    if (!row_ptr || (E > 0 && !col_idx) || !out || M <= 0 || N <= 0 || E < 0) return set_err(DNALDPC_ERR_ARG, "bad argument");
    if (row_ptr[0] != 0 || row_ptr[M] != E) return set_err(DNALDPC_ERR_ARG, "row_ptr does not span [0, E]");
    std::vector<int64_t> pairs;
    pairs.reserve((size_t)E);
    for (int i = 0; i < M; i++) {
        if (row_ptr[i + 1] < row_ptr[i]) return set_err(DNALDPC_ERR_ARG, "row_ptr not monotone");
        for (int e = row_ptr[i]; e < row_ptr[i + 1]; e++) {
            if (col_idx[e] < 0 || col_idx[e] >= N) return set_err(DNALDPC_ERR_ARG, "column index out of range");
            pairs.push_back(((int64_t)i << 32) | (uint32_t)col_idx[e]);
        }
    }
    std::unique_ptr<dnaldpc_code> h(new dnaldpc_code);
    std::string err = build_code(M, N, pairs, h->c);
    if (!err.empty()) return set_err(DNALDPC_ERR_ARG, err);
    *out = h.release();
    return DNALDPC_OK;
}

int dnaldpc_code_write_pchk(const dnaldpc_code *c, const char *path) {
    if (!c || !path) return set_err(DNALDPC_ERR_ARG, "null argument");
    std::string err;
    int rc = write_pchk(path, c->c, err);
    return rc ? set_err(DNALDPC_ERR_IO, err) : DNALDPC_OK;
}

void dnaldpc_code_free(dnaldpc_code *c) { delete c; }

int dnaldpc_code_dims(const dnaldpc_code *c, int *M, int *N, int *E) {
    if (!c) return set_err(DNALDPC_ERR_ARG, "null code");
    if (M) *M = c->c.M;
    if (N) *N = c->c.N;
    if (E) *E = c->c.E;
    return DNALDPC_OK;
}

int dnaldpc_code_export(const dnaldpc_code *c, int32_t *row_ptr, int32_t *col_idx, int32_t *col_ptr, int32_t *col_edge) {
    if (!c) return set_err(DNALDPC_ERR_ARG, "null code");
    const Code &k = c->c;
    if (row_ptr) memcpy(row_ptr, k.row_ptr.data(), k.row_ptr.size() * 4);
    if (col_idx) memcpy(col_idx, k.col_idx.data(), k.col_idx.size() * 4);
    if (col_ptr) memcpy(col_ptr, k.col_ptr.data(), k.col_ptr.size() * 4);
    if (col_edge) memcpy(col_edge, k.col_edge.data(), k.col_edge.size() * 4);
    return DNALDPC_OK;
}

int dnaldpc_code_check_regular(const dnaldpc_code *c, int *dv, int *regular_dv, int *dc, int *regular_dc) {
    if (!c) return set_err(DNALDPC_ERR_ARG, "null code");
    int a, b, x, y;
    check_regular(c->c, a, b, x, y);
    if (dv) *dv = a;
    if (regular_dv) *regular_dv = b;
    if (dc) *dc = x;
    if (regular_dc) *regular_dc = y;
    return DNALDPC_OK;
}

int dnaldpc_code_layers(const dnaldpc_code *c, int *n_layers, int32_t *layer_of_row) {
    if (!c || !n_layers) return set_err(DNALDPC_ERR_ARG, "null argument");
    const Layers &l = code_layers(c->c);
    *n_layers = l.n_layers;
    if (layer_of_row) memcpy(layer_of_row, l.layer_of_row.data(), l.layer_of_row.size() * 4);
    return DNALDPC_OK;
}

int dnaldpc_decoder_create(const dnaldpc_code *c, const dnaldpc_config *cfg, dnaldpc_decoder **out) {
    DeviceRestore restore_device;
    if (!c || !out) return set_err(DNALDPC_ERR_ARG, "null argument");
    dnaldpc_config k{};
    if (cfg) k = *cfg;
    if (k.n_devices < 0 || k.n_devices > 16) return set_err(DNALDPC_ERR_ARG, "n_devices out of range");
    if (k.precision != DNALDPC_PREC_F64 && k.precision != DNALDPC_PREC_F32) return set_err(DNALDPC_ERR_ARG, "unknown precision");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return set_err(DNALDPC_ERR_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(e) +
                                             " (this decoder has no CPU fallback)");
    std::vector<int> devs;
    if (k.n_devices == 0) {
        int cur = 0;
        cudaGetDevice(&cur);
        devs.push_back(cur);
    } else {
        for (int i = 0; i < k.n_devices; i++) {
            if (k.devices[i] < 0 || k.devices[i] >= ndev) return set_err(DNALDPC_ERR_ARG, "device ordinal out of range");
            devs.push_back(k.devices[i]);
        }
    }
    std::unique_ptr<dnaldpc_decoder> d(new dnaldpc_decoder);
    d->c = c->c;
    for (int dev : devs) {
        d->eng.emplace_back(new Engine(d->c, dev, k.precision, k.wave_frames));
        if (!d->eng.back()->ok()) {
            const std::string &m = d->eng.back()->error();
            return set_err(m.rfind("unsupported", 0) == 0 ? DNALDPC_ERR_UNSUPPORTED : DNALDPC_ERR_CUDA, m);
        }
    }
    *out = d.release();
    return DNALDPC_OK;
}

void dnaldpc_decoder_destroy(dnaldpc_decoder *d) {
    DeviceRestore restore_device;
    delete d;
}

int dnaldpc_set_minsum_scale(dnaldpc_decoder *d, double alpha) {
    if (!d) return set_err(DNALDPC_ERR_ARG, "null decoder");
    if (!(alpha > 0.0 && alpha <= 1.0)) return set_err(DNALDPC_ERR_ARG, "min-sum scale must be in (0, 1]");
    for (auto &e : d->eng) e->minsum_scale = alpha;
    return DNALDPC_OK;
}

// DNALDPC_FLAG_LAYERED exists for min-sum only (a layered sum-product is not implemented).
static int check_layered(int flags) {
    if ((flags & DNALDPC_FLAG_LAYERED) && !(flags & DNALDPC_FLAG_MINSUM))
        return set_err(DNALDPC_ERR_UNSUPPORTED, "DNALDPC_FLAG_LAYERED needs DNALDPC_FLAG_MINSUM (no layered sum-product)");
    return DNALDPC_OK;
}

static int check_input(const dnaldpc_input *in, int N) {
    if (!in) return set_err(DNALDPC_ERR_ARG, "null input descriptor");
    if (packed_stride(in->kind, N) == 0) return set_err(DNALDPC_ERR_ARG, "unknown input kind");
    if (in->kind == DNALDPC_IN_BSC_BITS && !(in->param > 0.0 && in->param < 1.0))
        return set_err(DNALDPC_ERR_ARG, "BSC crossover probability must be in (0,1)");
    if ((in->kind == DNALDPC_IN_AWGN_F32 || in->kind == DNALDPC_IN_AWGN_F64) && !(in->param > 0.0))
        return set_err(DNALDPC_ERR_ARG, "AWGN sigma must be positive");
    if (in->kind == DNALDPC_IN_VOTE_I8 && !in->table && !(in->param > 0.0 && in->param < 1.0))
        return set_err(DNALDPC_ERR_ARG, "vote-count eps must be in (0,1)");
    return check_layered(in->flags);
}

int dnaldpc_decode_batch(dnaldpc_decoder *d, const dnaldpc_input *in, int64_t F, int max_iter, const dnaldpc_output *out) {
    DeviceRestore restore_device;
    if (!d || !out) return set_err(DNALDPC_ERR_ARG, "null argument");
    int rc = check_input(in, d->c.N);
    if (rc) return rc;
    if (F < 0 || max_iter < 0) return set_err(DNALDPC_ERR_ARG, "negative frame count or max_iter");
    if (F > 0 && !in->data) return set_err(DNALDPC_ERR_ARG, "null input buffer");
    std::string err;
    rc = decode_host_batch(d->eng, *in, F, max_iter, *out, d->stats, err);
    return rc ? set_err(rc, err) : DNALDPC_OK;
}

int dnaldpc_decode_batch_device(dnaldpc_decoder *d, const dnaldpc_input *in, int64_t F, int max_iter,
                                const dnaldpc_output *out, void *stream) {
    DeviceRestore restore_device;
    if (!d || !out) return set_err(DNALDPC_ERR_ARG, "null argument");
    int rc = check_input(in, d->c.N);
    if (rc) return rc;
    if (F < 0 || max_iter < 0) return set_err(DNALDPC_ERR_ARG, "negative frame count or max_iter");
    if (F > 0 && !in->data) return set_err(DNALDPC_ERR_ARG, "null input buffer");
    if (in->flags & DNALDPC_FLAG_HOST_EXP) return set_err(DNALDPC_ERR_ARG, "HOST_EXP needs host buffers");
    std::string err;
    rc = decode_device_batch(d->eng, *in, F, max_iter, *out, (cudaStream_t)stream, d->stats, err);
    return rc ? set_err(rc, err) : DNALDPC_OK;
}

int dnaldpc_decode_window(dnaldpc_decoder *d, const dnaldpc_window *win, const double *lratio, int64_t F, int max_iter,
                          const dnaldpc_output *out) {
    DeviceRestore restore_device;
    if (!d || !win || !out) return set_err(DNALDPC_ERR_ARG, "null argument");
    // Frames are independent (DNA_main.cpp:629-651 splits them over ranks): with several devices every engine decodes
    // a contiguous share of the batch on its own thread, no exchange between them.
    const int nd = (int)std::min<int64_t>((int64_t)d->eng.size(), std::max<int64_t>(1, F / 64));
    if (nd <= 1) {
        const int rc = d->eng[0]->decode_window_host(d->c, *win, lratio, F, max_iter, *out);
        if (rc) return set_err(rc, d->eng[0]->error());
        d->stats = d->eng[0]->stats;
        return DNALDPC_OK;
    }
    const int N = d->c.N, M = d->c.M;
    const size_t wpf = (size_t)(N + 31) / 32;
    const int64_t share = ((F + nd - 1) / nd + 31) / 32 * 32;
    std::vector<int> rcs((size_t)nd, DNALDPC_OK);
    auto run = [&](int k) {
        const int64_t f0 = std::min<int64_t>(F, share * k), nf = std::min<int64_t>(share, F - f0);
        if (nf <= 0) { d->eng[(size_t)k]->stats = dnaldpc_stats{}; return; }
        dnaldpc_output o = *out;
        if (o.bits) o.bits += (size_t)f0 * wpf;
        if (o.dblk) o.dblk += (size_t)f0 * N;
        if (o.pchk) o.pchk += (size_t)f0 * M;
        if (o.iters) o.iters += f0;
        if (o.is_codeword) o.is_codeword += f0;
        rcs[(size_t)k] = d->eng[(size_t)k]->decode_window_host(d->c, *win, lratio + (size_t)f0 * N, nf, max_iter, o);
    };
    std::vector<std::thread> th;
    for (int k = 1; k < nd; k++) th.emplace_back(run, k);
    run(0);
    for (auto &t : th) t.join();
    d->stats = dnaldpc_stats{};
    for (int k = 0; k < nd; k++) {
        if (rcs[(size_t)k]) return set_err(rcs[(size_t)k], d->eng[(size_t)k]->error());
        const dnaldpc_stats &e = d->eng[(size_t)k]->stats;
        d->stats.frames += e.frames; d->stats.frame_iters += e.frame_iters; d->stats.kernel_launches += e.kernel_launches;
        d->stats.waves += e.waves;
    }
    return DNALDPC_OK;
}

int dnaldpc_run_bp_decoder(dnaldpc_decoder *d, const double *lratio, int max_iter, char *dblk, char *pchk,
                           int *is_codeword, int *iters) {
    if (!d || !lratio || !dblk) return set_err(DNALDPC_ERR_ARG, "null argument");
    dnaldpc_input in{};
    in.kind = DNALDPC_IN_LR_F64;
    in.data = lratio;
    dnaldpc_output out{};
    int32_t n = 0;
    uint8_t ok = 0;
    out.dblk = (uint8_t *)dblk;
    out.pchk = (uint8_t *)pchk;
    out.iters = &n;
    out.is_codeword = &ok;
    int rc = dnaldpc_decode_batch(d, &in, 1, max_iter, &out);
    if (rc) return rc;
    if (iters) *iters = n;
    if (is_codeword) *is_codeword = ok;
    return DNALDPC_OK;
}

// The sweep with libm exp on the host (bit-exact with the reference's exe): the failed frames of a round are gathered
// on the host, exponentiated there and decoded as a fresh host batch.
static int sweep_host_exp(dnaldpc_decoder *d, const dnaldpc_input &in0, int64_t F, int max_iter, const double *params,
                          int n_params, const dnaldpc_output *out, int32_t *rounds) {
    const int M = d->c.M, N = d->c.N;
    const size_t wpf = (size_t)(N + 31) / 32;
    const size_t stride = in0.frame_stride ? in0.frame_stride : (size_t)N * 8;
    std::vector<uint8_t> ok((size_t)F, 0);
    dnaldpc_input in = in0;
    in.param = params[0];
    dnaldpc_output o = *out;
    o.is_codeword = ok.data();
    int rc = dnaldpc_decode_batch(d, &in, F, max_iter, &o);  // round 0: every frame
    if (rc) return rc;
    if (rounds) for (int64_t f = 0; f < F; f++) rounds[f] = 0;
    dnaldpc_stats total = d->stats;
    std::vector<int64_t> failed;
    for (int r = 1; r < n_params; r++) {
        failed.clear();
        for (int64_t f = 0; f < F; f++) if (!ok[(size_t)f]) failed.push_back(f);
        if (failed.empty()) break;
        const size_t K = failed.size();
        std::vector<double> sub(K * (size_t)N);
        for (size_t k = 0; k < K; k++) memcpy(&sub[k * (size_t)N], (const char *)in0.data + (size_t)failed[k] * stride, (size_t)N * sizeof(double));
        std::vector<uint32_t> t_bits(out->bits ? K * wpf : 0);
        std::vector<uint8_t> t_dblk(out->dblk ? K * (size_t)N : 0), t_ok(K), t_pchk(out->pchk ? K * (size_t)M : 0);
        std::vector<int32_t> t_it(K);
        std::vector<double> t_post(out->posterior ? K * (size_t)N : 0);
        dnaldpc_input in2 = in;
        in2.data = sub.data();
        in2.frame_stride = 0;
        in2.param = params[r];
        dnaldpc_output o2{};
        o2.bits = out->bits ? t_bits.data() : nullptr;
        o2.dblk = out->dblk ? t_dblk.data() : nullptr;
        o2.iters = t_it.data();
        o2.is_codeword = t_ok.data();
        o2.posterior = out->posterior ? t_post.data() : nullptr;
        o2.pchk = out->pchk ? t_pchk.data() : nullptr;
        rc = dnaldpc_decode_batch(d, &in2, (int64_t)K, max_iter, &o2);
        if (rc) return rc;
        for (size_t k = 0; k < K; k++) {  // a frame keeps the result of its last round
            const size_t f = (size_t)failed[k];
            if (out->bits) memcpy(out->bits + f * wpf, &t_bits[k * wpf], wpf * 4);
            if (out->dblk) memcpy(out->dblk + f * N, &t_dblk[k * (size_t)N], (size_t)N);
            if (out->iters) out->iters[f] = t_it[k];
            if (out->posterior) memcpy(out->posterior + f * N, &t_post[k * (size_t)N], (size_t)N * 8);
            if (out->pchk) memcpy(out->pchk + f * M, &t_pchk[k * (size_t)M], (size_t)M);
            ok[f] = t_ok[k];
            if (rounds) rounds[f] = r;
        }
        total.frames += d->stats.frames; total.frame_iters += d->stats.frame_iters;
        total.kernel_launches += d->stats.kernel_launches; total.waves += d->stats.waves;
        total.compactions += d->stats.compactions;
    }
    if (out->is_codeword) memcpy(out->is_codeword, ok.data(), (size_t)F);
    d->stats = total;
    return DNALDPC_OK;
}

int dnaldpc_redecode_sweep_ex(dnaldpc_decoder *d, const dnaldpc_input *in, int64_t F, int max_iter, const double *params,
                              int n_params, const dnaldpc_output *out, int32_t *rounds) {
    DeviceRestore restore_device;
    if (!d || !in || !out || !params || n_params <= 0 || F < 0 || max_iter < 0) return set_err(DNALDPC_ERR_ARG, "bad argument");
    if (F > 0 && !in->data) return set_err(DNALDPC_ERR_ARG, "null input buffer");
    if (in->kind == DNALDPC_IN_LR_F64) return set_err(DNALDPC_ERR_ARG, "a sweep needs a parameter to vary: LR_F64 inputs have none");
    if (in->kind == DNALDPC_IN_VOTE_I8 && in->table) return set_err(DNALDPC_ERR_ARG, "a vote-count sweep builds its tables from params[]: table must be NULL");
    for (int r = 0; r < n_params; r++) {  // every round's parameter has to be valid for the kind
        dnaldpc_input t = *in;
        t.param = params[r];
        const int rc = check_input(&t, d->c.N);
        if (rc) return rc;
    }
    const bool host_exp = in->kind == DNALDPC_IN_LLR_F64 && (in->flags & DNALDPC_FLAG_HOST_EXP) && !(in->flags & DNALDPC_FLAG_MINSUM);
    if (host_exp) return sweep_host_exp(d, *in, F, max_iter, params, n_params, out, rounds);
    std::string err;
    const int rc = redecode_sweep_batch(d->eng, *in, F, max_iter, params, n_params, *out, rounds, d->stats, err);
    return rc ? set_err(rc, err) : DNALDPC_OK;
}

int dnaldpc_redecode_sweep(dnaldpc_decoder *d, const double *llr, int64_t F, int max_iter, const double *scales,
                           int n_scales, int flags, const dnaldpc_output *out, int32_t *rounds) {
    if (!d || !llr || !out || !scales || n_scales <= 0 || F < 0) return set_err(DNALDPC_ERR_ARG, "bad argument");
    dnaldpc_input in{};
    in.kind = DNALDPC_IN_LLR_F64;
    in.flags = flags & (DNALDPC_FLAG_HOST_EXP | DNALDPC_FLAG_FIXED_ITERS | DNALDPC_FLAG_MINSUM);
    in.data = llr;
    return dnaldpc_redecode_sweep_ex(d, &in, F, max_iter, scales, n_scales, out, rounds);
}

double dnaldpc_std_dev(double ebno_db, double rate) {  // channel.cpp:9-16
    const double enl = std::pow(10.0, ebno_db * 0.1);
    return 1 / std::sqrt(2 * rate * enl);
}

int dnaldpc_vote_table(double eps, double *t) {  // decoder.py:314 followed by DNA_main.cpp:1344
    if (!t || !(eps > 0.0 && eps < 1.0)) return set_err(DNALDPC_ERR_ARG, "bad argument");
    const double L = std::log((1 - eps) / eps);
    for (int k = -128; k < 128; k++) t[k + 128] = std::exp(k * L);
    return DNALDPC_OK;
}

int dnaldpc_bsc_table(double p, double *t) {  // channel.cpp:75-84
    if (!t || !(p > 0.0 && p < 1.0)) return set_err(DNALDPC_ERR_ARG, "bad argument");
    t[0] = (1 - p) / p;
    t[1] = p / (1 - p);
    return DNALDPC_OK;
}

int dnaldpc_synth_bsc_device(dnaldpc_decoder *d, const uint32_t *cw_bits, int n_cw, uint64_t seed, int64_t frame0,
                             int64_t F, double eps, uint32_t *out_bits, void *stream) {
    DeviceRestore restore_device;
    if (!d) return set_err(DNALDPC_ERR_ARG, "null decoder");
    int rc = d->eng[0]->synth_bsc(cw_bits, n_cw, seed, frame0, F, eps, out_bits, (cudaStream_t)stream);
    return rc ? set_err(rc, d->eng[0]->error()) : DNALDPC_OK;
}

int dnaldpc_synth_awgn_device(dnaldpc_decoder *d, const uint32_t *cw_bits, int n_cw, uint64_t seed, int64_t frame0,
                              int64_t F, double sigma, float *out_y, void *stream) {
    DeviceRestore restore_device;
    if (!d) return set_err(DNALDPC_ERR_ARG, "null decoder");
    int rc = d->eng[0]->synth_awgn(cw_bits, n_cw, seed, frame0, F, sigma, out_y, (cudaStream_t)stream);
    return rc ? set_err(rc, d->eng[0]->error()) : DNALDPC_OK;
}

int dnaldpc_synth_vote_device(dnaldpc_decoder *d, const uint32_t *cw_bits, int n_cw, uint64_t seed, int64_t frame0,
                              int64_t F, double mean_reads, double read_err, int8_t *out_k, void *stream) {
    DeviceRestore restore_device;
    if (!d) return set_err(DNALDPC_ERR_ARG, "null decoder");
    int rc = d->eng[0]->synth_vote(cw_bits, n_cw, seed, frame0, F, mean_reads, read_err, out_k, (cudaStream_t)stream);
    return rc ? set_err(rc, d->eng[0]->error()) : DNALDPC_OK;
}

int dnaldpc_code_systematic(const dnaldpc_code *c, int *K, int32_t *info_cols, int32_t *parity_cols) {
    if (!c || !K) return set_err(DNALDPC_ERR_ARG, "null argument");
    int rc = 0;
    std::string err;
    const Systematic *s = systematic_form(c->c, &rc, &err);
    if (!s) return set_err(rc, err);
    *K = s->K;
    if (info_cols) memcpy(info_cols, s->info_cols.data(), s->info_cols.size() * 4);
    if (parity_cols) memcpy(parity_cols, s->parity_cols.data(), s->parity_cols.size() * 4);
    return DNALDPC_OK;
}

// The decoder's encoder on its first device, created on first use.
static int first_encoder(dnaldpc_decoder *d) {
    if (!d->enc) {
        int rc = 0;
        std::string err;
        const Systematic *s = systematic_form(d->c, &rc, &err);
        if (!s) return set_err(rc, err);
        std::unique_ptr<Encoder> e(new Encoder(*s, d->c.N, d->eng[0]->device()));
        if (!e->ok()) return set_err(DNALDPC_ERR_CUDA, e->error());
        d->enc = std::move(e);
    }
    return DNALDPC_OK;
}

// Argument checks shared by the encode / extract entry points; *enc receives the decoder's encoder.
static int encoder_call(dnaldpc_decoder *d, const void *src, int64_t F, const void *dst, Encoder **enc) {
    *enc = nullptr;
    if (!d) return set_err(DNALDPC_ERR_ARG, "null decoder");
    if (F < 0) return set_err(DNALDPC_ERR_ARG, "negative frame count");
    if (F == 0) return DNALDPC_OK;
    if (!src || !dst) return set_err(DNALDPC_ERR_ARG, "null buffer");
    const int rc = first_encoder(d);
    if (rc) return rc;
    *enc = d->enc.get();
    return DNALDPC_OK;
}

int dnaldpc_encode_device(dnaldpc_decoder *d, const uint32_t *msg, int64_t F, uint32_t *cw, void *stream) {
    DeviceRestore restore_device;
    Encoder *e;
    int rc = encoder_call(d, msg, F, cw, &e);
    if (rc || !e) return rc;
    rc = e->encode(msg, F, cw, (cudaStream_t)stream);
    return rc ? set_err(rc, e->error()) : DNALDPC_OK;
}

int dnaldpc_encode(dnaldpc_decoder *d, const uint32_t *msg, int64_t F, uint32_t *cw) {
    DeviceRestore restore_device;
    Encoder *e;
    int rc = encoder_call(d, msg, F, cw, &e);
    if (rc || !e) return rc;
    rc = e->encode_host(msg, F, cw);
    return rc ? set_err(rc, e->error()) : DNALDPC_OK;
}

int dnaldpc_extract_device(dnaldpc_decoder *d, const uint32_t *cw, int64_t F, uint32_t *msg, void *stream) {
    DeviceRestore restore_device;
    Encoder *e;
    int rc = encoder_call(d, cw, F, msg, &e);
    if (rc || !e) return rc;
    rc = e->extract(cw, F, msg, (cudaStream_t)stream);
    return rc ? set_err(rc, e->error()) : DNALDPC_OK;
}

int dnaldpc_extract(dnaldpc_decoder *d, const uint32_t *cw, int64_t F, uint32_t *msg) {
    DeviceRestore restore_device;
    Encoder *e;
    int rc = encoder_call(d, cw, F, msg, &e);
    if (rc || !e) return rc;
    rc = e->extract_host(cw, F, msg);
    return rc ? set_err(rc, e->error()) : DNALDPC_OK;
}

int dnaldpc_simulate(dnaldpc_decoder *d, const dnaldpc_sim *s, dnaldpc_sim_result *r) {
    DeviceRestore restore_device;
    if (!d || !s || !r) return set_err(DNALDPC_ERR_ARG, "null argument");
    if (s->channel != DNALDPC_IN_BSC_BITS && s->channel != DNALDPC_IN_AWGN_F32 && s->channel != DNALDPC_IN_VOTE_I8)
        return set_err(DNALDPC_ERR_ARG, "unknown simulation channel (BSC_BITS, AWGN_F32 or VOTE_I8)");
    if (s->flags & ~(DNALDPC_FLAG_MINSUM | DNALDPC_FLAG_FIXED_ITERS | DNALDPC_FLAG_LAYERED))
        return set_err(DNALDPC_ERR_ARG, "unknown simulation flag");
    if (int rc = check_layered(s->flags)) return rc;
    if ((s->channel == DNALDPC_IN_BSC_BITS || s->channel == DNALDPC_IN_VOTE_I8) && !(s->param > 0.0 && s->param < 1.0))
        return set_err(DNALDPC_ERR_ARG, "error probability must be in (0,1)");
    if (s->channel == DNALDPC_IN_AWGN_F32 && !(s->param > 0.0)) return set_err(DNALDPC_ERR_ARG, "AWGN sigma must be positive");
    if (s->channel == DNALDPC_IN_VOTE_I8 && !(s->mean_reads > 0.0 && s->mean_reads <= 32.0))
        return set_err(DNALDPC_ERR_ARG, "mean reads must be in (0, 32]");
    if (s->max_iter < 0 || s->max_frames < 1 || s->target_frame_errors < 0)
        return set_err(DNALDPC_ERR_ARG, "max_iter < 0, max_frames < 1 or target_frame_errors < 0");
    int rc = 0;
    std::string err;
    const Systematic *sys = systematic_form(d->c, &rc, &err);
    if (!sys) return set_err(rc, err);
    // every device encodes its own frames: engine 0 with the decoder's encoder, the others with encoders of their own
    rc = first_encoder(d);
    if (rc) return rc;
    std::vector<Encoder *> encs{d->enc.get()};
    for (size_t k = 1; k < d->eng.size(); k++) {
        if (d->sim_enc.size() < k) {
            std::unique_ptr<Encoder> e(new Encoder(*sys, d->c.N, d->eng[k]->device()));
            if (!e->ok()) return set_err(DNALDPC_ERR_CUDA, e->error());
            d->sim_enc.push_back(std::move(e));
        }
        encs.push_back(d->sim_enc[k - 1].get());
    }
    rc = simulate_batch(d->eng, encs, *sys, *s, *r, d->stats, err);
    return rc ? set_err(rc, err) : DNALDPC_OK;
}

int dnaldpc_get_stats(const dnaldpc_decoder *d, dnaldpc_stats *s) {
    if (!d || !s) return set_err(DNALDPC_ERR_ARG, "null argument");
    *s = d->stats;
    return DNALDPC_OK;
}

int dnaldpc_set_profiling(dnaldpc_decoder *d, int on) {
    if (!d) return set_err(DNALDPC_ERR_ARG, "null decoder");
    for (auto &e : d->eng) { e->profiling = on == 1; e->trace_ticks_ = on == 2 ? 64 : 0; }
    return DNALDPC_OK;
}

int dnaldpc_get_trace(dnaldpc_decoder *d, double *row_ms, double *col_ms, double *sched_ms, int *ticks) {
    DeviceRestore restore_device;
    if (!d || !row_ms || !col_ms || !sched_ms) return set_err(DNALDPC_ERR_ARG, "null argument");
    const int n = d->eng[0]->trace_result(row_ms, col_ms, sched_ms);
    if (ticks) *ticks = n;
    return DNALDPC_OK;
}

int dnaldpc_selftest_math(int64_t n, uint64_t seed, int64_t *mismatches) {
    if (!mismatches || n < 0) return set_err(DNALDPC_ERR_ARG, "bad argument");
    std::string err;
    long long mm = 0;
    int rc = math_selftest(n, seed, &mm, err);
    if (rc) return set_err(rc, err);
    *mismatches = mm;
    return DNALDPC_OK;
}

}  // extern "C"
