// encoder.cu - systematic encoding P[F][R] = M[F][K] * A^T over GF(2) and bit placement (encode / extract).
//
// Parity kernel: a bit-packed GEMM whose multiply-add is one AND-XOR (LOP3.LUT 0x78) per 32 bit products. A CTA covers
// 128 frames x 128 parity rows; 32-word k-slices of the messages and of A are staged into shared memory with cp.async
// (two stages), and every thread keeps an 8 x 8 register tile of accumulators: per 2 k words it reads 16 x 8 bytes of
// shared memory and issues 128 LOP3. The parity of an accumulator's popcount is the parity bit.
// Placement kernel: one warp builds 32 output words at a time; lane l gathers bit l of each word through a per-column
// source table and __ballot_sync packs the bits. The same kernel with the inverse table extracts the message.
#include "encoder.h"

#include <algorithm>
#include <vector>

#include "../../include/dnaldpc.h"

namespace dnaldpc {

namespace {

constexpr int kBF = 128, kBR = 128, kBK = 32, kPad = 2, kThreads = 256;
// shared-memory row stride in words: the 8-byte reads of 16 rows tx + 16 j (tx = 0..15) start on banks 2 tx, no conflict
constexpr int kLd = kBK + kPad;
constexpr int kStageWords = (kBF + kBR) * kLd;
constexpr size_t kParitySmem = 2 * kStageWords * sizeof(uint32_t);

// Placement table entries: -1 = constant 0; otherwise word << 5 | bit of source row A, plus kSrcB for source row B.
constexpr int32_t kSrcB = 0x40000000;
constexpr int kPlaceFrames = 64, kPlaceWarps = 8;

__device__ __forceinline__ void cp_async8(uint32_t *dst, const uint32_t *src) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(d), "l"(src));
}
// 4-byte copy; src_bytes == 0 writes a zero word without reading `src`.
__device__ __forceinline__ void cp_async4(uint32_t *dst, const uint32_t *src, int src_bytes) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(d), "l"(src), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
__device__ __forceinline__ void cp_async_wait_1() { asm volatile("cp.async.wait_group 1;\n" ::); }
__device__ __forceinline__ void cp_async_wait_0() { asm volatile("cp.async.wait_group 0;\n" ::); }

// msg: [F][kw] (bits beyond K in the last word are multiplied by zero columns of A); A: [rpad][kwp], zero beyond R / K.
// par: [F][rpad / 32], bit r of frame f = parity row r. grid = (rpad / 128, ceil(F / 128)).
__global__ void __launch_bounds__(kThreads, 2)
encode_parity_kernel(const uint32_t *__restrict__ msg, long long F, int kw, const uint32_t *__restrict__ A, int kwp,
                     uint32_t *__restrict__ par, int par_words) {
    extern __shared__ __align__(16) uint32_t smem[];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int r0 = blockIdx.x * kBR;
    const long long f0 = (long long)blockIdx.y * kBF;
    const int ktiles = kwp / kBK;

    auto load = [&](int kt, int s) {
        uint32_t *sA = smem + s * kStageWords, *sM = sA + kBR * kLd;
#pragma unroll
        for (int q = 0; q < kBR * kBK / 2 / kThreads; q++) {  // A: 8-byte chunks, rows always in range (padded)
            const int idx = tid + q * kThreads, r = idx / (kBK / 2), c = idx % (kBK / 2);
            cp_async8(sA + r * kLd + c * 2, A + (size_t)(r0 + r) * kwp + (size_t)kt * kBK + c * 2);
        }
#pragma unroll
        for (int q = 0; q < kBF * kBK / kThreads; q++) {  // messages: words, a warp reads 32 consecutive words of a frame
            const int idx = tid + q * kThreads, fr = idx / kBK, k = idx % kBK;
            const long long f = f0 + fr;
            const int kg = kt * kBK + k;
            const bool in = f < F && kg < kw;
            cp_async4(sM + fr * kLd + k, in ? msg + (size_t)f * kw + kg : msg, in ? 4 : 0);
        }
    };

    uint32_t acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
        for (int j = 0; j < 8; j++) acc[i][j] = 0u;

    if (ktiles > 0) load(0, 0);
    cp_async_commit();
    for (int kt = 0; kt < ktiles; kt++) {
        const int s = kt & 1;
        if (kt + 1 < ktiles) load(kt + 1, s ^ 1);
        cp_async_commit();
        cp_async_wait_1();
        __syncthreads();
        const uint32_t *sA = smem + s * kStageWords, *sM = sA + kBR * kLd;
#pragma unroll
        for (int kk = 0; kk < kBK; kk += 2) {
            uint2 a[8];
#pragma unroll
            for (int j = 0; j < 8; j++) a[j] = *reinterpret_cast<const uint2 *>(sA + (tx + 16 * j) * kLd + kk);
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const uint2 m = *reinterpret_cast<const uint2 *>(sM + (ty + 16 * i) * kLd + kk);
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    uint32_t t = acc[i][j];
                    t ^= a[j].x & m.x;
                    t ^= a[j].y & m.y;
                    acc[i][j] = t;
                }
            }
        }
        __syncthreads();  // the stage read here is the one the next iteration refills
    }
    cp_async_wait_0();

    // Thread (tx, ty) holds rows tx + 16 j of frames ty + 16 i. Lanes 0-15 of a warp are one frame, lanes 16-31 the next:
    // word w of the tile (rows 32 w .. 32 w + 31) is j = 2 w in the low half and j = 2 w + 1 in the high half.
    const int lane = tid & 31;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const long long f = f0 + ty + 16 * i;
#pragma unroll
        for (int w = 0; w < 4; w++) {
            const unsigned b0 = __ballot_sync(0xffffffffu, __popc(acc[i][2 * w]) & 1);
            const unsigned b1 = __ballot_sync(0xffffffffu, __popc(acc[i][2 * w + 1]) & 1);
            const uint32_t word = lane == 0 ? (b0 & 0xffffu) | (b1 << 16) : (b0 >> 16) | (b1 & 0xffff0000u);
            if ((lane & 15) == 0 && f < F) par[(size_t)f * par_words + blockIdx.x * 4 + w] = word;
        }
    }
}

// out[f][w] for w < out_words: bit l = source bit table[w * 32 + l] (see kSrcB). grid = (ceil(out_words / 32),
// ceil(F / kPlaceFrames)), kPlaceWarps warps per block; each warp keeps the table entries of its 32 words in registers.
__global__ void __launch_bounds__(kPlaceWarps * 32)
place_bits_kernel(const uint32_t *__restrict__ srcA, long long strideA, const uint32_t *__restrict__ srcB, long long strideB,
                  const int32_t *__restrict__ table, int out_words, uint32_t *__restrict__ out, long long F) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int w0 = blockIdx.x * 32;
    int32_t ent[32];
#pragma unroll
    for (int i = 0; i < 32; i++) ent[i] = table[(size_t)(w0 + i) * 32 + lane];
    const long long fend = min(F, (long long)(blockIdx.y + 1) * kPlaceFrames);
    for (long long f = (long long)blockIdx.y * kPlaceFrames + warp; f < fend; f += kPlaceWarps) {
        const uint32_t *a = srcA + f * strideA, *b = srcB + f * strideB;
        uint32_t mine = 0;
#pragma unroll
        for (int i = 0; i < 32; i++) {
            const int32_t e = ent[i];
            unsigned v = 0;
            if (e >= 0) v = ((e & kSrcB) ? b : a)[(e & (kSrcB - 1)) >> 5] >> (e & 31) & 1u;
            const unsigned word = __ballot_sync(0xffffffffu, v);
            if (lane == i) mine = word;
        }
        if (w0 + lane < out_words) out[f * out_words + w0 + lane] = mine;
    }
}

int launch_place(const uint32_t *srcA, long long strideA, const uint32_t *srcB, long long strideB, const int32_t *table,
                 int out_words, uint32_t *out, long long F, cudaStream_t st) {
    if (out_words == 0 || F == 0) return 0;
    for (long long f0 = 0; f0 < F; f0 += 65535LL * kPlaceFrames) {  // grid.y limit
        const long long n = std::min(F - f0, 65535LL * kPlaceFrames);
        const dim3 grid((unsigned)((out_words + 31) / 32), (unsigned)((n + kPlaceFrames - 1) / kPlaceFrames));
        place_bits_kernel<<<grid, kPlaceWarps * 32, 0, st>>>(srcA + f0 * strideA, strideA, srcB ? srcB + f0 * strideB : nullptr,
                                                             strideB, table, out_words, out + f0 * out_words, n);
    }
    return 0;
}

}  // namespace

int Encoder::fail(cudaError_t e, const char *what) {
    err_ = std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what;
    return DNALDPC_ERR_CUDA;
}

#define CK(call)                                      \
    do {                                              \
        cudaError_t e_ = (call);                      \
        if (e_ != cudaSuccess) return fail(e_, #call); \
    } while (0)

Encoder::Encoder(const Systematic &s, int N, int device) : device_(device), N_(N), K_(s.K), R_(s.R), kw_(s.kw) {
    wpf_ = (N + 31) / 32;
    kwp_ = (kw_ + kBK - 1) / kBK * kBK;
    rpad_ = (R_ + kBR - 1) / kBR * kBR;
    auto chk = [&](cudaError_t e, const char *w) { if (e != cudaSuccess && err_.empty()) fail(e, w); };
    chk(cudaSetDevice(device_), "cudaSetDevice");
    if (!err_.empty()) return;
    // A, rows and words padded with zeros to whole tiles
    std::vector<uint32_t> a((size_t)rpad_ * kwp_, 0u);
    for (int i = 0; i < R_; i++)
        std::copy(s.A.begin() + (size_t)i * kw_, s.A.begin() + (size_t)(i + 1) * kw_, a.begin() + (size_t)i * kwp_);
    // codeword bit j <- message bit t (info column) or parity bit i (parity column); extraction: the inverse for info bits
    std::vector<int32_t> place((size_t)(wpf_ + 31) / 32 * 1024, -1), extract((size_t)(kw_ + 31) / 32 * 1024, -1);
    for (int t = 0; t < K_; t++) { place[(size_t)s.info_cols[(size_t)t]] = t; extract[(size_t)t] = s.info_cols[(size_t)t]; }
    for (int i = 0; i < R_; i++) place[(size_t)s.parity_cols[(size_t)i]] = kSrcB | i;
    auto up = [&](void **dst, const void *src, size_t bytes) {
        chk(cudaMalloc(dst, std::max<size_t>(bytes, 4)), "cudaMalloc(encoder tables)");
        if (err_.empty() && bytes) chk(cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice), "cudaMemcpy(encoder tables)");
    };
    up((void **)&d_A_, a.data(), a.size() * 4);
    up((void **)&d_place_, place.data(), place.size() * 4);
    up((void **)&d_extract_, extract.data(), extract.size() * 4);
    chk(cudaFuncSetAttribute(encode_parity_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kParitySmem),
        "cudaFuncSetAttribute(encode_parity_kernel)");
    chk(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking), "cudaStreamCreate");
}

Encoder::~Encoder() {
    if (cudaSetDevice(device_) != cudaSuccess) return;
    if (stream_) cudaStreamSynchronize(stream_);
    cudaFree(d_A_);
    cudaFree(d_place_);
    cudaFree(d_extract_);
    if (stream_) cudaStreamDestroy(stream_);
}

int Encoder::encode(const uint32_t *msg, int64_t F, uint32_t *cw, cudaStream_t st) {
    err_.clear();
    CK(cudaSetDevice(device_));
    if (F == 0) return DNALDPC_OK;
    const int par_words = rpad_ / 32;
    // parity bits go through a stream-ordered scratch of at most 64 MiB: chunks of frames
    const int64_t chunk = R_ ? std::max<int64_t>(kBF, ((64ll << 20) / ((int64_t)par_words * 4)) / kBF * kBF) : F;
    uint32_t *par = nullptr;
    if (R_) CK(cudaMallocAsync((void **)&par, (size_t)std::min(F, chunk) * par_words * 4, st));
    for (int64_t f0 = 0; f0 < F; f0 += chunk) {
        const int64_t n = std::min(F - f0, chunk);
        if (R_) {
            const dim3 grid((unsigned)(rpad_ / kBR), (unsigned)((n + kBF - 1) / kBF));
            encode_parity_kernel<<<grid, kThreads, kParitySmem, st>>>(msg + f0 * kw_, n, kw_, d_A_, kwp_, par, par_words);
        }
        launch_place(msg + f0 * kw_, kw_, par, par_words, d_place_, wpf_, cw + f0 * wpf_, n, st);
        CK(cudaGetLastError());
    }
    if (par) CK(cudaFreeAsync(par, st));
    return DNALDPC_OK;
}

int Encoder::extract(const uint32_t *cw, int64_t F, uint32_t *msg, cudaStream_t st) {
    err_.clear();
    CK(cudaSetDevice(device_));
    launch_place(cw, wpf_, nullptr, 0, d_extract_, kw_, msg, F, st);
    CK(cudaGetLastError());
    return DNALDPC_OK;
}

int Encoder::host_pass(bool enc, const uint32_t *in, int64_t F, uint32_t *out) {
    err_.clear();
    CK(cudaSetDevice(device_));
    if (F == 0) return DNALDPC_OK;
    const int in_w = enc ? kw_ : wpf_, out_w = enc ? wpf_ : kw_;
    const int64_t chunk = std::min<int64_t>(F, 32768);
    uint32_t *d_in = nullptr, *d_out = nullptr;
    CK(cudaMallocAsync((void **)&d_in, (size_t)chunk * std::max(in_w, 1) * 4, stream_));
    CK(cudaMallocAsync((void **)&d_out, (size_t)chunk * std::max(out_w, 1) * 4, stream_));
    int rc = DNALDPC_OK;
    for (int64_t f0 = 0; f0 < F && rc == DNALDPC_OK; f0 += chunk) {
        const int64_t n = std::min(F - f0, chunk);
        cudaError_t e = cudaMemcpyAsync(d_in, in + f0 * in_w, (size_t)n * in_w * 4, cudaMemcpyHostToDevice, stream_);
        if (e != cudaSuccess) { rc = fail(e, "cudaMemcpyAsync(H2D)"); break; }
        rc = enc ? encode(d_in, n, d_out, stream_) : extract(d_in, n, d_out, stream_);
        if (rc) break;
        e = cudaMemcpyAsync(out + f0 * out_w, d_out, (size_t)n * out_w * 4, cudaMemcpyDeviceToHost, stream_);
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream_);
        if (e != cudaSuccess) rc = fail(e, "cudaMemcpyAsync(D2H)");
    }
    cudaFreeAsync(d_in, stream_);
    cudaFreeAsync(d_out, stream_);
    const cudaError_t e = cudaStreamSynchronize(stream_);
    if (rc == DNALDPC_OK && e != cudaSuccess) rc = fail(e, "cudaStreamSynchronize");
    return rc;
}

int Encoder::encode_host(const uint32_t *msg, int64_t F, uint32_t *cw) { return host_pass(true, msg, F, cw); }
int Encoder::extract_host(const uint32_t *cw, int64_t F, uint32_t *msg) { return host_pass(false, cw, F, msg); }

}  // namespace dnaldpc
