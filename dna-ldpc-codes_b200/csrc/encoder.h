// encoder.h - systematic LDPC encoder and message extraction on one GPU (kernels in encoder.cu). Holds the dense parity
// part A of the systematic form (host/systematic.h) in HBM and the two bit-placement tables. Internal C++ interface
// behind dnaldpc_encode* / dnaldpc_extract* of include/dnaldpc.h.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <string>

#include "../host/systematic.h"

namespace dnaldpc {

class Encoder {
  public:
    Encoder(const Systematic &s, int N, int device);
    ~Encoder();
    bool ok() const { return err_.empty(); }
    const std::string &error() const { return err_; }

    // DEVICE buffers on this encoder's device, asynchronous on `stream`. msg: uint32 [F][kw], cw: uint32 [F][ceil(N/32)].
    int encode(const uint32_t *msg, int64_t F, uint32_t *cw, cudaStream_t stream);
    int extract(const uint32_t *cw, int64_t F, uint32_t *msg, cudaStream_t stream);
    // HOST buffers, blocking: moved through device memory in chunks.
    int encode_host(const uint32_t *msg, int64_t F, uint32_t *cw);
    int extract_host(const uint32_t *cw, int64_t F, uint32_t *msg);

  private:
    int fail(cudaError_t e, const char *what);
    int host_pass(bool enc, const uint32_t *in, int64_t F, uint32_t *out);

    std::string err_;
    int device_ = 0, N_ = 0, K_ = 0, R_ = 0;
    int kw_ = 0, wpf_ = 0;   // words of a message / of a codeword
    int kwp_ = 0, rpad_ = 0; // A in HBM: [rpad_][kwp_], rows and k words padded with zeros to whole tiles
    uint32_t *d_A_ = nullptr;
    int32_t *d_place_ = nullptr;    // codeword bit -> message / parity bit ([ceil(wpf/32) * 1024])
    int32_t *d_extract_ = nullptr;  // message bit -> codeword bit ([ceil(kw/32) * 1024])
    cudaStream_t stream_ = nullptr; // host forms
};

}  // namespace dnaldpc
