// sim.h - Monte-Carlo error-rate simulation behind dnaldpc_simulate (kernels and frame source in sim.cu).
// Internal C++ interface between capi.cu and the engines.
#pragma once
#include <string>
#include <vector>

#include "encoder.h"
#include "sources.h"

namespace dnaldpc {

// Simulates spec `s` on the engines (encoders[k] lives on eng[k]'s device). `r` receives the counters of the shortest
// prefix of frames the spec asks for; `st` every frame decoded, the discarded ones included. The spec has been checked.
int simulate_batch(EngineSet &eng, const std::vector<Encoder *> &encoders, const Systematic &sys, const dnaldpc_sim &s,
                   dnaldpc_sim_result &r, dnaldpc_stats &st, std::string &err);

}  // namespace dnaldpc
