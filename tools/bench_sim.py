#!/usr/bin/env python3
"""bench_sim.py - throughput of the Monte-Carlo simulator (dnaldpc_simulate) against its ceiling, on one GPU.

  python tools/bench_sim.py [--frames F] [--eps E] [--max-iter I] [--chunk C] [--out FILE]

n=18432 code, BSC, one process, the card's name and power limit read in the same run. Three ways to get the error
counts of the same F frames (random messages of RNG stream 1, seed 1):
  (a) simulate: dnaldpc_simulate, generation and counting inside one engine session;
  (b) ceiling:  dnaldpc_decode_batch_device over the same F frames, messages, codewords and channel bits generated
                beforehand (only the decode is timed);
  (c) chunked:  the Python composition encode_device -> synth_bsc_device -> decode_device -> frame-error count (torch) in
                chunks of C frames, messages already on the device (not timed).
All three must count the same frame errors. Also the in-pipeline trace of (a) and (b) (check pass, bit pass and
scheduler time per tick, decoder profiling mode 2, a separate shorter run) and the encoder's rate on these messages.
Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")):
    sys.path.insert(0, p)

import numpy as np  # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return {"name": q[0], "power_limit_w": float(q[1]), "sm_max_mhz": float(q[2])}
    except Exception:
        return {}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1000000)
    ap.add_argument("--eps", type=float, default=0.006)
    ap.add_argument("--max-iter", type=int, default=100)
    ap.add_argument("--chunk", type=int, default=65536)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_sim.py needs a CUDA device")
    import _pkg
    import oraclelib as ol
    import sim_oracle as so
    ldpc = _pkg.load()
    code = ldpc.Code(ol.PCHK_18432)
    dec = ldpc.Decoder(code, devices=[0])
    F, eps, it, seed = a.frames, a.eps, a.max_iter, a.seed
    N, K, wpf = code.N, dec.K, dec.words_per_frame
    kw = (K + 31) // 32
    res = {"gpu": gpu_info(), "code": "n18432_m2048", "N": N, "K": K, "channel": "bsc", "eps": eps, "max_iter": it,
           "frames": F, "seed": seed, "chunk": a.chunk}
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

    # messages of the simulator's frames, generated beforehand by the numpy twin (chunks keep the host memory small)
    msg = torch.empty((F, kw), dtype=torch.int32, device="cuda")
    for f0 in range(0, F, 65536):
        n = min(65536, F - f0)
        msg[f0:f0 + n] = torch.from_numpy(so.messages(seed, f0, n, K).view(np.int32)).cuda()
    cw = torch.empty((F, wpf), dtype=torch.int32, device="cuda")
    rx = torch.empty_like(cw)
    bits = torch.zeros_like(cw)
    for _ in range(2):  # warm-up of the encoder
        dec.encode_device(msg.data_ptr(), F, cw.data_ptr())
    e0, e1 = ev(), ev()
    e0.record()
    dec.encode_device(msg.data_ptr(), F, cw.data_ptr())
    e1.record()
    torch.cuda.synchronize()
    enc_ms = e0.elapsed_time(e1)
    res["encode"] = {"ms": round(enc_ms, 2), "frames_per_s": round(F / enc_ms * 1e3), "msg_gbit_per_s": round(F * K / enc_ms / 1e6, 2)}
    dec.synth_bsc_device(cw.data_ptr(), F, seed, 0, F, eps, rx.data_ptr())

    # warm-up of both paths (module loads, slot arrays, rings)
    dec.simulate(ldpc.IN_BSC_BITS, eps, it, 65536, seed=seed + 1)
    dec.decode_device(ldpc.IN_BSC_BITS, rx.data_ptr(), 65536, it, param=eps, bits_ptr=bits.data_ptr())
    torch.cuda.synchronize()

    # (a) the simulator
    t = time.perf_counter()
    r = dec.simulate(ldpc.IN_BSC_BITS, eps, it, F, seed=seed)
    a_s = time.perf_counter() - t
    st = dec.stats()
    res["a_simulate"] = {"s": round(a_s, 3), "frames_per_s": round(F / a_s), "result": r, "frames_decoded": st["frames"]}

    # (b) the ceiling: one device-resident batch of the same frames
    torch.cuda.synchronize()
    t = time.perf_counter()
    dec.decode_device(ldpc.IN_BSC_BITS, rx.data_ptr(), F, it, param=eps, bits_ptr=bits.data_ptr())
    torch.cuda.synchronize()
    b_s = time.perf_counter() - t
    b_fe = int((bits != cw).any(dim=1).sum().item())
    res["b_decode_device"] = {"s": round(b_s, 3), "frames_per_s": round(F / b_s), "frame_errors": b_fe,
                              "iterations": dec.stats()["frame_iters"]}
    res["b_decode_device"]["same_frame_errors_as_a"] = b_fe == r["frame_errors"]

    # (c) the chunked composition in Python
    C = a.chunk
    cw_c = torch.empty((C, wpf), dtype=torch.int32, device="cuda")
    rx_c, bits_c = torch.empty_like(cw_c), torch.empty_like(cw_c)
    fe = 0
    torch.cuda.synchronize()
    t = time.perf_counter()
    for f0 in range(0, F, C):
        n = min(C, F - f0)
        dec.encode_device(msg[f0].data_ptr(), n, cw_c.data_ptr())
        dec.synth_bsc_device(cw_c.data_ptr(), C, seed, f0, n, eps, rx_c.data_ptr())  # frame f0 + i reads row (f0 + i) % C = i
        dec.decode_device(ldpc.IN_BSC_BITS, rx_c.data_ptr(), n, it, param=eps, bits_ptr=bits_c.data_ptr())
        fe += int((bits_c[:n] != cw_c[:n]).any(dim=1).sum().item())
    torch.cuda.synchronize()
    c_s = time.perf_counter() - t
    res["c_chunked"] = {"s": round(c_s, 3), "frames_per_s": round(F / c_s), "frame_errors": fe}
    res["c_chunked"]["same_frame_errors_as_a"] = fe == r["frame_errors"]  # the same frames as (a) and (b)
    res["a_over_b"] = round(b_s / a_s, 4)
    res["a_over_c"] = round(c_s / a_s, 4)

    # in-pipeline trace (separate runs; profiling mode 2 records ticks 8..71 without synchronising)
    Ft = min(F, 262144)
    dec.set_profiling(2)
    dec.simulate(ldpc.IN_BSC_BITS, eps, it, Ft, seed=seed)
    ra = dec.trace()
    dec.set_profiling(2)
    dec.decode_device(ldpc.IN_BSC_BITS, rx.data_ptr(), Ft, it, param=eps, bits_ptr=bits.data_ptr())
    torch.cuda.synchronize()
    rb = dec.trace()
    dec.set_profiling(0)
    keys = ("check_ms", "bit_ms", "sched_ms", "ticks")
    res["trace_per_tick"] = {"simulate": dict(zip(keys, [round(x, 4) for x in ra[:3]] + [ra[3]])),
                             "decode_device": dict(zip(keys, [round(x, 4) for x in rb[:3]] + [rb[3]]))}
    line = json.dumps(res)
    print(line)
    if a.out:
        open(a.out, "w").write(line + "\n")
    dec.close()


if __name__ == "__main__":
    main()
