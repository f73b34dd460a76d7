#!/usr/bin/env python3
"""bench_encode.py - throughput of the systematic encoder (dnaldpc_encode_device / dnaldpc_encode) on one GPU.

  python tools/bench_encode.py [--reps R] [--out FILE]

Two codes: the n=18432 code of bench.py (K = 16572, R = 1860) and BASELINE configs[4] (gen_regular(65536, 6554, 3, 5):
K = 58982, R = 6554). Messages are random, device-resident and larger than the 126 MB L2 (262144 resp. 32768 frames);
every timed call encodes all of them. Work: F * R * ceil(K/32) AND-XOR word operations (one LOP3 each) per call.
The LOP3 ceiling is 148 SMs x 64 results per clock per SM (32-bit bitwise operations, compute capability 10.0, CUDA C++
Programming Guide throughput table) x the SM clock sampled during the timed window. Prints one JSON line.
"""
import argparse
import ctypes as C
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

LOP3_PER_CLK_PER_SM = 64
SMS = 148


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return {"name": q[0], "power_limit_w": float(q[1]), "sm_max_mhz": float(q[2])}
    except Exception:
        return {}


def bench_code(ldpc, torch, name, code, F, reps, host_frames):
    from bench import ClockSampler
    dec = ldpc.Decoder(code, devices=[0], wave_frames=32)
    K, N = dec.K, code.N
    R = N - K
    kw, wpf = (K + 31) // 32, dec.words_per_frame
    g = torch.Generator(device="cuda").manual_seed(1)
    msg = torch.randint(-2**31, 2**31 - 1, (F, kw), dtype=torch.int32, device="cuda", generator=g)
    cw = torch.empty((F, wpf), dtype=torch.int32, device="cuda")
    for _ in range(3):  # warm-up: module load, scratch pool
        dec.encode_device(msg.data_ptr(), F, cw.data_ptr())
    torch.cuda.synchronize()
    clk = ClockSampler(0, period_ms=100)
    clk.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        dec.encode_device(msg.data_ptr(), F, cw.data_ptr())
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    c = clk.stop()
    ops = F * R * kw
    sm_mhz = c["sm_mhz"]
    ceiling = SMS * LOP3_PER_CLK_PER_SM * sm_mhz * 1e6 if sm_mhz else None
    # host-buffer form: the same messages from pageable host memory, codewords back to it
    hm = msg[:host_frames].cpu().numpy()
    hc = np.empty((host_frames, wpf), np.int32)
    L = ldpc.lib()
    ldpc._check(L.dnaldpc_encode(dec._h, hm.ctypes.data, host_frames, hc.ctypes.data))  # warm-up
    t = time.perf_counter()
    ldpc._check(L.dnaldpc_encode(dec._h, hm.ctypes.data, host_frames, hc.ctypes.data))
    host_s = time.perf_counter() - t
    assert np.array_equal(hc, cw[:host_frames].cpu().numpy())
    dec.close()
    return {
        "code": name, "N": N, "K": K, "R": R, "frames": F, "reps": reps, "ms_per_call": round(ms, 3),
        "frames_per_s": round(F / ms * 1e3), "msg_gbit_per_s": round(F * K / ms / 1e6, 2),
        "codeword_gbit_per_s": round(F * N / ms / 1e6, 2), "word_ops_per_s": ops / ms * 1e3,
        "lop3_ceiling_per_s": ceiling, "fraction_of_lop3_ceiling": round(ops / ms * 1e3 / ceiling, 3) if ceiling else None,
        "sm_mhz": sm_mhz, "clock_reasons": c["reasons"], "clock_samples": c["samples"],
        "host_frames": host_frames, "host_frames_per_s": round(host_frames / host_s),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=0, help="timed calls per code (0 = about 3 s each)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_encode.py needs a CUDA device")
    import _pkg
    import gen_regular_pchk
    import oraclelib as ol
    ldpc = _pkg.load()
    res = {"gpu": gpu_info(), "codes": []}
    c18 = ldpc.Code(ol.PCHK_18432)
    rp, ci = gen_regular_pchk.gen_regular(65536, 6554, 3, 5)
    c4 = ldpc.Code(csr=(6554, 65536, rp, ci))
    for name, code, F, reps, hf in (("n18432_m2048", c18, 262144, a.reps or 100, 65536),
                                    ("configs4_n65536_m6554", c4, 32768, a.reps or 60, 16384)):
        t = time.perf_counter()
        code.systematic()
        sys_s = time.perf_counter() - t
        r = bench_code(ldpc, torch, name, code, F, reps, hf)
        r["systematic_form_s"] = round(sys_s, 2)
        res["codes"].append(r)
    line = json.dumps(res)
    print(line)
    if a.out:
        open(a.out, "w").write(line + "\n")


if __name__ == "__main__":
    main()
