#!/usr/bin/env python3
"""bench_layered.py - layered normalised min-sum (FLAG_MINSUM | FLAG_LAYERED) against flooding BP on the n=18432 code.

  python tools/bench_layered.py [--frames F] [--chunk C] [--max-iter I] [--alpha A] [--target T] [--out FILE]

One process on GPU 0; the card's name and power limit are read in the same run. Two parts:
  (a) throughput: device-resident decodes of F frames (default 2^20, in chunks of C frames generated on the device from
      the 272 fixture codewords) for BSC eps 0.006 and 0.008, vote counts (BASELINE configs[2]: 3.9 mean reads, read
      error 0.01, decoder eps 0.02) and AWGN (configs[3]: Eb/N0 4.6 dB), each with flooding BP fp64, layered fp64 and
      layered fp32 (alpha = --alpha). Reported: frames/s, decoded Gbit/s (N bits per frame), average iterations, FER
      (decoded != sent). Then, in separate shorter runs with per-tick profiling (mode 1), the layer passes' kernel time
      per tick and per layer pass next to the algorithmic bytes of the traffic model (DESIGN.md §5e) of one tick with
      every slot busy, read at the BSC 0.008 point where frames need many iterations.
  (b) error rates: dnaldpc_simulate with --target frame errors (capped), flooding BP against layered fp64 with alpha in
      {0.625, 0.6875, 0.75, 0.8125, 0.875, 1.0}, at BSC eps 0.006 / 0.008 and AWGN Eb/N0 3.6 / 4.0 dB.
Prints one JSON object and writes it to --out (default profiles/layered_b200.json).
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


def state_elems(esz, max_row_deg):
    """T-sized elements of one check's layered state (layered_kernels.cuh LayerState<T, DC>::W)."""
    dc = 8 if max_row_deg <= 8 else 32 if max_row_deg <= 32 else 72 if max_row_deg <= 72 else 128
    meta_words = 1 + (dc + 31) // 32
    return 2 + (meta_words * 4 + esz - 1) // esz


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1 << 20)
    ap.add_argument("--chunk", type=int, default=1 << 18)
    ap.add_argument("--max-iter", type=int, default=50)
    ap.add_argument("--alpha", type=float, default=0.75)
    ap.add_argument("--target", type=int, default=100, help="frame errors per simulated point")
    ap.add_argument("--sim-cap", type=int, default=400000, help="most frames per simulated point")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--skip-sim", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "layered_b200.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_layered.py needs a CUDA device")
    import _pkg
    import oraclelib as ol
    ldpc = _pkg.load()
    code = ldpc.Code(ol.PCHK_18432)
    M, N, E = code.M, code.N, code.E
    n_layers, _ = code.layers()
    dev = torch.device("cuda:0")
    cws = ol.load_codewords()
    d_cw = torch.from_numpy(ldpc._pack_bits(cws).view(np.int32)).to(dev)
    sent_all = torch.from_numpy(ldpc._pack_bits(cws).view(np.int32)).to(dev)
    W = (N + 31) // 32
    LAY = ldpc.FLAG_MINSUM | ldpc.FLAG_LAYERED
    decs = {"bp_f64": (ldpc.Decoder(code, devices=[0]), 0),
            "layered_f64": (ldpc.Decoder(code, devices=[0]), LAY),
            "layered_f32": (ldpc.Decoder(code, devices=[0], precision=ldpc.PREC_F32), LAY)}
    for name, (d, fl) in decs.items():
        d.set_minsum_scale(a.alpha)
    sigma46 = ldpc.std_dev(4.6, 1 - M / N)
    workloads = {
        "bsc_eps0.006": (ldpc.IN_BSC_BITS, torch.int32, W, 0.006, lambda d, f0, F, out: d.synth_bsc_device(d_cw.data_ptr(), 272, a.seed, f0, F, 0.006, out)),
        "bsc_eps0.008": (ldpc.IN_BSC_BITS, torch.int32, W, 0.008, lambda d, f0, F, out: d.synth_bsc_device(d_cw.data_ptr(), 272, a.seed, f0, F, 0.008, out)),
        "vote_c2": (ldpc.IN_VOTE_I8, torch.int8, N, 0.02, lambda d, f0, F, out: d.synth_vote_device(d_cw.data_ptr(), 272, a.seed, f0, F, 3.9, 0.01, out)),
        "awgn_c3_4.6dB": (ldpc.IN_AWGN_F32, torch.float32, N, sigma46, lambda d, f0, F, out: d.synth_awgn_device(d_cw.data_ptr(), 272, a.seed, f0, F, sigma46, out)),
    }
    res = {"gpu": gpu_info(), "code": "n=18432 m=2048 (decode_n18432_m2048_final.pchk), %d layers" % n_layers,
           "frames": a.frames, "chunk": a.chunk, "max_iter": a.max_iter, "alpha": a.alpha, "throughput": {}}
    C = min(a.chunk, a.frames)
    nchunks = (a.frames + C - 1) // C
    gen = decs["bp_f64"][0]
    for wname, (kind, dt, width, param, synth) in workloads.items():
        d_in = torch.empty((C, width), dtype=dt, device=dev)
        bits = torch.empty((C, W), dtype=torch.int32, device=dev)
        iters = torch.empty(C, dtype=torch.int32, device=dev)
        row = {}
        for name, (dec, fl) in decs.items():
            dec.decode_device(kind, d_in.data_ptr(), min(C, 4096), a.max_iter, param=param, bits_ptr=bits.data_ptr(),
                              iters_ptr=iters.data_ptr(), flags=fl)   # warm-up
            t_ms, it_sum, fe, frames = 0.0, 0, 0, 0
            for c in range(nchunks):
                F = min(C, a.frames - c * C)
                synth(gen, c * C, F, d_in.data_ptr())
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                dec.decode_device(kind, d_in.data_ptr(), F, a.max_iter, param=param, bits_ptr=bits.data_ptr(),
                                  iters_ptr=iters.data_ptr(), flags=fl)
                torch.cuda.synchronize()
                t_ms += (time.perf_counter() - t0) * 1e3
                it_sum += int(iters[:F].sum().item())
                rows = (torch.arange(F, device=dev) + c * C) % 272
                diff = (bits[:F] ^ sent_all[rows])
                diff[:, -1] &= (1 << (N % 32)) - 1 if N % 32 else -1
                fe += int((diff != 0).any(dim=1).sum().item())
                frames += F
            row[name] = {"ms": t_ms, "frames_per_s": frames / (t_ms * 1e-3), "gbit_per_s": frames * N / (t_ms * 1e-3) / 1e9,
                         "avg_iters": it_sum / frames, "fer": fe / frames}
            print(wname, name, json.dumps(row[name]), flush=True)
        res["throughput"][wname] = row
        del d_in, bits, iters
        torch.cuda.empty_cache()

    # per-tick layer-pass time with profiling (mode 1: events around the passes of every tick, host syncs)
    res["layer_pass_profile"] = {}
    Fp = 65536
    kind, dt, width, param, synth = workloads["bsc_eps0.008"]
    d_in = torch.empty((Fp, width), dtype=dt, device=dev)
    synth(gen, 0, Fp, d_in.data_ptr())
    for name, (dec, fl) in decs.items():
        dec.set_profiling(1)
        dec.decode_device(kind, d_in.data_ptr(), Fp, a.max_iter, param=param, flags=fl)
        torch.cuda.synchronize()
        st = dec.stats()
        dec.set_profiling(0)
        ticks = max(st["waves"], 1)
        slots = 4096
        if fl:
            esz = 8 if name.endswith("f64") else 4
            Wst = state_elems(esz, 72)
            # per tick, every slot busy: q read + written once per edge, the check state read + written once per check,
            # the decision words read-modify-written once per edge (one 4-byte word per 32 slots)
            bytes_tick = slots * (2 * E * esz + 2 * M * Wst * esz) + (slots // 32) * E * 8
            per_tick = st["row_ms"] / ticks
            res["layer_pass_profile"][name] = {"ticks": ticks, "layer_ms_per_tick": per_tick,
                                               "ms_per_layer_pass": per_tick / n_layers,
                                               "model_bytes_per_tick_all_slots_busy": bytes_tick,
                                               "model_gb_per_s": bytes_tick / (per_tick * 1e-3) / 1e9,
                                               "state_elems_per_check": Wst}
        else:
            per_tick = (st["row_ms"] + st["col_ms"]) / ticks
            bytes_tick = slots * (32 * E + 8.25 * N)   # B_iter of DESIGN.md §6 (fp64 flooding)
            res["layer_pass_profile"][name] = {"ticks": ticks, "check_plus_bit_ms_per_tick": per_tick,
                                               "model_bytes_per_tick_all_slots_busy": bytes_tick,
                                               "model_gb_per_s": bytes_tick / (per_tick * 1e-3) / 1e9}
        print("profile", name, json.dumps(res["layer_pass_profile"][name]), flush=True)
    del d_in
    torch.cuda.empty_cache()

    if not a.skip_sim:
        K = decs["bp_f64"][0].K
        points = [("bsc", ldpc.IN_BSC_BITS, 0.006), ("bsc", ldpc.IN_BSC_BITS, 0.008),
                  ("awgn_dB", ldpc.IN_AWGN_F32, 3.6), ("awgn_dB", ldpc.IN_AWGN_F32, 4.0)]
        res["simulate"] = {"target_frame_errors": a.target, "cap": a.sim_cap, "points": {}}
        for label, ch, x in points:
            param = x if ch == ldpc.IN_BSC_BITS else ldpc.std_dev(x, K / N)
            pt = {}
            runs = [("bp_f64", decs["bp_f64"][0], 0, None)] + \
                   [("layered_f64_a%g" % al, decs["layered_f64"][0], LAY, al) for al in (0.625, 0.6875, 0.75, 0.8125, 0.875, 1.0)]
            for rname, dec, fl, al in runs:
                if al is not None:
                    dec.set_minsum_scale(al)
                t0 = time.perf_counter()
                r = dec.simulate(ch, param, a.max_iter, a.sim_cap, target_frame_errors=a.target, seed=a.seed, flags=fl)
                s = time.perf_counter() - t0
                pt[rname] = {"frames": r["frames"], "frame_errors": r["frame_errors"], "fer": r["frame_errors"] / r["frames"],
                             "ber": r["bit_errors"] / (r["frames"] * N), "avg_iters": r["iterations"] / r["frames"],
                             "undetected": r["undetected"], "s": s}
                print("sim", label, x, rname, json.dumps(pt[rname]), flush=True)
            res["simulate"]["points"]["%s_%g" % (label, x)] = pt
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(a.out), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
