#!/usr/bin/env python3
"""bench.py - decoded Gbit/s of the B200 BP decoder on BASELINE.json's n=18432 code (contract: see DESIGN.md §Measurement).

  python bench.py --gpus N --steps K --warmup W            our arm (one rank per GPU; torchrun for N > 1)
  python bench.py --impl reference --gpus N ...            the reference's own CPU implementation on the host cores
  python bench.py ... --dump-outputs DIR                   also write the last timed step's outputs as DIR/<name>.npy

A step = one pass of the hot path over one batch: F frames (default 100 000, BASELINE configs[1]) of the
n=18432/m=2048 code, codeword[f % 272] through a BSC(eps), prprp max 100 iterations, decoded bits + iteration counts out.
`value` = whole-job decoded Gbit/s with inputs resident in HBM; `e2e` = same through the host-buffer C-ABI call.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only; the bench writes nothing into it
DUMP_FRAMES = 512              # --dump-outputs: frames whose decoded bits are written (18432 x 4 B each)
DUMP_SCALAR_FRAMES = 1 << 20   # --dump-outputs: frames whose iteration count and codeword flag are written (8 B each)
PCHK = os.path.join(ROOT, "tests", "golden", "decode_n18432_m2048_final.pchk")
CW_BITS = os.path.join(ROOT, "tests", "golden", "codewords_n18432_272.bits")
N, M, E = 18432, 2048, 147456
B_ROW = 16 * E                 # check-node pass: read pr + write lr, 8 B each per edge
B_COL = 16 * E + 8.25 * N      # bit-node pass: read lr + write pr, lratio, packed decisions
B_ITER = 32 * E + 8.25 * N     # SURVEY.md §8d: algorithmic bytes per frame-iteration (fp64)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index, period_ms=200):
        self.gpu = gpu_index
        self.period_ms = period_ms
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", str(self.period_ms)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, reasons = [], set()
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); out["sm_max_mhz"] = float(r[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out["sm_mhz"] = statistics.median(sm)
        out["reasons"] = sorted(reasons)
        out["samples"] = len(sm)
        return out


def shard(total_frames_per_gpu, rank):
    """Weak scaling: every rank decodes its own F frames; GLOBAL frame indices keep results independent of N."""
    return rank * total_frames_per_gpu, total_frames_per_gpu


def aggregate(ms, frame_iters, device, world):
    """Whole-job figures from per-rank ones: time = MAX over ranks (device time), work = SUM over ranks.
    The only cross-rank traffic of the whole job (two doubles); the data path has no collective."""
    if world <= 1:
        return float(ms), float(frame_iters)
    import torch
    import torch.distributed as dist
    t = torch.tensor([float(ms), float(frame_iters)], dtype=torch.float64, device=device)
    tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
    return float(tmax[0]), float(tsum[1])


def cpu_reference_run(frames_per_proc, eps, max_iter):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import cpu_baseline
    return cpu_baseline.run(PCHK, 0, frames_per_proc, eps, max_iter)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # bounded sample of the same workload: `fpp` frames per host core per step
    vals, info = [], None
    for s in range(args.warmup + args.steps):
        info = cpu_reference_run(args.ref_frames_per_core, args.eps, args.max_iter)
        if s >= args.warmup:
            vals.append(info["frames"] * N / info["decode_s"] / 1e9)
    v = statistics.mean(vals)
    line = {
        "impl": "reference", "metric": "decoded Gbit/s, n=18432 prprp", "value": v, "unit": "Gbit/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * info["decode_s"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, info["frames"]),
        "cpu_baseline": {"value": v, "unit": "Gbit/s", "cores": info["cores"], "kind": info["kind"],
                         "sample": "%d frames (%d per core) x max %d iterations, eps=%g; %.2f ms per iteration per core"
                                   % (info["frames"], args.ref_frames_per_core, args.max_iter, args.eps, info["ms_per_iter_per_core"])},
        "e2e": {"value": v, "unit": "Gbit/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


def workload_config(args, frames):
    return {"workload": "configs[1]: n=18432/m=2048 code (decode_n18432_m2048_final.pchk), %d-frame batch per GPU, "
                        "codeword[f%%272] + synthetic BSC eps=%g, prprp max %d iterations" % (frames, args.eps, args.max_iter),
            "frames_per_gpu": frames, "eps": args.eps, "max_iter": args.max_iter, "wave_frames": args.wave, "algorithm": args.alg,
            "l2": "inputs larger than L2: message working set %.1f GB per wave vs 126 MB L2" % (min(args.wave, frames) * E * 8 / 1e9)}


def _ev_time(torch, fn, reps=1):
    """CUDA-event time in ms of fn() on the current stream (fn blocks the host until its batch has drained)."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def _sample_frames(F, k):
    """All F frame indices, or k of them drawn with a fixed seed (sorted): the same frames on every run."""
    return np.arange(F) if F <= k else np.sort(np.random.default_rng(0).choice(F, k, replace=False))


def dump_outputs(out_dir, d_bits, d_it, d_ok):
    """What the caller of dnaldpc_decode_batch_device receives, as float .npy files: iteration counts and codeword flags
    (frames.npy: which frames, all of them up to DUMP_SCALAR_FRAMES) and the decoded bits, unpacked to 0/1, of
    DUMP_FRAMES frames (bits_frames.npy). Under 64 MB in all; the inputs depend on the arguments alone, so two builds run
    with the same arguments can be compared file by file."""
    import torch
    F = d_it.shape[0]
    os.makedirs(out_dir, exist_ok=True)
    idx = _sample_frames(F, DUMP_SCALAR_FRAMES)
    sel = torch.from_numpy(idx).to(d_it.device)
    np.save(os.path.join(out_dir, "frames.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "iters.npy"), d_it[sel].cpu().numpy().astype(np.float32))
    np.save(os.path.join(out_dir, "is_codeword.npy"), d_ok[sel].cpu().numpy().astype(np.float32))
    idx = _sample_frames(F, DUMP_FRAMES)
    words = d_bits[torch.from_numpy(idx).to(d_bits.device)].cpu().numpy()
    bits = np.unpackbits(words.view(np.uint8), axis=1, bitorder="little")[:, :N]
    np.save(os.path.join(out_dir, "bits_frames.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "bits.npy"), bits.astype(np.float32))


def secondary_regimes(ldpc, torch, dec, code, d_cw, args, peak):
    """The regimes the headline configuration never exercises (frames that converge: admission, refill-regime check pass,
    drain-tail compaction; BASELINE configs[2..4]; fp32; min-sum; host buffers of the wide input kinds). A few seconds
    each, CUDA-event timed after one warm-up pass; frac = B_iter x frame-iterations / time / measured HBM peak."""
    dev = torch.device("cuda", torch.cuda.current_device())
    st = torch.cuda.current_stream().cuda_stream
    W = (N + 31) // 32
    out = {}
    sel = set(args.secondary.split(","))
    want = lambda name: "all" in sel or name in sel  # noqa: E731

    def run_device(dc, kind, d_in, F, param, max_iter, n_, flags=0, b_iter=B_ITER, reps=1):
        d_bits = torch.empty((F, (n_ + 31) // 32), dtype=torch.int32, device=dev)
        d_it = torch.empty(F, dtype=torch.int32, device=dev)
        d_ok = torch.empty(F, dtype=torch.uint8, device=dev)

        def go():
            dc.decode_device(kind, d_in.data_ptr(), F, max_iter, param=param, bits_ptr=d_bits.data_ptr(), iters_ptr=d_it.data_ptr(),
                             ok_ptr=d_ok.data_ptr(), stream=st, flags=flags)
        go()  # warm-up (slot arrays, queue tables)
        ms = _ev_time(torch, go, reps)
        fi = float(d_it.sum().item())
        return {"frames": F, "ms": ms, "gbit_s": F * n_ / (ms * 1e-3) / 1e9, "frames_per_s": F / (ms * 1e-3),
                "frame_iters_per_s": fi / (ms * 1e-3), "avg_iters": fi / F, "fer": 1.0 - float(d_ok.float().mean().item()),
                "whole_step_gbs": b_iter * fi / (ms * 1e-3) / 1e9, "frac": b_iter * fi / (ms * 1e-3) / 1e9 / peak}

    # converging BSC frames (the pipeline's real regime), two batch sizes
    for F in (65536, 1000000) if want("bsc") else ():
        d_in = torch.empty((F, W), dtype=torch.int32, device=dev)
        dec.synth_bsc_device(d_cw.data_ptr(), 272, args.seed, 0, F, 0.006, d_in.data_ptr(), st)
        out["bsc_eps0.006_%d" % F] = run_device(dec, ldpc.IN_BSC_BITS, d_in, F, 0.006, args.max_iter, N)
        del d_in
    if want("vote"):
        # configs[2]: vote counts, 1M frames
        F = 1000000
        d_in = torch.empty((F, N), dtype=torch.int8, device=dev)
        dec.synth_vote_device(d_cw.data_ptr(), 272, args.seed, 0, F, 3.9, 0.01, d_in.data_ptr(), st)
        out["c3_vote_i8_1000000"] = run_device(dec, ldpc.IN_VOTE_I8, d_in, F, 0.02, args.max_iter, N)
        # the same frames through the host-buffer call (pinned memory, copies inside the timed region)
        Fh = 131072
        h_in = torch.empty((Fh, N), dtype=torch.int8).pin_memory(); h_in.copy_(d_in[:Fh])
        same_size = run_device(dec, ldpc.IN_VOTE_I8, d_in[:Fh], Fh, 0.02, args.max_iter, N)  # the ratio compares batches of one size
        del d_in
        out["c3_vote_i8_host_%d" % Fh] = host_leg(ldpc, torch, dec, ldpc.IN_VOTE_I8, h_in, Fh, 0.02, args.max_iter, same_size)
        del h_in
    if want("awgn"):
        # configs[3]: AWGN at Eb/N0 = 4.6 dB
        F = 262144
        sigma = ldpc.std_dev(4.6, 1 - M / N)
        d_in = torch.empty((F, N), dtype=torch.float32, device=dev)
        dec.synth_awgn_device(d_cw.data_ptr(), 272, args.seed, 0, F, sigma, d_in.data_ptr(), st)
        out["c4_awgn_f32_%d" % F] = run_device(dec, ldpc.IN_AWGN_F32, d_in, F, sigma, args.max_iter, N)
        Fh = 65536
        h_in = torch.empty((Fh, N), dtype=torch.float32).pin_memory(); h_in.copy_(d_in[:Fh])
        same_size = run_device(dec, ldpc.IN_AWGN_F32, d_in[:Fh], Fh, sigma, args.max_iter, N)
        del d_in
        out["c4_awgn_f32_host_%d" % Fh] = host_leg(ldpc, torch, dec, ldpc.IN_AWGN_F32, h_in, Fh, sigma, args.max_iter, same_size)
        del h_in
    if want("llr"):
        # LLR text-file style input: fp64 LLRs, exp on the host with libm (what the CLI does); bound by libm exp on the host cores
        Fh = 16384
        d_b = torch.empty((Fh, W), dtype=torch.int32, device=dev)
        dec.synth_bsc_device(d_cw.data_ptr(), 272, args.seed, 0, Fh, 0.006, d_b.data_ptr(), st)
        torch.cuda.synchronize()
        bits = np.unpackbits(d_b.cpu().numpy().view(np.uint8).reshape(Fh, W * 4), axis=1, bitorder="little")[:, :N]
        L = float(np.log((1 - 0.006) / 0.006))
        h_llr = torch.from_numpy(np.where(bits == 0, L, -L)).pin_memory()
        del d_b, bits
        out["llr_f64_host_exp_%d" % Fh] = host_leg(ldpc, torch, dec, ldpc.IN_LLR_F64, h_llr, Fh, 0.0, args.max_iter, None, flags=ldpc.FLAG_HOST_EXP)
        out["llr_f64_device_exp_%d" % Fh] = host_leg(ldpc, torch, dec, ldpc.IN_LLR_F64, h_llr, Fh, 0.0, args.max_iter, None)
        del h_llr
    if want("minsum_fp32"):
        # min-sum and fp32 at the headline operating point (no frame converges: pure kernel throughput)
        F = 16384
        d_in = torch.empty((F, W), dtype=torch.int32, device=dev)
        dec.synth_bsc_device(d_cw.data_ptr(), 272, args.seed, 0, F, args.eps, d_in.data_ptr(), st)
        out["minsum_eps%g_%d" % (args.eps, F)] = run_device(dec, ldpc.IN_BSC_BITS, d_in, F, args.eps, args.max_iter, N, flags=ldpc.FLAG_MINSUM)
        d32 = ldpc.Decoder(code, devices=[torch.cuda.current_device()], wave_frames=args.wave, precision=ldpc.PREC_F32)
        out["fp32_eps%g_%d" % (args.eps, F)] = run_device(d32, ldpc.IN_BSC_BITS, d_in, F, args.eps, args.max_iter, N, b_iter=0.5 * B_ITER)
        d32.close()
        del d_in
    if want("c5"):
        # configs[4]: Neal-style random regular code n=65536, column weight 3, rate 0.9
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import gen_regular_pchk
        n5, m5 = 65536, 6554
        row_ptr, col_idx = gen_regular_pchk.gen_regular(n5, m5, 3, 5)
        code5 = ldpc.Code(csr=(m5, n5, row_ptr, col_idx))
        dec5 = ldpc.Decoder(code5, devices=[torch.cuda.current_device()], wave_frames=args.wave)
        b5 = 32 * code5.E + 8.25 * n5
        for eps5, F5 in ((0.02, 8192), (0.004, 32768)):
            d_in = torch.empty((F5, n5 // 32), dtype=torch.int32, device=dev)
            dec5.synth_bsc_device(None, 0, args.seed, 0, F5, eps5, d_in.data_ptr(), st)  # all-zero codeword
            out["c5_n65536_eps%g_%d" % (eps5, F5)] = run_device(dec5, ldpc.IN_BSC_BITS, d_in, F5, eps5, 50, n5, b_iter=b5)
            del d_in
        dec5.close()
    if want("sw"):
        out["sw_z1024_l24_eps0.03_8192"] = sliding_window_leg(ldpc, torch, args)
    return out


def sliding_window_leg(ldpc, torch, args, Z=1024, Lc=24, win=6, F=8192, eps=0.03, max_iter=20):
    """dnaldpc_decode_window (Run_SW_Decoder, dec.cpp:2092-2196) on a terminated (3,6) SC-LDPC code from tools/gen_sc_pchk.py:
    all-zero codeword through a BSC, fp64 ratios in pinned host memory, host buffers out; the C-ABI call alone is timed."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import gen_sc_pchk
    Cc = ldpc.C
    Ms, Ns, row_ptr, col_idx, Mv, Mc = gen_sc_pchk.gen_sc(Z, Lc, 11)
    code = ldpc.Code(csr=(Ms, Ns, row_ptr, col_idx))
    dec = ldpc.Decoder(code, devices=[torch.cuda.current_device()], wave_frames=args.wave)
    dev = torch.device("cuda", torch.cuda.current_device())
    gen = torch.Generator(device=dev); gen.manual_seed(args.seed)
    h_lr = torch.empty((F, Ns), dtype=torch.float64).pin_memory()
    for f0 in range(0, F, 1024):  # ratios made on the device in slices, parked in pinned host memory
        fl = torch.rand((min(1024, F - f0), Ns), device=dev, generator=gen) < eps
        h_lr[f0:f0 + fl.shape[0]].copy_(torch.where(fl, eps / (1 - eps), (1 - eps) / eps).to(torch.float64))
    D = Lc + 3 - 1
    mv = np.ascontiguousarray(Mv[:D], dtype=np.int32); mc = np.ascontiguousarray(Mc[:D], dtype=np.int32)
    Ws = (Ns + 31) // 32
    h_bits = torch.zeros((F, Ws), dtype=torch.int32).pin_memory()
    h_it = torch.zeros(F, dtype=torch.int32).pin_memory()
    h_ok = torch.zeros(F, dtype=torch.uint8).pin_memory()
    wd = ldpc.Window(code_type=0, L=Lc, w=3, win=win, Mv=mv.ctypes.data, Mc=mc.ctypes.data)
    outp = ldpc.Output(bits=h_bits.data_ptr(), dblk=None, iters=h_it.data_ptr(), is_codeword=h_ok.data_ptr(), posterior=None, pchk=None)

    def go(nf):
        rc = ldpc.lib().dnaldpc_decode_window(dec._h, Cc.byref(wd), h_lr.data_ptr(), nf, max_iter, Cc.byref(outp))
        if rc:
            raise RuntimeError(ldpc.lib().dnaldpc_last_error())
    go(min(F, args.wave))
    torch.cuda.synchronize()
    sampler = ClockSampler(torch.cuda.current_device(), period_ms=50)
    sampler.start()
    dts = []
    for _ in range(2):
        t0 = time.perf_counter()
        go(F)
        dts.append(time.perf_counter() - t0)
    dt = min(dts)
    clocks = sampler.stop()
    stt = dec.stats()
    ok = h_ok.numpy()
    good = torch.from_numpy(ok.astype(bool))
    r = {"frames": F, "ms": dt * 1e3, "gbit_s": F * Ns / dt / 1e9, "frames_per_s": F / dt, "fer": 1.0 - float(ok.mean()),
         "code": {"Z": Z, "L": Lc, "N": Ns, "M": Ms, "window": win}, "max_extra_updates": max_iter, "ticks": stt["waves"],
         "kernel_launches": stt["kernel_launches"], "ms_runs": [x * 1e3 for x in dts], "clocks": clocks, "h2d_bytes": F * Ns * 8, "d2h_bytes": F * (Ws * 4 + 5),
         "flagged_frames": int(ok.sum()), "flagged_frames_with_bit_errors": int((h_bits[good] != 0).any(dim=1).sum().item()) if ok.any() else 0,
         "bit_errors_all_frames": int(np.unpackbits(h_bits.numpy().view(np.uint8)).sum())}
    dec.close()
    return r


def host_leg(ldpc, torch, dec, kind, h_in, F, param, max_iter, device_ref, flags=0):
    """One host-buffer batch through dnaldpc_decode_batch (pinned memory; H2D and D2H inside the timed region)."""
    Cc = ldpc.C
    W = (N + 31) // 32
    h_bits = torch.empty((F, W), dtype=torch.int32).pin_memory()
    h_it = torch.empty(F, dtype=torch.int32).pin_memory()
    h_ok = torch.empty(F, dtype=torch.uint8).pin_memory()
    inp = ldpc.Input(kind=kind, flags=flags, data=h_in.data_ptr(), frame_stride=0, param=param, table=None)
    outp = ldpc.Output(bits=h_bits.data_ptr(), dblk=None, iters=h_it.data_ptr(), is_codeword=h_ok.data_ptr(), posterior=None, pchk=None)

    def go():
        rc = ldpc.lib().dnaldpc_decode_batch(dec._h, Cc.byref(inp), F, max_iter, Cc.byref(outp))
        if rc:
            raise RuntimeError(ldpc.lib().dnaldpc_last_error())
    go()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    go()
    dt = time.perf_counter() - t0
    fi = float(h_it.sum().item())
    h2d = h_in.numel() * h_in.element_size()
    r = {"frames": F, "ms": dt * 1e3, "gbit_s": F * N / dt / 1e9, "frames_per_s": F / dt, "frame_iters_per_s": fi / dt,
         "avg_iters": fi / F, "h2d_bytes": h2d, "d2h_bytes": F * (W * 4 + 5), "pcie_gbs": (h2d + F * (W * 4 + 5)) / dt / 1e9}
    if device_ref is not None:
        r["vs_device_resident"] = r["frames_per_s"] / device_ref["frames_per_s"]
        r["device_resident_frames_per_s"] = device_ref["frames_per_s"]  # same kind, same number of frames
    return r


def inproc_multi(ldpc, torch, code, d_cw_np, args, world):
    """Rank 0 alone decodes ONE batch through the library's own multi-GPU dispatch (dnaldpc_config.devices[0..N)), host
    buffers, against the same call on one device. The other ranks have released their decoders and wait on the store."""
    F = args.inproc_frames
    W = (N + 31) // 32
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream().cuda_stream
    one = ldpc.Decoder(code, devices=[0], wave_frames=args.wave)
    d_cw = torch.from_numpy(d_cw_np).to(dev)
    d_in = torch.empty((F, W), dtype=torch.int32, device=dev)
    one.synth_bsc_device(d_cw.data_ptr(), 272, args.seed, 0, F, 0.006, d_in.data_ptr(), st)
    h_in = torch.empty((F, W), dtype=torch.int32).pin_memory(); h_in.copy_(d_in)
    del d_in
    res = {}
    outs = []
    for name, devs in (("one", [0]), ("many", list(range(world)))):
        dec = one if name == "one" else ldpc.Decoder(code, devices=devs, wave_frames=args.wave)
        h_bits = torch.empty((F, W), dtype=torch.int32).pin_memory()
        h_it = torch.empty(F, dtype=torch.int32).pin_memory()
        h_ok = torch.empty(F, dtype=torch.uint8).pin_memory()
        inp = ldpc.Input(kind=ldpc.IN_BSC_BITS, flags=0, data=h_in.data_ptr(), frame_stride=0, param=0.006, table=None)
        outp = ldpc.Output(bits=h_bits.data_ptr(), dblk=None, iters=h_it.data_ptr(), is_codeword=h_ok.data_ptr(), posterior=None, pchk=None)
        best = None
        for rep in range(3):  # first pass warms up (slot arrays and staging rings on every device)
            t0 = time.perf_counter()
            rc = ldpc.lib().dnaldpc_decode_batch(dec._h, ldpc.C.byref(inp), F, args.max_iter, ldpc.C.byref(outp))
            dt = time.perf_counter() - t0
            if rc:
                raise RuntimeError(ldpc.lib().dnaldpc_last_error())
            if rep > 0:
                best = dt if best is None else min(best, dt)
        res[name] = best
        outs.append((h_bits, h_it, h_ok))
        dec.close()
    same = all(bool(torch.equal(a, b)) for a, b in zip(outs[0], outs[1]))
    fi = float(outs[0][1].sum().item())
    return {"workload": "one batch of %d frames, BSC eps=0.006, max %d iterations, host buffers, rank 0 only" % (F, args.max_iter),
            "devices": world, "gbit_s": F * N / res["many"] / 1e9, "frame_iters_per_s": fi / res["many"],
            "one_device_gbit_s": F * N / res["one"] / 1e9, "speedup_vs_1": res["one"] / res["many"],
            "efficiency": res["one"] / res["many"] / world, "identical_to_one_device": same}


def run_ours(args):
    import torch
    import torch.distributed as dist
    import _pkg
    ldpc = _pkg.load()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the decoder has no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    code = ldpc.Code(PCHK)
    prec = ldpc.PREC_F32 if args.precision == "f32" else ldpc.PREC_F64
    bscale = 0.5 if args.precision == "f32" else 1.0   # fp32 messages / ratios are 4 bytes
    dec = ldpc.Decoder(code, devices=[local], wave_frames=args.wave, precision=prec)
    F = args.frames
    W = (N + 31) // 32
    frame0, _ = shard(F, rank)
    cw = np.fromfile(CW_BITS, dtype=np.uint8).view(np.int32).reshape(272, W)
    d_cw = torch.from_numpy(cw).to(dev)
    d_in = torch.empty((F, W), dtype=torch.int32, device=dev)
    d_bits = torch.empty((F, W), dtype=torch.int32, device=dev)
    d_it = torch.empty(F, dtype=torch.int32, device=dev)
    d_ok = torch.empty(F, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    dec.synth_bsc_device(d_cw.data_ptr(), 272, args.seed, frame0, F, args.eps, d_in.data_ptr(), stream)
    torch.cuda.synchronize()

    flags = ldpc.FLAG_MINSUM if args.alg == "minsum" else 0

    def step_device():
        inp_d = ldpc.Input(kind=ldpc.IN_BSC_BITS, flags=flags, data=d_in.data_ptr(), frame_stride=0, param=args.eps, table=None)
        out_d = ldpc.Output(bits=d_bits.data_ptr(), dblk=None, iters=d_it.data_ptr(), is_codeword=d_ok.data_ptr(), posterior=None, pchk=None)
        rc = ldpc.lib().dnaldpc_decode_batch_device(dec._h, ldpc.C.byref(inp_d), F, args.max_iter, ldpc.C.byref(out_d), stream)
        if rc:
            raise RuntimeError(ldpc.lib().dnaldpc_last_error())
        return dec.stats()["kernel_launches"]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_device()
    # in-pipeline trace (no synchronisation): real per-tick check-pass / bit-pass / scheduler times of a warm-up step
    dec.set_profiling(2)
    step_device()
    torch.cuda.synchronize()
    tr_row, tr_col, tr_sched, tr_ticks = dec.trace()
    dec.set_profiling(0)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    ev0.record()
    for _ in range(args.steps):
        launches += step_device()
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if rank == 0 else None
    frame_iters = int(d_it.sum().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_bits, d_it, d_ok)
    ms, frame_iters_all = aggregate(ms, frame_iters, dev, world)
    value = world * F * args.steps * N / (ms * 1e-3) / 1e9

    # ---- end to end through the host-buffer C-ABI call (pinned host memory, H2D + D2H inside the timed region)
    h_in = torch.empty((F, W), dtype=torch.int32).pin_memory()
    h_in.copy_(d_in)
    h_bits = torch.empty((F, W), dtype=torch.int32).pin_memory()
    h_it = torch.empty(F, dtype=torch.int32).pin_memory()
    h_ok = torch.empty(F, dtype=torch.uint8).pin_memory()
    C = ldpc.C
    inp = ldpc.Input(kind=ldpc.IN_BSC_BITS, flags=flags, data=h_in.data_ptr(), frame_stride=0, param=args.eps, table=None)
    out = ldpc.Output(bits=h_bits.data_ptr(), dblk=None, iters=h_it.data_ptr(), is_codeword=h_ok.data_ptr(), posterior=None, pchk=None)

    def step_host():
        rc = ldpc.lib().dnaldpc_decode_batch(dec._h, C.byref(inp), F, args.max_iter, C.byref(out))
        if rc:
            raise RuntimeError(ldpc.lib().dnaldpc_last_error())

    e2e_steps = max(1, args.e2e_steps if args.e2e_steps > 0 else args.steps)
    step_host()  # warm-up (staging buffers)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_host()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_val = world * F * e2e_steps * N / float(te[0]) / 1e9
    same = bool((h_it.to(dev) == d_it).all()) and bool((h_bits.to(dev) == d_bits).all())

    # ---- N > 1: the library's own multi-GPU dispatch is driven by rank 0 alone, later on; the other ranks free their
    # GPUs and wait on the store (no NCCL kernel is involved)
    want_inproc = world > 1 and args.inproc_frames > 0
    store = dist.distributed_c10d._get_default_store() if want_inproc else None
    if rank != 0 and want_inproc:
        import datetime
        del d_in, d_bits, d_it, d_ok, h_in, h_bits, h_it, h_ok, d_cw
        dec.close()
        torch.cuda.empty_cache()
        store.set("released_%d" % rank, "1")
        store.wait(["inproc_done"], datetime.timedelta(seconds=3000))
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel: per-launch CUDA-event timing (profiling mode syncs, so it runs apart from the timed region)
    peak, peak_src = peaks()
    pf = min(F, args.wave)
    dec.set_profiling(1)
    inp_p = ldpc.Input(kind=ldpc.IN_BSC_BITS, flags=flags, data=d_in.data_ptr(), frame_stride=0, param=args.eps, table=None)
    out_p = ldpc.Output(bits=d_bits.data_ptr(), dblk=None, iters=d_it.data_ptr(), is_codeword=d_ok.data_ptr(), posterior=None, pchk=None)
    ldpc.lib().dnaldpc_decode_batch_device(dec._h, C.byref(inp_p), pf, min(args.max_iter, 24), C.byref(out_p), stream)
    torch.cuda.synchronize()
    st = dec.stats()
    dec.set_profiling(0)
    n_it = max(1, int(d_it[:pf].max().item()))
    act_fi = float(d_it[:pf].sum().item())  # frame-iterations actually processed by those launches
    row_ms, col_ms = st["row_ms"] / n_it, st["col_ms"] / n_it
    frames_per_launch = act_fi / n_it
    if row_ms >= col_ms:
        kname, kms, kbytes = "row_pass_kernel (check-node)", row_ms, bscale * B_ROW * frames_per_launch
    else:
        kname, kms, kbytes = "col_pass_kernel (bit-node)", col_ms, bscale * B_COL * frames_per_launch
    achieved = kbytes / (kms * 1e-3) / 1e9
    roof = {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": None, "peak_source": peak_src, "launch_ms": kms, "frames_per_launch": frames_per_launch,
            "row_ms": row_ms, "col_ms": col_ms,
            "in_pipeline": {"row_ms": tr_row, "col_ms": tr_col, "scheduler_ms": tr_sched, "ticks": tr_ticks,
                            "note": "CUDA events inside the running pipeline (no sync): check pass, bit pass, and bit-pass end -> next check-pass start"},
            "iteration": {"achieved": bscale * B_ITER * frames_per_launch / ((row_ms + col_ms) * 1e-3) / 1e9,
                          "note": "B_iter=32E+8.25N per frame-iteration over row+col kernel time"},
            "whole_step": {"achieved": bscale * B_ITER * (frame_iters_all / world) / (ms / args.steps * 1e-3) / 1e9,
                           "note": "B_iter x frame-iterations of a step / step time (all kernels, launch gaps included)"}}
    tr = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tr):
        try:
            roof["traffic"] = json.load(open(tr)).get("row_per_frame" if row_ms >= col_ms else "col_per_frame") * frames_per_launch
            roof["traffic_source"] = "profiles/traffic.json: dram__bytes_read + dram__bytes_write of one ncu --set full capture of this kernel (profiles/r02/ncu_full_row_col.md), scaled to this launch; not re-measured in this run"
        except Exception:
            pass

    secondary = None
    if world == 1 and not args.no_secondary:
        secondary = secondary_regimes(ldpc, torch, dec, code, d_cw, args, peak)

    inproc = None
    if want_inproc:
        import datetime
        del d_in, d_bits, d_it, d_ok, h_in, h_bits, h_it, h_ok, d_cw
        dec.close()
        torch.cuda.empty_cache()
        try:
            store.wait(["released_%d" % r for r in range(1, world)], datetime.timedelta(seconds=600))
            inproc = inproc_multi(ldpc, torch, code, cw, args, world)
        except Exception as ex:  # reported, never fatal for the headline line
            inproc = {"error": repr(ex)}
        store.set("inproc_done", "1")

    cpu = None
    if not args.no_cpu and world == 1:
        info = cpu_reference_run(args.ref_frames_per_core, args.eps, args.max_iter)
        cpu = {"value": info["frames"] * N / info["decode_s"] / 1e9, "unit": "Gbit/s", "cores": info["cores"], "kind": info["kind"],
               "sample": "%d frames (%d per core, one pinned process per core) x max %d iterations, eps=%g; %.2f ms per iteration per core"
                         % (info["frames"], args.ref_frames_per_core, args.max_iter, args.eps, info["ms_per_iter_per_core"])}

    line = {
        "metric": "decoded Gbit/s, n=18432 prprp", "value": value, "unit": "Gbit/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": args.precision, "data": "synthetic", "config": workload_config(args, F),
        "frame_iters_per_s": frame_iters_all * args.steps / (ms * 1e-3),
        "avg_iters": frame_iters_all / (world * F),
        "e2e": {"value": e2e_val, "unit": "Gbit/s", "h2d_bytes_per_step": F * W * 4, "d2h_bytes_per_step": F * (W * 4 + 5),
                "steps": e2e_steps, "matches_device_path": same},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
    }
    if secondary is not None:
        line["secondary"] = secondary
    if inproc is not None:
        line["inproc_multi"] = inproc
    emit(line)
    if world > 1:
        dist.destroy_process_group()


_OUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout. Libraries write there too (NCCL prints its version banner on fd 1 when
    NCCL_DEBUG is set in the environment), so fd 1 is pointed at stderr for the whole run and the line goes to a private
    duplicate of the original stdout."""
    global _OUT
    sys.stdout.flush()
    _OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line):
    out = _OUT if _OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=100000, help="frames per GPU per step")
    ap.add_argument("--eps", type=float, default=0.02)
    ap.add_argument("--max-iter", type=int, default=100)
    ap.add_argument("--wave", type=int, default=4096)
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--e2e-steps", type=int, default=0, help="timed steps of the host-buffer leg (default: --steps)")
    ap.add_argument("--ref-frames-per-core", type=int, default=4)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary regimes (converging frames, configs 3-5, fp32, min-sum, host-buffer kinds)")
    ap.add_argument("--secondary", default="all", help="comma-separated subset of the secondary regimes: bsc,vote,awgn,llr,minsum_fp32,c5,sw (default all)")
    ap.add_argument("--inproc-frames", type=int, default=1000000, help="N > 1: frames of the one batch rank 0 decodes through the library's own multi-GPU dispatch")
    ap.add_argument("--alg", default="bp", choices=["bp", "minsum"], help="bp = sum-product (the metric); minsum = floating min-sum (SURVEY 8f-4)")
    ap.add_argument("--precision", default="f64", choices=["f64", "f32"], help="f64 = bit-exact mode (the metric); f32 = optional fast mode")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the decoded bits, iteration counts and codeword flags of the last timed step (rank 0) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3  # timing rule: W >= 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
