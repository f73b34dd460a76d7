"""The Monte-Carlo simulator (dnaldpc_simulate, pytest -m gpu) against the same frames rebuilt from public pieces: twin
messages (tests/sim_oracle.py) -> encode_device -> synth_*_device -> decode_device -> counters in numpy. Also: results
independent of the piece size, wave_frames and the number of GPUs; the stopping rule; random against fixture codewords
on the BSC; `ldpc --simulate`; argument errors."""
import ctypes as C
import json
import math
import os
import shutil
import subprocess

import numpy as np
import pytest

import _pkg
import oraclelib as ol
import sim_oracle as so

ldpc = _pkg.load()
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LDPC = os.path.join(ROOT, "dna-ldpc-codes_b200", "ldpc")
SMALL = os.path.join(ol.GOLDEN, "small_n120_m60.pchk")
pytestmark = pytest.mark.gpu

MAX_ITER = 50
SEED = 11
BSC, AWGN, VOTE = ldpc.IN_BSC_BITS, ldpc.IN_AWGN_F32, ldpc.IN_VOTE_I8
READ_ERR = 0.01
_codes, _decoders, _picked = {}, {}, {}


def _dec(name, wave=256, devices=(0,)):
    key = (name, wave, devices)
    if key not in _decoders:
        if name not in _codes:
            _codes[name] = ldpc.Code(ol.PCHK_18432 if name == "n18432" else SMALL)
        _decoders[key] = ldpc.Decoder(_codes[name], devices=list(devices), wave_frames=wave)
    return _decoders[key]


def _with_piece(piece, fn):
    old = os.environ.get("DNALDPC_SIM_PIECE")
    if piece is None:
        os.environ.pop("DNALDPC_SIM_PIECE", None)
    else:
        os.environ["DNALDPC_SIM_PIECE"] = str(piece)
    try:
        return fn()
    finally:
        if old is None:
            os.environ.pop("DNALDPC_SIM_PIECE", None)
        else:
            os.environ["DNALDPC_SIM_PIECE"] = old


def _spec(dec, channel, x):
    """(param, mean_reads) of a search point x: p for the BSC, Eb/N0 in dB for AWGN, mean reads for vote counts."""
    if channel == AWGN:
        return ldpc.std_dev(x, dec.K / dec.code.N), 0.0
    if channel == VOTE:
        return READ_ERR, x
    return x, 0.0


def compose(dec, channel, param, F, flags=0, mean_reads=0.0, seed=SEED, max_iter=MAX_ITER):
    """Per-frame counters of frames 0..F-1 built from the public entry points."""
    import torch
    code = dec.code
    N, K, wpf = code.N, dec.K, dec.words_per_frame
    info, _ = code.systematic()
    msg = torch.from_numpy(so.messages(seed, 0, F, K).view(np.int32)).cuda()
    cw = torch.empty((F, wpf), dtype=torch.int32, device="cuda")
    dec.encode_device(msg.data_ptr(), F, cw.data_ptr())
    if channel == BSC:
        rx = torch.empty_like(cw)
        dec.synth_bsc_device(cw.data_ptr(), F, seed, 0, F, param, rx.data_ptr())
    elif channel == AWGN:
        rx = torch.empty((F, N), dtype=torch.float32, device="cuda")
        dec.synth_awgn_device(cw.data_ptr(), F, seed, 0, F, param, rx.data_ptr())
    else:
        rx = torch.empty((F, N), dtype=torch.int8, device="cuda")
        dec.synth_vote_device(cw.data_ptr(), F, seed, 0, F, mean_reads, param, rx.data_ptr())
    bits = torch.zeros_like(cw)
    iters = torch.zeros(F, dtype=torch.int32, device="cuda")
    ok = torch.zeros(F, dtype=torch.uint8, device="cuda")
    dec.decode_device(channel, rx.data_ptr(), F, max_iter, param=param, bits_ptr=bits.data_ptr(),
                      iters_ptr=iters.data_ptr(), ok_ptr=ok.data_ptr(), flags=flags)
    torch.cuda.synchronize()
    sent = cw.cpu().numpy().view(np.uint32)
    if channel == BSC:
        hard = rx.cpu().numpy().view(np.uint32)
    else:
        hard = ldpc._pack_bits(rx.cpu().numpy() < 0)
    return so.frame_counters(sent, bits.cpu().numpy().view(np.uint32), ok.cpu().numpy(), iters.cpu().numpy(), hard, info, N)


def pick(name, channel, grid, flags=0, F=512, need_undetected=False):
    """First point of `grid` (easy to hard) whose FER over F simulated frames lies in [0.1, 0.9] (and, if asked, with
    undetected errors): deterministic for a given build, it keeps the checks in the regime where both outcomes occur."""
    key = (name, channel, flags, need_undetected)
    if key not in _picked:
        dec = _dec(name)
        seen = []
        for x in grid:
            param, reads = _spec(dec, channel, x)
            r = dec.simulate(channel, param, MAX_ITER, F, seed=SEED, flags=flags, mean_reads=reads)
            fer = r["frame_errors"] / r["frames"]
            seen.append((x, fer, r["undetected"]))
            if 0.1 <= fer <= 0.9 and (r["undetected"] > 0 or not need_undetected):
                _picked[key] = x
                break
        else:
            pytest.fail("no point of the grid in the waterfall: %s" % seen)
    return _picked[key]


BSC_GRID = [0.006, 0.007, 0.0075, 0.008, 0.0085, 0.009, 0.01, 0.012, 0.015]
AWGN_GRID = [4.2, 4.0, 3.8, 3.6, 3.4, 3.2, 3.0, 2.8, 2.6, 2.4, 2.2, 2.0, 1.5]
VOTE_GRID = [3.5, 3.4, 3.3, 3.25, 3.2, 3.15, 3.1, 3.05, 3.0, 2.9, 2.8]
SMALL_GRID = [0.04, 0.06, 0.08, 0.1, 0.12, 0.14, 0.16, 0.18, 0.2]
SMALL_AWGN_GRID = [6.0, 5.0, 4.5, 4.0, 3.5, 3.0, 2.5, 2.0, 1.5, 1.0, 0.5, 0.0]
GRIDS = {("n18432", BSC): BSC_GRID, ("n18432", AWGN): AWGN_GRID, ("n18432", VOTE): VOTE_GRID, ("small", BSC): SMALL_GRID,
         ("small", AWGN): SMALL_AWGN_GRID}


# Plain (unnormalised) min-sum does not converge on the n=18432 code (check degree ~72: FER 1 from 4.2 dB / eps 0.006
# down), so its cases run on the small code, where both outcomes occur.
@pytest.mark.parametrize("name,channel,flags,F", [
    ("n18432", BSC, 0, 2000), ("n18432", AWGN, 0, 1500), ("n18432", VOTE, 0, 1500),
    ("n18432", BSC, ldpc.FLAG_FIXED_ITERS, 1000), ("small", BSC, 0, 20000),
    ("small", BSC, ldpc.FLAG_MINSUM, 5000), ("small", AWGN, ldpc.FLAG_MINSUM, 5000)])
def test_exact_against_composition(name, channel, flags, F):
    dec = _dec(name)
    undet = name == "small" and flags == 0
    x = pick(name, channel, GRIDS[(name, channel)], flags, F=F if undet else 512, need_undetected=undet)
    param, reads = _spec(dec, channel, x)
    want = so.totals(compose(dec, channel, param, F, flags=flags, mean_reads=reads), F)
    got = dec.simulate(channel, param, MAX_ITER, F, seed=SEED, flags=flags, mean_reads=reads)
    assert got == want, (x, got, want)
    assert 0 < got["frame_errors"] < got["frames"] == F
    assert got["frame_errors"] == got["detected"] + got["undetected"]
    assert got["raw_frame_errors"] > 0 and got["raw_bit_errors"] > 0
    if flags & ldpc.FLAG_FIXED_ITERS:
        assert got["iterations"] == F * MAX_ITER
    if undet:
        assert got["undetected"] > 0


def _bsc_case():
    dec = _dec("n18432")
    eps = pick("n18432", BSC, BSC_GRID)
    return dec, eps, compose(dec, BSC, eps, 2000)


def test_invariant_to_piece_size_and_wave():
    dec, eps, pf = _bsc_case()
    F = 2000
    want = so.totals(pf, F)
    fails = np.flatnonzero(pf["frame_errors"])
    T = max(1, len(fails) // 2)
    want_t = so.totals(pf, int(fails[T - 1]) + 1)
    for wave in (256, 4096):
        d = _dec("n18432", wave=wave)
        for piece in (None, 100, 77, 1000, 4096):
            got = _with_piece(piece, lambda: d.simulate(BSC, eps, MAX_ITER, F, seed=SEED))
            assert got == want, (wave, piece)
            got = _with_piece(piece, lambda: d.simulate(BSC, eps, MAX_ITER, F, target_frame_errors=T, seed=SEED))
            assert got == want_t, (wave, piece)
            st = d.stats()
            assert st["frames"] >= want_t["frames"]   # discarded frames are decoded and reported, never counted


def test_invariant_to_gpu_count():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    dec, eps, pf = _bsc_case()
    F = 2000
    fails = np.flatnonzero(pf["frame_errors"])
    T = max(1, len(fails) // 2)
    d2 = _dec("n18432", wave=256, devices=(0, 1))
    for piece in (100, 77):
        assert _with_piece(piece, lambda: d2.simulate(BSC, eps, MAX_ITER, F, seed=SEED)) == so.totals(pf, F)
        got = _with_piece(piece, lambda: d2.simulate(BSC, eps, MAX_ITER, F, target_frame_errors=T, seed=SEED))
        assert got == so.totals(pf, int(fails[T - 1]) + 1)


def test_stopping_rule():
    dec, eps, pf = _bsc_case()
    F = 2000
    fails = np.flatnonzero(pf["frame_errors"])
    assert len(fails) >= 3
    for T in (1, 2, len(fails) // 2, len(fails)):
        stop = int(fails[T - 1]) + 1
        got = _with_piece(64, lambda: dec.simulate(BSC, eps, MAX_ITER, F, target_frame_errors=T, seed=SEED))
        assert got["frames"] == stop and got == so.totals(pf, stop), T
        assert got["frame_errors"] == T
        # a cap below that point stops exactly at the cap
        cap = max(1, stop - 1)
        got = _with_piece(64, lambda: dec.simulate(BSC, eps, MAX_ITER, cap, target_frame_errors=T, seed=SEED))
        assert got == so.totals(pf, cap), T
    # a target beyond the errors of the run: exactly max_frames
    got = dec.simulate(BSC, eps, MAX_ITER, F, target_frame_errors=len(fails) + 1, seed=SEED)
    assert got == so.totals(pf, F)


def test_random_vs_fixture_codewords():
    import torch
    dec = _dec("n18432", wave=4096)
    eps = pick("n18432", BSC, BSC_GRID)
    F = 4096
    r = dec.simulate(BSC, eps, MAX_ITER, F, seed=SEED)
    p1 = r["frame_errors"] / F
    cws = ol.load_codewords()
    cw = torch.from_numpy(ldpc._pack_bits(cws).view(np.int32)).cuda()
    rx = torch.empty((F, dec.words_per_frame), dtype=torch.int32, device="cuda")
    dec.synth_bsc_device(cw.data_ptr(), len(cws), SEED, 0, F, eps, rx.data_ptr())
    bits = torch.zeros_like(rx)
    dec.decode_device(BSC, rx.data_ptr(), F, MAX_ITER, param=eps, bits_ptr=bits.data_ptr())
    torch.cuda.synchronize()
    sent = np.ascontiguousarray(ldpc._pack_bits(cws)[np.arange(F) % len(cws)])
    diff = sent ^ bits.cpu().numpy().view(np.uint32)
    diff[:, -1] &= np.uint32((1 << (dec.code.N % 32)) - 1 if dec.code.N % 32 else 0xFFFFFFFF)
    p2 = float((so.popcount_rows(diff) > 0).mean())
    assert 0.1 <= p1 <= 0.9 and 0.1 <= p2 <= 0.9, (eps, p1, p2)
    p = (p1 + p2) / 2
    assert abs(p1 - p2) <= 2.576 * math.sqrt(p * (1 - p) * 2 / F), (eps, p1, p2)   # two-proportion, 99 %


def test_cli_simulate(tmp_path):
    d = str(tmp_path)
    shutil.copyfile(ol.PCHK_18432, os.path.join(d, "H.pchk"))
    dec = _dec("n18432", wave=4096)
    eps = pick("n18432", BSC, BSC_GRID)
    points = [eps, BSC_GRID[BSC_GRID.index(eps) + 1]]
    r = subprocess.run([LDPC, "--simulate", "H", "1", ",".join(repr(p) for p in points), str(SEED), str(MAX_ITER), "600",
                        "--timing"], cwd=d, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lines = [json.loads(l) for l in r.stderr.splitlines() if l.startswith("{")]
    assert len(lines) == 2
    for i, (p, j) in enumerate(zip(points, lines)):
        want = dec.simulate(BSC, p, MAX_ITER, 600, seed=SEED)
        assert {k: j[k] for k in want} == want, (p, j, want)
        assert "[%d]  frame_err              : %d\n" % (i, want["frame_errors"]) in r.stdout
        assert "[%d]  without coding (bit)   : %d\n" % (i, want["raw_bit_errors"]) in r.stdout
        assert "[%d]  undetected             : %d\n" % (i, want["undetected"]) in r.stdout
    r = subprocess.run([LDPC, "--simulate", "H", "1", repr(eps), str(SEED), str(MAX_ITER), "0", "7", "--max-frames",
                        "100000", "--timing"], cwd=d, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    j = json.loads([l for l in r.stderr.splitlines() if l.startswith("{")][0])
    want = dec.simulate(BSC, eps, MAX_ITER, 100000, target_frame_errors=7, seed=SEED)
    assert want["frame_errors"] == 7 and {k: j[k] for k in want} == want


def test_argument_errors():
    dec = _dec("small")
    L = ldpc.lib()
    before = dec.stats()
    good = dict(channel=BSC, flags=0, param=0.05, mean_reads=0.0, seed=1, max_iter=10, max_frames=10, target_frame_errors=0)
    bad = [dict(channel=ldpc.IN_LR_F64), dict(channel=7), dict(flags=ldpc.FLAG_HOST_EXP), dict(flags=64),
           dict(param=0.0), dict(param=1.0), dict(param=float("nan")), dict(channel=AWGN, param=0.0),
           dict(channel=AWGN, param=-1.0), dict(channel=VOTE, param=0.01, mean_reads=0.0),
           dict(channel=VOTE, param=0.01, mean_reads=33.0), dict(channel=VOTE, param=1.5, mean_reads=3.0),
           dict(max_iter=-1), dict(max_frames=0), dict(target_frame_errors=-1)]
    r = ldpc.SimResult()
    for b in bad:
        s = ldpc.Sim(**dict(good, **b))
        assert L.dnaldpc_simulate(dec._h, C.byref(s), C.byref(r)) == 1, b
    s = ldpc.Sim(**good)
    assert L.dnaldpc_simulate(None, C.byref(s), C.byref(r)) == 1
    assert L.dnaldpc_simulate(dec._h, None, C.byref(r)) == 1
    assert L.dnaldpc_simulate(dec._h, C.byref(s), None) == 1
    assert dec.stats() == before   # nothing ran
    assert L.dnaldpc_simulate(dec._h, C.byref(s), C.byref(r)) == 0 and r.frames == 10
    # a code over the systematic form's cap (R x K > 2^33 bits): unsupported, as for dnaldpc_encode
    M, N = 16384, 1 << 20
    big = ldpc.Code(csr=(M, N, np.arange(M + 1, dtype=np.int32), np.arange(M, dtype=np.int32)))
    dbig = ldpc.Decoder(big, devices=[0], wave_frames=32)
    with pytest.raises(ldpc.LdpcError) as ei:
        dbig.simulate(BSC, 0.01, 10, 10)
    assert ei.value.rc == 6
    dbig.close()
