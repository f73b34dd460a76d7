"""CPU-side checks of the Monte-Carlo simulator (dnaldpc_simulate): the numpy twin of its message generator against a
pure-Python evaluation of the RNG specification, and the `ldpc --simulate` argument and file errors, which come before
any CUDA call."""
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
M64 = (1 << 64) - 1


def _rng_u64_int(seed, frame, bit, stream):
    """DESIGN.md §9 with Python integers (the specification, independent of numpy's uint64 arithmetic)."""
    def mix(z):
        z &= M64
        z ^= z >> 30; z = (z * 0xBF58476D1CE4E5B9) & M64
        z ^= z >> 27; z = (z * 0x94D049BB133111EB) & M64
        z ^= z >> 31
        return z
    x = mix(seed * 0x9E3779B97F4A7C15 + frame + 0x632BE59BD9B4E019)
    return mix(x ^ ((bit * 0xD6E8FEB86659FD93 + stream * 0xA0761D6478BD642F + 0x2545F4914F6CDD1D) & M64))


@pytest.mark.parametrize("seed,f0,K", [(0, 0, 16572), (7, 123456, 60), (2**63 + 5, 2**40, 33), (1, 5, 32)])
def test_message_twin_matches_specification(seed, f0, K):
    F, kw = 3, (K + 31) // 32
    words = so.messages(seed, f0, F, K)
    assert words.shape == (F, kw) and words.dtype == np.uint32
    for i in range(F):
        for w in sorted({0, kw // 2, kw - 1}):
            want = _rng_u64_int(seed, f0 + i, w, 1) & 0xFFFFFFFF
            if w == kw - 1 and K % 32:
                want &= (1 << (K % 32)) - 1
            assert int(words[i, w]) == want, (seed, f0 + i, w)
    bits = ldpc._unpack_bits(words, kw * 32)
    assert not bits[:, K:].any()                 # bits at and past K are zero
    if K % 32:
        assert bits[:, K - (K % 32):K].any()     # the kept bits of the last word are random, not cleared


def test_message_stream_differs_from_the_channel_streams():
    w = np.arange(64, dtype=np.uint64)
    s1 = ol.rng_u64(3, 9, w, 1)
    for stream in (0, 2, 3, 4, 5):
        assert not np.array_equal(s1, ol.rng_u64(3, 9, w, stream))


def test_frame_counters_twin():
    N, F = 40, 4
    rng = np.random.default_rng(1)
    sent = rng.integers(0, 2, (F, N), dtype=np.int8)
    dec = sent.copy()
    dec[1, 3] ^= 1                  # one bit error in an info column
    dec[2, [30, 39]] ^= 1           # two in parity columns
    hard = sent.copy()
    hard[0, :5] ^= 1
    ok = np.array([1, 1, 0, 1])
    info = np.arange(0, 20)
    pack = ldpc._pack_bits
    pf = so.frame_counters(pack(sent), pack(dec), ok, [3, 4, 5, 6], pack(hard), info, N)
    t = so.totals(pf, F)
    assert t == dict(frames=4, iterations=18, frame_errors=2, bit_errors=3, msg_frame_errors=1, msg_bit_errors=1,
                     detected=1, undetected=1, raw_frame_errors=1, raw_bit_errors=5)


def test_cli_simulate_errors_before_cuda(tmp_path):
    d = str(tmp_path)
    shutil.copyfile(os.path.join(ol.GOLDEN, "small_n120_m60.pchk"), os.path.join(d, "S.pchk"))

    def run(*a):
        return subprocess.run([LDPC, "--simulate"] + [str(x) for x in a], cwd=d, capture_output=True, text=True)
    for args in [(), ("S", 1, 0.05, 1, 10), ("S", 1, 0.05, 1, 10, 100, 5), ("S", 1, 0.05, 1, 10, 0, 5, 6)]:
        r = run(*args)
        assert r.returncode == 1 and "usage: ldpc --simulate" in r.stderr, (args, r.stderr)
    r = run("S", 1, 0.05, 1, 10, 0)                                  # frame_num 0 without a target
    assert r.returncode == 1 and "needs <target_frame_err>" in r.stderr
    r = run("S", 2, 0.05, 1, 10, 100)                                # the BEC
    assert r.returncode == 1 and "channel type 2 (BEC) is not supported" in r.stderr
    r = run("S", 5, 0.05, 1, 10, 100)
    assert r.returncode == 1 and "unknown channel type 5" in r.stderr
    r = run("S", 3, 0.01, 1, 10, 100)                                # vote counts without --reads
    assert r.returncode == 1 and "needs --reads" in r.stderr
    r = run("S", 3, 0.01, 1, 10, 100, "--reads", 40)
    assert r.returncode == 1 and "--reads must be in (0, 32]" in r.stderr
    for p in ("0.05,1.2", "0", "-0.1", "1"):                          # p out of range
        r = run("S", 1, p, 1, 10, 100)
        assert r.returncode == 1 and "is not in (0,1)" in r.stderr, p
    r = run("S", 1, "0.05,x", 1, 10, 100)
    assert r.returncode == 1 and "bad channel parameter list" in r.stderr
    r = run("S", 1, 0.05, 1, 10, 0, 5, "--max-frames", 0)
    assert r.returncode == 1 and "--max-frames must be a positive integer" in r.stderr
    r = run("S", 1, 0.05, 1, 10, 100, "--decoder", 21)
    assert r.returncode == 1 and "--decoder must be 0" in r.stderr
    r = run("nosuch", 1, 0.05, 1, 10, 100)                           # missing .pchk
    assert r.returncode == 1 and "Can't open parity check file: nosuch.pchk" in r.stderr
    # the reference's positional decode line still refuses frame_num 0
    r = subprocess.run([LDPC, "0", "0", "1", "7", "20", "0", "5", "c", "s", "S", "0.05", "0", "0", "0"], cwd=d,
                       capture_output=True, text=True)
    assert r.returncode == 1 and "frame_num 0" in r.stderr
