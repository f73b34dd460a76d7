"""Pins the CPU restatement against the UNMODIFIED reference objects (oracle/_ref/libldpc_ref.so) on fresh seeded inputs -
beyond the committed golden vectors. CPU only.

The reference's results on these inputs are kept as digests in tests/golden/ref_seeded.json
(tools/make_golden_ref_seeded.py), so the comparison runs without the reference build; where oracle/_ref is built, every
case also goes through the live reference objects and must give the same digests."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import gen_sc_pchk
import oraclelib as ol

GOLDEN = os.path.join(ol.GOLDEN, "ref_seeded.json")
PCHK_SC = os.path.join(ol.GOLDEN, "sc_z32_l12.pchk")
BP_KEYS = ("n", "ok", "dblk", "pchk", "post", "pr", "lr")


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _digest(r, keys):
    """Integers as they are, arrays as the SHA-256 of their bytes (the bit patterns of the float64 ones)."""
    return {k: _sha(r[k]) if isinstance(r[k], np.ndarray) else int(r[k]) for k in keys}


def _compare(got, live):
    """`got` (the oracle's digests) against the stored reference digests and, where given, the live reference's."""
    want = json.load(open(GOLDEN))["cases"]
    for name, d in got.items():
        assert d == want[name], name
    if live is not None:
        assert live == got


# ---- the seeded cases; `dec` is an ol.Oracle or an ol.RefLib, which share these methods. name -> digest

def structure(dec):
    rp, ci = dec.export_csr() if isinstance(dec, ol.RefLib) else (dec.row_ptr, dec.col_idx)
    return {"structure": {"row_ptr": _sha(rp.astype(np.int32)), "col_idx": _sha(ci.astype(np.int32)),
                          "regular": list(dec.check_regular())}}


def random_frames(dec):
    cws = ol.load_codewords()
    rs = np.random.RandomState(2024)
    N = dec.N
    out = {}
    for t in range(8):
        f = int(rs.randint(272))
        kind = t % 4
        if kind == 0:
            eps = [0.005, 0.0075][t // 4 % 2]
            lr = np.where((cws[f] ^ ol.bsc_flips(100 + t, f, N, eps)) == 0, (1 - eps) / eps, eps / (1 - eps))
        elif kind == 1:
            sigma = 1 / np.sqrt(2 * (1 - 2048 / 18432) * 10 ** 0.42)
            lr = np.exp(2 * (np.where(cws[f] == 0, 1.0, -1.0) + sigma * rs.randn(N)) / sigma ** 2)
        elif kind == 2:
            k = rs.poisson(3.7, N) - 2 * rs.binomial(4, 0.02, N)
            lr = np.exp(np.where(cws[f] == 0, k, -k) * np.log(49.0))
        else:
            lr = np.exp(rs.uniform(-60, 60, N))  # garbage: exercises inf / NaN guards
        mi = [100, 30, 100, 12][kind]
        out["random_frames.%d" % t] = _digest(dec.decode(lr, mi, want_msgs=True), BP_KEYS)
    return out


def check_words(dec):
    rs = np.random.RandomState(5)
    d = (rs.rand(dec.N) < 0.3).astype(np.int8)
    w, p = dec.check(d)
    return {"check": {"weight": int(w), "pchk": _sha(p)}}


def fixed_iterations(dec):
    """Run_Belief_Propagation_Decoder_SAVE (dec.cpp:192-223): no early exit."""
    cws = ol.load_codewords()
    N = dec.N
    out = {}
    for f, eps, mi in [(3, 0.006, 9), (4, 0.0085, 5), (5, 0.004, 0)]:
        lr = np.where((cws[f] ^ ol.bsc_flips(77, f, N, eps)) == 0, (1 - eps) / eps, eps / (1 - eps))
        r = dec.decode_fixed(lr, mi)
        assert r["n"] == mi
        out["fixed.%d" % f] = _digest(r, ("n", "ok", "dblk", "pchk"))
    return out


def minsum(dec):
    """Run_MSA_Decoder_INF (dec.cpp:1216-1250): floating-point min-sum in the LLR domain."""
    cws = ol.load_codewords()
    N = dec.N
    rs = np.random.RandomState(12)
    sigma = 1 / np.sqrt(2 * (1 - 2048 / 18432) * 10 ** 0.5)
    cases = []
    for f, eps, mi in [(3, 0.004, 50), (4, 0.006, 30), (5, 0.004, 0), (6, 0.02, 3)]:
        cases.append((np.where((cws[f] ^ ol.bsc_flips(78, f, N, eps)) == 0, 1.0, -1.0) * np.log((1 - eps) / eps), mi))
    cases.append((2 * (np.where(cws[7] == 0, 1.0, -1.0) + sigma * rs.randn(N)) / sigma ** 2, 40))
    llr = np.where(cws[8] == 0, 1.0, -1.0) * rs.poisson(3.0, N) * np.log(49.0)   # many exact zeros and ties
    cases.append((llr, 25))
    return {"minsum.%d" % i: _digest(dec.decode_minsum(llr, mi), ("n", "ok", "dblk", "pchk", "post"))
            for i, (llr, mi) in enumerate(cases)}


def sliding_window(dec):
    """Run_SW_Decoder (dec.cpp:2092-2196) on the generated SC code (dec must hold sc_z32_l12.pchk), every final message."""
    M, N, rp, ci, Mv, Mc = gen_sc_pchk.gen_sc(32, 12, 11)
    rs = np.random.RandomState(99)
    out = {}
    for t in range(24):
        eps = [0.03, 0.05, 0.065, 0.08][t % 4]
        win = [3, 4, 6, 12][(t // 4) % 4]
        mi = [1, 8, 25][t % 3]
        llr = np.where(rs.rand(N) < eps, -1.0, 1.0) * rs.uniform(1.0, 4.0, N)
        llr[rs.rand(N) < 0.02] = 0.0
        r = dec.decode_sw(np.exp(llr), mi, 12, 3, win, Mv, Mc, want_msgs=True)
        out["sw.%d" % t] = _digest(r, ("n", "ok", "dblk", "pchk", "pr", "lr"))
    return out


@pytest.fixture(scope="module")
def pair():
    return ol.RefLib(ol.PCHK_18432) if ol.RefLib.available() else None, ol.Oracle(ol.PCHK_18432)


def _run(case, pair):
    ref, orc = pair
    _compare(case(orc), None if ref is None else case(ref))


def test_structure(pair):
    _run(structure, pair)


def test_bitexact_random_frames(pair):
    _run(random_frames, pair)


def test_check_matches(pair):
    _run(check_words, pair)


def test_fixed_iteration_variant(pair):
    _run(fixed_iterations, pair)


def test_minsum_variant(pair):
    _run(minsum, pair)


def test_sliding_window_variant_in_subprocess():
    """orc_sw_decode vs the reference's Run_SW_Decoder on fresh seeded inputs. The live reference runs in a child process:
    the reference object holds one .pchk per process."""
    got = sliding_window(ol.Oracle(PCHK_SC))
    live = None
    if ol.RefLib.available():
        here = os.path.dirname(os.path.abspath(__file__))
        code = ("import sys, json; sys.path[:0] = %r\nimport oraclelib as ol, test_oracle_vs_ref as t\n"
                "print(json.dumps(t.sliding_window(ol.RefLib(t.PCHK_SC))))" % [here, os.path.join(os.path.dirname(here), "tools")])
        res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
        assert res.returncode == 0, res.stderr
        live = json.loads(res.stdout.splitlines()[-1])
    _compare(got, live)
