"""CPU-side checks of the layered min-sum decoder: dnaldpc_code_layers against the oracle's first fit and against the
definition, the sequential oracle's fixed point on noiseless codewords, and the command line's --layered / --scale
errors, which come before any CUDA call."""
import os
import subprocess

import numpy as np
import pytest

import _pkg
import gen_regular_pchk
import layered_oracle as lo
import oraclelib as ol

ldpc = _pkg.load()
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LDPC = os.path.join(ROOT, "dna-ldpc-codes_b200", "ldpc")
CODES = {"n18432": ol.PCHK_18432, "small": os.path.join(ol.GOLDEN, "small_n120_m60.pchk"),
         "sc": os.path.join(ol.GOLDEN, "sc_z32_l12.pchk")}
N_LAYERS = {"n18432": 8, "small": 7, "sc": 3, "n65536": 23}


def _code(name):
    if name == "n65536":
        row_ptr, col_idx = gen_regular_pchk.gen_regular(65536, 6554, 3, 5)
        return ldpc.Code(csr=(6554, 65536, row_ptr, col_idx))
    return ldpc.Code(CODES[name])


@pytest.mark.parametrize("name", ["n18432", "small", "sc", "n65536"])
def test_layers_match_oracle_and_definition(name):
    code = _code(name)
    row_ptr, col_idx, _, _ = code.export()
    n, lay = code.layers()
    n_orc, lay_orc = lo.layers(code.M, code.N, row_ptr, col_idx)
    assert n == n_orc == N_LAYERS[name]
    assert np.array_equal(lay, lay_orc)
    assert lay.min() == 0 and lay.max() == n - 1
    # rows in ascending order: each lands in a layer whose columns so far it does not touch, and clashes with every
    # lower layer (first fit)
    cols_of = [np.zeros(code.N, bool) for _ in range(n)]
    for i in range(code.M):
        cols = col_idx[row_ptr[i]:row_ptr[i + 1]]
        assert not cols_of[lay[i]][cols].any(), (name, i)
        for l in range(lay[i]):
            assert cols_of[l][cols].any(), (name, i, l)
        cols_of[lay[i]][cols] = True


def test_n18432_layers_are_the_row_blocks():
    n, lay = _code("n18432").layers()
    assert n == 8 and np.array_equal(lay, np.arange(2048) // 256)


def test_layers_of_degenerate_rows():
    # an empty row goes to layer 0; rows sharing one column each need a layer of their own
    code = ldpc.Code(csr=(4, 5, np.array([0, 0, 2, 4, 6]), np.array([0, 1, 0, 2, 0, 3])))
    n, lay = code.layers()
    assert n == 3 and lay.tolist() == [0, 0, 1, 2]
    n_orc, lay_orc = lo.layers(4, 5, *code.export()[:2])
    assert n_orc == n and np.array_equal(lay_orc, lay)


@pytest.mark.parametrize("f32", [False, True])
@pytest.mark.parametrize("alpha", [1.0, 0.75])
def test_oracle_noiseless_codewords_stop_at_once(f32, alpha):
    code = ldpc.Code(ol.PCHK_18432)
    orc = lo.Layered(code.M, code.N, *code.export()[:2])
    cws = ol.load_codewords()[:4]
    llr = lo.llr_bsc(cws, 0.01)
    r = orc.decode(llr, 20, alpha=alpha, f32=f32)
    assert (r["iters"] == 0).all() and (r["ok"] == 1).all()
    assert np.array_equal(r["dblk"], cws.astype(np.uint8)) and not r["pchk"].any()
    want = llr.astype(np.float32).astype(np.float64) if f32 else llr
    assert np.array_equal(r["post"], want)


def test_oracle_clamps_and_zeroes_nan():
    code = ldpc.Code(os.path.join(ol.GOLDEN, "small_n120_m60.pchk"))
    orc = lo.Layered(code.M, code.N, *code.export()[:2])
    llr = np.full((1, code.N), 3.0)
    llr[0, :4] = [np.nan, 1e300, -np.inf, 2.0 ** 70]
    r = orc.decode(llr, 0)
    assert r["post"][0, :4].tolist() == [0.0, 2.0 ** 64, -2.0 ** 64, 2.0 ** 64]
    assert r["dblk"][0, :4].tolist() == [1, 0, 1, 0]


def test_cli_layered_errors_before_cuda(tmp_path):
    d = str(tmp_path)

    def decode(dtype, *extra):
        window = ["0", "2", "12", "3"] if dtype == 60 else []   # <code_type> <w> <L> <WIN> of the sliding window
        return subprocess.run([LDPC, "0", str(dtype), "1", "7", "20", "1", "c", "s", "S", "0.05", "0", "0", "0"] + window +
                              list(extra), cwd=d, capture_output=True, text=True)
    for dtype in (0, 60):
        r = decode(dtype, "--layered")
        assert r.returncode == 1 and "--layered needs a min-sum decoder" in r.stderr, (dtype, r.stderr)
    r = decode(20, "--scale", "0.75")
    assert r.returncode == 1 and "--scale needs --layered" in r.stderr
    for a in ("0", "1.5", "-0.5", "x", "nan"):
        r = decode(21, "--layered", "--scale", a)
        assert r.returncode == 1 and "--scale must be in (0, 1]" in r.stderr, a

    def simulate(*a):
        return subprocess.run([LDPC, "--simulate", "S", "1", "0.05", "1", "10", "100"] + list(a), cwd=d,
                              capture_output=True, text=True)
    r = simulate("--layered")
    assert r.returncode == 1 and "--layered needs a min-sum decoder" in r.stderr and "usage: ldpc --simulate" in r.stderr
    r = simulate("--decoder", "20", "--scale", "0.5")
    assert r.returncode == 1 and "--scale needs --layered" in r.stderr
    r = simulate("--decoder", "20", "--layered", "--scale", "2")
    assert r.returncode == 1 and "--scale must be in (0, 1]" in r.stderr
