"""CPU-side checks of the systematic form behind the encoder (dnaldpc_code_systematic): the parity / info columns equal
those of the independent numpy oracle (tests/encoder_oracle.py) on the test codes and on a rank-deficient matrix, the
size cap, and the `ldpc --encode` argument and file errors, which come before any CUDA call."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import _pkg
import encoder_oracle as eo
import oraclelib as ol

ldpc = _pkg.load()
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LDPC = os.path.join(ROOT, "dna-ldpc-codes_b200", "ldpc")


def _check_against_oracle(M, N, row_ptr, col_idx, info_o, par_o):
    info, par = ldpc.Code(csr=(M, N, row_ptr, col_idx)).systematic()
    assert np.array_equal(info, info_o) and np.array_equal(par, par_o)
    assert np.array_equal(np.sort(np.concatenate([info, par])), np.arange(N))
    return info, par


@pytest.mark.parametrize("name,K", [("small", 60), ("sc", 322), ("n18432", 16572), ("config4", 58982)])
def test_systematic_matches_oracle(name, K):
    M, N, row_ptr, col_idx = eo.csr_of(name)
    info_o, par_o, _ = eo.systematic_of(name)
    info, par = _check_against_oracle(M, N, row_ptr, col_idx, info_o, par_o)
    assert len(info) == K and len(par) == N - K
    if name == "n18432":  # the 272 fixture codewords are codewords of this systematic form
        cws = ol.load_codewords()
        _, _, A = eo.systematic_of(name)
        assert np.array_equal(eo.encode(A, info, par, N, cws[:16][:, info]), cws[:16])


def test_rank_deficient_duplicates_and_empty_column():
    """Rows 2 = row 0 + row 1 (rank 3 of 4), a duplicated entry, and column 5 without entries (always an info column)."""
    rows = [[0, 1, 4, 4], [1, 2, 6], [0, 2, 4, 6], [3, 7, 0]]
    M, N = 4, 8
    row_ptr = np.cumsum([0] + [len(r) for r in rows]).astype(np.int32)
    col_idx = np.array(sum(rows, []), np.int32)
    info_o, par_o, A = eo.systematic(M, N, row_ptr, col_idx)
    info, par = _check_against_oracle(M, N, row_ptr, col_idx, info_o, par_o)
    assert len(par) == 3 and 5 in info and 7 in par
    # every codeword of this code is reproduced from its info bits
    H = eo.dense(M, N, row_ptr, col_idx).astype(np.int64)
    words = np.array([[(x >> j) & 1 for j in range(N)] for x in range(1 << N)], np.int8)
    cws = words[~((words.astype(np.int64) @ H.T) % 2).any(axis=1)]
    assert len(cws) == 1 << (N - 3)
    assert np.array_equal(eo.encode(A, info, par, N, cws[:, info]), cws)


def test_size_cap():
    # R x K = 16384 x 1032192 bits > 2^33
    M, N = 16384, 1 << 20
    c = ldpc.Code(csr=(M, N, np.arange(M + 1, dtype=np.int32), np.arange(M, dtype=np.int32)))
    with pytest.raises(ldpc.LdpcError) as ei:
        c.systematic()
    assert ei.value.rc == 6 and "2^33" in str(ei.value)
    # M x M elimination transform > 2^33 bits
    M = 100000
    c = ldpc.Code(csr=(M, 8, np.zeros(M + 1, np.int32), np.zeros(0, np.int32)))
    with pytest.raises(ldpc.LdpcError) as ei:
        c.systematic()
    assert ei.value.rc == 6 and "2^33" in str(ei.value)


def test_cli_encode_errors_before_cuda(tmp_path):
    d = str(tmp_path)
    shutil.copyfile(os.path.join(ol.GOLDEN, "small_n120_m60.pchk"), os.path.join(d, "S.pchk"))

    def run(*a):
        return subprocess.run([LDPC, "--encode"] + list(a), cwd=d, capture_output=True, text=True)
    for args in [("S",), ("S", "m"), ("S", "m", "c", "x"), ("S", "m", "--list", "l")]:
        r = run(*args)
        assert r.returncode == 1 and "usage: ldpc --encode" in r.stderr, args
    r = run("nosuch", "m", "c")
    assert r.returncode == 1 and "Can't open parity check file: nosuch.pchk" in r.stderr
    r = run("S", "m", "c")
    assert r.returncode == 1 and "Can't open input file: m.txt" in r.stderr
    open(os.path.join(d, "short.txt"), "w").write("1 " * 59)
    r = run("S", "short", "c")
    assert r.returncode == 1 and "short.txt holds fewer than 60" in r.stderr
    open(os.path.join(d, "two.txt"), "w").write("2 " * 60)
    r = run("S", "two", "c")
    assert r.returncode == 1 and "other than 0 or 1" in r.stderr
    r = run("S", "--list", "nolist")
    assert r.returncode == 1 and "Can't open list file: nolist" in r.stderr
    open(os.path.join(d, "empty.lst"), "w").write("")
    r = run("S", "--list", "empty.lst")
    assert r.returncode == 1 and "holds no" in r.stderr
    assert not os.path.exists(os.path.join(d, "c.txt"))
