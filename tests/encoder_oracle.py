"""numpy oracle of the systematic form (include/dnaldpc.h, dnaldpc_code_systematic), written independently of the
library's elimination: Gauss-Jordan on dense bit rows of H with the column order reversed, pivots taken greedily
(rightmost column first). Test infrastructure only."""
import functools

import numpy as np


def dense(M, N, row_ptr, col_idx):
    """H as uint8 [M][N] (duplicate entries count once, as in the library's reader)."""
    H = np.zeros((M, N), np.uint8)
    H[np.repeat(np.arange(M), np.diff(row_ptr)), col_idx] = 1
    return H


def systematic(M, N, row_ptr, col_idx):
    """(info_cols, parity_cols, A) with A uint8 [R][K]: parity bit i = XOR_t A[i][t] m_t."""
    W = (N + 63) // 64
    rows = np.repeat(np.arange(M), np.diff(row_ptr))
    p = (N - 1 - np.asarray(col_idx, np.int64))            # position of column j in the reversed order
    B = np.zeros((M, W), np.uint64)
    np.bitwise_or.at(B, (rows, p // 64), np.left_shift(np.uint64(1), (p % 64).astype(np.uint64)))
    rank, piv_pos = 0, []
    for w in range(W):
        for b in range(64):
            pos = w * 64 + b
            if pos >= N or rank == M:
                break
            col = (B[rank:, w] >> np.uint64(b)) & np.uint64(1)
            nz = np.flatnonzero(col)
            if nz.size == 0:
                continue
            r = rank + nz[0]
            if r != rank:
                B[[rank, r]] = B[[r, rank]]
            hit = np.flatnonzero((B[:, w] >> np.uint64(b)) & np.uint64(1))
            hit = hit[hit != rank]
            if hit.size:                                    # the pivot row is zero before word w
                B[hit, w:] ^= B[rank, w:]
            piv_pos.append(pos)
            rank += 1
    R = rank
    parity_rev = np.array(piv_pos, np.int64)
    parity_cols = np.sort(N - 1 - parity_rev).astype(np.int32)
    is_par = np.zeros(N, bool)
    is_par[parity_cols] = True
    info_cols = np.flatnonzero(~is_par).astype(np.int32)
    # reduced row i has its pivot at reversed position piv_pos[i]; order rows by ascending parity column
    bits = np.unpackbits(B[:R].view(np.uint8), axis=1, bitorder="little")[:, :N]   # bit pos of reversed order
    red = bits[:, ::-1]                                                             # natural column order
    order = np.argsort(N - 1 - parity_rev)
    A = np.ascontiguousarray(red[order][:, info_cols])
    return info_cols, parity_cols, A


@functools.lru_cache(maxsize=None)
def systematic_of(name):
    """Cached oracle of the named test codes: 'n18432', 'small', 'sc', 'config4'."""
    return systematic(*csr_of(name))


@functools.lru_cache(maxsize=None)
def csr_of(name):
    import os
    import oraclelib as ol
    if name == "config4":
        import gen_regular_pchk
        row_ptr, col_idx = gen_regular_pchk.gen_regular(65536, 6554, 3, 5)
        return 6554, 65536, np.asarray(row_ptr, np.int32), np.asarray(col_idx, np.int32)
    path = {"n18432": ol.PCHK_18432, "small": os.path.join(ol.GOLDEN, "small_n120_m60.pchk"),
            "sc": os.path.join(ol.GOLDEN, "sc_z32_l12.pchk")}[name]
    o = ol.Oracle(path)
    return o.M, o.N, o.row_ptr.copy(), o.col_idx.copy()


def encode(A, info_cols, parity_cols, N, msg):
    """Codewords int8 [F][N] of message bits [F][K]: float32 products are exact (sums <= K < 2^24)."""
    msg = np.asarray(msg, np.float32)
    cw = np.zeros((msg.shape[0], N), np.int8)
    cw[:, info_cols] = msg
    if len(parity_cols):
        cw[:, parity_cols] = (msg @ A.T.astype(np.float32)).astype(np.int64) % 2
    return cw


def syndrome_ok(M, N, row_ptr, col_idx, cw):
    """True per frame when H c = 0 (sparse: XOR of the bits of every row)."""
    cw = np.asarray(cw, np.int64)
    s = np.add.reduceat(cw[:, col_idx], row_ptr[:-1], axis=1) if len(col_idx) else np.zeros((cw.shape[0], M), np.int64)
    empty = np.diff(row_ptr) == 0
    s[:, empty] = 0
    return ~(s % 2).any(axis=1)
