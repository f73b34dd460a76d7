"""ctypes wrapper of tests/layered_oracle.c, the sequential C restatement of the layered normalised min-sum decoder.

The shared library is compiled on first use into the system temporary directory (keyed by a hash of the source), so
the tests leave the tree untouched. Also: the channel LLRs of each input kind as the decoder computes them (the
LLR-domain setup of DNALDPC_FLAG_MINSUM), for feeding the oracle the same values."""
import ctypes as C
import hashlib
import math
import os
import subprocess
import tempfile

import numpy as np

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "layered_oracle.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(SRC, "rb").read()
        tag = hashlib.sha256(src).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "dnaldpc_layered_oracle_%d_%s.so" % (os.getuid(), tag))
        if not os.path.exists(so):
            tmp = "%s.%d.tmp" % (so, os.getpid())
            subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-std=c11", "-fPIC", "-shared", "-o", tmp, SRC, "-lm"])
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.lo_layers.restype = C.c_int
        L.lo_layers.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        for name in ("lo_layered_minsum_decode_f64", "lo_layered_minsum_decode_f32"):
            getattr(L, name).restype = None
            getattr(L, name).argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                         C.c_int, C.c_int, C.c_int, C.c_double] + [C.c_void_p] * 5
        _lib = L
    return _lib


def layers(M, N, row_ptr, col_idx):
    """(n_layers, layer_of_row int32 [M]) by first fit."""
    row_ptr = np.ascontiguousarray(row_ptr, np.int32)
    col_idx = np.ascontiguousarray(col_idx, np.int32)
    lay = np.zeros(M, np.int32)
    n = lib().lo_layers(M, N, row_ptr.ctypes.data, col_idx.ctypes.data, lay.ctypes.data)
    return n, lay


class Layered:
    """The oracle bound to one code (row_ptr / col_idx as exported by ldpc.Code.export())."""

    def __init__(self, M, N, row_ptr, col_idx):
        self.M, self.N = M, N
        self.row_ptr = np.ascontiguousarray(row_ptr, np.int32)
        self.col_idx = np.ascontiguousarray(col_idx, np.int32)
        self.n_layers, self.layer_of_row = layers(M, N, self.row_ptr, self.col_idx)

    def decode(self, llr, max_iter, alpha=1.0, fixed=False, f32=False):
        """llr: float64 [F][N] channel LLRs. Returns dict(iters, ok, dblk, pchk, post) like Decoder.decode."""
        llr = np.ascontiguousarray(np.atleast_2d(llr), np.float64)
        F, M, N = llr.shape[0], self.M, self.N
        res = dict(iters=np.zeros(F, np.int32), ok=np.zeros(F, np.uint8), dblk=np.zeros((F, N), np.uint8),
                   pchk=np.zeros((F, M), np.uint8), post=np.zeros((F, N), np.float64))
        fn = lib().lo_layered_minsum_decode_f32 if f32 else lib().lo_layered_minsum_decode_f64
        fn(M, N, self.row_ptr.ctypes.data, self.col_idx.ctypes.data, self.layer_of_row.ctypes.data, self.n_layers,
           llr.ctypes.data, F, max_iter, int(fixed), float(alpha), res["iters"].ctypes.data, res["ok"].ctypes.data,
           res["dblk"].ctypes.data, res["pchk"].ctypes.data, res["post"].ctypes.data)
        return res


# Channel LLRs as the decoder's min-sum setup computes them (bp_kernels.cuh load_llr, engine.cu tables; libm log).
def llr_bsc(recv_bits, p):
    t = np.array([math.log((1 - p) / p), math.log(p / (1 - p))])
    return t[np.asarray(recv_bits, np.int64)]


def llr_awgn_f32(y, sigma):
    return (2.0 * np.asarray(y, np.float32).astype(np.float64)) / (sigma * sigma)


def llr_vote(k, eps):
    L = math.log((1 - eps) / eps)
    return np.asarray(k, np.int64).astype(np.float64) * L
