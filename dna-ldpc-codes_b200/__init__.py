"""dna_ldpc_codes_b200 - thin ctypes binding over the C ABI (include/dnaldpc.h) of libdnaldpc.so.

The reference's decode path is compiled C++ with no library boundary; the product is the C-ABI shared library
(CUDA kernels + C++ host) and the `ldpc` CLI. This module only marshals numpy / torch buffers for tests and bench.py.
There is NO CPU fallback: if the library is missing, or no GPU is present when a decoder is created, it raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DNALDPC_LIB") or os.path.join(_HERE, "libdnaldpc.so")  # the override is for A/B runs of library builds

OK = 0
PREC_F64, PREC_F32 = 0, 1
IN_LR_F64, IN_LLR_F64, IN_BSC_BITS, IN_AWGN_F32, IN_AWGN_F64, IN_VOTE_I8 = range(6)
FLAG_HOST_EXP = 1
FLAG_FIXED_ITERS = 2
FLAG_MINSUM = 4

EXPORTS = [
    "dnaldpc_last_error", "dnaldpc_version", "dnaldpc_code_read_pchk", "dnaldpc_code_from_csr",
    "dnaldpc_code_write_pchk", "dnaldpc_code_free", "dnaldpc_code_dims", "dnaldpc_code_export",
    "dnaldpc_code_check_regular", "dnaldpc_decoder_create", "dnaldpc_decoder_destroy", "dnaldpc_decode_batch",
    "dnaldpc_decode_batch_device", "dnaldpc_run_bp_decoder", "dnaldpc_std_dev", "dnaldpc_vote_table",
    "dnaldpc_bsc_table", "dnaldpc_synth_bsc_device", "dnaldpc_get_stats", "dnaldpc_set_profiling",
    "dnaldpc_selftest_math", "dnaldpc_redecode_sweep", "dnaldpc_get_trace", "dnaldpc_decode_window",
    "dnaldpc_redecode_sweep_ex", "dnaldpc_synth_awgn_device", "dnaldpc_synth_vote_device", "dnaldpc_code_systematic",
    "dnaldpc_encode_device", "dnaldpc_encode", "dnaldpc_extract_device", "dnaldpc_extract", "dnaldpc_simulate",
]


class Config(C.Structure):
    _fields_ = [("n_devices", C.c_int32), ("devices", C.c_int32 * 16), ("precision", C.c_int32),
                ("wave_frames", C.c_int32), ("flags", C.c_int32)]


class Input(C.Structure):
    _fields_ = [("kind", C.c_int32), ("flags", C.c_int32), ("data", C.c_void_p), ("frame_stride", C.c_size_t),
                ("param", C.c_double), ("table", C.c_void_p)]


class Output(C.Structure):
    _fields_ = [("bits", C.c_void_p), ("dblk", C.c_void_p), ("iters", C.c_void_p), ("is_codeword", C.c_void_p),
                ("posterior", C.c_void_p), ("pchk", C.c_void_p)]


class Stats(C.Structure):
    _fields_ = [("frames", C.c_int64), ("frame_iters", C.c_int64), ("kernel_launches", C.c_int64),
                ("waves", C.c_int64), ("row_ms", C.c_double), ("col_ms", C.c_double), ("total_ms", C.c_double),
                ("compactions", C.c_int64)]


class Window(C.Structure):
    _fields_ = [("code_type", C.c_int32), ("L", C.c_int32), ("w", C.c_int32), ("win", C.c_int32),
                ("Mv", C.c_void_p), ("Mc", C.c_void_p)]


class Sim(C.Structure):
    _fields_ = [("channel", C.c_int32), ("flags", C.c_int32), ("param", C.c_double), ("mean_reads", C.c_double),
                ("seed", C.c_uint64), ("max_iter", C.c_int32), ("max_frames", C.c_int64), ("target_frame_errors", C.c_int64)]


class SimResult(C.Structure):
    _fields_ = [(k, C.c_int64) for k in ("frames", "iterations", "frame_errors", "bit_errors", "msg_frame_errors",
                                         "msg_bit_errors", "detected", "undetected", "raw_frame_errors", "raw_bit_errors")]


class LdpcError(RuntimeError):
    def __init__(self, rc, msg):
        super().__init__("dnaldpc error %d: %s" % (rc, msg))
        self.rc = rc


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("%s not built: run `make -C %s` (or __graft_entry__.build()); there is no CPU fallback"
                              % (LIB_PATH, _HERE))
        L = C.CDLL(LIB_PATH)
        L.dnaldpc_last_error.restype = C.c_char_p
        L.dnaldpc_version.restype = C.c_char_p
        L.dnaldpc_std_dev.restype = C.c_double
        L.dnaldpc_std_dev.argtypes = [C.c_double, C.c_double]
        L.dnaldpc_code_read_pchk.argtypes = [C.c_char_p, C.POINTER(C.c_void_p)]
        L.dnaldpc_code_from_csr.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]
        L.dnaldpc_code_write_pchk.argtypes = [C.c_void_p, C.c_char_p]
        L.dnaldpc_code_free.argtypes = [C.c_void_p]
        L.dnaldpc_code_free.restype = None
        L.dnaldpc_code_dims.argtypes = [C.c_void_p] + [C.POINTER(C.c_int)] * 3
        L.dnaldpc_code_export.argtypes = [C.c_void_p] * 5
        L.dnaldpc_code_check_regular.argtypes = [C.c_void_p] + [C.POINTER(C.c_int)] * 4
        L.dnaldpc_decoder_create.argtypes = [C.c_void_p, C.POINTER(Config), C.POINTER(C.c_void_p)]
        L.dnaldpc_decoder_destroy.argtypes = [C.c_void_p]
        L.dnaldpc_decoder_destroy.restype = None
        L.dnaldpc_decode_batch.argtypes = [C.c_void_p, C.POINTER(Input), C.c_int64, C.c_int, C.POINTER(Output)]
        L.dnaldpc_decode_batch_device.argtypes = [C.c_void_p, C.POINTER(Input), C.c_int64, C.c_int, C.POINTER(Output), C.c_void_p]
        L.dnaldpc_run_bp_decoder.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                             C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.dnaldpc_vote_table.argtypes = [C.c_double, C.c_void_p]
        L.dnaldpc_bsc_table.argtypes = [C.c_double, C.c_void_p]
        L.dnaldpc_synth_bsc_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_int64, C.c_int64,
                                               C.c_double, C.c_void_p, C.c_void_p]
        L.dnaldpc_get_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
        L.dnaldpc_set_profiling.argtypes = [C.c_void_p, C.c_int]
        L.dnaldpc_selftest_math.argtypes = [C.c_int64, C.c_uint64, C.POINTER(C.c_int64)]
        L.dnaldpc_get_trace.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int)]
        L.dnaldpc_redecode_sweep.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                             C.POINTER(Output), C.c_void_p]
        L.dnaldpc_redecode_sweep_ex.argtypes = [C.c_void_p, C.POINTER(Input), C.c_int64, C.c_int, C.c_void_p, C.c_int,
                                                C.POINTER(Output), C.c_void_p]
        L.dnaldpc_synth_awgn_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_int64, C.c_int64,
                                                C.c_double, C.c_void_p, C.c_void_p]
        L.dnaldpc_synth_vote_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_int64, C.c_int64,
                                                C.c_double, C.c_double, C.c_void_p, C.c_void_p]
        L.dnaldpc_decode_window.argtypes = [C.c_void_p, C.POINTER(Window), C.c_void_p, C.c_int64, C.c_int, C.POINTER(Output)]
        L.dnaldpc_code_systematic.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.c_void_p, C.c_void_p]
        for name in ("dnaldpc_encode_device", "dnaldpc_extract_device"):
            getattr(L, name).argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
        for name in ("dnaldpc_encode", "dnaldpc_extract"):
            getattr(L, name).argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
        L.dnaldpc_simulate.argtypes = [C.c_void_p, C.POINTER(Sim), C.POINTER(SimResult)]
        _lib = L
    return _lib


def _check(rc):
    if rc != OK:
        raise LdpcError(rc, lib().dnaldpc_last_error().decode(errors="replace"))


class Code:
    """Parity-check matrix (read_pchk, rcode.cpp:54-86)."""

    def __init__(self, pchk_path=None, csr=None):
        L = lib()
        self._h = C.c_void_p()
        if pchk_path is not None:
            _check(L.dnaldpc_code_read_pchk(os.fsencode(pchk_path), C.byref(self._h)))
        else:
            M, N, row_ptr, col_idx = csr
            row_ptr = np.ascontiguousarray(row_ptr, dtype=np.int32)
            col_idx = np.ascontiguousarray(col_idx, dtype=np.int32)
            _check(L.dnaldpc_code_from_csr(M, N, len(col_idx), row_ptr.ctypes.data, col_idx.ctypes.data, C.byref(self._h)))
        m, n, e = C.c_int(), C.c_int(), C.c_int()
        _check(L.dnaldpc_code_dims(self._h, C.byref(m), C.byref(n), C.byref(e)))
        self.M, self.N, self.E = m.value, n.value, e.value

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.dnaldpc_code_free(self._h)
            self._h = None

    def export(self):
        row_ptr = np.zeros(self.M + 1, np.int32); col_idx = np.zeros(self.E, np.int32)
        col_ptr = np.zeros(self.N + 1, np.int32); col_edge = np.zeros(self.E, np.int32)
        _check(lib().dnaldpc_code_export(self._h, row_ptr.ctypes.data, col_idx.ctypes.data, col_ptr.ctypes.data, col_edge.ctypes.data))
        return row_ptr, col_idx, col_ptr, col_edge

    def check_regular(self):
        v = [C.c_int() for _ in range(4)]
        _check(lib().dnaldpc_code_check_regular(self._h, *[C.byref(x) for x in v]))
        return tuple(x.value for x in v)

    def write_pchk(self, path):
        _check(lib().dnaldpc_code_write_pchk(self._h, os.fsencode(path)))

    def systematic(self):
        """(info_cols, parity_cols) of the systematic form (include/dnaldpc.h): K = len(info_cols) = N - rank(H)."""
        if getattr(self, "_sys", None) is None:
            K = C.c_int()
            info = np.zeros(self.N, np.int32); par = np.zeros(self.N, np.int32)
            _check(lib().dnaldpc_code_systematic(self._h, C.byref(K), info.ctypes.data, par.ctypes.data))
            self._sys = (info[:K.value].copy(), par[:self.N - K.value].copy())
        return self._sys


def _pack_bits(bits):
    """int8 / bool [F][n] -> uint32 [F][ceil(n/32)], LSB first."""
    bits = np.asarray(bits)
    F, n = bits.shape
    w = (n + 31) // 32
    b = np.zeros((F, w * 32), np.uint8)
    b[:, :n] = bits != 0
    return np.ascontiguousarray(np.packbits(b, axis=1, bitorder="little")).view(np.uint32)


def _unpack_bits(words, n):
    F = words.shape[0]
    return np.unpackbits(words.view(np.uint8).reshape(F, -1), axis=1, bitorder="little")[:, :n].astype(np.int8)


_KIND_DTYPE = {IN_LR_F64: np.float64, IN_LLR_F64: np.float64, IN_BSC_BITS: np.uint32, IN_AWGN_F32: np.float32,
               IN_AWGN_F64: np.float64, IN_VOTE_I8: np.int8}


class Decoder:
    """Batched BP decoder (Run_Belief_Propagation_Decoder, dec.cpp:583-605) on one or more GPUs."""

    def __init__(self, code, devices=None, precision=PREC_F64, wave_frames=0):
        self.code = code
        cfg = Config()
        if devices:
            cfg.n_devices = len(devices)
            for i, d in enumerate(devices):
                cfg.devices[i] = d
        cfg.precision = precision
        cfg.wave_frames = wave_frames
        self._h = C.c_void_p()
        _check(lib().dnaldpc_decoder_create(code._h, C.byref(cfg), C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.dnaldpc_decoder_destroy(self._h)
            self._h = None

    __del__ = close

    @property
    def words_per_frame(self):
        return (self.code.N + 31) // 32

    def decode(self, kind, data, max_iter, param=0.0, table=None, flags=0, want=("bits", "iters", "ok")):
        """HOST numpy buffers. data: [F][...] per `kind`. Returns dict of numpy arrays (bits unpacked to int8 [F][N])."""
        N, M = self.code.N, self.code.M
        data = np.ascontiguousarray(data, dtype=_KIND_DTYPE[kind])
        F = data.shape[0]
        inp = Input(kind=kind, flags=flags, data=data.ctypes.data, frame_stride=0, param=param, table=None)
        if table is not None:
            table = np.ascontiguousarray(table, dtype=np.float64)
            assert table.shape == (256,)
            inp.table = table.ctypes.data
        res, out = {}, Output()
        if "bits" in want:
            res["bits_packed"] = np.zeros((F, self.words_per_frame), np.uint32); out.bits = res["bits_packed"].ctypes.data
        if "dblk" in want:
            res["dblk"] = np.zeros((F, N), np.uint8); out.dblk = res["dblk"].ctypes.data
        if "iters" in want:
            res["iters"] = np.zeros(F, np.int32); out.iters = res["iters"].ctypes.data
        if "ok" in want:
            res["ok"] = np.zeros(F, np.uint8); out.is_codeword = res["ok"].ctypes.data
        if "post" in want:
            res["post"] = np.zeros((F, N), np.float64); out.posterior = res["post"].ctypes.data
        if "pchk" in want:
            res["pchk"] = np.zeros((F, M), np.uint8); out.pchk = res["pchk"].ctypes.data
        _check(lib().dnaldpc_decode_batch(self._h, C.byref(inp), F, max_iter, C.byref(out)))
        if "bits" in want:
            res["bits"] = np.unpackbits(res["bits_packed"].view(np.uint8).reshape(F, self.words_per_frame * 4), axis=1,
                                        bitorder="little")[:, :N].astype(np.int8)
        return res

    def redecode_sweep(self, llr, max_iter, scales, flags=0):
        """decoder.py:594-664 in one call: frames whose syndrome stays non-zero are re-decoded with LR = exp(scales[r]*LLR)."""
        llr = np.ascontiguousarray(llr, dtype=np.float64)
        scales = np.ascontiguousarray(scales, dtype=np.float64)
        F, N = llr.shape
        res = dict(bits_packed=np.zeros((F, self.words_per_frame), np.uint32), iters=np.zeros(F, np.int32),
                   ok=np.zeros(F, np.uint8), rounds=np.zeros(F, np.int32))
        out = Output(bits=res["bits_packed"].ctypes.data, iters=res["iters"].ctypes.data, is_codeword=res["ok"].ctypes.data)
        _check(lib().dnaldpc_redecode_sweep(self._h, llr.ctypes.data, F, max_iter, scales.ctypes.data, len(scales), flags,
                                            C.byref(out), res["rounds"].ctypes.data))
        res["bits"] = np.unpackbits(res["bits_packed"].view(np.uint8).reshape(F, self.words_per_frame * 4), axis=1,
                                    bitorder="little")[:, :N].astype(np.int8)
        return res

    def redecode_sweep_ex(self, kind, data, max_iter, params, flags=0, want=("bits", "iters", "ok")):
        """The sweep for any parameterised input kind: round r decodes with param = params[r]; inputs stay in HBM."""
        N, M = self.code.N, self.code.M
        data = np.ascontiguousarray(data, dtype=_KIND_DTYPE[kind])
        params = np.ascontiguousarray(params, dtype=np.float64)
        F = data.shape[0]
        inp = Input(kind=kind, flags=flags, data=data.ctypes.data, frame_stride=0, param=float(params[0]), table=None)
        res, out = dict(rounds=np.zeros(F, np.int32)), Output()
        if "bits" in want:
            res["bits_packed"] = np.zeros((F, self.words_per_frame), np.uint32); out.bits = res["bits_packed"].ctypes.data
        if "dblk" in want:
            res["dblk"] = np.zeros((F, N), np.uint8); out.dblk = res["dblk"].ctypes.data
        if "iters" in want:
            res["iters"] = np.zeros(F, np.int32); out.iters = res["iters"].ctypes.data
        if "ok" in want:
            res["ok"] = np.zeros(F, np.uint8); out.is_codeword = res["ok"].ctypes.data
        if "post" in want:
            res["post"] = np.zeros((F, N), np.float64); out.posterior = res["post"].ctypes.data
        if "pchk" in want:
            res["pchk"] = np.zeros((F, M), np.uint8); out.pchk = res["pchk"].ctypes.data
        _check(lib().dnaldpc_redecode_sweep_ex(self._h, C.byref(inp), F, max_iter, params.ctypes.data, len(params),
                                               C.byref(out), res["rounds"].ctypes.data))
        if "bits" in want:
            res["bits"] = np.unpackbits(res["bits_packed"].view(np.uint8).reshape(F, self.words_per_frame * 4), axis=1,
                                        bitorder="little")[:, :N].astype(np.int8)
        return res

    def decode_window(self, lratio, max_iter, L, w, win, Mv, Mc, code_type=0, want=("bits", "iters", "ok")):
        """Sliding-window BP for SC-LDPC codes (Run_SW_Decoder, dec.cpp:2092-2196). lratio: [F][N] p0/p1."""
        N, M = self.code.N, self.code.M
        lratio = np.ascontiguousarray(lratio, dtype=np.float64)
        Mv = np.ascontiguousarray(Mv, dtype=np.int32); Mc = np.ascontiguousarray(Mc, dtype=np.int32)
        F = lratio.shape[0]
        wd = Window(code_type=code_type, L=L, w=w, win=win, Mv=Mv.ctypes.data, Mc=Mc.ctypes.data)
        res, out = {}, Output()
        if "bits" in want:
            res["bits_packed"] = np.zeros((F, self.words_per_frame), np.uint32); out.bits = res["bits_packed"].ctypes.data
        if "dblk" in want:
            res["dblk"] = np.zeros((F, N), np.uint8); out.dblk = res["dblk"].ctypes.data
        if "iters" in want:
            res["iters"] = np.zeros(F, np.int32); out.iters = res["iters"].ctypes.data
        if "ok" in want:
            res["ok"] = np.zeros(F, np.uint8); out.is_codeword = res["ok"].ctypes.data
        if "pchk" in want:
            res["pchk"] = np.zeros((F, M), np.uint8); out.pchk = res["pchk"].ctypes.data
        _check(lib().dnaldpc_decode_window(self._h, C.byref(wd), lratio.ctypes.data, F, max_iter, C.byref(out)))
        if "bits" in want:
            res["bits"] = np.unpackbits(res["bits_packed"].view(np.uint8).reshape(F, self.words_per_frame * 4), axis=1,
                                        bitorder="little")[:, :N].astype(np.int8)
        return res

    def run_bp_decoder(self, lratio, max_iter):
        """One-frame drop-in with the reference's buffer contract (dec.h:80)."""
        lratio = np.ascontiguousarray(lratio, dtype=np.float64)
        dblk = np.zeros(self.code.N, np.int8); pchk = np.zeros(self.code.M, np.int8)
        ok, n = C.c_int(-1), C.c_int(-1)
        _check(lib().dnaldpc_run_bp_decoder(self._h, lratio.ctypes.data, max_iter, dblk.ctypes.data, pchk.ctypes.data,
                                            C.byref(ok), C.byref(n)))
        return dict(n=n.value, ok=ok.value, dblk=dblk, pchk=pchk)

    def decode_device(self, kind, data_ptr, F, max_iter, param=0.0, bits_ptr=None, iters_ptr=None, ok_ptr=None,
                      post_ptr=None, dblk_ptr=None, pchk_ptr=None, table_ptr=None, stream=None, frame_stride=0, flags=0):
        """DEVICE pointers (ints) of buffers on one GPU; the decoder's first device works on `stream` (a cudaStream_t as
        int, None = default stream), its other devices reach the buffers through peer access. `table_ptr` may be a host
        or a device pointer."""
        inp = Input(kind=kind, flags=flags, data=data_ptr, frame_stride=frame_stride, param=param, table=table_ptr)
        out = Output(bits=bits_ptr, dblk=dblk_ptr, iters=iters_ptr, is_codeword=ok_ptr, posterior=post_ptr, pchk=pchk_ptr)
        _check(lib().dnaldpc_decode_batch_device(self._h, C.byref(inp), F, max_iter, C.byref(out), stream))

    @property
    def K(self):
        return len(self.code.systematic()[0])

    def encode(self, msg):
        """HOST numpy: message bits int8 [F][K] -> codewords int8 [F][N] (systematic form of include/dnaldpc.h)."""
        msg = np.asarray(msg)
        assert msg.ndim == 2 and msg.shape[1] == self.K, msg.shape
        F = msg.shape[0]
        m = _pack_bits(msg)
        cw = np.zeros((F, self.words_per_frame), np.uint32)
        _check(lib().dnaldpc_encode(self._h, m.ctypes.data, F, cw.ctypes.data))
        return _unpack_bits(cw, self.code.N)

    def extract(self, bits):
        """HOST numpy: codeword bits int8 [F][N] -> message bits int8 [F][K] (the bits at the info columns)."""
        bits = np.asarray(bits)
        assert bits.ndim == 2 and bits.shape[1] == self.code.N, bits.shape
        F, K = bits.shape[0], self.K
        c = _pack_bits(bits)
        m = np.zeros((F, (K + 31) // 32), np.uint32)
        _check(lib().dnaldpc_extract(self._h, c.ctypes.data, F, m.ctypes.data))
        return _unpack_bits(m, K)

    def encode_device(self, msg_ptr, F, cw_ptr, stream=None):
        """DEVICE pointers (ints) on the decoder's first GPU: uint32 [F][ceil(K/32)] -> uint32 [F][ceil(N/32)]."""
        _check(lib().dnaldpc_encode_device(self._h, msg_ptr, F, cw_ptr, stream))

    def extract_device(self, cw_ptr, F, msg_ptr, stream=None):
        """DEVICE pointers (ints): uint32 [F][ceil(N/32)] -> uint32 [F][ceil(K/32)]."""
        _check(lib().dnaldpc_extract_device(self._h, cw_ptr, F, msg_ptr, stream))

    def synth_bsc_device(self, cw_bits_ptr, n_cw, seed, frame0, F, eps, out_bits_ptr, stream=None):
        _check(lib().dnaldpc_synth_bsc_device(self._h, cw_bits_ptr, n_cw, seed, frame0, F, eps, out_bits_ptr, stream))

    def synth_awgn_device(self, cw_bits_ptr, n_cw, seed, frame0, F, sigma, out_y_ptr, stream=None):
        _check(lib().dnaldpc_synth_awgn_device(self._h, cw_bits_ptr, n_cw, seed, frame0, F, sigma, out_y_ptr, stream))

    def synth_vote_device(self, cw_bits_ptr, n_cw, seed, frame0, F, mean_reads, read_err, out_k_ptr, stream=None):
        _check(lib().dnaldpc_synth_vote_device(self._h, cw_bits_ptr, n_cw, seed, frame0, F, mean_reads, read_err, out_k_ptr, stream))

    def simulate(self, channel, param, max_iter, max_frames, target_frame_errors=0, seed=0, flags=0, mean_reads=0.0):
        """Monte-Carlo error rates (dnaldpc_simulate): random codewords of the systematic encoder through the synthetic
        channel `channel` (IN_BSC_BITS p, IN_AWGN_F32 sigma, IN_VOTE_I8 read error probability + mean_reads), decoded
        and counted on the GPU; stops after the first `target_frame_errors` frame errors (0 = exactly max_frames)."""
        spec = Sim(channel=channel, flags=flags, param=param, mean_reads=mean_reads, seed=seed, max_iter=max_iter,
                   max_frames=max_frames, target_frame_errors=target_frame_errors)
        r = SimResult()
        _check(lib().dnaldpc_simulate(self._h, C.byref(spec), C.byref(r)))
        return {k: getattr(r, k) for k, _ in SimResult._fields_}

    def stats(self):
        s = Stats()
        _check(lib().dnaldpc_get_stats(self._h, C.byref(s)))
        return {k: getattr(s, k) for k, _ in Stats._fields_}

    def set_profiling(self, on):
        _check(lib().dnaldpc_set_profiling(self._h, int(on)))

    def trace(self):
        """(row_ms, col_ms, sched_ms, ticks) of the in-pipeline trace armed by set_profiling(2)."""
        r, c, g, n = C.c_double(), C.c_double(), C.c_double(), C.c_int()
        _check(lib().dnaldpc_get_trace(self._h, C.byref(r), C.byref(c), C.byref(g), C.byref(n)))
        return r.value, c.value, g.value, n.value


def selftest_math(n, seed=1):
    mm = C.c_int64(-1)
    _check(lib().dnaldpc_selftest_math(n, seed, C.byref(mm)))
    return mm.value


def std_dev(ebno_db, rate):
    return lib().dnaldpc_std_dev(ebno_db, rate)


def vote_table(eps):
    t = np.zeros(256, np.float64)
    _check(lib().dnaldpc_vote_table(eps, t.ctypes.data))
    return t


def bsc_table(p):
    t = np.zeros(2, np.float64)
    _check(lib().dnaldpc_bsc_table(p, t.ctypes.data))
    return t
