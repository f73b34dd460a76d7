"""The `ldpc` command line against outputs of the UNMODIFIED reference CLI (oracle/_ref/ldpc_ref, captured by
tools/make_golden.py): same argv (the pipeline's call, ex_decoder/def_func.py:49), same files in, byte-identical
stdout / dec_*.txt and identical result_*.txt apart from the two wall-clock lines."""
import hashlib
import json
import os
import shutil
import subprocess

import numpy as np
import pytest

import oraclelib as ol

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LDPC = os.path.join(ROOT, "dna-ldpc-codes_b200", "ldpc")


def _write_inputs(tmp, f, llr, cws):
    cwname, softname = "codeword_n18432_m1860_%d" % (f + 1), "soft_test_%d" % (f + 1)
    with open(os.path.join(tmp, cwname + ".txt"), "w") as fh:
        fh.write("".join("%d " % b for b in cws[f]))
    with open(os.path.join(tmp, softname + ".txt"), "w") as fh:
        fh.write("\n".join(str(float(x)) for x in llr))  # def_func.py:54-57 writes str(float)
    return cwname, softname


def _strip_times(txt):
    return [l for l in txt.splitlines() if not l.startswith(("start time", "end time", "simulation time"))]


@pytest.mark.parametrize("tag,f", [("a", 0), ("b", 1)])
def test_cli_matches_reference(tmp_path, tag, f):
    tmp = str(tmp_path)
    cws = ol.load_codewords()
    shutil.copyfile(ol.PCHK_18432, os.path.join(tmp, "decode_n18432_m2048_final.pchk"))
    llr = np.load(os.path.join(ol.GOLDEN, "cli_case_%s_llr.npy" % tag))
    cwname, softname = _write_inputs(tmp, f, llr, cws)
    res = subprocess.run([LDPC, "0", "0", "0", "7", "200", "1", cwname, softname, "decode_n18432_m2048_final", "0", "0", "0", "0"],
                         cwd=tmp, capture_output=True)
    assert res.returncode == 0, res.stderr
    assert res.stdout == open(os.path.join(ol.GOLDEN, "cli_case_%s_stdout.txt" % tag), "rb").read()
    dec = open(os.path.join(tmp, "dec_%s.txt" % cwname), "rb").read()
    assert hashlib.sha256(dec).hexdigest() == open(os.path.join(ol.GOLDEN, "cli_case_%s_dec.sha256" % tag)).read().strip()
    resname = "result_(%s.txt)_decode_n18432_m2048_final.pchk_0_0.000dB_0_200_7.txt" % softname
    got = open(os.path.join(tmp, resname)).read()
    want = open(os.path.join(ol.GOLDEN, "cli_case_%s_result.txt" % tag)).read()
    assert _strip_times(got) == _strip_times(want)


def test_cli_errors_and_batch_list(tmp_path):
    tmp = str(tmp_path)
    cws = ol.load_codewords()
    # argc mismatch -> "argc error!" + exit 1 (DNA_main.cpp:494-502); unreadable pchk -> exit 1 (rcode.cpp:60-64)
    r = subprocess.run([LDPC, "0", "0", "0", "7", "200", "1", "a", "b", "c", "0", "0", "0"], cwd=tmp, capture_output=True)
    assert r.returncode == 1 and b"argc error!" in r.stderr
    r = subprocess.run([LDPC, "0", "0", "0", "7", "200", "1", "a", "b", "nope", "0", "0", "0", "0"], cwd=tmp, capture_output=True)
    assert r.returncode == 1 and b"Can't open parity check file: nope.pchk" in r.stderr
    shutil.copyfile(ol.PCHK_18432, os.path.join(tmp, "H.pchk"))
    r = subprocess.run([LDPC, "0", "3", "0", "7", "200", "1", "a", "b", "H", "0", "0", "0", "0"], cwd=tmp, capture_output=True)
    assert r.returncode == 1 and b"not supported" in r.stderr
    r = subprocess.run([LDPC, "0", "0", "0", "7", "200", "1", "a", "b", "H", "0", "0", "0", "0"], cwd=tmp, capture_output=True)
    assert r.returncode == 1 and b"Can't open input file: a.txt" in r.stderr
    # --list: 5 frames in one process; every dec file equals the single-frame run's
    names = []
    for f in range(5):
        eps = 0.006
        llr = np.where((cws[f] ^ ol.bsc_flips(7, f, 18432, eps)) == 0, 1.0, -1.0) * np.log((1 - eps) / eps)
        names.append(_write_inputs(tmp, f, llr, cws))
    with open(os.path.join(tmp, "frames.lst"), "w") as fh:
        fh.write("".join("%s %s\n" % n for n in names))
    r = subprocess.run([LDPC, "0", "0", "0", "7", "200", "1", "x", "x", "H", "0", "0", "0", "0", "--list", "frames.lst", "--timing"],
                       cwd=tmp, capture_output=True)
    assert r.returncode == 0, r.stderr
    assert b'"frames": 5' in r.stderr
    for f, (cwname, _) in enumerate(names):
        got = np.array(open(os.path.join(tmp, "dec_%s.txt" % cwname)).read().split(), dtype=np.int8)
        assert np.array_equal(got, cws[f])
    assert b"frame_num              : 5" in r.stdout and b"bit_err                : 0" in r.stdout


# The side-by-side cases below compare our CLI with the unmodified reference CLI (oracle/_ref/ldpc_ref). What the
# reference printed and wrote for each case is kept in tests/golden/cli_side_by_side.json (tools/make_golden_cli_side.py),
# so the comparison runs without the reference build; where it is built, the live reference CLI is compared as well.
REF_CLI = os.path.join(ROOT, "oracle", "_ref", "ldpc_ref")
GOLDEN_SIDE = os.path.join(ol.GOLDEN, "cli_side_by_side.json")


def _record(r, d, dec_name, keep=lambda line: True):
    """stdout, SHA-256 of the dec file, result-file name and its body without the wall-clock lines: JSON-able."""
    assert r.returncode == 0, r.stderr
    res = [f for f in os.listdir(d) if f.startswith("result_")]
    assert len(res) == 1
    return {"stdout": r.stdout.decode("latin-1"),
            "dec_sha256": hashlib.sha256(open(os.path.join(d, dec_name), "rb").read()).hexdigest(),
            "result_name": res[0], "result": [line for line in _strip_times(open(os.path.join(d, res[0])).read()) if keep(line)]}


def _bp_case(exe, d, dectype):
    cws = ol.load_codewords()
    shutil.copyfile(ol.PCHK_18432, os.path.join(d, "H.pchk"))
    eps = 0.005
    llr = np.where((cws[3] ^ ol.bsc_flips(17, 3, 18432, eps)) == 0, 1.0, -1.0) * np.log((1 - eps) / eps) * np.linspace(0.7, 1.3, 18432)
    cwname, softname = _write_inputs(d, 3, llr, cws)
    r = subprocess.run([exe, "0", dectype, "0", "7", "60", "1", cwname, softname, "H", "0", "0", "0", "0"], cwd=d, capture_output=True)
    return _record(r, d, "dec_%s.txt" % cwname)


def _sw_case(exe, d, _=None):
    g = np.load(os.path.join(ol.GOLDEN, "golden_sw.npz"))
    N = 768
    rs = np.random.RandomState(8)
    llr = np.where(rs.rand(N) < 0.05, -1.0, 1.0) * rs.uniform(1.0, 4.0, N)
    shutil.copyfile(os.path.join(ol.GOLDEN, "sc_z32_l12.pchk"), os.path.join(d, "sc.pchk"))
    with open(os.path.join(d, "sc.txt"), "w") as fh:
        fh.write("".join("%d\n" % v for v in g["Mv"]) + "".join("%d\n" % v for v in g["Mc"]))
    with open(os.path.join(d, "cw.txt"), "w") as fh:
        fh.write("0 " * N)
    with open(os.path.join(d, "soft.txt"), "w") as fh:
        fh.write(" ".join(repr(float(x)) for x in llr))
    r = subprocess.run([exe, "0", "60", "0", "7", "20", "1", "cw", "soft", "sc", "0", "0", "0", "0", "0", "3", "12", "4"], cwd=d, capture_output=True)
    return _record(r, d, "dec_cw.txt", keep=lambda line: not line.startswith("BER["))


def _args_case(exe, d, args):
    N = 768
    rs = np.random.RandomState(12)
    llr = np.where(rs.rand(N) < 0.04, -1.0, 1.0) * rs.uniform(0.5, 4.0, N)
    shutil.copyfile(os.path.join(ol.GOLDEN, "sc_z32_l12.pchk"), os.path.join(d, "sc.pchk"))
    with open(os.path.join(d, "cw.txt"), "w") as fh:
        fh.write("0 " * N)
    with open(os.path.join(d, "soft.txt"), "w") as fh:
        fh.write(" ".join(repr(float(x)) for x in llr))
    r = subprocess.run([exe] + list(args), cwd=d, capture_output=True)
    return _record(r, d, "dec_cw.txt")


ARG_VARIANTS = [
    ("1", "0", "1", "7", "20", "3", "cw", "soft", "sc", "0.05", "0", "0", "0"),    # systematic count, BSC naming (%.4f), frame_num 3
    ("0", "0", "2", "5", "10", "1", "cw", "soft", "sc", "0.3", "0", "0", "0"),     # BEC naming / "Eps" lines
    ("0", "21", "0", "9", "15", "2", "cw", "soft", "sc", "1.5", "0", "0", "0"),    # min-sum type 21, Eb/N0 1.5 dB -> g_std_dev
    ("0", "0", "0", "7", "0", "1", "cw", "soft", "sc", "0", "0", "0", "0"),        # max_iter 0
]
# name -> (case, its parameter); the names key tests/golden/cli_side_by_side.json
SIDE_CASES = dict([("bp type 0", (_bp_case, "0")), ("bp type 20", (_bp_case, "20")), ("sw type 60", (_sw_case, None))]
                  + [("args " + " ".join(a), (_args_case, a)) for a in ARG_VARIANTS])


def _side_by_side(tmp_path, name):
    case, param = SIDE_CASES[name]
    outs = {}
    for who, exe in (("ours", LDPC), ("ref", REF_CLI)):
        if who == "ref" and not os.path.exists(REF_CLI):
            continue
        d = str(tmp_path / who)
        os.makedirs(d)
        outs[who] = case(exe, d, param)
    assert outs["ours"] == json.load(open(GOLDEN_SIDE))["cases"][name]
    if "ref" in outs:
        assert outs["ours"] == outs["ref"]


@pytest.mark.parametrize("dectype", ["0", "20"])
def test_cli_side_by_side_with_reference_binary(tmp_path, dectype):
    """Our CLI and the unmodified reference CLI on the same files: BP (type 0) and floating min-sum (type 20,
    Run_MSA_Decoder_INF)."""
    _side_by_side(tmp_path, "bp type " + dectype)


def test_cli_sliding_window_side_by_side(tmp_path):
    """Decoder type 60 (sliding-window BP, Run_SW_Decoder) with the reference's own argument block
    `<code_type> <w> <L> <WIN>` and node-count file <pchk_base>.txt: stdout, dec file, result-file name and the result
    file up to its BER lines (which the reference computes from an uninitialised counter, SURVEY section 5) must equal the
    unmodified reference CLI's. The POSITION_BER diagnostic file is not produced."""
    _side_by_side(tmp_path, "sw type 60")
    assert len(np.load(os.path.join(ol.GOLDEN, "golden_sw.npz"))["Mv"]) == 14


@pytest.mark.parametrize("args", ARG_VARIANTS)
def test_cli_argument_variants_side_by_side(tmp_path, args):
    """The positional arguments the pipeline never varies (bSystematic, channel type + parameter, frame_num, seed,
    max_iter 0) against the unmodified reference CLI on the small SC code: stdout, dec file, result-file name and body."""
    _side_by_side(tmp_path, "args " + " ".join(args))


def test_resident_worker_serves_the_unmodified_command_line(tmp_path):
    """`ldpc --serve` + the same binary as a thin client ($DNALDPC_SOCKET): the pipeline's serial one-process-per-codeword
    loop (ex_decoder/def_func.py:47-51) runs unchanged, every call answered by the worker with the stdout, the files
    and the exit code of a local run - also for the error cases and for two parity-check files in turn."""
    import json
    import time
    tmp = str(tmp_path)
    cws = ol.load_codewords()
    shutil.copyfile(ol.PCHK_18432, os.path.join(tmp, "H.pchk"))
    shutil.copyfile(os.path.join(ol.GOLDEN, "small_n120_m60.pchk"), os.path.join(tmp, "S.pchk"))
    names = []
    for f in range(6):
        eps = 0.006
        llr = np.where((cws[f] ^ ol.bsc_flips(7, f, 18432, eps)) == 0, 1.0, -1.0) * np.log((1 - eps) / eps)
        names.append(_write_inputs(tmp, f, llr, cws))
    rs = np.random.RandomState(5)
    with open(os.path.join(tmp, "cw_s.txt"), "w") as fh:
        fh.write("0 " * 120)
    with open(os.path.join(tmp, "soft_s.txt"), "w") as fh:
        fh.write("\n".join(str(float(x)) for x in rs.randn(120) + 2.0))
    sock = os.path.join(tmp, "w.sock")
    env = dict(os.environ, DNALDPC_SOCKET=sock)
    calls = [[LDPC, "0", "0", "0", "7", "200", "1", cw, sn, "H", "0", "0", "0", "0"] for cw, sn in names]
    calls.append([LDPC, "0", "0", "0", "7", "50", "1", "cw_s", "soft_s", "S", "0", "0", "0", "0"])
    calls.append([LDPC, "0", "0", "0", "7", "200", "1", "a", "b", "nope", "0", "0", "0", "0"])          # unreadable pchk
    calls.append([LDPC, "0", "0", "0", "7", "200", "1", "a", "b", "H", "0", "0", "0"])                  # argc error
    calls.append([LDPC, "0", "0", "0", "7", "200", "1", names[0][0], names[0][1], "H", "0", "0", "0", "0", "--timing"])
    local = []
    for c in calls:
        r = subprocess.run(c, cwd=tmp, capture_output=True)
        decs = {n: open(os.path.join(tmp, n), "rb").read() for n in sorted(os.listdir(tmp)) if n.startswith("dec_")}
        local.append((r.returncode, r.stdout, decs))
        for n in decs:
            os.unlink(os.path.join(tmp, n))
    worker = subprocess.Popen([LDPC, "--serve"], cwd="/", env=env, stderr=subprocess.PIPE)
    try:
        for _ in range(100):
            if os.path.exists(sock):
                break
            time.sleep(0.05)
        t_first = None
        for k, c in enumerate(calls):
            t0 = time.perf_counter()
            r = subprocess.run(c, cwd=tmp, capture_output=True, env=env)
            dt = time.perf_counter() - t0
            if k == 0:
                t_first = dt
            decs = {n: open(os.path.join(tmp, n), "rb").read() for n in sorted(os.listdir(tmp)) if n.startswith("dec_")}
            assert (r.returncode, r.stdout, decs) == local[k], (k, r.stderr)
            for n in decs:
                os.unlink(os.path.join(tmp, n))
            if k in (1, 2, 3, 4, 5):
                assert dt < 0.5 * max(t_first, 0.4), (k, dt, t_first)  # no CUDA context creation after the first call
        tj = json.loads(r.stderr.decode().strip().splitlines()[-1])
        assert tj["frames"] == 1 and len(tj["iterations"]) == 1 and tj["iterations"][0] == tj["total_iterations"]
        assert tj["gpu_init_ms"] == 0.0  # the decoder came from the worker's cache
    finally:
        subprocess.run([LDPC, "--shutdown"], env=env, capture_output=True)
        worker.wait(timeout=30)
    assert not os.path.exists(sock)


def test_cli_multi_gpu_list(tmp_path):
    """--gpus N: the frames of a --list batch decoded on every visible GPU by the library's own dispatcher; same dec files
    and stdout as on one GPU, per-frame iteration counts in the --timing line."""
    import json
    import torch
    nd = torch.cuda.device_count()
    if nd < 2:
        pytest.skip("needs at least 2 GPUs")
    tmp = str(tmp_path)
    cws = ol.load_codewords()
    shutil.copyfile(ol.PCHK_18432, os.path.join(tmp, "H.pchk"))
    names = []
    for f in range(96):
        eps = [0.004, 0.006, 0.0075][f % 3]
        llr = np.where((cws[f] ^ ol.bsc_flips(9, f, 18432, eps)) == 0, 1.0, -1.0) * np.log((1 - eps) / eps)
        names.append(_write_inputs(tmp, f, llr, cws))
    with open(os.path.join(tmp, "frames.lst"), "w") as fh:
        fh.write("".join("%s %s\n" % n for n in names))
    outs = []
    for g in (1, nd):
        r = subprocess.run([LDPC, "0", "0", "0", "7", "60", "1", "x", "x", "H", "0", "0", "0", "0", "--list", "frames.lst", "--timing",
                            "--gpus", str(g)], cwd=tmp, capture_output=True)
        assert r.returncode == 0, r.stderr
        tj = json.loads(r.stderr.decode().strip().splitlines()[-1])
        decs = [open(os.path.join(tmp, "dec_%s.txt" % cw), "rb").read() for cw, _ in names]
        outs.append((r.stdout, decs, tj["iterations"], tj["avg_iterations"]))
        assert tj["gpus"] == g and len(tj["iterations"]) == 96
    assert outs[0] == outs[1]
