"""Layered normalised min-sum (FLAG_MINSUM | FLAG_LAYERED, pytest -m gpu) against the sequential C oracle
(tests/layered_oracle.c): bit-exact decisions, iteration counts, flags, syndromes and posteriors in both precisions, for
every input kind at a waterfall point, normalised and not, with fixed iterations, on four codes; identical results over
host / device buffers, wave sizes and GPUs; re-decoding sweeps and the simulator; error paths and the command line."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import _pkg
import gen_regular_pchk
import layered_oracle as lo
import oraclelib as ol
import sim_oracle as so

ldpc = _pkg.load()
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LDPC = os.path.join(ROOT, "dna-ldpc-codes_b200", "ldpc")
pytestmark = pytest.mark.gpu

LAY = ldpc.FLAG_MINSUM | ldpc.FLAG_LAYERED
BSC, AWGN, VOTE, LLR = ldpc.IN_BSC_BITS, ldpc.IN_AWGN_F32, ldpc.IN_VOTE_I8, ldpc.IN_LLR_F64
MAX_ITER = 30
SEED = 5
READ_ERR = 0.01
WANT = ("bits", "dblk", "iters", "ok", "post", "pchk")
_codes, _decs, _orcs, _picked = {}, {}, {}, {}


def _code(name):
    if name not in _codes:
        if name == "n65536":
            row_ptr, col_idx = gen_regular_pchk.gen_regular(65536, 6554, 3, 5)
            _codes[name] = ldpc.Code(csr=(6554, 65536, row_ptr, col_idx))
        else:
            _codes[name] = ldpc.Code({"n18432": ol.PCHK_18432, "small": os.path.join(ol.GOLDEN, "small_n120_m60.pchk"),
                                      "sc": os.path.join(ol.GOLDEN, "sc_z32_l12.pchk")}[name])
    return _codes[name]


def _dec(name, f32=False, wave=0, devices=(0,)):
    key = (name, f32, wave, devices)
    if key not in _decs:
        _decs[key] = ldpc.Decoder(_code(name), devices=list(devices), precision=ldpc.PREC_F32 if f32 else ldpc.PREC_F64,
                                  wave_frames=wave)
    return _decs[key]


def _orc(name):
    if name not in _orcs:
        c = _code(name)
        _orcs[name] = lo.Layered(c.M, c.N, *c.export()[:2])
    return _orcs[name]


def _channel(kind, cws, x, seed=SEED):
    """Channel values of the codewords for a waterfall point x, as (decoder input, param, oracle LLRs)."""
    F, N = cws.shape
    if kind in (BSC, LLR):
        recv = np.stack([cws[f] ^ ol.bsc_flips(seed, f, N, x) for f in range(F)]).astype(np.uint8)
        llr = lo.llr_bsc(recv, x)
        return (ldpc._pack_bits(recv), x, llr) if kind == BSC else (llr, 1.0, llr)
    if kind == AWGN:
        sigma = ldpc.std_dev(x, 0.9)
        y = np.stack([ol.synth_awgn(cws[f], seed, f, N, sigma) for f in range(F)]).astype(np.float32)
        return y, sigma, lo.llr_awgn_f32(y, sigma)
    k = np.stack([ol.synth_vote(cws[f], seed, f, N, x, READ_ERR) for f in range(F)]).astype(np.int8)
    return k, READ_ERR, lo.llr_vote(k, READ_ERR)


GRIDS = {BSC: [0.006, 0.007, 0.008, 0.009, 0.01, 0.012, 0.015, 0.02],
         AWGN: [4.2, 4.0, 3.8, 3.6, 3.4, 3.2, 3.0, 2.8, 2.6, 2.4, 2.2, 2.0],
         VOTE: [3.5, 3.4, 3.3, 3.25, 3.2, 3.15, 3.1, 3.05, 3.0, 2.9, 2.8]}


def pick(kind, alpha=0.75):
    """First grid point (easy to hard) where layered fp64 fails on 10-90 % of the first 128 fixture codewords."""
    key = (kind, alpha)
    if key not in _picked:
        grid_kind = BSC if kind == LLR else kind
        dec = _dec("n18432")
        dec.set_minsum_scale(alpha)
        cws = ol.load_codewords()[:128]
        seen = []
        for x in GRIDS[grid_kind]:
            data, param, _ = _channel(grid_kind, cws, x)
            r = dec.decode(grid_kind, data, MAX_ITER, param=param, flags=LAY, want=("ok",))
            fer = 1 - r["ok"].mean()
            seen.append((x, fer))
            if 0.1 <= fer <= 0.9:
                _picked[key] = x
                break
        else:
            pytest.fail("no grid point in the waterfall: %s" % seen)
    return _picked[key]


def _check(got, want, what):
    for k in ("iters", "ok", "dblk", "pchk"):
        assert np.array_equal(got[k], want[k]), (what, k, np.flatnonzero((np.atleast_2d(got[k]) != np.atleast_2d(want[k])).any(axis=-1))[:8])
    assert np.array_equal(got["bits"].astype(np.uint8), want["dblk"]), what
    assert np.array_equal(got["post"].view(np.uint64), want["post"].view(np.uint64)), (what, "posterior")


@pytest.mark.parametrize("kind", [BSC, AWGN, VOTE, LLR])
@pytest.mark.parametrize("f32", [False, True])
@pytest.mark.parametrize("alpha", [1.0, 0.75])
def test_fixture_codewords_exact(kind, f32, alpha):
    x = pick(kind)
    cws = ol.load_codewords()
    data, param, llr = _channel(kind, cws, x)
    dec = _dec("n18432", f32)
    dec.set_minsum_scale(alpha)
    got = dec.decode(kind, data, MAX_ITER, param=param, flags=LAY, want=WANT)
    want = _orc("n18432").decode(llr, MAX_ITER, alpha=alpha, f32=f32)
    _check(got, want, (kind, f32, alpha))
    if alpha == 0.75 and not f32:
        assert 0 < (1 - got["ok"]).sum() < len(cws) and len(set(got["iters"].tolist())) > 3
    # n = 0: the posterior is the channel LLR as the oracle computes it
    z = dec.decode(kind, data, 0, param=param, flags=LAY, want=("post", "iters"))
    assert (z["iters"] == 0).all()
    assert np.array_equal(z["post"], llr.astype(np.float32).astype(np.float64) if f32 else llr)


@pytest.mark.parametrize("f32", [False, True])
def test_llr_nan_and_out_of_range(f32):
    """The setup's NaN -> 0 and +-2^64 clamp of the channel LLRs, at n = 0 and through the iterations."""
    recv, llr = _small_frames(256, 0.06, seed=9)
    llr[:, :4] = [np.nan, 1e300, -2.0 ** 80, -np.inf]
    dec = _dec("small", f32)
    dec.set_minsum_scale(0.75)
    z = dec.decode(LLR, llr, 0, flags=LAY, want=("post",))
    assert z["post"][0, :4].tolist() == [0.0, 2.0 ** 64, -2.0 ** 64, -2.0 ** 64], z["post"][0, :4]
    got = dec.decode(LLR, llr, MAX_ITER, flags=LAY, want=WANT)
    _check(got, _orc("small").decode(llr, MAX_ITER, alpha=0.75, f32=f32), f32)


@pytest.mark.parametrize("f32", [False, True])
def test_fixed_iterations_exact(f32):
    x = pick(BSC)
    cws = ol.load_codewords()[:96]
    data, param, llr = _channel(BSC, cws, x)
    dec = _dec("n18432", f32)
    dec.set_minsum_scale(0.8125)
    got = dec.decode(BSC, data, 12, param=param, flags=LAY | ldpc.FLAG_FIXED_ITERS, want=WANT)
    assert (got["iters"] == 12).all()
    _check(got, _orc("n18432").decode(llr, 12, alpha=0.8125, fixed=True, f32=f32), f32)


def _small_frames(F, p, seed=3):
    dec = _dec("small")
    rng = np.random.default_rng(seed)
    cws = dec.encode(rng.integers(0, 2, (F, dec.K), dtype=np.int8))
    recv = (cws ^ np.stack([ol.bsc_flips(seed, f, dec.code.N, p) for f in range(F)])).astype(np.uint8)
    return recv, lo.llr_bsc(recv, p)


@pytest.mark.parametrize("f32", [False, True])
def test_many_small_code_frames_with_compaction(f32):
    F = 20000
    recv, llr = _small_frames(F, 0.06)
    dec = _dec("small", f32, wave=4096)
    dec.set_minsum_scale(0.75)
    got = dec.decode(BSC, ldpc._pack_bits(recv), 40, param=0.06, flags=LAY, want=WANT)
    st = dec.stats()
    want = _orc("small").decode(llr, 40, alpha=0.75, f32=f32)
    _check(got, want, f32)
    assert st["compactions"] > 0 and len(set(got["iters"].tolist())) > 5
    assert 0 < (1 - got["ok"]).sum() < F


@pytest.mark.parametrize("name,p", [("n65536", 0.004), ("sc", 0.03)])
def test_other_codes_exact(name, p):
    code = _code(name)
    F = 192
    recv = np.stack([ol.bsc_flips(SEED, f, code.N, p) for f in range(F)]).astype(np.uint8)   # all-zero codeword
    llr = lo.llr_bsc(recv, p)
    dec = _dec(name, wave=256)
    for alpha in (1.0, 0.6875):
        dec.set_minsum_scale(alpha)
        got = dec.decode(BSC, ldpc._pack_bits(recv), MAX_ITER, param=p, flags=LAY, want=WANT)
        _check(got, _orc(name).decode(llr, MAX_ITER, alpha=alpha), (name, alpha))
        assert len(set(got["iters"].tolist())) > 2


def test_host_device_stream_and_wave_agree():
    import torch
    x = pick(AWGN)
    cws = ol.load_codewords()
    y, sigma, _ = _channel(AWGN, cws, x)
    F, N = y.shape
    ref = _dec("n18432")
    ref.set_minsum_scale(0.75)
    want = ref.decode(AWGN, y, MAX_ITER, param=sigma, flags=LAY, want=("bits", "iters", "ok", "post"))
    small = _dec("n18432", wave=256)
    small.set_minsum_scale(0.75)
    got = small.decode(AWGN, y, MAX_ITER, param=sigma, flags=LAY, want=("bits", "iters", "ok", "post"))
    for k in ("bits", "iters", "ok", "post"):
        assert np.array_equal(got[k], want[k]), ("wave 256", k)
    s = torch.cuda.Stream()
    yd = torch.from_numpy(y).cuda()
    bits = torch.zeros((F, ref.words_per_frame), dtype=torch.int32, device="cuda")
    it = torch.zeros(F, dtype=torch.int32, device="cuda")
    ok = torch.zeros(F, dtype=torch.uint8, device="cuda")
    post = torch.zeros((F, N), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    ref.decode_device(AWGN, yd.data_ptr(), F, MAX_ITER, param=sigma, bits_ptr=bits.data_ptr(), iters_ptr=it.data_ptr(),
                      ok_ptr=ok.data_ptr(), post_ptr=post.data_ptr(), stream=s.cuda_stream, flags=LAY)
    s.synchronize()
    assert np.array_equal(bits.cpu().numpy().view(np.uint32), want["bits_packed"])
    assert np.array_equal(it.cpu().numpy(), want["iters"]) and np.array_equal(ok.cpu().numpy(), want["ok"])
    assert np.array_equal(post.cpu().numpy(), want["post"])


def test_multi_gpu_identical():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    x = pick(BSC)
    cws = ol.load_codewords()
    data, param, _ = _channel(BSC, cws, x)
    one, two = _dec("n18432", wave=256), _dec("n18432", wave=256, devices=(0, 1))
    for d in (one, two):
        d.set_minsum_scale(0.75)
    a = one.decode(BSC, data, MAX_ITER, param=param, flags=LAY, want=("bits", "iters", "ok", "post"))
    b = two.decode(BSC, data, MAX_ITER, param=param, flags=LAY, want=("bits", "iters", "ok", "post"))
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def test_redecode_sweep_matches_oracle_rounds():
    x = pick(VOTE)
    cws = ol.load_codewords()
    k, _, _ = _channel(VOTE, cws, x)
    eps = [0.01, 0.0095, 0.009, 0.0085]
    dec = _dec("n18432")
    dec.set_minsum_scale(0.75)
    got = dec.redecode_sweep_ex(VOTE, k, MAX_ITER, eps, flags=LAY, want=("bits", "iters", "ok", "post"))
    orc = _orc("n18432")
    F = len(cws)
    rounds, todo = np.zeros(F, np.int32), np.arange(F)
    want = {key: None for key in ("iters", "ok", "dblk", "post")}
    for r, e in enumerate(eps):
        o = orc.decode(lo.llr_vote(k[todo], e), MAX_ITER, alpha=0.75)
        if r == 0:
            want = o
        else:
            for key in want:
                want[key][todo] = o[key]
            rounds[todo] = r
        todo = todo[o["ok"] == 0]
        if len(todo) == 0:
            break
    assert rounds.max() > 0
    assert np.array_equal(got["rounds"], rounds)
    for key in ("iters", "ok", "post"):
        assert np.array_equal(got[key], want[key]), key
    assert np.array_equal(got["bits"].astype(np.uint8), want["dblk"])


@pytest.mark.parametrize("channel,x", [(BSC, 0.1), (AWGN, 3.0)])
def test_simulate_matches_composition(channel, x):
    from test_gpu_sim import compose   # the same frames rebuilt from the public entry points
    dec = _dec("small", wave=256)
    dec.set_minsum_scale(0.75)
    param = x if channel == BSC else ldpc.std_dev(x, dec.K / dec.code.N)
    F = 5000
    want = so.totals(compose(dec, channel, param, F, flags=LAY, seed=SEED, max_iter=MAX_ITER), F)
    got = dec.simulate(channel, param, MAX_ITER, F, seed=SEED, flags=LAY)
    assert got == want
    assert 0 < got["frame_errors"] < F


def test_error_paths():
    dec = _dec("small")
    recv, llr = _small_frames(64, 0.06)
    L = ldpc.lib()
    with pytest.raises(ldpc.LdpcError) as ei:
        dec.decode(BSC, ldpc._pack_bits(recv), 10, param=0.06, flags=ldpc.FLAG_LAYERED)
    assert ei.value.rc == 6
    with pytest.raises(ldpc.LdpcError) as ei:
        dec.simulate(BSC, 0.06, 10, 10, flags=ldpc.FLAG_LAYERED)
    assert ei.value.rc == 6
    for a in (0.0, -0.5, 1.0000001, float("nan"), float("inf")):
        assert L.dnaldpc_set_minsum_scale(dec._h, a) == 1, a
    assert L.dnaldpc_set_minsum_scale(None, 0.5) == 1
    # the flooding min-sum decoder ignores the scale
    dec.set_minsum_scale(1.0)
    a = dec.decode(LLR, llr, 20, flags=ldpc.FLAG_MINSUM, want=("bits", "iters", "ok", "post"))
    dec.set_minsum_scale(0.75)
    b = dec.decode(LLR, llr, 20, flags=ldpc.FLAG_MINSUM, want=("bits", "iters", "ok", "post"))
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    o = ol.Oracle(os.path.join(ol.GOLDEN, "small_n120_m60.pchk")).decode_minsum(llr[0], 20)
    assert a["iters"][0] == o["n"]


def test_cli_layered_list_and_simulate(tmp_path):
    d = str(tmp_path)
    shutil.copyfile(ol.PCHK_18432, os.path.join(d, "H.pchk"))
    x = pick(BSC)
    cws = ol.load_codewords()[:6]
    _, _, llr = _channel(BSC, cws, x)
    names = []
    for f in range(len(cws)):
        with open(os.path.join(d, "cw%d.txt" % f), "w") as fh:
            fh.write("".join("%d " % b for b in cws[f]))
        with open(os.path.join(d, "llr%d.txt" % f), "w") as fh:
            fh.write("\n".join(repr(float(v)) for v in llr[f]))
        names.append(("cw%d" % f, "llr%d" % f))
    with open(os.path.join(d, "frames.lst"), "w") as fh:
        fh.write("".join("%s %s\n" % n for n in names))
    r = subprocess.run([LDPC, "0", "21", "0", "7", str(MAX_ITER), "1", "x", "x", "H", "0", "0", "0", "0", "--list", "frames.lst",
                        "--layered", "--scale", "0.6875"], cwd=d, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    dec = _dec("n18432")
    dec.set_minsum_scale(0.6875)
    want = dec.decode(LLR, llr, MAX_ITER, flags=LAY, want=("bits",))["bits"]
    for f, (cw, _) in enumerate(names):
        got = np.array(open(os.path.join(d, "dec_%s.txt" % cw)).read().split(), dtype=np.int8)
        assert np.array_equal(got, want[f]), f
    r = subprocess.run([LDPC, "--simulate", "H", "1", repr(x), "1", str(MAX_ITER), "200", "--decoder", "20", "--layered",
                        "--scale", "0.75"], cwd=d, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    dec.set_minsum_scale(0.75)
    want = dec.simulate(BSC, x, MAX_ITER, 200, seed=1, flags=LAY)
    assert "[0]  frame_err              : %d\n" % want["frame_errors"] in r.stdout
