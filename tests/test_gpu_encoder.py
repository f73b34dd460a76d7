"""The systematic encoder and message extraction on the GPU (pytest -m gpu), against the numpy oracle of
tests/encoder_oracle.py: the 272 fixture codewords, seeded random messages on four codes (every codeword also satisfies
H c = 0), unused high message bits, the round trip through the BSC generator and the decoder, the host and device
forms, and `ldpc --encode`."""
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
pytestmark = pytest.mark.gpu


def _decoder(name, **kw):
    M, N, row_ptr, col_idx = eo.csr_of(name)
    code = ldpc.Code(csr=(M, N, row_ptr, col_idx))
    return code, ldpc.Decoder(code, devices=[0], wave_frames=kw.get("wave_frames", 256))


def _words(bits):
    return ldpc._pack_bits(bits)


def _encode_device(dec, msg_words, stream=None):
    import torch
    F = msg_words.shape[0]
    m = torch.from_numpy(msg_words.view(np.int32)).cuda()
    cw = torch.full((F, dec.words_per_frame), -1, dtype=torch.int32, device="cuda")   # every word is written
    dec.encode_device(m.data_ptr(), F, cw.data_ptr(), stream=stream)
    torch.cuda.synchronize()
    return cw.cpu().numpy().view(np.uint32)


def test_fixture_codewords():
    code, dec = _decoder("n18432")
    info, par = code.systematic()
    cws = ol.load_codewords()
    assert np.array_equal(dec.encode(cws[:, info]), cws)
    assert np.array_equal(dec.extract(cws), cws[:, info])
    dec.close()


@pytest.mark.parametrize("name,Fs", [("small", (1, 31, 33, 300)), ("sc", (1, 33, 300)),
                                     ("n18432", (1, 31, 33, 4097, 20000)), ("config4", (300,))])
def test_random_messages_match_oracle(name, Fs):
    code, dec = _decoder(name)
    M, N, row_ptr, col_idx = eo.csr_of(name)
    info, par, A = eo.systematic_of(name)
    K, kw = len(info), (len(info) + 31) // 32
    rng = np.random.default_rng(len(name))
    for F in Fs:
        msg = rng.integers(0, 2, (F, K), dtype=np.int8)
        want = eo.encode(A, info, par, N, msg)
        words = _words(msg)
        if K % 32:  # garbage in the unused high bits of the last word must not change the output
            words[:, kw - 1] |= rng.integers(0, 1 << 32, F, dtype=np.uint64).astype(np.uint32) & np.uint32(~((1 << (K % 32)) - 1) & 0xffffffff)
        got = _encode_device(dec, words)
        if N % 32:
            assert not (got[:, -1] >> np.uint32(N % 32)).any()
        got = ldpc._unpack_bits(got, N)
        assert np.array_equal(got, want), (name, F)
        assert eo.syndrome_ok(M, N, row_ptr, col_idx, got).all(), (name, F)
    dec.close()


def test_round_trip_through_bsc_and_decoder():
    import torch
    code, dec = _decoder("n18432", wave_frames=4096)
    N, K, F = code.N, dec.K, 8192
    kw = (K + 31) // 32
    g = torch.Generator(device="cuda").manual_seed(5)
    msg = torch.randint(-2**31, 2**31 - 1, (F, kw), dtype=torch.int32, device="cuda", generator=g)
    msg[:, -1] &= (1 << (K % 32)) - 1
    cw = torch.empty((F, dec.words_per_frame), dtype=torch.int32, device="cuda")
    back = torch.empty_like(msg)
    dec.encode_device(msg.data_ptr(), F, cw.data_ptr())
    dec.extract_device(cw.data_ptr(), F, back.data_ptr())
    torch.cuda.synchronize()
    assert torch.equal(back, msg)
    # noise, decode, extract: every frame flagged as a codeword gives back its message
    recv = torch.empty_like(cw)
    dec.synth_bsc_device(cw.data_ptr(), F, 11, 0, F, 0.002, recv.data_ptr())
    bits = torch.empty_like(cw)
    ok = torch.zeros(F, dtype=torch.uint8, device="cuda")
    dec.decode_device(ldpc.IN_BSC_BITS, recv.data_ptr(), F, 100, param=0.002, bits_ptr=bits.data_ptr(), ok_ptr=ok.data_ptr())
    out = torch.empty_like(msg)
    dec.extract_device(bits.data_ptr(), F, out.data_ptr())
    torch.cuda.synchronize()
    good = ok.bool()
    assert torch.equal(out[good], msg[good])
    assert good.float().mean().item() >= 0.99, good.float().mean().item()
    dec.close()


def test_host_and_device_forms_agree_on_a_stream():
    import torch
    code, dec = _decoder("sc")
    N, K, F = code.N, dec.K, 5000
    rng = np.random.default_rng(9)
    msg = rng.integers(0, 2, (F, K), dtype=np.int8)
    host = dec.encode(msg)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        m = torch.from_numpy(_words(msg).view(np.int32)).cuda()
        cw = torch.zeros((F, dec.words_per_frame), dtype=torch.int32, device="cuda")
        back = torch.zeros_like(m)
        dec.encode_device(m.data_ptr(), F, cw.data_ptr(), stream=s.cuda_stream)
        dec.extract_device(cw.data_ptr(), F, back.data_ptr(), stream=s.cuda_stream)
    s.synchronize()
    assert np.array_equal(ldpc._unpack_bits(cw.cpu().numpy().view(np.uint32), N), host)
    assert np.array_equal(back.cpu().numpy(), m.cpu().numpy())
    assert np.array_equal(dec.extract(host), msg)
    # argument handling: F = 0 is a no-op, F < 0 and null buffers are errors
    dec.encode_device(0, 0, 0)
    for args in [(m.data_ptr(), -1, cw.data_ptr()), (0, 1, cw.data_ptr()), (m.data_ptr(), 1, 0)]:
        with pytest.raises(ldpc.LdpcError) as ei:
            dec.encode_device(*args)
        assert ei.value.rc == 1
    dec.close()


def test_cli_encode_list(tmp_path):
    d = str(tmp_path)
    shutil.copyfile(ol.PCHK_18432, os.path.join(d, "H.pchk"))
    code = ldpc.Code(ol.PCHK_18432)
    info, _ = code.systematic()
    cws = ol.load_codewords()[:16]
    with open(os.path.join(d, "enc.lst"), "w") as f:
        for k in range(16):
            open(os.path.join(d, "m%d.txt" % k), "w").write(" ".join(str(b) for b in cws[k, info]) + "\n")
            f.write("m%d c%d\n" % (k, k))
    r = subprocess.run([LDPC, "--encode", "H", "--list", "enc.lst", "--timing"], cwd=d, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert '"encode_ms"' in r.stderr
    for k in range(16):
        txt = open(os.path.join(d, "c%d.txt" % k)).read()
        assert txt == "".join("%d " % b for b in cws[k])                       # write_dec_txt format
        assert np.array_equal(np.array(txt.split(), np.int8), cws[k])
    # the decode command line reads them: noiseless LLRs, zero bit errors
    with open(os.path.join(d, "dec.lst"), "w") as f:
        for k in range(16):
            open(os.path.join(d, "s%d.txt" % k), "w").write(" ".join("-5.0" if b else "5.0" for b in cws[k]))
            f.write("c%d s%d\n" % (k, k))
    r = subprocess.run([LDPC, "0", "0", "0", "7", "20", "1", "c0", "s0", "H", "0", "0", "0", "0", "--list", "dec.lst"],
                       cwd=d, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "bit_err                : 0\n" in r.stdout and "frame_err              : 0\n" in r.stdout
