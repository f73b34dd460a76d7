"""tools/alist_to_pchk.py against the reference's own converter (oracle/_ref/alist_to_pchk_ref, built from
alist-to-pchk.cpp) and a pchk -> alist -> pchk round trip of the n=18432 matrix. CPU only."""
import hashlib
import os
import subprocess
import sys

import alist_to_pchk as a2p
import gen_regular_pchk
import oraclelib as ol

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_TOOL = os.path.join(ROOT, "oracle", "_ref", "alist_to_pchk_ref")
TOOL = os.path.join(ROOT, "tools", "alist_to_pchk.py")


def test_roundtrip_n18432(tmp_path):
    alist, back = str(tmp_path / "h.alist"), str(tmp_path / "h.pchk")
    assert a2p.main(["x", "--to-alist", ol.PCHK_18432, alist]) == 0
    assert a2p.main(["x", alist, back]) == 0
    assert open(back, "rb").read() == open(ol.PCHK_18432, "rb").read()


# SHA-256 of the .pchk the reference's converter writes for the alist below, without and with -t. Recorded from
# tools/alist_to_pchk.py, whose output this test had found byte-identical to the reference converter's.
REF_PCHK_SHA256 = {"": "7b36f71c03ba3ea5881c0640f78f2df3a4a978683c23d57ff6c81173dc743c14",
                   "-t": "1de25b365426a2fd37f063b689dffe6baab84e488bbb7fa31cc1d7f42d8422c9"}


def test_matches_reference_converter(tmp_path):
    """Against the reference converter's recorded outputs, and against the converter itself where oracle/_ref is built."""
    live = os.path.exists(REF_TOOL)
    row_ptr, col_idx = gen_regular_pchk.gen_regular(120, 60, 3, 4)
    rows = [sorted(col_idx[row_ptr[i]:row_ptr[i + 1]].tolist()) for i in range(60)]
    rows[7] = rows[7][:-1]  # make it irregular
    alist = str(tmp_path / "c.alist")
    a2p.write_alist(alist, 60, 120, rows)
    for flag in ([], ["-t"]):
        mine, ref = str(tmp_path / "mine.pchk"), str(tmp_path / "ref.pchk")
        assert subprocess.run([sys.executable, TOOL] + flag + [alist, mine]).returncode == 0
        assert hashlib.sha256(open(mine, "rb").read()).hexdigest() == REF_PCHK_SHA256[" ".join(flag)]
        if live:
            assert subprocess.run([REF_TOOL] + flag + [alist, ref]).returncode == 0
            assert open(mine, "rb").read() == open(ref, "rb").read()
    # malformed files are rejected by both with the same message
    bad = str(tmp_path / "bad.alist")
    txt = open(alist).read().split("\n")
    txt[4] = txt[4].replace(txt[4].split()[0], "121", 1)  # column index out of range
    open(bad, "w").write("\n".join(txt))
    r1 = subprocess.run([sys.executable, TOOL, bad, str(tmp_path / "x.pchk")], capture_output=True)
    assert r1.returncode == 1
    assert r1.stderr == b"Alist file doesn't have the right format\n"
    if live:
        r2 = subprocess.run([REF_TOOL, bad, str(tmp_path / "y.pchk")], capture_output=True)
        assert (r2.returncode, r2.stderr) == (r1.returncode, r1.stderr)
