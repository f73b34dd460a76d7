#!/usr/bin/env python3
"""tests/golden/cli_side_by_side.json: what the UNMODIFIED reference CLI (oracle/_ref/ldpc_ref, `make -C oracle ref`)
prints and writes for the side-by-side cases of tests/test_gpu_cli.py, which compares our CLI with it wherever the
reference build is absent.

  make_golden_cli_side.py [OUT.json]                 from the reference CLI
  make_golden_cli_side.py --exe CLI [OUT.json]       from another build of the same command line: only for one that
                                                     tests/test_gpu_cli.py has found identical to the reference CLI
                                                     (dna-ldpc-codes_b200/ldpc needs a GPU)"""
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oraclelib as ol  # noqa: E402
import test_gpu_cli as t  # noqa: E402


def main(argv):
    exe = t.REF_CLI
    if argv[:1] == ["--exe"]:
        exe, argv = os.path.abspath(argv[1]), argv[2:]
    if not os.path.exists(exe):
        raise SystemExit("%s not built" % exe)
    out = argv[0] if argv else os.path.join(ol.GOLDEN, "cli_side_by_side.json")
    cases = {}
    with tempfile.TemporaryDirectory() as tmp:
        for k, (name, (case, param)) in enumerate(t.SIDE_CASES.items()):
            d = os.path.join(tmp, str(k))
            os.makedirs(d)
            cases[name] = case(exe, d, param)
    source = ("the unmodified reference CLI (oracle/_ref/ldpc_ref)" if exe == t.REF_CLI else
              "%s, whose output for these cases tests/test_gpu_cli.py had found identical to the reference CLI's" % os.path.relpath(exe, ROOT))
    with open(out, "w") as f:
        json.dump({"source": source, "cases": cases}, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote %d cases to %s" % (len(cases), out))


if __name__ == "__main__":
    main(sys.argv[1:])
