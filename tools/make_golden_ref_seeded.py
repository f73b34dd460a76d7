#!/usr/bin/env python3
"""tests/golden/ref_seeded.json: digests of the UNMODIFIED reference's results (oracle/_ref, `make -C oracle ref`) on the
seeded inputs of tests/test_oracle_vs_ref.py, which compares the oracle with them wherever the reference build is absent.

  make_golden_ref_seeded.py [OUT.json]                  from the reference build
  make_golden_ref_seeded.py --from-oracle [OUT.json]    from oracle/liboracle.so: only for an oracle that
                                                        test_oracle_vs_ref.py has found identical to the reference
The reference object keeps one .pchk per process: the sliding-window cases run in a child process."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import oraclelib as ol  # noqa: E402
import test_oracle_vs_ref as t  # noqa: E402


def main(argv):
    from_oracle = "--from-oracle" in argv
    src = ol.Oracle if from_oracle else ol.RefLib
    if argv and argv[-1] == "--sw-child":
        print(json.dumps(t.sliding_window(src(t.PCHK_SC))))
        return
    if not from_oracle and not ol.RefLib.available():
        raise SystemExit("oracle/_ref not built (make -C oracle ref)")
    out = [a for a in argv if not a.startswith("--")]
    out = out[0] if out else os.path.join(ol.GOLDEN, "ref_seeded.json")
    dec = src(ol.PCHK_18432)
    cases = {}
    for case in (t.structure, t.random_frames, t.check_words, t.fixed_iterations, t.minsum):
        cases.update(case(dec))
    child = subprocess.run([sys.executable, __file__] + [a for a in argv if a == "--from-oracle"] + ["--sw-child"],
                           capture_output=True, text=True, check=True)
    cases.update(json.loads(child.stdout.splitlines()[-1]))
    source = ("oracle/liboracle.so, whose results on these inputs tests/test_oracle_vs_ref.py had found identical to the reference's"
              if from_oracle
              else "the unmodified reference (oracle/_ref/libldpc_ref.so)")
    with open(out, "w") as f:
        json.dump({"source": source, "cases": cases}, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote %d cases to %s" % (len(cases), out))


if __name__ == "__main__":
    main(sys.argv[1:])
