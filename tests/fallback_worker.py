"""Child process of tests/test_gpu_fallbacks.py: loads the library named by JRLQP_B200_LIB (built with
-DJRLQP_TEST_FALLBACKS), sets or clears the flag that makes every proof of correct rounding decline, runs the named
cases of fallback_cases.py and writes, per case, <out>/<case>.npz (the outputs) and the per-site fallback counts
(<out>/counts.json: case -> 3 x FB_NSITES counts, rows = the dense / large kernels, the structured decompositions,
BlockGI). No assertion here: the parent compares."""
import argparse
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (HERE, ROOT, os.path.join(ROOT, "oracle")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import ctypes as C  # noqa: E402

import numpy as np  # noqa: E402

import jrl_qp_b200  # noqa: F401,E402
from jrl_qp_b200 import solver as S  # noqa: E402
import fallback_cases as fc  # noqa: E402

NSITES = 11


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--decline", type=int, required=True)
    ap.add_argument("--out", required=True)
    ap.add_argument("cases", nargs="+")
    args = ap.parse_args()
    assert os.environ.get("JRLQP_B200_LIB"), "JRLQP_B200_LIB must name the test build"
    lib = S.load_library()
    lib.jrlqp_test_fallback_counts.argtypes = [C.POINTER(C.c_uint64)]
    lib.jrlqp_test_fallback_decline_all.argtypes = [C.c_int32]
    counts = (C.c_uint64 * (3 * NSITES))()
    assert lib.jrlqp_test_fallback_decline_all(args.decline) == 0
    assert lib.jrlqp_test_fallback_counts(counts) == 0
    os.makedirs(args.out, exist_ok=True)
    result = {}
    for name in args.cases:
        try:
            out = fc.ALL_CASES[name].run(S)
        except Exception as e:
            raise RuntimeError(f"case {name}: {e}") from e
        assert lib.jrlqp_test_fallback_counts(counts) == 0
        result[name] = [int(c) for c in counts]
        np.savez(os.path.join(args.out, name + ".npz"), **out)
    assert lib.jrlqp_test_fallback_decline_all(0) == 0
    with open(os.path.join(args.out, "counts.json"), "w") as fh:
        json.dump(result, fh)


if __name__ == "__main__":
    main()
