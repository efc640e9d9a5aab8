#!/usr/bin/env python
"""Development aid: build a variant of libjrlqp_b200.so, with extra -D flags on every source if any, in its own directory:
python scripts/build_variant.py <name> [-DJRLQP_TEST_FALLBACKS ...]  ->  _build/variants/<name>/libjrlqp_b200.so, copied to
_build/libjrlqp_b200_<name>.so (the name scripts/ab_variants.py looks for). Select it at run time with JRLQP_B200_LIB=<path>.
Tuning values are constants in the sources: to time a different value, build the variant from a branch that changes it."""
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import jrl_qp_b200  # noqa: F401,E402
from jrl_qp_b200 import build as B  # noqa: E402


def main():
    name, flags = sys.argv[1], sys.argv[2:]
    bad = [f for f in flags if not f.startswith("-D")]
    if bad:
        sys.exit(f"only -D flags are supported: {bad}")
    lib = B.build_cuda(defines=[f[2:] for f in flags], out_dir=os.path.join(B.OUT, "variants", name))
    log = open(os.path.join(os.path.dirname(lib), "capi.ptxas.log")).read()
    lines = log.splitlines()
    for i, ln in enumerate(lines):
        if "gi_dense_cta_kernelILi" in ln and "Compiling" in ln and "ELb0ELb0" in ln:
            print(ln.split("'")[1][:60], "|", lines[i + 2].strip(), "|", lines[i + 3].strip())
    out = os.path.join(B.OUT, f"libjrlqp_b200_{name}.so")
    shutil.copyfile(lib, out)
    print(out)


if __name__ == "__main__":
    main()
