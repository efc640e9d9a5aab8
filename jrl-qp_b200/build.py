"""In-tree build of the native libraries (no cmake, no torch extension machinery).

  _build/libjrlqp_b200.so         CUDA kernels + C-ABI (include/jrlqp_b200.h), nvcc, sm_100a only
  _build/libjrlqp_testsupport.so  host-side synthetic problem generator (g++)

The .so files are git-ignored but travel to the GPU box with the gpurun snapshot.
"""
import concurrent.futures
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT = os.path.join(HERE, "_build")
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(ROOT, "include")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-fmad=false",  # only the explicit fma() calls are fused: canonical arithmetic order (DESIGN.md)
    "-Xcompiler", "-fPIC", "-shared",
    "-Xptxas", "-v",
    "-I", INCLUDE, "-I", CSRC,
]


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def _listdir(d, exts):
    return sorted(os.path.join(d, f) for f in os.listdir(d) if f.endswith(exts))


def _includes(path, seen=None):
    """Transitive closure of the local #include "..." files of a source (for per-object staleness)."""
    seen = set() if seen is None else seen
    if path in seen or not os.path.exists(path):
        return seen
    seen.add(path)
    with open(path) as fh:
        for line in fh:
            line = line.strip()
            if line.startswith("#include \""):
                name = line.split("\"")[1]
                for d in (os.path.dirname(path), CSRC, INCLUDE):
                    cand = os.path.join(d, name)
                    if os.path.exists(cand):
                        _includes(cand, seen)
                        break
    return seen


def build_cuda(force=False, verbose=False, defines=(), out_dir=None):
    """One object per .cu (recompiled only when it or a header it includes changed), then one link. The objects compile
    in parallel. defines: extra -D flags (e.g. ["JRLQP_TEST_FALLBACKS"]) for a variant of the library, which then
    belongs in its own out_dir (default _build)."""
    out = out_dir or OUT
    os.makedirs(out, exist_ok=True)
    target = os.path.join(out, "libjrlqp_b200.so")
    flags = [f for f in NVCC_FLAGS if f != "-shared"] + ["-D" + d for d in defines]
    srcs = _listdir(CSRC, (".cu",))
    objs = [os.path.join(out, os.path.basename(src)[:-3] + ".o") for src in srcs]
    stale = [(src, obj) for src, obj in zip(srcs, objs) if force or _newer(obj, sorted(_includes(src)))]

    def compile_one(job):
        src, obj = job
        cmd = [NVCC] + flags + ["-c", src, "-o", obj]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        res = subprocess.run(cmd, capture_output=True, text=True)
        with open(obj[:-2] + ".ptxas.log", "w") as fh:
            fh.write(res.stdout + res.stderr)
        return src, res

    with concurrent.futures.ThreadPoolExecutor(max(1, min(len(stale), os.cpu_count() or 1))) as pool:
        results = list(pool.map(compile_one, stale))
    for src, res in results:
        if res.returncode != 0:
            sys.stderr.write(res.stdout + res.stderr)
            raise RuntimeError("nvcc failed on " + src)
    if stale or force or _newer(target, objs):
        cmd = [NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-fPIC"] + objs + ["-o", target]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            sys.stderr.write(res.stdout + res.stderr)
            raise RuntimeError("nvcc link failed")
    return target


def build_testsupport(force=False, verbose=False):
    os.makedirs(OUT, exist_ok=True)
    target = os.path.join(OUT, "libjrlqp_testsupport.so")
    srcs = _listdir(os.path.join(HERE, "testsupport"), (".cpp",))
    if force or _newer(target, srcs):
        cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-pthread", "-Wall", "-Wextra"] + srcs + ["-o", target]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        subprocess.run(cmd, check=True)
    return target


def build_all(force=False, verbose=False):
    return {"cuda": build_cuda(force, verbose), "testsupport": build_testsupport(force, verbose)}


if __name__ == "__main__":
    print(build_all(force="--force" in sys.argv, verbose=True))
