"""The stock-arithmetic fallbacks behind every proven quotient and square root (DESIGN.md §2, fp64_exact.cuh).

On the serial recurrences a division or square root comes from a hardware seed and one correction, and an exact remainder
test proves it correctly rounded; when a proof is declined the kernel redoes the work with the stock `/` and `sqrt`. Random
O(1) inputs almost never decline a proof, so this file reaches the recovery code on purpose, three ways:

(a) decline-all: the library built with -DJRLQP_TEST_FALLBACKS (test_fallbacks.cuh), with the flag that makes every proof
    decline, runs every kernel family in a child process (the library is loaded once per process); every output must
    equal the shipped library's and the oracle's bit for bit, and every fallback site must have been taken;
(b) count-only: the same build with the flag off, on the edge inputs of (c): each family must reach the sites listed in
    EDGE_SITES, which shows that the shipped-build tests of (c) do exercise the fallbacks;
(c) edge inputs on the shipped library: problems scaled by 2^-840 (every divisor of the factor of G and of R leaves the
    +-400-binade range of the proofs; structured factors also at 2^-980, below the range guard of the small-tile sqrt),
    and dyadic problems (G = I or 4 I, +-1 or equal-entry normals, integer bounds), whose quotients are often powers of
    two. Oracle parity, plus a relation that needs no oracle: scaling G and a by s leaves status, iterations, active set
    and x unchanged and scales u and f by s, bit for bit; a structured factor scales by sqrt(s) and its solves by
    1 / sqrt(s). The oracle side of the relation is checked without a GPU.
"""
import json
import os
import subprocess
import sys
import time

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

import fallback_cases as fc  # noqa: E402
import jrl_qp_b200  # noqa: F401,E402
from jrl_qp_b200 import build as B, problems as P  # noqa: E402

SITES = ["x=-G^-1a", "givens_link_slow", "givens_chain careful", "back_substitution_exact", "givens_recurrence careful",
         "givens_recurrence W=4 bad", "initial_point_blocked", "warm B=L^-1N", "block_solve_exact", "r_solve_blocked",
         "small-tile LLT vote"]
UNITS = ["dense/large", "structured", "blockgi"]
NS = len(SITES)
# (unit, site) every fallback, as the decline-all run must reach them
ALL_SITES = [(0, s) for s in range(8)] + [(1, 8), (1, 10), (2, 8), (2, 9)]
# sites the edge inputs of (c) reach with every proof attempted (count-only run of the test build)
EDGE_SITES = {
    "binade_A": [(0, 0), (0, 3)],
    "binade_B": [(0, 0), (0, 3)],
    "binade_D": [(0, 0), (0, 3)],
    "binade_n70": [(0, 0), (0, 3)],
    "binade_n300": [(0, 1)],
    "binade_n300_shared": [(0, 1), (0, 6)],
    "binade_warm_A": [(0, 3)],
    "binade_warm_B": [(0, 3)],
    "binade_warm_D": [(0, 1), (0, 7)],
    "binade_warm_n300_shared": [(0, 1), (0, 7)],
    "binade_structured_k2": [(1, 8), (1, 10)],  # (the general kernel 1 proves no quotient: nothing to fall back from)
    "binade_structured_k3": [(1, 8), (1, 10)],
    "binade_blockgi_ref": [(2, 9)],
    "binade_blockgi_wide": [(1, 10), (2, 8), (2, 9)],
    "dyadic_I_cold": [(0, 0), (0, 3), (0, 4)],
    "dyadic_4I_cold": [(0, 0), (0, 3), (0, 4)],
    "dyadic_I_warm": [(0, 3), (0, 4)],
    "dyadic_4I_warm": [(0, 4)],
    "dyadic_I_large": [(0, 1), (0, 2)],
    "dyadic_sequence": [(0, 3), (0, 4)],
}
# sites of the global-workspace kernel at four rows per thread, with every proof declined
# (initial_point_blocked runs only from the factor of a batch-shared G; a per-instance G takes the serial initial_point)
LARGE_N_SITES = {"large_n800_cold": [(0, 1)], "large_n800_warm": [(0, 7)], "large_n800_shared": [(0, 6)]}
# sites of the structured solver past n = 512 (blockgi_kernel<8>), with every proof declined: the small-tile factor, the
# warp-level block solves and the blocked R solve
BLOCKGI_N528_SITES = [(1, 10), (2, 8), (2, 9)]
# (warm starts of the scaled problems from the unscaled cold active set: oracle parity only — the oracle itself does not
# keep the relation there)
RELATION_QP = ["binade_A", "binade_B", "binade_D", "binade_n70", "binade_n300"]
RELATION_STRUCT = {"binade_structured_k1": fc.S840, "binade_structured_k2": fc.S980, "binade_structured_k3": fc.S980}
RELATION_BLOCK = ["binade_blockgi_ref", "binade_blockgi_wide"]


def _names(counts):
    return {f"{UNITS[u]}:{SITES[s]}": c for u in range(3) for s in range(NS) if (c := counts[u * NS + s])}


# ------------------------------------------------------------------------------------------------------------------------
# the test build, run in child processes (one per mode, all cases)
# ------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def variant(tmp_path_factory):
    t0 = time.perf_counter()
    # next to the shipped objects (incremental across runs), or in a temporary directory when the tree is read-only
    out_dir = os.path.join(B.OUT, "fallbacks") if os.access(B.OUT, os.W_OK) else str(tmp_path_factory.mktemp("fallbacks"))
    lib = B.build_cuda(defines=["JRLQP_TEST_FALLBACKS"], out_dir=out_dir)
    t_build = time.perf_counter() - t0
    runs = {}
    for mode, decline in (("decline", 1), ("count", 0)):
        out = str(tmp_path_factory.mktemp(mode))
        env = dict(os.environ, JRLQP_B200_LIB=lib)
        res = subprocess.run([sys.executable, os.path.join(HERE, "fallback_worker.py"), "--decline", str(decline), "--out", out]
                             + fc.RUN_CASES, env=env, capture_output=True, text=True)
        assert res.returncode == 0, res.stdout[-4000:] + res.stderr[-4000:]
        with open(os.path.join(out, "counts.json")) as fh:
            counts = json.load(fh)
        runs[mode] = (out, counts)
        print(f"\n[{mode}] per-site fallback counts (variant build {t_build:.0f} s):")
        for name, c in counts.items():
            print(f"  {name:28s} {_names(c)}")
    return runs


def _load(variant, mode, name):
    out, _ = variant[mode]
    with np.load(os.path.join(out, name + ".npz")) as d:
        return {k: d[k] for k in d.files}


_shipped_cache = {}


def _shipped(name):
    from jrl_qp_b200 import solver as S
    if name not in _shipped_cache:
        _shipped_cache[name] = fc.ALL_CASES[name].run(S)
    return _shipped_cache[name]


def _assert_equal(got, ref, what):
    for k in ref:
        assert np.array_equal(np.asarray(got[k]), np.asarray(ref[k])), f"{what}: {k} differs"


@pytest.mark.gpu
@pytest.mark.parametrize("name", fc.RUN_CASES)
def test_decline_all_matches_shipped_and_oracle(variant, name):
    """Every proof declined: each fallback recomputes what the fast path would have, so the outputs are the oracle's."""
    got = _load(variant, "decline", name)
    ship = _shipped(name)
    ref = fc.ALL_CASES[name].oracle()
    _assert_equal(ship, ref, "shipped library vs oracle")
    _assert_equal(got, ref, "every proof declined vs oracle")
    _assert_equal(got, ship, "every proof declined vs shipped library")


@pytest.mark.gpu
def test_decline_all_reaches_every_site(variant):
    _, counts = variant["decline"]
    total = np.sum([np.asarray(c, dtype=np.int64) for c in counts.values()], axis=0)
    missed = [f"{UNITS[u]}:{SITES[s]}" for u, s in ALL_SITES if total[u * NS + s] == 0]
    assert not missed, f"fallback sites never taken with every proof declined: {missed}"


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(LARGE_N_SITES))
def test_decline_all_reaches_the_large_kernel_sites_at_n_800(variant, name):
    _, counts = variant["decline"]
    c = counts[name]
    missed = [f"{UNITS[u]}:{SITES[s]}" for u, s in LARGE_N_SITES[name] if c[u * NS + s] == 0]
    assert not missed, f"{name} does not reach {missed} with every proof declined (counts {_names(c)})"


@pytest.mark.gpu
def test_decline_all_reaches_the_blockgi_sites_above_512_variables(variant):
    _, counts = variant["decline"]
    c = counts["blockgi_n528"]
    missed = [f"{UNITS[u]}:{SITES[s]}" for u, s in BLOCKGI_N528_SITES if c[u * NS + s] == 0]
    assert not missed, f"blockgi_n528 does not reach {missed} with every proof declined (counts {_names(c)})"


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(EDGE_SITES))
def test_edge_inputs_reach_their_sites(variant, name):
    _, counts = variant["count"]
    c = counts[name]
    missed = [f"{UNITS[u]}:{SITES[s]}" for u, s in EDGE_SITES[name] if c[u * NS + s] == 0]
    assert not missed, f"{name} no longer reaches {missed} (counts {_names(c)})"


# ------------------------------------------------------------------------------------------------------------------------
# (c) edge inputs on the shipped library: relations that need no oracle, and KKT
# ------------------------------------------------------------------------------------------------------------------------
def _unscaled(name):
    return fc.ALL_CASES[name.replace("binade_", "unscaled_")]


def _assert_qp_scaling(sc, un, s, what):
    for k in ("status", "iterations", "n_active", "active_set", "active_list", "x"):
        assert np.array_equal(sc[k], un[k]), f"{what}: {k} changes under the scaling"
    assert np.array_equal(sc["u"], un["u"] * s), f"{what}: u is not s u"
    assert np.array_equal(sc["f"], un["f"] * s), f"{what}: f is not s f"


def _not_subnormal(*arrays):
    for a in arrays:
        a = np.abs(np.asarray(a, dtype=np.float64))
        assert not ((a > 0) & (a < np.finfo(np.float64).tiny)).any(), "subnormal value"


@pytest.mark.gpu
@pytest.mark.parametrize("name", RELATION_QP + RELATION_BLOCK)
def test_binade_scaling_relation_gpu(name):
    sc = _shipped(name)
    un = _shipped(name.replace("binade_", "unscaled_"))
    _assert_qp_scaling(sc, un, fc.S840, name)


def _assert_factor_scaling(sc, un, s):
    """The factor's entries scale by sqrt(s); the entries the factorisation leaves untouched (upper triangles of the
    diagonal blocks in the packed storage) keep the input's scaling s."""
    kept = un["L"] == un["input"]
    assert np.array_equal(sc["input"], un["input"] * s)
    assert np.array_equal(sc["L"][~kept], un["L"][~kept] * np.sqrt(s)), "L is not sqrt(s) L"
    assert np.array_equal(sc["L"][kept], sc["input"][kept])


def _assert_solve_scaling(sc, un, k, r):
    """The solves over the whole vector scale by 1 / sqrt(s). (A hint window reads the entries outside it as they are,
    unscaled: no relation there; those solves are compared with the oracle only.)"""
    n = un["rhs"].shape[-1]
    if k not in (f"fwd0_{n}", f"bwd0_{n}"):
        return
    kept = un[k] == un["rhs"]
    assert np.array_equal(sc[k][~kept], un[k][~kept] / r), f"{k}: the solve does not scale by 1 / sqrt(s)"
    assert np.array_equal(sc[k][kept], sc["rhs"][kept]), k


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(RELATION_STRUCT))
def test_binade_structured_scaling_gpu(name):
    s = RELATION_STRUCT[name]
    sc = _shipped(name)
    un = _shipped(name.replace("binade_", "unscaled_"))
    assert sc["ok"].all() and un["ok"].all()
    _assert_factor_scaling(sc, un, s)
    r = np.sqrt(s)
    for k in sc:
        if k.startswith(("fwd", "bwd")):
            _assert_solve_scaling(sc, un, k, r)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["dyadic_I_cold", "dyadic_4I_cold", "dyadic_I_warm", "dyadic_4I_warm", "dyadic_I_large"])
def test_dyadic_kkt(name):
    g = _shipped(name)
    kind = {"dyadic_I_cold": "pm1_I", "dyadic_4I_cold": "equal_4I", "dyadic_I_warm": "equal_I", "dyadic_4I_warm": "pm1_4I",
            "dyadic_I_large": "pm1_I"}[name]
    pb = fc.dyadic_problem(kind, g["x"].shape[0], seed=len(kind))
    assert (g["status"] == 0).all()
    assert P.test_kkt(g["x"], g["u"], pb).all()


# ------------------------------------------------------------------------------------------------------------------------
# oracle side of the relations (no GPU)
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", RELATION_QP + RELATION_BLOCK)
def test_binade_scaling_relation_oracle(name):
    sc = fc.ALL_CASES[name].oracle()
    un = _unscaled(name).oracle()
    _not_subnormal(sc["x"], sc["u"], sc["f"])
    _assert_qp_scaling(sc, un, fc.S840, name)


@pytest.mark.parametrize("name", list(RELATION_STRUCT))
def test_binade_structured_scaling_oracle(name):
    s = RELATION_STRUCT[name]
    sc = fc.ALL_CASES[name].oracle()
    un = _unscaled(name).oracle()
    assert sc["ok"].all() and un["ok"].all()
    _not_subnormal(*sc.values())
    r = np.sqrt(s)
    assert r * r == s
    _assert_factor_scaling(sc, un, s)
    for k in sc:
        if k.startswith(("fwd", "bwd")):
            _assert_solve_scaling(sc, un, k, r)


@pytest.mark.parametrize("name", ["binade_A", "binade_n70", "binade_n300"])
def test_binade_factor_leaves_the_proof_range(name):
    """The scaled factor's diagonal lies outside +-400 binades, so that every quotient by it declines its proof."""
    s = fc.S840
    pb = fc.scaled(fc.dense_problem(name[len("binade_"):], 4), s)
    _not_subnormal(pb.G, pb.a)
    L = np.linalg.cholesky(pb.G)
    e = np.log2(np.abs(np.diagonal(L, axis1=1, axis2=2)))
    assert e.max() < -400 and e.min() > -1000
