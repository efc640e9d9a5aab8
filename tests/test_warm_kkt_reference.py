"""An extended-precision reference for the warm-start solver, independent of oracle/warm_oracle.cpp.

Whatever path the solver took, its result must be the solution of the equality-constrained QP on the active set it
reports: K [x; lam] = [-a; b] with K = [[G, -N^T], [N, 0]], N the normals of the active constraints (rows of C or unit
vectors) and b their active bounds. The warm start reaches that point through its own formulas (x = J1 beta - J2 alpha2,
u = R^-1 (alpha1 + beta), f = beta . (beta / 2 + alpha1) - |alpha2|^2 / 2), so this checks them against plain linear
algebra: K is solved in float64 and refined with residuals computed in 200-bit arithmetic (mpmath), which gives the
solution to float64 accuracy while cond(K) eps << 1. The solver's multipliers are u = -lam on the active entries and
exactly 0 elsewhere.

This module holds the reference and pins the oracle to it on the CPU; tests/test_gpu_warm_widths.py applies the same
check to the GPU's warm outputs."""
import os

import mpmath
import numpy as np
import pytest

import pyoracle as po
from fallback_cases import wrong_guess
from jrl_qp_b200 import problems as P

EPS = 2.0 ** -52
KAPPA_MAX = 1e8  # beyond this the bound 64 eps kappa says nothing
TOL_FACTOR = 64  # the oracle's worst error / (eps kappa max(1, |.|)) on this module's 368 instances: 0.58 for x, 0.84 for u
INACTIVE, LOWER, UPPER, EQUALITY, LOWER_BOUND, UPPER_BOUND, FIXED = range(7)

# CTA widths 1 ... 4 of the warm kernels, their slot boundaries, and the sizes whose warm layout no longer fits in shared
# memory (n >= 116 with mc = n and bounds)
WIDTHS = [1, 2, 31, 32, 33, 63, 64, 65, 77, 78, 96, 97, 100, 112, 115, 116, 120, 127, 128]


def slot_characteristics(n):
    """The generator recipe of test_gpu_parity.py::test_sizes_across_slot_boundaries: mc = n, bounds, double-sided."""
    ne = n // 5
    ni = n - ne
    return P.ProblemCharacteristics(n, ne, ni, min(ni, max(0, n // 4)), 0, min(n // 10, n - ne - min(ni, n // 4)), 0, True, True)


def _residual(rows, z, rhs):
    """rhs - K z, each entry computed in 200-bit arithmetic from the float64 entries, then rounded once."""
    zm = [mpmath.mpf(float(v)) for v in z]
    return np.array([float(mpmath.mpf(float(r)) - mpmath.fdot(vals, [zm[j] for j in cols])) for (cols, vals), r in zip(rows, rhs)])


def kkt_reference(G, a, C, bl, bu, xl, xu, act, refinements=3):
    """x*, u*, f* and cond(K) of one instance (arrays of one instance, layout of solve_batch) on the active set `act`."""
    n = a.shape[0]
    mc = 0 if C is None else C.shape[0]
    active = np.flatnonzero(act != INACTIVE)
    N = np.zeros((active.size, n))
    b = np.zeros(active.size)
    for r, i in enumerate(active):
        s = act[i]
        if i < mc:
            N[r] = C[i]
            b[r] = bu[i] if s == UPPER else bl[i]
        else:
            N[r, i - mc] = 1.0
            b[r] = xu[i - mc] if s == UPPER_BOUND else xl[i - mc]
    q = active.size
    K = np.block([[G, -N.T], [N, np.zeros((q, q))]])
    rhs = np.concatenate([-a, b])
    rows = []
    for row in K:
        cols = np.flatnonzero(row)
        rows.append((cols, [mpmath.mpf(float(v)) for v in row[cols]]))
    with mpmath.workprec(200):
        z = np.linalg.solve(K, rhs)
        for _ in range(refinements):
            z = z + np.linalg.solve(K, _residual(rows, z, rhs))
        xs = z[:n]
        xm = [mpmath.mpf(float(v)) for v in xs]
        Gx = [mpmath.fdot([mpmath.mpf(float(v)) for v in G[i]], xm) for i in range(n)]
        fs = float(mpmath.fdot(xm, Gx) / 2 + mpmath.fdot([mpmath.mpf(float(v)) for v in a], xm))
    us = np.zeros(act.size)
    us[active] = -z[n:]
    return xs, us, fs, np.linalg.cond(K)


def assert_matches_kkt_reference(pb, out, sample=8, what=""):
    """Up to `sample` successful instances of `out`, spread over the batch, against kkt_reference."""
    ok = np.flatnonzero(out["status"] == 0)
    assert ok.size > 0, f"{what}: no successful instance to check"
    pick = ok[np.unique(np.linspace(0, ok.size - 1, min(sample, ok.size)).astype(int))]
    for b in pick:
        G = pb.G[b] if pb.G.ndim == 3 else pb.G
        C = None if pb.mc == 0 else (pb.C[b] if pb.C.ndim == 3 else pb.C)
        bl, bu, xl, xu = ((None if v is None else (v[b] if v.ndim == 2 else v)) for v in (pb.bl, pb.bu, pb.xl, pb.xu))
        act = out["active_set"][b]
        xs, us, fs, kappa = kkt_reference(G, pb.a[b], C, bl, bu, xl, xu, act)
        tag = f"{what} instance {b}"
        assert kappa <= KAPPA_MAX, f"{tag}: cond(K) = {kappa:.3g}, the bound would be meaningless"
        tol = TOL_FACTOR * EPS * kappa
        x, u, f = out["x"][b], out["u"][b], float(out["f"][b])
        assert (u[act == INACTIVE] == 0).all(), f"{tag}: nonzero multiplier on an inactive constraint"
        ex = np.abs(x - xs).max(initial=0.0)
        eu = np.abs(u - us).max(initial=0.0)
        assert ex <= tol * max(1.0, np.abs(xs).max(initial=0.0)), f"{tag}: |x - x*| = {ex:.3g}, eps kappa = {EPS * kappa:.3g}"
        assert eu <= tol * max(1.0, np.abs(us).max(initial=0.0)), f"{tag}: |u - u*| = {eu:.3g}, eps kappa = {EPS * kappa:.3g}"
        assert abs(f - fs) <= tol * max(1.0, abs(fs)), f"{tag}: |f - f*| = {abs(f - fs):.3g}, eps kappa = {EPS * kappa:.3g}"


def oracle_cold(pb):
    return po.solve_batch(pb.G, pb.a, pb.C, pb.bl, pb.bu, pb.xl, pb.xu, nthreads=os.cpu_count())


def oracle_warm(pb, as_in, warm=True):
    return po.solve_batch(pb.G, pb.a, pb.C, pb.bl, pb.bu, pb.xl, pb.xu, nthreads=os.cpu_count(), experimental=True,
                          warm_start=warm, as_in=as_in)


def full_rank_problem(n, eq, B, seed):
    """q = n at the solution: `eq` equalities, then n - eq double-sided inequalities active on their lower side, with
    orthonormal normals (random normals make cond(K) reach 1e9 at n = 33), then four inactive rows; inactive bounds."""
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((B, n, n))
    G = A @ A.transpose(0, 2, 1) / n + np.eye(n)
    N = np.linalg.qr(rng.standard_normal((B, n, n)))[0].transpose(0, 2, 1)  # rows orthonormal
    x = rng.uniform(-1, 1, (B, n))
    u = np.concatenate([rng.standard_normal((B, eq)), -rng.uniform(0.5, 1.5, (B, n - eq))], axis=1)  # LOWER: u < 0
    a = -np.einsum("bij,bj->bi", G, x) - np.einsum("bji,bj->bi", N, u)
    Cm = np.concatenate([N, rng.standard_normal((B, 4, n))], axis=1)
    cx = np.einsum("bij,bj->bi", Cm, x)
    bl = cx - np.concatenate([np.zeros((B, n)), rng.uniform(1, 2, (B, 4))], axis=1)
    bu = cx + np.concatenate([np.zeros((B, eq)), rng.uniform(1, 2, (B, n - eq + 4))], axis=1)
    return P.ProblemBatch(G, a, Cm, bl, bu, x - rng.uniform(1, 2, (B, n)), x + rng.uniform(1, 2, (B, n)), x)


def test_kkt_reference_solves_a_known_problem():
    """tests/GoldfarbIdnaniSolverTest.cpp:51-73: x = (0.5, 1.5), u = (-5, 0, 0), f = 6.5 on the active set {LOWER}."""
    G = np.array([[4.0, -2.0], [-2.0, 4.0]])
    xs, us, fs, kappa = kkt_reference(G, np.array([6.0, 0.0]), np.array([[1.0, 1.0]]), np.array([2.0]), np.array([10.0]),
                                      np.zeros(2), np.full(2, 10.0), np.array([LOWER, INACTIVE, INACTIVE], dtype=np.int8))
    assert np.array_equal(xs, [0.5, 1.5]) and np.array_equal(us, [-5.0, 0.0, 0.0]) and fs == 6.5
    assert kappa < 10


@pytest.mark.parametrize("n", WIDTHS)
def test_oracle_warm_start_matches_extended_precision_kkt(n):
    """The oracle's warm start from the exact and from a wrong guess, every width of the GPU tests."""
    pb = P.random_problems(slot_characteristics(n), 16, seed=n)
    act = oracle_cold(pb)["active_set"]
    exact = oracle_warm(pb, act)
    assert (exact["iterations"] == 0).all()
    assert_matches_kkt_reference(pb, exact, what=f"n={n} exact")
    assert_matches_kkt_reference(pb, oracle_warm(pb, wrong_guess(act, pb.mc, seed=n)), what=f"n={n} wrong")


@pytest.mark.parametrize("n", [20, 33, 70, 100])
@pytest.mark.parametrize("eq", ["all", "half"])
def test_oracle_warm_start_with_n_active_constraints_matches_kkt(n, eq):
    """q = n: N fixes x alone and the multipliers come from the first block row."""
    pb = full_rank_problem(n, n if eq == "all" else n // 2, 8, seed=300 + n)
    act = oracle_cold(pb)["active_set"]
    r = oracle_warm(pb, act)
    assert (r["status"] == 0).all() and (r["n_active"] == n).all()
    assert_matches_kkt_reference(pb, r, what=f"n={n} q=n ({eq} equalities)")
