"""An extended-precision reference for the solver, independent of the oracles (oracle/gi_oracle.cpp, warm_oracle.cpp).

Whatever path the solver took, its result must be the solution of the equality-constrained QP on the active set it
reports: K [x; lam] = [-a; b] with K = [[G, -N^T], [N, 0]], N the normals of the active constraints (rows of C or unit
vectors) and b their active bounds. The warm start reaches that point through its own formulas (x = J1 beta - J2 alpha2,
u = R^-1 (alpha1 + beta), f = beta . (beta / 2 + alpha1) - |alpha2|^2 / 2), and the cold solver through a sequence of
rank-one updates, so this checks them against plain linear algebra: K is solved in float64 and refined with residuals
that are correctly rounded (each product exact as p + e by Dekker's split, each row summed by math.fsum), which gives
the solution to float64 accuracy while cond(K) eps << 1. The solver's multipliers are u = -lam on the active entries
and exactly 0 elsewhere.

This module holds the reference and pins the oracle to it on the CPU; tests/test_gpu_warm_widths.py and
tests/test_gpu_large_n.py apply the same check to the GPU's outputs."""
import functools
import math
import os
import time

import mpmath
import numpy as np
import pytest
import scipy.linalg as sla

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


_SPLIT = 134217729.0  # 2^27 + 1: Dekker's split of a double into two halves of at most 26 significant bits


def _two_products(A, z):
    """p, e with p + e = A * z exactly, elementwise (Dekker's product; numpy never contracts a * b + c into an FMA).
    Exact while no product over- or underflows, as with the O(1) data of these tests."""
    def split(v):
        c = _SPLIT * v
        hi = c - (c - v)
        return hi, v - hi
    p = A * z
    ah, al = split(A)
    zh, zl = split(z)
    return p, ((ah * zh - p) + ah * zl + al * zh) + al * zl


def _residual(K, z, rhs):
    """rhs - K z, each entry correctly rounded: math.fsum of rhs_i and the exact products of row i (its nonzeros)."""
    p, e = _two_products(K, z[None, :])
    out = np.empty(K.shape[0])
    for i, row in enumerate(K):
        nz = row != 0
        out[i] = math.fsum(np.concatenate([[rhs[i]], -p[i, nz], -e[i, nz]]).tolist())
    return out


def kkt_reference(G, a, C, bl, bu, xl, xu, act, refinements=3, residual=_residual):
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
    z = np.linalg.solve(K, rhs)
    for _ in range(refinements):
        z = z + np.linalg.solve(K, residual(K, z, rhs))
    xs = z[:n]
    # f* = x*.(G x*) / 2 + a.x*, with G x* rounded once per row and the rest summed exactly
    p, e = _two_products(np.concatenate([0.5 * xs, a]), np.concatenate([-_residual(G, xs, np.zeros(n)), xs]))
    fs = math.fsum(np.concatenate([p, e]).tolist())
    us = np.zeros(act.size)
    us[active] = -z[n:]
    # cond_2(K) from the symmetric [[G, N^T], [N, 0]] = K diag(I, -I), whose |eigenvalues| are the singular values of K: at
    # n = 1024 the eigenvalues take 0.1 s, the SVD of np.linalg.cond 0.5 s and numpy's own eigvalsh over 1 s
    ev = np.abs(sla.eigh(np.block([[G, N.T], [N, np.zeros((q, q))]]), eigvals_only=True))
    return xs, us, fs, ev.max() / ev.min()


def _sampled_instances(pb, out, sample, what):
    """(b, arguments of kkt_reference) of up to `sample` successful instances of `out`, spread over the batch."""
    ok = np.flatnonzero(out["status"] == 0)
    assert ok.size > 0, f"{what}: no successful instance to check"
    for b in ok[np.unique(np.linspace(0, ok.size - 1, min(sample, ok.size)).astype(int))]:
        G = pb.G[b] if pb.G.ndim == 3 else pb.G
        C = None if pb.mc == 0 else (pb.C[b] if pb.C.ndim == 3 else pb.C)
        bl, bu, xl, xu = ((None if v is None else (v[b] if v.ndim == 2 else v)) for v in (pb.bl, pb.bu, pb.xl, pb.xu))
        yield b, (G, pb.a[b], C, bl, bu, xl, xu, out["active_set"][b])


def assert_matches_kkt_reference(pb, out, sample=8, what=""):
    """Up to `sample` successful instances of `out`, spread over the batch, against kkt_reference. Returns the worst error
    of x, u and f in units of eps kappa max(1, |.|)."""
    worst = 0.0
    for b, args in _sampled_instances(pb, out, sample, what):
        act = args[-1]
        xs, us, fs, kappa = kkt_reference(*args)
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
        unit = EPS * kappa
        worst = max(worst, ex / (unit * max(1.0, np.abs(xs).max(initial=0.0))), eu / (unit * max(1.0, np.abs(us).max(initial=0.0))),
                    abs(f - fs) / (unit * max(1.0, abs(fs))))
    return worst


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


@functools.lru_cache(maxsize=None)
def _width_case(n):
    """16 instances of the slot recipe at n, and the oracle's warm starts from the exact and from a wrong guess."""
    pb = P.random_problems(slot_characteristics(n), 16, seed=n)
    act = oracle_cold(pb)["active_set"]
    return pb, act, oracle_warm(pb, act), oracle_warm(pb, wrong_guess(act, pb.mc, seed=n))


@functools.lru_cache(maxsize=None)
def _full_rank_case(n, eq):
    pb = full_rank_problem(n, n if eq == "all" else n // 2, 8, seed=300 + n)
    return pb, oracle_warm(pb, oracle_cold(pb)["active_set"])


@pytest.mark.parametrize("n", WIDTHS)
def test_oracle_warm_start_matches_extended_precision_kkt(n):
    """The oracle's warm start from the exact and from a wrong guess, every width of the GPU tests."""
    pb, act, exact, wrong = _width_case(n)
    assert (exact["iterations"] == 0).all()
    assert_matches_kkt_reference(pb, exact, what=f"n={n} exact")
    assert_matches_kkt_reference(pb, wrong, what=f"n={n} wrong")


@pytest.mark.parametrize("n", [20, 33, 70, 100])
@pytest.mark.parametrize("eq", ["all", "half"])
def test_oracle_warm_start_with_n_active_constraints_matches_kkt(n, eq):
    """q = n: N fixes x alone and the multipliers come from the first block row."""
    pb, r = _full_rank_case(n, eq)
    assert (r["status"] == 0).all() and (r["n_active"] == n).all()
    assert_matches_kkt_reference(pb, r, what=f"n={n} q=n ({eq} equalities)")


def _residual_mpmath(K, z, rhs):
    """rhs - K z, each entry computed in 200-bit arithmetic from the float64 entries, then rounded once."""
    with mpmath.workprec(200):
        zm = [mpmath.mpf(float(v)) for v in z]
        return np.array([float(mpmath.mpf(float(r)) - mpmath.fdot([mpmath.mpf(float(v)) for v in row[c]], [zm[j] for j in c]))
                         for row, r in zip(K, rhs) for c in (np.flatnonzero(row),)])


@pytest.mark.parametrize("case", [("slot", n) for n in WIDTHS] + [("q=n", n, eq) for n in (20, 33, 70, 100) for eq in ("all", "half")],
                         ids=lambda c: "-".join(map(str, c)))
def test_exact_residual_refines_to_the_same_bits_as_200_bit_arithmetic(case):
    """The correctly rounded residual (Dekker products, math.fsum) and a 200-bit mpmath residual lead the refinement to the
    same x* and u*, on every instance the tests above check."""
    if case[0] == "slot":
        pb, _, exact, wrong = _width_case(case[1])
        outs = [(pb, exact), (pb, wrong)]
    else:
        outs = [_full_rank_case(*case[1:])]
    for pb, out in outs:
        for b, args in _sampled_instances(pb, out, 8, str(case)):
            x1, u1, _, _ = kkt_reference(*args)
            x2, u2, _, _ = kkt_reference(*args, residual=_residual_mpmath)
            assert np.array_equal(x1, x2), f"{case} instance {b}: x* differs"
            assert np.array_equal(u1, u2), f"{case} instance {b}: u* differs"


def test_oracle_cold_matches_extended_precision_kkt_at_n_1024():
    """The cold oracle at the top of the supported range (slot recipe, up to 2000 iterations) against the reference,
    which stays fast enough there to sample many instances of a batch."""
    pb = P.random_problems(slot_characteristics(1024), 2, seed=1024)
    r = po.solve_batch(pb.G, pb.a, pb.C, pb.bl, pb.bu, pb.xl, pb.xu, nthreads=os.cpu_count(), max_iter=2000)
    assert (r["status"] == 0).all()
    t0 = time.perf_counter()
    assert_matches_kkt_reference(pb, r, what="n=1024 cold")
    print(f"kkt_reference at n = 1024: {(time.perf_counter() - t0) / pb.batch:.2f} s per instance")
