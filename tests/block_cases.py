"""Shared problem builders for the BlockGISolver tests (CPU oracle and GPU): seeded restatements of the
cases of the reference's tests/BlockGISolverTest.in.cpp — structured G (tests/structured_cases.py), a
block-diagonal C with double-sided inequalities built per block around a planted point
(:86-101: `randomProblem(ProblemCharacteristics(n_i, 0, 0, m_i).doubleSidedIneq(true))`), and the two
MultiIK fixtures split into blocks the way the tests do (:190-215, :286-303)."""
import os
import sys
import types

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "oracle"))
import pyoracle as po  # noqa: E402
from structured_cases import make_H  # noqa: E402

import jrl_qp_b200  # noqa: F401,E402
from jrl_qp_b200.structured import Structure, Type  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


class BlockProblem:
    """One batch: stG/stC describe the block layouts, Gdata/Cdata hold them, dense copies for the dense solver."""

    def __init__(self, stG, stC, Gdata, a, Cdata, bl, bu, xl=None, xu=None, Gdense=None, Cdense=None):
        self.stG, self.stC = stG, stC
        self.Gdata, self.a, self.Cdata, self.bl, self.bu, self.xl, self.xu = Gdata, a, Cdata, bl, bu, xl, xu
        self.Gdense, self.Cdense = Gdense, Cdense
        self.n, self.mc = stC.n, stC.mc


def random_block_problem(type, sizes, mi, batch, seed, bounds=False, active_frac=0.3, layout="packed", shift=0.0):
    """G = A A^T (tri-block-diagonal) or A^T A (arrow); per block i, m_i double-sided inequalities
    l <= C_i^T x_i <= u, optionally box bounds. Built around a planted optimum x* as the reference's generator does
    (src/test/randomProblems.cpp:150-225): a fraction `active_frac` of the constraints of every block (at most n_i,
    so that the active normals are independent) is active at x* on a random side with a multiplier in (0, 1],
    the others are strictly satisfied with slacks |U[-1,1]|, and a = -G x* + sum +/- lambda_j c_j."""
    rng = np.random.default_rng(seed)
    sizes = [int(s) for s in sizes]
    mi = [int(m) for m in mi]
    n, mc = sum(sizes), sum(mi)
    H = make_H(type, sizes, batch, seed + 7919, shift=shift)
    stG = Structure.packed(type, sizes) if layout == "packed" else Structure.dense(type, sizes)
    Gdata = stG.pack(H)
    if layout != "packed":  # dense layout: keep the full symmetric matrix in place
        Gdata = np.ascontiguousarray(H.transpose(0, 2, 1).reshape(batch, n * n))
    stC = po.CStructure.packed(sizes, mi) if layout == "packed" else po.CStructure.dense(sizes, mi)
    Cd = np.zeros((batch, mc, n))
    r0 = np.concatenate([[0], np.cumsum(sizes)])
    c0 = np.concatenate([[0], np.cumsum(mi)])
    act = np.zeros((batch, mc), dtype=bool)
    for i in range(len(sizes)):
        Cd[:, c0[i]:c0[i + 1], r0[i]:r0[i + 1]] = rng.standard_normal((batch, mi[i], sizes[i]))
        k = min(int(round(active_frac * mi[i])), sizes[i] - (1 if bounds else 0))
        for b in range(batch):
            act[b, c0[i] + rng.permutation(mi[i])[:k]] = True
    x0 = rng.uniform(-1, 1, (batch, n))
    cx = np.einsum("bjn,bn->bj", Cd, x0)
    upper = rng.uniform(0, 1, (batch, mc)) < 0.5
    lam = np.where(act, 1.0 - rng.uniform(0, 1, (batch, mc)), 0.0)
    lo = np.where(act & ~upper, 0.0, np.abs(rng.uniform(-1, 1, (batch, mc))) + 1e-3)
    hi = np.where(act & upper, 0.0, np.abs(rng.uniform(-1, 1, (batch, mc))) + 1e-3)
    bl, bu = cx - lo, cx + hi
    # stationarity: G x* + a = sum_{lower} lam c - sum_{upper} lam c
    a = -np.einsum("bij,bj->bi", H, x0) + np.einsum("bjn,bj->bn", Cd, np.where(upper, -lam, lam))
    Cdata = stC.pack(Cd)
    xl = xu = None
    if bounds:
        bact = rng.uniform(0, 1, (batch, n)) < 0.1
        bup = rng.uniform(0, 1, (batch, n)) < 0.5
        blam = np.where(bact, 1.0 - rng.uniform(0, 1, (batch, n)), 0.0)
        xl = x0 - np.where(bact & ~bup, 0.0, np.abs(rng.uniform(-1, 1, (batch, n))) + 1e-3)
        xu = x0 + np.where(bact & bup, 0.0, np.abs(rng.uniform(-1, 1, (batch, n))) + 1e-3)
        a = a + np.where(bup, -blam, blam)
    pb = BlockProblem(stG, stC, Gdata, a, Cdata, bl, bu, xl, xu, Gdense=H, Cdense=Cd)
    pb.x_planted = x0
    return pb


def dense_view(pb):
    """The dense copies of a batch with the attributes of a problems.ProblemBatch (G, a, C, bounds, mc), as
    tests/test_warm_kkt_reference.py reads them; C is None without constraints."""
    return types.SimpleNamespace(G=pb.Gdense, a=pb.a, C=pb.Cdense if pb.mc else None, bl=pb.bl, bu=pb.bu, xl=pb.xl, xu=pb.xu,
                                 mc=pb.mc)


def dense_solution(pb, nthreads=4):
    """The same problems through the dense solver restatement (GoldfarbIdnaniSolver)."""
    return po.solve_batch(pb.Gdense, pb.a, pb.Cdense, pb.bl, pb.bu, pb.xl, pb.xu, nthreads=nthreads)


def multiik_sequential(batch=1, seed=0, scale=0.0):
    """tests/BlockGISolverTest.in.cpp:172-217: 9 blocks of 43 dofs, tri-block-diagonal G, the constraints split by the
    block their first non-zero row falls in; l = -inf. G and C shared (stride 0); a perturbed per instance."""
    d = np.load(os.path.join(GOLDEN, "multiik_sequential.npz"))
    G, Cm, a, u = d["G"], d["C"], d["a"], d["u"]
    n, nd = G.shape[0], 43
    nb_cstr = []
    for i in range(Cm.shape[0]):
        j = int(np.flatnonzero(Cm[i])[0])
        if j >= len(nb_cstr) * nd:
            nb_cstr.append(1)
        else:
            nb_cstr[-1] += 1
    stG = Structure.dense(Type.TriBlockDiagonal, [nd] * 9)
    stC = po.CStructure.dense([nd] * 9, nb_cstr)
    rng = np.random.default_rng(seed)
    A = a[None, :] + scale * rng.standard_normal((batch, n)) * (np.arange(batch)[:, None] > 0)
    bl = np.full(Cm.shape[0], -np.inf)
    pb = BlockProblem(stG, stC, np.ascontiguousarray(G.T).ravel(), A, np.ascontiguousarray(Cm).ravel(), bl, u.copy(),
                      Gdense=G, Cdense=Cm)
    return pb, d


def multiik_simultaneous(batch=1, seed=0, scale=0.0):
    """tests/BlockGISolverTest.in.cpp:273-305: 5 blocks of 42 dofs, arrow-up G, 5 constraints per block, bounds."""
    d = np.load(os.path.join(GOLDEN, "multiik_simultaneous.npz"))
    G, Cm, a, u, xl, xu = d["G"], d["C"], d["a"], d["u"], d["xl"], d["xu"]
    n, nd = G.shape[0], 42
    stG = Structure.dense(Type.BlockArrowUp, [nd] * 5)
    stC = po.CStructure.dense([nd] * 5, [5] * 5)
    rng = np.random.default_rng(seed)
    A = a[None, :] + scale * rng.standard_normal((batch, n)) * (np.arange(batch)[:, None] > 0)
    bl = np.full(Cm.shape[0], -np.inf)
    pb = BlockProblem(stG, stC, np.ascontiguousarray(G.T).ravel(), A, np.ascontiguousarray(Cm).ravel(), bl, u.copy(),
                      xl.copy(), xu.copy(), Gdense=G, Cdense=Cm)
    return pb, d


def is_approx(a, b, prec):
    """Eigen isApprox: ||a - b|| <= prec * min(||a||, ||b||)."""
    return np.linalg.norm(a - b) <= prec * min(np.linalg.norm(a), np.linalg.norm(b))
