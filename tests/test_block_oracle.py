"""Pins the BlockGISolver restatement (oracle/block_oracle.cpp) the way the reference's own tests pin the solver
(tests/BlockGISolverTest.in.cpp): same termination status as the dense GoldfarbIdnaniSolver and a solution within
1e-8 (Eigen isApprox) on small tri-block-diagonal / arrow problems (:68-123, :125-170) and on the two MultiIK
fixtures (:172-230, :273-310; fixture solution to 1e-4, :188). CPU only."""
import numpy as np
import pytest

from block_cases import (dense_solution, dense_view, is_approx, multiik_sequential, multiik_simultaneous, po, random_block_problem)
from jrl_qp_b200.structured import Type


def _solve(pb, **kw):
    return po.block_solve_batch(pb.stG, pb.stC, pb.Gdata, pb.a, pb.Cdata, pb.bl, pb.bu, pb.xl, pb.xu, **kw)


@pytest.mark.parametrize("type", [Type.TriBlockDiagonal, Type.BlockArrowUp, Type.BlockArrowDown])
@pytest.mark.parametrize("layout", ["packed", "dense"])
def test_small_problem_matches_dense_solver(type, layout):
    # tests/BlockGISolverTest.in.cpp:68-170: n = {3,5,2,3}, 3 double-sided inequalities per block
    # (a small multiple of the identity keeps the random G = A A^T well conditioned: the unshifted matrices, which
    # reach cond(G) = 1e11, are checked below against the attainable eps * cond(G))
    pb = random_block_problem(type, [3, 5, 2, 3], [3, 3, 3, 3], 64, seed=11 + int(type), layout=layout, shift=0.05)
    rb = _solve(pb, nthreads=4)
    rd = dense_solution(pb)
    assert np.array_equal(rb["status"], rd["status"])
    assert (rb["status"] == 0).all()
    assert rb["iterations"].max() > 0  # the constraints do bite
    for k in range(64):
        assert is_approx(rb["x"][k], rd["x"][k], 1e-8), k
    assert np.allclose(rb["f"], rd["f"], rtol=1e-9, atol=1e-12)
    # same optimal active set and multipliers (the trajectories may differ: Householder vs Givens updates)
    assert np.array_equal(rb["active_set"], rd["active_set"])
    assert np.allclose(rb["u"], rd["u"], rtol=1e-7, atol=1e-9)


@pytest.mark.parametrize("type", [Type.TriBlockDiagonal, Type.BlockArrowUp, Type.BlockArrowDown])
def test_small_problem_unshifted(type):
    pb = random_block_problem(type, [3, 5, 2, 3], [3, 3, 3, 3], 64, seed=11 + int(type))
    rb = _solve(pb, nthreads=4)
    rd = dense_solution(pb)
    assert np.array_equal(rb["status"], rd["status"]) and (rb["status"] == 0).all()
    cond = np.linalg.cond(pb.Gdense)
    for k in range(64):
        assert is_approx(rb["x"][k], rd["x"][k], max(1e-8, 1e-15 * cond[k])), k


@pytest.mark.parametrize("type", [Type.TriBlockDiagonal, Type.BlockArrowUp, Type.BlockArrowDown])
def test_medium_problem_with_bounds(type):
    pb = random_block_problem(type, [6, 9, 4, 7, 5], [5, 6, 3, 5, 4], 32, seed=5 + int(type), bounds=True, shift=0.05)
    rb = _solve(pb, nthreads=4)
    rd = dense_solution(pb)
    assert np.array_equal(rb["status"], rd["status"]) and (rb["status"] == 0).all()
    for k in range(32):
        assert is_approx(rb["x"][k], rd["x"][k], 1e-8), k
    assert (rb["active_set"] >= 4).any()  # some bounds are active at the optimum


def test_mpc_shape_config_e():
    # BASELINE config 5: 32 blocks of 12 x 12, 12 double-sided constraints per block (reduced batch)
    pb = random_block_problem(Type.TriBlockDiagonal, [12] * 32, [12] * 32, 8, seed=3, active_frac=0.3, shift=0.05)
    rb = _solve(pb, nthreads=4)
    rd = dense_solution(pb)
    assert np.array_equal(rb["status"], rd["status"]) and (rb["status"] == 0).all()
    for k in range(8):
        assert is_approx(rb["x"][k], rd["x"][k], 1e-8), k
    assert rb["q_doubles"].max() > 0


def test_multiik_sequential():
    pb, d = multiik_sequential()
    rb = _solve(pb)
    rd = dense_solution(pb, nthreads=1)
    assert rb["status"][0] == 0 and rd["status"][0] == 0
    assert np.abs(d["sol"] - rd["x"][0]).max() <= 1e-4  # :188
    assert is_approx(rb["x"][0], rd["x"][0], 1e-8)  # :217


def test_multiik_simultaneous():
    pb, d = multiik_simultaneous()
    rb = _solve(pb)
    rd = dense_solution(pb, nthreads=1)
    assert rb["status"][0] == 0 and rd["status"][0] == 0
    assert is_approx(rb["x"][0], rd["x"][0], 1e-8)  # :305


def test_status_codes():
    pb = random_block_problem(Type.TriBlockDiagonal, [3, 4, 3], [2, 2, 2], 4, seed=1)
    # an equality in the data: the reference asserts (no active constraint may exist at the start) -> INCONSISTENT_INPUT
    bu = pb.bu.copy()
    bu[1, 2] = pb.bl[1, 2]
    r = po.block_solve_batch(pb.stG, pb.stC, pb.Gdata, pb.a, pb.Cdata, pb.bl, bu)
    assert list(r["status"]) == [0, 1, 0, 0] and (r["x"][1] == 0).all()
    # not positive definite
    G = pb.Gdata.copy()
    G[2, pb.stG.diag_offset[1]] = -1.0
    r = po.block_solve_batch(pb.stG, pb.stC, G, pb.a, pb.Cdata, pb.bl, pb.bu)
    assert list(r["status"]) == [0, 0, 2, 0]
    # infeasible: two parallel constraints with disjoint slabs
    Cd = pb.Cdense.copy()
    Cd[3, 1] = Cd[3, 0]
    bl, bu = pb.bl.copy(), pb.bu.copy()
    bl[3, 0], bu[3, 0] = 0.0, 1.0
    bl[3, 1], bu[3, 1] = 2.0, 3.0
    r = po.block_solve_batch(pb.stG, pb.stC, pb.Gdata, pb.a, pb.stC.pack(Cd), bl, bu)
    assert r["status"][3] == 3
    # iteration cap
    r = po.block_solve_batch(pb.stG, pb.stC, pb.Gdata, pb.a, pb.Cdata, pb.bl, pb.bu, max_iter=1)
    full = po.block_solve_batch(pb.stG, pb.stC, pb.Gdata, pb.a, pb.Cdata, pb.bl, pb.bu)
    assert ((r["status"] == 4) == (full["iterations"] >= 1)).all()


def test_oracle_at_n_1024_matches_kkt_reference_and_dense_solver():
    """The oracle the GPU tests trust, at the top of the structured solver's range: [16] * 64 with bounds against the
    extended-precision KKT solve on its active set (tests/test_warm_kkt_reference.py), the reference's testKKT and the
    dense solver."""
    from test_warm_kkt_reference import assert_matches_kkt_reference
    pb = random_block_problem(Type.TriBlockDiagonal, [16] * 64, [8] * 64, 2, seed=1024, bounds=True, shift=0.05)
    rb = _solve(pb, max_iter=1000, nthreads=2)
    assert (rb["status"] == 0).all() and (rb["active_set"] >= 4).any()
    flags, _, nfail = po.kkt_check_batch(rb["x"], rb["u"], pb.Gdense, pb.a, pb.Cdense, pb.bl, pb.bu, pb.xl, pb.xu, nthreads=2)
    assert nfail == 0, flags
    worst = assert_matches_kkt_reference(dense_view(pb), rb, sample=2, what="oracle n=1024")
    print(f"worst error {worst:.3g} eps cond(K)")
    rd = po.solve_batch(pb.Gdense, pb.a, pb.Cdense, pb.bl, pb.bu, pb.xl, pb.xu, max_iter=1000, nthreads=2)
    assert np.array_equal(rb["status"], rd["status"])
    for k in range(2):
        assert is_approx(rb["x"][k], rd["x"][k], 1e-8) and is_approx(rb["x"][k], pb.x_planted[k], 1e-6), k
