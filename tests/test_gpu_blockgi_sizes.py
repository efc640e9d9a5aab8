"""GPU tests of the structured solver (experimental::BlockGISolver, csrc/blockgi.cuh) over its whole size range, n = 512 ...
1024: the passes over Q with four and with eight entries of a reflector per thread (blockgi_kernel<4> up to n = 512,
blockgi_kernel<8> above), the fast paths switched one by one at n > 512, the three structures with and without bounds,
the block sizes where the structured factor changes its thread count (32 / 33, 64 / 65, 96), constraint matrices
without constraints, shared G and C, the entry points, and the size limit n <= 1024.

Each batch holds 7 distinct problems repeated in interleaved order (instance b is problem b % 7) and is 17 instances
longer than one wave of persistent CTAs, so that CTAs solve a second, different problem in a workspace that is not fresh.
The oracle (oracle/block_oracle.cpp) runs on the 7 distinct problems only, with the same iteration cap as the GPU, and
every copy must equal its problem's oracle result bit for bit.

Three checks that share no code with that oracle:
  * every instance passes the reference's testKKT (pyoracle.kkt_check_batch: primal feasibility, stationarity and the
    signs of the multipliers) on the dense copies of G and C;
  * a sample of each case equals the extended-precision solve of the KKT system on the reported active set
    (tests/test_warm_kkt_reference.py) within 64 eps cond(K);
  * a sample of each case matches the dense solver's oracle under the reference's own criterion (same status, x within
    1e-8, tests/BlockGISolverTest.in.cpp) and the planted optimum within 1e-6."""
import functools
import os

import numpy as np
import pytest
import torch

import block_cases as bc
import pyoracle as po
import jrl_qp_b200  # noqa: F401
from jrl_qp_b200 import solver as S
from jrl_qp_b200.blockgi import BatchedBlockGISolver, BlockGISolver, StructuredC
from jrl_qp_b200.structured import Structure, Type
from test_gpu_blockgi import KEYS
from test_warm_kkt_reference import assert_matches_kkt_reference

pytestmark = pytest.mark.gpu
DISTINCT = 7
TRI, DOWN, UP = Type.TriBlockDiagonal, Type.BlockArrowDown, Type.BlockArrowUp
MIXED_512 = [7, 33, 1, 64, 20, 96, 5, 40, 65, 12, 30, 50, 89]
MIXED_513 = [16, 1, 95, 32, 33, 8, 64, 2, 65, 12, 90, 95]
WORKSPACE_LIMIT = 5 << 30  # Q workspaces of one wave of CTAs: keep a test's footprint on a shared GPU to a few GB


def _half(sizes):
    return [s // 2 for s in sizes]  # constraints per block (none for a block of one variable)


# name: structure, block sizes, constraints per block, bounds, iteration cap (above the oracle's counts), layout / shared G
CASES = {
    # four -> eight entries of a reflector per thread at 512 -> 513
    "512_uniform": (TRI, [16] * 32, [8] * 32, False, 1000),
    "513_uniform": (TRI, [16] * 32 + [1], [8] * 32 + [1], True, 600),
    "512_mixed": (UP, MIXED_512, _half(MIXED_512), True, 1000),
    "513_mixed": (DOWN, MIXED_513, _half(MIXED_513), False, 1000),
    "516": (DOWN, [12] * 43, [6] * 43, True, 600),
    "640": (UP, [20] * 32, [10] * 32, True, 1000),
    # the top of the range, every structure with and without bounds
    "768": (TRI, [24] * 32, [12] * 32, True, 800),
    "1000": (DOWN, [40] * 25, [20] * 25, False, 1000),
    "1020": (TRI, [12] * 85, [6] * 85, True, 800),
    "1023": (UP, [33] * 31, [16] * 31, True, 1000),
    "1024_8": (TRI, [8] * 128, [4] * 128, True, 750),
    "1024_16": (TRI, [16] * 64, [8] * 64, False, 500),
    "1024_64": (DOWN, [64] * 16, [32] * 16, True, 1000),
    "1024_33": (UP, [33] * 31 + [1], [16] * 31 + [0], False, 1000),
    # largest block where the structured factor runs on 32 / 64 / 128 threads
    "nmax32": (TRI, [32] * 17, [16] * 17, True, 1000),
    "nmax33": (DOWN, [33] * 16 + [16], [16] * 16 + [8], False, 1000),
    "nmax64": (UP, [64] * 9, [32] * 9, True, 1000),
    "nmax65": (TRI, [65] * 9, [32] * 9, False, 1000),
    "nmax96": (TRI, [96] * 9, [48] * 9, False, 500),  # ~ 227 KB of shared memory at 500 iterations: fits, barely
    # structure edges
    "ncstr0": (TRI, [12] * 50, [0] * 50, True, 1000),  # blocks of C without constraints: the bounds are the only ones
    "single96": (TRI, [96], [48], True, 1000),
    "dense520": (TRI, [40] * 13, [20] * 13, True, 1000, "dense"),  # dense layout, one G shared by the batch
}
FAST_SHAPES = ["1024_8", "1020", "1024_16"]  # uniform dense tiles of 8 / 12 / 16: every fast path applies


def _seed(name):
    return 20261022 + sum(map(ord, name))


@functools.lru_cache(maxsize=None)
def _distinct(name):
    """The 7 distinct problems of a case and the oracle's results on them."""
    ty, sizes, mi, bounds, max_iter, *layout = CASES[name]
    dense = layout == ["dense"]
    pb = bc.random_block_problem(ty, sizes, mi, DISTINCT, seed=_seed(name), bounds=bounds, shift=0.05,
                                 layout="dense" if dense else "packed")
    if dense:
        # one G for the batch (the dense layout holds n^2 doubles per instance): problem 0's, with every linear term moved
        # by (G_k - G_0) x*_k so that x*_k stays the optimum of problem k
        G0 = np.repeat(pb.Gdense[:1], DISTINCT, axis=0)
        pb.a = pb.a + np.einsum("bij,bj->bi", pb.Gdense - G0, pb.x_planted)
        pb.Gdata, pb.Gdense = pb.Gdata[0], G0
    ref = po.block_solve_batch(pb.stG, pb.stC, pb.Gdata, pb.a, pb.Cdata, pb.bl, pb.bu, pb.xl, pb.xu, max_iter=max_iter,
                               nthreads=os.cpu_count())
    assert (ref["status"] == 0).all(), f"{name}: the oracle did not solve every problem within {max_iter} iterations"
    return pb, ref, max_iter


def _idx(B):
    return np.arange(B) % DISTINCT


def _per(v, i):
    return None if v is None else (v[i] if v.ndim == 2 else v)


def _solver(pb, max_iter, capacity):
    sv = BatchedBlockGISolver(pb.stG, pb.stC, pb.xl is not None, capacity)
    sv.options(S.SolverOptions().maxIter(max_iter))
    return sv


def _batch(pb, max_iter):
    """More than one wave of CTAs: the grid of a solver configured like the one under test, plus 17."""
    info = _solver(pb, max_iter, 1).info()
    assert info["workspace_bytes_per_cta"] * info["grid"] <= WORKSPACE_LIMIT, info
    return info["grid"] + 17, info


def _gpu(pb, max_iter, B, sv=None):
    i = _idx(B)
    sv = sv or _solver(pb, max_iter, B)
    before = S.launch_count()
    sv.solve(*(_per(v, i) for v in (pb.Gdata, pb.a, pb.Cdata, pb.bl, pb.bu, pb.xl, pb.xu)))
    assert S.launch_count() >= before + 2, "factorisation + solver kernels were not launched"
    return sv.last


def _expand(ref, B):
    return {k: ref[k][_idx(B)] for k in KEYS}


def _assert_same_bits(g, want, what):
    for k in KEYS:
        assert np.array_equal(g[k], want[k]), f"{what}: {k} differs"


def assert_kkt_every_instance(pb, g, what):
    """testKKT (tau = 1e-6) on every instance, against the dense copies of its problem's G and C."""
    i = _idx(g["x"].shape[0])
    for p in range(DISTINCT):
        sel = i == p
        C = pb.Cdense[p] if pb.mc else None
        flags, resid, nfail = po.kkt_check_batch(g["x"][sel], g["u"][sel], pb.Gdense[p], pb.a[p], C, _per(pb.bl, p),
                                                 _per(pb.bu, p), _per(pb.xl, p), _per(pb.xu, p), nthreads=os.cpu_count())
        assert nfail == 0, f"{what}: problem {p} fails testKKT (flags {np.unique(flags)}, residuals {resid[0]})"


def assert_dense_solver_sample(pb, out, max_iter, sample, what):
    """The dense solver's oracle on a sample: same status, x within 1e-8 (isApprox), and the planted optimum within 1e-6."""
    ks = np.unique(np.linspace(0, DISTINCT - 1, sample).astype(int))
    rd = po.solve_batch(pb.Gdense[ks], pb.a[ks], pb.Cdense[ks], _per(pb.bl, ks), _per(pb.bu, ks),
                        _per(pb.xl, ks), _per(pb.xu, ks), max_iter=max_iter, nthreads=os.cpu_count())
    for j, k in enumerate(ks):
        assert rd["status"][j] == out["status"][k], f"{what} problem {k}: status differs from the dense solver's"
        assert bc.is_approx(out["x"][k], rd["x"][j], 1e-8), f"{what} problem {k}: x differs from the dense solver's"
        if pb.x_planted is not None:
            assert bc.is_approx(out["x"][k], pb.x_planted[k], 1e-6), f"{what} problem {k}: x is not the planted optimum"


# ---------------------------------------------------------------------------------------------
# every shape: host entry, bit for bit, KKT, extended-precision reference, dense solver
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(CASES))
def test_matches_the_oracle_and_independent_references(name):
    pb, ref, max_iter = _distinct(name)
    B, info = _batch(pb, max_iter)
    g = _gpu(pb, max_iter, B)
    _assert_same_bits(g, _expand(ref, B), f"{name} vs oracle")
    assert_kkt_every_instance(pb, g, name)
    worst = assert_matches_kkt_reference(bc.dense_view(pb), {k: v[:DISTINCT] for k, v in g.items() if isinstance(v, np.ndarray)},
                                         sample=2, what=name)
    assert_dense_solver_sample(pb, ref, max_iter, 2, name)
    print(f"\n{name}: n = {pb.n}, mc = {pb.mc}, B = {B}, iterations {ref['iterations'].min()} ... {ref['iterations'].max()}, "
          f"smem {info['smem_bytes']} B, {info['ctas_per_sm']} CTA/SM, worst KKT error {worst:.3g} eps kappa")


@pytest.mark.parametrize("fast", range(8))
@pytest.mark.parametrize("name", FAST_SHAPES)
def test_fast_paths_above_512_variables(name, fast, monkeypatch):
    """JRLQP_BLOCKGI_FAST bits (warp-level solves fed by TMA, register-resident sequence, blocked R solve), every
    combination, on uniform tiles of 8, 12 and 16 at n = 1020 / 1024 (the switch is read when a solver is created)."""
    monkeypatch.setenv("JRLQP_BLOCKGI_FAST", str(fast))
    pb, ref, max_iter = _distinct(name)
    B, _ = _batch(pb, max_iter)
    _assert_same_bits(_gpu(pb, max_iter, B), _expand(ref, B), f"{name} JRLQP_BLOCKGI_FAST={fast}")


# ---------------------------------------------------------------------------------------------
# structure edges
# ---------------------------------------------------------------------------------------------
def test_constraint_matrix_without_blocks():
    """A C with no blocks at all is the problem whose blocks have no constraints: same bits, bounds the only constraints."""
    pb, ref, max_iter = _distinct("ncstr0")
    B, _ = _batch(pb, max_iter)
    i = _idx(B)
    sv = BatchedBlockGISolver(pb.stG, po.CStructure.packed([], []), True, B)
    sv.options(S.SolverOptions().maxIter(max_iter))
    assert sv.info()["mc"] == 0
    sv.solve(pb.Gdata[i], pb.a[i], np.zeros((B, 0)), np.zeros((B, 0)), np.zeros((B, 0)), pb.xl[i], pb.xu[i])
    _assert_same_bits(sv.last, _expand(ref, B), "C without blocks vs the oracle with empty blocks")
    assert (ref["n_active"] > 0).all()


def test_block_sizes_beyond_shared_memory_raise_at_creation():
    """[96] * 9 fits in the shared memory of one CTA at 500 iterations (test above); [96] * 10 does not, and says so when
    the solver is created rather than failing at launch."""
    pb = bc.random_block_problem(TRI, [96] * 10, [48] * 10, 1, seed=1, shift=0.05)
    with pytest.raises(S.JrlQpError, match="shared memory"):
        BatchedBlockGISolver(pb.stG, pb.stC, False, 1)


# ---------------------------------------------------------------------------------------------
# entry points at n > 512
# ---------------------------------------------------------------------------------------------
def _device_solve(sv, B, G, a, Cd, bl, bu, xl, xu, shared=()):
    dev = torch.device("cuda:0")
    n, m = sv.n, sv.m
    out = dict(x=torch.empty((B, n), dtype=torch.float64, device=dev), u=torch.empty((B, m), dtype=torch.float64, device=dev),
               f=torch.empty(B, dtype=torch.float64, device=dev), iterations=torch.empty(B, dtype=torch.int32, device=dev),
               status=torch.empty(B, dtype=torch.int32, device=dev), active_set=torch.empty((B, m), dtype=torch.int8, device=dev),
               active_list=torch.empty((B, n), dtype=torch.int32, device=dev), n_active=torch.empty(B, dtype=torch.int32, device=dev))
    sv.solve_device(B, G, a, Cd, bl, bu, xl, xu, shared=shared, stream=torch.cuda.current_stream().cuda_stream, **out)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def test_shared_G_and_C_through_the_device_entry():
    """G, C and bounds of problem 0 shared by the batch (stride 0), 7 linear terms: against per-instance copies through the
    device entry and against the oracle. The caller's shared G is left untouched; a per-instance G is factorised in place
    into the oracle's factor."""
    pb, _, max_iter = _distinct("1024_16")
    B, _ = _batch(pb, max_iter)
    i = _idx(B)
    a7 = pb.a[0] + 0.05 * np.random.default_rng(5).standard_normal((DISTINCT, pb.n))
    one = lambda v: np.repeat(v[:1], DISTINCT, axis=0)  # noqa: E731
    ref = po.block_solve_batch(pb.stG, pb.stC, one(pb.Gdata), a7, one(pb.Cdata), one(pb.bl), one(pb.bu), max_iter=max_iter,
                               nthreads=os.cpu_count(), want_L=True)
    assert (ref["status"] == 0).all()
    want = _expand(ref, B)
    dev = torch.device("cuda:0")
    t = lambda v: torch.from_numpy(np.ascontiguousarray(v)).to(dev)  # noqa: E731
    sv = _solver(pb, max_iter, B)
    G1 = t(pb.Gdata[0])
    g_sh = _device_solve(sv, B, G1, t(a7[i]), t(pb.Cdata[0]), t(pb.bl[0]), t(pb.bu[0]), None, None, shared=("G", "C", "bl", "bu"))
    _assert_same_bits(g_sh, want, "device entry, shared G and C")
    assert np.array_equal(G1.cpu().numpy(), pb.Gdata[0]), "the caller's shared G was modified"
    Gp = t(one(pb.Gdata)[i])
    g_rep = _device_solve(sv, B, Gp, t(a7[i]), t(one(pb.Cdata)[i]), t(one(pb.bl)[i]), t(one(pb.bu)[i]), None, None)
    _assert_same_bits(g_rep, want, "device entry, per-instance copies")
    assert np.array_equal(Gp.cpu().numpy(), ref["L"][i]), "a per-instance G does not hold the oracle's factor"
    sv.solve(pb.Gdata[0], a7[i], pb.Cdata[0], pb.bl[0], pb.bu[0])
    _assert_same_bits(sv.last, want, "host entry, shared G and C")


def test_single_problem_mirror_at_n_1024():
    pb, ref, max_iter = _distinct("1024_8")
    solver = BlockGISolver(pb.n, pb.mc, True)
    solver.options(S.SolverOptions().maxIter(max_iter))
    for k in (0, 3):
        rc = solver.solve((pb.stG, pb.Gdata[k]), pb.a[k], StructuredC(pb.stC, pb.Cdata[k]), pb.bl[k], pb.bu[k], pb.xl[k], pb.xu[k])
        assert int(rc) == 0
        assert np.array_equal(solver.solution(), ref["x"][k]) and np.array_equal(solver.multipliers(), ref["u"][k])
        assert solver.objectiveValue() == ref["f"][k] and solver.iterations() == ref["iterations"][k]
        assert [int(s) for s in solver.activeSet()] == list(ref["active_set"][k])


def test_iteration_cap_above_512_variables():
    pb, full, _ = _distinct("1020")
    cap = int(full["iterations"].min()) // 2
    ref = po.block_solve_batch(pb.stG, pb.stC, pb.Gdata, pb.a, pb.Cdata, pb.bl, pb.bu, pb.xl, pb.xu, max_iter=cap,
                               nthreads=os.cpu_count())
    assert (ref["status"] == 4).all()
    B, _ = _batch(pb, cap)
    _assert_same_bits(_gpu(pb, cap, B), _expand(ref, B), f"max_iter = {cap}")


# ---------------------------------------------------------------------------------------------
# the size limit
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sizes", [[12] * 85 + [5], [12] * 86], ids=["n1025", "n1032"])
def test_more_than_1024_variables_are_refused_at_creation(sizes):
    """Past n = 1024 the passes over Q would leave the entries k >= 1024 of every reflector and vector untouched."""
    stG = Structure.packed(TRI, sizes)
    stC = po.CStructure.packed(sizes, [s // 2 for s in sizes])
    with pytest.raises(S.JrlQpError, match="1024"):
        BatchedBlockGISolver(stG, stC, True, 1)
    with pytest.raises(S.JrlQpError, match="1024"):
        BlockGISolver(sum(sizes), stC.mc, True).solve((stG, np.zeros(stG.stride)), np.zeros(sum(sizes)),
                                                      StructuredC(stC, np.zeros(stC.stride)), np.zeros(stC.mc), np.zeros(stC.mc),
                                                      np.zeros(sum(sizes)), np.zeros(sum(sizes)))
    assert BatchedBlockGISolver(Structure.packed(TRI, [8] * 128), po.CStructure.packed([8] * 128, [4] * 128), True, 1).info()["n"] == 1024
