"""GPU tests of the global-workspace kernel at the top of its range, n = 511 ... 1024 (gi_large.cuh, 256 threads per QP):
two, three and four rows per thread in the Cholesky of G and in the prefactor of a batch-shared G (RP = 1024 / T), the
column ring off past n = 2 T = 512, the warm start without shared-memory slabs, the transposed batch-shared C at full
size, and the host entry's two-block upload of G at odd n.

Each batch holds 7 distinct problems repeated in interleaved order (instance b is problem b % 7) and is 17 instances
longer than one wave of persistent CTAs, so that CTAs solve a second, different problem in a workspace that is not fresh.
7 shares no factor with the grid (148 or 296 CTAs): the ticket one wave later is never the same problem. The oracle runs
on the 7 distinct problems only, and every copy must equal its problem's oracle result bit for bit. Both sides allow 2000
iterations: the slot recipe takes about 420 at n = 1024, close to the default cap of 500.

A sample of every cold and warm case is also compared with an extended-precision solve of the KKT system on the reported
active set (tests/test_warm_kkt_reference.py), which shares no code with the oracle."""
import contextlib
import functools
import os

import numpy as np
import pytest
import torch

import pyoracle as po
import jrl_qp_b200  # noqa: F401
from fallback_cases import ch_n, wrong_guess
from jrl_qp_b200 import problems as P, solver as S
from test_warm_kkt_reference import assert_matches_kkt_reference, slot_characteristics

pytestmark = pytest.mark.gpu
DISTINCT = 7
MAX_ITER = 2000
KEYS = ("x", "u", "f", "iterations", "status", "active_set", "active_list", "n_active")
# rows per thread 2 -> 3 (and the ring off) at 512 -> 513, 3 -> 4 at 768 -> 769, the top of the range
SIZES = [511, 512, 513, 640, 767, 768, 769, 1000, 1023, 1024]
SHAPES = {**{n: slot_characteristics(n) for n in SIZES},
          "n600_mc2n": ch_n(600, 60, 1140),   # mc = 2 n
          "n900_mc_quarter": ch_n(900, 25, 200)}  # mc = n / 4, a fraction of the bounds active


@contextlib.contextmanager
def _env(**values):
    """Environment switches of the large kernel, read when a handle configures it (create, or the first warm call)."""
    old = {k: os.environ.get(k) for k in values}
    os.environ.update(values)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k)
            else:
                os.environ[k] = v


def _oracle(pb, **kw):
    return po.solve_batch(pb.G, pb.a, pb.C, pb.bl, pb.bu, pb.xl, pb.xu, nthreads=os.cpu_count(), max_iter=MAX_ITER, **kw)


def _oracle_warm(pb, as_in, warm=True):
    return _oracle(pb, experimental=True, warm_start=warm, as_in=as_in)


def _grid(n, mc):
    return S.BatchedGoldfarbIdnaniSolver(n, mc, True, 1).kernel_info()["grid"]


def _idx(B):
    return np.arange(B) % DISTINCT


def _replicate(pb, B):
    """B instances, instance b a copy of problem b % 7 of pb."""
    i = _idx(B)
    return P.ProblemBatch(pb.G[i], pb.a[i], pb.C[i], pb.bl[i], pb.bu[i], pb.xl[i], pb.xu[i])


def _expand(ref, B):
    return {k: v[_idx(B)] for k, v in ref.items() if isinstance(v, np.ndarray)}


def _first(out):
    return {k: v[:DISTINCT] for k, v in out.items() if isinstance(v, np.ndarray)}


@functools.lru_cache(maxsize=None)
def _case(shape):
    """7 distinct problems of a shape, the oracle's cold results (factor of G included), and the batch size."""
    ch = SHAPES[shape]
    base = P.random_problems(ch, DISTINCT, seed=20261021 + ch.nVar + ch.nIneq)
    ref = _oracle(base, want_L=True)
    assert (ref["status"] == 0).all(), f"{shape}: the oracle did not solve every problem within {MAX_ITER} iterations"
    return base, ref, _grid(base.n, base.mc) + 17


def _solver(pb, warm=None):
    sv = S.BatchedGoldfarbIdnaniSolver(pb.n, pb.mc, True, pb.batch)
    o = S.SolverOptions().maxIter(MAX_ITER)
    if warm is not None:
        o.warmStart(warm)
    sv.options(o)
    return sv


def _gpu(pb, want_L=False):
    sv = _solver(pb)
    before = S.launch_count()
    sv.solve(pb.G, pb.a, pb.C, pb.bl, pb.bu, pb.xl, pb.xu, want_L=want_L)
    assert S.launch_count() > before, "no CUDA kernel was launched"
    return sv.last, sv.kernel_info()


def _gpu_warm(pb, as_in, warm=True):
    sv = _solver(pb, warm=warm)
    sv.solve(pb.G, pb.a, pb.C, pb.bl, pb.bu, pb.xl, pb.xu, experimental=True, as_in=as_in)
    return sv.last


def _device(sv, pb, shared=()):
    dev = torch.device("cuda:0")
    t = lambda v: torch.from_numpy(np.ascontiguousarray(v)).to(dev)  # noqa: E731
    B, n, m = pb.batch, pb.n, pb.mc + pb.nb
    out = dict(x=torch.empty((B, n), dtype=torch.float64, device=dev), u=torch.empty((B, m), dtype=torch.float64, device=dev),
               f=torch.empty(B, dtype=torch.float64, device=dev), iterations=torch.empty(B, dtype=torch.int32, device=dev),
               status=torch.empty(B, dtype=torch.int32, device=dev), active_set=torch.empty((B, m), dtype=torch.int8, device=dev),
               active_list=torch.empty((B, n), dtype=torch.int32, device=dev), n_active=torch.empty(B, dtype=torch.int32, device=dev))
    sv.solve_device(B, t(pb.G), t(pb.a), t(pb.C), t(pb.bl), t(pb.bu), t(pb.xl), t(pb.xu),
                    stream=torch.cuda.current_stream().cuda_stream, shared=shared, **out)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def _assert_same_bits(g, ref, what=""):
    for k in KEYS:
        assert np.array_equal(g[k], ref[k]), f"{what}: {k} differs"


def _assert_same_factor(L, L_ref, what):
    """Lower triangles of column-major factors equal, instance b of L against instance b % len(L_ref) of L_ref."""
    for b in range(L.shape[0]):
        assert np.array_equal(np.tril(L[b].T), np.tril(L_ref[b % L_ref.shape[0]].T)), f"{what}: instance {b}"


# ---------------------------------------------------------------------------------------------
# cold, automatic path
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", list(SHAPES), ids=str)
def test_cold_matches_the_oracle_at_two_three_and_four_rows_per_thread(shape):
    base, ref, B = _case(shape)
    pb = _replicate(base, B)
    want = _expand({k: v for k, v in ref.items() if k != "L"}, B)
    g, info = _gpu(pb, want_L=True)
    print(f"\n{shape}: n = {pb.n}, mc = {pb.mc}, B = {B}, kernel {info}")
    assert info["threads_per_qp"] == 256 and info["rows_per_thread"] == (pb.n + 255) // 256
    _assert_same_bits(g, want, "cold vs oracle")
    _assert_same_factor(g["L"], ref["L"], "factor of G vs the oracle's")
    assert_matches_kkt_reference(base, _first(g), sample=4, what=f"{shape} cold")
    # the column ring forced on where it fits (n <= 512) and off, warm slabs on and off: the same bits (past n = 512
    # neither can be used, so the switches must change nothing)
    for ring, slab in (("2", "1"), ("0", "0")):
        with _env(JRLQP_LARGE_RING=ring, JRLQP_LARGE_SLAB=slab):
            _assert_same_bits(_gpu(pb)[0], g, f"JRLQP_LARGE_RING={ring} JRLQP_LARGE_SLAB={slab}")


# ---------------------------------------------------------------------------------------------
# warm start: J = J Q thread = row over the workspace (no shared-memory slabs past n ~ 460)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [513, 769, 1024])
def test_warm_start_exact_wrong_and_off(n):
    base, ref, B = _case(n)
    pb = _replicate(base, B)
    i = _idx(B)
    act = ref["active_set"]
    wrong = wrong_guess(act, base.mc, seed=n)
    exact = _oracle_warm(base, act)
    g = _gpu_warm(pb, act[i])
    _assert_same_bits(g, _expand(exact, B), "exact guess")
    assert (g["iterations"] == 0).all() and np.array_equal(g["active_set"], act[i])
    assert_matches_kkt_reference(base, _first(g), sample=4, what=f"n={n} exact guess")
    ref_wrong = _expand(_oracle_warm(base, wrong), B)
    assert (ref_wrong["status"] == 0).all(), f"the oracle did not repair every wrong guess within {MAX_ITER} iterations"
    g = _gpu_warm(pb, wrong[i])
    _assert_same_bits(g, ref_wrong, "wrong guess")
    assert_matches_kkt_reference(base, _first(g), sample=4, what=f"n={n} wrong guess")
    _assert_same_bits(_gpu_warm(pb, wrong[i], warm=False), _expand(_oracle_warm(base, wrong, warm=False), B), "warmStart off")
    if n == 513:
        for slab in ("1", "0"):
            with _env(JRLQP_LARGE_SLAB=slab):
                _assert_same_bits(_gpu_warm(pb, wrong[i]), ref_wrong, f"JRLQP_LARGE_SLAB={slab}")


# ---------------------------------------------------------------------------------------------
# G and C shared by the batch: prefactor kernel, initial_point_blocked over 25 / 32 blocks, transposed shared C
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [769, 1024])
def test_batch_shared_G_and_C(n):
    base, _, B = _case(n)
    i = _idx(B)
    a7 = base.a[0] + 0.05 * np.random.default_rng(n).standard_normal((DISTINCT, n))
    sh = P.ProblemBatch(base.G[0], a7[i], base.C[0], base.bl[0], base.bu[0], base.xl[0], base.xu[0])
    one = lambda v: np.repeat(v[:1], DISTINCT, axis=0)  # noqa: E731
    ref = _oracle(P.ProblemBatch(one(base.G), a7, one(base.C), one(base.bl), one(base.bu), one(base.xl), one(base.xu)), want_L=True)
    assert (ref["status"] == 0).all()
    want = _expand({k: v for k, v in ref.items() if k != "L"}, B)
    before = S.launch_count()
    g_sh, _ = _gpu(sh, want_L=True)
    assert S.launch_count() >= before + 2, "prefactor kernel + solver kernel"
    _assert_same_bits(g_sh, want, "host entry, shared G and C")
    _assert_same_factor(g_sh["L"], ref["L"], "factor of the shared G vs the oracle's")
    _assert_same_bits(_device(_solver(sh), sh, shared=("G", "C", "bl", "bu", "xl", "xu")), want, "device entry, shared G and C")
    rep = _replicate(P.ProblemBatch(one(base.G), a7, one(base.C), one(base.bl), one(base.bu), one(base.xl), one(base.xu)), B)
    g_rep, _ = _gpu(rep, want_L=True)
    _assert_same_bits(g_rep, want, "G and C replicated per instance")
    _assert_same_factor(g_rep["L"], g_sh["L"], "per-instance factors vs the shared factor")
    g_bad, _ = _gpu(P.ProblemBatch(-sh.G, sh.a, sh.C, sh.bl, sh.bu, sh.xl, sh.xu))
    assert (g_bad["status"] == S.TerminationStatus.NON_POS_HESSIAN).all()


# ---------------------------------------------------------------------------------------------
# host entry at odd n: G crosses the link as its left n // 2 columns and the bottom-right block
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [769, 1023])
def test_host_entry_moves_only_the_lower_triangle_of_G_at_odd_n(n):
    base, ref, B = _case(n)
    pb = _replicate(base, B)
    want = _expand({k: v for k, v in ref.items() if k != "L"}, B)
    sv = _solver(pb)
    assert sv.host_g_bytes(False) == 8 * (n * (n // 2) + (n - n // 2) ** 2)
    dev = _device(sv, pb)
    _assert_same_bits(dev, want, "device entry")
    iu = np.triu_indices(n, 1)
    Gp = pb.G.copy()
    Gp[:, iu[1], iu[0]] = np.nan  # G [B][col][row]: entry (row < col) is the strict upper triangle
    sv.solve(Gp, pb.a, pb.C, pb.bl, pb.bu, pb.xl, pb.xu)
    _assert_same_bits(sv.last, dev, "host entry, upper triangle of G poisoned, vs device entry")


# ---------------------------------------------------------------------------------------------
# warm-started sequence with a shared G
# ---------------------------------------------------------------------------------------------
def test_warm_sequence_with_a_shared_G_at_n_700():
    """G, C and bounds of one problem shared by the batch, 7 distinct linear terms moving over three steps."""
    n, T = 700, 3
    base = P.random_problems(slot_characteristics(n), 1, seed=700)
    B = _grid(n, base.mc) + 17
    i = _idx(B)
    rng = np.random.default_rng(7)
    a0 = base.a[0] + 0.05 * rng.standard_normal((DISTINCT, n))
    a_seq = np.stack([a0 + 0.02 * t * rng.standard_normal((DISTINCT, n)) for t in range(T)])
    sv = S.BatchedGoldfarbIdnaniSolver(n, base.mc, True, B)
    sv.options(S.SolverOptions().maxIter(MAX_ITER).warmStart(True))
    sv.solve_sequence(base.G[0], np.ascontiguousarray(a_seq[:, i]), base.C[0], base.bl[0], base.bu[0], base.xl[0], base.xu[0],
                      warm=True, keep_steps=True)
    g = sv.last
    # the oracle's chain: step 0 cold through the warm-capable solver, every later step warm from the previous active set
    one = lambda v: np.repeat(v[:1], DISTINCT, axis=0)  # noqa: E731
    rep = lambda a: P.ProblemBatch(one(base.G), a, one(base.C), one(base.bl), one(base.bu), one(base.xl), one(base.xu))  # noqa: E731
    act = None
    for t in range(T):
        r = _oracle_warm(rep(a_seq[t]), act)
        for k in ("x", "u", "f", "iterations", "status"):
            assert np.array_equal(g[k][t], r[k][i]), f"step {t}: {k} differs from the oracle's chain"
        act = r["active_set"]
    assert np.array_equal(g["active_set"], act[i]) and (g["status_worst"] == 0).all()
    cold = _oracle(rep(a_seq[-1]))
    assert np.allclose(g["x"][-1], cold["x"][i], rtol=1e-9, atol=1e-11)


# ---------------------------------------------------------------------------------------------
# bounds of the API
# ---------------------------------------------------------------------------------------------
def test_size_limits_of_the_api():
    with pytest.raises(S.JrlQpError):
        S.BatchedGoldfarbIdnaniSolver(1025, 10, True, 1)
    sv = S.BatchedGoldfarbIdnaniSolver(1024, 10, True, 1)
    assert sv.kernel_info()["rows_per_thread"] == 4
    with pytest.raises(S.JrlQpError):
        sv.set_kernel_path(1)
    with pytest.raises(S.JrlQpError):
        S.BatchedGoldfarbIdnaniSolver(129, 10, True, 1).set_kernel_path(1)
