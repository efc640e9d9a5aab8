"""GPU tests of the warm-start solver (experimental::GoldfarbIdnaniSolver) at every CTA width of its shared-memory kernel
(gi_dense_cta_kernel<W, false, true>, W = 1 ... 4), at the slot boundaries of each width and past the size where its
layout stops fitting in shared memory (n >= 116 with mc = n and bounds), where automatic mode runs warm calls on the
global-workspace kernel.

Every result is compared with the oracle bit for bit (oracle/warm_oracle.cpp), and a sample of each is compared with an
extended-precision solve of the KKT system on the reported active set (tests/test_warm_kkt_reference.py), which does
not share the warm start's formulas. The batches are larger than one wave of persistent CTAs, so the ticket loop runs."""
import functools
import os

import numpy as np
import pytest
import torch

import jrl_qp_b200  # noqa: F401
from fallback_cases import ch_n, wrong_guess
from jrl_qp_b200 import problems as P, solver as S
from test_gpu_parity import assert_parity
from test_gpu_sequence import _oracle_sequence, _seq_with_env, _trajectory
from test_warm_kkt_reference import (WIDTHS, assert_matches_kkt_reference, full_rank_problem, oracle_cold, oracle_warm,
                                     slot_characteristics)

pytestmark = pytest.mark.gpu
LOWER, LOWER_BOUND = 1, 4
FITS = [n for n in WIDTHS if n <= 115]  # the shared-memory warm kernel fits (mc = n, bounds)
DOUBLE_SIDED = {"ds70": ch_n(70, 5, 150), "ds100": ch_n(100, 10, 110)}  # mc > n


def _warps(n):
    return min((n + 31) // 32, 4)


def _batch(n):
    """More instances than the warm kernel keeps resident on 148 SMs at this width."""
    return (2000, 1000, 400, 300)[_warps(n) - 1]


@functools.lru_cache(maxsize=None)
def _case(shape):
    """Problems of a shape (an n of WIDTHS or a name of DOUBLE_SIDED), the exact and a wrong guess, and the oracle."""
    if shape in DOUBLE_SIDED:
        ch = DOUBLE_SIDED[shape]
        pb = P.random_problems(ch, _batch(ch.nVar), seed=ch.nVar + 1)
    else:
        pb = P.random_problems(slot_characteristics(shape), _batch(shape), seed=shape)
    act = oracle_cold(pb)["active_set"]
    wrong = wrong_guess(act, pb.mc, seed=pb.n)
    ref = {"exact": oracle_warm(pb, act), "wrong": oracle_warm(pb, wrong), "off": oracle_warm(pb, wrong, warm=False)}
    return pb, act, wrong, ref


def _gpu_warm(pb, as_in, warm=True, path=0, scan_transposed=None):
    sv = S.BatchedGoldfarbIdnaniSolver(pb.n, pb.mc, pb.xl is not None, pb.batch)
    sv.set_kernel_path(path)
    if scan_transposed is not None:
        sv.set_scan_transposed(scan_transposed)
    sv.options(S.SolverOptions().warmStart(warm))
    before = S.launch_count()
    sv.solve(pb.G, pb.a, pb.C, pb.bl, pb.bu, pb.xl, pb.xu, experimental=True, as_in=as_in)
    assert S.launch_count() > before, "no CUDA kernel was launched"
    return sv.last


def _assert_same_bits(g1, g2):
    for k in ("x", "u", "f", "iterations", "status", "active_set", "active_list", "n_active"):
        assert np.array_equal(g1[k], g2[k]), f"{k} differs"


@pytest.mark.parametrize("shape", WIDTHS + list(DOUBLE_SIDED))
def test_warm_start_exact_wrong_and_off(shape):
    pb, act, wrong, ref = _case(shape)
    g = _gpu_warm(pb, act)
    assert_parity(g, ref["exact"])
    assert (g["status"] == 0).all() and (g["iterations"] == 0).all()
    assert np.array_equal(g["active_set"], act)
    assert_matches_kkt_reference(pb, g, what=f"{shape} exact")
    g = _gpu_warm(pb, wrong)
    assert_parity(g, ref["wrong"])
    assert_matches_kkt_reference(pb, g, what=f"{shape} wrong")
    assert_parity(_gpu_warm(pb, wrong, warm=False), ref["off"])  # the guess is ignored


@pytest.mark.parametrize("shape", FITS + list(DOUBLE_SIDED))
def test_kernel_paths_and_constraint_scans_agree(shape):
    """Where the shared-memory warm kernel fits, it and the global-workspace kernel compute the same bits; at W >= 3 the
    scan of the CTA's transposed copy of C and the scan of C in place do too."""
    pb, act, wrong, ref = _case(shape)
    shared = _gpu_warm(pb, wrong, path=1)
    _assert_same_bits(shared, _gpu_warm(pb, wrong, path=2))
    assert_parity(shared, ref["wrong"])
    if _warps(pb.n) >= 3:
        for on in (True, False):
            assert_parity(_gpu_warm(pb, act, path=1, scan_transposed=on), ref["exact"])
            assert_parity(_gpu_warm(pb, wrong, path=1, scan_transposed=on), ref["wrong"])


@pytest.mark.parametrize("n", [20, 33, 70, 100])
@pytest.mark.parametrize("eq", ["all", "half"])
def test_guess_of_n_active_constraints(n, eq):
    """q = n: the last Householder column has nothing below its diagonal (len == 0) and J2 is empty."""
    pb = full_rank_problem(n, n if eq == "all" else n // 2, _batch(n), seed=300 + n)
    act = oracle_cold(pb)["active_set"]
    g = _gpu_warm(pb, act)
    assert_parity(g, oracle_warm(pb, act))
    assert (g["status"] == 0).all() and (g["iterations"] == 0).all() and (g["n_active"] == n).all()
    assert_matches_kkt_reference(pb, g, what=f"n={n} q=n ({eq} equalities)")


@pytest.mark.parametrize("n", [20, 33, 70, 100])
def test_guess_of_more_than_n_constraints(n):
    """Every constraint and bound guessed LOWER: 2 n guesses, trimmed from the back to n, then dropped as needed."""
    pb = P.random_problems(slot_characteristics(n), _batch(n), seed=500 + n)
    guess = np.where(np.arange(pb.mc + pb.n) < pb.mc, LOWER, LOWER_BOUND).astype(np.int8)
    g = _gpu_warm(pb, guess)
    ref = oracle_warm(pb, np.broadcast_to(guess, (pb.batch, guess.size)).copy())
    assert_parity(g, ref)
    assert_matches_kkt_reference(pb, g, what=f"n={n} all guessed")


@pytest.mark.parametrize("n", [20, 33, 70, 100])
def test_degenerate_householder_reflectors(n):
    """G = 4 I and bounds guessed on the leading variables: L^-1 e_k has no entry below row k, so every reflector of the
    QR of B = L^-1 N is the identity (tau = 0)."""
    pb = P.random_problems(slot_characteristics(n), _batch(n), seed=600 + n)
    pb.G[:] = 4.0 * np.eye(n)
    guess = np.zeros((pb.batch, pb.mc + n), dtype=np.int8)
    guess[:, pb.mc:pb.mc + max(1, n // 4)] = LOWER_BOUND
    g = _gpu_warm(pb, guess)
    assert_parity(g, oracle_warm(pb, guess))
    assert_matches_kkt_reference(pb, g, what=f"n={n} G = 4I")


@pytest.mark.parametrize("n", [33, 70, 100, 116, 120, 128])
@pytest.mark.parametrize("fcache", ["1", "0"])
def test_warm_sequence_matches_stepwise_oracle(n, fcache):
    """jrlqp_solve_sequence_host, every step warm-started from the previous one, with the factor of step 0 re-read from
    HBM (JRLQP_SEQ_FCACHE=1) or recomputed (=0); n >= 116 runs on the global-workspace kernel."""
    B, T = (300, 6) if n <= 100 else (150, 4)
    pb = P.random_problems(slot_characteristics(n), B, seed=700 + n)
    a_seq = _trajectory(pb, T, n)

    def run():
        sv = S.BatchedGoldfarbIdnaniSolver(pb.n, pb.mc, True, B)
        sv.solve_sequence(pb.G, a_seq, pb.C, pb.bl, pb.bu, pb.xl, pb.xu, warm=True, keep_steps=True)
        return sv.last
    g = _seq_with_env(fcache, run)
    ref = _oracle_sequence(pb, a_seq, True)
    for t in range(T):
        for k in ("x", "u", "f", "iterations", "status"):
            assert np.array_equal(g[k][t], ref[t][k]), f"step {t}: {k} differs from the oracle"
    assert np.array_equal(g["active_set"], ref[-1]["active_set"])


# ---------------------------------------------------------------------------------------------
# automatic mode: warm starts whose shared-memory layout does not fit take the global-workspace kernel
# ---------------------------------------------------------------------------------------------
def _device_warm(sv, pb, as_in, shared=()):
    dev = torch.device("cuda:0")
    t = lambda v: None if v is None else torch.from_numpy(np.ascontiguousarray(v)).to(dev)  # noqa: E731
    B, n, m = pb.batch, pb.n, pb.mc + pb.nb
    out = dict(x=torch.empty((B, n), dtype=torch.float64, device=dev), u=torch.empty((B, m), dtype=torch.float64, device=dev),
               f=torch.empty(B, dtype=torch.float64, device=dev), iterations=torch.empty(B, dtype=torch.int32, device=dev),
               status=torch.empty(B, dtype=torch.int32, device=dev), active_set=torch.empty((B, m), dtype=torch.int8, device=dev),
               active_list=torch.empty((B, n), dtype=torch.int32, device=dev), n_active=torch.empty(B, dtype=torch.int32, device=dev))
    sv.solve_device(B, t(pb.G), t(pb.a), t(pb.C), t(pb.bl), t(pb.bu), t(pb.xl), t(pb.xu), stream=torch.cuda.current_stream().cuda_stream,
                    shared=shared, experimental=True, as_in=t(as_in), **out)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


@pytest.mark.parametrize("n", [116, 120, 128])
def test_automatic_mode_runs_warm_starts_that_do_not_fit_on_the_global_workspace_kernel(n):
    pb, act, wrong, ref = _case(n)
    sv = S.BatchedGoldfarbIdnaniSolver(n, pb.mc, True, pb.batch)
    sv.options(S.SolverOptions().warmStart(True))
    sv.solve(pb.G, pb.a, pb.C, pb.bl, pb.bu, pb.xl, pb.xu, experimental=True, as_in=wrong)
    auto = sv.last
    assert_parity(auto, ref["wrong"])
    assert sv.kernel_info()["threads_per_qp"] == 128  # cold calls keep the shared-memory kernel
    sv.solve(pb.G, pb.a, pb.C, pb.bl, pb.bu, pb.xl, pb.xu)
    assert_parity(sv.last, oracle_cold(pb))
    assert_parity(_device_warm(sv, pb, wrong), ref["wrong"])
    _assert_same_bits(auto, _gpu_warm(pb, wrong, path=2))
    with pytest.raises(S.JrlQpError):
        _gpu_warm(pb, wrong, path=1)
    # G shared by the batch: factorised once per call (prefactor), through both entry points
    sh = P.ProblemBatch(pb.G[0], pb.a, pb.C, pb.bl, pb.bu, pb.xl, pb.xu)
    ref_sh = oracle_warm(sh, act)
    sv.solve(sh.G, sh.a, sh.C, sh.bl, sh.bu, sh.xl, sh.xu, experimental=True, as_in=act)
    assert_parity(sv.last, ref_sh)
    assert_parity(_device_warm(sv, sh, act, shared=("G",)), ref_sh)


def test_warm_start_entries_at_n_120():
    """The class mirror and the multi-GPU warm entry (two shards on device 0) at a size the shared-memory warm kernel
    cannot hold."""
    pb, act, wrong, ref = _case(120)
    ws = S.experimental.GoldfarbIdnaniSolver(120, pb.mc, True)
    ws.options(S.SolverOptions().warmStart(True))
    assert ws.solve(pb.G[0].T.copy(), pb.a[0], pb.C[0].T, pb.bl[0], pb.bu[0], pb.xl[0], pb.xu[0], act[0]) == S.TerminationStatus.SUCCESS
    assert ws.iterations() == 0 and np.array_equal(ws.solution(), ref["exact"]["x"][0])
    mv = S.MultiGpuGoldfarbIdnaniSolver(120, pb.mc, True, pb.batch, devices=[0, 0])
    mv.options(S.SolverOptions().warmStart(True))
    mv.solve(pb.G, pb.a, pb.C, pb.bl, pb.bu, pb.xl, pb.xu, experimental=True, as_in=wrong)
    assert_parity(mv.last, ref["wrong"])
