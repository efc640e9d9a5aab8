"""One handle driven through a fixed script of reconfigurations: set_stage_c(0 / 1 / -1), then set_kernel_path 2 -> 0 -> 1
(at n > 128 a refused set_kernel_path(1)). After each step the handle runs every entry: cold host, cold device, warm host,
warm device (the device calls on two streams) and a warm-started sequence. Every result and kernel_info() must equal, bit
for bit, those of a fresh handle configured the same way.

Shapes: n = 50 (two warps), n = 70 (three warps: the register-capped choice), n = 120 (warm calls take the large-n kernel,
cold calls the shared-memory one) and n = 300 (large-n kernel, TMA column ring on). At n = 120 and 300, G and C are shared
by the batch, so the factor of the shared G and the transposed shared C are prepared by both kinds of entry."""
import numpy as np
import pytest
import torch

import jrl_qp_b200  # noqa: F401
from jrl_qp_b200 import solver as S, problems as P
from test_warm_kkt_reference import slot_characteristics

pytestmark = pytest.mark.gpu

B, T = 48, 3
SHARED = ("G", "C", "bl", "bu", "xl", "xu")
SHAPES = {50: False, 70: False, 120: True, 300: True}  # n: G, C and the bounds shared by the batch


def _inputs(n, shared):
    base = P.random_problems(slot_characteristics(n), B, seed=4100 + n)
    rng = np.random.default_rng(n)
    if shared:
        arrs = dict(G=base.G[0], a=base.a[0] + 0.05 * rng.standard_normal((B, n)), C=base.C[0], bl=base.bl[0], bu=base.bu[0],
                    xl=base.xl[0], xu=base.xu[0])
    else:
        arrs = dict(G=base.G, a=base.a, C=base.C, bl=base.bl, bu=base.bu, xl=base.xl, xu=base.xu)
    a_seq = np.stack([arrs["a"] + 0.02 * t * rng.standard_normal((B, n)) for t in range(T)])
    return base.mc, arrs, a_seq


def _solver(n, mc, stage=-1, path=0):
    sv = S.BatchedGoldfarbIdnaniSolver(n, mc, True, B)
    sv.options(S.SolverOptions().warmStart(True))
    if stage != -1:
        sv.set_stage_c(stage)
    if path != 0:
        sv.set_kernel_path(path)
    return sv


def _host(sv, h, **kw):
    sv.solve(h["G"], h["a"], h["C"], h["bl"], h["bu"], h["xl"], h["xu"], **kw)
    return dict(sv.last)


def _device(sv, d, shared, stream, **kw):
    dev = torch.device("cuda:0")
    n, m = sv.n, sv.m
    out = dict(x=torch.empty((B, n), dtype=torch.float64, device=dev), u=torch.empty((B, m), dtype=torch.float64, device=dev),
               f=torch.empty(B, dtype=torch.float64, device=dev), iterations=torch.empty(B, dtype=torch.int32, device=dev),
               status=torch.empty(B, dtype=torch.int32, device=dev), active_set=torch.empty((B, m), dtype=torch.int8, device=dev),
               active_list=torch.empty((B, n), dtype=torch.int32, device=dev), n_active=torch.empty(B, dtype=torch.int32, device=dev))
    sv.solve_device(B, d["G"], d["a"], d["C"], d["bl"], d["bu"], d["xl"], d["xu"], stream=stream.cuda_stream,
                    shared=SHARED if shared else (), **kw, **out)
    return out


def _outcome(call):
    """The call's result, or the message of its refusal (warm calls at n = 120 on the shared-memory path)."""
    try:
        return call()
    except S.JrlQpError as e:
        return str(e)


def _sequence(sv, h, a_seq):
    sv.solve_sequence(h["G"], a_seq, h["C"], h["bl"], h["bu"], h["xl"], h["xu"], warm=True, keep_steps=True)
    return dict(sv.last)


def _calls(sv, h, a_seq, guess, shared, streams):
    """Every entry once; the two device calls are enqueued back to back on two streams."""
    d = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in h.items()}
    d_guess = torch.from_numpy(guess).cuda()
    torch.cuda.synchronize()
    res = {"kernel_info": sv.kernel_info(), "cold host": _outcome(lambda: _host(sv, h))}
    dev = {"cold device": _outcome(lambda: _device(sv, d, shared, streams[0])),
           "warm device": _outcome(lambda: _device(sv, d, shared, streams[1], experimental=True, as_in=d_guess))}
    torch.cuda.synchronize()
    res.update({k: v if isinstance(v, str) else {kk: vv.cpu().numpy() for kk, vv in v.items()} for k, v in dev.items()})
    res["warm host"] = _outcome(lambda: _host(sv, h, experimental=True, as_in=guess))
    res["warm sequence"] = _outcome(lambda: _sequence(sv, h, a_seq))
    return res


def _assert_same(got, want, what):
    assert got["kernel_info"] == want["kernel_info"], f"{what}: kernel_info {got['kernel_info']} != {want['kernel_info']}"
    for call, ref in want.items():
        if call == "kernel_info":
            continue
        if isinstance(ref, str) or isinstance(got[call], str):
            assert got[call] == ref, f"{what}, {call}: {got[call]!r:.200} != {ref!r:.200}"
            continue
        assert ref["status"].shape[-1] == B  # (a sequence keeps [T, B])
        for k, v in ref.items():
            assert np.array_equal(got[call][k], v), f"{what}, {call}: {k} differs from a fresh handle's"


@pytest.mark.parametrize("n", sorted(SHAPES))
def test_reconfigured_handle_matches_a_fresh_one(n):
    shared = SHAPES[n]
    mc, h, a_seq = _inputs(n, shared)
    streams = (torch.cuda.Stream(), torch.cuda.Stream())
    # the warm start's guess: the active sets of the last step's linear terms (a few iterations away from the solutions)
    guess = _host(_solver(n, mc), dict(h, a=a_seq[-1]))["active_set"]
    script = [("stage_c", 0), ("stage_c", 1), ("stage_c", -1), ("path", 2), ("path", 0), ("path", 1)]
    sv = _solver(n, mc)
    stage, path = -1, 0
    for step, mode in [("create", None)] + script:
        if step == "stage_c":
            sv.set_stage_c(mode)
            stage = mode
        elif step == "path" and (mode != 1 or n <= 128):
            sv.set_kernel_path(mode)
            path = mode
        elif step == "path":
            with pytest.raises(S.JrlQpError, match="needs n <= 128"):
                sv.set_kernel_path(mode)
        got = _calls(sv, h, a_seq, guess, shared, streams)
        fresh = _solver(n, mc, stage, path)
        want = _calls(fresh, h, a_seq, guess, shared, streams)
        del fresh
        _assert_same(got, want, f"n = {n}, after {step}({mode})")
        # every call runs, except the warm ones at n = 120 once the shared-memory path is forced
        refused = [k for k, v in got.items() if isinstance(v, str)]
        assert refused == (["warm device", "warm host", "warm sequence"] if (n, path) == (120, 1) else []), refused
