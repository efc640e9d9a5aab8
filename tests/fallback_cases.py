"""Inputs of tests/test_gpu_fallbacks.py, shared by the test (shipped library, oracle) and by fallback_worker.py (the
library built with -DJRLQP_TEST_FALLBACKS, in a child process). Every case is deterministic: the same name gives the
same inputs in both processes. A case's `run(S)` solves on the GPU through the solver module S and returns a dict of
output arrays; `oracle()` returns the CPU oracle's outputs under the same keys (None where the oracle has no
counterpart of the call)."""
import os

import numpy as np

import block_cases as bc
import pyoracle as po
import structured_cases as sc
from jrl_qp_b200 import problems as P
from jrl_qp_b200.structured import Structure, Type

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
QP_KEYS = ("status", "iterations", "n_active", "active_set", "active_list", "x", "u", "f")
S840 = 2.0 ** -840  # moves every divisor of G's factor and of R out of the +-400-binade range of the proofs
S980 = 2.0 ** -980  # small-tile LLT: pivots below the sqrt sequence's range guard (biased exponent <= 64)
NCPU = os.cpu_count()


def _nthreads():
    return NCPU


# ------------------------------------------------------------------------------------------------------------------------
# problems
# ------------------------------------------------------------------------------------------------------------------------
def ch_n(n, ne, ni):
    return P.ProblemCharacteristics(n, ne, ni, nStrongActIneq=max(1, ni // 7), bounds=True, nStrongActBounds=max(1, n // 14),
                                    doubleSidedIneq=True)


def dense_problem(name, B):
    chs = {"B": P.config_B(), "A": P.config_A(), "D": P.config_D(), "n70": ch_n(70, 5, 150), "n90": ch_n(90, 9, 120),
           "n100": ch_n(100, 10, 110),
           "weak": P.ProblemCharacteristics(12, 2, 14, 3, 3, 1, 2, True, True), "n160": ch_n(160, 32, 128), "n300": ch_n(300, 60, 240),
           "n800": ch_n(800, 80, 720)}
    return P.random_problems(chs[name], B, seed=9000 + chs[name].nVar)


def scaled(pb, s):
    """G and a scaled by s: x is unchanged, u and f scale by s exactly (power-of-two s, nothing subnormal)."""
    return P.ProblemBatch(pb.G * s, pb.a * s, pb.C, pb.bl, pb.bu, pb.xl, pb.xu)


def wrong_guess(act, mc, seed):
    """A quarter of the entries of an active set flipped to the other side / activated (kinds of include/jrlqp_b200.h)."""
    rng = np.random.default_rng(seed)
    m = act.shape[1]
    swapped = act.copy()
    swapped[act == 1], swapped[act == 2], swapped[act == 4], swapped[act == 5] = 2, 1, 5, 4
    kind_lower = np.where(np.arange(m) < mc, 1, 4).astype(np.int8)
    swapped[act == 0] = np.broadcast_to(kind_lower, act.shape)[act == 0]
    return np.where(rng.random(act.shape) < 0.25, swapped, act).astype(np.int8)


def multiik(which, B, seed=0):
    d = np.load(os.path.join(GOLDEN, f"multiik_{which}.npz"))
    rng = np.random.default_rng(seed)
    a = d["a"][None] * (1.0 + 1e-3 * rng.standard_normal((B, d["a"].size)))
    a[0] = d["a"]
    bu = d["u"]
    xl, xu = (d["xl"], d["xu"]) if which == "simultaneous" else (None, None)
    return P.ProblemBatch(np.ascontiguousarray(d["G"].T), a, np.ascontiguousarray(d["C"]), np.full_like(bu, -np.inf), bu, xl, xu)


def dyadic_problem(kind, B, seed):
    """Textbook-shaped problems whose quotients are often powers of two: G = I or 4 I, constraint normals with equal
    entries or entries +-1, integer bounds."""
    rng = np.random.default_rng(seed)
    n, mc = 24, 30
    G = np.broadcast_to((4.0 if kind.endswith("4I") else 1.0) * np.eye(n), (B, n, n)).copy()
    if kind.startswith("equal"):
        # one value per row (1 ... 3, either sign) on a random half of the variables
        Cm = np.repeat((rng.integers(1, 4, (B, mc, 1)) * rng.choice([-1, 1], (B, mc, 1))).astype(float), n, axis=2)
        Cm *= rng.random((B, mc, n)) < 0.5
    else:
        Cm = rng.choice([-1.0, 1.0], (B, mc, n))
    bl = -rng.integers(1, 4, (B, mc)).astype(float)
    bu = rng.integers(0, 3, (B, mc)).astype(float)
    a = rng.integers(-8, 9, (B, n)).astype(float)
    xl = -np.ones((B, n)) * rng.integers(1, 3, (B, 1))
    xu = np.ones((B, n)) * rng.integers(1, 3, (B, 1))
    return P.ProblemBatch(G, a, Cm, bl, bu, xl, xu)


def sequence_workload(n, B, T, seed):
    """The shape of the warm-start benchmark (benchmarks/SolversWarmStart.cpp as bench.py --sequence runs it): G = I,
    n double-sided tangent-plane rows (unit normals) with bounds +-1, variable bounds +-1, a(t) rotating on a sphere."""
    rng = np.random.default_rng(seed)

    def unit(*shape):
        v = rng.standard_normal(shape)
        return v / np.linalg.norm(v, axis=-1, keepdims=True)
    Cm = unit(B, n, n)
    r = 2.0 * np.sqrt(n)
    p1, p2 = r * unit(B, n), r * unit(B, n)
    c = (p1 * p2).sum(-1, keepdims=True) / (p1 * p1).sum(-1, keepdims=True)
    v = p2 - c * p1
    v *= np.linalg.norm(p1, axis=-1, keepdims=True) / np.linalg.norm(v, axis=-1, keepdims=True)
    w = np.arccos(c)
    t = (np.arange(T) / T)[:, None, None]
    a_seq = np.cos(t * w) * p1 + np.sin(t * w) * v
    return dict(G=np.eye(n), C=Cm, bl=-np.ones(n), bu=np.ones(n), xl=-np.ones(n), xu=np.ones(n), a_seq=np.ascontiguousarray(a_seq))


# ------------------------------------------------------------------------------------------------------------------------
# GPU calls and their oracle counterparts
# ------------------------------------------------------------------------------------------------------------------------
def gpu_cold(S, pb, path=0, stage=-1, big_bnd=None, want_L=False):
    sv = S.BatchedGoldfarbIdnaniSolver(pb.n, pb.mc, pb.nb > 0, pb.batch)
    sv.set_kernel_path(path)
    sv.set_stage_c(stage)
    if big_bnd is not None:
        sv.options(S.SolverOptions().bigBnd(big_bnd))
    sv.solve(pb.G, pb.a, pb.C, pb.bl, pb.bu, pb.xl, pb.xu, want_L=want_L)
    return {k: sv.last[k] for k in QP_KEYS + (("L",) if want_L else ())}


def gpu_warm(S, pb, as_in, path=0, big_bnd=None, max_iter=500):
    sv = S.BatchedGoldfarbIdnaniSolver(pb.n, pb.mc, pb.nb > 0, pb.batch)
    sv.set_kernel_path(path)
    o = S.SolverOptions().warmStart(True).maxIter(max_iter)
    if big_bnd is not None:
        o.bigBnd(big_bnd)
    sv.options(o)
    sv.solve(pb.G, pb.a, pb.C, pb.bl, pb.bu, pb.xl, pb.xu, experimental=True, as_in=as_in)
    return {k: sv.last[k] for k in QP_KEYS}


def oracle_cold(pb, big_bnd=1e100):
    r = po.solve_batch(pb.G, pb.a, pb.C, pb.bl, pb.bu, pb.xl, pb.xu, big_bnd=big_bnd, nthreads=_nthreads())
    return {k: r[k] for k in QP_KEYS}


def oracle_warm(pb, as_in, big_bnd=1e100, max_iter=500):
    r = po.solve_batch(pb.G, pb.a, pb.C, pb.bl, pb.bu, pb.xl, pb.xu, big_bnd=big_bnd, nthreads=_nthreads(), experimental=True,
                       warm_start=True, as_in=as_in, max_iter=max_iter)
    return {k: r[k] for k in QP_KEYS}


def gpu_sequence(S, w, B):
    n = w["G"].shape[0]
    sv = S.BatchedGoldfarbIdnaniSolver(n, n, True, B)
    sv.options(S.SolverOptions().warmStart(True))
    sv.solve_sequence(w["G"], w["a_seq"], w["C"], w["bl"], w["bu"], w["xl"], w["xu"], warm=True, keep_steps=True)
    return {k: sv.last[k] for k in ("x", "u", "f", "iterations", "status", "active_set", "iterations_total", "status_worst")}


def oracle_sequence(w):
    """The sequence chained on the oracle: step 0 cold through the warm-capable solver with an empty guess, every later
    step warm-started from the active set the previous one ended with."""
    T, B, n = w["a_seq"].shape
    rep = lambda v: np.broadcast_to(v, (B,) + v.shape).copy()  # noqa: E731
    G, bl, bu, xl, xu = (rep(w[k]) for k in ("G", "bl", "bu", "xl", "xu"))
    Cm = w["C"]
    out = {k: [] for k in ("x", "u", "f", "iterations", "status")}
    act = None
    for t in range(T):
        r = po.solve_batch(G, w["a_seq"][t], Cm, bl, bu, xl, xu, nthreads=_nthreads(), experimental=True, warm_start=True,
                           as_in=act)
        for k in out:
            out[k].append(r[k])
        act = r["active_set"]
    res = {k: np.stack(v) for k, v in out.items()}
    res["active_set"] = act
    res["iterations_total"] = res["iterations"].sum(axis=0).astype(np.int32)
    res["status_worst"] = res["status"].max(axis=0)
    return res


def structured_factor(S, st, H, kernel):
    from jrl_qp_b200.structured import StructuredG
    g = StructuredG(st, st.pack(H))
    g.set_kernel(kernel)
    ok = g.lltInPlace()
    return g, ok


def structured_windows(n, size):
    return sorted({(0, n), (0, 1), (n - 1, n), (size // 2, n), (0, n - size // 2), (size, n), (0, size)})


def run_structured(S, size, blocks, batch, kernel, s, seed):
    st = Structure.packed(Type.TriBlockDiagonal, [size] * blocks)
    H = sc.make_H(Type.TriBlockDiagonal, [size] * blocks, batch, seed=seed, shift=1.0) * s
    g, ok = structured_factor(S, st, H, kernel)
    out = {"ok": np.asarray(ok), "L": g.data.copy(), "input": st.pack(H)}
    V = np.random.default_rng(seed + 1).uniform(-1, 1, (batch, 2, st.n))
    out["rhs"] = V
    for i, j in structured_windows(st.n, size):
        out[f"fwd{i}_{j}"] = g.solveL(V.copy(), i, j)
        out[f"bwd{i}_{j}"] = g.solveLTranspose(V.copy(), i, j)
    return out


def oracle_structured(size, blocks, batch, s, seed):
    st = Structure.packed(Type.TriBlockDiagonal, [size] * blocks)
    H = sc.make_H(Type.TriBlockDiagonal, [size] * blocks, batch, seed=seed, shift=1.0) * s
    data = st.pack(H)
    ok = po.decomp_llt(st, data, nthreads=_nthreads())
    out = {"ok": np.asarray(ok).astype(bool), "L": data, "input": st.pack(H)}
    V = np.random.default_rng(seed + 1).uniform(-1, 1, (batch, 2, st.n))
    out["rhs"] = V
    for i, j in structured_windows(st.n, size):
        out[f"fwd{i}_{j}"] = po.decomp_solve(st, data, V.copy(), transpose=False, start=i, end=j, nthreads=_nthreads())
        out[f"bwd{i}_{j}"] = po.decomp_solve(st, data, V.copy(), transpose=True, start=i, end=j, nthreads=_nthreads())
    return out


def block_problem(which, s=1.0):
    if which == "ref":
        pb = bc.random_block_problem(Type.TriBlockDiagonal, [3, 5, 2, 3], [3, 3, 3, 3], 32, seed=31, shift=0.05)
    elif which == "wide":
        pb = bc.random_block_problem(Type.TriBlockDiagonal, [12] * 6, [7] * 6, 16, seed=217, bounds=True, shift=0.05)
    elif which == "n528":
        pb = bc.random_block_problem(Type.TriBlockDiagonal, [12] * 44, [6] * 44, 4, seed=528, bounds=True, shift=0.05)
    else:
        pb, _ = bc.multiik_sequential(6, scale=1e-3)
    if s != 1.0:
        pb.Gdata = pb.Gdata * s
        pb.a = pb.a * s
    return pb


def gpu_block(S, pb, big_bnd=None):
    from jrl_qp_b200.blockgi import BatchedBlockGISolver
    B = pb.a.shape[0] if pb.a.ndim == 2 else 1
    sv = BatchedBlockGISolver(pb.stG, pb.stC, pb.xl is not None, B)
    if big_bnd is not None:
        sv.options(S.SolverOptions().bigBnd(big_bnd))
    sv.solve(pb.Gdata, pb.a, pb.Cdata, pb.bl, pb.bu, pb.xl, pb.xu)
    return {k: sv.last[k] for k in QP_KEYS}


def oracle_block(pb, big_bnd=1e100):
    r = po.block_solve_batch(pb.stG, pb.stC, pb.Gdata, pb.a, pb.Cdata, pb.bl, pb.bu, pb.xl, pb.xu, big_bnd=big_bnd,
                             nthreads=_nthreads())
    return {k: r[k] for k in QP_KEYS}


# ------------------------------------------------------------------------------------------------------------------------
# the cases
# ------------------------------------------------------------------------------------------------------------------------
class Case:
    def __init__(self, name, run, oracle):
        self.name, self.run, self.oracle = name, run, oracle


def _dense_cold(name, B, path=0, stage=-1, s=1.0, want_L=True):
    pb = lambda: scaled(dense_problem(name, B), s) if s != 1.0 else dense_problem(name, B)  # noqa: E731
    bb = None if s == 1.0 else 1e100 * s
    return (lambda S: gpu_cold(S, pb(), path, stage, bb, want_L)), (lambda: oracle_cold(pb(), 1e100 if bb is None else bb))


def _dense_warm(name, B, path, guess, s=1.0, max_iter=500):
    """Warm start from the oracle's cold active set ("exact") or from a wrong guess derived from it."""
    def inputs():
        pb0 = dense_problem(name, B)
        act = oracle_cold(pb0)["active_set"]
        as_in = act if guess == "exact" else wrong_guess(act, pb0.mc, seed=B)
        return (scaled(pb0, s) if s != 1.0 else pb0), as_in
    bb = None if s == 1.0 else 1e100 * s

    def run(S):
        pb, as_in = inputs()
        return gpu_warm(S, pb, as_in, path, bb, max_iter)

    def oracle():
        pb, as_in = inputs()
        return oracle_warm(pb, as_in, 1e100 if bb is None else bb, max_iter)
    return run, oracle


def _dense_shared(name, B):
    """G, C and bounds shared by the batch, a per instance: the large kernel factorises G once (prefactor kernel) and
    every CTA computes x = -G^-1 a from the shared factor in initial_point_blocked."""
    def sh():
        pb = dense_problem(name, B)
        a = pb.a[0] + 0.05 * np.random.default_rng(1).standard_normal(pb.a.shape)
        return P.ProblemBatch(pb.G[0], a, pb.C[0], pb.bl[0], pb.bu[0], pb.xl[0], pb.xu[0])
    return (lambda S: gpu_cold(S, sh(), 2)), (lambda: oracle_cold(_replicated(sh())))


def _multiik(which, B, warm):
    def run(S):
        pb = multiik(which, B)
        if not warm:
            return gpu_cold(S, pb, 0)
        return gpu_warm(S, pb, np.roll(oracle_cold(pb)["active_set"], 1, axis=0), 0)

    def oracle():
        pb = multiik(which, B)
        r = oracle_cold(pb)
        return oracle_warm(pb, np.roll(r["active_set"], 1, axis=0)) if warm else r
    return run, oracle


def _dyadic(kind, B, warm, path=0):
    def run(S):
        pb = dyadic_problem(kind, B, seed=len(kind))
        if not warm:
            return gpu_cold(S, pb, path)
        return gpu_warm(S, pb, wrong_guess(oracle_cold(pb)["active_set"], pb.mc, seed=5), path)

    def oracle():
        pb = dyadic_problem(kind, B, seed=len(kind))
        r = oracle_cold(pb)
        return oracle_warm(pb, wrong_guess(r["active_set"], pb.mc, seed=5)) if warm else r
    return run, oracle


def _seq(n, B, T):
    return (lambda S: gpu_sequence(S, sequence_workload(n, B, T, 20261018), B)), (lambda: oracle_sequence(sequence_workload(n, B, T, 20261018)))


def _structured(size, blocks, batch, kernel, s=1.0):
    return (lambda S: run_structured(S, size, blocks, batch, kernel, s, 11 + size)), (lambda: oracle_structured(size, blocks, batch, s, 11 + size))


def _block(which, s=1.0):
    bb = None if s == 1.0 else 1e100 * s
    return (lambda S: gpu_block(S, block_problem(which, s), bb)), (lambda: oracle_block(block_problem(which, s), 1e100 if bb is None else bb))


def _cases(spec):
    return [Case(e[0], *(e[1] if len(e) == 2 else e[1:])) for e in spec]


# Part (a): every kernel family, natural inputs; under the decline flag every fallback runs
FAMILY_CASES = _cases([
    ("dense_B", _dense_cold("B", 256)),                       # one warp per QP
    ("dense_A_staged", _dense_cold("A", 128, stage=1)),        # two warps
    ("dense_A_unstaged", _dense_cold("A", 128, stage=0)),
    ("dense_n70", _dense_cold("n70", 48)),                     # three warps, register-capped instantiation
    ("dense_n90", _dense_cold("n90", 48)),                     # three warps
    ("dense_D", _dense_cold("D", 32, stage=0)),                # four warps: branch-free Givens links
    ("dense_n100_staged", _dense_cold("n100", 32, stage=1)),
    ("dense_warm_A_wrong", _dense_warm("A", 128, 1, "wrong")),
    ("dense_warm_B_wrong", _dense_warm("B", 256, 1, "wrong")),
    ("dense_warm_n70_wrong", _dense_warm("n70", 48, 1, "wrong")),    # warm, three warps
    ("dense_warm_n100_wrong", _dense_warm("n100", 32, 1, "wrong")),  # warm, four warps: branch-free Givens links
    ("large_n160_cold", _dense_cold("n160", 12, path=2)),
    ("large_n160_warm", _dense_warm("n160", 12, 2, "wrong")),
    ("large_n300_cold", _dense_cold("n300", 6, path=2)),
    ("large_n300_warm", _dense_warm("n300", 6, 2, "wrong")),
    ("large_n800_cold", _dense_cold("n800", 3, path=2)),        # four rows per thread, no column ring
    ("large_n800_warm", _dense_warm("n800", 3, 2, "wrong", max_iter=2000)),  # warm, J = J Q without shared-memory slabs
                                                                              # (about 670 iterations)
    ("large_n800_shared", _dense_shared("n800", 3)),            # prefactor of the shared G, initial_point_blocked
    ("multiik_seq_cold", _multiik("sequential", 6, False)),    # G and C shared by the batch
    ("multiik_seq_warm", _multiik("sequential", 6, True)),
    ("multiik_sim_cold", _multiik("simultaneous", 6, False)),
    ("multiik_sim_warm", _multiik("simultaneous", 6, True)),
    ("sequence_fcache", _seq(20, 64, 6)),                      # warm sequence, factor cache on (default)
    ("structured_k1", _structured(12, 6, 37, 1)),
    ("structured_k2", _structured(8, 5, 37, 2)),
    ("structured_k3", _structured(16, 4, 37, 3)),
    ("blockgi_ref", _block("ref")),
    ("blockgi_wide", _block("wide")),
    ("blockgi_multiik", _block("multiik")),
    ("blockgi_n528", _block("n528")),                          # eight entries of a reflector per thread (n > 512)
])

# Part (b) / shipped-build edge tests: binade-shifted and dyadic inputs
EDGE_CASES = _cases([
    ("binade_A", _dense_cold("A", 64, s=S840)),
    ("binade_B", _dense_cold("B", 128, s=S840)),
    ("binade_D", _dense_cold("D", 16, s=S840)),
    ("binade_n70", _dense_cold("n70", 24, s=S840)),
    ("binade_n300", _dense_cold("n300", 4, s=S840)),
    ("binade_weak", _dense_cold("weak", 128, s=S840)),          # weakly active: absolute thresholds, parity only
    ("binade_n300_shared", (lambda S: gpu_cold(S, _shared_binade(), 0, -1, 1e100 * S840)),
     lambda: oracle_cold(_replicated(_shared_binade()), 1e100 * S840)),
    ("binade_warm_A", _dense_warm("A", 64, 1, "exact", s=S840)),
    ("binade_warm_B", _dense_warm("B", 128, 1, "exact", s=S840)),
    ("binade_warm_D", _dense_warm("D", 16, 2, "exact", s=S840)),
    ("binade_warm_n300_shared", (lambda S: gpu_warm(S, _shared_binade(), _shared_binade_guess(), 0, 1e100 * S840)),
     lambda: oracle_warm(_replicated(_shared_binade()), _shared_binade_guess(), 1e100 * S840)),
    ("binade_structured_k1", _structured(12, 6, 37, 1, S840)),
    ("binade_structured_k2", _structured(8, 5, 37, 2, S980)),
    ("binade_structured_k3", _structured(16, 4, 37, 3, S980)),
    ("binade_blockgi_ref", _block("ref", S840)),
    ("binade_blockgi_wide", _block("wide", S840)),
    ("dyadic_I_cold", _dyadic("pm1_I", 256, False)),
    ("dyadic_4I_cold", _dyadic("equal_4I", 256, False)),
    ("dyadic_I_warm", _dyadic("equal_I", 256, True)),
    ("dyadic_4I_warm", _dyadic("pm1_4I", 256, True)),
    ("dyadic_I_large", _dyadic("pm1_I", 32, False, path=2)),
    ("dyadic_sequence", _seq(20, 64, 6)),
])


def _shared_binade():
    """G, C and bounds shared by the batch (the large kernel factorises G once), n = 300, scaled by 2^-840."""
    pb = dense_problem("n300", 4)
    rng = np.random.default_rng(1)
    a = pb.a[0] + 0.05 * rng.standard_normal(pb.a.shape)
    return P.ProblemBatch(pb.G[0] * S840, a * S840, pb.C[0], pb.bl[0], pb.bu[0], pb.xl[0], pb.xu[0])


def _replicated(sh):
    B = sh.a.shape[0]
    rep = lambda v: np.repeat(v[None], B, axis=0)  # noqa: E731
    return P.ProblemBatch(rep(sh.G), sh.a, rep(sh.C), rep(sh.bl), rep(sh.bu), rep(sh.xl), rep(sh.xu))


def _shared_binade_guess():
    return oracle_cold(_replicated(_shared_binade()), 1e100 * S840)["active_set"]


# the unscaled twins of the binade-shifted cases (the relation scaled vs unscaled needs no oracle)
UNSCALED_CASES = _cases([
    ("unscaled_A", _dense_cold("A", 64)),
    ("unscaled_B", _dense_cold("B", 128)),
    ("unscaled_D", _dense_cold("D", 16)),
    ("unscaled_n70", _dense_cold("n70", 24)),
    ("unscaled_n300", _dense_cold("n300", 4)),
    ("unscaled_warm_A", _dense_warm("A", 64, 1, "exact")),
    ("unscaled_warm_B", _dense_warm("B", 128, 1, "exact")),
    ("unscaled_warm_D", _dense_warm("D", 16, 2, "exact")),
    ("unscaled_structured_k1", _structured(12, 6, 37, 1)),
    ("unscaled_structured_k2", _structured(8, 5, 37, 2)),
    ("unscaled_structured_k3", _structured(16, 4, 37, 3)),
    ("unscaled_blockgi_ref", _block("ref")),
    ("unscaled_blockgi_wide", _block("wide")),
])

RUN_CASES = [c.name for c in FAMILY_CASES + EDGE_CASES]  # what the test build runs, in both modes
ALL_CASES = {c.name: c for c in FAMILY_CASES + EDGE_CASES + UNSCALED_CASES}
