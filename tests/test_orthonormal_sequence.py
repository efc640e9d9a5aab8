"""Known-answer tests of internal::OrthonormalSequence / ElemOrthonormalSequence / SingleNZSegmentVector as the
structured solver uses them — the reference's tests/InternalTest.cpp:35-323 restated:
  * sequences of Householder reflectors and of Givens rotations against the DENSE orthogonal matrix they represent
    (built here with numpy from the same (essential, tau) / (c, s) data), both directions, to 1e-8, norm preserved;
  * vectors with a single non-zero segment [0; x; 0] at every position (SingleNZSegmentVector): the (start, size)
    hint of the reference only skips work on zeros, so the full application must give Q v for them;
  * a composite sequence of four embedded transformations (InternalTest.cpp:223-323);
  * sequences at n = 513, 700 and 1024, where the kernel holds 5 ... 8 entries of a reflector and of the vector per thread
    (blockgi_kernel<8>): reflectors over the whole vector and starting at the class boundaries 127 / 128, and Givens
    records on either side of MJ * 64 rotations, the longest a thread-private stage holds (longer ones are read from
    global memory by givens_record), up to n - 1 rotations.
CPU part: the restatement inside oracle/block_oracle.cpp (the checker of the BlockGI kernel). GPU part (-m gpu): the
kernel's own apply_q / apply_qt through jrlqp_blockgi_test_sequence, bit for bit against the oracle and to 1e-8
against the dense matrix."""
import ctypes as C
import functools
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import pyoracle as po  # noqa: E402

GIVENS_FLAG = -(1 << 31)


def _lib():
    L = po.lib()
    L.block_oracle_seq_create.restype = C.c_void_p
    L.block_oracle_seq_create.argtypes = [C.c_int]
    L.block_oracle_seq_destroy.argtypes = [C.c_void_p]
    L.block_oracle_seq_add_householder.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_double]
    L.block_oracle_seq_add_givens.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.block_oracle_seq_apply.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    L.block_oracle_make_householder.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    return L


def make_householder(x):
    """VectorXd::makeHouseholderInPlace as StructuredQR::add applies it: (essential, tau, beta)."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    ess = np.zeros(max(len(x) - 1, 1))
    tau, beta = C.c_double(), C.c_double()
    _lib().block_oracle_make_householder(x.ctypes.data, len(x), ess.ctypes.data, C.byref(tau), C.byref(beta))
    return ess[:len(x) - 1], tau.value, beta.value


def make_givens(p, q):
    """Eigen JacobiRotation::makeGivens, real case (SURVEY.md appendix B): (c, s)."""
    if q == 0:
        return (-1.0 if p < 0 else 1.0), 0.0
    if p == 0:
        return 0.0, (1.0 if q < 0 else -1.0)
    if abs(p) > abs(q):
        t = q / p
        u = np.sqrt(1 + t * t) * (-1 if p < 0 else 1)
        c = 1 / u
        return c, -t * c
    t = p / q
    u = np.sqrt(1 + t * t) * (-1 if q < 0 else 1)
    s = -1 / u
    return -t * s, s


class Sequence:
    """Records in addition order + the dense Q = E1 E2 ... they represent (Q.middleCols(start, size) *= E.toDense())."""

    def __init__(self, n):
        self.n, self.recs = n, []
        self.Q = np.eye(n)

    def householder(self, start, essential, tau):
        e = np.concatenate([[1.0], essential])
        cols = self.Q[:, start:start + len(e)]  # Q H = Q - tau (Q e) e^T on the columns the reflector touches
        cols -= tau * np.outer(cols @ e, e)
        self.recs.append(("h", start, np.asarray(essential, dtype=np.float64), float(tau)))

    def givens(self, start, cs):
        # ElemOrthonormalSequence of Givens: G_1 G_2 ... G_k, G_i acting on (start + i, start + i + 1);
        # applyOnTheLeft(i, i+1, G): [x; y] <- [c x + s y; -s x + c y]
        # Q G_i on columns a, a + 1, with G_i = [[c, s], [-s, c]] there
        for i, (c, s) in enumerate(cs):
            a = start + i
            qa, qb = self.Q[:, a].copy(), self.Q[:, a + 1].copy()
            self.Q[:, a], self.Q[:, a + 1] = c * qa - s * qb, s * qa + c * qb
        self.recs.append(("g", start, np.array([c for c, _ in cs]), np.array([s for _, s in cs])))

    def oracle_apply(self, v, transpose):
        L = _lib()
        h = L.block_oracle_seq_create(self.n)
        keep = []
        for r in self.recs:
            if r[0] == "h":
                ess = np.ascontiguousarray(r[2])
                keep.append(ess)
                L.block_oracle_seq_add_householder(h, r[1], len(ess) + 1, ess.ctypes.data if len(ess) else None, r[3])
            else:
                c, s = np.ascontiguousarray(r[2]), np.ascontiguousarray(r[3])
                keep += [c, s]
                L.block_oracle_seq_add_givens(h, r[1], len(c), c.ctypes.data, s.ctypes.data)
        out = np.ascontiguousarray(v, dtype=np.float64).copy()
        L.block_oracle_seq_apply(h, out.ctypes.data, int(transpose))
        L.block_oracle_seq_destroy(h)
        return out

    def device_records(self):
        rec, data = [], []
        for r in self.recs:
            off = len(data)
            if r[0] == "h":
                rec += [r[1], len(r[2]) + 1, off]
                data += [r[3]] + list(r[2])
            else:
                rec += [r[1] + GIVENS_FLAG, len(r[2]), off]
                data += list(r[2]) + list(r[3])
        return np.array(rec, dtype=np.int32), np.array(data, dtype=np.float64)


def _elem_householder(rng, n=8, k=3):
    seq = Sequence(n)
    for j in range(k):
        ess, tau, _ = make_householder(rng.uniform(-1, 1, n - j))
        seq.householder(j, ess, tau)
    return seq


def _elem_givens(n=8):
    seq = Sequence(n)
    seq.givens(0, [make_givens(1, 2), make_givens(3, 4), make_givens(5, 6), make_givens(7, 8), make_givens(9, 10)])
    return seq


def _composite(rng):
    """tests/InternalTest.cpp:223-262: four transformations embedded in a 16-vector."""
    seq = Sequence(16)
    for j, ln in enumerate((6, 5, 4)):
        ess, tau, _ = make_householder(rng.uniform(-1, 1, ln))
        seq.householder(2 + j, ess, tau)
    seq.givens(5, [make_givens(1, 2), make_givens(3, 4), make_givens(5, 6), make_givens(7, 8), make_givens(9, 10)])
    ess, tau, _ = make_householder(rng.uniform(-1, 1, 4))
    seq.householder(12, ess, tau)
    ess, tau, _ = make_householder(rng.uniform(-1, 1, 7))
    seq.householder(1, ess, tau)
    return seq


def _vectors(rng, n, seg=None):
    """full random vectors + single-non-zero-segment vectors [0; x; 0] at every position (past n = 300: at the ends and
    across the boundaries of the 128 classes)"""
    vs = [rng.uniform(-1, 1, n)]
    ln = seg or 3
    pos = range(n - ln + 1) if n <= 300 else sorted({p for c in range(0, n, 128) for p in (c - 2, c - 1, c, c + 1)
                                                     if 0 <= p <= n - ln} | {n - ln})
    for i in pos:
        v = np.zeros(n)
        v[i:i + ln] = rng.uniform(-1, 1, ln)
        vs.append(v)
    return np.array(vs)


def _random_givens(rng, k):
    return [make_givens(*rng.uniform(-1, 1, 2)) for _ in range(k)]


def _large(rng, n, kind):
    """Records of a sequence at n > 512. A thread-private stage holds the (c, s) of MJ * 64 rotations, MJ = ceil(n / 128)."""
    seq, staged = Sequence(n), 64 * ((n + 127) // 128)

    def h(start):
        ess, tau, _ = make_householder(rng.uniform(-1, 1, n - start))
        seq.householder(start, ess, tau)
    if kind == "householder":
        for start in (0, 127, 128, 500, n - 2):
            h(start)
    elif kind == "givens":
        for start, k in ((130, 40), (0, staged), (n - 2 - staged, staged + 1), (0, n - 1)):
            seq.givens(start, _random_givens(rng, k))
    else:
        h(0)
        seq.givens(5, _random_givens(rng, staged + 3))
        h(127)
        seq.givens(120, _random_givens(rng, 50))
        h(n - 2)
        seq.givens(0, _random_givens(rng, n - 1))
        h(128)
    return seq


@functools.lru_cache(maxsize=None)
def _sequences():
    rng = np.random.default_rng(20261018)
    seqs = {"householder x3": _elem_householder(rng), "householder x1": _elem_householder(rng, k=1), "givens x5": _elem_givens(),
            "composite": _composite(rng), "long householder": _elem_householder(rng, n=300, k=2)}
    for n in (513, 700, 1024):
        for kind in ("householder", "givens", "composite"):
            seqs[f"{kind} n={n}"] = _large(rng, n, kind)
    return seqs


@pytest.mark.parametrize("name", list(_sequences()))
def test_oracle_sequence_against_dense_q(name):
    seq = _sequences()[name]
    rng = np.random.default_rng(1)
    assert np.abs(seq.Q @ seq.Q.T - np.eye(seq.n)).max() < 1e-12  # the dense matrix is orthogonal: (tau, essential) / (c, s) are consistent
    for v in _vectors(rng, seq.n, 4 if name == "composite" else 3):
        for transpose in (False, True):
            want = (seq.Q.T if transpose else seq.Q) @ v
            got = seq.oracle_apply(v, transpose)
            assert np.abs(got - want).max() <= 1e-8 * max(1.0, np.abs(want).max()), (name, transpose)
            assert abs(np.linalg.norm(got) - np.linalg.norm(v)) <= 1e-12 * max(1.0, np.linalg.norm(v))


def test_make_householder_annihilates_the_tail():
    rng = np.random.default_rng(5)
    for ln in (1, 2, 7, 40):
        x = rng.uniform(-1, 1, ln)
        ess, tau, beta = make_householder(x)
        e = np.concatenate([[1.0], ess])
        Hx = x - tau * e * (e @ x)
        assert abs(Hx[0] - beta) <= 1e-14 * max(1, abs(beta)) and (np.abs(Hx[1:]) <= 1e-14).all()
        assert abs(abs(beta) - np.linalg.norm(x)) <= 1e-14 * np.linalg.norm(x)
    ess, tau, beta = make_householder(np.array([0.75, 0.0, 0.0]))  # tail below the smallest normal: tau = 0, beta = c0
    assert tau == 0.0 and beta == 0.75 and (ess == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("fast", [7, 0])  # vector in registers, one barrier per reflector (round 2) / the shared-memory pass
@pytest.mark.parametrize("threads", [128, 256])
@pytest.mark.parametrize("name", list(_sequences()))
def test_device_sequence_equals_oracle_and_dense_q(name, threads, fast, monkeypatch):
    monkeypatch.setenv("JRLQP_BLOCKGI_FAST", str(fast))
    import jrl_qp_b200  # noqa: F401
    from jrl_qp_b200 import solver as S
    lib = S.load_library()
    seq = _sequences()[name]
    rec, data = seq.device_records()
    rng = np.random.default_rng(2)
    V = _vectors(rng, seq.n, 4 if name == "composite" else 3)
    before = S.launch_count()
    for transpose in (False, True):
        out = np.ascontiguousarray(V.copy())
        rc = lib.jrlqp_blockgi_test_sequence(C.c_int32(0), C.c_int32(seq.n), C.c_int32(len(rec) // 3), rec.ctypes.data_as(C.c_void_p),
                                             data.ctypes.data_as(C.c_void_p), C.c_int64(len(data)), out.ctypes.data_as(C.c_void_p),
                                             C.c_int32(len(V)), C.c_int32(int(transpose)), C.c_int32(threads))
        assert rc == 0
        for v, g in zip(V, out):
            want = (seq.Q.T if transpose else seq.Q) @ v
            assert np.abs(g - want).max() <= 1e-8 * max(1.0, np.abs(want).max())
            assert np.array_equal(g, seq.oracle_apply(v, transpose)), "kernel and oracle differ in the last bits"
    assert S.launch_count() > before


@pytest.mark.gpu
def test_device_sequence_refuses_more_than_1024_entries():
    import jrl_qp_b200  # noqa: F401
    from jrl_qp_b200 import solver as S
    lib = S.load_library()
    seq = Sequence(1025)
    seq.givens(0, [make_givens(1, 2)])
    rec, data = seq.device_records()
    v = np.ones(1025)
    rc = lib.jrlqp_blockgi_test_sequence(C.c_int32(0), C.c_int32(1025), C.c_int32(1), rec.ctypes.data_as(C.c_void_p),
                                         data.ctypes.data_as(C.c_void_p), C.c_int64(len(data)), v.ctypes.data_as(C.c_void_p),
                                         C.c_int32(1), C.c_int32(0), C.c_int32(128))
    assert rc == -2  # JRLQP_ERR_ARG
