"""Sparse QCQP family (LFPSQP_FAM_SPARSE_QCQP) without a GPU: canonicalisation of the data, the data-form slack embedding
against host.slack_callbacks, and the ctypes mirror of the C descriptor."""
import ctypes
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from lfpsqp.jl_b200 import _lib, families, host

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def dense(t, shape):
    """(row, col, val) or (mat, row, col, val) -> dense array"""
    out = np.zeros(shape)
    np.add.at(out, tuple(t[:-1]), t[-1])
    return out


def test_symmetrised_and_duplicates_summed():
    sp = pytest.importorskip("scipy.sparse")
    rng = np.random.default_rng(0)
    n = 7
    A = rng.standard_normal((n, n)) * (rng.random((n, n)) < 0.4)
    fam = families.sparse_qcqp(P=A, q=np.ones(n))
    Ps = dense(fam.P, (n, n))
    assert np.array_equal(Ps, Ps.T)                                   # exactly symmetric
    assert np.allclose(Ps, 0.5 * (A + A.T), rtol=0, atol=1e-15)
    # duplicate coordinates are summed (scipy keeps them in a coo_matrix)
    rows, cols, vals = np.array([0, 0, 2, 1]), np.array([1, 1, 2, 0]), np.array([1.0, 2.0, 5.0, 4.0])
    M = sp.coo_matrix((vals, (rows, cols)), shape=(3, 3))
    f2 = families.sparse_qcqp(P=M)
    P2 = dense(f2.P, (3, 3))
    assert P2[0, 1] == P2[1, 0] == 0.5 * (3.0 + 4.0) and P2[2, 2] == 5.0
    # a scipy matrix and its dense form give the same canonical lists
    f3 = families.sparse_qcqp(P=M.toarray())
    assert all(np.array_equal(a, b) for a, b in zip(f2.P, f3.P))
    # entries are sorted by (row, col), without explicit zeros
    key = fam.P[0] * n + fam.P[1]
    assert np.all(np.diff(key) > 0) and np.all(fam.P[2] != 0)


def test_shapes_inferred():
    sp = pytest.importorskip("scipy.sparse")
    n = 12
    fam = families.sparse_qcqp(P=sp.eye(n), Qc=[sp.eye(n), 2 * np.eye(n)], Ac=sp.random(2, n, density=0.3, random_state=1),
                               bc=[1.0, 2.0], Qd=[sp.eye(n)], bd=[0.5])
    assert (fam.n, fam.m, fam.p) == (n, 2, 1)
    assert fam.c is not None and fam.d is not None
    assert np.array_equal(np.unique(fam.Qc[0]), [0, 1])
    fam2 = families.sparse_qcqp(q=np.zeros(5), Ad=np.ones((3, 5)))
    assert (fam2.n, fam2.m, fam2.p) == (5, 0, 3) and fam2.c is None


@pytest.mark.parametrize("kw, msg", [
    (dict(P=np.ones((3, 4))), "square"),
    (dict(P=np.eye(3), q=np.ones(4)), "n = "),
    (dict(Qc=[np.eye(3), np.eye(4)]), "n = "),
    (dict(Qc=[np.eye(3)], bc=[1.0, 2.0]), "m = "),
    (dict(P=np.eye(3), Ac=np.ones((2, 4))), "n = "),
    (dict(P=np.eye(3), bc=[1.0]), "need Qc or Ac"),
    (dict(P=np.eye(3), bd=[1.0]), "need Qd or Ad"),
    (dict(Qc=[np.ones(3)]), "matrix"),
    (dict(r=1.0), "n is unknown"),
])
def test_bad_shapes_rejected(kw, msg):
    with pytest.raises(_lib.LFPSQPError, match=msg):
        families.sparse_qcqp(**kw)


def _random_problem(seed, n=9, m=2, p=3):
    rng = np.random.default_rng(seed)
    def spd_like():
        A = rng.standard_normal((n, n)) * (rng.random((n, n)) < 0.5)
        return A + A.T
    return families.sparse_qcqp(P=spd_like(), q=rng.standard_normal(n), r=0.25, Qc=[spd_like() for _ in range(m)],
                                Ac=rng.standard_normal((m, n)) * (rng.random((m, n)) < 0.6), bc=rng.standard_normal(m),
                                Qd=[spd_like() for _ in range(p)], Ad=rng.standard_normal((p, n)), bd=rng.standard_normal(p))


@pytest.mark.parametrize("sides", ["finite", "infinite", "mixed"])
def test_slack_embedding_matches_slack_callbacks(sides):
    fam = _random_problem(3)
    n, m, p = fam.n, fam.m, fam.p
    rng = np.random.default_rng(4)
    dl = {"finite": -np.ones(p), "infinite": -np.inf * np.ones(p), "mixed": np.array([-np.inf, -1.0, 0.2])}[sides]
    du = {"finite": np.ones(p), "infinite": np.zeros(p), "mixed": np.array([0.5, np.inf, 3.0])}[sides]
    x0 = rng.standard_normal(n)
    xl, xu = -2 * np.ones(n), np.full(n, np.inf)
    cb = fam.callbacks()
    f_aux, grad_aux, c_aux, jac_aux, hess_aux, x0a, xla, xua = host.slack_callbacks(
        cb["f"], cb["grad"], cb["hess_vec"], cb["c"], cb["jac"], cb["chess_vec"], cb["d"], cb["djac"], cb["dhess_vec"],
        dl, du, x0, xl, xu, m, p)
    aug, x0b, xlb, xub = fam.slack_embedding(x0, xl, xu, dl, du)
    assert (aug.n, aug.m, aug.p) == (n + p, m + p, 0)
    assert np.allclose(x0b, x0a, rtol=1e-14, atol=1e-14)
    assert np.array_equal(xlb, xla) and np.array_equal(xub, xua)
    ca = aug.callbacks()
    for _ in range(3):
        x = rng.standard_normal(n + p)
        v = rng.standard_normal(n + p)
        lam = rng.standard_normal(m + p)
        assert abs(ca["f"](x) - f_aux(x)) <= 1e-13 * max(1.0, abs(f_aux(x)))
        c1 = np.zeros(m + p); c_aux(c1, x)
        c2 = np.zeros(m + p); ca["c"](c2, x)
        assert np.allclose(c2, c1, rtol=1e-13, atol=1e-13)
        J1 = np.zeros((m + p, n + p), order="F"); cv1 = np.zeros(m + p); jac_aux(J1, cv1, x)
        J2 = np.zeros((m + p, n + p), order="F"); cv2 = np.zeros(m + p); ca["jac"](J2, cv2, x)
        assert np.allclose(J2, J1, rtol=1e-13, atol=1e-13) and np.allclose(cv2, cv1, rtol=1e-13, atol=1e-13)
        h1 = np.zeros(n + p); hess_aux(h1, v, x, lam)
        h2 = np.zeros(n + p); t = np.zeros(n + p)
        ca["hess_vec"](h2, v, x); ca["chess_vec"](t, v, x, lam); h2 += t
        assert np.allclose(h2, h1, rtol=1e-13, atol=1e-13)
        g1 = np.zeros(n + p); grad_aux(g1, x)
        g2 = np.zeros(n + p); ca["grad"](g2, x)
        assert np.allclose(g2, g1, rtol=1e-13, atol=1e-13)


def test_callbacks_match_dense_formulas():
    fam = _random_problem(5)
    n, m, p = fam.n, fam.m, fam.p
    P = dense(fam.P, (n, n)); Qc = dense(fam.Qc, (m, n, n)); Ac = dense(fam.Ac, (m, n))
    Qd = dense(fam.Qd, (p, n, n)); Ad = dense(fam.Ad, (p, n))
    x = np.random.default_rng(6).standard_normal(n)
    cb = fam.callbacks()
    assert np.isclose(cb["f"](x), 0.5 * x @ P @ x + fam.q @ x + 0.25, rtol=1e-13)
    c = np.zeros(m); cb["c"](c, x)
    assert np.allclose(c, 0.5 * np.einsum("i,kij,j->k", x, Qc, x) + Ac @ x - fam.bc, rtol=1e-13, atol=1e-13)
    J = np.zeros((m, n), order="F"); cb["jac"](J, c, x)
    assert np.allclose(J, np.einsum("kij,j->ki", Qc, x) + Ac, rtol=1e-13, atol=1e-13)
    assert np.allclose(fam.d_values(x), 0.5 * np.einsum("i,kij,j->k", x, Qd, x) + Ad @ x - fam.bd, rtol=1e-13, atol=1e-13)


def test_package_does_not_import_scipy():
    code = "import sys, lfpsqp.jl_b200; sys.exit(1 if any(k.split('.')[0] == 'scipy' for k in sys.modules) else 0)"
    assert subprocess.run([sys.executable, "-c", code], cwd=ROOT).returncode == 0


def test_ctypes_descriptor_matches_header(tmp_path):
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "lfpsqp_b200.h"\n'
                   'int main(void) { printf("%d %d %d %d %d %d %d %d", (int)sizeof(lfpsqp_coo), (int)sizeof(lfpsqp_sparse_qcqp),\n'
                   '  (int)offsetof(lfpsqp_sparse_qcqp, q), (int)offsetof(lfpsqp_sparse_qcqp, r), (int)offsetof(lfpsqp_sparse_qcqp, Qc),\n'
                   '  (int)offsetof(lfpsqp_sparse_qcqp, Ac), (int)offsetof(lfpsqp_sparse_qcqp, bc), LFPSQP_FAM_SPARSE_QCQP); return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    S = _lib.CSparseQcqp
    want = [ctypes.sizeof(_lib.CCoo), ctypes.sizeof(S), S.q.offset, S.r.offset, S.Qc.offset, S.Ac.offset, S.bc.offset,
            families.SPARSE_QCQP]
    assert got == want


def test_batched_entry_points_name_optimize_large():
    import lfpsqp.jl_b200 as L
    fam = families.sparse_qcqp(P=np.eye(4), Qc=[np.eye(4)], bc=[0.5])
    for call in (lambda: L.optimize(fam.f, fam.c, np.ones(4), 1), lambda: L.optimize_batched(fam.f, fam.c, np.ones((2, 4)), 1)):
        with pytest.raises(_lib.LFPSQPError, match="optimize_large"):
            call()
