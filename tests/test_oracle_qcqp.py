"""The dense QCQP family in the CPU reference (the oracle with the family added, tests/qcqp_reference.py): callbacks
against numpy, known answers of its solves, and the encodings of the README families, which must reproduce the
registered families bit for bit (every extra term is an exact zero or an exact power-of-two scaling)."""
import numpy as np
import pytest
from scipy.optimize import brentq

BUILDS = (None, "fma", "seq")


def sym(rng, n, spd=False):
    M = rng.standard_normal((n, n))
    M = 0.5 * (M + M.T)
    return M @ M.T / n + np.eye(n) if spd else M


@pytest.fixture(scope="session")
def R():
    from tests import qcqp_reference
    qcqp_reference.build()
    return qcqp_reference


def qcqp_solve(R, n, m, p, x0, params=None, xl=None, xu=None, **arrays):
    x0 = np.atleast_2d(x0)
    fp, stride = R.qcqp_params(n, m, p, B=x0.shape[0], **arrays)
    if p and xl is None:
        xl, xu = -np.inf * np.ones(n), np.inf * np.ones(n)
    return R.optimize_batched("qcqp", n, m, p, x0, xl=xl, xu=xu, fam_params=fp, fam_stride=stride, params=params)


def tight(R):
    return R.default_params(eps_kkt=1e-10, eps_f=0.0, eps_c=1e-12, maxiter=2000)


# ------------------------------------------------------------------ callbacks
@pytest.mark.parametrize("parts", ["all", "no_quadratic_constraints", "no_linear_terms", "objective_only"])
def test_callbacks_match_numpy(R, parts):
    rng = np.random.default_rng(11)
    n, m, p = 7, 2, 3
    a = dict(P=sym(rng, n), q=rng.standard_normal(n), r=rng.standard_normal(),
             Qc=np.stack([sym(rng, n) for _ in range(m)]), Ac=rng.standard_normal((m, n)), bc=rng.standard_normal(m),
             Qd=np.stack([sym(rng, n) for _ in range(p)]), Ad=rng.standard_normal((p, n)), bd=rng.standard_normal(p))
    if parts == "no_quadratic_constraints":
        a.pop("Qc"); a.pop("Qd")
    elif parts == "no_linear_terms":
        for k in ("q", "r", "Ac", "Ad"):
            a.pop(k)
    elif parts == "objective_only":
        m = p = 0
        a = dict(P=a["P"], q=a["q"])
    z = lambda k, shape: a.get(k, np.zeros(shape))
    P, q, r = z("P", (n, n)), z("q", n), z("r", ())
    Qc, Ac, bc = z("Qc", (m, n, n)), z("Ac", (m, n)), z("bc", m)
    Qd, Ad, bd = z("Qd", (p, n, n)), z("Ad", (p, n)), z("bd", p)
    fp, _ = R.qcqp_params(n, m, p, **a)
    x, v = rng.standard_normal(n), rng.standard_normal(n)
    lam = rng.standard_normal(m + p)

    assert R.family_f("qcqp", n, m, p, x, fp) == pytest.approx(0.5 * x @ P @ x + q @ x + r, rel=1e-13, abs=1e-13)
    np.testing.assert_allclose(R.family_grad("qcqp", n, m, p, x, fp), P @ x + q, rtol=1e-13, atol=1e-13)
    J, cval = R.family_jac("qcqp", n, m, p, x, fp)
    Jref = np.concatenate([Qc @ x + Ac, Qd @ x + Ad]) if m + p else np.zeros((0, n))
    cref = np.concatenate([0.5 * np.einsum("j,ijk,k->i", x, Qc, x) + Ac @ x - bc,
                           0.5 * np.einsum("j,ijk,k->i", x, Qd, x) + Ad @ x - bd])
    np.testing.assert_allclose(J, Jref, rtol=1e-13, atol=1e-13)
    np.testing.assert_allclose(cval, cref, rtol=1e-13, atol=1e-13)
    H = P + np.einsum("i,ijk->jk", lam[:m], Qc) + np.einsum("i,ijk->jk", lam[m:], Qd)
    np.testing.assert_allclose(R.family_hess("qcqp", n, m, p, x, lam, v, fp), H @ v, rtol=1e-12, atol=1e-12)


# ------------------------------------------------------------------ known answers
def test_rayleigh_quotient_on_the_sphere(R):
    rng = np.random.default_rng(12)
    n, B = 12, 6
    A = sym(rng, n)
    x0 = rng.standard_normal((B, n)); x0 /= np.linalg.norm(x0, axis=1, keepdims=True)
    x, obj, olen, lam, term, _ = qcqp_solve(R, n, 1, 0, x0, params=tight(R), P=A, Qc=2 * np.eye(n)[None],
                                            bc=[1.0])
    fstar = 0.5 * np.linalg.eigvalsh(A)[0]
    f = obj[np.arange(B), olen - 1]
    np.testing.assert_allclose(f, fstar, rtol=1e-10)
    np.testing.assert_allclose(np.linalg.norm(x, axis=1), 1.0, atol=1e-10)


def stiefel(n, k):
    """constraints x_a . x_b = delta_ab (a <= b) on X = [x_1 .. x_k] (n x k, column-major into x)"""
    Qc, bc = [], []
    for a in range(k):
        for b in range(a, k):
            Q = np.zeros((n * k, n * k))
            if a == b:
                Q[a * n:(a + 1) * n, a * n:(a + 1) * n] = 2 * np.eye(n)
            else:
                Q[a * n:(a + 1) * n, b * n:(b + 1) * n] = np.eye(n)
                Q[b * n:(b + 1) * n, a * n:(a + 1) * n] = np.eye(n)
            Qc.append(Q); bc.append(1.0 if a == b else 0.0)
    return np.stack(Qc), np.array(bc)


def test_stiefel_trace_minimisation(R):
    rng = np.random.default_rng(13)
    n, k, B = 8, 3, 4
    A = sym(rng, n)
    Qc, bc = stiefel(n, k)
    x0 = np.stack([np.linalg.qr(rng.standard_normal((n, k)))[0].T.ravel() for _ in range(B)])
    x, obj, olen, lam, term, _ = qcqp_solve(R, n * k, len(bc), 0, x0, params=tight(R),
                                            P=np.kron(np.eye(k), A), Qc=Qc, bc=bc)
    fstar = 0.5 * np.linalg.eigvalsh(A)[:k].sum()
    np.testing.assert_allclose(obj[np.arange(B), olen - 1], fstar, rtol=1e-10)
    for xi in x:
        X = xi.reshape(k, n).T
        np.testing.assert_allclose(X.T @ X, np.eye(k), atol=1e-10)


def test_equality_constrained_convex_qp(R):
    rng = np.random.default_rng(14)
    n, m, B = 10, 3, 4
    P = sym(rng, n, spd=True); q = rng.standard_normal(n)
    Ac = rng.standard_normal((m, n)); bc = rng.standard_normal(m)
    K = np.block([[P, Ac.T], [Ac, np.zeros((m, m))]])
    xstar = np.linalg.solve(K, np.concatenate([-q, bc]))[:n]
    x, obj, olen, lam, term, _ = qcqp_solve(R, n, m, 0, rng.standard_normal((B, n)), params=tight(R),
                                            P=P, q=q, Ac=Ac, bc=bc)
    np.testing.assert_allclose(x, np.broadcast_to(xstar, x.shape), rtol=0, atol=1e-8 * np.linalg.norm(xstar))


def trust_region_answer(P, q, delta):
    x = -np.linalg.solve(P, q)
    if np.linalg.norm(x) <= delta:
        return x
    n = len(q)
    phi = lambda mu: np.linalg.norm(np.linalg.solve(P + mu * np.eye(n), q)) - delta   # secular equation
    hi = 1.0
    while phi(hi) > 0:
        hi *= 2
    mu = brentq(phi, 0.0, hi, xtol=1e-15, rtol=1e-15)
    return -np.linalg.solve(P + mu * np.eye(n), q)


@pytest.mark.parametrize("case", ["interior", "boundary"])
def test_convex_trust_region_subproblem(R, case):
    rng = np.random.default_rng(15)
    n, B = 8, 4
    P = sym(rng, n, spd=True); q = rng.standard_normal(n)
    unc = np.linalg.norm(np.linalg.solve(P, q))
    delta = 2.0 * unc if case == "interior" else 0.5 * unc
    xstar = trust_region_answer(P, q, delta)
    x0 = 0.1 * delta * rng.standard_normal((B, n)) / np.sqrt(n)
    x, obj, olen, lam, term, _ = qcqp_solve(R, n, 0, 1, x0, params=tight(R), P=P, q=q,
                                            Qd=np.eye(n)[None], bd=[0.5 * delta ** 2])
    np.testing.assert_allclose(x, np.broadcast_to(xstar, x.shape), rtol=0, atol=1e-7 * np.linalg.norm(xstar))


# ------------------------------------------------------------------ encodings of the registered families
def assert_same_result(a, b):
    x, obj, olen, lam, term, _ = a
    x2, obj2, olen2, lam2, term2, _ = b
    assert np.array_equal(olen, olen2)
    assert np.array_equal(term, term2)
    assert np.array_equal(x, x2)
    assert np.array_equal(lam, lam2)
    assert np.array_equal(obj, obj2, equal_nan=True)


@pytest.mark.parametrize("build", BUILDS)
def test_readme_equality_encoding_is_bitwise(R, build):
    rng = np.random.default_rng(16)
    n, B = 10, 6
    x0 = rng.standard_normal((B, n))
    ref = R.optimize_batched("readme_eq", n, 1, 0, x0, H=128, build=build)
    fp, stride = R.qcqp_params(n, 1, 0, B=B, P=2 * np.eye(n), Ac=np.eye(n)[:1], bc=[0.75])
    enc = R.optimize_batched("qcqp", n, 1, 0, x0, fam_params=fp, fam_stride=stride, H=128, build=build)
    assert (ref[4]["iter"] >= 1).all()
    assert_same_result(enc, ref)


# Not the FMA build: there the compiler contracts the registered family's inlined dot(x, x) differently from the same
# dot over a copy of x, so the two differ by an ulp in that build alone.
@pytest.mark.parametrize("build", [None, "seq"])
def test_readme_inequality_encoding_is_bitwise(R, build):
    rng = np.random.default_rng(17)
    n, B = 10, 6
    co = rng.standard_normal((B, n))
    x0 = 0.1 * rng.standard_normal((B, n))
    inf = np.inf * np.ones(n)
    kw = dict(xl=-inf, xu=inf, H=128, build=build)
    fp, stride = R.qcqp_params(n, 0, 1, B=B, q=co, Qd=2 * np.eye(n)[None], bd=[1.0])
    ref = R.optimize_batched("readme_ineq", n, 0, 1, x0, fam_params=co, fam_stride=n, **kw)
    enc = R.optimize_batched("qcqp", n, 0, 1, x0, fam_params=fp, fam_stride=stride, **kw)
    assert (ref[4]["iter"] >= 1).all()
    assert_same_result(enc, ref)
