"""CPU-only checks of the host side of the generic path (lfpsqp.jl_b200/host.py): the lfpsqp_host_callbacks layout, the
slack wrapper of src/optimize.jl:13-71 with explicit derivatives (checked against the oracle's family callbacks and by
finite differences), method dispatch, and the loud failure without a GPU (no CPU fallback)."""
import ctypes
import multiprocessing as mp

import numpy as np
import pytest


def test_host_callbacks_struct_layout():
    from lfpsqp.jl_b200 import host
    # include/lfpsqp_b200.h: void *user + 7 function pointers
    assert ctypes.sizeof(host.HostCallbacks) == 64
    assert [n for n, _ in host.HostCallbacks._fields_] == ["user", "f", "grad", "c", "jac", "hess_lag_vec", "callback", "randn"]


def _readme_ineq(coeff):
    def f(x): return float(coeff @ x)
    def grad(g, x): g[:] = coeff
    def hv(dest, src, x): dest[:] = 0.0
    def d(dv, x): dv[0] = x @ x - 1.0
    def djac(Jd, dv, x): Jd[0, :] = 2.0 * x; d(dv, x)
    def dhv(dest, src, x, lam): dest[:] = 2.0 * lam[0] * src
    return f, grad, hv, d, djac, dhv


def test_slack_wrapper_matches_oracle_family(oracle):
    # README.md:57-76 through the slack wrapper: augmented callbacks == the oracle's readme_ineq family + the slack columns
    from lfpsqp.jl_b200 import host
    n, p = 50, 1
    rng = np.random.default_rng(0)
    coeff = rng.standard_normal(n)
    f, grad, hv, d, djac, dhv = _readme_ineq(coeff)
    x0 = rng.standard_normal(n)
    fa, ga, ca, ja, ha, x0a, xla, xua = host.slack_callbacks(f, grad, hv, None, None, None, d, djac, dhv, [-np.inf], [0.0], x0,
                                                             None, None, 0, p)
    assert x0a.shape == (n + p,) and x0a[n] == pytest.approx(x0 @ x0 - 1.0)                 # s0 = d(x0), optimize.jl:26-28
    assert np.all(np.isneginf(xla)) and np.all(np.isposinf(xua[:n])) and xua[n] == 0.0     # [xl; dl], [xu; du]
    xa = np.concatenate([rng.standard_normal(n), [0.3]])
    assert fa(xa) == pytest.approx(oracle.family_f("readme_ineq", n, 0, p, xa[:n], fam_params=coeff))
    g = np.zeros(n + p); ga(g, xa)
    assert np.allclose(g[:n], oracle.family_grad("readme_ineq", n, 0, p, xa[:n], fam_params=coeff)) and g[n] == 0.0
    Jo, co = oracle.family_jac("readme_ineq", n, 0, p, xa[:n], fam_params=coeff)
    Jc = np.zeros((p, n + p), order="F"); cv = np.zeros(p); ja(Jc, cv, xa)
    assert np.allclose(Jc[:, :n], Jo) and Jc[0, n] == -1.0 and cv[0] == pytest.approx(co[0] - xa[n])   # d(x) - s
    cv2 = np.zeros(p); ca(cv2, xa)
    assert cv2[0] == cv[0]
    lam = np.array([0.7]); v = rng.standard_normal(n + p)
    out = np.zeros(n + p); ha(out, v, xa, lam)
    assert np.allclose(out[:n], oracle.family_hess("readme_ineq", n, 0, p, xa[:n], lam, v[:n], fam_params=coeff)) and out[n] == 0.0


def test_slack_wrapper_finite_differences():
    # m = 2 equalities + p = 2 inequalities with curvature: Jacobian and Lagrangian-Hessian action of the augmented problem
    from lfpsqp.jl_b200 import host
    n, m, p = 6, 2, 2
    rng = np.random.default_rng(1)
    Bm = rng.standard_normal((m, n)); Dm = rng.standard_normal((p, n)); t = rng.standard_normal(n)
    def f(x): return float(np.sum((x - t) ** 4))
    def grad(g, x): g[:] = 4 * (x - t) ** 3
    def hv(dest, src, x): dest[:] = 12 * (x - t) ** 2 * src
    def c(cv, x): cv[:] = Bm @ np.sin(x)
    def jac(Jc, cv, x): Jc[:, :] = Bm * np.cos(x)[None, :]; c(cv, x)
    def chv(dest, src, x, lam): dest[:] = -(lam @ Bm) * np.sin(x) * src
    def d(dv, x): dv[:] = Dm @ (x * x) - 1.0
    def djac(Jd, dv, x): Jd[:, :] = 2 * Dm * x[None, :]; d(dv, x)
    def dhv(dest, src, x, lam): dest[:] = 2 * (lam @ Dm) * src
    fa, ga, ca, ja, ha, x0a, xla, xua = host.slack_callbacks(f, grad, hv, c, jac, chv, d, djac, dhv, -np.ones(p), np.zeros(p),
                                                             rng.standard_normal(n), -2 * np.ones(n), 2 * np.ones(n), m, p)
    assert np.array_equal(xla, np.concatenate([-2 * np.ones(n), -np.ones(p)])) and np.array_equal(xua[n:], np.zeros(p))
    xa = rng.standard_normal(n + p); lam = rng.standard_normal(m + p); v = rng.standard_normal(n + p)
    Jc = np.zeros((m + p, n + p), order="F"); cv = np.zeros(m + p); ja(Jc, cv, xa)
    eps = 1e-6
    Jfd = np.zeros_like(Jc)
    for j in range(n + p):
        e = np.zeros(n + p); e[j] = eps
        cp = np.zeros(m + p); cm = np.zeros(m + p); ca(cp, xa + e); ca(cm, xa - e)
        Jfd[:, j] = (cp - cm) / (2 * eps)
    assert np.allclose(Jc, Jfd, atol=1e-7)
    def lag_grad(x):
        g = np.zeros(n + p); ga(g, x)
        J2 = np.zeros((m + p, n + p), order="F"); c2 = np.zeros(m + p); ja(J2, c2, x)
        return g + J2.T @ lam
    hfd = (lag_grad(xa + eps * v) - lag_grad(xa - eps * v)) / (2 * eps)
    out = np.zeros(n + p); ha(out, v, xa, lam)
    assert np.allclose(out, hfd, atol=1e-5 * max(1.0, np.abs(hfd).max()))


def _explicit_core_dispatch_and_no_cpu_fallback():
    import lfpsqp.jl_b200 as L
    f = lambda x: float(x @ x)
    def grad(g, x): g[:] = 2 * x
    def hlv(dest, src, x, lam): dest[:] = 2 * src
    # 9 positional arguments with a plain callable first = optimize(f, grad!, c!, jac!, hess_lag_vec!, x0, xl, xu, m) (optimize.jl:119)
    with pytest.raises(L.LFPSQPError, match="no CPU fallback"):
        L.optimize(f, grad, None, None, hlv, np.ones(3), None, None, 0)
    with pytest.raises(L.LFPSQPError, match="same length"):                               # optimize.jl:144-148 (checked before any device work)
        L.optimize(f, grad, None, None, hlv, np.ones(3), np.zeros(2), np.ones(2), 0)
    with pytest.raises(L.LFPSQPError, match="required when m > 0"):
        L.optimize(f, grad, None, None, hlv, np.ones(3), None, None, 1)
    with pytest.raises(TypeError):                                                        # device-family path still demands a family handle
        L.optimize(f, np.ones(3))


def test_explicit_core_dispatch_and_no_cpu_fallback(monkeypatch):
    # in a child process that sees no GPU, so that the check runs on a GPU machine as well
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    p = mp.get_context("spawn").Process(target=_explicit_core_dispatch_and_no_cpu_fallback)
    p.start()
    p.join(300)
    assert p.exitcode == 0
