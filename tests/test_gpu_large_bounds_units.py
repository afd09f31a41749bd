"""Large-n mode with finite bounds (the 2n embedding of src/inequality_helper.jl): the bound-embedding kernels one at a time,
through the unit-level entry points (factor, project, projcg, pcg, retract) on a bounded problem, each against a plain
reference of the same operation.  Every GPU case asserts through Context.large_dispatch that the path it targets ran.

References:
  weighted Gram   two-sided bounds with integer xl, xu and xu - xl even, each coordinate at its box midpoint (Dx = 0,
                  Dy = +-1 exactly) or at an active bound (Dy = 0 exactly), and integer J: G_w = J diag(Dy^2) J' must equal
                  numpy's J_S J_S' exactly, J_S = the midpoint columns (ineq_scale_cols_kernel + SYRK, spj_gram_kernel<true>)
  projection      C = [[J, 0], [diag(dx), diag(dy)]] in np.longdouble, (dx, dy) the unnormalised gradient of h: tangency
                  r1 = C pv and r2 = v - pv - C'[lambda ; lambda_y], componentwise against rounding bounds
                  (ineq_proj_pre_kernel, ineq_proj_tail, the lambda_y line of project())
  projcg! / pcg!  float64 transcriptions on the working Hessian / on B'B + mu I, B = [[diag(dx), diag(dy)], [J, 0]]
                  (ineq_cg_init / ineq_cg_update2, the bound terms of the DIAGQUAD Hessian, ineq_hess_aug_kernel,
                  ineq_pcg_z_kernel)
  retractions     float64 transcriptions of retract_nr / retract_pp as large.cu implements them (ineq_pp_rhs_kernel,
                  the bounded branches of both)
Host callbacks (LFPSQP_FAM_HOST) are not covered here: LargeProblem binds device families only.  The unmarked tests at
the end feed each checker corrupted copies of reference results and require every corruption to be rejected."""
import numpy as np
import pytest

from tests.test_gpu_large_boundaries import (C_BOUND, CG_TOL, SOLVE_PINV, SOLVE_TRIANGULAR, SYRK_SKIP, L, S, cg_tolerance, dim,
                                             disp, factor_ratios, gamma, pinv_reference, rel, worst)
from tests.test_gpu_large_bounds import bounds_for

SYRK_NARROW, SPARSE_GRAM = 4, 256
T = np.longdouble


@pytest.fixture(scope="module")
def O(oracle):
    return oracle


# ------------------------------------------------------------------ references
def grad_h(O, xl, xu, xaug):
    """(Dx, Dy, S) of the oracle and the unnormalised gradient (dx, dy) of h (inequality_helper.jl:125-141)"""
    Dx, Dy, Sv = O.ineq_gradient(xl, xu, xaug)
    q, r, s, t, _, _ = O.ineq_data(xl, xu)
    n = q.size
    dx = 2.0 * q * (xaug[:n] - r) + (q == 0.0)
    dy = 2.0 * s * (xaug[n:] - r) - (s == 0.0)
    return Dx, Dy, Sv, dx, dy


def closed_projection(J, Dx, Dy, Sv, v, Gsolve=None):
    """the device's closed form in float64: pv, lambda, lambda_y (large_ineq.cuh header)"""
    n = Dx.size
    vx, vy = v[:n], v[n:]
    Jw = J * Dy[None, :]
    t = J @ (Dy * (Dy * vx - Dx * vy))
    lam = (Gsolve or (lambda r: np.linalg.solve(Jw @ Jw.T, r)))(t) if J.shape[0] else np.zeros(0)
    w = J.T @ lam if J.shape[0] else np.zeros(n)
    a = Dx * vx + Dy * vy
    pv = np.concatenate([vx - (Dx * a + Dy * Dy * w), vy - (Dy * a - Dx * Dy * w)])
    lamy = -(Dx / Sv) * w + a / Sv
    return pv, lam, lamy


def embedded_projection_ratios(J, dx, dy, v, pv, lam, lamy):
    """r1 = C pv and r2 = v - pv - C'[lambda ; lambda_y] over rounding bounds, C = [[J, 0], [diag(dx), diag(dy)]].
    The closed form differs from the exact projector by the rounding of the Gram solve (as projection_ratios) and of the
    elementwise terms a = Dx v_x + Dy v_y, Dx a + Dy^2 w, Dy a - Dx Dy w, lambda_y = (a - Dx w) / S."""
    m, n = J.shape
    Jt, dxt, dyt, vt, pt, lt, lyt = (np.asarray(a).astype(T) for a in (J, dx, dy, v, pv, lam, lamy))
    St = np.sqrt(dxt * dxt + dyt * dyt)
    Dx, Dy = dxt / St, dyt / St
    vx, vy, px, py = vt[:n], vt[n:], pt[:n], pt[n:]
    aJ = np.abs(Jt)
    w = aJ.T @ np.abs(lt) if m else np.zeros(n, dtype=T)
    aa = np.abs(Dx * vx) + np.abs(Dy * vy)                       # |a| before cancellation
    ex = np.abs(vx) + np.abs(px) + np.abs(Dx) * aa + Dy * Dy * w   # magnitudes entering the x-half
    ey = np.abs(vy) + np.abs(py) + np.abs(Dy) * aa + np.abs(Dx * Dy) * w
    c = C_BOUND
    g = gamma(max(m, n) + 16)
    r1x = Jt @ px if m else np.zeros(0, dtype=T)
    b1x = c * g * (aJ @ ex) if m else np.zeros(0, dtype=T)
    r1y = dxt * px + dyt * py
    b1y = c * gamma(16) * (np.abs(dxt) * ex + np.abs(dyt) * ey)
    r2x = vx - px - ((Jt.T @ lt) if m else 0) - dxt * lyt
    r2y = vy - py - dyt * lyt
    gm = gamma(m + 16)
    lyb = (aa + np.abs(Dx) * w) / St                               # |lambda_y| before cancellation
    b2x = c * gm * (w + np.abs(dxt) * lyb + ex)
    b2y = c * gamma(16) * (np.abs(dyt) * lyb + ey)
    r1 = max(worst(r1x, b1x), worst(r1y, b1y))
    r2 = max(worst(r2x, b2x), worst(r2y, b2y))
    return r1, r2


def weighted_gram(J, Dy):
    Jw = J * Dy[None, :]
    return Jw @ Jw.T


def ref_projcg_op(hop, b, proj, K):
    """projcg! (projcg.jl:40-121) with c = 0, tol = 0, K iterations on the operator hop"""
    xs = np.zeros_like(b); r = proj(-b); d = -r; rg = r @ r
    for _ in range(K):
        Ad = hop(d); al = rg / (d @ Ad); xs = xs + al * d; rp = r + al * Ad; gp = proj(rp)
        be = (rp @ gp) / rg; d = be * d - gp; r = gp; rg = gp @ gp
    return xs


def ref_pcg_tol(op, b, tol, lim):
    """pcg! (retractions.jl:179-246) from x = 0 as large.cu's kernels stop it -> (x, iterations)"""
    x = np.zeros_like(b); r = b.copy(); p = np.zeros_like(b); rho_prev = 1.0; it = 0; first = True
    while True:
        rho = r @ r
        nr = np.inf if first else np.sqrt(rho)
        if not nr > tol or it >= lim:
            return x, it
        p = r + (rho / rho_prev) * p
        z = op(p); al = rho / (p @ z); x = x + al * p; r = r - al * z
        rho_prev = rho; it += 1; first = False


def ld_solver(Gw):
    """G_w^-1 t in np.longdouble: a float64 Cholesky solve and two steps of refinement with the residual in np.longdouble"""
    from scipy.linalg import cho_factor, cho_solve
    cf = cho_factor(Gw)
    Gl = Gw.astype(T)

    def solve(t):
        lam = cho_solve(cf, np.asarray(t, dtype=np.float64)).astype(T)
        for _ in range(2):
            lam = lam + cho_solve(cf, np.asarray(t - Gl @ lam, dtype=np.float64)).astype(T)
        return lam
    return solve


def cg_bar(ref, ref_ld):
    """cg_tolerance with the spread between the float64 reference and the same iteration in np.longdouble: how far
    float64 rounding alone moves the K-step iterate of this problem"""
    return cg_tolerance(rel(ref, np.asarray(ref_ld, dtype=np.float64)))


def bigA_ops(J, Dx, Dy, Sv):
    """(B, B') of the embedding: B' p = [S (Dx p_x + Dy p_y) ; J p_x], B [wh ; wc] = [J' wc + Dx S wh ; Dy S wh]"""
    n = Dx.size
    Bt = lambda p: np.concatenate([Sv * (Dx * p[:n] + Dy * p[n:]), J @ p[:n]])
    B = lambda u: np.concatenate([J.T @ u[n:] + Dx * Sv * u[:n], Dy * Sv * u[:n]])
    return B, Bt


# ------------------------------------------------------------------ problem builders
def exact_point(n, seed, active=0.4, runs=()):
    """bounds and a point at which Dy is exactly 0 or +-1: (xl, xu, x, y, mid).  Two-sided boxes [c - k, c + k] with
    integer c and k (r = c, rho = k): the midpoint with y = c +- k (Dx = 0, Dy = +-1), or x at a bound (y = c, Dy = 0);
    active one-sided bounds (x = xl or x = xu, y = r: Dy = 0).  runs: column ranges forced active."""
    rng = np.random.default_rng(seed)
    c = rng.integers(-2, 3, n).astype(np.float64); k = rng.integers(1, 3, n).astype(np.float64)
    kind = rng.choice(4, n, p=[1.0 - active, active / 2, active / 4, active / 4])   # 0 mid, 1 box bound, 2 lower, 3 upper
    for a, b in runs:
        kind[a:b] = 1
    xl, xu, x, y = c - k, c + k, c.copy(), c.copy()
    sgn = rng.choice([-1.0, 1.0], n)
    mid = kind == 0
    y[mid] = c[mid] + sgn[mid] * k[mid]
    box = kind == 1
    x[box] = c[box] + sgn[box] * k[box]
    lo, up = kind == 2, kind == 3
    xl[lo], xu[lo] = c[lo], np.inf
    xl[up], xu[up] = -np.inf, c[up]
    return xl, xu, x, y, mid


def int_diagquad_at(Lm, x, m, seed, mask=None, qzero=None):
    rng = np.random.default_rng(seed)
    n = x.size
    Q = rng.integers(-8, 9, (m, n)).astype(np.float64)
    A = rng.integers(-8, 9, (m, n)).astype(np.float64)
    if mask is not None:
        Q *= mask; A *= mask
    if qzero is not None:
        Q[:, qzero] = 0.0
    b = 0.5 * Q @ (x * x) + A @ x
    return Lm.families.diagquad(Q, A, b, np.zeros(n), np.ones(n)), Q * x[None, :] + A


def int_sparse_at(x, m, seed, jacobian="csr", long_row=False):
    import scipy.sparse as sp
    from lfpsqp.jl_b200 import families
    rng = np.random.default_rng(seed)
    n = x.size
    A = sp.random(m, n, density=min(1.0, 40.0 / n + 0.01), random_state=seed,
                  data_rvs=lambda k: rng.integers(1, 4, k).astype(float)).tolil()
    if long_row:
        A[m // 2, :] = rng.integers(1, 4, n).astype(float)[None]
    Ac = sp.csr_matrix(A)
    Qc = [sp.diags(rng.integers(-2, 3, n).astype(float) * (rng.random(n) < 0.01)) for _ in range(m)]
    fam = families.sparse_qcqp(q=np.zeros(n), Qc=Qc, Ac=Ac, jacobian=jacobian)
    return fam, jac_of(fam, x)


def jac_of(fam, x):
    Jc = np.zeros((fam.m, fam.n), order="F"); cv = np.zeros(fam.m)
    fam.callbacks()["jac"](Jc, cv, x)
    return np.ascontiguousarray(Jc)


def gram_ok(G, J, mid):
    want = J[:, mid] @ J[:, mid].T
    assert np.max(np.abs(want)) < 2.0 ** 53
    return np.array_equal(np.tril(G), np.tril(want))


# ------------------------------------------------------------------ a. exact weighted Gram
GRAM_MS = [1, 63, 64, 65, 129, "split"]


def split_m(S):
    return dim((2, 1), S)


@pytest.mark.gpu
@pytest.mark.parametrize("mspec", GRAM_MS)
@pytest.mark.parametrize("jac", ["dense", "csr"])
def test_weighted_gram_is_exact(L, S, O, mspec, jac):
    m = split_m(S) if mspec == "split" else mspec
    n = 8192 if mspec == "split" else (2048 if jac == "dense" else 1001)
    xl, xu, x, y, mid = exact_point(n, seed=m + n)
    if jac == "dense":
        fam, J = int_diagquad_at(L, x, m, seed=m)
    else:
        fam, J = int_sparse_at(x, m, seed=m)
    P = L.LargeProblem(fam)
    P.set_bounds(xl, xu)
    Dx, Dy, Sv, _, _ = grad_h(O, xl, xu, np.concatenate([x, y]))
    assert np.array_equal(Dy * Dy, mid.astype(np.float64)) and np.all(np.abs(O.ineq_h(xl, xu, np.concatenate([x, y]))) == 0)
    fac = P.factor(np.concatenate([x, y]))
    d = disp(L)
    assert d["fused_single"] == d["fused_general"] == d["fused_pcg"] == 0, d
    if jac == "csr":
        assert d["gemm"] & SPARSE_GRAM and not d["gemm"] & 15, d
    else:
        assert d["gemm"] & (SYRK_NARROW if m <= 64 else SYRK_SKIP), d
    assert gram_ok(fac["G"], J, mid), (m, n, jac)
    assert fac["rank_deficient"] == 0
    if m <= 512:
        r1, r2 = factor_ratios(J[:, mid] @ J[:, mid].T, fac["L"], fac["Linv"])
        assert r1 <= 1 and r2 <= 1, (r1, r2)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["long_row", "odd_dense", "zero_slabs"])
def test_weighted_gram_is_exact_at_the_edges(L, S, O, case):
    # long_row: a CSR row of more than 4096 entries (the chunked sparse Gram with weights); odd_dense: an odd column count
    # with the Jacobian stored dense (ineq_scale_cols' 8-byte tail, a y-half 8 bytes off 16-byte alignment); zero_slabs:
    # 64 consecutive active columns over all rows give J diag(Dy) all-zero (64 x 16) slabs that J does not have
    if case == "long_row":
        n, m = (1 << 16) + 1, 5
        xl, xu, x, y, mid = exact_point(n, seed=1)
        fam, J = int_sparse_at(x, m, seed=1, long_row=True)
        assert np.count_nonzero(J[m // 2]) > 4096
    elif case == "odd_dense":
        n, m = 1001, 65
        xl, xu, x, y, mid = exact_point(n, seed=2)
        fam, J = int_sparse_at(x, m, seed=2, jacobian="dense")
    else:
        n, m = 4096, 129
        xl, xu, x, y, mid = exact_point(n, seed=3, active=0.2, runs=[(1024, 1088), (2048, 2112), (3000, 3040)])
        fam, J = int_diagquad_at(L, x, m, seed=3)
        assert all(np.any(J[r:r + 64, c:c + 16]) for r in (0, 64) for c in range(1024, 1088, 16))   # J has no zero slab there
    P = L.LargeProblem(fam)
    P.set_bounds(xl, xu)
    fac = P.factor(np.concatenate([x, y]))
    d = disp(L)
    if case == "long_row":
        assert d["gemm"] & SPARSE_GRAM, d
    else:
        assert d["gemm"] & (SYRK_SKIP if m > 64 else SYRK_NARROW), d
    assert gram_ok(fac["G"], J, mid), case
    assert fac["rank_deficient"] == 0


# ------------------------------------------------------------------ b. structure changes through the bounds alone
def coupled_problem(L, zero_row=False):
    """m = 128: rows 0-63 on columns [0, 1024), rows 64-127 on [1024, 2048), and 8 coupling columns used by every row.
    Q is zero on the coupling columns, so J does not depend on where x sits there.  Point a: the coupling columns at an
    active bound (G_w block diagonal); point b: the same columns at their midpoint (G_w couples the two blocks)."""
    m, n = 128, 2048
    xl, xu, x, y, mid = exact_point(n, seed=11, active=0.3)
    cpl = np.arange(2040, 2048)
    mask = np.zeros((m, n)); mask[:64, :1024] = 1; mask[64:, 1024:2040] = 1; mask[:, cpl] = 1
    if zero_row:   # row 5 lives on coupling columns only: at point a its row of J diag(Dy) is zero
        mask[5, :] = 0; mask[5, cpl] = 1
    c = np.array([-2.0, -1.0, 0.0, 1.0, 2.0, 0.0, 1.0, -1.0])   # two-sided boxes [c - 1, c + 1] on the coupling columns
    xl[cpl], xu[cpl] = c - 1, c + 1
    x[cpl] = c + 1
    fam, J = int_diagquad_at(L, x, m, seed=12, mask=mask, qzero=cpl)
    pts = {}
    for key in ("a", "b"):
        xx, yy, mm = x.copy(), y.copy(), mid.copy()
        if key == "a":
            xx[cpl], yy[cpl], mm[cpl] = c + 1, c, False
        else:
            xx[cpl], yy[cpl], mm[cpl] = c, c + 1, True
        pts[key] = (np.concatenate([xx, yy]), mm)
    return fam, J, xl, xu, pts


@pytest.mark.gpu
def test_block_diagonal_chain_skip_tracks_bound_changes(L, O, monkeypatch):
    fam, J, xl, xu, pts = coupled_problem(L)
    for key, (xa, mm) in pts.items():
        assert np.array_equal(jac_of_diagquad(fam, xa[:J.shape[1]]), J), key   # J is the same at both points
    Ga = J[:, pts["a"][1]] @ J[:, pts["a"][1]].T
    assert not np.any(Ga[64:, :64]) and np.any((J[:, pts["b"][1]] @ J[:, pts["b"][1]].T)[64:, :64])
    # the references first: a context holds one large-n problem, so P (structure caches on) must be the last one set up
    fresh = {}
    monkeypatch.setenv("LFPSQP_GRAM_SKIP", "0")
    for key in ("a", "b"):
        Pf = L.LargeProblem(fam); Pf.set_bounds(xl, xu)
        fresh[key] = Pf.factor(pts[key][0])
        assert not disp(L)["gemm"] & SYRK_SKIP
    monkeypatch.delenv("LFPSQP_GRAM_SKIP", raising=False)
    P = L.LargeProblem(fam)
    P.set_bounds(xl, xu)
    for call, key in enumerate("aaabbaab"):
        fac = P.factor(pts[key][0])
        if call == 0:   # the structure caches are live: the first Gram scans J diag(Dy) for zero slabs
            assert disp(L)["gemm"] & SYRK_SKIP, disp(L)
        assert fac["rank_deficient"] == 0
        assert gram_ok(fac["G"], J, pts[key][1]), (call, key)
        for k in ("G", "L", "Linv"):
            assert np.array_equal(np.tril(fac[k]), np.tril(fresh[key][k])), (call, key, k)


def jac_of_diagquad(fam, x):
    m, n = fam.m, fam.n
    p = np.asarray(fam.params).ravel()
    Q, A = p[:m * n].reshape(m, n), p[m * n:2 * m * n].reshape(m, n)
    return Q * x[None, :] + A


@pytest.mark.gpu
def test_bounds_that_zero_a_constraint_row_take_the_pseudo_inverse(L, O):
    fam, J, xl, xu, pts = coupled_problem(L, zero_row=True)
    xa, mm = pts["a"]
    n = J.shape[1]
    P = L.LargeProblem(fam)
    P.set_bounds(xl, xu)
    fac = P.factor(xa)
    assert fac["rank_deficient"] == 1
    assert gram_ok(fac["G"], J, mm)
    Dx, Dy, Sv, dx, dy = grad_h(O, xl, xu, xa)
    Jw = J * Dy[None, :]
    Gp, defect = pinv_reference(Jw)
    assert defect == 1
    v = np.random.default_rng(4).standard_normal(2 * n)
    pv, lam = P.project(v)
    d = disp(L)
    assert d["solve"] & SOLVE_PINV and d["fused_single"] == d["fused_general"] == 0, d
    lam_x, lamy = lam[:fam.m], lam[fam.m:]
    rpv, rlam, rlamy = closed_projection(J, Dx, Dy, Sv, v, Gsolve=lambda t: Gp @ t)
    assert rel(lam_x, rlam) < 1e-8 and rel(pv, rpv) < 1e-10 and rel(lamy, rlamy) < 1e-8
    assert lam_x[5] == 0.0
    r1, r2 = embedded_projection_ratios(J, dx, dy, v, pv, lam_x, lamy)
    print("pinv projection: r1 %.2e r2 %.2e of the bound" % (r1, r2))
    assert r1 <= 1 and r2 <= 1, (r1, r2)


@pytest.mark.gpu
def test_working_length_follows_the_library(L):
    # the embedding is on unless every xl is -Inf and every xu +Inf (optimize.jl:151): a NaN entry switches it on although
    # no entry is finite, and the wrappers size and check their vectors by the library's decision
    n, m = 64, 4
    Q, A, b, xt, w, x0 = L.make_diagquad(n, m, seed=5, cond=50.0)
    P = L.LargeProblem(L.families.diagquad(Q, A, b, xt, w))
    assert P.nv == n
    xl, xu = -np.inf * np.ones(n), np.inf * np.ones(n)
    P.set_bounds(xl, xu)
    assert P.nv == n
    xl[3] = np.nan
    P.set_bounds(xl, xu)
    assert P.nv == 2 * n
    with pytest.raises(L.LFPSQPError, match="working length"):
        P.project(np.ones(n))
    P.set_bounds(None, None)
    assert P.nv == n


# ------------------------------------------------------------------ c. projection and multipliers
def general_point(L, O, n, m, seed, kind="mixed", active=0.25, jac="diagquad"):
    """a DIAGQUAD (or CSR sparse QCQP) problem at a feasible embedded point with all four bound classes and some bounds
    active -> (fam, J, xl, xu, xaug)"""
    rng = np.random.default_rng(seed)
    if jac == "diagquad":
        Q, A, b, xt, w, x0 = L.make_diagquad(n, m, seed=seed, cond=50.0)
    else:
        x0 = rng.standard_normal(n)
    xl, xu = bounds_for(x0, seed + 10, kind)
    act = rng.random(n) < active
    lo = act & np.isfinite(xl) & (rng.random(n) < 0.5)
    up = act & np.isfinite(xu) & ~lo
    x0 = np.where(lo, xl, np.where(up, xu, x0))
    if jac == "diagquad":
        b = 0.5 * Q @ (x0 * x0) + A @ x0
        fam = L.families.diagquad(Q, A, b, xt, w)
        J = Q * x0[None, :] + A
    else:
        import scipy.sparse as sp
        from lfpsqp.jl_b200 import families
        Pm = sp.diags(np.exp(rng.uniform(0, np.log(50.0), n)))
        if m > 0:
            Ac = sp.csr_matrix(sp.random(m, n, density=0.01, random_state=seed) + sp.eye(m, n))
            fam = families.sparse_qcqp(P=Pm, q=rng.standard_normal(n), Qc=[sp.diags(0.1 * rng.random(n))] * m, Ac=Ac,
                                       jacobian="csr")
            J = jac_of(fam, x0)
        else:
            fam = families.sparse_qcqp(P=Pm, q=rng.standard_normal(n), jacobian="csr")
            J = np.zeros((0, n))
    xaug = O.ineq_initial_y(xl, xu, x0)
    return fam, J, xl, xu, xaug


PROJ_CASES = [(2048, 65, "mixed", "diagquad"), (2048, 1, "box", "diagquad"), (300, 0, "mixed", "diagquad"),
              (4096, 129, "mixed", "diagquad"), (2001, 40, "mixed", "csr"), (1001, 0, "box", "csr")]


@pytest.mark.gpu
@pytest.mark.parametrize("n,m,kind,jac", PROJ_CASES)
def test_projection_and_multipliers(L, O, n, m, kind, jac):
    fam, J, xl, xu, xaug = general_point(L, O, n, m, seed=n + m, kind=kind, jac=jac)
    P = L.LargeProblem(fam)
    P.set_bounds(xl, xu)
    assert P.factor(xaug, want=())["rank_deficient"] == 0
    v = np.random.default_rng(n).standard_normal(2 * n)
    pv, lam = P.project(v)
    d = disp(L)
    assert d["fused_single"] == d["fused_general"] == 0, d
    if m > 0:
        assert d["solve"] & SOLVE_TRIANGULAR, d
    assert lam.shape == (m + n,)
    Dx, Dy, Sv, dx, dy = grad_h(O, xl, xu, xaug)
    r1, r2 = embedded_projection_ratios(J, dx, dy, v, pv, lam[:m], lam[m:])
    print("n = %d m = %d %s %s: r1 %.2e r2 %.2e of the bound" % (n, m, kind, jac, r1, r2))
    assert r1 <= 1 and r2 <= 1, (r1, r2)
    rpv, rlam, rlamy = closed_projection(J, Dx, Dy, Sv, v)
    assert rel(pv, rpv) < 1e-8 and rel(lam[m:], rlamy) < 1e-8


# ------------------------------------------------------------------ d. projcg! with bounds
def projcg_setup(L, O, n, m, seed, jac):
    fam, J, xl, xu, xaug = general_point(L, O, n, m, seed, kind="mixed", jac=jac)
    rng = np.random.default_rng(seed + 1)
    q, r, s, t, _, _ = O.ineq_data(xl, xu)
    lam = 0.1 * rng.standard_normal(m)
    # lambda_y with 2 lambda_y s in [1, 50] where s != 0: kappa(H) <= 100 on every line
    lamy = np.where(s != 0, s * rng.uniform(0.5, 25.0, n), 0.0)
    Dx, Dy, Sv, _, _ = grad_h(O, xl, xu, xaug)
    x = xaug[:n]
    if jac == "diagquad":
        p = np.asarray(fam.params).ravel()
        Q, w, xt = p[:m * n].reshape(m, n), p[2 * m * n + m + n:], p[2 * m * n + m:2 * m * n + m + n]
        g = w * (x - xt)
        hx = lambda v: (w + Q.T @ lam) * v
    else:
        cb = fam.callbacks()
        g = np.zeros(n); cb["grad"](g, x)

        def hx(v):
            a = np.zeros(n); b = np.zeros(n); v = np.asarray(v, dtype=np.float64)
            cb["hess_vec"](a, v, x); cb["chess_vec"](b, v, x, lam)
            return a + b
    hop = lambda v: np.concatenate([hx(v[:n]) + 2 * lamy * q * v[:n], 2 * lamy * s * v[n:]])
    Jw = J * Dy[None, :]
    Gw = Jw @ Jw.T
    proj = lambda v: closed_projection(J, Dx, Dy, Sv, v, Gsolve=lambda t: np.linalg.solve(Gw, t))[0]
    Jl, Dxl, Dyl, Sl, sol = J.astype(T), Dx.astype(T), Dy.astype(T), Sv.astype(T), ld_solver(Gw)
    proj_ld = lambda v: closed_projection(Jl, Dxl, Dyl, Sl, v, Gsolve=sol)[0]
    return fam, xl, xu, xaug, np.concatenate([lam, lamy]), np.concatenate([g, np.zeros(n)]), hop, proj, proj_ld


@pytest.mark.gpu
@pytest.mark.parametrize("n,m,K,jac", [(4096, 33, 40, "diagquad"), (4096, 33, 65, "diagquad"), (2001, 20, 40, "csr")])
def test_projcg_with_bounds_vs_float64(L, O, n, m, K, jac):
    fam, xl, xu, xaug, lam, g, hop, proj, proj_ld = projcg_setup(L, O, n, m, seed=n + K, jac=jac)
    P = L.LargeProblem(fam)
    P.set_bounds(xl, xu)
    P.factor(xaug, want=())
    out = P.projcg(xaug, lam=lam, tol=0.0, maxit=K)
    d = disp(L)
    assert d["fused_single"] == d["fused_general"] == 0 and d["solve"] & SOLVE_TRIANGULAR, d
    assert out["iters"] == K and out["status"] == 4, out
    ref = ref_projcg_op(hop, proj(-g), proj, K)
    ref_ld = ref_projcg_op(hop, proj_ld(-g.astype(T)), proj_ld, K)
    e, tol = rel(out["sol"], ref), cg_bar(ref, ref_ld)
    print("projcg n = %d m = %d K = %d %s: vs float64 reference %.2e, bar %.2e" % (n, m, K, jac, e, tol))
    assert e < tol, (e, tol)


@pytest.mark.gpu
def test_projcg_iteration_cap_with_bounds(L, O):
    # min(maxit, 3n + rank) (optimize.jl:366-372): boxes only, so the working Hessian is positive definite everywhere
    n, m = 16, 2
    fam, xl, xu, xaug, lam, g, hop, proj, _ = projcg_setup(L, O, n, m, seed=9, jac="diagquad")
    xl2, xu2 = bounds_for(xaug[:n], 3, "box")
    P = L.LargeProblem(fam)
    P.set_bounds(xl2, xu2)
    xaug2 = O.ineq_initial_y(xl2, xu2, xaug[:n])
    P.factor(xaug2, want=())
    lam2 = np.concatenate([lam[:m], np.full(n, 3.0)])
    out = P.projcg(xaug2, lam=lam2, tol=0.0, maxit=10 ** 6)
    assert out["iters"] == 3 * n + m and out["status"] == 4, out


# ------------------------------------------------------------------ e. pcg! with bounds
def pcg_cases():
    return [(4096, 9, "diagquad"), (2001, 20, "csr"), ((1024, -2), 3, "diagquad"), ((1024, 2), 3, "diagquad"),
            ((1024, -1), 3, "csr"), ((1024, 1), 3, "csr")]


@pytest.mark.gpu
@pytest.mark.parametrize("nspec,m,jac", pcg_cases())
def test_pcg_with_bounds_vs_float64(L, S, O, nspec, m, jac):
    # n = 1024 S +- 1 or 2 (256 x vgrid with vgrid at its cap of 4 SMs): the grid-stride loops take one and two strides
    n = dim(nspec, S)
    fam, J, xl, xu, xaug = general_point(L, O, n, m, seed=7 + m, kind="mixed", jac=jac)
    Dx, Dy, Sv, _, _ = grad_h(O, xl, xu, xaug)
    B, Bt = bigA_ops(J, Dx, Dy, Sv)
    mu, K = 0.5, 20
    b = np.random.default_rng(n).standard_normal(2 * n)
    P = L.LargeProblem(fam)
    P.set_bounds(xl, xu)
    x, r, flag, it = P.pcg(xaug, mu, b, tol=0.0, maxiter=K)
    d = disp(L)
    assert d["fused_pcg"] == 0, d
    assert it == K and flag == 1
    xr, itr = ref_pcg_tol(lambda p: B(Bt(p)) + mu * p, b, 0.0, K)
    Bl, Btl = bigA_ops(J.astype(T), Dx.astype(T), Dy.astype(T), Sv.astype(T))
    xl_ref, _ = ref_pcg_tol(lambda p: Bl(Btl(p)) + mu * p, b.astype(T), 0.0, K)
    e, tol = rel(x, xr), cg_bar(xr, xl_ref)
    print("pcg n = %d m = %d %s: vs float64 reference %.2e, bar %.2e" % (n, m, jac, e, tol))
    assert itr == K and e < tol, (e, tol)


# ------------------------------------------------------------------ f. retractions with bounds
def ref_retract(method, fam, O, xl, xu, xb, xt, prm):
    """float64 transcription of large.cu's retract_nr / retract_pp with bounds -> (flag, xnew, it1, it2)"""
    n, m = fam.n, fam.m
    p = np.asarray(fam.params).ravel()
    Q, A, bb = p[:m * n].reshape(m, n), p[m * n:2 * m * n].reshape(m, n), p[2 * m * n:2 * m * n + m]
    cfun = lambda x: 0.5 * Q @ (x * x) + A @ x - bb
    jac = lambda x: Q * x[None, :] + A
    eps_c, maxit = prm.eps_c, int(prm.maxiter_retract)
    if method == "nr":
        Dx, Dy, Sv = O.ineq_gradient(xl, xu, xb)
        J = jac(xb[:n]); Jw = J * Dy[None, :]
        Lc = np.linalg.cholesky(Jw @ Jw.T); Li = np.linalg.inv(Lc)
        xnew = O.y_retract(xl, xu, xb, xt.copy())
        cval = cfun(xnew[:n]); D = Li.copy(); i = 0
        while i < maxit:
            if np.max(np.abs(cval)) < eps_c:
                break
            delta = -(D @ cval)
            s = J.T @ (Li.T @ delta)
            xn = xnew.copy()
            xn[:n] = xnew[:n] + Dy * Dy * s; xn[n:] = xnew[n:] - Dx * Dy * s
            xnew = O.y_retract(xl, xu, xb, xn)
            t2 = cfun(xnew[:n]); dcv = t2 - cval; cval = t2
            u = D.T @ delta; den = u @ dcv
            t1 = delta - D @ dcv
            D = D + np.outer(t1, u) / den
            i += 1
        return (1 if i == maxit else 0), xnew, i, 0
    xnew = xt.copy(); mu = prm.mu0; i = 0; flag = 0; total = 0; cvc = np.zeros(m)
    hfun = lambda z: O.ineq_h(xl, xu, z)
    while i < maxit:
        cval = cfun(xnew[:n]); J = jac(xnew[:n])
        Dx, Dy, Sv = O.ineq_gradient(xl, xu, xnew)
        h = hfun(xnew)
        curtol = max(np.max(np.abs(h)), np.max(np.abs(cval)), np.max(np.abs(cvc)))
        cvc = cval.copy()
        cc, hh = cval @ cval, h @ h
        gv = xnew - xt; gg = gv @ gv
        if curtol < eps_c:
            break
        prev = (hh + cc) + mu * gg
        B, Bt = bigA_ops(J, Dx, Dy, Sv)
        rhs = B(np.concatenate([h, cval])) + mu * gv
        dx, it = ref_pcg_tol(lambda q: B(Bt(q)) + mu * q, rhs, eps_c, int(prm.maxiter_pcg))
        total += it
        if it == prm.maxiter_pcg:
            flag = 2
            break
        base = xnew.copy(); ar_dot = -(rhs @ dx)
        xnew = base - dx; dist2 = (xnew - xt) @ (xnew - xt)
        cn = cfun(xnew[:n]); cvc = cn.copy(); ccnew = cn @ cn
        hn = hfun(xnew); hhnew = hn @ hn
        alpha, cnt = 1.0, 0
        while (hhnew + ccnew) + mu * dist2 > prev + 1e-4 * alpha * ar_dot:
            alpha /= 2
            xnew = base - alpha * dx; dist2 = (xnew - xt) @ (xnew - xt)
            hn = hfun(xnew); hhnew = hn @ hn
            cnt += 1
            if cnt == 100:
                flag = 3
                break
        i += 1
        mu = min(mu * 0.1, np.sqrt(hhnew + ccnew))
    if i == maxit:
        flag = 1
    return flag, xnew, i, total


@pytest.mark.gpu
@pytest.mark.parametrize("method", ["nr", "pp"])
@pytest.mark.parametrize("step", [1e-3, 1e-2])
def test_retraction_with_bounds_vs_transcription(L, O, method, step):
    n, m = 256, 8
    Q, A, b, xt, w, x0 = L.make_diagquad(n, m, seed=21, cond=50.0)
    fam = L.families.diagquad(Q, A, b, xt, w)
    xl, xu = bounds_for(x0, 31, "mixed")
    xb = O.ineq_initial_y(xl, xu, x0)
    assert np.max(np.abs(O.ineq_h(xl, xu, xb))) < 1e-12 and np.max(np.abs(0.5 * Q @ (x0 * x0) + A @ x0 - b)) < 1e-12
    xtil = xb + step * np.random.default_rng(int(1 / step)).standard_normal(2 * n)
    prm = L.LFPSQPParams()
    P = L.LargeProblem(fam)
    P.set_bounds(xl, xu)
    flag, xnew, cval, it, pit = P.retract(method, xb, xtil, prm)
    d = disp(L)
    assert d["fused_pcg"] == 0 and d["fused_single"] == d["fused_general"] == 0, d
    rflag, rx, rit, rpit = ref_retract(method, fam, O, xl, xu, xb, xtil, prm)
    print("%s step %.0e: flag %d/%d iters %d/%d pcg %d/%d, xnew vs transcription %.2e"
          % (method, step, flag, rflag, it, rit, pit, rpit, rel(xnew, rx)))
    assert (flag, it, pit) == (rflag, rit, rpit)
    assert rel(xnew, rx) < 1e-9
    assert flag == 0
    assert np.max(np.abs(O.ineq_h(xl, xu, xnew))) < prm.eps_c
    assert np.max(np.abs(0.5 * Q @ (xnew[:n] ** 2) + A @ xnew[:n] - b)) < prm.eps_c


# ------------------------------------------------------------------ g. the checkers reject corrupted results (no GPU)
def _exact_case(n=512, m=40, seed=5):
    xl, xu, x, y, mid = exact_point(n, seed)
    rng = np.random.default_rng(seed)
    J = (rng.integers(-8, 9, (m, n)) * x + rng.integers(-8, 9, (m, n))).astype(np.float64)
    return xl, xu, np.concatenate([x, y]), mid, J


def test_gram_checker_rejects_wrong_weights(oracle):
    xl, xu, xaug, mid, J = _exact_case()
    Dx, Dy, Sv = oracle.ineq_gradient(xl, xu, xaug)
    assert np.any(Dy < 0) and np.any(Dy == 0) and np.any(Dx != 0)
    assert gram_ok(weighted_gram(J, Dy), J, mid)
    assert not gram_ok((J * Dy) @ J.T, J, mid)                     # Dy where Dy^2 belongs
    Dy1 = Dy.copy(); Dy1[np.flatnonzero(mid)[7]] = 0.0
    assert not gram_ok(weighted_gram(J, Dy1), J, mid)              # one weight dropped
    assert not gram_ok(weighted_gram(J, Dx), J, mid)               # Dx and Dy swapped
    assert not gram_ok(J @ J.T, J, mid)                            # weights not applied at all


def _general_case(oracle, n=300, m=12, seed=3):
    rng = np.random.default_rng(seed)
    x0 = rng.standard_normal(n)
    xl, xu = bounds_for(x0, seed, "mixed")
    act = rng.random(n) < 0.2
    x0 = np.where(act & np.isfinite(xl), xl, x0)
    xaug = oracle.ineq_initial_y(xl, xu, x0)
    J = rng.standard_normal((m, n)) / np.sqrt(n)
    Dx, Dy, Sv = oracle.ineq_gradient(xl, xu, xaug)
    return J, Dx, Dy, Sv, rng.standard_normal(2 * n)


def test_projection_checker_accepts_the_closed_form(oracle):
    for m in (12, 0):
        J, Dx, Dy, Sv, v = _general_case(oracle, m=m)
        pv, lam, lamy = closed_projection(J, Dx, Dy, Sv, v)
        r1, r2 = embedded_projection_ratios(J, Dx * Sv, Dy * Sv, v, pv, lam, lamy)
        assert r1 <= 1 and r2 <= 1, (m, r1, r2)


def test_projection_checker_rejects_corruptions(oracle):
    J, Dx, Dy, Sv, v = _general_case(oracle)
    n = Dx.size
    dx, dy = Dx * Sv, Dy * Sv
    ratios = lambda pv, lam, lamy: embedded_projection_ratios(J, dx, dy, v, pv, lam, lamy)
    pv, lam, lamy = closed_projection(J, Dx, Dy, Sv, v)
    # Dy in place of Dy^2 (operand and removed part)
    Jy = J * np.abs(Dy)[None, :]
    lb = np.linalg.solve(J @ (Jy.T), J @ (Dy * (Dy * v[:n] - Dx * v[n:])))
    w = J.T @ lb; a = Dx * v[:n] + Dy * v[n:]
    pvb = np.concatenate([v[:n] - (Dx * a + Dy * w), v[n:] - (Dy * a - Dx * Dy * w)])
    assert max(ratios(pvb, lb, -(Dx / Sv) * w + a / Sv)) > 1
    # one weight dropped from the Gram
    k = int(np.argmax(np.abs(Dy)))
    Dy1 = Dy.copy(); Dy1[k] = 0.0
    lb = np.linalg.solve(weighted_gram(J, Dy1), J @ (Dy * (Dy * v[:n] - Dx * v[n:])))
    pvb = closed_projection(J, Dx, Dy, Sv, v, Gsolve=lambda t: lb)[0]
    assert max(ratios(pvb, lb, lamy)) > 1
    # Dx and Dy swapped
    pvb, lb, lyb = closed_projection(J, Dy, Dx, Sv, v)
    assert max(ratios(pvb, lb, lyb)) > 1
    # lambda_y with the wrong sign, and without / S
    assert ratios(pv, lam, -lamy)[1] > 1
    assert ratios(pv, lam, lamy * Sv)[1] > 1
    # the y-half shifted by one entry
    pvs = pv.copy(); pvs[n:] = np.roll(pv[n:], 1)
    assert max(ratios(pvs, lam, lamy)) > 1


def test_projcg_reference_rejects_a_dropped_bound_term(oracle):
    # the 2 lambda_y q term of the x-half Hessian dropped: the K-step iterate moves by more than the widest CG bar
    J, Dx, Dy, Sv, v = _general_case(oracle, n=400, m=10, seed=8)
    n = Dx.size
    rng = np.random.default_rng(2)
    q = (np.abs(Dx) < 1).astype(np.float64)      # a nonzero q where the point is not on a line
    w = np.exp(rng.uniform(0.0, np.log(50.0), n))
    lamy = rng.uniform(0.5, 25.0, n)
    proj = lambda u: closed_projection(J, Dx, Dy, Sv, u)[0]
    good = lambda u: np.concatenate([(w + 2 * lamy * q) * u[:n], 2 * lamy * u[n:]])
    bad = lambda u: np.concatenate([w * u[:n], 2 * lamy * u[n:]])
    b = proj(np.concatenate([-rng.standard_normal(n), np.zeros(n)]))
    K = 30
    ref = ref_projcg_op(good, b, proj, K)
    assert rel(ref_projcg_op(good, b, proj, K), ref) < CG_TOL
    assert rel(ref_projcg_op(bad, b, proj, K), ref) > 1e-5
    # and a y-half shifted by one inside the projector
    shifted = lambda u: (lambda p: np.concatenate([p[:n], np.roll(p[n:], 1)]))(proj(u))
    assert rel(ref_projcg_op(good, b, shifted, K), ref) > 1e-5
