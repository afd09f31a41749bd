"""Large-n mode on the sparse QCQP family (LFPSQP_FAM_SPARSE_QCQP): whole solves against the dense QCQP oracle
(tests/qcqp_reference.py), against the DIAGQUAD family and against host callbacks at a size the dense oracle cannot
take; unit-level factor / project / projcg; bit-identical repeats; and the argument errors of the C ABI.
Parity bar as tests/test_gpu_large.py: same termination, iterations +-1, x within 1e-8 relative, final objective within
1e-10 relative, multipliers within 1e-6 relative."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

sp = pytest.importorskip("scipy.sparse")


@pytest.fixture(scope="module")
def L():
    import lfpsqp.jl_b200 as L
    L.default_context(0)
    return L


@pytest.fixture(scope="module")
def ref():
    from tests import qcqp_reference
    qcqp_reference.build()
    return qcqp_reference


def rel(a, b):
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def dense(t, shape):
    out = np.zeros(shape)
    np.add.at(out, tuple(t[:-1]), t[-1])
    return out


def laplacian_1d(n, shift=0.1):
    return sp.diags([-np.ones(n - 1), (2.0 + shift) * np.ones(n), -np.ones(n - 1)], [-1, 0, 1]).tocsr()


def laplacian_2d(k, shift=0.01):
    T = laplacian_1d(k, 0.0)
    I = sp.identity(k)
    return (sp.kron(I, T) + sp.kron(T, I) + shift * sp.identity(k * k)).tocsr()


def oracle_solve(ref, fam, x0, xl=None, xu=None, **kw):
    """the dense QCQP oracle on the densified data of fam (its own slack wrapper for d)"""
    n, m, p = fam.n, fam.m, fam.p
    arrays = dict(P=dense(fam.P, (n, n)), q=fam.q, r=np.array([fam.r]), Qc=dense(fam.Qc, (m, n, n)), Ac=dense(fam.Ac, (m, n)),
                  bc=fam.bc, Qd=dense(fam.Qd, (p, n, n)), Ad=dense(fam.Ad, (p, n)), bd=fam.bd)
    fp, _ = ref.qcqp_params(n, m, p, **arrays)
    if p and xl is None:
        xl, xu = -np.inf * np.ones(n), np.inf * np.ones(n)
    prm = ref.default_params(**{k: int(v) if isinstance(v, bool) else v for k, v in kw.items()})
    x, obj, olen, lam, term, stats = ref.optimize_batched("qcqp", n, m, p, x0[None], xl, xu, fam_params=fp, params=prm, H=4096)
    return x[0], obj[0, :int(olen[0])], lam[0], term[0]


def assert_parity(got, want):
    x, obj, lam, info = got
    ox, oobj, olam, ot = want
    assert int(info.condition) == int(ot["condition"]) and abs(info.iter - int(ot["iter"])) <= 1, (info, ot)
    assert rel(x, ox) <= 1e-8, rel(x, ox)
    assert abs(obj[-1] - oobj[-1]) <= 1e-10 * max(abs(oobj[-1]), 1e-300), (obj[-1], oobj[-1])
    if len(olam):
        assert rel(lam, olam) <= 1e-6, rel(lam, olam)


def args_of(fam, x0, xl=None, xu=None, dl=None, du=None):
    if fam.p:
        return [fam.f, fam.c, fam.d, dl, du, x0, xl, xu, fam.m, fam.p] if dl is not None else \
               [fam.f, fam.c, fam.d, x0, xl, xu, fam.m, fam.p]
    if xl is not None:
        return [fam.f, fam.c, x0, xl, xu, fam.m]
    return [fam.f, fam.c, x0, fam.m]


# ------------------------------------------------------------------------------------------------ a. dense oracle
def rayleigh(n=300, seed=1):
    rng = np.random.default_rng(seed)
    A = sp.random(n, n, density=4.0 / n, random_state=seed) + laplacian_1d(n, 0.0)
    A = (A + A.T).tocsr()
    fam = L_fam().sparse_qcqp(P=A, Qc=[sp.identity(n)], bc=[0.5])
    x0 = rng.standard_normal(n); x0 /= np.linalg.norm(x0)
    return fam, x0, A


def L_fam():
    from lfpsqp.jl_b200 import families
    return families


def test_rayleigh_quotient(L, ref):
    fam, x0, A = rayleigh()
    got = L.optimize_large(fam.f, fam.c, x0, 1)
    assert_parity(got, oracle_solve(ref, fam, x0))
    lmin = np.linalg.eigvalsh(A.toarray())[0]
    assert abs(got[1][-1] - 0.5 * lmin) <= 1e-5 * max(1.0, abs(lmin))


def convex_qp(n=256, m=12, seed=2):
    rng = np.random.default_rng(seed)
    Ac = sp.random(m, n, density=0.05, random_state=seed) + sp.eye(m, n)
    x0 = rng.standard_normal(n)
    return L_fam().sparse_qcqp(P=laplacian_1d(n), q=rng.standard_normal(n), r=1.5, Ac=Ac, bc=Ac @ x0), x0


@pytest.mark.parametrize("bounds", [False, True])
def test_convex_qp(L, ref, bounds):
    fam, x0 = convex_qp()
    xl = xu = None
    if bounds:
        xl, xu = -0.5 * np.ones(fam.n), 0.5 * np.ones(fam.n)
        x0 = np.clip(x0, -0.4, 0.4)
        fam = L_fam().sparse_qcqp(P=laplacian_1d(fam.n), q=fam.q, r=fam.r, Ac=dense(fam.Ac, (fam.m, fam.n)),
                                  bc=dense(fam.Ac, (fam.m, fam.n)) @ x0)
    got = L.optimize_large(*args_of(fam, x0, xl, xu))
    assert_parity(got, oracle_solve(ref, fam, x0, xl, xu))


def block_equalities(n=240, nblk=6, nlin=5, seed=3):
    rng = np.random.default_rng(seed)
    bs = n // nblk
    Qc = []
    for k in range(nblk):
        d = np.zeros(n); d[k * bs:(k + 1) * bs] = 1.0
        Qc.append(sp.diags(d))
    Ac = sp.vstack([sp.csr_matrix((nblk, n)), sp.random(nlin, n, density=0.1, random_state=seed)]).tocsr()
    Qc += [sp.csr_matrix((n, n))] * nlin
    x0 = rng.standard_normal(n)
    for k in range(nblk):
        x0[k * bs:(k + 1) * bs] /= np.linalg.norm(x0[k * bs:(k + 1) * bs])
    bc = np.concatenate([0.5 * np.ones(nblk), Ac[nblk:] @ x0])
    return L_fam().sparse_qcqp(P=laplacian_1d(n, 1.0), q=rng.standard_normal(n), Qc=Qc, Ac=Ac, bc=bc), x0


def test_block_quadratic_equalities(L, ref):
    fam, x0 = block_equalities()
    got = L.optimize_large(*args_of(fam, x0))
    assert_parity(got, oracle_solve(ref, fam, x0))


def balls(n=256, p=4, seed=4, lin=True):
    rng = np.random.default_rng(seed)
    bs = n // p
    Qd = []
    for k in range(p):
        d = np.zeros(n); d[k * bs:(k + 1) * bs] = 1.0
        Qd.append(sp.diags(d))
    Ac = sp.random(3, n, density=0.1, random_state=seed) if lin else None
    x0 = 0.05 * rng.standard_normal(n)
    kw = dict(Ac=Ac, bc=Ac @ x0) if lin else {}
    fam = L_fam().sparse_qcqp(P=laplacian_1d(n, 0.05), q=-rng.standard_normal(n), Qd=Qd, bd=0.5 * np.ones(p), **kw)
    return fam, x0


def test_inequalities_through_slack_variables(L, ref):
    fam, x0 = balls()
    got = L.optimize_large(*args_of(fam, x0))
    assert len(got[2]) == fam.m + fam.p
    assert_parity(got, oracle_solve(ref, fam, x0))


@pytest.mark.parametrize("variant", ["nr", "exact", "odd_n", "m0_bounds"])
def test_driver_variants(L, ref, variant):
    kw = {}
    xl = xu = None
    if variant == "nr":
        fam, x0 = block_equalities()
        kw = dict(do_project_retract=False)
    elif variant == "exact":
        fam, x0 = block_equalities(seed=5)
        kw = dict(linesearch=1)
    elif variant == "odd_n":
        fam, x0 = block_equalities(n=245, nblk=5, seed=6)
    else:
        rng = np.random.default_rng(7)
        n = 201
        fam = L_fam().sparse_qcqp(P=laplacian_1d(n), q=3 * rng.standard_normal(n))
        x0 = np.zeros(n)
        xl, xu = -np.ones(n), np.ones(n)
    got = L.optimize_large(*args_of(fam, x0, xl, xu), L.LFPSQPParams(**kw))
    assert_parity(got, oracle_solve(ref, fam, x0, xl, xu, **kw))


def test_beta_noise(L, ref):
    fam, x0 = block_equalities(seed=8)
    T = 20
    nz = np.random.default_rng(9).standard_normal((T, fam.n))
    kw = dict(beta=1e-3, t_beta=T)
    got = L.optimize_large(*args_of(fam, x0), L.LFPSQPParams(**kw), noise=nz)
    ref.set_noise(nz[None])
    try:
        want = oracle_solve(ref, fam, x0, **kw)
    finally:
        ref.set_noise(None)
    assert_parity(got, want)


# ------------------------------------------------------------------------------------------------ b. DIAGQUAD
def test_matches_diagquad(L):
    n, m = 8192, 256
    Q, A, b, xt, w, x0 = L.make_diagquad(n, m, seed=3, cond=100.0)
    dq = L.LargeProblem(L.families.diagquad(Q, A, b, xt, w)).solve(x0)
    fam = L.families.sparse_qcqp(P=sp.diags(w), q=-w * xt, r=0.5 * np.sum(w * xt * xt), Qc=[sp.diags(Q[i]) for i in range(m)],
                                 Ac=A, bc=b)
    got = L.optimize_large(fam.f, fam.c, x0, m)
    x, obj, lam, info = got
    assert int(info.condition) == int(dq[3].condition) and abs(info.iter - dq[3].iter) <= 1
    assert rel(x, dq[0]) <= 1e-8 and abs(obj[-1] - dq[1][-1]) <= 1e-10 * abs(dq[1][-1]) and rel(lam, dq[2]) <= 1e-6


# ------------------------------------------------------------------------------------------------ c, d. host callbacks
def _host(L, fam, x0, xl=None, xu=None, dl=None, du=None):
    cb = fam.callbacks()
    return L.optimize_slack(cb["f"], cb["grad"], cb["hess_vec"], cb["c"], cb["jac"], cb["chess_vec"], cb["d"], cb["djac"],
                            cb["dhess_vec"], dl, du, x0, xl, xu, fam.m, fam.p)


def _same_bar(got, want):
    x, obj, lam, info = got
    hx, hobj, hlam, hinfo = want
    assert int(info.condition) == int(hinfo.condition) and abs(info.iter - hinfo.iter) <= 1, (info, hinfo)
    assert rel(x, hx) <= 1e-8 and abs(obj[-1] - hobj[-1]) <= 1e-10 * abs(hobj[-1]) and rel(lam, hlam) <= 1e-6


def test_against_host_callbacks_at_scale(L):
    k, m = 256, 512
    n = k * k
    rng = np.random.default_rng(10)
    Ac = sp.random(m, n, density=64.0 / n, random_state=10, format="csr")
    x0 = 0.1 * rng.standard_normal(n)
    fam = L.families.sparse_qcqp(P=laplacian_2d(k), q=rng.standard_normal(n), Ac=Ac, bc=Ac @ x0 + 0.01)
    _same_bar(L.optimize_large(fam.f, fam.c, x0, m), _host(L, fam, x0))


def test_two_sided_inequalities_match_optimize_slack(L):
    fam, x0 = balls(seed=11)
    p = fam.p
    dl = np.array([-np.inf, -0.3, -1.0, -np.inf])
    du = np.array([0.0, np.inf, 0.2, 0.1])
    xl, xu = -np.ones(fam.n), np.inf * np.ones(fam.n)
    got = L.optimize_large(fam.f, fam.c, fam.d, dl, du, x0, xl, xu, fam.m, p)
    _same_bar(got, _host(L, fam, x0, xl, xu, dl, du))


# ------------------------------------------------------------------------------------------------ e. unit level
def test_factor_project_projcg(L):
    fam, x0 = block_equalities(n=480, nblk=8, nlin=9, seed=12)
    n, m = fam.n, fam.m
    P = L.LargeProblem(fam)
    J = np.zeros((m, n), order="F"); cv = np.zeros(m)
    fam.callbacks()["jac"](J, cv, x0)
    fac = P.factor(x0)
    G = J @ J.T
    assert fac["rank_deficient"] == 0 and rel(np.tril(fac["G"]), np.tril(G)) < 1e-14
    v = np.random.default_rng(13).standard_normal(n)
    pv, lam = P.project(v)
    u = np.linalg.solve(G, J @ v)
    assert rel(pv, v - J.T @ u) < 1e-12 and rel(lam, u) < 1e-11
    # projcg with the assembled H = P + sum lam_i Qc_i (test/test_cg.jl:23-28 properties)
    lam = 0.1 * np.random.default_rng(14).standard_normal(m)
    H = dense(fam.P, (n, n)) + np.einsum("k,kij->ij", lam, dense(fam.Qc, (m, n, n)))
    Pm = lambda w: w - J.T @ np.linalg.solve(G, J @ w)
    b = Pm(np.random.default_rng(15).standard_normal(n))
    c = np.random.default_rng(16).standard_normal(m)
    r = P.projcg_general(x0, lam, b, c, tol=1e-10, maxit=10000)
    assert r["status"] == 1
    x = r["sol"]
    Lc = np.linalg.cholesky(G)
    U = J.T @ np.linalg.inv(Lc).T                   # the orthonormal basis J' L^-T of range(J')
    assert np.allclose(U.T @ x, c, atol=1e-9)
    assert np.linalg.norm(Pm(H @ x - b)) < 1e-8
    assert rel(r["lam"], U.T @ (b - H @ x)) < 1e-8


def test_unbounded_solve_uses_fused_pcg(L):
    fam, x0 = block_equalities(seed=17)
    P = L.LargeProblem(fam)
    P.solve(x0)
    d = L.default_context(0).large_dispatch
    assert d["fused_pcg"] > 0 and d["fused_single"] == 0 and d["fused_general"] == 0


# ------------------------------------------------------------------------------------------------ f. determinism
def test_repeat_solves_are_bit_identical(L):
    fam, x0 = balls(n=512, p=8, seed=18)
    a = L.optimize_large(*args_of(fam, x0), return_stats=True)
    b = L.optimize_large(*args_of(fam, x0), return_stats=True)
    for u, v in zip(a[:3], b[:3]):
        assert np.array_equal(np.asarray(u).view(np.uint8), np.asarray(v).view(np.uint8))
    assert a[3] == b[3] and a[4] == b[4] and a[5] == b[5]


# ------------------------------------------------------------------------------------------------ g. errors
def _setup(L, fam, desc=None, n_loc=None, on_dev=0):
    ctx = L.default_context(0)
    pp, keep = fam.large_args()
    if desc is not None:
        pp = C.cast(C.pointer(desc), C.c_void_p)
    return ctx.lib.lfpsqp_large_setup(ctx.h, 102, fam.n, fam.m, 0, fam.n if n_loc is None else n_loc, pp, on_dev), ctx


def test_argument_errors(L):
    ERR_ARG, ERR_FAMILY = -1, -3
    fam = L.families.sparse_qcqp(P=laplacian_1d(6), q=np.ones(6), Qc=[sp.identity(6), 2 * sp.identity(6)], Ac=np.ones((2, 6)),
                                 bc=[0.5, 1.0])
    rc, ctx = _setup(L, fam)
    assert rc == 0

    def mutated(field, key, values):
        """a descriptor whose list `field` has array `key` replaced by `values` (the arrays stay alive in `hold`)"""
        pp, keep = fam.large_args()
        desc = keep[0]
        arr = np.ascontiguousarray(values)
        hold.append(arr)
        setattr(getattr(desc, field), key, None if values is None else arr.ctypes.data)
        hold.append(keep)
        return desc

    hold = []
    P0 = fam.P
    cases = {
        "out of range": mutated("P", "col", np.where(P0[1] == 5, 6, P0[1]).astype(np.int64)),
        "constraint index": mutated("Qc", "mat", np.where(np.arange(fam.Qc[0].size) == 2, 2, fam.Qc[0]).astype(np.int64)),
        "duplicate": mutated("Ac", "col", np.zeros(fam.Ac[1].size, np.int64)),
        "symmetric": mutated("P", "val", P0[2] + (P0[0] < P0[1]) * 1e-16 * 4),
        "NULL": mutated("Qc", "row", None),
        "finite": mutated("Ac", "val", np.where(np.arange(fam.Ac[2].size) == 3, np.nan, fam.Ac[2])),
    }
    for what, desc in cases.items():
        rc, ctx = _setup(L, fam, desc=desc)
        msg = ctx.lib.lfpsqp_last_error(ctx.h).decode()
        assert rc == ERR_ARG, (what, rc, msg)
        assert what in msg or what.split()[0] in msg.lower(), (what, msg)
    # on the device / sharded / batched
    assert _setup(L, fam, on_dev=1)[0] == ERR_ARG
    assert _setup(L, fam, n_loc=fam.n - 2)[0] == ERR_FAMILY
    pp, keep = fam.large_args()
    x0 = np.zeros((2, fam.n)); out = np.zeros((2, fam.n)); obj = np.zeros((2, 4)); olen = np.zeros(2, np.int64)
    lam = np.zeros((2, fam.m)); term = np.zeros(2, dtype=L._lib.TERM_DTYPE)
    cp = L.LFPSQPParams().to_c()
    rc = ctx.lib.lfpsqp_solve_batched(ctx.h, 102, fam.n, fam.m, 0, 2, pp, 0, L._lib.ptr(x0), None, None,
                                      C.cast(C.pointer(cp), C.c_void_p), L._lib.ptr(out), L._lib.ptr(obj), 4, L._lib.ptr(olen),
                                      L._lib.ptr(lam), L._lib.ptr(term), None)
    assert rc == ERR_FAMILY
    with pytest.raises(L.LFPSQPError, match="optimize_large"):
        L.optimize(fam.f, fam.c, np.zeros(fam.n), fam.m)
    # a valid problem binds again after the refusals
    assert _setup(L, fam)[0] == 0
