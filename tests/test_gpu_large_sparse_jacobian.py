"""Sparse QCQP family with its Jacobian kept sparse on the device (LFPSQP_FAM_SPARSE_QCQP_CSR, jacobian="csr"): parity with
the dense-Jacobian family and the dense QCQP oracle, the exact sparse Gram, projections and pcg! against extended-precision
and float64 references, the dispatch record, a problem whose dense Jacobian would not fit on the GPU, bit-identical repeats
and the argument errors.  Parity bar as tests/test_gpu_large_sparse_qcqp.py."""
import ctypes as C

import numpy as np
import pytest

from tests.test_gpu_large_boundaries import projection_ratios
from tests.test_gpu_large_sparse_qcqp import (L, args_of, assert_parity, balls, block_equalities, convex_qp, dense, laplacian_1d,
                                              oracle_solve, ref, rel, rayleigh)

pytestmark = pytest.mark.gpu

sp = pytest.importorskip("scipy.sparse")

SPARSE_GRAM, CSR_ROWS, CSC_COLS = 256, 64, 128
SOLVE_PINV = 4


def as_csr(fam):
    from lfpsqp.jl_b200 import families
    return families.SparseQCQPFamily(fam.n, fam.m, fam.p, fam.P, fam.q, fam.r, fam.Qc, fam.Ac, fam.bc, fam.Qd, fam.Ad, fam.bd,
                                     jacobian="csr")


def as_want(res):
    """an optimize_large result in the shape assert_parity takes as its reference"""
    x, obj, lam, info = res
    return x, obj, lam, dict(condition=int(info.condition), iter=info.iter)


def jac_of(fam, x):
    J = np.zeros((fam.m, fam.n), order="F"); cv = np.zeros(fam.m)
    fam.callbacks()["jac"](J, cv, x)
    return np.ascontiguousarray(J)


# ------------------------------------------------------------------------------------------------ 1. parity
@pytest.mark.parametrize("case", ["rayleigh", "qp", "qp_bounds", "blocks", "balls", "nr", "exact", "odd_n", "m0_bounds", "beta"])
def test_parity_with_dense_jacobian_and_oracle(L, ref, case):
    from lfpsqp.jl_b200 import families
    xl = xu = None
    kw = {}
    noise = None
    if case == "rayleigh":
        fam, x0, _ = rayleigh()
    elif case.startswith("qp"):
        fam, x0 = convex_qp()
        if case == "qp_bounds":
            xl, xu = -0.5 * np.ones(fam.n), 0.5 * np.ones(fam.n)
            x0 = np.clip(x0, -0.4, 0.4)
            A = dense(fam.Ac, (fam.m, fam.n))
            fam = families.sparse_qcqp(P=laplacian_1d(fam.n), q=fam.q, r=fam.r, Ac=A, bc=A @ x0)
    elif case == "blocks":
        fam, x0 = block_equalities()
    elif case == "balls":
        fam, x0 = balls()
    elif case == "nr":
        fam, x0 = block_equalities()
        kw = dict(do_project_retract=False)
    elif case == "exact":
        fam, x0 = block_equalities(seed=5)
        kw = dict(linesearch=1)
    elif case == "odd_n":
        fam, x0 = block_equalities(n=245, nblk=5, seed=6)
    elif case == "m0_bounds":
        rng = np.random.default_rng(7)
        n = 201
        fam = families.sparse_qcqp(P=laplacian_1d(n), q=3 * rng.standard_normal(n))
        x0, xl, xu = np.zeros(n), -np.ones(n), np.ones(n)
    else:
        fam, x0 = block_equalities(seed=8)
        kw = dict(beta=1e-3, t_beta=20)
        noise = np.random.default_rng(9).standard_normal((20, fam.n))
    cfam = as_csr(fam)
    assert cfam.id == 103 and fam.id == 102
    prm = L.LFPSQPParams(**kw)
    got = L.optimize_large(*args_of(cfam, x0, xl, xu), prm, noise=noise)
    assert_parity(got, as_want(L.optimize_large(*args_of(fam, x0, xl, xu), prm, noise=noise)))
    if noise is not None:
        ref.set_noise(noise[None])
    try:
        want = oracle_solve(ref, fam, x0, xl, xu, **kw)
    finally:
        ref.set_noise(None)
    assert_parity(got, want)


def test_two_sided_inequalities(L):
    fam, x0 = balls(seed=11)
    dl = np.array([-np.inf, -0.3, -1.0, -np.inf])
    du = np.array([0.0, np.inf, 0.2, 0.1])
    xl, xu = -np.ones(fam.n), np.inf * np.ones(fam.n)
    want = L.optimize_large(fam.f, fam.c, fam.d, dl, du, x0, xl, xu, fam.m, fam.p)
    cfam = as_csr(fam)
    assert_parity(L.optimize_large(cfam.f, cfam.c, cfam.d, dl, du, x0, xl, xu, cfam.m, cfam.p), as_want(want))


# ------------------------------------------------------------------------------------------------ 2. exact Gram
def gram_problem(kind, seed=0):
    """(family, x) with integer Qc, Ac and x: J = Qc_i x + Ac_i is integer and J J' exact in binary64"""
    from lfpsqp.jl_b200 import families
    rng = np.random.default_rng(seed)
    n, m, Qc = 1001, 8, None
    if isinstance(kind, int):
        m = kind
        Ac = sp.random(m, n, density=0.02, random_state=seed, data_rvs=lambda k: rng.integers(-3, 4, k).astype(float))
        Qc = [sp.diags(rng.integers(-2, 3, n).astype(float) * (rng.random(n) < 0.01)) for _ in range(m)]
    elif kind == "zero_row":
        Ac = sp.random(m, n, density=0.05, random_state=seed, data_rvs=lambda k: rng.integers(1, 4, k).astype(float)).tolil()
        Ac[3, :] = 0
    elif kind == "duplicate_rows":
        A = sp.random(m, n, density=0.05, random_state=seed, data_rvs=lambda k: rng.integers(1, 4, k).astype(float)).tolil()
        A[5, :] = A[1, :]
        A[6, :] = A[1, :]
        Ac = A
    elif kind == "long_row":
        n = (1 << 20) + 1
        A = sp.random(5, n, density=40.0 / n, random_state=seed, data_rvs=lambda k: rng.integers(1, 4, k).astype(float)).tolil()
        A[2, :] = rng.integers(1, 4, n).astype(float)[None]
        Ac, m = A, 5
    elif kind == "shared_column":
        A = sp.random(64, n, density=0.01, random_state=seed, data_rvs=lambda k: rng.integers(1, 4, k).astype(float)).tolil()
        A[:, 17] = rng.integers(1, 4, 64).astype(float)[:, None]
        Ac, m = A, 64
    Ac = sp.csr_matrix(Ac)
    m = Ac.shape[0]
    fam = families.sparse_qcqp(q=np.zeros(n), Qc=Qc, Ac=Ac, jacobian="csr")
    x = rng.integers(-2, 3, n).astype(float)
    return fam, x


@pytest.mark.parametrize("kind", [1, 63, 64, 65, 129, "zero_row", "duplicate_rows", "long_row", "shared_column"])
def test_gram_is_exact(L, kind):
    fam, x = gram_problem(kind)
    J = jac_of(fam, x)
    assert np.array_equal(J, np.round(J))
    P = L.LargeProblem(fam)
    fac = P.factor(x, want=("G",))
    d = L.default_context(0).large_dispatch
    assert d["gemm"] & SPARSE_GRAM and not d["gemm"] & 15, d
    want = np.tril(J @ J.T)
    assert np.array_equal(np.tril(fac["G"]).view(np.uint64), want.view(np.uint64))
    if kind in ("zero_row", "duplicate_rows"):
        assert fac["rank_deficient"] > 0
        P.project(np.random.default_rng(1).standard_normal(fam.n))
        assert L.default_context(0).large_dispatch["solve"] & SOLVE_PINV
    else:
        assert fac["rank_deficient"] == 0


# ------------------------------------------------------------------------------------------------ 3. projection and pcg!
def pass_problem(kind, seed=3):
    from lfpsqp.jl_b200 import families
    rng = np.random.default_rng(seed)
    n = 20001
    if kind == "long_row":      # one row over every column: 5 chunks of the row pass and of the Gram
        A = sp.random(40, n, density=0.003, random_state=seed).tolil()
        A[7, :] = rng.standard_normal(n)[None]
    else:                       # a few columns touched by every row
        A = sp.random(300, n, density=0.002, random_state=seed).tolil()
        for j in (0, 5, 9999, n - 1):
            A[:, j] = rng.standard_normal(300)[:, None]
    Ac = sp.csr_matrix(A)
    fam = families.sparse_qcqp(P=laplacian_1d(n), Qc=[sp.diags(rng.random(n) * (rng.random(n) < 0.1))] * Ac.shape[0], Ac=Ac,
                               jacobian="csr")
    return fam, rng.standard_normal(n)


@pytest.mark.parametrize("kind", ["long_row", "shared_columns"])
def test_projection_residuals(L, kind):
    fam, x = pass_problem(kind)
    J = jac_of(fam, x)
    P = L.LargeProblem(fam)
    assert P.factor(x, want=())["rank_deficient"] == 0
    v = np.random.default_rng(5).standard_normal(fam.n)
    pv, lam = P.project(v)
    d = L.default_context(0).large_dispatch
    assert d["rows_dot"] == CSR_ROWS | CSC_COLS, d
    r1, r2 = projection_ratios(J, v, pv, lam)
    assert r1 <= 1 and r2 <= 1, (r1, r2)


@pytest.mark.parametrize("kind", ["long_row", "shared_columns"])
def test_pcg_matches_float64_cg(L, kind):
    fam, x = pass_problem(kind, seed=4)
    J = sp.csr_matrix(jac_of(fam, x))
    mu = 0.5
    b = np.random.default_rng(6).standard_normal(fam.n)
    K = 20
    xs, r, fl, it = L.LargeProblem(fam).pcg(x, mu, b, tol=0.0, maxiter=K)
    assert it == K and fl == 1
    # float64 CG on (J'J + mu I) x = b, K steps from x = 0 (retractions.jl:179-246 without a preconditioner)
    A = lambda w: J.T @ (J @ w) + mu * w
    xr = np.zeros(fam.n); rr = b.copy(); p = np.zeros(fam.n); rho_prev = 1.0
    for _ in range(K):
        rho = rr @ rr
        p = rr + (rho / rho_prev) * p
        z = A(p)
        al = rho / (p @ z)
        xr += al * p; rr -= al * z; rho_prev = rho
    # K CG steps amplify the rounding of different summation orders; a dropped row or pass moves the iterate by O(1)
    assert rel(xs, xr) <= 1e-7, rel(xs, xr)


# ------------------------------------------------------------------------------------------------ 4. dispatch
def test_dispatch_record(L):
    fam, x0 = block_equalities(seed=17)        # unbounded, even n: the dense family takes the fused pcg! kernel
    assert fam.n % 2 == 0
    L.LargeProblem(fam).solve(x0)
    dd = dict(L.default_context(0).large_dispatch)
    assert dd["fused_pcg"] > 0 and dd["gemm"] & 15 and dd["rows_dot"] & 7 and not dd["gemm"] & SPARSE_GRAM
    assert not dd["rows_dot"] & (CSR_ROWS | CSC_COLS)
    L.LargeProblem(as_csr(fam)).solve(x0)
    d = L.default_context(0).large_dispatch
    assert d["gemm"] & SPARSE_GRAM and not d["gemm"] & 15, d
    assert d["rows_dot"] == CSR_ROWS | CSC_COLS, d
    assert d["fused_pcg"] == 0 and d["fused_single"] == 0 and d["fused_general"] == 0, d


# ------------------------------------------------------------------------------------------------ 5. beyond dense
def test_beyond_dense(L):
    import torch
    from lfpsqp.jl_b200 import families
    n, nlin, nsph, blk = 1 << 24, 2000, 47, 4096
    m = nlin + nsph + 1
    rng = np.random.default_rng(20)
    x0 = rng.standard_normal(n)
    rows = np.repeat(np.arange(nlin), 64)
    cols = rng.integers(0, n, nlin * 64)
    Alin = sp.csr_matrix((rng.standard_normal(nlin * 64), (rows, cols)), shape=(nlin, n))
    Alin.sum_duplicates()
    Ac = sp.vstack([Alin, sp.csr_matrix((nsph, n)), sp.csr_matrix(np.ones((1, n)))]).tocsr()   # last row: sum(x) = s
    Qc = [sp.coo_matrix((n, n))] * nlin
    for k in range(nsph):
        idx = np.arange(k * blk, (k + 1) * blk)
        Qc.append(sp.coo_matrix((np.ones(blk), (idx, idx)), shape=(n, n)))
    Qc.append(sp.coo_matrix((n, n)))
    bc = np.concatenate([Alin @ x0, [0.5 * x0[k * blk:(k + 1) * blk] @ x0[k * blk:(k + 1) * blk] for k in range(nsph)], [x0.sum()]])
    w = 1.0 + rng.random(n)
    xt = x0 + 1e-2 * rng.standard_normal(n)
    fam = families.sparse_qcqp(P=sp.diags(w), q=-w * xt, r=0.5 * np.sum(w * xt * xt), Qc=Qc, Ac=Ac, bc=bc, jacobian="csr")
    assert fam.m == m == 2048
    nnz = int(fam.Ac[2].size) + nsph * blk                       # structural entries of J (segments)
    assert 8 * m * n > 250e9                                     # a dense J would not fit
    torch.cuda.init()
    free0, _ = torch.cuda.mem_get_info(0)
    P = L.LargeProblem(fam)
    torch.cuda.synchronize()
    free1, _ = torch.cuda.mem_get_info(0)
    used = free0 - free1
    # CSR + CSC values and indices, the 12 working vectors (2n each), the P / H patterns and the x-sized spq structures
    shapes = 2 * 8 * nnz + 3 * 4 * nnz + 4 * (n + 1) + 12 * 8 * (2 * n + 2) + 2 * 8 * n
    assert used <= 3 * shapes, (used, shapes)
    x, obj, lam, info = P.solve(x0)
    assert info.condition in (L.TerminationCondition.f_tol, L.TerminationCondition.x_tol, L.TerminationCondition.kkt_tol), info
    Jq = sp.vstack([Alin, sp.csr_matrix((np.concatenate([x[k * blk:(k + 1) * blk] for k in range(nsph)]),
                                         (np.repeat(np.arange(nsph), blk), np.arange(nsph * blk))), shape=(nsph, n)),
                    sp.csr_matrix(np.ones((1, n)))]).tocsr()
    c = np.concatenate([Alin @ x, [0.5 * x[k * blk:(k + 1) * blk] @ x[k * blk:(k + 1) * blk] for k in range(nsph)], [x.sum()]]) - bc
    assert np.max(np.abs(c)) <= 1e-5, np.max(np.abs(c))
    kkt = w * (x - xt) + Jq.T @ lam
    assert np.max(np.abs(kkt)) <= 1e-4, np.max(np.abs(kkt))


# ------------------------------------------------------------------------------------------------ 6. determinism and errors
def test_repeat_solves_are_bit_identical(L):
    fam, x0 = balls(n=512, p=8, seed=18)
    cfam = as_csr(fam)
    a = L.optimize_large(*args_of(cfam, x0), return_stats=True)
    b = L.optimize_large(*args_of(cfam, x0), return_stats=True)
    for u, v in zip(a[:3], b[:3]):
        assert np.array_equal(np.asarray(u).view(np.uint8), np.asarray(v).view(np.uint8))
    assert a[3] == b[3] and a[4] == b[4] and a[5] == b[5]


def _setup(L, fam, desc=None, n_loc=None, on_dev=0):
    ctx = L.default_context(0)
    pp, keep = fam.large_args()
    if desc is not None:
        pp = C.cast(C.pointer(desc), C.c_void_p)
    return ctx.lib.lfpsqp_large_setup(ctx.h, 103, fam.n, fam.m, 0, fam.n if n_loc is None else n_loc, pp, on_dev), ctx


def test_argument_errors(L):
    ERR_ARG, ERR_FAMILY = -1, -3
    fam = L.families.sparse_qcqp(P=laplacian_1d(6), q=np.ones(6), Qc=[sp.identity(6), 2 * sp.identity(6)], Ac=np.ones((2, 6)),
                                 bc=[0.5, 1.0], jacobian="csr")
    rc, ctx = _setup(L, fam)
    assert rc == 0
    hold = []

    def mutated(field, key, values):
        pp, keep = fam.large_args()
        desc = keep[0]
        arr = np.ascontiguousarray(values)
        hold.append(arr)
        setattr(getattr(desc, field), key, None if values is None else arr.ctypes.data)
        hold.append(keep)
        return desc

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
    assert _setup(L, fam, on_dev=1)[0] == ERR_ARG
    assert _setup(L, fam, n_loc=fam.n - 2)[0] == ERR_FAMILY
    pp, keep = fam.large_args()
    x0 = np.zeros((2, fam.n)); out = np.zeros((2, fam.n)); obj = np.zeros((2, 4)); olen = np.zeros(2, np.int64)
    lam = np.zeros((2, fam.m)); term = np.zeros(2, dtype=L._lib.TERM_DTYPE)
    cp = L.LFPSQPParams().to_c()
    rc = ctx.lib.lfpsqp_solve_batched(ctx.h, 103, fam.n, fam.m, 0, 2, pp, 0, L._lib.ptr(x0), None, None,
                                      C.cast(C.pointer(cp), C.c_void_p), L._lib.ptr(out), L._lib.ptr(obj), 4, L._lib.ptr(olen),
                                      L._lib.ptr(lam), L._lib.ptr(term), None)
    assert rc == ERR_FAMILY
    with pytest.raises(L.LFPSQPError, match="optimize_large"):
        L.optimize(fam.f, fam.c, np.zeros(fam.n), fam.m)
    with pytest.raises(L.LFPSQPError, match="optimize_large"):
        L.optimize_batched(fam.f, fam.c, np.zeros((2, fam.n)), fam.m)
    assert _setup(L, fam)[0] == 0
