"""Large-n mode at its tile, split, row-pass and fallback boundaries (large.cu, large_gemm.cuh, large_kernels.cuh,
large_fused*.cu, large_eig.cu): each kernel is compared with a plain, more precise computation of the same operation, at
shapes just below, at and just above the boundary it targets.  Shapes are derived from the device's SM count, and every
GPU case asserts through lfpsqp_large_last_dispatch (Context.large_dispatch) that the path it targets is the one that ran.

References:
  Gram        integer J (DIAGQUAD with small-integer Q, A and an integer point): every product and partial sum of J J' is an
              integer below 2^53, exact in binary64 in any summation order, so G must equal numpy's J @ J.T bit for bit
  factor      componentwise backward-error bounds |G - L L'| <= c g_m |L||L'| and |L^-1 L - I| <= c g_m |L^-1||L|
  projection  r1 = J pv (tangency) and r2 = v - pv - J' lam (the removed part is J' lam with the returned multipliers)
  fused CG    the launch-per-phase loop, and a float64 CG on a Householder-QR projector (projcg!) or on J'J + mu I (pcg!)
  Jacobi      numpy's eigendecomposition of the Gram at the truncation rule of large_eig.cu
Residuals are evaluated in np.longdouble for m <= 512, in float64 with the bound doubled above that.  The unmarked tests
at the end feed the checkers corrupted copies of reference results and require each corruption to be rejected."""
import numpy as np
import pytest

from tests.test_gpu_large_bounds import bounds_for, check, diagquad_callbacks

U = np.finfo(np.float64).eps / 2
# c of the componentwise bounds.  Cholesky satisfies |G - L L'| <= g_{m+1} |L||L'| in any summation order (Higham, Accuracy
# and Stability of Numerical Algorithms, Thm 10.3), and a triangular inverse formed from products satisfies
# |X L - I| <= g_m |X||L| (ibid. 14.2).  The recursive-doubling inverse builds each off-diagonal block from two products,
# X21 = -(X22 L21) X11, which doubles the constant; 4 leaves a further factor of 2 for the extended-precision evaluation
# and for g_{m+1} vs g_m.  A dropped K chunk, a skipped block pair or a 1e-12 change of a row exceeds it by orders of magnitude.
C_BOUND = 4.0
EXT_MAX = 512          # residuals in np.longdouble up to this m, float64 with the bound doubled above
CG_TOL = 1e-9          # fixed-K CG vs the launch-per-phase loop and vs the float64 reference (kappa(H) <= 100, K <= 65)
CG_SENS_MAX = 1e-6     # largest loop-vs-reference spread at which a fixed-K CG case still judges anything
SYRK_LEAN, SYRK_EXT, SYRK_NARROW, SYRK_SKIP = 1, 2, 4, 8
SOLVE_EXPLICIT, SOLVE_TRIANGULAR, SOLVE_PINV = 1, 2, 4
FUSED_CHUNK = 64       # projcg iterations per fused launch at the default chunk (large.cu::projcg)


def gamma(k):
    return k * U / (1.0 - k * U)


def rel(a, b):
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def worst(R, B):
    """max |R| / B; an entry with B == 0 must be exactly 0"""
    R = np.abs(R)
    ok = B > 0
    r = np.where(ok, R / np.where(ok, B, 1), np.where(R != 0, np.inf, 0.0))
    return float(np.max(r)) if r.size else 0.0


def _prec(m):
    return (np.longdouble, C_BOUND) if m <= EXT_MAX else (np.float64, 2 * C_BOUND)


def factor_ratios(G, L, Linv):
    """worst |G - L L'| / (c g_m |L||L'|) and |L^-1 L - I| / (c g_m |L^-1||L|) over the lower triangle"""
    m = G.shape[0]
    T, c = _prec(m)
    Gl, Lt, Li = (np.tril(a).astype(T) for a in (G, L, Linv))
    aL, aLi = np.abs(Lt), np.abs(Li)
    r1 = worst(np.tril(Gl - Lt @ Lt.T), c * gamma(m) * np.tril(aL @ aL.T))
    r2 = worst(Li @ Lt - np.eye(m, dtype=T), c * gamma(m) * (aLi @ aL))
    return r1, r2


def projection_ratios(J, v, pv, lam):
    """r1 = J pv against c g_n (|J||v| + |J||J'||lam|) (rounding of t = J v and of the Gram solve), r2 = v - pv - J' lam
    against c g_m |J'||lam| + c u |pv| (the column pass and the final subtraction)"""
    m, n = J.shape
    T, c = _prec(m)
    Jt, vt, pt, lt = (np.asarray(a).astype(T) for a in (J, v, pv, lam))
    aJ = np.abs(Jt)
    Jl = aJ.T @ np.abs(lt)
    r1 = worst(Jt @ pt, c * gamma(n) * (aJ @ np.abs(vt) + aJ @ Jl))
    r2 = worst(vt - pt - Jt.T @ lt, c * gamma(m) * Jl + c * U * np.abs(pt))
    return r1, r2


def ref_projcg(hd, b, proj, K):
    """projcg! (projcg.jl:40-121) with c = 0, tol = 0, K iterations, on H = diag(hd) with the projector proj"""
    xs = np.zeros_like(b); r = proj(-b); d = -r; rg = r @ r
    for _ in range(K):
        Ad = hd * d; al = rg / (d @ Ad); xs = xs + al * d; rp = r + al * Ad; gp = proj(rp)
        be = (rp @ gp) / rg; d = be * d - gp; r = gp; rg = gp @ gp
    return xs


def cg_tolerance(spread):
    """Bar for a fixed-K CG result: CG_TOL, or 10 x the spread between two independent float64 implementations (the
    launch-per-phase loop and the numpy reference) where the K-step map amplifies rounding more than that.  Once the
    Krylov space has nearly converged (small n: a few hundred distinct eigenvalues), reordered sums alone move the iterate
    by ~1e-8 (B200, m = 3, n = 294, K = 65: loop vs reference 1.1e-8).  A dropped row, pass or block moves it by orders of
    magnitude more; CG_SENS_MAX keeps the bar from widening past that."""
    assert spread < CG_SENS_MAX, spread
    return max(CG_TOL, 10.0 * spread)


def ref_pcg(J, mu, b, K):
    """pcg! (retractions.jl:179-246) on (J'J + mu I) x = b from x = 0, tol = 0, K iterations"""
    x = np.zeros_like(b); r = b.copy(); p = np.zeros_like(b); rho = r @ r; rho_prev = 1.0
    for _ in range(K):
        p = r + (rho / rho_prev) * p
        z = J.T @ (J @ p) + mu * p
        al = rho / (p @ z); x = x + al * p; r = r - al * z
        rho_prev, rho = rho, r @ r
    return x


def qr_projector(J):
    Qj, _ = np.linalg.qr(J.T)
    return lambda v: v - Qj @ (Qj.T @ v)


def ragged_pairs(m, NB=64):
    """(B, B2r) of every level of the recursive-doubling inverse whose last pair is ragged (large.cu::factorize)"""
    out, B = [], NB
    while B < m:
        b2r = m - (m // (2 * B)) * 2 * B - B
        if b2r > 0:
            out.append((B, b2r))
        B *= 2
    return out


# ------------------------------------------------------------------ problem builders
def int_diagquad(L, m, n, seed, mask=None):
    """DIAGQUAD with Q, A in [-8, 8] and x in [-3, 3] (integers): J = Q o x + A is an integer matrix"""
    rng = np.random.default_rng(seed)
    Q = rng.integers(-8, 9, (m, n)).astype(np.float64)
    A = rng.integers(-8, 9, (m, n)).astype(np.float64)
    if mask is not None:
        Q *= mask; A *= mask
    x = rng.integers(-3, 4, n).astype(np.float64)
    b = 0.5 * Q @ (x * x) + A @ x
    return L.families.diagquad(Q, A, b, np.zeros(n), np.ones(n)), x, Q * x[None, :] + A


def band_mask(m, n, width):
    mask = np.zeros((m, n))
    for i in range(m):
        lo = (i * 13) % (n - width); mask[i, lo:lo + width] = 1.0
    return mask


_CG_CACHE = {}


def cg_problem(L, m, n, mmax):
    """DIAGQUAD for the fixed-K CG cases: J well conditioned (entries N(0, (1 + x^2) / n)), H = diag(w) with w in [1, 100].
    The problems of one n are the leading m of mmax rows, so one QR of the largest J' serves all of them."""
    if n not in _CG_CACHE:
        Q, A, b, xt, w, x0 = L.make_diagquad(n, mmax, seed=n, cond=100.0)
        J = Q * x0[None, :] + A
        # the Householder QR of J[:m]' is the leading part of the QR of J' (each reflector depends on its leading columns only)
        _CG_CACHE[n] = (Q, A, b, xt, w, x0, J, np.linalg.qr(J.T)[0])
    Q, A, b, xt, w, x0, J, Qfull = _CG_CACHE[n]
    Qj = Qfull[:, :m]
    fam = L.families.diagquad(Q[:m].copy(), A[:m].copy(), b[:m].copy(), xt, w)
    return fam, x0, J[:m], w, xt, (lambda v: v - Qj @ (Qj.T @ v))


# ------------------------------------------------------------------ GPU fixtures and shape helpers
@pytest.fixture(scope="module")
def L():
    import lfpsqp.jl_b200 as L
    L.default_context(0)
    return L


@pytest.fixture(scope="module")
def S():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def dim(spec, S):
    """an int, or (a, b) = a * SMs + b"""
    return spec if isinstance(spec, int) else spec[0] * S + spec[1]


def wave_m(S):
    """a ragged m (one row in the last tile row) whose lower SYRK has between SMs / 2 and SMs tiles: the wave split"""
    g = 1
    while g * (g + 1) // 2 * 2 <= S:
        g += 1
    assert g * (g + 1) // 2 < S
    return 128 * (g - 1) + 1


def ws_bytes(m):
    return max(16 * m * 64 * 8, min(m * m * 8 * 16, 1 << 30))


def lower_tiles(m):
    g, gx = -(-m // 128), -(-m // (64 if m <= 64 else 128))
    return (g * gx + g) // 2


def wave_factor(S, m, K):
    """large.cu::gemm_nt's wave split of an m x m lower SYRK over K"""
    tiles = lower_tiles(m)
    eff = lambda ks: tiles * ks / (-(-tiles * ks // S) * S)
    best = 1
    for ks in range(2, 17):
        if ks * m * (m + 1) * 8 > ws_bytes(m) or K // ks < 2048:
            break
        if eff(ks) > eff(best) + 0.02:
            best = ks
    return best


def disp(L):
    return L.default_context().large_dispatch


def syrk_bits(d):
    return d["gemm"] & 15


# ------------------------------------------------------------------ 1. Gram: exact, every SYRK branch
GRAM_CASES = [(1, 1022), (63, 1024), (64, 1026), (65, 1022), (65, 1024), (127, 1026), (128, 1024), (129, 1022),
              ((2, -1), 1024), ((2, 1), 1026), ((2, 1), 8190), ((2, -1), 8194), ("wave", 8190), ("wave", 8192), ("wave", 8194)]


@pytest.mark.gpu
@pytest.mark.parametrize("mspec,K", GRAM_CASES)
def test_gram_of_each_syrk_kernel_is_exact_at_every_branch(L, S, mspec, K):
    # factor() returns the G it factorises, from one SYRK per call: for m > 64 the scan-and-skip kernel on the first call, the
    # plain one on the next.  Both must equal J J' exactly (integer entries).
    m = wave_m(S) if mspec == "wave" else dim(mspec, S)
    fam, x, J = int_diagquad(L, m, K, seed=m + K)
    G = J @ J.T
    assert np.max(np.abs(G)) < 2.0 ** 53
    P = L.LargeProblem(fam)
    tiles = lower_tiles(m)
    grid = 2 * tiles <= S and K >= 1024
    wave = (not grid) and K >= 8192 and tiles < S
    first = None
    for call in range(2):   # first call: the SYRK scans for zero slabs and skips them; later calls know J is dense
        fac = P.factor(x)
        d = disp(L)
        assert np.array_equal(np.tril(fac["G"]), np.tril(G)), (m, K, call)
        if m <= 64:
            assert syrk_bits(d) == SYRK_NARROW
        else:
            assert syrk_bits(d) == (SYRK_SKIP if call == 0 else SYRK_LEAN), (call, d)
        assert (d["ksplit_grid"] > 1) == grid, d
        if wave:
            assert d["ksplit_wave"] == wave_factor(S, m, K) > 1, d
        else:
            assert d["ksplit_wave"] == 0, d
        assert fac["rank_deficient"] == 0
        if first is None:
            first = fac
        else:   # the dense plain SYRK and the slab-skipping one agree, and the factor does not depend on the call
            for key in ("L", "Linv"):
                assert np.array_equal(np.tril(fac[key]), np.tril(first[key])), (m, K, key)
    if m <= EXT_MAX:
        r1, r2 = factor_ratios(G, fac["L"], fac["Linv"])
        assert r1 <= 1 and r2 <= 1, (r1, r2)


@pytest.mark.gpu
@pytest.mark.parametrize("mspec", [129, (2, 1), 321])
def test_gram_skip_matches_dense_on_block_sparse_j(L, S, monkeypatch, mspec):
    # zero-slab skipping (SYRK, rows_dot, cols_dot) vs the dense kernels at ragged m: the same bits.  Integer entries, so the
    # Gram is also exact.
    m, n = dim(mspec, S), 4096
    fam, x, J = int_diagquad(L, m, n, seed=m, mask=band_mask(m, n, 600))
    v = np.random.default_rng(m).standard_normal(n)
    out = {}
    for mode in ("dense", "skip"):
        if mode == "dense":
            monkeypatch.setenv("LFPSQP_GRAM_SKIP", "0")
        P = L.LargeProblem(fam)
        fac = P.factor(x)
        d = disp(L)
        assert bool(syrk_bits(d) & SYRK_SKIP) == (mode == "skip"), d
        pv, lam = P.project(v)
        dp = disp(L)
        R = 4 if m >= 8 * S else 2 if m >= 2 * S else 1
        assert dp["rows_dot"] == (R << 3 if mode == "skip" else R), dp
        out[mode] = (fac, pv, lam)
        monkeypatch.delenv("LFPSQP_GRAM_SKIP", raising=False)
    for key in ("G", "L", "Linv"):
        assert np.array_equal(np.tril(out["skip"][0][key]), np.tril(out["dense"][0][key])), key
    assert np.array_equal(np.tril(out["skip"][0]["G"]), np.tril(J @ J.T))
    assert np.array_equal(out["skip"][1], out["dense"][1]) and np.array_equal(out["skip"][2], out["dense"][2])
    r1, r2 = projection_ratios(J, v, out["skip"][1], out["skip"][2])
    assert r1 <= 1 and r2 <= 1, (r1, r2)


# ------------------------------------------------------------------ 2. factor residuals across block and doubling boundaries
# 65, 193, 321: last pair of the B = 64 level is ragged with B2r = 1 (129, 385 at B = 128; 257, 769 at B = 256);
# 127, 255, 511: B2r = B - 1
FACTOR_MS = [1, 63, 64, 65, 127, 128, 129, 193, 255, 256, 257, 321, 385, 511, 512, 513, 769]


@pytest.mark.gpu
@pytest.mark.parametrize("m", FACTOR_MS)
def test_factor_componentwise_and_repeatable(L, m):
    n = 2048
    fam, x, J = int_diagquad(L, m, n, seed=3 * m)
    G = J @ J.T
    P = L.LargeProblem(fam)
    a = P.factor(x)
    b = P.factor(x)   # a look-ahead race between the side stream and the trailing update would show as different bits
    assert a["rank_deficient"] == 0
    for key in ("L", "Linv"):
        assert np.array_equal(np.tril(a[key]), np.tril(b[key])), key
    assert np.array_equal(np.tril(a["G"]), np.tril(G))
    r1, r2 = factor_ratios(G, a["L"], a["Linv"])
    print("m = %d ragged pairs %s: |G - LL'| %.2e, |L^-1 L - I| %.2e of the bound" % (m, ragged_pairs(m), r1, r2))
    assert r1 <= 1 and r2 <= 1, (r1, r2)


# ------------------------------------------------------------------ 3. projection
def cols_dot_split(m, n, S):
    """(row splits, rows in the last split) of the column pass (lfpsqp_large_setup)"""
    coltiles = -(-n // 512)
    want = max(1, -(-4 * S // coltiles))
    ns = max(1, min(want, max(1, m // 32), 64))
    rps = -(-m // ns)
    ns = -(-m // rps)
    return ns, m - (ns - 1) * rps


def one_row_last_split(n, S, lo=200):
    m = lo
    while cols_dot_split(m, n, S)[1] != 1:
        m += 1
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("mspec,n", [((2, -1), 4096), ((2, 1), 4096), ((8, -1), 4096), ((8, 1), 4096), ("split1", 2048),
                                     (6200, 8192)])
def test_projection_residuals(L, S, mspec, n):
    # rows_dot R = 1 / 2 / 4 across 2 SMs and 8 SMs, a column pass whose last row split has one row, and m = 6200 (the staged
    # m-vector of the triangular passes needs more than 48 KB of shared memory)
    m = one_row_last_split(n, S) if mspec == "split1" else dim(mspec, S)
    if mspec == "split1":
        assert cols_dot_split(m, n, S)[0] > 1
    Q, A, b, xt, w, x0 = L.make_diagquad(n, m, seed=m, cond=100.0)
    J = Q * x0[None, :] + A
    P = L.LargeProblem(L.families.diagquad(Q, A, b, xt, w))
    P.factor(x0, want=())
    v = np.random.default_rng(m).standard_normal(n)
    pv, lam = P.project(v)
    d = disp(L)
    R = 4 if m >= 8 * S else 2 if m >= 2 * S else 1
    assert d["rows_dot"] == R and d["solve"] == SOLVE_TRIANGULAR, d
    r1, r2 = projection_ratios(J, v, pv, lam)
    print("m = %d n = %d: r1 %.2e r2 %.2e of the bound" % (m, n, r1, r2))
    assert r1 <= 1 and r2 <= 1, (r1, r2)


@pytest.mark.gpu
@pytest.mark.parametrize("npts", [33, 101, 333])
def test_thomson_odd_column_count(L, S, monkeypatch, npts):
    # n = 3 npts odd: the SYRK's 8-byte tail, the odd tails of rows_dot / cols_dot, with and without zero-slab skipping.
    # Integer coordinates: J = 2 x is an integer matrix and the Gram is exact.
    rng = np.random.default_rng(npts)
    x = rng.integers(1, 4, 3 * npts) * rng.choice([-1.0, 1.0], 3 * npts)
    n = x.size
    J = np.zeros((npts, n))
    for i in range(npts):
        J[i, 3 * i:3 * i + 3] = 2.0 * x[3 * i:3 * i + 3]
    v = rng.standard_normal(n)
    out = {}
    for mode in ("dense", "skip"):
        if mode == "dense":
            monkeypatch.setenv("LFPSQP_GRAM_SKIP", "0")
        P = L.LargeProblem(L.families.thomson(npts))
        fac = P.factor(x)
        pv, lam = P.project(v)
        d = disp(L)
        R = 4 if npts >= 8 * S else 2 if npts >= 2 * S else 1
        assert d["rows_dot"] == (R << 3 if mode == "skip" and npts > 64 else R), d   # no zero-slab map for m <= 64
        out[mode] = (fac, pv, lam)
        monkeypatch.delenv("LFPSQP_GRAM_SKIP", raising=False)
    fac, pv, lam = out["skip"]
    assert np.array_equal(np.tril(fac["G"]), np.tril(J @ J.T))
    for key in ("L", "Linv"):
        assert np.array_equal(np.tril(fac[key]), np.tril(out["dense"][0][key])), key
    assert np.array_equal(pv, out["dense"][1]) and np.array_equal(lam, out["dense"][2])
    r1, r2 = factor_ratios(J @ J.T, fac["L"], fac["Linv"])
    assert r1 <= 1 and r2 <= 1, (r1, r2)
    r1, r2 = projection_ratios(J, v, pv, lam)
    assert r1 <= 1 and r2 <= 1, (r1, r2)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["mixed", "box"])
def test_host_family_odd_n_with_bounds_vs_oracle(L, oracle, kind):
    # host callbacks at odd n with finite bounds: J diag(Dy) (ineq_scale_cols, odd tail), the SYRK's 8-byte tail and the odd
    # tails of the streaming passes inside a whole solve
    n, m, seed = 301, 17, 2
    Q, A, b, xt, w, x0 = L.make_diagquad(n, m, seed=seed, cond=50.0)
    fam = L.families.diagquad(Q, A, b, xt, w)
    xl, xu = bounds_for(x0, seed + 10, kind)
    got = L.optimize(*diagquad_callbacks(Q, A, b, xt, w), x0, xl, xu, m, return_stats=True)
    d = disp(L)
    assert d["rows_dot"] == 1 and d["solve"] & SOLVE_TRIANGULAR and d["fused_single"] == d["fused_general"] == 0, d
    orc = oracle.optimize("diagquad", n, m, 0, x0, xl=xl, xu=xu, fam_params=fam.params)
    with oracle.variant("fma"):
        orc_fma = oracle.optimize("diagquad", n, m, 0, x0, xl=xl, xu=xu, fam_params=fam.params)
    check(got, orc, orc_fma)


# ------------------------------------------------------------------ 4. fused projcg! and pcg!
# (m, n, K): the row phase's passes of 16 rows per CTA (m around 16 SMs and past 32 SMs), odd m (the solve phase's tail),
# n / 2 at the 2048-pair chunk of the row phase and one pair either side, fewer column pairs than CTAs, K across a chunk
FUSED_CASES = [((16, -1), 8192, 65), ((16, 0), 8192, 65), ((16, 1), 8192, 65), ((32, 1), 10240, 65), (3, 4094, 65),
               (129, 4096, 64), (129, 4096, 65), (129, 4098, 65), (3, (2, -2), 65), (129, (2, -2), 65)]


def fused_mmax(n, S):
    return max(dim(c[0], S) for c in FUSED_CASES if dim(c[1], S) == n)


def _fused_id(c):
    f = lambda s: str(s) if isinstance(s, int) else "%dS%+d" % s
    return "m%s-n%s-K%d" % (f(c[0]), f(c[1]), c[2])


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["explicit", "triangular"])
@pytest.mark.parametrize("case", FUSED_CASES, ids=_fused_id)
def test_fused_projcg_boundaries(L, S, monkeypatch, case, form):
    ms, ns, K = case
    m, n = dim(ms, S), dim(ns, S)
    fam, x0, J, w, xt, proj = cg_problem(L, m, n, fused_mmax(n, S))
    res = {}
    for path in ("fused", "unfused"):
        if path == "unfused":
            monkeypatch.setenv("LFPSQP_FUSED_PROJCG", "0")
        if form == "triangular":
            monkeypatch.setenv("LFPSQP_EXPLICIT_INVERSE", "0")
        P = L.LargeProblem(fam)
        assert P.factor(x0, want=())["rank_deficient"] == 0
        out = P.projcg(x0, lam=np.zeros(m), tol=0.0, maxit=K)
        d = disp(L)
        monkeypatch.delenv("LFPSQP_FUSED_PROJCG", raising=False)
        monkeypatch.delenv("LFPSQP_EXPLICIT_INVERSE", raising=False)
        assert out["iters"] == K and out["status"] == 4, out
        launches = -(-K // FUSED_CHUNK)
        if path == "unfused":
            assert d["fused_single"] == d["fused_general"] == 0, d
        elif form == "explicit":
            assert d["fused_single"] == launches and d["fused_general"] == 0 and d["solve"] & SOLVE_EXPLICIT, d
        else:
            assert d["fused_general"] == launches and d["fused_single"] == 0 and not d["solve"] & SOLVE_EXPLICIT, d
        res[path] = out["sol"]
    ref = ref_projcg(w, proj(-(w * (x0 - xt))), proj, K)
    e_loop, e_ref, spread = rel(res["fused"], res["unfused"]), rel(res["fused"], ref), rel(res["unfused"], ref)
    print("m = %d n = %d K = %d %s: vs loop %.2e, vs QR reference %.2e, loop vs reference %.2e"
          % (m, n, K, form, e_loop, e_ref, spread))
    tol = cg_tolerance(spread)
    assert e_loop < tol and e_ref < tol, (e_loop, e_ref, tol)


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c for c in FUSED_CASES if c[2] == 65], ids=lambda c: _fused_id(c).rsplit("-K", 1)[0])
def test_fused_pcg_boundaries(L, S, monkeypatch, case):
    ms, ns, _ = case
    m, n = dim(ms, S), dim(ns, S)
    fam, x0, J, w, xt, proj = cg_problem(L, m, n, fused_mmax(n, S))
    K, mu = 24, 1e-2
    rhs = np.random.default_rng(n).standard_normal(n)
    res = {}
    for path in ("fused", "unfused"):
        if path == "unfused":
            monkeypatch.setenv("LFPSQP_FUSED_PROJCG", "0")
        P = L.LargeProblem(fam)
        x, r, flag, it = P.pcg(x0, mu, rhs, tol=0.0, maxiter=K)
        d = disp(L)
        monkeypatch.delenv("LFPSQP_FUSED_PROJCG", raising=False)
        assert it == K and flag == 1
        assert d["fused_pcg"] == (1 if path == "fused" else 0), d
        res[path] = x
    ref = ref_pcg(J, mu, rhs, K)
    e_loop, e_ref, spread = rel(res["fused"], res["unfused"]), rel(res["fused"], ref), rel(res["unfused"], ref)
    print("pcg m = %d n = %d: vs loop %.2e, vs reference %.2e, loop vs reference %.2e" % (m, n, e_loop, e_ref, spread))
    tol = cg_tolerance(spread)
    assert e_loop < tol and e_ref < tol, (e_loop, e_ref, tol)


# ------------------------------------------------------------------ 5. Jacobi pseudo-inverse
def pinv_reference(J, eps_rank=1e-10):
    """G^+ at large_eig.cu's rule: keep lambda_k >= max(eps_rank^2, 1e-13 lambda_max)"""
    lam, V = np.linalg.eigh(J @ J.T)
    keep = lam >= max(eps_rank ** 2, 1e-13 * lam.max())
    return (V[:, keep] / lam[keep]) @ V[:, keep].T, int(np.sum(~keep))


@pytest.mark.gpu
@pytest.mark.parametrize("mspec,zero_row", [(129, False), (129, True), ((4, 48), False), ((4, 48), True)])
def test_jacobi_pseudo_inverse(L, S, monkeypatch, mspec, zero_row):
    # odd m (the round-robin tournament's dummy player), more pairs than CTAs (m > 2 x the 2-SM grid), an all-zero
    # constraint row (den = 0), two groups of duplicated rows
    m, n = dim(mspec, S), 2048
    Q, A, b, xt, w, x0 = L.make_diagquad(n, m, seed=m, cond=50.0)
    for k in range(8):            # group 1: the last 8 rows repeat rows 0..7
        Q[m - 8 + k] = Q[k]; A[m - 8 + k] = A[k]; b[m - 8 + k] = b[k]
    for k in (21, 22):            # group 2: row 20 three times
        Q[k] = Q[20]; A[k] = A[20]; b[k] = b[20]
    if zero_row:
        Q[10] = 0.0; A[10] = 0.0; b[10] = 0.0
    J = Q * x0[None, :] + A
    Gp, defect = pinv_reference(J)
    assert defect == 10 + (1 if zero_row else 0)
    fam = L.families.diagquad(Q, A, b, xt, w)
    P = L.LargeProblem(fam)
    assert P.factor(x0, want=())["rank_deficient"] == defect
    v = np.random.default_rng(1).standard_normal(n)
    pv, lam = P.project(v)
    assert disp(L)["solve"] == SOLVE_PINV
    lam_ref = Gp @ (J @ v)
    assert rel(pv, v - J.T @ lam_ref) < 1e-10 and rel(lam, lam_ref) < 1e-8
    assert np.linalg.norm(J @ pv) < 1e-9 * np.linalg.norm(v)
    tol = 1e-8 * np.max(np.abs(lam))
    assert np.allclose(lam[:8], lam[m - 8:], rtol=0, atol=tol)          # minimum-norm multipliers: copies share equally
    assert np.allclose(lam[21:23], lam[20], rtol=0, atol=tol)
    if zero_row:
        assert lam[10] == 0.0                                           # a null row is never rotated: its multiplier is 0
    # fused projcg applies G^+ through the explicit-inverse kernel; the launch-per-phase loop through its own pass
    K = 12
    a = P.projcg(x0, lam=np.zeros(m), tol=0.0, maxit=K)
    d = disp(L)
    assert d["fused_single"] == 1 and d["solve"] & SOLVE_PINV, d
    monkeypatch.setenv("LFPSQP_FUSED_PROJCG", "0")
    P2 = L.LargeProblem(fam)
    P2.factor(x0, want=())
    b_ = P2.projcg(x0, lam=np.zeros(m), tol=0.0, maxit=K)
    assert disp(L)["fused_single"] == 0
    assert a["iters"] == b_["iters"] == K and rel(a["sol"], b_["sol"]) < CG_TOL
    assert np.linalg.norm(J @ a["sol"]) < 1e-9 * np.linalg.norm(a["sol"])


# ------------------------------------------------------------------ the checkers reject corrupted results (no GPU)
def _exact_reference(m=129, n=1024, seed=5):
    rng = np.random.default_rng(seed)
    J = (rng.integers(-8, 9, (m, n)) * rng.integers(-3, 4, n) + rng.integers(-8, 9, (m, n))).astype(np.float64)
    G = J @ J.T
    Lc = np.linalg.cholesky(G)
    return J, G, Lc, np.linalg.inv(Lc)


def test_checkers_accept_reference_results():
    J, G, Lc, Li = _exact_reference()
    r1, r2 = factor_ratios(G, Lc, Li)
    assert r1 <= 1 and r2 <= 1, (r1, r2)
    v = np.random.default_rng(0).standard_normal(J.shape[1])
    lam = np.linalg.solve(G, J @ v)
    r1, r2 = projection_ratios(J, v, v - J.T @ lam, lam)
    assert r1 <= 1 and r2 <= 1, (r1, r2)


def test_checkers_reject_a_dropped_k_chunk():
    # one 16-column K chunk missing from one 128 x 128 tile of the SYRK: the Gram is no longer exact, and L no longer factors it
    J, G, Lc, Li = _exact_reference()
    Gc = G.copy()
    Gc[:128, :128] -= J[:128, 512:528] @ J[:128, 512:528].T
    assert not np.array_equal(np.tril(Gc), np.tril(J @ J.T))
    assert factor_ratios(Gc, Lc, Li)[0] > 1
    Lbad = np.linalg.cholesky(Gc[:128, :128])       # a consistent factor of the corrupted tile: the residual vs G rejects it
    L2 = Lc.copy(); L2[:128, :128] = Lbad
    assert factor_ratios(G, L2, np.linalg.inv(L2))[0] > 1


def test_checkers_reject_a_perturbed_ragged_row_of_the_inverse():
    # the last row of m = 129 (the ragged pair of the B = 128 level, B2r = 1), relative change 1e-12
    J, G, Lc, Li = _exact_reference()
    assert ragged_pairs(129) == [(128, 1)]
    Lb = Li.copy()
    Lb[128, :] *= 1.0 + 1e-12
    assert factor_ratios(G, Lc, Lb)[1] > 1


def test_checkers_reject_a_missing_second_row_pass():
    # one t_i of the second row pass of the fused kernel (row 16 x SMs, with 8 SMs here) left at zero in every projection
    m, n, K = 16 * 8 + 3, 512, 65
    rng = np.random.default_rng(3)
    J = rng.standard_normal((m, n)) / np.sqrt(n)
    w = np.exp(rng.uniform(0.0, np.log(100.0), n))
    bvec = rng.standard_normal(n)
    good = qr_projector(J)
    G = J @ J.T
    i = 16 * 8 + 1

    def bad(v):
        t = J @ v; t[i] = 0.0
        return v - J.T @ np.linalg.solve(G, t)
    ref = ref_projcg(w, good(bvec), good, K)
    assert rel(ref_projcg(w, good(bvec), good, K), ref) < CG_TOL     # deterministic reference
    assert rel(ref_projcg(w, good(bvec), bad, K), ref) > 10 * CG_SENS_MAX   # rejected at the widest bar cg_tolerance allows
    v = rng.standard_normal(n)
    t = J @ v; t[i] = 0.0
    lam = np.linalg.solve(G, t)
    assert projection_ratios(J, v, v - J.T @ lam, lam)[0] > 1
