"""One-GPU benchmark of the sparse QCQP family in large-n mode, on a problem of the size a user would pose:

    f      = 1/2 x'(L + 0.01 I)x + q.x        L = 5-point Laplacian on a 512 x 512 grid (n = 262,144)
    c_i    = Ac_i.x - bc_i = 0                512 sparse rows, about 256 non-zeros each
    d_k    = 1/2 |x_Bk|^2 - 1/2 <= 0          512 balls on disjoint 64-variable blocks (slack variables, as data)
    -1 <= x_j <= 1                           on every tenth variable

Reports the device solve in each storage of the constraint Jacobian (jacobian="dense" and "csr", alternated --rounds times
in one process: wall time, lfpsqp_large_phase_ms split, projcg iterations per second, the Gram's device time, bytes per
projcg iteration from shapes and the resulting share of HBM bandwidth, and the largest difference between the two
solutions), and the same problem through host callbacks (optimize_slack), capped at --host-maxiter outer iterations
(0 skips it).  A second problem only the CSR storage can hold ("beyond dense"):

    f      = 1/2 (x - xt)' diag(w) (x - xt)   n = 2^24, w in [1, 2]
    c      = 2000 sparse linear rows of 64 entries, 47 spheres |x_Bk|^2 = const on 4096-variable blocks, sum(x) = s   (m = 2048)

whose dense J would take 275 GB; its setup time, solve time and the device memory setup took are reported.  GPU name and
power limit are read in the same run.  Writes one JSON file (default profiles/sparse_qcqp_bench_1gpu.json).

    python tools/sparse_qcqp_bench.py [--out PATH] [--jacobian dense|csr|both] [--rounds R] [--host-maxiter K] [--no-beyond]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import scipy.sparse as sp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_TBPS = 7.7   # HGX B200 data sheet, one GPU


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return dict(gpu=name, power_limit=power)
    except Exception as e:   # the number is still stated, with what is known about the card
        return dict(gpu="unknown (%s)" % e, power_limit="unknown")


def problem(L, k=512, m=512, nnz_row=256, p=512, block=64, seed=0):
    rng = np.random.default_rng(seed)
    n = k * k
    T = sp.diags([-np.ones(k - 1), 2.0 * np.ones(k), -np.ones(k - 1)], [-1, 0, 1])
    P = (sp.kron(sp.identity(k), T) + sp.kron(T, sp.identity(k)) + 0.01 * sp.identity(n)).tocsr()
    Ac = sp.random(m, n, density=nnz_row / n, random_state=seed, format="csr")
    x0 = 0.01 * rng.standard_normal(n)
    Qd = []
    for b in range(p):
        idx = np.arange(b * block, (b + 1) * block)
        Qd.append(sp.coo_matrix((np.ones(block), (idx, idx)), shape=(n, n)))
    fam = L.families.sparse_qcqp(P=P, q=rng.standard_normal(n), Ac=Ac, bc=Ac @ x0, Qd=Qd, bd=0.5 * np.ones(p))
    xl, xu = -np.inf * np.ones(n), np.inf * np.ones(n)
    xl[::10], xu[::10] = -1.0, 1.0
    return fam, x0, xl, xu


def bytes_per_projcg_iter(aug, jacobian):
    """bytes one projcg iteration moves, from shapes: the two passes over J (dense: all of the m x n array twice; CSR:
    values, 32-bit indices and pointers of the CSR row pass and the CSC column pass, one gathered read of the source vector
    per entry and one write of each result) and the CSR pass over the assembled Lagrangian Hessian"""
    na, ma = aug.n, aug.m
    nnz_h = int(np.unique(np.concatenate([aug.P[0] * na + aug.P[1], aug.Qc[1] * na + aug.Qc[2]])).size)
    h_bytes = nnz_h * 12 + (na + 1) * 4 + 2 * na * 8
    if jacobian == "dense":
        j_bytes = 2 * ma * na * 8
    else:
        nnz_j = int(np.unique(np.concatenate([aug.Ac[0] * na + aug.Ac[1], aug.Qc[0] * na + aug.Qc[1]])).size)
        rows = nnz_j * (8 + 4 + 8) + (ma + 1) * 4 + ma * 8
        cols = nnz_j * (8 + 4 + 8) + (na + 1) * 4 + na * 8
        j_bytes = rows + cols
    return dict(J_passes=j_bytes, H_spmv=h_bytes, total=j_bytes + h_bytes, nnz_H=nnz_h)


def run_storage(L, ctx, fam, x0, xl, xu, jacobian):
    aug, x0a, xla, xua = fam.slack_embedding(x0, xl, xu)
    aug = L.families.SparseQCQPFamily(aug.n, aug.m, 0, aug.P, aug.q, aug.r, aug.Qc, aug.Ac, aug.bc, aug.Qd, aug.Ad, aug.bd,
                                      jacobian=jacobian)
    t0 = time.perf_counter()
    prob = L.LargeProblem(aug, ctx=ctx)
    setup = time.perf_counter() - t0
    prob.factor(x0a, want=())                                      # warm-up of the Gram
    gram_ms = prob.factor(x0a, want=())["gram_ms"]                 # device time of J J' (the solve's Gram is J diag(Dy^2) J')
    prob.set_bounds(xla, xua)
    param = L.LFPSQPParams()
    prob.solve(x0a, param, return_stats=True)                      # warm-up: module loads, first allocations
    t0 = time.perf_counter()
    x, obj, lam, info, stats, status = prob.solve(x0a, param, return_stats=True)
    wall = time.perf_counter() - t0
    ph = prob.phase_ms()
    it = stats["projcg_iters"]
    its = it / (ph["projcg"] / 1e3) if ph["projcg"] > 0 else float("nan")
    b = bytes_per_projcg_iter(aug, jacobian)
    res = dict(wall_s=wall, setup_s=setup, phase_ms=ph, gram_ms=gram_ms, iterations=info.iter, condition=info.condition.name,
               status=status, stats=stats, objective=float(obj[-1]), projcg_iters_per_s=its, bytes_per_projcg_iter=b,
               projcg_hbm_share=b["total"] * its / (HBM_TBPS * 1e12), s_per_outer_iteration=wall / max(info.iter, 1),
               max_equality_violation=float(np.max(np.abs(_c(fam, x[:fam.n])))), max_ball_violation=float(np.max(fam.d_values(x[:fam.n]))))
    del prob
    return res, x[:fam.n]


def beyond_dense(L, ctx, seed=20):
    """the CSR-only problem of the module docstring: setup time, solve time and the device memory setup took"""
    import torch
    n, nlin, nsph, blk = 1 << 24, 2000, 47, 4096
    rng = np.random.default_rng(seed)
    x0 = rng.standard_normal(n)
    Alin = sp.csr_matrix((rng.standard_normal(nlin * 64), (np.repeat(np.arange(nlin), 64), rng.integers(0, n, nlin * 64))),
                         shape=(nlin, n))
    Alin.sum_duplicates()
    Ac = sp.vstack([Alin, sp.csr_matrix((nsph, n)), sp.csr_matrix(np.ones((1, n)))]).tocsr()
    Qc = [sp.coo_matrix((n, n))] * nlin
    for k in range(nsph):
        idx = np.arange(k * blk, (k + 1) * blk)
        Qc.append(sp.coo_matrix((np.ones(blk), (idx, idx)), shape=(n, n)))
    Qc.append(sp.coo_matrix((n, n)))
    blocks = [x0[k * blk:(k + 1) * blk] for k in range(nsph)]
    bc = np.concatenate([Alin @ x0, [0.5 * b @ b for b in blocks], [x0.sum()]])
    w = 1.0 + rng.random(n)
    xt = x0 + 1e-2 * rng.standard_normal(n)
    fam = L.families.sparse_qcqp(P=sp.diags(w), q=-w * xt, r=0.5 * np.sum(w * xt * xt), Qc=Qc, Ac=Ac, bc=bc, jacobian="csr")
    nnz_j = int(fam.Ac[2].size) + nsph * blk
    torch.cuda.synchronize()
    free0, total = torch.cuda.mem_get_info(0)
    t0 = time.perf_counter()
    prob = L.LargeProblem(fam, ctx=ctx)
    setup = time.perf_counter() - t0
    free1, _ = torch.cuda.mem_get_info(0)
    t0 = time.perf_counter()
    x, obj, lam, info, stats, status = prob.solve(x0, return_stats=True)
    solve = time.perf_counter() - t0
    ph = prob.phase_ms()
    del prob
    return dict(n=n, m=fam.m, nnz_J=nnz_j, dense_J_bytes=8 * fam.m * n, csr_csc_bytes=nnz_j * (2 * 8 + 3 * 4) + 4 * (n + 1),
                setup_s=setup, setup_device_bytes=int(free0 - free1), solve_s=solve, phase_ms=ph, iterations=info.iter,
                condition=info.condition.name, status=status, stats=stats, objective=float(obj[-1]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sparse_qcqp_bench_1gpu.json"))
    ap.add_argument("--jacobian", choices=("dense", "csr", "both"), default="both")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--host-maxiter", type=int, default=3)
    ap.add_argument("--no-beyond", action="store_true")
    a = ap.parse_args()
    import lfpsqp.jl_b200 as L
    ctx = L.default_context(0)
    res = gpu_info()
    t0 = time.perf_counter()
    fam, x0, xl, xu = problem(L)
    res["build_problem_s"] = time.perf_counter() - t0
    n, m, p = fam.n, fam.m, fam.p
    res["shape"] = dict(n=n, m=m, p=p, n_working=n + p, m_working=m + p, nnz_P=int(fam.P[2].size), nnz_Ac=int(fam.Ac[2].size),
                        nnz_Qd=int(fam.Qd[3].size), bounded=int(np.isfinite(xl).sum()))
    storages = ("dense", "csr") if a.jacobian == "both" else (a.jacobian,)
    runs = {s: [] for s in storages}
    xs = {}
    for _ in range(a.rounds):                                      # alternated: the storages see the same machine state
        for s in storages:
            r, xs[s] = run_storage(L, ctx, fam, x0, xl, xu, s)
            runs[s].append(r)
    res["device"] = {s: dict(runs=runs[s], wall_s_min=min(r["wall_s"] for r in runs[s]),
                             projcg_iters_per_s_max=max(r["projcg_iters_per_s"] for r in runs[s]),
                             gram_ms_min=min(r["gram_ms"] for r in runs[s])) for s in storages}
    if len(storages) == 2:
        d = xs["dense"] - xs["csr"]
        res["max_abs_x_difference"] = float(np.max(np.abs(d)))
        res["rel_x_difference"] = float(np.linalg.norm(d) / np.linalg.norm(xs["dense"]))
    if a.host_maxiter > 0:
        # the same problem through host callbacks (lfpsqp_solve_host: dense m x n Jc uploaded per jac!, one host round trip
        # per projcg iteration), capped at --host-maxiter outer iterations
        cb = fam.callbacks()
        hp = L.LFPSQPParams(maxiter=a.host_maxiter)
        t0 = time.perf_counter()
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            hx, hobj, hlam, hinfo = L.optimize_slack(cb["f"], cb["grad"], cb["hess_vec"], cb["c"], cb["jac"], cb["chess_vec"],
                                                     cb["d"], cb["djac"], cb["dhess_vec"], -np.inf * np.ones(p), np.zeros(p), x0, xl,
                                                     xu, m, p, hp)
        hwall = time.perf_counter() - t0
        res["host_callbacks"] = dict(wall_s=hwall, iterations=hinfo.iter, capped_at=a.host_maxiter, condition=hinfo.condition.name,
                                     s_per_outer_iteration=hwall / max(hinfo.iter, 1), objective=float(hobj[-1]))
    if not a.no_beyond and "csr" in storages:
        res["beyond_dense"] = beyond_dense(L, ctx)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1, default=float)
    print(json.dumps(res, default=float))


def _c(fam, x):
    c = np.zeros(fam.m)
    fam.callbacks()["c"](c, x)
    return c


if __name__ == "__main__":
    main()
