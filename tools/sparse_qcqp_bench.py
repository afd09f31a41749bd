"""One-GPU benchmark of the sparse QCQP family in large-n mode, on a problem of the size a user would pose:

    f      = 1/2 x'(L + 0.01 I)x + q.x        L = 5-point Laplacian on a 512 x 512 grid (n = 262,144)
    c_i    = Ac_i.x - bc_i = 0                512 sparse rows, about 256 non-zeros each
    d_k    = 1/2 |x_Bk|^2 - 1/2 <= 0          512 balls on disjoint 64-variable blocks (slack variables, as data)
    -1 <= x_j <= 1                           on every tenth variable

Reports the device solve (wall time, lfpsqp_large_phase_ms split, projcg iterations per second, bytes per projcg iteration
from shapes and the resulting share of HBM bandwidth) and the same problem through host callbacks (optimize_slack), the
only route such a problem had before; that route is capped at --host-maxiter outer iterations.  GPU name and power limit
are read in the same run.  Writes one JSON file (default profiles/sparse_qcqp_bench_1gpu.json).

    python tools/sparse_qcqp_bench.py [--out PATH] [--host-maxiter K]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sparse_qcqp_bench_1gpu.json"))
    ap.add_argument("--host-maxiter", type=int, default=3)
    a = ap.parse_args()
    import lfpsqp.jl_b200 as L
    ctx = L.default_context(0)
    res = gpu_info()
    t0 = time.perf_counter()
    fam, x0, xl, xu = problem(L)
    aug, x0a, xla, xua = fam.slack_embedding(x0, xl, xu)
    res["build_problem_s"] = time.perf_counter() - t0
    n, m, p = fam.n, fam.m, fam.p
    na, ma = aug.n, aug.m
    res["shape"] = dict(n=n, m=m, p=p, n_working=na, m_working=ma, nnz_P=int(fam.P[2].size), nnz_Ac=int(fam.Ac[2].size),
                        nnz_Qd=int(fam.Qd[3].size), bounded=int(np.isfinite(xl).sum()))
    t0 = time.perf_counter()
    prob = L.LargeProblem(aug, ctx=ctx)
    prob.set_bounds(xla, xua)
    res["setup_s"] = time.perf_counter() - t0
    param = L.LFPSQPParams()
    prob.solve(x0a, param, return_stats=True)                      # warm-up: module loads, first allocations
    t0 = time.perf_counter()
    x, obj, lam, info, stats, status = prob.solve(x0a, param, return_stats=True)
    wall = time.perf_counter() - t0
    ph = prob.phase_ms()
    it = stats["projcg_iters"]
    # bytes of one projcg iteration from shapes: the two passes over the dense m x n J of the working problem (J v and
    # J' u; with bounds the passes are not skipped), and the CSR pass over the assembled Lagrangian Hessian (values,
    # 32-bit column indices, row pointers, one gathered read of the source vector and one write of the result)
    nnz_h = int(np.unique(np.concatenate([aug.P[0] * na + aug.P[1], aug.Qc[1] * na + aug.Qc[2]])).size)
    j_bytes = 2 * ma * na * 8
    h_bytes = nnz_h * 12 + (na + 1) * 4 + 2 * na * 8
    per_it = j_bytes + h_bytes
    its = it / (ph["projcg"] / 1e3) if ph["projcg"] > 0 else float("nan")
    res["device"] = dict(wall_s=wall, phase_ms=ph, iterations=info.iter, condition=info.condition.name, status=status,
                         stats=stats, objective=float(obj[-1]), projcg_iters_per_s=its, nnz_H=nnz_h,
                         bytes_per_projcg_iter=dict(J_passes=j_bytes, H_spmv=h_bytes, total=per_it),
                         projcg_hbm_share=per_it * its / (HBM_TBPS * 1e12),
                         max_equality_violation=float(np.max(np.abs(_c(fam, x)))),
                         max_ball_violation=float(np.max(fam.d_values(x))))
    # the same problem through host callbacks (lfpsqp_solve_host: dense m x n Jc uploaded per jac!, one host round trip per
    # projcg iteration), capped at --host-maxiter outer iterations
    cb = fam.callbacks()
    hp = L.LFPSQPParams(maxiter=a.host_maxiter)
    t0 = time.perf_counter()
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        hx, hobj, hlam, hinfo = L.optimize_slack(cb["f"], cb["grad"], cb["hess_vec"], cb["c"], cb["jac"], cb["chess_vec"], cb["d"],
                                                 cb["djac"], cb["dhess_vec"], -np.inf * np.ones(p), np.zeros(p), x0, xl, xu, m, p, hp)
    hwall = time.perf_counter() - t0
    res["host_callbacks"] = dict(wall_s=hwall, iterations=hinfo.iter, capped_at=a.host_maxiter, condition=hinfo.condition.name,
                                 s_per_outer_iteration=hwall / max(hinfo.iter, 1), objective=float(hobj[-1]))
    res["device"]["s_per_outer_iteration"] = wall / max(info.iter, 1)
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
