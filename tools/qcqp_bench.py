"""Dense QCQP family (LFPSQP_FAM_QCQP) in batched mode: two workloads on either side of the data-path question.

  S1  shared matrices: orthogonality-constrained trace minimisation, X 16 x 3 (n = 48, m = 6); P = I3 (x) A and the six
      Qc matrices are shared by the batch, only x0 varies per instance.  The matrices stay in L2 for the whole launch.
  S2  per-instance matrices: trust-region subproblems, n = 32, p = 1; P (SPD), q and bd = Delta^2/2 per instance,
      Qd = I shared.  Every instance streams its own 8 KB P from HBM.

For each: the device-resident rate (lfpsqp_solve_batched_dev) and kernel time, the end-to-end rate through the host
entry point (copies and the symmetry check included), the FP64 share of the measured DFMA peak (algorithmic flops =
the instrumented count of the CPU oracle with the family added, tests/qcqp_reference.py, on a sample), the matrix
bytes each instance reads in Hessian and Jacobian products (from the solver's counters; f and c evaluations not
counted) over kernel time, and that CPU oracle on every host core.

    python tools/qcqp_bench.py [--B 65536] [--reps 5] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def stiefel(n, k):
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


def s1(B, rng):
    nrow, k = 16, 3
    A = rng.standard_normal((nrow, nrow)); A = 0.5 * (A + A.T)
    Qc, bc = stiefel(nrow, k)
    x0 = np.linalg.qr(rng.standard_normal((B, nrow, k)))[0].transpose(0, 2, 1).reshape(B, nrow * k)
    return dict(name="S1 Stiefel trace minimisation (shared P, Qc)", n=nrow * k, m=len(bc), p=0, x0=np.ascontiguousarray(x0),
                arrays=dict(P=np.kron(np.eye(k), A), Qc=Qc, bc=bc))


def s2(B, rng):
    n = 32
    G = rng.standard_normal((B, n, n))
    P = G @ G.transpose(0, 2, 1) / n + 0.5 * np.eye(n)
    q = rng.standard_normal((B, n))
    delta = rng.uniform(0.2, 2.0, B)
    x0 = 0.1 * delta[:, None] * rng.standard_normal((B, n)) / np.sqrt(n)
    return dict(name="S2 trust-region subproblems (per-instance P, q, bd)", n=n, m=0, p=1, x0=x0,
                arrays=dict(P=P, q=q, Qd=np.eye(n)[None], bd=(0.5 * delta ** 2)[:, None]))


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [s.strip() for s in out.split(",")]
        return dict(gpu=name, power_limit=power, sm_max_clock=clk)
    except Exception as e:   # the numbers below stay valid; only the label is missing
        return dict(gpu_query_error=repr(e))


def run(w, L, O, reps):
    import torch
    n, m, p, x0 = w["n"], w["m"], w["p"], w["x0"]
    B = x0.shape[0]
    fam = L.families.qcqp(**w["arrays"])
    inf = np.inf * np.ones(n)
    args = [fam.f, fam.c] + ([fam.d] if p else []) + [x0] + ([-inf, inf] if p else []) + [m] + ([p] if p else [])
    ctx = L.default_context()
    H = 64
    # end-to-end through the host entry point
    host = L.optimize_batched(*args, history=H, return_stats=True)
    t0 = time.perf_counter()
    for _ in range(reps):
        L.optimize_batched(*args, history=H)
    e2e = (time.perf_counter() - t0) / reps
    # device-resident
    dev = {k: torch.from_numpy(a).cuda() for k, (a, _) in fam.arrays.items()}
    desc = L._lib.CQcqp()
    for k, (a, per) in fam.arrays.items():
        setattr(desc, k, dev[k].data_ptr()); setattr(desc, k + "_stride", a[0].size if per else 0)
    dx0 = torch.from_numpy(x0).cuda()
    xo = torch.empty((B, n), dtype=torch.float64, device="cuda"); obj = torch.empty((B, H), dtype=torch.float64, device="cuda")
    olen = torch.empty(B, dtype=torch.int64, device="cuda"); lam = torch.empty((B, max(m + p, 1)), dtype=torch.float64, device="cuda")
    term = torch.empty((B, 40), dtype=torch.uint8, device="cuda")
    cp = L.LFPSQPParams().to_c()
    xl = L._lib.ptr(-inf) if p else None
    xu = L._lib.ptr(inf) if p else None
    keep = (-inf, inf)

    def dev_call():
        ctx.check(ctx.lib.lfpsqp_solve_batched_dev(ctx.h, L.families.QCQP, n, m, p, B, C.cast(C.pointer(desc), C.c_void_p), 0,
                                                   dx0.data_ptr(), xl, xu, C.cast(C.pointer(cp), C.c_void_p), xo.data_ptr(),
                                                   obj.data_ptr(), H, olen.data_ptr(), lam.data_ptr(), term.data_ptr(), None))
    torch.cuda.synchronize()
    dev_call()
    t0 = time.perf_counter(); kms = []
    for _ in range(reps):
        dev_call(); kms.append(ctx.last_kernel_ms)
    dt = (time.perf_counter() - t0) / reps
    del keep
    assert np.array_equal(xo.cpu().numpy(), host[0]), "host and device-resident entry points disagree"
    kernel = ctx.last_kernel
    kms = float(np.median(kms))
    # algorithmic flops (oracle count) and CPU reference on a sample
    S = min(B, 2048)
    fp, stride = O.qcqp_params(n, m, p, B=S, **{k: (a[:S] if per else a) for k, (a, per) in fam.arrays.items()})
    cores = os.cpu_count() or 1
    t0 = time.perf_counter()
    orc = O.optimize_batched("qcqp", n, m, p, x0[:S], xl=-inf if p else None, xu=inf if p else None, fam_params=fp,
                             fam_stride=stride, H=H, nthreads=cores)
    cpu_rate = S / (time.perf_counter() - t0)
    flops = float(orc[5]["flops"].mean())
    dfma = ctx.fp64_peak("dfma")
    st = host[5]
    nmat_h = (1 if "P" in fam.arrays else 0) + (m if "Qc" in fam.arrays else 0) + (p if "Qd" in fam.arrays else 0)
    nmat_j = (m if "Qc" in fam.arrays else 0) + (p if "Qd" in fam.arrays else 0)
    hess = float(st["projcg_iters"].mean()); jac = float((st["factorizations"] + st["retract_outer"]).mean())
    mbytes = (hess * nmat_h + jac * nmat_j) * n * n * 8.0
    per_instance_matrix_bytes = sum(a[0].nbytes for a, per in fam.arrays.values() if per)
    return dict(workload=w["name"], B=B, n=n, m=m, p=p, kernel=list(kernel),
                shared=[k for k, (a, per) in fam.arrays.items() if not per],
                per_instance=[k for k, (a, per) in fam.arrays.items() if per],
                dev_instances_per_s=B / dt, dev_call_ms=dt * 1e3, kernel_ms=kms, kernel_instances_per_s=B / (kms * 1e-3),
                e2e_instances_per_s=B / e2e, e2e_call_ms=e2e * 1e3,
                iterations_mean=float(host[4]["iter"].mean()), hess_products_mean=hess, jac_products_mean=jac,
                flops_per_instance=flops, achieved_tflops=flops * B / (kms * 1e-3) / 1e12, dfma_peak_tflops=dfma,
                fp64_share_of_dfma_peak=flops * B / (kms * 1e-3) / 1e12 / dfma,
                matrix_bytes_per_instance=mbytes, matrix_read_GBps=mbytes * B / (kms * 1e-3) / 1e9,
                per_instance_input_bytes=per_instance_matrix_bytes,
                unique_input_GBps=per_instance_matrix_bytes * B / (kms * 1e-3) / 1e9,
                oracle_sample=S, oracle_threads=cores, oracle_instances_per_s=cpu_rate,
                speedup_dev_vs_oracle=(B / dt) / cpu_rate)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import lfpsqp.jl_b200 as L
    from tests import qcqp_reference as O   # the CPU oracle with the QCQP family added
    L.default_context(0)
    rng = np.random.default_rng(0)
    res = dict(info=gpu_info(), results=[run(w, L, O, a.reps) for w in (s1(a.B, rng), s2(a.B, rng))])
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
