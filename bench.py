#!/usr/bin/env python
"""bench.py -- headline benchmark of the LFPSQP hot path on B200 (contract: see the task's bench section).

A "step" is one pass of the hot path over one batch of synthetic input: BASELINE.json config C2, the README
inequality example batched (n=50, p=1, 65,536 independent instances per GPU, seeded N(0,1) coefficients).
    value : instances solved / s, whole job, inputs already resident in HBM (lfpsqp_solve_batched_dev)
    e2e   : the same through the host-buffer C-ABI call (pinned host memory; H2D + kernel + D2H inside the timed region)
Multi-GPU: the path shards by instances with no collective (weak scaling: every rank solves its own B instances).
`--impl reference` times the CPU oracle port of the reference (Julia is absent from this image) on all host cores.
`--dump-outputs DIR` writes what the last timed step returned for rank 0's instances (x, obj_values, obj_len, lambda,
term_*) as DIR/<name>.npy in float64, about 39 MB, all finite; the inputs are seeded, so two builds can be compared file
for file.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

N_VARS = 50
B_PER_GPU = 65536
HIST = 16
SEED = 0
METRIC = "SQP instances solved/sec (batched, README inequality example n=50 p=1)"
UNIT = "instances/s"


def make_inputs(rank, B):
    rng = np.random.Generator(np.random.Philox(key=SEED + 1000 * rank))
    coeff = rng.standard_normal((B, N_VARS))
    x0 = np.zeros((B, N_VARS))
    return coeff, x0


def dump_outputs(d, x, obj, olen, lam, term):
    """One batched solve's results as float64 .npy files.  The solver leaves obj entries past an instance's history
    length unwritten (it always records f(x0), so the length is at least 1): they are stored as the last recorded
    objective, which keeps every value finite and loses nothing next to obj_len."""
    os.makedirs(d, exist_ok=True)
    H = obj.shape[1]
    obj = obj[np.arange(obj.shape[0])[:, None], np.minimum(np.arange(H)[None, :], np.minimum(olen, H)[:, None] - 1)]
    out = {"x": x, "obj_values": obj, "obj_len": olen, "lambda": lam}
    out.update({"term_" + k: term[k] for k in term.dtype.names})
    for k, v in out.items():
        np.save(os.path.join(d, k + ".npy"), np.asarray(v, dtype=np.float64))


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_oracle_rate(coeff, x0, seconds_target=12.0, nthreads=None):
    """Times the CPU oracle (port of the reference, analytic derivatives) on a bounded sample of the workload."""
    from oracle import oracle as O
    nthreads = nthreads or host_cores()
    n = N_VARS
    inf = np.inf * np.ones(n)
    # calibrate
    S = min(2048, coeff.shape[0])
    t0 = time.perf_counter()
    O.optimize_batched("readme_ineq", n, 0, 1, x0[:S], xl=-inf, xu=inf, fam_params=coeff[:S], fam_stride=n, H=HIST,
                       nthreads=nthreads)
    dt = time.perf_counter() - t0
    S2 = int(min(coeff.shape[0], max(S, S * seconds_target / max(dt, 1e-3))))
    t0 = time.perf_counter()
    out = O.optimize_batched("readme_ineq", n, 0, 1, x0[:S2], xl=-inf, xu=inf, fam_params=coeff[:S2], fam_stride=n,
                             H=HIST, nthreads=nthreads)
    dt = time.perf_counter() - t0
    flops = float(out[5]["flops"].mean())
    return S2 / dt, S2, nthreads, dt, flops


class ClockSampler:
    def __init__(self, gpu_index):
        self.rows = []
        self.stop = False
        self.gpu = gpu_index
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.th = threading.Thread(target=self._read, daemon=True)
        self.th.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def finish(self, t_begin, t_end):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, line in self.rows:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                mhz = float(parts[0]); smax = float(parts[1])
            except ValueError:
                continue
            if t_begin - 0.05 <= t <= t_end + 0.05:
                sm.append(mhz)
                for nm, v in zip(names, parts[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def _traffic(kernel, key):
    """DRAM bytes of `kernel` from the committed ncu --set full capture (profiles/traffic.json), or None."""
    try:
        return float(json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[kernel][key])
    except Exception:
        return None


def large_n_section(L, ctx, torch, dev, with_cpu, dist=None, rank=0, world=1, weak=False):
    """Secondary metric of BASELINE.json: large-n projcg iterations/s on config C5 (n=65536, m=2048 dense random
    diagonal-quadratic equality constraints, definition pinned in DESIGN.md), fixed-K projcg (tol=0) through the
    unit-level export, plus the FP64 DMMA Gram.  Inputs are generated on the device (2 GB of parameters).
    With world > 1 the instance is column-sharded (strong scaling): NCCL all-reduces the Gram, J v and the CG scalars."""
    from lfpsqp.jl_b200 import dist as D
    n, m, K = 65536 * (world if weak else 1), 2048, 64
    col0, nloc = D.column_range(n, world, rank)
    if world > 1 and ctx.lib.lfpsqp_comm_mode(ctx.h) == 0:
        D.init_comm(ctx, dist)
    g = torch.Generator(device=dev); g.manual_seed(SEED)     # same stream on every rank; each keeps its column shard

    def shard_rand():
        full = torch.randn((m, n), dtype=torch.float64, device=dev, generator=g) / np.sqrt(n)
        return full[:, col0:col0 + nloc].contiguous()
    Q = shard_rand(); A = shard_rand()
    x0 = torch.randn(n, dtype=torch.float64, device=dev, generator=g)[col0:col0 + nloc].contiguous()
    xt = torch.randn(n, dtype=torch.float64, device=dev, generator=g)[col0:col0 + nloc]
    w = torch.exp(torch.rand(n, dtype=torch.float64, device=dev, generator=g) * np.log(1e4))[col0:col0 + nloc]
    b = 0.5 * Q @ (x0 * x0) + A @ x0
    if world > 1:
        dist.all_reduce(b)
    blob = torch.cat([Q.reshape(-1), A.reshape(-1), b, xt, w]).contiguous()
    del Q, A
    torch.cuda.synchronize()
    fam = L.families.Family(L.families.DIAGQUAD, "diagquad", n, m, 0)
    P = L.LargeProblem(fam, ctx, col0=col0, n_loc=nloc, n_global=n, params_dev_ptr=blob.data_ptr())
    x0h = x0.cpu().numpy()
    lam0 = np.zeros(m)
    gram_ms = []
    for _ in range(3):
        gram_ms.append(P.factor(x0h, want=())["gram_ms"])
    gram_ms = float(np.min(gram_ms[1:]))
    for _ in range(3):  # warm-up
        P.projcg(x0h, lam=lam0, tol=0.0, maxit=8, chunk=16, want_solution=False)
    per = []
    launches = 0
    for _ in range(5):
        if world > 1:
            dist.barrier()
        r = P.projcg(x0h, lam=lam0, tol=0.0, maxit=K, chunk=16, want_solution=False)
        assert r["iters"] == K
        ms = r["ms"]
        if world > 1:   # device time, max over ranks
            t = torch.tensor([ms], dtype=torch.float64, device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item())
        per.append(ms / K)
        launches = ctx.last_launches
    ms_it = float(np.median(per))
    # the retraction's inner loop: pcg! (retractions.jl:179-246) on (J'J + mu I) dx = b, fixed 100 iterations (tol = 0)
    rhs = np.random.default_rng(5 + rank).standard_normal(nloc)
    pcg_per = []
    pcg_launches = 0
    for rep in range(4):
        if world > 1:
            dist.barrier()
        _, _, _, pit = P.pcg(x0h, 1e-2, rhs, tol=0.0, maxiter=100)
        ms = ctx.last_kernel_ms / max(pit, 1) * 100.0    # normally all 100 iterations run (tol = 0)
        if world > 1:
            tt = torch.tensor([ms], dtype=torch.float64, device=dev); dist.all_reduce(tt, op=dist.ReduceOp.MAX); ms = float(tt.item())
        if rep > 0:
            pcg_per.append(ms / 100)
        pcg_launches = ctx.last_launches
    pcg_ms = float(np.median(pcg_per))
    pcg_bytes = 16.0 * m * nloc + 96.0 * nloc     # two passes over J + 12 vector sweeps (p, r, z, dx)
    bytes_it = 16.0 * m * nloc + 8.0 * m * m + 104.0 * nloc   # per GPU; SURVEY.md 8(d): two passes over J + two triangular GEMVs + vector sweeps
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    ach = bytes_it / (ms_it * 1e-3) / 1e9
    out = {"metric": "large-n projcg iterations/s", "value": 1e3 / ms_it, "unit": "iterations/s",
           "config": {"workload": "C5 large dense: n=65536, m=2048, c_i = 1/2 sum_j Q_ij x_j^2 + A_i.x - b_i, "
                                  "f = 1/2 (x-xt)' diag(w) (x-xt), fixed K=%d projcg iterations (tol=0), column-sharded over %d GPU(s)" % (K, world),
                      "scaling": ("weak (n = 65536 per GPU, m fixed)" if weak else "strong (total work fixed, J and x sharded by columns)"),
                      "n": n, "comm": {0: "none", 1: "NCCL", 2: "peer-memory all-reduce kernels (CUDA IPC over NVLink) + NCCL for the Gram"}[ctx.lib.lfpsqp_comm_mode(ctx.h)],
                      "l2": "J alone is 1 GiB per pass (>> 126 MB L2)"},
           "ms_per_iteration": ms_it, "gpu_launches_per_iteration": launches / K,
           "roofline": {"bound": "hbm", "kernels": ("fused_projcg_kernel (persistent cooperative kernel: grid barriers, in-kernel peer-memory all-reduce)"
                                                    if launches / K < 1.0 else "rows_dot_kernel + cols_dot_kernel (+ tri_gemv, cg_update*)"),
                        "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm,
                        "algorithmic_bytes_per_iteration_per_gpu": bytes_it,
                        "traffic": (_traffic("fused_projcg_kernel" if launches / K < 1.0 else "rows_dot_kernel+cols_dot_kernel", "bytes_per_iteration")
                                    if (world == 1 and not weak) else None),
                        "peak_source": "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"}}
    out["retraction_pcg"] = {"metric": "ProjPenalty pcg! iterations/s (retractions.jl:179-246)", "value": 1e3 / pcg_ms, "unit": "iterations/s",
                             "ms_per_iteration": pcg_ms, "gpu_launches_per_iteration": pcg_launches / 100.0,
                             "roofline": {"bound": "hbm", "kernel": ("fused_pcg_kernel (one cooperative launch per pcg! call)" if pcg_launches < 50
                                                                     else "pcg_a + rows_dot + cols_dot + pcg_z + pcg_x"),
                                          "achieved": pcg_bytes / (pcg_ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                                          "frac": pcg_bytes / (pcg_ms * 1e-3) / 1e9 / hbm, "algorithmic_bytes_per_iteration_per_gpu": pcg_bytes,
                                          "traffic": (_traffic("fused_pcg_kernel", "bytes_per_iteration") if (world == 1 and not weak) else None)}}
    try:
        dmma = ctx.fp64_peak("dmma")
        flops = float(m) * (m + 1) * nloc
        out["gram"] = {"kernel": "dgemm_nt_kernel<128> (SYRK, lower tiles, mma.sync.m8n8k4.f64)", "ms": gram_ms, "flops": flops,
                       "bound": "tensor", "achieved": flops / (gram_ms * 1e-3) / 1e12, "peak": dmma, "unit": "TFLOP/s",
                       "frac": flops / (gram_ms * 1e-3) / 1e12 / dmma,
                       "peak_source": "DMMA (mma.sync.m8n8k4.f64) microbenchmark measured in this run",
                       "peak_method": "lfpsqp_bench_fp64_peak(which=1), csrc/microbench.cu: 148*8 CTAs x 256 threads, 4096 iterations of "
                                      "32 register-only mma.sync.m8n8k4.f64 per warp (4 independent accumulator pairs), 512 flops "
                                      "per instruction per warp, CUDA-event timed, best of 3 after one warm-up"}
    except Exception as e:  # noqa
        out["gram"] = {"error": str(e)}
    if with_cpu:
        # CPU baseline: the ORACLE's own projcg! (oracle/lfpsqp_oracle.cpp::projcg, src/projcg.jl:40-121) on a C5-shaped
        # problem -- orthonormal n x m basis U (the reference's SVD factor; made here by a QR on the GPU, which is setup,
        # not timed), diagonal Lagrangian Hessian with the benchmark's spectrum, fixed iteration count (tol = 0).
        from oracle import oracle as O
        Uq = torch.linalg.qr(torch.randn((n, m), dtype=torch.float64, device=dev, generator=g)).Q
        Uh = Uq.T.contiguous().cpu().numpy().T          # (n, m) column-major, as the reference holds U
        del Uq
        hdh = np.exp(np.random.default_rng(2).uniform(0.0, np.log(1e4), n))
        bh = np.random.default_rng(3).standard_normal(n)
        bh -= Uh @ (Uh.T @ bh)
        t0 = time.perf_counter(); O.projcg_diag(hdh, Uh, bh, np.zeros(m), tol=0.0, maxit=3); t3 = time.perf_counter() - t0
        kc = int(max(4, min(64, 10.0 / max(t3 / 3, 1e-3))))
        t0 = time.perf_counter()
        _, _, itc, _ = O.projcg_diag(hdh, Uh, bh, np.zeros(m), tol=0.0, maxit=kc)
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": itc / dt, "unit": "iterations/s", "cores": 1, "kind": "port",
                               "sample": "%d iterations of the oracle's projcg! (scalar C++ port of src/projcg.jl) on a C5-shaped problem: "
                                         "orthonormal %dx%d basis, diagonal Hessian, %.1f s" % (itc, n, m, dt)}
        del Uh
    del blob
    return out


def c4_sharded_section(L, ctx, dist, rank, world):
    """BASELINE config C4 (Thomson N = 4096, n = 12288, m = 4096, dense-treated J) column-sharded over `world` GPUs: whole
    points per rank, x / v all-gathered per callback evaluation (SURVEY.md 8e-iv); first 10 outer iterations of the real solve."""
    import warnings
    from lfpsqp.jl_b200 import dist as D
    npts = 4096
    rng = np.random.Generator(np.random.Philox(key=SEED + 4))
    p0 = rng.standard_normal((npts, 3)); p0 /= np.linalg.norm(p0, axis=1, keepdims=True); p0 = p0.ravel()
    col0, nloc = D.thomson_point_range(npts, world, rank)
    P = L.LargeProblem(L.families.thomson(npts), ctx, col0=col0, n_loc=nloc, n_global=3 * npts)
    best = None
    for rep in range(2):
        dist.barrier()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            t0 = time.perf_counter()
            x, obj, lam, info, st, status = P.solve(p0[col0:col0 + nloc], L.LFPSQPParams(maxiter=10, disp=L.off), return_stats=True)
            wall = time.perf_counter() - t0
        if best is None or wall < best[0]:
            best = (wall, P.phase_ms(), st, float(obj[0]), float(obj[-1]), status)
    return {"workload": "Thomson N=4096 column-sharded over %d GPUs (whole points per rank), first 10 outer iterations, default params" % world,
            "wall_s": best[0], "phase_ms": best[1], "stats": best[2], "f_first_last": [best[3], best[4]], "status": best[5],
            "note": "the m x m Cholesky / triangular inverse is replicated on every rank (only the Gram partials shard), so the "
                    "factorisation bounds the scaling of this configuration"}


def extras_section(L, ctx, torch, dev, with_cpu):
    """Parity-test configurations of BASELINE.json reported as extra lines (not the headline): C3 Rosenbrock batched
    (1,048,576 instances, thread-per-instance kernel) and C4 Thomson N=4096 (n=12288, m=4096, J treated dense as the
    reference does) -- first 10 outer iterations of the real solve, split by phase."""
    import ctypes as C
    from lfpsqp.jl_b200 import _lib
    out = {}
    # ---- C3
    B = 1 << 20
    rng = np.random.Generator(np.random.Philox(key=SEED + 3))
    x0 = rng.uniform(-2.0, 2.0, (B, 2)); x0[0] = 0.0            # instance 0 = the README start (golden vector)
    H = 64
    d_x0 = torch.from_numpy(x0).to(dev); d_x = torch.empty((B, 2), dtype=torch.float64, device=dev)
    d_obj = torch.empty((B, H), dtype=torch.float64, device=dev); d_len = torch.empty(B, dtype=torch.int64, device=dev)
    d_lam = torch.empty((B, 1), dtype=torch.float64, device=dev); d_term = torch.empty(B * 40, dtype=torch.uint8, device=dev)
    prm = L.LFPSQPParams(disp=L.off).to_c(); pprm = C.cast(C.pointer(prm), C.c_void_p)
    ms = []
    for k in range(6):
        ctx.check(ctx.lib.lfpsqp_solve_batched_dev(ctx.h, L.families.ROSENBROCK, 2, 0, 0, B, None, 0, d_x0.data_ptr(), None, None, pprm,
                                                   d_x.data_ptr(), d_obj.data_ptr(), H, d_len.data_ptr(), d_lam.data_ptr(), d_term.data_ptr(), None))
        if k >= 2:
            ms.append(ctx.last_kernel_ms)
    lens = d_len.cpu().numpy()
    term0 = np.frombuffer(d_term[:40].cpu().numpy().tobytes(), dtype=_lib.TERM_DTYPE)[0]
    kms = float(np.median(ms))
    io = float(B * (16 + 16 + 8 + 40) + 8 * np.minimum(lens, H).sum())
    out["c3_rosenbrock_batched"] = {"metric": "SQP instances solved/sec", "value": B / (kms * 1e-3), "unit": UNIT, "instances": B,
                                    "kernel": "batched_tiny_kernel<FamRosenbrock,2> (one thread per instance)", "kernel_ms": kms,
                                    "mean_outer_iterations": float(lens.mean() - 1),
                                    "golden_instance0": {"iter": int(term0["iter"]), "condition": int(term0["condition"]), "f_diff": float(term0["f_diff"])},
                                    "hbm_io_gbs": io / (kms * 1e-3) / 1e9}
    try:   # binding roof of the thread-per-instance kernel: FP64 issue (HBM sees 0.05 of its peak)
        from oracle import oracle as O
        fl = float(O.optimize_batched("rosenbrock", 2, 0, 0, x0[:1 << 14], H=H, nthreads=host_cores())[5]["flops"].mean())
        dfma = ctx.fp64_peak("dfma")
        out["c3_rosenbrock_batched"]["roofline"] = {"bound": "fp64-issue", "flops_per_instance": fl, "achieved": fl * B / (kms * 1e-3) / 1e12,
                                                    "peak": dfma, "unit": "TFLOP/s", "frac": fl * B / (kms * 1e-3) / 1e12 / dfma,
                                                    "peak_source": "DFMA microbenchmark measured in this run",
                                                    "note": "algorithmic flops = the oracle's instrumented FP64 op count; n = 2, so the work per "
                                                            "instance is divisions, square roots and branches of the driver, not vector arithmetic"}
    except Exception as e:  # noqa
        out["c3_rosenbrock_batched"]["roofline"] = {"error": repr(e)}
    if with_cpu:
        from oracle import oracle as O
        S = 1 << 17
        t0 = time.perf_counter()
        O.optimize_batched("rosenbrock", 2, 0, 0, x0[:S], H=H, nthreads=host_cores())
        dt = time.perf_counter() - t0
        out["c3_rosenbrock_batched"]["cpu_baseline"] = {"value": S / dt, "unit": UNIT, "cores": host_cores(), "kind": "port",
                                                        "sample": "%d of the %d instances" % (S, B)}
    del d_x0, d_x, d_obj, d_len, d_lam, d_term
    # ---- C4
    npts = 4096
    rng = np.random.Generator(np.random.Philox(key=SEED + 4))
    p0 = rng.standard_normal((npts, 3)); p0 /= np.linalg.norm(p0, axis=1, keepdims=True)
    P = L.LargeProblem(L.families.thomson(npts), ctx)
    gram_ms = min(P.factor(p0.ravel(), want=())["gram_ms"] for _ in range(2))
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        t0 = time.perf_counter()
        x, obj, lam, info, st, status = P.solve(p0.ravel(), L.LFPSQPParams(maxiter=10, disp=L.off), return_stats=True)
        wall = time.perf_counter() - t0
    ph = P.phase_ms()
    n, m = 3 * npts, npts
    bytes_it = 16.0 * m * n + 8.0 * m * m + 104.0 * n
    it_s = st["projcg_iters"] / (ph["projcg"] * 1e-3) if ph["projcg"] > 0 else None
    out["c4_thomson_4096"] = {"workload": "Thomson N=4096: n=12288, m=4096, dense J (402 MB), first 10 outer iterations, default params",
                              "outer_iterations": info.iter, "wall_s": wall, "phase_ms": ph, "stats": st, "status": status,
                              "f_first_last": [float(obj[0]), float(obj[-1])],
                              "gram": {"ms": gram_ms, "dense_equivalent_tflops": m * (m + 1.0) * n / (gram_ms * 1e-3) / 1e12,
                                       "note": "J is stored dense (402 MB) but Thomson's rows are block-sparse: one scan marks the all-zero "
                                               "64 x 16 slabs and the SYRK skips them (bit-identical result); the dense-equivalent rate is "
                                               "not a tensor-pipe figure -- the dense Gram roofline is the C5 number under large_n"},
                              "projcg_iterations_per_s_in_solve": it_s,
                              "projcg_roofline_frac_in_solve": (bytes_it * it_s / 1e9 / 6543.4) if it_s else None,
                              "note": "in-solve projcg rate includes the start-up projection, Thomson's O(N^2) pairwise Hessian kernel and one host sync per chunk"}
    return out


def run_reference(args):
    """Reference arm: the reference's CPU implementation of the path = the oracle port (kind "port"), all host threads,
    same config/metric; one step = all instances of one GPU-arm step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    coeff, x0 = make_inputs(0, B_PER_GPU)
    from oracle import oracle as O
    nthreads = host_cores()
    n = N_VARS
    inf = np.inf * np.ones(n)
    S = B_PER_GPU  # one step = the whole instance set of the GPU arm's step (0.2 s on 16 host threads): same config, and the
                   # threads are not starved by small slices (8192-instance slices ran at 0.6x this rate)
    for _ in range(max(1, min(args.warmup, 2))):
        O.optimize_batched("readme_ineq", n, 0, 1, x0[:1024], xl=-inf, xu=inf, fam_params=coeff[:1024], fam_stride=n,
                           H=HIST, nthreads=nthreads)
    t0 = time.perf_counter()
    for k in range(args.steps):
        lo = (k * S) % (B_PER_GPU - S + 1)
        res = O.optimize_batched("readme_ineq", n, 0, 1, x0[lo:lo + S], xl=-inf, xu=inf, fam_params=coeff[lo:lo + S],
                                 fam_stride=n, H=HIST, nthreads=nthreads)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *res[:5])
    value = S * args.steps / dt
    sample = "%d of the %d instances per step, %d steps, %d host threads" % (S, B_PER_GPU, args.steps, nthreads)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "C2 README inequality example batched: n=50, p=1, m=0, x0=0, coeff~N(0,1) seeded",
                       "instances_per_step": S, "note": "Julia is not installed in this image; the reference arm is the "
                       "CPU oracle port of LFPSQP.jl (analytic derivatives, same dgesvd), i.e. faster than the AD-based original"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": nthreads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def bind_to_gpu_cpus(gpu_index):
    """N ranks x 90 MB of pinned traffic per step: keep every rank's host buffers and its calling thread on the CPU socket its
    GPU hangs off (NVML's ideal CPU affinity), so that the copies do not cross the socket interconnect."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        before = len(os.sched_getaffinity(0))
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return {"method": "nvmlDeviceSetCpuAffinity", "cpus_before": before, "cpus": len(os.sched_getaffinity(0))}
    except Exception as e:  # noqa
        return {"method": "none", "error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip-large", action="store_true", help="skip the secondary large-n (C5) section")
    ap.add_argument("--no-numa-bind", action="store_true", help="N > 1: do not bind each rank to the CPUs next to its GPU (A/B)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results for rank 0's instances as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import ctypes as C
    import lfpsqp.jl_b200 as L
    from lfpsqp.jl_b200 import _lib

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    host_placement = None
    if world > 1 and not args.no_numa_bind:
        host_placement = bind_to_gpu_cpus(local_rank)   # before the pinned buffers are allocated (first touch = local node)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        cpu_group = dist.new_group(backend="gloo")   # host-side waits (an NCCL barrier would keep a kernel spinning on the idle GPUs)
    dev = torch.device("cuda", local_rank)
    ctx = L.Context(local_rank)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)

    B, n, H = B_PER_GPU, N_VARS, HIST
    coeff, x0 = make_inputs(rank, B)
    inf = np.inf * np.ones(n)
    xl = -inf; xu = inf
    prm = L.LFPSQPParams(disp=L.off).to_c()
    pprm = C.cast(C.pointer(prm), C.c_void_p)

    # ---- device-resident buffers (torch owns the memory; the library gets raw pointers)
    d_coeff = torch.from_numpy(coeff).to(dev); d_x0 = torch.from_numpy(x0).to(dev)
    d_x = torch.empty((B, n), dtype=torch.float64, device=dev); d_obj = torch.empty((B, H), dtype=torch.float64, device=dev)
    d_len = torch.empty(B, dtype=torch.int64, device=dev); d_lam = torch.empty((B, 1), dtype=torch.float64, device=dev)
    d_term = torch.empty(B * 40, dtype=torch.uint8, device=dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # 256 MiB > 126 MB L2

    def step_dev():
        rc = ctx.lib.lfpsqp_solve_batched_dev(ctx.h, L.families.README_INEQ, n, 0, 1, B, d_coeff.data_ptr(), n,
                                              d_x0.data_ptr(), _lib.ptr(xl), _lib.ptr(xu), pprm, d_x.data_ptr(),
                                              d_obj.data_ptr(), H, d_len.data_ptr(), d_lam.data_ptr(), d_term.data_ptr(), None)
        ctx.check(rc)

    # ---- pinned host buffers for the end-to-end arm
    def pinned(shape, dtype):
        t = torch.empty(shape, dtype=dtype).pin_memory()
        return t, t.numpy()
    _, h_coeff = pinned((B, n), torch.float64); h_coeff[:] = coeff
    _, h_x0 = pinned((B, n), torch.float64); h_x0[:] = x0
    _, h_x = pinned((B, n), torch.float64); _, h_obj = pinned((B, H), torch.float64)
    _, h_len = pinned((B,), torch.int64); _, h_lam = pinned((B, 1), torch.float64)
    _, h_term = pinned((B * 40,), torch.uint8)
    h2d = h_coeff.nbytes + h_x0.nbytes
    d2h = h_x.nbytes + h_obj.nbytes + h_len.nbytes + h_lam.nbytes + h_term.nbytes

    def step_e2e():
        rc = ctx.lib.lfpsqp_solve_batched(ctx.h, L.families.README_INEQ, n, 0, 1, B, _lib.ptr(h_coeff), n, _lib.ptr(h_x0),
                                          _lib.ptr(xl), _lib.ptr(xu), pprm, _lib.ptr(h_x), _lib.ptr(h_obj), H,
                                          _lib.ptr(h_len), _lib.ptr(h_lam), _lib.ptr(h_term), None)
        ctx.check(rc)
        return float(h_obj[0, 0])  # the step's result is read on the host

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if dist is None:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- warm-up
    for _ in range(max(args.warmup, 3)):
        step_dev()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)

    # ---- timed: K steps, device events around every step, L2 flushed between steps (flush not timed)
    K = args.steps
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    kern_ms = []
    barrier()
    t_begin = time.perf_counter()
    for k in range(K):
        flush.zero_()
        ev[k][0].record(stream)
        step_dev()
        ev[k][1].record(stream)
        kern_ms.append(ctx.last_kernel_ms)
    barrier()
    t_end = time.perf_counter()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = max_over_ranks(float(sum(step_ms)))
    value = world * B * K / (total_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_x.cpu().numpy(), d_obj.cpu().numpy(), d_len.cpu().numpy(), d_lam.cpu().numpy(),
                     np.frombuffer(d_term.cpu().numpy().tobytes(), dtype=_lib.TERM_DTYPE))

    # ---- end-to-end through the host-buffer C-ABI call (pinned host memory, copies inside the timed region)
    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for k in range(K):
        step_e2e()
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_value = world * B * K / e2e_s
    e2e_modes = {"per_process": e2e_value}
    if world > 1:
        # the same end-to-end step as ONE host call: rank 0 owns a multi-GPU context (lfpsqp_ctx_create_multi) over all N
        # devices and lfpsqp_solve_batched shards the N*B instances inside the library (one host thread + stream pipeline
        # per device, no collective); the other ranks only wait.
        barrier()
        dist.barrier(group=cpu_group)
        one_call = 0.0
        if rank == 0:
            mc = L.MultiContext(list(range(world)))
            BW = world * B
            call = [make_inputs(r, B) for r in range(world)]
            _, g_coeff = pinned((BW, n), torch.float64); g_coeff[:] = np.concatenate([c[0] for c in call])
            _, g_x0 = pinned((BW, n), torch.float64); g_x0[:] = 0.0
            _, g_x = pinned((BW, n), torch.float64); _, g_obj = pinned((BW, H), torch.float64)
            _, g_len = pinned((BW,), torch.int64); _, g_lam = pinned((BW, 1), torch.float64)
            _, g_term = pinned((BW * 40,), torch.uint8)

            def step_one():
                rc = mc.lib.lfpsqp_solve_batched(mc.h, L.families.README_INEQ, n, 0, 1, BW, _lib.ptr(g_coeff), n, _lib.ptr(g_x0),
                                                 _lib.ptr(xl), _lib.ptr(xu), pprm, _lib.ptr(g_x), _lib.ptr(g_obj), H,
                                                 _lib.ptr(g_len), _lib.ptr(g_lam), _lib.ptr(g_term), None)
                mc.check(rc)
                return float(g_obj[0, 0])
            for _ in range(2):
                step_one()
            t0 = time.perf_counter()
            for k in range(K):
                step_one()
            one_call = BW * K / (time.perf_counter() - t0)
            assert np.array_equal(g_x[:B], h_x), "multi-GPU one-call result differs from the per-process result"
            mc.close()
        dist.barrier(group=cpu_group)     # the other ranks wait on the host: their GPUs are driven by rank 0's context meanwhile
        barrier()
        e2e_modes["one_call_multi_ctx"] = max_over_ranks(one_call)
        e2e_value = max(e2e_modes.values())
    clocks = sampler.finish(t_begin, t_end) if rank == 0 else None

    # ---- roofline of the dominant (only) kernel: batched_reg_kernel<SepReadmeIneq,2,1,true> (register-resident warp solver)
    d_len_h = d_len.cpu().numpy()
    io_bytes = float(B * (n * 8 + n * 8 + n * 8 + 8 + 8 + 40) + 8 * np.minimum(d_len_h, H).sum())  # coeff,x0 in; x,len,lam,term,obj out
    kms = float(np.mean(kern_ms))
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    achieved = io_bytes / (kms * 1e-3) / 1e9
    hbm_roof = {"bound": "hbm (NOT binding)", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                "peak_source": peak_src, "io_bytes_per_instance": io_bytes / B,
                "note": "per-instance state lives on-chip; HBM only sees the instance I/O"}
    # the BINDING roof of this kernel is FP64 issue: algorithmic flops = the oracle's instrumented FP64 operation count per
    # instance (mean over a sample of the same instance set) against the DFMA peak measured in this run by
    # lfpsqp_bench_fp64_peak (csrc/microbench.cu: 8 independent DFMA chains per thread, 2 flops per DFMA, every SM full,
    # CUDA-event timed) -- MEASURED_PEAKS.json carries no FP64 figure
    from oracle import oracle as O
    S_fl = min(4096, B)
    flops = float(O.optimize_batched("readme_ineq", n, 0, 1, x0[:S_fl], xl=-inf, xu=inf, fam_params=coeff[:S_fl], fam_stride=n, H=HIST,
                                     nthreads=host_cores())[5]["flops"].mean())
    try:
        dfma = ctx.fp64_peak("dfma")
    except Exception:  # noqa
        dfma = float("nan")
    ach_tf = flops * B / (kms * 1e-3) / 1e12
    roofline = {"bound": "fp64-issue", "kernel": "batched_reg_kernel<SepReadmeIneq, LW=8 lanes/instance, NPL=7, ME=1, INEQ, SPARSE> "
                                                 "(register-resident, 4 instances per warp)",
                "achieved": ach_tf, "peak": dfma, "unit": "TFLOP/s", "frac": ach_tf / dfma,
                "traffic": _traffic("batched_reg_kernel", "bytes_per_launch"), "kernel_ms": kms,
                "flops_per_instance": flops, "peak_source": "DFMA microbenchmark measured in this run (lfpsqp_bench_fp64_peak)",
                "peak_method": "lfpsqp_bench_fp64_peak(which=0), csrc/microbench.cu: 148*8 CTAs x 256 threads, 4096 iterations of 64 "
                               "DFMA per thread in 8 independent chains, 2 flops per DFMA, CUDA-event timed, best of 3 after one "
                               "warm-up; flops_per_instance = the oracle's instrumented FP64 operation count (mean of 4096 instances)",
                "hbm": hbm_roof}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": max(args.warmup, 3),
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": "C2 README inequality example batched: n=50, p=1, m=0, x0=0, coeff~N(0,1) seeded "
                                   "(Philox), working size N=102, M=52 after slack+bound embedding",
                       "instances_per_gpu": B, "history": H, "params": "defaults (src/LFPSQP.jl:57-81)",
                       "l2": "256 MiB buffer written between timed iterations (flush not timed)",
                       "parallelism": "instances sharded over %d GPU(s), no collective" % world},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "modes": e2e_modes, "host_placement": host_placement,
                    "note": "bytes are per GPU per step; value = best of the listed ways to drive N GPUs through the C ABI "
                            "(one process per GPU, or one host call on a multi-GPU context)"},
            "gpu_launches": int(K), "clocks": clocks, "roofline": roofline}

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        rate, S2, nth, dt, flops = cpu_oracle_rate(coeff, x0)
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": nth, "kind": "port",
                                "sample": "%d of the %d instances, %.1f s, one instance per thread" % (S2, B, dt)}
    if not args.skip_large:
        try:
            line["large_n"] = large_n_section(L, ctx, torch, dev, (not args.no_cpu_baseline) and world == 1 and rank == 0,
                                              dist, rank, world)
            if world > 1:
                line["large_n_weak"] = large_n_section(L, ctx, torch, dev, False, dist, rank, world, weak=True)
                line["c4_thomson_sharded"] = c4_sharded_section(L, ctx, dist, rank, world)
        except Exception as e:  # noqa
            line["large_n"] = {"error": repr(e)}
    if world == 1 and not args.skip_large:
        try:
            line["extras"] = extras_section(L, ctx, torch, dev, not args.no_cpu_baseline)
        except Exception as e:  # noqa
            line["extras"] = {"error": repr(e)}
    try:   # per-instance parity verdict of the last full-size GPU sweep (tests/test_gpu_parity_fullsize.py)
        pr = json.load(open(os.path.join(ROOT, "profiles", "parity_r2.json")))
        line["parity"] = {"verdict": pr.get("parity"), "failures_total": pr.get("failures_total"),
                          "records": {k: {q: r.get(q) for q in ("instances", "within_tolerance", "within_tolerance_frac", "outside_tolerance",
                                                                 "tagged_rounding_sensitive", "failures", "x_err_max", "f_err_max")}
                                      for k, r in pr.get("records", {}).items()},
                          "source": "profiles/parity_r2.json (copy of the record written by pytest -m gpu on a B200)"}
    except Exception:  # noqa
        line["parity"] = None
    if rank == 0:
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
