"""ctypes binding of liblfpsqp_b200.so -- exactly the C ABI of include/lfpsqp_b200.h (what Julia's ccall binds).

There is no CPU fallback: a missing library or a missing GPU raises."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LFPSQP_LIB_PATH") or os.path.join(_HERE, "liblfpsqp_b200.so")


class CParams(C.Structure):  # lfpsqp_params == LFPSQPParams, src/LFPSQP.jl:57-81
    _fields_ = [("alpha", C.c_double), ("beta", C.c_double), ("t_beta", C.c_int64), ("s", C.c_double),
                ("sigma", C.c_double), ("eps_c", C.c_double), ("eps_f", C.c_double), ("eps_x", C.c_double),
                ("eps_kkt", C.c_double), ("eps_rank", C.c_double), ("maxiter", C.c_int64),
                ("maxiter_retract", C.c_int64), ("maxiter_pcg", C.c_int64), ("mu0", C.c_double),
                ("disable_linesearch", C.c_int32), ("do_project_retract", C.c_int32), ("disp", C.c_int32),
                ("linesearch", C.c_int32), ("do_newton", C.c_int32), ("_pad", C.c_int32),
                ("tn_maxiter", C.c_int64), ("tn_kappa", C.c_double), ("callback_period", C.c_int64)]


QCQP_FIELDS = ("P", "q", "r", "Qc", "Ac", "bc", "Qd", "Ad", "bd")


class CQcqp(C.Structure):  # lfpsqp_qcqp: nine {const double*, int64 batch stride} pairs
    _fields_ = [f for name in QCQP_FIELDS for f in ((name, C.c_void_p), (name + "_stride", C.c_int64))]


TERM_DTYPE = np.dtype([("condition", "<i4"), ("status", "<i4"), ("f_diff", "<f8"), ("step_diff", "<f8"),
                       ("kkt_diff", "<f8"), ("iter", "<i8")])
STATS_FIELDS = ("projcg_iters", "projcg_negcurv", "armijo_trials", "retract_outer", "retract_pcg", "pp_backtracks",
                "newton_accepted", "factorizations", "f_evals", "flag_last")
STATS_DTYPE = np.dtype([(k, "<i8") for k in STATS_FIELDS])

EXPORTS = [
    "lfpsqp_version", "lfpsqp_default_params", "lfpsqp_ctx_create", "lfpsqp_ctx_destroy", "lfpsqp_last_error",
    "lfpsqp_ctx_set_stream", "lfpsqp_last_kernel_ms", "lfpsqp_last_launches", "lfpsqp_solve_batched",
    "lfpsqp_solve_batched_dev", "lfpsqp_bench_fp64_peak", "lfpsqp_solve_large", "lfpsqp_large_setup",
    "lfpsqp_large_solve", "lfpsqp_large_factor", "lfpsqp_large_project", "lfpsqp_large_projcg",
    "lfpsqp_comm_unique_id", "lfpsqp_comm_init", "lfpsqp_comm_destroy", "lfpsqp_large_retract", "lfpsqp_large_pcg",
    "lfpsqp_ineq_op", "lfpsqp_large_phase_ms", "lfpsqp_comm_ipc_export", "lfpsqp_comm_ipc_import", "lfpsqp_comm_mode",
    "lfpsqp_large_set_bounds", "lfpsqp_solve_host", "lfpsqp_linesearch", "lfpsqp_aug_hess_vec", "lfpsqp_large_projcg_general",
    "lfpsqp_ctx_create_multi", "lfpsqp_ctx_device_count", "lfpsqp_ctx_set_noise", "lfpsqp_last_kernel",
]

_lib = None


def load():
    """Load the shared library (no GPU needed for this step)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("liblfpsqp_b200.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'`); "
                               "there is no CPU fallback")
        lib = C.CDLL(LIB_PATH)
        lib.lfpsqp_version.restype = C.c_char_p
        lib.lfpsqp_last_error.restype = C.c_char_p
        lib.lfpsqp_last_error.argtypes = [C.c_void_p]
        lib.lfpsqp_last_kernel_ms.restype = C.c_double
        lib.lfpsqp_last_kernel_ms.argtypes = [C.c_void_p]
        lib.lfpsqp_last_launches.restype = C.c_int64
        lib.lfpsqp_last_launches.argtypes = [C.c_void_p]
        lib.lfpsqp_last_kernel.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
        lib.lfpsqp_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        lib.lfpsqp_ctx_destroy.argtypes = [C.c_void_p]
        lib.lfpsqp_ctx_create_multi.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]
        lib.lfpsqp_ctx_device_count.argtypes = [C.c_void_p]
        lib.lfpsqp_ctx_set_noise.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64]
        lib.lfpsqp_ctx_set_stream.argtypes = [C.c_void_p, C.c_void_p]
        P = C.c_void_p
        I = C.c_int64
        sig = [P, C.c_int, I, I, I, I, P, I, P, P, P, P, P, P, I, P, P, P, P]
        lib.lfpsqp_solve_batched.argtypes = sig
        lib.lfpsqp_solve_batched_dev.argtypes = sig
        lib.lfpsqp_bench_fp64_peak.argtypes = [P, C.c_int, C.POINTER(C.c_double)]
        lib.lfpsqp_solve_large.argtypes = [P, C.c_int, I, I, P, P, P, P, P, P, P, I, P, P, P, P]
        lib.lfpsqp_large_setup.argtypes = [P, C.c_int, I, I, I, I, P, C.c_int]
        lib.lfpsqp_large_solve.argtypes = [P, P, P, P, P, I, P, P, P, P]
        lib.lfpsqp_large_factor.argtypes = [P, P, P, P, P, P, P]
        lib.lfpsqp_large_project.argtypes = [P, P, P, P]
        lib.lfpsqp_large_projcg.argtypes = [P, P, P, C.c_double, I, C.c_int, P, P, P, P, P]
        lib.lfpsqp_comm_unique_id.argtypes = [P, C.c_char_p]
        lib.lfpsqp_comm_init.argtypes = [P, C.c_int, C.c_int, P, C.c_char_p]
        lib.lfpsqp_comm_destroy.argtypes = [P]
        lib.lfpsqp_large_retract.argtypes = [P, C.c_int, P, P, P, P, P, P, P, P]
        lib.lfpsqp_large_pcg.argtypes = [P, P, C.c_double, P, C.c_double, I, P, P, P, P]
        lib.lfpsqp_ineq_op.argtypes = [P, C.c_int, I, I, P, P, P, P, I, P, I]
        lib.lfpsqp_large_phase_ms.argtypes = [P, P]
        lib.lfpsqp_comm_ipc_export.argtypes = [P, P]
        lib.lfpsqp_comm_ipc_import.argtypes = [P, P]
        lib.lfpsqp_comm_mode.argtypes = [P]
        lib.lfpsqp_large_set_bounds.argtypes = [P, P, P]
        lib.lfpsqp_solve_host.argtypes = [P, P, I, I, P, P, P, P, P, P, I, P, P, P, P]
        lib.lfpsqp_linesearch.argtypes = [P, C.c_int, C.c_int, I, I, P, P, P, P, P, P, P, P, P]
        lib.lfpsqp_aug_hess_vec.argtypes = [P, C.c_int, I, I, P, P, P, P, P, P, P, P]
        lib.lfpsqp_large_projcg_general.argtypes = [P, P, P, P, P, C.c_double, I, P, P, P, P, P]
        _lib = lib
    return _lib


class LFPSQPError(RuntimeError):
    """Mirrors the reference's error() exceptions (optimize.jl:19-21, :144-148, :160-162)."""


class Context:
    """One lfpsqp_ctx (one GPU, one host thread)."""

    def __init__(self, device=0):
        self.lib = load()
        h = C.c_void_p()
        rc = self.lib.lfpsqp_ctx_create(int(device), C.byref(h))
        if rc != 0:
            raise LFPSQPError(self.lib.lfpsqp_last_error(None).decode())
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.lfpsqp_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc):
        if rc != 0:
            raise LFPSQPError("%s (rc=%d)" % (self.lib.lfpsqp_last_error(self.h).decode(), rc))

    def set_stream(self, cuda_stream_ptr):
        self.check(self.lib.lfpsqp_ctx_set_stream(self.h, C.c_void_p(cuda_stream_ptr)))

    def fp64_peak(self, which):
        """measured FP64 peak in TFLOP/s: which = 'dfma' | 'dmma'"""
        v = C.c_double()
        self.check(self.lib.lfpsqp_bench_fp64_peak(self.h, 0 if which == "dfma" else 1, C.byref(v)))
        return v.value

    @property
    def last_kernel_ms(self):
        return self.lib.lfpsqp_last_kernel_ms(self.h)

    @property
    def last_launches(self):
        return self.lib.lfpsqp_last_launches(self.h)

    @property
    def last_kernel(self):
        """(kind, LW, NPL, SPARSE) of the last batched launch: kind 0 thread per instance, 1 warp solver, 2 register
        solver, -1 none"""
        out = (C.c_int * 4)()
        self.check(self.lib.lfpsqp_last_kernel(self.h, out))
        return tuple(out)


class MultiContext(Context):
    """lfpsqp_ctx_create_multi: one ctx over a device list; lfpsqp_solve_batched shards the instances over the devices
    from one host call (one host thread per device inside the library, no collective)."""

    def __init__(self, devices):
        self.lib = load()
        devs = (C.c_int * len(devices))(*[int(d) for d in devices])
        h = C.c_void_p()
        rc = self.lib.lfpsqp_ctx_create_multi(devs, len(devices), C.byref(h))
        if rc != 0:
            raise LFPSQPError(self.lib.lfpsqp_last_error(None).decode() or "lfpsqp_ctx_create_multi failed (rc=%d)" % rc)
        self.h = h
        self.device = int(devices[0])
        self.devices = [int(d) for d in devices]

    @property
    def device_count(self):
        return self.lib.lfpsqp_ctx_device_count(self.h)


_default_ctx = {}


def default_context(device=0):
    if device not in _default_ctx:
        _default_ctx[device] = Context(device)
    return _default_ctx[device]


def ptr(a):
    """host numpy array -> void* (None -> NULL)"""
    return None if a is None else C.c_void_p(a.ctypes.data)
