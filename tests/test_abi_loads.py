"""CPU-only checks of the boundary: the C-ABI library loads and exports every symbol include/lfpsqp_b200.h declares,
and fails loudly (no CPU fallback) when there is no GPU."""
import ctypes
import multiprocessing as mp
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "lfpsqp_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(lfpsqp_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    import lfpsqp.jl_b200 as L
    lib = L.load()
    syms = _declared_symbols()
    assert len(syms) >= 10
    for s in syms:
        assert hasattr(lib, s), "missing export %s" % s
    assert b"sm_100a" in lib.lfpsqp_version()


def test_default_params_match_reference_defaults():
    # src/LFPSQP.jl:57-81
    import lfpsqp.jl_b200 as L
    from lfpsqp.jl_b200 import _lib
    p = _lib.CParams()
    L.load().lfpsqp_default_params(ctypes.byref(p))
    assert (p.alpha, p.beta, p.t_beta, p.s, p.sigma) == (1.0, 0.0, 0, 0.5, 1e-4)
    assert (p.eps_c, p.eps_f, p.eps_x, p.eps_kkt, p.eps_rank) == (1e-6, 1e-6, 0.0, 1e-6, 1e-10)
    assert (p.maxiter, p.maxiter_retract, p.maxiter_pcg, p.mu0) == (10000, 100, 100, 1e-2)
    assert (p.disable_linesearch, p.do_project_retract, p.linesearch, p.do_newton) == (0, 1, 0, 1)
    assert (p.tn_maxiter, p.tn_kappa, p.callback_period) == (10000, 0.5, 100)
    q = L.LFPSQPParams().to_c()
    for name, _ in _lib.CParams._fields_:
        assert getattr(p, name) == getattr(q, name), name
    assert L.LFPSQPParams(ϵ_c=1e-8).eps_c == 1e-8 and L.LFPSQPParams(eps_c=1e-8).ϵ_c == 1e-8
    assert ctypes.sizeof(_lib.CParams) == 160 and _lib.TERM_DTYPE.itemsize == 40


def _no_cpu_fallback():
    import lfpsqp.jl_b200 as L
    with pytest.raises(L.LFPSQPError, match="no CPU fallback"):
        L.Context(0)


def test_no_cpu_fallback(monkeypatch):
    # in a child process that sees no GPU, so that the check runs on a GPU machine as well
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    p = mp.get_context("spawn").Process(target=_no_cpu_fallback)
    p.start()
    p.join(300)
    assert p.exitcode == 0


def test_method_shapes_resolve():
    # optimize.jl:13, :83, :88, :107, :112 -- argument parsing only (no device work)
    from lfpsqp.jl_b200 import api, families
    fam = families.readme_inequality(np.ones(5))
    f, c, d, dl, du, x0, xl, xu, m, p, prm = api._parse((fam.f, None, fam.d, np.zeros(5), None, None, 0, 1))
    assert (m, p) == (0, 1) and d is fam.d and isinstance(prm, api.LFPSQPParams)
    f, c, d, dl, du, x0, xl, xu, m, p, prm = api._parse((fam.f, np.zeros(5), api.LFPSQPParams(maxiter=3)))
    assert (m, p, prm.maxiter) == (0, 0, 3)
    with pytest.raises(TypeError):
        api._parse((fam.f, 1, 2))
    with pytest.raises(TypeError):
        api._family_of(lambda x: 0.0, None, None)


def test_header_is_plain_c(tmp_path):
    # the boundary is a C ABI: the header must compile as C99 (what a cgo / ccall / ctypes binder assumes), no C++-isms
    import shutil
    import subprocess
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    src = tmp_path / "use_header.c"
    src.write_text('#include "lfpsqp_b200.h"\n'
                   'int probe(lfpsqp_ctx *c, const lfpsqp_host_callbacks *cb, lfpsqp_params *p) {\n'
                   '  lfpsqp_default_params(p);\n'
                   '  return (int)sizeof(lfpsqp_term) + (int)sizeof(lfpsqp_stats) + (cb && c ? LFPSQP_FAM_HOST : LFPSQP_OK);\n'
                   '}\n')
    r = subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-fsyntax-only",
                        "-I", os.path.join(ROOT, "include"), str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
