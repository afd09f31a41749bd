"""Sparse QCQP family with its Jacobian kept sparse (LFPSQP_FAM_SPARSE_QCQP_CSR) without a GPU: the jacobian= choice of
families.sparse_qcqp, the family id it selects, and its survival through slack_embedding and equalities."""
import os
import subprocess

import numpy as np
import pytest

from lfpsqp.jl_b200 import _lib, families

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def small(**kw):
    n = 6
    return families.sparse_qcqp(P=np.eye(n), q=np.ones(n), Qc=[np.eye(n)], Ac=np.ones((1, n)), bc=[0.5],
                                Qd=[2 * np.eye(n)], Ad=np.arange(n, dtype=float)[None], bd=[1.0], **kw)


def test_default_is_dense():
    fam = small()
    assert fam.jacobian == "dense" and fam.id == families.SPARSE_QCQP == 102


def test_csr_selects_family_103():
    fam = small(jacobian="csr")
    assert fam.jacobian == "csr" and fam.id == families.SPARSE_QCQP_CSR == 103
    assert fam.f.family is fam


@pytest.mark.parametrize("bad", ["CSR", "sparse", "", None, 1])
def test_other_values_are_refused(bad):
    with pytest.raises(_lib.LFPSQPError, match="jacobian"):
        small(jacobian=bad)


@pytest.mark.parametrize("jac", ["dense", "csr"])
def test_choice_survives_slack_embedding_and_equalities(jac):
    fam = small(jacobian=jac)
    aug, x0, xl, xu = fam.slack_embedding(np.zeros(fam.n))
    assert aug.jacobian == jac and aug.id == fam.id and (aug.n, aug.m, aug.p) == (fam.n + 1, 2, 0)
    eq = fam.equalities()
    assert eq.jacobian == jac and eq.id == fam.id and (eq.n, eq.m, eq.p) == (fam.n, 1, 0)


def test_same_data_in_both_storages():
    a, b = small(), small(jacobian="csr")
    for name in ("P", "Qc", "Ac", "Qd", "Ad"):
        for u, v in zip(getattr(a, name), getattr(b, name)):
            assert np.array_equal(u, v)
    for name in ("q", "bc", "bd"):
        assert np.array_equal(getattr(a, name), getattr(b, name))


def test_header_constant_matches():
    """LFPSQP_FAM_SPARSE_QCQP_CSR in the C header is the id the Python layer passes"""
    src = ('#include <stdio.h>\n#include "lfpsqp_b200.h"\n'
           'int main(void) { printf("%d", LFPSQP_FAM_SPARSE_QCQP_CSR); return 0; }\n')
    cc = os.environ.get("CC", "cc")
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        with open(os.path.join(d, "t.c"), "w") as fh:
            fh.write(src)
        exe = os.path.join(d, "t")
        try:
            subprocess.check_call([cc, "-I", os.path.join(ROOT, "include"), "-o", exe, os.path.join(d, "t.c")])
        except (OSError, subprocess.CalledProcessError):
            pytest.skip("no C compiler")
        assert int(subprocess.check_output([exe]).decode()) == families.SPARSE_QCQP_CSR


def test_julia_binding_declares_the_id():
    with open(os.path.join(ROOT, "lfpsqp.jl_b200", "julia", "LFPSQPB200.jl")) as fh:
        assert "const LFPSQP_FAM_SPARSE_QCQP_CSR = 103" in fh.read()
