"""GPU tests of the large-N fallback: when the multishift iteration reaches its round cap
((256 + 100 n / D) maxitfac / 30 rounds) it drains the bulges in flight and returns status 1, and
the single-bulge team kernel (gpschur_team_kernel) finishes the problem from that state.  Also the
team path without multishift (p = 13..16, above the multishift's largest period), which no other
test reaches at N >= 192."""
import os
import sys

import numpy as np
import pytest

import psd_checks as K

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "ms_emul"))
import emul  # noqa: E402

pytestmark = pytest.mark.gpu
EPS = np.finfo(float).eps


def _round_bound(n, p, maxitfac):
    """largest number of rounds of a capped run: the cap, the round that sees it, the drain"""
    g = emul.geom(p)  # csrc/psd_ms_core.cuh:geom_for, compiled for the CPU
    W, D = g["W"], g["D"]
    return (256 + 100 * n // D) * maxitfac // 30 + 1 + (n + W) // D + 4


def _pairs_first_positive(lam):
    n = lam.shape[0]
    k = 0
    while k < n:
        if lam[k].imag != 0:
            assert lam[k].imag > 0 and lam[k + 1] == np.conj(lam[k]), k
            k += 2
        else:
            k += 1


def _trace(A, left):
    p = A.shape[0]
    order = range(p) if not left else range(p - 1, -1, -1)
    P = np.linalg.multi_dot([K.M(A[j]) for j in order]) if p > 1 else K.M(A[0])
    return P


def _check_fallback(psd, A, lr, wantT, wantZ, maxitfac):
    """one capped call: the fallback ran, and its result matches a default call"""
    n, p = A.shape[2], A.shape[1]
    left = lr == "L"
    T, Z, lam, info = psd.pschur_batched(A, lr, wantT=wantT, wantZ=wantZ, maxitfac=maxitfac)
    st = psd.default_handle().large_stats()
    assert st["status"] == 1, st
    assert 0 < st["rounds"] <= _round_bound(n, p, maxitfac), st
    assert info[0] == 0
    if wantZ:
        K.pschur_check(A[0], T[0], Z[0], lam[0], left=left, tol=40, check_lambda=False)
    elif wantT:
        js = p - 1 if left else 0
        for j in range(p):
            assert not np.tril(K.M(T[0, j]), -2 if j == js else -1).any(), j
    _pairs_first_positive(lam[0])
    _, _, lam0, info0 = psd.pschur_batched(A, lr, wantT=False, wantZ=False)
    assert info0[0] == 0 and psd.default_handle().large_stats()["status"] == 0
    scale = np.max(np.abs(lam0[0]))
    assert K.match_eigs(lam0[0], lam[0]) <= 100 * n * EPS * scale
    P = _trace(A[0], left)
    tr = np.trace(P)
    assert abs(lam[0].sum() - tr) <= 1e-10 * np.abs(lam0[0]).sum()


# Uncapped rounds of these inputs (CPU emulation, tests/test_ms_giveup.py; the GPU's shift choice
# depends on timing and needs about as many): N = 256, p = 2: 140; N = 300, p = 1: 250.  The caps
# at maxitfac = 1 / 2 are 35 / 70 and 39 / 79 rounds, so every call below gives up with a margin
# of a factor of two or more.
@pytest.mark.parametrize("maxitfac", [1, 2])
@pytest.mark.parametrize("n,p,lr,wantT,wantZ", [(256, 2, "R", True, True), (300, 1, "L", True, False),
                                               (256, 2, "R", False, False)])
def test_capped_multishift_falls_back(psd, oracle, maxitfac, n, p, lr, wantT, wantZ):
    A = oracle.gen_real(1234, n, p, 1)
    _check_fallback(psd, A, lr, wantT, wantZ, maxitfac)


def test_capped_multishift_batch(psd, oracle):
    """batch > 1: each problem falls back on its own (team kernel and postscale per problem)"""
    n, p = 200, 3
    A = oracle.gen_real(1234, n, p, 2)
    T, Z, lam, info = psd.pschur_batched(A, "R", maxitfac=1)
    assert psd.default_handle().large_stats()["status"] == 1
    assert (info == 0).all()
    for b in range(2):
        K.pschur_check(A[b], T[b], Z[b], lam[b], tol=40, check_lambda=False)
        _pairs_first_positive(lam[b])
        ref = np.linalg.eigvals(_trace(A[b], False))
        assert K.match_eigs(ref, lam[b]) <= 1e-8 * np.max(np.abs(ref))


@pytest.mark.parametrize("scale", [1e-160, 1e160])
def test_capped_multishift_badly_scaled(psd, oracle, scale):
    """one factor tiny / huge: the power-of-two prescale before the reduction and the postscale
    after the team kernel (reached only through the fallback)"""
    n, p = 256, 2
    A = oracle.gen_real(1234, n, p, 1)
    As = A.copy()
    As[:, 0] *= scale
    T, Z, lam, info = psd.pschur_batched(As, "R", maxitfac=1)
    assert psd.default_handle().large_stats()["status"] == 1
    assert info[0] == 0 and np.isfinite(T).all() and np.isfinite(Z).all()
    K.pschur_check(As[0], T[0], Z[0], lam[0], tol=40, check_lambda=False)
    _, _, lam1, info1 = psd.pschur_batched(A, "R", wantT=False, wantZ=False)
    assert info1[0] == 0
    s1 = np.max(np.abs(lam1[0]))
    assert K.match_eigs(lam1[0], lam[0] / scale) <= 1e-8 * s1


@pytest.mark.parametrize("n,p,lr", [(192, 13, "R"), (200, 16, "L")])
def test_team_path_long_periods(psd, oracle, n, p, lr):
    """p > 12 at N >= 192: blocked reduction, then the team kernel directly"""
    left = lr == "L"
    A = oracle.gen_real(4000 + 10 * p + n, n, p, 1)
    T, Z, lam, info = psd.pschur_batched(A, lr)
    assert info[0] == 0
    K.pschur_check(A[0], T[0], Z[0], lam[0], left=left, tol=40, check_lambda=False)
    _pairs_first_positive(lam[0])
    _, _, lo, io, _ = oracle.rpschur_batched(A, left=left, wantT=False, wantZ=False)
    assert io[0] == 0
    scale = np.max(np.abs(lo[0]))
    assert K.match_eigs(lo[0], lam[0]) <= 100 * n * EPS * scale
