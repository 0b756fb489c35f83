"""CPU tests of the give-up path of the large-N multishift iteration (csrc/psd_ms_driver.hpp)
through the emulation harness (tests/ms_emul/).  When the iteration stops early (round cap from
maxitfac, or an explicit cap on the driver's rounds) it returns status 1 and the library hands
the factors to the single-bulge team iteration, which assumes a Hessenberg-triangular form with
Z accumulated.  So the returned state must be exactly that: every bulge still in flight drained,
exact zeros below the structure, Z orthogonal, A_j = Z_j H_j Z_{j+1}' to rounding, and
finishing it with the reference algorithm must give a correct periodic Schur form."""
import os
import sys

import numpy as np
import pytest

import psd_checks as K

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "ms_emul"))
import emul  # noqa: E402

EPS = np.finfo(float).eps

# Emulated rounds of the uncapped iteration on these inputs: (256, 2) 140, (300, 1) 250,
# (200, 3) 60, (192, 4) 61.  maxitfac = 1 caps them at (256 + 100 n / D) / 30 = 35, 40, 29, 31,
# so every case below gives up with packets in flight.
SHAPES = [(256, 2, 140), (300, 1, 250), (200, 3, 60), (192, 4, 61)]
CAPS = [dict(maxitfac=1), dict(max_rounds=1), dict(max_rounds=2), "half"]


def _problem(oracle, n, p):
    A = oracle.gen_real(1234, n, p, 1)
    H, Q = oracle.rphess_batched(A)
    return A[0], H[0], Q[0]


def _caps():
    for n, p, full in SHAPES:
        for cap in CAPS:
            kw = dict(max_rounds=full // 2) if cap == "half" else cap
            yield pytest.param(n, p, kw, id=f"{n}x{p}-" + "-".join(f"{k}{v}" for k, v in kw.items()))


def _check_structure(H):
    p = H.shape[0]
    for j in range(p):
        low = np.tril(K.M(H[j]), -2 if j == 0 else -1)
        assert not low.any(), f"factor {j}: {np.count_nonzero(low)} non-zeros below the structure, " \
                              f"largest {np.abs(low).max():.3g}"


def _product(A):
    p = A.shape[0]
    return np.linalg.multi_dot([K.M(A[j]) for j in range(p)]) if p > 1 else K.M(A[0])


def _check_eigs(A, lam):
    P = _product(A)
    ref = np.linalg.eigvals(P)
    assert K.match_eigs(ref, lam) <= 1e-9 * np.max(np.abs(ref))
    tr = np.trace(P)
    assert abs(lam.sum() - tr) <= 1e-10 * np.abs(ref).sum()


@pytest.mark.parametrize("n,p,cap", list(_caps()))
def test_giveup_leaves_hessenberg_triangular_form(oracle, n, p, cap):
    A, H, Q = _problem(oracle, n, p)
    T, Z, _, info, st = emul.run(H, Q, **cap)
    assert st["status"] == 1 and info == 0, st
    if "max_rounds" in cap:
        assert st["rounds"] <= cap["max_rounds"] + 1 + (n + emul.geom(p)["W"]) // emul.geom(p)["D"] + 4
    _check_structure(T)
    for j in range(p):
        Zj, Zn = K.M(Z[j]), K.M(Z[(j + 1) % p])
        assert np.linalg.norm(Zj.T @ Zj - np.eye(n)) < 10 * EPS * n
        res = np.linalg.norm(K.M(A[j]) - Zj @ K.M(T[j]) @ Zn.T)
        assert res <= 40 * EPS * np.linalg.norm(K.M(A[j]), 1), (j, res / (EPS * np.linalg.norm(K.M(A[j]), 1)))
    # finish with the reference algorithm: a periodic Schur form of A
    T2, Z2, lam, info2 = oracle.rpschur_hessut(T)
    assert info2 == 0
    Zt = np.stack([(K.M(Z[j]) @ K.M(Z2[j])).T for j in range(p)])
    K.pschur_check(A, T2, Zt, lam, tol=48, check_lambda=False)
    _check_eigs(A, lam)


@pytest.mark.parametrize("n,p,cap", [(256, 2, dict(maxitfac=1)), (200, 3, dict(maxitfac=1)),
                                     (300, 1, dict(max_rounds=2)), (192, 4, dict(max_rounds=30))])
def test_giveup_eigenvalues_only(oracle, n, p, cap):
    """without T and Z the updates stay inside the active blocks; the returned factors still have
    exact zeros below the structure and the eigenvalues of the product"""
    A, H, _ = _problem(oracle, n, p)
    T, _, _, info, st = emul.run(H, None, wantT=False, wantZ=False, **cap)
    assert st["status"] == 1 and info == 0, st
    _check_structure(T)
    _, _, lam, info2 = oracle.rpschur_hessut(T, wantT=False, wantZ=False)
    assert info2 == 0
    _check_eigs(A, lam)


@pytest.mark.parametrize("n,p", [(256, 2), (200, 3)])
def test_default_maxitfac_is_unchanged(oracle, n, p):
    """maxitfac = 30 is the default: same cap, same result bit for bit"""
    A, H, Q = _problem(oracle, n, p)
    T0, Z0, lam0, info0, st0 = emul.run(H, Q)
    T1, Z1, lam1, info1, st1 = emul.run(H, Q, maxitfac=30)
    assert st0["status"] == 0 and st0 == st1 and info0 == info1 == 0
    assert np.array_equal(T0, T1) and np.array_equal(Z0, Z1) and np.array_equal(lam0, lam1)


def test_maxitfac_scales_the_round_cap(oracle):
    """the cap is (256 + 100 n / D) maxitfac / 30 rounds: maxitfac = 1 stops (256, 2) after at
    most 35 + 1 rounds plus the drain, maxitfac = 2 after at most 71 + 1 plus the drain; both
    leave a usable state"""
    n, p = 256, 2
    g = emul.geom(p)
    drain = (n + g["W"]) // g["D"] + 4
    A, H, Q = _problem(oracle, n, p)
    for fac in (1, 2):
        cap = (256 + 100 * n // g["D"]) * fac // 30
        T, Z, _, info, st = emul.run(H, Q, maxitfac=fac)
        assert st["status"] == 1 and info == 0
        assert cap - 8 <= st["rounds"] <= cap + 1 + drain, (fac, cap, st)
        _check_structure(T)
