"""CPU checks of the per-eigenvalue accuracy gate (tests/eigacc.py) and of its ground truth
(tests/golden/eigacc_golden.json): the inputs still come out of their recipes, the ground truth is
converged, the CPU oracle passes the gate with margin, a gate that only looks at the largest
eigenvalue would not catch what this one catches, and the exponent bookkeeping of the
power-of-two normalisation done before the eigenvalue-only iteration."""
import math

import numpy as np
import pytest

import eigacc as EA
import psd_checks as K

GOLD = {g["id"]: g for g in EA.load()["problems"]}
IDS = [pid for pid, _ in EA.PROBLEMS]


def test_golden_covers_every_problem():
    assert IDS == [g["id"] for g in EA.load()["problems"]]
    for pid, rec in EA.PROBLEMS:
        assert GOLD[pid]["recipe"] == rec, pid


@pytest.mark.parametrize("pid", IDS)
def test_golden_inputs_and_convergence(oracle, pid):
    g = GOLD[pid]
    A = EA.inputs(oracle, g["recipe"])
    assert np.isfinite(A).all()
    assert EA.sha(A) == g["sha256"], "the recipe no longer gives the inputs the ground truth was computed for"
    ref, kappa = EA.truth(g)
    assert len(ref) == g["recipe"]["n"] and (kappa >= 1.0).all()
    assert g["agreement"] <= 1e-30
    assert g["dps_check"] >= 1.5 * g["dps"]
    spread = np.log10(np.abs(ref).max() / np.abs(ref).min())
    assert g["dps"] >= 40 + spread
    # the ground truth of a real product: complex eigenvalues in conjugate pairs
    assert sorted(ref[ref.imag > 0].tolist(), key=abs) == sorted(np.conj(ref[ref.imag < 0]).tolist(), key=abs)


@pytest.mark.parametrize("want_tz", [False, True], ids=["eig", "TZ"])
@pytest.mark.parametrize("pid", IDS)
def test_oracle_passes_the_gate(oracle, pid, want_tz):
    """The CPU oracle meets the gate on every problem, with a margin of 4 on the first-order branch;
    with T, its eigenvalues agree with the diagonal blocks of T."""
    g = GOLD[pid]
    rec = g["recipe"]
    A = EA.inputs(oracle, rec)
    T, lam_s, shift, info = EA.oracle_run(oracle, rec, A, want_tz)
    assert info == 0
    lam = EA.unshift(lam_s, shift)
    ref, kappa = EA.truth(g)
    err, allowed, cond = EA.check(ref, kappa, lam, rec["n"], what=pid)
    assert (err[cond] <= allowed[cond] / 4).all(), np.max(err[cond] / allowed[cond])
    EA.check_output_order(lam, ref)
    if want_tz:
        EA.check_against_T(T, lam_s, rec["left"], EA.T_tolerance(ref, kappa, lam, rec["p"]))


def _smallest_checked(ref, kappa, n, below):
    """index of the smallest-magnitude real eigenvalue on the first-order branch whose allowed
    relative error is below `below`"""
    allowed, cond = EA.bounds(ref, kappa, n)
    ok = [k for k in range(len(ref)) if cond[k] and ref[k].imag == 0 and allowed[k] < below]
    assert ok
    return min(ok, key=lambda k: abs(ref[k]))


@pytest.mark.parametrize("pid", ["n32p8R-b0", "n32p8L-b1", "n24p7-b0"])
def test_gate_catches_one_small_eigenvalue_off(oracle, pid):
    """A relative error of 1e-9 in one small eigenvalue fails the gate; an absolute gate at
    100 N eps |lambda|max (the one the other eigenvalue tests use) lets it through."""
    g = GOLD[pid]
    rec = g["recipe"]
    n = rec["n"]
    ref, kappa = EA.truth(g)
    _, lam, shift, _ = EA.oracle_run(oracle, rec, EA.inputs(oracle, rec), False)
    lam = EA.unshift(lam, shift)
    EA.check(ref, kappa, lam, n)
    k = _smallest_checked(ref, kappa, n, 1e-10)
    assert abs(ref[k]) < 1e-6 * np.abs(ref).max()  # several decades below the largest
    bad = lam.copy()
    i = EA.match(ref, lam)[k]
    bad[i] = bad[i].real * (1 + 1e-9)
    with pytest.raises(AssertionError, match="outside the gate"):
        EA.check(ref, kappa, bad, n)
    assert K.match_eigs(ref, bad) <= 100 * n * EA.EPS * np.abs(ref).max()


@pytest.mark.parametrize("factor", [2.0 ** -13, 2.0 ** 13, 2.0 ** -29])
@pytest.mark.parametrize("pid", ["tiny305-n32p8-b0", "tiny310-n16p3-b0", "n3p3-b0"])
def test_gate_catches_a_wrong_exponent(oracle, pid, factor):
    """all eigenvalues off by a power of two, as a wrongly recorded normalisation makes them"""
    g = GOLD[pid]
    rec = g["recipe"]
    ref, kappa = EA.truth(g)
    _, lam, shift, _ = EA.oracle_run(oracle, rec, EA.inputs(oracle, rec), False)
    lam = EA.unshift(lam, shift)
    with pytest.raises(AssertionError, match="outside the gate"):
        EA.check(ref, kappa, lam * factor, rec["n"])


def test_gate_catches_a_missing_pair():
    ref = np.array([2.0 + 1.0j, 2.0 - 1.0j, 0.5])
    with pytest.raises(AssertionError, match="complex pairs"):
        EA.check_output_order(np.array([2.0, 2.0, 0.5], dtype=complex), ref)
    with pytest.raises(AssertionError, match="does not open a pair"):
        EA.check_output_order(np.array([2.0 - 1.0j, 2.0 + 1.0j, 0.5]), ref)


def _normalise(m):
    """Python restatement of the normalisation before the eigenvalue-only iteration
    (psd_device.cuh pow2_shift and its callers): the factor is multiplied by 2^s, with the shift
    capped at 2^1000, and -s is recorded; the eigenvalues are multiplied back by 2^(recorded)."""
    _, e = math.frexp(m)
    s = 1000 if -e > 1000 else -e
    return s, -s, e


@pytest.mark.parametrize("m", [1.0, 1e-150, 4.6e-302, 1e-305, 1e-310, 5e-324, 1e300, 1.6e308])
def test_normalisation_records_the_applied_shift(m):
    s, recorded, e = _normalise(m)
    scaled = math.ldexp(m, s)
    assert 0.0 < scaled < 1.0 and math.ldexp(scaled, recorded) == m  # exact both ways
    if m >= 2.0 ** -1000:
        assert recorded == e and 0.5 <= scaled  # nothing changes above the cap
    else:
        # below the cap the unclamped exponent (what was recorded before) is off by 2^(-e-1000)
        assert recorded != e and math.ldexp(scaled, e) == m * 2.0 ** (e + 1000)
