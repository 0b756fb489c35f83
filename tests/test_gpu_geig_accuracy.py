"""Every eigenvalue of the generalized paths (complex and real periodic QZ) against high-precision
ground truth (tests/golden/geigacc_golden.json; gate in tests/geigacc.py), compared from the raw
(alpha, beta, alphascale) triple: each finite eigenvalue must be accurate relative to its own
structured condition number, and zero and infinite eigenvalues must come back as exact zeros of
alpha and beta, as many as the ground truth has.

The cases are chosen by the kernel variant they reach (dispatch: psd_capi.cu launch_gen_t); each
case asserts the memory mode through the handle's statistics.
  shared memory ("smem"): the factors (and Z) of one problem fit in one CTA's shared memory; the
      256-thread gpschur_kernel runs the reduction and the QZ sweeps there.
  global memory ("global"): the factors stay in global memory; the 512-thread ("wide") kernel runs
      the blocked Stage 1 and the windowed Stage 2 of the reduction (full entry only; the
      Hessenberg-triangular entry skips the reduction), windowed QZ sweeps, and, complex only, the
      table-driven "deep" rotation chases.
  With Z, real p = 10 leaves shared memory near N = 38 and complex p = 6 near N = 34; without Z
  (eigenvalues only, or T only) at about 1.4 times those orders.
Signatures: all true (allT), alternating (alt, C5 pattern [F,T,...] with :L), single minus
(oneminus), the C3 pattern [T,F,T,T,F,T] (C3); the N = 40 - 64 cases stand in for the benchmark
sizes C3 (N = 128) and C5 (N = 512), where mpmath is too slow for ground truth.  The scale cases
put whole factors at 1e+-300 so that the eigenvalues lie beyond 1e+-308 (big / small), one factor
subnormal throughout, direct (sub0) or inverted (sub1), or one factor's largest entry at 1.75e308
(huge), or take N = 1 and 2 with factors at 1.75e308, subnormal and 1e-300 (edgeA / edgeB); see
the comment on the scale cases below.  The hole cases plant exact zeros on the diagonal of a
direct or an inverted triangular factor.

Golden problems sit at the first, an inner and the last index of a prime-sized batch of seeded
filler problems, which only have to converge."""
import numpy as np
import pytest

import geigacc as GA
import gpsd_cases as GC

pytestmark = pytest.mark.gpu
EPS = np.finfo(np.float64).eps

GOLD = {g["id"]: g for g in GA.load()["problems"]}
BATCH = 37
POSITIONS = (0, 17, BATCH - 1)


def _c(groups, modes, where):
    return [(g, m, w) for g in groups for m, w in zip(modes, where)]


S, G = "smem", "global"
# Scale cases (SCALE below): every factor whose largest entry lies outside [2^-500, 2^500] is
# normalised by an exact power of two before the reduction (psd_cplx_qz.cuh factor_scale_exponents).
# Without it (the parent of that change, B200), the QZ, like the reference algorithm, failed on each:
#   big-n8p3, big-n40p10      7 of 8 / 39 of 40 eigenvalues infinite (beta = 0): the diagonal of the
#                             inverted factor at 1e-300 is below smlnum and taken for zeros
#   small-n8p3, small-n40p10  every eigenvalue wrong, relative errors 0.3 to 2e9
#   sub0-n12p3                every eigenvalue NaN (the products of subnormal diagonals overflowed)
#   sub1-n12p3, huge-n12p3    info = n (no convergence)
#   edge*-n1p3, edge*-n2p3    every eigenvalue inf or NaN: the products of diagonals at 1.75e308 and
#                             subnormal ones left the double range
HOLES5 = [f"{c}-hole{k}" for c in "rc" for k in range(len(GC.HOLE_CASES))]
# (problem group, outputs: eig = eigenvalues only, T = T only, TZ = T and Z; memory mode reached)
CASES = (
    _c(["c-n5p5-allT", "r-n5p5-allT"], ["eig", "T", "TZ"], [S, S, S]) +
    _c(["c-n12p6-C3", "c-n20p4-altL", "c-n24p4-oneminus", "c-graded-n16p4",
        "r-n12p3-alt", "r-n20p4-oneminus", "r-n24p10-C5L", "r-graded-n16p4"], ["eig", "TZ"], [S, S]) +
    _c(["c-n40p6-C3"], ["eig", "T", "TZ"], [S, S, G]) +
    _c(["c-n56p6-C3", "r-n64p10-C5L"], ["eig", "TZ"], [G, G]) +
    _c(["r-n40p10-C5L"], ["eig", "TZ"], [S, G]) +
    _c(["c-hessut-n40p6", "r-hessut-n40p10"], ["eig", "TZ"], [S, G]) +
    _c(HOLES5, ["TZ"], [S]) +
    _c([f"{c}-hole-n40p{p}-{k}" for c, p in (("c", 6), ("r", 10)) for k in ("direct", "inverted")],
       ["eig", "TZ"], [S, G]) +
    _c([f"{c}-{k}-n8p3" for c in "cr" for k in ("big", "small")] +
       [f"{c}-sub{j}-n12p3" for c in "cr" for j in (0, 1)] + ["c-huge-n12p3", "r-huge-n12p3"] +
       [f"{c}-{k}-n{n}p3" for c in "cr" for n in (1, 2) for k in ("edgeA", "edgeB")],
       ["eig", "TZ"], [S, S]) +
    _c([f"r-{k}-n40p10" for k in ("big", "small")], ["eig", "TZ"], [S, G]) +
    _c([f"c-{k}-n40p10" for k in ("big", "small")], ["eig", "TZ"], [G, G])
)


def _members(group):
    return [pid for pid, _ in GA.PROBLEMS if pid == group or pid.rsplit("-b", 1)[0] == group]


def _placed_batch(group, seed):
    pids = _members(group)
    rec = GOLD[pids[0]]["recipe"]
    dt = np.complex128 if rec["cplx"] else np.float64
    A = np.stack([GA.inputs(rec, seed=seed + b) for b in range(BATCH)]).astype(dt)
    placed = {}
    for k, pos in enumerate(POSITIONS):
        placed[pos] = pids[k % len(pids)]
        A[pos] = GA.inputs(GOLD[placed[pos]]["recipe"])
    return A, placed


@pytest.mark.parametrize("group,mode,where", CASES, ids=[f"{g}-{m}-{w}" for g, m, w in CASES])
def test_eigenvalues_against_ground_truth(psd, group, mode, where):
    A, placed = _placed_batch(group, 5151)
    rec0 = GOLD[placed[0]]["recipe"]
    h = psd.Handle([0])
    wantT, wantZ = mode != "eig", mode == "TZ"
    T, _, al, be, sc, info = psd.gpschur_batched(A, rec0["S"], "L" if rec0["left"] else "R", wantZ=wantZ,
                                                 wantT=wantT, handle=h, hessut=rec0["hessut"])
    st = h.stats()
    assert st["problems_smem" if where == S else "problems_global"] == BATCH, st
    assert (info == 0).all(), {i: int(info[i]) for i in np.flatnonzero(info)}
    worst = 0.0
    for pos, pid in placed.items():
        g = GOLD[pid]
        rec = g["recipe"]
        err, allowed, _ = GA.check(g, al[pos], be[pos], sc[pos], what=f"{pid} at index {pos}")
        worst = max(worst, float(np.max(err / allowed)) if len(err) else 0.0)
        if not rec["cplx"]:
            GA.check_pairs(al[pos], be[pos], sc[pos], g)
        if wantT:
            GA.check_against_T(T[pos], al[pos], be[pos], sc[pos], rec["S"], rec["left"],
                               GA.T_tolerance(g, al[pos], be[pos], sc[pos]))
    print(f"worst error / allowed {group} {mode} {where}: {worst:.3g}")


@pytest.mark.parametrize("cplx", [False, True], ids=["real", "complex"])
@pytest.mark.parametrize("n", [2, 3])
def test_subnormal_diagonal_beside_normal_entries(psd, n, cplx):
    """An inverted triangular factor whose diagonal holds one subnormal entry beside entries of order
    one, e.g. [[0.8, 0.6], [0, 1e-310]]: the entry lies below the deflation tolerance
    (ulp times its neighbours), so the QZ sets it to an exact zero, as the reference does, and the
    eigenvalue comes back infinite (beta = 0) with every other one finite; no inf or NaN reaches
    alpha, and the eigenvalues agree with the diagonal blocks of T."""
    S = [1, 0, 1]
    A = GC.hessut_storage(8600 + n, n, 3, 1, cplx)
    A[0, 1, n - 1, n - 1] = 1e-310
    T, _, al, be, sc, info = psd.gpschur_batched(A, S, "R", hessut=True)
    assert info[0] == 0
    assert np.isfinite(al[0]).all() and np.isfinite(be[0]).all()
    assert np.count_nonzero(be[0] == 0) == 1 and np.count_nonzero(al[0] == 0) == 0
    assert not T[0, 1].diagonal().all()
    GA.check_against_T(T[0], al[0], be[0], sc[0], S, False, np.full(n, 1e3 * EPS))
