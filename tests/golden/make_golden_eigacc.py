"""Generates tests/golden/eigacc_golden.json: eigenvalues of the periodic product F_1 F_2 ... F_p
(F = A_1..A_p for :R, A_p..A_1 for :L) of every problem in tests/eigacc.py:PROBLEMS in mpmath,
with the relative structured condition number of each eigenvalue (see tests/eigacc.py) from the
left and right eigenvectors.

Precision: at least 40 + log10(|lambda|max / |lambda|min) digits (a first pass at 60 digits finds
the spread; too few digits give wrong small eigenvalues of graded products).  The eigenvalues are
computed again at 1.5x the digits, the two sets are matched, and their relative agreement must be
below 1e-30; both figures are stored.  Problems run in parallel, one per core.
Run:  python tests/golden/make_golden_eigacc.py
"""
import json
import math
import multiprocessing as mproc
import os
import sys

import mpmath as mp
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import eigacc as EA  # noqa: E402
from oracle import oracle as O  # noqa: E402

AGREE = 1e-30


def factors(A, left):
    """Math matrices of the factors in product order, exact in mpmath."""
    F = [mp.matrix(a.T.tolist()) for a in A]
    return F[::-1] if left else F


def product(F):
    P = F[0]
    for f in F[1:]:
        P = P * f
    return P


def sorted_eigs(E):
    return sorted(E, key=lambda z: (-abs(z), -mp.im(z)))


def agreement(E1, E2):
    """max relative distance between two eigenvalue sets, greedy matching largest first"""
    rem = list(E2)
    worst = mp.mpf(0)
    for z in sorted_eigs(E1):
        d = [abs(z - w) / abs(z) for w in rem]
        k = min(range(len(d)), key=lambda i: d[i])
        worst = max(worst, d[k])
        rem.pop(k)
    return worst


def norm2(a):
    """spectral norm, from float64 after an exact power-of-two normalisation (subnormal or huge
    factors); only its leading digits enter kappa"""
    m = np.abs(a).max()
    if m == 0:
        return mp.mpf(0)
    _, e = math.frexp(m)
    return mp.ldexp(mp.mpf(float(np.linalg.norm(np.ldexp(a, -e), 2))), e)


def kappas(F, E, EL, ER, fnorms):
    """relative structured condition numbers, all eigenvalues at once:
    rows of EL F_1..F_{j-1} and columns of F_{j+1}..F_p ER."""
    p, n = len(F), len(E)
    pre, suf = [None] * p, [None] * p
    L = EL
    for j in range(p):
        pre[j] = L
        L = L * F[j]
    R = ER
    for j in range(p - 1, -1, -1):
        suf[j] = R
        R = F[j] * R
    out = []
    for k in range(n):
        s = mp.mpf(0)
        for j in range(p):
            s += mp.norm(pre[j][k, :]) * fnorms[j] * mp.norm(suf[j][:, k])
        d = abs((EL[k, :] * ER[:, k])[0, 0]) * abs(E[k])
        out.append(s / d)
    return out


def solve(item):
    pid, rec = item
    O.lib()
    A = EA.inputs(O, rec)
    fnorms = [norm2(a.T) for a in A]
    fnorms = fnorms[::-1] if rec["left"] else fnorms
    dps = 60
    while True:
        mp.mp.dps = dps
        F = factors(A, rec["left"])
        E, EL, ER = mp.eig(product(F), left=True, right=True)
        mags = [abs(z) for z in E]
        need = 40 + int(math.ceil(float(mp.log10(max(mags) / min(mags)))))
        if need <= dps:
            break
        dps = need
    kap = kappas(F, E, EL, ER, fnorms)
    dps_check = int(math.ceil(1.5 * dps))
    mp.mp.dps = dps_check
    E2 = mp.eig(product(factors(A, rec["left"])), left=False, right=False)
    agree = float(agreement(E, E2))
    assert agree <= AGREE, (pid, agree)
    mp.mp.dps = dps
    order = sorted(range(len(E)), key=lambda k: (-abs(E[k]), -mp.im(E[k])))
    eig, kappa = [], []
    for k in order:
        z = E[k]
        im = 0.0 if abs(mp.im(z)) <= EA.REAL_TOL * abs(z) else float(mp.im(z))
        eig.append([float(mp.re(z)), im])
        kappa.append(float(kap[k]))
    return pid, dict(id=pid, recipe=rec, sha256=EA.sha(A), dps=dps, dps_check=dps_check, agreement=agree, eig=eig, kappa=kappa)


def main():
    O.build()
    work = sorted(EA.PROBLEMS, key=lambda it: -(it[1]["n"] ** 3) * it[1]["p"])  # largest first
    with mproc.Pool(os.cpu_count()) as pool:
        res = dict(pool.imap_unordered(solve, work))
    out = {"problems": [res[pid] for pid, _ in EA.PROBLEMS]}
    with open(EA.GOLDEN, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print("wrote", len(out["problems"]), "problems; worst agreement",
          max(g["agreement"] for g in out["problems"]), "; max digits", max(g["dps"] for g in out["problems"]))


if __name__ == "__main__":
    main()
