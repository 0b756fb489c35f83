"""Generates tests/golden/geigacc_golden.json: the eigenvalues of prod A_j^{s_j} (A_1^{s_1}..A_p^{s_p}
for :R, A_p^{s_p}..A_1^{s_1} for :L) of every problem in tests/geigacc.py:PROBLEMS in mpmath, with
the relative structured condition number of each finite non-zero eigenvalue (see tests/geigacc.py)
and the exact counts of zero and infinite eigenvalues.

Without a singular inverted factor the eigenvalues are those of the product, formed in mpmath.  With
one (an exact zero on the diagonal of a triangular factor B with s = false), the cycle is rotated so
that the product reads M B^-1, and the eigenvalues are those of the pencil (M, B), by shift and
invert: mu = eig((M - sigma B)^-1 B) for a sigma that is no eigenvalue, lambda = sigma + 1/mu, and
mu = 0 is an infinite eigenvalue.  Those problems carry no condition numbers (the gate then takes
its fallback).  The eigenvalues (values of mu) that the planted holes make exactly zero must come
out below 10^(-dps/2) of the smallest of the others.

Precision: at least 40 + log10(|lambda|max / |lambda|min) digits (a first pass at 60 digits finds
the spread).  The eigenvalues are computed again at 1.5x the digits and their relative agreement
must be below 1e-30; both figures are stored.  Eigenvalues are stored as decimal strings, so that
values beyond 1e+-308 survive.  Problems run in parallel, one per core.
Run:  python tests/golden/make_golden_geigacc.py
"""
import json
import math
import multiprocessing as mproc
import os
import sys
import time

import mpmath as mp
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import geigacc as GA  # noqa: E402
from make_golden_eigacc import agreement  # noqa: E402

AGREE = 1e-30
SIGMA = mp.mpf(3) / 7   # shift of the shift-and-invert step (no eigenvalue of any problem)


def norm2(a):
    """spectral norm, from float64 after an exact power-of-two normalisation (subnormal or huge
    factors); only its leading digits enter kappa"""
    m = np.abs(a).max()
    if m == 0:
        return mp.mpf(0)
    _, e = math.frexp(m)
    s = np.ldexp(a.real, -e) + 1j * np.ldexp(a.imag, -e) if np.iscomplexobj(a) else np.ldexp(a, -e)
    return mp.ldexp(mp.mpf(float(np.linalg.norm(s, 2))), e)


def _mat(a):
    return mp.matrix([[mp.mpc(complex(x)) if np.iscomplexobj(a) else mp.mpf(float(x)) for x in row] for row in a])


def factors(A, rec):
    """[(math matrix, s_j)] in product order, exact in mpmath"""
    order = list(range(rec["p"]))[::-1] if rec["left"] else list(range(rec["p"]))
    return [(_mat(A[j].T), bool(rec["S"][j]), j) for j in order]


def inverse(a):
    """mp.inverse, by back substitution for an upper triangular matrix (mp.inverse calls one with a
    diagonal entry far below its norm, such as a subnormal one, singular)"""
    n = a.rows
    if any(a[i, j] != 0 for j in range(n) for i in range(j + 1, n)):
        return mp.inverse(a)
    X = mp.zeros(n, n)
    for c in range(n):
        for i in range(c, -1, -1):
            s = (1 if i == c else 0) - mp.fsum(a[i, k] * X[k, c] for k in range(i + 1, c + 1))
            X[i, c] = s / a[i, i]
    return X


def product(F):
    P = mp.eye(F[0][0].rows)
    for a, s, _ in F:
        P = P * (a if s else inverse(a))
    return P


def singular_inverted(rec):
    return [j for j, _, v in rec["diag"] if v == 0 and not rec["S"][j]]


def _drop_smallest(E, count, tiny):
    """indices of E without its `count` smallest members, which must lie below tiny times the
    smallest of the rest (the exact zeros the recipe planted)"""
    order = sorted(range(len(E)), key=lambda k: abs(E[k]))
    keep = sorted(order[count:])
    if count:
        assert abs(E[order[count - 1]]) < tiny * abs(E[order[count]]), "a planted zero is not separated"
    if count < len(E) - 1:
        assert abs(E[order[count]]) >= tiny * abs(E[order[-1]]) or count == 0, "an unplanted zero"
    return keep


def eigs(A, rec, vectors):
    """(eigenvalues, indices of the finite non-zero ones, zero count, infinite count, left / right
    eigenvectors or None, factors in product order)"""
    F = factors(A, rec)
    tiny = mp.mpf(10) ** (-mp.mp.dps // 2)
    nz, ni = GA.holes(rec)
    if ni:
        k = [f[2] for f in F].index(singular_inverted(rec)[0])
        F = F[k + 1:] + F[:k + 1]
        M, B = product(F[:-1]), F[-1][0]
        mu = mp.eig(inverse(M - SIGMA * B) * B, left=False, right=False)
        keep = _drop_smallest(mu, ni, tiny)
        return [SIGMA + 1 / mu[k] for k in keep], None, nz, ni, None, F
    P = product(F)
    if P.rows == 1:  # (mp.eig does not take a 1 x 1 matrix)
        E, EL, ER = [P[0, 0]], mp.eye(1), mp.eye(1)
    elif vectors:
        E, EL, ER = mp.eig(P, left=True, right=True)
    else:
        E, EL, ER = mp.eig(P, left=False, right=False), None, None
    return E, _drop_smallest(E, nz, tiny), nz, ni, (EL, ER), F


def kappas(F, E, EL, ER, keep, fnorms):
    """relative structured condition numbers of the eigenvalues E[keep]: rows of EL F_1..F_{j-1}
    and columns of F_{j+1}..F_p ER, with A_j^{-1} applied on both sides for an inverted factor"""
    p = len(F)
    Fm = [a if s else inverse(a) for a, s, _ in F]
    pre, suf = [None] * p, [None] * p
    L = EL
    for j in range(p):
        pre[j] = L
        L = L * Fm[j]
    R = ER
    for j in range(p - 1, -1, -1):
        suf[j] = R
        R = Fm[j] * R
    out = []
    for k in keep:
        s = mp.mpf(0)
        for j in range(p):
            y, x = pre[j][k, :], suf[j][:, k]
            if not F[j][1]:
                y, x = y * Fm[j], Fm[j] * x
            s += mp.norm(y) * fnorms[F[j][2]] * mp.norm(x)
        d = abs((EL[k, :] * ER[:, k])[0, 0]) * abs(E[k])
        out.append(s / d)
    return out


def solve(item):
    pid, rec = item
    t0 = time.time()
    A = GA.inputs(rec)
    fnorms = [norm2(a.T) for a in A]
    dps = 60
    while True:
        mp.mp.dps = dps
        E, keep, nz, ni, vec, F = eigs(A, rec, vectors=True)
        fin = E if keep is None else [E[k] for k in keep]
        mags = [abs(z) for z in fin]
        need = 40 + int(math.ceil(float(mp.log10(max(mags) / min(mags)))))
        if need <= dps:
            break
        dps = need
    kap = None if vec is None else kappas(F, E, vec[0], vec[1], keep, fnorms)
    dps_check = int(math.ceil(1.5 * dps))
    mp.mp.dps = dps_check
    E2, keep2, _, _, _, _ = eigs(A, rec, vectors=False)
    fin2 = E2 if keep2 is None else [E2[k] for k in keep2]
    agree = float(agreement(fin, fin2))
    assert agree <= AGREE, (pid, agree)
    mp.mp.dps = dps
    order = sorted(range(len(fin)), key=lambda k: (-abs(fin[k]), -mp.im(fin[k])))
    eig, kappa = [], []
    for k in order:
        z = fin[k]
        im = mp.mpf(0) if abs(mp.im(z)) <= GA.REAL_TOL * abs(z) else mp.im(z)
        eig.append([mp.nstr(mp.re(z), 25), mp.nstr(im, 25)])
        if kap is not None:
            kappa.append(float(kap[k]))
    return pid, dict(id=pid, recipe=rec, sha256=GA.sha(A), dps=dps, dps_check=dps_check, agreement=agree,
                     nzero=nz, ninf=ni, eig=eig, kappa=kappa if kap is not None else None), time.time() - t0


def main():
    t0 = time.time()
    work = sorted(GA.PROBLEMS, key=lambda it: -(it[1]["n"] ** 3) * (it[1]["p"] + 4) * (2 if it[1]["cplx"] else 1))
    with mproc.Pool(os.cpu_count()) as pool:
        res = {pid: (g, t) for pid, g, t in pool.imap_unordered(solve, work)}
    out = {"problems": [res[pid][0] for pid, _ in GA.PROBLEMS]}
    with open(GA.GOLDEN, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    slow = max(res, key=lambda k: res[k][1])
    print("wrote", len(out["problems"]), "problems; worst agreement",
          max(g["agreement"] for g in out["problems"]), "; max digits", max(g["dps"] for g in out["problems"]),
          f"; {time.time() - t0:.0f} s ({os.cpu_count()} processes; slowest {slow} {res[slow][1]:.0f} s)")


if __name__ == "__main__":
    main()
