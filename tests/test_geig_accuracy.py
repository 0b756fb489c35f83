"""CPU checks of the per-eigenvalue gate of the generalized paths (tests/geigacc.py) and of its ground
truth (tests/golden/geigacc_golden.json): the inputs still come out of their recipes, the ground
truth is converged, the numpy oracle passes the gate where it can represent the problem, the gate
catches what a gate relative to the largest eigenvalue does not, and the exponent bookkeeping of the
eigenvalue products (safeprod, tri_block_product in the CUDA kernels) stays exact at the ends of the
double range."""
import math

import mpmath as mp
import numpy as np
import pytest

import geigacc as GA
import psd_checks as K

GOLD = {g["id"]: g for g in GA.load()["problems"]}
IDS = [pid for pid, _ in GA.PROBLEMS]
ORACLE_MAX_N = 24   # the numpy oracle takes seconds per problem at N = 24, minutes at N = 64

# Problems on which the numpy oracle, a restatement of the reference algorithm, fails.  It does not
# normalise the factors: with a factor subnormal throughout or near the largest double its QZ does
# not converge ("info") or returns wrong eigenvalues, and with whole factors at 1e+-300 it returns
# infinite or wrong eigenvalues ("gate").  r-sub1 and the N = 1, 2 edge cases (NaN, wrong
# eigenvalues, or minutes of iteration) are not run.  (Its eigenvalue products
# also multiply and divide by the raw diagonal entries, gpsd_common.py safeprod, which overflows or
# loses bits at the ends of the range; the CUDA kernels split every entry into mantissa and exponent
# first, DESIGN.md section 6.)
ORACLE_FAILS = {**{f"{c}-{k}-n12p3": "info" for c, k in (("c", "sub0"), ("c", "sub1"), ("c", "huge"), ("r", "huge"))},
                **{f"{c}-{k}-n8p3": "gate" for c in "cr" for k in ("big", "small")}, "r-sub0-n12p3": "gate"}
ORACLE_SKIP = {"r-sub1-n12p3"} | {pid for pid in IDS if "-edge" in pid}


def test_golden_covers_every_problem():
    assert IDS == [g["id"] for g in GA.load()["problems"]]
    for pid, rec in GA.PROBLEMS:
        assert GOLD[pid]["recipe"] == rec, pid


@pytest.mark.parametrize("pid", IDS)
def test_golden_inputs_and_convergence(pid):
    g = GOLD[pid]
    rec = g["recipe"]
    A = GA.inputs(rec)
    assert np.isfinite(A).all()
    assert GA.sha(A) == g["sha256"], "the recipe no longer gives the inputs the ground truth was computed for"
    ref, kappa = GA.truth(g)
    assert len(ref) + g["nzero"] + g["ninf"] == rec["n"]
    assert (g["nzero"], g["ninf"]) == GA.holes(rec)
    assert (kappa is None) == (g["ninf"] > 0)
    assert kappa is None or (kappa >= 1.0).all()
    assert g["agreement"] <= 1e-30 and g["dps_check"] >= 1.5 * g["dps"]
    mags = [abs(z) for z in ref]
    assert g["dps"] >= 40 + float(mp.log10(max(mags) / min(mags)))
    if not rec["cplx"]:  # conjugate pairs
        up = sorted((z for z in ref if mp.im(z) > 0), key=abs)
        down = sorted((mp.conj(z) for z in ref if mp.im(z) < 0), key=abs)
        assert len(up) == len(down) and all(abs(a - b) <= 1e-20 * abs(a) for a, b in zip(up, down))


def _oracle(oracle, rec, A, want_tz, maxitfac=None):
    from oracle import gpsd as OG
    f = OG.cpschur_batched if rec["cplx"] else OG.rgpschur_batched
    kw = {} if maxitfac is None else {"maxitfac": maxitfac}
    T, _, al, be, sc, info = f(A[None], rec["S"], left=rec["left"], hessut=rec["hessut"], wantT=want_tz,
                               wantZ=want_tz, **kw)
    return T[0], al[0], be[0], sc[0], int(info[0])


SMALL = [pid for pid in IDS if GOLD[pid]["recipe"]["n"] <= ORACLE_MAX_N and pid not in ORACLE_SKIP]


@pytest.mark.parametrize("want_tz", [False, True], ids=["eig", "TZ"])
@pytest.mark.parametrize("pid", SMALL)
def test_oracle_passes_the_gate(oracle, pid, want_tz):
    """The numpy oracle meets the gate with a margin of 4 on the first-order branch, and its
    eigenvalues agree with the diagonal blocks of its T; on the problems of ORACLE_FAILS it fails."""
    g = GOLD[pid]
    rec = g["recipe"]
    if ORACLE_FAILS.get(pid) == "info":  # (an iteration limit of 10 per eigenvalue keeps it quick)
        assert _oracle(oracle, rec, GA.inputs(rec), want_tz, maxitfac=10)[4] == rec["n"]
        return
    if ORACLE_FAILS.get(pid) == "gate":
        T, al, be, sc, info = _oracle(oracle, rec, GA.inputs(rec), want_tz)
        assert info == 0
        with pytest.raises(AssertionError, match="eigenvalues"):
            GA.check(g, al, be, sc, what=pid)
        return
    T, al, be, sc, info = _oracle(oracle, rec, GA.inputs(rec), want_tz)
    assert info == 0
    err, allowed, cond = GA.check(g, al, be, sc, what=pid)
    assert (err[cond] <= allowed[cond] / 4).all(), np.max(err[cond] / allowed[cond])
    if not rec["cplx"]:
        GA.check_pairs(al, be, sc, g)
    if want_tz:
        GA.check_against_T(T, al, be, sc, rec["S"], rec["left"], GA.T_tolerance(g, al, be, sc))


def _oracle_values(oracle, pid):
    g = GOLD[pid]
    rec = g["recipe"]
    _, al, be, sc, info = _oracle(oracle, rec, GA.inputs(rec), False)
    assert info == 0
    GA.check(g, al, be, sc)
    return g, al, be, sc


@pytest.mark.parametrize("pid", ["r-n24p10-C5L-b0", "c-n24p4-oneminus-b1", "r-n24p10-C5L-b1"])
def test_gate_catches_one_small_eigenvalue_off(oracle, pid):
    """A relative error of 1e-9 in one small eigenvalue fails the gate; an absolute gate at
    100 N eps |lambda|max (the one of the oracle parity tests) lets it through."""
    g, al, be, sc = _oracle_values(oracle, pid)
    n = g["recipe"]["n"]
    ref, kappa = GA.truth(g)
    allowed, cond = GA.bounds(kappa, len(ref), n)
    k = min((k for k in range(len(ref)) if cond[k] and allowed[k] < 1e-10), key=lambda k: abs(ref[k]))
    assert abs(ref[k]) < 1e-3 * max(abs(z) for z in ref)
    i = GA.match(ref, GA.values(al, be, sc))[k]
    bad = al.copy()
    bad[i] *= 1 + 1e-9
    with pytest.raises(AssertionError, match="outside the gate"):
        GA.check(g, bad, be, sc)
    lam = [complex(v) for v in GA.values(bad, be, sc)]
    assert K.match_eigs([complex(z) for z in ref], lam) <= 100 * n * GA.EPS * max(abs(complex(z)) for z in ref)


@pytest.mark.parametrize("pid", ["r-n12p3-alt-b0", "c-n12p6-C3-b0", "c-hole1"])
def test_gate_catches_an_alphascale_off_by_one(oracle, pid):
    g, al, be, sc = _oracle_values(oracle, pid)
    for i in (0, len(sc) - 1):
        bad = sc.copy()
        bad[i] += 1
        with pytest.raises(AssertionError, match="outside the gate"):
            GA.check(g, al, be, bad)


@pytest.mark.parametrize("pid", ["r-hole2", "c-hole3"])
def test_gate_catches_a_missing_infinite_eigenvalue(oracle, pid):
    g, al, be, sc = _oracle_values(oracle, pid)
    assert g["ninf"] == 1
    i = int(np.flatnonzero(be == 0)[0])
    bad = be.copy()
    bad[i] = 1.0
    with pytest.raises(AssertionError, match="infinite eigenvalues"):
        GA.check(g, al, bad, sc)
    bad = al.copy()
    bad[i] = 0.0  # 0 / 0
    with pytest.raises(AssertionError, match="undefined"):
        GA.check(g, bad, be, sc)


def test_gate_catches_a_missing_pair():
    g = GOLD["r-n12p3-alt-b0"]
    al = np.array([2 + 1j, 2 - 1j, 0.5])
    one, zero = np.ones(3), np.zeros(3, dtype=np.int64)
    with pytest.raises(AssertionError, match="does not open a pair"):
        GA.check_pairs(al[[1, 0, 2]], one, zero, g)
    with pytest.raises(AssertionError, match="not a conjugate pair"):
        GA.check_pairs(al, one, np.array([0, 1, 0]), g)


# ---- exponent bookkeeping of the eigenvalue products (psd_gen_common.cuh safeprod,
# psd_cplx_qz.cuh tri_block_product), restated ----

def split(x):
    """x = m 2^k exactly with the larger of |Re m|, |Im m| in [0.5, 1) (psd_gen_common.cuh pow2_split)"""
    big = max(abs(x.real), abs(x.imag)) if isinstance(x, complex) else abs(x)
    if big == 0 or not math.isfinite(big):
        return x, 0
    _, k = math.frexp(big)
    if isinstance(x, complex):
        return complex(math.ldexp(x.real, -k), math.ldexp(x.imag, -k)), k
    return math.ldexp(x, -k), k


def safeprod(S, xs):
    """safeprod of the kernels: prod x_i^{s_i} = alpha / beta 2^scale, |alpha| in [1, 2) or 0,
    beta in {0, 1}; every x_i is split into mantissa and exponent before it enters the product."""
    alpha, beta, scale = (1 + 0j) if any(isinstance(x, complex) for x in xs) else 1.0, 1, 0
    for s, x in zip(S, xs):
        if not s and x == 0:
            beta = 0
        else:
            m, k = split(x)
            alpha = alpha * m if s else alpha / m
            scale += k if s else -k
        aa = abs(alpha)
        if aa == 0:
            alpha, scale = alpha * 0, 0
            if beta == 0:
                return alpha, beta, scale
        else:
            _, e = math.frexp(aa)
            alpha = alpha * 2.0 ** -(e - 1)
            if abs(alpha) >= 2.0:
                alpha, e = alpha * 0.5, e + 1
            elif abs(alpha) < 1.0:
                alpha, e = alpha * 2.0, e - 1
            scale += e - 1
    return alpha, beta, scale


def tri_block_product(S, blocks):
    """tri_block_product of the kernels: Tm 2^e = prod_l U_l^{s_l} of upper triangular K x K blocks.
    A direct block is split into mantissas and one exponent before the product; an inverted one entry
    by entry, and the quotients keep one exponent per entry (N = q 2^x): each entry's terms are summed
    at the exponent of the largest and divided by the mantissa of the diagonal.  Then renormalised."""
    K = len(blocks[0])
    Tm, e = np.eye(K), 0
    for s, U in zip(S, blocks):
        U = np.triu(np.array(U, dtype=float))
        if s:
            _, ku = math.frexp(np.abs(U).max())
            U = np.ldexp(U, -ku)
            N = Tm @ U
            e += ku
            _, ex = math.frexp(np.abs(N).max())
            Tm = np.ldexp(N, -ex)
        else:
            q, x = np.zeros((K, K)), np.zeros((K, K), dtype=int)
            for r in range(K):
                for c in range(r, K):
                    sp = [split(float(U[k, c])) for k in range(K)]
                    terms = [k for k in range(r, c) if q[r, k] != 0 and U[k, c] != 0]
                    xm = max([0] * int(Tm[r, c] != 0) + [int(x[r, k]) + sp[k][1] for k in terms], default=0)
                    acc = math.ldexp(Tm[r, c], -xm)
                    for k in range(r, c):
                        sh = int(x[r, k]) + sp[k][1] - xm if k in terms else 0
                        acc = acc - q[r, k] * math.ldexp(sp[k][0], sh)
                    md, kd = math.frexp(U[c, c])
                    q[r, c], x[r, c] = acc / md, xm - kd
            ex = max(math.frexp(q[r, c])[1] + int(x[r, c]) for r in range(K) for c in range(r, K) if q[r, c] != 0)
            Tm = np.array([[math.ldexp(q[r, c], int(x[r, c]) - ex) for c in range(K)] for r in range(K)])
        e += ex
    return Tm, e


def _tri_inv(M):
    """inverse of an upper triangular mpmath matrix by back substitution (mp.inverse calls one with
    a diagonal entry far below its norm singular)"""
    K = M.rows
    X = mp.zeros(K, K)
    for c in range(K):
        for i in range(c, -1, -1):
            X[i, c] = ((1 if i == c else 0) - mp.fsum(M[i, k] * X[k, c] for k in range(i + 1, c + 1))) / M[i, i]
    return X


def _mp_prod(S, xs):
    with mp.workdps(50):
        v = mp.mpf(1)
        for s, x in zip(S, xs):
            v = v * mp.mpc(x) if s else v / mp.mpc(x)
        return v


EDGE = [1.75e308, 9.5e307, 1e-310, 5e-324, 2.2250738585072014e-308, 3e-320, 1.0, 0.7]


@pytest.mark.parametrize("cplx", [False, True])
@pytest.mark.parametrize("S", [[1, 1, 1], [1, 0, 1], [1, 0, 0], [0, 0, 0]])
def test_safeprod_exponents_at_the_range_edges(S, cplx):
    """The products of diagonals at the ends of the double range (above 9e307, subnormal) agree
    with mpmath to a few eps; the raw product of the reference overflows or loses bits there."""
    rng = np.random.default_rng(3)
    for trial in range(200):
        xs = [float(rng.choice(EDGE)) * float(rng.uniform(0.5, 1.0)) * rng.choice([-1, 1]) for _ in S]
        if cplx:
            xs = [complex(x, x * float(rng.uniform(-1, 1))) for x in xs]
        a, b, sc = safeprod(S, xs)
        assert b == 1 and 1.0 <= abs(a) < 2.0
        want = _mp_prod(S, xs)
        got = mp.mpc(a) * mp.ldexp(1, sc)
        assert float(abs(got - want) / abs(want)) <= 4 * len(S) * GA.EPS, (xs, a, sc)


def test_safeprod_zero_and_infinite():
    assert safeprod([1, 0, 1], [1e-310, 0.0, 3.0])[1] == 0
    a, b, sc = safeprod([1, 0, 1], [0.0, 2.0, 1e308])
    assert a == 0 and b == 1 and sc == 0


@pytest.mark.parametrize("K", [2, 3])
@pytest.mark.parametrize("S", [[1, 1, 1], [1, 0, 1], [0, 0, 1]])
def test_tri_block_product_at_the_range_edges(S, K):
    """The product of triangular blocks, some inverted, with diagonals subnormal or near overflow, or
    an inverted block with one diagonal entry far below the rest (its inverse then has entries near
    1e+310 beside ones of order one), against mpmath: finite, a few eps relative to the largest entry.
    (The running product keeps one exponent, so its entries more than 2^1074 below its largest flush
    to zero; a second such block later in the chain could need them.)"""
    rng = np.random.default_rng(5 + K)
    for trial in range(50):
        blocks = []
        mixed = trial % 2 and 0 in S
        for j, s in enumerate(S):
            U = np.triu(rng.uniform(0.5, 1.0, (K, K)) * rng.choice([-1, 1], (K, K)))
            U = U * float(rng.choice([1.7e308, 1e-310, 3e-320, 1.0]))
            if mixed and j == S.index(0):  # one diagonal entry far below the rest of its block
                i = int(rng.integers(K))
                U[i, i] = float(rng.choice([1e-310, 3e-320, 1e-300])) * rng.uniform(0.5, 1.0)
            blocks.append(U)
        Tm, e = tri_block_product(S, blocks)
        assert np.isfinite(Tm).all() and 0.5 <= np.abs(Tm).max() < 1.0
        with mp.workdps(50):
            P = mp.eye(K)
            for s, U in zip(S, blocks):
                M = mp.matrix(U.tolist())
                P = P * (M if s else _tri_inv(M))
            got = mp.matrix(Tm.tolist()) * mp.ldexp(1, e)
            scale = max(abs(P[r, c]) for r in range(K) for c in range(K))
            for r in range(K):
                for c in range(r, K):
                    assert float(abs(got[r, c] - P[r, c]) / scale) <= 16 * len(S) * GA.EPS, (r, c)
