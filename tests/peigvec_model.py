"""Numpy model of the device eigenvector algorithm (csrc/psd_eigvecs.cuh): periodic
back-substitution on a periodic Schur form, per-row cyclic systems solved by a structured Givens QR
after power-of-two row scaling, eps pivot replacement, 2x2 blocks of the real Schur factor, factor
and chain scaling.  It is where the numerics are debugged without a GPU, and its worst backward
error on the test cases sets the GPU gate (MODEL_WORST_BE).  Also the checks the GPU tests share.

Storage layout throughout: T, Z, V [p][n][n] with each matrix column-major ([col][row]), user
factor order."""
import numpy as np

EPS = np.finfo(np.float64).eps
EV_LIM = 900
# worst ||A_l v_{l+1} - mu_l v_l|| / (n eps ||A_l||_F) the model reaches on the cases of
# tests/test_eigvecs_model.py (measured: 6.55, at n = 2, p = 8, :L, where n eps is small
# against the decomposition's own backward error); the GPU gate is 10x this
MODEL_WORST_BE = 6.6

# how often the rare branches ran since the last reset (the tests make sure each one is reached):
# a pivot replaced by eps with a nonzero right-hand side, a rescale inside the back-substitution,
# a common rescale of a vector's whole chain
COUNTS = {"pivot": 0, "solve_rescale": 0, "chain_shift": 0}


def _exp(a):
    return int(np.frexp(a)[1]) if a > 0 and np.isfinite(a) else 0


def _amax(z):
    return max(abs(z.real), abs(z.imag))


def _givens(f, g):
    """[c s; -conj(s) c] [f; g] = [r; 0] (zlartg)."""
    if g == 0:
        return 1.0, 0j, f
    if f == 0:
        return 0.0, np.conj(g) / abs(g), complex(abs(g))
    af, h = abs(f), np.hypot(abs(f), abs(g))
    return af / h, (f / af) * np.conj(g) / h, (f / af) * h


def cyclic_solve(D, mu, rhs):
    """-mu_l u_l + D_l u_{l+1} = rhs_l (l = 0..p-1, u_p = u_0), D [p][B][B], rhs [p][B].
    Returns (u [p][B], E) with the solution u * 2^E."""
    p, B = len(mu), D.shape[1]

    def entry(l, r, cb, c):
        v = -mu[l] if (cb == l and r == c) else 0j
        if cb == (l + 1) % p:
            v = v + D[l][r][c]
        return v

    def rowexp(l, r):
        mx = 0.0
        for c in range(B):
            mx = max(mx, _amax(entry(l, r, l, c)))
            if p > 1:
                mx = max(mx, _amax(entry(l, r, (l + 1) % p, c)))
        return _exp(mx)

    ex = [_exp(_amax(rhs[l][r])) - rowexp(l, r) for l in range(p) for r in range(B) if rhs[l][r] != 0]
    Er = max(ex) if ex else 0

    def load(l):
        Ad = np.zeros((B, B), complex); Bn = np.zeros((B, B), complex); rr = np.zeros(B, complex)
        for r in range(B):
            e = rowexp(l, r)
            for c in range(B):
                Ad[r, c] = np.ldexp(entry(l, r, l, c).real, -e) + 1j * np.ldexp(entry(l, r, l, c).imag, -e)
                if p > 1:
                    v = entry(l, r, (l + 1) % p, c)
                    Bn[r, c] = np.ldexp(v.real, -e) + 1j * np.ldexp(v.imag, -e)
            rr[r] = np.ldexp(rhs[l][r].real, -e - Er) + 1j * np.ldexp(rhs[l][r].imag, -e - Er)
        return Ad, Bn, rr

    G, S, rs = load(p - 1)
    rows = []
    for l in range(p - 1):
        A, Bm, r = load(l)
        F = np.zeros((B, B), complex)
        if l + 2 == p:
            F, Bm = Bm, np.zeros((B, B), complex)
        Sn = np.zeros((B, B), complex)
        for cc in range(B):
            for ss in range(B):
                if S[ss, cc] == 0:
                    continue
                c, s, rv = _givens(A[cc, cc], S[ss, cc])
                top = np.concatenate([A[cc], Bm[cc], F[cc], [r[cc]]])
                bot = np.concatenate([S[ss], Sn[ss], G[ss], [rs[ss]]])
                nt, nb = c * top + s * bot, c * bot - np.conj(s) * top
                A[cc], Bm[cc], F[cc], r[cc] = nt[:B], nt[B:2 * B], nt[2 * B:3 * B], nt[3 * B]
                S[ss], Sn[ss], G[ss], rs[ss] = nb[:B], nb[B:2 * B], nb[2 * B:3 * B], nb[3 * B]
                A[cc, cc], S[ss, cc] = rv, 0
        rows.append((A, Bm, F, r))
        S = Sn
    if B == 2 and G[1, 0] != 0:
        c, s, rv = _givens(G[0, 0], G[1, 0])
        t = np.array([G[0, 1], rs[0]]); bt = np.array([G[1, 1], rs[1]])
        nt, nb = c * t + s * bt, c * bt - np.conj(s) * t
        G[0, 1], rs[0], G[1, 1], rs[1] = nt[0], nt[1], nb[0], nb[1]
        G[0, 0], G[1, 0] = rv, 0
    u = np.zeros((p, B), complex)
    state = {"se": 0}

    def solve_tri(U, y, l):
        for rr in range(B - 1, -1, -1):
            num = y[rr] - sum(U[rr, c] * y[c] for c in range(rr + 1, B))
            pv = U[rr, rr] if abs(U[rr, rr]) >= EPS else complex(EPS)
            if abs(U[rr, rr]) < EPS and num != 0:
                COUNTS["pivot"] += 1
            if _amax(num) > 2.0 ** 900 * _amax(pv):
                COUNTS["solve_rescale"] += 1
                k = _exp(_amax(num)) - _exp(_amax(pv)) - EV_LIM + 2
                u[:] = np.ldexp(u.real, -k) + 1j * np.ldexp(u.imag, -k)
                for q in range(len(rows)):
                    rows[q] = rows[q][:3] + (rows[q][3] * 2.0 ** -k,)
                y[:] = y * 2.0 ** -k
                num = num * 2.0 ** -k
                state["se"] += k
            y[rr] = num / pv
        return y

    u[p - 1] = solve_tri(G, rs.copy(), p - 1)
    for l in range(p - 2, -1, -1):
        A, Bm, F, r = rows[l]
        y = r - Bm @ u[l + 1] - F @ u[p - 1]
        u[l] = solve_tri(A, y, l)
    return u, Er + state["se"]


def _maps(p, lr):
    fac = (lambda j: p - 1 - j) if lr == "L" else (lambda j: j)
    uvec = (lambda j: (p - j) % p) if lr == "L" else (lambda j: j)
    return fac, uvec


def effective_selection(T, lr, select=None):
    """Columns that get vectors: selected ones, and both members of a pair when either is."""
    p, n = T.shape[0], T.shape[1]
    T1 = T[p - 1 if lr == "L" else 0].T
    real = not np.iscomplexobj(T)
    out, c = [], 0
    while c < n:
        pair = real and c + 1 < n and T1[c + 1, c] != 0
        want = select is None or select[c] or (pair and select[c + 1])
        if want:
            out += [c, c + 1] if pair else [c]
        c += 2 if pair else 1
    return out


def eigvecs(T, Z, lr="R", select=None):
    """Model of one problem of psd_reigvecs_batched / psd_ceigvecs_batched; V [p][n][n] complex."""
    p, n = T.shape[0], T.shape[1]
    fac, uvec = _maps(p, lr)
    real = not np.iscomplexobj(T)
    R = [T[fac(j)].T.astype(complex) for j in range(p)]  # math orientation
    V = np.zeros((p, n, n), complex)
    cols = effective_selection(T, lr, select)
    # factor scales over the leading part up to the last vector (upper part and first subdiagonal)
    kk = max(cols) + 1 if cols else 0
    sc = []
    for j in range(p):
        Rl = np.triu(R[j][:kk, :kk], -1)
        mx = np.max(np.maximum(np.abs(Rl.real), np.abs(Rl.imag)), initial=0.0)
        sc.append(2.0 ** -min(1000, max(-1000, _exp(mx))) if mx > 0 else 1.0)
    Rs = [R[j] * sc[j] for j in range(p)]
    for c in cols:
        pair = real and c + 1 < n and R[0][c + 1, c] != 0
        if real and c > 0 and R[0][c, c - 1] != 0:
            continue  # second member: conjugate of the first
        top = c + 1 if pair else c
        x = np.zeros((p, n), complex)
        s = np.zeros((p, n), complex)
        mu = np.zeros(p, complex)
        r = top
        while r >= 0:
            two = real and r >= 1 and R[0][r, r - 1] != 0
            i0, bs = (r - 1, 2) if two else (r, 1)
            if i0 == c:
                if bs == 1:
                    mu = np.array([Rs[j][c, c] for j in range(p)])
                    x[:, c] = 1.0
                else:
                    Pm = np.eye(2)
                    for j in range(p):
                        Pm = Pm @ Rs[j][c:c + 2, c:c + 2].real
                        Pm = np.ldexp(Pm, -_exp(np.abs(Pm).max()))
                    t = 0.5 * (Pm[0, 0] + Pm[1, 1])
                    h = 0.5 * (Pm[0, 0] - Pm[1, 1])
                    lam = complex(t, np.sqrt(max(0.0, -(h * h + Pm[0, 1] * Pm[1, 0]))))
                    lmd = lam - Pm[1, 1]
                    y1 = (lam - Pm[0, 0]) / Pm[0, 1] if abs(Pm[0, 1]) >= abs(lmd) else Pm[1, 0] / lmd
                    x[0, c], x[0, c + 1] = 1.0, y1
                    nx = y1
                    for j in range(p - 1, -1, -1):
                        B = Rs[j][c:c + 2, c:c + 2]
                        z0 = B[0, 0] + B[0, 1] * nx
                        z1 = B[1, 0] + B[1, 1] * nx
                        mu[j] = z0
                        if j > 0:
                            nx = z1 / z0
                            x[j, c], x[j, c + 1] = 1.0, nx
            else:
                D = np.array([Rs[j][i0:i0 + bs, i0:i0 + bs] for j in range(p)])
                u, E = cyclic_solve(D, mu, -s[:, i0:i0 + bs])
                nz = [_exp(_amax(v)) for v in u.ravel() if v != 0]
                if nz and E + max(nz) > EV_LIM:
                    COUNTS["chain_shift"] += 1
                    sh = E + max(nz) - EV_LIM
                    x, s = x * 2.0 ** -sh, s * 2.0 ** -sh
                    E -= sh
                x[:, i0:i0 + bs] = np.ldexp(u.real, E) + 1j * np.ldexp(u.imag, E)
            for j in range(p):
                s[j, :i0] += Rs[j][:i0, i0:i0 + bs] @ x[(j + 1) % p, i0:i0 + bs]
            r = i0 - 1
        for j in range(p):
            u = uvec(j)
            v = Z[u].T.astype(complex) @ x[j]
            am = np.abs(v)
            im = int(np.argmax(am))
            w = v * 2.0 ** -_exp(am[im])
            w = w * (np.conj(w[im]) / abs(w[im])) / np.linalg.norm(w)
            w[im] = abs(w[im])
            if real and not pair:
                w = w.real + 0j
            V[u, c] = w
            if pair:
                V[u, c + 1] = np.conj(w)
    return V


# ---------------------------------------------------------------------------------------------
# checks shared with the GPU tests
# ---------------------------------------------------------------------------------------------
def check_contract(T, V, lam, lr, cols=None):
    """Unit norms, phase rule, exact zeros, exact conjugate pairs, real vectors of real eigenvalues."""
    p, n = T.shape[0], T.shape[1]
    real = not np.iscomplexobj(T)
    T1 = T[p - 1 if lr == "L" else 0].T
    cols = effective_selection(T, lr) if cols is None else cols
    for c in range(n):
        for l in range(p):
            v = V[l, c]
            if c not in cols:
                assert not v.any(), c
                continue
            assert abs(np.linalg.norm(v) - 1.0) <= 1e-14, (c, l, np.linalg.norm(v))
            a = np.abs(v)
            i = int(np.argmax(a))
            if not (v[i].imag == 0 and v[i].real > 0):  # a near-tie decided by the device's hypot
                j = [k for k in range(n) if a[k] >= a.max() * (1 - 4 * EPS) and v[k].imag == 0 and v[k].real > 0]
                assert j, (c, l)
            if real:
                first = c + 1 < n and T1[c + 1, c] != 0
                second = c > 0 and T1[c, c - 1] != 0
                if second:
                    assert np.array_equal(v, np.conj(V[l, c - 1]))
                elif not first:
                    assert not v.imag.any()
    return 0.0


def _pow2(A):
    """A times the power of two bringing its largest entry into [0.5, 1), and that exponent."""
    mx = np.abs(A).max()
    e = _exp(mx) if mx > 0 else 0
    return (np.ldexp(A.real, -e) + (1j * np.ldexp(A.imag, -e) if np.iscomplexobj(A) else 0)), e


def backward_errors(A, V, lr, cols=None):
    """||A_l v_{l+1} - mu_l v_l|| / (n eps ||A_l||_F) (:R; :L  A_l v_l - mu_l v_{l+1}) with
    mu_l = v_l^H A_l v_{l+1} (:L  v_{l+1}^H A_l v_l), every A_l taken at the power of two that
    brings its largest entry into [0.5, 1) (the ratio does not depend on it).  Returns (ratios
    [len(cols)][p], {k: prod mu_l} for the unscaled factors)."""
    p, n = A.shape[0], A.shape[1]
    cols = range(n) if cols is None else cols
    As = []
    shift = 0
    for l in range(p):
        a, e = _pow2(A[l].T)
        As.append(a)
        shift += e
    out, prods = [], {}
    for k in cols:
        row = []
        m, ex = 1.0 + 0j, 0
        for l in range(p):
            ln = (l + 1) % p
            if lr == "R":
                y = As[l] @ V[ln, k]
                mu = np.vdot(V[l, k], y)
                r = y - mu * V[l, k]
            else:
                y = As[l] @ V[l, k]
                mu = np.vdot(V[ln, k], y)
                r = y - mu * V[ln, k]
            nA = np.linalg.norm(As[l])
            row.append(np.linalg.norm(r) / (n * EPS * nA) if nA > 0 else np.linalg.norm(r))
            m *= mu
            e = _exp(abs(m)) if m != 0 else 0
            m, ex = m * 2.0 ** -e, ex + e
        prods[k] = m * 2.0 ** (ex + shift) if m != 0 else 0j
        out.append(row)
    return np.array(out), prods


def sine(x, v):
    """Sine of the angle between unit vectors x and v (the projection residual: no cancellation)."""
    return float(np.linalg.norm(v - np.vdot(x, v) * x))


def angle_to_mpmath(A, V, lam, lr, mp, dps=40):
    """Largest angle (sine) between v_l and the mpmath eigenvector of the l-th cyclic product."""
    p, n = A.shape[0], A.shape[1]
    worst = 0.0
    with mp.workdps(dps):
        Am = [mp.matrix(A[l].T.tolist()) for l in range(p)]
        for l in range(p):
            order = ([(l + i) % p for i in range(p)] if lr == "R" else
                     [(l - 1 - i) % p for i in range(p)])
            Pm = mp.eye(n)
            for j in order:
                Pm = Pm * Am[j]
            E, ER = mp.eig(Pm)
            Ec = np.array([complex(e) for e in E])
            for k in range(n):
                j = int(np.argmin(np.abs(Ec - lam[k])))
                x = np.array([complex(ER[i, j]) for i in range(n)])
                x /= np.linalg.norm(x)
                worst = max(worst, sine(x, V[l, k]))
    return worst


def planted_blocks(n, p, batch, seed):
    """Real periodic Schur forms (:R) with complex-pair 2x2 blocks at rows 0-1 and n-2..n-1,
    random orthogonal Z; returns (T, Z, A) in storage layout, A_l = Z_l T_l Z_{l+1}'."""
    rng = np.random.default_rng(seed)
    T = np.zeros((batch, p, n, n)); Z = np.zeros_like(T); A = np.zeros_like(T)
    for b in range(batch):
        Tm = [np.triu(rng.standard_normal((n, n))) for _ in range(p)]
        for i0 in (0, n - 2):
            Tm[0][i0 + 1, i0] = 1.0 + rng.random()
            Tm[0][i0, i0 + 1] = -(1.0 + rng.random())  # a rotation-like block: complex eigenvalues
            Tm[0][i0, i0] = Tm[0][i0 + 1, i0 + 1] = 0.3
            for j in range(1, p):  # the other blocks a multiple of I: the product keeps complex eigenvalues
                Tm[j][i0, i0] = Tm[j][i0 + 1, i0 + 1] = 0.5 + rng.random()
                Tm[j][i0, i0 + 1] = 0.0
        Zm = [np.linalg.qr(rng.standard_normal((n, n)))[0] for _ in range(p)]
        for l in range(p):
            T[b, l] = Tm[l].T
            Z[b, l] = Zm[l].T
            A[b, l] = (Zm[l] @ Tm[l] @ Zm[(l + 1) % p].T).T
    return T, Z, A


def planted_defective(n, p, batch, seed, cplx=False):
    """Exactly defective periodic Schur forms (:R): T_1 = 2 I + random strictly upper, the other
    factors unit upper triangular, random orthogonal (unitary) Z, so every eigenvalue is 2 exactly
    and every cyclic system of the back-substitution is singular.  Returns (T, Z, A) in storage
    layout, A_l = Z_l T_l Z_{l+1}'."""
    rng = np.random.default_rng(seed)
    dt = complex if cplx else float
    T = np.zeros((batch, p, n, n), dt); Z = np.zeros_like(T); A = np.zeros_like(T)

    def g(*s):
        return rng.standard_normal(s) + (1j * rng.standard_normal(s) if cplx else 0)
    for b in range(batch):
        Tm = [np.triu(g(n, n), 1) + (2.0 if l == 0 else 1.0) * np.eye(n) for l in range(p)]
        Zm = [np.linalg.qr(g(n, n))[0] for _ in range(p)]
        for l in range(p):
            T[b, l] = Tm[l].T
            Z[b, l] = Zm[l].T
            A[b, l] = (Zm[l] @ Tm[l] @ Zm[(l + 1) % p].conj().T).T
    return T, Z, A


def planted_singular_chain(n, p, batch, seed):
    """Periodic Schur forms (:R) with a repeated zero eigenvalue from singular factors: the last row
    has a zero diagonal entry in every factor, the other rows have 1 in factors 1..p-1 and 0 in
    factor p, random strictly upper parts, random orthogonal Z.  The cyclic systems of the last
    vector then have p eps pivots in a row (growth about eps^-p), which needs the rescale inside
    the back-substitution for p >= 18.  Returns (T, Z, A) in storage layout."""
    rng = np.random.default_rng(seed)
    T = np.zeros((batch, p, n, n)); Z = np.zeros_like(T); A = np.zeros_like(T)
    for b in range(batch):
        Tm = []
        for l in range(p):
            d = np.full(n, 1.0 if l < p - 1 else 0.0)
            d[-1] = 0.0
            Tm.append(np.triu(rng.standard_normal((n, n)), 1) + np.diag(d))
        Zm = [np.linalg.qr(rng.standard_normal((n, n)))[0] for _ in range(p)]
        for l in range(p):
            T[b, l] = Tm[l].T
            Z[b, l] = Zm[l].T
            A[b, l] = (Zm[l] @ Tm[l] @ Zm[(l + 1) % p].T).T
    return T, Z, A


def schur_eigs(T, lr):
    """Eigenvalues of a real periodic Schur form (pairs: positive imaginary part first)."""
    p, n = T.shape[0], T.shape[1]
    fac, _ = _maps(p, lr)
    R = [T[fac(j)].T for j in range(p)]
    lam = np.zeros(n, complex)
    c = 0
    while c < n:
        if c + 1 < n and R[0][c + 1, c] != 0:
            P = np.eye(2)
            for j in range(p):
                P = P @ R[j][c:c + 2, c:c + 2]
            w = np.linalg.eigvals(P)
            w = w[np.argsort(-w.imag)]
            lam[c:c + 2] = w
            c += 2
        else:
            lam[c] = np.prod([R[j][c, c] for j in range(p)])
            c += 1
    return lam
