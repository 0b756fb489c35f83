"""Eigenvectors of periodic Schur results on the device (psd_reigvecs_batched,
psd_ceigvecs_batched): backward error per factor and vector, eigenvalue consistency, high-precision
ground truth, shapes, edge cases and the output contract.  Every problem goes through the real
pschur entry points first; the checked problems sit at the first, an inner and the last index of
a prime-sized batch."""
import numpy as np
import pytest

import eigacc as EA
import peigvec_model as M

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
# ||A_l v_{l+1} - mu_l v_l|| <= C_BE n eps ||A_l||_F.  The numpy model of the same algorithm
# (tests/peigvec_model.py, tests/test_eigvecs_model.py) reaches at most M.MODEL_WORST_BE (6.6, measured 6.55) on
# these cases; C_BE is 10x that.
C_BE = 10 * M.MODEL_WORST_BE
BATCH = 7


def _schur(psd, A, lr):
    if A.dtype == np.complex128:
        T, Z, al, be, sc, info = psd.gpschur_batched(A, [True] * A.shape[1], lr)
        lam = psd.gvalues(al, be, sc)
    else:
        T, Z, lam, info = psd.pschur_batched(A, lr)
    assert (info == 0).all()
    return T, Z, lam


def _rand(seed, n, p, count, cplx):
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((count, p, n, n))
    if cplx:
        A = A + 1j * rng.standard_normal((count, p, n, n))
    return A


def _run(psd, A, lr, select=None):
    T, Z, lam = _schur(psd, A, lr)
    V, info = psd.eigvecs_batched(T, Z, lr, select)
    assert (info == 0).all()
    return T, Z, lam, V


def _check(A, T, V, lam, lr, cols=None, eig_rel=None):
    """Contract and backward error of one problem (storage layout); returns worst gate ratio."""
    n = A.shape[1]
    worst = M.check_contract(T, V, lam, lr, cols)
    be, prods = M.backward_errors(A, V, lr, cols)
    assert be.max(initial=0.0) <= C_BE, be.max()
    if eig_rel is not None:
        for k, pr in prods.items():
            assert abs(pr - lam[k]) <= eig_rel * abs(lam[k]) + 1e-300, (k, pr, lam[k])
    return max(worst, be.max(initial=0.0))


@pytest.mark.parametrize("cplx", [False, True])
@pytest.mark.parametrize("lr", ["R", "L"])
@pytest.mark.parametrize("n,p", [(1, 1), (2, 2), (5, 3), (32, 8), (50, 3), (64, 8), (5, 1), (32, 2), (2, 8)])
def test_shapes(psd, n, p, lr, cplx):
    A = _rand(1000 + 7 * n + p, n, p, BATCH, cplx)
    T, Z, lam, V = _run(psd, A, lr)
    for b in (0, 3, BATCH - 1):
        _check(A[b], T[b], V[b], lam[b], lr, eig_rel=1e-8)


@pytest.mark.parametrize("cplx", [False, True])
@pytest.mark.parametrize("lr", ["R", "L"])
def test_selection_and_structure(psd, lr, cplx):
    n, p = 12, 3
    A = _rand(77, n, p, BATCH, cplx)
    T, Z, lam = _schur(psd, A, lr)
    rng = np.random.default_rng(5)
    sel = rng.random((BATCH, n)) < 0.4
    V, info = psd.eigvecs_batched(T, Z, lr, sel)
    assert (info == 0).all()
    Vall, _ = psd.eigvecs_batched(T, Z, lr)
    for b in range(BATCH):
        cols = M.effective_selection(T[b], lr, sel[b])
        for c in range(n):
            if c in cols:
                assert np.array_equal(V[b, :, c], Vall[b, :, c])  # per-column work: same bits
            else:
                assert not V[b, :, c].any()
        _check(A[b], T[b], V[b], lam[b], lr, cols)


@pytest.mark.parametrize("lr", ["R", "L"])
@pytest.mark.parametrize("cplx", [False, True])
def test_ground_truth_mpmath(psd, lr, cplx):
    mp = pytest.importorskip("mpmath")
    n, p = 8, 3
    A = _rand(4242, n, p, BATCH, cplx)
    T, Z, lam, V = _run(psd, A, lr)
    for b in (0, 3, BATCH - 1):
        worst = M.angle_to_mpmath(A[b], V[b], lam[b], lr, mp)
        assert worst <= 1e-10, worst


@pytest.mark.parametrize("cplx", [False, True])
def test_ground_truth_p1_scipy(psd, cplx):
    import scipy.linalg as sl
    n = 10
    A = _rand(99, n, 1, BATCH, cplx)
    T, Z, lam, V = _run(psd, A, "R")
    for b in (0, 3, BATCH - 1):
        w, X = sl.eig(A[b, 0].T)
        for k in range(n):
            j = int(np.argmin(np.abs(w - lam[b, k])))
            x = X[:, j] / np.linalg.norm(X[:, j])
            assert M.sine(x, V[b, 0, k]) <= 1e-10


def test_blocks_in_first_and_last_rows(psd):
    """A hand-made real periodic Schur form with 2x2 blocks at rows 0-1 and n-2..n-1."""
    n, p = 9, 3
    T, Z, A = M.planted_blocks(n, p, BATCH, seed=3)
    V, info = psd.eigvecs_batched(T, Z, "R")
    assert (info == 0).all()
    for b in (0, 3, BATCH - 1):
        lam = M.schur_eigs(T[b], "R")
        _check(A[b], T[b], V[b], lam, "R", eig_rel=1e-10)


def test_n32_p8_eigenvalue_path_batch(psd):
    """The N = 32, p = 8 shape that the eigenvalue-only kernels serve, with T and Z from the T/Z call."""
    n, p, batch = 32, 8, 37
    A = _rand(31, n, p, batch, False)
    T, Z, lam, V = _run(psd, A, "R")
    for b in (0, 17, batch - 1):
        _check(A[b], T[b], V[b], lam[b], "R", eig_rel=1e-8)


def test_large_n1024(psd):
    n, p = 1024, 4
    A = _rand(1024, n, p, 1, False)
    T, Z, lam = _schur(psd, A, "R")
    pairs = np.flatnonzero(np.abs(lam[0].imag) > 0)
    sel = np.zeros((1, n), dtype=bool)
    sel[0, np.linspace(0, n - 1, 14).astype(int)] = True
    sel[0, pairs[0]] = True  # one member of a complex pair
    V, info = psd.eigvecs_batched(T, Z, "R", sel)
    assert info[0] == 0
    cols = M.effective_selection(T[0], "R", sel[0])
    assert len(cols) >= 16 and pairs[0] in cols
    for c in range(n):
        if c not in cols:
            assert not V[0, :, c].any()
    _check(A[0], T[0], V[0], lam[0], "R", cols, eig_rel=1e-6)


@pytest.mark.parametrize("n,p,cplx,nsel", [(24, 2, False, None), (40, 3, False, None), (24, 3, True, None),
                                          (200, 2, False, 6), (200, 2, True, 6)])
def test_exactly_defective(psd, n, p, cplx, nsel):
    """Planted forms whose eigenvalues are all exactly 2 (tests/peigvec_model.py: planted_defective):
    eps pivots with nonzero right-hand sides and chain rescales in every vector, in the
    shared-memory kernel and, at n = 200 with a few vectors, in global memory."""
    batch = 3 if n >= 192 else BATCH
    T, Z, A = M.planted_defective(n, p, batch, seed=n + p, cplx=cplx)
    sel = None
    if nsel:
        sel = np.zeros((batch, n), dtype=bool)
        sel[:, np.linspace(0, n - 1, nsel).astype(int)] = True
    V, info = psd.eigvecs_batched(T, Z, "R", sel)
    assert (info == 0).all()
    lam = np.full(n, 2.0 + 0j)
    for b in (0, batch // 2, batch - 1):
        cols = M.effective_selection(T[b], "R", None if sel is None else sel[b])
        _check(A[b], T[b], V[b], lam, "R", cols)


def test_singular_chain(psd):
    """A repeated zero eigenvalue from singular factors with p = 24 eps pivots in one cyclic system
    (tests/peigvec_model.py: planted_singular_chain): the rescale inside the back-substitution."""
    T, Z, A = M.planted_singular_chain(4, 24, BATCH, seed=7)
    V, info = psd.eigvecs_batched(T, Z, "R")
    assert (info == 0).all()
    for b in (0, 3, BATCH - 1):
        _check(A[b], T[b], V[b], np.zeros(4, complex), "R")


@pytest.mark.parametrize("cplx,lr", [(True, "R"), (True, "L"), (False, "L")])
def test_global_memory_complex_and_left(psd, cplx, lr):
    """n = 256 (DMMA back-transformation): the complex four-product path and :L indexing."""
    n, p = 256, 2
    A = _rand(256 + int(cplx), n, p, 1, cplx)
    T, Z, lam = _schur(psd, A, lr)
    sel = np.zeros((1, n), dtype=bool)
    sel[0, [0, 1, 77, 128, 200, 255]] = True
    V, info = psd.eigvecs_batched(T, Z, lr, sel)
    assert info[0] == 0
    cols = M.effective_selection(T[0], lr, sel[0])
    _check(A[0], T[0], V[0], lam[0], lr, cols, eig_rel=1e-6)


@pytest.mark.parametrize("case", ["zero_column", "identity", "defective", "scaled", "graded"])
def test_edge_cases(psd, case):
    n, p = 10, 3
    A = _rand(555, n, p, BATCH, False)
    for b in range(BATCH):
        if case == "zero_column":
            A[b, 1, 4] = 0.0  # column 4 of A_2: a zero eigenvalue
        elif case == "identity":
            A[b] = np.eye(n)
        elif case == "defective":
            Q, _ = np.linalg.qr(A[b, 0])
            J = 2.0 * np.eye(n) + np.diag(np.ones(n - 1), 1)
            A[b, 0] = (Q @ J @ Q.T).T
            A[b, 1] = np.eye(n)
            A[b, 2] = np.eye(n)
        elif case == "scaled":
            A[b, 0] *= 1e160
            A[b, 2] *= 1e-160
        elif case == "graded":
            d = 10.0 ** (-8.0 * np.arange(n) / n)
            for j in range(p):
                A[b, j] *= d[None, :] if j % 2 == 0 else d[:, None]
    if case == "scaled":
        # the decomposition runs on the factors normalised by exact powers of two (as in
        # tests/eigacc.py); T_l times the same powers is a periodic Schur form of the scaled A_l
        e = np.frexp(np.abs(A).max(axis=(2, 3)))[1]
        T, Z, lam = _schur(psd, np.ldexp(A, -e[:, :, None, None]), "R")
        T = np.ldexp(T, e[:, :, None, None])
        lam = lam * np.exp2(e.sum(axis=1).astype(float))[:, None]
        V, info = psd.eigvecs_batched(T, Z, "R")
        assert (info == 0).all()
    else:
        T, Z, lam, V = _run(psd, A, "R")
    for b in (0, 3, BATCH - 1):
        _check(A[b], T[b], V[b], lam[b], "R")


def test_eigacc_golden(psd, oracle):
    """Eigenvalue consistency on the golden problems: prod mu_l against the ground truth, held to
    the per-eigenvalue gate of tests/eigacc.py; backward error as everywhere."""
    g = {rec["id"]: rec for rec in EA.load()["problems"]}
    for pid, rec in EA.PROBLEMS:
        A = EA.inputs(oracle, rec)
        lr = "L" if rec["left"] else "R"
        shift = 0
        if rec["scale"] or rec["peak"]:  # normalised factors, as the eigenvalue tests run them
            A, shift = EA.normalise(A)
        T, Z, lam = _schur(psd, A[None], lr)
        V, info = psd.eigvecs_batched(T, Z, lr)
        assert info[0] == 0, pid
        be, prods = M.backward_errors(A, V[0], lr)
        assert be.max() <= C_BE, (pid, be.max())
        ref, kappa = EA.truth(g[pid])
        lam_v = EA.unshift([prods[k] for k in range(rec["n"])], shift)
        EA.check(ref, kappa, lam_v, rec["n"], what=pid)


def test_malformed_problem_sets_info_alone(psd):
    n, p = 8, 3
    A = _rand(8, n, p, BATCH, False)
    T, Z, lam = _schur(psd, A, "R")
    T[3, 0, 1, 2] = 1.0   # T_1[2, 1]
    T[3, 0, 2, 3] = 1.0   # T_1[3, 2]: two adjacent nonzero subdiagonal entries
    V, info = psd.eigvecs_batched(T, Z, "R")
    assert info.tolist() == [0, 0, 0, 1, 0, 0, 0]
    assert not V[3].any()
    for b in (0, BATCH - 1):
        _check(A[b], T[b], V[b], lam[b], "R")


def test_eigvecs_struct(psd):
    n, p = 6, 2
    rng = np.random.default_rng(1)
    As = [rng.standard_normal((n, n)) for _ in range(p)]
    P = psd.pschur(As, "L")
    select = [True, False, False, False, False, True]
    Vs = psd.eigvecs(P, select=select)
    cols = M.effective_selection(np.stack([P.T[0].T, P.T1.T]), "L", select)  # T in storage layout
    m = len(cols)
    assert len(Vs) == p and all(V.shape == (n, m) for V in Vs)
    # the backward-error relation on the returned matrices against the input factors
    A = np.stack([a.T for a in As])
    V = np.stack([v.T for v in Vs])
    be, prods = M.backward_errors(A, V, "L", range(m))
    assert be.max() <= C_BE, be.max()
    lam = P.values[cols]
    for k in range(m):
        assert abs(prods[k] - lam[k]) <= 1e-8 * abs(lam[k])
