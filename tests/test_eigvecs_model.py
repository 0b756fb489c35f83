"""CPU checks of the eigenvector algorithm through its numpy model (tests/peigvec_model.py) on
oracle decompositions, against the gates of the GPU tests; and the argument checks of the two
eigenvector entry points, which need no device."""
import ctypes as C

import numpy as np
import pytest

import peigvec_model as M

EPS = np.finfo(np.float64).eps


def _cases(oracle):
    """(name, A, T, Z, lam, lr): real oracle decompositions of the shapes and edge cases the GPU
    tests use, and complex ones from the numpy QZ oracle."""
    from oracle import gpsd as OG
    out = []
    for n, p, lr in [(1, 1, "R"), (2, 2, "L"), (5, 3, "R"), (8, 3, "L"), (12, 1, "R"), (16, 8, "R"), (10, 3, "L")]:
        A = oracle.gen_real(900 + n + p, n, p, 1) - 0.5
        T, Z, lam, info, _ = oracle.rpschur_batched(A, left=(lr == "L"))
        assert info[0] == 0
        out.append((f"real-n{n}p{p}{lr}", A[0], T[0], Z[0], lam[0], lr))
    for n, p in [(2, 2), (5, 3), (2, 8), (32, 8)]:  # inputs of test_gpu_eigvecs.py::test_shapes
        for lr in ("R", "L"):
            for b in (0, 6):
                A = np.random.default_rng(1000 + 7 * n + p).standard_normal((7, p, n, n))[b:b + 1]
                T, Z, lam, info, _ = oracle.rpschur_batched(A, left=(lr == "L"))
                assert info[0] == 0
                out.append((f"real-shapes-n{n}p{p}{lr}b{b}", A[0], T[0], Z[0], lam[0], lr))
    rng = np.random.default_rng(3)
    for case in ("zero_column", "identity", "defective", "scaled", "graded"):
        n, p = 10, 3
        A = rng.standard_normal((1, p, n, n))
        if case == "zero_column":
            A[0, 1, 4] = 0.0
        elif case == "identity":
            A[0] = np.eye(n)
        elif case == "defective":
            Q, _ = np.linalg.qr(A[0, 0])
            A[0, 0] = (Q @ (2.0 * np.eye(n) + np.diag(np.ones(n - 1), 1)) @ Q.T).T
            A[0, 1] = A[0, 2] = np.eye(n)
        elif case == "scaled":
            A[0, 0] *= 1e160
            A[0, 2] *= 1e-160
        else:
            d = 10.0 ** (-8.0 * np.arange(n) / n)
            for j in range(p):
                A[0, j] *= d[None, :] if j % 2 == 0 else d[:, None]
        As = A
        shift = 0
        if case == "scaled":  # the oracle runs on the normalised factors (tests/eigacc.py)
            As = A.copy()
            for j in range(p):
                e = int(np.frexp(np.abs(As[0, j]).max())[1])
                As[0, j] = np.ldexp(As[0, j], -e)
                shift += e
        T, Z, lam, info, _ = oracle.rpschur_batched(As)
        assert info[0] == 0
        if case == "scaled":
            T = T.copy()
            for j in range(p):
                e = int(np.frexp(np.abs(A[0, j]).max())[1])
                T[0, j] = np.ldexp(T[0, j], e)
        out.append((case, A[0], T[0], Z[0], lam[0], "R"))
    T, Z, A = M.planted_blocks(9, 3, 1, seed=3)
    out.append(("planted-blocks", A[0], T[0], Z[0], M.schur_eigs(T[0], "R"), "R"))
    for n, p, lr in [(6, 3, "R"), (8, 3, "L"), (5, 1, "R")]:
        Ac = rng.standard_normal((1, p, n, n)) + 1j * rng.standard_normal((1, p, n, n))
        T, Z, al, be, sc, info = OG.cpschur_batched(Ac, [True] * p, left=(lr == "L"))
        assert info[0] == 0
        lam = al[0] / be[0] * np.exp2(sc[0].astype(float))
        out.append((f"complex-n{n}p{p}{lr}", Ac[0], T[0], Z[0], lam, lr))
    return out


def test_model_backward_error_and_contract(oracle):
    worst = 0.0
    for name, A, T, Z, lam, lr in _cases(oracle):
        V = M.eigvecs(T, Z, lr)
        M.check_contract(T, V, lam, lr)
        be, prods = M.backward_errors(A, V, lr)
        worst = max(worst, be.max())
        assert be.max() <= M.MODEL_WORST_BE, (name, be.max())
        if name.startswith(("real", "complex", "planted")):
            for k, pr in prods.items():
                assert abs(pr - lam[k]) <= 1e-8 * abs(lam[k]), (name, k, pr, lam[k])
    print("model worst backward error ratio", worst)


@pytest.mark.parametrize("n,p,cplx", [(24, 2, False), (40, 3, False), (24, 3, True)])
def test_model_exactly_defective(n, p, cplx):
    """Every eigenvalue exactly repeated: eps pivots with nonzero right-hand sides, rescales inside
    the back-substitution and chain shifts all run, and the backward error and contract hold."""
    for k in M.COUNTS:
        M.COUNTS[k] = 0
    T, Z, A = M.planted_defective(n, p, 1, seed=n + p)
    lam = np.full(n, 2.0 + 0j)
    V = M.eigvecs(T[0], Z[0], "R")
    M.check_contract(T[0], V, lam, "R")
    be, _ = M.backward_errors(A[0], V, "R")
    assert be.max() <= M.MODEL_WORST_BE, be.max()
    assert M.COUNTS["pivot"] > 0 and M.COUNTS["chain_shift"] > 0, M.COUNTS


def test_model_singular_chain():
    """p eps pivots in one cyclic system: the rescale inside the back-substitution runs."""
    for k in M.COUNTS:
        M.COUNTS[k] = 0
    T, Z, A = M.planted_singular_chain(4, 24, 1, seed=7)
    V = M.eigvecs(T[0], Z[0], "R")
    M.check_contract(T[0], V, np.zeros(4, complex), "R")
    be, _ = M.backward_errors(A[0], V, "R")
    assert be.max() <= M.MODEL_WORST_BE, be.max()
    assert M.COUNTS["solve_rescale"] > 0 and M.COUNTS["pivot"] > 0, M.COUNTS


def test_model_ground_truth(oracle):
    mp = pytest.importorskip("mpmath")
    for lr in ("R", "L"):
        A = oracle.gen_real(4242, 8, 3, 1) - 0.5
        T, Z, lam, info, _ = oracle.rpschur_batched(A, left=(lr == "L"))
        V = M.eigvecs(T[0], Z[0], lr)
        assert M.angle_to_mpmath(A[0], V, lam[0], lr, mp) <= 1e-10


def test_model_selection(oracle):
    A = oracle.gen_real(17, 12, 3, 1) - 0.5
    T, Z, lam, info, _ = oracle.rpschur_batched(A)
    sel = np.zeros(12, dtype=bool)
    pairs = np.flatnonzero(lam[0].imag > 0)
    sel[[0, 5]] = True
    if pairs.size:
        sel[pairs[0] + 1] = True  # the second member selects the whole pair
    V = M.eigvecs(T[0], Z[0], "R", sel)
    cols = M.effective_selection(T[0], "R", sel)
    if pairs.size:
        assert pairs[0] in cols and pairs[0] + 1 in cols
    M.check_contract(T[0], V, lam[0], "R", cols)


@pytest.mark.parametrize("name", ["psd_reigvecs_batched", "psd_ceigvecs_batched"])
def test_bad_arguments_need_no_device(psd, name):
    f = getattr(psd.lib(), name)
    buf = np.zeros(64)
    info = np.zeros(4, dtype=np.int32)
    vp = C.c_void_p
    d, i = vp(buf.ctypes.data), vp(info.ctypes.data)
    cases = [((None, 0, 1, 1, 0, d, d, None, d, i), "n, p"),
             ((None, 2, 0, 1, 0, d, d, None, d, i), "n, p"),
             ((None, 2, 1, -1, 0, d, d, None, d, i), "batch"),
             ((None, 2, 1, 1, 2, d, d, None, d, i), "orientation"),
             ((None, 2, 1, 1, 0, None, d, None, d, i), "NULL"),
             ((None, 2, 1, 1, 0, d, d, None, None, i), "NULL"),
             ((None, 2, 1, 1, 0, d, d, None, d, None), "NULL"),
             ((None, 2, 1, 1, 0, d, d, None, d, i), "handle")]
    for args, what in cases:
        assert f(*args) == -1  # PSD_ERR_BAD_ARG
        assert what in psd.lib().psd_last_error_string().decode()
