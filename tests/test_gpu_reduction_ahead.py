"""Bit-for-bit checks of the small-N periodic Hessenberg-triangular reduction
(rphess_ahead32_kernel_t: the reflector chain on one warp, the trailing updates on others, up to
p-2 steps behind).  Reordering independent work must not change a single bit, so the
eigenvalue-only fast path is compared exactly against golden results of the build before that
kernel (tests/golden/make_golden_reduction.py): eigenvalues, info and iteration counts.  The
chain-ahead kernel runs for p >= 7 where it keeps as many problems resident per SM as the two-warp
kernel (here N = 31, 32 at p = 8); the other cases pin the two-warp kernel and, for p = 2, the path
that serves p = 2 (the eigenvalue-only fast path starts at p = 3).  The `zeros` and `rescale`
cases take the H = I and power-of-two rescale branches of the reflector."""
import numpy as np
import pytest

import reduction_cases as RC

pytestmark = pytest.mark.gpu

_EO, _BO = RC.offsets()


def _golden(i):
    kind, n, p = RC.CASES[i]
    eig = np.load(RC.golden_path("eig"))[_EO[i]:_EO[i] + RC.BATCH * n].reshape(RC.BATCH, n)
    info = np.load(RC.golden_path("info"))[_BO[i]:_BO[i] + RC.BATCH]
    iters = np.load(RC.golden_path("iters"))[_BO[i]:_BO[i] + RC.BATCH]
    return eig, info, iters


def _run(psd, A):
    _, _, lam, info, iters = psd.pschur_batched(A, "R", wantZ=False, wantT=False, return_iters=True)
    return lam, info, iters


@pytest.mark.parametrize("i", range(len(RC.CASES)), ids=[RC.case_id(c) for c in RC.CASES])
def test_reduction_bitwise_golden(psd, oracle, i):
    A = RC.inputs(oracle, RC.CASES[i])
    lam, info, iters = _run(psd, A)
    eig0, info0, iters0 = _golden(i)
    assert np.array_equal(info, info0)
    assert np.array_equal(iters, iters0)
    assert np.array_equal(lam, eig0, equal_nan=True), np.argwhere(~((lam == eig0) | (np.isnan(lam) & np.isnan(eig0))))


def test_golden_cases_take_the_rare_branches(oracle):
    """The zeros / rescale inputs really contain zero tails and tiny tails after normalisation."""
    A = RC.inputs(oracle, ("zeros", 17, 3))
    assert (A[-1, 1][np.tril_indices(17, -1)[::-1]] == 0.0).all()
    A = RC.inputs(oracle, ("rescale", 17, 3))
    col = A[1, 0][0]
    assert np.abs(col[9:]).max() < 1e-140 * np.abs(A[1, 0]).max()


@pytest.mark.parametrize("n,p", [(32, 8), (17, 3), (31, 4)])
def test_reduction_repeatable(psd, oracle, n, p):
    """A race between the chain warp and the update warps would show up as a difference between
    two runs of the same batch (large enough to fill every SM several times)."""
    A = oracle.gen_real(77, n, p, 3001)
    r1 = _run(psd, A)
    r2 = _run(psd, A)
    for x, y in zip(r1, r2):
        assert np.array_equal(x, y, equal_nan=True)
