"""Inputs of the bit-for-bit checks of the small-N periodic Hessenberg-triangular reduction
(tests/test_gpu_reduction_ahead.py, golden results from tests/golden/make_golden_reduction.py).

The eigenvalue-only fast path (N <= 32) reduces every problem and then runs the QR iteration on
the packed factors.  The same packed factors give the same iterations, so equal eigenvalues,
`info` and iteration counts pin the reduction bit for bit.  Each case is one seeded batch:
  plain   - oracle.gen_real inputs;
  zeros   - some factors already triangular (factor 1: Hessenberg), so many reflector steps see an
            exactly zero tail (H = I);
  rescale - whole factors scaled by 1e+160 or 1e-160 and the lower half of the rows by another
            1e-160, so tails of the later columns are tiny next to the factor's largest entry and
            take the power-of-two rescale of the reflector.
BATCH is prime: no launch shape divides it, so the last CTA of every launch is partly empty."""
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SEED = 4242
BATCH = 13

CASES = ([("plain", n, p) for p in (2, 3, 4, 8) for n in (3, 4, 5, 17, 31, 32)] +
         [("zeros", n, p) for p in (2, 3, 8) for n in (5, 17, 32)] +
         [("rescale", n, p) for p in (2, 3, 8) for n in (5, 17, 32)])


def case_id(c):
    return f"{c[0]}-n{c[1]}-p{c[2]}"


def inputs(oracle, case):
    """A [BATCH][p][col][row] of one case (deterministic)."""
    kind, n, p = case
    seed = SEED + 1000 * ("plain", "zeros", "rescale").index(kind) + 37 * n + p
    A = oracle.gen_real(seed, n, p, BATCH)
    rows = np.arange(n)
    if kind == "zeros":
        below = rows[None, :] > rows[:, None]           # [col][row]: strictly below the diagonal
        below_h = rows[None, :] > rows[:, None] + 1     # below the subdiagonal
        for b in range(BATCH):
            for j in range(p):
                if (b + j) % 3 == 0 or b == BATCH - 1:  # the last problem is fully reduced already
                    A[b, j][below_h if j == 0 else below] = 0.0
            c = b % n
            A[b, b % p, c, c + 1:] = 0.0  # and one column with a zero tail in every problem
    elif kind == "rescale":
        for b in range(BATCH):
            for j in range(p):
                A[b, j] *= 1e160 if (b + j) % 2 else 1e-160
                if (b + 2 * j) % 3:
                    A[b, j][:, n // 2:] *= 1e-160
    return A


def golden_path(name):
    return os.path.join(GOLDEN, f"reduction_{name}.npy")


def offsets():
    """Start of each case's rows in the concatenated golden arrays (eigenvalues: BATCH * n rows)."""
    eo, bo, e, b = [], [], 0, 0
    for _, n, _ in CASES:
        eo.append(e)
        bo.append(b)
        e += BATCH * n
        b += BATCH
    return eo, bo
