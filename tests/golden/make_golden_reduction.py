"""Generates tests/golden/reduction_{eig,info,iters}.npy: eigenvalues (complex128), info and QR
iteration counts (int32) of the eigenvalue-only fast path for the cases of
tests/reduction_cases.py, concatenated in case order.  These are results of a build, not ground
truth: they pin the small-N reduction bit for bit across changes that must not alter it (the
last such change reordered independent work only).  Regenerate only when the arithmetic of the
path changes on purpose.
Run (on a GPU, with the build to be pinned):  python tests/golden/make_golden_reduction.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]
import psd_b200  # noqa: E402
import reduction_cases as RC  # noqa: E402
from oracle import oracle as O  # noqa: E402


def main():
    O.build()
    h = psd_b200.Handle([0])
    eig, info, iters = [], [], []
    for case in RC.CASES:
        A = RC.inputs(O, case)
        _, _, lam, inf, it = psd_b200.pschur_batched(A, "R", wantZ=False, wantT=False, handle=h,
                                                     return_iters=True)
        eig.append(lam.reshape(-1))
        info.append(inf)
        iters.append(it)
    np.save(RC.golden_path("eig"), np.concatenate(eig))
    np.save(RC.golden_path("info"), np.concatenate(info).astype(np.int32))
    np.save(RC.golden_path("iters"), np.concatenate(iters).astype(np.int32))
    print(f"{len(RC.CASES)} cases x {RC.BATCH} problems written to {RC.GOLDEN}")


if __name__ == "__main__":
    main()
