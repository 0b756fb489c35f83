#!/usr/bin/env python
"""SHA-256 digests of everything the generalized paths return, (alpha, beta, alphascale, info, T, Z)
and the eigenvalue-only triple, on the inputs of the generalized GPU tests (test_gpu_complex.py,
test_gpu_rgeneralized.py) and at the C3 / C5 benchmark shapes.  Two libraries give the same digests
exactly when their results agree bit for bit.

  python scripts/gen_outputs_digest.py OUT.json
"""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import gpsd_cases as GC  # noqa: E402
import psd_b200  # noqa: E402


def cases():
    for c in (True, False):
        for p, S, left in [(5, [1] * 5, False), (5, [1] * 5, True), (4, [1, 0, 1, 0], False), (4, [0, 1, 0, 1], True),
                           (1, [1], False), (2, [1, 0], False), (6, [1, 0, 1, 1, 0, 1], False), (3, [0, 1, 1], True)]:
            yield f"n5p{p}", GC.rand_storage(1234, 5, p, 6, c), S, left, False
        for p in (2, 3, 5):
            yield f"hessut-n5p{p}", GC.hessut_storage(79, 5, p, 4, c), [1, 0] + [1] * (p - 2), False, True
        for S, hole in GC.HOLE_CASES:
            yield f"hole{hole}", GC.hessut_storage(80 + hole[0] * 10 + hole[1], 5, 5, 4, c, hole=hole), S, False, True
        yield "hole-n32p4", GC.hessut_storage(99, 32, 4, 2, c, hole=(2, 3)), [1, 0, 1, 0], False, True
        for n, p in [(1, 3), (2, 2), (3, 4), (16, 3), (33, 2), (40, 2), (24, 6)]:
            S = [1] + [(k % 2) for k in range(1, p)]
            yield f"n{n}p{p}", GC.rand_storage(7, n, p, 3, c), S, False, False
            yield f"n{n}p{p}L", GC.rand_storage(7, n, p, 3, c), S[::-1] if S[-1] else [1] * p, True, False
        for p, S, left in [(1, [1], False), (2, [1, 0], False), (2, [0, 1], True), (3, [1, 1, 1], True)]:
            yield f"windowed-p{p}", GC.rand_storage(4242 + p, 150 if c else 200, p, 2, c), S, left, False
    yield "C3-n128", GC.rand_storage(1234, 128, 6, 2, True), [1, 0, 1, 1, 0, 1], False, False
    yield "C5-n64", GC.rand_storage(1234, 64, 10, 2, False), [k % 2 for k in range(10)], True, False
    yield "C5-n512", GC.rand_storage(1234, 512, 10, 1, False), [k % 2 for k in range(10)], True, False


def digest(arrays):
    h = hashlib.sha256()
    for a in arrays:
        if a is not None:
            h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def main():
    out = {}
    for name, A, S, left, hessut in cases():
        key = f"{'c' if A.dtype == np.complex128 else 'r'}-{name}-{'L' if left else 'R'}{'-'.join(map(str, S))}"
        for wT, wZ in ((True, True), (False, False)):
            r = psd_b200.gpschur_batched(A, S, "L" if left else "R", wantZ=wZ, wantT=wT, hessut=hessut)
            out[f"{key}-{'TZ' if wT else 'eig'}"] = digest(r[:2] if wT else ()) + " " + digest(r[2:])
    with open(sys.argv[1], "w") as f:
        json.dump(out, f, indent=1)
    print(len(out), "digests")


if __name__ == "__main__":
    main()
