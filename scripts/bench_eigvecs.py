"""Eigenvectors of periodic Schur results on the device (psd_reigvecs_batched): one JSON line per
workload with the device name and power limit read in the same run.

  kernel_ms   device time of the eigenvector kernels of one call (CUDA events around every launch
              sequence, psd_set_profiling; N >= 192 includes the DMMA GEMMs of the
              back-transformation and the normalisation kernel), averaged over the timed calls
  call_ms     end to end through the host call (copies of T, Z in and V out), warmed up
  pschur_ms   psd_rpschur_batched with T and Z on the same batch, for scale

Workloads: the headline shape (p = 8, N = 32, 10 000 problems) and config C1 (p = 3, N = 50,
4096 problems) with every eigenvector, and one N = 1024, p = 4 problem with 16 vectors selected
and then with all of them.

Usage: python scripts/bench_eigvecs.py [--reps R] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import psd_b200 as psd  # noqa: E402


def device_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True)
    name, power = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
    return name, power


def run(h, name, n, p, batch, nsel, reps, dev):
    rng = np.random.default_rng(n * 100 + p)
    A = rng.standard_normal((batch, p, n, n))
    psd.pschur_batched(A[: min(batch, 4)], "R", handle=h)  # warm-up of the decomposition kernels
    t0 = time.perf_counter()
    T, Z, lam, info = psd.pschur_batched(A, "R", handle=h)
    pschur_ms = (time.perf_counter() - t0) * 1e3
    assert (info == 0).all()
    sel = None
    if nsel is not None:
        sel = np.zeros((batch, n), dtype=bool)
        sel[:, np.linspace(0, n - 1, nsel - 1).astype(int)] = True
        sel[:, int(np.flatnonzero(lam[0].imag > 0)[0])] = True  # and one complex pair
    V, vinfo = psd.eigvecs_batched(T, Z, "R", sel, handle=h)  # warm-up
    assert (vinfo == 0).all()
    h.set_profiling(True)
    h.kernel_times()
    call = []
    for _ in range(reps):
        t0 = time.perf_counter()
        psd.eigvecs_batched(T, Z, "R", sel, handle=h)
        call.append((time.perf_counter() - t0) * 1e3)
    kt = h.kernel_times()
    h.set_profiling(False)
    vectors = int(np.count_nonzero(np.any(V[:, 0] != 0, axis=2)))
    return {"workload": name, "n": n, "p": p, "batch": batch, "vectors": vectors,
            "kernel_ms": kt["iterate_ms"] / reps, "call_ms": float(np.median(call)),
            "call_ms_min": float(np.min(call)), "pschur_ms": pschur_ms, "reps": reps,
            "device": dev[0], "power_limit": dev[1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = device_info()
    h = psd.Handle([0])
    lines = []
    for name, n, p, batch, nsel in [("p8_n32_all", 32, 8, 10000, None), ("c1_p3_n50_all", 50, 3, 4096, None),
                                    ("p4_n1024_sel16", 1024, 4, 1, 16), ("p4_n1024_all", 1024, 4, 1, None)]:
        line = json.dumps(run(h, name, n, p, batch, nsel, a.reps, dev))
        print(line, flush=True)
        lines.append(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
