#!/usr/bin/env python
"""Per-kernel time of the headline workload, split by occupancy phase.

The handle's timer reports the occupancy phases of the eigenvalue-only iteration
(`rpqr_eig32_kernel_t<32,8>` for order 32, then the register-capped kernel for orders 28..12) as
one "iterate" figure.  This script runs the `bench.py` workload (real p = 8, N = 32, 100 000
problems, eigenvalues only, device-resident) under torch.profiler with CUDA activities and prints
the summed duration per step of the reduction kernel and of each phase, with the GPU name and
power limit read in the same run.  A problem batch is launched in chunks; within a chunk the
phases run in order after the reduction, which is how launches of the same kernel are told apart.

  python scripts/eig32_phase_times.py [--steps 3] [--warmup 2] [--batch 100000]

Tracing slows the host, so take end-to-end numbers from bench.py, not from this script.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

N, P, SEED = 32, 8, 1234
PHASE_ORDERS = [32, 28, 24, 20, 16, 12]  # launch_real_eig32: n - k * (n / 8), k = 0..5


def gpu_info(index: int) -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader", "-i", str(index)],
                             capture_output=True, text=True, check=True).stdout.strip()
        name, plim, smax = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": plim, "sm_max_clock": smax}
    except Exception as e:  # report, do not guess
        return {"name": None, "error": str(e)}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--batch", type=int, default=100_000)
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile
    import psd_b200

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    L = psd_b200.lib()
    h = psd_b200.Handle([0])
    B = args.batch
    dA = torch.empty((B, P, N, N), dtype=torch.float64, device=dev)
    dE = torch.empty((B, N, 2), dtype=torch.float64, device=dev)
    dI = torch.empty(B, dtype=torch.int32, device=dev)
    ts = torch.cuda.Stream(device=dev)
    psd_b200.capi.check(L.psd_fill_uniform_dev(C.c_void_p(ts.cuda_stream), SEED, N, P, B, 0, 0,
                                               C.c_void_p(dA.data_ptr())))

    def step():
        psd_b200.capi.check(L.psd_rpschur_batched_dev(
            h.ptr, 0, C.c_void_p(ts.cuda_stream), N, P, B, 0, 0, 0, 30,
            C.c_void_p(dA.data_ptr()), None, C.c_void_p(dE.data_ptr()), C.c_void_p(dI.data_ptr())))

    with torch.cuda.stream(ts):
        for _ in range(args.warmup):
            step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        with torch.cuda.stream(ts):
            for _ in range(args.steps):
                step()
        torch.cuda.synchronize()
    info = gpu_info(0)
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    kern = sorted((e for e in events if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    reduce_us = 0.0
    n_reduce = 0
    phase_us = [0.0] * len(PHASE_ORDERS)
    phase_n = [0] * len(PHASE_ORDERS)
    phase_name = [None] * len(PHASE_ORDERS)
    k = None
    for e in kern:
        name = e["name"]
        if "rphess_" in name:
            reduce_us += e["dur"]
            n_reduce += 1
            k = 0
        elif "rpqr_eig32" in name:
            if k is None or k >= len(PHASE_ORDERS):
                raise SystemExit(f"unexpected launch order at {name}")
            phase_us[k] += e["dur"]
            phase_n[k] += 1
            phase_name[k] = name
            k += 1
    fails = int((dI != 0).sum().item())
    s = args.steps
    res = {
        "gpu": info,
        "steps": s,
        "batch": B,
        "fails": fails,
        "reduce_ms_per_step": round(reduce_us / s / 1e3, 3),
        "reduce_launches_per_step": n_reduce / s,
        "phases": [{"order": o, "kernel": phase_name[i], "launches_per_step": phase_n[i] / s,
                    "ms_per_step": round(phase_us[i] / s / 1e3, 3)} for i, o in enumerate(PHASE_ORDERS)],
        "iterate_ms_per_step": round(sum(phase_us) / s / 1e3, 3),
    }
    print(json.dumps(res))


if __name__ == "__main__":
    main()
