#!/usr/bin/env python
"""bench.py — headline benchmark of the dense pschur! hot path on B200.

Workload (BASELINE.json configs[1]): batched real Float64 pschur!, p=8, N=32, 100 000
independent problems per GPU, eigenvalues only (wantT=wantZ=false), uniform [0,1) synthetic
inputs from the counter-based generator (seed 1234).  One "step" = one pass of the hot path
over the whole batch.

  python bench.py --gpus N --steps K --warmup W            (ours; torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  (CPU restatement of the reference)
  python bench.py ... --dump-outputs DIR                   (also write the last step's results)

Prints ONE JSON line on rank 0.  `value` is device-resident throughput (inputs already in
HBM), `e2e` goes through the reference-facing C-ABI call with pinned HOST buffers (H2D and
D2H inside the timed region).  Weak scaling: every rank owns its own 100k-problem shard, no
data-path collective (SURVEY.md §8(e)).

--dump-outputs DIR writes what the device-resident path returned in its last timed step, so
that two builds run with the same arguments (hence the same inputs) can be compared output
for output: eigenvalues.npy [problems][N][2] (real, imaginary parts), info.npy [problems] and
problem_index.npy [problems] (index of each problem in the batch), all float64.  Above 64 MiB
in all, a fixed seeded sample of the problems is written.  With N > 1 GPUs, rank 0's shard.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: no __pycache__ next to the sources

N_ORDER = 32
PERIOD = 8
SEED = 1234
# SURVEY.md §8(d): compulsory bytes per problem = read 8*32*32*8 + write 32*16
BYTES_PER_PROBLEM = PERIOD * N_ORDER * N_ORDER * 8 + N_ORDER * 16
FLOPS_PER_PROBLEM = 10 * PERIOD * N_ORDER ** 3


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def bench_config(batch_per_gpu: int, world: int) -> dict:
    """The workload description, identical for both arms (the CPU arm times a bounded sample of it,
    stated in its cpu_baseline.sample)."""
    return {"workload": "real pschur! p=8 N=32 eigenvalues only (BASELINE configs[1])",
            "batch_per_gpu": batch_per_gpu, "inputs": "uniform[0,1) seed 1234",
            "l2": "input 6.55 GB per GPU >> 126 MB L2 (no flush needed)",
            "parallelism": f"batch shards x{world}, no collective"}


def host_cores() -> int:
    """Host threads this process may use (torchrun exports OMP_NUM_THREADS=1, so the OpenMP
    default cannot be trusted: the thread count is always passed explicitly)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def cpu_reference_rate(sample: int, nthreads: int = 0):
    """Time the CPU restatement of the reference (oracle, OpenMP over the batch) on `sample`
    problems of the same workload.  Returns (problems/s, cores, seconds)."""
    from oracle import oracle as O
    nthreads = nthreads or host_cores()
    A = O.gen_real(SEED, N_ORDER, PERIOD, sample)
    t0 = time.perf_counter()
    _, _, _, info, _ = O.rpschur_batched(A, left=False, wantT=False, wantZ=False, nthreads=nthreads)
    dt = time.perf_counter() - t0
    assert (info == 0).all()
    return sample / dt, nthreads, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = host_cores()
    # bounded sample per step: ~2-4 s of CPU work
    probe_rate, _, _ = cpu_reference_rate(max(64, 32 * cores))
    sample = int(max(256, min(args.batch, probe_rate * 3.0)))
    for _ in range(args.warmup):
        cpu_reference_rate(sample)
    t = 0.0
    for _ in range(args.steps):
        _, _, dt = cpu_reference_rate(sample)
        t += dt
    rate = sample * args.steps / t
    line = {
        "impl": "reference", "metric": "pschur!/sec batched (p=8,N=32); large-N FP64 % peak in large_n", "value": rate,
        "unit": "problems/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": bench_config(args.batch, args.gpus),
        "cpu_baseline": {"value": rate, "unit": "problems/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} problems per step, C++ restatement of the reference "
                                   f"(Julia unavailable), OpenMP over the batch"},
        "e2e": {"value": rate, "unit": "problems/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


LARGE_N, LARGE_P = 4096, 4   # BASELINE configs[3]


def cublas_dgemm_tflops(torch, dev, m=8192, reps=5):
    """FP64 tensor-core denominator (SURVEY.md section 8(d)): cuBLAS DGEMM m^3, best of `reps`,
    measured in this very run."""
    x = torch.randn(m, m, dtype=torch.float64, device=dev)
    y = torch.randn(m, m, dtype=torch.float64, device=dev)
    torch.matmul(x, y)
    best = 1e30
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(x, y); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del x, y
    torch.cuda.empty_cache()
    return 2.0 * m ** 3 / (best * 1e-3) / 1e12


def large_n_block(torch, psd_b200, L, h, dev, n=LARGE_N, p=LARGE_P):
    """Second half of BASELINE's metric ("large-N FP64 % peak"): one full real pschur! with T and
    Z at p = 4, N = 4096 on device-resident buffers through psd_rpschur_batched_dev; standard flop
    count against the cuBLAS DGEMM rate of the same run; the FP64 tensor-core (DMMA) window
    updates of the iteration and the GEMM updates of the reduction against it separately;
    residual and orthogonality checked on the device."""
    peak = cublas_dgemm_tflops(torch, dev)
    nn = n * n
    A0 = torch.empty((1, p, n, n), dtype=torch.float64, device=dev)
    st = torch.cuda.Stream(device=dev)  # a real stream handle (NULL would select the library's own)
    psd_b200.capi.check(L.psd_fill_uniform_dev(C.c_void_p(st.cuda_stream), SEED, n, p, 1, 0, 0, C.c_void_p(A0.data_ptr())))
    T = torch.empty_like(A0)
    Z = torch.empty_like(A0)
    E = torch.empty((1, n, 2), dtype=torch.float64, device=dev)
    I = torch.empty(1, dtype=torch.int32, device=dev)

    torch.cuda.synchronize()

    def run():
        T.copy_(A0)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        psd_b200.capi.check(L.psd_rpschur_batched_dev(h.ptr, 0, C.c_void_p(st.cuda_stream), n, p, 1, 0, 1, 1, 30,
                                                      C.c_void_p(T.data_ptr()), C.c_void_p(Z.data_ptr()),
                                                      C.c_void_p(E.data_ptr()), C.c_void_p(I.data_ptr())))
        e1.record(st)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e-3

    h.set_profiling(False)
    run()                     # warm-up (workspaces, module load)
    secs = min(run(), run())  # timed without per-launch events
    h.set_profiling(True); h.kernel_times()
    run()                     # one more pass with CUDA events around every launch, for the split
    kt = h.kernel_times()
    ls = h.large_stats()
    h.set_profiling(False)
    # residual / orthogonality on the device (storage is column-major: tensor [c][r] = M^T)
    eps = 2.220446049250313e-16
    res = orth = 0.0
    for j in range(p):
        Aj, Tj, Zj, Zn = A0[0, j].T, T[0, j].T, Z[0, j].T, Z[0, (j + 1) % p].T
        res = max(res, float(torch.linalg.norm(Aj - Zj @ Tj @ Zn.T) / torch.linalg.norm(Aj)))
        orth = max(orth, float(torch.linalg.norm(Zj @ Zj.T - torch.eye(n, dtype=torch.float64, device=dev))))
    low = max(float(torch.tril(T[0, j].T, -2 if j == 0 else -1).abs().max()) for j in range(p))
    flops = 25.0 * p * n ** 3
    upd_tf = ls["apply_flops"] / max(1e-9, ls["apply_ms"] * 1e-3) / 1e12
    red_tf = kt["large_gemm_flops"] / max(1e-9, kt["large_gemm_ms"] * 1e-3) / 1e12
    return {
        "workload": f"real pschur! p={p} N={n} :R with T and Z, single problem (BASELINE configs[3])",
        "seconds": secs, "info": int(I.item()),
        "standard_flops": flops, "tflops_standard_count": flops / secs / 1e12,
        "dgemm_cublas_tflops_same_run": peak, "frac_of_dgemm": flops / secs / 1e12 / peak,
        "reduction_ms": kt["large_panel_ms"] + kt["large_gemm_ms"], "iteration_ms": kt["iterate_ms"],
        "iteration": {k: ls[k] for k in ("status", "sweeps", "rounds", "windows", "shift_pairs", "final_blocks",
                                         "chase_ms", "apply_ms", "scan_ms", "final_ms")},
        "dmma_window_updates": {"flops": ls["apply_flops"], "ms": ls["apply_ms"], "tflops": upd_tf,
                                "frac_of_dgemm": upd_tf / peak, "kernel": "psd::ms::ms_apply_kernel",
                                "note": "sum of the launch durations inside the pipeline, where the far updates share "
                                        "the GPU with the chase of the next round (two streams); 'isolated' = the same "
                                        "kernel alone on one synthetic N=4096 round (scripts/ubench/apply_bench)",
                                "isolated": isolated_update_rate(peak)},
        "dmma_reduction_updates": {"flops": kt["large_gemm_flops"], "ms": kt["large_gemm_ms"], "tflops": red_tf,
                                   "frac_of_dgemm": red_tf / peak, "kernel": "psd::dgemm_dmma_kernel"},
        "residual_over_n_eps": res / (n * eps), "orthogonality_over_n_eps": orth / (n * eps),
        "largest_entry_below_structure": low,
        "gates": "BASELINE: residual <= 10 N eps, ||Z'Z - I|| <= 10 N eps, exact quasi-triangular structure",
    }


def isolated_update_rate(peak):
    """Window-update kernel alone: one synthetic round of the N = 4096, p = 4 pipeline (13 windows of
    order 56), CUDA events, 20 repetitions (scripts/ubench/apply_bench.cu, built by build())."""
    exe = os.path.join(os.path.dirname(os.path.abspath(__file__)), "scripts", "ubench", "apply_bench")
    if not os.path.exists(exe):
        return None
    try:
        out = subprocess.run([exe, "4096", "13"], capture_output=True, text=True, timeout=120).stdout
        best = None
        for ln in out.splitlines():
            if ln.startswith("unsplit,"):
                f = ln.split()
                us, tf = float(f[f.index("us") - 1]), float(f[f.index("TFLOP/s") - 1])
                if best is None or tf > best[1]:
                    best = (us, tf, " ".join(f[:6]))
        if best is None:
            return None
        return {"us_per_round": best[0], "tflops": best[1], "frac_of_dgemm": best[1] / peak, "variant": best[2],
                "split_matches_unsplit_bitwise": "max |diff| 0.000e+00" in out}
    except Exception as ex:  # measurement tool only
        return {"error": repr(ex)}


def cpu_large_baseline(n_small=384, p=LARGE_P):
    """CPU restatement of the reference on the same kind of problem at a small order, with the
    N^3-extrapolated figure for N = 4096 (the reference's unblocked BLAS-1/2 algorithm needs hours
    there; a single problem does not thread).  SURVEY.md section 8(d)."""
    from oracle import oracle as O
    A = O.gen_real(SEED, n_small, p, 1)
    t0 = time.perf_counter()
    _, _, _, info, _ = O.rpschur_batched(A, nthreads=1)
    dt = time.perf_counter() - t0
    return {"seconds_measured": dt, "n_measured": n_small, "cores": 1, "kind": "port",
            "seconds_extrapolated_n4096": dt * (LARGE_N / n_small) ** 3,
            "sample": f"one p={p} N={n_small} problem with T and Z on one core (C++ restatement of the reference, "
                      f"Julia unavailable); N=4096 figure = measured x (4096/{n_small})^3, an extrapolation"}


def config1_block(psd_b200, h, reps=20):
    """BASELINE configs[0]: one real p=3 N=50 problem with Schur vectors - latency through the host
    call, with the CPU restatement of the reference (one core) timed beside it."""
    import numpy as np
    from oracle import oracle as O
    A = O.gen_real(SEED, 50, 3, 1)
    psd_b200.pschur_batched(A, "R", handle=h)
    t0 = time.perf_counter()
    for _ in range(reps):
        T, Z, lam, info = psd_b200.pschur_batched(A, "R", handle=h)
    gpu_ms = (time.perf_counter() - t0) / reps * 1e3
    t0 = time.perf_counter()
    for _ in range(reps):
        To, Zo, lo, io, _ = O.rpschur_batched(A, nthreads=1)
    cpu_ms = (time.perf_counter() - t0) / reps * 1e3
    # a small batch of the same shape (what the GPU is for)
    Ab = O.gen_real(SEED, 50, 3, 4096)
    psd_b200.pschur_batched(Ab, "R", handle=h)  # (first call of a shape allocates the pinned staging buffers)
    h.set_profiling(True); h.kernel_times()
    t0 = time.perf_counter()
    psd_b200.pschur_batched(Ab, "R", handle=h)
    gpu_batch = 4096 / (time.perf_counter() - t0)
    kt = h.kernel_times()
    h.set_profiling(False)
    gpu_batch_kernels = 4096 / max(1e-9, (kt["iterate_ms"] + kt["reduce_ms"]) * 1e-3)
    nb = 64 * host_cores()
    t0 = time.perf_counter()
    O.rpschur_batched(Ab[:nb], nthreads=host_cores())
    cpu_batch = nb / (time.perf_counter() - t0)
    return {"workload": "real pschur! p=3 N=50 :R with T and Z (BASELINE configs[0])",
            "single_problem_ms": gpu_ms, "info": int(info[0]),
            "cpu_single_problem_ms": cpu_ms, "cpu_cores_single": 1,
            "batch_4096_problems_per_s": gpu_batch, "batch_4096_problems_per_s_kernels_only": gpu_batch_kernels,
            "cpu_batch_problems_per_s": cpu_batch,
            "cpu_cores_batch": host_cores(),
            "note": "host call with pageable numpy buffers, copies included (second call of the shape: staging buffers exist); kernels_only sums the durations of chunk launches that overlap on three streams; CPU = C++ restatement of the reference"}


def pinned_input(L, psd_b200, torch, local_rank, shape):
    """Input buffer of the end-to-end leg.  With PSD_BENCH_WC_INPUT=1: page-locked, write-combined
    (the host only writes it, the GPU reads it over PCIe every step), allocated while the process is
    bound to the CPUs next to its GPU so that the pages land on that NUMA node (first touch)."""
    import numpy as np
    if not os.environ.get("PSD_BENCH_WC_INPUT"):
        # default: torch's pinned allocator.  The write-combined / affinity variant below was
        # measured at 8 GPUs: 1.648 M instead of 1.630 M problems/s end to end (noise); the GPU boxes
        # are VMs with one NUMA node, and 8 x 13.4 GB/s = 107 GB/s is what their host side delivers.
        return torch.empty(shape, dtype=torch.float64, pin_memory=True)
    old = None
    try:
        import pynvml
        pynvml.nvmlInit()
        hnd = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        words = pynvml.nvmlDeviceGetCpuAffinity(hnd, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            old = os.sched_getaffinity(0)
            os.sched_setaffinity(0, cpus)
    except Exception:
        old = None
    try:
        count = int(np.prod(shape))
        ptr = C.c_void_p()
        psd_b200.capi.check(L.psd_host_alloc(count * 8, 1, C.byref(ptr)))
        arr = np.ctypeslib.as_array((C.c_double * count).from_address(ptr.value)).reshape(shape)
        t = torch.from_numpy(arr)  # (lives until the process exits)
    except Exception:
        t = torch.empty(shape, dtype=torch.float64, pin_memory=True)
    finally:
        if old:
            os.sched_setaffinity(0, old)
    return t


def multi_device_handle_leg(psd_b200, L, torch, world, B, n, p):
    """The library's own multi-GPU path: ONE psd_rpschur_batched call on a handle that owns all
    `world` devices (one host thread + streams per device inside the library, contiguous batch
    shards, host-side gather; no collective), pinned host buffers, H2D/D2H inside the timed region."""
    import psutil
    need = world * B * (p * n * n * 8 + n * 16 + 4)
    if psutil.virtual_memory().available < 2.5 * need:
        return {"skipped": f"needs {need / 2**30:.1f} GiB of pinned host memory"}
    hA = torch.empty((world * B, p, n, n), dtype=torch.float64, pin_memory=True)
    psd_b200.capi.check(L.psd_fill_uniform_host(SEED, n, p, world * B, 0, 0, C.c_void_p(hA.data_ptr())))
    hE = torch.empty((world * B, n, 2), dtype=torch.float64, pin_memory=True)
    hI = torch.empty(world * B, dtype=torch.int32, pin_memory=True)
    hh = psd_b200.Handle(list(range(world)))

    def step():
        psd_b200.capi.check(L.psd_rpschur_batched(hh.ptr, n, p, world * B, 0, 0, 0, 30, C.c_void_p(hA.data_ptr()),
                                                  None, C.c_void_p(hE.data_ptr()), C.c_void_p(hI.data_ptr())))
    step()
    t0 = time.perf_counter()
    step(); step()
    dt = (time.perf_counter() - t0) / 2
    st = hh.stats()
    out = {"value": world * B / dt, "unit": "problems/s", "devices": world, "seconds_per_call": dt,
           "h2d_bytes_per_call": st["h2d_bytes"], "d2h_bytes_per_call": st["d2h_bytes"],
           "unconverged": int((hI != 0).sum().item()),
           "what": "one psd_rpschur_batched call on Handle(range(N)), rank 0 only, other ranks idle"}
    hh.close()
    return out


DUMP_LIMIT_BYTES = 64_000_000
NPY_HEADER_BYTES = 4096  # allowance per file, far above numpy's actual header size


def dump_outputs(out_dir, E, I):
    """Write the device-resident path's results E [B][n][2] and I [B] (see --dump-outputs): every
    problem when they fit DUMP_LIMIT_BYTES, else a seeded sample of problems in batch order."""
    import numpy as np
    import torch
    B = E.shape[0]
    per_problem = (E[0].numel() + 2) * 8   # eigenvalues, info and index, as float64
    budget = DUMP_LIMIT_BYTES - 3 * NPY_HEADER_BYTES
    if B * per_problem <= budget:
        idx = np.arange(B)
    else:
        idx = np.sort(np.random.default_rng(SEED).choice(B, budget // per_problem, replace=False))
    sel = torch.from_numpy(idx).to(E.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "eigenvalues.npy"), E[sel].cpu().numpy())
    np.save(os.path.join(out_dir, "info.npy"), I[sel].cpu().numpy().astype(np.float64))
    np.save(os.path.join(out_dir, "problem_index.npy"), idx.astype(np.float64))


def run_ours(args):
    import numpy as np
    import torch
    import psd_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    L = psd_b200.lib()
    h = psd_b200.Handle([local_rank])
    n, p, B = N_ORDER, PERIOD, args.batch
    first_b = rank * B

    # ---- inputs: pinned host master copy + device copy (6.55 GB per GPU at B=100k > L2) ----
    hA = pinned_input(L, psd_b200, torch, local_rank, (B, p, n, n))
    psd_b200.capi.check(L.psd_fill_uniform_host(SEED, n, p, B, first_b, 0, C.c_void_p(hA.data_ptr())))
    hE = torch.empty((B, n, 2), dtype=torch.float64, pin_memory=True)
    hI = torch.empty(B, dtype=torch.int32, pin_memory=True)
    dA = hA.to(dev)
    dE = torch.empty((B, n, 2), dtype=torch.float64, device=dev)
    dI = torch.empty(B, dtype=torch.int32, device=dev)
    ts = torch.cuda.Stream(device=dev)

    def step_dev():
        psd_b200.capi.check(L.psd_rpschur_batched_dev(
            h.ptr, 0, C.c_void_p(ts.cuda_stream), n, p, B, 0, 0, 0, 30,
            C.c_void_p(dA.data_ptr()), None, C.c_void_p(dE.data_ptr()), C.c_void_p(dI.data_ptr())))

    # eigenvalues-only mode never writes A back (wantT=false), so the HBM-resident input is
    # reused as is; it is 52x larger than L2, so every step streams it from HBM again.
    with torch.cuda.stream(ts):
        for _ in range(args.warmup):
            step_dev()
    barrier()
    h.set_profiling(True)   # CUDA events around every kernel launch, on the launching stream
    h.kernel_times()        # drop anything recorded so far
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    evs = []
    with torch.cuda.stream(ts):
        for _ in range(args.steps):
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            step_dev()
            e1.record()
            evs.append((e0, e1))
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    kt = h.kernel_times()
    h.set_profiling(False)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dE, dI)
    kernel_ms = [a.elapsed_time(b) for a, b in evs]
    total_ms = evs[0][0].elapsed_time(evs[-1][1])
    total_ms = max_over_ranks(total_ms)
    fails = int((dI != 0).sum().item())
    ms_per_step = total_ms / args.steps
    value = world * B / (ms_per_step * 1e-3)

    # ---- end to end through the host C-ABI call (pinned host buffers, H2D + D2H inside) ----
    def step_e2e():
        psd_b200.capi.check(L.psd_rpschur_batched(
            h.ptr, n, p, B, 0, 0, 0, 30, C.c_void_p(hA.data_ptr()), None,
            C.c_void_p(hE.data_ptr()), C.c_void_p(hI.data_ptr())))

    e2e_steps = args.steps
    step_e2e()  # warm-up (allocates the handle's device buffers)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_e2e()
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0) / e2e_steps
    st = h.stats()
    e2e_value = world * B / e2e_s
    # e2e result check: same eigenvalues as the device-resident path
    same = bool(torch.equal(hE, dE.cpu()))

    # the library's in-process multi-device path, measured by rank 0 while the other ranks wait
    handle_leg = None
    if world > 1:
        del dA
        torch.cuda.empty_cache()
        barrier()
        # the waiting ranks must not touch their GPUs: a NCCL barrier spins a kernel on every device
        # (measured: 218 k instead of 430 k problems/s on 2 GPUs), so they wait in a gloo barrier
        cpu_pg = dist.new_group(backend="gloo")
        if rank == 0:
            try:
                handle_leg = multi_device_handle_leg(psd_b200, L, torch, world, B, n, p)
            except Exception as ex:
                handle_leg = {"error": repr(ex)}
        dist.barrier(group=cpu_pg)

    if rank != 0:
        return 0

    peak, peak_kind = _peaks()
    step_ms = sum(kernel_ms) / len(kernel_ms)
    # dominant kernel: the eigenvalue-only periodic QR iteration (psd::rpqr_eig32_kernel_t); its
    # launches each process min(B, 65536) problems.  achieved = SURVEY.md §8(d) bytes per
    # problem x problems per launch / average launch duration (CUDA events on its stream).
    n_it = max(1, kt["iterate_launches"])
    k_ms = kt["iterate_ms"] / n_it
    units_per_launch = B * args.steps / n_it
    achieved = BYTES_PER_PROBLEM * units_per_launch / (k_ms * 1e-3) / 1e9
    traffic = None
    fp64_issue = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            with open(tpath) as f:
                tj = json.load(f)
            traffic = tj.get("rpqr_eig32_dram_bytes_per_problem")
            ph = tj.get("rpqr_eig32_phases", [])
            wi = tj.get("warp_instructions_per_problem_iteration")
            if ph and wi:
                tms = sum(x["ms"] for x in ph)
                # second roofline of the dominant kernel: it is bound by the FP64 pipe / issue slots,
                # not by HBM.  Counters from the committed ncu capture of the final kernels
                # (profiles/r2_c2_final_kernels_ncu_full_raw.csv), time-weighted over the six phases.
                fp64_issue = {
                    "bound": "fp64 pipe / issue slots (latency-bound dependent chain)",
                    "pipe_fp64_cycles_active_pct": sum(x["pipe_fp64_active_pct"] * x["ms"] for x in ph) / tms,
                    "issue_active_pct": sum(x["issue_active_pct"] * x["ms"] for x in ph) / tms,
                    "warps_active_pct": sum(x["warps_active_pct"] * x["ms"] for x in ph) / tms,
                    "executed_warp_instructions_per_problem": wi,
                    "standard_flops_per_problem": FLOPS_PER_PROBLEM,
                    "source": "ncu --set full, launches of one 20000-problem step (profiles/traffic.json)"}
        except Exception:
            traffic = None
    line = {
        "metric": "pschur!/sec batched (p=8,N=32); large-N FP64 % peak in large_n", "value": value, "unit": "problems/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": bench_config(B, world),
        "e2e": {"value": e2e_value, "unit": "problems/s", "h2d_bytes_per_step": st["h2d_bytes"],
                "d2h_bytes_per_step": st["d2h_bytes"], "steps": e2e_steps,
                "matches_device_path": same},
        "gpu_launches": kt["iterate_launches"] + kt["reduce_launches"] + kt["extra_launches"],
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak,
                     "traffic": (traffic * units_per_launch) if traffic else None,
                     "traffic_note": ("DRAM bytes of the six phase launches that one timed 'launch' stands for "
                                      "(ncu capture of the final kernels, profiles/traffic.json, written by "
                                      "scripts/ncu_traffic.py): %.1f KB per problem = %.1fx the path-level "
                                      "%d B, because every phase hands the packed prefixes to the next one "
                                      "through HBM" % (traffic / 1e3, traffic / BYTES_PER_PROBLEM, BYTES_PER_PROBLEM))
                                     if traffic else None,
                     "fp64_issue": fp64_issue,
                     "peak_kind": f"of {peak_kind}",
                     "kernel": "psd::rpqr_eig32_kernel_t (six occupancy phases, orders 32..12, timed together)",
                     "kernel_ms": k_ms,
                     "problems_per_launch": units_per_launch,
                     "kernel_share_of_step": kt["iterate_ms"] / (kt["iterate_ms"] + kt["reduce_ms"]),
                     "reduce_kernel": "psd::rphess_pair32_kernel_t<32,8>",
                     "reduce_kernel_ms": kt["reduce_ms"] / max(1, kt["reduce_launches"]),
                     "step_ms_device": step_ms,
                     "fp64_gflops_standard_count": FLOPS_PER_PROBLEM * B / (step_ms * 1e-3) / 1e9,
                     "note": "latency-bound serial bulge-chase chain per problem; see DESIGN.md"},
        "clocks": clocks,
        "unconverged": fails,
    }
    if handle_leg is not None:
        line["e2e_single_call_all_devices"] = handle_leg
    if world == 1:
        try:
            line["config1"] = config1_block(psd_b200, h)
        except Exception as ex:
            line["config1"] = {"error": repr(ex)}
    if world == 1 and not args.no_large:
        try:
            del dA, dE, dI
            torch.cuda.empty_cache()
            line["large_n"] = large_n_block(torch, psd_b200, L, h, dev)
            line["large_n"]["cpu_baseline"] = cpu_large_baseline()
            line["large_n"]["speedup_vs_cpu_extrapolated"] = (
                line["large_n"]["cpu_baseline"]["seconds_extrapolated_n4096"] / line["large_n"]["seconds"])
        except Exception as ex:  # the headline line must still be printed
            line["large_n"] = {"error": repr(ex)}
    if world == 1:
        # bounded CPU sample: ~10-20 s on the box's host cores
        probe, cores, _ = cpu_reference_rate(max(64, 32 * host_cores()))
        sample = int(max(512, min(B, probe * 12.0)))
        rate, cores, dt = cpu_reference_rate(sample)
        line["cpu_baseline"] = {
            "value": rate, "unit": "problems/s", "cores": cores, "kind": "port",
            "sample": f"{sample} problems of the same workload in {dt:.1f} s; C++ restatement of "
                      f"the reference (Julia unavailable), OpenMP over the batch"}
    print(json.dumps(line))
    return 0


def _shutdown():
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            dist.destroy_process_group()
    except Exception:
        pass


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=100000, help="problems per GPU per step")
    ap.add_argument("--no-large", dest="no_large", action="store_true",
                    help="skip the large-N (p=4, N=4096) block of the N=1 line")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR",
                    help="write the results of the last timed step as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    try:
        return run_ours(args)
    finally:
        _shutdown()


if __name__ == "__main__":
    sys.exit(main())
