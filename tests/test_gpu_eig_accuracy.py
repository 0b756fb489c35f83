"""Every eigenvalue of the real standard path against high-precision ground truth
(tests/golden/eigacc_golden.json; gate in tests/eigacc.py): each must be accurate relative to its
own structured condition number, not only relative to the largest eigenvalue of its problem.

The cases are chosen by the kernel they reach (dispatch: psd_capi.cu launch_real and
launch_real_eig32).  Eigenvalue-only, N <= 32, p >= 3: periodic Hessenberg-triangular reduction
(rphess_pair32 / rphess_ahead32) and the warp-per-problem QR (rpqr_eig32) over its occupancy phases:
  n3p3, n5p4       pair reduction, one phase
  n17p8            p >= 7 but the pair kernel keeps more problems resident
  n23p3            largest order without occupancy phases
  n24p3, n24p7     phases 24 -> 21 -> ... -> 9; p = 7 is the first p that considers the ahead kernel
  n31p8, n32p7     ahead kernel <0,0>, phases, the r168 kernel of the later phases
  n32p8, n32p12    the <32,8> specialisations; the largest p
  hessut           eigenvalue-only on Hessenberg-triangular input: rpschur_kernel packs, then eig32
Everything else takes the one-CTA rpschur_kernel: eigenvalue-only at p <= 2 (n20p1, n32p2), every
call with T and Z, and N = 64 in global-memory mode.  The scale cases put one factor below 2^-1000
(1e-305: normal, 1e-310: subnormal) or at 1.75e308, where the normalisation before the
eigenvalue-only iteration is capped or reaches its largest shift; the graded cases make many
eigenvalues ill-conditioned.  The one-CTA kernel does not normalise the factors and, like the
reference algorithm it restates (and the CPU oracle), does not converge on the scale cases, so
they run eigenvalue-only here.

Golden problems sit at the first, an inner and the last index of a prime-sized batch of seeded
filler problems, which only have to converge."""
import ctypes as C

import numpy as np
import pytest

import eigacc as EA

pytestmark = pytest.mark.gpu

GOLD = {g["id"]: g for g in EA.load()["problems"]}
BATCH = 101
POSITIONS = (0, 37, BATCH - 1)

# (problem group, path): eig = eigenvalues only, TZ = with T and Z; hessut* = Hessenberg-triangular input
CASES = ([(g, "eig") for g in ("n3p3", "n5p4", "n8p3", "n17p8", "n23p3", "n24p3", "n24p7", "n31p8R", "n31p8L",
                               "n32p7", "n32p8R", "n32p8L", "n32p12", "n20p1", "n32p2", "n64p8")] +
         [(g, "TZ") for g in ("n32p8R", "n32p8L", "n50p3", "n64p8", "n3p3", "n17p8")] +
         [(g, "hessut") for g in ("hessut-n17p3", "hessut-n32p8")] +
         [("hessut-n17p3", "hessut-TZ")] +
         [(g, "eig") for g in ("tiny305-n16p3", "tiny305-n32p8", "tiny310-n16p3", "tiny310-n32p8",
                               "huge-n16p3", "huge-n32p8")] +
         [(g, "hessut") for g in ("tiny305-hessut-n17p3", "tiny310-hessut-n17p3")] +
         [(g, path) for g in ("graded-n12p5", "graded-n32p4") for path in ("eig", "TZ")])


def _members(group):
    return [pid for pid, _ in EA.PROBLEMS if pid.rsplit("-b", 1)[0] == group]


def _filler(oracle, rec, batch, seed):
    A = oracle.gen_real(seed, rec["n"], rec["p"], batch)
    if rec["hessut"]:
        A = np.stack([EA.inputs(oracle, dict(rec, seed=seed, b=b, scale=[], peak=None, grade=0.0))
                      for b in range(batch)])
    return A


def _placed_batch(oracle, group, batch, positions, seed):
    pids = _members(group)
    A = _filler(oracle, GOLD[pids[0]]["recipe"], batch, seed)
    placed = {}
    for k, pos in enumerate(positions):
        placed[pos] = pids[k % len(pids)]
        A[pos] = EA.inputs(oracle, GOLD[placed[pos]]["recipe"])
    return A, placed


def _run_gpu(psd, rec, A, want_tz):
    if rec["hessut"]:
        T, _, lam, info = psd.pschur_hessut_batched(A, wantZ=want_tz, wantT=want_tz)
    else:
        T, _, lam, info = psd.pschur_batched(A, "L" if rec["left"] else "R", wantZ=want_tz, wantT=want_tz)
    return T, lam, info


@pytest.mark.parametrize("group,path", CASES, ids=[f"{g}-{p}" for g, p in CASES])
def test_eigenvalues_against_ground_truth(psd, oracle, group, path):
    pids = _members(group)
    rec0 = GOLD[pids[0]]["recipe"]
    n, p = rec0["n"], rec0["p"]
    want_tz = path.endswith("TZ")
    A, placed = _placed_batch(oracle, group, BATCH, POSITIONS, 4243)
    T, lam, info = _run_gpu(psd, rec0, A, want_tz)
    assert (info == 0).all(), np.flatnonzero(info)
    for pos, pid in placed.items():
        g = GOLD[pid]
        rec = g["recipe"]
        ref, kappa = EA.truth(g)
        _, lam_o, shift, info_o = EA.oracle_run(oracle, rec, A[pos], want_tz)
        assert info_o == 0
        err_o = EA.rel_errors(ref, EA.unshift(lam_o, shift))
        EA.check(ref, kappa, lam[pos], n, err_oracle=err_o, what=f"{pid} at index {pos}")
        EA.check_output_order(lam[pos], ref)
        if want_tz:
            EA.check_against_T(T[pos], lam[pos], rec["left"], EA.T_tolerance(ref, kappa, lam[pos], p, err_o))


def test_batch_across_the_eig_chunk_device_resident(psd, oracle):
    """More problems than one reduction + QR launch pair takes (65536): golden problems at 65535
    and 65536, on both sides of the boundary, and at the last index.  The device-resident entry
    keeps the whole batch in one call (the host entry splits a batch this large into copies)."""
    import torch
    B = 65539
    pos = (0, 65535, 65536, B - 1)
    A, placed = _placed_batch(oracle, "n8p3", B, pos, 4244)
    n, p = 8, 3
    h = psd.Handle([0])
    dA = torch.from_numpy(A).cuda()
    dE = torch.full((B, n, 2), np.nan, dtype=torch.float64, device="cuda")
    dI = torch.full((B,), -1, dtype=torch.int32, device="cuda")
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    psd.capi.check(psd.lib().psd_rpschur_batched_dev(
        h.ptr, 0, C.c_void_p(st.cuda_stream), n, p, B, 0, 0, 0, 30,
        C.c_void_p(dA.data_ptr()), None, C.c_void_p(dE.data_ptr()), C.c_void_p(dI.data_ptr())))
    torch.cuda.synchronize()
    info = dI.cpu().numpy()
    E = dE.cpu().numpy()
    lam = E[..., 0] + 1j * E[..., 1]
    assert (info == 0).all(), np.flatnonzero(info)
    assert np.isfinite(E).all()
    _, _, lam1, info1 = psd.pschur_batched(np.stack([A[i] for i in pos]), "R", wantZ=False, wantT=False, handle=h)
    assert (info1 == 0).all()
    for k, i in enumerate(pos):
        g = GOLD[placed[i]]
        ref, kappa = EA.truth(g)
        EA.check(ref, kappa, lam[i], n, what=f"{placed[i]} at index {i}")
        assert np.array_equal(lam[i], lam1[k]), i  # the same problem alone gives the same bits


def test_batch_across_the_eig_chunk_iteration_counts(psd, oracle):
    """The same boundary through the host entry (a batch this small is one launch), with the
    per-problem iteration counts: eigenvalues, info and iterations of the golden problems at
    65535, 65536 and the last index must be those of the same problems run alone."""
    B = 65539
    pos = (0, 65535, 65536, B - 1)
    A, placed = _placed_batch(oracle, "n3p3", B, pos, 4245)
    _, _, lam, info, iters = psd.pschur_batched(A, "R", wantZ=False, wantT=False, return_iters=True)
    assert (info == 0).all(), np.flatnonzero(info)
    assert (iters > 0).sum() > B // 2
    _, _, lam1, info1, iters1 = psd.pschur_batched(np.stack([A[i] for i in pos]), "R", wantZ=False, wantT=False,
                                                   return_iters=True)
    for k, i in enumerate(pos):
        g = GOLD[placed[i]]
        ref, kappa = EA.truth(g)
        EA.check(ref, kappa, lam[i], 3, what=f"{placed[i]} at index {i}")
        assert np.array_equal(lam[i], lam1[k]) and info[i] == info1[k] and iters[i] == iters1[k], i
