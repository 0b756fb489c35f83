"""Host-side mirror of the reference's dense periodic Schur interface.

Reference methods mirrored (file:line relative to the reference repository):
  pschur(A, lr; kwargs...)                      PeriodicSchurDecompositions.jl:108-113
  pschur!(A, lr; wantZ, wantT, maxitfac)        PeriodicSchurDecompositions.jl:120-152
  PeriodicSchur                                  PeriodicSchurDecompositions.jl:59-92
  char_lr / throw_lr                             PeriodicSchurDecompositions.jl:155-177
  phessenberg!(A)                                PeriodicSchurDecompositions.jl:213-259

Storage convention: the C ABI takes column-major factors (Julia `Matrix`).  A numpy matrix `M`
(math orientation) is therefore handed over as `M.T` made C-contiguous; the batched functions
take/return arrays already in that storage layout, [batch][p][col][row].
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

from . import capi
from .capi import PsdError, check, lib


def shard_bounds(batch: int, world: int, rank: int):
    """Contiguous batch shard [lo, hi) owned by `rank` of `world` (SURVEY.md §8(e)); the same
    split the C library applies across the devices of a handle (batch*d/nd)."""
    return batch * rank // world, batch * (rank + 1) // world


def char_lr(lr) -> str:
    """PeriodicSchurDecompositions.jl:155-177"""
    if lr in ("R", ":R", "r"):
        return "R"
    if lr in ("L", ":L", "l"):
        return "L"
    raise ValueError("orientation argument must be either :R (right) or :L (left)")


@dataclass
class PeriodicSchur:
    """Mirror of the reference result struct (PeriodicSchurDecompositions.jl:59-92).

    T1: the quasi-triangular Schur factor T_k, k = schurindex; T: the other p-1 triangular
    factors in order; Z: the p orthogonal factors; values: eigenvalues of the product.
    All matrices are numpy arrays in math orientation."""
    T1: np.ndarray
    T: List[np.ndarray]
    Z: List[np.ndarray]
    values: np.ndarray
    orientation: str = "R"
    schurindex: int = 1
    info: int = 0
    extra: dict = field(default_factory=dict)

    @property
    def period(self) -> int:
        return len(self.T) + 1


@dataclass
class GeneralizedPeriodicSchur:
    """Mirror of the reference result struct (generalized.jl:31-85): S, schurindex, T1, T, Z,
    alpha, beta, alphascale, orientation; values = alpha ./ beta .* 2^alphascale (:75-76)."""
    S: List[bool]
    schurindex: int
    T1: np.ndarray
    T: List[np.ndarray]
    Z: List[np.ndarray]
    alpha: np.ndarray
    beta: np.ndarray
    alphascale: np.ndarray
    orientation: str = "R"
    info: int = 0

    @property
    def period(self) -> int:
        return len(self.S)

    @property
    def values(self) -> np.ndarray:
        return gvalues(self.alpha, self.beta, self.alphascale)


def gvalues(alpha, beta, alphascale):
    """alpha ./ beta .* 2^alphascale (generalized.jl:75-76); beta == 0 gives a non-finite value."""
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        return alpha / beta * np.exp2(np.asarray(alphascale, dtype=np.float64))


class Handle:
    """Owns a psd_handle_t (streams, device workspaces, pinned staging)."""

    def __init__(self, devices: Optional[Sequence[int]] = None):
        self._h = C.c_void_p()
        if devices is None:
            check(lib().psd_create(C.byref(self._h), 0, None))
        else:
            arr = (C.c_int * len(devices))(*devices)
            check(lib().psd_create(C.byref(self._h), len(devices), arr))

    @property
    def ptr(self):
        return self._h

    @property
    def ndev(self) -> int:
        return int(lib().psd_handle_device_count(self._h))

    def stats(self):
        s = (C.c_int64 * 8)()
        check(lib().psd_last_stats(self._h, s))
        return {"launches": s[0], "problems_smem": s[1], "problems_global": s[2],
                "h2d_bytes": s[3], "d2h_bytes": s[4], "wall_us": s[5]}

    def set_profiling(self, on: bool):
        check(lib().psd_set_profiling(self._h, int(on)))

    def kernel_times(self):
        """Device time (ms) of the kernels launched since the last call, by kind."""
        ms = (C.c_double * 8)()
        check(lib().psd_kernel_times(self._h, ms))
        return {"reduce_ms": ms[0], "iterate_ms": ms[1], "reduce_launches": int(ms[2]),
                "iterate_launches": int(ms[3]), "large_panel_ms": ms[4], "large_gemm_ms": ms[5],
                "large_gemm_flops": ms[6], "extra_launches": int(ms[7])}

    def large_stats(self):
        """Counters of the most recent large-N multishift iteration (psd_large_stats)."""
        o = (C.c_double * 16)()
        check(lib().psd_large_stats(self._h, o))
        names = ["status", "sweeps", "rounds", "windows", "shift_pairs", "exceptional", "final_blocks",
                 "launches", "apply_flops", "chase_ms", "apply_ms", "shifts_ms", "scan_ms", "final_ms", "rounds_ms", "wall_s"]
        return {k: (o[i] if k.endswith(("_ms", "_flops", "_s")) else int(o[i])) for i, k in enumerate(names)}

    def close(self):
        if self._h:
            lib().psd_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default: Optional[Handle] = None


def default_handle() -> Handle:
    global _default
    if _default is None:
        _default = Handle()
    return _default


def _vp(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def pschur_batched(A: np.ndarray, lr="R", wantZ: bool = True, wantT: bool = True,
                   maxitfac: int = 30, handle: Optional[Handle] = None, overwrite: bool = False,
                   return_iters: bool = False):
    """Batched real periodic Schur decomposition through psd_rpschur_batched.

    A: float64 [batch][p][n][n], each factor column-major (storage layout), user factor order.
    Returns (T, Z, values, info): T is A overwritten (a copy unless overwrite=True), Z is None
    when wantZ is False, values complex128 [batch][n], info int32 [batch].  return_iters=True
    appends the QR iterations per problem (psd_set_iters_output; int32 [batch])."""
    orient = char_lr(lr)
    if A.dtype != np.float64 or A.ndim != 4 or A.shape[2] != A.shape[3]:
        raise ValueError("A must be float64 with shape [batch][p][n][n]")  # DimensionMismatch, :220
    h = handle or default_handle()
    batch, p, n, _ = A.shape
    T = A if (overwrite and A.flags.c_contiguous) else np.ascontiguousarray(A).copy()
    Z = np.empty_like(T) if wantZ else None
    vals = np.empty((batch, n), dtype=np.complex128)
    info = np.empty(batch, dtype=np.int32)
    iters = np.zeros(batch, dtype=np.int32) if return_iters else None
    if return_iters:
        check(lib().psd_set_iters_output(h.ptr, _vp(iters)))
    try:
        check(lib().psd_rpschur_batched(h.ptr, n, p, batch, 1 if orient == "L" else 0, int(wantT),
                                        int(wantZ), int(maxitfac), _vp(T), _vp(Z), _vp(vals),
                                        _vp(info)))
    finally:
        if return_iters:
            lib().psd_set_iters_output(h.ptr, None)
    if return_iters:
        return T, Z, vals, info, iters
    return T, Z, vals, info


def phessenberg_packed_batched(A: np.ndarray, handle: Optional[Handle] = None):
    """phessenberg!(A) with the result in the reference's packed form (:229-253): returns (F, tau),
    F[b][j] = H_j in the upper part and the Householder vectors below it, tau [batch][p][n]."""
    h = handle or default_handle()
    batch, p, n, _ = A.shape
    F = np.ascontiguousarray(A, dtype=np.float64).copy()
    tau = np.empty((batch, p, n))
    check(lib().psd_rphess_packed_batched(h.ptr, n, p, batch, _vp(F), _vp(tau)))
    return F, tau


def checkpsd_batched(A: np.ndarray, T: np.ndarray, Z: np.ndarray, lr="R", thresh: float = 100.0,
                     strict: bool = True, handle: Optional[Handle] = None):
    """checkpsd(P, Hs) (diagnostics.jl:190-263) for batched real results, norms computed on the
    device (psd_rcheckpsd_batched).  Returns (ok [batch] bool, err [batch][p], tri, orth)."""
    orient = char_lr(lr)
    h = handle or default_handle()
    batch, p, n, _ = A.shape
    A = np.ascontiguousarray(A, dtype=np.float64)
    T = np.ascontiguousarray(T, dtype=np.float64)
    Z = np.ascontiguousarray(Z, dtype=np.float64)
    err = np.empty((batch, p)); tri = np.empty((batch, p)); orth = np.empty((batch, p))
    check(lib().psd_rcheckpsd_batched(h.ptr, n, p, batch, 1 if orient == "L" else 0, _vp(A), _vp(T), _vp(Z),
                                      _vp(err), _vp(tri), _vp(orth)))
    eps = np.finfo(np.float64).eps
    cmp = 0.0 if strict else 10 * eps * n          # ttol, :212, 225
    ok = (tri <= cmp).all(axis=1) & (orth <= 10 * eps * n).all(axis=1) & (err <= thresh).all(axis=1)
    return ok, err, tri, orth


def eigvecs_batched(T: np.ndarray, Z: np.ndarray, lr="R", select=None, handle: Optional[Handle] = None):
    """Eigenvectors of batched periodic Schur results (psd_reigvecs_batched for float64 T and Z,
    psd_ceigvecs_batched for complex128), by periodic back-substitution on the Schur form.

    T, Z: [batch][p][n][n] storage layout, user factor order, as pschur_batched / gpschur_batched
    (S all true) return them.  select: [batch][n] (or [n] for every problem) booleans, None = all.
    Returns (V, info): V complex128 [batch][p][n][n] with column k of V[b, l] the unit vector v_l of
    eigenvalue k (zero where not selected), info int32 [batch] (1 = T not in periodic Schur form)."""
    orient = char_lr(lr)
    if T.ndim != 4 or T.shape[2] != T.shape[3] or T.shape != Z.shape or T.dtype != Z.dtype \
            or T.dtype not in (np.float64, np.complex128):
        raise ValueError("T and Z must be float64 or complex128 with equal shape [batch][p][n][n]")
    h = handle or default_handle()
    batch, p, n, _ = T.shape
    T = np.ascontiguousarray(T)
    Z = np.ascontiguousarray(Z)
    sel = None
    if select is not None:
        sel = np.ascontiguousarray(np.broadcast_to(np.asarray(select, dtype=bool), (batch, n)).astype(np.uint8))
    V = np.empty((batch, p, n, n), dtype=np.complex128)
    info = np.empty(batch, dtype=np.int32)
    f = lib().psd_ceigvecs_batched if T.dtype == np.complex128 else lib().psd_reigvecs_batched
    check(f(h.ptr, n, p, batch, 1 if orient == "L" else 0, _vp(T), _vp(Z), _vp(sel), _vp(V), _vp(info)))
    return V, info


def eigvecs(P: PeriodicSchur, select=None, handle: Optional[Handle] = None) -> List[np.ndarray]:
    """Eigenvectors of a PeriodicSchur result: p matrices (n x m, math orientation), matrix l holding
    v_l of every selected eigenvalue (all when select is None) in eigenvalue order; a complex pair
    is kept whole when either member is selected.  :R  A_l v_{l+1} = mu_l v_l,
    :L  A_l v_l = mu_l v_{l+1}, prod mu_l = values[k]."""
    p = P.period
    n = P.T1.shape[0]
    if len(P.Z) != p or P.Z[0].shape != (n, n):
        raise ValueError("eigvecs needs the Schur vectors (pschur with wantZ)")
    dt = np.complex128 if np.iscomplexobj(P.T1) else np.float64
    Ts = [P.T1] + list(P.T) if P.orientation == "R" else list(P.T) + [P.T1]
    T = np.empty((1, p, n, n), dtype=dt)
    Z = np.empty((1, p, n, n), dtype=dt)
    for j in range(p):
        T[0, j] = Ts[j].T
        Z[0, j] = P.Z[j].T
    V, info = eigvecs_batched(T, Z, P.orientation, None if select is None else np.asarray(select, bool)[None],
                              handle)
    if info[0] == 1:
        raise ValueError("the factors are not in periodic Schur form")
    if info[0] == 2:
        raise FloatingPointError("an eigenvector came out zero or not finite")
    # the columns the library fills: the selected ones, and a complex pair (exactly nonzero
    # subdiagonal of the Schur factor) whole when either member is selected
    keep = np.zeros(n, dtype=bool) if select is not None else np.ones(n, dtype=bool)
    if select is not None:
        sel = np.asarray(select, dtype=bool)
        c = 0
        while c < n:
            pair = dt == np.float64 and c + 1 < n and P.T1[c + 1, c] != 0
            w = 2 if pair else 1
            keep[c:c + w] = sel[c:c + w].any()
            c += w
    return [np.ascontiguousarray(V[0, l].T[:, keep]) for l in range(p)]


def pschur_hessut_batched(H: np.ndarray, wantZ: bool = True, wantT: bool = True, maxitfac: int = 30,
                          handle: Optional[Handle] = None, Q: Optional[np.ndarray] = None):
    """Inner method pschur!(H1, Hs; ...) (PeriodicSchurDecompositions.jl:322) on Hessenberg /
    triangular input, rightwards order, Z starting from the identity - or, with Q given (storage
    layout of H), accumulated onto it (the `Q` keyword of the reference, :326): Z = Q_j Z_j."""
    h = handle or default_handle()
    batch, p, n, _ = H.shape
    T = np.ascontiguousarray(H).copy()
    vals = np.empty((batch, n), dtype=np.complex128)
    info = np.empty(batch, dtype=np.int32)
    if Q is not None:
        if Q.shape != H.shape:
            raise ValueError("Q must have the shape of H")
        Z = np.ascontiguousarray(Q, dtype=np.float64).copy()
        check(lib().psd_rpschur_hessut_q_batched(h.ptr, n, p, batch, int(wantT), int(maxitfac),
                                                 _vp(T), _vp(Z), _vp(vals), _vp(info)))
        return T, Z, vals, info
    Z = np.empty_like(T) if wantZ else None
    check(lib().psd_rpschur_hessut_batched(h.ptr, n, p, batch, int(wantT), int(wantZ),
                                           int(maxitfac), _vp(T), _vp(Z), _vp(vals), _vp(info)))
    return T, Z, vals, info


def phessenberg_batched(A: np.ndarray, wantQ: bool = True, handle: Optional[Handle] = None):
    """phessenberg!(A) + explicit Q (PeriodicSchurDecompositions.jl:213-259, 136-140), batched,
    storage layout.  Returns (H, Q)."""
    h = handle or default_handle()
    batch, p, n, _ = A.shape
    H = np.ascontiguousarray(A).copy()
    Q = np.empty_like(H) if wantQ else None
    check(lib().psd_rphess_batched(h.ptr, n, p, batch, int(wantQ), _vp(H), _vp(Q)))
    return H, Q


def rphessenberg_rowwise_batched(Ap: np.ndarray, A: Optional[np.ndarray], Q: Optional[np.ndarray],
                                 handle: Optional[Handle] = None):
    """_rphessenberg!(Ap, A, Q) (rhessx.jl:53-109), batched, storage layout:
    Ap [batch][n][m] (column-major m x n, m = n or n+1), A [batch][p-1][n][n] or None,
    Q [batch][p][n][qrows] or None.  Returns updated copies (Ap, A, Q)."""
    h = handle or default_handle()
    batch, n, m = Ap.shape
    if m not in (n, n + 1):
        raise ValueError("only implemented for square or 1 extra row")  # rhessx.jl:60
    p = 1 if A is None else A.shape[1] + 1
    Ap2 = np.ascontiguousarray(Ap, dtype=np.float64).copy()
    A2 = None if A is None else np.ascontiguousarray(A, dtype=np.float64).copy()
    Q2 = None if Q is None else np.ascontiguousarray(Q, dtype=np.float64).copy()
    qrows = 0 if Q is None else Q.shape[3]
    check(lib().psd_rphess_rowwise_batched(h.ptr, n, int(m == n + 1), p, qrows, batch, _vp(Ap2),
                                           _vp(A2), _vp(Q2)))
    return Ap2, A2, Q2


def _sig(S, p):
    S = np.ascontiguousarray(np.asarray(S, dtype=bool).astype(np.uint8))
    if S.shape != (p,):
        raise ValueError("DimensionMismatch: S must have one entry per factor")
    return S


def gphessenberg_batched(A: np.ndarray, S, wantQ: bool = True, handle: Optional[Handle] = None):
    """_phessenberg!(A, S; wantQ) (generalized.jl:988-1082), batched, storage layout, float64 or
    complex128.  Returns (H, Q)."""
    h = handle or default_handle()
    batch, p, n, _ = A.shape
    Sb = _sig(S, p)
    H = np.ascontiguousarray(A).copy()
    Q = np.empty_like(H) if wantQ else None
    try:
        check(lib().psd_gphess_batched(h.ptr, int(A.dtype == np.complex128), n, p, batch, _vp(Sb),
                                       int(wantQ), _vp(H), _vp(Q)))
    except PsdError as e:
        if e.code == -4:
            raise ValueError("The first entry in S must be true") from e  # generalized.jl:990
        raise
    return H, Q


def gpschur_batched(A: np.ndarray, S, lr="R", wantZ: bool = True, wantT: bool = True,
                    maxitfac: int = 0, handle: Optional[Handle] = None, hessut: bool = False):
    """Batched generalized periodic Schur decomposition (psd_cpschur_batched for complex128 A;
    psd_rgpschur_batched for float64 A).  A: [batch][p][n][n] storage layout, user factor order;
    S: signature, user order.  hessut=True calls the inner entry point on Hessenberg-triangular
    input (rightwards order).  Returns (T, Z, alpha, beta, alphascale, info)."""
    orient = char_lr(lr)
    if A.ndim != 4 or A.shape[2] != A.shape[3] or A.dtype not in (np.complex128, np.float64):
        raise ValueError("A must be complex128 or float64 with shape [batch][p][n][n]")
    h = handle or default_handle()
    batch, p, n, _ = A.shape
    Sb = _sig(S, p)
    cplx = A.dtype == np.complex128
    T = np.ascontiguousarray(A).copy()
    Z = np.empty_like(T) if wantZ else None
    alpha = np.empty((batch, n), dtype=np.complex128)
    beta = np.empty((batch, n), dtype=np.complex128 if cplx else np.float64)
    scale = np.empty((batch, n), dtype=np.int64)
    info = np.empty(batch, dtype=np.int32)
    L = lib()
    if hessut:
        if orient != "R":
            raise ValueError("the Hessenberg-triangular entry point is rightwards only")
        f = L.psd_cpschur_hessut_batched if cplx else L.psd_rgpschur_hessut_batched
        check(f(h.ptr, n, p, batch, _vp(Sb), int(wantT), int(wantZ), int(maxitfac), _vp(T), _vp(Z),
                _vp(alpha), _vp(beta), _vp(scale), _vp(info)))
    else:
        f = L.psd_cpschur_batched if cplx else L.psd_rgpschur_batched
        check(f(h.ptr, n, p, batch, 1 if orient == "L" else 0, _vp(Sb), int(wantT), int(wantZ),
                int(maxitfac), _vp(T), _vp(Z), _vp(alpha), _vp(beta), _vp(scale), _vp(info)))
    return T, Z, alpha, beta, scale, info


def gpschur_(A: List[np.ndarray], S, lr="R", wantZ: bool = True, wantT: bool = True,
             handle: Optional[Handle] = None) -> GeneralizedPeriodicSchur:
    """pschur!(A, S, lr; wantZ, wantT) (generalized.jl:108-148 complex, rgeneralized.jl:3-45 real):
    overwrites A with the T factors and returns the reference's result struct."""
    orient = char_lr(lr)
    p = len(A)
    n = A[0].shape[0]
    dt = A[0].dtype
    for Aj in A:
        if Aj.ndim != 2 or Aj.shape != (n, n) or Aj.dtype != dt:
            raise ValueError("DimensionMismatch: all factors must be square of equal order and type")
    stor = np.empty((1, p, n, n), dtype=dt)
    for j in range(p):
        stor[0, j] = A[j].T
    try:
        T, Z, alpha, beta, scale, info = gpschur_batched(stor, S, orient, wantZ, wantT, 0, handle)
    except PsdError as e:
        if e.code == -4:
            raise ValueError("The leftmost entry in S must be true") from e  # ArgumentError
        raise
    if info[0] != 0:
        raise RuntimeError(f"convergence failed at level {int(info[0])}")
    for j in range(p):
        A[j][...] = T[0, j].T
    if orient == "R":
        T1, Ts, sidx = A[0], [A[j] for j in range(1, p)], 1
    else:
        T1, Ts, sidx = A[p - 1], [A[j] for j in range(0, p - 1)], p
    Zs = [np.ascontiguousarray(Z[0, j].T) for j in range(p)] if wantZ else []
    return GeneralizedPeriodicSchur([bool(x) for x in S], sidx, T1, Ts, Zs, alpha[0].copy(),
                                    beta[0].copy(), scale[0].copy(), orient, int(info[0]))


def cpschur_std_(A: List[np.ndarray], lr="R", wantZ: bool = True, wantT: bool = True,
                 handle: Optional[Handle] = None) -> PeriodicSchur:
    """Complex standard pschur!(A, lr) (PeriodicSchurDecompositions.jl:1106-1111): S = trues,
    result repackaged as PeriodicSchur with values = alpha ./ beta .* 2^alphascale."""
    F = gpschur_(A, [True] * len(A), lr, wantZ, wantT, handle)
    return PeriodicSchur(F.T1, F.T, F.Z, F.values, F.orientation, F.schurindex, F.info)


def pschur_(A: List[np.ndarray], lr="R", wantZ: bool = True, wantT: bool = True,
            maxitfac: int = 30, handle: Optional[Handle] = None) -> PeriodicSchur:
    """pschur!(A, lr; wantZ, wantT, maxitfac) (PeriodicSchurDecompositions.jl:120-152): the input
    matrices are used as workspace / overwritten with the T factors; T1 aliases A[0] (:R) or
    A[p-1] (:L) as in the reference (:265, :1078-1093)."""
    orient = char_lr(lr)
    p = len(A)
    if p < 1:
        raise ValueError("A must hold at least one matrix")
    n = A[0].shape[0]
    for Aj in A:
        if Aj.ndim != 2 or Aj.shape != (n, n):
            raise ValueError("DimensionMismatch: all factors must be square of equal order")
        if Aj.dtype not in (np.float64, np.complex128):
            raise TypeError("float64 or complex128 matrices expected")
    if A[0].dtype == np.complex128:
        return cpschur_std_(A, orient, wantZ, wantT, handle)
    for Aj in A:
        if Aj.dtype != np.float64:
            raise TypeError("all factors must have the same element type")
    stor = np.empty((1, p, n, n), dtype=np.float64)
    for j in range(p):
        stor[0, j] = A[j].T
    T, Z, vals, info = pschur_batched(stor, orient, wantZ, wantT, maxitfac, handle, overwrite=True)
    if info[0] != 0:
        raise RuntimeError(f"convergence failed at level {int(info[0])}")  # :891-893
    for j in range(p):
        A[j][...] = T[0, j].T
    if orient == "R":
        T1 = A[0]
        Ts = [A[j] for j in range(1, p)]
        sidx = 1
    else:
        T1 = A[p - 1]
        Ts = [A[j] for j in range(0, p - 1)]
        sidx = p
    if wantZ:
        Zs = [np.ascontiguousarray(Z[0, j].T) for j in range(p)]
    else:
        Zs = [np.zeros((0, 0))]  # :1074-1076
    return PeriodicSchur(T1, Ts, Zs, vals[0].copy(), orient, sidx, int(info[0]))


def pschur(A: Sequence[np.ndarray], lr="R", **kwargs) -> PeriodicSchur:
    """pschur(A, lr; kwargs...) (PeriodicSchurDecompositions.jl:108-113): copying wrapper."""
    dt = np.complex128 if any(np.iscomplexobj(Aj) for Aj in A) else np.float64
    return pschur_([np.array(Aj, dtype=dt, copy=True) for Aj in A], lr, **kwargs)


def gpschur(A: Sequence[np.ndarray], S, lr="R", **kwargs) -> GeneralizedPeriodicSchur:
    """pschur(A, S, lr; kwargs...) (generalized.jl:87-91): copying wrapper."""
    dt = np.complex128 if any(np.iscomplexobj(Aj) for Aj in A) else np.float64
    return gpschur_([np.array(Aj, dtype=dt, copy=True) for Aj in A], S, lr, **kwargs)
