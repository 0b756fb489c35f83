"""The chunked, slot-pipelined shard loop behind every batched host call (psd_capi.cu, run_shard):
for each entry family, one call on a batch of at least three chunks must return, bit for bit,
what separate calls on slices around the chunk boundaries return, on pageable and on pinned host
buffers; h2d_bytes and d2h_bytes must match their closed forms."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SM_COUNT = 148  # B200: a generalized chunk is a whole number of waves of 2 * SM_COUNT problems


def real_chunks(count, per, pinned):
    """chunk sizes of the real standard path (plan_real_chunks) for per bytes of factors"""
    chunk = max(1, (2048 << 20) // per)
    if not pinned:
        chunk = max(1, min(chunk, (512 << 20) // per))
    chunk = min(chunk, count)
    if not pinned and count * per >= (64 << 20) and count >= 8:
        chunk = min(chunk, (count + 3) // 4)
    out, nxt = [], (max(1, chunk // (16 if pinned else 2)) if count > chunk else chunk)
    while sum(out) < count:
        out.append(min(nxt, count - sum(out)))
        nxt = min(chunk, nxt * 4)
    return out


def gen_chunks(count, per):
    """chunk sizes of the generalized paths (plan_gen_chunks); the device-memory cap does not
    bind at these sizes"""
    wave = 2 * SM_COUNT
    chunk = min(-(-max(1, (512 << 20) // per) // wave) * wave, count)
    return [min(chunk, count - o) for o in range(0, count, chunk)]


def around_cuts(B, plan, halo, ndev=1):
    """slices around every chunk boundary of every device's share, plus the first and last
    problems; every share must span at least three chunks"""
    cuts = []
    for d in range(ndev):
        lo, hi = B * d // ndev, B * (d + 1) // ndev
        chunks = plan(hi - lo)
        assert len(chunks) >= 3
        cuts += [lo] if d else []
        cuts += [lo + int(c) for c in np.cumsum(chunks)[:-1]]
    return [slice(0, halo)] + [slice(c - halo, c + halo) for c in cuts] + [slice(B - halo, B)]


def vp(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def fill(psd, A, first=0):
    """uniform factors of problems first.. (the library's counter-based generator, seed 7)"""
    batch, p, n, _ = A.shape
    psd.capi.check(psd.lib().psd_fill_uniform_host(7, n, p, batch, first, int(A.dtype == np.complex128),
                                                   A.ctypes.data))
    return A


def inputs(psd, sl, p, n, dtype):
    return fill(psd, np.empty((sl.stop - sl.start, p, n, n), dtype), sl.start)


@pytest.fixture
def pinned(psd):
    """allocator of page-locked numpy arrays (psd_host_alloc), freed after the test"""
    L = psd.lib()
    ptrs = []

    def empty(shape, dtype):
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        ptr = C.c_void_p()
        psd.capi.check(L.psd_host_alloc(nbytes, 0, C.byref(ptr)))
        ptrs.append(ptr)
        return np.frombuffer((C.c_char * nbytes).from_address(ptr.value), dtype=dtype).reshape(shape)

    yield empty
    for ptr in ptrs:
        L.psd_host_free(ptr)


@pytest.mark.parametrize("mode", ["pageable", "pinned"])
def test_real_eigenvalues_only(psd, pinned, mode):
    n, p = 32, 8
    per = p * n * n * 8
    B = 40000 if mode == "pinned" else 9001  # pinned chunks hold up to 2 GiB of factors
    alloc = pinned if mode == "pinned" else np.empty
    A = fill(psd, alloc((B, p, n, n), np.float64))
    eig, info = alloc((B, n), np.complex128), alloc(B, np.int32)
    h = psd.Handle()
    psd.capi.check(psd.lib().psd_rpschur_batched(h.ptr, n, p, B, 0, 0, 0, 30, vp(A), None, vp(eig), vp(info)))
    st = h.stats()
    assert st["h2d_bytes"] == B * per and st["d2h_bytes"] == B * (16 * n + 4)
    for sl in around_cuts(B, lambda c: real_chunks(c, per, mode == "pinned"), 40):
        _, _, e, i = psd.pschur_batched(A[sl], "R", wantT=False, wantZ=False)
        assert np.array_equal(eig[sl], e) and np.array_equal(info[sl], i)
    h.close()


@pytest.mark.parametrize("mode", ["pageable", "pinned"])
def test_real_T_Z_iters(psd, pinned, mode):
    """pageable: a handle that lists device 0 twice, so that two pipelines share the GPU; pinned:
    the iteration counts are pinned too and copied without staging"""
    if mode == "pinned":
        n, p, B, ndev = 16, 8, 140000, 1
        A, Z = fill(psd, pinned((B, p, n, n), np.float64)), pinned((B, p, n, n), np.float64)
        eig, info, it = pinned((B, n), np.complex128), pinned(B, np.int32), pinned(B, np.int32)
        h = psd.Handle()
        L = psd.lib()
        psd.capi.check(L.psd_set_iters_output(h.ptr, vp(it)))
        try:
            psd.capi.check(L.psd_rpschur_batched(h.ptr, n, p, B, 0, 1, 1, 30, vp(A), vp(Z), vp(eig), vp(info)))
        finally:
            L.psd_set_iters_output(h.ptr, None)
        T = A
    else:
        n, p, B, ndev = 20, 3, 16000, 2
        h = psd.Handle([0, 0])
        T, Z, eig, info, it = psd.pschur_batched(fill(psd, np.empty((B, p, n, n))), "R", handle=h,
                                                 return_iters=True)
    per = p * n * n * 8
    st = h.stats()
    assert st["h2d_bytes"] == B * per and st["d2h_bytes"] == B * (2 * per + 16 * n + 4)  # iters not counted
    assert (it > 0).all()
    for sl in around_cuts(B, lambda c: real_chunks(c, per, mode == "pinned"), 40, ndev):
        Ts, Zs, es, i, its = psd.pschur_batched(inputs(psd, sl, p, n, np.float64), "R", return_iters=True)
        for x, y in ((T, Ts), (Z, Zs), (eig, es), (info, i), (it, its)):
            assert np.array_equal(x[sl], y)
    h.close()


def test_real_hessut_q(psd):
    """Z goes in (the caller's Q) as well as out"""
    n, p, B = 20, 3, 8000
    per = p * n * n * 8
    H, Q = psd.phessenberg_batched(fill(psd, np.empty((B, p, n, n))))
    h = psd.Handle()
    T, Z, eig, info = psd.pschur_hessut_batched(H, Q=Q, handle=h)
    st = h.stats()
    assert st["h2d_bytes"] == 2 * B * per and st["d2h_bytes"] == B * (2 * per + 16 * n + 4)
    for sl in around_cuts(B, lambda c: real_chunks(c, per, False), 40):
        out = psd.pschur_hessut_batched(H[sl], Q=Q[sl])
        for x, y in zip((T, Z, eig, info), out):
            assert np.array_equal(x[sl], y)
    h.close()


def test_real_reduce_only(psd):
    """psd_rphess_batched returns H and Q only: no eigenvalue or info bytes come back"""
    n, p, B = 20, 3, 8000
    per = p * n * n * 8
    A = fill(psd, np.empty((B, p, n, n)))
    h = psd.Handle()
    H, Q = psd.phessenberg_batched(A, handle=h)
    st = h.stats()
    assert st["h2d_bytes"] == B * per and st["d2h_bytes"] == 2 * B * per
    for sl in around_cuts(B, lambda c: real_chunks(c, per, False), 40):
        Hs, Qs = psd.phessenberg_batched(A[sl])
        assert np.array_equal(H[sl], Hs) and np.array_equal(Q[sl], Qs)
    h.close()


S16 = [1, 1, 0, 1] * 4


@pytest.mark.parametrize("mode", ["pageable", "pinned"])
def test_complex_T_Z(psd, pinned, mode):
    n, p, B = 64, 16, 1300  # 1 MiB of factors per problem: chunks of 592
    per = p * n * n * 16
    if mode == "pinned":
        A, Z = fill(psd, pinned((B, p, n, n), np.complex128)), pinned((B, p, n, n), np.complex128)
        alpha, beta = pinned((B, n), np.complex128), pinned((B, n), np.complex128)
        scale, info = pinned((B, n), np.int64), pinned(B, np.int32)
        h = psd.Handle()
        S = np.array(S16, dtype=np.uint8)
        psd.capi.check(psd.lib().psd_cpschur_batched(h.ptr, n, p, B, 0, vp(S), 1, 1, 0, vp(A), vp(Z), vp(alpha),
                                                     vp(beta), vp(scale), vp(info)))
        out = (A, Z, alpha, beta, scale, info)
    else:
        h = psd.Handle()
        out = psd.gpschur_batched(fill(psd, np.empty((B, p, n, n), np.complex128)), S16, handle=h)
    st = h.stats()
    assert st["h2d_bytes"] == B * per and st["d2h_bytes"] == B * (2 * per + 40 * n + 4)
    for sl in around_cuts(B, lambda c: gen_chunks(c, per), 8):
        ref = psd.gpschur_batched(inputs(psd, sl, p, n, np.complex128), S16)
        for x, y in zip(out, ref):
            assert np.array_equal(x[sl], y)
    h.close()


def test_real_generalized(psd):
    n, p, B = 64, 16, 2500  # 512 KiB of factors per problem: chunks of 1184
    per = p * n * n * 8
    h = psd.Handle()
    out = psd.gpschur_batched(fill(psd, np.empty((B, p, n, n))), S16, handle=h)
    st = h.stats()
    assert st["h2d_bytes"] == B * per and st["d2h_bytes"] == B * (2 * per + 32 * n + 4)
    for sl in around_cuts(B, lambda c: gen_chunks(c, per), 8):
        ref = psd.gpschur_batched(inputs(psd, sl, p, n, np.float64), S16)
        for x, y in zip(out, ref):
            assert np.array_equal(x[sl], y)
    h.close()


@pytest.mark.parametrize("dtype,n,B", [
    (np.complex128, 64, 1300),  # chunks of 592 staged through pinned buffers
    (np.float64, 180, 800),     # chunks of 296 problems, 1.2 GB: copied directly from pageable memory
])
def test_generalized_reduce_only(psd, dtype, n, B):
    """psd_gphess_batched returns H and Q only: no alpha, beta, alphascale or info bytes"""
    p = 16
    per = p * n * n * np.dtype(dtype).itemsize
    A = fill(psd, np.empty((B, p, n, n), dtype))
    h = psd.Handle()
    H, Q = psd.gphessenberg_batched(A, S16, handle=h)
    st = h.stats()
    assert st["h2d_bytes"] == B * per and st["d2h_bytes"] == 2 * B * per
    for sl in around_cuts(B, lambda c: gen_chunks(c, per), 8):
        Hs, Qs = psd.gphessenberg_batched(A[sl], S16)
        assert np.array_equal(H[sl], Hs) and np.array_equal(Q[sl], Qs)
    h.close()
