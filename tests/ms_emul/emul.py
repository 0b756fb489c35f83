"""TEST INFRASTRUCTURE ONLY: ctypes loader of tests/ms_emul/libms_emul.so (CPU emulation of the
large-N multishift iteration, built from the product's own host/device headers)."""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libms_emul.so")
_lib = None


def build():
    src = os.path.join(_HERE, "ms_emul.cpp")
    root = os.path.dirname(os.path.dirname(_HERE))
    deps = [src] + [os.path.join(root, "periodicschurdecompositions.jl_b200", "csrc", f)
                    for f in ("psd_ms_core.cuh", "psd_ms_driver.hpp")] + \
           [os.path.join(root, "oracle", f) for f in ("psdo_real.hpp", "psdo_common.hpp")]
    if not os.path.exists(_SO) or any(os.path.getmtime(d) > os.path.getmtime(_SO) for d in deps):
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-fopenmp", "-ffp-contract=off", "-Wall",
                        "-Wno-unused-function", "-shared", "-o", _SO, src], check=True)
    return _SO


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
    return _lib


def geom(p):
    out = (C.c_int * 4)()
    lib().ms_emul_geom(p, out)
    return {"W": out[0], "D": out[1], "NB": out[2], "LD": out[3]}


def run(H, Z, wantT=True, wantZ=True, nsw=0, rep_max=0, maxitfac=0, max_rounds=0):
    """H, Z: [p][n][n] storage (column-major factors), Hessenberg-triangular / preset Q.
    maxitfac: the caller's budget factor as psd_rpschur_batched takes it (<= 0: 30);
    max_rounds > 0: cap on the driver's rounds (the emulated kernels keep working).
    Returns (T, Z, eig, info, stats)."""
    p, n, _ = H.shape
    T = np.ascontiguousarray(H).copy()
    Zo = np.ascontiguousarray(Z).copy() if Z is not None else None
    eig = np.zeros((n, 2))
    info = C.c_int(0)
    stats = (C.c_longlong * 10)()
    dp = C.POINTER(C.c_double)
    lib().ms_emul_run(n, p, T.ctypes.data_as(dp), Zo.ctypes.data_as(dp) if Zo is not None else None,
                      int(wantT), int(wantZ), nsw, rep_max, int(maxitfac), C.c_longlong(max_rounds),
                      eig.ctypes.data_as(dp), C.byref(info), stats)
    names = ["sweeps", "rounds", "windows", "shift_pairs", "exceptional", "final_blocks", "bulge_steps", "status",
             "bulges_left_behind", "held_windows"]
    return T, Zo, eig[:, 0] + 1j * eig[:, 1], info.value, dict(zip(names, list(stats)))
