"""periodicschurdecompositions.jl_b200 — host-side mirror of the dense `pschur!` interface of
RalphAS/PeriodicSchurDecompositions.jl on top of the sm_100a C-ABI library libpsd_b200.so.

The reference's host language is Julia (julia/PeriodicSchurB200.jl holds the ccall glue a
maintainer drops into the package); Julia is not available in this image, so this Python
module mirrors the same operator interface (names, argument meaning, result structs, error
behaviour) over the identical C ABI so that the parity tests read like the reference's tests.

Import name: the directory contains a dot, so it is loaded through the `psd_b200` shim at the
repository root (`import psd_b200`).

There is NO CPU fallback: every compute entry point raises if libpsd_b200.so is missing or no
B200 is visible.
"""
from __future__ import annotations

from .capi import (  # noqa: F401
    PsdError,
    device_count,
    lib,
    lib_path,
    library_available,
    version,
)
from .pschur import (  # noqa: F401
    PeriodicSchur,
    GeneralizedPeriodicSchur,
    Handle,
    gpschur,
    gpschur_,
    gpschur_batched,
    gphessenberg_batched,
    gvalues,
    default_handle,
    phessenberg_batched,
    rphessenberg_rowwise_batched,
    pschur,
    pschur_,
    pschur_batched,
    pschur_hessut_batched,
    checkpsd_batched,
    eigvecs,
    eigvecs_batched,
    phessenberg_packed_batched,
    shard_bounds,
)

__all__ = [
    "PsdError", "device_count", "lib", "lib_path", "library_available", "version",
    "PeriodicSchur", "GeneralizedPeriodicSchur", "gpschur", "gpschur_", "gpschur_batched", "gphessenberg_batched", "gvalues", "Handle", "default_handle", "phessenberg_batched", "rphessenberg_rowwise_batched", "pschur", "pschur_",
    "pschur_batched", "pschur_hessut_batched", "checkpsd_batched", "eigvecs", "eigvecs_batched", "phessenberg_packed_batched", "shard_bounds",
]
