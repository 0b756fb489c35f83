# PeriodicSchurB200.jl — Julia glue between PeriodicSchurDecompositions.jl and libpsd_b200.so.
#
# Drop this file next to the reference package (or `include` it after `using
# PeriodicSchurDecompositions`): it adds methods of `pschur!` for the concrete BLAS element types
# that are MORE SPECIFIC than the reference's generic methods
#   pschur!(A::AbstractVector{<:AbstractMatrix{T}}, lr)            PeriodicSchurDecompositions.jl:120
#   pschur!(A, S, lr) where T<:Complex                             generalized.jl:108
#   pschur!(A, S, lr) where T<:Real                                rgeneralized.jl:3
#   pschur!(A::Vector{<:Matrix{<:Complex}}, lr)                    PeriodicSchurDecompositions.jl:1106
# so dispatch prefers them, packs the factors into one contiguous (n,n,p,batch) array (which IS
# the device layout), calls the C ABI of include/psd_b200.h with `ccall`, copies the results back
# into the caller's matrices (T1 aliases A[1] / A[p] exactly as in the reference, :265,
# :1078-1093) and builds the reference's own result structs.  `ordschur!`, `eigvecs`,
# `partial_pschur` keep running as the reference code on those structs.
#
# There is no CPU fallback: if the library cannot be loaded or no B200 is visible these methods
# throw.  NOTE: written without a Julia runtime at hand (none exists in the build image); the
# same ABI is exercised end to end by the Python mirror in ../pschur.py and the tests.
module PeriodicSchurB200

using LinearAlgebra
using PeriodicSchurDecompositions
using PeriodicSchurDecompositions: PeriodicSchur, GeneralizedPeriodicSchur
import PeriodicSchurDecompositions: pschur!

const libpsd = get(ENV, "PSD_B200_LIB", joinpath(@__DIR__, "..", "libpsd_b200.so"))

const PSD_ERR_SIGNATURE = -4

mutable struct Handle
    ptr::Ptr{Cvoid}
    function Handle(devices::Vector{Cint} = Cint[])
        r = Ref{Ptr{Cvoid}}(C_NULL)
        rc = ccall((:psd_create, libpsd), Cint, (Ref{Ptr{Cvoid}}, Cint, Ptr{Cint}),
                   r, length(devices), isempty(devices) ? C_NULL : pointer(devices))
        rc == 0 || error(lasterror(rc))
        h = new(r[])
        finalizer(x -> ccall((:psd_destroy, libpsd), Cint, (Ptr{Cvoid},), x.ptr), h)
        h
    end
end

lasterror(rc) = "psd_b200 error $rc: " *
                unsafe_string(ccall((:psd_last_error_string, libpsd), Cstring, ()))

const _default = Ref{Union{Nothing, Handle}}(nothing)
default_handle() = (_default[] === nothing && (_default[] = Handle()); _default[]::Handle)

orient_code(lr::Symbol) = lr === :R ? Cint(0) : lr === :L ? Cint(1) :
    throw(ArgumentError("orientation argument must be either :R (right) or :L (left)"))

function _pack(A::Vector{Matrix{T}}) where {T}
    p = length(A)
    n = LinearAlgebra.checksquare(A[1])
    for j in 2:p
        LinearAlgebra.checksquare(A[j]) == n || throw(DimensionMismatch())
    end
    buf = Array{T, 3}(undef, n, n, p)
    for j in 1:p
        copyto!(view(buf, :, :, j), A[j])
    end
    return buf, n, p
end

_unpack!(A, buf) = (for j in eachindex(A); copyto!(A[j], view(buf, :, :, j)); end; A)

function _split(A, lr)
    p = length(A)
    lr === :R ? (A[1], [A[j] for j in 2:p], 1) : (A[p], [A[j] for j in 1:(p - 1)], p)
end

# ---- real standard: PeriodicSchurDecompositions.jl:120-152 -------------------------------------
function pschur!(A::Vector{Matrix{Float64}}, lr::Symbol = :R; wantZ::Bool = true,
                 wantT::Bool = true, maxitfac = 30, handle::Handle = default_handle())
    o = orient_code(lr)
    buf, n, p = _pack(A)
    Z = wantZ ? Array{Float64, 3}(undef, n, n, p) : Array{Float64, 3}(undef, 0, 0, 0)
    vals = Vector{ComplexF64}(undef, n)
    info = Ref{Int32}(0)
    rc = ccall((:psd_rpschur_batched, libpsd), Cint,
               (Ptr{Cvoid}, Cint, Cint, Int64, Cint, Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64},
                Ptr{ComplexF64}, Ref{Int32}),
               handle.ptr, n, p, 1, o, wantT, wantZ, maxitfac, buf, wantZ ? Z : C_NULL, vals, info)
    rc == 0 || error(lasterror(rc))
    info[] == 0 || throw(ErrorException("convergence failed at level $(info[])"))
    wantT && _unpack!(A, buf)
    T1, Ts, sidx = _split(A, lr)
    Zs = wantZ ? [Z[:, :, j] for j in 1:p] : [Matrix{Float64}(undef, 0, 0)]
    return PeriodicSchur(T1, Ts, Zs, vals, lr === :R ? 'R' : 'L', sidx)
end

# ---- generalized: generalized.jl:108-148 (complex), rgeneralized.jl:3-45 (real) ---------------
for (T, Tb, fn) in ((ComplexF64, ComplexF64, :psd_cpschur_batched),
                    (Float64, Float64, :psd_rgpschur_batched))
    @eval function pschur!(A::Vector{Matrix{$T}}, S::AbstractVector{Bool}, lr::Symbol = :R;
                           wantZ::Bool = true, wantT::Bool = true, aggressive::Bool = false,
                           handle::Handle = default_handle())
        aggressive && throw(ArgumentError("aggressive deflation is not offered by the B200 path"))
        o = orient_code(lr)
        buf, n, p = _pack(A)
        length(S) == p || throw(DimensionMismatch("S must have one entry per factor"))
        Sb = UInt8.(S)
        Z = wantZ ? Array{$T, 3}(undef, n, n, p) : Array{$T, 3}(undef, 0, 0, 0)
        α = Vector{ComplexF64}(undef, n)
        β = Vector{$Tb}(undef, n)
        αscale = Vector{Int64}(undef, n)
        info = Ref{Int32}(0)
        rc = ccall(($(QuoteNode(fn)), libpsd), Cint,
                   (Ptr{Cvoid}, Cint, Cint, Int64, Cint, Ptr{UInt8}, Cint, Cint, Cint, Ptr{$T},
                    Ptr{$T}, Ptr{ComplexF64}, Ptr{$Tb}, Ptr{Int64}, Ref{Int32}),
                   handle.ptr, n, p, 1, o, Sb, wantT, wantZ, 0, buf, wantZ ? Z : C_NULL, α, β,
                   αscale, info)
        rc == PSD_ERR_SIGNATURE && throw(ArgumentError("The leftmost entry in S must be true"))
        rc == 0 || error(lasterror(rc))
        info[] == 0 || throw(ErrorException("convergence failed at level $(info[])"))
        wantT && _unpack!(A, buf)
        T1, Ts, sidx = _split(A, lr)
        Zs = wantZ ? [Z[:, :, j] for j in 1:p] : Vector{Matrix{$T}}(undef, 0)
        return GeneralizedPeriodicSchur(collect(Bool, S), sidx, T1, Ts, Zs, α, β,
                                        Vector{Int}(αscale), lr === :R ? 'R' : 'L')
    end
end

# ---- complex standard: PeriodicSchurDecompositions.jl:1106-1111 --------------------------------
function pschur!(A::Vector{Matrix{ComplexF64}}, lr::Symbol = :R; kwargs...)
    F = pschur!(A, trues(length(A)), lr; kwargs...)
    return PeriodicSchur(F.T1, F.T, F.Z, F.values, F.orientation, F.schurindex)
end

# ---- batched entry points (new; the reference has none) ----------------------------------------
"""
    pschur_batched!(A::Array{Float64,4}, lr=:R; wantZ, wantT, maxitfac) -> (Z, values, info)

`A` is (n, n, p, batch): the device layout.  `A` is overwritten with the T factors in the user's
factor order; `values` is n x batch; `info[b] > 0` marks a problem that did not converge.
"""
function pschur_batched!(A::Array{Float64, 4}, lr::Symbol = :R; wantZ::Bool = true,
                         wantT::Bool = true, maxitfac = 30, handle::Handle = default_handle())
    n, n2, p, B = size(A)
    n == n2 || throw(DimensionMismatch())
    Z = wantZ ? similar(A) : Array{Float64, 4}(undef, 0, 0, 0, 0)
    vals = Matrix{ComplexF64}(undef, n, B)
    info = Vector{Int32}(undef, B)
    rc = ccall((:psd_rpschur_batched, libpsd), Cint,
               (Ptr{Cvoid}, Cint, Cint, Int64, Cint, Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64},
                Ptr{ComplexF64}, Ptr{Int32}),
               handle.ptr, n, p, B, orient_code(lr), wantT, wantZ, maxitfac, A,
               wantZ ? Z : C_NULL, vals, info)
    rc == 0 || error(lasterror(rc))
    return Z, vals, info
end

"""
    gpschur_batched!(A::Array{T,4}, S, lr=:R; wantZ, wantT) -> (Z, α, β, αscale, info)

Batched generalized periodic Schur decomposition, `T` = `Float64` or `ComplexF64`.
"""
function gpschur_batched!(A::Array{T, 4}, S::AbstractVector{Bool}, lr::Symbol = :R;
                          wantZ::Bool = true, wantT::Bool = true,
                          handle::Handle = default_handle()) where {T <: Union{Float64, ComplexF64}}
    n, n2, p, B = size(A)
    n == n2 || throw(DimensionMismatch())
    Z = wantZ ? similar(A) : Array{T, 4}(undef, 0, 0, 0, 0)
    α = Matrix{ComplexF64}(undef, n, B)
    β = Matrix{T}(undef, n, B)
    αscale = Matrix{Int64}(undef, n, B)
    info = Vector{Int32}(undef, B)
    Sb = UInt8.(S)
    fn = T <: Complex ? :psd_cpschur_batched : :psd_rgpschur_batched
    rc = if T <: Complex
        ccall((:psd_cpschur_batched, libpsd), Cint,
              (Ptr{Cvoid}, Cint, Cint, Int64, Cint, Ptr{UInt8}, Cint, Cint, Cint, Ptr{T}, Ptr{T},
               Ptr{ComplexF64}, Ptr{T}, Ptr{Int64}, Ptr{Int32}),
              handle.ptr, n, p, B, orient_code(lr), Sb, wantT, wantZ, 0, A, wantZ ? Z : C_NULL, α,
              β, αscale, info)
    else
        ccall((:psd_rgpschur_batched, libpsd), Cint,
              (Ptr{Cvoid}, Cint, Cint, Int64, Cint, Ptr{UInt8}, Cint, Cint, Cint, Ptr{T}, Ptr{T},
               Ptr{ComplexF64}, Ptr{T}, Ptr{Int64}, Ptr{Int32}),
              handle.ptr, n, p, B, orient_code(lr), Sb, wantT, wantZ, 0, A, wantZ ? Z : C_NULL, α,
              β, αscale, info)
    end
    rc == PSD_ERR_SIGNATURE && throw(ArgumentError("The leftmost entry in S must be true"))
    rc == 0 || error(lasterror(rc))
    return Z, α, β, αscale, info
end

"""
    pschur_hessut_batched!(H::Array{Float64,4}; Q = nothing, wantT = true, maxitfac = 30)
        -> (Z, values, info)

Inner method of the reference on Hessenberg-triangular input (`pschur!(H1, Hs; Q, wantZ, wantT)`,
PeriodicSchurDecompositions.jl:322), batched, rightwards order.  With `Q` (same shape as `H`) the
Schur vectors are accumulated onto it, as the `Q` keyword of the reference does (:326, 432-437;
used by the Krylov-Schur driver, krylov.jl:583-591); `Q` is overwritten and returned.
"""
function pschur_hessut_batched!(H::Array{Float64, 4}; Q::Union{Nothing, Array{Float64, 4}} = nothing,
                                wantT::Bool = true, maxitfac = 30, handle::Handle = default_handle())
    n, n2, p, B = size(H)
    n == n2 || throw(DimensionMismatch())
    vals = Matrix{ComplexF64}(undef, n, B)
    info = Vector{Int32}(undef, B)
    if Q === nothing
        Z = similar(H)
        rc = ccall((:psd_rpschur_hessut_batched, libpsd), Cint,
                   (Ptr{Cvoid}, Cint, Cint, Int64, Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64},
                    Ptr{ComplexF64}, Ptr{Int32}),
                   handle.ptr, n, p, B, wantT, true, maxitfac, H, Z, vals, info)
    else
        size(Q) == size(H) || throw(DimensionMismatch("Q must have the shape of H"))
        Z = Q
        rc = ccall((:psd_rpschur_hessut_q_batched, libpsd), Cint,
                   (Ptr{Cvoid}, Cint, Cint, Int64, Cint, Cint, Ptr{Float64}, Ptr{Float64},
                    Ptr{ComplexF64}, Ptr{Int32}),
                   handle.ptr, n, p, B, wantT, maxitfac, H, Z, vals, info)
    end
    rc == 0 || error(lasterror(rc))
    return Z, vals, info
end

"""
    large_stats(handle) -> NamedTuple

Report of the last large-N (N >= 192) real decomposition on `handle`: status (0 = the multishift
iteration finished), shift sets, rounds, window-rounds, shift pairs, exceptional sets, final blocks,
kernel launches - the counterpart of the `niter` report of the reference (:458-459, 1077).
"""
function large_stats(handle::Handle = default_handle())
    out = Vector{Float64}(undef, 16)
    rc = ccall((:psd_large_stats, libpsd), Cint, (Ptr{Cvoid}, Ptr{Float64}), handle.ptr, out)
    rc == 0 || error(lasterror(rc))
    return (status = Int(out[1]), sets = Int(out[2]), rounds = Int(out[3]), windows = Int(out[4]),
            shift_pairs = Int(out[5]), exceptional = Int(out[6]), final_blocks = Int(out[7]),
            launches = Int(out[8]), update_flops = out[9])
end

"""
    checkpsd_batched(A, T, Z, lr = :R; thresh = 100, strict = true) -> (ok, err)

`checkpsd` (diagnostics.jl:190-263) for batched real results in the device layout (n, n, p, batch):
the normalized factorization errors, the triangularity and the orthogonality norms are formed on
the GPU; `ok[b]` applies the reference's thresholds.
"""
function checkpsd_batched(A::Array{Float64, 4}, T::Array{Float64, 4}, Z::Array{Float64, 4},
                          lr::Symbol = :R; thresh = 100, strict::Bool = true,
                          handle::Handle = default_handle())
    n, n2, p, B = size(A)
    (n == n2 && size(T) == size(A) && size(Z) == size(A)) || throw(DimensionMismatch())
    err = Matrix{Float64}(undef, p, B); tri = similar(err); orth = similar(err)
    rc = ccall((:psd_rcheckpsd_batched, libpsd), Cint,
               (Ptr{Cvoid}, Cint, Cint, Int64, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
               handle.ptr, n, p, B, orient_code(lr), A, T, Z, err, tri, orth)
    rc == 0 || error(lasterror(rc))
    cmp = strict ? 0.0 : 10 * eps(Float64) * n
    ok = [all(tri[:, b] .<= cmp) && all(orth[:, b] .<= 10 * eps(Float64) * n) && all(err[:, b] .<= thresh)
          for b in 1:B]
    return ok, err
end

"""
    phessenberg!(A::Vector{Matrix{Float64}}) -> (H1::Hessenberg, pH::Vector{<:QR})

Drop-in for the reference's `phessenberg!` (PeriodicSchurDecompositions.jl:213-259): the reduction
runs on the GPU and comes back in the reference's own packed form (reflector vectors below the
(sub)diagonal, `tau`), from which the same `Hessenberg` / `QR` objects are built (:249-253).
"""
function phessenberg!(A::Vector{Matrix{Float64}}; handle::Handle = default_handle())
    buf, n, p = _pack(A)
    tau = Matrix{Float64}(undef, n, p)
    rc = ccall((:psd_rphess_packed_batched, libpsd), Cint,
               (Ptr{Cvoid}, Cint, Cint, Int64, Ptr{Float64}, Ptr{Float64}),
               handle.ptr, n, p, 1, buf, tau)
    rc == 0 || error(lasterror(rc))
    _unpack!(A, buf)
    H1 = LinearAlgebra.Hessenberg(A[1], tau[1:(n - 1), 1])
    pH = [LinearAlgebra.QR(A[j], tau[:, j]) for j in 2:p]
    return H1, pH
end

# ---- eigenvectors of PeriodicSchur results (psd_reigvecs_batched / psd_ceigvecs_batched) -------
"""
    eigvecs_batched(T, Z, lr = :R; select = nothing, handle) -> (V, info)

Eigenvectors of `batch` periodic Schur results at once, by periodic back-substitution on the Schur
form.  `T` and `Z` are `(n, n, p, batch)` arrays of `Float64` or `ComplexF64` in user factor order
(the layout `pschur!` packs for the device); `select` an `(n, batch)` `Bool` array or `nothing`
for every eigenvalue.  `V[:, k, l, b]` is the unit vector `v_l` of eigenvalue `k` of problem `b`
(`:R`: `A_l v_{l+1} = mu_l v_l`, `:L`: `A_l v_l = mu_l v_{l+1}`, `prod(mu) = values[k]`), with its
entry of largest modulus real and positive; unselected columns are zero and a complex pair is
filled whole when either member is selected.  `info[b] == 1`: `T` of problem `b` is not in periodic
Schur form.

This is deliberately the module's own function and not a method of `LinearAlgebra.eigvecs` for the
reference's structs: the reference computes its vectors by reordering with `ordschur!`, and the
normalisation and layout of its return value cannot be confirmed here.  Like the rest of this file
the glue has not been executed; the same ABI is exercised by the Python mirror (`../pschur.py`).
"""
function eigvecs_batched(T::Array{E, 4}, Z::Array{E, 4}, lr::Symbol = :R;
                         select::Union{Nothing, AbstractMatrix{Bool}} = nothing,
                         handle::Handle = default_handle()) where {E <: Union{Float64, ComplexF64}}
    o = orient_code(lr)
    n, n2, p, batch = size(T)
    (n == n2 && size(Z) == size(T)) || throw(DimensionMismatch("T and Z must be (n, n, p, batch)"))
    sel = select === nothing ? C_NULL : convert(Array{UInt8}, select)
    select === nothing || size(select) == (n, batch) || throw(DimensionMismatch("select must be (n, batch)"))
    V = zeros(ComplexF64, n, n, p, batch)
    info = zeros(Int32, batch)
    rc = GC.@preserve sel begin
        if E === Float64
            ccall((:psd_reigvecs_batched, libpsd), Cint,
                  (Ptr{Cvoid}, Cint, Cint, Int64, Cint, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{UInt8},
                   Ptr{ComplexF64}, Ptr{Int32}),
                  handle.ptr, n, p, batch, o, T, Z, sel, V, info)
        else
            ccall((:psd_ceigvecs_batched, libpsd), Cint,
                  (Ptr{Cvoid}, Cint, Cint, Int64, Cint, Ptr{ComplexF64}, Ptr{ComplexF64}, Ptr{UInt8},
                   Ptr{ComplexF64}, Ptr{Int32}),
                  handle.ptr, n, p, batch, o, T, Z, sel, V, info)
        end
    end
    rc == 0 || error(lasterror(rc))
    return V, info
end

end # module
