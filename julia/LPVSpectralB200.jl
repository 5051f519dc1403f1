# LPVSpectralB200.jl -- drop-in Julia shim over liblpvs.so (include/lpvs.h).
#
# Same names / signatures / kwargs as LPVSpectral.jl's least-squares estimators
# (src/lsfft.jl:62-80,112-126,140-156,176-193,239-259; src/lasso.jl:27-126), but every flop runs in the
# sm_100a CUDA library.  The shim only marshals: collect ranges into Vector{Float64}, validate exactly where the
# reference validates, evaluate window_func on the host, map proxg objects to (kind, param), allocate outputs,
# `ccall`, and wrap results.  There is NO CPU fallback: unsupported `estimator`/`proxg` throw ArgumentError.
#
# NOTE: Julia is not installed in the build image or on the GPU box, so this file is syntax-reviewed only; the
# identical C ABI is exercised end to end from Python ctypes (lpvspectral.jl_b200/_api.py mirrors this file line
# for line) by tests/ and bench.py.
module LPVSpectralB200

using LinearAlgebra, Statistics, Printf
import LPVSpectral: SpectralExt, default_freqs, check_freq   # host-side pieces stay untouched Julia
import DSP: rect, hanning

export ls_spectral, tls_spectral, ls_windowpsd, ls_windowcsd, ls_cohere, ls_sparse_spectral, ls_spectral_lpv,
       ls_sparse_spectral_lpv, ls_windowpsd_lpv, mapwindows_b200, ls_windowpsd_multi, ls_windowcsd_matrix, ls_cohere_matrix,
       ls_sparse_windowpsd_multi, ls_sparse_windowcsd_matrix, ls_sparse_cohere_matrix, ls_spectral_multi

const liblpvs = get(ENV, "LIBLPVS", "liblpvs")
const WIN_PSD, WIN_CSD, WIN_COHERE = Cint(0), Cint(1), Cint(2)
const PROX_L1, PROX_L0, PROX_BALL_L0 = Cint(0), Cint(1), Cint(2)

mutable struct Ctx
    h::Ptr{Cvoid}
end
const CTX = Ref{Union{Nothing,Ctx}}(nothing)

function ctx()
    if CTX[] === nothing
        h = Ref{Ptr{Cvoid}}(C_NULL)
        dev = parse(Int, get(ENV, "LOCAL_RANK", "0"))
        rc = ccall((:lpvs_init, liblpvs), Cint, (Cint, Ptr{Ptr{Cvoid}}), dev, h)
        rc == 0 || error("lpvs_init failed ($rc): no usable B200 (there is no CPU fallback)")
        c = Ctx(h[])
        finalizer(c -> ccall((:lpvs_destroy, liblpvs), Cvoid, (Ptr{Cvoid},), c.h), c)
        CTX[] = c
    end
    CTX[].h
end

lasterr() = unsafe_string(ccall((:lpvs_last_error, liblpvs), Cstring, (Ptr{Cvoid},), ctx()))
function check(rc)
    rc == 0 && return
    msg = lasterr()
    rc == -1 && throw(ArgumentError(msg))
    rc == -2 && throw(PosDefException(1))
    error("liblpvs error $rc: $msg")
end

# LPVS_OPT_ADMM_M32 (include/lpvs.h): ADMM problems created while set keep their inverse in single precision.  The Float32
# instantiations of the sparse estimators switch it on around the create call.
const OPT_ADMM_M32 = Cint(7)
setopt(key, v) = check(ccall((:lpvs_set_option, liblpvs), Cint, (Ptr{Cvoid}, Cint, Float64), ctx(), key, Float64(v)))
# LPVS_OPT_PHASE_MODE (include/lpvs.h, enum lpvs_phase_mode): how the Fourier basis / its Gram matrix is formed.  The default
# (:auto) reproduces the reference's phase rounding fl(fl(2 pi f) t) (src/lsfft.jl:34,41); :structured_ref gives the same
# results from the trigonometric-sum Gram matrix + a half-precision tensor-core correction, 2.6x faster on uniform grids.
const OPT_PHASE_MODE = Cint(0)
const PHASE_MODES = (auto = 0, chain = 1, direct = 2, chain_ref = 3, structured = 4, structured_ref = 5)
"phase_mode!(:auto | :chain | :direct | :chain_ref | :structured | :structured_ref) -- applies to every later call."
phase_mode!(mode::Symbol) = setopt(OPT_PHASE_MODE, getproperty(PHASE_MODES, mode))
"Give the context's grow-only device workspaces back (re-allocated on demand by the next call)."
release_workspace() = check(ccall((:lpvs_release_workspace, liblpvs), Cint, (Ptr{Cvoid},), ctx()))
function with_m32(fn, T)
    T === Float32 || return fn()
    setopt(OPT_ADMM_M32, 1)
    try
        return fn()
    finally
        setopt(OPT_ADMM_M32, 0)
    end
end

vecf(x) = collect(Float64, x)
nullable(x) = x === nothing ? Ptr{Float64}(C_NULL) : pointer(x)
# Float32 instantiation of the generic signatures (e.g. src/lasso.jl:85 `AbstractArray{T}`): results carry the signal's
# eltype.  The device arithmetic is the FP64 path on the up-converted inputs (there are no FP32 kernels), so a Float32
# caller gets the correctly rounded-to-single FP64 answer.
like(y, x::AbstractArray{<:Complex}) = eltype(y) === Float32 ? ComplexF32.(x) : x
like(y, x::AbstractArray{<:Real}) = eltype(y) === Float32 ? Float32.(x) : x
like(y, x) = x

# ---- ls_spectral (src/lsfft.jl:62-80) ---------------------------------------------------------------------
function ls_spectral(y, t, f=default_freqs(t); λ=1e-10, verbose=false)
    _ls_spectral(y, t, f, nothing, λ)
end
function ls_spectral(y, t, f, W::AbstractVector; λ=1e-10, verbose=false)
    _ls_spectral(y, t, f, W, λ)
end
function _ls_spectral(y, t, f, W, λ)
    check_freq(f)                                    # ArgumentError site, src/lsfft.jl:22
    yv, tv, fv = vecf(y), vecf(t), vecf(f)
    length(yv) == length(tv) || throw(ArgumentError("y and t has to be the same length"))
    Wv = W === nothing ? nothing : vecf(W)
    x = Vector{ComplexF64}(undef, length(fv))
    info = Ref{Cint}(0)
    GC.@preserve yv tv fv Wv x begin
        check(ccall((:lpvs_ls_spectral, liblpvs), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}, Cint, Ptr{Float64}, Float64,
             Ptr{ComplexF64}, Ptr{Cint}),
            ctx(), yv, tv, length(yv), fv, length(fv), nullable(Wv), Float64(λ), x, info))
    end
    # info 1: a WEIGHTED problem was numerically singular and re-factorised with a jitter ridge (the reference's LU returns
    # something there too); info 2 (informational): the unweighted solve took the QR-class path of csrc/lsq.cu
    info[] == 1 && @warn "weighted Gram matrix numerically singular: solved with a jitter ridge (DESIGN.md section 1)"
    like(y, x), f                                    # the caller's own f object, untouched
end

# ---- ls_spectral of every column of Y (N x C) at the shared t: one Gram matrix and one factor for all channels ----------
# (no reference equivalent; column c is ls_spectral(Y[:,c], t, f[, W]; λ)).  Returns (X::Matrix{ComplexF64} Nf x C, f).
function ls_spectral_multi(Y::AbstractMatrix, t, f=default_freqs(t); λ=1e-10)
    _ls_spectral_multi(Y, t, f, nothing, λ)
end
function ls_spectral_multi(Y::AbstractMatrix, t, f, W::AbstractVector; λ=1e-10)
    _ls_spectral_multi(Y, t, f, W, λ)
end
function _ls_spectral_multi(Y, t, f, W, λ)
    check_freq(f)
    Yv, tv, fv = Matrix{Float64}(Y), vecf(t), vecf(f)    # column-major: channel c at c*N
    N, C = size(Yv)
    C >= 1 || throw(ArgumentError("Y must have at least one column"))
    N == length(tv) || throw(ArgumentError("Y and t has to be the same length"))
    Wv = W === nothing ? nothing : vecf(W)
    Wv === nothing || length(Wv) == N || throw(ArgumentError("W and Y has to be the same length"))
    X = Matrix{ComplexF64}(undef, length(fv), C)
    info = zeros(Cint, C)
    GC.@preserve Yv tv fv Wv X info begin
        check(ccall((:lpvs_ls_spectral_multi, liblpvs), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Cint, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Cint, Ptr{Float64}, Float64,
             Ptr{ComplexF64}, Ptr{Cint}),
            ctx(), Yv, C, N, tv, N, fv, length(fv), nullable(Wv), Float64(λ), X, info))
    end
    any(==(1), info) && @warn "weighted Gram matrix numerically singular: solved with a jitter ridge (DESIGN.md section 1)"
    X, f
end

# ---- tls_spectral (src/lsfft.jl:87-99) ---------------------------------------------------------------------
function tls_spectral(y, t, f=default_freqs(t)[1:end-1])
    check_freq(f)
    yv, tv, fv = vecf(y), vecf(t), vecf(f)
    length(yv) == length(tv) || throw(ArgumentError("y and t has to be the same length"))
    x = Vector{ComplexF64}(undef, length(fv))
    its = Ref{Cint}(0)
    GC.@preserve yv tv fv x begin
        check(ccall((:lpvs_tls_spectral, liblpvs), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}, Cint, Ptr{ComplexF64}, Ptr{Cint}),
            ctx(), yv, tv, length(yv), fv, length(fv), x, its))
    end
    like(y, x), f
end

# ---- mapwindows / merge (src/windows.jl:50-70): the closure runs on the host as in the reference, the overlap-average
# re-assembly on the device ------------------------------------------------------------------------------------
function mapwindows_b200(fn::Function, y, t, n::Integer, noverlap::Integer=-1)
    yv, tv = vecf(y), vecf(t)
    length(yv) == length(tv) || throw(AssertionError("y and t has to be the same length"))   # src/windows.jl:31
    noverlap < 0 && (noverlap = n >> 1)
    noverlap < n || throw(ArgumentError("noverlap must be smaller than the window length n"))
    hop = n - noverlap
    K = length(yv) >= n ? (length(yv) - n) ÷ hop + 1 : 0
    pieces = Matrix{Float64}(undef, n, K)             # column k = window k: K x n row-major for the C side
    for k in 0:K-1
        r = k*hop+1:k*hop+n
        pieces[:, k+1] = fn(yv[r], tv[r])
    end
    out = Vector{Float64}(undef, length(yv))
    GC.@preserve pieces out begin
        check(ccall((:lpvs_merge_windows, liblpvs), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Int64, Cint, Cint, Int64, Ptr{Float64}),
            ctx(), pieces, K, n, noverlap, length(yv), out))
    end
    like(y, out)
end

# ---- windowed estimators (src/lsfft.jl:112-193) -----------------------------------------------------------
function _windowed(kind, y, u, t, freqs, nw, noverlap, window_func, estimator, kwargs)
    n = length(y) ÷ nw                               # src/lsfft.jl:113
    freqs === nothing && (freqs = default_freqs(t, n))
    check_freq(freqs)
    estimator === ls_spectral ||
        return _windowed_generic(kind, y, u, t, freqs, n, noverlap, window_func, estimator, kwargs)
    λ = get(kwargs, :λ, 1e-10)
    yv, tv, fv = vecf(y), vecf(t), vecf(freqs)
    uv = u === nothing ? nothing : vecf(u)
    length(yv) == length(tv) || throw(AssertionError("y and t has to be the same length"))  # src/windows.jl:31
    noverlap < 0 && (noverlap = n >> 1)
    noverlap < n || throw(ArgumentError("noverlap must be smaller than the window length n"))  # DSP.arraysplit
    Wv = vecf(window_func(n))
    length(Wv) == n || throw(DimensionMismatch("window_func(n) must return n = $n weights, got $(length(Wv))"))
    out = kind == WIN_CSD ? Vector{ComplexF64}(undef, length(fv)) : Vector{Float64}(undef, length(fv))
    K = Ref{Int64}(0); info = Ref{Cint}(0)
    GC.@preserve yv uv tv fv Wv out begin
        check(ccall((:lpvs_ls_window, liblpvs), Cint,
            (Ptr{Cvoid}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}, Cint, Ptr{Float64},
             Cint, Cint, Float64, Ptr{Cvoid}, Ptr{Int64}, Ptr{Cint}),
            ctx(), kind, yv, nullable(uv), tv, length(yv), fv, length(fv), Wv, n, noverlap, Float64(λ), out, K, info))
    end
    like(y, out), freqs
end

# estimator = ls_sparse_spectral (test/test_lasso.jl:36).  Without init / callback / periodic prints all windows run
# in ONE device pass (lpvs_ls_window_sparse_sums: batched Gram, Cholesky and inverse, one CTA per window iterates to
# its own stop test); otherwise one device ADMM solve per window through the single-problem entry point.
function _windowed_generic(kind, y, u, t, freqs, n, noverlap, window_func, estimator, kwargs)
    estimator === ls_sparse_spectral ||
        throw(ArgumentError("estimator must be ls_spectral or ls_sparse_spectral (no CPU fallback)"))
    noverlap < 0 && (noverlap = n >> 1)
    noverlap < n || throw(ArgumentError("noverlap must be smaller than the window length n"))  # DSP.arraysplit
    W = vecf(window_func(n)); hop = n - noverlap
    length(W) == n || throw(DimensionMismatch("window_func(n) must return n = $n weights, got $(length(W))"))
    # K == 0 (signal shorter than one window): empty sums divided by K^2 / K give NaN spectra, as in the reference
    K = length(y) >= n ? (length(y) - n) ÷ hop + 1 : 0
    kw = Dict{Symbol,Any}(kwargs)
    iters = get(kw, :iters, 10000); tol = get(kw, :tol, 1e-5); printerval = get(kw, :printerval, 100)
    if !get(kw, :init, false) && get(kw, :cb, nothing) === nothing && printerval >= iters
        λ = get(kw, :λ, 1.0); μ = get(kw, :μ, 0.05)
        0 ≤ μ ≤ 1 || throw(AssertionError("μ should be ≤ 1"))                   # src/lasso.jl:143
        pg = get(kw, :proxg, nothing)
        pk, pp = pg === nothing ? (PROX_L1, Float64(λ)) : proxdesc(pg)                 # Q15
        yv, tv, fv = vecf(y), vecf(t), vecf(freqs)
        uv = u === nothing ? nothing : vecf(u)
        nrhs = kind == WIN_PSD ? 1 : 2
        sums = zeros((kind == WIN_PSD ? 1 : kind == WIN_CSD ? 2 : 4) * length(fv))
        its = zeros(Int64, max(K, 1) * nrhs); res = zeros(max(K, 1) * nrhs); info = Ref{Cint}(0)
        GC.@preserve yv uv tv fv W sums its res begin
            K > 0 && check(ccall((:lpvs_ls_window_sparse_sums, liblpvs), Cint,
                (Ptr{Cvoid}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}, Cint, Ptr{Float64},
                 Cint, Cint, Cint, Float64, Float64, Int64, Float64, Int64, Int64, Ptr{Float64}, Ptr{Int64},
                 Ptr{Float64}, Ptr{Cint}),
                ctx(), kind, yv, nullable(uv), tv, length(yv), fv, length(fv), W, n, noverlap, pk, Float64(pp),
                Float64(μ), iters, Float64(tol), 0, K, sums, its, res, info))
        end
        for k in 1:K*nrhs                       # the line the reference prints when a window stops (src/lasso.jl:164)
            res[k] < tol && @printf("%d ||x-z||₂ %.10f\n", its[k], res[k])
        end
        out = kind == WIN_CSD ? Vector{ComplexF64}(undef, length(fv)) : Vector{Float64}(undef, length(fv))
        check(ccall((:lpvs_ls_window_finalize, liblpvs), Cint, (Cint, Ptr{Float64}, Cint, Int64, Ptr{Cvoid}),
                    kind, sums, length(fv), K, out))
        return like(y, out), freqs
    end
    Syy = zeros(length(freqs)); Suu = zeros(length(freqs)); Syu = zeros(ComplexF64, length(freqs))
    for k in 0:K-1
        r = k*hop+1:k*hop+n
        xy = estimator(y[r], t[r], freqs, W; kwargs...)[1]
        Syy .+= abs2.(xy)
        if u !== nothing
            xu = estimator(u[r], t[r], freqs, W; kwargs...)[1]
            Suu .+= abs2.(xu); Syu .+= xy .* conj.(xu)
        end
    end
    kind == WIN_PSD && return Syy ./ K^2, freqs
    kind == WIN_CSD && return Syu ./ K, freqs
    abs2.(Syu) ./ (Suu .* Syy), freqs
end

ls_windowpsd(y, t, freqs=nothing; nw=8, noverlap=-1, window_func=rect, estimator=ls_spectral, kwargs...) =
    _windowed(WIN_PSD, y, nothing, t, freqs, nw, noverlap, window_func, estimator, kwargs)
ls_windowcsd(y, u, t, freqs=nothing; nw=10, noverlap=-1, window_func=rect, estimator=ls_spectral, kwargs...) =
    _windowed(WIN_CSD, y, u, t, freqs, nw, noverlap, window_func, estimator, kwargs)
ls_cohere(y, u, t, freqs=nothing; nw=10, noverlap=-1, estimator=ls_spectral, kwargs...) =
    _windowed(WIN_COHERE, y, u, t, freqs, nw, noverlap, hanning, estimator, kwargs)   # hanning hard-coded (:182)

# ---- many channels of one record (the columns of Y, shared t): no reference equivalent.  Per window ONE Gram matrix and
# ONE factor for all channels; entry [f, i, j] equals ls_windowcsd(Y[:, i], Y[:, j], t, ...) / ls_cohere(...), column c of
# the PSD ls_windowpsd(Y[:, c], t, ...).  New names: the reference's own names keep their vector methods only.
# `sparse = (proxg, μ, iters, tol)`: estimator = ls_sparse_spectral per channel (lpvs_ls_window_matrix_sparse_sums: one
# inverse per window, each channel's ADMM once), λ then the NormL1 weight of the default proxg.
function _windowed_matrix(kind, Y::AbstractMatrix, t, freqs, nw, noverlap, window_func, λ; sparse=nothing)
    N, nch = size(Y)
    length(t) == N || throw(AssertionError("y and t has to be the same length"))
    n = N ÷ nw
    freqs === nothing && (freqs = default_freqs(t, n))
    check_freq(freqs)
    noverlap < 0 && (noverlap = n >> 1)
    noverlap < n || throw(ArgumentError("noverlap must be smaller than the window length n"))
    Yv = Matrix{Float64}(Y)                          # column-major: channel c starts at c*N, so ldY = N
    tv, fv = vecf(t), vecf(freqs)
    Wv = vecf(window_func(n))
    length(Wv) == n || throw(DimensionMismatch("window_func(n) must return n = $n weights, got $(length(Wv))"))
    K = N >= n ? (N - n) ÷ (n - noverlap) + 1 : 0
    sums = zeros(ComplexF64, nch, nch, length(fv))   # C order [f][i][j] = Julia index (j, i, f)
    info = Ref{Cint}(0)
    if sparse === nothing
        GC.@preserve Yv tv fv Wv sums begin
            K > 0 && check(ccall((:lpvs_ls_window_matrix_sums, liblpvs), Cint,
                (Ptr{Cvoid}, Ptr{Float64}, Cint, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Cint, Ptr{Float64}, Cint, Cint,
                 Float64, Int64, Int64, Ptr{ComplexF64}, Ptr{Cint}),
                ctx(), Yv, nch, N, tv, N, fv, length(fv), Wv, n, noverlap, Float64(λ), 0, K, sums, info))
        end
    else
        pg, μ, iters, tol = sparse
        0 ≤ μ ≤ 1 || throw(AssertionError("μ should be ≤ 1"))                   # src/lasso.jl:143
        pk, pp = pg === nothing ? (PROX_L1, Float64(λ)) : proxdesc(pg)
        its = zeros(Int64, nch, max(K, 1)); res = zeros(nch, max(K, 1))     # C order [window][channel]
        GC.@preserve Yv tv fv Wv sums its res begin
            K > 0 && check(ccall((:lpvs_ls_window_matrix_sparse_sums, liblpvs), Cint,
                (Ptr{Cvoid}, Ptr{Float64}, Cint, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Cint, Ptr{Float64}, Cint, Cint,
                 Cint, Float64, Float64, Int64, Float64, Int64, Int64, Ptr{ComplexF64}, Ptr{Int64}, Ptr{Float64},
                 Ptr{Cint}),
                ctx(), Yv, nch, N, tv, N, fv, length(fv), Wv, n, noverlap, pk, Float64(pp), Float64(μ), iters,
                Float64(tol), 0, K, sums, its, res, info))
        end
    end
    info[] == 1 && @warn "a window's Gram matrix was numerically singular: solved with a jitter ridge (DESIGN.md section 1)"
    out = kind == WIN_PSD ? Matrix{Float64}(undef, nch, length(fv)) :
          kind == WIN_CSD ? Array{ComplexF64}(undef, nch, nch, length(fv)) : Array{Float64}(undef, nch, nch, length(fv))
    GC.@preserve sums out begin
        check(ccall((:lpvs_ls_window_matrix_finalize, liblpvs), Cint, (Cint, Ptr{ComplexF64}, Cint, Cint, Int64, Ptr{Cvoid}),
                    kind, sums, length(fv), nch, K, out))
    end
    res = kind == WIN_PSD ? permutedims(out, (2, 1)) : permutedims(out, (3, 2, 1))   # Nf x C, Nf x C x C
    like(Y, res), freqs
end

ls_windowpsd_multi(Y::AbstractMatrix, t, freqs=nothing; nw=8, noverlap=-1, window_func=rect, λ=1e-10) =
    _windowed_matrix(WIN_PSD, Y, t, freqs, nw, noverlap, window_func, λ)
ls_windowcsd_matrix(Y::AbstractMatrix, t, freqs=nothing; nw=10, noverlap=-1, window_func=rect, λ=1e-10) =
    _windowed_matrix(WIN_CSD, Y, t, freqs, nw, noverlap, window_func, λ)
ls_cohere_matrix(Y::AbstractMatrix, t, freqs=nothing; nw=10, noverlap=-1, λ=1e-10) =
    _windowed_matrix(WIN_COHERE, Y, t, freqs, nw, noverlap, hanning, λ)   # hanning hard-coded, as ls_cohere
ls_sparse_windowpsd_multi(Y::AbstractMatrix, t, freqs=nothing; nw=8, noverlap=-1, window_func=rect, proxg=nothing, λ=1.0,
                          μ=0.05, iters=10000, tol=1e-5) =
    _windowed_matrix(WIN_PSD, Y, t, freqs, nw, noverlap, window_func, λ; sparse=(proxg, μ, iters, tol))
ls_sparse_windowcsd_matrix(Y::AbstractMatrix, t, freqs=nothing; nw=10, noverlap=-1, window_func=rect, proxg=nothing,
                           λ=1.0, μ=0.05, iters=10000, tol=1e-5) =
    _windowed_matrix(WIN_CSD, Y, t, freqs, nw, noverlap, window_func, λ; sparse=(proxg, μ, iters, tol))
ls_sparse_cohere_matrix(Y::AbstractMatrix, t, freqs=nothing; nw=10, noverlap=-1, proxg=nothing, λ=1.0, μ=0.05,
                        iters=10000, tol=1e-5) =
    _windowed_matrix(WIN_COHERE, Y, t, freqs, nw, noverlap, hanning, λ; sparse=(proxg, μ, iters, tol))

# ---- LPV (src/lsfft.jl:239-259) -----------------------------------------------------------------------------
function ls_spectral_lpv(Y::AbstractVector, X::AbstractVector, V::AbstractVector, w, Nv::Integer;
                         λ=1e-8, coulomb=false, normalize=true)
    Yv, Xv, Vv, wv = vecf(Y), vecf(X), vecf(V), vecf(w[:])
    ncc = length(wv) * (coulomb ? 2Nv : Nv)
    params = Vector{ComplexF64}(undef, ncc)
    Σ = Matrix{Float64}(undef, 2ncc, 2ncc)
    fva = Ref{Float64}(0.0); info = Ref{Cint}(0)
    GC.@preserve Yv Xv Vv wv params Σ begin
        check(ccall((:lpvs_ls_spectral_lpv, liblpvs), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}, Cint, Cint, Float64, Cint,
             Cint, Ptr{ComplexF64}, Ptr{Float64}, Ptr{Float64}, Ptr{Cint}),
            ctx(), Yv, Xv, Vv, length(Yv), wv, length(wv), Nv, Float64(λ), coulomb, normalize, params, Σ, fva, info))
    end
    fva[] < 0.9 && @warn("Fraction of variance explained = $(fva[])")       # src/lsfft.jl:256
    SpectralExt(Y, X, V, wv, Nv, λ, coulomb, normalize, like(Y, params), like(Y, Σ))
end

# ---- ls_windowpsd_lpv (src/lsfft.jl:267-277): rect windows (Windows3), S = Σ_windows |Σ_k x[f,k]|², not normalised ----
function ls_windowpsd_lpv(Y::AbstractVector, X::AbstractVector, V::AbstractVector, w, Nv::Integer, nw::Int=10,
                          noverlap=0; λ=1e-8, coulomb=false, normalize=true)
    length(Y) == length(X) == length(V) || throw(AssertionError("y, t and v has to be the same length"))  # src/windows.jl:96
    Yv, Xv, Vv, wv = vecf(Y), vecf(X), vecf(V), vecf(w[:])
    n = length(Yv) ÷ nw
    Kw = ccall((:lpvs_window_count, liblpvs), Int64, (Int64, Cint, Cint), length(Yv), n, noverlap)
    S = zeros(length(wv)); fva = ones(max(Kw, 1))
    K = Ref{Int64}(0); info = Ref{Cint}(0)
    GC.@preserve Yv Xv Vv wv S fva begin
        check(ccall((:lpvs_ls_windowpsd_lpv, liblpvs), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}, Cint, Cint, Cint, Cint, Float64,
             Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Cint}),
            ctx(), Yv, Xv, Vv, length(Yv), wv, length(wv), Nv, n, noverlap, Float64(λ), coulomb, normalize, S, fva, K,
            info))
    end
    for k in 1:K[]
        fva[k] < 0.9 && @warn("Fraction of variance explained = $(fva[k])")  # src/lsfft.jl:256, once per window
    end
    like(Y, S)
end

# ---- ADMM-backed sparse estimators (src/lasso.jl) ---------------------------------------------------------------
# proxg objects are ProximalOperators types; only their (kind, parameter) crosses the ABI.
proxdesc(p) = begin
    T = string(nameof(typeof(p)))
    T == "NormL1" && return PROX_L1, Float64(p.lambda)
    T == "NormL0" && return PROX_L0, Float64(p.lambda)
    T == "IndBallL0" && return PROX_BALL_L0, Float64(p.r)
    throw(ArgumentError("proxg must be NormL1, NormL0 or IndBallL0 (no CPU fallback for other operators)"))
end

# Drives the device loop in chunks of `printerval` so prints and cb(x,z) match src/lasso.jl:158-167 (SURVEY H6).
function run_admm(h, n; iters=10000, tol=1e-5, printerval=100, cb=nothing, μ=nothing)
    done = 0; res = Ref{Float64}(Inf); conv = Ref{Cint}(0); it = Ref{Int64}(0)
    while done < iters && conv[] == 0
        chunk = min(printerval - done % printerval, iters - done)
        check(ccall((:lpvs_admm_run, liblpvs), Cint, (Ptr{Cvoid}, Int64, Float64, Ptr{Int64}, Ptr{Float64}, Ptr{Cint}),
                    h, chunk, Float64(tol), it, res, conv))
        done += it[]
        if done % printerval == 0                                               # src/lasso.jl:158-163
            @printf("%d ||x-z||₂ %.10f\n", done, res[])
            if cb !== nothing
                x = Vector{Float64}(undef, n); z = similar(x)
                check(ccall((:lpvs_admm_get, liblpvs), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}), h, x, z))
                cb(x, z)
            end
        end
        if conv[] != 0                                # :164-168 (a stop on a print iteration prints the line twice)
            @printf("%d ||x-z||₂ %.10f\n", done, res[])
            @info("||x-z||₂ ≤ tol")
        end
    end
end

function ls_sparse_spectral(y::AbstractArray{T}, t, f=default_freqs(t), W=nothing;
                            init=false, λ=T(1), proxg=nothing, μ=T(0.05), kwargs...) where T
    @assert 0 ≤ μ ≤ 1 "μ should be ≤ 1"                                  # src/lasso.jl:143
    check_freq(f)
    kind, param = proxg === nothing ? (PROX_L1, Float64(λ)) : proxdesc(proxg)   # Q15
    yv, tv, fv = vecf(y), vecf(t), vecf(f)
    Wv = W === nothing ? nothing : vecf(W)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve yv tv fv Wv with_m32(T) do
        check(ccall((:lpvs_admm_create_fourier, liblpvs), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}, Cint, Ptr{Float64}, Cint, Float64, Float64,
             Ptr{Float64}, Cint, Float64, Ptr{Ptr{Cvoid}}),
            ctx(), yv, tv, length(yv), fv, length(fv), nullable(Wv), kind, param, Float64(μ), C_NULL, init,
            Float64(λ), h))
    end
    params = Vector{ComplexF64}(undef, length(fv))
    try
        run_admm(h[], ccall((:lpvs_admm_size, liblpvs), Cint, (Ptr{Cvoid},), h[]); kwargs...)
        check(ccall((:lpvs_admm_result, liblpvs), Cint, (Ptr{Cvoid}, Ptr{ComplexF64}), h[], params))
    finally
        ccall((:lpvs_admm_free, liblpvs), Cvoid, (Ptr{Cvoid},), h[])
    end
    like(y, params), f
end

function ls_sparse_spectral_lpv(y::AbstractVector{S}, X::AbstractVector{S}, V::AbstractVector{S}, w, Nv::Integer;
                                λ=1, coulomb=false, normalize=true, μ=S(0.05), kwargs...) where S
    yv, Xv, Vv, wv = vecf(y), vecf(X), vecf(V), vecf(w[:])
    h = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve yv Xv Vv wv with_m32(S) do
        check(ccall((:lpvs_admm_create_lpv, liblpvs), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}, Cint, Cint, Cint, Cint,
             Float64, Float64, Ptr{Ptr{Cvoid}}),
            ctx(), yv, Xv, Vv, length(yv), wv, length(wv), Nv, coulomb, normalize, Float64(λ), Float64(μ), h))
    end
    params = Vector{ComplexF64}(undef, length(wv) * (coulomb ? 2Nv : Nv))
    try
        try
            run_admm(h[], ccall((:lpvs_admm_size, liblpvs), Cint, (Ptr{Cvoid},), h[]); kwargs...)
        catch e
            e isa InterruptException || rethrow(e)                          # src/lasso.jl:57-66 (Q17)
            @info "Aborting"
        end
        check(ccall((:lpvs_admm_result, liblpvs), Cint, (Ptr{Cvoid}, Ptr{ComplexF64}), h[], params))
    finally
        ccall((:lpvs_admm_free, liblpvs), Cvoid, (Ptr{Cvoid},), h[])
    end
    SpectralExt(y, X, V, wv, Nv, λ, coulomb, normalize, like(y, params), nothing)
end

end # module
