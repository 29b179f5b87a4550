# LSCuda.jl - Julia host side of the B200-native Lippmann-Schwinger hot path.
#
# Drop-in for the reference's operator objects: the types below carry the same fields and the same
# method table as `FastM` (src/FastConvolution.jl:11-154), `FastM3D` (src/FastConvolution3D.jl:7-63)
# and `SparsifyingPreconditioner` (src/preconditioner.jl:27-58,132-170), but every apply ends in a
# `ccall` into libls_cuda.so (include/ls_cuda.h).  `IterativeSolvers.gmres!(u, A, rhs, Pl=precond)`
# (examples/example.jl:85) takes them unchanged because it only needs `mul!`, `size`, `eltype`
# and `ldiv!`; `gmres_gpu!` additionally keeps the whole Krylov basis on the device.
#
# NOT EXECUTED IN THIS REPOSITORY'S CI: the build image has no Julia.  The same C-ABI calls are
# exercised by the Python/ctypes mirror (fast_solver_lippmann_schwinger_b200/), see INTEGRATION.md.
module LSCuda

using LinearAlgebra, SparseArrays
import Base: *, \, size, eltype
import LinearAlgebra: mul!, ldiv!

const libls = get(ENV, "LS_CUDA_LIB", "libls_cuda.so")

const LS_MEM_HOST, LS_MEM_DEVICE = Cint(0), Cint(1)
const LS_FLAG_FORCE_GENERIC, LS_FLAG_PAD4, LS_FLAG_EMBED = Cint(1), Cint(2), Cint(4)
const LS_ORTH = Dict("ModifiedGramSchmidt" => Cint(0), "ClassicalGramSchmidt" => Cint(1), "DGKS" => Cint(2))
const LS_QUAD = Dict("trapezoidal" => Cint(0), "Greengard_Vico" => Cint(1))

struct LSCudaError <: Exception
    code::Cint
    msg::String
end

function check(rc::Cint)
    rc == 0 && return nothing
    throw(LSCudaError(rc, unsafe_string(ccall((:ls_last_error, libls), Cstring, ()))))
end

mutable struct Handle
    ptr::Ptr{Cvoid}
    function Handle(p::Ptr{Cvoid})
        h = new(p)
        finalizer(h -> (h.ptr != C_NULL && ccall((:ls_destroy, libls), Cint, (Ptr{Cvoid},), h.ptr); h.ptr = C_NULL), h)
        return h
    end
end

set_device(dev::Integer) = check(ccall((:ls_set_device, libls), Cint, (Cint,), dev))

# ---------------------------------------------------------------------------------- FastM (2-D)
struct GPUFastM
    h::Handle
    nu::Vector{Float64}
    ne::Int64; me::Int64; n::Int64; m::Int64
    omega::Float64
    quadRule::String
end

"""
    GPUFastM(GFFT, nu, ne, me, n, m, k; quadRule, embed=false)

Same constructor as FastM (FastConvolution.jl:24).  `embed=true` (LS_FLAG_EMBED) runs any grid with n, m <= 4096 on the
power-of-two kernels with the grid zero-embedded (h = 1/1000: n = 1001, beyond the Bluestein general path).
"""
function GPUFastM(GFFT::Array{ComplexF64,2}, nu::Vector{Float64}, ne, me, n, m, k; quadRule::String="trapezoidal",
                  embed::Bool=false)
    size(GFFT) == (ne, me) || throw(DimensionMismatch("GFFT is $(size(GFFT)), expected ($ne, $me)"))
    length(nu) == n * m || throw(DimensionMismatch("nu has $(length(nu)) entries, expected $(n*m)"))
    out = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:ls_op2d_create, libls), Cint,
                (Ref{Ptr{Cvoid}}, Int64, Int64, Int64, Int64, Ptr{Float64}, Ptr{ComplexF64}, Float64, Cint, Cint),
                out, n, m, ne, me, nu, GFFT, Float64(k), LS_QUAD[quadRule], embed ? LS_FLAG_EMBED : Cint(0)))
    return GPUFastM(Handle(out[]), nu, ne, me, n, m, Float64(k), quadRule)
end
"Move an existing reference operator to the GPU."
GPUFastM(M) = GPUFastM(M.GFFT, M.nu, M.ne, M.me, M.n, M.m, M.omega; quadRule=M.quadRule)
"""
    GPUFastM(x, y, h, k, nu)

GPU twin of `buildFastConvolution(x, y, h, k, nu, quadRule = "Greengard_Vico")` (FastConvolution.jl:185-231) that never
builds GFFT on the host: the spectrum Gtruncated2D(L, k, S) is evaluated on the device (ls_op2d_create_gv).
"""
function GPUFastM(x::AbstractVector, y::AbstractVector, h::Real, k::Real, nu::Function; embed::Bool=false)
    (n, m) = length(x), length(y)
    Lp = 4 * (abs(x[end] - x[1]) + h); L = 1.5 * (abs(x[end] - x[1]) + h)
    X = repeat(x, 1, m)[:]; Y = repeat(y', n, 1)[:]
    nuv = Vector{Float64}(nu(X, Y))
    out = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:ls_op2d_create_gv, libls), Cint, (Ref{Ptr{Cvoid}}, Int64, Int64, Ptr{Float64}, Float64, Float64, Float64, Cint),
                out, n, m, nuv, Float64(k), Float64(L), Float64(Lp), embed ? LS_FLAG_EMBED : Cint(0)))
    return GPUFastM(Handle(out[]), nuv, 4n, 4m, n, m, Float64(k), "Greengard_Vico")
end

"(route: 0 power of two / 1 Bluestein / 2 zero-embedded, line lengths the kernels run, padding factor in use)"
function op2d_info(M::GPUFastM)
    r = Ref{Cint}(0); nl = Ref{Int64}(0); ml = Ref{Int64}(0); p = Ref{Cint}(0)
    check(ccall((:ls_op2d_info, libls), Cint, (Ptr{Cvoid}, Ref{Cint}, Ref{Int64}, Ref{Int64}, Ref{Cint}), M.h.ptr, r, nl, ml, p))
    return (route=r[], n_line=nl[], m_line=ml[], padding=p[])
end

size(M::GPUFastM, dim) = length(M.nu)                       # FastConvolution.jl:31-33
size(M::GPUFastM) = (size(M.nu), size(M.nu))                # :35-37 (tuple of tuples, kept)
eltype(M::GPUFastM) = ComplexF64                            # :39-41

function apply!(y::StridedVector{ComplexF64}, M::GPUFastM, b::StridedVector{ComplexF64}, mode::Integer)
    length(b) == length(M.nu) == length(y) || throw(DimensionMismatch("vector length"))
    (stride(b, 1) == 1 && stride(y, 1) == 1) || throw(ArgumentError("unit stride required"))
    check(ccall((:ls_op2d_apply, libls), Cint, (Ptr{Cvoid}, Ptr{ComplexF64}, Ptr{ComplexF64}, Cint, Cint),
                M.h.ptr, b, y, mode, LS_MEM_HOST))
    return y
end
fastconvolution(M::GPUFastM, b::AbstractVector{ComplexF64}) = apply!(similar(b, ComplexF64), M, b, 0)   # :58-107
FFTconvolution(M::GPUFastM, b::Vector{ComplexF64}) = apply!(similar(b), M, b, 1)                        # :110-154
*(M::GPUFastM, b::AbstractVector{ComplexF64}) = fastconvolution(M, b)                                   # :43-48
mul!(Y::AbstractVector{ComplexF64}, M::GPUFastM, b::AbstractVector{ComplexF64}) = apply!(Y, M, b, 0)    # :50-54

# several right-hand sides: the N x K columns through one ls_op_apply_batch (each column with the bits of the single apply)
function apply!(Y::Matrix{ComplexF64}, M, B::Matrix{ComplexF64}, mode::Integer)
    size(Y) == size(B) && size(B, 1) == length(M.nu) || throw(DimensionMismatch("B is $(size(B)), Y is $(size(Y))"))
    N, K = size(B)
    check(ccall((:ls_op_apply_batch, libls), Cint, (Ptr{Cvoid}, Ptr{ComplexF64}, Int64, Ptr{ComplexF64}, Int64, Cint, Cint, Cint),
                M.h.ptr, B, N, Y, N, K, mode, LS_MEM_HOST))
    return Y
end
*(M::GPUFastM, B::Matrix{ComplexF64}) = apply!(similar(B), M, B, 0)
mul!(Y::Matrix{ComplexF64}, M::GPUFastM, B::Matrix{ComplexF64}) = apply!(Y, M, B, 0)

# -------------------------------------------------------------------------------- FastM3D (3-D)
struct GPUFastM3D
    h::Handle
    nu::Vector{Float64}
    ne::Int64; me::Int64; le::Int64; n::Int64; m::Int64; l::Int64
    omega::Float64
    quadRule::String
end

"""GFFT === nothing: the Greengard-Vico spectrum is generated on the device from (L, Lp) (FastConvolution3D.jl:72-99).
`embed=true` (LS_FLAG_EMBED) runs any n = m, l <= 512 on the power-of-two kernels with the grid zero-embedded."""
function GPUFastM3D(GFFT, nu::Vector{Float64}, ne, me, le, n, m, l, k; L=0.0, Lp=0.0, quadRule="Greengard_Vico",
                    embed::Bool=false)
    out = Ref{Ptr{Cvoid}}(C_NULL)
    g = GFFT === nothing ? Ptr{ComplexF64}(C_NULL) : pointer(GFFT)
    GC.@preserve GFFT check(ccall((:ls_op3d_create, libls), Cint,
                (Ref{Ptr{Cvoid}}, Int64, Int64, Int64, Int64, Int64, Int64, Ptr{Float64}, Ptr{ComplexF64}, Float64, Float64, Float64, Cint),
                out, n, m, l, ne, me, le, nu, g, Float64(k), Float64(L), Float64(Lp), embed ? LS_FLAG_EMBED : Cint(0)))
    return GPUFastM3D(Handle(out[]), nu, ne, me, le, n, m, l, Float64(k), quadRule)
end
"GPUFastM3D(M) - GPU twin of a reference `FastM3D`."
GPUFastM3D(M) = GPUFastM3D(M.GFFT, M.nu, M.ne, M.me, M.le, M.n, M.m, M.l, M.omega; quadRule=M.quadRule)
size(M::GPUFastM3D, dim) = length(M.nu)       # not defined upstream (Q4) - required by gmres!
size(M::GPUFastM3D) = (size(M.nu), size(M.nu))
eltype(M::GPUFastM3D) = ComplexF64
function apply!(y::StridedVector{ComplexF64}, M::GPUFastM3D, b::StridedVector{ComplexF64}, mode::Integer)
    check(ccall((:ls_op3d_apply, libls), Cint, (Ptr{Cvoid}, Ptr{ComplexF64}, Ptr{ComplexF64}, Cint, Cint),
                M.h.ptr, b, y, mode, LS_MEM_HOST))
    return y
end
*(M::GPUFastM3D, b::Array{ComplexF64,1}; verbose::Bool=false) = apply!(similar(b), M, b, 0)     # FastConvolution3D.jl:31-37
FFTconvolution(M::GPUFastM3D, b::Array{ComplexF64,1}; verbose::Bool=false) = apply!(similar(b), M, b, 1)   # :39-63
mul!(Y::AbstractVector{ComplexF64}, M::GPUFastM3D, b::AbstractVector{ComplexF64}) = apply!(Y, M, b, 0)
*(M::GPUFastM3D, B::Matrix{ComplexF64}) = apply!(similar(B), M, B, 0)
mul!(Y::Matrix{ComplexF64}, M::GPUFastM3D, B::Matrix{ComplexF64}) = apply!(Y, M, B, 0)

# ---------------------------------------------------- FastM3D slab-decomposed over several GPUs
# One Julia process per GPU (Distributed.jl / MPI.jl).  Rank 0 calls nccl_unique_id() and broadcasts the
# 128 bytes; every rank then builds the operator with its z slab of nu (planes [rank*l/P, (rank+1)*l/P))
# and applies it to its slab of the vectors.  gmres_gpu! on such an operator all-reduces its dot products.
function nccl_unique_id()
    id = zeros(UInt8, 128)
    check(ccall((:ls_nccl_unique_id, libls), Cint, (Ptr{UInt8},), id))
    return id
end
function GPUFastM3DSharded(nu_slab::Vector{Float64}, n, m, l, k, L, Lp, rank::Integer, nranks::Integer,
                           id::Vector{UInt8}; pad4::Bool=false, embed::Bool=false)
    out = Ref{Ptr{Cvoid}}(C_NULL)
    flags = (pad4 ? LS_FLAG_PAD4 : Cint(0)) | (embed ? LS_FLAG_EMBED : Cint(0))
    check(ccall((:ls_op3d_create_dist, libls), Cint,
                (Ref{Ptr{Cvoid}}, Int64, Int64, Int64, Ptr{Float64}, Float64, Float64, Float64, Cint, Cint, Ptr{UInt8}, Cint),
                out, n, m, l, nu_slab, Float64(k), Float64(L), Float64(Lp), rank, nranks, id, flags))
    return GPUFastM3D(Handle(out[]), nu_slab, 4n, 4m, 4l, n, m, l, Float64(k), "Greengard_Vico")
end

"(padding factor in use, x-slot chunks, transpose route: 0 single GPU / 1 NCCL send-recv / 2 copy-engine pushes)"
function op3d_info(M::GPUFastM3D)
    p = Ref{Cint}(0); c = Ref{Cint}(0); x = Ref{Cint}(0)
    check(ccall((:ls_op3d_info, libls), Cint, (Ptr{Cvoid}, Ref{Cint}, Ref{Cint}, Ref{Cint}), M.h.ptr, p, c, x))
    return (padding=p[], chunks=c[], exchange=x[])
end

"(route: 0 power of two / 1 Bluestein / 2 zero-embedded, line lengths the kernels run along x, y, z)"
function op3d_lines(M::GPUFastM3D)
    r = Ref{Cint}(0); nl = Ref{Int64}(0); ml = Ref{Int64}(0); ll = Ref{Int64}(0)
    check(ccall((:ls_op3d_lines, libls), Cint, (Ptr{Cvoid}, Ref{Cint}, Ref{Int64}, Ref{Int64}, Ref{Int64}), M.h.ptr, r, nl, ml, ll))
    return (route=r[], n_line=nl[], m_line=ml[], l_line=ll[])
end

"""
Row slab of the sparsifier next to a sharded operator: `Ablk` is `As[rows, (first(rows)-halo):(last(rows)+halo)]`
(columns outside the matrix empty), `rows` the rank's slab of `M`.  `As_sh * x` is collective: the halo of x
comes from the two z-neighbours.
"""
function GPUSparseMatrixCSCSharded(Ablk::SparseMatrixCSC{ComplexF64,Int64}, M::GPUFastM3D, halo::Integer)
    out = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:ls_spm_create_dist, libls), Cint,
                (Ref{Ptr{Cvoid}}, Ptr{Cvoid}, Int64, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{ComplexF64}),
                out, M.h.ptr, Ablk.m, halo, Ablk.colptr, Ablk.rowval, Ablk.nzval))
    return GPUSparseMatrixCSC(Handle(out[]), Ablk.m, Ablk.m)
end

# ---------------------------------------------------------------- sparsifying preconditioner
struct GPUSparseMatrixCSC
    h::Handle
    m::Int64; n::Int64
end
function GPUSparseMatrixCSC(A::SparseMatrixCSC{ComplexF64,Int64})
    out = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:ls_spm_create, libls), Cint, (Ref{Ptr{Cvoid}}, Int64, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{ComplexF64}),
                out, A.m, A.n, A.colptr, A.rowval, A.nzval))
    return GPUSparseMatrixCSC(Handle(out[]), A.m, A.n)
end
"y <- alpha*A*x + beta*y; the cscmv! of sparseblas.jl:14-25 with transa = 'N'."
function cscmv!(alpha::ComplexF64, A::GPUSparseMatrixCSC, x::Vector{ComplexF64}, beta::ComplexF64, y::Vector{ComplexF64})
    length(x) == A.n || throw(DimensionMismatch("Matrix with $(A.n) columns multiplied with vector of length $(length(x))"))
    length(y) == A.m || throw(DimensionMismatch("Vector of length $(A.m) added to vector of length $(length(y))"))
    check(ccall((:ls_spm_mv, libls), Cint, (Ptr{Cvoid}, ComplexF64, Ptr{ComplexF64}, ComplexF64, Ptr{ComplexF64}, Cint),
                A.h.ptr, alpha, x, beta, y, LS_MEM_HOST))
    return y
end
*(A::GPUSparseMatrixCSC, x::Vector{ComplexF64}) = cscmv!(1.0 + 0im, A, x, 0.0 + 0im, zeros(ComplexF64, A.m))

"""
`lu(Msp)` (preconditioner.jl:35) on the GPU: nested-dissection factorisation of the 9-point matrix Msp of the
n x m grid, or (with `l`) of the 27-point matrix of the n x m x l grid (examples/example3D.jl:56-61).  `F \\ b` solves on host vectors; inside `gmres_gpu!` the solve never leaves the device.
"""
struct GPUMspFactorization
    h::Handle
    N::Int64
end
function GPUMspFactorization(Msp::SparseMatrixCSC{ComplexF64,Int64}, n::Integer, m::Integer)
    size(Msp, 1) == size(Msp, 2) == n * m || throw(DimensionMismatch("Msp is $(size(Msp)), the grid has $(n*m) unknowns"))
    out = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:ls_msp_factor, libls), Cint, (Ref{Ptr{Cvoid}}, Int64, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{ComplexF64}),
                out, n, m, Msp.colptr, Msp.rowval, Msp.nzval))
    return GPUMspFactorization(Handle(out[]), n * m)
end
function GPUMspFactorization(Msp::SparseMatrixCSC{ComplexF64,Int64}, n::Integer, m::Integer, l::Integer)
    size(Msp, 1) == size(Msp, 2) == n * m * l || throw(DimensionMismatch("Msp is $(size(Msp)), the grid has $(n*m*l) unknowns"))
    out = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:ls_msp_factor3d, libls), Cint, (Ref{Ptr{Cvoid}}, Int64, Int64, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{ComplexF64}),
                out, n, m, l, Msp.colptr, Msp.rowval, Msp.nzval))
    return GPUMspFactorization(Handle(out[]), n * m * l)
end
function \(F::GPUMspFactorization, b::Vector{ComplexF64})
    x = similar(b)
    check(ccall((:ls_msp_solve, libls), Cint, (Ptr{Cvoid}, Ptr{ComplexF64}, Ptr{ComplexF64}, Cint), F.h.ptr, b, x, LS_MEM_HOST))
    return x
end
"`F \\ B` for an N x K matrix: the K right-hand sides in one ls_msp_solve_batch (each factor block read once per chunk of columns)."
function \(F::GPUMspFactorization, B::Matrix{ComplexF64})
    X = similar(B)
    check(ccall((:ls_msp_solve_batch, libls), Cint, (Ptr{Cvoid}, Ptr{ComplexF64}, Int64, Ptr{ComplexF64}, Int64, Cint, Cint),
                F.h.ptr, B, size(B, 1), X, size(X, 1), size(B, 2), LS_MEM_HOST))
    return X
end
function msp_info(F::GPUMspFactorization)
    fb = Ref{Int64}(0); dep = Ref{Cint}(0); sec = Ref{Float64}(0.0)
    check(ccall((:ls_msp_info, libls), Cint, (Ptr{Cvoid}, Ref{Int64}, Ref{Cint}, Ref{Float64}), F.h.ptr, fb, dep, sec))
    return (factor_bytes=fb[], depth=dep[], factor_seconds=sec[])
end
function msp_plan(F::GPUMspFactorization)
    buf = Vector{UInt8}(undef, 8192)
    check(ccall((:ls_msp_plan, libls), Cint, (Ptr{Cvoid}, Ptr{UInt8}, Int64), F.h.ptr, buf, length(buf)))
    return unsafe_string(pointer(buf))
end

struct GPUSparsifyingPreconditioner      # preconditioner.jl:27-58
    Msp::SparseMatrixCSC{ComplexF64,Int64}
    As::GPUSparseMatrixCSC
    MspInv                                 # lu(Msp): UMFPACK on the host, or GPUMspFactorization (solverType = "GPU")
    solverType::String
end
"solverType = \"UMFPACK\" / \"MKLPARDISO\" as upstream (host LU, reached through the ls_solve_cb callback), or \"GPU\" with grid = (n, m) or (n, m, l)."
GPUSparsifyingPreconditioner(Msp, As; solverType::String="UMFPACK", grid=nothing) =
    GPUSparsifyingPreconditioner(Msp, GPUSparseMatrixCSC(As),
                                 solverType == "GPU" ? GPUMspFactorization(Msp, grid...) : lu(Msp), solverType)
\(M::GPUSparsifyingPreconditioner, b::Array{ComplexF64,1}) = M.MspInv \ (M.As * b)                     # :132-145
function ldiv!(M::GPUSparsifyingPreconditioner, b::AbstractArray{ComplexF64,1})                        # :147-166
    b[:] = M.MspInv \ (M.As * Vector(b))
end
# several right-hand sides: with solverType = "GPU" the Msp^-1 of all columns is one batched solve
function ldiv!(M::GPUSparsifyingPreconditioner, B::Matrix{ComplexF64})
    AB = reduce(hcat, [M.As * B[:, j] for j in 1:size(B, 2)])
    B[:, :] = M.MspInv isa GPUMspFactorization ? M.MspInv \ AB : reduce(hcat, [M.MspInv \ AB[:, j] for j in 1:size(B, 2)])
    return B
end

# ------------------------------------------------------- device-resident GMRES (whole loop on GPU)
"""
    gmres_gpu!(x, A, b; Pl=nothing, abstol, reltol, restart, maxiter, log, initially_zero)

Same keywords and history semantics as `IterativeSolvers.gmres!`; the Krylov basis, the modified
Gram-Schmidt sweeps and the operator applies stay on the device; `Msp^-1` runs on the device too when the
preconditioner was built with solverType = "GPU", else it is reached through a host callback.
"""
function gmres_gpu!(x::Vector{ComplexF64}, A, b::Vector{ComplexF64}; Pl=nothing, abstol=0.0,
                    reltol=sqrt(eps(Float64)), restart=min(20, length(b)), maxiter=length(b), log=false,
                    initially_zero=false, orth_meth="ModifiedGramSchmidt")
    N = length(b)
    kh = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:ls_krylov_create, libls), Cint, (Ref{Ptr{Cvoid}}, Int64), kh, N))
    K = Handle(kh[])
    check(ccall((:ls_krylov_set_orth, libls), Cint, (Ptr{Cvoid}, Cint), K.ptr, LS_ORTH[orth_meth]))
    hist = zeros(Float64, maxiter); niter = Ref{Int64}(0); conv = Ref{Cint}(0); mv = Ref{Int64}(0)
    cb = C_NULL; as = C_NULL
    if Pl !== nothing && Pl.MspInv isa GPUMspFactorization      # Msp^-1 (As v) entirely on the device
        check(ccall((:ls_gmres_msp, libls), Cint,
            (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{ComplexF64}, Ptr{ComplexF64}, Cint, Int64,
             Float64, Float64, Cint, Ptr{Float64}, Int64, Ref{Int64}, Ref{Cint}, Ref{Int64}, Cint),
            K.ptr, A.h.ptr, Pl.As.h.ptr, Pl.MspInv.h.ptr, b, x, restart, maxiter,
            reltol, abstol, initially_zero, hist, maxiter, niter, conv, mv, LS_MEM_HOST))
        return log ? (x, (resnorm=hist[1:niter[]], iters=niter[], isconverged=conv[] != 0, mvps=mv[])) : x
    end
    if Pl !== nothing
        solve = function (user::Ptr{Cvoid}, v::Ptr{ComplexF64}, n::Int64)::Cint
            w = unsafe_wrap(Array, v, n)
            w[:] = Pl.MspInv \ copy(w)
            return 0
        end
        cb = @cfunction($solve, Cint, (Ptr{Cvoid}, Ptr{ComplexF64}, Int64))
        as = Pl.As.h.ptr
    end
    GC.@preserve cb check(ccall((:ls_gmres, libls), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{ComplexF64}, Ptr{ComplexF64}, Cint, Int64,
         Float64, Float64, Cint, Ptr{Float64}, Int64, Ref{Int64}, Ref{Cint}, Ref{Int64}, Cint),
        K.ptr, A.h.ptr, as, cb isa Ptr ? cb : Base.unsafe_convert(Ptr{Cvoid}, cb), C_NULL, b, x, restart, maxiter,
        reltol, abstol, initially_zero, hist, maxiter, niter, conv, mv, LS_MEM_HOST))
    return log ? (x, (resnorm=hist[1:niter[]], iters=niter[], isconverged=conv[] != 0, mvps=mv[])) : x
end

"""
    gmres_gpu!(X::Matrix, A, B::Matrix; Pl, abstol, reltol, restart, maxiter, log, initially_zero)

K independent gmres! runs for the columns of B (several incident fields) in lockstep on the device: with Pl = I
(ls_gmres_batch) or with Pl built with solverType = "GPU" (ls_gmres_msp_batch); each system gets the history and x that
gmres_gpu! gives it alone, the operator applies of all active systems are multi-column applies and, with Pl, the
Msp^-1 of all active systems is one batched solve per iteration.
With log = true the second result is a vector of K histories.
"""
function gmres_gpu!(X::Matrix{ComplexF64}, A, B::Matrix{ComplexF64}; Pl=I, abstol=0.0, reltol=sqrt(eps(Float64)),
                    restart=min(20, size(B, 1)), maxiter=size(B, 1), log=false, initially_zero=false)
    N, K = size(B)
    size(X) == (N, K) || throw(DimensionMismatch("X is $(size(X)), B is $(size(B))"))
    Pl === I || Pl.MspInv isa GPUMspFactorization ||
        throw(ArgumentError("several right-hand sides need Pl = I or Pl with solverType = \"GPU\""))
    kh = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:ls_krylov_create, libls), Cint, (Ref{Ptr{Cvoid}}, Int64), kh, N))
    W = Handle(kh[])
    cap = min(maxiter, 1_000_000)                 # history rows kept, as in the Python mirror
    hist = zeros(Float64, cap, K); niter = zeros(Int64, K); conv = zeros(Cint, K); mv = zeros(Int64, K)
    if Pl === I
        check(ccall((:ls_gmres_batch, libls), Cint,
            (Ptr{Cvoid}, Ptr{Cvoid}, Cint, Ptr{ComplexF64}, Int64, Ptr{ComplexF64}, Int64, Cint, Int64,
             Float64, Float64, Cint, Ptr{Float64}, Int64, Ptr{Int64}, Ptr{Cint}, Ptr{Int64}, Cint),
            W.ptr, A.h.ptr, K, B, N, X, N, restart, maxiter, reltol, abstol, initially_zero, hist, cap, niter, conv, mv,
            LS_MEM_HOST))
    else
    check(ccall((:ls_gmres_msp_batch, libls), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Cint, Ptr{ComplexF64}, Int64, Ptr{ComplexF64}, Int64, Cint, Int64,
         Float64, Float64, Cint, Ptr{Float64}, Int64, Ptr{Int64}, Ptr{Cint}, Ptr{Int64}, Cint),
        W.ptr, A.h.ptr, Pl.As.h.ptr, Pl.MspInv.h.ptr, K, B, N, X, N, restart, maxiter,
        reltol, abstol, initially_zero, hist, cap, niter, conv, mv, LS_MEM_HOST))
    end
    log || return X
    return X, [(resnorm=hist[1:min(niter[q], cap), q], iters=niter[q], isconverged=conv[q] != 0, mvps=mv[q]) for q in 1:K]
end

export GPUFastM, op2d_info, GPUFastM3D, GPUFastM3DSharded, op3d_lines, nccl_unique_id, GPUSparsifyingPreconditioner, GPUSparseMatrixCSC, GPUMspFactorization, msp_info, fastconvolution, FFTconvolution,
       gmres_gpu!, cscmv!, set_device

end # module
