# EnlsipB200.jl -- Julia host layer over the C ABI of include/enlsip_b200.h.
#
# Keeps the exported names of the reference (src/cnls_model.jl:1-3, src/solver.jl:1):
#     CnlsModel, solve!, status, solution, sum_sq_residuals, total_nb_constraints, dict_status_codes
# and calls the B200 engine with `ccall`.  The reference's closures (residuals, jacobians,
# constraints) cannot cross to the GPU, so a model names a device problem `family` compiled into
# libenlsip_b200.so and carries its data arrays; one model object is a BATCH of B independent
# problems (row b of `starting_point` is the starting point of problem b).
#
# NOT EXECUTED in the build container (no Julia binary in the image; see DESIGN.md).  The ctypes
# binding in enlsip.jl_b200/capi.py binds the same symbols with the same argument lists and is what
# the tests exercise.
module EnlsipB200

export CnlsModel, LargeCnlsModel, solve!, status, solution, sum_sq_residuals, total_nb_constraints, dict_status_codes

const libenlsip = get(ENV, "ENLSIP_B200_LIB", joinpath(@__DIR__, "..", "lib", "libenlsip_b200.so"))

const FAMILY_HS65 = Cint(0)
const FAMILY_GAUSS_PEAKS = Cint(1)
const JAC_ANALYTIC = Cint(0)
const JAC_FORWARD_DIFF = Cint(1)

# struct enlsipb200_options (include/enlsip_b200.h) == keyword arguments of solve! (solver.jl:62-63)
struct Options
    max_iter::Cint
    scaling::Cint
    jac_mode::Cint
    reserved::Cint
    time_limit::Cdouble
    abs_tol::Cdouble
    rel_tol::Cdouble
    c_tol::Cdouble
    x_tol::Cdouble
end

const dict_status_codes = Dict(          # cnls_model.jl:180-186
    0 => :unsolved,
    1 => :found_first_order_stationary_point,
    -1 => :failed,
    -2 => :maximum_iterations_exceeded,
    -11 => :time_limit_exceeded,
)

last_error() = unsafe_string(ccall((:enlsipb200_last_error, libenlsip), Cstring, ()))
check(rc::Cint) = rc == 0 || error("enlsip_b200 error $rc: $(last_error())")

# ---- user problems: the reference's closure arguments as CUDA C++ source (include/enlsip_b200.h) ----
using Libdl
const FAMILY_USER = Cint(64)
const stock_handle = Ref{Ptr{Cvoid}}(C_NULL)
stocklib() = (stock_handle[] == C_NULL && (stock_handle[] = Libdl.dlopen(libenlsip)); stock_handle[])
# entry point `name` of the stock library (lib == C_NULL) or of a library written by compile_family
fsym(lib::Ptr{Cvoid}, name::Symbol) = Libdl.dlsym(lib == C_NULL ? stocklib() : lib, name)

"""
    compile_family(source; n, m, nb_eqcons=0, nb_ineqcons=0, stride0=0, stride1=0, has_jacobians=false)

Device-side counterpart of the closures `residuals`, `eq_constraints`, `ineq_constraints`, `jacobian_*` of the
reference constructor (cnls_model.jl:345-359): `source` defines `enl_user::residual`, `enl_user::constraints` (and
optionally `jac_residual`, `jac_constraints`); the engine compiles its solver around them and returns the handle of a
library with the same C ABI.  Pass it to `CnlsModel(lib, starting_point; ...)`.
"""
function compile_family(source::String; n::Integer, m::Integer, nb_eqcons::Integer=0, nb_ineqcons::Integer=0,
                        stride0::Integer=0, stride1::Integer=0, has_jacobians::Bool=false,
                        work_dir::String=mktempdir(), out::String=joinpath(work_dir, "libenlsip_b200_user.so"))
    check(ccall((:enlsipb200_compile_family, libenlsip), Cint,
                (Cstring, Cint, Cint, Cint, Cint, Cint, Cint, Cint, Cstring, Cstring),
                source, n, m, nb_eqcons, nb_ineqcons, stride0, stride1, has_jacobians ? 1 : 0, out, work_dir))
    return Libdl.dlopen(out)
end

mutable struct CnlsModel{T<:Float64}
    handle::Ptr{Cvoid}
    lib::Ptr{Cvoid}                  # C_NULL: stock library; else the library of a user family (compile_family)
    family::Symbol
    nb_parameters::Int
    nb_residuals::Int
    nb_eqcons::Int
    nb_constraints::Int
    lmax::Int
    starting_point::Matrix{T}        # n x B  (column b = problem b; column major == the ABI's [B,n] row major)
    x_low::Vector{T}
    x_upp::Vector{T}
    jacobian::Symbol                 # :analytic | :forward_diff  (cnls_model.jl:65-82)
    status_code::Vector{Cint}
    exit_code::Vector{Cint}
    sol::Matrix{T}
    obj_value::Vector{T}
    iterations::Vector{Cint}
    nb_active::Vector{Cint}
    active::Matrix{Cint}             # lmax x B, 1-based constraint ids of the final working set, 0 padded
    data::Vector{Any}                # the family's data arrays: enlsipb200_set_data with host pointers only RECORDS the pointer
                                     # (the upload happens inside the next solve), so the model must keep the arrays alive
end

"""
    CnlsModel(family, starting_point; data=(), x_low, x_upp, jacobian=:analytic)

`family` is `:hs65` or `:gauss_peaks`; `data` are the family's arrays in slot order
(`:gauss_peaks`: `y` (128 x B) and `S` (B)).  Mirrors the assertions of cnls_model.jl:363-369.
"""
function CnlsModel(family::Symbol, starting_point::Matrix{Float64}; kwargs...)
    fam = family === :hs65 ? FAMILY_HS65 : family === :gauss_peaks ? FAMILY_GAUSS_PEAKS :
          error("A device problem family must be provided")
    return CnlsModel(C_NULL, fam, family, starting_point; kwargs...)
end
# user family: `lib` comes from compile_family; without jacobian_* the engine differentiates by forward differences
CnlsModel(lib::Ptr{Cvoid}, starting_point::Matrix{Float64}; jacobian::Symbol=:forward_diff, kwargs...) =
    CnlsModel(lib, FAMILY_USER, :user, starting_point; jacobian=jacobian, kwargs...)

function CnlsModel(lib::Ptr{Cvoid}, fam::Cint, family::Symbol, starting_point::Matrix{Float64}; data=(),
                   x_low=fill(-Inf, size(starting_point, 1)), x_upp=fill(Inf, size(starting_point, 1)),
                   jacobian::Symbol=:analytic, device::Integer=-1)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall(fsym(lib, :enlsipb200_create), Cint, (Cint, Ptr{Cdouble}, Ptr{Cdouble}, Cint, Ptr{Ptr{Cvoid}}),
                fam, x_low, x_upp, Cint(device), h))
    n, m, q, l, lmax = Ref{Cint}(0), Ref{Cint}(0), Ref{Cint}(0), Ref{Cint}(0), Ref{Cint}(0)
    check(ccall(fsym(lib, :enlsipb200_dims), Cint, (Ptr{Cvoid}, Ptr{Cint}, Ptr{Cint}, Ptr{Cint}, Ptr{Cint}, Ptr{Cint}),
                h[], n, m, q, l, lmax))
    @assert size(starting_point, 1) == n[] "starting_point must be n x B"
    B = size(starting_point, 2)
    kept = Any[arr for arr in data]
    for (slot, arr) in enumerate(kept)
        check(ccall(fsym(lib, :enlsipb200_set_data), Cint, (Ptr{Cvoid}, Cint, Ptr{Cdouble}, Clonglong, Cint, Ptr{Cvoid}),
                    h[], Cint(slot - 1), arr, length(arr), Cint(0), C_NULL))
    end
    model = CnlsModel{Float64}(h[], lib, family, n[], m[], q[], l[], lmax[], starting_point, x_low, x_upp, jacobian,
                               zeros(Cint, B), zeros(Cint, B), copy(starting_point), fill(NaN, B), zeros(Cint, B),
                               zeros(Cint, B), zeros(Cint, lmax[], B), kept)
    finalizer(m -> ccall(fsym(m.lib, :enlsipb200_destroy), Cint, (Ptr{Cvoid},), m.handle), model)
    return model
end

"""
    solve!(model; silent=true, max_iter=100, scaling=false, time_limit=1e3, abs_tol=eps(), rel_tol=√abs_tol,
           c_tol=rel_tol, x_tol=rel_tol)

Same keyword arguments and defaults as the reference (solver.jl:62-63); fills `status_code`, `sol`,
`obj_value` like solver.jl:84-87 and returns `nothing`.
"""
function solve!(model::CnlsModel; silent::Bool=true, max_iter::Int=100, scaling::Bool=false, time_limit::Float64=1e3,
                abs_tol::Float64=eps(Float64), rel_tol::Float64=sqrt(abs_tol), c_tol::Float64=rel_tol, x_tol::Float64=rel_tol)
    B = size(model.starting_point, 2)
    opt = Ref(Options(max_iter, scaling, model.jacobian === :forward_diff ? JAC_FORWARD_DIFF : JAC_ANALYTIC, 0,
                      time_limit, abs_tol, rel_tol, c_tol, x_tol))
    data = model.data
    GC.@preserve data begin          # the recorded host pointers of the data slots are read inside this call
        check(ccall(fsym(model.lib, :enlsipb200_solve_batch), Cint,
                    (Ptr{Cvoid}, Clonglong, Ptr{Cdouble}, Ptr{Options}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cint}, Ptr{Cint}, Ptr{Cint},
                     Ptr{Cint}, Ptr{Cint}, Ptr{Cint}, Ptr{Cdouble}, Cint, Cint, Ptr{Cvoid}),
                    model.handle, B, model.starting_point, opt, model.sol, model.obj_value, model.exit_code, model.status_code,
                    model.iterations, model.nb_active, model.active, C_NULL, C_NULL, Cint(0), Cint(0), C_NULL))
    end
    silent || println("solved $B problems: ", count(==(1), model.status_code), " converged")
    return
end

status(model::CnlsModel) = [dict_status_codes[Int(c)] for c in model.status_code]     # cnls_model.jl:206
solution(model::CnlsModel) = model.sol                                                # cnls_model.jl:213
sum_sq_residuals(model::CnlsModel) = model.obj_value                                  # cnls_model.jl:221
total_nb_constraints(model::CnlsModel) = model.nb_constraints                         # cnls_model.jl:238

# ---------------------------------------------------------------------------------------------------
# Large-Jacobian regime (one problem, m >> n; include/enlsip_b200.h, "Large-Jacobian regime"):
# the same `solve!` / `status` / `solution` / `sum_sq_residuals` surface for B = 1.
# ---------------------------------------------------------------------------------------------------
const FAMILY_SINGLE_INDEX = Cint(16)
const FAMILY_LARGE_CHAINED_ROSENBROCK = Cint(17)
const LARGE_FACTOR_TSQR = Cint(0x100)      # OR-ed into the family of a row family: TSQR of [J | r], row sharding
const LARGE_MIDSIZE = Cint(0x200)          # OR-ed into the family of a row family with n + m < 1000: Newton steps (EF:2658)

"""
    large_compile_family(source; m, nb_eqcons=0, nb_ineqcons=0, has_jacobians=false) -> library handle

User problems of the large regime (n + m >= 1000, or smaller with m >= n + 1 and Newton steps): `source` defines `enl_user::residual` / `enl_user::constraint` as
templates over a point accessor (and optionally `jac_residual` / `jac_constraint`), see include/enlsip_b200.h.  Pass the
handle to `LargeCnlsModel(lib, starting_point; m=..., nb_eqcons=..., nb_ineqcons=..., data=(...))`.
"""
function large_compile_family(source::String; m::Integer, nb_eqcons::Integer=0, nb_ineqcons::Integer=0,
                              has_jacobians::Bool=false, work_dir::String=mktempdir(),
                              out::String=joinpath(work_dir, "libenlsip_b200_large_user.so"))
    check(ccall((:enlsipb200_large_compile_family, libenlsip), Cint,
                (Cstring, Clonglong, Cint, Cint, Cint, Cstring, Cstring),
                source, m, nb_eqcons, nb_ineqcons, has_jacobians ? 1 : 0, out, work_dir))
    return Libdl.dlopen(out)
end

mutable struct LargeCnlsModel{T<:AbstractFloat}
    handle::Ptr{Cvoid}
    lib::Ptr{Cvoid}                 # C_NULL: stock library; else the library of a user row family
    jacobian::Symbol                # :analytic | :forward_diff (general row families)
    nb_parameters::Int
    nb_residuals::Int               # global m (all row shards)
    nb_eqcons::Int
    nb_constraints::Int
    starting_point::Vector{T}
    status_code::Base.RefValue{Cint}
    exit_code::Base.RefValue{Cint}
    sol::Vector{T}
    obj_value::Base.RefValue{T}
    iterations::Base.RefValue{Cint}
    nb_active::Base.RefValue{Cint}
    active::Vector{Cint}
end

"""
    LargeCnlsModel(:single_index, starting_point; W, y, rho, ineq=false, x_low, x_upp, m_global=size(W,2))

`W` is `n x rows` (column major = the ABI's row-major `[rows, n]`), `y` has `rows` entries: the rows held by THIS
process (a row shard when `m_global > rows`).  Constraints: `rho[k]` for the k-th block of 4 parameters
(equalities, or inequalities with `ineq=true`), plus finite bounds -- ordered as cnls_model.jl:402-403.
"""
function LargeCnlsModel(family::Symbol, starting_point::Vector{Float64}; W::Matrix{Float64}, y::Vector{Float64},
                        rho::Vector{Float64}, ineq::Bool=false, x_low=fill(-Inf, length(starting_point)),
                        x_upp=fill(Inf, length(starting_point)), m_global::Integer=size(W, 2), device::Integer=-1)
    family === :single_index || error("A device problem family must be provided")
    n, rows = length(starting_point), size(W, 2)
    @assert size(W, 1) == n && length(y) == rows "W must be n x rows and y of length rows"
    h = Ref{Ptr{Cvoid}}(C_NULL)
    checkl(ccall((:enlsipb200_large_create, libenlsip), Cint,
                 (Cint, Cint, Clonglong, Clonglong, Cint, Cint, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Cint, Ptr{Ptr{Cvoid}}),
                 FAMILY_SINGLE_INDEX, n, rows, m_global, length(rho), ineq, rho, x_low, x_upp, Cint(device), h))
    for (slot, arr) in ((0, W), (1, y))
        checkl(ccall((:enlsipb200_large_set_data, libenlsip), Cint, (Ptr{Cvoid}, Cint, Ptr{Cdouble}, Clonglong, Cint),
                     h[], Cint(slot), arr, length(arr), Cint(0)))
    end
    l = length(rho) + count(isfinite, x_low) + count(isfinite, x_upp)
    model = LargeCnlsModel{Float64}(h[], C_NULL, :analytic, n, m_global, ineq ? 0 : length(rho), l, starting_point, Ref(Cint(0)),
                                    Ref(Cint(0)), copy(starting_point), Ref(NaN), Ref(Cint(0)), Ref(Cint(0)), zeros(Cint, max(l, 1)))
    finalizer(m -> ccall((:enlsipb200_large_destroy, libenlsip), Cint, (Ptr{Cvoid},), m.handle), model)
    return model
end

"""
    LargeCnlsModel(:chained_rosenbrock, starting_point; x_low, x_upp, jacobian=:analytic, factor=:householder, shard=nothing)
    LargeCnlsModel(lib, starting_point; m, nb_eqcons=0, nb_ineqcons=0, data=(), x_low, x_upp, jacobian=:forward_diff,
                   factor=:householder, shard=nothing)

General row families: the reference's own chained Rosenbrock test (test/problems/chained_rosenbrock.jl, any n; the
reference runs n = 1000), or a user family compiled by `large_compile_family`.  `data`: up to two Float64 arrays
handed to the family's functions (copied to the device here; whole on every rank).  `factor=:tsqr` compresses [J | r]
with the tall-skinny QR (LARGE_FACTOR_TSQR); with it, `shard=(rank, nranks)` gives this process the rows of
`shard_rows(m, rank, nranks)`, after which every rank calls `join!`.  With n + m < 1000 the problem is solved with
Newton steps, as the reference decides by size (EF:2658; LARGE_MIDSIZE); such a problem takes neither `factor=:tsqr`
nor `shard`.
"""
function LargeCnlsModel(family::Symbol, starting_point::Vector{Float64}; x_low=fill(-Inf, length(starting_point)),
                        x_upp=fill(Inf, length(starting_point)), jacobian::Symbol=:analytic, device::Integer=-1,
                        factor::Symbol=:householder, shard=nothing)
    family === :chained_rosenbrock || error("row families: :chained_rosenbrock, or a library from large_compile_family")
    n = length(starting_point)
    return _row_family_model(C_NULL, FAMILY_LARGE_CHAINED_ROSENBROCK, starting_point, 2 * (n - 1), n - 2, 0, (), x_low, x_upp,
                             jacobian, device, factor, shard)
end
LargeCnlsModel(lib::Ptr{Cvoid}, starting_point::Vector{Float64}; m::Integer, nb_eqcons::Integer=0, nb_ineqcons::Integer=0,
               data=(), x_low=fill(-Inf, length(starting_point)), x_upp=fill(Inf, length(starting_point)),
               jacobian::Symbol=:forward_diff, device::Integer=-1, factor::Symbol=:householder, shard=nothing) =
    _row_family_model(lib, FAMILY_USER, starting_point, m, nb_eqcons, nb_ineqcons, data, x_low, x_upp, jacobian, device,
                      factor, shard)

"Rows (row0, rows) of `rank` among `nranks` shards of m rows: multiples of 256 (one level-0 TSQR subtile), the last rank takes the remainder."
function shard_rows(m::Integer, rank::Integer, nranks::Integer)
    0 <= rank < nranks || error("shard must be (rank, nranks) with 0 <= rank < nranks")
    chunk = max(256, div(div(m, nranks), 256) * 256)
    row0 = min(rank * chunk, m)
    return row0, rank == nranks - 1 ? m - row0 : min(chunk, m - row0)
end

function _row_family_model(lib, fam, starting_point, m, q, ni, data, x_low, x_upp, jacobian, device, factor=:householder,
                           shard=nothing)
    factor in (:householder, :tsqr) || error("factor must be :householder or :tsqr")
    shard === nothing || factor === :tsqr || error("shard=(rank, nranks) needs factor=:tsqr")
    n = length(starting_point)
    midsize = n + m < 1000      # second_derivatives of the reference (EF:2658)
    midsize && (factor === :tsqr || shard !== nothing) && error("n + m < 1000 (Newton steps): neither factor=:tsqr nor shard")
    rows = shard === nothing ? m : shard_rows(m, shard...)[2]
    flag = (factor === :tsqr ? LARGE_FACTOR_TSQR : Cint(0)) | (midsize ? LARGE_MIDSIZE : Cint(0))
    h = Ref{Ptr{Cvoid}}(C_NULL)
    checkl(ccall(fsym(lib, :enlsipb200_large_create), Cint,
                 (Cint, Cint, Clonglong, Clonglong, Cint, Cint, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Cint, Ptr{Ptr{Cvoid}}),
                 fam | flag, n, rows, m, 0, 0, C_NULL, x_low, x_upp, Cint(device), h))
    for (slot, arr) in enumerate(data)      # copied host -> device inside the call: nothing to keep alive
        checkl(ccall(fsym(lib, :enlsipb200_large_set_data), Cint, (Ptr{Cvoid}, Cint, Ptr{Cdouble}, Clonglong, Cint),
                     h[], Cint(slot - 1), arr, length(arr), Cint(0)))
    end
    l = q + ni + count(isfinite, x_low) + count(isfinite, x_upp)
    model = LargeCnlsModel{Float64}(h[], lib, jacobian, n, m, q, l, starting_point, Ref(Cint(0)), Ref(Cint(0)),
                                    copy(starting_point), Ref(NaN), Ref(Cint(0)), Ref(Cint(0)), zeros(Cint, max(l, 1)))
    finalizer(mm -> ccall(fsym(mm.lib, :enlsipb200_large_destroy), Cint, (Ptr{Cvoid},), mm.handle), model)
    return model
end

checkl(rc) = rc == 0 ? nothing :
    error("enlsip_b200 (large regime) error $rc: ", unsafe_string(ccall((:enlsipb200_large_last_error, libenlsip), Cstring, ())))

"Join the row shards of `nranks` processes (one per GPU): `id` is the 128-byte NCCL id made by rank 0 (`large_comm_id()`), distributed by the caller (MPI.jl / Distributed)."
large_comm_id() = (id = zeros(UInt8, 128); checkl(ccall((:enlsipb200_large_comm_id, libenlsip), Cint, (Ptr{UInt8},), id)); id)
join!(model::LargeCnlsModel, id::Vector{UInt8}, rank::Integer, nranks::Integer) =
    checkl(ccall((:enlsipb200_large_comm_init, libenlsip), Cint, (Ptr{Cvoid}, Ptr{UInt8}, Cint, Cint), model.handle, id, rank, nranks))

function solve!(model::LargeCnlsModel; silent::Bool=true, max_iter::Int=100, scaling::Bool=false, time_limit::Float64=1e3,
                abs_tol::Float64=eps(Float64), rel_tol::Float64=sqrt(abs_tol), c_tol::Float64=rel_tol, x_tol::Float64=rel_tol)
    opt = Ref(Options(max_iter, scaling, model.jacobian === :forward_diff ? JAC_FORWARD_DIFF : JAC_ANALYTIC, 0, time_limit,
                      abs_tol, rel_tol, c_tol, x_tol))
    checkl(ccall(fsym(model.lib, :enlsipb200_large_solve), Cint,
                 (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Options}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cint}, Ptr{Cint}, Ptr{Cint}, Ptr{Cint},
                  Ptr{Cint}, Ptr{Cdouble}, Cint),
                 model.handle, model.starting_point, opt, model.sol, model.obj_value, model.exit_code, model.status_code,
                 model.iterations, model.nb_active, model.active, C_NULL, Cint(0)))
    silent || println("exit code ", model.exit_code[], " after ", model.iterations[], " iterations")
    return
end

status(model::LargeCnlsModel) = dict_status_codes[Int(model.status_code[])]
solution(model::LargeCnlsModel) = model.sol
sum_sq_residuals(model::LargeCnlsModel) = model.obj_value[]
total_nb_constraints(model::LargeCnlsModel) = model.nb_constraints

end # module
