# IsingModelB200.jl — Julia host side of libising_b200.so.  Keeps the reference's module, type and method names
# (src/IsingModel.jl:3-15) so that user code written for Wandao123/IsingModel.jl — its own test/runtests.jl
# included — runs unchanged; only the arithmetic moves behind `ccall`.
#
#   using IsingModelB200                       # instead of `using IsingModel`
#   ss = SpinSystems.SpinSystem(s, J, h)       # src/SpinSystems.jl:19-51 (same checks, warnings, errors)
#   ua = SingleSpinFlip.GlauberDynamics(deepcopy(ss), T)
#   SingleSpinFlip.update!(ua, node, fluct)    # src/SingleSpinFlip.jl:46-55, one isb_ssf_run call
#   for ua in SamplingHelper.makeSampler!(ua, n; annealingSchedule, rng) ... end
#
# No julia binary exists in the build image: this file is checked statically (tests/test_julia_shim.py: every ccall
# signature against include/ising_b200.h, the constants against the header's enums, the presence of every reference
# method) and the same C ABI is exercised from C (tests/c_abi_replay.c) and from Python ctypes in tests/.
#
# How the reference's mutable-struct semantics are kept on top of device-resident state
#   * `ss.spinConfiguration` (and `hiddenLayer`) are ordinary host arrays, as in the reference.  The device copy is
#     tracked by a shadow (`_dev`, what the device holds).  Before every device operation the host array is compared
#     with the shadow and pushed when it differs — so assignments (`setproperty!`), the five setters
#     (src/SpinSystems.jl:62-66,129-137) and even in-place writes `ss.spinConfiguration[i] = -1` all reach the device.
#   * `ss.couplingCoefficients = J`, `ss.externalMagneticField = h`, `ss.auxiliaryBias = b` rebuild the device model.
#   * `deepcopy(ss)` gives an independent ensemble on the shared immutable model (isb_model_retain + isb_ens_clone):
#     test/runtests.jl:22-24,30-31 copy one system into several algorithms.
#   * finalizers release the ensemble and the model (handles are reference counted inside the library).
#
# Extension: `spinConfiguration` may be an N x R matrix (R replicas, one per column).
module IsingModelB200

export SpinSystems, SingleSpinFlip, MultiSpinFlip, OnBipartiteGraph, SamplingHelper

@enum IsingSpin DownSpin = -1 UpSpin = +1     # src/IsingModel.jl:9

const libisb = get(ENV, "ISING_B200_LIB", joinpath(@__DIR__, "..", "libising_b200.so"))

# ------------------------------------------------------------------ raw C ABI (include/ising_b200.h)
module CABI
import ..libisb
const Ctx = Ptr{Cvoid}; const Model = Ptr{Cvoid}; const Ens = Ptr{Cvoid}
const RULE_HOPFIELD, RULE_GLAUBER, RULE_METROPOLIS = Cint(0), Cint(1), Cint(2)
const BIP_SCA, BIP_MA = Cint(0), Cint(1)
const ORDER_SEQUENTIAL, ORDER_LIST, ORDER_RANDOM, ORDER_CHECKERBOARD = Cint(0), Cint(1), Cint(2), Cint(3)
const FLUCT_PHILOX, FLUCT_SHARED, FLUCT_PER_REPLICA = Cint(0), Cint(1), Cint(2)
const PREC_F64, PREC_F32, PREC_AUTO, PREC_BF16X3, PREC_BF16X1, PREC_BF16X2 = Cint(0), Cint(1), Cint(2), Cint(3), Cint(4), Cint(5)
const PREC_FP16X2, PREC_FP16X1 = Cint(6), Cint(7)
const PREC_I8X3, PREC_I8X2, PREC_I8X4 = Cint(8), Cint(9), Cint(10)

lasterror(ctx) = unsafe_string(ccall((:isb_last_error, libisb), Cstring, (Ctx,), ctx))
check(rc, ctx) = rc == 0 ? nothing : error(lasterror(ctx))

function create(device::Integer)
    h = Ref{Ctx}(C_NULL)
    rc = ccall((:isb_create, libisb), Cint, (Cint, Ref{Ctx}), device, h)
    rc == 0 || error(lasterror(C_NULL))
    h[]
end
const _ctx = Ref{Ctx}(C_NULL)
context() = (_ctx[] == C_NULL && (_ctx[] = create(parse(Int, get(ENV, "LOCAL_RANK", "0")))); _ctx[])

function model_dense(J::Matrix{Float64}, h::Vector{Float64}; prec = PREC_AUTO)
    m = Ref{Model}(C_NULL); w = Ref{Cint}(0)
    check(ccall((:isb_model_dense, libisb), Cint,
                (Ctx, Cint, Ptr{Float64}, Int64, Ptr{Float64}, Cint, Ref{Cint}, Ref{Model}),
                context(), size(J, 1), J, stride(J, 2), h, prec, w, m), context())
    m[]
end
# SparseMatrixCSC couplings (what the reference's tests and demo pass) stay sparse: 0-based CSC across the ABI
function model_sparse(n::Integer, colptr::Vector{Int64}, rowval::Vector{Int32}, nzval::Vector{Float64}, h::Vector{Float64})
    m = Ref{Model}(C_NULL); w = Ref{Cint}(0)
    check(ccall((:isb_model_sparse, libisb), Cint,
                (Ctx, Cint, Ptr{Int64}, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}, Ref{Cint}, Ref{Model}),
                context(), n, colptr, rowval, nzval, h, w, m), context())
    m[]
end
function model_bipartite(W::Matrix{Float64}, h::Vector{Float64}, b::Vector{Float64}; prec = PREC_F64)
    m = Ref{Model}(C_NULL)
    check(ccall((:isb_model_bipartite, libisb), Cint,
                (Ctx, Cint, Cint, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}, Cint, Ref{Model}),
                context(), size(W, 1), size(W, 2), W, stride(W, 2), h, b, prec, m), context())
    m[]
end
model_retain(m::Model) = check(ccall((:isb_model_retain, libisb), Cint, (Model,), m), context())
model_destroy(m::Model) = ccall((:isb_model_destroy, libisb), Cvoid, (Model,), m)
function ensemble(m::Model, R::Integer)
    e = Ref{Ens}(C_NULL)
    check(ccall((:isb_ens_create, libisb), Cint, (Model, Cint, Ref{Ens}), m, R, e), context())
    e[]
end
function ens_clone(src::Ens)
    e = Ref{Ens}(C_NULL)
    check(ccall((:isb_ens_clone, libisb), Cint, (Ens, Ref{Ens}), src, e), context())
    e[]
end
ens_destroy(e::Ens) = ccall((:isb_ens_destroy, libisb), Cvoid, (Ens,), e)
# spins cross the ABI as Int8, one replica per column of an N x R matrix (== [R][ld] replica-major in C)
set_spins!(e, S::Matrix{Int8}) = check(ccall((:isb_ens_set_spins, libisb), Cint, (Ens, Ptr{Int8}, Int64), e, S, stride(S, 2)), context())
get_spins!(e, S::Matrix{Int8}) = (check(ccall((:isb_ens_get_spins, libisb), Cint, (Ens, Ptr{Int8}, Int64), e, S, stride(S, 2)), context()); S)
set_hidden!(e, S::Matrix{Int8}) = check(ccall((:isb_ens_set_hidden, libisb), Cint, (Ens, Ptr{Int8}, Int64), e, S, stride(S, 2)), context())
get_hidden!(e, S::Matrix{Int8}) = (check(ccall((:isb_ens_get_hidden, libisb), Cint, (Ens, Ptr{Int8}, Int64), e, S, stride(S, 2)), context()); S)
energy(e, R) = (E = Vector{Float64}(undef, R); check(ccall((:isb_ens_energy, libisb), Cint, (Ens, Ptr{Float64}), e, E), context()); E)
function local_field(e, n, R)
    F = Matrix{Float64}(undef, n, R)
    check(ccall((:isb_ens_local_field, libisb), Cint, (Ens, Ptr{Float64}, Int64), e, F, n), context()); F
end
function local_aux_bias(e, n, R)
    F = Matrix{Float64}(undef, n, R)
    check(ccall((:isb_ens_local_aux_bias, libisb), Cint, (Ens, Ptr{Float64}, Int64), e, F, n), context()); F
end
_optr(::Nothing, T) = Ptr{T}(C_NULL)
_optr(a::Array, T) = a
# nodes are 1-based on the Julia side, 0-based across the ABI.  With `snap` (an N x R x ntr Int8 array) the call is
# isb_ssf_run_snap: the state after every `trace_every`-th step is recorded (and its energy into `E`, R x ntr).
# `checkerboard = true` (periodic L x L lattices given as sparse J): ISB_ORDER_CHECKERBOARD, `start` = first position of the
# two-colour sweep order.
function ssf_run!(e, rule, nsteps; nodes = nothing, start = 1, fluct = nothing, per_replica = false, seed = 0,
                  step_offset = 0, T = Float64[], steps_per_T = 1, trace_every = 0, E = nothing, snap = nothing,
                  checkerboard = false)
    n0 = nodes === nothing ? nothing : Vector{Int32}(nodes .- 1)
    order = nodes === nothing ? (checkerboard ? ORDER_CHECKERBOARD : ORDER_SEQUENTIAL) : ORDER_LIST
    mode = fluct === nothing ? FLUCT_PHILOX : (per_replica ? FLUCT_PER_REPLICA : FLUCT_SHARED)
    f = fluct === nothing ? nothing : Vector{Float64}(vec(fluct))
    Tv = Vector{Float64}(T)
    if snap === nothing
        check(ccall((:isb_ssf_run, libisb), Cint,
                    (Ens, Cint, Int64, Cint, Ptr{Int32}, Cint, Cint, Ptr{Float64}, UInt64, UInt64, Ptr{Float64}, Int64,
                     Int64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}),
                    e, rule, nsteps, order, _optr(n0, Int32), start - 1, mode, _optr(f, Float64), seed, step_offset, Tv,
                    length(Tv), steps_per_T, trace_every, _optr(E, Float64), C_NULL, C_NULL), context())
    else
        check(ccall((:isb_ssf_run_snap, libisb), Cint,
                    (Ens, Cint, Int64, Cint, Ptr{Int32}, Cint, Cint, Ptr{Float64}, UInt64, UInt64, Ptr{Float64}, Int64,
                     Int64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Int8}, Int64),
                    e, rule, nsteps, order, _optr(n0, Int32), start - 1, mode, _optr(f, Float64), seed, step_offset, Tv,
                    length(Tv), steps_per_T, trace_every, _optr(E, Float64), C_NULL, C_NULL, snap, size(snap, 1)), context())
    end
end
# Parallel tempering with the round loop inside the library (isb_ssf_run_pt).  `level_of` (Vector{Int32}, one 0-based
# level per replica, replica = ladder * length(levels) + slot) is updated in place.  E / M: levels x ladders x rounds
# (column-major == the ABI's [rounds][levels][ladders]), Q: levels x ladders/2 x rounds, accepted: levels - 1, flips: R.
function ssf_run_pt!(e, rule, levels, rounds, steps_per_round, level_of::Vector{Int32}; order = ORDER_SEQUENTIAL,
                     start = 1, seed = 0, step_offset = 0, round_offset = 0, E = nothing, M = nothing, Q = nothing,
                     accepted = nothing, flips = nothing)
    lv = Vector{Float64}(levels)
    check(ccall((:isb_ssf_run_pt, libisb), Cint,
                (Ens, Cint, Cint, Ptr{Float64}, Int64, Int64, Cint, Cint, UInt64, UInt64, UInt64, Ptr{Int32},
                 Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Int64}),
                e, rule, length(lv), lv, rounds, steps_per_round, order, start - 1, seed, step_offset, round_offset,
                level_of, _optr(E, Float64), _optr(M, Float64), _optr(Q, Float64), _optr(accepted, Int64),
                _optr(flips, Int64)), context())
    level_of
end
# Replica r takes the state of replica src[r] (1-based on the Julia side, 0-based across the ABI), spins and cached
# fields bit for bit (isb_ens_select_replicas).
function select_replicas!(e, src)
    s0 = Vector{Int32}(src .- 1)
    check(ccall((:isb_ens_select_replicas, libisb), Cint, (Ens, Ptr{Int32}), e, s0), context())
    e
end
# Population annealing with the temperature loop inside the library (isb_ssf_run_pa): R = n_pop * P replicas,
# population p = replicas p*P+1 .. (p+1)*P.  `family` (Vector{Int32} labels or nothing) is updated in place.
# E / M: R x nT (column-major == the ABI's [nT][R]), lnQ: n_pop x (nT - 1 + (T_next > 0)), flips: R.
function ssf_run_pa!(e, rule, n_pop, T, steps_per_T; T_next = 0.0, order = ORDER_SEQUENTIAL, start = 1, seed = 0,
                     step_offset = 0, T_offset = 0, family = nothing, E = nothing, M = nothing, lnQ = nothing,
                     flips = nothing)
    Tv = Vector{Float64}(T)
    check(ccall((:isb_ssf_run_pa, libisb), Cint,
                (Ens, Cint, Cint, Int64, Ptr{Float64}, Float64, Int64, Cint, Cint, UInt64, UInt64, UInt64, Ptr{Int32},
                 Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}),
                e, rule, n_pop, length(Tv), Tv, T_next, steps_per_T, order, start - 1, seed, step_offset, T_offset,
                _optr(family, Int32), _optr(E, Float64), _optr(M, Float64), _optr(lnQ, Float64), _optr(flips, Int64)),
          context())
    family
end
# Fv / Fh: (units, steps) column-major == [steps][units].  With snapV / snapH (units x R x ntr Int8) the call is
# isb_bip_run_snap.
function bip_run!(e, rule, nsteps; Fv = nothing, Fh = nothing, per_replica = false, seed = 0, step_offset = 0,
                  T = Float64[], steps_per_T = 1, trace_every = 0, E = nothing, snapV = nothing, snapH = nothing)
    mode = Fv === nothing ? FLUCT_PHILOX : (per_replica ? FLUCT_PER_REPLICA : FLUCT_SHARED)
    fv = Fv === nothing ? nothing : Vector{Float64}(vec(Fv))
    fh = Fh === nothing ? nothing : Vector{Float64}(vec(Fh))
    Tv = Vector{Float64}(T)
    if snapV === nothing && snapH === nothing
        check(ccall((:isb_bip_run, libisb), Cint,
                    (Ens, Cint, Int64, Cint, Ptr{Float64}, Ptr{Float64}, UInt64, UInt64, Ptr{Float64}, Int64, Int64,
                     Int64, Ptr{Float64}),
                    e, rule, nsteps, mode, _optr(fv, Float64), _optr(fh, Float64), seed, step_offset, Tv, length(Tv),
                    steps_per_T, trace_every, _optr(E, Float64)), context())
    else
        check(ccall((:isb_bip_run_snap, libisb), Cint,
                    (Ens, Cint, Int64, Cint, Ptr{Float64}, Ptr{Float64}, UInt64, UInt64, Ptr{Float64}, Int64, Int64,
                     Int64, Ptr{Float64}, Ptr{Int8}, Int64, Ptr{Int8}, Int64),
                    e, rule, nsteps, mode, _optr(fv, Float64), _optr(fh, Float64), seed, step_offset, Tv, length(Tv),
                    steps_per_T, trace_every, _optr(E, Float64), snapV, size(snapV, 1), snapH, size(snapH, 1)), context())
    end
end
# ---- row-sharded synchronous SCA (BASELINE config 5): one process per GPU, the step loop inside the library
const ShardRun = Ptr{Cvoid}
const EXCH_LOCAL, EXCH_NCCL, EXCH_COPY = Cint(0), Cint(1), Cint(2)
function shard_model_sk(n::Integer, n_blocks::Integer, block::Integer, seed::Integer, q::Real; prec = PREC_I8X3)
    m = Ref{Model}(C_NULL)
    check(ccall((:isb_shard_model_sk, libisb), Cint, (Ctx, Cint, Cint, Cint, UInt64, Float64, Cint, Ref{Model}),
                context(), n, n_blocks, block, seed, q, prec, m), context())
    m[]
end
# Wrows: the rows [block nb + 1, (block + 1) nb] of the symmetric W as an n x nb Julia matrix (column r = row r of the
# block: the C side reads [nb][n] row-major); wmax = largest off-diagonal |W| of the WHOLE matrix (int8 planes)
function shard_model_rows(n::Integer, n_blocks::Integer, block::Integer, Wrows::Matrix{Float64}, h_blk::Vector{Float64},
                          b_blk::Vector{Float64}; prec = PREC_I8X3, wmax = 0.0)
    m = Ref{Model}(C_NULL)
    check(ccall((:isb_shard_model_rows_q, libisb), Cint,
                (Ctx, Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Cint, Float64, Ref{Model}),
                context(), n, n_blocks, block, Wrows, h_blk, b_blk, prec, wmax, m), context())
    m[]
end
function shard_run_create(m::Model, R::Integer, exchange::Cint)
    s = Ref{ShardRun}(C_NULL)
    check(ccall((:isb_shard_run_create, libisb), Cint, (Model, Cint, Cint, Ref{ShardRun}), m, R, exchange, s), context())
    s[]
end
shard_run_destroy(s::ShardRun) = ccall((:isb_shard_run_destroy, libisb), Cvoid, (ShardRun,), s)
nccl_unique_id() = (id = Vector{UInt8}(undef, 128); check(ccall((:isb_nccl_unique_id, libisb), Cint, (Ptr{UInt8},), id), C_NULL); id)
shard_run_init_nccl(s::ShardRun, id::Vector{UInt8}) = check(ccall((:isb_shard_run_init_nccl, libisb), Cint, (ShardRun, Ptr{UInt8}), s, id), context())
shard_run_set_nccl_comm(s::ShardRun, comm::Ptr{Cvoid}) = check(ccall((:isb_shard_run_set_nccl_comm, libisb), Cint, (ShardRun, Ptr{Cvoid}), s, comm), context())
shard_run_ipc_export(s::ShardRun) = (h = Vector{UInt8}(undef, 64); check(ccall((:isb_shard_run_ipc_export, libisb), Cint, (ShardRun, Ptr{UInt8}), s, h), context()); h)
shard_run_ipc_import(s::ShardRun, rank::Integer, h::Vector{UInt8}) = check(ccall((:isb_shard_run_ipc_import, libisb), Cint, (ShardRun, Cint, Ptr{UInt8}), s, rank, h), context())
shard_run_barrier(s::ShardRun) = check(ccall((:isb_shard_run_barrier, libisb), Cint, (ShardRun,), s), context())
shard_run_set_spins!(s::ShardRun, S::Matrix{Int8}) = check(ccall((:isb_shard_run_set_spins, libisb), Cint, (ShardRun, Ptr{Int8}, Int64), s, S, stride(S, 2)), context())
shard_run_get_spins!(s::ShardRun, layer::Integer, S::Matrix{Int8}) = (check(ccall((:isb_shard_run_get_spins, libisb), Cint, (ShardRun, Cint, Ptr{Int8}, Int64), s, layer, S, stride(S, 2)), context()); S)
shard_run_steps!(s::ShardRun, rule::Cint, nsteps::Integer, T::Vector{Float64}; seed = 0, step_offset = 0) =
    check(ccall((:isb_shard_run_steps, libisb), Cint, (ShardRun, Cint, Int64, Ptr{Float64}, Int64, UInt64, UInt64),
                s, rule, nsteps, T, length(T), seed, step_offset), context())
end # module CABI

# ------------------------------------------------------------------ SpinSystems (src/SpinSystems.jl)
module SpinSystems
export SpinSystem, UpdatingAlgorithm, getSpinConfiguration, getCouplingCoefficients, getExternalMagneticField
export calcEnergy, calcLocalMagneticField, SpinSystemOnBipartiteGraph, UpdatingAlgorithmOnBipartiteGraph
export getHiddenLayer, getAuxiliaryBias, calcLocalAuxiliaryBias
using LinearAlgebra
using SparseArrays
import ..CABI

_int8(a) = Matrix{Int8}(reshape(a, size(a, 1), :))
_like(a, S::Matrix{Int8}, T) = ndims(a) == 1 ? Vector{T}(vec(S)) : Matrix{T}(S)

mutable struct SpinSystem
    spinConfiguration::AbstractVecOrMat{<:Number}
    couplingCoefficients::AbstractMatrix{<:AbstractFloat}
    externalMagneticField::AbstractVector{<:AbstractFloat}
    model::CABI.Model
    ens::CABI.Ens
    _dev::Matrix{Int8}          # what the device ensemble currently holds (N x R)
    function SpinSystem(spinConfiguration, couplingCoefficients, externalMagneticField)
        # the reference's checks, in its order and with its messages (src/SpinSystems.jl:19-49)
        numNodes = size(spinConfiguration, 1)
        (row, column) = size(couplingCoefficients)
        if row != column
            error("The coupling-coefficient matrix is not a square matrix: $(row)rows ≠ $(column)columns.")
        elseif numNodes < row
            @warn "The size of the spin-configuration vector is too smaller than the size of the coupling-coefficient matrix.  The incorresponding components of the coupling-coefficient matrix are ignored."
            couplingCoefficients = couplingCoefficients[1:numNodes, 1:numNodes]
        elseif numNodes > row
            @warn "The size of the spin-configuration vector is too bigger than the size of the coupling-coefficient matrix.  The incorresponding components of the spin-configuration vector are ignored."
            spinConfiguration = ndims(spinConfiguration) == 1 ? spinConfiguration[1:row] : spinConfiguration[1:row, :]
        elseif !issymmetric(couplingCoefficients)
            @warn "The coupling-coefficient matrix should be symmetric.  It is symmetrized by its upper-triangular components automatically."
            couplingCoefficients = Symmetric(couplingCoefficients, :U)
        end
        if any(diag(couplingCoefficients) .!= 0)
            @warn "The diagonal components of the coupling-coefficient matrix should be zero.  Their non-zero components are ignored."
            couplingCoefficients -= Diagonal(couplingCoefficients)
        end
        numBias = length(externalMagneticField)
        if row != numBias                   # the ORIGINAL row count, as the reference compares (:41)
            error("The size of the coupling-coefficient matrix does not match the size of the external-magnetic-field vector: $(row) ≠ $(numBias).")
        elseif numNodes < numBias
            @warn "The size of the spin-configuration vector is too smaller than the size of the external-magnetic-field vector.  The incorresponding components of the external-magnetic-field vector are ignored."
            externalMagneticField = externalMagneticField[1:numNodes]
        elseif numNodes > numBias
            @warn "The size of the spin-configuration vector is too bigger than the size of the external-magnetic-field vector.  The incorresponding components of the spin-configuration vector are ignored."
            spinConfiguration = ndims(spinConfiguration) == 1 ? spinConfiguration[1:numBias] : spinConfiguration[1:numBias, :]
        end
        J = float.(couplingCoefficients); h = float.(externalMagneticField)
        ss = new(spinConfiguration, J, h, C_NULL, C_NULL, Matrix{Int8}(undef, 0, 0))
        _build!(ss)
        finalizer(_release!, ss)
    end
    # deepcopy: a second object on the same (retained) model with a cloned ensemble
    function SpinSystem(src::SpinSystem, dict::IdDict)
        _sync!(src)
        CABI.model_retain(src.model)
        ss = new(Base.deepcopy_internal(getfield(src, :spinConfiguration), dict),
                 Base.deepcopy_internal(getfield(src, :couplingCoefficients), dict),
                 Base.deepcopy_internal(getfield(src, :externalMagneticField), dict),
                 src.model, CABI.ens_clone(src.ens), copy(getfield(src, :_dev)))
        finalizer(_release!, ss)
    end
end
Base.deepcopy_internal(ss::SpinSystem, dict::IdDict) = haskey(dict, ss) ? dict[ss] : (dict[ss] = SpinSystem(ss, dict))

function _release!(ss)
    e = getfield(ss, :ens); m = getfield(ss, :model)
    e != C_NULL && CABI.ens_destroy(e)
    m != C_NULL && CABI.model_destroy(m)
    setfield!(ss, :ens, convert(CABI.Ens, C_NULL)); setfield!(ss, :model, convert(CABI.Model, C_NULL))
    nothing
end
# (re)build the device model + ensemble from the host fields
function _build!(ss::SpinSystem)
    _release!(ss)
    Jh = getfield(ss, :couplingCoefficients); h = Vector{Float64}(getfield(ss, :externalMagneticField))
    if Jh isa SparseMatrixCSC
        J = SparseMatrixCSC{Float64,Int64}(Jh)
        m = CABI.model_sparse(size(J, 1), J.colptr .- 1, Int32.(J.rowval .- 1), J.nzval, h)
    else
        m = CABI.model_dense(Matrix{Float64}(Jh), h)
    end
    S = _int8(getfield(ss, :spinConfiguration))
    e = CABI.ensemble(m, size(S, 2)); CABI.set_spins!(e, S)
    setfield!(ss, :model, m); setfield!(ss, :ens, e); setfield!(ss, :_dev, S)
    ss
end
# host -> device when the host array no longer equals what the device holds (assignment or in-place writes)
function _sync!(ss::SpinSystem)
    S = _int8(getfield(ss, :spinConfiguration))
    if S != getfield(ss, :_dev)
        CABI.set_spins!(ss.ens, S); setfield!(ss, :_dev, S)
    end
    ss
end
# device -> host after a run; the host array keeps the reference's shape (Vector for one replica) and element type
function _pull!(ss::SpinSystem)
    old = getfield(ss, :spinConfiguration)
    S = CABI.get_spins!(ss.ens, Matrix{Int8}(undef, length(ss.externalMagneticField), size(old, 2)))
    _adopt!(ss, S)
end
# the host array is updated IN PLACE (the reference mutates spinConfiguration[i], src/SingleSpinFlip.jl:32,51,70),
# so references a caller holds to it keep seeing the current state
function _adopt!(ss::SpinSystem, S::AbstractMatrix{Int8}; dev = S)
    old = getfield(ss, :spinConfiguration)
    if size(old, 1) == size(S, 1) && size(old, 2) == size(S, 2)
        old[:] .= vec(S)
    else
        setfield!(ss, :spinConfiguration, _like(old, Matrix{Int8}(S), Int))
    end
    dev === nothing || setfield!(ss, :_dev, Matrix{Int8}(dev))
    ss
end
function Base.setproperty!(ss::SpinSystem, name::Symbol, v)
    if name === :couplingCoefficients || name === :externalMagneticField
        setfield!(ss, name, float.(v)); _build!(ss)      # the couplings / fields live on the device: rebuild
    else
        setfield!(ss, name, convert(fieldtype(SpinSystem, name), v))   # spinConfiguration: pushed by the next _sync!
    end
    v
end

abstract type UpdatingAlgorithm end

getSpinConfiguration(ua::UpdatingAlgorithm) = ua.spinSystem.spinConfiguration
setSpinConfiguration(ua::UpdatingAlgorithm, spinConfiguration::AbstractVecOrMat{<:Number}) = (ua.spinSystem.spinConfiguration = spinConfiguration)
getCouplingCoefficients(ua::UpdatingAlgorithm) = ua.spinSystem.couplingCoefficients
setCouplingCoefficients(ua::UpdatingAlgorithm, couplingCoefficient::AbstractMatrix{<:AbstractFloat}) = (ua.spinSystem.couplingCoefficients = couplingCoefficient)
getExternalMagneticField(ua::UpdatingAlgorithm) = ua.spinSystem.externalMagneticField
setExternalMagneticField(ua::UpdatingAlgorithm, externalMagneticField::AbstractVector{<:AbstractFloat}) = (ua.spinSystem.externalMagneticField = externalMagneticField)
_nrep(ss) = size(getfield(ss, :spinConfiguration), 2)
_scalar(ss, v) = ndims(getfield(ss, :spinConfiguration)) == 1 ? v[1] : v
calcEnergy(ss::SpinSystem) = (_sync!(ss); _scalar(ss, CABI.energy(ss.ens, _nrep(ss))))                  # :68-71
calcEnergy(ua::UpdatingAlgorithm) = calcEnergy(ua.spinSystem)
function calcLocalMagneticField(ss::SpinSystem)                                                          # :75-78
    _sync!(ss)
    F = CABI.local_field(ss.ens, length(ss.externalMagneticField), _nrep(ss))
    ndims(getfield(ss, :spinConfiguration)) == 1 ? vec(F) : F
end
calcLocalMagneticField(ss::SpinSystem, nodeIndex::Integer) =                                            # :80-83
    (_sync!(ss); _scalar(ss, CABI.local_field(ss.ens, length(ss.externalMagneticField), _nrep(ss))[nodeIndex, :]))
calcLocalMagneticField(ua::UpdatingAlgorithm) = calcLocalMagneticField(ua.spinSystem)
calcLocalMagneticField(ua::UpdatingAlgorithm, x::Integer) = calcLocalMagneticField(ua.spinSystem, x)

mutable struct SpinSystemOnBipartiteGraph
    spinConfiguration::AbstractVecOrMat{<:Number}
    hiddenLayer::AbstractVecOrMat{<:Number}
    couplingCoefficients::AbstractMatrix{<:AbstractFloat}
    externalMagneticField::AbstractVector{<:AbstractFloat}
    auxiliaryBias::AbstractVector{<:AbstractFloat}
    model::CABI.Model
    ens::CABI.Ens
    prec::Cint
    _devV::Matrix{Int8}
    _devH::Matrix{Int8}
    function SpinSystemOnBipartiteGraph(spinConfiguration, hiddenLayer, couplingCoefficients, externalMagneticField, auxiliaryBias; prec = CABI.PREC_F64)
        numVisibleNodes = size(spinConfiguration, 1); numHiddenNodes = size(hiddenLayer, 1)              # :97-118
        (row, column) = size(couplingCoefficients)
        if row != numVisibleNodes
            error("The size of the coupling-coefficient matrix does not match the number of visible and hidden nodes: $(numVisibleNodes)nodes ≠ $(row)rows.")
        elseif column != numHiddenNodes
            error("The size of the coupling-coefficient matrix does not match the number of visible and hidden nodes: $(numHiddenNodes)nodes ≠ $(column)columns.")
        end
        numFields = length(externalMagneticField); numBias = length(auxiliaryBias)
        if numFields != numVisibleNodes
            error("The size of the external-magnetic-field vector does not match the number of visible nodes: $(numFields) ≠ $(numVisibleNodes).")
        elseif numBias != numHiddenNodes
            error("The size of the eauxiliary-bias vector does not match the number of hidden nodes: $(numBias) ≠ $(numHiddenNodes).")
        end
        ss = new(spinConfiguration, hiddenLayer, float.(couplingCoefficients), float.(externalMagneticField), float.(auxiliaryBias),
                 C_NULL, C_NULL, prec, Matrix{Int8}(undef, 0, 0), Matrix{Int8}(undef, 0, 0))
        _build!(ss)
        finalizer(_release!, ss)
    end
    function SpinSystemOnBipartiteGraph(src::SpinSystemOnBipartiteGraph, dict::IdDict)
        _sync!(src)
        CABI.model_retain(src.model)
        ss = new(Base.deepcopy_internal(getfield(src, :spinConfiguration), dict),
                 Base.deepcopy_internal(getfield(src, :hiddenLayer), dict),
                 Base.deepcopy_internal(getfield(src, :couplingCoefficients), dict),
                 Base.deepcopy_internal(getfield(src, :externalMagneticField), dict),
                 Base.deepcopy_internal(getfield(src, :auxiliaryBias), dict),
                 src.model, CABI.ens_clone(src.ens), src.prec, copy(getfield(src, :_devV)), copy(getfield(src, :_devH)))
        finalizer(_release!, ss)
    end
end
Base.deepcopy_internal(ss::SpinSystemOnBipartiteGraph, dict::IdDict) =
    haskey(dict, ss) ? dict[ss] : (dict[ss] = SpinSystemOnBipartiteGraph(ss, dict))
function _build!(ss::SpinSystemOnBipartiteGraph)
    _release!(ss)
    m = CABI.model_bipartite(Matrix{Float64}(getfield(ss, :couplingCoefficients)), Vector{Float64}(getfield(ss, :externalMagneticField)),
                             Vector{Float64}(getfield(ss, :auxiliaryBias)); prec = getfield(ss, :prec))
    S = _int8(getfield(ss, :spinConfiguration)); T = _int8(getfield(ss, :hiddenLayer))
    e = CABI.ensemble(m, size(S, 2)); CABI.set_spins!(e, S); CABI.set_hidden!(e, T)
    setfield!(ss, :model, m); setfield!(ss, :ens, e); setfield!(ss, :_devV, S); setfield!(ss, :_devH, T)
    ss
end
function _sync!(ss::SpinSystemOnBipartiteGraph)
    S = _int8(getfield(ss, :spinConfiguration)); T = _int8(getfield(ss, :hiddenLayer))
    S != getfield(ss, :_devV) && (CABI.set_spins!(ss.ens, S); setfield!(ss, :_devV, S))
    T != getfield(ss, :_devH) && (CABI.set_hidden!(ss.ens, T); setfield!(ss, :_devH, T))
    ss
end
function _pull!(ss::SpinSystemOnBipartiteGraph)
    R = _nrep(ss)
    S = CABI.get_spins!(ss.ens, Matrix{Int8}(undef, length(ss.externalMagneticField), R))
    T = CABI.get_hidden!(ss.ens, Matrix{Int8}(undef, length(ss.auxiliaryBias), R))
    _adopt!(ss, S, T)
end
# the reference REPLACES both layers by fresh Vector{Float64} in every update (src/OnBipartiteGraph.jl:35-42)
function _adopt!(ss::SpinSystemOnBipartiteGraph, S::AbstractMatrix{Int8}, T::AbstractMatrix{Int8}; devV = S, devH = T)
    setfield!(ss, :spinConfiguration, _like(getfield(ss, :spinConfiguration), Matrix{Int8}(S), Float64))
    setfield!(ss, :hiddenLayer, _like(getfield(ss, :hiddenLayer), Matrix{Int8}(T), Float64))
    devV === nothing || setfield!(ss, :_devV, Matrix{Int8}(devV))
    devH === nothing || setfield!(ss, :_devH, Matrix{Int8}(devH))
    ss
end
function Base.setproperty!(ss::SpinSystemOnBipartiteGraph, name::Symbol, v)
    if name === :couplingCoefficients || name === :externalMagneticField || name === :auxiliaryBias
        setfield!(ss, name, float.(v)); _build!(ss)
    else
        setfield!(ss, name, convert(fieldtype(SpinSystemOnBipartiteGraph, name), v))
    end
    v
end

abstract type UpdatingAlgorithmOnBipartiteGraph end
getSpinConfiguration(ua::UpdatingAlgorithmOnBipartiteGraph) = ua.spinSystem.spinConfiguration
setSpinConfiguration(ua::UpdatingAlgorithmOnBipartiteGraph, spinConfiguration::AbstractVecOrMat{<:Number}) = (ua.spinSystem.spinConfiguration = spinConfiguration)
getHiddenLayer(ua::UpdatingAlgorithmOnBipartiteGraph) = ua.spinSystem.hiddenLayer
setHiddenLayer(ua::UpdatingAlgorithmOnBipartiteGraph, hiddenLayer::AbstractVecOrMat{<:Number}) = (ua.spinSystem.hiddenLayer = hiddenLayer)
getCouplingCoefficients(ua::UpdatingAlgorithmOnBipartiteGraph) = ua.spinSystem.couplingCoefficients
setCouplingCoefficients(ua::UpdatingAlgorithmOnBipartiteGraph, couplingCoefficients::AbstractMatrix{<:AbstractFloat}) = (ua.spinSystem.couplingCoefficients = couplingCoefficients)
getExternalMagneticField(ua::UpdatingAlgorithmOnBipartiteGraph) = ua.spinSystem.externalMagneticField
setExternalMagneticField(ua::UpdatingAlgorithmOnBipartiteGraph, externalMagneticField::AbstractVector{<:AbstractFloat}) = (ua.spinSystem.externalMagneticField = externalMagneticField)
getAuxiliaryBias(ua::UpdatingAlgorithmOnBipartiteGraph) = ua.spinSystem.auxiliaryBias
setAuxiliaryBias(ua::UpdatingAlgorithmOnBipartiteGraph, auxiliaryBias::AbstractVector{<:AbstractFloat}) = (ua.spinSystem.auxiliaryBias = auxiliaryBias)
calcEnergy(ss::SpinSystemOnBipartiteGraph) = (_sync!(ss); _scalar(ss, CABI.energy(ss.ens, _nrep(ss))))   # :139-143
calcEnergy(ua::UpdatingAlgorithmOnBipartiteGraph) = calcEnergy(ua.spinSystem)
function calcLocalMagneticField(ss::SpinSystemOnBipartiteGraph)                                           # :147-150
    _sync!(ss)
    F = CABI.local_field(ss.ens, length(ss.externalMagneticField), _nrep(ss))
    ndims(getfield(ss, :spinConfiguration)) == 1 ? vec(F) : F
end
calcLocalMagneticField(ua::UpdatingAlgorithmOnBipartiteGraph) = calcLocalMagneticField(ua.spinSystem)
function calcLocalAuxiliaryBias(ss::SpinSystemOnBipartiteGraph)                                           # :154-157
    _sync!(ss)
    A = CABI.local_aux_bias(ss.ens, length(ss.auxiliaryBias), _nrep(ss))
    ndims(getfield(ss, :spinConfiguration)) == 1 ? vec(A) : A
end
calcLocalAuxiliaryBias(ua::UpdatingAlgorithmOnBipartiteGraph) = calcLocalAuxiliaryBias(ua.spinSystem)
heaviside(x::T; c::T = one(T)) where {T<:Number} = x > zero(T) ? one(T) : (x < zero(T) ? zero(T) : c)   # :163-171
end # module SpinSystems

# ------------------------------------------------------------------ SingleSpinFlip (src/SingleSpinFlip.jl)
module SingleSpinFlip
export update!, AsynchronousHopfieldNetwork, GlauberDynamics, MetropolisMethod
using LinearAlgebra
using Random, Distributions
using ..SpinSystems
import ..CABI
abstract type SingleSpinUpdatingAlgorithm <: UpdatingAlgorithm end
mutable struct AsynchronousHopfieldNetwork <: SingleSpinUpdatingAlgorithm
    spinSystem::SpinSystem
    distribution::ContinuousUnivariateDistribution
    AsynchronousHopfieldNetwork(spinSystem::SpinSystem) = new(spinSystem, Uniform())
end
mutable struct GlauberDynamics <: SingleSpinUpdatingAlgorithm
    spinSystem::SpinSystem
    temperature::AbstractFloat
    distribution::ContinuousUnivariateDistribution
    GlauberDynamics(spinSystem::SpinSystem, temperature::AbstractFloat) = new(spinSystem, temperature, Logistic())
end
mutable struct MetropolisMethod <: SingleSpinUpdatingAlgorithm
    spinSystem::SpinSystem
    temperature::AbstractFloat
    distribution::ContinuousUnivariateDistribution
    MetropolisMethod(spinSystem::SpinSystem, temperature::AbstractFloat) = new(spinSystem, temperature, Exponential())
end
rule(::AsynchronousHopfieldNetwork) = CABI.RULE_HOPFIELD
rule(::GlauberDynamics) = CABI.RULE_GLAUBER
rule(::MetropolisMethod) = CABI.RULE_METROPOLIS
temperature(ua) = hasproperty(ua, :temperature) ? Float64(ua.temperature) : 0.0
# update!(ua, updatedNode, fluctuation): src/SingleSpinFlip.jl:31-36, 46-55, 65-74
function update!(ua::SingleSpinUpdatingAlgorithm, updatedNode::Integer, fluctuation::AbstractFloat = 0.0)
    temperature(ua) < 0 && @warn "$(ua.temperature) is negative."
    ss = ua.spinSystem
    SpinSystems._sync!(ss)
    CABI.ssf_run!(ss.ens, rule(ua), 1; nodes = [updatedNode], fluct = [Float64(fluctuation)], T = [temperature(ua)])
    SpinSystems._pull!(ss)
    s = ss.spinConfiguration
    ndims(s) == 1 ? s[updatedNode] : s[updatedNode, :]
end
end # module SingleSpinFlip

# ------------------------------------------------------------------ OnBipartiteGraph (src/OnBipartiteGraph.jl)
module OnBipartiteGraph
export update!, makeSampler!, StochasticCellularAutomata
using LinearAlgebra
using Random, Distributions
using ..SpinSystems
import ..CABI
mutable struct StochasticCellularAutomata <: UpdatingAlgorithmOnBipartiteGraph
    spinSystem::SpinSystemOnBipartiteGraph
    temperature::AbstractFloat
    distribution::ContinuousUnivariateDistribution
    StochasticCellularAutomata(spinSystem::SpinSystemOnBipartiteGraph, temperature::AbstractFloat) = new(spinSystem, temperature, Logistic())
end
mutable struct MomentumAnnealing <: UpdatingAlgorithmOnBipartiteGraph
    spinSystem::SpinSystemOnBipartiteGraph
    temperature::AbstractFloat
    distribution::ContinuousUnivariateDistribution
    MomentumAnnealing(spinSystem::SpinSystemOnBipartiteGraph, temperature::AbstractFloat) = new(spinSystem, temperature, Exponential())
end
rule(::StochasticCellularAutomata) = CABI.BIP_SCA
rule(::MomentumAnnealing) = CABI.BIP_MA
# update!(ua, Fv, Fh): src/OnBipartiteGraph.jl:30-43, 53-66
function update!(ua::UpdatingAlgorithmOnBipartiteGraph, fluctuationForSpinConfiguration::AbstractVector{<:AbstractFloat},
                 fluctuationForHiddenLayer::AbstractVector{<:AbstractFloat})
    ua.temperature < 0 && @warn "$(ua.temperature) is negative."
    ss = ua.spinSystem
    SpinSystems._sync!(ss)
    CABI.bip_run!(ss.ens, rule(ua), 1; Fv = fluctuationForSpinConfiguration, Fh = fluctuationForHiddenLayer,
                  T = [Float64(ua.temperature)])
    SpinSystems._pull!(ss)
    ss.spinConfiguration
end
end # module OnBipartiteGraph

# ------------------------------------------------------------------ MultiSpinFlip (stub in the reference: src/MultiSpinFlip.jl)
module MultiSpinFlip
export update!, makeSampler!, StochasticCellularAutomata
using LinearAlgebra
using Random, Distributions
using ..SpinSystems
import ..OnBipartiteGraph
abstract type MultiSpinUpdatingAlgorithm <: UpdatingAlgorithm end          # src/MultiSpinFlip.jl:9
# The reference defines no concrete multi-spin algorithm (SamplingHelper.jl:64-91 calls an update! that does not
# exist).  The one it demonstrates is the SCA of a general graph as the bipartite embedding of demo.jl:82-90:
# W = (J + qI)/2, biases h/2, sigma = tau = s.
mutable struct StochasticCellularAutomata <: MultiSpinUpdatingAlgorithm
    spinSystem::SpinSystem
    temperature::AbstractFloat
    distribution::ContinuousUnivariateDistribution
    bipartite::OnBipartiteGraph.StochasticCellularAutomata
    pinningParameter::Float64
    _J::Any                    # the couplings / fields the embedding was built from (identity-compared)
    _h::Any
    function StochasticCellularAutomata(ss::SpinSystem, temperature::AbstractFloat;
                                        pinningParameter = 0.5 * eigmax(Symmetric(Matrix(ss.couplingCoefficients))),
                                        prec = OnBipartiteGraph.CABI.PREC_F64)
        ua = new(ss, temperature, Logistic())
        ua.pinningParameter = pinningParameter
        _embed!(ua; prec = prec)
        ua
    end
end
function _embed!(ua::StochasticCellularAutomata; prec = ua.bipartite.spinSystem.prec)
    ss = ua.spinSystem
    s = ss.spinConfiguration; J = ss.couplingCoefficients; h = ss.externalMagneticField
    b = SpinSystemOnBipartiteGraph(copy(s), copy(s), 0.5 * (Matrix(J) + ua.pinningParameter * I), 0.5 * h, 0.5 * h; prec = prec)
    ua.bipartite = OnBipartiteGraph.StochasticCellularAutomata(b, ua.temperature)
    ua._J = J; ua._h = h
    ua
end
# changes made to the general-graph system since the last step (setters, assignments, in-place writes) reach the embedding
function _sync_in!(ua::StochasticCellularAutomata)
    ss = ua.spinSystem
    (ss.couplingCoefficients === ua._J && ss.externalMagneticField === ua._h) || _embed!(ua)
    b = ua.bipartite.spinSystem
    if SpinSystems._int8(ss.spinConfiguration) != SpinSystems._int8(b.spinConfiguration)
        b.spinConfiguration = copy(ss.spinConfiguration); b.hiddenLayer = copy(ss.spinConfiguration)
    end
    ua.bipartite.temperature = ua.temperature
    ua
end
_sync_out!(ua::StochasticCellularAutomata) =
    (SpinSystems._adopt!(ua.spinSystem, SpinSystems._int8(ua.bipartite.spinSystem.spinConfiguration); dev = nothing); ua)
# one synchronous step with explicit fluctuations for the two copies (the 3-argument form of OnBipartiteGraph.update!)
function update!(ua::StochasticCellularAutomata, Fv::AbstractVector{<:AbstractFloat}, Fh::AbstractVector{<:AbstractFloat})
    _sync_in!(ua)
    OnBipartiteGraph.update!(ua.bipartite, Fv, Fh)
    _sync_out!(ua)
    ua.spinSystem.spinConfiguration
end
# The same synchronous SCA for a model too large for one GPU (BASELINE config 5): rank `block` of `n_blocks` processes
# (one per GPU) owns n / n_blocks rows of W = (J + qI)/2; the freshly sampled blocks are exchanged after every half-step
# inside the library (isb_shard_run_steps).  `wire!` carries the NCCL id (128 bytes, from rank 0) or the IPC handles
# (64 bytes per rank) between the processes with whatever the application uses (MPI.jl: `bcast` / `Allgather`).
mutable struct ShardedStochasticCellularAutomata <: MultiSpinUpdatingAlgorithm
    temperature::AbstractFloat
    n::Int
    replicas::Int
    block::Int
    n_blocks::Int
    model::Ptr{Cvoid}
    run::Ptr{Cvoid}
    # synthetic Sherrington-Kirkpatrick instance generated on the device (never materialised in full)
    function ShardedStochasticCellularAutomata(n::Integer, replicas::Integer, temperature::AbstractFloat; block::Integer,
                                               n_blocks::Integer, seed::Integer, pinningParameter::Real = 1.0,
                                               exchange = OnBipartiteGraph.CABI.EXCH_NCCL, prec = OnBipartiteGraph.CABI.PREC_I8X3)
        C = OnBipartiteGraph.CABI
        m = C.shard_model_sk(n, n_blocks, block, seed, pinningParameter; prec = prec)
        r = C.shard_run_create(m, replicas, n_blocks == 1 ? C.EXCH_LOCAL : exchange)
        ua = new(temperature, n, replicas, block, n_blocks, m, r)
        finalizer(ua) do u
            u.run != C_NULL && C.shard_run_destroy(u.run)
            u.model != C_NULL && C.model_destroy(u.model)
            u.run = C_NULL; u.model = C_NULL
        end
    end
end
# every rank: wire!(ua; nccl_id = the 128 bytes drawn on rank 0)   or   wire!(ua; ipc_handles = all ranks' 64-byte handles)
function wire!(ua::ShardedStochasticCellularAutomata; nccl_id = nothing, ipc_handles = nothing)
    C = OnBipartiteGraph.CABI
    nccl_id === nothing || C.shard_run_init_nccl(ua.run, Vector{UInt8}(nccl_id))
    if ipc_handles !== nothing
        for (q, h) in enumerate(ipc_handles)
            q - 1 == ua.block || C.shard_run_ipc_import(ua.run, q - 1, Vector{UInt8}(h))
        end
    end
    ua
end
ipcHandle(ua::ShardedStochasticCellularAutomata) = OnBipartiteGraph.CABI.shard_run_ipc_export(ua.run)
ncclUniqueId() = OnBipartiteGraph.CABI.nccl_unique_id()
# S: n x replicas (+-1), the same on every rank
setSpinConfiguration!(ua::ShardedStochasticCellularAutomata, S::AbstractMatrix{<:Number}) =
    OnBipartiteGraph.CABI.shard_run_set_spins!(ua.run, Matrix{Int8}(S))
getSpinConfiguration(ua::ShardedStochasticCellularAutomata) =
    Int.(OnBipartiteGraph.CABI.shard_run_get_spins!(ua.run, 0, Matrix{Int8}(undef, ua.n, ua.replicas)))
# nsteps synchronous steps, step k at annealingSchedule(k) (collective: every rank calls it with the same arguments)
function run!(ua::ShardedStochasticCellularAutomata, nsteps::Integer; annealingSchedule::Function = k -> ua.temperature,
              seed::Integer = 0, stepOffset::Integer = 0)
    T = Float64[annealingSchedule(k) for k in 1:nsteps]
    OnBipartiteGraph.CABI.shard_run_steps!(ua.run, OnBipartiteGraph.CABI.BIP_SCA, nsteps, T; seed = seed, step_offset = stepOffset)
    nsteps > 0 && (ua.temperature = T[end])
    ua
end
end # module MultiSpinFlip

# ------------------------------------------------------------------ SamplingHelper (src/SamplingHelper.jl)
module SamplingHelper
export update!, makeSampler!
using Random
using ..SpinSystems
using ..SingleSpinFlip
using ..MultiSpinFlip
using ..OnBipartiteGraph
import ..CABI

function update!(ua::SingleSpinFlip.SingleSpinUpdatingAlgorithm; rng::AbstractRNG = Random.default_rng())   # :22-26
    updatedNode = rand(rng, axes(getSpinConfiguration(ua), 1))
    fluctuation = rand(rng, ua.distribution)
    SingleSpinFlip.update!(ua, updatedNode, fluctuation)
end
function update!(ua::MultiSpinFlip.MultiSpinUpdatingAlgorithm; rng::AbstractRNG = Random.default_rng())     # :64-67
    n = size(getSpinConfiguration(ua), 1)
    Fv = rand(rng, ua.distribution, n)
    Fh = rand(rng, ua.distribution, n)
    MultiSpinFlip.update!(ua, Fv, Fh)
end
function update!(ua::UpdatingAlgorithmOnBipartiteGraph; rng::AbstractRNG = Random.default_rng())            # :104-108
    fluctuationForSpinConfiguration = rand(rng, ua.distribution, size(ua.spinSystem.spinConfiguration, 1))
    fluctuationForHiddenLayer = rand(rng, ua.distribution, size(ua.spinSystem.hiddenLayer, 1))
    OnBipartiteGraph.update!(ua, fluctuationForSpinConfiguration, fluctuationForHiddenLayer)
end

# Steps per library call of the streaming samplers: the kernels record the state after EVERY step of a chunk
# (isb_ssf_run_snap / isb_bip_run_snap, trace_every = 1) and the Channel contract — n + 1 items, each the same mutable
# object showing the state after its step, temperature set before the step — is replayed from those snapshots.
# The Channel stays unbuffered: the consumer sees step k when it takes item k.  If the consumer changes the spins (or,
# with the default schedule, the temperature) between two items, the rest of the chunk is discarded and the run
# resumes from the consumer's state, as the reference's step-by-step loop would.
const CHUNK = Ref(4096)
_chunk(maxMCSteps, k, bytes_per_step) = max(1, min(maxMCSteps - k, CHUNK[], (256 << 20) ÷ max(1, bytes_per_step)))

# makeSampler!(ua::SingleSpinUpdatingAlgorithm, n; annealingSchedule, rng): src/SamplingHelper.jl:28-51
function makeSampler!(updatingAlgorithm::SingleSpinFlip.SingleSpinUpdatingAlgorithm, maxMCSteps::Integer;
                      annealingSchedule::Function = n -> updatingAlgorithm.temperature,
                      rng::AbstractRNG = Random.default_rng())::Channel{SpinSystems.UpdatingAlgorithm}
    if maxMCSteps < 0
        @warn "$maxMCSteps is negative."
    end
    ua = updatingAlgorithm
    hasT = hasproperty(ua, :temperature)
    updatedNodes = rand(rng, axes(getSpinConfiguration(ua), 1), max(maxMCSteps, 0))      # :39
    fluctuations = rand(rng, ua.distribution, max(maxMCSteps, 0))                        # :40
    Channel{SpinSystems.UpdatingAlgorithm}() do channel
        hasT && (ua.temperature = annealingSchedule(0))                                   # :43
        put!(channel, ua)                                                                 # :44
        ss = ua.spinSystem
        N = length(ss.externalMagneticField); R = size(ss.spinConfiguration, 2)
        k = 0
        while k < maxMCSteps
            m = _chunk(maxMCSteps, k, N * R)
            T = hasT ? Float64[annealingSchedule(j) for j in k+1:k+m] : Float64[0.0]      # :46, evaluated per step
            snap = Array{Int8,3}(undef, N, R, m)
            SpinSystems._sync!(ss)
            CABI.ssf_run!(ss.ens, SingleSpinFlip.rule(ua), m; nodes = updatedNodes[k+1:k+m], fluct = fluctuations[k+1:k+m],
                          T = T, steps_per_T = hasT ? 1 : m, trace_every = 1, snap = snap)
            lastS = snap[:, :, m]
            done = m
            for j in 1:m
                SpinSystems._adopt!(ss, view(snap, :, :, j); dev = lastS)                 # host shows step k+j, device holds k+m
                hasT && (ua.temperature = T[j])
                put!(channel, ua)                                                         # :48
                touched = SpinSystems._int8(ss.spinConfiguration) != view(snap, :, :, j) ||
                          (hasT && j < m && annealingSchedule(k + j + 1) != T[j+1])
                if touched && j < m
                    done = j; break       # _sync! pushes the consumer's state before the next chunk
                end
            end
            k += done
        end
    end
end

# makeSampler!(ua::MultiSpinUpdatingAlgorithm, n, annealingSchedule; rng): src/SamplingHelper.jl:69-91 (the schedule is
# POSITIONAL here, as in the reference)
function makeSampler!(updatingAlgorithm::MultiSpinFlip.MultiSpinUpdatingAlgorithm, maxMCSteps::Integer,
                      annealingSchedule::Function = n -> updatingAlgorithm.temperature;
                      rng::AbstractRNG = Random.default_rng())::Channel{SpinSystems.UpdatingAlgorithm}
    if maxMCSteps < 0
        @warn "$maxMCSteps is negative."
    end
    ua = updatingAlgorithm
    n = size(getSpinConfiguration(ua), 1)
    Fv = rand(rng, ua.distribution, (n, max(maxMCSteps, 0)))
    Fh = rand(rng, ua.distribution, (n, max(maxMCSteps, 0)))
    Channel{SpinSystems.UpdatingAlgorithm}() do channel
        ua.temperature = annealingSchedule(0)
        put!(channel, ua)
        R = size(ua.spinSystem.spinConfiguration, 2)
        k = 0
        while k < maxMCSteps
            m = _chunk(maxMCSteps, k, 2 * n * R)
            T = Float64[annealingSchedule(j) for j in k+1:k+m]
            MultiSpinFlip._sync_in!(ua)
            b = ua.bipartite.spinSystem
            SpinSystems._sync!(b)
            snapV = Array{Int8,3}(undef, n, R, m); snapH = Array{Int8,3}(undef, n, R, m)
            CABI.bip_run!(b.ens, OnBipartiteGraph.rule(ua.bipartite), m; Fv = Fv[:, k+1:k+m], Fh = Fh[:, k+1:k+m], T = T,
                          trace_every = 1, snapV = snapV, snapH = snapH)
            lastV = snapV[:, :, m]; lastH = snapH[:, :, m]
            done = m
            for j in 1:m
                SpinSystems._adopt!(b, view(snapV, :, :, j), view(snapH, :, :, j); devV = lastV, devH = lastH)
                MultiSpinFlip._sync_out!(ua)
                ua.temperature = T[j]
                put!(channel, ua)
                touched = SpinSystems._int8(ua.spinSystem.spinConfiguration) != view(snapV, :, :, j) ||
                          (j < m && annealingSchedule(k + j + 1) != T[j+1])
                if touched && j < m
                    done = j; break
                end
            end
            k += done
        end
    end
end

# makeSampler!(ua::UpdatingAlgorithmOnBipartiteGraph, n; annealingSchedule, rng): src/SamplingHelper.jl:110-133
function makeSampler!(updatingAlgorithm::UpdatingAlgorithmOnBipartiteGraph, maxMCSteps::Integer;
                      annealingSchedule::Function = n -> updatingAlgorithm.temperature,
                      rng::AbstractRNG = Random.default_rng())::Channel{SpinSystems.UpdatingAlgorithmOnBipartiteGraph}
    if maxMCSteps < 0
        @warn "$maxMCSteps is negative."
    end
    ua = updatingAlgorithm
    nv = size(getSpinConfiguration(ua), 1); nh = size(getHiddenLayer(ua), 1)
    fluctuationsForSpinConfiguration = rand(rng, ua.distribution, (nv, max(maxMCSteps, 0)))   # :121
    fluctuationsForHiddenLayer = rand(rng, ua.distribution, (nh, max(maxMCSteps, 0)))         # :122
    Channel{SpinSystems.UpdatingAlgorithmOnBipartiteGraph}() do channel
        ua.temperature = annealingSchedule(0)                                                  # :125
        put!(channel, ua)                                                                      # :126
        ss = ua.spinSystem
        R = size(ss.spinConfiguration, 2)
        k = 0
        while k < maxMCSteps
            m = _chunk(maxMCSteps, k, (nv + nh) * R)
            T = Float64[annealingSchedule(j) for j in k+1:k+m]                                 # :128
            SpinSystems._sync!(ss)
            snapV = Array{Int8,3}(undef, nv, R, m); snapH = Array{Int8,3}(undef, nh, R, m)
            CABI.bip_run!(ss.ens, OnBipartiteGraph.rule(ua), m; Fv = fluctuationsForSpinConfiguration[:, k+1:k+m],
                          Fh = fluctuationsForHiddenLayer[:, k+1:k+m], T = T, trace_every = 1, snapV = snapV, snapH = snapH)
            lastV = snapV[:, :, m]; lastH = snapH[:, :, m]
            done = m
            for j in 1:m
                SpinSystems._adopt!(ss, view(snapV, :, :, j), view(snapH, :, :, j); devV = lastV, devH = lastH)
                ua.temperature = T[j]
                put!(channel, ua)                                                              # :130
                touched = SpinSystems._int8(ss.spinConfiguration) != view(snapV, :, :, j) ||
                          SpinSystems._int8(ss.hiddenLayer) != view(snapH, :, :, j) ||
                          (j < m && annealingSchedule(k + j + 1) != T[j+1])
                if touched && j < m
                    done = j; break
                end
            end
            k += done
        end
    end
end
end # module SamplingHelper

end # module IsingModelB200
