# DLRMB200.jl -- Julia host glue that puts libdlrm_b200.so (C ABI: include/dlrm_b200.h) BEHIND the
# entry points the unmodified DLRM.jl model and training loop already call.
#
# STATUS: written against the reference's call sites, NOT EXECUTED.  There is no `julia` binary in the
# build image or on the GPU box, and DLRM.jl's path dependencies (EmbeddingTables, OneDNN, CachedArrays;
# Manifest.toml:79-83,246-250,522-526) are not vendored.  Every ccall below is exercised instead through
# the Python ctypes binding (dlrm_jl_b200/_lib.py), which binds the same symbols with the same argument
# lists; tests/test_abi_cpu.py checks this file's ccall names and arities against the header.
#
# What dispatches where (paths relative to the DLRM.jl checkout; nothing in DLRM.jl is edited):
#
#   DLRM.jl line                                           method added here
#   ----------------------------------------------------   -------------------------------------------------
#   src/model/model.jl:117-122  embeddings::Vector{E}       E = B200Embedding{Static{D},Float32}: one element per
#                                                           table, every element a view (slab, k) of ONE device
#                                                           handle, so a single launch still serves all tables
#   src/model/model.jl:96-110   create_embeddings(finish..) `embedding_constructor = B200Embedding{Static{D}}` is the
#   src/model/model.jl:185,202  finish(init(ncols, nrows))  `finish` hook: called once per table with the host matrix
#   src/model/model.jl:161      maplookup(strategy,         EmbeddingTables.maplookup(::PreallocationStrategy /
#                               D.embeddings, sparse)       ::DefaultStrategy, ::Vector{<:B200Embedding}, sparse)
#   test/model/embedding_update.jl:22-40  Zygote._pullback  ChainRulesCore.rrule(::typeof(maplookup), ...) returning
#                               of maplookup                (nothing, nothing, Vector{SparseEmbeddingUpdate}, nothing)
#   src/train/train.jl:137-150  DLRMGrads.embeddings::      the pullback's elements ARE EmbeddingTables.
#                               Vector{SparseEmbeddingUpdate} SparseEmbeddingUpdate{Static{D}}(delta_view, indices), so
#                               + gather_embeddings! :177   `append!` into that vector type-checks
#   src/train/train.jl:283-290  EmbeddingTables.update!(opt, EmbeddingTables.update!(::Flux.Descent,
#                               param_embeddings,            ::Vector{<:B200Embedding}, ::Vector{<:SparseEmbeddingUpdate},
#                               grads_embeddings, indexers;  indexers; num_splits, nthreads)
#                               num_splits, nthreads)
#   src/validation.jl:138       isapprox(reference,          Base.isapprox(::AbstractMatrix, ::B200Embedding),
#                               model.embeddings[i])         Base.Array / Base.collect / size / getindex
#   src/model/model.jl:119,163  D.interaction(x, y)          (dot::B200DotInteraction)(x, y) + ChainRulesCore.rrule,
#   src/model/interact.jl:390-447                            passed as `interaction = B200DotInteraction()` to `dlrm`
#
# Assumed from the upstream EmbeddingTables.jl (v0.1.0, not available here -- [unverifiable]):
#   abstract type AbstractEmbeddingTable{S<:AbstractLookupType,T} <: AbstractArray{T,2}; Static{N} / Dynamic lookup
#   types; featuresize(table); SparseEmbeddingUpdate{S}(delta::AbstractMatrix, indices) with fields .delta/.indices
#   (constructor form used in src/playground.jl:44); PreallocationStrategy has a `prependrows` field.
# If a name differs upstream, only the few lines marked `# [upstream name]` need to follow it.
#
# The model in DLRM.jl is CPU-resident (OneDNN MLPs), so this glue uses the `_host` entry points: Julia
# arrays go in and come out, the copies happen inside the call.  Column-major Julia arrays are passed as
# they are: a `D x N` Julia matrix is the C array [N][D] the library expects; indices stay 1-based.
module DLRMB200

import ChainRulesCore
import ChainRulesCore: NoTangent
import Flux
import EmbeddingTables
import EmbeddingTables: AbstractEmbeddingTable, Static, SparseEmbeddingUpdate, PreallocationStrategy, DefaultStrategy

export B200Embedding, B200DotInteraction

const libdlrm_b200 = get(ENV, "DLRM_B200_LIB",
                         joinpath(@__DIR__, "..", "dlrm_jl_b200", "lib", "libdlrm_b200.so"))

struct B200Error <: Exception
    status::Int32
    msg::String
end
Base.showerror(io::IO, e::B200Error) = print(io, "libdlrm_b200 status ", e.status, ": ", e.msg)

function check(rc::Int32)
    rc == 0 && return nothing
    msg = unsafe_string(ccall((:dlrmb_last_error, libdlrm_b200), Cstring, ()))
    throw(B200Error(rc, msg))
end

#####
##### Storage: one device slab for all tables of a model, one B200Embedding per table
#####

"All tables of one model behind one `dlrmb_tables` handle (created lazily, see `materialize!`)."
mutable struct B200Slab
    handle::Ptr{Cvoid}
    device::Int32
    rows::Vector{Int64}
    featuresize::Int
    max_lookups::Int
    pending::Vector{Matrix{Float32}}     # host data of the tables until the handle exists
end

"""
    B200Embedding{Static{D}}(data)            # the `embedding_constructor` / `finish` hook

One embedding table of an HBM-resident model: a `(slab, k)` view.  `dlrm(...; embedding_constructor =
B200Embedding{Static{D}})` calls this once per table with the `D x nrows` host matrix
(src/model/model.jl:96-110,202-206); tables built one after the other join the slab that is still
collecting (`DLRMB200.new_model!()` starts a fresh one).  The device handle is created, and the data
uploaded, when the vector of tables is first used (`materialize!`), because only then are the number
of tables and the batch size known.
"""
struct B200Embedding{S,T} <: AbstractEmbeddingTable{S,T}        # [upstream name]
    slab::B200Slab
    k::Int                                                        # 1-based position in the slab
end

const COLLECTING = Ref{Union{Nothing,B200Slab}}(nothing)
const DEVICE = Ref{Int32}(0)

"Start a fresh slab: call before constructing a second model in the same process."
new_model!(; device::Integer = 0) = (DEVICE[] = Int32(device); COLLECTING[] = nothing)

function B200Embedding{Static{D}}(data::AbstractMatrix) where {D}
    @assert size(data, 1) == D
    slab = COLLECTING[]
    if slab === nothing || slab.handle != C_NULL || slab.featuresize != D
        slab = B200Slab(C_NULL, DEVICE[], Int64[], D, 0, Matrix{Float32}[])
        finalizer(slab) do s
            s.handle == C_NULL || ccall((:dlrmb_tables_destroy, libdlrm_b200), Int32, (Ptr{Cvoid},), s.handle)
            s.handle = C_NULL
        end
        COLLECTING[] = slab
    end
    push!(slab.rows, size(data, 2))
    push!(slab.pending, Matrix{Float32}(data))        # contiguous D x nrows == C [nrows][D]
    return B200Embedding{Static{D},Float32}(slab, length(slab.rows))
end
B200Embedding(data::AbstractMatrix) = B200Embedding{Static{size(data, 1)}}(data)

EmbeddingTables.featuresize(t::B200Embedding) = t.slab.featuresize          # [upstream name]
Base.size(t::B200Embedding) = (t.slab.featuresize, Int(t.slab.rows[t.k]))

"Create the device handle for `tables` (all views of one slab, in slab order) and upload the pending data."
function materialize!(tables::AbstractVector{<:B200Embedding}, max_lookups::Integer)
    slab = first(tables).slab
    @assert all(t -> t.slab === slab, tables) && [t.k for t in tables] == collect(1:length(slab.rows)) "the model's embeddings must be the tables of one slab, in construction order"
    if slab.handle == C_NULL
        out = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:dlrmb_tables_create, libdlrm_b200), Int32,
                    (Int32, Int32, Ptr{Int64}, Int32, Int64, Ptr{Ptr{Cvoid}}),
                    slab.device, length(slab.rows), slab.rows, slab.featuresize, max_lookups, out))
        slab.handle = out[]
        slab.max_lookups = max_lookups
        for (k, m) in enumerate(slab.pending)
            check(ccall((:dlrmb_tables_upload, libdlrm_b200), Int32, (Ptr{Cvoid}, Int32, Ptr{Float32}),
                        slab.handle, k - 1, m))
        end
        empty!(slab.pending)
        COLLECTING[] === slab && (COLLECTING[] = nothing)
    elseif max_lookups > slab.max_lookups        # a larger batch than any before: grow the workspaces only
        check(ccall((:dlrmb_tables_reserve, libdlrm_b200), Int32, (Ptr{Cvoid}, Int64), slab.handle, max_lookups))
        slab.max_lookups = max_lookups
    end
    return slab
end

"`Array(table)`: the `D x nrows` matrix of the table (validate_embeddings, src/validation.jl:138)."
function Base.Array(t::B200Embedding{S,T}) where {S,T}
    slab = t.slab
    slab.handle == C_NULL && return copy(slab.pending[t.k])
    A = Matrix{Float32}(undef, slab.featuresize, slab.rows[t.k])
    check(ccall((:dlrmb_tables_download, libdlrm_b200), Int32, (Ptr{Cvoid}, Int32, Ptr{Float32}),
                slab.handle, t.k - 1, A))
    return A
end
Base.collect(t::B200Embedding) = Array(t)
# element access downloads the table: fine for the REPL and tests, never used by the hot path
Base.getindex(t::B200Embedding, i::Int, j::Int) = Array(t)[i, j]
Base.isapprox(a::AbstractMatrix, t::B200Embedding; kw...) = isapprox(a, Array(t); kw...)
Base.isapprox(t::B200Embedding, a::AbstractMatrix; kw...) = isapprox(Array(t), a; kw...)
Base.isapprox(a::B200Embedding, b::B200Embedding; kw...) = isapprox(Array(a), Array(b); kw...)

#####
##### Index containers -> table-major [ntab][B][P]
#####

# `sparse` is DACLoader's B x ntab UInt32 matrix (src/data/criteo.jl:320-326) or a vector of per-table
# index vectors / P x B matrices (src/data/criteo.jl:551-557).  Both are already the table-major layout
# the library wants once concatenated; indices stay 1-based (idx_base = 1).  When the tables' widths
# differ (multi-hot with per-table hotness) the result is the flat reduce(vcat, vec.(sparse)) and the
# vector of pooling factors, for the `_mp` entry points.
_pack(sparse::AbstractMatrix{<:Integer}) = (Matrix(sparse), 1)                        # B x ntab, P = 1
function _pack(sparse::AbstractVector)
    Ps = [ndims(s) == 1 ? 1 : size(s, 1) for s in sparse]
    all(==(first(Ps)), Ps) && return (reduce(hcat, [vec(s) for s in sparse]), first(Ps))   # (P*B) x ntab
    return (reduce(vcat, [vec(s) for s in sparse]), Int32.(Ps))                       # sum(P)*B, P per table
end
_batch(idx, P::Integer) = div(size(idx, 1), P)
_batch(idx, P::AbstractVector) = div(length(idx), sum(P))
_table_indices(sparse::AbstractMatrix{<:Integer}, k) = view(sparse, :, k)
_table_indices(sparse::AbstractVector, k) = sparse[k]
_idxbytes(::AbstractArray{T}) where {T} = Int32(sizeof(T))
_prepend(s::PreallocationStrategy) = s.prependrows                                   # [upstream name]

#####
##### maplookup (src/model/model.jl:161) + pullback
#####

function _lookup(tables::AbstractVector{<:B200Embedding}, sparse, prependrows::Integer)
    idx, P = _pack(sparse)
    B = _batch(idx, P)
    slab = materialize!(tables, B * maximum(P))
    D = slab.featuresize
    @assert iszero(mod(prependrows, D))
    slot0 = div(prependrows, D)
    slots = slot0 + length(tables)
    out = zeros(Float32, slots * D, B)                                                # == C [B][slots][D]
    if P isa Integer
        check(ccall((:dlrmb_embedding_fwd_host, libdlrm_b200), Int32,
                    (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Int32, Int32, Int32, Ptr{Float32}, Int32, Int32),
                    slab.handle, idx, _idxbytes(idx), 1, B, P, out, slots, slot0))
    else
        check(ccall((:dlrmb_embedding_fwd_mp_host, libdlrm_b200), Int32,
                    (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Int32, Int32, Ptr{Int32}, Ptr{Float32}, Int32, Int32),
                    slab.handle, idx, _idxbytes(idx), 1, B, P, out, slots, slot0))
    end
    return out, slot0
end

function EmbeddingTables.maplookup(strategy::PreallocationStrategy, tables::AbstractVector{<:B200Embedding}, sparse)
    return first(_lookup(tables, sparse, _prepend(strategy)))
end

function EmbeddingTables.maplookup(::DefaultStrategy, tables::AbstractVector{<:B200Embedding}, sparse)
    out, _ = _lookup(tables, sparse, 0)
    D = first(tables).slab.featuresize
    return [out[((k - 1) * D + 1):(k * D), :] for k in eachindex(tables)]             # one D x B matrix per table
end
EmbeddingTables.maplookup(tables::AbstractVector{<:B200Embedding}, sparse) =
    EmbeddingTables.maplookup(DefaultStrategy(), tables, sparse)

# The lookup pullback does no arithmetic: per table, the rows of the incoming gradient that belong to it
# and that table's indices (src/train/train.jl:144; shape pinned by test/model/embedding_update.jl:36-40).
function _updates(Δ::AbstractMatrix, tables, sparse, slot0::Integer)
    D = first(tables).slab.featuresize
    return [SparseEmbeddingUpdate{Static{D}}(view(Δ, ((slot0 + k - 1) * D + 1):((slot0 + k) * D), :),
                                             _table_indices(sparse, k)) for k in eachindex(tables)]
end

function ChainRulesCore.rrule(::typeof(EmbeddingTables.maplookup), strategy::PreallocationStrategy,
                              tables::AbstractVector{<:B200Embedding}, sparse)
    out, slot0 = _lookup(tables, sparse, _prepend(strategy))
    function maplookup_pullback(Δ)
        dy = Δ isa Matrix{Float32} ? Δ : Matrix{Float32}(ChainRulesCore.unthunk(Δ))
        return (NoTangent(), NoTangent(), _updates(dy, tables, sparse, slot0), NoTangent())
    end
    return out, maplookup_pullback
end

function ChainRulesCore.rrule(::typeof(EmbeddingTables.maplookup), ::DefaultStrategy,
                              tables::AbstractVector{<:B200Embedding}, sparse)
    ys = EmbeddingTables.maplookup(DefaultStrategy(), tables, sparse)
    D = first(tables).slab.featuresize
    function maplookup_pullback(Δs)
        dy = reduce(vcat, [Matrix{Float32}(ChainRulesCore.unthunk(d)) for d in Δs])   # (ntab*D) x B
        return (NoTangent(), NoTangent(), _updates(dy, tables, sparse, 0), NoTangent())
    end
    return ys, maplookup_pullback
end

#####
##### EmbeddingTables.update! (src/train/train.jl:283-290)
#####

# If every update's delta is the matching row range of ONE parent matrix (what the pullbacks above
# build, and what the interaction pullback hands them), that matrix goes to the library as it is.
function _shared_parent(grads, D)
    p = parent(first(grads).delta)
    p isa Matrix{Float32} || return nothing
    first_row = first(parentindices(first(grads).delta)[1])
    iszero(mod(first_row - 1, D)) || return nothing
    slot0 = div(first_row - 1, D)
    for (k, g) in enumerate(grads)
        g.delta isa SubArray && parent(g.delta) === p || return nothing
        rows, cols = parentindices(g.delta)
        (first(rows) == (slot0 + k - 1) * D + 1 && length(rows) == D && cols == Base.Slice(axes(p, 2))) || return nothing
    end
    return p, slot0
end

function EmbeddingTables.update!(opt::Flux.Descent, tables::AbstractVector{<:B200Embedding},
                                 grads::AbstractVector{<:SparseEmbeddingUpdate}, indexers = nothing;
                                 num_splits = 8, nthreads = 12)
    @assert length(tables) == length(grads)
    D = first(tables).slab.featuresize
    idx, P = _pack([g.indices for g in grads])
    B = _batch(idx, P)
    slab = materialize!(tables, B * maximum(P))
    shared = _shared_parent(grads, D)
    if shared === nothing      # updates built one by one: pack into one (ntab*D) x B matrix
        delta, slot0 = reduce(vcat, [Matrix{Float32}(g.delta) for g in grads]), 0
    else
        delta, slot0 = shared
    end
    slots = div(size(delta, 1), D)
    # `indexers`, `num_splits`, `nthreads` steer the reference's CPU dedup / threading; here the dedup is
    # the device-side sort and the whole update is one launch, so they are accepted and ignored
    if P isa Integer
        check(ccall((:dlrmb_embedding_bwd_sgd_host, libdlrm_b200), Int32,
                    (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Int32, Int32, Int32, Ptr{Float32}, Int32, Int32, Float32),
                    slab.handle, idx, _idxbytes(idx), 1, B, P, delta, slots, slot0, Float32(opt.eta)))
    else
        check(ccall((:dlrmb_embedding_bwd_sgd_mp_host, libdlrm_b200), Int32,
                    (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Int32, Int32, Ptr{Int32}, Ptr{Float32}, Int32, Int32, Float32),
                    slab.handle, idx, _idxbytes(idx), 1, B, P, delta, slots, slot0, Float32(opt.eta)))
    end
    return nothing
end

#####
##### DotInteraction (src/model/interact.jl:369-447)
#####

"""
    B200DotInteraction(; pad_to_mul = 1, device = 0)

Callable for `DLRMModel.interaction` (pass as `interaction = B200DotInteraction()` to `dlrm` /
`kaggle_dlrm`).  `(dot)(x, ys)` with `ys` the PreallocationStrategy matrix (x is copied into its first
rows, the reference's `fast_vcat`, src/model/interact.jl:271-281) or a vector of `D x B` matrices
(DefaultStrategy, src/model/interact.jl:503-513).
"""
mutable struct B200DotInteraction
    staging::Ptr{Cvoid}          # a one-row table handle: owns the stream / device buffers of the host calls
    pad_to_mul::Int              # POST_INTERACTION_PAD_TO_MUL, src/model/model.jl:32
end

function B200DotInteraction(; pad_to_mul::Integer = 1, device::Integer = 0)
    out = Ref{Ptr{Cvoid}}(C_NULL)
    rows = Int64[1]
    check(ccall((:dlrmb_tables_create, libdlrm_b200), Int32,
                (Int32, Int32, Ptr{Int64}, Int32, Int64, Ptr{Ptr{Cvoid}}), device, 1, rows, 4, 4, out))
    dot = B200DotInteraction(out[], pad_to_mul)
    finalizer(dot) do d
        d.staging == C_NULL || ccall((:dlrmb_tables_destroy, libdlrm_b200), Int32, (Ptr{Cvoid},), d.staging)
        d.staging = C_NULL
    end
    return dot
end

_width(F, d, m) = m * cld(d + div(F * (F - 1), 2), m)

function _fwd!(dot::B200DotInteraction, T::Matrix{Float32}, x, d, B)
    F = div(size(T, 1), d)
    out = Matrix{Float32}(undef, _width(F, d, dot.pad_to_mul), B)
    check(ccall((:dlrmb_interaction_fwd_host, libdlrm_b200), Int32,
                (Ptr{Cvoid}, Ptr{Float32}, Ptr{Float32}, Int32, Int32, Int32, Int32, Ptr{Float32}),
                dot.staging, T, x === nothing ? C_NULL : x, B, F, d, dot.pad_to_mul, out))
    return out
end

function _bwd(dot::B200DotInteraction, Δ, T::Matrix{Float32}, d, B)
    F = div(size(T, 1), d)
    dT = similar(T)
    dx = Matrix{Float32}(undef, d, B)
    check(ccall((:dlrmb_interaction_bwd_host, libdlrm_b200), Int32,
                (Ptr{Cvoid}, Ptr{Float32}, Ptr{Float32}, Int32, Int32, Int32, Int32, Ptr{Float32}, Ptr{Float32}),
                dot.staging, Matrix{Float32}(ChainRulesCore.unthunk(Δ)), T, B, F, d, dot.pad_to_mul, dT, dx))
    return dx, dT
end

# PreallocationStrategy: ys is (d*F) x B with its first d rows reserved for x
function (dot::B200DotInteraction)(x::AbstractMatrix{Float32}, ys::Matrix{Float32})
    d, B = size(x)
    return _fwd!(dot, ys, Matrix{Float32}(x), d, B)        # x lands in slot 0 of ys inside the kernel
end

function ChainRulesCore.rrule(dot::B200DotInteraction, x::AbstractMatrix{Float32}, ys::Matrix{Float32})
    d, B = size(x)
    out = _fwd!(dot, ys, Matrix{Float32}(x), d, B)         # ys now holds x in slot 0: it is the saved `t`
    function dot_pullback(Δ)
        dx, dT = _bwd(dot, Δ, ys, d, B)
        return (NoTangent(), dx, dT)   # dy is the whole (d*F) x B matrix, slot 0 included (src/model/interact.jl:428-435)
    end
    return out, dot_pullback
end

# DefaultStrategy: ys is a vector of D x B matrices
function (dot::B200DotInteraction)(x::AbstractMatrix{Float32}, ys::AbstractVector{<:AbstractMatrix})
    d, B = size(x)
    return _fwd!(dot, Matrix{Float32}(reduce(vcat, [x, ys...])), nothing, d, B)
end

function ChainRulesCore.rrule(dot::B200DotInteraction, x::AbstractMatrix{Float32}, ys::AbstractVector{<:AbstractMatrix})
    d, B = size(x)
    T = Matrix{Float32}(reduce(vcat, [x, ys...]))
    out = _fwd!(dot, T, nothing, d, B)
    function dot_pullback(Δ)
        dx, dT = _bwd(dot, Δ, T, d, B)      # dx = Δ[1:d, :] + dT[1:d, :]: both roles of x (concat pass-through + Gram row)
        return (NoTangent(), dx, [dT[(f * d + 1):((f + 1) * d), :] for f in 1:length(ys)])
    end
    return out, dot_pullback
end

#####
##### Multi-GPU (BASELINE config 4) from Julia: see INTEGRATION.md, "Sharded tables from a Julia host"
#####

"`owner[k]` = 0-based rank owning table k (table count balanced first, bytes second)."
function shard_plan(rows::Vector{Int64}, world::Integer)
    owner = Vector{Int32}(undef, length(rows))
    check(ccall((:dlrmb_shard_plan, libdlrm_b200), Int32, (Int32, Ptr{Int64}, Int32, Ptr{Int32}),
                length(rows), rows, world, owner))
    return owner
end

"""Per-table pooling factors `P[k]`: equal P gives `shard_plan(rows, world)`; mixed P deals the tables longest
first (descending P, rows, id), each to the rank with the smallest sum of P so far (ties: fewer rows, lower rank)."""
function shard_plan(rows::Vector{Int64}, world::Integer, P::Vector{Int32})
    owner = Vector{Int32}(undef, length(rows))
    check(ccall((:dlrmb_shard_plan_mp, libdlrm_b200), Int32, (Int32, Ptr{Int64}, Ptr{Int32}, Int32, Ptr{Int32}),
                length(rows), rows, P, world, owner))
    return owner
end

"Rank 0: the 128-byte NCCL id to hand to the other ranks (file, socket, MPI.bcast ...)."
function comm_unique_id()
    id = Vector{UInt8}(undef, 128)
    check(ccall((:dlrmb_comm_unique_id, libdlrm_b200), Int32, (Ptr{UInt8},), id))
    return id
end

function comm_create(device::Integer, id::Vector{UInt8}, rank::Integer, world::Integer)
    out = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:dlrmb_comm_create, libdlrm_b200), Int32, (Int32, Ptr{UInt8}, Int32, Int32, Ptr{Ptr{Cvoid}}),
                device, id, rank, world, out))
    return out[]
end

comm_destroy(comm::Ptr{Cvoid}) = check(ccall((:dlrmb_comm_destroy, libdlrm_b200), Int32, (Ptr{Cvoid},), comm))

end # module
