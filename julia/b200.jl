# b200.jl -- the B200 scan path of DataFrameDBs.jl: `ccall` binding of libdfdb_b200.so (include/dfdb_b200.h).
#
# This file is meant to live INSIDE the reference package (src/gpu/b200.jl, `include`d from src/DataFrameDBs.jl after
# tables/*.jl and io/*.jl; INTEGRATION.md shows the five-line patch), so the methods it adds belong to the package that owns
# the functions -- nothing is overwritten from outside.  The lazy API (open_table, DFTable, DFView, DFColumn, t[pred, cols],
# broadcasting) is untouched: it only builds plan objects.  The consumers that pull from BlocksIterator -- nrow,
# materialize, the reductions over a DFColumn -- ask `B200.enabled(table)` first and hand the view's plan to the library
# when the table was given to the GPU with `B200.enable!(table)`.
#
# NOT EXECUTED IN THIS REPOSITORY: the build image has no julia binary (probed).  tests/test_julia_binding.py parses every
# `ccall` below and checks symbol, arity and integer widths against include/dfdb_b200.h; the wire format and the call
# sequences are the ones the Python twin (dataframedbs.jl_b200/{_capi,api,plan}.py) drives in the parity tests.
# Reference line numbers refer to waralex/DataFrameDBs.jl.
module B200

using ..DataFrameDBs
using ..DataFrameDBs: DFTable, DFView, DFColumn, BlockBroadcasting, ColRef
using ..DataFrameDBs.FlatStringsVectors: FlatStringsVector
import DataFrames
import Statistics

const LIB = get(ENV, "DFDB_B200_LIB", "libdfdb_b200.so")

# ---- status -> exception (the classes the reference throws in the same situation) ---------------------------
last_error() = unsafe_string(ccall((:dfdb_last_error, LIB), Cstring, ()))
function check(rc::Int32)
    rc == 0 && return
    msg = last_error()
    rc == 4 && throw(ArgumentError(msg))            # selection.jl:54, selection.jl:73
    rc == 5 && throw(ArgumentError("unsupported on the GPU path: " * msg))
    rc == 6 && throw(KeyError(msg))                 # table.jl:54
    rc == 7 && throw(DivideError())
    rc == 3 && throw(AssertionError(msg))           # BlockStreams.jl:112 "decompression error"
    error(msg)                                      # creators.jl:8-9, filesystem.jl:47-58
end

# ---- runtime / table handles -----------------------------------------------------------------------------------
mutable struct TableHandle
    ptr::Ptr{Cvoid}
end
close_handle(h::TableHandle) = (h.ptr == C_NULL || ccall((:dfdb_table_close, LIB), Int32, (Ptr{Cvoid},), h.ptr); h.ptr = C_NULL; nothing)

# weak keys: a table that is no longer referenced drops its handle, whose finalizer closes the device copy
const TABLES = WeakKeyDict{DFTable,TableHandle}()
const STARTED = Ref(false)

function start()
    STARTED[] && return
    check(ccall((:dfdb_init, LIB), Int32, (Int32,), parse(Int32, get(ENV, "LOCAL_RANK", "0"))))
    STARTED[] = true
    nothing
end

enabled(t::DFTable) = haskey(TABLES, t)

"""
    B200.enable!(t::DFTable; mode = 1, rank = 0, world = 1)

Give the table to the GPU: parses the headers (open_table, creators.jl:7-16), takes the block-range shard `rank` of
`world` and loads its compressed blocks (`mode` 0 = pinned host memory, 1 = HBM, 2 = HBM + decoded bodies cached).
From then on `nrow`, `materialize` and the reductions over views of `t` run on the device.
"""
function enable!(t::DFTable; mode::Integer = 1, rank::Integer = 0, world::Integer = 1)
    start()
    enabled(t) && return t
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:dfdb_table_open, LIB), Int32, (Cstring, Ref{Ptr{Cvoid}}), t.path, h))
    th = TableHandle(h[])
    finalizer(close_handle, th)
    world > 1 && check(ccall((:dfdb_table_set_shard, LIB), Int32, (Ptr{Cvoid}, Int32, Int32), th.ptr, Int32(rank), Int32(world)))
    check(ccall((:dfdb_table_load, LIB), Int32, (Ptr{Cvoid}, Ptr{Int64}, Int32, Int32), th.ptr, C_NULL, Int32(0), Int32(mode)))
    TABLES[t] = th
    t
end
disable!(t::DFTable) = (enabled(t) && close_handle(pop!(TABLES, t)); t)
handle(t::DFTable) = TABLES[t].ptr

# ---- multi-GPU: one Julia process per GPU; the id travels by whatever the launcher has (MPI.bcast, a shared file) ----
comm_unique_id() = (start(); id = zeros(UInt8, 128); check(ccall((:dfdb_comm_unique_id, LIB), Int32, (Ptr{UInt8},), id)); id)
comm_init(rank::Integer, world::Integer, id::Vector{UInt8}) =
    (start(); check(ccall((:dfdb_comm_init, LIB), Int32, (Int32, Int32, Ptr{UInt8}), Int32(rank), Int32(world), id)))
comm_destroy() = check(ccall((:dfdb_comm_destroy, LIB), Int32, ()))

# ---- plan serialisation (wire format: INTEGRATION.md, dataframedbs.jl_b200/plan.py) ---------------------------------
const OPS = Dict{Any,UInt8}(
    (==) => 0x10, (!=) => 0x11, (<) => 0x12, (<=) => 0x13, (>) => 0x14, (>=) => 0x15,
    (&) => 0x20, (|) => 0x21, xor => 0x22, (!) => 0x23,
    (+) => 0x30, (-) => 0x31, (*) => 0x32, (/) => 0x33, (%) => 0x34, rem => 0x34,
    ismissing => 0x40, coalesce => 0x41, startswith => 0x50, endswith => 0x51)

colid(t::DFTable, name::Symbol) = DataFrameDBs.getmeta(t, name).id

function emit!(io::IO, t::DFTable, a)::Int
    if a isa ColRef
        write(io, 0x01, Int64(colid(t, a.name))); return 1
    elseif a isa BlockBroadcasting
        if a.f === in
            n = emit!(io, t, a.args[1])
            c = a.args[2][]                                   # Ref(collection)
            if c isa Vector{Int64}
                write(io, 0x60, UInt32(length(c))); write(io, c)
            else
                # Ref(::AbstractSet) is isequal (semantics 1), vectors and tuples are `==` (0)
                write(io, 0x61, UInt8(c isa AbstractSet), UInt32(length(c)))
                for x in c
                    if x isa Bool
                        write(io, 0x05, UInt8(x))
                    elseif x isa Signed
                        write(io, 0x01, Int64(x))
                    elseif x isa Unsigned
                        write(io, 0x02, UInt64(x))
                    elseif x isa AbstractFloat
                        write(io, 0x03, Float64(x))
                    elseif x isa AbstractString
                        s = String(x); write(io, 0x04, UInt32(sizeof(s))); write(io, s)
                    elseif x === missing
                        write(io, 0x06)
                    else
                        throw(ArgumentError("in() element of type $(typeof(x)) is not available on the GPU path"))
                    end
                end
            end
            return n + 1
        end
        op = get(OPS, a.f, nothing)
        # closures of the Pair form (view.jl:64-70) are opaque: no CPU fallback in the library, tell the user
        op === nothing && throw(ArgumentError("function $(a.f) is not available on the GPU path"))
        (a.f === (-) && length(a.args) == 1) && (op = 0x35)
        n = sum(emit!(io, t, x) for x in a.args)
        write(io, op); return n + 1
    elseif a isa Base.RefValue{String}
        s = a[]; write(io, 0x04, UInt32(sizeof(s))); write(io, s); return 1
    elseif a isa Bool
        write(io, 0x05, UInt8(a)); return 1
    elseif a isa Integer
        write(io, 0x02, Int64(a)); return 1
    elseif a isa AbstractFloat
        write(io, 0x03, Float64(a)); return 1
    end
    throw(ArgumentError("cannot serialise $(typeof(a))"))
end

function expr_bytes(t::DFTable, e)
    body = IOBuffer(); n = emit!(body, t, e)
    io = IOBuffer(); write(io, UInt32(n)); write(io, take!(body)); take!(io)
end

function plan_bytes(v::DFView)
    io = IOBuffer()
    write(io, 0x31504644 % UInt32, UInt32(length(v.selection.queue)))
    for el in v.selection.queue
        if el isa BlockBroadcasting
            write(io, 0x03); write(io, expr_bytes(v.table, el))
        elseif el isa AbstractRange
            write(io, 0x01, Int64(first(el)), Int64(step(el)), Int64(last(el)))
        elseif el isa Integer
            write(io, 0x01, Int64(el), Int64(1), Int64(el))
        else
            idx = collect(Int64, el); write(io, 0x02, UInt32(length(idx))); write(io, idx)
        end
    end
    write(io, UInt32(length(v.projection.cols)))
    for c in values(v.projection.cols)
        if c isa ColRef
            write(io, 0x01, Int64(colid(v.table, c.name)))
        else
            write(io, 0x02); write(io, expr_bytes(v.table, c))
        end
    end
    take!(io)
end

function with_scan(f, v::DFView)
    plan = plan_bytes(v)
    s = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:dfdb_scan_prepare, LIB), Int32, (Ptr{Cvoid}, Ptr{UInt8}, Int64, Ref{Ptr{Cvoid}}), handle(v.table), plan, Int64(length(plan)), s))
    try
        f(s[])
    finally
        ccall((:dfdb_scan_free, LIB), Int32, (Ptr{Cvoid},), s[])
    end
end

# ---- consumers -------------------------------------------------------------------------------------------------------
# nrow(v): view.jl:192-206.  On a sharded table the count is over all shards (ncclAllGather inside the library).
function nrow(v::DFView)
    with_scan(v) do s
        n = Ref{Int64}(0)
        check(ccall((:dfdb_scan_count_all, LIB), Int32, (Ptr{Cvoid}, Ref{Int64}), s, n))
        Int(n[])
    end
end

struct OutCol
    values::Ptr{Cvoid}; missing::Ptr{UInt8}; str_sizes::Ptr{Int32}; str_chars::Ptr{UInt8}
end

# Result vectors come from the library's page-locked result arena (dfdb_host_alloc): dfdb_scan_materialize then fills them
# with one device-to-host copy at full PCIe rate.  The Array does not own the memory; a finalizer hands it back.
function pinned_vector(::Type{T}, n::Integer) where {T}
    p = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:dfdb_host_alloc, LIB), Int32, (Int64, Ref{Ptr{Cvoid}}), Int64(max(n, 1) * sizeof(T)), p))
    a = unsafe_wrap(Array, Ptr{T}(p[]), n; own = false)
    finalizer(_ -> ccall((:dfdb_host_free, LIB), Int32, (Ptr{Cvoid},), p[]), a)
    a
end

# A FlatStringsVector as the reference lays it out (FlatStringsVectors.jl:5-9: offsets::Vector{Int64}, sizes::Vector{Int32},
# data::String, datasize::Int).  `data` is a Julia String, so the gathered chars are copied once (unsafe_string); sizes are
# copied out of the arena into an ordinary Vector{Int32} because the struct keeps them and may resize them (push!).  The
# fields are filled directly: the inner constructor's `total == offsets[end] + sizes[end]` assertion
# (FlatStringsVectors.jl:18-28) does not hold when the last element is missing (size -1), and the keyword constructor
# (:54-59) passes uninitialised offsets to it.
function flat_strings(::Type{T}, sizes::Vector{Int32}, chars::Vector{UInt8}, nbytes::Integer) where {T}
    r = FlatStringsVector{T}(sizehint = 0)
    r.sizes = copy(sizes)
    r.offsets = Vector{Int64}(undef, length(sizes))
    off = Int64(0)
    @inbounds for i in eachindex(sizes)                       # unsafe_remake_offsets!, FlatStringsVectors.jl:61-70
        r.offsets[i] = off
        off += max(sizes[i], Int32(0))
    end
    r.data = GC.@preserve chars unsafe_string(pointer(chars), nbytes)
    r.datasize = Int(nbytes)
    r
end

# materialize(v::DFView): materialization.jl:27-40 (sizes first = the reference's nrow pass, then fill)
function materialize(v::DFView)
    names = keys(v.projection)
    types = [DataFrameDBs.coltype(v.projection, i) for i in 1:length(names)]
    with_scan(v) do s
        n = Ref{Int64}(0); sb = zeros(Int64, length(names))
        check(ccall((:dfdb_scan_materialize_sizes, LIB), Int32, (Ptr{Cvoid}, Ref{Int64}, Ptr{Int64}), s, n, sb))
        bufs = Any[]; outs = OutCol[]
        for (i, T) in enumerate(types)
            B = Base.nonmissingtype(T)
            if B === String
                sizes = pinned_vector(Int32, n[]); chars = pinned_vector(UInt8, sb[i])
                push!(bufs, (sizes, chars)); push!(outs, OutCol(C_NULL, C_NULL, pointer(sizes), pointer(chars)))
            else
                vals = pinned_vector(B, n[]); miss = T === B ? UInt8[] : pinned_vector(UInt8, n[])
                push!(bufs, (vals, miss)); push!(outs, OutCol(pointer(vals), T === B ? C_NULL : pointer(miss), C_NULL, C_NULL))
            end
        end
        GC.@preserve bufs check(ccall((:dfdb_scan_materialize, LIB), Int32, (Ptr{Cvoid}, Ptr{OutCol}, Int32), s, outs, Int32(length(outs))))
        cols = map(enumerate(zip(types, bufs))) do (i, (T, b))
            B = Base.nonmissingtype(T)
            if B === String
                flat_strings(T, b[1], b[2], sb[i])
            elseif T === B
                b[1]
            else
                r = Vector{T}(b[1]); r[b[2] .!= 0] .= missing; r
            end
        end
        DataFrames.DataFrame(collect(cols), collect(names), copycols = false)
    end
end
materialize(c::DFColumn) = materialize(c.view)[!, 1]     # materialization.jl:46-52

struct Agg
    count::Int64; nmissing::Int64; sum_i64::Int64; sum_f64::Float64; sum_f64_lo::Float64
    min_i64::Int64; max_i64::Int64; min_f64::Float64; max_f64::Float64; has_nan::Int32; value_class::Int32
end

# one fused GPU pass instead of the Base folds over iterate(::DFColumn) (column.jl:102-126); on a sharded table the
# per-shard partials are combined inside the library (dfdb_scan_aggregate_all: ncclAllGather + fixed rank-order fold)
function aggregate(c::DFColumn)
    with_scan(c.view) do s
        a = Ref{Agg}()
        check(ccall((:dfdb_scan_aggregate_all, LIB), Int32, (Ptr{Cvoid}, Int32, Ref{Agg}), s, Int32(0), a))
        a[]
    end
end

function sum(c::DFColumn{T}) where {T}
    a = aggregate(c)
    a.nmissing > 0 && return missing
    Base.nonmissingtype(T) <: AbstractFloat ? a.sum_f64 + a.sum_f64_lo : a.value_class == 2 ? reinterpret(UInt64, a.sum_i64) : a.sum_i64
end
function _extreme(c::DFColumn{T}, pick_i, pick_f) where {T}
    a = aggregate(c)
    a.count == 0 && throw(ArgumentError("reducing over an empty collection is not allowed"))
    a.nmissing > 0 && return missing
    Base.nonmissingtype(T) <: AbstractFloat ? pick_f(a) : convert(Base.nonmissingtype(T), pick_i(a))
end
minimum(c::DFColumn) = _extreme(c, a -> a.min_i64, a -> a.min_f64)
maximum(c::DFColumn) = _extreme(c, a -> a.max_i64, a -> a.max_f64)

# Base.unique over iterate(::DFColumn) (column.jl:102-126): the distinct values in order of first appearance, isequal, as a
# Vector{eltype(c)}.  Group table on the device per shard; on a sharded table the shards' results are all-gathered inside the
# library and merged on the device (dfdb_scan_unique_all), so every rank returns the whole column's result.
function unique(c::DFColumn{T}) where {T}
    B = Base.nonmissingtype(T)
    with_scan(c.view) do s
        n = Ref{Int64}(0); nb = Ref{Int64}(0)
        check(ccall((:dfdb_scan_unique_all, LIB), Int32, (Ptr{Cvoid}, Int32, Ref{Int64}, Ref{Int64}), s, Int32(0), n, nb))
        if B === String
            sizes = Vector{Int32}(undef, n[]); chars = Vector{UInt8}(undef, max(nb[], 1))
            GC.@preserve sizes chars check(ccall((:dfdb_scan_unique_values, LIB), Int32, (Ptr{Cvoid}, Ref{OutCol}),
                                                 s, OutCol(C_NULL, C_NULL, pointer(sizes), pointer(chars))))
            r = Vector{T}(undef, n[]); off = 0
            for i in 1:n[]
                if sizes[i] < 0
                    r[i] = missing
                else
                    r[i] = GC.@preserve chars unsafe_string(pointer(chars) + off, sizes[i]); off += sizes[i]
                end
            end
            r
        else
            vals = Vector{B}(undef, n[]); miss = zeros(UInt8, T === B ? 0 : n[])
            GC.@preserve vals miss check(ccall((:dfdb_scan_unique_values, LIB), Int32, (Ptr{Cvoid}, Ref{OutCol}),
                                               s, OutCol(pointer(vals), T === B ? C_NULL : pointer(miss), C_NULL, C_NULL)))
            T === B ? vals : (r = Vector{T}(vals); r[miss .!= 0] .= missing; r)
        end
    end
end
# the two halves of dfdb_scan_unique_all for hosts that carry the per-rank results with their own transport: the shard-local
# pass on scan `s`, and the merge of the ranks' results (`parts` in rank order, laid out as dfdb_scan_unique_values fills them)
unique_local!(s::Ptr{Cvoid}, n::Ref{Int64}, nb::Ref{Int64}) =
    check(ccall((:dfdb_scan_unique, LIB), Int32, (Ptr{Cvoid}, Int32, Ref{Int64}, Ref{Int64}), s, Int32(0), n, nb))
unique_merge!(s::Ptr{Cvoid}, parts::Vector{OutCol}, part_n::Vector{Int64}, part_nb::Vector{Int64}, n::Ref{Int64}, nb::Ref{Int64}) =
    check(ccall((:dfdb_scan_unique_merge, LIB), Int32, (Ptr{Cvoid}, Ptr{OutCol}, Ptr{Int64}, Ptr{Int64}, Int32, Ref{Int64}, Ref{Int64}),
                s, parts, part_n, part_nb, Int32(length(parts)), n, nb))

# Statistics.median / Statistics.quantile over iterate(::DFColumn) (column.jl:102-126; Statistics collects the column and sorts
# it on the host): the exact order statistics come from the device (MSD radix select over the gathered values,
# dfdb_scan_order_*), the Statistics arithmetic stays here.  On a sharded table only the aggs and each round's bin counts
# travel between the ranks, inside the library, and every rank returns the same value.
const ORDER_MAX_RANKS = 4096            # DFDB_ORDER_MAX_RANKS
function order_prepare(s::Ptr{Cvoid})
    a = Ref{Agg}()
    check(ccall((:dfdb_scan_order_prepare_all, LIB), Int32, (Ptr{Cvoid}, Int32, Ref{Agg}), s, Int32(0), a))
    a[]
end
# the ranks[i]-th smallest non-missing value (isless) of the prepared column, as a B
function order_stats(s::Ptr{Cvoid}, ranks::Vector{Int64}, ::Type{B}) where {B}
    out = Vector{B}(undef, length(ranks))
    for lo in 1:ORDER_MAX_RANKS:length(ranks)
        r = ranks[lo:min(lo + ORDER_MAX_RANKS - 1, end)]
        v = Vector{B}(undef, length(r))
        GC.@preserve r v check(ccall((:dfdb_scan_order_stats_all, LIB), Int32, (Ptr{Cvoid}, Ptr{Int64}, Int32, Ptr{Cvoid}),
                                     s, r, Int32(length(r)), v))
        out[lo:lo + length(r) - 1] = v
    end
    out
end
# one radix-select round and the values, for hosts that carry the per-round counts with their own transport (the first round
# of a query passes `global_counts` = C_NULL; see dfdb_scan_order_round)
order_prepare_local!(s::Ptr{Cvoid}, a::Ref{Agg}) = check(ccall((:dfdb_scan_order_prepare, LIB), Int32, (Ptr{Cvoid}, Int32, Ref{Agg}), s, Int32(0), a))
order_round!(s::Ptr{Cvoid}, whole::Ref{Agg}, ranks::Vector{Int64}, global_counts, nglobal::Integer, local_counts::Vector{Int64}, nlocal::Ref{Int64}) =
    check(ccall((:dfdb_scan_order_round, LIB), Int32, (Ptr{Cvoid}, Ref{Agg}, Ptr{Int64}, Int32, Ptr{Int64}, Int64, Ptr{Int64}, Int64, Ref{Int64}),
                s, whole, ranks, Int32(length(ranks)), global_counts, Int64(nglobal), local_counts, Int64(length(local_counts)), nlocal))
order_values!(s::Ptr{Cvoid}, values::Vector) = check(ccall((:dfdb_scan_order_values, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}), s, values))

function median(c::DFColumn{T}, skip::Bool) where {T}
    B = Base.nonmissingtype(T)
    with_scan(c.view) do s
        a = order_prepare(s)
        n = a.count - a.nmissing
        a.count == 0 && throw(ArgumentError("median of an empty collection is undefined, median(Any[])"))
        a.nmissing > 0 && !skip && return missing
        n == 0 && throw(ArgumentError("median of an empty collection is undefined, median(Any[])"))
        a.has_nan != 0 && return convert(B, NaN)
        isodd(n) ? Statistics.middle(order_stats(s, [(n + 1) ÷ 2], B)[1]) : Statistics.middle(order_stats(s, [n ÷ 2, n ÷ 2 + 1], B)...)
    end
end
# Statistics._quantile with alpha = beta = 1, restated: only v[j] and v[j + 1] of the sorted values are read
function quantile(c::DFColumn{T}, p, skip::Bool) where {T}
    B = Base.nonmissingtype(T)
    ps = p isa Real ? [p] : collect(p)
    all(x -> 0 <= x <= 1, ps) || throw(ArgumentError("input probability out of [0,1] range"))
    with_scan(c.view) do s
        a = order_prepare(s)
        n = a.count - a.nmissing
        (a.count == 0 || n == 0) && throw(ArgumentError("empty data vector"))
        (a.nmissing > 0 && !skip || a.has_nan != 0) && throw(ArgumentError("quantiles are undefined in presence of NaNs or missing values"))
        js = [clamp(trunc(Int, fma(n, x, 1 - x)), 1, n - 1) for x in ps]
        ranks = n == 1 ? [1] : sort!(unique!(vcat(js, js .+ 1)))
        pick = Dict(zip(ranks, order_stats(s, ranks, B)))
        out = map(ps) do x
            aleph = fma(n, x, 1 - x)
            j = clamp(trunc(Int, aleph), 1, n - 1)
            γ = clamp(aleph - j, 0, 1)
            va, vb = n == 1 ? (pick[1], pick[1]) : (pick[j], pick[j + 1])
            isfinite(va) && isfinite(vb) && va ≈ vb ? va + γ * (vb - va) : (1 - γ) * va + γ * vb
        end
        p isa Real ? out[1] : out
    end
end

# ---- the rows beyond the scan path (SURVEY.md 8f): zone maps, write path, group-by ----------------------------------------
"""
    B200.build_zonemaps!(t::DFTable)

Per-block (min, max, null count) of every fixed-width numeric column, computed on the device and written beside the column
files as the optional sidecar `<id>.zmap` (the reference ignores it).  Predicates of `column <cmp> constant` terms then skip
the blocks their constants rule out; `open_table` + `enable!` pick the sidecars up again later.
"""
build_zonemaps!(t::DFTable) = (check(ccall((:dfdb_table_build_zonemaps, LIB), Int32, (Ptr{Cvoid}, Ptr{Int64}, Int32), handle(t), C_NULL, Int32(0))); t)

# write_column (columns.jl:65-84) for a Vector of a stored bits type: bodies assembled, LZ4-compressed and compacted on the
# device, framed on the host (make_column_file + commit_block_write!).  add_column! (table.jl:96-124) calls it instead of
# write_column_from_iterator when B200 is enabled; meta.bin is still written by the reference's own write_table_meta.
function write_column_file(t::DFTable, id::Integer, data::Vector{T}) where {T}
    start()
    isbitstype(T) || throw(ArgumentError("$(T) is not written by the device path"))
    comp = Ref{Int64}(0); unc = Ref{Int64}(0)
    GC.@preserve data check(ccall((:dfdb_write_column_file, LIB), Int32,
        (Cstring, Int64, Cstring, Int64, Int64, Ptr{Cvoid}, Ptr{UInt8}, Ptr{Int32}, Ptr{UInt8}, Int64, Ref{Int64}, Ref{Int64}),
        t.path, Int64(id), DataFrameDBs.ColumnTypes.typestring(T), Int64(DataFrameDBs.blocksize(t)), Int64(length(data)),
        pointer(data), C_NULL, C_NULL, C_NULL, Int64(0), comp, unc))
    (compressed = comp[], uncompressed = unc[])
end

# groupreduce(view, by; cols...) -- finishes the stub in src/tables/aggregate.jl:1-36, over every shard: each rank's groups are
# all-gathered inside the library, merged on the device and folded in rank order (dfdb_scan_groupreduce_all), so every rank
# returns the whole table's groups.  Returns the key values (one vector per key column, `missing` where flagged), the 1-based
# table rows where the groups first appear and one Agg per (value column, group).
function groupreduce(v::DFView, by::Tuple{Vararg{Symbol}}, vals::Tuple{Vararg{Symbol}})
    gv = v[:, [by..., vals...]]
    with_scan(gv) do s
        ng = Ref{Int64}(0)
        kp = Int32.(0:length(by)-1); vp = Int32.(length(by):length(by)+length(vals)-1)
        check(ccall((:dfdb_scan_groupreduce_all, LIB), Int32, (Ptr{Cvoid}, Ptr{Int32}, Int32, Ptr{Int32}, Int32, Ref{Int64}),
                    s, kp, Int32(length(kp)), vp, Int32(length(vp)), ng))
        first = Vector{Int64}(undef, ng[]); aggs = Vector{Agg}(undef, ng[] * length(vals))
        check(ccall((:dfdb_scan_group_results, LIB), Int32, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Agg}), s, first, aggs))
        (keys = group_keys(s, gv, length(by), ng[]), first_rows = first, aggs = reshape(aggs, length(vals), :))
    end
end
# the key columns of the handle's group-by result, as Vector{eltype(column)}
function group_keys(s::Ptr{Cvoid}, gv::DFView, nkeys::Int, n::Int64)
    nb = zeros(Int64, nkeys)
    check(ccall((:dfdb_scan_group_key_bytes, LIB), Int32, (Ptr{Cvoid}, Ptr{Int64}), s, nb))
    Ts = [DataFrameDBs.coltype(gv.projection, k) for k in 1:nkeys]
    bufs = map(1:nkeys) do k
        B = Base.nonmissingtype(Ts[k])
        B === String ? (Vector{Int32}(undef, n), Vector{UInt8}(undef, max(nb[k], 1))) : (Vector{B}(undef, n), zeros(UInt8, n))
    end
    outs = [Ts[k] <: Union{String, Missing} ? OutCol(C_NULL, C_NULL, pointer(bufs[k][1]), pointer(bufs[k][2])) :
                                               OutCol(pointer(bufs[k][1]), pointer(bufs[k][2]), C_NULL, C_NULL) for k in 1:nkeys]
    GC.@preserve bufs check(ccall((:dfdb_scan_group_keys, LIB), Int32, (Ptr{Cvoid}, Ptr{OutCol}, Int32), s, outs, Int32(nkeys)))
    map(1:nkeys) do k
        T = Ts[k]; a, b = bufs[k]
        if Base.nonmissingtype(T) === String
            r = Vector{T}(undef, n); off = 0
            for i in 1:n
                a[i] < 0 ? (r[i] = missing) : (r[i] = GC.@preserve b unsafe_string(pointer(b) + off, a[i]); off += a[i])
            end
            r
        else
            T === eltype(a) ? a : (r = Vector{T}(a); r[b .!= 0] .= missing; r)
        end
    end
end
# the two halves of dfdb_scan_groupreduce_all for hosts that carry the per-rank results with their own transport: the
# shard-local pass on scan `s` (read it back with dfdb_scan_group_results / _group_key_bytes / _group_keys), and the merge of
# the ranks' results (`keys` nparts x nkeys in rank order, laid out as dfdb_scan_group_keys fills them; `first` and `aggs`
# concatenated in rank order)
groupreduce_local!(s::Ptr{Cvoid}, kp::Vector{Int32}, vp::Vector{Int32}, ng::Ref{Int64}) =
    check(ccall((:dfdb_scan_groupreduce, LIB), Int32, (Ptr{Cvoid}, Ptr{Int32}, Int32, Ptr{Int32}, Int32, Ref{Int64}),
                s, kp, Int32(length(kp)), vp, Int32(length(vp)), ng))
groupreduce_merge!(s::Ptr{Cvoid}, kp::Vector{Int32}, nvals::Integer, keys::Vector{OutCol}, first::Vector{Int64}, aggs::Vector{Agg},
                   part_n::Vector{Int64}, part_nb::Vector{Int64}, ng::Ref{Int64}) =
    check(ccall((:dfdb_scan_groupreduce_merge, LIB), Int32,
                (Ptr{Cvoid}, Ptr{Int32}, Int32, Int32, Ptr{OutCol}, Ptr{Int64}, Ptr{Agg}, Ptr{Int64}, Ptr{Int64}, Int32, Ref{Int64}),
                s, kp, Int32(length(kp)), Int32(nvals), keys, first, aggs, part_n, part_nb, Int32(length(part_n)), ng))

end # module B200

# ---- the hooks: methods of the package's own generic functions (this file is part of the package) --------------------------
# nrow(::DFView) and materialize(::DFView) get their one-line hooks from the patch in INTEGRATION.md; length / size of a
# DFColumn go through nrow (column.jl:46-52) and need nothing.  The reductions do not exist in the reference at all (they are
# Base's generic folds over iterate(::DFColumn), column.jl:102-126), so these methods are new, not overwritten; off the GPU
# they fall through to the same generic fold.
Base.sum(c::DFColumn) = B200.enabled(c.view.table) ? B200.sum(c) : invoke(Base.sum, Tuple{Any}, c)
Base.minimum(c::DFColumn) = B200.enabled(c.view.table) ? B200.minimum(c) : invoke(Base.minimum, Tuple{Any}, c)
Base.maximum(c::DFColumn) = B200.enabled(c.view.table) ? B200.maximum(c) : invoke(Base.maximum, Tuple{Any}, c)
Base.unique(c::DFColumn) = B200.enabled(c.view.table) ? B200.unique(c) : invoke(Base.unique, Tuple{Any}, c)
# Statistics.median / quantile (and their skipmissing forms) collect the column and sort it; on the GPU the order statistics
# come from the device.  Non-default alpha / beta fall through to the generic method.
import Statistics
Statistics.median(c::DFColumn) = B200.enabled(c.view.table) ? B200.median(c, false) : invoke(Statistics.median, Tuple{Any}, c)
Statistics.median(c::Base.SkipMissing{<:DFColumn}) =
    B200.enabled(c.x.view.table) ? B200.median(c.x, true) : invoke(Statistics.median, Tuple{Any}, c)
Statistics.quantile(c::DFColumn, p; sorted::Bool = false, alpha::Real = 1.0, beta::Real = alpha) =
    B200.enabled(c.view.table) && alpha == 1 && beta == 1 ? B200.quantile(c, p, false) :
    invoke(Statistics.quantile, Tuple{Any,Any}, c, p; sorted = sorted, alpha = alpha, beta = beta)
Statistics.quantile(c::Base.SkipMissing{<:DFColumn}, p; sorted::Bool = false, alpha::Real = 1.0, beta::Real = alpha) =
    B200.enabled(c.x.view.table) && alpha == 1 && beta == 1 ? B200.quantile(c.x, p, true) :
    invoke(Statistics.quantile, Tuple{Any,Any}, c, p; sorted = sorted, alpha = alpha, beta = beta)
