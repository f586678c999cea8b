# DynamicSparseArraysB200 — Julia glue over libdsa.so (include/dsa.h).
#
# Drop-in for DynamicSparseArrays.jl's hot path: same exported names (src/DynamicSparseArrays.jl:5-16), the structures
# live in B200 HBM behind opaque handles, every hot operation is one `ccall`.  Written against the C ABI; Julia is not
# installed in the build image, so this file is NOT executed by the test-suite — the executable statement of the same
# glue logic is dynamicsparsearrays.jl_b200/api.py (tested through tests/test_gpu_parity.py).
module DynamicSparseArraysB200

using SparseArrays

export DynamicSparseVector, DynamicSparseMatrix, DynamicMatrixColView, dynamicsparsevec, dynamicsparse, nbpartitions,
       deletecolumn!, deleterow!, addrow!, closefillmode!, shrink_size!,
       set_batch!, stage_batch!, apply_staged!        # additions: batched and double-buffered writes (no reference counterpart)
export spmspv                                          # addition: sparse product in the reference's summation order

const libdsa = get(ENV, "LIBDSA", joinpath(@__DIR__, "..", "dynamicsparsearrays.jl_b200", "libdsa.so"))
const COMBINE = Dict{Any,Cint}(+ => 0, * => 1, max => 5, min => 4)

function _check(code::Cint)
    code == 0 && return
    msg = unsafe_string(ccall((:dsa_last_error, libdsa), Cstring, ()))
    code == 1 && throw(ArgumentError(msg))       # DSA_ERR_ARGUMENT  (pcsr.jl:208, vector.jl:50)
    code == 2 && throw(BoundsError(msg))         # DSA_ERR_BOUNDS    (pcsr.jl:190)
    error(msg)                                   # DSA_ERR_ERROR / CUDA / OOM -> ErrorException
end

# ------------------------------------------------------------------------------------------ vector (vector.jl)
mutable struct DynamicSparseVector <: AbstractSparseVector{Float64,Int64}
    h::Ptr{Cvoid}
    pk::Vector{Int64}      # queued single writes, flushed as one batch before any read
    pv::Vector{Float64}
    function DynamicSparseVector(h)
        v = new(h, Int64[], Float64[])
        finalizer(x -> ccall((:dsa_vec_destroy, libdsa), Cint, (Ptr{Cvoid},), x.h), v)
        return v
    end
end

function dynamicsparsevec(I::Vector{Int64}, V::Vector{Float64}, combine::Function = +, n = nothing)   # vector.jl:44-62
    length(I) == length(V) || throw(ArgumentError("keys & nonzeros vectors must have same length."))
    h = Ref{Ptr{Cvoid}}()
    _check(ccall((:dsa_vec_build, libdsa), Cint, (Ptr{Int64}, Ptr{Float64}, Int64, Cint, Int64, Cint, Ref{Ptr{Cvoid}}),
                 I, V, length(I), COMBINE[combine], n === nothing ? 0 : n, n === nothing ? 0 : 1, h))
    return DynamicSparseVector(h[])
end

function flush!(v::DynamicSparseVector)
    isempty(v.pk) && return
    _check(ccall((:dsa_vec_set_batch, libdsa), Cint, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Float64}, Int64), v.h, v.pk, v.pv, length(v.pk)))
    empty!(v.pk); empty!(v.pv)
    return
end

function Base.setindex!(v::DynamicSparseVector, value, key::Integer)   # vector.jl:76-81
    push!(v.pk, key); push!(v.pv, value)
    return v
end

function Base.getindex(v::DynamicSparseVector, key::Integer)            # vector.jl:72
    flush!(v)
    out = Ref{Float64}(0.0)
    _check(ccall((:dsa_vec_get_batch, libdsa), Cint, (Ptr{Cvoid}, Ref{Int64}, Int64, Ref{Float64}), v.h, Ref(Int64(key)), 1, out))
    return out[]
end
Base.getindex(v::DynamicSparseVector, ::Colon) = v

function _info(v::DynamicSparseVector)
    flush!(v)
    out = Vector{Int64}(undef, 6)
    _check(ccall((:dsa_vec_info, libdsa), Cint, (Ptr{Cvoid}, Ptr{Int64}), v.h, out))
    return out   # capacity, segment_capacity, nb_segments, nnz, height, n
end
Base.length(v::DynamicSparseVector) = _info(v)[6]
Base.size(v::DynamicSparseVector) = (length(v),)
SparseArrays.nnz(v::DynamicSparseVector) = _info(v)[4]

function _nonzeros(v::DynamicSparseVector)                               # vector.jl:93-109
    n = nnz(v)
    k = Vector{Int64}(undef, n); x = Vector{Float64}(undef, n); cnt = Ref{Int64}(0)
    _check(ccall((:dsa_vec_nonzeros, libdsa), Cint, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Float64}, Int64, Ref{Int64}), v.h, k, x, n, cnt))
    return k, x
end
SparseArrays.nonzeroinds(v::DynamicSparseVector) = _nonzeros(v)[1]
SparseArrays.nonzeros(v::DynamicSparseVector) = _nonzeros(v)[2]
Base.iterate(v::DynamicSparseVector) = (kv = collect(zip(_nonzeros(v)...)); isempty(kv) ? nothing : (kv[1], (kv, 2)))
Base.iterate(::DynamicSparseVector, st) = st[2] > length(st[1]) ? nothing : (st[1][st[2]], (st[1], st[2] + 1))

function shrink_size!(v::DynamicSparseVector)                            # vector.jl:64
    flush!(v)
    out = Ref{Int64}(0)
    _check(ccall((:dsa_vec_shrink_size, libdsa), Cint, (Ptr{Cvoid}, Ref{Int64}), v.h, out))
    return out[]
end
Base.copy(::DynamicSparseVector) = error("copy of a dynamic sparse vector not implemented.")   # vector.jl:90
function Base.deepcopy_internal(v::DynamicSparseVector, ::IdDict)
    flush!(v)
    h = Ref{Ptr{Cvoid}}()
    _check(ccall((:dsa_vec_clone, libdsa), Cint, (Ptr{Cvoid}, Ref{Ptr{Cvoid}}), v.h, h))
    return DynamicSparseVector(h[])
end

# ------------------------------------------------------------------------------------------ matrix (matrix.jl, buffer.jl)
mutable struct Buffer                                                    # buffer.jl:1-4 — stays on the host
    rowmajor_coo::Dict{Int64,Tuple{Vector{Int64},Vector{Float64}}}
    length::Int
end
Buffer() = Buffer(Dict{Int64,Tuple{Vector{Int64},Vector{Float64}}}(), 0)

mutable struct DynamicSparseMatrix
    h::Ptr{Cvoid}
    m::Int64
    n::Int64
    fillmode::Bool
    buffer::Union{Buffer,Nothing}
    pr::Vector{Int64}; pc::Vector{Int64}; pv::Vector{Float64}           # queued single writes
    staged::Vector{Any}                                                  # host arrays of the batches staged in the library, oldest first
    function DynamicSparseMatrix(h, fillmode)
        A = new(h, 0, 0, fillmode, fillmode ? Buffer() : nothing, Int64[], Int64[], Float64[], Any[])
        finalizer(x -> x.h != C_NULL && ccall((:dsa_matrix_destroy, libdsa), Cint, (Ptr{Cvoid},), x.h), A)
        return A
    end
end

function dynamicsparse(I::Vector{Int64}, J::Vector{Int64}, V::Vector{Float64}, m = nothing, n = nothing)   # matrix.jl:15-19
    length(I) == length(J) == length(V) || throw(ArgumentError("rows, columns, and nonzeros do not have same length."))
    h = Ref{Ptr{Cvoid}}()
    _check(ccall((:dsa_matrix_build_coo, libdsa), Cint,
                 (Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Int64, Int64, Int64, Cint, Cint, Ref{Ptr{Cvoid}}),
                 I, J, V, length(I),
                 # each missing dimension defaults on its own: m = _guess_length(I), n = _guess_length(J)  (matrix.jl:15, vector.jl:6)
                 m === nothing ? maximum(I; init = 0) : m, n === nothing ? maximum(J; init = 0) : n,
                 (m === nothing && n === nothing) ? 0 : 1, 0, h))
    return DynamicSparseMatrix(h[], false)
end

function dynamicsparse(::Type{Int64}, ::Type{Int64}, ::Type{Float64}; fill_mode = true)                  # matrix.jl:31-41
    fill_mode && return DynamicSparseMatrix(C_NULL, true)
    h = Ref{Ptr{Cvoid}}()
    _check(ccall((:dsa_matrix_create, libdsa), Cint, (Ref{Ptr{Cvoid}},), h))
    return DynamicSparseMatrix(h[], false)
end

# Everything written so far becomes visible, in arrival order: staged batches first (stage_batch! flushes the queue in front
# of itself, so they are older than any queued write), then the queued single writes.  The queue is emptied only once the
# library has applied it: a failed flush loses nothing.
function flush!(A::DynamicSparseMatrix)
    while !isempty(A.staged)
        apply_staged!(A)
    end
    isempty(A.pv) && return
    _check(ccall((:dsa_matrix_set_batch, libdsa), Cint, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Int64),
                 A.h, A.pr, A.pc, A.pv, length(A.pv)))
    empty!(A.pr); empty!(A.pc); empty!(A.pv)
    return
end

# Batched setindex! (no reference counterpart: the reference loops, matrix.jl:119-121): last writer wins, 0.0 deletes.
function set_batch!(A::DynamicSparseMatrix, rows::Vector{Int64}, cols::Vector{Int64}, vals::Vector{Float64})
    A.fillmode && error("Cannot apply a batch in fill mode")
    length(rows) == length(cols) == length(vals) || throw(ArgumentError("rows, columns, and nonzeros do not have same length."))
    flush!(A)
    _check(ccall((:dsa_matrix_set_batch, libdsa), Cint, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Int64),
                 A.h, rows, cols, vals, length(vals)))
    return A
end

# Double-buffered flush: stage_batch! starts the host->device copy of a batch and returns; apply_staged! applies the oldest
# staged batch (two slots).  The arrays must stay reachable until their apply_staged! has returned (GC.@preserve / keep a reference).
function stage_batch!(A::DynamicSparseMatrix, rows::Vector{Int64}, cols::Vector{Int64}, vals::Vector{Float64})
    A.fillmode && error("Cannot apply a batch in fill mode")
    length(rows) == length(cols) == length(vals) || throw(ArgumentError("rows, columns, and nonzeros do not have same length."))
    isempty(A.pv) || flush!(A)                                          # earlier single writes (and the batches staged before them) go first
    _check(ccall((:dsa_matrix_stage_batch, libdsa), Cint, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Int64),
                 A.h, rows, cols, vals, length(vals)))
    push!(A.staged, (rows, cols, vals))                                 # keeps the host arrays reachable until the copy is consumed
    return A
end
function apply_staged!(A::DynamicSparseMatrix)                           # reads, writes, deletes and copies drain staged batches through flush!
    _check(ccall((:dsa_matrix_apply_staged, libdsa), Cint, (Ptr{Cvoid},), A.h))
    isempty(A.staged) || popfirst!(A.staged)
    return A
end

function Base.setindex!(A::DynamicSparseMatrix, val, row::Integer, col::Integer)                          # matrix.jl:43-62
    if A.fillmode
        if !iszero(val)
            A.m = max(A.m, row); A.n = max(A.n, col)
        end
        r = get!(A.buffer.rowmajor_coo, row, (Int64[], Float64[]))                                        # buffer.jl:20-31
        push!(r[1], col); push!(r[2], val); A.buffer.length += 1
    else
        # device contract: the error fires at the offending write, like the reference's setindex! would
        (row >= 1 && col >= 1) || throw(ArgumentError("row and column keys must be >= 1 (key 0 is the semaphore key, pcsr.jl:23)"))
        push!(A.pr, row); push!(A.pc, col); push!(A.pv, val)
    end
    return A
end

function Base.getindex(A::DynamicSparseMatrix, row::Integer, col::Integer)                                # matrix.jl:64-68
    A.fillmode && error("getindex(row, col) is not available in fill mode")
    flush!(A)
    out = Ref{Float64}(0.0)
    _check(ccall((:dsa_matrix_get_batch, libdsa), Cint, (Ptr{Cvoid}, Cint, Ref{Int64}, Ref{Int64}, Int64, Ref{Float64}),
                 A.h, 0, Ref(Int64(row)), Ref(Int64(col)), 1, out))
    return out[]
end

function _minfo(A::DynamicSparseMatrix, which)
    flush!(A)
    out = Vector{Int64}(undef, 10)
    _check(ccall((:dsa_matrix_info, libdsa), Cint, (Ptr{Cvoid}, Cint, Ptr{Int64}), A.h, which, out))
    return out
end
Base.size(A::DynamicSparseMatrix) = A.fillmode ? (A.m, A.n) : (i = _minfo(A, 0); (i[8], i[9]))
Base.size(A::DynamicSparseMatrix, d) = size(A)[d]
SparseArrays.nnz(A::DynamicSparseMatrix) = _minfo(A, 1)[10]                                               # matrix.jl:91
struct Orientation; A::DynamicSparseMatrix; which::Cint; end
Base.getproperty(A::DynamicSparseMatrix, s::Symbol) =
    s === :colmajor ? Orientation(A, 0) : s === :rowmajor ? Orientation(A, 1) : getfield(A, s)
nbpartitions(o::Orientation) = _minfo(o.A, o.which)[6]                                                    # pcsr.jl:21-22

function closefillmode!(A::DynamicSparseMatrix)                                                           # matrix.jl:126-134
    A.fillmode || error("Cannot close fill mode because matrix is not in fill mode.")
    I = Int64[]; J = Int64[]; V = Float64[]
    for (rowid, (cols, vals)) in A.buffer.rowmajor_coo                                                    # buffer.jl:33-50
        append!(I, fill(rowid, length(vals))); append!(J, cols); append!(V, vals)
    end
    h = Ref{Ptr{Cvoid}}()
    _check(ccall((:dsa_matrix_build_coo, libdsa), Cint,
                 (Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Int64, Int64, Int64, Cint, Cint, Ref{Ptr{Cvoid}}),
                 I, J, V, length(I), A.m, A.n, 1, 0, h))
    A.h = h[]; A.fillmode = false; A.buffer = nothing
    return true
end

function addrow!(A::DynamicSparseMatrix, row::Integer, colids::Vector{Int64}, vals::Vector{Float64})      # matrix.jl:113-124
    if A.fillmode
        haskey(A.buffer.rowmajor_coo, row) && error("Row with id $row already written in dynamic sparse matrix buffer.")
        p = sortperm(colids)
        A.buffer.rowmajor_coo[row] = (colids[p], vals[p]); A.buffer.length += length(vals)
    else
        for j in eachindex(colids); A[row, colids[j]] = vals[j]; end
    end
    return true
end

function _delete!(A::DynamicSparseMatrix, sym::Symbol, ids::Vector{Int64})
    A.fillmode && error("Cannot delete a column in fill mode")
    flush!(A)
    if sym === :dsa_matrix_delete_columns
        _check(ccall((:dsa_matrix_delete_columns, libdsa), Cint, (Ptr{Cvoid}, Ptr{Int64}, Int64), A.h, ids, length(ids)))
    else
        _check(ccall((:dsa_matrix_delete_rows, libdsa), Cint, (Ptr{Cvoid}, Ptr{Int64}, Int64), A.h, ids, length(ids)))
    end
    return true
end
deletecolumn!(A::DynamicSparseMatrix, col::Integer) = _delete!(A, :dsa_matrix_delete_columns, Int64[col])   # matrix.jl:95-102
deletecolumn!(A::DynamicSparseMatrix, cols::Vector{Int64}) = _delete!(A, :dsa_matrix_delete_columns, cols)
deleterow!(A::DynamicSparseMatrix, row::Integer) = _delete!(A, :dsa_matrix_delete_rows, Int64[row])        # matrix.jl:104-111
deleterow!(A::DynamicSparseMatrix, rows::Vector{Int64}) = _delete!(A, :dsa_matrix_delete_rows, rows)

struct DynamicMatrixColView                                                                               # views.jl:3-9
    keys::Vector{Int64}
    vals::Vector{Float64}
end
Base.iterate(v::DynamicMatrixColView, i = 1) = i > length(v.keys) ? nothing : ((v.keys[i], v.vals[i]), i + 1)
Base.length(v::DynamicMatrixColView) = length(v.keys)

function _span(A::DynamicSparseMatrix, row_not_col::Bool, id)
    flush!(A)
    cnt = Ref{Int64}(0)
    f(k, v, cap) = row_not_col ?
        ccall((:dsa_matrix_row, libdsa), Cint, (Ptr{Cvoid}, Int64, Ptr{Int64}, Ptr{Float64}, Int64, Ref{Int64}), A.h, id, k, v, cap, cnt) :
        ccall((:dsa_matrix_column, libdsa), Cint, (Ptr{Cvoid}, Int64, Ptr{Int64}, Ptr{Float64}, Int64, Ref{Int64}), A.h, id, k, v, cap, cnt)
    _check(f(C_NULL, C_NULL, 0))
    k = Vector{Int64}(undef, cnt[]); v = Vector{Float64}(undef, cnt[])
    cnt[] > 0 && _check(f(k, v, cnt[]))
    return DynamicMatrixColView(k, v)
end
function Base.view(A::DynamicSparseMatrix, ::Colon, col::Integer)                                         # matrix.jl:83-88
    A.fillmode && error("View of a column not available in fill mode.")
    return _span(A, false, col)
end
function Base.view(A::DynamicSparseMatrix, row::Integer, ::Colon)                                         # matrix.jl:70-81
    A.fillmode && error("Matrix is in fill mode, cannot create a view. However, you can use the view method on the buffer.")
    return _span(A, true, row)
end

# ------------------------------------------------------------------------------------------ products (operations.jl)
struct Transposed; array::DynamicSparseMatrix; end
Base.transpose(A::DynamicSparseMatrix) = Transposed(A)                                                    # operations.jl:5
Base.size(t::Transposed) = reverse(size(t.array))

function _mul(A::DynamicSparseMatrix, trans::Bool, xk::Vector{Int64}, xv::Vector{Float64}, n)
    flush!(A)
    cap = _minfo(A, trans ? 0 : 1)[7]
    yk = Vector{Int64}(undef, cap); yv = Vector{Float64}(undef, cap); cnt = Ref{Int64}(0)
    _check(ccall((:dsa_matrix_spmv, libdsa), Cint,
                 (Ptr{Cvoid}, Cint, Ptr{Int64}, Ptr{Float64}, Int64, Ptr{Int64}, Ptr{Float64}, Int64, Ref{Int64}),
                 A.h, trans ? 1 : 0, xk, xv, length(xk), yk, yv, cap, cnt))
    return SparseVector(n, yk[1:cnt[]], yv[1:cnt[]])                                                      # operations.jl:11-12
end
_xs(v::DynamicSparseVector) = _nonzeros(v)
_xs(v::SparseVector{Float64,Int64}) = (v.nzind, v.nzval)
const VecLike = Union{DynamicSparseVector,SparseVector{Float64,Int64}}
Base.:(*)(A::DynamicSparseMatrix, v::VecLike) = _mul(A, false, _xs(v)..., size(A, 1))                     # operations.jl:14-24
Base.:(*)(t::Transposed, v::VecLike) = _mul(t.array, true, _xs(v)..., size(t.array, 2))                   # operations.jl:26-36
Base.:(*)(v::VecLike, t::Transposed) = _mul(t.array, false, _xs(v)..., size(t.array, 1))                  # operations.jl:38-48
Base.:(*)(v::VecLike, A::DynamicSparseMatrix) = _mul(A, true, _xs(v)..., size(A, 2))                      # operations.jl:50-60

# The same products driven by v's entries, in the reference's own loop order (_mul_dyn_mat_col_loop!, operations.jl:62-105):
# the cost is the stored cells of the columns (rows) v selects, and the result is bit for bit the reference's `mat * v`.
function _spmspv(A::DynamicSparseMatrix, trans::Bool, xk::Vector{Int64}, xv::Vector{Float64}, n)
    A.fillmode && error("Matrix is in fill mode")
    flush!(A)
    cap = _minfo(A, trans ? 0 : 1)[7]
    yk = Vector{Int64}(undef, cap); yv = Vector{Float64}(undef, cap); cnt = Ref{Int64}(0)
    _check(ccall((:dsa_matrix_spmspv, libdsa), Cint,
                 (Ptr{Cvoid}, Cint, Ptr{Int64}, Ptr{Float64}, Int64, Ptr{Int64}, Ptr{Float64}, Int64, Ref{Int64}),
                 A.h, trans ? 1 : 0, xk, xv, length(xk), yk, yv, cap, cnt))
    return SparseVector(n, yk[1:cnt[]], yv[1:cnt[]])
end
spmspv(A::DynamicSparseMatrix, v::VecLike) = _spmspv(A, false, _xs(v)..., size(A, 1))                     # operations.jl:14-24
spmspv(t::Transposed, v::VecLike) = _spmspv(t.array, true, _xs(v)..., size(t.array, 2))                   # operations.jl:26-36

# k sparse right-hand sides in one call: column c of the result equals spmspv(A, X[:, c]) bit for bit.  X's row r is key r; the
# library returns key-space CSC with 0-based pointers, shifted here to SparseMatrixCSC's 1-based ones.  A result key above n
# (entries stored outside size(A)) throws a BoundsError.
function _spmspm(A::DynamicSparseMatrix, trans::Bool, X::SparseMatrixCSC, n)
    A.fillmode && error("Matrix is in fill mode")
    flush!(A)
    k = size(X, 2)
    xp = Vector{Int64}(X.colptr) .- 1; xk = Vector{Int64}(rowvals(X)); xv = Vector{Float64}(nonzeros(X))
    cnt = Ref{Int64}(0)
    f(yp, yk, yv, cap) = ccall((:dsa_matrix_spmspm, libdsa), Cint,
                               (Ptr{Cvoid}, Cint, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Int64, Int64, Ptr{Int64}, Ptr{Int64},
                                Ptr{Float64}, Int64, Ref{Int64}),
                               A.h, trans ? 1 : 0, xp, xk, xv, k, length(xk), yp, yk, yv, cap, cnt)
    _check(f(C_NULL, C_NULL, C_NULL, 0))                                                                  # size query: nnz
    yp = Vector{Int64}(undef, k + 1); yk = Vector{Int64}(undef, cnt[]); yv = Vector{Float64}(undef, cnt[])
    _check(f(yp, yk, yv, length(yk)))
    isempty(yk) || maximum(yk) <= n || throw(BoundsError(A, maximum(yk)))
    return SparseMatrixCSC(n, k, yp .+ 1, yk, yv)
end
spmspv(A::DynamicSparseMatrix, X::SparseMatrixCSC) = _spmspm(A, false, X, size(A, 1))                     # size (size(A, 1), k)
spmspv(t::Transposed, X::SparseMatrixCSC) = _spmspm(t.array, true, X, size(t.array, 2))                   # size (size(A, 2), k)

# k dense right-hand sides in one call (one pass over the matrix per 32 columns); column c of the result equals the product
# with X[:, c] bit for bit.  The library takes row-major buffers: permutedims turns the column-major X into one (ldx = k).
function _mul_dense(A::DynamicSparseMatrix, trans::Bool, X::Matrix{Float64})
    A.fillmode && error("Matrix is in fill mode")
    flush!(A)
    nx, k = size(X)
    ny = size(A, trans ? 2 : 1)
    Xr = permutedims(X)
    Yr = Matrix{Float64}(undef, k, ny)
    _check(ccall((:dsa_matrix_spmm_dense, libdsa), Cint,
                 (Ptr{Cvoid}, Cint, Ptr{Float64}, Int64, Int64, Int64, Ptr{Float64}, Int64, Int64),
                 A.h, trans ? 1 : 0, Xr, nx, k, k, Yr, ny, k))
    return permutedims(Yr)
end
Base.:(*)(A::DynamicSparseMatrix, X::Matrix{Float64}) = _mul_dense(A, false, X)                           # size (size(A, 1), k)
Base.:(*)(t::Transposed, X::Matrix{Float64}) = _mul_dense(t.array, true, X)                               # size (size(A, 2), k)

# ------------------------------------------------------------------------------------------ compressed snapshot
# The column-major orientation compacted on the device with 1-based pointers (dim = n, idim = m): colptr, rowval and nzval come
# back exactly as SparseMatrixCSC stores them (sorted row indices, stored zeros kept).  Entries outside size(A)
# (dynamicsparse(I, J, V, m, n) with m < maximum(I)) throw a BoundsError.
function SparseArrays.SparseMatrixCSC(A::DynamicSparseMatrix)
    A.fillmode && error("Matrix is in fill mode")
    flush!(A)
    m, n = size(A)
    cnt = Ref{Int64}(0)
    f(colptr, rowval, nzval, cap) = ccall((:dsa_matrix_compress_dense, libdsa), Cint,
                                          (Ptr{Cvoid}, Cint, Int64, Int64, Cint, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Int64, Ref{Int64}),
                                          A.h, 0, n, m, 1, colptr, rowval, nzval, cap, cnt)
    _check(f(C_NULL, C_NULL, C_NULL, 0))                                                                  # size query: nnz
    colptr = Vector{Int64}(undef, n + 1); rowval = Vector{Int64}(undef, cnt[]); nzval = Vector{Float64}(undef, cnt[])
    _check(f(colptr, rowval, nzval, length(nzval)))
    return SparseMatrixCSC(m, n, colptr, rowval, nzval)
end
SparseArrays.sparse(A::DynamicSparseMatrix) = SparseMatrixCSC(A)


# ------------------------------------------------------------------------------------------ multi-GPU (include/dsa.h "multi-GPU")
# One Julia process per GPU (e.g. under MPI.jl or Distributed).  A ShardedDynamicSparseMatrix is the same DynamicSparseMatrix
# (matrix.jl:1-8) sharded by key range over the group; every method below is a collective: all ranks call it in the same order.
# The 128-byte group id is drawn on rank 0 with dist_unique_id() and handed to the other ranks by the host program
# (MPI.Bcast!, a file, a socket ...).
export DistContext, ShardedDynamicSparseMatrix, dist_unique_id

function dist_unique_id()
    id = Vector{UInt8}(undef, 128)
    _check(ccall((:dsa_dist_unique_id, libdsa), Cint, (Ptr{Cvoid},), id))
    return id
end

mutable struct DistContext
    h::Ptr{Cvoid}
    rank::Int
    world::Int
    function DistContext(id::Vector{UInt8}, rank::Integer, world::Integer; device::Integer = rank)
        _check(ccall((:dsa_set_device, libdsa), Cint, (Cint,), device))
        h = Ref{Ptr{Cvoid}}()
        _check(ccall((:dsa_dist_init, libdsa), Cint, (Ptr{Cvoid}, Cint, Cint, Ref{Ptr{Cvoid}}), id, rank, world, h))
        c = new(h[], rank, world)
        finalizer(x -> ccall((:dsa_dist_destroy, libdsa), Cint, (Ptr{Cvoid},), x.h), c)
        return c
    end
end

mutable struct ShardedDynamicSparseMatrix
    h::Ptr{Cvoid}
    ctx::DistContext          # keeps the group alive as long as the matrix
    m::Int64
    n::Int64
    function ShardedDynamicSparseMatrix(ctx::DistContext, m::Integer, n::Integer; max_share::Integer,
                                        row_split::Union{Nothing,Vector{Int64}} = nothing, col_split::Union{Nothing,Vector{Int64}} = nothing)
        h = Ref{Ptr{Cvoid}}()
        _check(ccall((:dsa_dmatrix_create, libdsa), Cint, (Ptr{Cvoid}, Int64, Int64, Ptr{Int64}, Ptr{Int64}, Int64, Ref{Ptr{Cvoid}}),
                     ctx.h, m, n, row_split === nothing ? C_NULL : row_split, col_split === nothing ? C_NULL : col_split, max_share, h))
        A = new(h[], ctx, m, n)
        finalizer(x -> ccall((:dsa_dmatrix_destroy, libdsa), Cint, (Ptr{Cvoid},), x.h), A)
        return A
    end
end
Base.size(A::ShardedDynamicSparseMatrix) = (A.m, A.n)

# dynamicsparse(I, J, V, m, n) over the group (matrix.jl:15-19): every rank passes ITS share of the global COO
function dynamicsparse(ctx::DistContext, I::Vector{Int64}, J::Vector{Int64}, V::Vector{Float64}, m::Integer, n::Integer; max_share::Integer)
    length(I) == length(J) == length(V) || throw(ArgumentError("rows, columns, and nonzeros do not have same length."))
    A = ShardedDynamicSparseMatrix(ctx, m, n; max_share = max_share)
    _check(ccall((:dsa_dmatrix_build_coo, libdsa), Cint, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Int64, Cint),
                 A.h, I, J, V, length(V), 0))
    return A
end

# batched setindex! (matrix.jl:43-62): this rank's share of ONE global batch (op order: rank-major, then arrival)
function set_batch!(A::ShardedDynamicSparseMatrix, rows::Vector{Int64}, cols::Vector{Int64}, vals::Vector{Float64})
    length(rows) == length(cols) == length(vals) || throw(ArgumentError("rows, columns, and nonzeros do not have same length."))
    _check(ccall((:dsa_dmatrix_set_batch, libdsa), Cint, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Int64),
                 A.h, rows, cols, vals, length(vals)))
    return A
end
Base.setindex!(A::ShardedDynamicSparseMatrix, val, row::Integer, col::Integer) =
    set_batch!(A, Int64[row], Int64[col], Float64[val])      # a collective of one op: the other ranks pass empty shares

function Base.getindex(A::ShardedDynamicSparseMatrix, row::Integer, col::Integer)                         # matrix.jl:64-68
    out = Ref{Float64}(0.0)
    _check(ccall((:dsa_dmatrix_get_batch, libdsa), Cint, (Ptr{Cvoid}, Cint, Ref{Int64}, Ref{Int64}, Int64, Ref{Float64}),
                 A.h, 0, Ref(Int64(row)), Ref(Int64(col)), 1, out))
    return out[]
end

function _dmul(A::ShardedDynamicSparseMatrix, trans::Bool, x::Vector{Float64})                            # operations.jl:14-36
    y = Vector{Float64}(undef, trans ? A.n : A.m)
    _check(ccall((:dsa_dmatrix_spmv_dense, libdsa), Cint, (Ptr{Cvoid}, Cint, Ptr{Float64}, Int64, Ptr{Float64}, Int64),
                 A.h, trans ? 1 : 0, x, length(x), y, length(y)))
    return y
end
struct TransposedSharded; array::ShardedDynamicSparseMatrix; end
Base.transpose(A::ShardedDynamicSparseMatrix) = TransposedSharded(A)
Base.:(*)(A::ShardedDynamicSparseMatrix, x::Vector{Float64}) = _dmul(A, false, x)
Base.:(*)(t::TransposedSharded, x::Vector{Float64}) = _dmul(t.array, true, x)

function deletecolumn!(A::ShardedDynamicSparseMatrix, cols::Vector{Int64})                                # matrix.jl:95-102, same list on every rank
    _check(ccall((:dsa_dmatrix_delete_columns, libdsa), Cint, (Ptr{Cvoid}, Ptr{Int64}, Int64), A.h, cols, length(cols)))
    return true
end
deletecolumn!(A::ShardedDynamicSparseMatrix, col::Integer) = deletecolumn!(A, Int64[col])
function deleterow!(A::ShardedDynamicSparseMatrix, rows::Vector{Int64})                                   # matrix.jl:104-111
    _check(ccall((:dsa_dmatrix_delete_rows, libdsa), Cint, (Ptr{Cvoid}, Ptr{Int64}, Int64), A.h, rows, length(rows)))
    return true
end
deleterow!(A::ShardedDynamicSparseMatrix, row::Integer) = deleterow!(A, Int64[row])

function SparseArrays.nnz(A::ShardedDynamicSparseMatrix)                                                  # matrix.jl:91, summed over the shards
    out = Vector{Int64}(undef, 8)
    _check(ccall((:dsa_dmatrix_info, libdsa), Cint, (Ptr{Cvoid}, Ptr{Int64}), A.h, out))
    return out[3]
end

# How a batched setindex! is applied (include/dsa.h "tuning"): 0 = random-access pipeline only, 1 = dense batches are
# tile-streamed (default), 2 = tile-streamed whenever possible.  Same layout either way; returns the previous mode.
set_tile_mode!(mode::Integer) = ccall((:dsa_set_tile_mode, libdsa), Cint, (Cint,), mode)

end # module
