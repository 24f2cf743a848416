# CoverageCUDA.jl -- Julia `ccall` binding of libcoverage_cuda (include/coverage_cuda.h).
#
# Drop-in for the reference's objective factory: `CoverageCUDA.createObjective(cells, N, r_max)`
# returns a closure `AreaMaxObjective(x::Vector{Float64})::Float64` with the value semantics of
# src/TDM_STATIC_opt.jl:82-100, so `SetObjective(p, obj)` (src/TDM_STATIC_opt.jl:125) and
# src/FullSimulation.jl:84-97 keep working with only the factory swapped.  A batched entry
# (`objective_batch`) serves a poll-set-at-a-time MADS driver.
#
# NOT EXECUTED in this repository's CI: Julia is not installed in the build container or on the GPU
# box.  The same C entry points are exercised from Python ctypes in tests/test_gpu_parity.py.
module CoverageCUDA

const LIB = get(ENV, "LIBCOVERAGE_CUDA", joinpath(@__DIR__, "..", "libcoverage_cuda.so"))

struct CovError <: Exception
    code::Cint
    msg::String
end

mutable struct Handle
    ptr::Ptr{Cvoid}
    N::Int
    ncells::Int # nx * ny of the lattice last set through this binding (0: none yet)
    function Handle(device::Integer = 0)
        out = Ref{Ptr{Cvoid}}(C_NULL)
        rc = ccall((:cov_create, LIB), Cint, (Cint, Ref{Ptr{Cvoid}}), device, out)
        rc == 0 || throw(CovError(rc, unsafe_string(ccall((:cov_last_error, LIB), Cstring, (Ptr{Cvoid},), C_NULL))))
        h = new(out[], 0, 0)
        finalizer(h -> (h.ptr == C_NULL || ccall((:cov_destroy, LIB), Cvoid, (Ptr{Cvoid},), h.ptr); h.ptr = C_NULL), h)
        return h
    end
    Handle(ptr::Ptr{Cvoid}, N::Int) = new(ptr, N, 0) # borrowed (a MultiHandle's shard): never destroyed here
end

check(h::Handle, rc::Cint) =
    rc == 0 || throw(CovError(rc, unsafe_string(ccall((:cov_last_error, LIB), Cstring, (Ptr{Cvoid},), h.ptr))))

"Upload the reference's own point list (`Vector{Vector{Float64}}` of [x, y, area, weight, covered])."
function set_points!(h::Handle, points::Vector{Vector{Float64}}; nx = 100, ny = 100, dx = 5.0, dy = 5.0)
    flat = Vector{Float64}(undef, 5 * length(points))
    @inbounds for (p, pt) in enumerate(points), k in 1:5
        flat[5 * (p - 1) + k] = pt[k]
    end
    GC.@preserve flat check(h, ccall((:cov_set_points, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Int64, Float64, Float64),
        h.ptr, flat, length(points), nx, ny, dx, dy))
    h.ncells = nx * ny
end

"createPOI(dx, dy, nx, ny) built on the device (src/AreaCoverageCalculation.jl:11-21)."
function set_grid_full!(h::Handle, nx, ny, dx, dy)
    check(h, ccall((:cov_set_grid_full, LIB), Cint, (Ptr{Cvoid}, Int64, Int64, Float64, Float64), h.ptr, nx, ny, dx, dy))
    h.ncells = nx * ny
end

"rmvCoveredPOI on the device-resident store (src/CellFunctions.jl:81-108); returns entries removed."
function remove_covered!(h::Handle, xyR::Vector{Float64})
    removed = Ref{Int64}(0)
    GC.@preserve xyR check(h, ccall((:cov_remove_covered, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Int64, Ref{Int64}),
        h.ptr, xyR, length(xyR) ÷ 3, removed))
    return removed[]
end

"update_POI on the device-resident store (src/CellFunctions.jl:59-77): append list entries, duplicates add up."
function add_points!(h::Handle, points::Vector{Vector{Float64}})
    flat = Vector{Float64}(undef, 5 * length(points))
    @inbounds for (p, pt) in enumerate(points), k in 1:5
        flat[5 * (p - 1) + k] = pt[k]
    end
    GC.@preserve flat check(h, ccall((:cov_add_points, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Int64),
        h.ptr, flat, length(points)))
end

"""
    fire_init!(h, state; dx = 5.0, dy = 5.0, push_initial = true)
    fire_step!(h, wind_speed, wind_direction, prob_spread; seed = 0, step = 0, append = true)

The forest-fire automaton of src/DynamicArea.jl:17-86 on the device: `state` is the `nx x ny` `UInt8` grid
(0 EMPTY, 1 TREE, 2 FIRE); every step pushes the newly ignited cells straight into the cell store that the
objective reads (no xlsx hand-off). `fire_step!` returns the number of entries pushed.
"""
function fire_init!(h::Handle, state::Matrix{UInt8}; dx = 5.0, dy = 5.0, push_initial = true)
    nx, ny = size(state)
    GC.@preserve state check(h, ccall((:cov_fire_init, LIB), Cint,
        (Ptr{Cvoid}, Int64, Int64, Float64, Float64, Ptr{UInt8}, Int32), h.ptr, nx, ny, dx, dy, state, push_initial ? 1 : 0))
    h.ncells = nx * ny
end
function fire_step!(h::Handle, wind_speed, wind_direction, prob_spread; seed = 0, step = 0, append = true)
    pushed = Ref{Int64}(0)
    check(h, ccall((:cov_fire_step, LIB), Cint,
        (Ptr{Cvoid}, Float64, Float64, Float64, UInt64, Int64, Int32, Ref{Int64}),
        h.ptr, wind_speed, wind_direction, prob_spread, seed, step, append ? 1 : 0, pushed))
    return pushed[]
end

"Exact area of the union of the discs of every column of `X` (3N x B, [x; y; R]); no grid involved."
function union_area(h::Handle, X::Matrix{Float64})
    N = size(X, 1) ÷ 3; B = size(X, 2)
    area = Vector{Float64}(undef, B)
    GC.@preserve X area check(h, ccall((:cov_union_area_batch, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Ptr{Float64}), h.ptr, X, B, N, area))
    return area
end

"Captured variables of createObjective / create_cons3 / cons8 / cons7."
function set_params!(h::Handle, N::Integer, r_max::Vector{Float64}; penalty = 1e5,
                     prev::Union{Nothing,Vector{Float64}} = nothing, d_lim::Vector{Float64} = fill(10.0, N),
                     FOV = 100 / 180 * π, sep_min = 0.0, use_cons7 = false)
    prevp = prev === nothing ? Ptr{Float64}(C_NULL) : pointer(prev)
    GC.@preserve r_max prev d_lim check(h, ccall((:cov_set_params, LIB), Cint,
        (Ptr{Cvoid}, Int64, Ptr{Float64}, Float64, Ptr{Float64}, Ptr{Float64}, Float64, Float64, Int32),
        h.ptr, N, r_max, penalty, prevp, d_lim, tan(FOV / 2), sep_min, use_cons7 ? 1 : 0))
    h.N = N
end

"One candidate: AreaMaxObjective(x) (src/TDM_STATIC_opt.jl:83-98)."
function eval_one(h::Handle, x::Vector{Float64})
    obj = Ref{Float64}(0.0)
    GC.@preserve x check(h, ccall((:cov_eval_one, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ref{Float64}), h.ptr, x, obj))
    return obj[]
end

"A whole poll set: X is 3N x B (one candidate [x;y;R] per COLUMN, i.e. candidate-major in memory).
Allocates plain (pageable) outputs; for large or repeated batches use `BatchBuffers` + `objective_batch!` (pinned)."
function objective_batch(h::Handle, X::Matrix{Float64})
    B = size(X, 2)
    obj = Vector{Float64}(undef, B); count = Vector{Int64}(undef, B); feasible = Vector{UInt8}(undef, B)
    GC.@preserve X obj count feasible check(h, ccall((:cov_eval_batch, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Int64}, Ptr{UInt8}),
        h.ptr, X, B, obj, count, feasible))
    return obj, count, feasible
end

"""
    pinned_matrix(h, rows, cols) / pinned_vector(h, T, n)

Page-locked host arrays owned by the library (`cov_host_alloc`), wrapped without a copy. `cov_eval_batch` DMAs pinned
buffers in place; a plain `Matrix` goes through the library's pinned staging instead (measured on B200, 1 M candidates
x 5 UAVs: 2.45 ms pinned vs 3.3 ms pageable per call). The arrays stay valid until `free_pinned!` or until the handle
is destroyed -- keep the handle alive as long as they are in use.
"""
function pinned_vector(h::Handle, ::Type{T}, n::Integer) where {T}
    out = Ref{Ptr{Cvoid}}(C_NULL)
    check(h, ccall((:cov_host_alloc, LIB), Cint, (Ptr{Cvoid}, Int64, Ref{Ptr{Cvoid}}), h.ptr, max(n * sizeof(T), 1), out))
    return unsafe_wrap(Array, Ptr{T}(out[]), (Int(n),); own = false)
end
function pinned_matrix(h::Handle, rows::Integer, cols::Integer)
    out = Ref{Ptr{Cvoid}}(C_NULL)
    check(h, ccall((:cov_host_alloc, LIB), Cint, (Ptr{Cvoid}, Int64, Ref{Ptr{Cvoid}}), h.ptr, max(rows * cols * 8, 1), out))
    return unsafe_wrap(Array, Ptr{Float64}(out[]), (Int(rows), Int(cols)); own = false)
end
free_pinned!(h::Handle, a::Array) = check(h, ccall((:cov_host_free, LIB), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), h.ptr, pointer(a)))

"Reusable pinned buffers for poll sets of up to `B` candidates: fill `X[:, 1:b]`, call `objective_batch!(h, bufs, b)`."
struct BatchBuffers
    X::Matrix{Float64}        # 3N x B, one candidate per column
    obj::Vector{Float64}
    count::Vector{Int64}
    feasible::Vector{UInt8}
end
BatchBuffers(h::Handle, B::Integer) = BatchBuffers(pinned_matrix(h, 3 * h.N, B), pinned_vector(h, Float64, B),
                                                   pinned_vector(h, Int64, B), pinned_vector(h, UInt8, B))
function objective_batch!(h::Handle, b::BatchBuffers, n::Integer = size(b.X, 2))
    check(h, ccall((:cov_eval_batch, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Int64}, Ptr{UInt8}),
        h.ptr, b.X, n, b.obj, b.count, b.feasible))
    return view(b.obj, 1:n), view(b.count, 1:n), view(b.feasible, 1:n)
end

"""
    objective_batch_best!(h, bufs, n; barrier = true) -> (obj, count, feasible, best_obj, best_column)

`objective_batch!` plus the poll winner reduced on the device (`cov_eval_batch_best`): the 16 bytes a process
contributes when the candidates of one poll are sharded over several GPUs (one Julia process per GPU, e.g. under
MPI.jl or Distributed: `MPI.Allgather((best_obj, first_column + best_column))`, smallest objective wins, ties to the
smallest column). `best_column` is 1-based, 0 when no candidate is feasible.
"""
function objective_batch_best!(h::Handle, b::BatchBuffers, n::Integer = size(b.X, 2); barrier = true)
    bo = Ref{Float64}(Inf); bi = Ref{Int64}(-1)
    check(h, ccall((:cov_eval_batch_best, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Int64}, Ptr{UInt8}, Int32, Ref{Float64}, Ref{Int64}),
        h.ptr, b.X, n, b.obj, b.count, b.feasible, barrier ? 1 : 0, bo, bi))
    return view(b.obj, 1:n), view(b.count, 1:n), view(b.feasible, 1:n), bo[], bi[] + 1
end

_pack_code(::Type{Float32}) = Int32(1)
_pack_code(::Type{Int32}) = Int32(2)
_pack_code(::Type{Int16}) = Int32(3)

"Pinned `rows x cols` matrix of packed candidate values (`Int16`, `Int32` or `Float32`) for `objective_batch_packed`."
function pinned_packed(h::Handle, ::Type{T}, rows::Integer, cols::Integer) where {T<:Union{Int16,Int32,Float32}}
    out = Ref{Ptr{Cvoid}}(C_NULL)
    check(h, ccall((:cov_host_alloc, LIB), Cint, (Ptr{Cvoid}, Int64, Ref{Ptr{Cvoid}}), h.ptr, max(rows * cols * sizeof(T), 1), out))
    return unsafe_wrap(Array, Ptr{T}(out[]), (Int(rows), Int(cols)); own = false)
end

"""
    objective_batch_packed(h, Q, granularity = 1.0; winner = false, barrier = true)

Poll / search sets whose trial points sit on the MADS mesh, sent PACKED (`cov_eval_batch_packed`): `Q` is `3N x B` of
`Int16` or `Int32` mesh indices (candidate = `q * granularity`; granularity 1.0 on every variable in
`TDM_STATIC_opt.optimize`, src/TDM_STATIC_opt.jl:131-137) or of `Float32` values. A quarter or half of the bytes cross
PCIe, the kernels see the same `Float64` candidates, the results are bit for bit those of `objective_batch` on
`Float64.(Q) .* granularity` (measured on B200, 1 M candidates x 5 UAVs from pinned buffers: 2.40 ms -> 1.11 ms per
call with `Int16`). `Q` from `pinned_packed(h, T, 3N, B)` is DMA'd in place. With `winner = true` also returns
`(best_obj, best_column)` like `objective_batch_best!`.
"""
function objective_batch_packed(h::Handle, Q::Matrix{T}, granularity::Real = 1.0; winner = false, barrier = true) where {T<:Union{Int16,Int32,Float32}}
    B = size(Q, 2)
    obj = Vector{Float64}(undef, B); count = Vector{Int64}(undef, B); feasible = Vector{UInt8}(undef, B)
    if !winner
        GC.@preserve Q obj count feasible check(h, ccall((:cov_eval_batch_packed, LIB), Cint,
            (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Float64, Int64, Ptr{Float64}, Ptr{Int64}, Ptr{UInt8}, Int32, Ptr{Float64}, Ptr{Int64}),
            h.ptr, Q, _pack_code(T), Float64(granularity), B, obj, count, feasible, 0, C_NULL, C_NULL))
        return obj, count, feasible
    end
    bo = Ref{Float64}(Inf); bi = Ref{Int64}(-1)
    GC.@preserve Q obj count feasible check(h, ccall((:cov_eval_batch_packed, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Float64, Int64, Ptr{Float64}, Ptr{Int64}, Ptr{UInt8}, Int32, Ref{Float64}, Ref{Int64}),
        h.ptr, Q, _pack_code(T), Float64(granularity), B, obj, count, feasible, barrier ? 1 : 0, bo, bi))
    return obj, count, feasible, bo[], bi[] + 1
end

"The store's weight classes in the device's numbering (the `class_count` columns of `cov_eval_batch_ex`)."
function class_weights(h::Handle)
    w = zeros(Float64, 4)
    check(h, ccall((:cov_get_class_weights, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Int64), h.ptr, w, 4))
    return w
end

"""
    create_cons1_progressive(N, r_max) / create_cons2_progressive / create_cons3_progressive

The progressive constraints of src/TDM_Constraints.jl:182-221 (`x -> Real`, for `AddProgressiveConstraint`):
`sum_i max(R_i - r_max_i, 0.0)`, and the same term for UAV 2 / UAV 3 alone. `COV_OPT_PROGRESSIVE_INDEX` (10) selects
which one the `progressive` output of `cov_eval_batch_ex` carries; `.batch(X)`-style use: `progressive_batch`.
"""
function progressive_batch(h::Handle, X::Matrix{Float64}, which::Integer)
    B = size(X, 2)
    obj = Vector{Float64}(undef, B); prog = Vector{Float64}(undef, B)
    check(h, ccall((:cov_set_option, LIB), Cint, (Ptr{Cvoid}, Cint, Int64), h.ptr, 10, which))
    GC.@preserve X obj prog check(h, ccall((:cov_eval_batch_ex, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Int64}, Ptr{UInt8}, Ptr{Int64}, Ptr{Float64}),
        h.ptr, X, B, obj, C_NULL, C_NULL, C_NULL, prog))
    return prog
end
function _create_progressive(which::Integer, N::Integer, r_max; handle::Handle = Handle())
    set_grid_full!(handle, 1, 1, 1.0, 1.0)          # constraints do not look at the cell store
    set_params!(handle, N, collect(Float64, r_max); penalty = 0.0)
    return x -> progressive_batch(handle, reshape(collect(Float64, x), :, 1), which)[1]
end
create_cons1_progressive(N, r_max; kw...) = _create_progressive(0, N, r_max; kw...)
create_cons2_progressive(N, r_max; kw...) = _create_progressive(2, N, r_max; kw...)
create_cons3_progressive(N, r_max; kw...) = _create_progressive(3, N, r_max; kw...)

"Poll winner with the extreme barrier: (best objective, 1-based column) or (Inf, 0)."
function argmin_batch(h::Handle, X::Matrix{Float64}; barrier = true)
    bo = Ref{Float64}(Inf); bi = Ref{Int64}(-1)
    GC.@preserve X check(h, ccall((:cov_argmin, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int32, Ref{Float64}, Ref{Int64}), h.ptr, X, size(X, 2), barrier ? 1 : 0, bo, bi))
    return bo[], bi[] + 1
end

"""
    mads_solve(h, x0; N_iter = 100, granularity = 1.0, seed = 0)

The whole MADS solve inside the library (same settings as `TDM_STATIC_opt.optimize`, src/TDM_STATIC_opt.jl:118-222;
the constraints given to `set_params!` act as extreme barrier). Returns `(result, objective, runtime_seconds)`.
"""
function mads_solve(h::Handle, x0::Vector{Float64}; N_iter = 100, granularity = 1.0, seed = 0)
    out = similar(x0); obj = Ref{Float64}(0.0); stats = zeros(Int64, 4)
    t = @elapsed GC.@preserve x0 out stats check(h, ccall((:cov_mads_solve, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Float64, UInt64, Ptr{Float64}, Ref{Float64}, Ptr{Int64}),
        h.ptr, x0, N_iter, granularity, seed, out, obj, stats))
    return out, obj[], t
end

"""
    mads_solve_batch(h, X0; N_iter = 100, granularity = 1.0, seed = 0)

S independent MADS solves in one launch on the device (`cov_mads_solve_batch`), one start per column of `X0`
(3N x S); solve k (1-based) draws its directions from the Philox key `seed + k - 1`. Returns
`(X_out, objectives, stats, runtime_seconds)`: `X_out` 3N x S, `stats` 4 x S with rows iterations, evaluations,
successes, converged.
"""
function mads_solve_batch(h::Handle, X0::Matrix{Float64}; N_iter = 100, granularity = 1.0, seed = 0)
    S = size(X0, 2)
    out = similar(X0); obj = zeros(Float64, S); stats = zeros(Int64, 4, S)
    t = @elapsed GC.@preserve X0 out obj stats check(h, ccall((:cov_mads_solve_batch, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Float64, UInt64, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}),
        h.ptr, X0, S, N_iter, granularity, seed, out, obj, stats))
    return out, obj, stats, t
end

"""
    with_list_order(f, h, on)

`f()` with `COV_OPT_LIST_ORDER_HORIZON` (11) at 1 on `h` (a `MultiHandle`: on every shard) when `on`, so that the
horizon calls accept a store whose area depends on the list order (non-dyadic weights); the previous value is put back
afterwards, also when `f` throws. `on = false` leaves the option as it is.
"""
function with_list_order(f, h::Handle, on::Bool)
    on || return f()
    prev = Ref{Int64}(0)
    check(h, ccall((:cov_get_option, LIB), Cint, (Ptr{Cvoid}, Cint, Ref{Int64}), h.ptr, 11, prev))
    check(h, ccall((:cov_set_option, LIB), Cint, (Ptr{Cvoid}, Cint, Int64), h.ptr, 11, 1))
    try
        return f()
    finally
        ccall((:cov_set_option, LIB), Cint, (Ptr{Cvoid}, Cint, Int64), h.ptr, 11, prev[])
    end
end
with_list_order(f, m, on::Bool) = foldr((s, g) -> () -> with_list_order(g, s, on), m.shards; init = f)()

"""
    run_horizon(h, x_start; T, S = 1, spread = 3.0, N_iter = 100, granularity = 1.0, seed = 0,
                boxes = zeros(Float64, 4, 0), h_focus = 15.0, h_max = 30.0)

T timesteps of FullSimulation's MADS loop on the device in one call (`cov_run_horizon`): per timestep
rmvCoveredPOI of the current swarm, the r_max rule near the boxes (columns [x_LB; x_UB; y_LB; y_UB]), cons3 from the
current swarm, S solves (from the swarm and S - 1 perturbations of it) and the best as the next swarm. Needs
`set_params!` with a previous swarm. Returns `(X, objectives, stats, step_ms)`: `X` 3N x T, `stats` 4 x T with rows
winner, evaluations, feasible solves, entries removed; `step_ms` the device time of every timestep.
"""
function run_horizon(h::Handle, x_start::Vector{Float64}; T, S = 1, spread = 3.0, N_iter = 100, granularity = 1.0,
                     seed = 0, boxes::Matrix{Float64} = zeros(Float64, 4, 0), h_focus = 15.0, h_max = 30.0,
                     list_order = false)
    n = length(x_start); K = size(boxes, 2)
    X = zeros(Float64, n, T); obj = zeros(Float64, T); stats = zeros(Int64, 4, T); ms = zeros(Float64, T)
    with_list_order(h, list_order) do
        GC.@preserve x_start boxes X obj stats ms check(h, ccall((:cov_run_horizon, LIB), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Float64, Int64, Float64, UInt64, Ptr{Float64}, Int64, Float64,
             Float64, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Float64}),
            h.ptr, x_start, T, S, spread, N_iter, granularity, seed, K == 0 ? C_NULL : pointer(boxes), K, h_focus, h_max,
            X, obj, stats, ms))
    end
    return X, obj, stats, ms
end

"""
    run_horizon_points(h, x_start, appends; S = 1, spread = 3.0, N_iter = 100, granularity = 1.0, seed = 0,
                       boxes = zeros(Float64, 4, 0), h_focus = 15.0, h_max = 30.0, nx = 100, ny = 100)

`run_horizon` with the reference's fire list (`cov_run_horizon_points`): `appends` holds T matrices of reference
points (5 x n_t, columns [x; y; area; weight; covered]), timestep t appending `appends[t]` before its rmvCoveredPOI
(update_POI's push!). Returns `(X, objectives, stats, step_ms, last_removed)`: `stats` 5 x T with the entries appended
as row 5, `last_removed` (nx*ny of the store's lattice, index (i-1) + nx*(j-1)) the last timestep that removed entries
from each cell (0: none).
"""
function run_horizon_points(h::Handle, x_start::Vector{Float64}, appends::Vector{Matrix{Float64}}; S = 1,
                            spread = 3.0, N_iter = 100, granularity = 1.0, seed = 0,
                            boxes::Matrix{Float64} = zeros(Float64, 4, 0), h_focus = 15.0, h_max = 30.0, nx = 100,
                            ny = 100, list_order = false)
    T = length(appends); n = length(x_start); K = size(boxes, 2)
    offsets = zeros(Int64, T + 1)
    for t in 1:T
        offsets[t + 1] = offsets[t] + size(appends[t], 2)
    end
    pts = T == 0 ? zeros(Float64, 5, 0) : reduce(hcat, appends)  # column p = the 5-tuple of entry p
    last = zeros(Cint, nx * ny)
    X = zeros(Float64, n, T); obj = zeros(Float64, T); stats = zeros(Int64, 5, T); ms = zeros(Float64, T)
    with_list_order(h, list_order) do
        GC.@preserve x_start boxes pts offsets X obj stats ms last check(h, ccall((:cov_run_horizon_points, LIB), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Float64, Int64, Float64, UInt64, Ptr{Float64}, Int64, Float64,
             Float64, Ptr{Float64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Float64}, Ptr{Cint}),
            h.ptr, x_start, T, S, spread, N_iter, granularity, seed, K == 0 ? C_NULL : pointer(boxes), K, h_focus, h_max,
            offsets[end] == 0 ? C_NULL : pointer(pts), offsets, X, obj, stats, ms, last))
    end
    return X, obj, stats, ms, last
end

"""
    run_horizon_fire(h, x_start, fire_steps; wind_speed = 4.0, wind_direction = deg2rad(270.0), prob_spread = 0.5,
                     fire_seed = 0, first_step = 1, S = 1, spread = 3.0, N_iter = 100, granularity = 1.0, seed = 0,
                     boxes = zeros(Float64, 4, 0), h_focus = 15.0, h_max = 30.0)

`run_horizon` with the device forest-fire automaton (`cov_run_horizon_fire`, after `fire_init!`): timestep t first
runs `fire_steps[t]` automaton steps with append, numbered from `first_step`. Returns `(X, objectives, stats,
step_ms)` with `stats` 5 x T, row 5 the entries each timestep's steps pushed.
"""
function run_horizon_fire(h::Handle, x_start::Vector{Float64}, fire_steps::Vector{Int64}; wind_speed = 4.0,
                          wind_direction = deg2rad(270.0), prob_spread = 0.5, fire_seed = 0, first_step = 1, S = 1,
                          spread = 3.0, N_iter = 100, granularity = 1.0, seed = 0,
                          boxes::Matrix{Float64} = zeros(Float64, 4, 0), h_focus = 15.0, h_max = 30.0)
    T = length(fire_steps); n = length(x_start); K = size(boxes, 2)
    X = zeros(Float64, n, T); obj = zeros(Float64, T); stats = zeros(Int64, 5, T); ms = zeros(Float64, T)
    GC.@preserve x_start boxes fire_steps X obj stats ms check(h, ccall((:cov_run_horizon_fire, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Float64, Int64, Float64, UInt64, Ptr{Float64}, Int64, Float64,
         Float64, Ptr{Int64}, Float64, Float64, Float64, UInt64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Int64},
         Ptr{Float64}),
        h.ptr, x_start, T, S, spread, N_iter, granularity, seed, K == 0 ? C_NULL : pointer(boxes), K, h_focus, h_max,
        fire_steps, wind_speed, wind_direction, prob_spread, fire_seed, first_step, X, obj, stats, ms))
    return X, obj, stats, ms
end

"""
    run_horizon_ensemble(h, x_starts; T, S = 1, spread = 3.0, N_iter = 100, granularity = 1.0, seed = 0,
                         boxes = zeros(Float64, 4, 0), h_focus = 15.0, h_max = 30.0, want_cells = false)

E independent `run_horizon` scenarios in one call (`cov_run_horizon_ensemble`), each on a private copy of the
handle's current store and parameters: column e of `x_starts` (3N x E) starts scenario e, which equals `run_horizon`
with `seed + (e - 1) * T * S`. The handle is left unchanged. Returns `(X, objectives, stats, step_ms, cells)`: `X`
3N x T x E, `objectives` T x E, `stats` 4 x T x E (`run_horizon`'s rows), `step_ms` the device time of every timestep
of the whole ensemble, `cells` (nx*ny x E, with `want_cells`; else `nothing`) the multiplicities each scenario leaves. `want_cells` needs the
lattice set through this binding (`set_points!`, `set_grid_full!` or `fire_init!`), which sizes `cells`.
"""
function run_horizon_ensemble(h::Handle, x_starts::Matrix{Float64}; T, S = 1, spread = 3.0, N_iter = 100,
                              granularity = 1.0, seed = 0, boxes::Matrix{Float64} = zeros(Float64, 4, 0),
                              h_focus = 15.0, h_max = 30.0, want_cells = false, list_order = false)
    n, E = size(x_starts); K = size(boxes, 2)
    X = zeros(Float64, n, T, E); obj = zeros(Float64, T, E); stats = zeros(Int64, 4, T, E); ms = zeros(Float64, T)
    cells = want_cells ? zeros(UInt8, lattice_cells(h), E) : nothing
    with_list_order(h, list_order) do
        GC.@preserve x_starts boxes X obj stats ms cells check(h, ccall((:cov_run_horizon_ensemble, LIB), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Int64, Float64, Int64, Float64, UInt64, Ptr{Float64}, Int64, Float64,
             Float64, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Float64}, Ptr{UInt8}),
            h.ptr, x_starts, E, T, S, spread, N_iter, granularity, seed, K == 0 ? C_NULL : pointer(boxes), K, h_focus,
            h_max, X, obj, stats, ms, want_cells ? pointer(cells) : C_NULL))
    end
    return X, obj, stats, ms, cells
end

"""
    run_horizon_fire_ensemble(h, x_starts, fire_steps; winds = [4.0, deg2rad(270.0), 0.5], fire_seed = 0,
                              fire_seed_stride = 1, first_step = 1, S = 1, spread = 3.0, N_iter = 100,
                              granularity = 1.0, seed = 0, boxes = zeros(Float64, 4, 0), h_focus = 15.0, h_max = 30.0,
                              want_cells = false, want_states = false)

E independent `run_horizon_fire` scenarios in one call (`cov_run_horizon_fire_ensemble`, after `fire_init!`), each on
a private copy of the handle's current store, parameters and automaton state: column e of `x_starts` (3N x E) starts
scenario e, column e of `winds` (3 x E rows wind_speed, wind_direction, prob_spread; a 3-vector: the same wind for
every scenario) is its wind, and it equals `run_horizon_fire` with `seed + (e - 1) * T * S` and
`fire_seed + (e - 1) * fire_seed_stride` (stride 1: independent fires, 0: the same fire). The handle is left
unchanged. Returns `(X, objectives, stats, step_ms, cells, states)`: `X` 3N x T x E, `objectives` T x E, `stats`
5 x T x E (`run_horizon_fire`'s rows), `step_ms` the device time of every timestep of the whole ensemble, `cells` and
`states` (nx*ny x E, with `want_cells` / `want_states`; else `nothing`) the multiplicities and the automaton state
each scenario leaves.
"""
function run_horizon_fire_ensemble(h::Handle, x_starts::Matrix{Float64}, fire_steps::Vector{Int64};
                                   winds::VecOrMat{Float64} = [4.0, deg2rad(270.0), 0.5], fire_seed = 0,
                                   fire_seed_stride = 1, first_step = 1, S = 1, spread = 3.0, N_iter = 100,
                                   granularity = 1.0, seed = 0, boxes::Matrix{Float64} = zeros(Float64, 4, 0),
                                   h_focus = 15.0, h_max = 30.0, want_cells = false, want_states = false)
    n, E = size(x_starts); K = size(boxes, 2); T = length(fire_steps)
    W = fire_winds(winds, E)
    X = zeros(Float64, n, T, E); obj = zeros(Float64, T, E); stats = zeros(Int64, 5, T, E); ms = zeros(Float64, T)
    cells = want_cells ? zeros(UInt8, lattice_cells(h), E) : nothing
    states = want_states ? zeros(UInt8, lattice_cells(h), E) : nothing
    GC.@preserve x_starts boxes fire_steps W X obj stats ms cells states check(h,
        ccall((:cov_run_horizon_fire_ensemble, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Int64, Float64, Int64, Float64, UInt64, Ptr{Float64}, Int64, Float64,
         Float64, Ptr{Int64}, Ptr{Float64}, UInt64, UInt64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Float64},
         Ptr{UInt8}, Ptr{UInt8}),
        h.ptr, x_starts, E, T, S, spread, N_iter, granularity, seed, K == 0 ? C_NULL : pointer(boxes), K, h_focus,
        h_max, fire_steps, W, fire_seed, fire_seed_stride, first_step, X, obj, stats, ms,
        want_cells ? pointer(cells) : C_NULL, want_states ? pointer(states) : C_NULL))
    return X, obj, stats, ms, cells, states
end

"""
    run_horizon_points_ensemble(h, x_starts, schedules; list_of = zeros(Int64, size(x_starts, 2)), S = 1, spread = 3.0,
                                N_iter = 100, granularity = 1.0, seed = 0, boxes = zeros(Float64, 4, 0),
                                h_focus = 15.0, h_max = 30.0, want_cells = false, want_last_removed = false)

E independent `run_horizon_points` scenarios in one call (`cov_run_horizon_points_ensemble`), each on a private copy
of the handle's current store and parameters: `schedules` holds L fire schedules, each T matrices as
`run_horizon_points` takes them (the same T for all); column e of `x_starts` (3N x E) starts scenario e, which appends
schedule `list_of[e] + 1` (0-based indices, as the C call takes them) and equals `run_horizon_points` with
`seed + (e - 1) * T * S`. The handle is left unchanged. Returns `(X, objectives, stats, step_ms, cells, last_removed)`:
`X` 3N x T x E, `objectives` T x E, `stats` 5 x T x E (`run_horizon_points`' rows), `step_ms` the device time of every
timestep of the whole ensemble, `cells` and `last_removed` (nx*ny x E, with `want_cells` / `want_last_removed`; else
`nothing`) the multiplicities each scenario leaves and what `run_horizon_points` returns as `last_removed` for it.
"""
function run_horizon_points_ensemble(h::Handle, x_starts::Matrix{Float64}, schedules::Vector{Vector{Matrix{Float64}}};
                                     list_of::Vector{Int64} = zeros(Int64, size(x_starts, 2)), S = 1, spread = 3.0,
                                     N_iter = 100, granularity = 1.0, seed = 0,
                                     boxes::Matrix{Float64} = zeros(Float64, 4, 0), h_focus = 15.0, h_max = 30.0,
                                     want_cells = false, want_last_removed = false, list_order = false)
    n, E = size(x_starts); K = size(boxes, 2)
    T, L, pts, offsets = fire_schedules(schedules)
    X = zeros(Float64, n, T, E); obj = zeros(Float64, T, E); stats = zeros(Int64, 5, T, E); ms = zeros(Float64, T)
    cells = want_cells ? zeros(UInt8, lattice_cells(h), E) : nothing
    last = want_last_removed ? zeros(Cint, lattice_cells(h), E) : nothing
    with_list_order(h, list_order) do
        GC.@preserve x_starts boxes pts offsets list_of X obj stats ms cells last check(h,
            ccall((:cov_run_horizon_points_ensemble, LIB), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Int64, Float64, Int64, Float64, UInt64, Ptr{Float64}, Int64, Float64,
             Float64, Ptr{Float64}, Ptr{Int64}, Int64, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Float64},
             Ptr{UInt8}, Ptr{Cint}),
            h.ptr, x_starts, E, T, S, spread, N_iter, granularity, seed, K == 0 ? C_NULL : pointer(boxes), K, h_focus,
            h_max, offsets[end] == 0 ? C_NULL : pointer(pts), offsets, L, list_of, X, obj, stats, ms,
            want_cells ? pointer(cells) : C_NULL, want_last_removed ? pointer(last) : C_NULL))
    end
    return X, obj, stats, ms, cells, last
end

"The L fire schedules of the fire-list ensembles concatenated: (T, L, 5 x P entries, the L * T + 1 offsets)."
function fire_schedules(schedules::Vector{Vector{Matrix{Float64}}})
    L = length(schedules)
    L >= 1 || throw(CovError(-1, "schedules must hold at least one schedule"))
    T = length(schedules[1])
    all(s -> length(s) == T, schedules) || throw(CovError(-1, "every schedule must have the same number of timesteps"))
    rows = [a for s in schedules for a in s]
    offsets = zeros(Int64, L * T + 1)
    for q in 1:L * T
        offsets[q + 1] = offsets[q] + size(rows[q], 2)
    end
    pts = offsets[end] == 0 ? zeros(Float64, 5, 0) : reduce(hcat, rows)
    return T, L, pts, offsets
end

"The 3 x E winds of the fire ensembles: a 3-vector repeated for every scenario, or 3 x E as given."
function fire_winds(winds::VecOrMat{Float64}, E::Integer)
    W = winds isa Vector ? repeat(winds, 1, E) : winds
    size(W) == (3, E) || throw(CovError(-2, "winds must be 3 x E or a 3-vector"))
    return W
end

"The cells of the lattice set through the binding on h (`cells_out` rows of the ensemble calls)."
function lattice_cells(h::Handle)
    h.ncells > 0 || throw(CovError(-2, "want_cells needs the lattice set through set_points!, set_grid_full! or fire_init!"))
    return h.ncells
end

"Several devices of one box (`cov_multi_create`): one handle per device, borrowed with `shard_handle`."
mutable struct MultiHandle
    ptr::Ptr{Cvoid}
    shards::Vector{Handle} # borrowed views of the shards' handles, one per device
    function MultiHandle(devices::Vector{Cint})
        out = Ref{Ptr{Cvoid}}(C_NULL)
        rc = ccall((:cov_multi_create, LIB), Cint, (Ptr{Cint}, Cint, Ref{Ptr{Cvoid}}), devices, length(devices), out)
        rc == 0 || throw(CovError(rc, unsafe_string(ccall((:cov_last_error, LIB), Cstring, (Ptr{Cvoid},), C_NULL))))
        m = new(out[], Handle[])
        for k in 0:length(devices) - 1
            push!(m.shards, Handle(ccall((:cov_multi_handle, LIB), Ptr{Cvoid}, (Ptr{Cvoid}, Cint), m.ptr, k), 0))
        end
        finalizer(m -> (m.ptr == C_NULL || ccall((:cov_multi_destroy, LIB), Cvoid, (Ptr{Cvoid},), m.ptr);
                        m.ptr = C_NULL), m)
        return m
    end
end

check(m::MultiHandle, rc::Cint) =
    rc == 0 || throw(CovError(rc, unsafe_string(ccall((:cov_multi_last_error, LIB), Cstring, (Ptr{Cvoid},), m.ptr))))

"""
    shard_handle(m, k)

Shard k's handle (0-based), owned by `m`: set the same store and parameters on every shard through it. Keep `m`
alive while it is used.
"""
function shard_handle(m::MultiHandle, k::Integer)
    0 <= k < length(m.shards) || throw(CovError(-1, "no shard $k"))
    return m.shards[k + 1]
end

"""
    multi_run_horizon_ensemble(m, x_starts; T, S = 1, spread = 3.0, N_iter = 100, granularity = 1.0, seed = 0,
                               boxes = zeros(Float64, 4, 0), h_focus = 15.0, h_max = 30.0, want_cells = false)

`run_horizon_ensemble` over the devices of `m` (`cov_multi_run_horizon_ensemble`): contiguous shards of scenarios,
each with the keys it has in the single-device call, so the results are the same bits. Returns `(X, objectives,
stats, cells)`.
"""
function multi_run_horizon_ensemble(m::MultiHandle, x_starts::Matrix{Float64}; T, S = 1, spread = 3.0, N_iter = 100,
                                    granularity = 1.0, seed = 0, boxes::Matrix{Float64} = zeros(Float64, 4, 0),
                                    h_focus = 15.0, h_max = 30.0, want_cells = false, list_order = false)
    n, E = size(x_starts); K = size(boxes, 2)
    X = zeros(Float64, n, T, E); obj = zeros(Float64, T, E); stats = zeros(Int64, 4, T, E)
    cells = nothing
    if want_cells # every shard's lattice, as set through the binding, must be the same
        nc = lattice_cells(m.shards[1])
        all(s -> lattice_cells(s) == nc, m.shards) || throw(CovError(-2, "the shards hold different lattices"))
        cells = zeros(UInt8, nc, E)
    end
    with_list_order(m, list_order) do
        GC.@preserve x_starts boxes X obj stats cells check(m, ccall((:cov_multi_run_horizon_ensemble, LIB), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Int64, Float64, Int64, Float64, UInt64, Ptr{Float64}, Int64, Float64,
             Float64, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{UInt8}),
            m.ptr, x_starts, E, T, S, spread, N_iter, granularity, seed, K == 0 ? C_NULL : pointer(boxes), K, h_focus,
            h_max, X, obj, stats, want_cells ? pointer(cells) : C_NULL))
    end
    return X, obj, stats, cells
end

"""
    multi_run_horizon_fire_ensemble(m, x_starts, fire_steps; winds = [4.0, deg2rad(270.0), 0.5], fire_seed = 0,
                                    fire_seed_stride = 1, first_step = 1, S = 1, spread = 3.0, N_iter = 100,
                                    granularity = 1.0, seed = 0, boxes = zeros(Float64, 4, 0), h_focus = 15.0,
                                    h_max = 30.0, want_cells = false, want_states = false)

`run_horizon_fire_ensemble` over the devices of `m` (`cov_multi_run_horizon_fire_ensemble`): contiguous shards of
scenarios, each with the keys, fire seeds and winds it has in the single-device call, so the results are the same
bits. Call `fire_init!` and set the same parameters on every `shard_handle` first. Returns `(X, objectives, stats,
cells, states)`.
"""
function multi_run_horizon_fire_ensemble(m::MultiHandle, x_starts::Matrix{Float64}, fire_steps::Vector{Int64};
                                         winds::VecOrMat{Float64} = [4.0, deg2rad(270.0), 0.5], fire_seed = 0,
                                         fire_seed_stride = 1, first_step = 1, S = 1, spread = 3.0, N_iter = 100,
                                         granularity = 1.0, seed = 0, boxes::Matrix{Float64} = zeros(Float64, 4, 0),
                                         h_focus = 15.0, h_max = 30.0, want_cells = false, want_states = false)
    n, E = size(x_starts); K = size(boxes, 2); T = length(fire_steps)
    W = fire_winds(winds, E)
    X = zeros(Float64, n, T, E); obj = zeros(Float64, T, E); stats = zeros(Int64, 5, T, E)
    cells = states = nothing
    if want_cells || want_states # every shard's lattice, as set through the binding, must be the same
        nc = lattice_cells(m.shards[1])
        all(s -> lattice_cells(s) == nc, m.shards) || throw(CovError(-2, "the shards hold different lattices"))
        cells = want_cells ? zeros(UInt8, nc, E) : nothing
        states = want_states ? zeros(UInt8, nc, E) : nothing
    end
    GC.@preserve x_starts boxes fire_steps W X obj stats cells states check(m,
        ccall((:cov_multi_run_horizon_fire_ensemble, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Int64, Float64, Int64, Float64, UInt64, Ptr{Float64}, Int64, Float64,
         Float64, Ptr{Int64}, Ptr{Float64}, UInt64, UInt64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{UInt8},
         Ptr{UInt8}),
        m.ptr, x_starts, E, T, S, spread, N_iter, granularity, seed, K == 0 ? C_NULL : pointer(boxes), K, h_focus,
        h_max, fire_steps, W, fire_seed, fire_seed_stride, first_step, X, obj, stats,
        want_cells ? pointer(cells) : C_NULL, want_states ? pointer(states) : C_NULL))
    return X, obj, stats, cells, states
end

"""
    multi_run_horizon_points_ensemble(m, x_starts, schedules; list_of = zeros(Int64, size(x_starts, 2)), S = 1,
                                      spread = 3.0, N_iter = 100, granularity = 1.0, seed = 0,
                                      boxes = zeros(Float64, 4, 0), h_focus = 15.0, h_max = 30.0, want_cells = false,
                                      want_last_removed = false)

`run_horizon_points_ensemble` over the devices of `m` (`cov_multi_run_horizon_points_ensemble`): contiguous shards of
scenarios, each with the keys and schedules it has in the single-device call, so the results are the same bits. Set
the same store and parameters on every `shard_handle` first. Returns `(X, objectives, stats, cells, last_removed)`.
"""
function multi_run_horizon_points_ensemble(m::MultiHandle, x_starts::Matrix{Float64},
                                           schedules::Vector{Vector{Matrix{Float64}}};
                                           list_of::Vector{Int64} = zeros(Int64, size(x_starts, 2)), S = 1,
                                           spread = 3.0, N_iter = 100, granularity = 1.0, seed = 0,
                                           boxes::Matrix{Float64} = zeros(Float64, 4, 0), h_focus = 15.0, h_max = 30.0,
                                           want_cells = false, want_last_removed = false, list_order = false)
    n, E = size(x_starts); K = size(boxes, 2)
    T, L, pts, offsets = fire_schedules(schedules)
    X = zeros(Float64, n, T, E); obj = zeros(Float64, T, E); stats = zeros(Int64, 5, T, E)
    cells = last = nothing
    if want_cells || want_last_removed # every shard's lattice, as set through the binding, must be the same
        nc = lattice_cells(m.shards[1])
        all(s -> lattice_cells(s) == nc, m.shards) || throw(CovError(-2, "the shards hold different lattices"))
        cells = want_cells ? zeros(UInt8, nc, E) : nothing
        last = want_last_removed ? zeros(Cint, nc, E) : nothing
    end
    with_list_order(m, list_order) do
        GC.@preserve x_starts boxes pts offsets list_of X obj stats cells last check(m,
            ccall((:cov_multi_run_horizon_points_ensemble, LIB), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Int64, Float64, Int64, Float64, UInt64, Ptr{Float64}, Int64, Float64,
             Float64, Ptr{Float64}, Ptr{Int64}, Int64, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{UInt8},
             Ptr{Cint}),
            m.ptr, x_starts, E, T, S, spread, N_iter, granularity, seed, K == 0 ? C_NULL : pointer(boxes), K, h_focus,
            h_max, offsets[end] == 0 ? C_NULL : pointer(pts), offsets, L, list_of, X, obj, stats,
            want_cells ? pointer(cells) : C_NULL, want_last_removed ? pointer(last) : C_NULL))
    end
    return X, obj, stats, cells, last
end

"""
    set_region!(h, x_lo, y_lo, x_hi, y_hi, covered)

The grid-free static objective's region: the domain rectangle and the discs already covered, `covered` a 3 x M
matrix with columns [x; y; R] (0 columns: nothing covered yet).
"""
function set_region!(h::Handle, x_lo, y_lo, x_hi, y_hi, covered::Matrix{Float64} = zeros(Float64, 3, 0))
    M = size(covered, 2)
    xyR = vec(permutedims(covered))  # [x_1..x_M; y_1..y_M; R_1..R_M]
    GC.@preserve xyR check(h, ccall((:cov_set_region, LIB), Cint,
        (Ptr{Cvoid}, Float64, Float64, Float64, Float64, Ptr{Float64}, Int64),
        h.ptr, x_lo, y_lo, x_hi, y_hi, M == 0 ? C_NULL : pointer(xyR), M))
end

"Objective, newly covered area and feasibility of every column of `X` (3N x B) on the region (`set_region!`)."
function objective_region_batch(h::Handle, X::Matrix{Float64})
    B = size(X, 2)
    obj = Vector{Float64}(undef, B); area = Vector{Float64}(undef, B); feasible = Vector{UInt8}(undef, B)
    GC.@preserve X obj area feasible check(h, ccall((:cov_eval_region_batch, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{UInt8}, Int32, Ptr{Float64}, Ptr{Int64}),
        h.ptr, X, B, obj, area, feasible, 1, C_NULL, C_NULL))
    return obj, area, feasible
end

"`mads_solve_batch` on the region objective of `objective_region_batch` (no cell store needed)."
function mads_solve_batch_region(h::Handle, X0::Matrix{Float64}; N_iter = 100, granularity = 1.0, seed = 0)
    S = size(X0, 2)
    out = similar(X0); obj = zeros(Float64, S); stats = zeros(Int64, 4, S)
    t = @elapsed GC.@preserve X0 out obj stats check(h, ccall((:cov_mads_solve_batch_region, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Float64, UInt64, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}),
        h.ptr, X0, S, N_iter, granularity, seed, out, obj, stats))
    return out, obj, stats, t
end

"""
    run_horizon_region(h, x_start; T, S = 1, spread = 3.0, N_iter = 100, granularity = 1.0, seed = 0,
                       boxes = zeros(Float64, 4, 0), h_focus = 15.0, h_max = 30.0)

`run_horizon` on the region objective (`cov_run_horizon_region`): per timestep the current swarm's discs with R > 0
join the region's covered set, then the r_max rule, cons3 from the current swarm, S `mads_solve_batch_region` solves
and the best as the next swarm. Needs `set_region!` and `set_params!` with a previous swarm. Returns
`(X, objectives, stats, step_ms)`: `X` 3N x T, `stats` 4 x T with rows winner, evaluations, feasible solves, arcs of
the covered set's boundary.
"""
function run_horizon_region(h::Handle, x_start::Vector{Float64}; T, S = 1, spread = 3.0, N_iter = 100,
                            granularity = 1.0, seed = 0, boxes::Matrix{Float64} = zeros(Float64, 4, 0), h_focus = 15.0,
                            h_max = 30.0)
    n = length(x_start); K = size(boxes, 2)
    X = zeros(Float64, n, T); obj = zeros(Float64, T); stats = zeros(Int64, 4, T); ms = zeros(Float64, T)
    GC.@preserve x_start boxes X obj stats ms check(h, ccall((:cov_run_horizon_region, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Float64, Int64, Float64, UInt64, Ptr{Float64}, Int64, Float64,
         Float64, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Float64}),
        h.ptr, x_start, T, S, spread, N_iter, granularity, seed, K == 0 ? C_NULL : pointer(boxes), K, h_focus, h_max,
        X, obj, stats, ms))
    return X, obj, stats, ms
end

"""
    createObjective(cells, N, r_max; handle = Handle())

Same signature and value as the reference's `TDM_STATIC_opt.createObjective` (src/TDM_STATIC_opt.jl:82):
uploads `cells.points_of_interest` once and returns `AreaMaxObjective(x)`.
"""
function createObjective(cells, N, r_max; handle::Handle = Handle(), nx = 100, ny = 100, dx = 5.0, dy = 5.0)
    set_points!(handle, cells.points_of_interest; nx = nx, ny = ny, dx = dx, dy = dy)
    set_params!(handle, N, collect(Float64, r_max))
    AreaMaxObjective(x) = eval_one(handle, x)
    return AreaMaxObjective
end

end # module
