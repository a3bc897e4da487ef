# PAMG.jl — thin `ccall` shim from PartitionedArrays.jl objects to libpamg.so (include/pamg.h).
#
# STATUS: EXPERIMENTAL, NOT EXECUTED.  Julia is not installed in the build image and PartitionedArrays.jl is
# not vendored in the reference snapshot (/root/reference holds README.md:1-2 and LICENSE only), so every
# PartitionedArrays accessor name below is [RECALL-UNVERIFIED] (SURVEY.md App. A).  What CAN be checked is the
# marshalling arithmetic: tests/julia_shim_emulation.py restates `part_rows`, `ghost_permutation` and the
# local-vector permutation of `device_consistent!` / `device_assemble!` line by line in numpy on the same kind of
# inputs (1-based Int64 CSC blocks of the split local matrix, ghosts in discovery order) and
# tests/test_julia_shim_marshalling.py feeds the result to pamg_set_part_rows / pamg_consistent and compares with
# the oracle bit for bit.  All other logic lives below the C ABI.
#
# Usage (debug backend: all parts in this process; MPI backend: one rank per GPU of one node):
#   S = PAMG.setup(A)                 # A::PSparseMatrix (assembled, split format)   ~ setup(amg(), x, A, b)
#   PAMG.solve!(x, S, b)              # AMG-preconditioned CG to rtol                ~ solve!(x, S, b)
#   PAMG.vcycle!(z, S, r)             # one preconditioner application               ~ ldiv!(z, P, r)
#   PAMG.finalize!(S)
module PAMG

using PartitionedArrays
using SparseArrays

const lib = get(ENV, "PAMG_LIB", joinpath(@__DIR__, "..", "parallel_amg_b200", "libpamg.so"))

struct Options            # mirrors pamg_options (include/pamg.h); filled by pamg_default_options
    struct_size::Int32; eps_strength::Float64; coarse_size::Int32; max_levels::Int32
    smoother::Int32; omega_jacobi::Float64; nu_pre::Int32; nu_post::Int32; cheb_degree::Int32
    cheb_lo_frac::Float64; cheb_hi_frac::Float64; spmv_format::Int32; use_graph::Int32
    lanes_per_row::Int32; tail_rows::Int32; sell_sigma::Int32; sell_rows_per_thread::Int32; fuse_halo::Int32
    cycle::Int32
end

mutable struct Setup
    ctx::Ptr{Cvoid}
    nparts::Int
    local_parts::Vector{Int}          # 1-based part ids driven by this process
    ghost_perm::Dict{Int,Vector{Int}} # part => perm with lib_ghost[k] = pa_ghost[perm[k]] (level 0)
end

function check(ctx, st)
    st == 0 && return
    msg = ctx == C_NULL ? "" : unsafe_string(ccall((:pamg_last_error, lib), Cstring, (Ptr{Cvoid},), ctx))
    error("pamg status $st: $msg")          # -5 (PAMG_ERR_NOTCONV) is handled by the caller
end

default_options() = (r = Ref{Options}(); ccall((:pamg_default_options, lib), Cvoid, (Ref{Options},), r); r[])

is_mpi(a) = nameof(typeof(a)) == :MPIArray      # one item per process; DebugArray / Vector: every item is here

# CSR of the OWN ROWS of one part with GLOBAL 0-based column ids, from the split local matrix:
#   Aoo = own_own_values(A)   (n_own x n_own,   SparseMatrixCSC, 1-based)
#   Aog = own_ghost_values(A) (n_own x n_ghost, SparseMatrixCSC, 1-based)
# A CSC matrix lists, per COLUMN, the rows that hold an entry; the rows we need are the columns of the
# transposes, so both blocks are transposed once (no symmetry assumption) and row i is the concatenation of
# column i of transpose(Aoo) (own-local column ids -> own_to_global) and of transpose(Aog) (ghost-local column
# ids -> ghost_to_global).  The library sorts each row by global column id itself.
function part_rows(Aoo::SparseMatrixCSC, Aog::SparseMatrixCSC, row_ids, col_ids)
    o2g_rows = Int64.(own_to_global(row_ids)) .- 1
    o2g = Int64.(own_to_global(col_ids)) .- 1
    g2g = Int64.(ghost_to_global(col_ids)) .- 1
    nown = length(o2g_rows)
    Too = sparse(transpose(Aoo))               # column i of Too = row i of Aoo
    Tog = sparse(transpose(Aog))
    rowptr = zeros(Int64, nown + 1)
    for i in 1:nown
        rowptr[i+1] = rowptr[i] + (Too.colptr[i+1] - Too.colptr[i]) + (Tog.colptr[i+1] - Tog.colptr[i])
    end
    colgid = Vector{Int64}(undef, rowptr[end])
    val = Vector{Float64}(undef, rowptr[end])
    for i in 1:nown
        q = rowptr[i]
        for k in Too.colptr[i]:Too.colptr[i+1]-1
            q += 1; colgid[q] = o2g[Too.rowval[k]]; val[q] = Too.nzval[k]
        end
        for k in Tog.colptr[i]:Tog.colptr[i+1]-1
            q += 1; colgid[q] = g2g[Tog.rowval[k]]; val[q] = Tog.nzval[k]
        end
    end
    (o2g_rows, rowptr, colgid, val)
end

# The library orders the ghosts of a part by (owner part, global id); PartitionedArrays keeps discovery order.
# perm[k] = position in the PartitionedArrays ghost list of the library's ghost k (both lists hold the same ids).
function ghost_permutation(lib_ghost_gid0::Vector{Int64}, pa_ghost_gid1)
    pos = Dict{Int64,Int}(Int64(g) - 1 => k for (k, g) in enumerate(pa_ghost_gid1))
    [pos[g] for g in lib_ghost_gid0]
end

# level-0 ghost ids of a part in the library's order (0-based); NULL outputs are skipped by the C side
function lib_ghost_to_global(ctx, part0, n_ghost)
    gh = Vector{Int64}(undef, n_ghost)
    check(ctx, ccall((:pamg_get_index_maps, lib), Cint, (Ptr{Cvoid}, Int32, Int32, Ptr{Int64}, Ptr{Int64}, Ptr{Int32}),
                     ctx, 0, part0, C_NULL, gh, C_NULL))
    gh
end

# nullspace: optional n x k matrix (global row order) of near-nullspace vectors, e.g. the 6 rigid-body modes from
# `nullspace_linear_elasticity`; block_size: DOFs per node (3 for 3-D elasticity).
# devices: GPU id per LOCAL part (debug backend default 0:np-1; MPI backend default [local rank of this process]).
function setup(A::PSparseMatrix; devices = nothing, opts::Options = default_options(), nullspace = nothing, block_size = 1,
               rhs_capacity = 1)
    rows, cols = partition(axes(A, 1)), partition(axes(A, 2))
    np = length(rows)
    ranks = linear_indices(rows)
    mpi = is_mpi(rows)
    # rows of every part, marshalled where the part lives, then all-gathered (the host setup is replicated and
    # deterministic: every process builds the same hierarchy and uploads only the parts it drives)
    data = map(part_rows, own_own_values(A), own_ghost_values(A), rows, cols)
    all_o2g = gather(map(d -> d[1], data); destination = :all)
    all_ptr = gather(map(d -> d[2], data); destination = :all)
    all_col = gather(map(d -> d[3], data); destination = :all)
    all_val = gather(map(d -> d[4], data); destination = :all)
    pa_ghosts = map(c -> collect(ghost_to_global(c)), cols)
    out = map(ranks, all_o2g, all_ptr, all_col, all_val) do rank, o2gs, ptrs, colss, vals
        (mpi || rank == 1) || return nothing                     # debug backend: one context for all parts
        r = Ref{Ptr{Cvoid}}(C_NULL)
        check(C_NULL, ccall((:pamg_create, lib), Cint, (Int32, Ref{Ptr{Cvoid}}), np, r))
        ctx = r[]
        for p in 1:np
            o2g, rowptr, colgid, val = collect(o2gs[p]), collect(ptrs[p]), collect(colss[p]), collect(vals[p])
            check(ctx, ccall((:pamg_set_part_rows, lib), Cint,
                             (Ptr{Cvoid}, Int32, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}),
                             ctx, p - 1, length(o2g), o2g, rowptr, colgid, val))
        end
        if nullspace !== nothing
            B = permutedims(Matrix{Float64}(nullspace))           # row-major n x k for the C side
            check(ctx, ccall((:pamg_set_near_nullspace, lib), Cint, (Ptr{Cvoid}, Int32, Int32, Ptr{Float64}),
                             ctx, block_size, size(nullspace, 2), B))
        end
        check(ctx, ccall((:pamg_setup, lib), Cint, (Ptr{Cvoid}, Ref{Options}), ctx, Ref(opts)))
        check(ctx, ccall((:pamg_set_rhs_capacity, lib), Cint, (Ptr{Cvoid}, Int32), ctx, rhs_capacity))
        locals = mpi ? [rank] : collect(1:np)
        devs = devices === nothing ? (mpi ? Int32[parse(Int, get(ENV, "LOCAL_RANK", "0"))] : Int32.(0:np-1)) : Int32.(devices)
        check(ctx, ccall((:pamg_device_init, lib), Cint, (Ptr{Cvoid}, Int32, Ptr{Int32}, Ptr{Int32}),
                         ctx, length(locals), Int32.(locals .- 1), devs))
        Setup(ctx, np, locals, Dict{Int,Vector{Int}}())
    end
    if mpi
        # with_mpi: all-gather one opaque peer-memory handle per rank, map the others' arenas (INTEGRATION.md §4)
        nb = ccall((:pamg_comm_handle_bytes, lib), Int32, ())
        blobs = map(ranks, out) do rank, S
            blob = zeros(UInt8, nb)
            check(S.ctx, ccall((:pamg_comm_export, lib), Cint, (Ptr{Cvoid}, Int32, Ptr{UInt8}), S.ctx, rank - 1, blob))
            blob
        end
        allblobs = gather(blobs; destination = :all)
        map(ranks, out, allblobs) do rank, S, bl
            for q in 1:np
                q == rank && continue
                check(S.ctx, ccall((:pamg_comm_import, lib), Cint, (Ptr{Cvoid}, Int32, Ptr{UInt8}), S.ctx, q - 1, collect(bl[q])))
            end
            check(S.ctx, ccall((:pamg_comm_connect, lib), Cint, (Ptr{Cvoid},), S.ctx))
        end
    end
    # ghost order: library (owner, gid) vs PartitionedArrays discovery order, per local part
    S = nothing
    map(ranks, out, pa_ghosts) do rank, s, gh
        s === nothing || (S = s)
    end
    map(ranks, pa_ghosts) do rank, gh
        (S !== nothing && rank in S.local_parts) || return
        S.ghost_perm[rank] = ghost_permutation(lib_ghost_to_global(S.ctx, rank - 1, length(gh)), gh)
    end
    S
end

# nparts pointers to the contiguous OWN blocks; NULL for parts another process drives
function own_ptrs(v::PVector, S::Setup)
    ptrs = fill(Ptr{Float64}(C_NULL), S.nparts)
    map(linear_indices(partition(axes(v, 1))), own_values(v)) do rank, o
        rank in S.local_parts && (ptrs[rank] = pointer(o))
    end
    ptrs
end

function solve!(x::PVector, S::Setup, b::PVector; rtol = 1e-8, maxiter = 200, precond = true)
    iters = Ref{Int32}(0)
    hist = zeros(Float64, maxiter + 2)
    bp, xp = own_ptrs(b, S), own_ptrs(x, S)
    st = GC.@preserve b x ccall((:pamg_pcg, lib), Cint,
        (Ptr{Cvoid}, Ptr{Ptr{Float64}}, Ptr{Ptr{Float64}}, Float64, Int32, Int32, Ref{Int32}, Ptr{Float64}),
        S.ctx, bp, xp, rtol, maxiter, precond ? 1 : 0, iters, hist)
    st == -5 || check(S.ctx, st)
    wait(consistent!(x))                       # ghosts of the returned PVector (host side)
    (iterations = Int(iters[]), converged = st == 0, residuals = hist[1:iters[]+1])
end

# flexible AMG-preconditioned CG (pamg_fcg) and restarted flexible GMRES (pamg_fgmres): same result tuple as solve!
function solve_fcg!(x::PVector, S::Setup, b::PVector; rtol = 1e-8, maxiter = 200)
    iters = Ref{Int32}(0)
    hist = zeros(Float64, maxiter + 2)
    bp, xp = own_ptrs(b, S), own_ptrs(x, S)
    st = GC.@preserve b x ccall((:pamg_fcg, lib), Cint,
        (Ptr{Cvoid}, Ptr{Ptr{Float64}}, Ptr{Ptr{Float64}}, Float64, Int32, Ref{Int32}, Ptr{Float64}),
        S.ctx, bp, xp, rtol, maxiter, iters, hist)
    st == -5 || check(S.ctx, st)
    wait(consistent!(x))
    (iterations = Int(iters[]), converged = st == 0, residuals = hist[1:iters[]+1])
end

function solve_gmres!(x::PVector, S::Setup, b::PVector; rtol = 1e-8, maxiter = 200, restart = 30, precond = true)
    iters = Ref{Int32}(0)
    hist = zeros(Float64, maxiter + 2)
    bp, xp = own_ptrs(b, S), own_ptrs(x, S)
    st = GC.@preserve b x ccall((:pamg_fgmres, lib), Cint,
        (Ptr{Cvoid}, Ptr{Ptr{Float64}}, Ptr{Ptr{Float64}}, Float64, Int32, Int32, Int32, Ref{Int32}, Ptr{Float64}),
        S.ctx, bp, xp, rtol, maxiter, restart, precond ? 1 : 0, iters, hist)
    st == -5 || check(S.ctx, st)
    wait(consistent!(x))
    (iterations = Int(iters[]), converged = st == 0, residuals = hist[1:iters[]+1])   # residuals: the Arnoldi estimates
end

# k solve! calls sharing one setup (pamg_pcg_multi; setup(...; rhs_capacity >= k)): xs[j] and the j-th result tuple are
# bit-identical to solve!(xs[j], S, bs[j]); mode 0 CG, 1 AMG-PCG, 2 flexible AMG-PCG
function solve_multi!(xs::Vector{<:PVector}, S::Setup, bs::Vector{<:PVector}; rtol = 1e-8, maxiter = 200, mode = 1)
    k = length(bs)
    iters = zeros(Int32, k)
    conv = zeros(Int32, k)
    hist = zeros(Float64, maxiter + 1, k)          # column j = row j of the C k x (maxiter + 1) array
    bp = reduce(vcat, [own_ptrs(b, S) for b in bs])
    xp = reduce(vcat, [own_ptrs(x, S) for x in xs])
    st = GC.@preserve bs xs ccall((:pamg_pcg_multi, lib), Cint,
        (Ptr{Cvoid}, Int32, Ptr{Ptr{Float64}}, Ptr{Ptr{Float64}}, Float64, Int32, Int32, Ptr{Int32}, Ptr{Int32}, Ptr{Float64}),
        S.ctx, k, bp, xp, rtol, maxiter, mode, iters, conv, hist)
    st == -5 || check(S.ctx, st)
    foreach(x -> wait(consistent!(x)), xs)
    [(iterations = Int(iters[j]), converged = conv[j] == 1, residuals = hist[1:iters[j]+1, j]) for j in 1:k]
end

function vcycle!(z::PVector, S::Setup, r::PVector)
    rp, zp = own_ptrs(r, S), own_ptrs(z, S)
    GC.@preserve r z check(S.ctx, ccall((:pamg_vcycle, lib), Cint,
        (Ptr{Cvoid}, Ptr{Ptr{Float64}}, Ptr{Ptr{Float64}}), S.ctx, rp, zp))
    z
end

# device halo exchange of a level-0 vector.  The C side takes LOCAL values as [own ; ghosts in LIBRARY order], so the
# ghost segment is permuted on the way in and out: lib_ghost[k] = pa_ghost[perm[k]].
function device_halo!(fname::Symbol, v::PVector, S::Setup)
    bufs = Dict{Int,Vector{Float64}}()
    ptrs = fill(Ptr{Float64}(C_NULL), S.nparts)
    ranks = linear_indices(partition(axes(v, 1)))
    map(ranks, own_values(v), ghost_values(v)) do rank, o, g
        rank in S.local_parts || return
        bufs[rank] = vcat(collect(o), collect(g)[S.ghost_perm[rank]])
        ptrs[rank] = pointer(bufs[rank])
    end
    GC.@preserve bufs check(S.ctx, ccall((fname, lib), Cint, (Ptr{Cvoid}, Int32, Ptr{Ptr{Float64}}), S.ctx, 0, ptrs))
    map(ranks, own_values(v), ghost_values(v)) do rank, o, g
        rank in S.local_parts || return
        no = length(o)
        o .= view(bufs[rank], 1:no)
        g[S.ghost_perm[rank]] .= view(bufs[rank], no+1:no+length(g))
    end
    v
end
device_consistent!(v::PVector, S::Setup) = device_halo!(:pamg_consistent, v, S)   # consistent!(v) |> wait
device_assemble!(v::PVector, S::Setup) = device_halo!(:pamg_assemble, v, S)       # assemble!(v) |> wait

finalize!(S::Setup) = (ccall((:pamg_destroy, lib), Cvoid, (Ptr{Cvoid},), S.ctx); S.ctx = C_NULL; nothing)

end # module
