# device_hierarchy.jl - the reference-side binding of libamg1d.so (C ABI: include/amg1d.h).
#
# To be included in the reference's module after solvers.jl (src/AgglomerationMultigrid1D.jl):
#
#     include( "device_hierarchy.jl" )
#
# It keeps the package's entry points - multigrid_v_cycle, multigrid, ldiv!, apply_smoother - and adds
# methods for `DeviceHierarchy`, the uploaded form of a `MeshHierarchy`; every method is one ccall.
# Names used from the module: MeshHierarchy, CgMesh, DgMesh, AgglomeratedDgMesh1, AgglomeratedDgMeshN,
# JacobiSmoother, BlockJacobi, and its aliases `sp` (SparseArrays) and `la` (LinearAlgebra).
#
# NOT EXECUTED in this repository's build environment (no Julia there).  It targets exactly the ABI that
# the tested Python driver uses (agglomerationmultigrid1d_b200/_capi.py, device.py, blocks.py), call for
# call; INTEGRATION.md maps each reference call (file:line) to its ABI call.

const libamg1d = "libamg1d.so"     # on LD_LIBRARY_PATH, or an absolute path

mutable struct DeviceHierarchy
    handle::Ptr{Cvoid}
    nDof::Vector{Int64}
end

function amg1d_check(h::Ptr{Cvoid}, rc::Cint)
    rc == 0 && return
    msg = unsafe_string(ccall((:amg1d_last_error, libamg1d), Cstring, (Ptr{Cvoid},), h))
    rc == 1 ? throw(ArgumentError(msg)) : error("libamg1d error $rc: $msg")
end

# slot map of a level: slots[i, e] = DOF held by row i of element block e (0 = padding)
level_slots(m::Union{DgMesh, AgglomeratedDgMesh1, AgglomeratedDgMeshN}) =
    hcat([collect(el.mNodesInd) for el in m.mElements]...)
function level_slots(m::CgMesh)                 # [vertex_k, interior nodes of element k], k = 1..n+1
    n, p = length(m.mElements), m.mP
    s = zeros(Int64, p, n + 1)
    for (k, el) in enumerate(m.mElements)
        s[1, k] = el.mNodesInd[1]
        s[2:p, k] = el.mNodesInd[3:end]
    end
    s[1, n + 1] = m.mElements[end].mNodesInd[2]
    return s
end

# block-tridiagonal blocks of A in the grouping `slots` (column-major blocks, element-major outside)
function level_blocks(A::sp.SparseMatrixCSC{Float64,Int64}, slots::Matrix{Int64})
    m, n = size(slots)
    elemOf = zeros(Int64, size(A, 1)); locOf = zeros(Int64, size(A, 1))
    for e in 1:n, i in 1:m
        slots[i, e] > 0 && (elemOf[slots[i, e]] = e; locOf[slots[i, e]] = i)
    end
    lo = zeros(m, m, n); di = zeros(m, m, n); up = zeros(m, m, n)
    rows = sp.rowvals(A); vals = sp.nonzeros(A)
    for col in 1:size(A, 2), k in sp.nzrange(A, col)
        r = rows[k]; d = elemOf[col] - elemOf[r]
        abs(d) <= 1 || vals[k] == 0.0 || throw(ArgumentError("operator is not block tridiagonal"))
        blk = d == -1 ? lo : (d == 0 ? di : up)
        blk[locOf[r], locOf[col], elemOf[r]] += vals[k]
    end
    for e in 1:n, i in 1:m
        slots[i, e] == 0 && (di[i, i, e] = 1.0)          # padding rows: identity
    end
    return lo, di, up
end

smoother_inverse(S::JacobiSmoother, slots, di) =
    ([slots[i, e] > 0 ? 1.0 / S.mJac[slots[i, e], slots[i, e]] : 1.0
      for i in 1:size(slots, 1), e in 1:size(slots, 2)], 1)
smoother_inverse(S::BlockJacobi, slots, di) =
    (cat([inv(Matrix(b)) for b in S.mBlocks]...; dims = 3), 0)

# (parent, P0, P1) of an interpolation matrix L (src/interpolation.jl) in the groupings `fs` (fine) and
# `cs` (coarse):  x_f[e] += P0[:, :, e] * x_c[parent[e]] + P1[:, :, e] * x_c[parent[e] + 1].
# parent is 0-based and non-decreasing; P1 === nothing for single-parent transfers (dg_dg, aggdg_dg,
# aggdg_aggdg); cg_cg / dg_cg / aggdg_cg rows at shared vertices reach into the next coarse group.
function transfer_blocks(L::sp.SparseMatrixCSC{Float64,Int64}, fs::Matrix{Int64}, cs::Matrix{Int64})
    mf, nf = size(fs); mc, nc = size(cs)
    eF = zeros(Int64, size(L, 1)); lF = zeros(Int64, size(L, 1))
    eC = zeros(Int64, size(L, 2)); lC = zeros(Int64, size(L, 2))
    for e in 1:nf, i in 1:mf
        fs[i, e] > 0 && (eF[fs[i, e]] = e; lF[fs[i, e]] = i)
    end
    for e in 1:nc, i in 1:mc
        cs[i, e] > 0 && (eC[cs[i, e]] = e; lC[cs[i, e]] = i)
    end
    rows = sp.rowvals(L); vals = sp.nonzeros(L)
    pmin = fill(typemax(Int64), nf); pmax = zeros(Int64, nf)
    for col in 1:size(L, 2), k in sp.nzrange(L, col)
        vals[k] == 0.0 && continue
        e = eF[rows[k]]
        pmin[e] = min(pmin[e], eC[col]); pmax[e] = max(pmax[e], eC[col])
    end
    for e in 1:nf                                   # all-zero row blocks inherit the left neighbour's parent
        if pmax[e] == 0
            pmin[e] = e > 1 ? pmin[e - 1] : 1
            pmax[e] = pmin[e]
        end
    end
    all(pmax .- pmin .<= 1) || throw(ArgumentError("a fine element depends on more than two adjacent coarse elements"))
    issorted(pmin) || throw(ArgumentError("transfer parents are not monotone"))
    two = any(pmax .> pmin)
    P0 = zeros(mf, mc, nf); P1 = two ? zeros(mf, mc, nf) : nothing
    for col in 1:size(L, 2), k in sp.nzrange(L, col)
        vals[k] == 0.0 && continue
        e = eF[rows[k]]
        blk = eC[col] == pmin[e] ? P0 : P1
        blk[lF[rows[k]], lC[col], e] += vals[k]
    end
    return pmin .- 1, P0, P1
end

function DeviceHierarchy(H::MeshHierarchy; device::Integer = 0)
    nL = length(H.mMeshes)
    href = Ref{Ptr{Cvoid}}(C_NULL)
    amg1d_check(C_NULL, ccall((:amg1d_create, libamg1d), Cint,
                              (Ref{Ptr{Cvoid}}, Cint, Cint, Ptr{Cvoid}), href, nL, device, C_NULL))
    h = href[]
    slots = [level_slots(m) for m in H.mMeshes]
    for l in 1:nL
        lo, di, up = level_blocks(H.mStiffness[l], slots[l])
        dinv, isdiag = smoother_inverse(H.mSmoothers[l], slots[l], di)
        m, n = size(slots[l])
        perm = vec(slots[l]) .- 1                                  # 0-based, -1 = padding
        permptr = perm == collect(0:(m * n - 1)) ? C_NULL : pointer(perm)
        GC.@preserve perm amg1d_check(h, ccall((:amg1d_set_level, libamg1d), Cint,
            (Ptr{Cvoid}, Cint, Int64, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
             Cint, Ptr{Int64}, Int64),
            h, l - 1, n, m, lo, di, up, dinv, isdiag, permptr, size(H.mStiffness[l], 1)))
    end
    for l in 1:(nL - 1)
        parent, P0, P1 = transfer_blocks(H.mInterpolation[l], slots[l], slots[l + 1])  # as blocks.py
        amg1d_check(h, ccall((:amg1d_set_transfer, libamg1d), Cint,
            (Ptr{Cvoid}, Cint, Int64, Cint, Cint, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}),
            h, l - 1, size(slots[l], 2), size(slots[l], 1), size(slots[l + 1], 1), parent, P0,
            P1 === nothing ? C_NULL : P1))
    end
    amg1d_check(h, ccall((:amg1d_finalize, libamg1d), Cint, (Ptr{Cvoid},), h))
    D = DeviceHierarchy(h, [size(A, 1) for A in H.mStiffness])
    finalizer(d -> ccall((:amg1d_destroy, libamg1d), Cint, (Ptr{Cvoid},), d.handle), D)
    return D
end

# ---- the hot path: same names and arguments as src/solvers.jl ----------------------------------
function multigrid_v_cycle(D::DeviceHierarchy, x0::AbstractVector, b::AbstractVector;
                           nPre::Integer = 3, nPost::Integer = 3, alpha::AbstractFloat = 2.0 / 3.0)
    x = Vector{Float64}(x0); bb = Vector{Float64}(b)
    amg1d_check(D.handle, ccall((:amg1d_vcycle, libamg1d), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Cint, Cint, Float64), D.handle, x, bb, nPre, nPost, alpha))
    return x
end

function multigrid(D::DeviceHierarchy, H::MeshHierarchy, x0, b, maxiter::Integer, tol::AbstractFloat)
    x = Vector{Float64}(x0); bb = Vector{Float64}(b)
    uExact = H.mStiffness[1] \ bb                      # error history only, as in src/solvers.jl:120
    res = zeros(maxiter); err = zeros(maxiter); it = Ref{Cint}(0)
    amg1d_check(D.handle, ccall((:amg1d_solve, libamg1d), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Cint, Float64, Cint, Cint, Float64, Ref{Cint},
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        D.handle, x, bb, maxiter, tol, 3, 3, 2.0 / 3.0, it, res, err, uExact))
    return x, Int(it[]), res[1:it[]], err[1:it[]]
end

function ldiv!(y::AbstractVector, D::DeviceHierarchy, b::AbstractVector)
    yy = Vector{Float64}(undef, length(b)); bb = Vector{Float64}(b)
    amg1d_check(D.handle, ccall((:amg1d_ldiv, libamg1d), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Cint, Cint, Float64), D.handle, yy, bb, 3, 3, 2.0 / 3.0))
    y[:] = yy
    return
end
ldiv!(D::DeviceHierarchy, b::AbstractVector) = ldiv!(b, D, b)

# CG with the hierarchy as preconditioner, entirely on the device (what cg(A, b; Pl = H) would do
# through ldiv!, minus one host <-> device round trip per iteration)
function pcg(D::DeviceHierarchy, x0::AbstractVector, b::AbstractVector, maxiter::Integer, tol::AbstractFloat)
    x = Vector{Float64}(x0); bb = Vector{Float64}(b); res = zeros(maxiter); it = Ref{Cint}(0)
    amg1d_check(D.handle, ccall((:amg1d_pcg, libamg1d), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Cint, Float64, Cint, Cint, Float64, Ref{Cint}, Ptr{Float64}),
        D.handle, x, bb, maxiter, tol, 3, 3, 2.0 / 3.0, it, res))
    return x, Int(it[]), res[1:it[]]
end

# One V-cycle per (x0, b) pair of a stream of independent problems, pipelined over PCIe inside the library (upload
# of problem k + 1, cycle of k, download of k - 1 overlap).  zeroGuess = true is the ldiv! form.  X is overwritten.
function multigrid_v_cycle!(D::DeviceHierarchy, X::Vector{Vector{Float64}}, B::Vector{Vector{Float64}};
                            zeroGuess::Bool = false, nPre::Integer = 3, nPost::Integer = 3,
                            alpha::AbstractFloat = 2.0 / 3.0)
    xp = [pointer(x) for x in X]; bp = [pointer(b) for b in B]
    GC.@preserve X B amg1d_check(D.handle, ccall((:amg1d_vcycle_batch, libamg1d), Cint,
        (Ptr{Cvoid}, Cint, Ptr{Ptr{Float64}}, Ptr{Ptr{Float64}}, Cint, Cint, Cint, Float64),
        D.handle, length(X), xp, bp, zeroGuess ? 1 : 0, nPre, nPost, alpha))
    return X
end

# multigrid(H, x0, b, maxiter, tol) on a problem that already lives on the device (amg1d_dev_set_problem or
# amg1d_dev_assemble_rhs): no vector crosses PCIe; fetch the solution with dev_solution.
function multigrid_resident(D::DeviceHierarchy, maxiter::Integer, tol::AbstractFloat)
    res = zeros(maxiter); it = Ref{Cint}(0)
    amg1d_check(D.handle, ccall((:amg1d_dev_solve, libamg1d), Cint,
        (Ptr{Cvoid}, Cint, Float64, Cint, Cint, Float64, Ref{Cint}, Ptr{Float64}),
        D.handle, maxiter, tol, 3, 3, 2.0 / 3.0, it, res))
    return Int(it[]), res[1:it[]]
end
dev_solution(D::DeviceHierarchy) = (x = Vector{Float64}(undef, D.nDof[1]);
    amg1d_check(D.handle, ccall((:amg1d_dev_get_solution, libamg1d), Cint, (Ptr{Cvoid}, Ptr{Float64}), D.handle, x)); x)

# ---- up to AMG1D_MAX_COLS right-hand sides per V-cycle (multi-column resident set) -------------------------------
# UNVERIFIED like the rest of this file (no Julia in this repository's build environment); the Python driver
# (device.py: dev_set_problems ... dev_get_solutions, solvers.ldiv with a 2-D b) is the tested path.
const AMG1D_MAX_COLS = 8
dev_set_problems!(D::DeviceHierarchy, X0::Union{Nothing,AbstractMatrix}, B::AbstractMatrix) =
    (Bd = Matrix{Float64}(B); Xd = X0 === nothing ? Ptr{Float64}(C_NULL) : Matrix{Float64}(X0);
     GC.@preserve Bd Xd amg1d_check(D.handle, ccall((:amg1d_dev_set_problems, libamg1d), Cint,
        (Ptr{Cvoid}, Cint, Ptr{Float64}, Ptr{Float64}), D.handle, size(Bd, 2), Xd, Bd)))
dev_fill_rhs_random_multi!(D::DeviceHierarchy, k::Integer, seed::Integer) =
    amg1d_check(D.handle, ccall((:amg1d_dev_fill_rhs_random_multi, libamg1d), Cint, (Ptr{Cvoid}, Cint, UInt64),
                                D.handle, k, seed))
dev_vcycle_multi!(D::DeviceHierarchy; nPre::Integer = 3, nPost::Integer = 3, alpha::AbstractFloat = 2.0 / 3.0,
                  zeroGuess::Bool = false, withResidualNorms::Bool = false) =
    amg1d_check(D.handle, ccall((:amg1d_dev_vcycle_multi, libamg1d), Cint, (Ptr{Cvoid}, Cint, Cint, Float64, Cint, Cint),
                                D.handle, nPre, nPost, alpha, zeroGuess ? 1 : 0, withResidualNorms ? 1 : 0))
dev_residual_norms(D::DeviceHierarchy) = (res = zeros(get_info(D, "multi_columns"));
    amg1d_check(D.handle, ccall((:amg1d_dev_residual_norms, libamg1d), Cint, (Ptr{Cvoid}, Ptr{Float64}), D.handle, res)); res)
function multigrid_resident_multi(D::DeviceHierarchy, maxiter::Integer, tol::AbstractFloat)
    k = get_info(D, "multi_columns"); res = zeros(maxiter, k); it = zeros(Cint, k)
    amg1d_check(D.handle, ccall((:amg1d_dev_solve_multi, libamg1d), Cint,
        (Ptr{Cvoid}, Cint, Float64, Cint, Cint, Float64, Ptr{Cint}, Ptr{Float64}),
        D.handle, maxiter, tol, 3, 3, 2.0 / 3.0, it, res))
    return Int.(it), [res[1:it[c], c] for c in 1:k]
end
# pcg on every column of the set; the right-hand sides are consumed, the solutions stay on the device (dev_solutions)
function pcg_resident_multi(D::DeviceHierarchy, maxiter::Integer, tol::AbstractFloat)
    k = get_info(D, "multi_columns"); res = zeros(maxiter, k); it = zeros(Cint, k)
    amg1d_check(D.handle, ccall((:amg1d_dev_pcg_multi, libamg1d), Cint,
        (Ptr{Cvoid}, Cint, Float64, Cint, Cint, Float64, Ptr{Cint}, Ptr{Float64}),
        D.handle, maxiter, tol, 3, 3, 2.0 / 3.0, it, res))
    return Int.(it), [res[1:it[c], c] for c in 1:k]
end
dev_solutions(D::DeviceHierarchy) = (X = Matrix{Float64}(undef, D.nDof[1], get_info(D, "multi_columns"));
    amg1d_check(D.handle, ccall((:amg1d_dev_get_solutions, libamg1d), Cint, (Ptr{Cvoid}, Ptr{Float64}), D.handle, X)); X)

# ldiv!(Y, H, B): every column as ldiv!(y, H, b), up to AMG1D_MAX_COLS columns per V-cycle
function ldiv!(Y::AbstractMatrix, D::DeviceHierarchy, B::AbstractMatrix)
    size(Y) == size(B) || throw(DimensionMismatch("Y $(size(Y)) vs B $(size(B))"))
    for c0 in 1:AMG1D_MAX_COLS:size(B, 2)
        cols = c0:min(c0 + AMG1D_MAX_COLS - 1, size(B, 2))
        dev_set_problems!(D, nothing, B[:, cols])
        dev_vcycle_multi!(D; zeroGuess = true)
        Y[:, cols] = dev_solutions(D)
    end
    return
end

# pcg(D, X0, B, ...): every column as pcg(D, x0, b, ...), up to AMG1D_MAX_COLS columns sharing each V-cycle
function pcg(D::DeviceHierarchy, X0::AbstractMatrix, B::AbstractMatrix, maxiter::Integer, tol::AbstractFloat)
    size(X0) == size(B) || throw(DimensionMismatch("X0 $(size(X0)) vs B $(size(B))"))
    X = similar(B, Float64); iters = Int[]; res = Vector{Vector{Float64}}()
    for c0 in 1:AMG1D_MAX_COLS:size(B, 2)
        cols = c0:min(c0 + AMG1D_MAX_COLS - 1, size(B, 2))
        dev_set_problems!(D, X0[:, cols], B[:, cols])
        it, r = pcg_resident_multi(D, maxiter, tol)
        X[:, cols] = dev_solutions(D)
        append!(iters, it); append!(res, r)
    end
    return X, iters, res
end

function apply_smoother(D::DeviceHierarchy, level::Integer, B::AbstractVecOrMat; alpha::Float64 = 1.0)
    Bd = Matrix{Float64}(reshape(Array(B), size(B, 1), :)); Y = similar(Bd)
    amg1d_check(D.handle, ccall((:amg1d_apply_smoother, libamg1d), Cint,
        (Ptr{Cvoid}, Cint, Ptr{Float64}, Ptr{Float64}, Int64, Float64),
        D.handle, level - 1, Y, Bd, size(Bd, 2), alpha))
    return B isa AbstractVector ? vec(Y) : Y
end

function iterative_smoother_solve(D::DeviceHierarchy, level::Integer, x0::AbstractVector, b::AbstractVector;
                                  maxiter::Integer = 1000, tol::AbstractFloat = 1e-6,
                                  alpha::AbstractFloat = 1.0, uExact = nothing)
    x = Vector{Float64}(x0); bb = Vector{Float64}(b)
    res = zeros(maxiter); err = zeros(maxiter); it = Ref{Cint}(0)
    ue = uExact === nothing ? direct_solve(D, level, bb) : Vector{Float64}(uExact)   # A \ b, src/solvers.jl:194
    amg1d_check(D.handle, ccall((:amg1d_smoother_solve, libamg1d), Cint,
        (Ptr{Cvoid}, Cint, Ptr{Float64}, Ptr{Float64}, Cint, Float64, Float64, Ref{Cint}, Ptr{Float64},
         Ptr{Float64}, Ptr{Float64}),
        D.handle, level - 1, x, bb, maxiter, tol, alpha, it, res, err, ue))
    return x, Int(it[]), res[1:it[]], err[1:it[]]
end

# ---- the level operations the reference's scripts use directly (H.mStiffness[k] * u, L' * r, L * u, A \ b) ----
matvec(D::DeviceHierarchy, l::Integer, x) = (y = Vector{Float64}(undef, D.nDof[l]);
    amg1d_check(D.handle, ccall((:amg1d_matvec, libamg1d), Cint, (Ptr{Cvoid}, Cint, Ptr{Float64}, Ptr{Float64}),
                                D.handle, l - 1, y, Vector{Float64}(x))); y)
residual(D::DeviceHierarchy, l::Integer, x, b) = (r = Vector{Float64}(undef, D.nDof[l]);
    amg1d_check(D.handle, ccall((:amg1d_residual, libamg1d), Cint,
                                (Ptr{Cvoid}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                                D.handle, l - 1, r, Vector{Float64}(x), Vector{Float64}(b))); r)
restrict(D::DeviceHierarchy, l::Integer, rf) = (rc = Vector{Float64}(undef, D.nDof[l + 1]);      # L_l' * rf
    amg1d_check(D.handle, ccall((:amg1d_restrict, libamg1d), Cint, (Ptr{Cvoid}, Cint, Ptr{Float64}, Ptr{Float64}),
                                D.handle, l - 1, rc, Vector{Float64}(rf))); rc)
prolong(D::DeviceHierarchy, l::Integer, xc) = (xf = Vector{Float64}(undef, D.nDof[l]);           # L_l * xc
    amg1d_check(D.handle, ccall((:amg1d_prolong, libamg1d), Cint, (Ptr{Cvoid}, Cint, Ptr{Float64}, Ptr{Float64}),
                                D.handle, l - 1, xf, Vector{Float64}(xc))); xf)
direct_solve(D::DeviceHierarchy, l::Integer, b) = (x = Vector{Float64}(undef, D.nDof[l]);        # A_l \ b (BCR)
    amg1d_check(D.handle, ccall((:amg1d_direct_solve, libamg1d), Cint, (Ptr{Cvoid}, Cint, Ptr{Float64}, Ptr{Float64}),
                                D.handle, l - 1, x, Vector{Float64}(b))); x)

set_option!(D::DeviceHierarchy, key::AbstractString, value::Integer) =
    amg1d_check(D.handle, ccall((:amg1d_set_option, libamg1d), Cint, (Ptr{Cvoid}, Cstring, Int64),
                                D.handle, key, value))
get_info(D::DeviceHierarchy, key::AbstractString) =
    ccall((:amg1d_get_info, libamg1d), Int64, (Ptr{Cvoid}, Cstring), D.handle, key)

# ---- drop-in: the reference's own signatures, so that its scripts run unchanged ----------------------------
# tests/*_heirarchy_test.jl call aggmg.multigrid(H, x0, b, 100, 1e-10) with H::MeshHierarchy.  Including this
# file after solvers.jl REPLACES those four methods (same signatures as src/solvers.jl:19-20, :63, :84, :116-117)
# by versions that upload H on first use (cached per hierarchy object) and run on the device.  Delete this
# block to keep the CPU methods next to the DeviceHierarchy ones.
const DEVICE_CACHE = IdDict{MeshHierarchy,DeviceHierarchy}()
device(H::MeshHierarchy) = get!(() -> DeviceHierarchy(H), DEVICE_CACHE, H)

multigrid_v_cycle(H::MeshHierarchy, x0::AbstractVector, b::AbstractVector;
                  nPre::Integer = 3, nPost::Integer = 3, alpha::AbstractFloat = 2.0 / 3.0) =
    multigrid_v_cycle(device(H), x0, b; nPre = nPre, nPost = nPost, alpha = alpha)
multigrid(H::MeshHierarchy, x0::AbstractVector, b::AbstractVector, maxiter::Integer, tol::AbstractFloat) =
    multigrid(device(H), H, x0, b, maxiter, tol)
ldiv!(y::AbstractVector, H::MeshHierarchy, b::AbstractVector) = ldiv!(y, device(H), b)
ldiv!(H::MeshHierarchy, b::AbstractVector) = ldiv!(b, device(H), b)
ldiv!(Y::AbstractMatrix, H::MeshHierarchy, B::AbstractMatrix) = ldiv!(Y, device(H), B)
