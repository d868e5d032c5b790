# UNEXECUTED in this repository's environment (no Julia in the image); kept in sync with INTEGRATION.md section 2.
# lto_b200.jl -- ccall binding of liblto_b200.so (include/lto_b200.h)
module LtoB200
const lib = get(ENV, "LTO_B200_LIB", "liblto_b200.so")

mutable struct DirectParams            # == lto_direct_params (7 doubles, 4 int32)
    MU::Cdouble; DU::Cdouble; TU::Cdouble; Isp::Cdouble; g0::Cdouble; default_mass::Cdouble; tol::Cdouble
    mode::Int32; err_norm::Int32; max_attempts::Int32; kernel::Int32
    DirectParams() = (p = new(); ccall((:lto_direct_params_default, lib), Cvoid, (Ref{DirectParams},), p); p)
end
mutable struct IndirectParams          # == lto_indirect_params (12 doubles, 4 int32)
    MU::Cdouble; DU::Cdouble; TU::Cdouble; thrustLimit::Cdouble; mass::Cdouble; time_direction::Cdouble
    p::Cdouble; rho::Cdouble; Isp::Cdouble; g0::Cdouble; reltol::Cdouble; abstol::Cdouble
    controller::Int32; err_norm::Int32; max_attempts::Int32; kernel::Int32
    IndirectParams() = (p = new(); ccall((:lto_indirect_params_default, lib), Cvoid, (Ref{IndirectParams},), p); p)
end

const handle = Ref{Ptr{Cvoid}}(C_NULL)
function init(devices::Vector{Int32} = Int32[0])
    rc = ccall((:lto_init_devices, lib), Cint, (Cint, Ptr{Int32}, Ref{Ptr{Cvoid}}), length(devices), devices, handle)
    rc == 0 || error("lto_init_devices: ", unsafe_string(ccall((:lto_last_error, lib), Cstring, (Ptr{Cvoid},), C_NULL)))
end
check(rc) = rc == 0 || error("liblto_b200: ", unsafe_string(ccall((:lto_last_error, lib), Cstring, (Ptr{Cvoid},), handle[])))

# ---- pinned (page-locked) result arrays.  The device-to-host copy of the Jacobian / STM blocks is most of a call's bytes; into a
# pinned array it runs asynchronously at the PCIe rate and overlaps the kernels, into an ordinary (pageable) Julia array the driver
# stages it and the pipeline serialises (bench.py `e2e.pageable`).  Blocks are recycled through a small pool (cudaHostAlloc costs
# milliseconds); a finalizer gives the block back when the array is collected.
const _pool = Dict{Int, Vector{Ptr{Cvoid}}}()
const _pool_lock = ReentrantLock()
_size_class(n) = (c = 4096; while c < n; c <<= 1; end; c)
function pinned_array(::Type{T}, dims::Int...) where {T}
    nbytes = sizeof(T) * prod(dims)
    nbytes == 0 && return zeros(T, dims...)
    sz = _size_class(nbytes)
    ptr = lock(_pool_lock) do
        v = get(_pool, sz, nothing)
        (v === nothing || isempty(v)) ? C_NULL : pop!(v)
    end
    if ptr == C_NULL
        ptr = ccall((:lto_host_alloc, lib), Ptr{Cvoid}, (Csize_t,), sz)
        ptr == C_NULL && return zeros(T, dims...)          # pinned memory exhausted: a pageable array is still correct
    end
    a = unsafe_wrap(Array, Ptr{T}(ptr), dims; own = false)
    finalizer(a) do _
        lock(_pool_lock) do
            push!(get!(_pool, sz, Ptr{Cvoid}[]), ptr)
        end
    end
    a                                                       # contents unspecified: every caller below has the library overwrite all of it
end

# ---- direct: replaces defectCalc (multiShoot_CRTBP_direct.jl:66-109)
function defectCalc(X_all::Matrix{Float64}, u_all::Matrix{Float64}, t_TU::Vector{Float64}, nstate, n_nodes, nsteps, Isp, MU, DU, TU)
    p = DirectParams(); p.MU, p.DU, p.TU, p.Isp = MU, DU, TU, Isp
    defect = pinned_array(Float64, nstate, n_nodes - 1); errors = pinned_array(Float64, n_nodes - 1); status = pinned_array(Int32, n_nodes - 1)
    GC.@preserve X_all u_all t_TU defect errors status check(ccall((:lto_direct_defect_traj, lib), Cint,
        (Ptr{Cvoid}, Ref{DirectParams}, Int64, Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
        handle[], p, 1, n_nodes, nstate, nsteps, X_all, u_all, t_TU, defect, errors, status))
    (defect, errors)
end

# ---- direct: replaces jacobianCalc (:111-166); `defect`, `pert` become unused (variational equations)
function jacobianCalc(X_all, u_all, t_TU, nstate, n_nodes, nsteps, Isp, MU, DU, TU)
    p = DirectParams(); p.MU, p.DU, p.TU, p.Isp = MU, DU, TU, Isp
    nvar = 2 * (nstate + 3)
    defect = pinned_array(Float64, nstate, n_nodes - 1); errors = pinned_array(Float64, n_nodes - 1); status = pinned_array(Int32, n_nodes - 1)
    blocks = pinned_array(Float64, nstate, nvar, n_nodes - 1)              # block i == Jac_temp[(i-1)n+1 : i n, :]  (:139-140)
    GC.@preserve X_all u_all t_TU defect errors status blocks check(ccall((:lto_direct_defect_jac_traj, lib), Cint,
        (Ptr{Cvoid}, Ref{DirectParams}, Int64, Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Float64}),
        handle[], p, 1, n_nodes, nstate, nsteps, X_all, u_all, t_TU, defect, errors, status, blocks))
    Jac_full = zeros(nstate * (n_nodes - 1), n_nodes * (nstate + 3))                      # :146
    for i = 1:(n_nodes - 1)                                                               # :147-162, unchanged
        rows = ((i - 1) * nstate + 1):(i * nstate)
        Jac_full[rows, ((i - 1) * nstate + 1):((i + 1) * nstate)] = blocks[:, 1:(2 * nstate), i]
        c0 = nstate * n_nodes + 3 * (i - 1)
        Jac_full[rows, (c0 + 1):(c0 + 6)] = blocks[:, (2 * nstate + 1):end, i]
    end
    Jac_full
end

# ---- indirect: replaces defectCalc (multiShoot_CRTBP_indirect.jl:63-90) and jacobianCalc (:93-146)
function iparams(params)
    (MU, DU, TU, thrustLimit, mass, td, pp, rho) = params                                 # :260
    p = IndirectParams(); p.MU, p.DU, p.TU = MU, DU, TU
    p.thrustLimit, p.mass, p.time_direction, p.p, p.rho = thrustLimit, mass, td, pp, rho
    p
end
function defectCalc_indirect(XC_all::Matrix{Float64}, t_TU::Vector{Float64}, nstate, n_nodes, params)
    m = 2 * nstate; defect = pinned_array(Float64, m, n_nodes - 1); status = pinned_array(Int32, n_nodes - 1)
    GC.@preserve XC_all t_TU defect status check(ccall((:lto_indirect_defect_traj, lib), Cint,
        (Ptr{Cvoid}, Ref{IndirectParams}, Int64, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}),
        handle[], iparams(params), 1, n_nodes, m, XC_all, t_TU, C_NULL, C_NULL, defect, status, C_NULL))
    (defect, zeros(n_nodes - 1))                                                          # errors == 0 (:85)
end
function jacobianCalc_indirect(XC_all, t_TU, nstate, n_nodes, params)
    m = 2 * nstate; defect = pinned_array(Float64, m, n_nodes - 1); status = pinned_array(Int32, n_nodes - 1); phi = pinned_array(Float64, m, m, n_nodes - 1)
    GC.@preserve XC_all t_TU defect status phi check(ccall((:lto_indirect_defect_jac_traj, lib), Cint,
        (Ptr{Cvoid}, Ref{IndirectParams}, Int64, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}, Ptr{Float64}),
        handle[], iparams(params), 1, n_nodes, m, XC_all, t_TU, C_NULL, C_NULL, defect, status, C_NULL, phi))
    Jac_full = zeros(m * (n_nodes - 1), n_nodes * m)                                      # :127
    for i = 1:(n_nodes - 1)                                                               # :128-138
        r = ((i - 1) * m + 1):(i * m)
        Jac_full[r, ((i - 1) * m + 1):(i * m)] = phi[:, :, i]
        for k = 1:m; Jac_full[r[k], i * m + k] = -1.0; end                                # hcat(Phi_i, -I) without LinearAlgebra's `I`
    end
    Jac_full[:, 1:nstate] .= 0.0; Jac_full[:, (end - 2 * nstate + 1):(end - nstate)] .= 0.0   # :141-142
    Jac_full
end
# ---- densify (HelperFunctions.jl:51-101): every dense time is its own propagation (node i, t_TU[i]) -> t, all of them in ONE call
# (pairs form of lto_indirect_defect, x_target = NULL returns x(t1)); the reference evaluates Vern8's dense-output interpolant instead.
function densify(XC_all::Matrix{Float64}, t_TU::Vector{Float64}, params, n_desired)
    m = size(XC_all, 1); N = size(XC_all, 2)
    t_dense = collect(LinRange(t_TU[1], t_TU[end], n_desired))
    seg = [searchsortedlast(t_TU, t) for t in t_dense]
    keep = seg .<= N - 1                                                                  # t < t_TU[end] (:64)
    seg = vcat(seg[keep], N - 1); t1 = vcat(t_dense[keep], t_TU[end])                     # + the last segment's end state (:94-97)
    x0 = XC_all[:, seg]; t0 = t_TU[seg]; n = length(seg)
    xend = pinned_array(Float64, m, n); status = pinned_array(Int32, n)
    GC.@preserve x0 t0 t1 xend status check(ccall((:lto_indirect_defect, lib), Cint,
        (Ptr{Cvoid}, Ref{IndirectParams}, Int64, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}),
        handle[], iparams(params), n, m, x0, t0, t1, C_NULL, C_NULL, C_NULL, xend, status, C_NULL))
    (xend, t_dense)
end

# ---- indirect: the linear step of optimizeTraj_OLS (multiShoot_CRTBP_indirect.jl:181-182, :207) on the device.
# `phi` is what jacobianCalc_blocks returns (m x m x (n_nodes-1)); Jac_full is never formed.  m = 12, or 14 for the system with mass
# ([r v m | lr lv lm]; end pins r, v, m first / r, v, lm last, see lto_b200.h): the dimension is taken from the arrays.
function jacobianCalc_blocks(XC_all, t_TU, nstate, n_nodes, params)
    m = 2 * nstate; defect = pinned_array(Float64, m, n_nodes - 1); status = pinned_array(Int32, n_nodes - 1); phi = pinned_array(Float64, m, m, n_nodes - 1)
    GC.@preserve XC_all t_TU defect status phi check(ccall((:lto_indirect_defect_jac_traj, lib), Cint,
        (Ptr{Cvoid}, Ref{IndirectParams}, Int64, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}, Ptr{Float64}),
        handle[], iparams(params), 1, n_nodes, m, XC_all, t_TU, C_NULL, C_NULL, defect, status, C_NULL, phi))
    phi
end
function newtonUpdate(phi::Array{Float64,3}, defect::Matrix{Float64}, n_nodes, flag_adjointsOnly::Bool)
    m = size(phi, 1)
    (size(phi) == (m, m, n_nodes - 1) && size(defect) == (m, n_nodes - 1)) || throw(ArgumentError("phi must be m x m x (n_nodes-1), defect m x (n_nodes-1)"))
    xc_update = zeros(m, n_nodes); status = zeros(Int32, 1)               # == reshape(xc_update2, 2*nstate, n_nodes) (:185)
    GC.@preserve phi defect xc_update status check(ccall((:lto_indirect_newton_nd, lib), Cint,
        (Ptr{Cvoid}, Cint, Int64, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
        handle[], m, 1, n_nodes, flag_adjointsOnly ? 1 : 0, phi, defect, xc_update, status))
    xc_update
end

# ---- indirect: multiShoot_CRTBP_indirect (:58-345) for a BATCH of trajectories, iterated on the device.
# XC_batch: m x n_nodes x n_traj (m = 12, or 14 with mass: Isp enters its mass flow), t_batch: n_nodes x n_traj; thrustLimit / rho:
# per-trajectory vectors (continuation ladders).
function multiShoot_CRTBP_indirect_batch(XC_batch::Array{Float64,3}, t_batch::Matrix{Float64}, MU, DU, TU, mass0, thrustLimit::Vector{Float64},
                                         flag_adjointsOnly::Bool, maxIter, p, rho::Vector{Float64}; Isp = 2000.0)
    m = size(XC_batch, 1); n_nodes = size(XC_batch, 2); n_traj = size(XC_batch, 3)
    XC = copy(XC_batch); defect = zeros(m, n_nodes - 1, n_traj)
    status_flag = zeros(Int32, n_traj); iters = zeros(Int32, n_traj); er = zeros(n_traj)
    prm = iparams((MU, DU, TU, thrustLimit[1], mass0, 1.0, p, rho[1])); prm.Isp = Isp
    GC.@preserve XC t_batch thrustLimit rho defect status_flag iters er check(ccall((:lto_indirect_solve_batch_nd, lib), Cint,
        (Ptr{Cvoid}, Ref{IndirectParams}, Cint, Int64, Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Ptr{Int32}, Ptr{Float64}),
        handle[], prm, m, n_traj, n_nodes, maxIter, flag_adjointsOnly ? 1 : 0, XC, t_batch, thrustLimit, rho, defect, status_flag, iters, er))
    (XC, defect, status_flag)
end
# ---- indirect: reduceFuel_indirect (HelperFunctions.jl:105-193) for a BATCH of rho ladders in ONE call; the ladder logic runs on the device.
# XC_batch: m x n_nodes x n_traj starts (m = 12, or 14 with mass), t_batch: n_nodes x n_traj; thrustLimit, rho_current, rho_target: per-trajectory
# vectors; backoff: 100 x n_traj draws in [0, 1) for the back-off rho *= 3(1 + rand()) (:182), consumed in order (rand(rng, 100) per trajectory).
# maxIter is per solver call (the reference uses 10).  status: the last call's status_flag, or 3 when a ladder gave up after 100 rungs.
function reduceFuel_indirect_batch(XC_batch::Array{Float64,3}, t_batch::Matrix{Float64}, MU, DU, TU, mass, thrustLimit::Vector{Float64},
                                   rho_current::Vector{Float64}, rho_target::Vector{Float64}, backoff::Matrix{Float64}; maxIter = 10, Isp = 2000.0)
    m = size(XC_batch, 1); n_nodes = size(XC_batch, 2); n_traj = size(XC_batch, 3)
    XC = copy(XC_batch); defect = zeros(m, n_nodes - 1, n_traj); status = zeros(Int32, n_traj)
    calls = zeros(Int32, n_traj); newton_iters = zeros(Int32, n_traj); rho_last = zeros(n_traj)
    prm = iparams((MU, DU, TU, thrustLimit[1], mass, 1.0, 1.0, 1.0)); prm.Isp = Isp
    GC.@preserve XC t_batch thrustLimit rho_current rho_target backoff defect status calls newton_iters rho_last check(ccall((:lto_indirect_reduce_fuel_batch, lib), Cint,
        (Ptr{Cvoid}, Ref{IndirectParams}, Cint, Int64, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ptr{Float64}),
        handle[], prm, m, n_traj, n_nodes, maxIter, XC, t_batch, thrustLimit, rho_current, rho_target, backoff, defect, status, calls, newton_iters, rho_last))
    (XC, defect, status, calls)
end
# ---- direct: multiShoot_CRTBP_direct (:465-594) for a BATCH of trajectories, iterated on the device (flagEnd = false, allowImpulsive = false).
# X_batch: nstate x n_nodes x n_traj, u_batch: 3 x n_nodes x n_traj, t_batch: n_nodes x n_traj, state_0 / state_f: 6 x n_traj (interpEndStates, :483)
function multiShoot_CRTBP_direct_batch(X_batch::Array{Float64,3}, u_batch::Array{Float64,3}, t_batch::Matrix{Float64}, state_0::Matrix{Float64},
                                       state_f::Matrix{Float64}, MU, DU, TU, nsteps, mass, Isp, maxIter)
    nstate = size(X_batch, 1); n_nodes = size(X_batch, 2); n_traj = size(X_batch, 3)
    p = DirectParams(); p.MU, p.DU, p.TU, p.Isp = MU, DU, TU, Isp
    X = copy(X_batch); u = copy(u_batch); defect = zeros(nstate, n_nodes - 1, n_traj); iters = zeros(Int32, n_traj); er = zeros(n_traj)
    GC.@preserve X u t_batch state_0 state_f defect iters er check(ccall((:lto_direct_solve_batch, lib), Cint,
        (Ptr{Cvoid}, Ref{DirectParams}, Int64, Cint, Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Cdouble,
         Ptr{Float64}, Ptr{Int32}, Ptr{Float64}),
        handle[], p, n_traj, n_nodes, nstate, nsteps, maxIter, X, u, t_batch, state_0, state_f, mass, defect, iters, er))
    (X, u, defect, iters)
end
# ---- trajectory stacking (CRTBP_Multishoot_direct_demo.jl:117-157) for a BATCH of transfers in ONE call: splines, both ballistic arcs and
# both find_τ scans on the device.  X0_states / Xf_states: the 6 x n orbit tables; tau1, t_split: per transfer; t_batch: n_nodes x n_traj.
# Returns (XC 12 x n_nodes x n_traj, tau2, state_0 6 x n_traj, state_f 6 x n_traj, status); XC[1:6, :, :], state_0 and state_f feed
# multiShoot_CRTBP_direct_batch below.  Like the rest of this shim, not run under Julia here (the same ABI is exercised from Python).
function trajectory_stack_guess_batch(X0_states::Matrix{Float64}, Xf_states::Matrix{Float64}, tau1::Vector{Float64}, t_batch::Matrix{Float64},
                                      t_split::Vector{Float64}, MU, DU, TU)
    n_nodes = size(t_batch, 1); n_traj = size(t_batch, 2)
    XC = zeros(12, n_nodes, n_traj); tau2 = zeros(n_traj); state_0 = zeros(6, n_traj); state_f = zeros(6, n_traj); status = zeros(Int32, n_traj)
    prm = iparams((MU, DU, TU, 0.0, 1e3, 1.0, 1.0, 1.0))
    GC.@preserve X0_states Xf_states tau1 t_batch t_split XC tau2 state_0 state_f status check(ccall((:lto_stack_guess_batch, lib), Cint,
        (Ptr{Cvoid}, Ref{IndirectParams}, Int64, Cint, Ptr{Float64}, Cint, Ptr{Float64}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
        handle[], prm, n_traj, n_nodes, X0_states, size(X0_states, 2), Xf_states, size(Xf_states, 2), tau1, t_batch, t_split,
        XC, tau2, state_0, state_f, status))
    (XC, tau2, state_0, state_f, status)
end
# ---- control cost of 12-dim indirect trajectories in ONE call (lto_indirect_cost_batch): the defect-only kernel's steps with the quadratures
# of |a_u| and |a_u|^2 on them.  XC_batch: 12 x n_nodes x n_traj; t_batch: n_nodes x n_traj; thrustLimit, rho: per trajectory.
# Returns (dv in m/s, energy in N^2 TU, status).  Like the rest of this shim, not run under Julia here (the same ABI is exercised from Python).
function indirect_cost_batch(XC_batch::Array{Float64,3}, t_batch::Matrix{Float64}, MU, DU, TU, mass, thrustLimit::Vector{Float64}, p,
                             rho::Vector{Float64})
    n_nodes = size(XC_batch, 2); n_traj = size(XC_batch, 3)
    size(XC_batch, 1) == 12 || error("indirect_cost_batch: XC_batch must have 12 rows (the 14-dim cost is exact from the node masses)")
    dv = zeros(n_traj); energy = zeros(n_traj); status = zeros(Int32, n_traj)
    prm = iparams((MU, DU, TU, thrustLimit[1], mass, 1.0, p, rho[1]))
    GC.@preserve XC_batch t_batch thrustLimit rho dv energy status check(ccall((:lto_indirect_cost_batch, lib), Cint,
        (Ptr{Cvoid}, Ref{IndirectParams}, Int64, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Ptr{Int32}),
        handle[], prm, n_traj, n_nodes, XC_batch, t_batch, thrustLimit, rho, dv, energy, C_NULL, status))
    (dv, energy, status)
end
# ---- costates of nstate-6 direct solutions in ONE call (lto_direct_costates_batch): the direct QP's multipliers at (X, u), mapped to the
# node costates of the 12-dim p = 2 system.  X_batch 6 x n_nodes x n_traj, u_batch 3 x n_nodes x n_traj, t_batch n_nodes x n_traj,
# state_0 / state_f 6 x n_traj.  Returns (XC 12 x n_nodes x n_traj: X bitwise and the costates, multipliers 6 x (n_nodes-1) x n_traj,
# du_max in N, status); XC with the end states pinned is a start for multiShoot_CRTBP_indirect at p = 2.  Like the rest of this shim, not run
# under Julia here (the same ABI is exercised from Python).
function direct_costates_batch(X_batch::Array{Float64,3}, u_batch::Array{Float64,3}, t_batch::Matrix{Float64}, state_0::Matrix{Float64},
                               state_f::Matrix{Float64}, MU, DU, TU; nsteps=10)
    size(X_batch, 1) == 6 || error("direct_costates_batch: X_batch must have 6 rows (nstate 7 has no costate map)")
    n_nodes = size(X_batch, 2); n_traj = size(X_batch, 3)
    p = DirectParams(); p.MU, p.DU, p.TU = MU, DU, TU
    XC = zeros(12, n_nodes, n_traj); mult = zeros(6, n_nodes - 1, n_traj); du = zeros(n_traj); status = zeros(Int32, n_traj)
    GC.@preserve X_batch u_batch t_batch state_0 state_f XC mult du status check(ccall((:lto_direct_costates_batch, lib), Cint,
        (Ptr{Cvoid}, Ref{DirectParams}, Int64, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
        handle[], p, n_traj, n_nodes, nsteps, X_batch, u_batch, t_batch, state_0, state_f, XC, mult, du, status))
    (XC, mult, du, status)
end
# ---- switch times of 12-dim p = 1 indirect trajectories in ONE call (lto_indirect_switch_batch): the sign changes of |lv| - 1 (thrust on
# where > 0) located on the defect-only kernel's steps, with the node rule between segments.  XC_batch: 12 x n_nodes x n_traj; t_batch:
# n_nodes x n_traj; thrustLimit, rho: per trajectory.  Returns (t_switch max_switch x n_traj in TU (NaN unused), direction (+1 a burn starts,
# -1 it ends, 0 unused), n_switch (the true count, -1 where status is not OK), on_start, status).  Like the rest of this shim, not run under
# Julia here (the same ABI is exercised from Python).
function indirect_switch_batch(XC_batch::Array{Float64,3}, t_batch::Matrix{Float64}, MU, DU, TU, mass, thrustLimit::Vector{Float64},
                               rho::Vector{Float64}; max_switch=16)
    n_nodes = size(XC_batch, 2); n_traj = size(XC_batch, 3)
    size(XC_batch, 1) == 12 || error("indirect_switch_batch: XC_batch must have 12 rows")
    t_sw = zeros(max_switch, n_traj); dir = zeros(Int32, max_switch, n_traj)
    n_sw = zeros(Int32, n_traj); on = zeros(Int32, n_traj); status = zeros(Int32, n_traj)
    prm = iparams((MU, DU, TU, thrustLimit[1], mass, 1.0, 1.0, rho[1]))
    GC.@preserve XC_batch t_batch thrustLimit rho t_sw dir n_sw on status check(ccall((:lto_indirect_switch_batch, lib), Cint,
        (Ptr{Cvoid}, Ref{IndirectParams}, Int64, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Cint, Ptr{Float64}, Ptr{Int32},
         Ptr{Int32}, Ptr{Int32}, Ptr{Float64}, Ptr{Int32}),
        handle[], prm, n_traj, n_nodes, XC_batch, t_batch, thrustLimit, rho, max_switch, t_sw, dir, n_sw, on, C_NULL, status))
    (t_sw, dir, n_sw, on, status)
end
end # module
