"""Host-side mirror of the reference's two outer solvers, for running BASELINE configs 1-2
(the demo scripts) end to end without Julia / Ipopt / SuiteSparse.

    multiShoot_CRTBP_direct      src/multiShoot_CRTBP_direct.jl:58-594   (+ multiShoot_CRTBP_direct_batch: many trajectories, QP on the device)
    multiShoot_CRTBP_indirect    src/multiShoot_CRTBP_indirect.jl:58-345
    reduceFuel_indirect          src/HelperFunctions.jl:105-193   (+ reduceFuel_indirect_batch: many trajectories, one device call per round)
    trajectory_stack_guess       CRTBP_Multishoot_direct_demo.jl:117-157   (+ trajectory_stack_guess_batch: many transfers in one device call,
                                                                        direct_transfer_sweep: those guesses solved by the batched direct solver)
    indirect_transfer_sweep      CRTBP_Multishoot_indirect_demo.jl:166-281 over a direct_transfer_sweep, batched, with each result's
                                 transfer_cost_indirect (delta-v and control energy; no reference counterpart)
    thrust_arcs_indirect         the burns of p = 1 indirect solutions (switch times of |lv| - 1; no reference counterpart on the
                                 shooting path)
    densify, jacobiConstant, interpInitialStates, find_tau   src/HelperFunctions.jl:10-101

Same names, argument order and return values.  Arrays use the reference's shapes
(nstate x n_nodes etc.).  What stays on the host is only the small dense linear algebra of
the update step; EVERY propagation goes through a `backend` -- by default `GpuBackend`
(liblto_b200.so on the B200; there is no CPU propagation in this package).  The line
searches and the two t_f-perturbed defect evaluations are issued as ONE batched call
each (n_traj = 20 / 10 / 2) instead of the reference's sequential loops.

Deliberate, documented substitutions for third-party solvers that are not part of the hot path:
  * direct QP (JuMP + Ipopt, :264-386): with flagEnd = false (what the demo runs) every bound
    collapses to an equality, the problem is an equality-constrained convex QP and is solved
    exactly through its KKT system.  flagEnd = true needs bound constraints -> NotImplementedError.
  * indirect step (`-sparse(J) \\ defect`, SuiteSparseQR, :181-182): dense least squares; the
    system has full column rank once the structurally empty columns are dropped (SURVEY App. B).
"""
import numpy as np

from . import capi
from .capi import DAY
from .synthetic import interp_initial_states, load_orbit


# --------------------------------------------------------------------------- backends
class GpuBackend:
    """All propagation on the GPU through the C ABI (lowthrustopt_b200.capi.Handle)."""

    def __init__(self, handle=None, device=0):
        self.h = handle or capi.Handle(device)
        self.calls = 0

    # direct: X (B, N, n), U (B, N, 3), t (B, N)
    def direct_defect(self, X, U, t, nsteps, Isp, MU, DU, TU):
        self.calls += 1
        r = self.h.direct_traj(X, U, t, nsteps=nsteps, params=capi.direct_params(Isp=Isp, MU_=MU, DU_=DU, TU_=TU), jac=False)
        B, N, n = X.shape
        return r["defect"].reshape(B, N - 1, n), r["errors"].reshape(B, N - 1)

    def direct_blocks(self, X, U, t, nsteps, Isp, MU, DU, TU):
        self.calls += 1
        r = self.h.direct_traj(X, U, t, nsteps=nsteps, params=capi.direct_params(Isp=Isp, MU_=MU, DU_=DU, TU_=TU), jac=True)
        B, N, n = X.shape
        return r["defect"].reshape(B, N - 1, n), r["errors"].reshape(B, N - 1), r["jac"].reshape(B, N - 1, 2 * (n + 3), n).transpose(0, 1, 3, 2)

    # indirect: XC (B, N, m), t (B, N); params = the reference's tuple
    def _ip(self, params, **kw):
        MU, DU, TU, thrustLimit, mass, td, p, rho = params[:8]
        if len(params) > 8:                                                # 14-dim extension: the tuple carries Isp as a ninth entry
            kw.setdefault("Isp", params[8])
        if not (p == 0 or p >= 1):
            raise ValueError("Invalid value of p!")                       # CRTBP_stateCostate_deriv.jl:52
        return capi.indirect_params(thrustLimit=thrustLimit, mass=mass, time_direction=td, p=p, rho=rho, MU_=MU, DU_=DU, TU_=TU, **kw)

    def indirect_defect(self, XC, t, params):
        self.calls += 1
        r = self.h.indirect_traj(XC, t, params=self._ip(params), jac=False)
        B, N, m = XC.shape
        return r["defect"].reshape(B, N - 1, m)

    def indirect_blocks(self, XC, t, params):
        self.calls += 1
        r = self.h.indirect_traj(XC, t, params=self._ip(params), jac=True)
        B, N, m = XC.shape
        return r["defect"].reshape(B, N - 1, m), r["phi"].reshape(B, N - 1, m, m).transpose(0, 1, 3, 2)

    def propagate(self, x0, t0, t1, params):
        """x(t1) for independent rows x0 (B, m): solve(ODEProblem(odefun, x0, (t0, t1), params), Vern8(), 1e-13)[:, end]."""
        self.calls += 1
        return self.h.indirect(x0, t0, t1, params=self._ip(params), jac=False)["defect"]

    def direct_qp(self, blocks_cm, defect, u_all, t, b0, bf):
        """optimizeTraj's QP on the device (lto_direct_qp): blocks_cm (B, N-1, 2(n+3), n) column-major Jacobian blocks."""
        self.calls += 1
        return self.h.direct_qp(blocks_cm, defect, u_all, t, b0, bf)

    def indirect_newton(self, phi, defect, flag_adjointsOnly):
        """-sparse(Jac_full) \\ defect_vec on the device (lto_indirect_newton); phi (B, N-1, m, m) [.., row, col] -> (B, N, m)."""
        self.calls += 1
        upd, status = self.h.indirect_newton(np.ascontiguousarray(phi.transpose(0, 1, 3, 2)), defect, flag_adjointsOnly)
        return upd

    def indirect_solve_batch(self, XC, t, params, thrustLimit=None, rho=None, max_iter=50, flag_adjointsOnly=False):
        self.calls += 1
        return self.h.indirect_solve_batch(XC, t, params=self._ip(params), thrustLimit=thrustLimit, rho=rho, max_iter=max_iter,
                                           flag_adjointsOnly=flag_adjointsOnly)

    def indirect_reduce_fuel_batch(self, XC, t, params, rho_current, rho_target, backoff_uniform, thrustLimit=None, max_iter=10):
        self.calls += 1
        return self.h.indirect_reduce_fuel_batch(XC, t, rho_current, rho_target, backoff_uniform, params=self._ip(params),
                                                 thrustLimit=thrustLimit, max_iter=max_iter)

    def stack_guess_batch(self, X0_states, Xf_states, tau1, t_TU, t_split, params):
        """trajectory_stack_guess for many transfers in one device call (lto_stack_guess_batch); params = the reference's tuple."""
        self.calls += 1
        return self.h.stack_guess_batch(X0_states, Xf_states, tau1, t_TU, t_split, params=self._ip(params))

    def indirect_cost(self, XC, t, params, thrustLimit=None, rho=None, defect=False):
        """delta-v and control energy of 12-dim trajectories XC (B, N, 12) in one device call (lto_indirect_cost_batch)."""
        self.calls += 1
        return self.h.indirect_cost_batch(XC, t, params=self._ip(params), thrustLimit=thrustLimit, rho=rho, defect=defect)

    def indirect_switches(self, XC, t, params, thrustLimit=None, rho=None, max_switch=16, defect=False):
        """Switch times of p = 1 12-dim trajectories XC (B, N, 12) in one device call (lto_indirect_switch_batch)."""
        self.calls += 1
        return self.h.indirect_switch_batch(XC, t, params=self._ip(params), thrustLimit=thrustLimit, rho=rho, max_switch=max_switch,
                                            defect=defect)

    def direct_solve_batch(self, X, U, t, state_0, state_f, mass, nsteps, max_iter, Isp, MU, DU, TU):
        self.calls += 1
        return self.h.direct_solve_batch(X, U, t, state_0, state_f, mass=mass, nsteps=nsteps, max_iter=max_iter,
                                         params=capi.direct_params(Isp=Isp, MU_=MU, DU_=DU, TU_=TU))

    def direct_costates(self, X, U, t, state_0, state_f, nsteps, Isp, MU, DU, TU):
        """Costates of nstate-6 direct solutions X (B, N, 6), U (B, N, 3) in one device call (lto_direct_costates_batch)."""
        self.calls += 1
        return self.h.direct_costates_batch(X, U, t, state_0, state_f, nsteps=nsteps, params=capi.direct_params(Isp=Isp, MU_=MU, DU_=DU, TU_=TU))


_default_backend = None


def default_backend():
    global _default_backend
    if _default_backend is None:
        _default_backend = GpuBackend()
    return _default_backend


# --------------------------------------------------------------------------- endpoint helpers
def _orbit_states(X_states):
    """Accept the reference's 6 x 100 table (X0_states) and return a tau -> state(6) function:
    interpolating natural cubic spline on LinRange(0, 1, 100), tau wrapped to [0, 1]
    (HelperFunctions.jl:18-35, multiShoot_CRTBP_direct.jl:434-461)."""
    from scipy.interpolate import CubicSpline
    X_states = np.asarray(X_states, dtype=np.float64)
    sp = CubicSpline(np.linspace(0.0, 1.0, X_states.shape[1]), X_states.T, bc_type="natural")

    def wrap(tau):
        tau = float(tau)
        while tau > 1:
            tau -= 1
        while tau < 0:
            tau += 1
        return tau
    return lambda tau: sp(wrap(tau))


def interpInitialStates(p1, X0_times, X0_states, MU=None):
    return _orbit_states(X0_states)(p1)


def interpEndStates(tau1, tau2, X0_times, X0_states, Xf_times, Xf_states, MU=None):
    return _orbit_states(X0_states)(tau1), _orbit_states(Xf_states)(tau2)


def find_tau(X_times, X_states, state, MU=None):
    """find_τ (HelperFunctions.jl:38-48): the first of 1001 uniform tau with the smallest distance."""
    f = _orbit_states(X_states)
    tau_trial = np.linspace(0.0, 1.0, 1001)
    d = np.array([np.linalg.norm(f(tt) - state) for tt in tau_trial])
    return float(tau_trial[np.argmin(d)])


def jacobiConstant(state, MU, DU=None):
    """Jacobi constant of every column of `state` (6 x K) -- HelperFunctions.jl:10-15."""
    state = np.asarray(state, dtype=np.float64).reshape(6, -1)
    r1 = np.sqrt((state[0] + MU) ** 2 + state[1] ** 2 + state[2] ** 2)
    r2 = np.sqrt((state[0] + MU - 1) ** 2 + state[1] ** 2 + state[2] ** 2)
    v2 = np.sum(state[3:6] ** 2, axis=0)
    return state[0] ** 2 + state[1] ** 2 + 2 * (1 - MU) / r1 + 2 * MU / r2 - v2


def densify(XC_all, t_TU, params, n_desired, backend=None):
    """densify (HelperFunctions.jl:51-101): the trajectory on LinRange(t_TU[1], t_TU[end], n_desired).  Every dense time t with
    t_TU[i] <= t < t_TU[i+1] takes its column from segment i's solution (:64-75); after the last segment its end state -- the
    propagated one, not the node -- is appended (:94-97).  Returns (XC_dense, t_dense) like the reference.

    The reference evaluates each segment's Vern8 dense-output interpolant; here every dense point is its own segment
    propagation (node i, t_TU[i]) -> t at the solver tolerance, all n_desired of them in ONE batched call of the propagation path."""
    be = backend or default_backend()
    XC_all = np.asarray(XC_all, dtype=np.float64); t_TU = np.asarray(t_TU, dtype=np.float64)
    N = XC_all.shape[1]
    t_dense = np.linspace(t_TU[0], t_TU[-1], int(n_desired))
    seg = np.searchsorted(t_TU, t_dense, side="right") - 1
    keep = (seg >= 0) & (seg <= N - 2)                                    # t < t_TU[end]; the end point is added below
    seg = np.append(seg[keep], N - 2)
    t1 = np.append(t_dense[keep], t_TU[-1])
    x = be.propagate(np.ascontiguousarray(XC_all[:, seg].T), np.ascontiguousarray(t_TU[seg]), t1, params)
    return np.ascontiguousarray(x.T), t_dense


def controlLaw_cart(lambda_v, thrustLimit, p, rho, mass, DU=capi.DU, TU=capi.TU):
    """Control [N] from the primer vector (multiShoot_CRTBP_indirect.jl:389-440); post-processing only."""
    n = np.linalg.norm(lambda_v)
    aL = thrustLimit / mass / 1e3 * TU ** 2 / DU
    if p == 0:
        umag = aL
    elif p == 1:
        umag = 0.5 * (1 + np.tanh((n - 1) / (2 * rho))) * aL
    elif p > 1:
        umag = min((n / p) ** (1 / (p - 1)), aL)
    else:
        raise ValueError("Invalid value of p!")
    if not n > 0 or np.isnan(umag):
        return np.zeros(3)
    return -umag * np.asarray(lambda_v) / n * mass * DU * 1e3 / TU ** 2


def trajectory_stack_guess(X0_states, Xf_states, MU=capi.MU, DU=capi.DU, TU=capi.TU, n_nodes=30, tof1_days=10.0, tof2_days=10.0,
                           tau1=0.75, backend=None):
    """The demos' trajectory-stacking initial guess (CRTBP_Multishoot_direct_demo.jl:117-157): two ballistic
    arcs (thrustLimit = 0), the second starting at the point of the final orbit closest to the end of the
    first.  The reference samples two dense-output solutions; here every node is its own propagation
    from the arc's start (one batched call per arc), which agrees to the integration tolerance.
    Returns (XC_trajectoryStack 12 x n_nodes, t_TU, tau1, tau2, state_0, state_f)."""
    be = backend or default_backend()
    tof1 = tof1_days * DAY / TU; tof2 = tof2_days * DAY / TU; tof = tof1 + tof2
    t_TU = np.linspace(0.0, tof, n_nodes)
    t1 = t_TU[t_TU < tof1]; t2 = t_TU[t_TU >= tof1]
    params = (MU, DU, TU, 0.0, 1e3, 1.0, 1.0, 1.0)
    state_0 = np.concatenate([_orbit_states(X0_states)(tau1), np.zeros(6)])
    ends = np.concatenate([t1, [tof1]])
    arc1 = be.propagate(np.tile(state_0, (ends.size, 1)), np.zeros(ends.size), ends, params)
    tau2_0 = find_tau(None, Xf_states, arc1[-1, :6])
    state_f0 = np.concatenate([_orbit_states(Xf_states)(tau2_0), np.zeros(6)])
    ends2 = np.concatenate([t2, [tof1 + tof2]])
    arc2 = be.propagate(np.tile(state_f0, (ends2.size, 1)), np.full(ends2.size, tof1), ends2, params)
    tau2 = find_tau(None, Xf_states, arc2[-1, :6])
    state_f = np.concatenate([_orbit_states(Xf_states)(tau2), np.zeros(6)])
    XC = np.vstack([arc1[:-1], arc2[:-1]]).T.copy()
    XC[:, 0] = state_0
    XC[:, -1] = state_f
    return XC, t_TU, tau1, tau2, state_0, state_f


def trajectory_stack_guess_batch(X0_states, Xf_states, MU=capi.MU, DU=capi.DU, TU=capi.TU, n_nodes=30, tof1_days=10.0, tof2_days=10.0,
                                 tau1=0.75, backend=None):
    """trajectory_stack_guess for a BATCH of transfers in one device call (lto_stack_guess_batch): the spline lookups, both ballistic
    arcs and both find_tau scans of every transfer run on the device.  tau1, tof1_days, tof2_days: scalars or (T,) arrays; per row the
    same arithmetic as trajectory_stack_guess (t_TU = linspace(0, tof1 + tof2, n_nodes), the arcs split at tof1).
    Returns (XC (T, 12, n_nodes), t_TU (T, n_nodes), tau1 (T,), tau2 (T,), state_0 (T, 12), state_f (T, 12))."""
    be = backend or default_backend()
    tau1, tof1_days, tof2_days = np.broadcast_arrays(*[np.atleast_1d(np.asarray(a, dtype=np.float64)) for a in (tau1, tof1_days, tof2_days)])
    if tau1.ndim != 1:
        raise ValueError("tau1, tof1_days and tof2_days must be scalars or (T,) arrays")
    T = tau1.shape[0]
    t_TU = np.empty((T, n_nodes)); t_split = np.empty(T)
    for j in range(T):
        tof1 = float(tof1_days[j]) * DAY / TU; tof2 = float(tof2_days[j]) * DAY / TU
        t_TU[j] = np.linspace(0.0, tof1 + tof2, n_nodes)
        t_split[j] = tof1
    tau1 = np.ascontiguousarray(tau1)
    r = be.stack_guess_batch(X0_states, Xf_states, tau1, t_TU, t_split, (MU, DU, TU, 0.0, 1e3, 1.0, 1.0, 1.0))
    z = np.zeros((T, 6))
    return (r["XC_all"].transpose(0, 2, 1).copy(), t_TU, tau1.copy(), r["tau2"], np.concatenate([r["state_0"], z], axis=1),
            np.concatenate([r["state_f"], z], axis=1))


def _quad_cost(u_all, t_TU):
    """quadCost of optimizeTraj (multiShoot_CRTBP_direct.jl:367-368, dV = 0) at the controls u_all (T, 3, N): the node weights dt_temp
    of _qp_direct (:323-325) on the solver's fixed time grid."""
    t0 = t_TU[:, :1]; tf = t_TU[:, -1:]
    tau = (t_TU - t0) / (tf - t0) * 2 - 1
    t_fixed = t0 + (tau + 1) / 2 * (tf - t0)
    dt = np.diff(t_fixed, axis=1)
    z = np.zeros((t_TU.shape[0], 1))
    w = np.concatenate([dt / 2, dt[:, -1:] / 2], axis=1) + np.concatenate([z, dt[:, :-1] / 2, z], axis=1)
    return np.sum(u_all ** 2 * w[:, None, :], axis=(1, 2))


def direct_transfer_sweep(X0_states, Xf_states, tau1, tof1_days, tof2_days, n_nodes=30, nsteps=10, nstate=6, mass=1e3, Isp=2000.0,
                          maxIter=100, backend=None):
    """A trade study over departure phase and flight times: the trajectory-stacking guesses of every (tau1, tof1_days, tof2_days) row
    (trajectory_stack_guess_batch), then multiShoot_CRTBP_direct on all of them at once on the device (lto_direct_solve_batch; the demo's
    setting: flagEnd = false, allowImpulsive = false, u_all = 0 to start, nstate 7 adds a mass row of `mass`).  Two library calls.
    Returns dict(X_all (T, nstate, N), u_all (T, 3, N), t_TU (T, N), tau2 (T,), iters (T,), er (T,), converged (T,) = er <= 1e-6,
    cost (T,) = quadCost at the returned controls, state_0 / state_f (T, 6): the end states the solutions are pinned to)."""
    be = backend or default_backend()
    MU, DU, TU = capi.MU, capi.DU, capi.TU
    if nstate not in (6, 7):
        raise ValueError("nstate must be 6 or 7 (got %r)" % (nstate,))
    XC, t_TU, tau1, tau2, s0, sf = trajectory_stack_guess_batch(X0_states, Xf_states, MU, DU, TU, n_nodes, tof1_days, tof2_days, tau1,
                                                                backend=be)
    T = XC.shape[0]
    X = XC[:, :6].transpose(0, 2, 1)
    if nstate == 7:
        X = np.concatenate([X, np.full((T, n_nodes, 1), float(mass))], axis=2)
    r = be.direct_solve_batch(np.ascontiguousarray(X), np.zeros((T, n_nodes, 3)), t_TU, np.ascontiguousarray(s0[:, :6]),
                              np.ascontiguousarray(sf[:, :6]), mass, nsteps, maxIter, Isp, MU, DU, TU)
    u_all = r["u_all"].transpose(0, 2, 1).copy()
    return dict(X_all=r["X_all"].transpose(0, 2, 1).copy(), u_all=u_all, t_TU=t_TU, tau2=tau2, iters=r["iters"], er=r["er"],
                converged=r["er"] <= 1e-6, cost=_quad_cost(u_all, t_TU), state_0=s0[:, :6].copy(), state_f=sf[:, :6].copy())


def direct_costates(X_all, u_all, t_TU, state_0, state_f, nsteps=10, backend=None):
    """Costates of nstate-6 direct solutions in one device call (lto_direct_costates_batch): the multipliers of the direct QP's defect rows
    at (X_all, u_all), mapped to the node costates of the 12-dim p = 2 system (_direct_costate_map is the host mirror).  At a converged
    direct solution they are that energy-optimal problem's discrete costates, a start for multiShoot_CRTBP_indirect at a thrust limit that
    does not bind.  X_all (T, 6, N), u_all (T, 3, N), t_TU (T, N), state_0 / state_f (T, 6): direct_transfer_sweep's results.
    Returns dict(XC_all (T, 12, N): X_all bitwise and the costates (NaN where status != 0), multipliers (T, 6, N-1), du_max (T,): max |du|
    in N of the QP step at the given point, status (T,): the worst LTO_ST_* of K1's segments and the QP)."""
    be = backend or default_backend()
    X = np.asarray(X_all, dtype=np.float64)
    if X.ndim != 3 or X.shape[1] != 6:
        raise ValueError("X_all must be (T, 6, n_nodes) (got %s)" % (X.shape,))
    r = be.direct_costates(np.ascontiguousarray(X.transpose(0, 2, 1)), np.ascontiguousarray(np.asarray(u_all, dtype=np.float64).transpose(0, 2, 1)),
                           t_TU, state_0, state_f, nsteps, 2000.0, capi.MU, capi.DU, capi.TU)
    return dict(XC_all=r["XC_all"].transpose(0, 2, 1).copy(), multipliers=r["multipliers"].transpose(0, 2, 1).copy(), du_max=r["du_max"],
                status=r["status"])


G0 = 9.81                                          # the mass flow's g0 (CRTBP_prop_EP_deriv.jl:41; lto_indirect_params.g0)


def transfer_cost_indirect(XC_all, t_TU, MU, DU, TU, mass, thrustLimit, p, rho, Isp=2000.0, backend=None):
    """The cost of indirect trajectories XC_all (T, 12 or 14, N) on the time grids t_TU (T, N); thrustLimit and rho: scalars or (T,).
      12 rows (constant mass): ONE device call (lto_indirect_cost_batch) integrates every segment with the quadratures of |a_u| and
          |a_u|^2 along its adaptive steps: dv = int |a_u| dt in m/s and energy = int (|a_u| mass)^2 dt in N^2 TU, the units of the direct
          method's quadCost (direct_transfer_sweep's cost).  propellant: the rocket equation's mass for that dv at `Isp`.
      14 rows: no device call.  The mass is a state, so propellant = m0 - m_f from the node values and dv = Isp g0 ln(m0 / m_f), which
          is exact for the 14-dim dynamics (mdot = -|T| / (Isp g0), |a_u| = |T| / m); energy is not available (NaN).
    Returns dict(dv (T,), energy (T,), propellant (T,), status (T,): the worst LTO_ST_* of a trajectory's segments (14 rows: LTO_ST_NAN
    where a node mass is not finite))."""
    XC = np.asarray(XC_all, dtype=np.float64)
    if XC.ndim != 3 or XC.shape[1] not in (12, 14) or XC.shape[2] < 2:
        raise ValueError("XC_all must be (T, 12 or 14, n_nodes >= 2) (got %s)" % (XC.shape,))
    T, m, N = XC.shape
    t_TU = np.asarray(t_TU, dtype=np.float64)
    if t_TU.shape != (T, N):
        raise ValueError("t_TU must be (T, n_nodes) = %s (got %s)" % ((T, N), t_TU.shape))
    if m == 14:
        m0, mf = XC[:, 6, 0], XC[:, 6, -1]
        with np.errstate(divide="ignore", invalid="ignore"):
            dv = Isp * G0 * np.log(m0 / mf)
        ok = np.isfinite(m0) & np.isfinite(mf)
        return dict(dv=dv, energy=np.full(T, np.nan), propellant=m0 - mf, status=np.where(ok, 0, 1).astype(np.int32))   # LTO_ST_NAN
    be = backend or default_backend()
    tl = np.broadcast_to(np.asarray(thrustLimit, dtype=np.float64), (T,)).copy()
    rh = np.broadcast_to(np.asarray(rho, dtype=np.float64), (T,)).copy()
    params = (MU, DU, TU, float(tl[0]) if T else 0.0, mass, 1.0, p, float(rh[0]) if T else 1.0)
    r = be.indirect_cost(np.ascontiguousarray(XC.transpose(0, 2, 1)), t_TU, params, thrustLimit=tl, rho=rh)
    return dict(dv=r["dv"], energy=r["energy"], propellant=mass * -np.expm1(-r["dv"] / (Isp * G0)), status=r["status"])


def thrust_arcs_indirect(XC_all, t_TU, MU, DU, TU, mass, thrustLimit, rho, max_switch=16, backend=None):
    """The burns of p = 1 indirect trajectories XC_all (T, 12, N) on the time grids t_TU (T, N); thrustLimit and rho: scalars or (T,)
    (for a sweep's rows: its XC_all, t_TU and rho_last).  ONE device call (lto_indirect_switch_batch) locates the switches of
    S = |lv| - 1 (thrust on where S > 0) on every segment's adaptive steps, with the node rule between segments.
    Returns dict(t_switch (T, max_switch) TU, direction (T, max_switch) (+1 a burn starts, -1 it ends), n_switch (T,) (the true count;
    -1 where status is not OK), on_start (T,), status (T,), and per row: arcs, a (k, 2) array of [t_on, t_off] in TU clipped to
    [t_TU[0], t_TU[-1]] (None where the status is not OK or n_switch > max_switch), n_burns (k; -1 where arcs is None) and on_time
    (the total burn time in TU; NaN where arcs is None))."""
    XC = np.asarray(XC_all, dtype=np.float64)
    if XC.ndim != 3 or XC.shape[1] != 12 or XC.shape[2] < 2:
        raise ValueError("XC_all must be (T, 12, n_nodes >= 2): switch times are located in the 12-dim system (got %s)" % (XC.shape,))
    T, _, N = XC.shape
    t_TU = np.asarray(t_TU, dtype=np.float64)
    if t_TU.shape != (T, N):
        raise ValueError("t_TU must be (T, n_nodes) = %s (got %s)" % ((T, N), t_TU.shape))
    be = backend or default_backend()
    tl = np.broadcast_to(np.asarray(thrustLimit, dtype=np.float64), (T,)).copy()
    rh = np.broadcast_to(np.asarray(rho, dtype=np.float64), (T,)).copy()
    params = (MU, DU, TU, float(tl[0]) if T else 0.0, mass, 1.0, 1.0, float(rh[0]) if T else 1.0)
    r = be.indirect_switches(np.ascontiguousarray(XC.transpose(0, 2, 1)), t_TU, params, thrustLimit=tl, rho=rh, max_switch=max_switch)
    arcs, n_burns, on_time = [], np.full(T, -1, dtype=np.int64), np.full(T, np.nan)
    for j in range(T):
        n = int(r["n_switch"][j])
        if r["status"][j] != 0 or n < 0 or n > max_switch:
            arcs.append(None)
            continue
        t0, tf = t_TU[j, 0], t_TU[j, -1]
        on, begin, a = bool(r["on_start"][j]), t0, []
        for ts, d in zip(r["t_switch"][j, :n], r["direction"][j, :n]):
            if d > 0 and not on:
                on, begin = True, ts
            elif d < 0 and on:
                on = False
                a.append((begin, ts))
        if on:
            a.append((begin, tf))
        a = np.clip(np.array(a, dtype=np.float64).reshape(-1, 2), t0, tf)
        arcs.append(a)
        n_burns[j] = len(a)
        on_time[j] = float(np.sum(a[:, 1] - a[:, 0]))
    return dict(t_switch=r["t_switch"], direction=r["direction"], n_switch=r["n_switch"], on_start=r["on_start"], status=r["status"],
                arcs=arcs, n_burns=n_burns, on_time=on_time)


def indirect_transfer_sweep(X0_states, Xf_states, tau1, tof1_days, tof2_days, thrustLimit=0.05, rho_target=1e-4, seeds=None, n_nodes=30,
                            nsteps=10, mass=1e3, Isp=2000.0, maxIter_direct=100, backend=None, start="seeded"):
    """Fuel-optimal transfers for a grid of departure phases and flight times: the indirect demo's chain
    (CRTBP_Multishoot_indirect_demo.jl:166-281) run on every row of direct_transfer_sweep (nstate 6), each stage as one batched device call:
      start = "seeded" (the default), as the demo:
        start   per row j: costates 0.1 * N(0, 1) from np.random.default_rng(seeds[j]), end states pinned to state_0 / state_f,
                1e-10 jitter on the interior nodes (seeds default to 0 .. T-1);
        stage 1 adjoints-only solve, p = 2, 10 N, maxIter 10 (status 1 is expected there; only NaN fails the stage);
      start = "direct":
        stage 1 direct_costates of the direct solutions (the direct QP's multipliers: the discrete costates of the energy-optimal problem
                stage 2 solves), end states pinned to state_0 / state_f, no jitter; a row whose costate status is not 0 fails here;
      stage 2 full solve, p = 2, 10 N, maxIter 50;
      stage 3 p = 1 at thrustLimit, rho = 1, maxIter 30;
      stage 4 reduceFuel_indirect_batch(device_ladder=True) to rho_target, back-off draws from a fresh np.random.default_rng(seeds[j]);
      then transfer_cost_indirect of every surviving row (p = 1, its last rho).
    A row that fails a stage (status != 0) enters no later stage: stage_failed (T,) is that stage (1-4), 0 for a row that came through; its
    dv and energy are NaN.  Each row's result does not depend on the other rows.
    Returns dict(XC_all (T, 12, N): each row's last solution, t_TU, tau2, state_0, state_f, stage_failed, status and rho_last of the ladder
    (-1 / NaN for rows that did not reach it), dv (m/s), energy (N^2 TU), energy_p2: the stage-2 solution's energy at 10 N (NaN if it
    failed), and the direct sweep's cost / converged / iters alongside)."""
    MU, DU, TU = capi.MU, capi.DU, capi.TU
    shape = np.broadcast(*[np.atleast_1d(np.asarray(a, dtype=np.float64)) for a in (tau1, tof1_days, tof2_days)]).shape
    if len(shape) != 1:
        raise ValueError("tau1, tof1_days and tof2_days must be scalars or (T,) arrays")
    T = shape[0]
    seeds = list(range(T)) if seeds is None else [int(s) for s in np.atleast_1d(seeds)]
    if len(seeds) != T:
        raise ValueError("seeds must have one entry per row (%d, got %d)" % (T, len(seeds)))
    if not (np.isfinite(thrustLimit) and thrustLimit > 0):
        raise ValueError("thrustLimit must be a positive number of newtons (got %r)" % (thrustLimit,))
    if not (np.isfinite(rho_target) and 0 < rho_target <= 1):
        raise ValueError("rho_target must be in (0, 1] (got %r)" % (rho_target,))
    if n_nodes < 3:
        raise ValueError("n_nodes must be >= 3 (got %r)" % (n_nodes,))
    if start not in ("seeded", "direct"):
        raise ValueError("start must be 'seeded' or 'direct' (got %r)" % (start,))
    be = backend or default_backend()
    d = direct_transfer_sweep(X0_states, Xf_states, tau1, tof1_days, tof2_days, n_nodes=n_nodes, nsteps=nsteps, nstate=6, mass=mass, Isp=Isp,
                              maxIter=maxIter_direct, backend=be)
    t_TU = d["t_TU"]
    N = t_TU.shape[1]
    stage_failed = np.zeros(T, dtype=np.int32)
    if start == "direct":
        c = direct_costates(d["X_all"], d["u_all"], t_TU, d["state_0"], d["state_f"], nsteps=nsteps, backend=be)
        XC = c["XC_all"]
        XC[:, :6, 0] = d["state_0"]; XC[:, :6, -1] = d["state_f"]
        stage_failed[c["status"] != 0] = 1
    else:
        XC = np.empty((T, 12, N))
        for j in range(T):
            rng = np.random.default_rng(seeds[j])
            XC[j] = np.vstack([d["X_all"][j], 0.1 * rng.standard_normal((6, N))])
            XC[j, :6, 0] = d["state_0"][j]; XC[j, :6, -1] = d["state_f"][j]
            XC[j, :, 1:-1] += 1e-10 * rng.standard_normal((12, N - 2))

    def solve(stage, thrust, p, rho, max_iter, adjoints_only, fail_on):
        idx = np.flatnonzero(stage_failed == 0)
        if idx.size == 0:
            return
        Xn, _, st, _ = multiShoot_CRTBP_indirect_batch(XC[idx], t_TU[idx], MU, DU, TU, N, mass, thrust, adjoints_only, max_iter, p, rho,
                                                       backend=be)
        XC[idx] = Xn
        stage_failed[idx[np.isin(st, fail_on)]] = stage

    if start == "seeded":
        solve(1, 10.0, 2.0, 1.0, 10, True, (2,))
    solve(2, 10.0, 2.0, 1.0, 50, False, (1, 2))
    alive = np.flatnonzero(stage_failed == 0)
    energy_p2 = np.full(T, np.nan)
    if alive.size:
        energy_p2[alive] = transfer_cost_indirect(XC[alive], t_TU[alive], MU, DU, TU, mass, 10.0, 2.0, 1.0, Isp, backend=be)["energy"]
    solve(3, thrustLimit, 1.0, 1.0, 30, False, (1, 2))
    status = np.full(T, -1, dtype=np.int32); rho_last = np.full(T, np.nan)
    dv = np.full(T, np.nan); energy = np.full(T, np.nan)
    idx = np.flatnonzero(stage_failed == 0)
    if idx.size:
        # reduceFuel_indirect_batch(device_ladder=True) with its back-off draws taken the same way; called directly for rho_last
        draws = np.array([np.random.default_rng(seeds[j]).random(100) for j in idx], dtype=np.float64).reshape(idx.size, 100)
        r = be.indirect_reduce_fuel_batch(np.ascontiguousarray(XC[idx].transpose(0, 2, 1)), t_TU[idx], (MU, DU, TU, float(thrustLimit), mass,
                                          1.0, 1.0, 1.0), np.ones(idx.size), np.full(idx.size, float(rho_target)), draws,
                                          thrustLimit=np.full(idx.size, float(thrustLimit)), max_iter=10)
        st = r["status"]
        XC[idx] = r["XC_all"].transpose(0, 2, 1)
        status[idx] = st
        rho_last[idx] = r["rho_last"]
        stage_failed[idx[st != 0]] = 4
        ok = idx[st == 0]
        if ok.size:
            c = transfer_cost_indirect(XC[ok], t_TU[ok], MU, DU, TU, mass, thrustLimit, 1.0, rho_last[ok], Isp, backend=be)
            dv[ok] = c["dv"]; energy[ok] = c["energy"]
    return dict(XC_all=XC, t_TU=t_TU, tau2=d["tau2"], state_0=d["state_0"], state_f=d["state_f"], stage_failed=stage_failed, status=status,
                rho_last=rho_last, dv=dv, energy=energy, energy_p2=energy_p2, cost=d["cost"], direct_converged=d["converged"],
                direct_iters=d["iters"])


# --------------------------------------------------------------------------- direct method
def _band_direct(blocks, n, N):
    """Scatter of jacobianCalc (multiShoot_CRTBP_direct.jl:146-162): blocks (N-1, n, 2(n+3)) -> Jac_full."""
    J = np.zeros((n * (N - 1), N * (n + 3)))
    for i in range(N - 1):
        rows = slice(i * n, (i + 1) * n)
        J[rows, i * n:(i + 2) * n] = blocks[i][:, :2 * n]
        c0 = n * N + 3 * i
        J[rows, c0:c0 + 6] = blocks[i][:, 2 * n:]
    return J


def _qp_direct(X_all, u_all, dV1, dV2, defect, Jac_full, n, N, state_0, state_f, mass, tau, t0_TU, tf_TU, DU, TU, allowImpulsive,
               multipliers=False):
    """optimizeTraj (:248-403) for flagEnd = false: variables [X_jump | u_jump | dV1_jump | dV2_jump]
    (tf_jump, p1_jump, p2_jump are pinned to 0 by their bounds, :288-293).
    multipliers: also return the KKT multipliers of the linearised dynamics rows, (N-1, n) -- lambda of K7's K_L unknowns."""
    nX, nU = n * N, 3 * N
    nz = nX + nU + 6
    t_fixed = t0_TU + (tau + 1) / 2 * (tf_TU - t0_TU)
    dt = np.diff(t_fixed)
    dt_temp = np.concatenate([dt / 2, [dt[-1] / 2]]) + np.concatenate([[0.0], dt[:-1] / 2, [0.0]])      # :323-325
    w = np.repeat(dt_temp, 3)
    s = (DU / TU) ** 2
    H = np.zeros(nz); g = np.zeros(nz)
    H[nX:nX + nU] = 2 * w; g[nX:nX + nU] = 2 * w * u_all.T.ravel()
    H[nX + nU:] = 2 * s; g[nX + nU:] = 2 * s * np.concatenate([dV1, dV2])
    rows = []; rhs = []
    A_dyn = np.zeros((Jac_full.shape[0], nz)); A_dyn[:, :nX + nU] = -Jac_full[:, :nX + nU]                 # :337
    rows.append(A_dyn); rhs.append(defect.T.ravel())
    E = np.zeros((12, nz))
    for k in range(6):
        E[k, k] = 1.0; E[6 + k, (N - 1) * n + k] = 1.0
    for k in range(3):
        E[3 + k, nX + nU + k] = 1.0; E[9 + k, nX + nU + 3 + k] = 1.0
    b0 = state_0 - X_all[:6, 0] - np.concatenate([np.zeros(3), dV1])                                       # :374-375
    bf = state_f - X_all[:6, -1] - np.concatenate([np.zeros(3), dV2])
    rows.append(E); rhs.append(np.concatenate([b0, bf]))
    if n == 7:
        M = np.zeros((1, nz)); M[0, 6] = 1.0
        rows.append(M); rhs.append(np.array([mass - X_all[6, 0]]))                                        # :270
    if not allowImpulsive:
        Z = np.zeros((6, nz)); Z[np.arange(6), nX + nU + np.arange(6)] = 1.0
        rows.append(Z); rhs.append(np.zeros(6))                                                           # :301-302
    A = np.vstack(rows); b = np.concatenate(rhs)
    nc = A.shape[0]
    K = np.zeros((nz + nc, nz + nc))
    K[np.arange(nz), np.arange(nz)] = H
    K[:nz, nz:] = A.T; K[nz:, :nz] = A
    r = np.concatenate([-g, b])
    try:
        sol = np.linalg.solve(K, r)
        if not np.all(np.isfinite(sol)):
            raise np.linalg.LinAlgError
    except np.linalg.LinAlgError:
        sol = np.linalg.lstsq(K, r, rcond=None)[0]
    z = sol[:nz]
    x_update = z[:nX].reshape(N, n).T
    u_update = z[nX:nX + nU].reshape(N, 3).T
    dV1_update = z[nX + nU:nX + nU + 3]; dV2_update = z[nX + nU + 3:]
    cost = float(np.sum((u_all.T.ravel() + z[nX:nX + nU]) ** 2 * w) + s * np.sum((dV1 + dV1_update) ** 2) + s * np.sum((dV2 + dV2_update) ** 2))
    if multipliers:
        return x_update, u_update, dV1_update, dV2_update, cost, sol[nz:nz + n * (N - 1)].reshape(N - 1, n)
    return x_update, u_update, dV1_update, dV2_update, cost


def _direct_costate_map(blocks, lam, mass, DU, TU):
    """Host mirror of k_direct_qp_dual's epilogue: the multipliers lam (N-1, 6) of the direct QP's defect rows -> node costates
    [lr; lv] (6, N) of the 12-dim p = 2 system.  blocks (N-1, 6, 18) [.., row, col] = [X_i, X_{i+1}, u_i, u_{i+1}] columns.
    p_i = Jx(i, i)^T lam_i (i < N-1), p_{N-1} = -Jx(N-2, N-1)^T lam_{N-2}; costate = -p / kappa^2, kappa = mass DU 1e3 / TU^2
    (u in N = kappa x the nondimensional acceleration)."""
    blocks = np.asarray(blocks, dtype=np.float64); lam = np.asarray(lam, dtype=np.float64)
    Nm1 = lam.shape[0]
    p = np.empty((6, Nm1 + 1))
    for i in range(Nm1):
        p[:, i] = blocks[i][:, :6].T @ lam[i]
    p[:, Nm1] = -(blocks[Nm1 - 1][:, 6:12].T @ lam[Nm1 - 1])
    kappa = mass / (TU * TU / DU / 1e3)
    return -p / (kappa * kappa)


def multiShoot_CRTBP_direct(X_all, u_all, tau1, tau2, t_TU, dV1, dV2, MU, DU, TU, n_nodes, nsteps, mass, Isp, X0_times, X0_states,
                            Xf_times, Xf_states, plot_yn=False, flagEnd=False, beta=0.0, allowImpulsive=False, maxIter=100,
                            backend=None, log=None, device_qp=False):
    """(X_all, u_all, tau1, tau2, t_TU, dV1, dV2, defect) = multiShoot_CRTBP_direct(...)   (:58-60, :593).
    `log`, if a list, receives one dict per SQP iteration (iter, er, cost, alpha).
    device_qp: solve the QP on the GPU (lto_direct_qp, banded KKT) instead of the dense host KKT solve (allowImpulsive = false only)."""
    if flagEnd:
        raise NotImplementedError("flagEnd = true makes the subproblem a bound-constrained NLP (Ipopt, :286-298); only the "
                                  "demo's flagEnd = false equality-constrained QP is mirrored")
    be = backend or default_backend()
    X_all = np.array(X_all, dtype=np.float64); u_all = np.array(u_all, dtype=np.float64); t_TU = np.array(t_TU, dtype=np.float64)
    dV1 = np.array(dV1, dtype=np.float64); dV2 = np.array(dV2, dtype=np.float64)
    n = X_all.shape[0]; N = n_nodes
    t0_TU = t_TU[0]; tf_TU = t_TU[-1]
    tau = (t_TU - t0_TU) / (tf_TU - t0_TU) * 2 - 1                                                        # :481

    def defectCalc(X, U, t):
        d, e = be.direct_defect(X.T[None], U.T[None], t[None], nsteps, Isp, MU, DU, TU)
        return d[0].T.copy(), e[0]

    defect, errors = defectCalc(X_all, u_all, t_TU)                                                       # :486
    iterCount = 0; er = 1.0
    while er > 1e-6:                                                                                      # :491
        iterCount += 1
        if iterCount > maxIter:
            break
        _, _, blocks = be.direct_blocks(X_all.T[None], u_all.T[None], t_TU[None], nsteps, Isp, MU, DU, TU)   # :500
        Jac_full = _band_direct(blocks[0], n, N)
        pert_tf = 1e-3                                                                                    # :504
        t0_TU = t_TU[0]; tf_TU = t_TU[-1]
        t_mod = np.stack([t0_TU + (tau + 1) / 2 * (tf_TU + pert_tf - t0_TU), t0_TU + (tau + 1) / 2 * (tf_TU - pert_tf - t0_TU)])
        dm, _ = be.direct_defect(np.stack([X_all.T] * 2), np.stack([u_all.T] * 2), t_mod, nsteps, Isp, MU, DU, TU)   # :511-512 (one batch)
        ddefect_dt = (dm[0] - dm[1]) / (2 * pert_tf)
        Jac_full = np.hstack([Jac_full, ddefect_dt.ravel()[:, None]])                                     # :516
        state_0, state_f = interpEndStates(tau1, tau2, X0_times, X0_states, Xf_times, Xf_states, MU)
        if device_qp and not allowImpulsive:
            b0 = state_0 - X_all[:6, 0] - np.concatenate([np.zeros(3), dV1]); bf = state_f - X_all[:6, -1] - np.concatenate([np.zeros(3), dV2])
            if n == 7:
                b0 = np.concatenate([b0, [mass - X_all[6, 0]]])
            t_fixed = t0_TU + (tau + 1) / 2 * (tf_TU - t0_TU)
            xu, uu, st = be.direct_qp(np.ascontiguousarray(blocks.transpose(0, 1, 3, 2)), defect.T[None], u_all.T[None], t_fixed[None], b0[None], bf[None])
            x_update, u_update = xu[0].T, uu[0].T
            dV1_update = np.zeros(3); dV2_update = np.zeros(3)
            dt_ = np.diff(t_fixed); w_ = np.repeat(np.concatenate([dt_ / 2, [dt_[-1] / 2]]) + np.concatenate([[0.0], dt_[:-1] / 2, [0.0]]), 3)
            cost = float(np.sum((u_all.T.ravel() + u_update.T.ravel()) ** 2 * w_) + (DU / TU) ** 2 * (np.sum(dV1 ** 2) + np.sum(dV2 ** 2)))
        else:
            x_update, u_update, dV1_update, dV2_update, cost = _qp_direct(X_all, u_all, dV1, dV2, defect, Jac_full, n, N, state_0, state_f,
                                                                          mass, tau, t0_TU, tf_TU, DU, TU, allowImpulsive)
        alpha = 1.0
        if iterCount > 10:                                                                                # :559-561, lineSearch :405-430
            alpha_all = np.linspace(0.1, 1.0, 10)
            Xt = np.stack([(X_all + x_update * a).T for a in alpha_all]); Ut = np.stack([(u_all + u_update * a).T for a in alpha_all])
            dd, _ = be.direct_defect(Xt, Ut, np.stack([t_TU] * 10), nsteps, Isp, MU, DU, TU)
            ers = np.sum(dd.reshape(10, -1) ** 2, axis=1)
            alpha = float(alpha_all[np.argmin(ers)])
        X_all = X_all + x_update * alpha; u_all = u_all + u_update * alpha                                # :563-569
        dV1 = dV1 + dV1_update * alpha; dV2 = dV2 + dV2_update * alpha
        t_TU = t0_TU + (tau + 1) / 2 * (tf_TU - t0_TU)                                                    # :582
        defect, errors = defectCalc(X_all, u_all, t_TU)                                                   # :585
        er = float(np.max(np.abs(defect)))
        if log is not None:
            log.append(dict(iter=iterCount, er=er, cost=cost, alpha=alpha))
    return X_all, u_all, tau1, tau2, t_TU, dV1, dV2, defect


def multiShoot_CRTBP_direct_batch(X_all, u_all, tau1, tau2, t_TU, MU, DU, TU, n_nodes, nsteps, mass, Isp, X0_times, X0_states, Xf_times, Xf_states,
                                  maxIter=100, backend=None, log=None):
    """multiShoot_CRTBP_direct (:465-594; flagEnd = false, allowImpulsive = false, dV = 0: the demo's setting) for a BATCH of independent
    trajectories with every heavy step on the device: per SQP iteration ONE launch for all defects + Jacobian blocks
    (lto_direct_defect_jac_traj), ONE launch for all QPs (lto_direct_qp), one launch for the 10-point line searches of all
    trajectories (from iteration 11 on, :559-561), one launch for the defect check (:585).  A trajectory stops when its
    max defect <= 1e-6 (:491) or after maxIter iterations; the others go on.
    X_all: (T, n, N), u_all: (T, 3, N), t_TU: (T, N), tau1 / tau2: scalars or (T,).
    Returns (X_all, u_all, defect (T, n, N-1), iters (T,))."""
    be = backend or default_backend()
    X = np.array(X_all, dtype=np.float64).transpose(0, 2, 1).copy(); U = np.array(u_all, dtype=np.float64).transpose(0, 2, 1).copy()
    t = np.array(t_TU, dtype=np.float64)
    T, N, n = X.shape
    t1 = np.broadcast_to(np.asarray(tau1, dtype=np.float64), (T,)); t2 = np.broadcast_to(np.asarray(tau2, dtype=np.float64), (T,))
    ends = [interpEndStates(float(t1[j]), float(t2[j]), X0_times, X0_states, Xf_times, Xf_states, MU) for j in range(T)]
    s0 = np.stack([e[0] for e in ends]); sf = np.stack([e[1] for e in ends])
    defect, _ = be.direct_defect(X, U, t, nsteps, Isp, MU, DU, TU)                                          # :486
    er = np.ones(T)                                                                                         # `er = 1.0` (:490): one iteration always runs
    iters = np.zeros(T, dtype=np.int32)
    active = er > 1e-6
    it = 0
    while active.any() and it < maxIter:
        it += 1
        idx = np.nonzero(active)[0]
        Xa, Ua, ta = X[idx], U[idx], t[idx]
        d, _, blocks = be.direct_blocks(Xa, Ua, ta, nsteps, Isp, MU, DU, TU)                                # :500 (blocks [.., row, col])
        b0 = s0[idx] - Xa[:, 0, :6]; bf = sf[idx] - Xa[:, -1, :6]                                           # :374-375 (dV = 0)
        if n == 7:
            b0 = np.concatenate([b0, (mass - Xa[:, 0, 6])[:, None]], axis=1)                                # :270
        xu, uu, st = be.direct_qp(np.ascontiguousarray(blocks.transpose(0, 1, 3, 2)), d, Ua, ta, b0, bf)    # optimizeTraj (:248-403)
        alpha = np.ones(len(idx))
        if it > 10:                                                                                         # lineSearch (:405-430), all trajectories at once
            al = np.linspace(0.1, 1.0, 10)
            Xt = (Xa[None] + al[:, None, None, None] * xu[None]).reshape(-1, N, n); Ut = (Ua[None] + al[:, None, None, None] * uu[None]).reshape(-1, N, 3)
            dd, _ = be.direct_defect(Xt, Ut, np.tile(ta, (10, 1)), nsteps, Isp, MU, DU, TU)
            ers = np.sum(dd.reshape(10, len(idx), -1) ** 2, axis=2)
            alpha = al[np.argmin(ers, axis=0)]
        X[idx] = Xa + alpha[:, None, None] * xu; U[idx] = Ua + alpha[:, None, None] * uu                    # :563-569
        dn, _ = be.direct_defect(X[idx], U[idx], ta, nsteps, Isp, MU, DU, TU)                               # :585
        defect[idx] = dn
        er[idx] = np.max(np.abs(dn), axis=(1, 2))
        iters[idx] = it
        if log is not None:
            log.append(dict(iter=it, n_active=len(idx), er=er.copy(), alpha=alpha.copy()))
        active = er > 1e-6
    return X.transpose(0, 2, 1).copy(), U.transpose(0, 2, 1).copy(), defect.transpose(0, 2, 1).copy(), iters


# --------------------------------------------------------------------------- indirect method
def _end_pins(nstate):
    """Components held at the first / last node (:141-142, :324-325).  12-dim: the 6 states of both ends.  14-dim ([r v m | lr lv lm]):
    position, velocity and mass at the start; position, velocity and lm at the end -- the final mass is free (it follows from the
    control history), and lm, which enters no right-hand side, is fixed by its end value lm(t_f) (any constant offset of lm solves
    the defect equations, so one value must be held or the band is rank deficient)."""
    first = list(range(nstate))
    last = list(range(6)) + ([2 * nstate - 1] if nstate == 7 else [])
    return first, last


def _band_indirect(phi, nstate, N):
    """Band assembly of jacobianCalc (multiShoot_CRTBP_indirect.jl:127-142): phi (N-1, m, m) -> Jac_full."""
    m = 2 * nstate
    J = np.zeros((m * (N - 1), N * m))
    eye = np.eye(m)
    for i in range(N - 1):
        J[i * m:(i + 1) * m, i * m:(i + 1) * m] = phi[i]
        J[i * m:(i + 1) * m, (i + 1) * m:(i + 2) * m] = -eye
    first, last = _end_pins(nstate)
    J[:, first] = 0.0                                                                                     # :141
    J[:, [(N - 1) * m + c for c in last]] = 0.0                                                           # :142
    return J


def multiShoot_CRTBP_indirect(XC_all, t_TU, MU, DU, TU, n_nodes, mass0, thrustLimit, plot_yn=False, flag_adjointsOnly=False,
                              maxIter=50, p=1.0, rho=1.0, backend=None, log=None, device_newton=False, Isp=2000.0):
    """(XC_all, defect, status_flag) = multiShoot_CRTBP_indirect(...)   (:58-59, :344).
    device_newton: solve the update on the GPU (lto_indirect_newton_nd, either system) instead of the dense host least squares.

    XC_all with 12 rows is the reference's system.  With 14 rows ([r v m | lr lv lm], BASELINE configs[1] as north_star words it) the
    same loop runs on the 14-dim system with mass: nstate = 7, the band blocks are 14 x 14, and the end pins of :324-325 become
    7-element (`_end_pins`: r, v, m at the first node; r, v and lm at the last -- the final mass is free).  The reference has no such solver -- its loop
    hard-codes the 12-dim RHS (:258) and 6-element pins -- so this is the same algorithm on the larger system, not a mirror of
    existing code; `Isp` enters the mass flow (GeneralCode/twoBody_stateCostate_mass_deriv.jl:61)."""
    be = backend or default_backend()
    XC_all = np.array(XC_all, dtype=np.float64); t_TU = np.asarray(t_TU, dtype=np.float64)
    nstate = XC_all.shape[0] // 2; m = 2 * nstate; N = n_nodes
    if nstate not in (6, 7):
        raise ValueError("XC_all must have 12 rows (the reference's system) or 14 ([r v m | lr lv lm])")
    params = (MU, DU, TU, thrustLimit, mass0, 1.0, p, rho) + ((Isp,) if nstate == 7 else ())              # :260
    status_flag = 0
    pin0, pinf = _end_pins(nstate)
    state_0 = XC_all[pin0, 0].copy(); state_f = XC_all[pinf, -1].copy()

    def defectCalc(XC):
        return be.indirect_defect(XC.T[None], t_TU[None], params)[0].T.copy()

    keep = np.ones(N * m, dtype=bool)
    if flag_adjointsOnly:                                                                                 # :169-178
        for ind in range(N - 1):
            keep[ind * m:ind * m + nstate] = False

    def solve(J, dvec):
        """-sparse(J) \\ d (:181-182): least squares over the structurally non-empty columns, 0 elsewhere."""
        if device_newton:
            return be.indirect_newton(phi, dvec.reshape(1, N - 1, m), flag_adjointsOnly)[0].T
        Jk = J[:, keep]
        live = np.any(Jk != 0.0, axis=0)
        sol = np.zeros(Jk.shape[1])
        sol[live] = -np.linalg.lstsq(Jk[:, live], dvec, rcond=None)[0]
        full = np.zeros(N * m)
        full[keep] = sol
        return full.reshape(N, m).T

    defect = defectCalc(XC_all)                                                                           # :274
    iterCount = 0; er = 1.0
    while er > 1e-10:                                                                                     # :280
        iterCount += 1
        if iterCount > maxIter:
            status_flag = 1
            break
        _, phi = be.indirect_blocks(XC_all.T[None], t_TU[None], params)                                   # :290
        Jac_full = None if device_newton else _band_indirect(phi[0], nstate, N)
        xc_update = solve(Jac_full, defect.T.ravel())
        if np.max(np.abs(xc_update)) < 1e-1:                                                              # SOC :190-214
            d_soc = defectCalc(XC_all + xc_update)
            xc_update = xc_update + solve(Jac_full, d_soc.T.ravel())
        alpha = 1.0
        if iterCount > 3:                                                                                 # :300-302, lineSearch :221-246
            alpha_all = np.linspace(0.1, 1.0, 20)
            trial = np.stack([(XC_all + xc_update * a).T for a in alpha_all])
            dd = be.indirect_defect(trial, np.stack([t_TU] * 20), params)
            ers = np.sum(dd.reshape(20, -1) ** 2, axis=1)
            alpha = float(alpha_all[np.argmin(ers)])
        XC_all = XC_all + xc_update * alpha                                                               # :304
        XC_all[pin0, 0] = state_0; XC_all[pinf, -1] = state_f                                             # :324-325
        defect = defectCalc(XC_all)                                                                       # :328
        er = float(np.max(np.abs(defect)))
        if log is not None:
            log.append(dict(iter=iterCount, er=er, alpha=alpha))
        if not er <= 1e3:                                                                                 # :333-336 (also catches NaN)
            iterCount += 100
            if np.isnan(er):
                break
    # :339-341 tests XC_all[1,1] only -- a pinned entry whose update is exactly 0, so it can never be NaN (a latent bug of the
    # reference, not mirrored): a trajectory whose defects or nodes went non-finite is reported as such, never as "converged"
    if np.isnan(er) or not np.all(np.isfinite(XC_all)):
        status_flag = 2
    return XC_all, defect, status_flag


def multiShoot_CRTBP_indirect_batch(XC_all, t_TU, MU, DU, TU, n_nodes, mass0, thrustLimit, flag_adjointsOnly=False, maxIter=50, p=1.0,
                                    rho=1.0, backend=None, Isp=2000.0):
    """multiShoot_CRTBP_indirect for a BATCH of independent trajectories, iterated entirely on the device
    (lto_indirect_solve_batch_nd).  XC_all: (n_traj, m, n_nodes) in the reference's per-trajectory shape, m = 12 or 14 (the system
    with mass, same end pins as multiShoot_CRTBP_indirect; `Isp` enters its mass flow); t_TU: (n_traj, n_nodes);
    thrustLimit / rho: scalars or per-trajectory arrays (continuation ladders).  Returns (XC_all, defect (n_traj, m, n_nodes-1),
    status_flag (n_traj,), iters (n_traj,))."""
    be = backend or default_backend()
    XC = np.ascontiguousarray(np.asarray(XC_all, dtype=np.float64).transpose(0, 2, 1))
    T, _, m = XC.shape
    if m not in (12, 14):
        raise ValueError("XC_all must be (n_traj, 12 or 14, n_nodes) (got %s)" % (np.shape(XC_all),))
    tl = np.broadcast_to(np.asarray(thrustLimit, dtype=np.float64), (T,)).copy()
    rh = np.broadcast_to(np.asarray(rho, dtype=np.float64), (T,)).copy()
    params = (MU, DU, TU, float(tl[0]), mass0, 1.0, p, float(rh[0])) + ((Isp,) if m == 14 else ())
    r = be.indirect_solve_batch(XC, np.asarray(t_TU, dtype=np.float64), params, thrustLimit=tl, rho=rh, max_iter=maxIter,
                                flag_adjointsOnly=flag_adjointsOnly)
    return r["XC_all"].transpose(0, 2, 1).copy(), r["defect"].transpose(0, 2, 1).copy(), r["status_flag"], r["iters"]


def _reduceFuel_steps(XC_all, rho_current, rho_target, rng):
    """The rho-continuation ladder of reduceFuel_indirect (HelperFunctions.jl:105-193) as a coroutine: yields (XC_start, rho) for
    every call of multiShoot_CRTBP_indirect it wants (maxIter = 10, p = 1) and is sent back (XC_new, defect, status); returns the
    function's result.  Shared by the one-trajectory mirror and the batched driver, so both follow the reference line by line."""
    if rho_target > rho_current:
        rho_target = rho_current
    rho_temp = rho_current
    XC_new, defect, status = yield XC_all, rho_temp
    if status == 0 and rho_current == rho_target:
        return XC_new, defect, status
    while status != 0 and rho_temp < 1:                                                                   # :131-141
        rho_temp = min(rho_temp * 5, 1.0)
        XC_new, defect, status = yield XC_all, rho_temp
    if rho_temp == 1 and status != 0:
        return XC_new, defect, status
    if status == 0:
        XC_all = XC_new.copy()
    count = 0
    while rho_temp > rho_target or status != 0:                                                           # :155-187
        count += 1
        if count > 100:
            return XC_new, defect, 3
        if status == 0:
            XC_all = XC_new.copy()
            rho_temp = max(rho_temp / 2, rho_target)
        else:
            rho_temp *= 3 * (1 + rng.random())                                                            # :182
        XC_new, defect, status = yield XC_all, rho_temp
    return XC_new, defect, status


def reduceFuel_indirect(XC_all, t_TU, MU, DU, TU, n_nodes, mass, thrustLimit, rho_current, rho_target, backend=None, rng=None,
                        log=None, Isp=2000.0):
    """rho-continuation driver (HelperFunctions.jl:105-193).  `rng` supplies the rand() of the back-off (:182).
    XC_all: 12 or 14 rows (multiShoot_CRTBP_indirect); `Isp` enters the mass flow of the 14-dim system."""
    gen = _reduceFuel_steps(np.array(XC_all, dtype=np.float64), rho_current, rho_target, rng or np.random.default_rng(0))
    req = next(gen)
    while True:
        XC, rho = req
        out = multiShoot_CRTBP_indirect(XC, t_TU, MU, DU, TU, n_nodes, mass, thrustLimit, False, False, 10, 1.0, rho, backend=backend, Isp=Isp)
        if log is not None:
            log.append(dict(rho=rho, status=out[2], er=float(np.max(np.abs(out[1])))))
        try:
            req = gen.send(out)
        except StopIteration as fin:
            return fin.value


def reduceFuel_indirect_batch(XC_all, t_TU, MU, DU, TU, n_nodes, mass, thrustLimit, rho_current, rho_target, backend=None, rngs=None,
                              log=None, Isp=2000.0, device_ladder=False):
    """reduceFuel_indirect for a BATCH of independent trajectories (SURVEY 8(f) row 3): every trajectory walks its own rho ladder
    (halving on success, x 3(1 + rand) back-off on failure, :155-187); each round, the solver calls all unfinished trajectories
    ask for are issued as ONE lto_indirect_solve_batch call with per-trajectory rho / thrustLimit.
    XC_all: (n_traj, m, n_nodes), m = 12 or 14 (`Isp` enters the mass flow of the 14-dim system); t_TU: (n_traj, n_nodes);
    thrustLimit, rho_current, rho_target: scalars or (n_traj,).
    Returns (XC_new (n_traj, m, n_nodes), defect (n_traj, m, n_nodes-1), status (n_traj,), rounds).
    device_ladder: run the whole ladder in ONE device call (lto_indirect_reduce_fuel_batch): a trajectory's next solver call starts
    as soon as its last one ends.  Same results; each trajectory's 100 back-off draws are taken up front with rng.random(100), the
    same values as its successive rng.random() calls.  `rounds` is then the most solver calls any trajectory made, the round count
    of the default driver; `log` is not supported."""
    be = backend or default_backend()
    XC_all = np.asarray(XC_all, dtype=np.float64); t_TU = np.asarray(t_TU, dtype=np.float64)
    T = XC_all.shape[0]
    tl = np.broadcast_to(np.asarray(thrustLimit, dtype=np.float64), (T,)).copy()
    r0 = np.broadcast_to(np.asarray(rho_current, dtype=np.float64), (T,)); r1 = np.broadcast_to(np.asarray(rho_target, dtype=np.float64), (T,))
    rngs = rngs or [np.random.default_rng(j) for j in range(T)]
    if device_ladder:
        if log is not None:
            raise ValueError("log is not available with device_ladder=True: the ladder has no rounds on the device")
        m = XC_all.shape[1]
        if m not in (12, 14):
            raise ValueError("XC_all must be (n_traj, 12 or 14, n_nodes) (got %s)" % (XC_all.shape,))
        draws = np.array([rngs[j].random(100) for j in range(T)], dtype=np.float64).reshape(T, 100)
        params = (MU, DU, TU, float(tl[0]) if T else 0.0, mass, 1.0, 1.0, 1.0) + ((Isp,) if m == 14 else ())
        r = be.indirect_reduce_fuel_batch(np.ascontiguousarray(XC_all.transpose(0, 2, 1)), t_TU, params, r0, r1, draws, thrustLimit=tl,
                                          max_iter=10)
        rounds = int(r["calls"].max()) if T else 0
        return r["XC_all"].transpose(0, 2, 1).copy(), r["defect"].transpose(0, 2, 1).copy(), r["status"], rounds
    gens = [_reduceFuel_steps(XC_all[j].copy(), float(r0[j]), float(r1[j]), rngs[j]) for j in range(T)]
    req = {j: next(gens[j]) for j in range(T)}
    res = [None] * T
    rounds = 0
    while req:
        rounds += 1
        idx = sorted(req)
        XC = np.stack([req[j][0] for j in idx]); rho = np.array([req[j][1] for j in idx])
        Xn, dn, st, it = multiShoot_CRTBP_indirect_batch(XC, t_TU[idx], MU, DU, TU, n_nodes, mass, tl[idx], False, 10, 1.0, rho, backend=be,
                                                         Isp=Isp)
        if log is not None:
            log.append(dict(round=rounds, n=len(idx), rho=rho.copy(), status=np.asarray(st).copy()))
        for k, j in enumerate(idx):
            try:
                req[j] = gens[j].send((Xn[k], dn[k], int(st[k])))
            except StopIteration as fin:
                res[j] = fin.value
                del req[j]
    return (np.stack([r[0] for r in res]), np.stack([r[1] for r in res]), np.array([r[2] for r in res], dtype=np.int32), rounds)


def demo_fixtures():
    """(X0_times, X0_states, Xf_times, Xf_states) as the demos load them (CRTBP_Multishoot_direct_demo.jl:68-71)."""
    X0 = load_orbit(1); Xf = load_orbit(2)
    return np.linspace(0, 1, X0.shape[1]), X0, np.linspace(0, 1, Xf.shape[1]), Xf
