"""GPU: the transfer cost of indirect trajectories (lto_indirect_cost_batch, solvers.transfer_cost_indirect) and the indirect transfer
sweep (solvers.indirect_transfer_sweep).

The reference computes no cost of an indirect trajectory, so nothing in it pins these numbers.  What does:
  * same steps: the cost pass is K4 with two quadratures outside the error norm, so its defects are BITWISE those of the defect-only call;
  * closed form: with p = 0 the thrust is aL wherever lv != 0, so dv and energy are aL and aL^2 times the time span;
  * an independent integrator: scipy's DOP853 on the augmented system [x; int |a_u| dt; int |a_u|^2 dt], node to node."""
import numpy as np
import pytest
from scipy.integrate import solve_ivp

from lowthrustopt_b200 import capi, solvers as S, synthetic

pytestmark = pytest.mark.gpu
MU, DU, TU = capi.MU, capi.DU, capi.TU
DEMO = (0.75, 10.0, 10.0)


@pytest.fixture(scope="module")
def gpu(lto):
    return S.GpuBackend(handle=lto)


@pytest.fixture(scope="module")
def demo(gpu):
    """The demo row's chain (CRTBP_Multishoot_indirect_demo.jl:166-281) stage by stage, with the sweep's start for seed 42: the p = 2 and the
    p = 1 (rho = 1) solutions, and the ladder's results at rho = 1e-2 and 1e-4 from the same p = 1 solution."""
    fx = S.demo_fixtures()
    d = S.direct_transfer_sweep(fx[1], fx[3], DEMO[0], DEMO[1], DEMO[2], backend=gpu)
    t = d["t_TU"]
    rng = np.random.default_rng(42)
    XC = np.vstack([d["X_all"][0], 0.1 * rng.standard_normal((6, 30))])
    XC[:6, 0] = d["state_0"][0]; XC[:6, -1] = d["state_f"][0]
    XC[:, 1:-1] += 1e-10 * rng.standard_normal((12, 28))
    XC = XC[None]
    XC, _, st, _ = S.multiShoot_CRTBP_indirect_batch(XC, t, MU, DU, TU, 30, 1e3, 10.0, True, 10, 2.0, 1.0, backend=gpu)
    assert st[0] in (0, 1)
    p2, _, st, _ = S.multiShoot_CRTBP_indirect_batch(XC, t, MU, DU, TU, 30, 1e3, 10.0, False, 50, 2.0, 1.0, backend=gpu)
    assert st[0] == 0
    p1, _, st, _ = S.multiShoot_CRTBP_indirect_batch(p2, t, MU, DU, TU, 30, 1e3, 0.05, False, 30, 1.0, 1.0, backend=gpu)
    assert st[0] == 0
    out = dict(t=t, p2=p2, p1=p1, cost=d["cost"][0])
    for target in (1e-2, 1e-4):
        Xr, _, st, _ = S.reduceFuel_indirect_batch(p1, t, MU, DU, TU, 30, 1e3, 0.05, 1.0, target, backend=gpu,
                                                   rngs=[np.random.default_rng(42)], device_ladder=True)
        assert st[0] == 0
        out[target] = Xr
    return out


def _params(tl, p, rho):
    return capi.indirect_params(thrustLimit=tl, p=p, rho=rho)


def _same_steps(h, XC, t, tl, p, rho):
    prm = _params(float(tl[0]), p, rho)
    c = h.indirect_cost_batch(XC, t, params=prm, thrustLimit=tl, rho=rho, defect=True)
    ref = h.indirect_traj(XC, t, params=prm, thrustLimit=tl, rho=rho, jac=False)
    n = XC.shape[0]
    assert np.array_equal(c["defect"], ref["defect"].reshape(c["defect"].shape))
    assert np.array_equal(c["status"], ref["status"].reshape(n, -1).max(axis=1))
    return c


@pytest.mark.parametrize("tl,p,rho", [(10.0, 2.0, 1.0), (0.05, 1.0, 1.0), (0.05, 1.0, 1e-2)])
def test_cost_pass_takes_the_defect_passes_steps(lto, tl, p, rho):
    c = synthetic.continuation_batch(n_traj=24, n_seg_per_traj=29, ndim=12, seed=31)
    r = _same_steps(lto, c["XC_all"], c["t_TU"], np.full(24, tl), p, rho)
    assert (r["status"] == 0).all() and np.isfinite(r["dv"]).all() and (r["dv"] >= 0).all() and np.array_equal(r["dv"] == 0, r["energy"] == 0)
    # p = 2 and p = 1 at rho = 1 thrust wherever |lv| > 0.  At rho = 1e-2 these costates (|lv| ~ 0.1-0.3, far below the switch at 1) give
    # tanh((|lv| - 1) / (2 rho)) = -1 exactly: no thrust, and a cost of exactly zero is the right answer there.
    if p == 2.0 or rho == 1.0:
        assert (r["dv"] > 0).all() and (r["energy"] > 0).all()


def test_cost_pass_takes_the_defect_passes_steps_on_the_demo_solution(lto, demo):
    _same_steps(lto, demo[1e-4].transpose(0, 2, 1), demo["t"], np.array([0.05]), 1.0, 1e-4)


def test_constant_thrust_closed_form(lto):
    """p = 0: |a_u| = aL = thrustLimit k / mass wherever lv != 0, so dv = aL (t_N - t_1) DU 1e3 / TU and energy = thrustLimit^2 (t_N - t_1)."""
    c = synthetic.continuation_batch(n_traj=8, n_seg_per_traj=29, ndim=12, seed=5)
    tl = np.geomspace(0.05, 10.0, 8)
    r = lto.indirect_cost_batch(c["XC_all"], c["t_TU"], params=_params(0.05, 0.0, 1.0), thrustLimit=tl)
    span = c["t_TU"][:, -1] - c["t_TU"][:, 0]
    aL = tl * (TU * TU / DU / 1e3) / 1000.0
    assert (r["status"] == 0).all()
    np.testing.assert_allclose(r["dv"], aL * span * DU * 1e3 / TU, rtol=1e-13, atol=0)
    np.testing.assert_allclose(r["energy"], (aL * 1000.0 * DU * 1e3 / TU ** 2) ** 2 * span, rtol=1e-13, atol=0)


def _rhs(tl, p, rho, mass=1000.0):
    """CRTBP_stateCostate_deriv! (CRTBP_stateCostate_deriv.jl:9-90) with |a_u| and |a_u|^2 appended (rows 12, 13)."""
    aL = tl * (TU * TU / DU / 1e3) / mass

    def f(_, y):
        r, v, lr, lv = y[0:3], y[3:6], y[6:9], y[9:12]
        d1 = np.array([r[0] + MU, r[1], r[2]]); d2 = d1 - [1.0, 0.0, 0.0]
        n1, n2 = np.linalg.norm(d1), np.linalg.norm(d2)
        n = np.linalg.norm(lv)
        if p == 0:
            u = aL
        elif p == 1:
            u = 0.5 * (1 + np.tanh((n - 1) / (2 * rho))) * aL
        else:
            u = min((n / p) ** (1 / (p - 1)), aL)
        if not n > 0:
            u = 0.0
        a_u = -u * lv / n if n > 0 else np.zeros(3)
        g = -(1 - MU) * d1 / n1 ** 3 - MU * d2 / n2 ** 3
        acc = g + [r[0] + 2 * v[1], r[1] - 2 * v[0], 0.0] + a_u
        G = ((1 - MU) * (3 * np.outer(d1, d1) / n1 ** 5 - np.eye(3) / n1 ** 3) + MU * (3 * np.outer(d2, d2) / n2 ** 5 - np.eye(3) / n2 ** 3)
             + np.diag([1.0, 1.0, 0.0]))
        dlr = -G @ lv
        dlv = -lr - np.array([-2 * lv[1], 2 * lv[0], 0.0])
        return np.concatenate([v, acc, dlr, dlv, [u, u * u]])
    return f


def _dop853_cost(XC, t, tl, p, rho):
    """XC (12, N): per segment from node i over [t_i, t_i+1], summed in segment order; returns (dv, energy, end states (N-1, 12))."""
    f = _rhs(tl, p, rho)
    q = np.zeros(2); ends = []
    for i in range(XC.shape[1] - 1):
        s = solve_ivp(f, (t[i], t[i + 1]), np.concatenate([XC[:, i], [0.0, 0.0]]), method="DOP853", rtol=1e-13, atol=1e-15)
        assert s.success
        q += s.y[12:, -1]; ends.append(s.y[:12, -1])
    return q[0] * DU * 1e3 / TU, q[1] * (1000.0 * DU * 1e3 / TU ** 2) ** 2, np.array(ends)


@pytest.mark.parametrize("case", ["p2", "p1", 1e-2, 1e-4])
def test_cost_matches_an_independent_dop853_integration(lto, demo, case):
    tl, p, rho = {"p2": (10.0, 2.0, 1.0), "p1": (0.05, 1.0, 1.0)}.get(case, (0.05, 1.0, case))
    XC, t = demo[case][0], demo["t"][0]
    r = lto.indirect_cost_batch(XC.T[None], t[None], params=_params(tl, p, rho), defect=True)
    dv, e, ends = _dop853_cost(XC, t, tl, p, rho)
    x_gpu = r["defect"][0] + XC[:, 1:].T                                    # x(t_i+1) = defect + node i+1
    ddv, de = abs(r["dv"][0] - dv) / dv, abs(r["energy"][0] - e) / e
    dx = np.abs(x_gpu - ends).max() / max(1.0, np.abs(ends).max())
    print("\n[cost vs DOP853] %s: dv %.6f m/s rel %.2e | energy %.6e N^2 TU rel %.2e | end states %.2e" % (case, r["dv"][0], ddv, r["energy"][0],
                                                                                                     de, dx))
    # rho = 1e-4: a switch narrower than the stage spacing limits any order-8 pair to the ~1e-8 state accuracy of DESIGN.md section 5
    # (measured on a B200: dv 1.0e-8, energy 1.2e-10 relative)
    bar = 2e-8 if case == 1e-4 else 1e-9
    assert r["status"][0] == 0 and ddv <= bar and de <= bar, (ddv, de)


def test_rows_do_not_depend_on_their_batch(lto):
    c = synthetic.continuation_batch(n_traj=64, n_seg_per_traj=29, ndim=12, seed=9)
    XC, t, tl = c["XC_all"], c["t_TU"], c["thrustLimit"]
    p = _params(0.05, 1.0, 1e-2)
    full = lto.indirect_cost_batch(XC, t, params=p, thrustLimit=tl, rho=1e-2, defect=True)
    for j in (0, 17, 63):
        one = lto.indirect_cost_batch(XC[j:j + 1], t[j:j + 1], params=p, thrustLimit=tl[j:j + 1], rho=1e-2, defect=True)
        for k in ("dv", "energy", "status", "defect"):
            assert np.array_equal(one[k][0], full[k][j]), (j, k)
    bad = XC.copy(); bad[17, 5, 9] = np.nan
    nan = lto.indirect_cost_batch(bad, t, params=p, thrustLimit=tl, rho=1e-2, defect=True)
    assert nan["status"][17] == 1 and np.isnan(nan["dv"][17])            # LTO_ST_NAN
    keep = np.arange(64) != 17
    for k in ("dv", "energy", "status", "defect"):
        assert np.array_equal(nan[k][keep], full[k][keep]), k
    empty = lto.indirect_cost_batch(np.zeros((0, 30, 12)), np.zeros((0, 30)), params=p)
    assert empty["dv"].shape == (0,) and empty["status"].shape == (0,)


def test_library_refuses_what_the_wrapper_would(lto):
    import ctypes as C
    L = capi.lib()
    XC = np.zeros((1, 3, 12)); t = np.array([[0.0, 1.0, 0.5]]); dv = np.zeros(1); e = np.zeros(1)
    p = _params(0.05, 1.0, 1.0)
    rc = L.lto_indirect_cost_batch(lto._h, C.addressof(p), 1, 3, XC.ctypes.data, t.ctypes.data, None, None, dv.ctypes.data, e.ctypes.data, None, None)
    assert rc == -2 and b"trajectory 0" in L.lto_last_error(lto._h)
    p.controller = capi.LTO_CTRL_ODE78
    t = np.array([[0.0, 0.5, 1.0]])
    rc = L.lto_indirect_cost_batch(lto._h, C.addressof(p), 1, 3, XC.ctypes.data, t.ctypes.data, None, None, dv.ctypes.data, e.ctypes.data, None, None)
    assert rc == -2


def test_two_device_handle_splits_whole_trajectories(lto):
    if capi.lib().lto_device_count() < 2:
        pytest.skip("needs two GPUs")
    hm = capi.Handle([0, 1])
    try:
        c = synthetic.continuation_batch(n_traj=33, n_seg_per_traj=29, ndim=12, seed=4)
        p = _params(0.05, 1.0, 1e-2)
        a = lto.indirect_cost_batch(c["XC_all"], c["t_TU"], params=p, thrustLimit=c["thrustLimit"], rho=1e-2, defect=True)
        b = hm.indirect_cost_batch(c["XC_all"], c["t_TU"], params=p, thrustLimit=c["thrustLimit"], rho=1e-2, defect=True)
        for k in a:
            assert np.array_equal(a[k], b[k]), k
    finally:
        hm.close()


GRID_TAU1 = np.repeat([0.65, 0.7, 0.75, 0.8], 4)
GRID_TOF = np.tile([[10.0, 10.0], [9.0, 11.0], [11.0, 9.0], [10.0, 12.0]], (4, 1))
GRID_SEEDS = np.arange(34, 50)                                             # the demo row (8) gets the demo's seed 42


@pytest.fixture(scope="module")
def sweep(gpu):
    fx = S.demo_fixtures()
    return S.indirect_transfer_sweep(fx[1], fx[3], GRID_TAU1, GRID_TOF[:, 0], GRID_TOF[:, 1], seeds=GRID_SEEDS, backend=gpu)


def test_sweep_rows_equal_the_sweep_of_that_row_alone(gpu, sweep):
    fx = S.demo_fixtures()
    print("\n[sweep] stage_failed %s" % sweep["stage_failed"].tolist())
    for j in range(16):
        one = S.indirect_transfer_sweep(fx[1], fx[3], GRID_TAU1[j:j + 1], GRID_TOF[j:j + 1, 0], GRID_TOF[j:j + 1, 1], seeds=GRID_SEEDS[j:j + 1],
                                        backend=gpu)
        for k in ("XC_all", "stage_failed", "status", "rho_last", "dv", "energy", "energy_p2", "cost"):
            assert np.array_equal(one[k][0], sweep[k][j], equal_nan=True), (j, k)
        print("[sweep] row %2d tau1 %.2f tof %4.1f + %4.1f d: stage_failed %d | direct cost %.6e | p = 2 energy %.6e | rho %.0e dv %.4f m/s "
              "energy %.6e" % (j, GRID_TAU1[j], GRID_TOF[j, 0], GRID_TOF[j, 1], sweep["stage_failed"][j], sweep["cost"][j], sweep["energy_p2"][j],
                               sweep["rho_last"][j], sweep["dv"][j], sweep["energy"][j]))


def test_sweep_demo_row_is_the_device_ladder_from_the_demo_p1_solution(sweep, demo):
    j = int(np.flatnonzero((GRID_TAU1 == DEMO[0]) & (GRID_TOF[:, 0] == DEMO[1]) & (GRID_TOF[:, 1] == DEMO[2]))[0])
    assert GRID_SEEDS[j] == 42 and sweep["stage_failed"][j] == 0 and sweep["rho_last"][j] == 1e-4
    assert np.array_equal(sweep["XC_all"][j], demo[1e-4][0])
    c = S.transfer_cost_indirect(demo[1e-4], demo["t"], MU, DU, TU, 1e3, 0.05, 1.0, 1e-4)
    assert c["dv"][0] == sweep["dv"][j] and c["energy"][0] == sweep["energy"][j]
