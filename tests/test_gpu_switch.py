"""GPU: switch times of p = 1 indirect trajectories (lto_indirect_switch_batch, solvers.thrust_arcs_indirect).

The reference locates no switches on the shooting path, so nothing in it pins these numbers.  What does:
  * same steps: the switch pass is K4 with a scan outside the error norm, so its defects are BITWISE those of the defect-only call;
  * an independent integrator: scipy's DOP853 with the event |lv| - 1 = 0, node to node, with the node rule applied on the host;
  * the definition's invariants: times in order inside the span, alternating directions starting opposite to on_start, and a burn time
    that matches the delta-v of lto_indirect_cost_batch at rho = 1e-4 (near bang-bang: dv ~ aL x burn time)."""
import numpy as np
import pytest
from scipy.integrate import solve_ivp

from lowthrustopt_b200 import capi, solvers as S, synthetic

pytestmark = pytest.mark.gpu
MU, DU, TU = capi.MU, capi.DU, capi.TU
DEMO = (0.75, 10.0, 10.0)
AL = 0.05 * (TU * TU / DU / 1e3) / 1000.0                                  # aL of 0.05 N on 1000 kg, DU/TU^2


@pytest.fixture(scope="module")
def gpu(lto):
    return S.GpuBackend(handle=lto)


@pytest.fixture(scope="module")
def demo(gpu):
    """The demo row's p = 1 solutions as in test_gpu_transfer_cost.py: rho = 1, and the ladder's results at rho = 1e-2 and 1e-4."""
    fx = S.demo_fixtures()
    d = S.direct_transfer_sweep(fx[1], fx[3], DEMO[0], DEMO[1], DEMO[2], backend=gpu)
    t = d["t_TU"]
    rng = np.random.default_rng(42)
    XC = np.vstack([d["X_all"][0], 0.1 * rng.standard_normal((6, 30))])
    XC[:6, 0] = d["state_0"][0]; XC[:6, -1] = d["state_f"][0]
    XC[:, 1:-1] += 1e-10 * rng.standard_normal((12, 28))
    XC = XC[None]
    XC, _, st, _ = S.multiShoot_CRTBP_indirect_batch(XC, t, MU, DU, TU, 30, 1e3, 10.0, True, 10, 2.0, 1.0, backend=gpu)
    p2, _, st, _ = S.multiShoot_CRTBP_indirect_batch(XC, t, MU, DU, TU, 30, 1e3, 10.0, False, 50, 2.0, 1.0, backend=gpu)
    assert st[0] == 0
    p1, _, st, _ = S.multiShoot_CRTBP_indirect_batch(p2, t, MU, DU, TU, 30, 1e3, 0.05, False, 30, 1.0, 1.0, backend=gpu)
    assert st[0] == 0
    out = dict(t=t, p1=p1)
    for target in (1e-2, 1e-4):
        Xr, _, st, _ = S.reduceFuel_indirect_batch(p1, t, MU, DU, TU, 30, 1e3, 0.05, 1.0, target, backend=gpu,
                                                   rngs=[np.random.default_rng(42)], device_ladder=True)
        assert st[0] == 0
        out[target] = Xr
    return out


def _params(rho, tl=0.05):
    return capi.indirect_params(thrustLimit=tl, p=1.0, rho=rho)


def _crossing_batch(n_traj, seed):
    """continuation_batch with its costates scaled by 6: |lv| ~ 1 at the nodes, so every row crosses |lv| = 1."""
    c = synthetic.continuation_batch(n_traj=n_traj, n_seg_per_traj=29, ndim=12, seed=seed)
    c["XC_all"][:, :, 6:] *= 6.0
    return c


def _check_invariants(r, t):
    for j in range(len(r["n_switch"])):
        n = int(r["n_switch"][j])
        if n < 0:
            continue
        k = min(n, r["t_switch"].shape[1])
        ts, d = r["t_switch"][j, :k], r["direction"][j, :k]
        assert np.all(np.diff(ts) >= 0) and np.all(ts >= t[j, 0]) and np.all(ts <= t[j, -1]), (j, ts)
        want = np.where(np.arange(k) % 2 == 0, -1, 1) * (1 if r["on_start"][j] else -1)
        assert np.array_equal(d, want), (j, d, r["on_start"][j])
        assert np.isnan(r["t_switch"][j, k:]).all() and (r["direction"][j, k:] == 0).all()


def _same_steps(h, XC, t, tl, rho):
    prm = _params(rho, float(tl[0]))
    r = h.indirect_switch_batch(XC, t, params=prm, thrustLimit=tl, rho=rho, max_switch=64, defect=True)
    ref = h.indirect_traj(XC, t, params=prm, thrustLimit=tl, rho=rho, jac=False)
    n = XC.shape[0]
    assert np.array_equal(r["defect"], ref["defect"].reshape(r["defect"].shape))
    assert np.array_equal(r["status"], ref["status"].reshape(n, -1).max(axis=1))
    return r


@pytest.mark.parametrize("rho", [1.0, 1e-2])
def test_switch_pass_takes_the_defect_passes_steps(lto, rho):
    c = _crossing_batch(24, 31)
    r = _same_steps(lto, c["XC_all"], c["t_TU"], np.full(24, 0.05), rho)
    assert (r["status"] == 0).all() and (r["n_switch"] >= 1).all(), r["n_switch"]
    _check_invariants(r, c["t_TU"])
    print("\n[switch] synthetic rho %g: switches per row %s" % (rho, r["n_switch"].tolist()))


def test_switch_pass_takes_the_defect_passes_steps_on_the_demo_solution(lto, demo):
    r = _same_steps(lto, demo[1e-4].transpose(0, 2, 1), demo["t"], np.array([0.05]), 1e-4)
    assert r["status"][0] == 0


def _host_switches(XC, t, rho):
    """DOP853 (rtol 1e-13, atol 1e-15) from each node to the next with the event |lv| - 1 = 0 (directions from the slope of |lv|), and the
    node rule between segments.  Returns (times, directions, on_start, sdot at each time)."""
    f = _rhs_p1(rho)
    ev = lambda _, y: np.linalg.norm(y[9:12]) - 1.0
    times, dirs, sdot = [], [], []
    side = lambda y: bool(np.linalg.norm(y[9:12]) > 1.0)
    end_prev = None
    for i in range(XC.shape[1] - 1):
        x0 = XC[:, i]
        if end_prev is not None and side(x0) != end_prev:
            times.append(t[i]); dirs.append(1 if side(x0) else -1); sdot.append(np.nan)
        s = solve_ivp(f, (t[i], t[i + 1]), x0, method="DOP853", rtol=1e-13, atol=1e-15, events=ev)
        assert s.success
        for te, ye in zip(s.t_events[0], s.y_events[0]):
            lv, ld = ye[9:12], f(te, ye)[9:12]
            sd = np.dot(lv, ld) / np.linalg.norm(lv)
            times.append(te); dirs.append(1 if sd > 0 else -1); sdot.append(sd)
        end_prev = side(s.y[:, -1])
    return np.array(times), np.array(dirs), side(XC[:, 0]), np.array(sdot)


def _rhs_p1(rho, tl=0.05, mass=1000.0):
    """CRTBP_stateCostate_deriv! (CRTBP_stateCostate_deriv.jl:9-90), p = 1."""
    aL = tl * (TU * TU / DU / 1e3) / mass

    def f(_, y):
        r, v, lr, lv = y[0:3], y[3:6], y[6:9], y[9:12]
        d1 = np.array([r[0] + MU, r[1], r[2]]); d2 = d1 - [1.0, 0.0, 0.0]
        n1, n2 = np.linalg.norm(d1), np.linalg.norm(d2)
        n = np.linalg.norm(lv)
        u = 0.5 * (1 + np.tanh((n - 1) / (2 * rho))) * aL
        g = -(1 - MU) * d1 / n1 ** 3 - MU * d2 / n2 ** 3
        acc = g + [r[0] + 2 * v[1], r[1] - 2 * v[0], 0.0] - u * lv / n
        G = ((1 - MU) * (3 * np.outer(d1, d1) / n1 ** 5 - np.eye(3) / n1 ** 3) + MU * (3 * np.outer(d2, d2) / n2 ** 5 - np.eye(3) / n2 ** 3)
             + np.diag([1.0, 1.0, 0.0]))
        return np.concatenate([v, acc, -G @ lv, -lr - np.array([-2 * lv[1], 2 * lv[0], 0.0])])
    return f


@pytest.mark.parametrize("case", ["p1", 1e-2, 1e-4])
def test_switches_match_an_independent_dop853_integration(lto, demo, case):
    rho = 1.0 if case == "p1" else case
    XC, t = demo[case][0], demo["t"][0]
    r = lto.indirect_switch_batch(XC.T[None], t[None], params=_params(rho), max_switch=64, defect=True)
    n = int(r["n_switch"][0])
    ht, hd, hon, sdot = _host_switches(XC, t, rho)
    gt, gd = r["t_switch"][0, :n], r["direction"][0, :n]
    print("\n[switch vs DOP853] rho %g: %d switches (host %d), on_start %d" % (rho, n, len(ht), r["on_start"][0]))
    assert r["status"][0] == 0 and n == len(ht) and np.array_equal(gd, hd) and bool(r["on_start"][0]) == hon, (gt, ht, gd, hd)
    dt = np.abs(gt - ht)
    # |delta lv| / |S'| at each switch: the end-state distance to DOP853 carried to time (DESIGN.md section 5's sharp-switch accuracy)
    x_gpu = r["defect"][0] + XC[:, 1:].T
    ends = np.array([solve_ivp(_rhs_p1(rho), (t[i], t[i + 1]), XC[:, i], method="DOP853", rtol=1e-13, atol=1e-15).y[:, -1]
                     for i in range(len(t) - 1)])
    dlv = np.abs(x_gpu[:, 9:12] - ends[:, 9:12]).max()
    for k in range(n):
        print("[switch vs DOP853]   %+d at %.12f TU: |dt| %.2e TU, |S'| %.3e, |dlv|/|S'| %.2e" % (gd[k], gt[k], dt[k], abs(sdot[k]),
                                                                                               dlv / abs(sdot[k]) if sdot[k] == sdot[k] else 0.0))
    bar = 1e-7 if rho == 1e-4 else 1e-9
    assert dt.max(initial=0.0) <= bar, dt


def test_invariants_and_burn_time_on_the_demo_solution(lto, gpu, demo):
    t = demo["t"]
    r = S.thrust_arcs_indirect(demo[1e-4], t, MU, DU, TU, 1e3, 0.05, 1e-4, max_switch=64, backend=gpu)
    raw = dict(t_switch=r["t_switch"], direction=r["direction"], n_switch=r["n_switch"], on_start=r["on_start"])
    _check_invariants(raw, t)
    c = S.transfer_cost_indirect(demo[1e-4], t, MU, DU, TU, 1e3, 0.05, 1.0, 1e-4, backend=gpu)
    burn = c["dv"][0] / (AL * DU * 1e3 / TU)
    rel = abs(r["on_time"][0] - burn) / burn
    print("\n[switch] demo rho 1e-4: %d switches, %d burns, on_start %d, on_time %.6f TU vs dv / aL %.6f TU (rel %.2e)\n[switch] arcs %s"
          % (r["n_switch"][0], r["n_burns"][0], r["on_start"][0], r["on_time"][0], burn, rel, r["arcs"][0].tolist()))
    assert rel <= 1e-2, rel


def test_a_node_on_a_switch_counts_it_once(lto, demo):
    """Insert a node at a located switch (its state from the pairs-form propagation of the node before it): the switch is found once, at
    that node or within 1e-9 TU of it, and the other switches stay where they were."""
    XC, t = demo[1e-2][0], demo["t"][0]
    prm = _params(1e-2)
    r = lto.indirect_switch_batch(XC.T[None], t[None], params=prm, max_switch=64)
    n = int(r["n_switch"][0])
    assert n >= 1
    ts = r["t_switch"][0, 0]
    i = int(np.searchsorted(t, ts, side="right") - 1)
    assert t[i] < ts < t[i + 1]
    xs = lto.indirect(XC[:, i][None], np.array([t[i]]), np.array([ts]), params=prm, jac=False)["defect"][0]
    XC2 = np.insert(XC, i + 1, xs, axis=1)
    t2 = np.insert(t, i + 1, ts)
    r2 = lto.indirect_switch_batch(XC2.T[None], t2[None], params=prm, max_switch=64)
    n2 = int(r2["n_switch"][0])
    t_new = r2["t_switch"][0, :n2]
    near = np.abs(t_new - ts) <= 1e-9
    print("\n[switch] node at %.12f TU: %d switches (before %d), distance %.2e TU" % (ts, n2, n, np.abs(t_new - ts).min()))
    assert n2 == n and near.sum() == 1
    assert np.array_equal(r2["direction"][0, :n2], r["direction"][0, :n])
    assert np.abs(t_new - r["t_switch"][0, :n]).max() <= 1e-9


def test_rows_do_not_depend_on_their_batch(lto):
    c = _crossing_batch(64, 9)
    XC, t, tl = c["XC_all"], c["t_TU"], np.full(64, 0.05)
    p = _params(1e-2)
    full = lto.indirect_switch_batch(XC, t, params=p, thrustLimit=tl, rho=1e-2, defect=True)
    keys = ("t_switch", "direction", "n_switch", "on_start", "status", "defect")
    for j in (0, 17, 63):
        one = lto.indirect_switch_batch(XC[j:j + 1], t[j:j + 1], params=p, thrustLimit=tl[j:j + 1], rho=1e-2, defect=True)
        for k in keys:
            assert np.array_equal(one[k][0], full[k][j], equal_nan=True), (j, k)
    bad = XC.copy(); bad[17, 5, 9] = np.nan
    nan = lto.indirect_switch_batch(bad, t, params=p, thrustLimit=tl, rho=1e-2, defect=True)
    assert nan["status"][17] == 1 and nan["n_switch"][17] == -1 and np.isnan(nan["t_switch"][17]).all()   # LTO_ST_NAN
    keep = np.arange(64) != 17
    for k in keys:
        assert np.array_equal(nan[k][keep], full[k][keep], equal_nan=True), k
    empty = lto.indirect_switch_batch(np.zeros((0, 30, 12)), np.zeros((0, 30)), params=p)
    assert empty["t_switch"].shape == (0, 16) and empty["n_switch"].shape == (0,)
    one = lto.indirect_switch_batch(XC, t, params=p, thrustLimit=tl, rho=1e-2, max_switch=1)
    assert np.array_equal(one["n_switch"], full["n_switch"]) and (one["n_switch"] > 1).any()
    assert np.array_equal(one["t_switch"][:, 0], full["t_switch"][:, 0], equal_nan=True)
    assert np.array_equal(one["direction"][:, 0], full["direction"][:, 0])


def test_library_refuses_what_the_wrapper_would(lto):
    import ctypes as C
    L = capi.lib()
    XC = np.zeros((1, 3, 12)); ts = np.zeros(64); d = np.zeros(64, dtype=np.int32); n = np.zeros(1, dtype=np.int32); on = np.zeros(1, dtype=np.int32)

    def call(p, t, m=16):
        return L.lto_indirect_switch_batch(lto._h, C.addressof(p), 1, 3, XC.ctypes.data, t.ctypes.data, None, None, m, ts.ctypes.data,
                                           d.ctypes.data, n.ctypes.data, on.ctypes.data, None, None)
    good = np.array([[0.0, 0.5, 1.0]])
    assert call(_params(1.0), np.array([[0.0, 1.0, 0.5]])) == -2 and b"trajectory 0" in L.lto_last_error(lto._h)
    assert call(_params(1.0), np.array([[0.0, np.nan, 1.0]])) == -2 and b"trajectory 0" in L.lto_last_error(lto._h)
    assert call(capi.indirect_params(p=2.0), good) == -2
    assert call(_params(1.0), good, 0) == -2 and call(_params(1.0), good, 65) == -2
    p = _params(1.0); p.controller = capi.LTO_CTRL_ODE78
    assert call(p, good) == -2


def test_two_device_handle_splits_whole_trajectories(lto):
    if capi.lib().lto_device_count() < 2:
        pytest.skip("needs two GPUs")
    hm = capi.Handle([0, 1])
    try:
        c = _crossing_batch(33, 4)
        p = _params(1e-2)
        a = lto.indirect_switch_batch(c["XC_all"], c["t_TU"], params=p, rho=1e-2, defect=True)
        b = hm.indirect_switch_batch(c["XC_all"], c["t_TU"], params=p, rho=1e-2, defect=True)
        for k in a:
            assert np.array_equal(a[k], b[k], equal_nan=True), k
    finally:
        hm.close()
