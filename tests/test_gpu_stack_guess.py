"""GPU: the trajectory-stacking initial guess for a batch of transfers in one device call (lto_stack_guess_batch,
solvers.trajectory_stack_guess_batch) and the direct-method sweep built on it (solvers.direct_transfer_sweep), against the per-transfer
host path (solvers.trajectory_stack_guess: host splines and find_tau, one propagation call per arc; multiShoot_CRTBP_direct).

The arcs run through the same propagation kernels as the host path, so they agree with it to the last bits of the start states;
the spline lookups agree with scipy's to <= 1e-15 and find_τ picks the same candidate."""
import numpy as np
import pytest

from lowthrustopt_b200 import capi, solvers as S

pytestmark = pytest.mark.gpu
MU, DU, TU, DAY = capi.MU, capi.DU, capi.TU, capi.DAY
FX = S.demo_fixtures()
X0, XF = FX[1], FX[3]
LTO_ST_MAXSTEPS = 3


@pytest.fixture(scope="module")
def gpu(lto):
    return S.GpuBackend(handle=lto)


def _grid(N, n, seed):
    """n seeded rows (tau1, tof1_days, tof2_days): tau1 across [0, 1) and the wrap cases -0.25, 1.0, 1.75; flight times in 6-14 days."""
    rng = np.random.default_rng(seed)
    tau1 = np.concatenate([rng.random(n - 3), [-0.25, 1.0, 1.75]])
    tof1 = rng.uniform(6.0, 14.0, n); tof2 = rng.uniform(6.0, 14.0, n)
    if N == 41:
        tof1[5] = tof2[5] = 6.0                               # t_split == t_TU[20] exactly: node 20 starts arc 2
    return tau1, tof1, tof2


def _times(tof1_days, tof2_days, N):
    t = np.stack([np.linspace(0.0, (a * DAY / TU) + (b * DAY / TU), N) for a, b in zip(tof1_days, tof2_days)])
    return t, np.asarray(tof1_days) * DAY / TU


def _host_rows(gpu, tau1, tof1, tof2, N):
    return [S.trajectory_stack_guess(X0, XF, MU, DU, TU, N, float(a), float(b), float(t), backend=gpu) for t, a, b in zip(tau1, tof1, tof2)]


def _check_rows(out, host, tau1):
    XC, _, _, tau2, s0, sf = out
    worst = 0.0
    for j, (XCh, _, _, tau2h, _, _) in enumerate(host):
        assert tau2[j] == tau2h, (j, tau2[j], tau2h)
        e0, ef = S.interpEndStates(float(tau1[j]), tau2h, *FX)
        assert np.abs(s0[j, :6] - e0).max() <= 1e-15 and np.abs(sf[j, :6] - ef).max() <= 1e-15, j
        assert np.all(s0[j, 6:] == 0) and np.all(sf[j, 6:] == 0)
        worst = max(worst, float(np.abs(XC[j] - XCh).max()))
    # observed on one B200: 0 (bitwise) on the demo row and both grids -- the arcs start from the same states as the host path's
    assert worst <= 1e-12, "max |XC - host XC| = %.3e (0 observed on a B200)" % worst
    return worst


def test_demo_row_matches_host(gpu):
    out = S.trajectory_stack_guess_batch(X0, XF, MU, DU, TU, 30, 10.0, 10.0, 0.75, backend=gpu)
    assert out[3][0] == 0.274                                 # the host's tau2 (test_gpu_solvers.py)
    worst = _check_rows(out, _host_rows(gpu, [0.75], [10.0], [10.0], 30), [0.75])
    print("demo row: max |XC - host XC| = %.3e" % worst)


@pytest.mark.parametrize("N,seed", [(30, 11), (41, 12)])
def test_grid_matches_host_loop(gpu, N, seed):
    tau1, tof1, tof2 = _grid(N, 32, seed)
    out = S.trajectory_stack_guess_batch(X0, XF, MU, DU, TU, N, tof1, tof2, tau1, backend=gpu)
    assert out[0].shape == (32, 12, N) and out[1].shape == (32, N)
    if N == 41:
        t, ts = _times(tof1, tof2, N)
        assert t[5, 20] == ts[5]
        assert np.all(out[0][5, 6:, 20] == 0)                 # node 20 is arc 2's start: a point of the final orbit, zero costates
    worst = _check_rows(out, _host_rows(gpu, tau1, tof1, tof2, N), tau1)
    print("grid N=%d: max |XC - host XC| = %.3e" % (N, worst))


def test_batch_composition_invariance(lto):
    tau1, tof1, tof2 = _grid(30, 32, 13)
    t, ts = _times(tof1, tof2, 30)
    full = lto.stack_guess_batch(X0, XF, tau1, t, ts)
    sub = [3, 7, 8, 20]
    part = lto.stack_guess_batch(X0, XF, tau1[sub], t[sub], ts[sub])
    one = lto.stack_guess_batch(X0, XF, tau1[5:6], t[5:6], ts[5:6])
    for k in full:
        assert np.array_equal(part[k], full[k][sub]), k
        assert np.array_equal(one[k], full[k][5:6]), k
    assert np.all(full["status"] == 0)


def test_failing_row_leaves_the_others_alone(lto):
    tau1, tof1, tof2 = _grid(30, 16, 14)
    t, ts = _times(tof1, tof2, 30)
    # max_attempts: 3x the steps of a 14-day ballistic arc (host path), longer than any clean segment and far short of the bad row's
    # first 59-day segment of its second arc
    p0 = capi.indirect_params(thrustLimit=0.0, mass=1e3)
    seg = lto.indirect(np.concatenate([X0[:, 0], np.zeros(6)])[None], [0.0], [14.0 * DAY / TU], params=p0, jac=False)
    p = capi.indirect_params(thrustLimit=0.0, mass=1e3)
    p.max_attempts = int(3 * seg["nsteps"][0, 1])
    clean = lto.stack_guess_batch(X0, XF, tau1, t, ts, params=p)
    assert np.all(clean["status"] == 0)
    tb, tsb = _times([10.0], [2000.0], 30)
    at = 6
    ins = lambda a, v: np.concatenate([a[:at], v, a[at:]])
    bad = lto.stack_guess_batch(X0, XF, ins(tau1, [0.5]), ins(t, tb), ins(ts, tsb), params=p)
    assert bad["status"][at] == LTO_ST_MAXSTEPS
    keep = [j for j in range(17) if j != at]
    for k in clean:
        assert np.array_equal(bad[k][keep], clean[k]), k


def test_edge_cases(lto):
    e = lto.stack_guess_batch(X0, XF, np.zeros(0), np.zeros((0, 30)), np.zeros(0))
    assert e["XC_all"].shape == (0, 30, 12) and e["tau2"].shape == (0,) and e["status"].shape == (0,)
    tau1, tof1, tof2 = _grid(30, 3, 15)
    t, ts = _times(tof1, tof2, 30)
    cases = []
    tt = t.copy(); tt[1, 7] = tt[1, 6]; cases.append((tau1, tt, ts))                      # not strictly increasing
    tt = t.copy(); tt[1, 7] = np.nan; cases.append((tau1, tt, ts))                         # non-finite time
    s = ts.copy(); s[1] = t[1, 0]; cases.append((tau1, t, s))                              # t_split == t_TU[0]
    s = ts.copy(); s[1] = t[1, -1] * (1 + 1e-15); cases.append((tau1, t, s))               # t_split past t_TU[end]
    a = tau1.copy(); a[1] = np.nan; cases.append((a, t, ts))
    a = tau1.copy(); a[1] = 1000.5; cases.append((a, t, ts))                               # |tau1| > 1e3
    for a, tt, s in cases:
        with pytest.raises(capi.LtoError, match=r"error -2: trajectory 1\b"):
            lto.stack_guess_batch(X0, XF, a, tt, s)
    for x0, xf, tt in ((X0[:, :2], XF, t), (X0, XF[:, :2], t), (X0, XF, t[:, :1])):       # short tables, one node
        with pytest.raises(capi.LtoError, match="error -2"):
            lto.stack_guess_batch(x0, xf, tau1, tt, np.minimum(ts, tt[:, -1]))
    bad = XF.copy(); bad[3, 40] = np.inf
    with pytest.raises(capi.LtoError, match="error -2"):
        lto.stack_guess_batch(X0, bad, tau1, t, ts)


def test_multi_device_handle_stack_guess(lto):
    if capi.lib().lto_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    tau1, tof1, tof2 = _grid(30, 32, 16)
    t, ts = _times(tof1, tof2, 30)
    hm = capi.Handle([0, 1])
    try:
        a = lto.stack_guess_batch(X0, XF, tau1, t, ts)
        b = hm.stack_guess_batch(X0, XF, tau1, t, ts)
    finally:
        hm.close()
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def _host_quad_cost(u_all, t_TU):
    """quadCost (multiShoot_CRTBP_direct.jl:367-368, dV = 0) with _qp_direct's node weights on the host chain's time grid."""
    tau = (t_TU - t_TU[0]) / (t_TU[-1] - t_TU[0]) * 2 - 1
    t_fixed = t_TU[0] + (tau + 1) / 2 * (t_TU[-1] - t_TU[0])
    dt = np.diff(t_fixed)
    w = np.repeat(np.concatenate([dt / 2, [dt[-1] / 2]]) + np.concatenate([[0.0], dt[:-1] / 2, [0.0]]), 3)
    return float(np.sum(u_all.T.ravel() ** 2 * w))


def test_direct_sweep_matches_host_chain(gpu):
    tau1, tof1, tof2 = _grid(30, 16, 17)
    sw = S.direct_transfer_sweep(X0, XF, tau1, tof1, tof2, backend=gpu)
    assert sw["X_all"].shape == (16, 6, 30) and sw["u_all"].shape == (16, 3, 30)
    for j in range(16):
        XC, t_TU, a, tau2, s0, sf = S.trajectory_stack_guess(X0, XF, MU, DU, TU, 30, float(tof1[j]), float(tof2[j]), float(tau1[j]), backend=gpu)
        assert sw["tau2"][j] == tau2
        log = []
        out = S.multiShoot_CRTBP_direct(XC[:6].copy(), np.zeros((3, 30)), a, tau2, t_TU, np.zeros(3), np.zeros(3), MU, DU, TU, 30, 10, 1e3, 2000.0,
                                        *FX, backend=gpu, log=log)
        conv = float(np.abs(out[7]).max()) <= 1e-6
        assert sw["iters"][j] == len(log) and bool(sw["converged"][j]) == conv, (j, sw["iters"][j], len(log), conv)
        assert np.abs(sw["X_all"][j] - out[0]).max() < 1e-8 and np.abs(sw["u_all"][j] - out[1]).max() < 1e-8, j
        c = _host_quad_cost(out[1], out[4])
        assert abs(sw["cost"][j] - c) <= 1e-7 * abs(c), (j, sw["cost"][j], c)
    print("sweep: %d of 16 converged, iterations %s" % (int(sw["converged"].sum()), np.bincount(sw["iters"]).tolist()))
