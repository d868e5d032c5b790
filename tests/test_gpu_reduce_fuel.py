"""GPU: the rho continuation of reduceFuel_indirect in one device call (lto_indirect_reduce_fuel_batch,
solvers.reduceFuel_indirect_batch(device_ladder=True)).

Every solver call of a ladder is a call of lto_indirect_solve_batch_nd, and a trajectory's result does not depend on the rest of
its batch, so the device ladder must agree BITWISE with the round-based driver (one lto_indirect_solve_batch call per round):
same XC_all, defects, statuses, solver calls and last rho."""
import numpy as np
import pytest

from lowthrustopt_b200 import capi, solvers as S

pytestmark = pytest.mark.gpu
MU, DU, TU = capi.MU, capi.DU, capi.TU


@pytest.fixture(scope="module")
def gpu(lto):
    return S.GpuBackend(handle=lto)


@pytest.fixture(scope="module")
def demo_p1(gpu):
    """The demo pipeline (CRTBP_Multishoot_indirect_demo.jl:166-192) up to p = 1, rho = 1 solutions, for 4 costate seeds."""
    fx = S.demo_fixtures()
    XCg, t_TU, tau1, tau2, s0, sf = S.trajectory_stack_guess(fx[1], fx[3], backend=gpu)
    X_all = S.multiShoot_CRTBP_direct(XCg[:6].copy(), np.zeros((3, 30)), tau1, tau2, t_TU, np.zeros(3), np.zeros(3), MU, DU, TU, 30, 10, 1e3,
                                      2000.0, *fx, backend=gpu)[0]
    p1 = []
    for seed in (42, 43, 44, 45):
        rng = np.random.default_rng(seed)
        XC0 = np.vstack([X_all, 0.1 * rng.standard_normal((6, 30))])
        XC0[:6, 0] = s0[:6]; XC0[:6, -1] = sf[:6]
        XC0[:, 1:-1] += 1e-10 * rng.standard_normal((12, 28))
        XC, d, st = S.multiShoot_CRTBP_indirect(XC0, t_TU, MU, DU, TU, 30, 1e3, 10.0, False, False, 50, 2.0, 1.0, backend=gpu)
        assert st == 0
        XC, d, st = S.multiShoot_CRTBP_indirect(XC, t_TU, MU, DU, TU, 30, 1e3, 0.05, False, False, 30, 1.0, 1.0, backend=gpu)
        assert st == 0
        p1.append(XC)
    return t_TU, np.stack(p1)


@pytest.fixture(scope="module")
def starts14(oracle):
    from test_solvers_cpu import _guess14
    gs = [_guess14(oracle, 1e-2, seed) for seed in (3, 4, 5, 6)]
    return np.stack([g[0] for g in gs]), gs[0][1], gs[0][2]


class _Draws:
    """rng stand-in for _reduceFuel_steps: the given draws in order, counted."""

    def __init__(self, u):
        self.u, self.n = u, 0

    def random(self):
        self.n += 1
        return float(self.u[self.n - 1])


def _round_ladders(h, XC, t, r0, r1, draws, tl, max_iter, Isp=2000.0):
    """The round-based reference: _reduceFuel_steps per trajectory, each round's calls as one Handle.indirect_solve_batch.
    XC: (n_traj, n_nodes, m) rows.  Returns XC_all, defect, status, calls, rho_last, draws consumed, and each ladder's rho sequence."""
    T = XC.shape[0]
    rngs = [_Draws(draws[j]) for j in range(T)]
    gens = [S._reduceFuel_steps(XC[j].copy(), float(r0[j]), float(r1[j]), rngs[j]) for j in range(T)]
    req = {j: next(gens[j]) for j in range(T)}
    res, calls, rho_last, rhos = [None] * T, np.zeros(T, dtype=np.int32), np.zeros(T), [[] for _ in range(T)]
    p = capi.indirect_params(p=1.0, Isp=Isp)
    while req:
        idx = sorted(req)
        rho = np.array([req[j][1] for j in idx])
        r = h.indirect_solve_batch(np.stack([req[j][0] for j in idx]), t[idx], params=p, thrustLimit=tl[idx], rho=rho, max_iter=max_iter)
        for k, j in enumerate(idx):
            calls[j] += 1; rho_last[j] = rho[k]; rhos[j].append(rho[k])
            try:
                req[j] = gens[j].send((r["XC_all"][k].copy(), r["defect"][k].copy(), int(r["status_flag"][k])))
            except StopIteration as fin:
                res[j] = fin.value
                del req[j]
    return (np.stack([x[0] for x in res]), np.stack([x[1] for x in res]), np.array([x[2] for x in res], dtype=np.int32), calls, rho_last,
            np.array([g.n for g in rngs]), rhos)


def _device(h, XC, t, r0, r1, draws, tl, max_iter, Isp=2000.0):
    return h.indirect_reduce_fuel_batch(XC, t, r0, r1, draws, params=capi.indirect_params(p=1.0, Isp=Isp), thrustLimit=tl, max_iter=max_iter)


def _assert_same(d, ref):
    X, D, st, calls, rho_last = ref[:5]
    assert np.array_equal(d["status"], st), (d["status"], st)
    assert np.array_equal(d["calls"], calls), (d["calls"], calls)
    assert np.array_equal(d["rho_last"], rho_last)
    assert np.array_equal(d["XC_all"], X) and np.array_equal(d["defect"], D)


def _rows(p1):
    return np.ascontiguousarray(p1.transpose(0, 2, 1))


def test_device_ladder_matches_round_driver_demo12(gpu, demo_p1):
    t_TU, p1 = demo_p1
    T = p1.shape[0]
    tt = np.broadcast_to(t_TU, (T, 30)).copy()
    target = np.array([1e-2, 0.125, 0.05, 0.5]); tl = 0.05 * np.array([1.0, 1.1, 0.9, 1.0])
    Xr, dr, sr, rr = S.reduceFuel_indirect_batch(p1, tt, MU, DU, TU, 30, 1e3, tl, 1.0, target, backend=gpu,
                                                 rngs=[np.random.default_rng(j) for j in range(T)])
    Xd, dd, sd, rd = S.reduceFuel_indirect_batch(p1, tt, MU, DU, TU, 30, 1e3, tl, 1.0, target, backend=gpu,
                                                 rngs=[np.random.default_rng(j) for j in range(T)], device_ladder=True)
    assert np.all(sr == 0) and rr >= 2
    assert np.array_equal(Xd, Xr) and np.array_equal(dd, dr) and np.array_equal(sd, sr) and rd == rr
    draws = np.array([np.random.default_rng(j).random(100) for j in range(T)])
    r = _device(gpu.h, _rows(p1), tt, np.ones(T), target, draws, tl, 10)
    for j in range(T):
        log = []
        Xh, dh, sh = S.reduceFuel_indirect(p1[j], t_TU, MU, DU, TU, 30, 1e3, float(tl[j]), 1.0, float(target[j]), backend=gpu,
                                           rng=np.random.default_rng(j), log=log)
        assert sh == 0 and r["calls"][j] == len(log), (j, r["calls"][j], len(log))
    assert np.all(r["newton_iters"] > 0)
    assert np.array_equal(r["rho_last"], target)


def test_give_up_after_100_rungs(gpu, demo_p1):
    """max_iter = 0 from converged starts: the first call succeeds (0 iterations), every later call fails -> 100 back-off rungs."""
    t_TU, p1 = demo_p1
    T = p1.shape[0]
    tt = np.broadcast_to(t_TU, (T, 30)).copy(); tl = np.full(T, 0.05)
    r0, r1 = np.ones(T), np.full(T, 1e-2)
    draws = np.random.default_rng(7).random((T, 100))
    ref = _round_ladders(gpu.h, _rows(p1), tt, r0, r1, draws, tl, 0)
    d = _device(gpu.h, _rows(p1), tt, r0, r1, draws, tl, 0)
    assert np.all(ref[2] == 3) and np.all(ref[3] == 101) and np.all(ref[5] == 99)
    _assert_same(d, ref)
    assert np.all(d["newton_iters"] == 0)


def test_backoff_and_ramp_paths(gpu, demo_p1):
    t_TU, p1 = demo_p1
    T = p1.shape[0]
    tt = np.broadcast_to(t_TU, (T, 30)).copy(); tl = 0.05 * np.array([1.0, 1.2, 0.8, 1.0])
    draws = np.random.default_rng(11).random((T, 100))
    # max_iter = 2: halving steps that do not converge in 2 iterations back off
    r0, r1 = np.ones(T), np.array([1e-2, 0.05, 0.02, 0.1])
    ref = _round_ladders(gpu.h, _rows(p1), tt, r0, r1, draws, tl, 2)
    assert ref[5].max() >= 1
    _assert_same(_device(gpu.h, _rows(p1), tt, r0, r1, draws, tl, 2), ref)
    # starts converged at rho = 1, asked for at rho_current = 0.04 with max_iter = 2: the first call fails, the x5 ramp follows
    r0, r1 = np.full(T, 0.04), np.full(T, 0.02)
    ref = _round_ladders(gpu.h, _rows(p1), tt, r0, r1, draws, tl, 2)
    assert any(len(q) >= 2 and q[1] == min(0.04 * 5, 1.0) for q in ref[6])
    _assert_same(_device(gpu.h, _rows(p1), tt, r0, r1, draws, tl, 2), ref)


def test_device_ladder14_matches_round_driver(gpu, starts14):
    XS, t, tl = starts14
    T = 3
    conv = []
    for j in range(T):
        XC, d, st = S.multiShoot_CRTBP_indirect(XS[j], t, MU, DU, TU, 30, 1000.0, tl, False, False, 30, 1.0, 1e-2, backend=gpu)
        assert st == 0
        conv.append(XC)
    conv = np.stack(conv)
    tt = np.broadcast_to(t, (T, 30)).copy()
    out = [S.reduceFuel_indirect_batch(conv, tt, MU, DU, TU, 30, 1000.0, tl, 1e-2, 5e-3, backend=gpu,
                                       rngs=[np.random.default_rng(j) for j in range(T)], device_ladder=dl) for dl in (False, True)]
    (Xr, dr, sr, rr), (Xd, dd, sd, rd) = out
    assert Xd.shape == (T, 14, 30) and np.all(sr == 0)
    assert np.array_equal(Xd, Xr) and np.array_equal(dd, dr) and np.array_equal(sd, sr) and rd == rr


def test_independence_and_edge_cases(gpu, demo_p1):
    t_TU, p1 = demo_p1
    h = gpu.h
    T = p1.shape[0]
    X = _rows(p1); tt = np.broadcast_to(t_TU, (T, 30)).copy(); tl = 0.05 * np.array([1.0, 1.1, 0.9, 1.0])
    r0, r1 = np.ones(T), np.array([1e-2, 0.125, 0.05, 0.5])
    draws = np.random.default_rng(3).random((T, 100))
    full = _device(h, X, tt, r0, r1, draws, tl, 10)
    sub = [1, 3]
    part = _device(h, X[sub], tt[sub], r0[sub], r1[sub], draws[sub], tl[sub], 10)
    for k in full:
        assert np.array_equal(part[k], full[k][sub]), k
    # empty batch
    e = _device(h, np.zeros((0, 30, 12)), np.zeros((0, 30)), np.zeros(0), np.zeros(0), np.zeros((0, 100)), np.zeros(0), 10)
    assert e["XC_all"].shape == (0, 30, 12) and e["status"].shape == (0,) and e["defect"].shape == (0, 29, 12)
    # rho_target above rho_current: clamped, one call
    one = _device(h, X, tt, r0, np.full(T, 2.0), draws, tl, 10)
    assert np.all(one["calls"] == 1) and np.all(one["status"] == 0) and np.all(one["rho_last"] == 1.0)
    # a NaN interior costate: that ladder ends with status 2, its neighbours are those of a batch without it
    bad = X.copy(); bad[2, 10, 8] = np.nan
    rb = _device(h, bad, tt, r0, r1, draws, tl, 10)
    keep = [0, 1, 3]
    rk = _device(h, X[keep], tt[keep], r0[keep], r1[keep], draws[keep], tl[keep], 10)
    assert rb["status"][2] == 2
    for k in rb:
        assert np.array_equal(rb[k][keep], rk[k]), k
    # rho is only a homotopy parameter at p = 1
    with pytest.raises(capi.LtoError):
        h.indirect_reduce_fuel_batch(X, tt, r0, r1, draws, params=capi.indirect_params(p=2.0), thrustLimit=tl)


def test_multi_device_handle_reduce_fuel(lto, demo_p1):
    if capi.lib().lto_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    t_TU, p1 = demo_p1
    T = p1.shape[0]
    X = _rows(p1); tt = np.broadcast_to(t_TU, (T, 30)).copy(); tl = np.full(T, 0.05)
    r0, r1 = np.ones(T), np.array([1e-2, 0.125, 0.05, 0.5])
    draws = np.random.default_rng(5).random((T, 100))
    hm = capi.Handle([0, 1])
    try:
        a = _device(lto, X, tt, r0, r1, draws, tl, 10)
        b = _device(hm, X, tt, r0, r1, draws, tl, 10)
    finally:
        hm.close()
    for k in a:
        assert np.array_equal(a[k], b[k]), k
