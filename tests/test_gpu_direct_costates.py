"""GPU: costates of direct solutions (lto_direct_costates_batch, solvers.direct_costates) and the sweep's multiplier-based start
(solvers.indirect_transfer_sweep(start="direct")).

What pins the device numbers:
  * the dense KKT system of _qp_direct's formulation and the host map solvers._direct_costate_map, on the same K1 blocks;
  * K7's own primal step: du_max is max |u_update| of lto_direct_qp on the same inputs;
  * the KKT identities (u-stationarity, equal one-sided interior costates) on the device output;
  * a full p = 2 indirect solve from the mapped start, against the seeded chain's stage-2 solution."""
import numpy as np
import pytest

from lowthrustopt_b200 import capi, solvers as S
from test_direct_costates_cpu import identities, kkt_multipliers

pytestmark = pytest.mark.gpu
MU, DU, TU = capi.MU, capi.DU, capi.TU
DEMO = (0.75, 10.0, 10.0)


@pytest.fixture(scope="module")
def gpu(lto):
    return S.GpuBackend(handle=lto)


@pytest.fixture(scope="module")
def perturbed(lto, gpu):
    """5 perturbed demo trajectories, as test_direct_qp_vs_host_kkt builds them, with their K1 blocks and end-state right-hand sides."""
    fx = S.demo_fixtures()
    XC, t_TU, tau1, tau2, s0, sf = S.trajectory_stack_guess(fx[1], fx[3], backend=gpu)
    N, T = 30, 5
    rng = np.random.default_rng(8)
    state_0, state_f = S.interpEndStates(tau1, tau2, *fx, MU)
    X = np.stack([(XC[:6] + 1e-3 * rng.standard_normal((6, N))).T for _ in range(T)])
    U = np.stack([(0.02 * rng.standard_normal((3, N))).T for _ in range(T)])
    t = np.broadcast_to(t_TU, (T, N)).copy()
    s0b, sfb = np.tile(state_0, (T, 1)), np.tile(state_f, (T, 1))
    r = lto.direct_traj(X, U, t, nsteps=10, params=capi.direct_params(Isp=2000.0), jac=True)
    jac = r["jac"].reshape(T, N - 1, 18, 6); dfc = r["defect"].reshape(T, N - 1, 6)
    return dict(X=X, U=U, t=t, s0=s0b, sf=sfb, jac=jac, defect=dfc, b0=s0b - X[:, 0], bf=sfb - X[:, -1])


def _rel(a, b):
    return np.abs(a - b).max() / np.abs(b).max()


def test_multipliers_and_costates_match_the_dense_kkt_and_the_host_map(lto, perturbed):
    P = perturbed
    c = lto.direct_costates_batch(P["X"], P["U"], P["t"], P["s0"], P["sf"])
    assert (c["status"] == 0).all()
    assert np.array_equal(c["XC_all"][:, :, :6], P["X"])
    for j in range(5):
        blocks = P["jac"][j].transpose(0, 2, 1)
        _, _, lam = kkt_multipliers(blocks, P["defect"][j], P["X"][j].T, P["U"][j].T, P["t"][j], P["s0"][j], P["sf"][j])
        cs = S._direct_costate_map(blocks, lam, 1e3, DU, TU)
        em, ec = _rel(c["multipliers"][j], lam), _rel(c["XC_all"][j, :, 6:].T, cs)
        print("\n[dual] row %d: multipliers %.1e costates %.1e (relative)" % (j, em, ec), end="")
        assert em <= 1e-10 and ec <= 1e-10, (j, em, ec)


def test_du_max_is_the_primal_step_of_lto_direct_qp(lto, perturbed):
    P = perturbed
    c = lto.direct_costates_batch(P["X"], P["U"], P["t"], P["s0"], P["sf"])
    _, uu, st = lto.direct_qp(P["jac"], P["defect"], P["U"], P["t"], P["b0"], P["bf"])
    assert (st == 0).all()
    ref = np.abs(uu).max(axis=(1, 2))
    print("\n[dual] du_max %s, bitwise equal to lto_direct_qp: %s" % (c["du_max"], np.array_equal(c["du_max"], ref)))
    np.testing.assert_allclose(c["du_max"], ref, rtol=1e-14, atol=0)


@pytest.fixture(scope="module")
def grid64(gpu):
    """The demo's converged direct solution (row 0) and 63 more rows of a seeded grid, solved by the batched direct sweep."""
    rng = np.random.default_rng(64)
    tau1 = np.concatenate([[DEMO[0]], rng.uniform(0.0, 1.0, 63)])
    tof = np.concatenate([[DEMO[1:]], rng.uniform(8.0, 12.0, (63, 2))])
    fx = S.demo_fixtures()
    return S.direct_transfer_sweep(fx[1], fx[3], tau1, tof[:, 0], tof[:, 1], backend=gpu)


def test_kkt_identities_hold_on_the_device_output(lto, gpu, grid64):
    d = grid64
    T = d["X_all"].shape[0]
    X, U = d["X_all"].transpose(0, 2, 1).copy(), d["u_all"].transpose(0, 2, 1).copy()
    c = S.direct_costates(d["X_all"], d["u_all"], d["t_TU"], d["state_0"], d["state_f"], backend=gpu)
    r = lto.direct_traj(X, U, d["t_TU"], nsteps=10, params=capi.direct_params(Isp=2000.0), jac=True)
    jac = r["jac"].reshape(T, 29, 18, 6)
    _, du, st = lto.direct_qp(jac, r["defect"].reshape(T, 29, 6), U, d["t_TU"], d["state_0"] - X[:, 0], d["state_f"] - X[:, -1])
    assert d["converged"][0] and (c["status"] == 0).all() and (st == 0).all()
    worst = np.zeros(2)
    for j in range(T):
        ra, rb = identities(jac[j].transpose(0, 2, 1), c["multipliers"][j].T, U[j], du[j], d["t_TU"][j])
        worst = np.maximum(worst, [ra, rb])
        assert ra <= 1e-10 and rb <= 1e-10, (j, ra, rb)
    print("\n[dual] 64 rows: u-stationarity %.1e, interior one-sided costates %.1e; du_max %.1e N at most" % (*worst, c["du_max"].max()))


def test_full_p2_solve_from_the_mapped_start_matches_the_seeded_chain(gpu):
    fx = S.demo_fixtures()
    d = S.direct_transfer_sweep(fx[1], fx[3], *DEMO, backend=gpu)
    t = d["t_TU"]
    # the seeded chain of test_gpu_transfer_cost.py's fixture, seed 42: adjoints-only, then full p = 2 at 10 N
    rng = np.random.default_rng(42)
    XC = np.vstack([d["X_all"][0], 0.1 * rng.standard_normal((6, 30))])
    XC[:6, 0] = d["state_0"][0]; XC[:6, -1] = d["state_f"][0]
    XC[:, 1:-1] += 1e-10 * rng.standard_normal((12, 28))
    XC, _, st, _ = S.multiShoot_CRTBP_indirect_batch(XC[None], t, MU, DU, TU, 30, 1e3, 10.0, True, 10, 2.0, 1.0, backend=gpu)
    seeded, _, st, it_s = S.multiShoot_CRTBP_indirect_batch(XC, t, MU, DU, TU, 30, 1e3, 10.0, False, 50, 2.0, 1.0, backend=gpu)
    assert st[0] == 0
    c = S.direct_costates(d["X_all"], d["u_all"], t, d["state_0"], d["state_f"], backend=gpu)
    XM = c["XC_all"].copy()
    XM[:, :6, 0] = d["state_0"]; XM[:, :6, -1] = d["state_f"]
    mapped, _, st, it_m = S.multiShoot_CRTBP_indirect_batch(XM, t, MU, DU, TU, 30, 1e3, 10.0, False, 50, 2.0, 1.0, backend=gpu)
    dist = np.abs(mapped - seeded).max() / max(1.0, np.abs(seeded).max())
    start = np.abs(XM[0, 6:] - seeded[0, 6:]).max() / np.abs(seeded[0, 6:]).max()
    print("\n[dual] demo row: mapped start %.2e from the p = 2 costates; p = 2 solve from it: status %d, %d iterations (seeded chain: %d), "
          "solutions %.1e apart" % (start, st[0], it_m[0], it_s[0], dist))
    assert st[0] == 0 and dist <= 1e-8


GRID_TAU1 = np.repeat([0.65, 0.7, 0.75, 0.8], 4)
GRID_TOF = np.tile([[10.0, 10.0], [9.0, 11.0], [11.0, 9.0], [10.0, 12.0]], (4, 1))
GRID_SEEDS = np.arange(34, 50)
KEYS = ("XC_all", "stage_failed", "status", "rho_last", "dv", "energy", "energy_p2", "cost")


def test_direct_start_sweep_rows_equal_single_row_sweeps(gpu):
    fx = S.demo_fixtures()
    sw = S.indirect_transfer_sweep(fx[1], fx[3], GRID_TAU1, GRID_TOF[:, 0], GRID_TOF[:, 1], seeds=GRID_SEEDS, backend=gpu, start="direct")
    print("\n[sweep direct] stage_failed %s" % sw["stage_failed"].tolist())
    for j in range(16):
        one = S.indirect_transfer_sweep(fx[1], fx[3], GRID_TAU1[j:j + 1], GRID_TOF[j:j + 1, 0], GRID_TOF[j:j + 1, 1], seeds=GRID_SEEDS[j:j + 1],
                                        backend=gpu, start="direct")
        for k in KEYS:
            assert np.array_equal(one[k][0], sw[k][j], equal_nan=True), (j, k)


def _old_seeded_sweep(fx, be, tau1, tof1, tof2, seeds, thrustLimit=0.05, rho_target=1e-4, mass=1e3):
    """indirect_transfer_sweep as it was before the start keyword, stage by stage."""
    d = S.direct_transfer_sweep(fx[1], fx[3], tau1, tof1, tof2, backend=be)
    t = d["t_TU"]; T, N = t.shape
    XC = np.empty((T, 12, N))
    for j in range(T):
        rng = np.random.default_rng(seeds[j])
        XC[j] = np.vstack([d["X_all"][j], 0.1 * rng.standard_normal((6, N))])
        XC[j, :6, 0] = d["state_0"][j]; XC[j, :6, -1] = d["state_f"][j]
        XC[j, :, 1:-1] += 1e-10 * rng.standard_normal((12, N - 2))
    failed = np.zeros(T, dtype=np.int32)
    for stage, tl, p, it, adj, fail_on in ((1, 10.0, 2.0, 10, True, (2,)), (2, 10.0, 2.0, 50, False, (1, 2)), (3, thrustLimit, 1.0, 30, False, (1, 2))):
        idx = np.flatnonzero(failed == 0)
        Xn, _, st, _ = S.multiShoot_CRTBP_indirect_batch(XC[idx], t[idx], MU, DU, TU, N, mass, tl, adj, it, p, 1.0, backend=be)
        XC[idx] = Xn
        failed[idx[np.isin(st, fail_on)]] = stage
    idx = np.flatnonzero(failed == 0)
    draws = np.array([np.random.default_rng(seeds[j]).random(100) for j in idx]).reshape(idx.size, 100)
    r = be.indirect_reduce_fuel_batch(np.ascontiguousarray(XC[idx].transpose(0, 2, 1)), t[idx], (MU, DU, TU, thrustLimit, mass, 1.0, 1.0, 1.0),
                                      np.ones(idx.size), np.full(idx.size, rho_target), draws, thrustLimit=np.full(idx.size, thrustLimit), max_iter=10)
    XC[idx] = r["XC_all"].transpose(0, 2, 1)
    failed[idx[r["status"] != 0]] = 4
    return XC, failed


def test_seeded_start_is_unchanged(gpu):
    fx = S.demo_fixtures()
    sw = S.indirect_transfer_sweep(fx[1], fx[3], GRID_TAU1, GRID_TOF[:, 0], GRID_TOF[:, 1], seeds=GRID_SEEDS, backend=gpu, start="seeded")
    XC, failed = _old_seeded_sweep(fx, gpu, GRID_TAU1, GRID_TOF[:, 0], GRID_TOF[:, 1], GRID_SEEDS)
    assert np.array_equal(sw["stage_failed"], failed)
    assert np.array_equal(sw["XC_all"], XC, equal_nan=True)


def test_rows_do_not_depend_on_their_batch(lto, grid64):
    d = grid64
    X, U, t = d["X_all"].transpose(0, 2, 1).copy(), d["u_all"].transpose(0, 2, 1).copy(), d["t_TU"]
    s0, sf = d["state_0"], d["state_f"]
    full = lto.direct_costates_batch(X, U, t, s0, sf)
    for j in (0, 17, 63):
        one = lto.direct_costates_batch(X[j:j + 1], U[j:j + 1], t[j:j + 1], s0[j:j + 1], sf[j:j + 1])
        for k in full:
            assert np.array_equal(one[k][0], full[k][j]), (j, k)
    bad = X.copy(); bad[17, 9, 2] = np.nan
    nan = lto.direct_costates_batch(bad, U, t, s0, sf)
    assert nan["status"][17] == 1 and np.isnan(nan["XC_all"][17, :, 6:]).all()          # LTO_ST_NAN
    keep = np.arange(64) != 17
    for k in full:
        assert np.array_equal(nan[k][keep], full[k][keep]), k
    empty = lto.direct_costates_batch(np.zeros((0, 30, 6)), np.zeros((0, 30, 3)), np.zeros((0, 30)), np.zeros((0, 6)), np.zeros((0, 6)))
    assert empty["XC_all"].shape == (0, 30, 12) and empty["status"].shape == (0,)


def test_library_refuses_what_the_wrapper_would(lto):
    import ctypes as C
    L = capi.lib()
    p = capi.direct_params()
    X = np.zeros((2, 3, 6)); U = np.zeros((2, 3, 3)); s = np.zeros((2, 6)); XC = np.zeros((2, 3, 12))
    t = np.array([[0.0, 0.5, 1.0], [0.0, 0.5, 0.5]])
    args = lambda tt: (lto._h, C.addressof(p), 2, 3, 10, X.ctypes.data, U.ctypes.data, tt.ctypes.data, s.ctypes.data, s.ctypes.data,
                       XC.ctypes.data, None, None, None)
    assert L.lto_direct_costates_batch(*args(t)) == -2 and b"trajectory 1" in L.lto_last_error(lto._h)
    t[1, 2] = 1.0; t[0, 1] = np.nan
    assert L.lto_direct_costates_batch(*args(t)) == -2 and b"trajectory 0" in L.lto_last_error(lto._h)
    t[0, 1] = 0.5
    p.mode = capi.LTO_ADAPTIVE
    assert L.lto_direct_costates_batch(*args(t)) == -2


def test_two_device_handle_splits_whole_trajectories(lto, grid64):
    if capi.lib().lto_device_count() < 2:
        pytest.skip("needs two GPUs")
    d = grid64
    X, U = d["X_all"].transpose(0, 2, 1).copy(), d["u_all"].transpose(0, 2, 1).copy()
    hm = capi.Handle([0, 1])
    try:
        a = lto.direct_costates_batch(X[:33], U[:33], d["t_TU"][:33], d["state_0"][:33], d["state_f"][:33])
        b = hm.direct_costates_batch(X[:33], U[:33], d["t_TU"][:33], d["state_0"][:33], d["state_f"][:33])
        for k in a:
            assert np.array_equal(a[k], b[k]), k
    finally:
        hm.close()
