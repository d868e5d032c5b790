"""GPU: the device-side Newton update and the batched indirect solver on the 14-dim system [r v m | lr lv lm] (state + costate + mass,
BASELINE configs[1]), and the 12-dim path through the dimension-taking entry points.

  * lto_indirect_newton_nd(14, ...)  vs  the host loop's least-squares step on the assembled band (solvers._band_indirect with the
    7-element pins of solvers._end_pins(7)), both modes.
  * lto_indirect_solve_batch_nd(14, ...)  vs  solvers.multiShoot_CRTBP_indirect on 14 rows run once per trajectory (GPU propagation,
    host lstsq): same status flags and iteration counts, XC_all within 1e-8, mass within 1e-9 relative (north_star).
  * ndim = 12 through the new entry points is bit-identical to the existing ones.
"""
import ctypes as C

import numpy as np
import pytest

from lowthrustopt_b200 import capi, solvers as S, synthetic

pytestmark = pytest.mark.gpu
MU, DU, TU = capi.MU, capi.DU, capi.TU
TOL_TRAJ = 1e-8
TOL_MASS = 1e-9
PIN_FIRST = list(range(7))                 # r, v, m of the first node
PIN_LAST = list(range(6)) + [13]           # r, v, lm of the last node (the final mass is free)


def _lstsq_update(phi_rc, d, adjoints_only, nstate):
    """The host loop's step: phi_rc (N-1, m, m) [row, col], d (N-1, m) -> xc_update (N, m)."""
    N = phi_rc.shape[0] + 1
    m = 2 * nstate
    J = S._band_indirect(phi_rc, nstate, N)
    keep = np.ones(N * m, dtype=bool)
    if adjoints_only:                                                     # the state columns of nodes 0..N-2 (:169-178)
        for i in range(N - 1):
            keep[i * m:i * m + nstate] = False
    Jk = J[:, keep]
    live = np.any(Jk != 0.0, axis=0)
    sol = np.zeros(Jk.shape[1])
    sol[live] = -np.linalg.lstsq(Jk[:, live], d.ravel(), rcond=None)[0]
    full = np.zeros(N * m)
    full[keep] = sol
    return full.reshape(N, m)


def _blocks14(lto, n_traj, n_seg, seed):
    """K3-14 blocks and defects of a 14-dim continuation slab: phi (n_traj, n_seg, 14, 14) [.., col, row], d (n_traj, n_seg, 14)."""
    c = synthetic.continuation_batch(n_traj=n_traj, n_seg_per_traj=n_seg, ndim=14, seed=seed)
    r = lto.indirect_traj(c["XC_all"], c["t_TU"], params=capi.indirect_params(p=1.0, rho=1.0, thrustLimit=0.05), thrustLimit=c["thrustLimit"])
    return r["phi"].reshape(n_traj, n_seg, 14, 14), r["defect"].reshape(n_traj, n_seg, 14)


@pytest.mark.parametrize("n_traj,n_seg", [(9, 29), (5, 200), (3, 1), (2, 2)])
@pytest.mark.parametrize("adjoints_only", [False, True])
def test_newton14_update_vs_least_squares(lto, n_traj, n_seg, adjoints_only):
    phi, d = _blocks14(lto, n_traj, n_seg, seed=11 + n_seg)
    upd, status = lto.indirect_newton(phi, d, adjoints_only)
    assert upd.shape == (n_traj, n_seg + 1, 14) and np.all(status == 0)
    for j in range(n_traj):
        ref = _lstsq_update(phi[j].transpose(0, 2, 1), d[j], adjoints_only, 7)
        scale = max(1.0, np.abs(ref).max())
        assert np.abs(upd[j] - ref).max() <= 1e-9 * scale, (j, np.abs(upd[j] - ref).max(), scale)
    # structurally empty columns get exact zeros
    if adjoints_only:
        assert np.all(upd[:, :-1, :7] == 0.0)
    else:
        assert np.all(upd[:, 0, PIN_FIRST] == 0.0)
    assert np.all(upd[:, -1, PIN_LAST] == 0.0)
    assert np.any(upd[:, -1, 6] != 0.0)                                   # the final mass is an unknown in both modes


@pytest.mark.parametrize("adjoints_only", [False, True])
def test_newton14_resolve_reuses_the_factorisation(lto, adjoints_only):
    import torch
    n_traj, n_seg = 7, 200
    phi_h, d_h = _blocks14(lto, n_traj, n_seg, seed=5)
    dev = torch.device("cuda", 0)
    phi = torch.from_numpy(np.ascontiguousarray(phi_h)).to(dev); d1 = torch.from_numpy(np.ascontiguousarray(d_h)).to(dev)
    d2 = torch.from_numpy(np.random.default_rng(3).standard_normal(d_h.shape) * 1e-3).to(dev)
    u1 = torch.empty((n_traj, n_seg + 1, 14), dtype=torch.float64, device=dev); u2 = torch.empty_like(u1); u2b = torch.empty_like(u1)
    st = torch.zeros(n_traj, dtype=torch.int32, device=dev)
    lto.indirect_newton_dev(n_traj, n_seg + 1, adjoints_only, phi.data_ptr(), d1.data_ptr(), u1.data_ptr(), ndim=14)
    lto.indirect_newton_resolve_dev(n_traj, n_seg + 1, adjoints_only, d2.data_ptr(), u2.data_ptr(), st.data_ptr(), ndim=14)
    with pytest.raises(capi.LtoError):                                    # same shape and mode, other dimension: not the factorisation held
        lto.indirect_newton_resolve_dev(n_traj, n_seg + 1, adjoints_only, d2.data_ptr(), u2b.data_ptr(), ndim=12)
    lto.indirect_newton_dev(n_traj, n_seg + 1, adjoints_only, phi.data_ptr(), d2.data_ptr(), u2b.data_ptr(), ndim=14)   # afresh
    lto.sync()
    assert int(st.abs().max()) == 0
    a, b = u2.cpu().numpy(), u2b.cpu().numpy()
    assert np.abs(a - b).max() <= 1e-11 * max(1.0, np.abs(b).max())
    ref = _lstsq_update(phi_h[0].transpose(0, 2, 1), d2.cpu().numpy()[0], adjoints_only, 7)
    assert np.abs(a[0] - ref).max() <= 1e-9 * max(1.0, np.abs(ref).max())
    # and the other way round: a 12-dim factorisation of the same n_traj / n_nodes does not serve a 14-dim resolve
    phi12 = torch.zeros((n_traj, n_seg, 12, 12), dtype=torch.float64, device=dev); phi12[:] = torch.eye(12, dtype=torch.float64, device=dev)
    d12 = torch.zeros((n_traj, n_seg, 12), dtype=torch.float64, device=dev); u12 = torch.empty((n_traj, n_seg + 1, 12), dtype=torch.float64, device=dev)
    lto.indirect_newton_dev(n_traj, n_seg + 1, adjoints_only, phi12.data_ptr(), d12.data_ptr(), u12.data_ptr())
    with pytest.raises(capi.LtoError):
        lto.indirect_newton_resolve_dev(n_traj, n_seg + 1, adjoints_only, d2.data_ptr(), u2.data_ptr(), ndim=14)
    lto.sync()


def test_newton14_flags_singular_systems(lto):
    phi = np.zeros((2, 4, 14, 14)); d = np.ones((2, 4, 14))
    phi[1] = np.eye(14)                                                   # trajectory 0: Phi = 0 (singular)
    for r in range(7):
        phi[1, :, 7 + r, r] = 1.0                                         # trajectory 1: Phi = [[I, I], [0, I]] ([col, row] storage): well posed
    upd, status = lto.indirect_newton(phi, d, False)
    assert status[0] == 1 and status[1] == 0                              # LTO_ST_NAN = 1
    assert np.all(np.isfinite(upd[1]))


def _u64(a):
    return np.ascontiguousarray(a).view(np.uint64)


@pytest.mark.parametrize("adjoints_only", [False, True])
def test_ndim12_entry_points_are_bit_identical(lto, adjoints_only):
    L = capi.lib()
    c = synthetic.continuation_batch(n_traj=6, n_seg_per_traj=29, ndim=12, seed=7)
    r = lto.indirect_traj(c["XC_all"], c["t_TU"], params=capi.indirect_params(p=2.0, thrustLimit=10.0))
    phi = np.ascontiguousarray(r["phi"]); d = np.ascontiguousarray(r["defect"])
    ua, ub = np.empty((6, 30, 12)), np.empty((6, 30, 12))
    sa, sb = np.empty(6, np.int32), np.empty(6, np.int32)
    P = lambda a: a.ctypes.data
    lto._ck(L.lto_indirect_newton(lto._h, 6, 30, int(adjoints_only), P(phi), P(d), P(ua), P(sa)))
    lto._ck(L.lto_indirect_newton_nd(lto._h, 12, 6, 30, int(adjoints_only), P(phi), P(d), P(ub), P(sb)))
    assert np.array_equal(_u64(ua), _u64(ub)) and np.array_equal(sa, sb)
    with pytest.raises(capi.LtoError):
        lto._ck(L.lto_indirect_newton_nd(lto._h, 13, 6, 30, int(adjoints_only), P(phi), P(d), P(ub), P(sb)))


def test_ndim12_solve_batch_is_bit_identical(lto):
    """lto_indirect_solve_batch_nd(12, ...) on the input of test_gpu_newton.py::test_solve_batch_continuation_slab."""
    L = capi.lib()
    c = synthetic.continuation_batch(n_traj=16, n_seg_per_traj=200, ndim=12)
    XC = c["XC_all"].copy(); XC[:, :, 6:] *= 0.01
    t = np.ascontiguousarray(c["t_TU"])
    p = capi.indirect_params(p=2.0, thrustLimit=10.0)
    out = []
    for nd_call in (False, True):
        X = XC.copy(); D = np.empty((16, 200, 12)); F = np.empty(16, np.int32); I = np.empty(16, np.int32); E = np.empty(16)
        args = (16, 201, 12, 0, X.ctypes.data, t.ctypes.data, None, None, D.ctypes.data, F.ctypes.data, I.ctypes.data, E.ctypes.data)
        if nd_call:
            lto._ck(L.lto_indirect_solve_batch_nd(lto._h, C.addressof(p), 12, *args))
        else:
            lto._ck(L.lto_indirect_solve_batch(lto._h, C.addressof(p), *args))
        out.append((X, D, F, I, E))
    for a, b in zip(*out):
        assert np.array_equal(_u64(a) if a.dtype == np.float64 else a, _u64(b) if b.dtype == np.float64 else b)
    assert (out[0][2] == 0).sum() >= 8


# ------------------------------------------------------------------ the solvers on 14 rows
@pytest.fixture(scope="module")
def gpu(lto):
    return S.GpuBackend(handle=lto)


@pytest.fixture(scope="module")
def starts14(oracle):
    from test_solvers_cpu import _guess14
    gs = [_guess14(oracle, 1e-2, seed) for seed in (3, 4, 5, 6)]
    return np.stack([g[0] for g in gs]), gs[0][1], gs[0][2]


def _rel(a, b):
    return float((np.abs(a - b) / np.maximum(1.0, np.abs(b))).max())


def test_host_loop_with_device_newton14_matches_host_lstsq(gpu, starts14):
    XS, t, tl = starts14
    res = []
    for dn in (False, True):
        log = []
        XC, d, st = S.multiShoot_CRTBP_indirect(XS[0].copy(), t, MU, DU, TU, 30, 1000.0, tl, False, False, 30, 1.0, 1e-2, backend=gpu, log=log,
                                                device_newton=dn)
        res.append((XC, st, len(log)))
    (Xh, sh, nh), (Xd, sd, nd) = res
    print("host loop, 14-dim: device update vs host lstsq: iters %d / %d, XC rel %.3g, mass rel %.3g"
          % (nh, nd, _rel(Xd, Xh), np.abs(Xd[6] / Xh[6] - 1).max()))
    assert sh == sd == 0 and nh == nd
    assert _rel(Xd, Xh) < TOL_TRAJ
    assert np.abs(Xd[6] / Xh[6] - 1.0).max() < TOL_MASS and abs(Xd[6, -1] / Xh[6, -1] - 1.0) < TOL_MASS


@pytest.mark.parametrize("adjoints_only,max_iters", [(False, (30, 2)), (True, (10,))])
def test_solve_batch14_matches_per_trajectory_host_loops(gpu, starts14, adjoints_only, max_iters):
    XS, t, tl0 = starts14
    T = XS.shape[0]
    rho = np.array([1e-2, 1.2e-2, 1e-2, 8e-3]); tl = tl0 * np.array([1.0, 1.0, 1.1, 1.0])
    tt = np.broadcast_to(t, (T, 30)).copy()
    for max_iter in max_iters:
        Xb, db, fb, ib = S.multiShoot_CRTBP_indirect_batch(XS, tt, MU, DU, TU, 30, 1000.0, tl, adjoints_only, max_iter, 1.0, rho, backend=gpu)
        assert Xb.shape == XS.shape and db.shape == (T, 14, 29)
        for j in range(T):
            log = []
            Xh, dh, fh = S.multiShoot_CRTBP_indirect(XS[j], t, MU, DU, TU, 30, 1000.0, float(tl[j]), False, adjoints_only, max_iter, 1.0,
                                                     float(rho[j]), backend=gpu, log=log)
            print("batch14 adj=%s max_iter=%d traj %d: flag %d/%d iters %d/%d XC rel %.3g mass rel %.3g"
                  % (adjoints_only, max_iter, j, fb[j], fh, ib[j], len(log), _rel(Xb[j], Xh), np.abs(Xb[j, 6] / Xh[6] - 1).max()))
            assert fb[j] == fh and ib[j] == len(log), (max_iter, j, fb[j], fh, ib[j], len(log))
            assert _rel(Xb[j], Xh) < TOL_TRAJ, (max_iter, j, _rel(Xb[j], Xh))
            assert np.abs(Xb[j, 6] / Xh[6] - 1.0).max() < TOL_MASS
            if fh == 0:
                assert np.abs(db[j]).max() <= 1e-10
            assert np.array_equal(Xb[j, PIN_FIRST, 0], XS[j, PIN_FIRST, 0]) and np.array_equal(Xb[j, PIN_LAST, -1], XS[j, PIN_LAST, -1])
            assert Xb[j, 6, -1] != XS[j, 6, -1]                          # the final mass was solved for


def test_continuation_ladder14_matches_per_trajectory(gpu, starts14):
    """reduceFuel_indirect_batch on 14 rows (rho 1e-2 -> 5e-3) against reduceFuel_indirect run once per trajectory."""
    XS, t, tl = starts14
    T = 3
    conv = []
    for j in range(T):
        XC, d, st = S.multiShoot_CRTBP_indirect(XS[j], t, MU, DU, TU, 30, 1000.0, tl, False, False, 30, 1.0, 1e-2, backend=gpu)
        assert st == 0
        conv.append(XC)
    conv = np.stack(conv)
    tt = np.broadcast_to(t, (T, 30)).copy()
    Xb, db, sb, rounds = S.reduceFuel_indirect_batch(conv, tt, MU, DU, TU, 30, 1000.0, tl, 1e-2, 5e-3, backend=gpu,
                                                     rngs=[np.random.default_rng(j) for j in range(T)])
    assert Xb.shape == (T, 14, 30)
    for j in range(T):
        Xh, dh, sh = S.reduceFuel_indirect(conv[j], t, MU, DU, TU, 30, 1000.0, tl, 1e-2, 5e-3, backend=gpu, rng=np.random.default_rng(j))
        print("ladder14 traj %d: status %d/%d XC rel %.3g" % (j, sb[j], sh, _rel(Xb[j], Xh)))
        assert sb[j] == sh
        assert _rel(Xb[j], Xh) < TOL_TRAJ, (j, _rel(Xb[j], Xh))


def test_solve_batch14_continuation_slab(lto):
    c = synthetic.continuation_batch(n_traj=16, n_seg_per_traj=200, ndim=14)
    XC = c["XC_all"].copy(); XC[:, :, 7:] *= 0.01                         # small costates: near-ballistic start
    r = lto.indirect_solve_batch(XC, c["t_TU"], params=capi.indirect_params(p=2.0, thrustLimit=10.0), max_iter=12)
    f = r["status_flag"]; ok = f == 0
    print("slab14: %d of 16 converged, flags %s, iters %s" % (ok.sum(), f.tolist(), r["iters"].tolist()))
    assert np.all(ok | (f == 1) | (f == 2))
    assert np.all(r["er"][ok] <= 1e-10)
    assert np.array_equal(r["XC_all"][:, 0, PIN_FIRST], XC[:, 0, PIN_FIRST]) and np.array_equal(r["XC_all"][:, -1, PIN_LAST], XC[:, -1, PIN_LAST])
    for j in np.nonzero(ok)[0]:
        assert np.all(np.diff(r["XC_all"][j, :, 6]) <= 1e-9), j           # thrusting only burns mass


def test_solve_batch14_edge_cases(lto, gpu, starts14):
    p = capi.indirect_params(p=2.0, thrustLimit=10.0)
    c = synthetic.continuation_batch(n_traj=3, n_seg_per_traj=200, ndim=14)
    c = dict(XC_all=c["XC_all"][:, :2].copy(), t_TU=c["t_TU"][:, :2].copy())         # two nodes: one (short) segment per trajectory
    r = lto.indirect_solve_batch(c["XC_all"], c["t_TU"], params=p, max_iter=0)
    assert np.all(r["status_flag"] == 1) and np.all(r["iters"] == 0) and np.array_equal(r["XC_all"], c["XC_all"])
    r = lto.indirect_solve_batch(c["XC_all"], c["t_TU"], params=p, max_iter=20)
    print("two-node 14-dim batch: flags %s er %s" % (r["status_flag"].tolist(), r["er"].tolist()))
    assert np.all(r["status_flag"] == 0) and np.all(r["er"] <= 1e-10)
    assert np.array_equal(r["XC_all"][:, 0, PIN_FIRST], c["XC_all"][:, 0, PIN_FIRST])
    assert np.array_equal(r["XC_all"][:, -1, PIN_LAST], c["XC_all"][:, -1, PIN_LAST])
    r = lto.indirect_solve_batch(np.zeros((0, 5, 14)), np.zeros((0, 5)), params=p)  # empty batch
    assert r["XC_all"].shape == (0, 5, 14) and r["status_flag"].shape == (0,)
    with pytest.raises(capi.LtoError):
        lto.indirect_solve_batch(np.zeros((1, 1, 14)), np.zeros((1, 1)), params=p)  # n_nodes < 2
    # a NaN in an interior costate of one trajectory: flag 2, its neighbours still converge
    XS, t, tl = starts14
    bad = XS[:3].copy(); bad[1, 9, 7] = np.nan                                        # lr_z of node 7 ([trajectory, component, node])
    Xb, db, fb, ib = S.multiShoot_CRTBP_indirect_batch(bad, np.broadcast_to(t, (3, 30)).copy(), MU, DU, TU, 30, 1000.0, tl, False, 30, 1.0,
                                                       1e-2, backend=gpu)
    assert fb[1] == 2 and fb[0] == 0 and fb[2] == 0, fb
    # ndim 13 is refused by the C entry point
    L = capi.lib()
    X = np.zeros((1, 5, 13)); tt = np.tile(np.linspace(0, 0.4, 5), (1, 1))
    with pytest.raises(capi.LtoError):
        lto._ck(L.lto_indirect_solve_batch_nd(lto._h, C.addressof(p), 13, 1, 5, 3, 0, X.ctypes.data, tt.ctypes.data, None, None, None, None,
                                              None, None))


def test_multi_device_handle_solve_batch14(lto):
    ndev = capi.lib().lto_device_count()
    if ndev < 2:
        pytest.skip("needs 2 GPUs")
    hm = capi.Handle([0, 1])
    c = synthetic.continuation_batch(n_traj=11, n_seg_per_traj=200, ndim=14)
    XC = c["XC_all"].copy(); XC[:, :, 7:] *= 0.01
    p = capi.indirect_params(p=2.0, thrustLimit=10.0)
    s1 = lto.indirect_solve_batch(XC, c["t_TU"], params=p, max_iter=8)
    sm = hm.indirect_solve_batch(XC, c["t_TU"], params=p, max_iter=8)
    assert np.array_equal(s1["status_flag"], sm["status_flag"]) and np.array_equal(s1["iters"], sm["iters"])
    assert np.abs(s1["XC_all"] - sm["XC_all"]).max() < 1e-11
    tt1 = lto.indirect_traj(XC, c["t_TU"], params=p)
    u1, st1 = lto.indirect_newton(tt1["phi"].reshape(11, 200, 14, 14), tt1["defect"].reshape(11, 200, 14))
    um, stm = hm.indirect_newton(tt1["phi"].reshape(11, 200, 14, 14), tt1["defect"].reshape(11, 200, 14))
    assert np.array_equal(u1, um) and np.array_equal(st1, stm)
    hm.close()
