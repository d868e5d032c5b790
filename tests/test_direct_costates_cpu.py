"""CPU-side checks of the direct solution's costates (lto_direct_costates_batch, solvers.direct_costates) and of the sweep's multiplier-based
start (solvers.indirect_transfer_sweep(start="direct")): the sm_100a build of the dual kernel, wrapper validation, the sign and scale of the
multiplier -> costate map on the CPU oracle, and the sweep's stage gating against a fake backend (no GPU needed)."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from lowthrustopt_b200 import capi, solvers as S
from oracle_backend import OracleBackend
from test_transfer_cost_cpu import _SweepBackend

MU, DU, TU = capi.MU, capi.DU, capi.TU
KAPPA = 1e3 / (TU * TU / DU / 1e3)                 # default_mass / kthr: u in N = KAPPA x the nondimensional acceleration


def test_dual_kernel_builds_for_sm100a(tmp_path):
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    from lowthrustopt_b200 import build
    obj = str(tmp_path / "lto_direct_qp.o")
    cmd = [build._nvcc()] + build.ARCH + build.NVCC_FLAGS + ["-I", build.INC, "-I", build.CSRC, "-c",
                                                             os.path.join(build.CSRC, "lto_direct_qp.cu"), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "sm_100a" in subprocess.run([cuobjdump, "-lelf", obj], capture_output=True, text=True).stdout
    usage = subprocess.run([cuobjdump, "-res-usage", obj], capture_output=True, text=True).stdout
    found = dict(re.findall(r"Function (_ZN3lto3dqp\w+):\s*\n\s*(REG:.*)", usage))
    dual = [v for k, v in found.items() if "16k_direct_qp_dual" in k]
    assert len(dual) == 1, sorted(found)
    assert "STACK:0 " in dual[0] and "LOCAL:0 " in dual[0], dual[0]
    assert len([k for k in found if "11k_direct_qpILi" in k]) == 2, sorted(found)     # k_direct_qp<6>, <7> keep their names


def _unbound_handle():
    """A Handle object that never reached lto_init: the argument checks run before any library call."""
    return capi.Handle.__new__(capi.Handle)


def test_costate_wrapper_refuses_bad_arguments():
    h = _unbound_handle()
    T, N = 2, 5
    X, U = np.zeros((T, N, 6)), np.zeros((T, N, 3))
    t = np.tile(np.linspace(0.0, 1.0, N), (T, 1))
    s = np.zeros((T, 6))
    with pytest.raises(ValueError, match="nstate 6"):
        h.direct_costates_batch(np.zeros((T, N, 7)), U, t, s, s)                       # nstate 7: no lm map
    with pytest.raises(ValueError):
        h.direct_costates_batch(X[0], U[0], t[0], s[0], s[0])                          # not a batch
    with pytest.raises(ValueError):
        h.direct_costates_batch(X, U[:, :4], t, s, s)
    with pytest.raises(ValueError):
        h.direct_costates_batch(X, U, t[:, :4], s, s)
    with pytest.raises(ValueError):
        h.direct_costates_batch(X, U, t, s[:1], s)
    with pytest.raises(ValueError):
        h.direct_costates_batch(X[:, :1], U[:, :1], t[:, :1], s, s)                    # no segment
    with pytest.raises(ValueError, match="LTO_FIXED"):
        h.direct_costates_batch(X, U, t, s, s, params=capi.DirectParams(mode=capi.LTO_ADAPTIVE))
    flat = t.copy(); flat[1, 3] = flat[1, 2]
    with pytest.raises(ValueError, match="trajectory 1"):
        h.direct_costates_batch(X, U, flat, s, s)
    bad = t.copy(); bad[0, 2] = np.inf
    with pytest.raises(ValueError, match="trajectory 0"):
        h.direct_costates_batch(X, U, bad, s, s)
    with pytest.raises(ValueError):
        S.direct_costates(np.zeros((T, 7, N)), np.zeros((T, 3, N)), t, s, s, backend=object())


# --------------------------------------------------------------------------- the map, on the CPU oracle
def _node_weights(t):
    dt = np.diff(t)
    return np.concatenate([dt / 2, [dt[-1] / 2]]) + np.concatenate([[0.0], dt[:-1] / 2, [0.0]])


def kkt_multipliers(blocks, defect, X, U, t, s0, sf):
    """The dense KKT system of _qp_direct's formulation (optimizeTraj, flagEnd = false, dV = 0) at (X, U): (x_update, u_update, lambda)."""
    n, N = 6, X.shape[1]
    Jf = np.hstack([S._band_direct(blocks, n, N), np.zeros((n * (N - 1), 1))])
    tau = (t - t[0]) / (t[-1] - t[0]) * 2 - 1
    xu, uu, _, _, _, lam = S._qp_direct(X, U, np.zeros(3), np.zeros(3), defect.T, Jf, n, N, s0, sf, 1e3, tau, t[0], t[-1], DU, TU, False,
                                        multipliers=True)
    return xu, uu, lam


def identities(blocks, lam, U, du, t):
    """(a) u-stationarity 2 w_i (u_i + du_i) = (J^T lambda)_{u_i}; (b) Jx(i, i)^T lambda_i = -Jx(i-1, i)^T lambda_{i-1} at interior nodes.
    U, du: (N, 3).  Returns the two relative residuals."""
    N = U.shape[0]
    g = np.zeros((N, 3))
    for i in range(N - 1):
        g[i] += blocks[i][:, 12:15].T @ lam[i]
        g[i + 1] += blocks[i][:, 15:18].T @ lam[i]
    ra = np.abs(2 * _node_weights(t)[:, None] * (U + du) - g).max() / np.abs(g).max()
    fwd = np.stack([blocks[i][:, :6].T @ lam[i] for i in range(1, N - 1)])
    bwd = np.stack([-(blocks[i - 1][:, 6:12].T @ lam[i - 1]) for i in range(1, N - 1)])
    rb = np.abs(fwd - bwd).max() / np.abs(fwd).max()
    return ra, rb


@pytest.fixture(scope="module")
def demo():
    """The demo's direct problem solved with the oracle backend, and the multipliers of its QP at the solution."""
    be = OracleBackend()
    X0t, X0, Xft, Xf = S.demo_fixtures()
    XC, t, tau1, tau2, s0, sf = S.trajectory_stack_guess(X0, Xf, backend=be)
    out = S.multiShoot_CRTBP_direct(XC[:6].copy(), np.zeros((3, 30)), tau1, tau2, t, np.zeros(3), np.zeros(3), MU, DU, TU, 30, 10, 1e3, 2000.0,
                                    X0t, X0, Xft, Xf, backend=be)
    X, U, t = out[0], out[1], out[4]
    d, _, blocks = be.direct_blocks(X.T[None], U.T[None], t[None], 10, 2000.0, MU, DU, TU)
    xu, uu, lam = kkt_multipliers(blocks[0], d[0], X, U, t, s0[:6], sf[:6])
    return dict(be=be, X=X, U=U, t=t, s0=s0[:6], sf=sf[:6], blocks=blocks[0], lam=lam, du=uu)


def test_kkt_identities_hold_at_the_direct_solution(demo):
    ra, rb = identities(demo["blocks"], demo["lam"], demo["U"].T, demo["du"].T, demo["t"])
    print("\n[oracle] u-stationarity %.1e | interior one-sided costates %.1e | max |du| %.1e N" % (ra, rb, np.abs(demo["du"]).max()))
    assert ra <= 1e-10 and rb <= 1e-10


def test_mapped_lv_is_minus_two_u_over_kappa(demo):
    """The p = 2 law a = -lv / 2 and u = KAPPA a give lv = -2 u / KAPPA: the sign everywhere, the value to the discretisation level."""
    cs = S._direct_costate_map(demo["blocks"], demo["lam"], 1e3, DU, TU)
    ref = -2 * demo["U"] / KAPPA
    rel = np.abs(cs[3:] - ref).max() / np.abs(ref).max()
    print("\n[oracle] lv vs -2u/kappa: %.3e relative" % rel)
    assert np.array_equal(np.sign(cs[3:]), np.sign(ref))
    assert rel < 0.06                                                         # the oracle gives 4.4e-2 on the demo's 30 nodes


def test_full_p2_solve_from_the_mapped_start_converges(demo):
    cs = S._direct_costate_map(demo["blocks"], demo["lam"], 1e3, DU, TU)
    XC = np.vstack([demo["X"], cs])
    XC[:6, 0] = demo["s0"]; XC[:6, -1] = demo["sf"]
    log = []
    Xs, _, st = S.multiShoot_CRTBP_indirect(XC, demo["t"], MU, DU, TU, 30, 1e3, 10.0, False, False, 50, 2.0, 1.0, backend=demo["be"], log=log)
    print("\n[oracle] full p = 2 solve from the mapped start: status %d after %d iterations" % (st, len(log)))
    assert st == 0


# --------------------------------------------------------------------------- the sweep's start="direct", against a fake backend
class _DirectStartBackend(_SweepBackend):
    def __init__(self, statuses, costate_status):
        super().__init__(statuses)
        self.costate_status = costate_status          # row -> status of direct_costates
        self.draws = None

    def direct_costates(self, X, U, t, state_0, state_f, nsteps, Isp, MU, DU, TU):
        rows = [int(r) for r in X[:, 0, 0]]
        self.calls.append(("costates", rows))
        B, N, _ = X.shape
        XC = np.concatenate([X, np.full((B, N, 6), 0.25)], axis=2)
        st = np.array([self.costate_status.get(r, 0) for r in rows], dtype=np.int32)
        XC[st != 0, :, 6:] = np.nan
        return dict(XC_all=XC, multipliers=np.zeros((B, N - 1, 6)), du_max=np.zeros(B), status=st)

    def indirect_solve_batch(self, XC, t, params, thrustLimit=None, rho=None, max_iter=50, flag_adjointsOnly=False):
        if max_iter == 50:
            self.p2_start = XC.copy()
        return super().indirect_solve_batch(XC, t, params, thrustLimit, rho, max_iter, flag_adjointsOnly)

    def indirect_reduce_fuel_batch(self, XC, t, params, rho_current, rho_target, backoff_uniform, thrustLimit=None, max_iter=10):
        self.draws = backoff_uniform.copy()
        return super().indirect_reduce_fuel_batch(XC, t, params, rho_current, rho_target, backoff_uniform, thrustLimit, max_iter)


def test_direct_start_gates_on_the_costate_status():
    be = _DirectStartBackend({"p2": {3: 1}, "ladder": {5: 3}}, {1: 1, 4: 3})
    X0 = np.zeros((6, 10))
    seeds = [11, 12, 13, 14, 15, 16, 17]
    r = S.indirect_transfer_sweep(X0, X0, np.arange(7.0), 5.0, 5.0, thrustLimit=0.07, rho_target=1e-3, n_nodes=8, backend=be, seeds=seeds,
                                  start="direct")
    assert [c[0] for c in be.calls] == ["costates", "p2", "cost_p2", "p1", "ladder", "cost_p1"]    # no adjoints-only solve
    calls = dict(be.calls)
    assert calls["costates"] == [0, 1, 2, 3, 4, 5, 6]
    assert calls["p2"] == [0, 2, 3, 5, 6]                                      # rows 1 and 4 failed at stage 1 and entered nothing else
    assert calls["ladder"] == [0, 2, 5, 6] and calls["cost_p1"] == [0, 2, 6]
    assert r["stage_failed"].tolist() == [0, 1, 0, 2, 1, 4, 0]
    assert np.isnan(r["XC_all"][[1, 4], 6:]).all() and np.isnan(r["dv"][[1, 4]]).all()
    # stage 2 starts from the mapped costates, the end states pinned, no jitter
    start = be.p2_start.transpose(0, 2, 1)
    assert np.all(start[:, 6:] == 0.25)
    assert np.array_equal(start[:, 0, 1:-1], np.array([[0.0, 2.0, 3.0, 5.0, 6.0]]).T * np.ones((1, 6)))
    # the ladder's back-off draws still come from the seeds
    want = np.array([np.random.default_rng(seeds[j]).random(100) for j in (0, 2, 5, 6)])
    assert np.array_equal(be.draws, want)


def test_sweep_refuses_an_unknown_start():
    X0 = np.zeros((6, 10))
    for bad in ("random", None, "Direct"):
        with pytest.raises(ValueError, match="start"):
            S.indirect_transfer_sweep(X0, X0, 0.1, 5.0, 5.0, backend=object(), start=bad)
