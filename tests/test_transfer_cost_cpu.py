"""CPU-side checks of the transfer cost (lto_indirect_cost_batch, solvers.transfer_cost_indirect) and of the indirect transfer sweep
(solvers.indirect_transfer_sweep): the sm_100a build of the new kernels, wrapper validation, the 14-dim closed form and the sweep's stage
gating against a fake backend (no GPU needed)."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from lowthrustopt_b200 import capi, solvers as S

MU, DU, TU = capi.MU, capi.DU, capi.TU


def _unbound_handle():
    """A Handle object that never reached lto_init: the argument checks run before any library call."""
    return capi.Handle.__new__(capi.Handle)


def test_cost_kernels_build_for_sm100a(tmp_path):
    """k_cost_sum uses no stack and no local memory.  k_indirect_state_cost uses no local memory; like K4 itself (k_indirect_state,
    255 registers at two CTAs of 128 threads per SM) it keeps a spill / call frame, at most 64 bytes larger than K4's."""
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    from lowthrustopt_b200 import build
    obj = str(tmp_path / "lto_indirect_cw.o")
    cmd = [build._nvcc()] + build.ARCH + build.NVCC_FLAGS + ["-I", build.INC, "-I", build.CSRC, "-c",
                                                             os.path.join(build.CSRC, "lto_indirect_cw.cu"), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "sm_100a" in subprocess.run([cuobjdump, "-lelf", obj], capture_output=True, text=True).stdout
    usage = subprocess.run([cuobjdump, "-res-usage", obj], capture_output=True, text=True).stdout
    found = dict(re.findall(r"Function (_ZN3lto3icw\w+):\s*\n\s*(REG:.*)", usage))

    def one(tag):
        hits = [v for k, v in found.items() if tag in k]
        assert len(hits) == 1, (tag, sorted(found))
        return hits[0]

    s = one("10k_cost_sum")
    assert "STACK:0 " in s and "LOCAL:0 " in s, s
    q, k4 = one("21k_indirect_state_costE"), one("16k_indirect_stateE")
    assert "LOCAL:0 " in q and "LOCAL:0 " in k4, (q, k4)
    stack = lambda u: int(re.search(r"STACK:(\d+)", u).group(1))
    assert stack(q) <= stack(k4) + 64, (q, k4)


def test_cost_wrapper_refuses_bad_arguments():
    h = _unbound_handle()
    t = np.tile(np.linspace(0.0, 1.0, 5), (2, 1))
    with pytest.raises(ValueError):
        h.indirect_cost_batch(np.zeros((2, 5, 14)), t)                              # 14-dim: the node masses give the cost
    with pytest.raises(ValueError):
        h.indirect_cost_batch(np.zeros((5, 12)), t[0])                              # not a batch
    with pytest.raises(ValueError):
        h.indirect_cost_batch(np.zeros((2, 5, 12)), t[:, :4])                       # one time short
    with pytest.raises(ValueError):
        h.indirect_cost_batch(np.zeros((2, 1, 12)), t[:, :1])                       # no segment
    with pytest.raises(ValueError):
        h.indirect_cost_batch(np.zeros((2, 5, 12)), t, params=capi.IndirectParams(controller=capi.LTO_CTRL_ODE78))
    rev = t.copy(); rev[1, 3] = 0.1
    with pytest.raises(ValueError, match="trajectory 1"):
        h.indirect_cost_batch(np.zeros((2, 5, 12)), rev)
    bad = t.copy(); bad[0, 2] = np.nan
    with pytest.raises(ValueError, match="trajectory 0"):
        h.indirect_cost_batch(np.zeros((2, 5, 12)), bad)
    with pytest.raises(ValueError):
        h.indirect_cost_batch(np.zeros((2, 5, 12)), t, thrustLimit=np.ones(3))
    with pytest.raises(ValueError):
        S.transfer_cost_indirect(np.zeros((2, 13, 5)), t, MU, DU, TU, 1e3, 0.05, 1.0, 1.0, backend=object())
    with pytest.raises(ValueError):
        S.transfer_cost_indirect(np.zeros((2, 12, 5)), t[:, :4], MU, DU, TU, 1e3, 0.05, 1.0, 1.0, backend=object())


def test_14dim_cost_is_the_rocket_equation_on_the_node_masses():
    rng = np.random.default_rng(7)
    T, N = 6, 9
    XC = rng.standard_normal((T, 14, N))
    m0 = 1000.0 + rng.random(T); mf = m0 - 50.0 * rng.random(T)
    XC[:, 6, 0] = m0; XC[:, 6, -1] = mf; XC[:, 6, 1:-1] = 1e9                 # only the end masses count
    XC[5, 6, -1] = np.nan
    t = np.tile(np.linspace(0.0, 2.0, N), (T, 1))
    r = S.transfer_cost_indirect(XC, t, MU, DU, TU, 1e3, 0.05, 1.0, 1e-3, Isp=3000.0, backend=object())   # no device call
    assert np.array_equal(r["propellant"][:5], m0[:5] - mf[:5])
    np.testing.assert_allclose(r["dv"][:5], 3000.0 * 9.81 * np.log(m0[:5] / mf[:5]), rtol=1e-15)
    assert np.isnan(r["energy"]).all()
    assert r["status"].tolist() == [0, 0, 0, 0, 0, 1] and np.isnan(r["dv"][5])


class _SweepBackend:
    """Fake backend for indirect_transfer_sweep: row j of the grid is the one with tau1 = j, which the fake guess writes into x of node 0
    (pinned through every stage), so each call can see which rows it was given and answer with the statuses it was told to."""

    def __init__(self, statuses):
        self.statuses = statuses                      # call name -> {row: status}
        self.calls = []

    def stack_guess_batch(self, X0_states, Xf_states, tau1, t_TU, t_split, params):
        T, N = t_TU.shape
        s0 = np.zeros((T, 6)); s0[:, 0] = tau1
        XC = np.zeros((T, N, 12)); XC[:, :, 0] = tau1[:, None]
        return dict(XC_all=XC, tau2=np.zeros(T), state_0=s0, state_f=s0.copy(), status=np.zeros(T, dtype=np.int32))

    def direct_solve_batch(self, X, U, t, state_0, state_f, mass, nsteps, max_iter, Isp, MU, DU, TU):
        T = X.shape[0]
        return dict(X_all=X.copy(), u_all=U.copy(), defect=None, iters=np.ones(T, dtype=np.int32), er=np.zeros(T))

    def _answer(self, name, XC):
        rows = [int(r) for r in XC[:, 0, 0]]
        self.calls.append((name, rows))
        return rows, np.array([self.statuses.get(name, {}).get(r, 0) for r in rows], dtype=np.int32)

    def indirect_solve_batch(self, XC, t, params, thrustLimit=None, rho=None, max_iter=50, flag_adjointsOnly=False):
        name = {(2.0, True, 10): "adjoints", (2.0, False, 50): "p2", (1.0, False, 30): "p1"}[(params[6], bool(flag_adjointsOnly), max_iter)]
        assert np.all(thrustLimit == (0.07 if name == "p1" else 10.0)) and np.all(rho == 1.0)
        rows, st = self._answer(name, XC)
        B, N, m = XC.shape
        return dict(XC_all=XC.copy(), defect=np.zeros((B, N - 1, m)), status_flag=st, iters=np.ones(B, dtype=np.int32), er=np.zeros(B))

    def indirect_reduce_fuel_batch(self, XC, t, params, rho_current, rho_target, backoff_uniform, thrustLimit=None, max_iter=10):
        assert np.all(rho_current == 1.0) and np.all(rho_target == 1e-3) and np.all(thrustLimit == 0.07) and backoff_uniform.shape == (len(XC), 100)
        rows, st = self._answer("ladder", XC)
        return dict(XC_all=XC.copy(), status=st, rho_last=np.where(st == 0, 1e-3, 0.5))

    def indirect_cost(self, XC, t, params, thrustLimit=None, rho=None, defect=False):
        rows, _ = self._answer("cost_p%g" % params[6], XC)
        r = np.array(rows, dtype=np.float64)
        return dict(dv=100.0 + r, energy=200.0 + r, status=np.zeros(len(rows), dtype=np.int32))


def test_sweep_gates_each_stage_on_the_previous_one():
    be = _SweepBackend({"adjoints": {1: 2, 2: 1}, "p2": {3: 1}, "p1": {4: 2}, "ladder": {5: 3}})
    X0 = np.zeros((6, 10))
    r = S.indirect_transfer_sweep(X0, X0, np.arange(7.0), 5.0, 5.0, thrustLimit=0.07, rho_target=1e-3, n_nodes=8, backend=be)
    calls = dict(be.calls)
    assert [c[0] for c in be.calls] == ["adjoints", "p2", "cost_p2", "p1", "ladder", "cost_p1"]
    assert calls["adjoints"] == [0, 1, 2, 3, 4, 5, 6]
    assert calls["p2"] == [0, 2, 3, 4, 5, 6]                                  # status 1 of the adjoints-only solve is expected
    assert calls["cost_p2"] == calls["p1"] == [0, 2, 4, 5, 6]
    assert calls["ladder"] == [0, 2, 5, 6] and calls["cost_p1"] == [0, 2, 6]
    assert r["stage_failed"].tolist() == [0, 1, 0, 2, 3, 4, 0]
    assert r["status"].tolist() == [0, -1, 0, -1, -1, 3, 0]
    ok = np.array([0, 2, 6])
    assert np.array_equal(r["dv"][ok], 100.0 + ok) and np.array_equal(r["energy"][ok], 200.0 + ok)
    assert np.isnan(np.delete(r["dv"], ok)).all() and np.isnan(np.delete(r["energy"], ok)).all()
    assert np.array_equal(r["energy_p2"][[0, 2, 4, 5, 6]], [200.0, 202.0, 204.0, 205.0, 206.0]) and np.isnan(r["energy_p2"][[1, 3]]).all()
    assert r["rho_last"][5] == 0.5 and r["rho_last"][0] == 1e-3 and np.isnan(r["rho_last"][1])
    assert r["XC_all"].shape == (7, 12, 8) and np.array_equal(r["XC_all"][:, 0, 0], np.arange(7.0))


def test_sweep_start_is_the_demo_start():
    """Row j's start: the direct solution, costates 0.1 N(0, 1) and the 1e-10 interior jitter from default_rng(seeds[j]), as the demo."""
    be = _SweepBackend({"adjoints": {0: 2, 1: 2}})
    starts = []
    be.indirect_solve_batch = lambda XC, *a, **k: (starts.append(XC.copy()), _SweepBackend.indirect_solve_batch(be, XC, *a, **k))[1]
    S.indirect_transfer_sweep(np.zeros((6, 10)), np.zeros((6, 10)), [0.0, 1.0], 5.0, 5.0, seeds=[42, 9], n_nodes=8, backend=be)
    for j, seed in enumerate((42, 9)):
        rng = np.random.default_rng(seed)
        XC0 = np.vstack([np.zeros((6, 8)), 0.1 * rng.standard_normal((6, 8))])
        XC0[:6, 0] = XC0[:6, -1] = [j, 0, 0, 0, 0, 0]
        XC0[:, 1:-1] += 1e-10 * rng.standard_normal((12, 6))
        XC0[0, 1:-1] += j                                                       # the fake direct solution's x row
        assert np.array_equal(starts[0][j].T, XC0)


def test_sweep_refuses_bad_arguments():
    be = object()                                                               # nothing may reach a backend
    X0 = np.zeros((6, 10))
    with pytest.raises(ValueError):
        S.indirect_transfer_sweep(X0, X0, [0.1, 0.2], 5.0, 5.0, seeds=[1], backend=be)
    with pytest.raises(ValueError):
        S.indirect_transfer_sweep(X0, X0, [0.1, 0.2], [5.0, 6.0, 7.0], 5.0, backend=be)
    with pytest.raises(ValueError):
        S.indirect_transfer_sweep(X0, X0, 0.1, 5.0, 5.0, thrustLimit=0.0, backend=be)
    with pytest.raises(ValueError):
        S.indirect_transfer_sweep(X0, X0, 0.1, 5.0, 5.0, rho_target=2.0, backend=be)
    with pytest.raises(ValueError):
        S.indirect_transfer_sweep(X0, X0, 0.1, 5.0, 5.0, n_nodes=2, backend=be)
