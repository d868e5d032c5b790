"""GPU: parity of liblto_b200.so (through the C ABI) with the CPU oracle, the committed golden
vectors, and size-independent properties at the benchmark sizes.

Tolerances (BASELINE.json north_star): segment end states / defects 1e-10, Jacobian / STM
entries 1e-8, both relative to max(1, |value scale|).  FIXED-mode results come from the same
discrete map as the oracle, so they are held to much tighter bounds below.
"""
import os

import numpy as np
import pytest

from lowthrustopt_b200 import capi, synthetic as S

pytestmark = pytest.mark.gpu
ROOT = os.path.normpath(os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

TOL_STATE = 1e-10
TOL_JAC = 1e-8


def rel(a, b, scale=None):
    sc = np.maximum(1.0, np.abs(b) if scale is None else scale)
    return (np.abs(a - b) / sc).max() if a.size else 0.0


# ------------------------------------------------------------------ direct
@pytest.mark.parametrize("kernel", [capi.LTO_KERNEL_GENERIC, capi.LTO_KERNEL_AUTO])
@pytest.mark.parametrize("ns", [6, 7])
def test_direct_fixed_vs_oracle(ns, kernel, lto, oracle):
    n = 1000 + 37                                      # ragged: not a multiple of any tile size
    b = S.direct_batch(n, nstate=ns, seed=101)
    r = lto.direct(b["Xa"], b["Xb"], b["ua"], b["ub"], b["ta"], b["tb"], nsteps=10, params=capi.direct_params(kernel=kernel))
    do, eo, Jo, so = oracle.direct_jac_var(b["Xa"], b["Xb"], b["ua"], b["ub"], b["ta"], b["tb"], nthreads=oracle.num_threads())
    xscale = np.maximum(np.abs(b["Xa"]), np.abs(b["Xb"]))
    assert rel(r["defect"], do, xscale) < 1e-13
    assert rel(r["jac"].transpose(0, 2, 1), Jo) < 1e-12
    assert np.abs(r["errors"] - eo).max() < 2e-14     # rounding-level quantity (mass ~1e3)
    assert np.all(r["status"] == 0)
    # defect-only entry point gives the same defect
    r2 = lto.direct(b["Xa"], b["Xb"], b["ua"], b["ub"], b["ta"], b["tb"], nsteps=10, params=capi.direct_params(kernel=kernel), jac=False)
    assert rel(r2["defect"], r["defect"], xscale) < 1e-14


def test_direct_vs_golden(lto, golden):
    for g in golden["direct"]:
        r = lto.direct([g["Xa"]], [g["Xb"]], [g["ua"]], [g["ub"]], [g["ta"]], [g["tb"]], nsteps=g["nsteps"],
                       params=capi.direct_params(Isp=g["Isp"]))
        sc = np.maximum(1.0, np.abs(np.array(g["Xa"])))
        assert (np.abs(r["defect"][0] - np.array(g["defect"])) / sc).max() < TOL_STATE
        J = r["jac"][0].T
        Jr = np.array(g["jac_richardson"])
        rows = slice(0, 6) if np.all(np.array(g["ua"]) == 0) else slice(0, g["nstate"])
        assert rel(J[rows], Jr[rows]) < TOL_JAC * (1 if g["nstate"] == 6 else 10)   # Richardson truth is itself ~1e-8 on mass rows
        # distance to the reference's own FD Jacobian = the reference's FD noise (SURVEY D1), reported not gated tightly
        assert np.abs(J[:6] - np.array(g["jac_fd"])[:6]).max() < 5e-6


@pytest.mark.parametrize("ns", [6, 7])
def test_direct_adaptive_vs_oracle(ns, lto, oracle):
    n = 257
    b = S.direct_batch(n, nstate=ns, seed=102)
    for norm in (capi.LTO_NORM_STATE, capi.LTO_NORM_STATE_SENS):
        p = capi.direct_params(mode=capi.LTO_ADAPTIVE, tol=1e-12, err_norm=norm)
        r = lto.direct(b["Xa"], b["Xb"], b["ua"], b["ub"], b["ta"], b["tb"], params=p)
        do, eo, Jo, so = oracle.direct_jac_var(b["Xa"], b["Xb"], b["ua"], b["ub"], b["ta"], b["tb"], mode=1, tol=1e-12,
                                              with_partials=bool(norm), nthreads=oracle.num_threads())
        xscale = np.maximum(np.abs(b["Xa"]), np.abs(b["Xb"]))
        assert rel(r["defect"], do, xscale) < TOL_STATE
        assert rel(r["jac"].transpose(0, 2, 1), Jo) < TOL_JAC
        assert np.all(r["status"] == 0)


def test_direct_traj_form_equals_pairs_form(lto):
    n_traj, n_nodes, ns = 7, 30, 7
    rng = np.random.default_rng(7)
    X = np.empty((n_traj, n_nodes, ns)); t = np.empty((n_traj, n_nodes))
    for j in range(n_traj):
        tau = rng.uniform() + np.linspace(0, 4.6, n_nodes) / S.PERIODS[0]
        X[j, :, :6] = S.interp_initial_states(tau, 1) + 1e-3 * rng.standard_normal((n_nodes, 6))
        X[j, :, 6] = 1000.0 - np.linspace(0, 1, n_nodes)
        t[j] = np.linspace(0, 4.6, n_nodes) + rng.uniform()
    U = 0.05 * rng.standard_normal((n_traj, n_nodes, 3))
    rt = lto.direct_traj(X, U, t)
    rp = lto.direct(X[:, :-1].reshape(-1, ns), X[:, 1:].reshape(-1, ns), U[:, :-1].reshape(-1, 3), U[:, 1:].reshape(-1, 3),
                    t[:, :-1].ravel(), t[:, 1:].ravel())
    assert np.array_equal(rt["defect"], rp["defect"]) and np.array_equal(rt["jac"], rp["jac"])


def test_direct_edge_cases(lto, oracle):
    # empty batch
    z = np.zeros((0, 7))
    r = lto.direct(z, z, np.zeros((0, 3)), np.zeros((0, 3)), np.zeros(0), np.zeros(0))
    assert r["defect"].shape == (0, 7) and r["jac"].shape == (0, 20, 7)
    # |u| = 0 (the demo's first iteration): one-sided mass-flow slope, everything finite
    b = S.direct_batch(33, nstate=7, seed=5, zero_control=True)
    r = lto.direct(b["Xa"], b["Xb"], b["ua"], b["ub"], b["ta"], b["tb"])
    do, eo, Jo, so = oracle.direct_jac_var(b["Xa"], b["Xb"], b["ua"], b["ub"], b["ta"], b["tb"])
    assert np.all(np.isfinite(r["jac"])) and rel(r["jac"].transpose(0, 2, 1), Jo) < 1e-12
    # bad arguments are errors, not crashes
    with pytest.raises(capi.LtoError):
        lto.direct(np.zeros((1, 5)), np.zeros((1, 5)), np.zeros((1, 3)), np.zeros((1, 3)), np.zeros(1), np.ones(1))
    with pytest.raises(capi.LtoError):
        lto.direct(b["Xa"], b["Xb"], b["ua"], b["ub"], b["ta"], b["tb"], nsteps=1)


def test_direct_full_size_properties(lto):
    """65,536 segments (BASELINE config 3): properties that need no oracle."""
    n = 65536
    b = S.direct_batch(n, nstate=7)
    r = lto.direct(b["Xa"], b["Xb"], b["ua"], b["ub"], b["ta"], b["tb"])
    assert np.all(r["status"] == 0) and np.all(np.isfinite(r["jac"]))
    # (1) batch-position invariance, bitwise: a permuted batch gives the permuted result
    perm = np.random.default_rng(1).permutation(n)
    rp = lto.direct(b["Xa"][perm], b["Xb"][perm], b["ua"][perm], b["ub"][perm], b["ta"][perm], b["tb"][perm])
    assert np.array_equal(rp["defect"], r["defect"][perm]) and np.array_equal(rp["jac"], r["jac"][perm])
    # (2) mirror symmetry of the CRTBP, (x,y,z,vx,vy,vz,t) -> (x,-y,z,-vx,vy,-vz,-t) =: M, which the RK map
    #     inherits: for ballistic segments, swapping the nodes and mirroring them negates the mirrored defect
    bz = S.direct_batch(4096, nstate=6, seed=9, zero_control=True)
    r1 = lto.direct(bz["Xa"], bz["Xb"], bz["ua"], bz["ub"], bz["ta"], bz["tb"], jac=False)
    M = np.array([1, -1, 1, -1, 1, -1.0])
    r2 = lto.direct(bz["Xb"] * M, bz["Xa"] * M, bz["ub"], bz["ua"], bz["ta"], bz["tb"], jac=False)
    assert np.abs(r2["defect"] + r1["defect"] * M).max() < 1e-13
    # (3) Liouville: the (r, v) block of Phi_f has determinant 1 (trace of the 6x6 dynamics matrix is 0)
    J = rp["jac"][:256].transpose(0, 2, 1)      # (n, 7, 20)
    Phi_f = J[:, :6, :6]
    assert np.abs(np.linalg.det(Phi_f) - 1.0).max() < 1e-9


# ------------------------------------------------------------------ indirect
LAWS = [dict(p=1.0, rho=1.0, thrustLimit=0.05), dict(p=2.0, rho=1.0, thrustLimit=10.0), dict(p=1.0, rho=1e-2, thrustLimit=0.05),
        dict(p=0.0, rho=1.0, thrustLimit=0.05), dict(p=2.0, rho=1.0, thrustLimit=1e-3)]


@pytest.mark.parametrize("kernel", [capi.LTO_KERNEL_GENERIC, capi.LTO_KERNEL_AUTO])
@pytest.mark.parametrize("nd", [12, 14])
@pytest.mark.parametrize("law", LAWS)
def test_indirect_vs_oracle(nd, law, kernel, lto, oracle):
    n = 300 + 11
    b = S.indirect_batch(n, ndim=nd, seed=202)
    lv = slice(9, 12) if nd == 12 else slice(10, 13)
    b["x0"][::3, lv] *= 8.0                      # a third of the batch sits near the |lv| = 1 switch
    xt = b["x0"] + 0.01
    p = capi.indirect_params(kernel=kernel, **law)
    r = lto.indirect(b["x0"], b["t0"], b["t1"], x_target=xt, params=p)
    ip = oracle.iparams(law["thrustLimit"], p=law["p"], rho=law["rho"])
    xo, Po, so, nao, nto = oracle.indirect_prop_jac(b["x0"], b["t0"], b["t1"], ip, nthreads=oracle.num_threads())
    assert np.all(r["status"] == 0) and np.all(so == 0)
    assert rel(r["defect"] + xt, xo) < TOL_STATE
    assert rel(r["phi"].transpose(0, 2, 1), Po, np.abs(Po).max(axis=(1, 2), keepdims=True)) < TOL_JAC
    assert np.abs(r["nsteps"][:, 0] - nao).max() <= 2
    # defect-only path (state-only step control, like the reference's plain solve)
    r0 = lto.indirect(b["x0"], b["t0"], b["t1"], x_target=xt, params=p, jac=False)
    xo0, so0, _, _ = oracle.indirect_prop(b["x0"], b["t0"], b["t1"], ip, nthreads=oracle.num_threads())
    assert rel(r0["defect"] + xt, xo0) < TOL_STATE


_HC_CHILD = r"""
import sys, numpy as np
sys.path.insert(0, %r)
from lowthrustopt_b200 import capi, synthetic as S
h = capi.Handle(0)
out = {}
for i, law in enumerate(%r):
    b = S.indirect_batch(4096 + 37, ndim=12, seed=303)
    b["x0"][::3, 9:12] *= 8.0
    r = h.indirect(b["x0"], b["t0"], b["t1"], params=capi.indirect_params(**law))
    out["d%%d" %% i] = r["defect"]; out["p%%d" %% i] = r["phi"]; out["s%%d" %% i] = r["status"]; out["n%%d" %% i] = r["nsteps"]
np.savez(sys.argv[1], **out)
h.close()
"""


@pytest.mark.parametrize("layout", ["hc", "wl", "hc2"])
def test_k3_experimental_layouts_match_default(layout, lto, oracle, tmp_path):
    """The two round-2 rebuilds of K3 that were measured and not adopted (DESIGN.md section 4: hc = second-order half-column formulation with
    setmaxnreg and three tiles; wl = warp-local, every warp owns 8 slots) live in tools/experiments/ and are NOT in the product library; a library
    built by build.build_experiments() (tools/experiments/lib/liblto_k3x.so, made by build()) contains them.  Each runs in a child process (the
    layout is selected once per process) and is held to the same bars against the oracle as the default K3, and to 1e-10 against the default K3."""
    import subprocess
    import sys
    from lowthrustopt_b200 import build
    xlib = build.build_experiments()
    laws = LAWS[:3]
    f = str(tmp_path / "hc.npz")
    env = dict(os.environ, LTO_K3=layout, LTO_B200_LIB=xlib)
    cp = subprocess.run([sys.executable, "-c", _HC_CHILD % (ROOT, laws), f], env=env, capture_output=True, text=True, timeout=300)
    assert cp.returncode == 0, cp.stderr[-2000:]
    z = np.load(f)
    for i, law in enumerate(laws):
        b = S.indirect_batch(4096 + 37, ndim=12, seed=303)
        b["x0"][::3, 9:12] *= 8.0
        r = lto.indirect(b["x0"], b["t0"], b["t1"], params=capi.indirect_params(**law))
        ip = oracle.iparams(law["thrustLimit"], p=law["p"], rho=law["rho"])
        xo, Po, so, nao, nto = oracle.indirect_prop_jac(b["x0"], b["t0"], b["t1"], ip, nthreads=oracle.num_threads())
        sp = np.abs(Po).max(axis=(1, 2), keepdims=True)
        assert np.all(z["s%d" % i] == 0)
        assert rel(z["d%d" % i], xo) < TOL_STATE and rel(z["p%d" % i].transpose(0, 2, 1), Po, sp) < TOL_JAC
        assert rel(z["d%d" % i], r["defect"]) < TOL_STATE
        assert np.abs(z["n%d" % i][:, 0].astype(np.int64) - r["nsteps"][:, 0]).max() <= 2


def test_indirect_vs_golden(lto, golden):
    for g in golden["indirect"]:
        p = capi.indirect_params(thrustLimit=g["thrustLimit"], mass=g["mass"], time_direction=g["td"], p=g["p"], rho=g["rho"])
        r = lto.indirect([g["x0"]], [g["t0"]], [g["t1"]], params=p)
        assert np.abs(r["defect"][0] - np.array(g["xend"])).max() < TOL_STATE
        if "phi_richardson" in g:
            assert np.abs(r["phi"][0].T - np.array(g["phi_richardson"])).max() < 5e-8


def test_indirect14_vs_golden(lto, golden14):
    """K3-14 / K4-14 against the symbolically derived 14-dim system (tests/golden/make_golden14.py): end states 1e-10 relative
    (north_star), STM against the Richardson differences of the DOP853 flow."""
    for g in golden14["indirect14"]:
        p = capi.indirect_params(thrustLimit=g["thrustLimit"], time_direction=g["td"], p=g["p"], rho=g["rho"], Isp=g["Isp"])
        want = np.array(g["xend"]); sc = np.maximum(1.0, np.abs(want))
        r = lto.indirect([g["x0"]], [g["t0"]], [g["t1"]], params=p)
        assert r["status"][0] == 0 and (np.abs(r["defect"][0] - want) / sc).max() < TOL_STATE
        r0 = lto.indirect([g["x0"]], [g["t0"]], [g["t1"]], params=p, jac=False)
        assert (np.abs(r0["defect"][0] - want) / sc).max() < TOL_STATE
        if "phi_richardson" in g:
            P = np.array(g["phi_richardson"])
            assert np.abs(r["phi"][0].T - P).max() < 5e-8 * max(1.0, np.abs(P).max() / 10)


def test_indirect_ode78_controller_and_per_segment_params(lto, oracle):
    n = 64
    b = S.indirect_batch(n, ndim=12, seed=203)
    tl = np.geomspace(10.0, 0.05, n); rho = np.geomspace(1.0, 1e-3, n)
    p = capi.indirect_params(p=1.0, controller=capi.LTO_CTRL_ODE78)
    r = lto.indirect(b["x0"], b["t0"], b["t1"], params=p, thrustLimit=tl, rho=rho)
    ip = oracle.iparams(0.05, p=1.0)
    xo, Po, so, _, _ = oracle.indirect_prop_jac(b["x0"], b["t0"], b["t1"], ip, thrustLimit=tl, rho=rho, controller=1)
    assert rel(r["defect"], xo) < TOL_STATE and rel(r["phi"].transpose(0, 2, 1), Po) < TOL_JAC


def test_indirect_traj_form_and_edge_cases(lto):
    c = S.continuation_batch(n_traj=5, n_seg_per_traj=12, ndim=12)
    p = capi.indirect_params(p=1.0, rho=1.0)
    rt = lto.indirect_traj(c["XC_all"], c["t_TU"], params=p, thrustLimit=c["thrustLimit"])
    X = c["XC_all"]
    rp = lto.indirect(X[:, :-1].reshape(-1, 12), c["t_TU"][:, :-1].ravel(), c["t_TU"][:, 1:].ravel(), x_target=X[:, 1:].reshape(-1, 12),
                      params=p, thrustLimit=np.repeat(c["thrustLimit"], 12))
    assert np.array_equal(rt["defect"], rp["defect"]) and np.array_equal(rt["phi"], rp["phi"])
    # empty
    r = lto.indirect(np.zeros((0, 12)), np.zeros(0), np.zeros(0), params=p)
    assert r["phi"].shape == (0, 12, 12)
    # invalid control-law exponent is an error like the reference's error("Invalid value of p!")
    with pytest.raises(capi.LtoError, match="Invalid value of p"):
        lto.indirect(np.ones((1, 12)), np.zeros(1), np.ones(1), params=capi.indirect_params(p=0.5))
    # a reversed span is refused, not silently treated as empty (ADVICE r1); a zero-length span is fine (x0, Phi = I)
    with pytest.raises(capi.LtoError, match="reversed spans"):
        lto.indirect(np.ones((2, 12)), np.array([0.0, 0.3]), np.array([0.1, 0.2]), params=p)
    rz = lto.indirect(np.ones((1, 12)) * 0.5, np.array([0.2]), np.array([0.2]), params=p)
    assert rz["status"][0] == 0 and np.array_equal(rz["defect"][0], np.full(12, 0.5)) and np.array_equal(rz["phi"][0], np.eye(12))
    # NaN input -> status 1, not a crash
    bad = S.indirect_batch(4, ndim=12)
    bad["x0"][2, 0] = np.nan
    r = lto.indirect(bad["x0"], bad["t0"], bad["t1"], params=p)
    assert r["status"][2] == 1 and np.all(r["status"][[0, 1, 3]] == 0)


def test_indirect_symplectic_property(lto):
    """With a smooth control law the 12-dim system is Hamiltonian in (r, v | lr, lv) up to the
    Coriolis coupling; det(Phi) = 1 (Liouville: trace of A vanishes)."""
    b = S.indirect_batch(4096, ndim=12, seed=204)
    r = lto.indirect(b["x0"], b["t0"], b["t1"], params=capi.indirect_params(p=2.0, thrustLimit=10.0))
    det = np.linalg.det(r["phi"])
    assert np.abs(det - 1.0).max() < 1e-8


@pytest.mark.parametrize("nd,n", [(12, 40000), (14, 40000)])
def test_indirect_multi_chunk_host_pipeline(nd, n, lto):
    """Host-buffer calls above 8 MiB of output are cut into chunks (lto_host_chunk_plan) whose H2D copies, kernels and D2H copies
    run on their own streams: every segment must come back exactly as the one-launch call of a small batch computes it
    (bitwise -- a segment's arithmetic does not depend on its batch position)."""
    plan = capi.host_chunk_plan("indirect", n, nvar=nd)
    assert len(plan) >= 2 and sum(plan) == n
    b = S.indirect_batch(n, ndim=nd, seed=77)
    p = capi.indirect_params(p=1.0, rho=1.0, thrustLimit=0.05)
    r = lto.indirect(b["x0"], b["t0"], b["t1"], params=p)
    assert np.all(r["status"] == 0) and np.all(np.isfinite(r["phi"])) and np.all(r["nsteps"][:, 0] > 0)
    for lo in (0, plan[0] - 1500, n - 3000):                              # inside the first chunk, across a chunk boundary, the tail
        sl = slice(lo, lo + 3000)
        q = lto.indirect(b["x0"][sl], b["t0"][sl], b["t1"][sl], params=p)   # 3000 segments: one launch
        assert capi.host_chunk_plan("indirect", 3000, nvar=nd) == [3000]
        for k in ("defect", "phi", "status", "nsteps"):
            assert np.array_equal(q[k], r[k][sl]), (k, lo)
    # defect-only calls (K4: step control on the state alone) agree with the STM pass (joint control) far inside the 1e-10 bar
    # except where a segment passes a primary closely (measured max over 40,000 segments: 3.5e-10)
    d = lto.indirect(b["x0"], b["t0"], b["t1"], params=p, jac=False)
    err = np.abs(d["defect"] - r["defect"]).max(axis=1)
    assert np.median(err) < 1e-12 and err.max() < 1e-8


# ------------------------------------------------------------------ reference-interface mirror
def test_reference_closures_mirror(lto, oracle):
    from lowthrustopt_b200 import direct, indirect
    direct.set_handle(lto)
    n_nodes, ns = 30, 6
    t = np.linspace(0, 20 * 86400 / capi.TU, n_nodes)
    X = S.interp_initial_states(0.75 + t / S.PERIODS[0], 1).T.copy()          # (6, 30) like the demo's X_all
    U = np.zeros((3, n_nodes))
    defect, errors = direct.defectCalc(X, U, t, ns, n_nodes, 10, 2000.0, None)
    assert defect.shape == (6, 29) and errors.shape == (29,)
    Jf = direct.jacobianCalc(X, U, t, defect, ns, n_nodes, 10, 2000.0, None, 1e-8)
    assert Jf.shape == (6 * 29, 30 * 9)
    do, eo, Jo, _ = oracle.direct_jac_var(X.T[:-1], X.T[1:], U.T[:-1], U.T[1:], t[:-1], t[1:])
    assert np.abs(defect.T - do).max() < 1e-13
    assert np.abs(Jf[6:12, 6:18] - Jo[1][:, :12]).max() < 1e-12 and np.abs(Jf[6:12, 180 + 3:180 + 9] - Jo[1][:, 12:]).max() < 1e-12
    XC = np.vstack([X, 0.1 * np.random.default_rng(0).standard_normal((6, n_nodes))])
    params = (capi.MU, capi.DU, capi.TU, 10.0, 1000.0, 1.0, 2.0, 1.0)
    d2, e2 = indirect.defectCalc(XC, t, 6, n_nodes, None, params)
    J2 = indirect.jacobianCalc(XC, t, 6, n_nodes, None, params)
    assert d2.shape == (12, 29) and np.all(e2 == 0) and J2.shape == (12 * 29, 12 * 30)
    assert np.all(J2[:, :6] == 0) and np.array_equal(J2[12:24, 24:36], -np.eye(12))


# ------------------------------------------------------------------ one handle over several GPUs (the Julia drop-in's multi-GPU form)
def test_multi_device_handle_equals_single_device(lto):
    ndev = capi.lib().lto_device_count()
    with pytest.raises(capi.LtoError):
        capi.Handle([0, 0])                                 # a device may be listed once
    one = capi.Handle([0])
    assert one.n_devices == 1
    one.close()
    if ndev < 2:
        pytest.skip("needs 2 GPUs")
    hm = capi.Handle(list(range(min(ndev, 4))))
    assert hm.n_devices == min(ndev, 4)
    b = S.direct_batch(1000 + 37, nstate=7, seed=11)
    r1 = lto.direct(b["Xa"], b["Xb"], b["ua"], b["ub"], b["ta"], b["tb"])
    rm = hm.direct(b["Xa"], b["Xb"], b["ua"], b["ub"], b["ta"], b["tb"])
    assert np.array_equal(r1["defect"], rm["defect"]) and np.array_equal(r1["jac"], rm["jac"]) and np.array_equal(r1["errors"], rm["errors"])
    c = S.continuation_batch(n_traj=9, n_seg_per_traj=12, ndim=12)
    p = capi.indirect_params(p=1.0, rho=1.0)
    t1 = lto.indirect_traj(c["XC_all"], c["t_TU"], params=p, thrustLimit=c["thrustLimit"])
    tm = hm.indirect_traj(c["XC_all"], c["t_TU"], params=p, thrustLimit=c["thrustLimit"])
    assert np.array_equal(t1["defect"], tm["defect"]) and np.array_equal(t1["nsteps"], tm["nsteps"])
    assert np.abs(t1["phi"] - tm["phi"]).max() < 1e-12      # step control is slot-order independent; allow rounding-level differences only
    d1 = lto.direct_traj(np.zeros((3, 5, 6)) + 1.0, np.zeros((3, 5, 3)), np.tile(np.linspace(0, 0.4, 5), (3, 1)), jac=False)
    dm = hm.direct_traj(np.zeros((3, 5, 6)) + 1.0, np.zeros((3, 5, 3)), np.tile(np.linspace(0, 0.4, 5), (3, 1)), jac=False)
    assert np.array_equal(d1["defect"], dm["defect"])
    with pytest.raises(capi.LtoError):
        hm.direct_dev(capi.direct_params(), 1, 0, 7, 10, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1)   # device-pointer calls need a single-device handle
    # Newton update and batched solver: whole trajectories per device, same results as one device
    c2 = S.continuation_batch(n_traj=11, n_seg_per_traj=200, ndim=12)
    XC = c2["XC_all"].copy(); XC[:, :, 6:] *= 0.1
    p2 = capi.indirect_params(p=2.0, thrustLimit=10.0)
    s1 = lto.indirect_solve_batch(XC, c2["t_TU"], params=p2, max_iter=8)
    sm = hm.indirect_solve_batch(XC, c2["t_TU"], params=p2, max_iter=8)
    assert np.array_equal(s1["status_flag"], sm["status_flag"]) and np.array_equal(s1["iters"], sm["iters"])
    assert np.abs(s1["XC_all"] - sm["XC_all"]).max() < 1e-11
    tt1 = lto.indirect_traj(XC, c2["t_TU"], params=p2)
    u1, st1 = lto.indirect_newton(tt1["phi"].reshape(11, 200, 12, 12), tt1["defect"].reshape(11, 200, 12))
    um, stm = hm.indirect_newton(tt1["phi"].reshape(11, 200, 12, 12), tt1["defect"].reshape(11, 200, 12))
    assert np.array_equal(u1, um) and np.array_equal(st1, stm)
    assert hm.launches > 0
    hm.close()


def test_sumsq_dev_and_sharded_line_search_single_rank(lto):
    """lto_sumsq_dev = the line searches' er[ind] = sum(defect[:].^2); the sharded layer's "sumsq" mode (world 1) equals
    the defect-only pass reduced on the host."""
    import torch
    from lowthrustopt_b200 import sharded
    dev = torch.device("cuda", 0)
    v = torch.randn((37, 2400), dtype=torch.float64, device=dev)
    out = torch.empty(37, dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    lto.sumsq_dev(v.data_ptr(), 37, 2400, out.data_ptr()); lto.sync()
    ref = (v.cpu().numpy() ** 2).sum(axis=1)
    assert np.abs(out.cpu().numpy() / ref - 1.0).max() < 1e-14
    c = S.continuation_batch(n_traj=11, n_seg_per_traj=20, ndim=12)
    sh = sharded.ShardedIndirect(lto, 11, 21, 12, dev, n_chunks=2)
    sh.load(c["XC_all"], c["t_TU"], c["thrustLimit"], 1.0)
    p = capi.indirect_params(p=1.0, rho=1.0)
    d, _ = sh.run(p, jac=False)
    ls, _ = sh.run(p, mode="sumsq")
    r = lto.indirect_traj(c["XC_all"], c["t_TU"], params=p, thrustLimit=c["thrustLimit"], jac=False)
    assert np.array_equal(d["defect"].cpu().numpy().reshape(-1, 12), r["defect"])
    assert np.abs(ls["sumsq"].cpu().numpy() / (r["defect"].reshape(11, -1) ** 2).sum(axis=1) - 1.0).max() < 1e-13
    assert int(ls["bad"].max()) == 0
    j, _ = sh.run(p, jac=True)
    rj = lto.indirect_traj(c["XC_all"], c["t_TU"], params=p, thrustLimit=c["thrustLimit"], jac=True)
    assert np.abs(j["phi"].cpu().numpy().reshape(-1, 12, 12) - rj["phi"]).max() < 1e-12
