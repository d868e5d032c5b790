"""GPU: the direct kernels past their first round, against the CPU oracle and against themselves.

K1 (fixed grid) and K2 (ode78 controller) are persistent: a CTA takes pairs of 16-segment tiles, so one round is n_sm x 32 segments,
and each tile's step counter and 2-slot mbarrier ring carry over from one pair to the next.  K4 (defect only) grid-strides over
n_sm x 16 blocks x 4 warps x 16 segments per pass.  Every test below derives its sizes from the SM count and asserts its own geometry
(several rounds / passes, a partial last one, an odd tile count, n % 16 != 0) before it checks a number, so it cannot shrink to one
round on another part.  Besides the oracle, results are compared BITWISE with the same rows launched in slices of at most one round
(one pair per CTA): a change that only touches round 2 and later and stays inside the oracle's bar is caught there.

Device tensors go through Handle.direct_dev, so one call is one launch of known shape.  With LTO_TEST_REPORT_DIR set, the worst error
of every case (and its segment) is written to $LTO_TEST_REPORT_DIR/direct_scale.json (profiles/r09_direct_scale.json is such a report).
"""
import json
import os

import numpy as np
import pytest

from lowthrustopt_b200 import capi, synthetic as S

pytestmark = pytest.mark.gpu
TOL_STATE, TOL_JAC = 1e-10, 1e-8
ST_OK, ST_NAN, ST_HMIN, ST_MAXSTEPS = 0, 1, 2, 3
REPORT = {}


def _note(key, **kw):
    REPORT[key] = {k: (float(v) if isinstance(v, (float, np.floating)) else int(v) if isinstance(v, (int, np.integer)) else v) for k, v in kw.items()}
    out = os.environ.get("LTO_TEST_REPORT_DIR")
    if not out:
        return
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, "direct_scale.json"), "w") as f:
        json.dump(REPORT, f, indent=1, sort_keys=True)


# ------------------------------------------------------------------ geometry
@pytest.fixture(scope="module")
def n_sm():
    import torch
    return int(torch.cuda.get_device_properties(0).multi_processor_count)


def _cw_round(n_sm):
    return n_sm * 32                                        # K1 / K2: segments per round (one pair of 16-segment tiles per CTA)


def _k4_pass(n_sm):
    return n_sm * 16 * 4 * 16                               # K4: blocks x warps x segments per grid-stride pass


def _cw_size(n_sm, rounds=3.3):
    """About `rounds` rounds, n % 16 != 0 and an odd tile count (the last pair has a tile past n_tiles)."""
    n = int(rounds * _cw_round(n_sm))
    n = n - n % 16 + 5
    if ((n + 15) // 16) % 2 == 0:
        n += 16
    return n


def _assert_cw_geometry(n, n_sm, min_rounds=3):
    n_tiles = (n + 15) // 16
    n_pairs = (n_tiles + 1) // 2
    rounds = -(-n_pairs // n_sm)
    assert n % 16 != 0 and n_tiles % 2 == 1, (n, n_tiles)
    assert rounds >= min_rounds and n_pairs % n_sm != 0, (n, n_pairs, n_sm)     # several rounds, the last one partial
    return rounds


def _assert_k4_geometry(n, n_sm):
    n_warps = (n + 15) // 16
    per_pass = n_sm * 16 * 4
    passes = -(-n_warps // per_pass)
    assert n % 16 != 0 and passes >= 3 and n_warps % per_pass != 0, (n, n_warps, per_pass)
    return passes


def _slices(n, step):
    return [slice(lo, min(n, lo + step)) for lo in range(0, n, step)]


# ------------------------------------------------------------------ device calls
def _dev(lto, b, ns, nsteps, params, jac=True, rows=None):
    """One direct_dev launch (pairs form) over the rows `rows` (default: all) of batch b; numpy results."""
    import torch
    dev = torch.device("cuda", 0)
    sl = rows if rows is not None else slice(None)
    t = {k: torch.from_numpy(np.ascontiguousarray(b[k][sl])).to(dev) for k in ("Xa", "Xb", "ua", "ub", "ta", "tb")}
    n = t["Xa"].shape[0]
    o = dict(defect=torch.full((n, ns), -1.0, dtype=torch.float64, device=dev), errors=torch.full((n,), -1.0, dtype=torch.float64, device=dev),
             status=torch.full((n,), -1, dtype=torch.int32, device=dev))
    if jac:
        o["jac"] = torch.full((n, 2 * (ns + 3), ns), -1.0, dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    lto.direct_dev(params, n, 0, ns, nsteps, t["Xa"].data_ptr(), t["Xb"].data_ptr(), t["ua"].data_ptr(), t["ub"].data_ptr(),
                   t["ta"].data_ptr(), t["tb"].data_ptr(), o["defect"].data_ptr(), o["errors"].data_ptr(), o["status"].data_ptr(),
                   o["jac"].data_ptr() if jac else None)
    lto.sync()
    return {k: v.cpu().numpy() for k, v in o.items()}


def _dev_traj(lto, X, U, T, ns, nsteps, params, jac=True):
    """One direct_dev launch in the trajectory form (n_nodes > 0)."""
    import torch
    dev = torch.device("cuda", 0)
    n_traj, n_nodes = T.shape
    n = n_traj * (n_nodes - 1)
    x, u, t = (torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (X, U, T))
    o = dict(defect=torch.full((n, ns), -1.0, dtype=torch.float64, device=dev), errors=torch.full((n,), -1.0, dtype=torch.float64, device=dev),
             status=torch.full((n,), -1, dtype=torch.int32, device=dev))
    if jac:
        o["jac"] = torch.full((n, 2 * (ns + 3), ns), -1.0, dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    lto.direct_dev(params, n, n_nodes, ns, nsteps, x.data_ptr(), None, u.data_ptr(), None, t.data_ptr(), None, o["defect"].data_ptr(),
                   o["errors"].data_ptr(), o["status"].data_ptr(), o["jac"].data_ptr() if jac else None)
    lto.sync()
    return {k: v.cpu().numpy() for k, v in o.items()}


def _bitwise(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


def _first_diff(a, b):
    d = np.ascontiguousarray(a).view(np.uint8).reshape(len(a), -1) != np.ascontiguousarray(b).view(np.uint8).reshape(len(b), -1)
    rows = np.nonzero(d.any(axis=1))[0]
    return (len(rows), int(rows[0]) if len(rows) else -1)


def _assert_equal_results(r, q, keys, what):
    for k in keys:
        assert _bitwise(r[k], q[k]), (what, k, "rows differing, first:", _first_diff(r[k], q[k]))


def _sliced(lto, b, ns, nsteps, params, step, jac=True):
    """The same rows, launched in slices of `step` segments; concatenated."""
    parts = [_dev(lto, b, ns, nsteps, params, jac=jac, rows=sl) for sl in _slices(len(b["ta"]), step)]
    return {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}


def _batch(n, ns, seed):
    b = S.direct_batch(n, nstate=ns, seed=seed)
    b["ua"][::23] = 0.0                                     # |u| = 0 rows: the one-sided mass-flow slope
    b["ub"][5::37] = 0.0
    return b


def _xscale(b):
    return np.maximum(1.0, np.maximum(np.abs(b["Xa"]), np.abs(b["Xb"])))


# ------------------------------------------------------------------ a. K1 past one round
K1_CASES = [(ns, k) for ns in (6, 7) for k in (2, 3, 10, 11)] + [(7, 25)]


@pytest.mark.parametrize("ns,nsteps", K1_CASES)
def test_k1_multi_round_vs_oracle_and_one_round_slices(ns, nsteps, n_sm, lto, oracle):
    n = _cw_size(n_sm)
    rounds = _assert_cw_geometry(n, n_sm)
    b = _batch(n, ns, seed=3100 + 10 * ns + nsteps)
    p = capi.direct_params()
    r = _dev(lto, b, ns, nsteps, p)
    do, eo, Jo, so = oracle.direct_jac_var(b["Xa"], b["Xb"], b["ua"], b["ub"], b["ta"], b["tb"], nsteps=nsteps, nthreads=oracle.num_threads())
    ed = (np.abs(r["defect"] - do) / _xscale(b)).max(axis=1)
    ej = (np.abs(r["jac"].transpose(0, 2, 1) - Jo) / np.maximum(1.0, np.abs(Jo))).reshape(n, -1).max(axis=1)
    ee = np.abs(r["errors"] - eo)
    q = _sliced(lto, b, ns, nsteps, p, _cw_round(n_sm))
    same = all(_bitwise(r[k], q[k]) for k in ("defect", "errors", "status", "jac"))
    _note("k1_ns%d_nsteps%d" % (ns, nsteps), n=n, rounds=rounds, defect_max=ed.max(), defect_argmax=int(ed.argmax()), jac_max=ej.max(),
          jac_argmax=int(ej.argmax()), errors_max=ee.max(), bitwise_one_round_slices=same)
    assert np.all(r["status"] == ST_OK) and np.all(so == 0)
    assert ed.max() < 1e-13 and ej.max() < 1e-12 and ee.max() < 2e-14
    _assert_equal_results(r, q, ("defect", "errors", "status", "jac"), "K1 vs one-round slices")


@pytest.mark.parametrize("ns,nsteps", [(7, 10), (6, 11)])
def test_k1_trajectory_form_multi_round_equals_pairs_form(ns, nsteps, n_sm, lto):
    n_nodes = 30
    n_traj = _cw_size(n_sm) // (n_nodes - 1) | 1
    while (((n_traj * (n_nodes - 1)) + 15) // 16) % 2 == 0:
        n_traj += 2
    n = n_traj * (n_nodes - 1)
    rounds = _assert_cw_geometry(n, n_sm)
    rng = np.random.default_rng(3200 + ns)
    X = np.empty((n_traj, n_nodes, ns)); T = np.empty((n_traj, n_nodes))
    tau0 = rng.uniform(size=n_traj)
    grid = np.linspace(0.0, 4.6, n_nodes)
    X[:, :, :6] = S.interp_initial_states((tau0[:, None] + grid[None] / S.PERIODS[0]).ravel(), 1).reshape(n_traj, n_nodes, 6)
    X[:, :, :6] += 1e-3 * rng.standard_normal((n_traj, n_nodes, 6))
    if ns == 7:
        X[:, :, 6] = 1000.0 - np.linspace(0.0, 1.0, n_nodes)
    T[:] = grid[None] + rng.uniform(size=(n_traj, 1))
    U = 0.05 * rng.standard_normal((n_traj, n_nodes, 3))
    U[::7, 3] = 0.0
    p = capi.direct_params()
    rt = _dev_traj(lto, X, U, T, ns, nsteps, p)
    b = dict(Xa=X[:, :-1].reshape(-1, ns), Xb=X[:, 1:].reshape(-1, ns), ua=U[:, :-1].reshape(-1, 3), ub=U[:, 1:].reshape(-1, 3),
             ta=T[:, :-1].ravel(), tb=T[:, 1:].ravel())
    rp = _dev(lto, b, ns, nsteps, p)
    _note("k1_traj_ns%d_nsteps%d" % (ns, nsteps), n=n, n_traj=n_traj, n_nodes=n_nodes, rounds=rounds)
    assert np.all(rt["status"] == ST_OK)
    _assert_equal_results(rt, rp, ("defect", "errors", "status", "jac"), "K1 trajectory form vs pairs form")


# ------------------------------------------------------------------ b. K2 past one round, divergent step counts
def _k2_batch(n, ns, seed):
    """Tiles of short legs (spans 1e-4 .. 1e-2 TU: 4-5 attempts, h is capped at span / 2.5) and tiles that mix them with long legs
    (1 .. 4 TU: up to ~150 attempts), spans of exactly 0 and 1e-9 TU, controls of 0 and up to 1 N.  Long tiles are drawn at random,
    so the two tiles of a CTA often finish at different steps."""
    rng = np.random.default_rng(seed)
    b = S.direct_batch(n, nstate=ns, seed=seed)
    k = np.arange(n)
    long_tile = rng.uniform(size=(n + 15) // 16) < 0.5
    span = np.exp(rng.uniform(np.log(1e-4), np.log(1e-2), n))
    lng = long_tile[k // 16] & (rng.uniform(size=n) < 0.5)
    span[lng] = np.exp(rng.uniform(np.log(1.0), np.log(4.0), int(lng.sum())))
    span[rng.uniform(size=n) < 0.04] = 0.0
    span[rng.uniform(size=n) < 0.04] = 1e-9
    mag = np.where(rng.uniform(size=(n, 1)) < 0.25, 0.0, rng.uniform(0.0, 1.0, (n, 1)))
    d = rng.standard_normal((n, 3)); d /= np.linalg.norm(d, axis=1, keepdims=True)
    e = rng.standard_normal((n, 3)); e /= np.linalg.norm(e, axis=1, keepdims=True)
    b["ua"] = mag * d; b["ub"] = mag * e
    b["tb"] = b["ta"] + span
    return b


def _k2_params(tol=1e-12, max_attempts=0, kernel=capi.LTO_KERNEL_AUTO):
    p = capi.direct_params(mode=capi.LTO_ADAPTIVE, tol=tol, err_norm=capi.LTO_NORM_STATE, kernel=kernel)
    p.max_attempts = max_attempts
    return p


# The controller accepts a step when its error estimate is below tol * max(|x|, 1) (ode.jl:513).  With nstate 7, |x| is the mass
# (~1e3 kg), so tol = 1e-12 would hold r and v to ~1e-9 only: the oracle itself then moves by more than 1e-10 between tol and tol / 100 on
# a quarter of these legs (measured on the CPU: 3 588 of 15 621 rows).  nstate 7 runs at 1e-14 (16 such rows).  Not 1e-15: its tol / 100
# run is at the rounding floor of r and v, so it no longer measures the oracle's own error.
K2_TOL = {6: 1e-12, 7: 1e-14}


@pytest.mark.parametrize("ns", [6, 7])
def test_k2_multi_round_divergent_steps(ns, n_sm, lto, oracle):
    n = _cw_size(n_sm)
    rounds = _assert_cw_geometry(n, n_sm)
    b = _k2_batch(n, ns, seed=3300 + ns)
    args = (b["Xa"], b["Xb"], b["ua"], b["ub"], b["ta"], b["tb"])
    nth = oracle.num_threads()
    tol = K2_TOL[ns]
    _, _, so_d, att = oracle.direct_defect(*args, mode=1, tol=tol, nthreads=nth)             # attempts per leg [forward, backward]
    assert np.all(so_d == 0)
    # the spread is real: legs of one tile finish many steps apart, and the two tiles of a CTA at different steps
    ta_ = att[: n // 16 * 16].reshape(-1, 32)
    tmax, tmin = ta_.max(axis=1), ta_.min(axis=1)
    spread = tmax / np.maximum(tmin, 1)
    pair_max = tmax[: len(tmax) // 2 * 2].reshape(-1, 2)
    frac_spread, frac_pair = np.mean(spread >= 10), np.mean(pair_max[:, 0] != pair_max[:, 1])
    assert frac_spread >= 0.2 and frac_pair >= 0.5 and att.max() >= 50, (frac_spread, frac_pair, att.max())

    p = _k2_params(tol=tol)
    r = _dev(lto, b, ns, 10, p)
    do, eo, Jo, so = oracle.direct_jac_var(*args, mode=1, tol=tol, nthreads=nth)
    xs = _xscale(b)
    ed = (np.abs(r["defect"] - do) / xs).max(axis=1)
    ej = (np.abs(r["jac"].transpose(0, 2, 1) - Jo) / np.maximum(1.0, np.abs(Jo))).reshape(n, -1).max(axis=1)
    # Two correct order-8 runs whose step sequences differ (the kernel's error estimate is the Nystrom form's) may differ by more than
    # the bar after long legs: there the kernel is held to 5 x the oracle's own distance from a run at tol / 100.
    out = np.nonzero((ed >= TOL_STATE) | (ej >= TOL_JAC))[0]
    exc_ok = True
    if len(out):
        sub = tuple(a[out] for a in args)
        d2, _, J2, s2 = oracle.direct_jac_var(*sub, mode=1, tol=tol / 100, nthreads=nth)
        bd = np.maximum(TOL_STATE, 5.0 * (np.abs(do[out] - d2) / xs[out]).max(axis=1))
        bj = np.maximum(TOL_JAC, 5.0 * (np.abs(Jo[out] - J2) / np.maximum(1.0, np.abs(Jo[out]))).reshape(len(out), -1).max(axis=1))
        exc_ok = bool(np.all(ed[out] < bd) and np.all(ej[out] < bj))

    # bitwise against one-round slices
    q = _sliced(lto, b, ns, 10, p, _cw_round(n_sm))
    same = all(_bitwise(r[k], q[k]) for k in ("defect", "status", "jac"))

    # max_attempts: legs clearly above the cap fail with LTO_ST_MAXSTEPS; rows whose legs are clearly below it are bitwise the uncapped run
    cap, margin = 30, 3
    rc = _dev(lto, b, ns, 10, _k2_params(tol=tol, max_attempts=cap))
    amax = att.max(axis=1)
    above, below = amax >= cap + margin, amax <= cap - margin
    excluded = int((~above & ~below).sum())
    _note("k2_ns%d" % ns, n=n, rounds=rounds, tol=tol, attempts_max=int(att.max()), tiles_spread10=frac_spread, pairs_differ=frac_pair,
          defect_max=ed.max(), defect_argmax=int(ed.argmax()), jac_max=ej.max(), jac_argmax=int(ej.argmax()), beyond_bar_judged_vs_tol100=len(out),
          beyond_bar_rows=[int(i) for i in out[:20]],
          bitwise_one_round_slices=same, cap=cap, cap_rows_above=int(above.sum()), cap_rows_below=int(below.sum()), cap_rows_excluded=excluded)
    assert np.all(r["status"] == ST_OK) and np.all(so == 0)
    assert exc_ok and len(out) <= max(5, n // 1000), out[:20]
    _assert_equal_results(r, q, ("defect", "errors", "status", "jac"), "K2 vs one-round slices")
    assert above.sum() >= 50 and below.sum() >= n // 2 and excluded <= n // 20, (above.sum(), below.sum(), excluded)
    assert np.all(rc["status"][above] == ST_MAXSTEPS)
    for k in ("defect", "errors", "status", "jac"):
        assert _bitwise(rc[k][below], r[k][below]), ("capped vs uncapped", k, _first_diff(rc[k][below], r[k][below]))


# ------------------------------------------------------------------ c. K4 past one pass
@pytest.mark.parametrize("ns", [6, 7])
def test_k4_multi_pass_vs_oracle_and_host_chunks(ns, n_sm, lto, oracle):
    n = int(2.5 * _k4_pass(n_sm))
    n = n - n % 16 + 7
    passes = _assert_k4_geometry(n, n_sm)
    nsteps = 4
    b = _batch(n, ns, seed=3400 + ns)
    p = capi.direct_params()
    r = _dev(lto, b, ns, nsteps, p, jac=False)
    do, eo, so, _ = oracle.direct_defect(b["Xa"], b["Xb"], b["ua"], b["ub"], b["ta"], b["tb"], nsteps=nsteps, nthreads=oracle.num_threads())
    ed = (np.abs(r["defect"] - do) / _xscale(b)).max(axis=1)
    ee = np.abs(r["errors"] - eo)
    plan = capi.host_chunk_plan("direct", n, nvar=ns, nsteps=nsteps, jac=False, n_sm=n_sm)
    h = lto.direct(b["Xa"], b["Xb"], b["ua"], b["ub"], b["ta"], b["tb"], nsteps=nsteps, jac=False)   # pageable: staged two-wave chunks
    _note("k4_ns%d" % ns, n=n, passes=passes, defect_max=ed.max(), defect_argmax=int(ed.argmax()), errors_max=ee.max(),
          host_plan_pinned=len(plan), bitwise_host=all(_bitwise(r[k], h[k]) for k in ("defect", "errors", "status")))
    assert len(plan) >= 2 and max(plan) < _k4_pass(n_sm) and 2 * _cw_round(n_sm) < _k4_pass(n_sm)   # host launches stay inside one pass
    assert np.all(r["status"] == ST_OK) and np.all(so == 0)
    assert ed.max() < 1e-13 and ee.max() < 2e-14
    _assert_equal_results(r, h, ("defect", "errors", "status"), "K4 direct_dev vs host chunks")


# ------------------------------------------------------------------ d. host pipeline
def _host_rounds(n_sm):
    """Rounds of a host-pipeline batch: at least 6.3, and at least 30 000 segments (about four times the 8 MiB one-shot limit)."""
    return max(6.3, 30000.0 / _cw_round(n_sm))


def _staged_plan(n, unit, n_sm):
    """The chunks of a host call with pageable inputs: the library stages them itself, in equal two-wave chunks of whole units."""
    c = max(unit, -(-2 * _cw_round(n_sm) // unit) * unit)
    plan, left = [], n
    while left > 0:
        take = left if left < c + c // 2 else c
        plan.append(take); left -= take
    return plan


def _pinned(a):
    o = capi._POOL.empty(a.shape, a.dtype)
    o[...] = a
    return o


def _check_chunks(r, q, plan, keys, what):
    """Every chunk boundary of the plan, explicitly: the rows on both sides agree (the whole arrays are compared as well)."""
    b0 = 0
    for c in plan[:-1]:
        b0 += c
        sl = slice(max(0, b0 - 40), b0 + 40)
        for k in keys:
            assert _bitwise(r[k][sl], q[k][sl]), (what, "chunk boundary", b0, k)
    _assert_equal_results(r, q, keys, what)


@pytest.mark.parametrize("ns,pinned,mode", [(6, False, 0), (7, False, 0), (7, True, 0), (7, True, 1)])
def test_host_pairs_pipeline_equals_dev(ns, pinned, mode, n_sm, lto):
    n = _cw_size(n_sm, rounds=_host_rounds(n_sm))
    _assert_cw_geometry(n, n_sm, min_rounds=6)
    b = _k2_batch(n, ns, seed=3500 + ns) if mode else _batch(n, ns, seed=3500 + ns)
    p = _k2_params() if mode else capi.direct_params()
    plan_pinned = capi.host_chunk_plan("direct", n, nvar=ns, nsteps=10, mode=mode, n_sm=n_sm)
    plan = plan_pinned if pinned else _staged_plan(n, 1, n_sm)
    assert len(plan) >= 3 and sum(plan) == n, plan
    args = [_pinned(b[k]) if pinned else b[k] for k in ("Xa", "Xb", "ua", "ub", "ta", "tb")]
    r = lto.direct(*args, nsteps=10, params=p)
    q = _dev(lto, b, ns, 10, p)
    _note("host_pairs_ns%d_%s_%s" % (ns, "pinned" if pinned else "pageable", "adaptive" if mode else "fixed"), n=n, chunks=len(plan))
    assert np.all(q["status"] == ST_OK)
    _check_chunks(r, q, plan, ("defect", "errors", "status", "jac"), "host pairs form vs direct_dev")


@pytest.mark.parametrize("pinned", [False, True])
def test_host_traj_pipeline_equals_dev(pinned, n_sm, lto):
    ns, n_nodes = 7, 31                                     # 30 segments per trajectory: does not divide the wave
    assert (n_sm * 32) % (n_nodes - 1) != 0
    n_traj = (_cw_size(n_sm, rounds=_host_rounds(n_sm)) // (n_nodes - 1)) | 1
    n = n_traj * (n_nodes - 1)
    rng = np.random.default_rng(3600 + pinned)
    grid = np.linspace(0.0, 3.0, n_nodes)
    tau0 = rng.uniform(size=n_traj)
    X = np.empty((n_traj, n_nodes, ns))
    X[:, :, :6] = S.interp_initial_states((tau0[:, None] + grid[None] / S.PERIODS[1]).ravel(), 2).reshape(n_traj, n_nodes, 6)
    X[:, :, :6] += 1e-3 * rng.standard_normal((n_traj, n_nodes, 6))
    X[:, :, 6] = 1000.0 - np.linspace(0.0, 2.0, n_nodes)
    U = 0.05 * rng.standard_normal((n_traj, n_nodes, 3))
    T = grid[None] + rng.uniform(size=(n_traj, 1))
    plan = capi.host_chunk_plan("direct", n, n_nodes=n_nodes, nvar=ns, nsteps=10, n_sm=n_sm)
    assert len(plan) >= 2 and all(c % (n_nodes - 1) == 0 for c in plan), plan           # whole trajectories per chunk
    args = [_pinned(a) if pinned else a for a in (X, U, T)]
    r = lto.direct_traj(*args, nsteps=10)
    q = _dev_traj(lto, X, U, T, ns, 10, capi.direct_params())
    if not pinned:
        plan = _staged_plan(n, n_nodes - 1, n_sm)
    _note("host_traj_ns%d_%s" % (ns, "pinned" if pinned else "pageable"), n=n, n_traj=n_traj, chunks=len(plan))
    assert np.all(q["status"] == ST_OK)
    _check_chunks(r, q, plan, ("defect", "errors", "status", "jac"), "host trajectory form vs direct_dev")


# ------------------------------------------------------------------ e. spans
NAN, INF = float("nan"), float("inf")


def _special_rows(n, round_):
    """Row -> (ta, tb) replacement: NaN ta, NaN tb, +-inf, zero length, reversed; in the first round and in tiles past it."""
    kinds = [("nan_ta", lambda ta, tb: (NAN, tb)), ("nan_tb", lambda ta, tb: (ta, NAN)), ("inf_tb", lambda ta, tb: (ta, INF)),
             ("minus_inf_ta", lambda ta, tb: (-INF, tb)), ("inf_ta", lambda ta, tb: (INF, tb)), ("inf_minus_inf", lambda ta, tb: (INF, -INF)),
             ("zero", lambda ta, tb: (ta, ta)), ("reversed", lambda ta, tb: (tb, ta))]
    rows = {}
    for i, (name, f) in enumerate(kinds):
        for base in (37, round_ + 101, 2 * round_ + 515, 3 * round_ + 17):
            if base + 3 * len(kinds) < n:
                rows[base + 3 * i] = (name, f)
    return rows


def _apply_spans(b, rows):
    c = {k: v.copy() for k, v in b.items()}
    for i, (name, f) in rows.items():
        c["ta"][i], c["tb"][i] = f(b["ta"][i], b["tb"][i])
    return c


def _check_spans(r, r0, c, rows, mode, oracle, ns, nsteps, jac, what):
    idx = np.array(sorted(rows))
    names = np.array([rows[i][0] for i in idx])
    clean = np.ones(len(r["status"]), bool); clean[idx] = False
    keys = ("defect", "errors", "status") + (("jac",) if jac else ())
    for k in keys:
        assert _bitwise(r[k][clean], r0[k][clean]), (what, "clean rows changed", k, _first_diff(r[k][clean], r0[k][clean]))
    st = r["status"][idx]
    nonfinite = np.array([n not in ("zero", "reversed") for n in names])
    assert np.all(st[nonfinite] == ST_NAN), (what, list(zip(names[nonfinite], st[nonfinite])))
    rev = names == "reversed"
    if mode == 1:
        assert np.all(st[rev] != ST_OK), (what, st[rev])
        ok = names == "zero"
    else:
        ok = (names == "zero") | rev
    assert np.all(st[ok] == ST_OK), (what, list(zip(names[ok], st[ok])))
    sub = idx[ok]
    args = tuple(c[k][sub] for k in ("Xa", "Xb", "ua", "ub", "ta", "tb"))
    do, eo, Jo, so = oracle.direct_jac_var(*args, nsteps=nsteps, mode=mode, tol=1e-12)
    xs = np.maximum(1.0, np.maximum(np.abs(args[0]), np.abs(args[1])))
    assert (np.abs(r["defect"][sub] - do) / xs).max() < 1e-13, what
    if jac:
        assert (np.abs(r["jac"][sub].transpose(0, 2, 1) - Jo) / np.maximum(1.0, np.abs(Jo))).max() < 1e-12, what
    if mode == 0:
        assert np.abs(r["errors"][sub] - eo).max() < 2e-14, what


SPAN_PATHS = [("K1", 0, True, capi.LTO_KERNEL_AUTO), ("K2", 1, True, capi.LTO_KERNEL_AUTO), ("K4", 0, False, capi.LTO_KERNEL_AUTO),
              ("generic_fixed", 0, True, capi.LTO_KERNEL_GENERIC), ("generic_fixed_nojac", 0, False, capi.LTO_KERNEL_GENERIC),
              ("generic_adaptive", 1, True, capi.LTO_KERNEL_GENERIC), ("generic_adaptive_nojac", 1, False, capi.LTO_KERNEL_GENERIC)]


@pytest.mark.parametrize("name,mode,jac,kernel", SPAN_PATHS)
@pytest.mark.parametrize("ns", [6, 7])
def test_direct_special_spans(ns, name, mode, jac, kernel, n_sm, lto, oracle):
    nsteps = 10
    if name == "K4":
        n = int(2.5 * _k4_pass(n_sm)); n = n - n % 16 + 7
        _assert_k4_geometry(n, n_sm)
        rows = _special_rows(n, _k4_pass(n_sm))
    else:
        n = _cw_size(n_sm)
        _assert_cw_geometry(n, n_sm)
        rows = _special_rows(n, _cw_round(n_sm))
    b = _batch(n, ns, seed=3700 + ns)
    c = _apply_spans(b, rows)
    p = _k2_params(kernel=kernel) if mode else capi.direct_params(kernel=kernel)
    # device entry point
    r0 = _dev(lto, b, ns, nsteps, p, jac=jac)
    r = _dev(lto, c, ns, nsteps, p, jac=jac)
    _check_spans(r, r0, c, rows, mode, oracle, ns, nsteps, jac, name + " direct_dev")
    # host pairs form (chunked for the Jacobian paths)
    h0 = lto.direct(*(b[k] for k in ("Xa", "Xb", "ua", "ub", "ta", "tb")), nsteps=nsteps, params=p, jac=jac)
    h = lto.direct(*(c[k] for k in ("Xa", "Xb", "ua", "ub", "ta", "tb")), nsteps=nsteps, params=p, jac=jac)
    _check_spans(h, h0, c, rows, mode, oracle, ns, nsteps, jac, name + " host pairs")
    _note("spans_%s_ns%d" % (name, ns), n=n, special_rows=len(rows), statuses=sorted(set((rows[i][0], int(r["status"][i])) for i in rows)))


@pytest.mark.parametrize("name,mode,jac,kernel", SPAN_PATHS)
def test_direct_special_spans_traj_form(name, mode, jac, kernel, n_sm, lto, oracle):
    """Trajectory form (host and device): a NaN node time makes both segments that share the node NaN; a reversed or zero-length
    node interval is one segment."""
    ns, n_nodes = 7, 31
    n_traj = (_cw_size(n_sm) // (n_nodes - 1)) | 1
    n = n_traj * (n_nodes - 1)
    _assert_cw_geometry(n, n_sm)
    rng = np.random.default_rng(3800)
    grid = np.linspace(0.0, 3.0, n_nodes)
    X = np.empty((n_traj, n_nodes, ns))
    X[:, :, :6] = S.interp_initial_states((rng.uniform(size=(n_traj, 1)) + grid[None] / S.PERIODS[0]).ravel(), 1).reshape(n_traj, n_nodes, 6)
    X[:, :, 6] = 1000.0 - np.linspace(0.0, 1.0, n_nodes)
    U = 0.05 * rng.standard_normal((n_traj, n_nodes, 3))
    T0 = grid[None] + rng.uniform(size=(n_traj, 1))
    T = T0.copy()
    last = n_traj - 2                                       # a trajectory in the last round
    T[1, 5] = NAN; T[last, 7] = NAN; T[last, 20] = INF
    T[2, 9] = T[2, 8]                                       # zero-length segment 8
    T[last, 12] = T[last, 11] - 0.05                        # reversed segment 11 (segment 12 gets longer, still forwards)
    special = {1 * 30 + 4: "nan", 1 * 30 + 5: "nan", last * 30 + 6: "nan", last * 30 + 7: "nan", last * 30 + 19: "nan", last * 30 + 20: "nan",
               2 * 30 + 8: "zero", 2 * 30 + 9: "changed", last * 30 + 11: "reversed", last * 30 + 12: "changed"}
    p = _k2_params(kernel=kernel) if mode else capi.direct_params(kernel=kernel)
    for how in ("dev", "host"):
        if how == "dev":
            r0 = _dev_traj(lto, X, U, T0, ns, 10, p, jac=jac); r = _dev_traj(lto, X, U, T, ns, 10, p, jac=jac)
        else:
            r0 = lto.direct_traj(X, U, T0, nsteps=10, params=p, jac=jac); r = lto.direct_traj(X, U, T, nsteps=10, params=p, jac=jac)
        clean = np.ones(n, bool); clean[list(special)] = False
        for k in ("defect", "errors", "status") + (("jac",) if jac else ()):
            assert _bitwise(r[k][clean], r0[k][clean]), (name, how, k, _first_diff(r[k][clean], r0[k][clean]))
        for s, kind in special.items():
            st = int(r["status"][s])
            if kind == "nan":
                assert st == ST_NAN, (name, how, s, st)
            elif kind == "reversed" and mode == 1:
                assert st != ST_OK, (name, how, s, st)
            else:
                assert st == ST_OK, (name, how, s, kind, st)
        chk = [s for s, kind in special.items() if kind in ("zero", "changed") or (kind == "reversed" and mode == 0)]
        j, k_ = np.array(chk) // 30, np.array(chk) % 30
        do, eo, Jo, so = oracle.direct_jac_var(X[j, k_], X[j, k_ + 1], U[j, k_], U[j, k_ + 1], T[j, k_], T[j, k_ + 1], mode=mode, tol=1e-12)
        xs = np.maximum(1.0, np.maximum(np.abs(X[j, k_]), np.abs(X[j, k_ + 1])))
        tol = 1e-13 if mode == 0 else TOL_STATE                # the adaptive "changed" segment is a longer leg: ode78 vs the oracle
        assert (np.abs(r["defect"][chk] - do) / xs).max() < tol, (name, how)
    _note("spans_traj_%s" % name, n=n, n_traj=n_traj)


@pytest.mark.parametrize("nd", [12, 14])
def test_indirect_host_refuses_nonfinite_spans(nd, lto):
    b = S.indirect_batch(8, ndim=nd, seed=3900)
    p = capi.indirect_params(p=1.0, rho=1.0, thrustLimit=0.05)
    for field, val in (("t0", NAN), ("t1", NAN), ("t1", INF), ("t0", -INF)):
        for jac in (True, False):
            t0, t1 = b["t0"].copy(), b["t1"].copy()
            (t0 if field == "t0" else t1)[5] = val
            with pytest.raises(capi.LtoError, match="segment 5 has a non-finite or reversed span"):
                lto.indirect(b["x0"], t0, t1, params=p, jac=jac)
    c = S.continuation_batch(n_traj=3, n_seg_per_traj=12, ndim=nd)
    for node, seg in ((4, 3), (0, 0), (12, 11)):
        t = c["t_TU"].copy(); t[1, node] = NAN
        with pytest.raises(capi.LtoError, match="segment %d has a non-finite or reversed span" % (12 + seg)):
            lto.indirect_traj(c["XC_all"], t, params=p, thrustLimit=c["thrustLimit"])
    r = lto.indirect(b["x0"], b["t0"], b["t1"], params=p)                # the clean batch still runs
    assert np.all(r["status"] == ST_OK)
