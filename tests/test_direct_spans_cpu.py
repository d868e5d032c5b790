"""CPU: the span rules of the generic arithmetic (lto_prop_generic.cuh), built for the host as a TEST-ONLY library.

The adaptive controllers' loop conditions (t < tfinal, h >= hmin) are false for a NaN end time and for a reversed span; a leg must
then be flagged, never handed back as x0 with status OK:
  * direct, adaptive: non-finite span -> LTO_ST_NAN, reversed -> LTO_ST_HMIN, zero-length -> OK with x0;
  * direct, fixed grid: non-finite span -> LTO_ST_NAN, reversed -> integrated backwards, OK and equal to the oracle's ode7_8;
  * indirect, both controllers (RMS = drive_rk8, ODE78 = drive_ode78): non-finite span -> not OK.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import ptr
from lowthrustopt_b200 import synthetic as S

ST_OK, ST_NAN, ST_HMIN = 0, 1, 2
NAN, INF = float("nan"), float("inf")
NONFINITE = [(NAN, 0.1), (0.1, NAN), (NAN, NAN), (0.1, INF), (INF, 0.1), (-INF, 0.1), (0.1, -INF), (INF, -INF), (-INF, INF), (INF, INF)]


def _leg(hostcheck, oracle, ns, x0, u, back, t0, t1, mode, sens=1):
    xe = np.full(ns, -7.0); Sm = np.full((ns + 3, ns), -7.0); me = C.c_double(-1.0); na = C.c_int(-1)
    st = hostcheck.hc_ep_leg(ns, sens, ptr(x0), ptr(u), back, C.c_double(t0), C.c_double(t1), mode, 10, C.c_double(1e-12), 0,
                             ptr(oracle.dparams()), ptr(xe), ptr(Sm), C.byref(me), C.byref(na))
    return st, xe, Sm, me.value, na.value


@pytest.mark.parametrize("ns", [6, 7])
@pytest.mark.parametrize("span", NONFINITE)
def test_direct_nonfinite_span_is_nan(span, ns, oracle, hostcheck):
    b = S.direct_batch(2, nstate=ns, seed=41)
    t0, t1 = span
    for mode in (0, 1):
        for back in (0, 1):
            st, xe, Sm, me, na = _leg(hostcheck, oracle, ns, b["Xa"][back], b["ua"][back], back, t0, t1, mode)
            assert st == ST_NAN, (mode, back, span, st)
            if mode == 1:
                assert na == 0                              # never integrated


@pytest.mark.parametrize("ns", [6, 7])
def test_direct_adaptive_reversed_and_zero_span(ns, oracle, hostcheck):
    b = S.direct_batch(3, nstate=ns, seed=42)
    for s in range(3):
        for back in (0, 1):
            x0 = b["Xa"][s] if back == 0 else b["Xb"][s]
            u = b["ua"][s] if back == 0 else b["ub"][s]
            ta = b["ta"][s]
            st, xe, Sm, me, na = _leg(hostcheck, oracle, ns, x0, u, back, ta, ta - 0.07, 1)
            assert st == ST_HMIN and na == 0, (s, back, st, na)
            st, xe, Sm, me, na = _leg(hostcheck, oracle, ns, x0, u, back, ta, ta, 1)
            assert st == ST_OK and na == 0
            assert np.array_equal(xe, x0)                   # both legs are returned in the defect's frame: x0 itself
            assert np.array_equal(Sm.T, np.hstack([np.eye(ns), np.zeros((ns, 3))]))


@pytest.mark.parametrize("ns", [6, 7])
def test_direct_segment_spans_vs_oracle(ns, oracle, hostcheck):
    """Whole segments (both legs, the defect) at the host-compiled arithmetic: a reversed span on the fixed grid is the oracle's backwards
    ode7_8, a zero span is OK in both modes and an adaptive reversed span is flagged."""
    n = 6
    b = S.direct_batch(n, nstate=ns, seed=43)
    ta = b["ta"].copy(); tb = b["tb"].copy()
    tb[:3] = ta[:3] - (tb[:3] - ta[:3])                  # reversed
    tb[3:] = ta[3:]                                        # zero length
    for mode in (0, 1):
        do, eo, so, steps = oracle.direct_defect(b["Xa"], b["Xb"], b["ua"], b["ub"], ta, tb, mode=mode, tol=1e-12)
        for s in range(n):
            tm = ta[s] + (tb[s] - ta[s]) / 2.0
            sf, xf, _, mf, _ = _leg(hostcheck, oracle, ns, b["Xa"][s], b["ua"][s], 0, ta[s], tm, mode, sens=0)
            sb, xb, _, mb, _ = _leg(hostcheck, oracle, ns, b["Xb"][s], b["ub"][s], 1, ta[s], tm, mode, sens=0)
            st = sf or sb
            if mode == 1 and tb[s] < ta[s]:
                assert st == ST_HMIN, (s, st)
                continue
            assert st == ST_OK and so[s] == 0, (mode, s, st, so[s])
            scale = np.maximum(1.0, np.maximum(np.abs(b["Xa"][s]), np.abs(b["Xb"][s])))
            assert (np.abs((xf - xb) - do[s]) / scale).max() < 1e-13, (mode, s)
            if tb[s] < ta[s]:
                assert np.abs(xf - b["Xa"][s]).max() > 1e-3   # really integrated (backwards), not handed back
                assert abs(max(mf, mb) - eo[s]) < 2e-14


@pytest.mark.parametrize("nd", [12, 14])
@pytest.mark.parametrize("controller", [0, 1])
@pytest.mark.parametrize("span", [(NAN, 0.1), (0.0, NAN), (0.0, INF), (-INF, 0.1)])
def test_indirect_nonfinite_span_not_ok(span, controller, nd, oracle, hostcheck):
    b = S.indirect_batch(1, ndim=nd, seed=44)
    ip = oracle.iparams(0.05, p=1.0, rho=1.0)
    t0, t1 = span
    for sens in (0, 1):
        xe = np.zeros(nd); Phi = np.zeros((nd, nd)); na = C.c_int(-1); nt = C.c_int(-1)
        st = hostcheck.hc_sc_seg(nd, sens, ptr(b["x0"][0]), C.c_double(t0), C.c_double(t1), C.c_double(1e-13), C.c_double(1e-13), controller, 1,
                                 ptr(ip), ptr(xe), ptr(Phi), C.byref(na), C.byref(nt))
        assert st == ST_NAN and nt.value == 0, (sens, st, nt.value)


@pytest.mark.parametrize("controller", [0, 1])
def test_indirect_reversed_span_not_ok(controller, oracle, hostcheck):
    b = S.indirect_batch(1, ndim=12, seed=45)
    ip = oracle.iparams(0.05, p=1.0, rho=1.0)
    xe = np.zeros(12); Phi = np.zeros((12, 12)); na = C.c_int(-1); nt = C.c_int(-1)
    st = hostcheck.hc_sc_seg(12, 1, ptr(b["x0"][0]), C.c_double(0.2), C.c_double(0.1), C.c_double(1e-13), C.c_double(1e-13), controller, 1,
                             ptr(ip), ptr(xe), ptr(Phi), C.byref(na), C.byref(nt))
    assert st == ST_HMIN and nt.value == 0
