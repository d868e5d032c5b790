"""CPU-side checks of the switch times of p = 1 indirect trajectories (lto_indirect_switch_batch, solvers.thrust_arcs_indirect): the
interpolant and root search of csrc/lto_switch.h compiled for the host (polynomials, scipy DOP853 steps of the 12-dim system), the sm_100a
build of the new kernels, wrapper validation and the arc assembly against a fake backend (no GPU needed)."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
from scipy.integrate import solve_ivp
from scipy.optimize import brentq

from lowthrustopt_b200 import capi, solvers as S, synthetic

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "lowthrustopt_b200", "csrc")
MU, DU, TU = capi.MU, capi.DU, capi.TU

# stdin, repeated cases:
#   0  e0 (lv lv' lv'': 9) e1 (9) h m theta_1..m      -> m lines: the interpolant's lv at theta
#   1  e0 (9) e1 (9) t h cap                           -> count, then min(count, cap) lines "time direction"
#   2  x0 (12) x1 (12) mu m1 omega t h cap             -> as 1, with the end values from sw_end of the two states
_DRIVER = r"""
#include "lto_switch.h"
#include <cstdio>
static int rd(double* v, int n) { for (int i = 0; i < n; ++i) if (scanf("%lf", v + i) != 1) return 0; return 1; }
static void ends(const double* v, SwEnd& e) { for (int q = 0; q < 3; ++q) { e.lv[q] = v[q]; e.ld[q] = v[3 + q]; e.la[q] = v[6 + q]; } }
static void scan(const SwEnd& e0, const SwEnd& e1, double t, double h, int cap) {
    double ts[64]; int32_t d[64];
    const int n = sw_scan(e0, e1, t, h, 0, cap, ts, d);
    printf("%d\n", n);
    for (int k = 0; k < n && k < cap; ++k) printf("%.17g %d\n", ts[k], (int)d[k]);
}
int main() {
    int mode;
    while (scanf("%d", &mode) == 1) {
        SwEnd e0, e1;
        if (mode == 0) {
            double v[19]; int m; if (!rd(v, 19) || scanf("%d", &m) != 1) return 1;
            ends(v, e0); ends(v + 9, e1);
            double c[3][6]; sw_fit(e0, e1, v[18], c);
            for (int j = 0; j < m; ++j) {
                double th, p[3], dp[3]; if (!rd(&th, 1)) return 1;
                sw_eval(c, th, p, dp);
                printf("%.17g %.17g %.17g\n", p[0], p[1], p[2]);
            }
        } else if (mode == 1) {
            double v[21]; if (!rd(v, 21)) return 1;
            ends(v, e0); ends(v + 9, e1);
            scan(e0, e1, v[18], v[19], (int)v[20]);
        } else {
            double v[30]; if (!rd(v, 30)) return 1;
            sw_end(v[0], v[1], v[2], v[6], v[7], v[8], v[9], v[10], v[11], v[24], v[25], v[26], e0);
            sw_end(v[12], v[13], v[14], v[18], v[19], v[20], v[21], v[22], v[23], v[24], v[25], v[26], e1);
            scan(e0, e1, v[27], v[28], (int)v[29]);
        }
    }
    return 0;
}
"""


@pytest.fixture(scope="module")
def sw(tmp_path_factory):
    d = tmp_path_factory.mktemp("switch")
    src = d / "driver.cpp"
    src.write_text(_DRIVER)
    exe = str(d / "driver")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-ffp-contract=off", "-I", CSRC, "-o", exe, str(src)])
    return exe


def _fmt(v):
    return " ".join("%.17g" % x for x in np.ravel(v))


def _run(exe, text):
    return subprocess.run([exe], input=text, capture_output=True, text=True, check=True).stdout.split()


def _scans(exe, cases):
    """cases: input lines of mode 1 or 2; returns per case the list of (time, direction)."""
    out = iter(_run(exe, "\n".join(cases) + "\n"))
    res = []
    for _ in cases:
        n = int(next(out))
        res.append([(float(next(out)), int(next(out))) for _ in range(n)])
    return res


def _poly_ends(c, t0, h):
    """lv(t) = q((t - t0) / h), q_k = polyval(c[k], theta): (lv, lv', lv'') at theta = 0 and 1 in physical time."""
    e = []
    for th in (0.0, 1.0):
        e.append(np.concatenate([[np.polyval(q, th) for q in c], [np.polyval(np.polyder(q), th) / h for q in c],
                                 [np.polyval(np.polyder(q, 2), th) / h ** 2 for q in c]]))
    return e


def _poly_roots(c):
    """The roots of |q(theta)|^2 - 1 in (0, 1) from numpy.roots, each polished by two Newton steps on that polynomial."""
    g = np.polysub(sum(np.polymul(q, q) for q in c), [1.0])
    r = np.roots(g)
    r = np.sort(r[(np.abs(r.imag) < 1e-9) & (r.real > 0.0) & (r.real < 1.0)].real)
    dg = np.polyder(g)
    for _ in range(2):
        r = r - np.polyval(g, r) / np.polyval(dg, r)
    return r


def test_interpolant_reproduces_a_quintic_and_finds_its_roots(sw):
    rng = np.random.default_rng(11)
    th = np.linspace(0.0, 1.0, 41)
    t0, h = 2.5, 0.37
    worst_fit, worst_root, used = 0.0, 0.0, 0
    for case in range(400):
        deg = int(rng.integers(1, 6))
        c = [rng.standard_normal(deg + 1) * 0.6 for _ in range(3)]
        c[0][-1] += 0.7
        e0, e1 = _poly_ends(c, t0, h)
        vals = np.array(_run(sw, "0 %s %s %.17g %d %s\n" % (_fmt(e0), _fmt(e1), h, len(th), _fmt(th))), dtype=float).reshape(-1, 3)
        ref = np.array([[np.polyval(q, x) for q in c] for x in th])
        worst_fit = max(worst_fit, np.abs(vals - ref).max() / max(1.0, np.abs(ref).max()))
        roots = _poly_roots(c)
        # the scan sees a root when it is the only one between two samples k/8 and not within 1e-6 of a sample, and |q| crosses 1 there
        k = np.floor(roots * 8)
        g = np.polysub(sum(np.polymul(q, q) for q in c), [1.0])
        if len(np.unique(k)) != len(k) or (np.abs(roots * 8 - np.round(roots * 8)) < 1e-6).any() or \
                (np.abs(np.polyval(np.polyder(g), roots)) < 1e-3).any():
            continue
        used += 1
        got = _scans(sw, ["1 %s %s %.17g %.17g 64" % (_fmt(e0), _fmt(e1), t0, h)])[0]
        assert len(got) == len(roots), (case, got, roots)
        thg = (np.array([x for x, _ in got]) - t0) / h
        worst_root = max(worst_root, np.abs(thg - roots).max(initial=0.0))
        slope = np.polyval(np.polyder(g), roots)
        assert [d for _, d in got] == [1 if s > 0 else -1 for s in slope]
    print("\n[switch] quintic: interpolant %.2e, roots %.2e in theta over %d cases with roots" % (worst_fit, worst_root, used))
    assert used >= 100
    assert worst_fit <= 1e-14 and worst_root <= 1e-14, (worst_fit, worst_root)


def test_two_crossings_inside_one_step_are_both_found(sw):
    # |lv| = lv_x = 1.2 - 4 (theta - 0.5)^2 crosses 1 at theta = 0.5 -+ sqrt(0.05): both inside one step, in different eighths
    c = [np.array([-4.0, 4.0, 0.2]), np.zeros(1), np.zeros(1)]
    e0, e1 = _poly_ends(c, 0.0, 1.0)
    got = _scans(sw, ["1 %s %s 0 1 64" % (_fmt(e0), _fmt(e1))])[0]
    want = [0.5 - np.sqrt(0.05), 0.5 + np.sqrt(0.05)]
    assert [d for _, d in got] == [1, -1]
    assert np.abs(np.array([x for x, _ in got]) - want).max() <= 1e-15
    # a touch (max |lv| exactly 1) is no switch; the cap keeps the count
    assert _scans(sw, ["1 %s %s 0 1 64" % (_fmt(_poly_ends([np.array([-4.0, 4.0, 0.0]), np.zeros(1), np.zeros(1)], 0, 1)[0]),
                                          _fmt(_poly_ends([np.array([-4.0, 4.0, 0.0]), np.zeros(1), np.zeros(1)], 0, 1)[1]))])[0] == []
    out = _run(sw, "1 %s %s 0 1 1\n" % (_fmt(e0), _fmt(e1)))
    assert int(out[0]) == 2 and len(out) == 3


def _rhs12(tl, rho, mass=1000.0):
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


def _switching_starts():
    """Starts on L2_Anderson_2 at 0.22 DU from the Moon (|lv| = 0.95, four lr): each crosses |lv| = 1 once within 2 TU."""
    c = synthetic.continuation_batch(n_traj=1, n_seg_per_traj=40, ndim=12, seed=3)
    out = []
    for lr in ([0.4, -0.3, 0.1], [0.2, -0.6, 0.1], [1.0, 0.5, 0.0], [-0.5, 0.5, 0.2]):
        x = c["XC_all"][0, 11].copy()
        x[6:9] = lr
        x[9:12] = 0.95 * np.array([0.6, 0.8, 0.0])
        out.append(x)
    return out


@pytest.mark.parametrize("h", [0.02, 0.1])
def test_roots_on_dop853_steps_match_brentq_on_its_dense_output(sw, h):
    """Steps of length h from scipy's DOP853 (rtol 1e-13): the scan on each step's end states against brentq on that step's dense output.
    The interpolant's error is h^6 |lv^(6)| / 46080 at most, and lv^(6) grows with U's derivatives near the Moon: from a start at 0.12 DU
    the h = 0.02 distance was 1.9e-11 TU, against the 5.7e-13 TU measured here at 0.22 DU."""
    f = _rhs12(0.05, 1e-2)
    cases, refs = [], []
    for x in _switching_starts():
        for k in range(int(round(2.0 / h))):
            t = k * h
            s = solve_ivp(f, (t, t + h), x, method="DOP853", rtol=1e-13, atol=1e-15, dense_output=True)
            assert s.success
            x1 = s.y[:, -1]
            cases.append("2 %s %s %.17g %.17g 1 %.17g %.17g 64" % (_fmt(x), _fmt(x1), MU, 1.0 - MU, t, h))
            Sf = lambda tt: np.linalg.norm(s.sol(tt)[9:12]) - 1.0
            grid = np.linspace(t, t + h, 65)
            vals = np.array([Sf(g) for g in grid])
            vals[0], vals[-1] = np.linalg.norm(x[9:12]) - 1.0, np.linalg.norm(x1[9:12]) - 1.0
            refs.append([(brentq(Sf, grid[i], grid[i + 1], xtol=1e-15, rtol=1e-15), 1 if vals[i + 1] > 0 else -1)
                         for i in range(64) if (vals[i] > 0) != (vals[i + 1] > 0)])
            x = x1
    got = _scans(sw, cases)
    n_sw = sum(len(r) for r in refs)
    worst = 0.0
    for g, r in zip(got, refs):
        assert [d for _, d in g] == [d for _, d in r], (g, r)
        if r:
            worst = max(worst, np.abs(np.array([a for a, _ in g]) - [a for a, _ in r]).max())
    print("\n[switch] DOP853 steps h = %g TU: %d switches, max |t - t_brentq| = %.2e TU" % (h, n_sw, worst))
    assert n_sw == 4
    # measured 5.7e-13 TU (h = 0.02) and 5.9e-9 TU (h = 0.1)
    assert worst <= (1e-11 if h == 0.02 else 1e-8), worst


def test_switch_kernels_build_for_sm100a(tmp_path):
    """k_switch_gather uses no stack and no local memory.  k_indirect_state_switch uses no local memory; like K4 (k_indirect_state, 255
    registers at two CTAs of 128 threads per SM) it keeps a spill / call frame, here at most 64 bytes larger than K4's."""
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

    g = one("15k_switch_gather")
    assert "STACK:0 " in g and "LOCAL:0 " in g, g
    s, k4 = one("23k_indirect_state_switchE"), one("16k_indirect_stateE")
    assert "LOCAL:0 " in s, s
    stack = lambda u: int(re.search(r"STACK:(\d+)", u).group(1))
    print("\n[switch] k_indirect_state_switch: %s\n[switch] k_indirect_state: %s\n[switch] k_switch_gather: %s" % (s, k4, g))
    assert stack(s) <= stack(k4) + 64, (s, k4)


def _unbound_handle():
    """A Handle object that never reached lto_init: the argument checks run before any library call."""
    return capi.Handle.__new__(capi.Handle)


def test_switch_wrapper_refuses_bad_arguments():
    h = _unbound_handle()
    t = np.tile(np.linspace(0.0, 1.0, 5), (2, 1))
    z = np.zeros((2, 5, 12))
    with pytest.raises(ValueError):
        h.indirect_switch_batch(np.zeros((2, 5, 14)), t)                            # 14-dim: a different kernel
    with pytest.raises(ValueError, match="p = 1"):
        h.indirect_switch_batch(z, t, params=capi.indirect_params(p=2.0))
    for m in (0, 65):
        with pytest.raises(ValueError, match="max_switch"):
            h.indirect_switch_batch(z, t, max_switch=m)
    with pytest.raises(ValueError):
        h.indirect_switch_batch(z, t, params=capi.IndirectParams(controller=capi.LTO_CTRL_ODE78, p=1.0))
    rev = t.copy(); rev[1, 3] = 0.1
    with pytest.raises(ValueError, match="trajectory 1"):
        h.indirect_switch_batch(z, rev)
    bad = t.copy(); bad[0, 2] = np.nan
    with pytest.raises(ValueError, match="trajectory 0"):
        h.indirect_switch_batch(z, bad)
    with pytest.raises(ValueError):
        h.indirect_switch_batch(np.zeros((5, 12)), t[0])                            # not a batch
    with pytest.raises(ValueError):
        h.indirect_switch_batch(z, t[:, :4])                                        # one time short
    with pytest.raises(ValueError):
        h.indirect_switch_batch(np.zeros((2, 1, 12)), t[:, :1])                     # no segment
    with pytest.raises(ValueError):
        h.indirect_switch_batch(z, t, thrustLimit=np.ones(3))
    with pytest.raises(ValueError):
        S.thrust_arcs_indirect(np.zeros((2, 14, 5)), t, MU, DU, TU, 1e3, 0.05, 1e-4, backend=object())
    with pytest.raises(ValueError):
        S.thrust_arcs_indirect(np.zeros((2, 12, 5)), t[:, :4], MU, DU, TU, 1e3, 0.05, 1e-4, backend=object())


class _SwitchBackend:
    """Fake backend: answers indirect_switches with the rows it was built with."""

    def __init__(self, rows, K):
        self.rows, self.K = rows, K

    def indirect_switches(self, XC, t, params, thrustLimit=None, rho=None, max_switch=16, defect=False):
        assert params[6] == 1.0 and max_switch == self.K and XC.shape[2] == 12
        T = len(self.rows)
        ts = np.full((T, self.K), np.nan); dr = np.zeros((T, self.K), dtype=np.int32)
        for j, (st, on, times, dirs, n) in enumerate(self.rows):
            ts[j, :len(times)] = times; dr[j, :len(dirs)] = dirs
        return dict(t_switch=ts, direction=dr, n_switch=np.array([r[4] for r in self.rows], dtype=np.int32),
                    on_start=np.array([r[1] for r in self.rows], dtype=np.int32), status=np.array([r[0] for r in self.rows], dtype=np.int32))


def test_arcs_are_assembled_from_the_switches():
    K = 3
    rows = [(0, 1, [1.0, 2.0], [-1, 1], 2),                       # on at the start: [0, 1] and [2, 4]
            (0, 0, [0.5, 1.5, 3.0], [1, -1, 1], 3),               # off at the start: [0.5, 1.5] and [3, 4]
            (0, 0, [0.5, 1.5, 3.0], [1, -1, 1], 4),               # truncated: 4 switches, 3 slots
            (1, 0, [], [], -1),                                   # failed row
            (0, 1, [], [], 0),                                    # on throughout
            (0, 0, [], [], 0)]                                    # coasting throughout
    T = len(rows)
    t = np.tile(np.linspace(0.0, 4.0, 5), (T, 1))
    r = S.thrust_arcs_indirect(np.zeros((T, 12, 5)), t, MU, DU, TU, 1e3, 0.05, 1e-4, max_switch=K, backend=_SwitchBackend(rows, K))
    assert np.array_equal(r["arcs"][0], [[0.0, 1.0], [2.0, 4.0]]) and np.array_equal(r["arcs"][1], [[0.5, 1.5], [3.0, 4.0]])
    assert r["arcs"][2] is None and r["arcs"][3] is None
    assert np.array_equal(r["arcs"][4], [[0.0, 4.0]]) and r["arcs"][5].shape == (0, 2)
    assert r["n_burns"].tolist() == [2, 2, -1, -1, 1, 0]
    np.testing.assert_array_equal(r["on_time"], [3.0, 2.0, np.nan, np.nan, 4.0, 0.0])
    assert r["n_switch"].tolist() == [2, 3, 4, -1, 0, 0] and r["status"].tolist() == [0, 0, 0, 1, 0, 0]
