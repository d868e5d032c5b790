"""CPU-side checks of the batched trajectory-stacking guess (lto_stack_guess_batch): the orbit lookups of csrc/lto_orbit.h, compiled
for the host, against the host mirror's scipy spline and find_tau on both orbit tables; wrapper validation; and the sm_100a build of
lto_guess.cu's kernels with no stack or local memory (no GPU needed)."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from lowthrustopt_b200 import capi, solvers as S, synthetic

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "lowthrustopt_b200", "csrc")

# stdin: n, the 6 x n table (column-major), m, m values of tau, q, q states (6 each)
# stdout: per tau the 6 spline values of the wrapped tau; per state the index of find_τ's first nearest candidate
_DRIVER = r"""
#include "lto_orbit.h"
#include <cstdio>
#include <vector>
int main() {
    int n; if (scanf("%d", &n) != 1) return 1;
    std::vector<double> X(6 * n), coef((n - 1) * 24), work(4 * n);
    for (double& v : X) if (scanf("%lf", &v) != 1) return 1;
    orbit_fit(X.data(), n, coef.data(), work.data());
    int m; if (scanf("%d", &m) != 1) return 1;
    for (int j = 0; j < m; ++j) {
        double t; if (scanf("%lf", &t) != 1) return 1;
        t = orbit_wrap(t);
        for (int k = 0; k < 6; ++k) printf("%.17g%c", orbit_eval(coef.data(), n, t, k), k == 5 ? '\n' : ' ');
    }
    std::vector<double> cand(LTO_ORBIT_NTAU * 6);
    for (int c = 0; c < LTO_ORBIT_NTAU; ++c)
        for (int k = 0; k < 6; ++k) cand[c * 6 + k] = orbit_eval(coef.data(), n, orbit_tau_candidate(c), k);
    int q; if (scanf("%d", &q) != 1) return 1;
    for (int j = 0; j < q; ++j) {
        double x[6]; for (double& v : x) if (scanf("%lf", &v) != 1) return 1;
        double best = 0.0; int kb = -1;
        for (int c = 0; c < LTO_ORBIT_NTAU; ++c) {
            const double d = orbit_distance(&cand[c * 6], x);
            if (kb < 0 || orbit_before(d, c, best, kb)) { best = d; kb = c; }
        }
        printf("%d\n", kb);
    }
    return 0;
}
"""


@pytest.fixture(scope="module")
def orbit_driver(tmp_path_factory):
    d = tmp_path_factory.mktemp("orbit")
    src = d / "driver.cpp"
    src.write_text(_DRIVER)
    exe = str(d / "driver")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-ffp-contract=off", "-I", CSRC, "-o", exe, str(src)])
    return exe


def _run(exe, X, taus, states):
    text = ("%d\n" % X.shape[1] + " ".join("%.17g" % v for v in X.T.ravel()) + "\n%d\n" % len(taus) + " ".join("%.17g" % t for t in taus)
            + "\n%d\n" % len(states) + " ".join("%.17g" % v for v in np.asarray(states).ravel()) + "\n")
    out = subprocess.run([exe], input=text, capture_output=True, text=True, check=True).stdout.splitlines()
    vals = np.array([[float(x) for x in line.split()] for line in out[:len(taus)]]).reshape(len(taus), 6)
    return vals, np.array([int(line) for line in out[len(taus):]], dtype=int)


@pytest.mark.parametrize("which", [1, 2])
def test_orbit_spline_matches_scipy(orbit_driver, which):
    X = synthetic.load_orbit(which)
    n = X.shape[1]
    rng = np.random.default_rng(100 + which)
    wraps = [-0.25, 1.75, 1.0]
    taus = np.concatenate([rng.random(10000), np.linspace(0.0, 1.0, n), [0.0, 1.0], wraps])
    vals, _ = _run(orbit_driver, X, taus, np.zeros((0, 6)))
    sp = synthetic.orbit_spline(which)
    ref = sp(np.concatenate([taus[:-3], [0.75, 0.75, 1.0]]))                  # -0.25 and 1.75 wrap to 0.75; 1.0 stays 1
    assert np.abs(vals - ref).max() <= 1e-15
    host = np.array([S._orbit_states(X)(t) for t in taus[-3:]])             # the host mirror's own wrap loop
    assert np.abs(vals[-3:] - host).max() <= 1e-15
    assert np.abs(vals[10000:10000 + n] - X.T).max() <= 1e-15                  # it interpolates the table


@pytest.mark.parametrize("which", [1, 2])
def test_find_tau_index_matches_host(orbit_driver, which):
    X = synthetic.load_orbit(which)
    rng = np.random.default_rng(200 + which)
    sp = synthetic.orbit_spline(which)
    states = sp(rng.random(300)) + 0.05 * rng.standard_normal((300, 6))
    _, idx = _run(orbit_driver, X, np.zeros(0), states)
    cand = np.linspace(0.0, 1.0, 1001)
    ref = np.array([S.find_tau(None, X, s) for s in states])
    assert np.array_equal(cand[idx], ref)


def _unbound_handle():
    """A Handle object that never reached lto_init: the shape checks run before any library call."""
    return capi.Handle.__new__(capi.Handle)


def test_stack_guess_wrapper_refuses_bad_shapes():
    h = _unbound_handle()
    X0 = synthetic.load_orbit(1)
    t = np.tile(np.linspace(0.0, 1.0, 5), (2, 1))
    with pytest.raises(ValueError):
        h.stack_guess_batch(X0.T, X0, np.zeros(2), t, np.full(2, 0.5))              # tables are (6, n)
    with pytest.raises(ValueError):
        h.stack_guess_batch(X0, X0, np.zeros(3), t, np.full(2, 0.5))                # tau1 for 3 transfers
    with pytest.raises(ValueError):
        h.stack_guess_batch(X0, X0, np.zeros(2), t, np.full(3, 0.5))
    with pytest.raises(ValueError):
        h.stack_guess_batch(X0, X0, np.zeros(2), t[0], np.full(2, 0.5))             # t_TU is (n_traj, n_nodes)
    with pytest.raises(ValueError):
        S.trajectory_stack_guess_batch(X0, X0, tau1=np.zeros((2, 2)), backend=object())
    with pytest.raises(ValueError):
        S.direct_transfer_sweep(X0, X0, 0.75, 10.0, 10.0, nstate=5, backend=object())


def test_sm100a_build_of_the_guess_kernels(tmp_path):
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    from lowthrustopt_b200 import build
    obj = str(tmp_path / "lto_guess.o")
    cmd = [build._nvcc()] + build.ARCH + build.NVCC_FLAGS + ["-I", build.INC, "-I", build.CSRC, "-c", os.path.join(build.CSRC, "lto_guess.cu"),
                                                             "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    elfs = subprocess.run([cuobjdump, "-lelf", obj], capture_output=True, text=True).stdout
    assert set(re.findall(r"\.(sm_\w+)\.cubin", elfs)) == {"sm_100a"}
    usage = subprocess.run([cuobjdump, "-res-usage", obj], capture_output=True, text=True).stdout
    found = dict(re.findall(r"Function (_ZN3lto3gss\w+):\s*\n\s*(REG:.*)", usage))
    for kern in ("12k_orbit_eval", "13k_orbit_table", "11k_arc_table", "10k_find_tau", "10k_assemble"):
        hits = [v for k, v in found.items() if kern in k]
        assert len(hits) == 1, (kern, sorted(found))
        assert "STACK:0 " in hits[0] and "LOCAL:0 " in hits[0], (kern, hits[0])
