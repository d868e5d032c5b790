"""CPU-side checks of the device rho continuation (lto_indirect_reduce_fuel_batch): the ladder state machine of
csrc/lto_ladder.h, compiled for the host, against solvers._reduceFuel_steps on random status sequences; wrapper validation; and
the sm_100a build carrying the new kernels with no stack or local memory (no GPU needed)."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from lowthrustopt_b200 import capi, solvers as S

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "lowthrustopt_b200", "csrc")

# stdin: n_cases, then per case: rho_current rho_target n_status status... draws[100]
# stdout per case: one line "rho start" per call (start: -1 the original start, k the XC_new of call k), then "end status draws"
_DRIVER = r"""
#include "lto_ladder.h"
#include <cstdio>
#include <vector>
int main() {
    int n; if (scanf("%d", &n) != 1) return 1;
    for (int c = 0; c < n; ++c) {
        double r0, r1; int ns; if (scanf("%lf %lf %d", &r0, &r1, &ns) != 3) return 1;
        std::vector<int> st(ns); for (int& s : st) if (scanf("%d", &s) != 1) return 1;
        double draws[LADDER_DRAWS]; for (double& d : draws) if (scanf("%lf", &d) != 1) return 1;
        LadderState s; int start = -1;
        double rho = ladder_init(&s, r0, r1);
        for (int k = 0;; ++k) {
            printf("%.17g %d\n", rho, start);
            if (k >= ns) return 2;
            int accept = 0, fin = 0;
            if (!ladder_step(&s, st[k], draws, &accept, &fin)) { printf("end %d %d\n", fin, s.draws); break; }
            if (accept) start = k;
            rho = s.rho;
        }
    }
    return 0;
}
"""


@pytest.fixture(scope="module")
def ladder_driver(tmp_path_factory):
    d = tmp_path_factory.mktemp("ladder")
    src = d / "driver.cpp"
    src.write_text(_DRIVER)
    exe = str(d / "driver")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-I", CSRC, "-o", exe, str(src)])
    return exe


class _Draws:
    """rng stand-in: hands out the given draws in order and counts them."""

    def __init__(self, u):
        self.u, self.n = u, 0

    def random(self):
        self.n += 1
        return float(self.u[self.n - 1])


def _reference(r0, r1, statuses, draws):
    rng = _Draws(draws)
    gen = S._reduceFuel_steps(np.array([-1.0]), r0, r1, rng)
    calls = []
    req = next(gen)
    k = 0
    while True:
        start, rho = req
        calls.append((rho, int(start[0])))
        try:
            req = gen.send((np.array([float(k)]), None, statuses[k]))
        except StopIteration as fin:
            return calls, (fin.value[2], rng.n)
        k += 1


def test_ladder_header_matches_reduceFuel_steps(ladder_driver):
    rng = np.random.default_rng(2026)
    cases = []
    for i in range(3000):
        r0 = float(10.0 ** rng.uniform(-4, 0.8))                      # includes rho > 1
        r1 = float(10.0 ** rng.uniform(-5, 0.8)) if i % 10 else r0 * 2  # and targets above rho_current
        p_fail = rng.choice([0.0, 0.2, 0.5, 0.9, 1.0])
        st = np.where(rng.random(400) < p_fail, rng.choice([1, 2], 400), 0).astype(int)
        cases.append((r0, r1, st, rng.random(100)))
    text = "%d\n" % len(cases) + "".join("%.17g %.17g %d %s %s\n" % (r0, r1, len(st), " ".join(map(str, st)), " ".join("%.17g" % u for u in d))
                                        for r0, r1, st, d in cases)
    out = subprocess.run([ladder_driver], input=text, capture_output=True, text=True, check=True).stdout.splitlines()
    pos = 0
    ends = set()
    for r0, r1, st, d in cases:
        ref_calls, (ref_status, ref_draws) = _reference(r0, r1, st, d)
        for rho, start in ref_calls:
            got_rho, got_start = out[pos].split(); pos += 1
            assert float(got_rho) == rho and int(got_start) == start, (r0, r1, rho, start, out[pos - 1])
        tag, status, ndraws = out[pos].split(); pos += 1
        assert tag == "end" and int(status) == ref_status and int(ndraws) == ref_draws, (r0, r1, out[pos - 1], ref_status, ref_draws)
        ends.add(ref_status)
    assert pos == len(out)
    assert ends == {0, 1, 2, 3}                                           # every way out of the ladder was taken


def _unbound_handle():
    """A Handle object that never reached lto_init: the shape checks run before any library call."""
    return capi.Handle.__new__(capi.Handle)


def test_reduce_fuel_wrapper_refuses_bad_shapes():
    h = _unbound_handle()
    X, t, u = np.zeros((2, 5, 12)), np.zeros((2, 5)), np.zeros((2, 100))
    with pytest.raises(ValueError):
        h.indirect_reduce_fuel_batch(np.zeros((2, 5, 13)), t, 1.0, 0.1, u)           # no such system
    with pytest.raises(ValueError):
        h.indirect_reduce_fuel_batch(X, np.zeros((2, 4)), 1.0, 0.1, u)               # one node short
    with pytest.raises(ValueError):
        h.indirect_reduce_fuel_batch(X, t, np.ones(3), 0.1, u)                       # rho_current for 3 trajectories
    with pytest.raises(ValueError):
        h.indirect_reduce_fuel_batch(X, t, 1.0, np.ones((2, 1)), u)
    with pytest.raises(ValueError):
        h.indirect_reduce_fuel_batch(X, t, 1.0, 0.1, np.zeros((2, 99)))              # the draws table is (n_traj, 100)
    with pytest.raises(ValueError):
        h.indirect_reduce_fuel_batch(X, t, 1.0, 0.1, u, thrustLimit=np.ones(3))
    with pytest.raises(ValueError):
        S.reduceFuel_indirect_batch(np.zeros((2, 12, 5)), t, capi.MU, capi.DU, capi.TU, 5, 1000.0, 0.05, 1.0, 0.1, backend=object(),
                                    log=[], device_ladder=True)


def test_sm100a_build_carries_the_ladder_kernels(tmp_path):
    """A forced build into a scratch directory: the engine's and the ladder's kernels are sm_100a code with no stack or local memory."""
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    from lowthrustopt_b200 import build
    so = build.build_lib(force=True, lib=str(tmp_path / "liblto_b200.so"), obj_dir=str(tmp_path / "_build"))
    elfs = subprocess.run([cuobjdump, "-lelf", so], capture_output=True, text=True).stdout
    assert set(re.findall(r"\.(sm_\w+)\.cubin", elfs)) == {"sm_100a"}
    usage = subprocess.run([cuobjdump, "-res-usage", so], capture_output=True, text=True).stdout
    found = dict(re.findall(r"Function (_ZN3lto3slv\w+):\s*\n\s*(REG:.*)", usage))
    for kern in ("13k_ladder_hook", "13k_ladder_init", "10k_call_end", "8k_select", "10k_index_of", "13k_gather_rows", "14k_scatter_rows",
                 "11k_ls_trials", "16k_pick_alpha_sel"):
        hits = [v for k, v in found.items() if kern in k]
        assert len(hits) == 1, (kern, sorted(found))
        assert "STACK:0 " in hits[0] and "LOCAL:0 " in hits[0], (kern, hits[0])
