"""CPU-side checks of the 14-dim device Newton update: wrapper validation, the host loop's dispatch of the update to the backend on
14 rows, and the sm_100a build carrying the 14-dim kernels with no local memory (no GPU needed)."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from lowthrustopt_b200 import capi, solvers as S
from oracle_backend import OracleBackend

MU, DU, TU = capi.MU, capi.DU, capi.TU


def _unbound_handle():
    """A Handle object that never reached lto_init: the shape checks run before any library call."""
    return capi.Handle.__new__(capi.Handle)


def test_wrappers_refuse_inconsistent_14dim_shapes():
    h = _unbound_handle()
    with pytest.raises(ValueError):
        h.indirect_newton(np.zeros((2, 5, 14, 14)), np.zeros((2, 5, 12)))     # 14 x 14 blocks, 12-wide defects
    with pytest.raises(ValueError):
        h.indirect_newton(np.zeros((2, 5, 14, 12)), np.zeros((2, 5, 14)))     # not square
    with pytest.raises(ValueError):
        h.indirect_newton(np.zeros((2, 5, 13, 13)), np.zeros((2, 5, 13)))     # no such system
    with pytest.raises(ValueError):
        h.indirect_newton(np.zeros((2, 5, 14, 14)), np.zeros((2, 4, 14)))     # one segment short
    with pytest.raises(ValueError):
        h.indirect_solve_batch(np.zeros((2, 5, 13)), np.zeros((2, 5)), params=capi.IndirectParams())
    with pytest.raises(ValueError):
        h.indirect_solve_batch(np.zeros((2, 5, 14)), np.zeros((2, 4)), params=capi.IndirectParams())
    with pytest.raises(ValueError):
        S.multiShoot_CRTBP_indirect_batch(np.zeros((2, 13, 5)), np.zeros((2, 5)), MU, DU, TU, 5, 1000.0, 0.05, backend=object())


class _RecordingBackend(OracleBackend):
    """Oracle propagation; the Newton update is recorded and answered with the host loop's own least squares."""

    def __init__(self):
        super().__init__()
        self.newton_calls = []

    def indirect_newton(self, phi, defect, flag_adjointsOnly):
        self.newton_calls.append((phi.shape, defect.shape, flag_adjointsOnly))
        B, n_seg, m, _ = phi.shape
        N = n_seg + 1
        J = S._band_indirect(phi[0], m // 2, N)
        live = np.any(J != 0.0, axis=0)
        sol = np.zeros(N * m)
        sol[live] = -np.linalg.lstsq(J[:, live], defect[0].ravel(), rcond=None)[0]
        return sol.reshape(1, N, m)


def test_host_loop_sends_the_14dim_update_to_the_backend(oracle):
    from test_solvers_cpu import _guess14
    XC0, t, tl = _guess14(oracle)
    be = _RecordingBackend()
    la, lb = [], []
    Xa, da, sa = S.multiShoot_CRTBP_indirect(XC0.copy(), t, MU, DU, TU, 30, 1000.0, tl, False, False, 3, 1.0, 1e-2, backend=be, log=la,
                                             device_newton=True)
    assert be.newton_calls and all(c == ((1, 29, 14, 14), (1, 29, 14), False) for c in be.newton_calls)
    Xb, db, sb = S.multiShoot_CRTBP_indirect(XC0.copy(), t, MU, DU, TU, 30, 1000.0, tl, False, False, 3, 1.0, 1e-2, backend=OracleBackend(),
                                             log=lb)
    assert sa == sb and len(la) == len(lb)
    assert np.abs(Xa - Xb).max() <= 1e-8 * max(1.0, np.abs(Xb).max())


def test_sm100a_build_carries_the_14dim_newton_kernels(tmp_path):
    """python -m lowthrustopt_b200.build --force (same nvcc commands, into a scratch directory so that the library the other tests
    loaded stays untouched): k_indirect_newton<14> / <7> and their resolve kernels are there as sm_100a code with no local memory."""
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    from lowthrustopt_b200 import build
    so = build.build_lib(force=True, lib=str(tmp_path / "liblto_b200.so"), obj_dir=str(tmp_path / "_build"))
    elfs = subprocess.run([cuobjdump, "-lelf", so], capture_output=True, text=True).stdout
    assert set(re.findall(r"\.(sm_\w+)\.cubin", elfs)) == {"sm_100a"}
    usage = subprocess.run([cuobjdump, "-res-usage", so], capture_output=True, text=True).stdout
    found = dict(re.findall(r"Function (_ZN3lto3nwt\w+):\s*\n\s*(REG:.*)", usage))
    for kern in ("17k_indirect_newtonILi14E", "17k_indirect_newtonILi7E", "25k_indirect_newton_resolveILi14E", "25k_indirect_newton_resolveILi7E",
                 "17k_indirect_newtonILi12E", "17k_indirect_newtonILi6E"):
        hits = [v for k, v in found.items() if kern in k]
        assert len(hits) == 1, (kern, sorted(found))
        assert "STACK:0 " in hits[0] and "LOCAL:0 " in hits[0], (kern, hits[0])
