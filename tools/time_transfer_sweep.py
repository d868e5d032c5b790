"""Times solvers.indirect_transfer_sweep on the 1 024-transfer grid of tools/time_stack_guess.py, stage by stage (each stage is one
library call that ends in a device synchronise, so a host clock around it is its wall time), and compares the cost pass
(lto_indirect_cost_batch: K4 plus the two quadratures) with a plain defect pass (lto_indirect_defect_traj: K4) on the same batch --
the sweep's final rho_target trajectories -- alternated, medians over --runs runs.  Also reports, for the rows that converged at p = 2,
the indirect p = 2 control energy next to the direct method's quadCost (a comparison, not a check: the direct cost is a 30-node
trapezoid sum of the direct method's controls).

    python tools/time_transfer_sweep.py [--runs 5] [--rows 1024] [--out profiles/r06_transfer_sweep.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from lowthrustopt_b200 import capi, solvers as S  # noqa: E402
from time_stack_guess import grid  # noqa: E402


class TimedBackend(S.GpuBackend):
    """GpuBackend that records the wall time of every call, in call order."""

    def __init__(self, handle):
        super().__init__(handle=handle)
        self.log = []

    def _timed(name):
        def wrap(self, *a, **k):
            t0 = time.perf_counter()
            out = getattr(S.GpuBackend, name)(self, *a, **k)
            self.log.append((name, time.perf_counter() - t0))
            return out
        return wrap

    stack_guess_batch = _timed("stack_guess_batch")
    direct_solve_batch = _timed("direct_solve_batch")
    indirect_solve_batch = _timed("indirect_solve_batch")
    indirect_cost = _timed("indirect_cost")
    indirect_reduce_fuel_batch = _timed("indirect_reduce_fuel_batch")


STAGES = ["guess (lto_stack_guess_batch)", "direct solve (lto_direct_solve_batch)", "stage 1: adjoints-only p = 2, 10 N",
          "stage 2: p = 2, 10 N", "cost of the p = 2 solutions", "stage 3: p = 1, rho = 1", "stage 4: device ladder to rho_target",
          "cost of the rho_target solutions"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--rows", type=int, default=1024)
    ap.add_argument("--out", default="profiles/r06_transfer_sweep.json")
    a = ap.parse_args()
    gpu_q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    fx = S.demo_fixtures()
    h = capi.Handle(0)
    be = TimedBackend(h)
    tau1, tof1, tof2 = (x[:a.rows] for x in grid())
    T = tau1.size
    S.indirect_transfer_sweep(fx[1], fx[3], tau1[:8], tof1[:8], tof2[:8], backend=be)          # warm-up: module load, first launches
    be.log.clear()
    t0 = time.perf_counter()
    sw = S.indirect_transfer_sweep(fx[1], fx[3], tau1, tof1, tof2, backend=be)
    wall = time.perf_counter() - t0
    names = [n for n, _ in be.log]
    assert names == ["stack_guess_batch", "direct_solve_batch"] + ["indirect_solve_batch"] * 2 + ["indirect_cost", "indirect_solve_batch",
                                                                                                   "indirect_reduce_fuel_batch", "indirect_cost"], names
    stages = {s: w for s, (_, w) in zip(STAGES, be.log)}
    ok = np.flatnonzero(sw["stage_failed"] == 0)
    XC = np.ascontiguousarray(sw["XC_all"][ok].transpose(0, 2, 1)); t = sw["t_TU"][ok]
    p = capi.indirect_params(thrustLimit=0.05, p=1.0, rho=1e-4)
    wc, wd, kc, kd = [], [], [], []
    h.indirect_cost_batch(XC, t, params=p); h.indirect_traj(XC, t, params=p, jac=False)
    for _ in range(a.runs):
        t1 = time.perf_counter(); c = h.indirect_cost_batch(XC, t, params=p, defect=True); wc.append(time.perf_counter() - t1); kc.append(h.last_kernel_ms)
        t1 = time.perf_counter(); d = h.indirect_traj(XC, t, params=p, jac=False); wd.append(time.perf_counter() - t1); kd.append(h.last_kernel_ms)
    same = bool(np.array_equal(c["defect"], d["defect"].reshape(c["defect"].shape)))
    p2 = np.isfinite(sw["energy_p2"])
    ratio = sw["energy_p2"][p2] / sw["cost"][p2]
    report = dict(
        gpu=gpu_q.splitlines()[0] if gpu_q else "unknown",
        grid=dict(n_traj=T, n_nodes=30, tau1="32 values k/32", tof_days="32 seeded (tof1, tof2) pairs in [6, 14]", thrustLimit_N=0.05,
                  rho_target=1e-4, seeds="row index"),
        sweep=dict(wall_s=wall, stage_wall_s=stages,
                   stage_failed={int(k): int(v) for k, v in zip(*np.unique(sw["stage_failed"], return_counts=True))},
                   direct_converged=int(sw["direct_converged"].sum())),
        cost_vs_defect_pass=dict(rows=int(ok.size), segments=int(ok.size * 29), runs=a.runs, defects_bitwise_equal=same,
                                 cost_device_ms_median=float(np.median(kc)), defect_device_ms_median=float(np.median(kd)),
                                 cost_wall_ms_median=float(np.median(wc)) * 1e3, defect_wall_ms_median=float(np.median(wd)) * 1e3,
                                 cost_device_ms_runs=kc, defect_device_ms_runs=kd),
        p2_energy_vs_direct_cost=dict(rows=int(p2.sum()), ratio_median=float(np.median(ratio)) if p2.any() else None,
                                      ratio_min=float(ratio.min()) if p2.any() else None, ratio_max=float(ratio.max()) if p2.any() else None),
        dv_m_s=dict(median=float(np.nanmedian(sw["dv"])) if ok.size else None, min=float(np.nanmin(sw["dv"])) if ok.size else None,
                    max=float(np.nanmax(sw["dv"])) if ok.size else None),
    )
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report, indent=1))
    h.close()
    assert same


if __name__ == "__main__":
    main()
