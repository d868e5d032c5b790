"""Measures lto_indirect_switch_batch on the rows of the 1 024-transfer grid of tools/time_stack_guess.py (30 nodes, thrustLimit 0.05 N,
rho_target 1e-4) that come through solvers.indirect_transfer_sweep:
  * the switch call against lto_indirect_cost_batch and lto_indirect_defect_traj on the same batch (the sweep's XC_all, t_TU and
    rho_last), alternated after a warm-up: wall (host clock around the call, which ends in a device synchronise) and device time (the
    call's kernel events), medians over --runs runs;
  * solvers.thrust_arcs_indirect on that batch: the distribution of switch and burn counts, and the agreement of each row's burn time with
    dv / (aL DU 1e3 / TU) from the cost call (near bang-bang at rho = 1e-4, the thrust is aL wherever it is on).

    python tools/time_thrust_arcs.py [--runs 5] [--rows 1024] [--max-switch 16] [--out profiles/r08_thrust_arcs.json]"""
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

MU, DU, TU = capi.MU, capi.DU, capi.TU


def _counts(a):
    return {int(k): int(v) for k, v in zip(*np.unique(a, return_counts=True))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--rows", type=int, default=1024)
    ap.add_argument("--max-switch", type=int, default=16)
    ap.add_argument("--out", default="profiles/r08_thrust_arcs.json")
    a = ap.parse_args()
    gpu_q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    fx = S.demo_fixtures()
    h = capi.Handle(0)
    be = S.GpuBackend(handle=h)
    tau1, tof1, tof2 = (x[:a.rows] for x in grid())
    t0 = time.perf_counter()
    sw = S.indirect_transfer_sweep(fx[1], fx[3], tau1, tof1, tof2, thrustLimit=0.05, rho_target=1e-4, backend=be)
    sweep_s = time.perf_counter() - t0
    ok = np.flatnonzero(sw["stage_failed"] == 0)
    XC = np.ascontiguousarray(sw["XC_all"][ok].transpose(0, 2, 1))                   # (n, 30, 12)
    t, rho = sw["t_TU"][ok], sw["rho_last"][ok]
    n = len(ok)
    p = capi.indirect_params(thrustLimit=0.05, p=1.0, rho=1e-4)
    calls = dict(
        switch=lambda: h.indirect_switch_batch(XC, t, params=p, thrustLimit=0.05, rho=rho, max_switch=a.max_switch),
        cost=lambda: h.indirect_cost_batch(XC, t, params=p, thrustLimit=0.05, rho=rho),
        defect=lambda: h.indirect_traj(XC, t, params=p, thrustLimit=0.05, rho=rho, jac=False))
    for f in calls.values():                                                           # warm-up
        f()
    wall = {k: [] for k in calls}; dev = {k: [] for k in calls}
    out = {}
    for _ in range(a.runs):
        for k, f in calls.items():
            t0 = time.perf_counter(); out[k] = f(); wall[k].append((time.perf_counter() - t0) * 1e3)
            dev[k].append(float(h.last_kernel_ms))
    ar = S.thrust_arcs_indirect(sw["XC_all"][ok], t, MU, DU, TU, 1e3, 0.05, rho, max_switch=a.max_switch, backend=be)
    aL = 0.05 * (TU * TU / DU / 1e3) / 1e3
    burn = out["cost"]["dv"] / (aL * DU * 1e3 / TU)
    good = ar["n_burns"] >= 0
    rel = np.abs(ar["on_time"][good] - burn[good]) / burn[good]
    report = dict(
        gpu=gpu_q.splitlines()[0] if gpu_q else "unknown",
        grid=dict(n_traj=int(tau1.size), n_nodes=30, thrustLimit_N=0.05, rho_target=1e-4, rows_through_sweep=n, sweep_wall_s=sweep_s,
                  rho_last={"%g" % k: int(v) for k, v in zip(*np.unique(rho, return_counts=True))}),
        timing={k: dict(runs=a.runs, wall_ms_median=float(np.median(wall[k])), device_ms_median=float(np.median(dev[k])), wall_ms_runs=wall[k],
                        device_ms_runs=dev[k]) for k in calls},
        max_switch=a.max_switch,
        status=_counts(ar["status"]),
        n_switch=_counts(ar["n_switch"]),
        truncated_rows=int((ar["n_switch"] > a.max_switch).sum()),
        n_burns=_counts(ar["n_burns"]),
        on_start=_counts(ar["on_start"]),
        on_time_TU=dict(median=float(np.median(ar["on_time"][good])), min=float(ar["on_time"][good].min()), max=float(ar["on_time"][good].max())),
        on_time_vs_dv_over_aL=dict(rows=int(good.sum()), rel_median=float(np.median(rel)), rel_max=float(rel.max()),
                                   rel_p99=float(np.quantile(rel, 0.99))),
    )
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report, indent=1))
    h.close()


if __name__ == "__main__":
    main()
