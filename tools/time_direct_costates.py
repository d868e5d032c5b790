"""Measures lto_direct_costates_batch and the sweep's two starts on the 1 024-transfer grid of tools/time_stack_guess.py (30 nodes,
thrustLimit 0.05 N, rho_target 1e-4):
  * lto_direct_costates_batch on the direct sweep's 1 024 solutions: wall (host clock around the call, which ends in a device
    synchronise) and device time (the call's kernel events), alternated with the stage it replaces -- the seeded start's adjoints-only
    p = 2 solve (lto_indirect_solve_batch, maxIter 10) -- medians over --runs runs;
  * solvers.indirect_transfer_sweep with start="seeded" and start="direct", alternated: wall time, per-stage failure counts, stage-2
    iteration counts, and dv / energy agreement on the rows both bring through.

    python tools/time_direct_costates.py [--runs 3] [--rows 1024] [--out profiles/r07_direct_costates.json]"""
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


class Stage2Backend(S.GpuBackend):
    """GpuBackend that keeps the per-row iteration counts of the stage-2 solve (full p = 2, maxIter 50) of the last sweep."""

    def indirect_solve_batch(self, XC, t, params, thrustLimit=None, rho=None, max_iter=50, flag_adjointsOnly=False):
        r = super().indirect_solve_batch(XC, t, params, thrustLimit=thrustLimit, rho=rho, max_iter=max_iter, flag_adjointsOnly=flag_adjointsOnly)
        if max_iter == 50 and not flag_adjointsOnly:
            self.stage2 = (r["iters"].copy(), r["status_flag"].copy())
        return r


def _counts(a):
    return {int(k): int(v) for k, v in zip(*np.unique(a, return_counts=True))}


def _rel_agreement(a, b):
    r = np.abs(a - b) / np.abs(b)
    return dict(rows=int(r.size), max=float(r.max()) if r.size else None, median=float(np.median(r)) if r.size else None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--rows", type=int, default=1024)
    ap.add_argument("--out", default="profiles/r07_direct_costates.json")
    a = ap.parse_args()
    gpu_q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    fx = S.demo_fixtures()
    h = capi.Handle(0)
    be = Stage2Backend(handle=h)
    tau1, tof1, tof2 = (x[:a.rows] for x in grid())
    T = tau1.size

    # ---- the call against the stage it replaces
    d = S.direct_transfer_sweep(fx[1], fx[3], tau1, tof1, tof2, backend=be)
    X, U, t = d["X_all"].transpose(0, 2, 1).copy(), d["u_all"].transpose(0, 2, 1).copy(), d["t_TU"]
    XC_seed = np.empty((T, 12, 30))
    for j in range(T):
        rng = np.random.default_rng(j)
        XC_seed[j] = np.vstack([d["X_all"][j], 0.1 * rng.standard_normal((6, 30))])
        XC_seed[j, :6, 0] = d["state_0"][j]; XC_seed[j, :6, -1] = d["state_f"][j]
        XC_seed[j, :, 1:-1] += 1e-10 * rng.standard_normal((12, 28))
    XC_seed = np.ascontiguousarray(XC_seed.transpose(0, 2, 1))
    p2 = capi.indirect_params(thrustLimit=10.0, p=2.0, rho=1.0)
    c = h.direct_costates_batch(X, U, t, d["state_0"], d["state_f"])                                  # warm-up of both
    h.indirect_solve_batch(XC_seed, t, params=p2, max_iter=10, flag_adjointsOnly=True)
    wc, kc, ws = [], [], []
    for _ in range(a.runs):
        t0 = time.perf_counter(); c = h.direct_costates_batch(X, U, t, d["state_0"], d["state_f"]); wc.append(time.perf_counter() - t0)
        kc.append(h.last_kernel_ms)
        t0 = time.perf_counter(); h.indirect_solve_batch(XC_seed, t, params=p2, max_iter=10, flag_adjointsOnly=True); ws.append(time.perf_counter() - t0)

    # ---- the two sweeps, alternated
    S.indirect_transfer_sweep(fx[1], fx[3], tau1[:8], tof1[:8], tof2[:8], backend=be, start="direct")      # warm-up
    walls = {"seeded": [], "direct": []}
    sweeps, it2 = {}, {}
    for _ in range(a.runs):
        for start in ("seeded", "direct"):
            t0 = time.perf_counter()
            sweeps[start] = S.indirect_transfer_sweep(fx[1], fx[3], tau1, tof1, tof2, backend=be, start=start)
            walls[start].append(time.perf_counter() - t0)
            it2[start] = be.stage2
    sd, dd = sweeps["seeded"], sweeps["direct"]
    both = (sd["stage_failed"] == 0) & (dd["stage_failed"] == 0)
    both_p2 = np.isfinite(sd["energy_p2"]) & np.isfinite(dd["energy_p2"])

    def sweep_report(start):
        s = sweeps[start]; iters, flag = it2[start]
        ok = iters[flag == 0]
        return dict(wall_s_median=float(np.median(walls[start])), wall_s_runs=walls[start], stage_failed=_counts(s["stage_failed"]),
                    stage2=dict(rows_entered=int(iters.size), converged=int((flag == 0).sum()), iterations_of_converged=_counts(ok),
                                iterations_mean=float(ok.mean()) if ok.size else None))

    report = dict(
        gpu=gpu_q.splitlines()[0] if gpu_q else "unknown",
        grid=dict(n_traj=T, n_nodes=30, tau1="32 values k/32", tof_days="32 seeded (tof1, tof2) pairs in [6, 14]", thrustLimit_N=0.05,
                  rho_target=1e-4, seeds="row index", direct_converged=int(d["converged"].sum())),
        direct_costates_batch=dict(runs=a.runs, wall_ms_median=float(np.median(wc)) * 1e3, device_ms_median=float(np.median(kc)),
                                   wall_ms_runs=[w * 1e3 for w in wc], device_ms_runs=kc, status=_counts(c["status"]),
                                   du_max_N=dict(median=float(np.median(c["du_max"])), max=float(c["du_max"].max()))),
        seeded_stage1_adjoints_only=dict(runs=a.runs, wall_ms_median=float(np.median(ws)) * 1e3, wall_ms_runs=[w * 1e3 for w in ws]),
        sweep=dict(seeded=sweep_report("seeded"), direct=sweep_report("direct")),
        agreement=dict(rows_both_through=int(both.sum()),
                       dv=_rel_agreement(dd["dv"][both], sd["dv"][both]), energy=_rel_agreement(dd["energy"][both], sd["energy"][both]),
                       p2_energy=_rel_agreement(dd["energy_p2"][both_p2], sd["energy_p2"][both_p2]),
                       only_seeded_through=int(((sd["stage_failed"] == 0) & (dd["stage_failed"] != 0)).sum()),
                       only_direct_through=int(((dd["stage_failed"] == 0) & (sd["stage_failed"] != 0)).sum())),
    )
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report, indent=1))
    h.close()


if __name__ == "__main__":
    main()
