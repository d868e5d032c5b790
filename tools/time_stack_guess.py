"""Times the trajectory-stacking initial guess for a trade-study grid: (a) the host loop of solvers.trajectory_stack_guess on the GPU
backend (host splines and find_tau, one propagation call per arc; timed on a subset and reported per transfer), (b) one
lto_stack_guess_batch call for the whole grid (solvers.trajectory_stack_guess_batch), and (c) the whole sweep, guess + batched direct
solve (solvers.direct_transfer_sweep).  (a) and (b) alternate in one process; medians over --runs runs.  Checks (a) against (b) on the
rows (a) ran: tau2 identical, XC within 1e-12.  Reports how many transfers of (c) converged and its iteration histogram.

    python tools/time_stack_guess.py [--runs 3] [--host-rows 128] [--out profiles/r05_stack_guess.json]

Grid: 32 values of tau1 in [0, 1) x 32 (tof1, tof2) pairs in 6-14 days (seeded), 30 nodes -- 1 024 distinct transfers between the
two demo orbits."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from lowthrustopt_b200 import capi, solvers as S  # noqa: E402

MU, DU, TU = capi.MU, capi.DU, capi.TU


def grid(seed=2026):
    rng = np.random.default_rng(seed)
    tau = np.arange(32) / 32.0
    tofs = rng.uniform(6.0, 14.0, (32, 2))
    tau1 = np.repeat(tau, 32)
    tof1 = np.tile(tofs[:, 0], 32); tof2 = np.tile(tofs[:, 1], 32)
    return tau1, tof1, tof2


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--host-rows", type=int, default=128)
    ap.add_argument("--out", default="profiles/r05_stack_guess.json")
    a = ap.parse_args()
    fx = S.demo_fixtures()
    X0, Xf = fx[1], fx[3]
    h = capi.Handle(0)
    gpu = S.GpuBackend(handle=h)
    tau1, tof1, tof2 = grid()
    T, N = tau1.size, 30
    sub = np.linspace(0, T - 1, a.host_rows).astype(int)

    def host():
        t0 = time.perf_counter()
        out = [S.trajectory_stack_guess(X0, Xf, MU, DU, TU, N, float(tof1[j]), float(tof2[j]), float(tau1[j]), backend=gpu) for j in sub]
        return out, time.perf_counter() - t0

    def device():
        t0 = time.perf_counter()
        out = S.trajectory_stack_guess_batch(X0, Xf, MU, DU, TU, N, tof1, tof2, tau1, backend=gpu)
        return out, time.perf_counter() - t0, h.last_kernel_ms

    device(); host()                                                      # warm-up: module load, first launches
    t_host, t_dev, k_dev = [], [], []
    for _ in range(a.runs):
        ho, w = host(); t_host.append(w)
        do, w, k = device(); t_dev.append(w); k_dev.append(k)
    tau2_same = all(do[3][j] == ho[i][3] for i, j in enumerate(sub))
    xc_err = max(float(np.abs(do[0][j] - ho[i][0]).max()) for i, j in enumerate(sub))
    t_sweep = []
    for _ in range(a.runs):
        t0 = time.perf_counter()
        sw = S.direct_transfer_sweep(X0, Xf, tau1, tof1, tof2, n_nodes=N, backend=gpu)
        t_sweep.append(time.perf_counter() - t0)
    gpu_q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    report = dict(
        gpu=gpu_q.splitlines()[0] if gpu_q else "unknown",
        grid=dict(n_traj=T, n_nodes=N, tau1="32 values k/32", tof_days="32 seeded (tof1, tof2) pairs in [6, 14]"),
        host_loop=dict(rows=int(len(sub)), wall_s_median=float(np.median(t_host)), wall_s_runs=t_host,
                       ms_per_transfer=float(np.median(t_host)) / len(sub) * 1e3,
                       extrapolated_s_for_grid=float(np.median(t_host)) / len(sub) * T),
        device_guess=dict(wall_ms_median=float(np.median(t_dev)) * 1e3, wall_ms_runs=[x * 1e3 for x in t_dev],
                          device_ms_median=float(np.median(k_dev)), device_ms_runs=k_dev),
        check=dict(tau2_identical=bool(tau2_same), max_abs_xc_diff=xc_err),
        sweep=dict(wall_s_median=float(np.median(t_sweep)), wall_s_runs=t_sweep, converged=int(sw["converged"].sum()),
                   iteration_histogram={int(k): int(v) for k, v in zip(*np.unique(sw["iters"], return_counts=True))}),
    )
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report, indent=1))
    h.close()
    assert tau2_same and xc_err <= 1e-12, (tau2_same, xc_err)


if __name__ == "__main__":
    main()
