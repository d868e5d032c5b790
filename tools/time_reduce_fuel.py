"""Times the rho continuation of reduceFuel_indirect on the GPU: the device ladder (reduceFuel_indirect_batch(device_ladder=True),
one lto_indirect_reduce_fuel_batch call) against the round-based driver (one lto_indirect_solve_batch call per round), alternated
in one process on the same inputs and back-off draws, and checks that both return bitwise-equal outputs.

Demo size: n_traj ladders of the demo's 30-node transfer, from p = 1, rho = 1 solutions built with the batched solvers (demo
pipeline: direct solve, then p = 2 and p = 1 indirect batches from seeded costates), thrustLimit geomspace(0.05, 0.2) N and targets
geomspace(1e-1, 1e-4) spread across the trajectories so that the ladders differ in length.

    python tools/time_reduce_fuel.py [--n-traj 1024] [--runs 3] [--out profiles/r04_reduce_fuel.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from lowthrustopt_b200 import capi, solvers as S  # noqa: E402

MU, DU, TU = capi.MU, capi.DU, capi.TU


class CountingBackend(S.GpuBackend):
    """Records, per round of the host driver, the slowest trajectory's Newton iterations and the call's device time."""

    def __init__(self, h):
        super().__init__(handle=h)
        self.rounds = []

    def indirect_solve_batch(self, *a, **k):
        r = super().indirect_solve_batch(*a, **k)
        self.rounds.append((int(r["iters"].max()), int(r["iters"].sum()), self.h.last_kernel_ms, int(r["iters"].size)))
        return r


def demo_starts(gpu, n):
    fx = S.demo_fixtures()
    XCg, t_TU, tau1, tau2, s0, sf = S.trajectory_stack_guess(fx[1], fx[3], backend=gpu)
    X_all = S.multiShoot_CRTBP_direct(XCg[:6].copy(), np.zeros((3, 30)), tau1, tau2, t_TU, np.zeros(3), np.zeros(3), MU, DU, TU, 30, 10, 1e3,
                                      2000.0, *fx, backend=gpu)[0]
    rng = np.random.default_rng(0)
    XC0 = np.repeat(np.vstack([X_all, np.zeros((6, 30))])[None], n, axis=0)
    XC0[:, 6:] = 0.1 * rng.standard_normal((n, 6, 30))
    XC0[:, :6, 0] = s0[:6]; XC0[:, :6, -1] = sf[:6]
    XC0[:, :, 1:-1] += 1e-10 * rng.standard_normal((n, 12, 28))
    tt = np.broadcast_to(t_TU, (n, 30)).copy()
    tl = np.geomspace(0.05, 0.2, n)
    X2, _, s2, _ = S.multiShoot_CRTBP_indirect_batch(XC0, tt, MU, DU, TU, 30, 1e3, 10.0, False, 50, 2.0, 1.0, backend=gpu)
    X1, _, s1, _ = S.multiShoot_CRTBP_indirect_batch(X2, tt, MU, DU, TU, 30, 1e3, tl, False, 30, 1.0, 1.0, backend=gpu)
    ok = np.flatnonzero((s2 == 0) & (s1 == 0))
    if ok.size == 0:
        raise RuntimeError("no start converged")
    pick = ok[np.arange(n) % ok.size]                 # converged starts, repeated (with their own thrustLimit) up to n ladders
    return X1[pick], tt, tl[pick], int(ok.size)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-traj", type=int, default=1024)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--out", default="profiles/r04_reduce_fuel.json")
    a = ap.parse_args()
    h = capi.Handle(0)
    gpu = CountingBackend(h)
    X1, tt, tl, n_conv = demo_starts(gpu, a.n_traj)
    T = X1.shape[0]
    target = np.random.default_rng(1).permutation(np.geomspace(1e-1, 1e-4, T))
    draws_rngs = lambda: [np.random.default_rng(j) for j in range(T)]  # noqa: E731

    def host():
        gpu.rounds = []
        t0 = time.perf_counter()
        out = S.reduceFuel_indirect_batch(X1, tt, MU, DU, TU, 30, 1e3, tl, 1.0, target, backend=gpu, rngs=draws_rngs())
        return out, time.perf_counter() - t0, sum(r[2] for r in gpu.rounds)

    def device():
        t0 = time.perf_counter()
        out = S.reduceFuel_indirect_batch(X1, tt, MU, DU, TU, 30, 1e3, tl, 1.0, target, backend=gpu, rngs=draws_rngs(), device_ladder=True)
        return out, time.perf_counter() - t0, h.last_kernel_ms

    host(); device()                                  # warm-up
    res = {"host": [], "device": []}
    for _ in range(a.runs):
        for name, f in (("host", host), ("device", device)):
            out, wall, dev_ms = f()
            res[name].append(dict(wall_s=wall, device_ms=dev_ms))
            if name == "host":
                ho, host_rounds = out, list(gpu.rounds)
            else:
                do = out
    draws = np.stack([r.random(100) for r in draws_rngs()])
    rd = h.indirect_reduce_fuel_batch(np.ascontiguousarray(X1.transpose(0, 2, 1)), tt, 1.0, target, draws, params=capi.indirect_params(p=1.0),
                                      thrustLimit=tl, max_iter=10)
    gpu_q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    med = lambda v: float(np.median(v))  # noqa: E731
    report = dict(
        gpu=gpu_q.splitlines()[0] if gpu_q else "unknown",
        n_traj=T, n_nodes=30, converged_distinct_starts=n_conv, runs=a.runs,
        host_driver=dict(wall_s=[r["wall_s"] for r in res["host"]], device_ms=[r["device_ms"] for r in res["host"]],
                         wall_s_median=med([r["wall_s"] for r in res["host"]]), rounds=int(ho[3]), solver_calls=int(sum(r[3] for r in host_rounds)),
                         sum_of_round_max_newton_iters=int(sum(r[0] for r in host_rounds)), newton_iters=int(sum(r[1] for r in host_rounds))),
        device_ladder=dict(wall_s=[r["wall_s"] for r in res["device"]], device_ms=[r["device_ms"] for r in res["device"]],
                           wall_s_median=med([r["wall_s"] for r in res["device"]]), solver_calls=int(rd["calls"].sum()),
                           newton_iters=int(rd["newton_iters"].sum()), max_newton_iters_of_one_ladder=int(rd["newton_iters"].max()),
                           launches_per_call=None),
        status_counts={str(s): int((ho[2] == s).sum()) for s in range(4)},
        bitwise_equal=bool(np.array_equal(ho[0], do[0]) and np.array_equal(ho[1], do[1]) and np.array_equal(ho[2], do[2]) and ho[3] == do[3]),
    )
    l0 = h.launches
    h.indirect_reduce_fuel_batch(np.ascontiguousarray(X1.transpose(0, 2, 1)), tt, 1.0, target, draws, params=capi.indirect_params(p=1.0),
                                 thrustLimit=tl, max_iter=10)
    report["device_ladder"]["launches_per_call"] = h.launches - l0
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report, indent=1))


if __name__ == "__main__":
    main()
