"""Timing of the 14-dim device Newton update and of the batched 14-dim solve on one GPU; prints ONE JSON line.

    python tools/time_indirect14_solve.py [--out FILE]

  * k_indirect_newton<14> and <12> (full mode) and their re-solves, 1,024 trajectories x 201 nodes, CUDA events on lto_stream,
    the two dimensions alternated in the same process (Phi blocks and defects from one STM pass of each system);
  * lto_indirect_solve_batch_nd(14) on synthetic.continuation_batch(1024, 200, ndim=14) with bench.py continuation_solve's settings
    (p = 2, thrustLimit 10, max_iter 8, max_attempts 5000): host wall clock around the blocking call and its device time
    (lto_last_kernel_ms), trajectories converged, largest iteration count;
  * the GPU's name and power limit, read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np
import torch

from lowthrustopt_b200 import capi, synthetic


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().split(", ")
    return {"gpu": q[0] if q else torch.cuda.get_device_name(0), "power_limit": q[1] if len(q) > 1 else None,
            "max_sm_clock": q[2] if len(q) > 2 else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    ap.add_argument("--n-traj", type=int, default=1024)
    args = ap.parse_args()
    T, spu = args.n_traj, 200
    N = spu + 1
    dev = torch.device("cuda", 0)
    h = capi.Handle(0)
    stream = torch.cuda.ExternalStream(h.stream, device=dev)
    p = capi.indirect_params(p=2.0, thrustLimit=10.0, rho=1.0); p.max_attempts = 5000

    # ---- Newton update kernels: inputs from one STM pass of each system
    sets = {}
    for nd in (12, 14):
        c = synthetic.continuation_batch(n_traj=T, n_seg_per_traj=spu, ndim=nd)
        dXC = torch.from_numpy(c["XC_all"]).to(dev); dT = torch.from_numpy(c["t_TU"]).to(dev)
        d_def = torch.empty((T * spu, nd), dtype=torch.float64, device=dev); d_phi = torch.empty((T * spu, nd, nd), dtype=torch.float64, device=dev)
        d_ns = torch.empty((T * spu, 2), dtype=torch.int32, device=dev)
        h.indirect_dev(p, T * spu, N, nd, dXC.data_ptr(), dT.data_ptr(), None, None, None, None, d_def.data_ptr(), None, d_ns.data_ptr(),
                       d_phi.data_ptr())
        d2 = (d_def * 0.5).contiguous()
        upd = torch.empty((T, N, nd), dtype=torch.float64, device=dev); upd2 = torch.empty_like(upd)
        st = torch.zeros(T, dtype=torch.int32, device=dev)
        sets[nd] = (d_phi, d_def, d2, upd, upd2, st)
    h.sync()

    def timed(fn, reps=10):
        for _ in range(2):
            fn()
        h.sync()
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            a.record()
            for _ in range(reps):
                fn()
            b.record()
        h.sync()
        return a.elapsed_time(b) / reps

    samples = {k: [] for k in ("newton12", "newton14", "resolve12", "resolve14")}
    nan_status = {}
    for _ in range(5):                                                    # the two dimensions alternated
        for nd in (12, 14):
            d_phi, d_def, d2, upd, upd2, st = sets[nd]
            fact = lambda: h.indirect_newton_dev(T, N, 0, d_phi.data_ptr(), d_def.data_ptr(), upd.data_ptr(), st.data_ptr(), ndim=nd)
            samples["newton%d" % nd].append(timed(fact))
            fact()                                                        # the factorisation the re-solve replays
            samples["resolve%d" % nd].append(timed(lambda: h.indirect_newton_resolve_dev(T, N, 0, d2.data_ptr(), upd2.data_ptr(), ndim=nd)))
            nan_status[nd] = int((st != 0).sum().item())
    ms = {k: statistics.median(v) for k, v in samples.items()}

    # ---- the batched 14-dim solve (continuation_solve's settings)
    c = synthetic.continuation_batch(n_traj=T, n_seg_per_traj=spu, ndim=14)
    walls, devs = [], []
    for rep in range(4):
        XC = c["XC_all"].copy()
        t0 = time.perf_counter()
        r = h.indirect_solve_batch(XC, c["t_TU"], params=p, max_iter=8)
        wall = (time.perf_counter() - t0) * 1e3
        if rep > 0:                                                       # the first call allocates the solver's arrays
            walls.append(wall); devs.append(h.last_kernel_ms)
    line = {"what": "14-dim device Newton update and batched solve", "n_traj": T, "n_nodes": N,
            "newton_full_ms": {"k_indirect_newton<12>": ms["newton12"], "k_indirect_newton<14>": ms["newton14"],
                               "ratio_14_over_12": ms["newton14"] / ms["newton12"]},
            "resolve_full_ms": {"k_indirect_newton_resolve<12>": ms["resolve12"], "k_indirect_newton_resolve<14>": ms["resolve14"]},
            "newton_samples_ms": samples, "newton_nonzero_status": nan_status,
            "solve14": {"call": "lto_indirect_solve_batch_nd(ndim=14)", "p": 2.0, "thrustLimit": 10.0, "max_iter": 8, "max_attempts": 5000,
                        "wall_ms_median": statistics.median(walls), "last_kernel_ms_median": statistics.median(devs), "wall_ms": walls,
                        "last_kernel_ms": devs, "converged": int((r["status_flag"] == 0).sum()), "flag_counts": np.bincount(r["status_flag"], minlength=3).tolist(),
                        "iters_max": int(r["iters"].max())},
            "timing": "kernels: CUDA events on lto_stream, mean of 10 launches, median of 5 alternated rounds; solve: host wall clock around the "
                      "blocking call, median of 3 after one warm-up call",
            "machine": gpu_info(), "torch": torch.__version__}
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")
    h.close()


if __name__ == "__main__":
    main()
