#!/usr/bin/env python
"""bench.py -- segment-propagations/s (fp64 state + STM) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic segments.  Default
workload (BASELINE.json configs[2]): 65,536 direct-method segments per GPU, 7-state + STM
+ control sensitivities, the reference's FIXED RKF7(8) grid (nsteps = 10, what
multiShoot_CRTBP_direct actually runs; `--workload direct7_adaptive` runs the ode78
controller instead).  Weak scaling: every rank owns its own 65,536 segments, no data-path
collective (segments are independent).

Prints ONE JSON line (rank 0).  `value` times the kernel(s) with inputs resident in HBM
(CUDA events on the launching stream, L2 flushed between iterations); `e2e` times the
C-ABI host-buffer call (pinned host memory, H2D + kernels + D2H inside the timed region).
`--dump-outputs DIR` writes what the timed path returned in its last step (dump_outputs); the inputs are seeded, so two
builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# Algorithmic FLOPs per unit: profiles/flops_per_unit.json, written by tools/flopcount/count.py -- the kernels' own host-device
# arithmetic compiled with a FLOP-counting scalar (SURVEY.md 7.1 / 8(d)); `used` = min(survey-time figure, every counted formulation).
def _flop_table():
    with open(os.path.join(ROOT, "profiles", "flops_per_unit.json")) as f:
        return json.load(f)


FLOP_TABLE = _flop_table()
FLOPS_PER_SEG = {"direct7": float(FLOP_TABLE["used"]["direct7_segment"]), "direct6": float(FLOP_TABLE["used"]["direct6_segment"])}
FLOPS_PER_STEP_INDIRECT = {12: float(FLOP_TABLE["used"]["indirect12_step"]), 14: float(FLOP_TABLE["used"]["indirect14_step"])}
FLOPS_COUNTED = {"direct7": FLOP_TABLE["counted"]["direct7_segment"]["flops"], "direct6": FLOP_TABLE["counted"]["direct6_segment"]["flops"],
                 12: min(FLOP_TABLE["counted"]["indirect12_step_first_order"]["flops"], FLOP_TABLE["counted"]["indirect12_step_half_column"]["flops"]),
                 14: FLOP_TABLE["counted"]["indirect14_step_first_order"]["flops"]}
# Algorithmic HBM bytes per unit (SURVEY.md 8(d))
BYTES_PER_SEG = {"direct7": 1360.0, "direct6": (2 * 6 + 6 + 2 + 6 + 1 + 6 * 18) * 8.0, 12: 1360.0, 14: 1808.0}

WORKLOADS = ["direct7_fixed", "direct6_fixed", "direct7_adaptive", "indirect12", "indirect14", "indirect12_1m", "continuation",
             "continuation_solve"]
SHARDED = ("indirect12_1m", "continuation")      # strong-scaling workloads: fixed total, sharded + all-gathered (lowthrustopt_b200/sharded.py)
DUMP_BYTES = 60_000_000                          # --dump-outputs: data of all files together (the .npy headers keep it under 64 MB)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="direct7_fixed", choices=WORKLOADS)
    ap.add_argument("--n-seg", type=int, default=0, help="segments per GPU (default: 65536 direct / 131072 indirect)")
    ap.add_argument("--kernel", default="auto", choices=["auto", "generic", "fast"])
    ap.add_argument("--err-norm", default="joint", choices=["joint", "state"], help="indirect step-control norm: x+Phi (ForwardDiff semantics) or x only")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample", type=int, default=0)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU time of the cpu_baseline leg")
    ap.add_argument("--chunks", type=int, default=4, help="all-gather / compute overlap chunks of the sharded paths")
    ap.add_argument("--single-process", action="store_true",
                    help="ONE process drives --gpus devices through lto_init_devices (the form the Julia drop-in uses): host-buffer calls only, "
                         "no torch.distributed; prints one JSON line whose value is the end-to-end rate")
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"],
                    help="sharded workloads: deliver results to the solver rank by the kernels' own stores into its HBM over NVLink "
                         "peer memory (fused, default) or by a chunked NCCL all-gather")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the arrays the timed path returned in its last step as DIR/<name>.npy (float64; "
                         "a fixed, seeded sample of units when they exceed 60 MB)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; --impl reference has none")
    return a


def dump_outputs(directory, arrays, seed=20180005):
    """DIR/<name>.npy in float64 for every array the timed path returned in its last step.  Every array is indexed by unit (segment or
    trajectory) along its first axis; when together they exceed DUMP_BYTES, the same seeded sample of units is kept of each, and the
    sampled unit indices are written as DIR/sample_index.npy."""
    host = {k: (v.cpu().numpy() if hasattr(v, "cpu") else np.asarray(v)).astype(np.float64) for k, v in arrays.items()}
    n = len(next(iter(host.values())))
    if sum(a.nbytes for a in host.values()) > DUMP_BYTES:
        per_unit = sum(a[0].nbytes for a in host.values()) + 8
        keep = np.sort(np.random.default_rng(seed).choice(n, DUMP_BYTES // per_unit, replace=False))
        host = {k: a[keep] for k, a in host.items()}
        host["sample_index"] = keep.astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(directory, k + ".npy"), a)


def make_batch(workload, n_seg, rank):
    from lowthrustopt_b200 import synthetic as S
    if workload.startswith("direct"):
        ns = 7 if workload.startswith("direct7") else 6
        return S.direct_batch(n_seg, nstate=ns, seed=20180001 + rank)
    nd = 12 if workload == "indirect12" else 14
    return S.indirect_batch(n_seg, ndim=nd, seed=20180002 + rank)


class ClockSampler(threading.Thread):
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index; self.rows = []; self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        busy = [x for x in sm if x > 0.5 * (max(mx) if mx else 1)] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------- NUMA placement of the pinned host buffers
def _cpulist(txt):
    cpus = set()
    for part in txt.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        cpus.update(range(int(a), int(b or a) + 1))
    return cpus


def numa_bind(device_index):
    """Before the pinned host buffers of the e2e leg are allocated: move this thread onto the CPUs of the NUMA node the GPU hangs off, so
    that cudaHostAlloc places the pages there (PCIe DMA into the other socket's memory crosses the inter-socket link).  Returns
    (previous affinity or None, note for the JSON line); never raises -- on any doubt nothing is changed."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(device_index)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        with open("/sys/bus/pci/devices/%s/numa_node" % bdf) as f:
            node = int(f.read().strip())
        if node < 0:
            return None, "no NUMA information for %s" % bdf
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpus = _cpulist(f.read())
        old = os.sched_getaffinity(0)
        want = old & cpus
        if not want:
            return None, "GPU %s is on NUMA node %d, none of its CPUs is available to this process" % (bdf, node)
        os.sched_setaffinity(0, want)
        return old, "pinned host buffers allocated from a CPU of NUMA node %d (the node of GPU %s)" % (node, bdf)
    except Exception as e:                                                   # noqa: BLE001
        return None, "NUMA placement skipped (%s)" % type(e).__name__


def numa_restore(old):
    try:
        if old:
            os.sched_setaffinity(0, old)
    except Exception:                                                        # noqa: BLE001
        pass


# --------------------------------------------------------------------------- CPU legs (oracle = checker / baseline only)
def host_threads():
    """Threads the CPU legs use: every CPU this process may run on.  NOT the OpenMP default -- torch.distributed.run exports
    OMP_NUM_THREADS=1 into its workers, which silently turned the N > 1 reference arm of round 1 into a 1-thread run; the oracle's
    entry points take the count explicitly (an `omp parallel for num_threads(n)` clause overrides the environment)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_variational_pass(batch, n, nthreads):
    """One pass of the SAME MATHS as the GPU path on the host (BASELINE.md section 4, mode 2): the state and its variational
    equations [Phi | Gamma] in one RKF7(8) integration per leg, structural zeros skipped -- the kernels' own __host__ __device__
    arithmetic compiled for the host cores (oracle_direct_variational_host) -- instead of the reference's 2(n+3) finite-difference
    re-propagations.  Direct workloads only -- for the indirect ones the reference algorithm (dual numbers) already is this."""
    from oracle import oracle as O
    sl = {k: v[:n] for k, v in batch.items()}
    t = time.perf_counter()
    O.direct_variational_host(sl["Xa"], sl["Xb"], sl["ua"], sl["ub"], sl["ta"], sl["tb"], nthreads=nthreads)
    return time.perf_counter() - t


def cpu_reference_pass(workload, batch, n, nthreads):
    """One pass of the REFERENCE ALGORITHM on the host: direct = defectCalc + forward-FD jacobianCalc
    (multiShoot_CRTBP_direct.jl:66-143, pert 1e-8, both legs re-propagated per variable); indirect = dual numbers
    through the adaptive solver (multiShoot_CRTBP_indirect.jl:93-124).  Returns seconds."""
    from oracle import oracle as O
    t = time.perf_counter()
    if workload.startswith("direct"):
        sl = {k: v[:n] for k, v in batch.items()}
        mode = 1 if workload.endswith("adaptive") else 0
        d, e, st, _ = O.direct_defect(sl["Xa"], sl["Xb"], sl["ua"], sl["ub"], sl["ta"], sl["tb"], mode=mode, nthreads=nthreads)
        O.direct_jac_fd(sl["Xa"], sl["Xb"], sl["ua"], sl["ub"], sl["ta"], sl["tb"], d, mode=mode, nthreads=nthreads)
    else:
        ip = O.iparams(0.05, p=1.0, rho=1.0)
        O.indirect_prop_jac(batch["x0"][:n], batch["t0"][:n], batch["t1"][:n], ip, nthreads=nthreads)
    return time.perf_counter() - t


def cpu_baseline(workload, batch, sample, seconds=12.0):
    """The reference ALGORITHM on the host cores for about `seconds` of CPU work: repeated passes over the first
    `sample` segments of the same batch."""
    from oracle import oracle as O
    O.build()
    nthreads = host_threads()
    n = min(sample, len(next(iter(batch.values()))))
    cpu_reference_pass(workload, batch, min(n, 256), nthreads)        # warm the thread pool
    dt, passes = 0.0, 0
    while dt < seconds and passes < 10000:
        dt += cpu_reference_pass(workload, batch, n, nthreads); passes += 1
    out = {"value": n * passes / dt, "unit": "segment-propagations/s", "cores": nthreads, "kind": "port",
           "sample": "%d passes over the first %d segments of the same batch, reference algorithm (%s) restated in C++ (oracle/), "
                     "OpenMP over segments on %d threads, %.1f s"
                     % (passes, n, "defectCalc + forward-FD jacobianCalc, pert 1e-8" if workload.startswith("direct") else
                        "dual numbers through the adaptive RK8", nthreads, dt)}
    if workload.endswith("_fixed"):                                   # equal-algorithm comparison next to the reference-algorithm one
        dv, pv = 0.0, 0
        while dv < seconds / 3.0 and pv < 10000:
            dv += cpu_variational_pass(batch, n, nthreads); pv += 1
        out["variational"] = {"value": n * pv / dv, "unit": "segment-propagations/s", "cores": nthreads, "kind": "port",
                              "sample": "%d passes over the same %d segments, the GPU path's own maths (state + variational equations in one "
                                        "RKF7(8) integration per leg: the kernels' host-device arithmetic compiled for the host), %.1f s" % (pv, n, dv)}
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O
    O.build()
    nthreads = host_threads()
    if args.workload == "continuation_solve":
        from lowthrustopt_b200 import synthetic as S
        c = S.continuation_batch(n_traj=64, n_seg_per_traj=200, ndim=12)
        cb = cpu_solve_baseline(c["XC_all"], c["t_TU"], 64, args.cpu_seconds)
        print(json.dumps({"impl": "reference", "metric": "segment-propagations/s (fp64 state+STM)", "value": cb["value"], "unit": cb["unit"],
                          "n_gpus": args.gpus, "steps": 1, "warmup": 0, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                          "dtype": "f64", "data": "synthetic", "config": {"workload": "continuation_solve"}, "cpu_baseline": cb,
                          "e2e": {"value": cb["value"], "unit": cb["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}), flush=True)
        return
    n_seg = args.n_seg or (65536 if args.workload.startswith("direct") else 131072)
    sample = args.cpu_sample or (16384 if args.workload.startswith("direct") else 4096)
    batch = make_batch(args.workload, sample, 0)
    for _ in range(max(1, min(args.warmup, 1))):
        cpu_reference_pass(args.workload, batch, min(sample, 512), nthreads)
    t = 0.0
    for _ in range(args.steps):
        t += cpu_reference_pass(args.workload, batch, sample, nthreads)
    v = sample * args.steps / t
    line = {"impl": "reference", "metric": "segment-propagations/s (fp64 state+STM)", "value": v, "unit": "segment-propagations/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args.workload, n_seg, args.gpus),
            "cpu_baseline": {"value": v, "unit": "segment-propagations/s", "cores": nthreads, "kind": "port",
                             "sample": "%d segments per step; the reference is Julia (not installed here or on the GPU box), so this is its "
                                       "algorithm restated in C++ (oracle/), OpenMP over segments on all host threads" % sample},
            "e2e": {"value": v, "unit": "segment-propagations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def workload_config(workload, n_seg, n_gpus, gather="peer"):
    if workload in SHARDED:
        desc = {"indirect12_1m": "BASELINE configs[3]: 1,048,576 perturbed indirect-shooting guesses (12-dim reference RHS, adaptive RK8 1e-13, "
                                 "12x12 STM) in TOTAL, sharded across the GPUs, defects + STM blocks delivered to the solver rank",
                "continuation": "BASELINE configs[4]: 1,024 trajectories x 200 segments (L2_Anderson_2 ballistic stack, thrustLimit ladder 10 -> 0.05 N); "
                                "one step = one Newton iteration of multiShoot_CRTBP_indirect = 1 STM pass + 22 defect-only passes (SOC, check, and the "
                                "20 line-search points as ONE batched pass of 20,480 trial trajectories reduced to sum(defect^2) on the device); "
                                "results delivered to the solver rank"}[workload]
        return {"workload": workload, "description": desc, "segments_total": n_seg, "segments_per_gpu": n_seg // n_gpus,
                "l2": "not flushed: each pass writes more output than the 126 MB L2 holds",
                "parallelism": ("contiguous slabs of units on %d GPU(s), one launch per rank and pass; the kernels store their slab into the solver "
                                "rank's HBM over NVLink peer memory (no collective)" % n_gpus if gather == "peer" else
                                "units interleaved across %d GPU(s) in chunks; NCCL all-gather of each chunk overlapped with the next chunk's "
                                "kernel" % n_gpus)}
    desc = {
        "direct7_fixed": "BASELINE configs[2]: synthetic batch of 65,536 direct-method segments per GPU, nstate 7 + STM + control "
                         "sensitivities (7x20 Jacobian block), FIXED RKF7(8) grid nsteps=10 both legs (reference ode7_8 path)",
        "direct6_fixed": "direct-method segments, nstate 6 (the demo's size), FIXED RKF7(8) nsteps=10",
        "direct7_adaptive": "BASELINE configs[2] with the ode78 adaptive controller, tol 1e-13",
        "indirect12": "BASELINE configs[3] (12-dim reference RHS): perturbed indirect-shooting guesses, adaptive RK8 1e-13, 12x12 STM",
        "indirect14": "BASELINE configs[3] (14-dim extension): adaptive RK8 1e-13, 14x14 STM",
    }[workload]
    return {"workload": workload, "description": desc, "segments_per_gpu": n_seg, "segments_total": n_seg * n_gpus,
            "l2": "flushed between timed iterations (256 MiB write)", "parallelism": "segments sharded across %d GPU(s), no collective" % n_gpus}


# --------------------------------------------------------------------------- GPU arm
def dist_setup():
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    return world, rank, local


def executed_flops(wl, units_per_launch, kernel_ms, peak, attempted=None):
    """What ncu counted for the dominant kernel of this workload (profiles/executed.json: thread-level DFMA/DMUL/DADD executed per
    unit and FP64-pipe-active %, from the committed --set full capture of the same build) next to the algorithmic figure: the
    achieved rate in EXECUTED flops and its fraction of the measured peak.  None when no capture is on file for the workload."""
    try:
        with open(os.path.join(ROOT, "profiles", "executed.json")) as f:
            e = json.load(f).get(wl)
    except Exception:
        e = None
    if not e:
        return None
    per_unit = e["flops_per_unit"]
    if e.get("attempted_steps_per_unit"):                      # adaptive kernels: the capture's count scales with the attempted steps of THIS batch
        if attempted is None:
            return None
        per_unit = per_unit / e["attempted_steps_per_unit"] * attempted
    ach = per_unit * units_per_launch / (kernel_ms * 1e-3) / 1e12
    return {"flops_per_unit": per_unit, "achieved": ach, "frac": ach / (peak / 1e12), "fp64_pipe_active_pct": e.get("fp64_pipe_active_pct"),
            "source": e.get("source")}


def fp64_roofline(h, flops_unit, units_per_launch, kernel_ms, bytes_unit, wl, flops_counted=None, attempted=None):
    peak_burst, _ = h.fp64_peak_probe(2048)
    peak_sust, ms_p = h.fp64_peak_probe(200000)
    achieved = flops_unit * units_per_launch / (kernel_ms * 1e-3) / 1e12
    hbm = None
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            hbm = json.load(f).get("hbm_gbs")
    except Exception:
        pass
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic = json.load(f).get(wl)
    except Exception:
        pass
    gbs = bytes_unit * units_per_launch / (kernel_ms * 1e-3) / 1e9
    return {"bound": "fp64", "achieved": achieved, "peak": peak_sust / 1e12, "unit": "TFLOP/s", "frac": achieved / (peak_sust / 1e12),
            "traffic": traffic,
            "peak_source": "DFMA issue-rate probe (lto_fp64_peak_probe) run on this GPU in this process: sustained %.2f TFLOP/s over %.0f ms, "
                           "burst %.2f; MEASURED_PEAKS.json carries no FP64 figure; spec 148 SM x 64 DFMA/clk x 2 x 1.965 GHz = 37.2"
                           % (peak_sust / 1e12, ms_p, peak_burst / 1e12),
            "flops_per_unit": flops_unit, "units_per_launch": units_per_launch, "kernel_ms": kernel_ms,
            "flops_source": "profiles/flops_per_unit.json (tools/flopcount/count.py: the kernels' host-device arithmetic compiled with a counting "
                            "scalar); used = min(SURVEY 8(d) figure, every counted formulation)",
            "flops_per_unit_counted": flops_counted,
            "executed": executed_flops(wl, units_per_launch, kernel_ms, peak_sust, attempted),
            "hbm": {"algorithmic_bytes_per_unit": bytes_unit, "achieved_gbs": gbs, "peak_gbs": hbm, "frac": (gbs / hbm) if hbm else None}}


def run_sharded(args):
    """Strong-scaling workloads through lowthrustopt_b200.sharded (results delivered to the solver rank: peer stores, or --gather nccl)."""
    import torch
    import torch.distributed as dist
    from lowthrustopt_b200 import capi, sharded, synthetic as S

    world, rank, local = dist_setup()
    dev = torch.device("cuda", local)
    h = capi.Handle(local)
    wl = args.workload
    nd = 12
    if wl == "indirect12_1m":
        n_units = args.n_seg or (1 << 20); n_nodes = 2; passes_def = 0
        b = S.indirect_batch(n_units, ndim=nd, seed=20180002) if rank == 0 else None
        if rank == 0:
            XC = np.zeros((n_units, 2, nd)); XC[:, 0] = b["x0"]
            tt = np.stack([b["t0"], b["t1"]], axis=1)
            tl = 0.05
    else:
        n_units = args.n_seg or 1024; n_nodes = 201; passes_def = 22
        if rank == 0:
            c = S.continuation_batch(n_traj=n_units, n_seg_per_traj=n_nodes - 1, ndim=nd)
            XC, tt, tl = c["XC_all"], c["t_TU"], c["thrustLimit"]
    spu = n_nodes - 1
    n_seg = n_units * spu
    peer = args.gather == "peer"
    if peer:
        sh = sharded.PeerIndirect(h, n_units, n_nodes, nd, dev)
    else:
        sh = sharded.ShardedIndirect(h, n_units, n_nodes, nd, dev, n_chunks=args.chunks)
    p = capi.indirect_params(p=1.0, rho=1.0, thrustLimit=0.05)
    N_ALPHA = 20                                               # lineSearch: alpha_all = LinRange(0.1, 1, 20) (:227)
    sh_ls = upd = alphas = None
    if passes_def:
        # the 20 trial trajectories of every line search form ONE batched pass (n_traj = 20 x 1024) whose merit values
        # sum(defect^2) are reduced on the device; the trial update is a fixed synthetic direction (Newton steps are host-side)
        sh_ls = (sharded.PeerIndirect(h, n_units * N_ALPHA, n_nodes, nd, dev) if peer else
                 sharded.ShardedIndirect(h, n_units * N_ALPHA, n_nodes, nd, dev, n_chunks=1))
        upd = torch.empty((n_units, n_nodes, nd), dtype=torch.float64, device=dev)
        if rank == 0:
            upd.copy_(torch.from_numpy(1e-4 * np.random.default_rng(20180004).standard_normal((n_units, n_nodes, nd))))
        sharded._bcast(upd, 0, None)
        alphas = torch.linspace(0.1, 1.0, N_ALPHA, dtype=torch.float64, device=dev)
    pin_in = pin_out = None
    if rank == 0:
        pin_in = {"XC": capi.PinnedBuffer(XC.shape), "t": capi.PinnedBuffer(tt.shape)}
        pin_in["XC"].array[...] = XC; pin_in["t"].array[...] = tt
        pin_out = {"defect": torch.empty((n_units, spu, nd), dtype=torch.float64).pin_memory(),
                   "phi": torch.empty((n_units, spu, nd, nd), dtype=torch.float64).pin_memory(),
                   "status": torch.empty((n_units, spu), dtype=torch.int32).pin_memory()}
        sh.load(pin_in["XC"].array, pin_in["t"].array, tl, 1.0)
    else:
        sh.load()
    if sh_ls is not None:
        sh_ls.t.view(N_ALPHA, n_units, n_nodes).copy_(sh.t.unsqueeze(0).expand(N_ALPHA, -1, -1))
        sh_ls.tl.view(N_ALPHA, n_units).copy_(sh.tl.unsqueeze(0).expand(N_ALPHA, -1)); sh_ls.rho.fill_(1.0)

    def step_peer():
        out = sh.run(p, jac=True, wait=not passes_def)                        # jacobianCalc (:290)
        if passes_def:
            sh.run(p, jac=False, wait=False)                                  # SOC defectCalc (:197)
            torch.add(sh.XC.unsqueeze(0), alphas.view(-1, 1, 1, 1) * upd.unsqueeze(0), out=sh_ls.XC.view(N_ALPHA, n_units, n_nodes, nd))
            sh_ls.run(p, mode="sumsq", wait=False)                            # lineSearch, 20 alphas in one pass (:232-241)
            sh.run(p, jac=False, wait=True)                                   # check defectCalc (:328); flags are monotone: all earlier passes have landed too
            sh_ls.pg_ls.wait_all()
        h.sync()
        return out

    def step():
        """One Newton iteration's worth of hot-path calls (multiShoot_CRTBP_indirect.jl:290-328)."""
        if peer:
            return step_peer()
        out, plan = sh.run(p, jac=True, sync=False)                           # jacobianCalc (:290)
        if passes_def:
            sh.run(p, jac=False, sync=False)                                  # SOC defectCalc (:197)
            torch.add(sh.XC.unsqueeze(0), alphas.view(-1, 1, 1, 1) * upd.unsqueeze(0), out=sh_ls.XC.view(N_ALPHA, n_units, n_nodes, nd))
            sh_ls.run(p, mode="sumsq", sync=False)                            # lineSearch, 20 alphas in one pass (:232-241)
            sh.run(p, jac=False, sync=False)                                  # check defectCalc (:328)
            sh_ls.finish()
        sh.finish()
        return out

    host_call = None
    if world == 1 and not passes_def:
        # one GPU: the user's call is the blocking host-buffer C-ABI entry point itself (chunked H2D -> kernel -> D2H pipeline)
        hb_in = {k: capi.PinnedBuffer(v.shape) for k, v in (("x0", b["x0"]), ("t0", b["t0"]), ("t1", b["t1"]))}
        for k in hb_in:
            hb_in[k].array[...] = b[k]
        hb_out = {"defect": pin_out["defect"].numpy().reshape(n_seg, nd), "status": pin_out["status"].numpy().reshape(n_seg),
                  "nsteps": capi.PinnedBuffer((n_seg, 2), np.int32), "phi": pin_out["phi"].numpy().reshape(n_seg, nd, nd)}
        hb_keep = hb_out["nsteps"]
        hb_out["nsteps"] = hb_keep.array

        def host_call():
            r = h.indirect(hb_in["x0"].array, hb_in["t0"].array, hb_in["t1"].array, params=p, jac=True, out=hb_out)
            return float(r["defect"][0, 0])

    def step_e2e():
        if host_call is not None:
            return host_call()
        if rank == 0:
            sh.load(pin_in["XC"].array, pin_in["t"].array, tl, 1.0)
        else:
            sh.load()
        out = step()
        r = 0.0
        if rank == 0:
            for k in pin_out:
                pin_out[k].copy_(out[k], non_blocking=True)
            torch.cuda.synchronize()
            r = float(pin_out["defect"][0, 0, 0])
        if peer and world > 1:
            dist.barrier()                                    # the solver rank has consumed the arrays: peers may overwrite them
        return r

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local); sampler.start(); time.sleep(0.3)
    l0 = h.launches
    if not peer:
        sh.run_jac.timing = []
    stream = sh.stream
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        out = step()
    e1.record(stream)
    barrier()
    launches = h.launches - l0
    t_total = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_total, op=dist.ReduceOp.MAX)
    ms_per_step = float(t_total.item()) / args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)
    if peer:
        # the dominant kernel alone: this rank's STM launch into its own (local) scratch, CUDA events on the library stream
        u0, u1 = sh.pg.slab()
        cnt = u1 - u0
        sc = {k: torch.empty((cnt,) + tuple(sp), dtype=dt, device=dev) for k, (sp, dt) in sh.spec_jac.items()}
        ka, kb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 3
        for i in range(reps + 1):
            if i == 1:
                ka.record(stream)
            h.indirect_dev(p, cnt * spu, n_nodes, nd, sh.XC[u0].data_ptr(), sh.t[u0].data_ptr(), None, None, sh.tl[u0:].data_ptr(),
                           sh.rho[u0:].data_ptr(), sc["defect"].data_ptr(), sc["status"].data_ptr(), sc["nsteps"].data_ptr(), sc["phi"].data_ptr())
        kb.record(stream); h.sync()
        kernel_ms = ka.elapsed_time(kb) / reps; units_per_launch = cnt * spu
        nst = sc["nsteps"].cpu().numpy().reshape(-1, 2)
    else:
        kt = [(a.elapsed_time(b), cnt) for a, b, cnt in sh.run_jac.timing]
        sh.run_jac.timing = None
        kernel_ms = float(np.mean([x[0] for x in kt])); units_per_launch = int(np.mean([x[1] for x in kt])) * spu
        nst = out["nsteps"].cpu().numpy().reshape(-1, 2)
    attempted = float(nst[:, 1].mean()); accepted = float(nst[:, 0].mean())
    passes = 1 + passes_def
    value = n_seg * passes / (ms_per_step * 1e-3)
    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    t_e2e = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    barrier()
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    clocks = sampler.stop()
    roof = fp64_roofline(h, FLOPS_PER_STEP_INDIRECT[nd] * attempted, units_per_launch, kernel_ms, BYTES_PER_SEG[nd], "indirect12",
                         FLOPS_COUNTED[nd] * attempted, attempted)
    roof["attempted_steps_per_segment"] = attempted; roof["accepted_steps_per_segment"] = accepted
    roof["kernel"] = "k_indirect_cw (the STM pass); launches of %d segments" % units_per_launch
    gathered = n_seg * (nd * 8 + nd * nd * 8 + 12) + (2 * n_seg * (nd * 8 + 12) + n_units * N_ALPHA * 12 if passes_def else 0)
    line = {"metric": "segment-propagations/s (fp64 state+STM)", "value": value, "unit": "segment-propagations/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(wl, n_seg, world, args.gather), "clocks": clocks,
            "passes_per_step": {"stm": 1, "defect_only": passes_def},
            "collective": ({"kind": "none: kernels store their slab into the solver rank's HBM over NVLink peer memory (CUDA IPC), "
                                    "stream-ordered completion flags", "bytes_into_solver_rank_per_step": int(gathered * (world - 1) // world)}
                           if peer else
                           {"kind": "ncclAllGather (torch.distributed all_gather_into_tensor)", "chunks": args.chunks,
                            "bytes_gathered_per_rank_per_step": int(gathered)}),
            "e2e": {"value": n_seg * passes * args.steps / float(t_e2e.item()), "unit": "segment-propagations/s",
                    "h2d_bytes_per_step": int(n_seg * (nd + 2) * 8 if host_call is not None else n_units * n_nodes * (nd + 1) * 8),
                    "d2h_bytes_per_step": int(n_seg * (nd * 8 + nd * nd * 8 + 4 + (8 if host_call is not None else 0))),
                    "timing": ("host wall clock around the blocking lto_indirect_defect_jac call, pinned host buffers" if host_call is not None else
                               "host wall clock on the solver rank: pinned host inputs -> H2D -> broadcast -> sharded passes + delivery to the solver rank -> "
                               "D2H of defect/STM/status into pinned memory; max over ranks")},
            "gpu_launches": int(launches), "roofline": roof, "kernel": args.kernel}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if peer:
        for o in (sh, sh_ls):
            if o is not None:
                o.pg.close()
                if o.pg_ls is not None:
                    o.pg_ls.close()
    h.close()
    if world > 1:
        dist.destroy_process_group()


def allgather_leg(args, h, dev, wl, n_seg, world, rank, batch, p):
    """The same weak-scaling batch (n_seg segments per GPU) with every rank's defects + Jacobian/STM blocks all-gathered
    so the solver rank holds the full set (north_star); chunked so the NCCL all-gather overlaps the next chunk's kernel."""
    import torch
    import torch.distributed as dist
    from lowthrustopt_b200 import sharded
    total = n_seg * world
    if wl.startswith("direct"):
        ns = 7 if wl.startswith("direct7") else 6
        sh = sharded.ShardedDirect(h, total, ns, dev, n_chunks=args.chunks)
        # every rank contributes its own batch: all-gather the inputs once (untimed set-up), globally ordered like the shard plan
        for k, dst in sh.inp.items():
            loc = torch.from_numpy(np.ascontiguousarray(batch[k])).to(dev)
            dist.all_gather_into_tensor(dst, loc)
        per_unit = ns * 8 + 8 + 4 + ns * 2 * (ns + 3) * 8
    else:
        nd = 12 if wl == "indirect12" else 14
        sh = sharded.ShardedIndirect(h, total, 2, nd, dev, n_chunks=args.chunks)
        XC = np.zeros((n_seg, 2, nd)); XC[:, 0] = batch["x0"]
        dist.all_gather_into_tensor(sh.XC, torch.from_numpy(XC).to(dev))
        dist.all_gather_into_tensor(sh.t, torch.from_numpy(np.stack([batch["t0"], batch["t1"]], axis=1)).to(dev))
        sh.tl.fill_(0.05); sh.rho.fill_(1.0)
        per_unit = nd * 8 + 12 + nd * nd * 8
    for _ in range(3):
        sh.run(p, jac=True)
    torch.cuda.synchronize(); dist.barrier()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(sh.stream)
    for _ in range(args.steps):
        sh.run(p, jac=True)
    e1.record(sh.stream)
    torch.cuda.synchronize(); dist.barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / args.steps
    res = {"value": total / (ms * 1e-3), "unit": "segment-propagations/s", "ms_per_step": ms, "chunks": args.chunks,
           "bytes_received_per_rank_per_step": int(per_unit * n_seg * (world - 1)),
           "what": "same batch, outputs of all ranks all-gathered (NCCL over NVLink) into every rank's HBM, max over ranks"}
    # ---- fused alternative: every rank's kernel stores its slab straight into the solver rank's HBM (NVLink peer memory)
    if wl.startswith("direct"):
        pe = sharded.PeerDirect(h, total, ns, dev)
        for k in pe.inp:
            pe.inp[k].copy_(sh.inp[k])
    else:
        pe = sharded.PeerIndirect(h, total, 2, nd, dev)
        pe.XC.copy_(sh.XC); pe.t.copy_(sh.t); pe.tl.copy_(sh.tl); pe.rho.copy_(sh.rho)
    torch.cuda.synchronize()
    for _ in range(3):
        pe.run(p, jac=True)
    h.sync(); dist.barrier()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(pe.stream)
    for _ in range(args.steps):
        out = pe.run(p, jac=True)
    e1.record(pe.stream)
    h.sync(); dist.barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms2 = float(t.item()) / args.steps
    # the gathered arrays on the solver rank must equal the all-gathered ones
    ok = torch.ones(1, dtype=torch.int32, device=dev)
    if rank == 0:
        ref, _ = sh.run(p, jac=True)
        key = "jac" if wl.startswith("direct") else "phi"
        same = torch.equal(out["defect"].reshape(-1), ref["defect"].reshape(-1)) and bool(((out[key].reshape(-1) - ref[key].reshape(-1)).abs().max() < 1e-11).item())
        ok[0] = 1 if same else 0
    else:
        sh.run(p, jac=True)
    dist.broadcast(ok, src=0)
    res["peer_gather"] = {"value": total / (ms2 * 1e-3), "unit": "segment-propagations/s", "ms_per_step": ms2,
                          "bytes_into_solver_rank_per_step": int(per_unit * n_seg * (world - 1)), "matches_allgather": bool(ok.item()),
                          "what": "same batch, one launch per rank, kernels store their slab into the solver rank's HBM over NVLink peer memory; "
                                  "timed on the library streams incl. the solver rank's wait for every rank's completion flag, max over ranks"}
    pe.pg.close()
    return res


def solve_passes(it_max):
    """Propagation passes a trajectory goes through in lto_indirect_solve_batch when it iterates it_max times: first nominal run
    + per iteration STM, SOC, check (+ 20 line-search trials from iteration 4)."""
    return 1 + sum(3 + (20 if it > 3 else 0) for it in range(1, it_max + 1))


def cpu_solve_baseline(XC, tt, n_traj, seconds):
    """The reference's solver loop (multiShoot_CRTBP_indirect.jl:254-345) on the host for the first trajectories of the same batch:
    propagation = the C++ restatement (oracle/, dual numbers, OpenMP over segments), linear step = scipy's sparse direct solve of the
    band system standing in for SuiteSparseQR."""
    import scipy.sparse as sp
    import scipy.sparse.linalg as spl
    from oracle import oracle as O
    O.build()
    nthreads = host_threads()
    ip = O.iparams(10.0, p=2.0, rho=1.0)
    N = XC.shape[1]; m = 12

    def defect(X):
        xe = O.indirect_prop(X[:-1], tt[0, :-1], tt[0, 1:], ip, nthreads=nthreads)[0]
        return xe - X[1:]

    def solve(phi, d):
        rows, cols, vals = [], [], []
        for i in range(N - 1):
            r, c = np.meshgrid(np.arange(m), np.arange(m), indexing="ij")
            rows.append((i * m + r).ravel()); cols.append((i * m + c).ravel()); vals.append(phi[i].ravel())
            rows.append(i * m + np.arange(m)); cols.append((i + 1) * m + np.arange(m)); vals.append(-np.ones(m))
        J = sp.csc_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(m * (N - 1), m * N))
        keep = np.ones(m * N, dtype=bool); keep[:6] = False; keep[-12:-6] = False
        sol = np.zeros(m * N); sol[keep] = -spl.spsolve(J[:, keep].tocsc(), d.ravel())
        return sol.reshape(N, m)

    t0 = time.perf_counter(); done = 0; props = 0
    while done < n_traj and (time.perf_counter() - t0 < seconds or done == 0):
        X = XC[done].copy(); d = defect(X); props += N - 1; it = 0
        while np.abs(d).max() > 1e-10 and it < 8:
            it += 1
            xe, phi, *_ = O.indirect_prop_jac(X[:-1], tt[0, :-1], tt[0, 1:], ip, nthreads=nthreads); props += N - 1
            upd = solve(phi, d)
            if np.abs(upd).max() < 1e-1:
                upd = upd + solve(phi, defect(X + upd)); props += N - 1
            alpha = 1.0
            if it > 3:
                al = np.linspace(0.1, 1.0, 20); er = [np.sum(defect(X + upd * a) ** 2) for a in al]; props += 20 * (N - 1)
                alpha = float(al[int(np.argmin(er))])
            X = X + upd * alpha; d = defect(X); props += N - 1
        done += 1
    dt = time.perf_counter() - t0
    return {"value": props / dt, "unit": "segment-propagations/s", "cores": nthreads, "kind": "port", "trajectories_per_s": done / dt,
            "sample": "the reference's solver loop run to convergence on the first %d trajectories of the same batch, one after the other "
                      "(propagation: C++ restatement in oracle/, dual numbers, OpenMP over the 200 segments on %d threads; linear step: scipy sparse "
                      "direct solve standing in for SuiteSparseQR), %.1f s" % (done, nthreads, dt)}


def run_solve(args):
    """BASELINE configs[4] solved END TO END on the device: lto_indirect_solve_batch = multiShoot_CRTBP_indirect's whole iteration loop
    (STM pass, banded-QR Newton update, SOC, 20-point line search, checks) for every trajectory of the batch; trajectories are sharded
    over the ranks (independent solver instances, no collective)."""
    import torch
    import torch.distributed as dist
    from lowthrustopt_b200 import capi, synthetic as S

    world, rank, local = dist_setup()
    dev = torch.device("cuda", local)
    h = capi.Handle(local)
    n_traj_total = args.n_seg or 1024
    n_nodes = 201; nd = 12; spu = n_nodes - 1
    c = S.continuation_batch(n_traj=n_traj_total, n_seg_per_traj=spu, ndim=nd)
    u0, u1 = n_traj_total * rank // world, n_traj_total * (rank + 1) // world
    XC0 = c["XC_all"][u0:u1].copy(); tt = c["t_TU"][u0:u1].copy()
    T = u1 - u0
    p = capi.indirect_params(p=2.0, thrustLimit=10.0, rho=1.0); p.max_attempts = 5000
    max_iter = 8
    pin = capi.PinnedBuffer(XC0.shape); pin_t = capi.PinnedBuffer(tt.shape); pin_t.array[...] = tt
    pin_out = {"defect": capi.PinnedBuffer((T, spu, nd)), "status_flag": capi.PinnedBuffer((T,), np.int32), "iters": capi.PinnedBuffer((T,), np.int32),
               "er": capi.PinnedBuffer((T,))}
    outs = {k: b.array for k, b in pin_out.items()}

    def step():
        pin.array[...] = XC0                                     # the solver works in place on the caller's XC_all (pinned, like every output)
        return h.indirect_solve_batch(pin.array, pin_t.array, params=p, max_iter=max_iter, inplace=True, out=outs)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        r = step()
    barrier()
    sampler = ClockSampler(local); sampler.start(); time.sleep(0.3)
    l0 = h.launches
    dev_ms = 0.0
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r = step()
        dev_ms += h.last_kernel_ms
    wall = time.perf_counter() - t0
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, r)
    launches = h.launches - l0
    tm = torch.tensor([dev_ms, wall * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    ms_per_step = float(tm[0].item()) / args.steps; wall_ms = float(tm[1].item()) / args.steps
    it_max = int(r["iters"].max())
    its = torch.tensor([it_max], dtype=torch.int64, device=dev); conv = torch.tensor([int((r["status_flag"] == 0).sum())], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(its, op=dist.ReduceOp.MAX); dist.all_reduce(conv)
    passes = solve_passes(it_max)
    # a trajectory is propagated only while it iterates (the solver compacts its work set): count what was actually propagated
    segs = torch.tensor([float(spu * sum(solve_passes(int(k)) for k in r["iters"]))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(segs)
    total_props = float(segs.item())
    clocks = sampler.stop()
    # ---- the two dominant kernels alone, device-resident (CUDA events on the library stream)
    stream = torch.cuda.ExternalStream(h.stream, device=dev)
    dXC = torch.from_numpy(XC0).to(dev); dT = torch.from_numpy(tt).to(dev)
    d_def = torch.empty((T * spu, nd), dtype=torch.float64, device=dev); d_ns = torch.empty((T * spu, 2), dtype=torch.int32, device=dev)
    d_phi = torch.empty((T * spu, nd, nd), dtype=torch.float64, device=dev); d_upd = torch.empty((T, n_nodes, nd), dtype=torch.float64, device=dev)

    def timed(fn, reps=5):
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
    stm_ms = timed(lambda: h.indirect_dev(p, T * spu, n_nodes, nd, dXC.data_ptr(), dT.data_ptr(), None, None, None, None, d_def.data_ptr(), None,
                                          d_ns.data_ptr(), d_phi.data_ptr()))
    nwt_ms = timed(lambda: h.indirect_newton_dev(T, n_nodes, 0, d_phi.data_ptr(), d_def.data_ptr(), d_upd.data_ptr()))
    nst = d_ns.cpu().numpy()
    attempted = float(nst[:, 1].mean()); accepted = float(nst[:, 0].mean())
    roof = fp64_roofline(h, FLOPS_PER_STEP_INDIRECT[nd] * attempted, T * spu, stm_ms, BYTES_PER_SEG[nd], "indirect12", FLOPS_COUNTED[nd] * attempted, attempted)
    roof["attempted_steps_per_segment"] = attempted; roof["accepted_steps_per_segment"] = accepted
    roof["kernel"] = "k_indirect_cw (the STM pass of every iteration); launches of %d segments" % (T * spu)
    # Newton update: HBM-side accounting (factor rows written once, read once; Phi and defects read once; update written once)
    nwt_bytes = T * (spu * (nd * nd + nd) * 8 + n_nodes * nd * 8 + 2 * n_nodes * 12 * 26 * 8)
    line = {"metric": "segment-propagations/s (fp64 state+STM)", "value": total_props / (ms_per_step * 1e-3), "unit": "segment-propagations/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "continuation_solve",
                       "description": "BASELINE configs[4]: 1,024 trajectories x 200 segments (L2_Anderson_2 ballistic stack, costates 0.1 N(0,1), p = 2, "
                                      "thrustLimit 10 N) SOLVED to the reference's 1e-10 defect threshold by lto_indirect_solve_batch: one step = the whole "
                                      "multiShoot_CRTBP_indirect loop for all trajectories, every array resident on the device (STM pass, banded-QR Newton "
                                      "update, SOC, line search, checks; trajectories leave the work set when they stop iterating); value counts the segment propagations actually done",
                       "trajectories_total": n_traj_total, "segments_total": n_traj_total * spu, "l2": "not flushed: each pass streams more than the 126 MB L2 holds",
                       "parallelism": "whole trajectories split over %d GPU(s), independent solver instances, no collective" % world},
            "clocks": clocks, "iterations_max": int(its.item()), "trajectories_converged": int(conv.item()), "passes_of_the_longest_trajectory": passes,
            "trajectories_per_s": n_traj_total / (wall_ms * 1e-3),
            "e2e": {"value": total_props / (wall_ms * 1e-3), "unit": "segment-propagations/s", "ms_per_step": wall_ms,
                    "h2d_bytes_per_step": int(XC0.nbytes + tt.nbytes), "d2h_bytes_per_step": int(XC0.nbytes + T * spu * nd * 8 + T * 16),
                    "timing": "host wall clock around the blocking lto_indirect_solve_batch call (pinned XC_all in, converged XC_all + defects + flags out), max over ranks"},
            "gpu_launches": int(launches), "roofline": roof,
            "newton_update": {"kernel": "k_indirect_newton<12>: banded Householder QR + back substitution, one warp per trajectory", "ms": nwt_ms,
                              "trajectories": T, "nodes": n_nodes, "hbm_bytes": int(nwt_bytes), "hbm_gbs": nwt_bytes / (nwt_ms * 1e-3) / 1e9,
                              "bound": "latency: a dependent chain of 12 reflections per node, %d warps per SM" % max(1, T // 148)},
            "stm_pass_ms": stm_ms, "kernel": args.kernel}
    if rank == 0 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_solve_baseline(c["XC_all"], c["t_TU"], min(512, n_traj_total), args.cpu_seconds)
    if rank == 0:
        print(json.dumps(line), flush=True)
    h.close()
    if world > 1:
        dist.destroy_process_group()


def run_ours(args):
    import torch
    import torch.distributed as dist
    from lowthrustopt_b200 import capi

    if args.workload in SHARDED:
        return run_sharded(args)
    if args.workload == "continuation_solve":
        return run_solve(args)

    world, rank, local = dist_setup()
    dev = torch.device("cuda", local)
    h = capi.Handle(local)
    stream = torch.cuda.ExternalStream(h.stream, device=dev)
    kern = {"auto": capi.LTO_KERNEL_AUTO, "generic": capi.LTO_KERNEL_GENERIC, "fast": capi.LTO_KERNEL_FAST}[args.kernel]

    wl = args.workload
    direct = wl.startswith("direct")
    n_seg = args.n_seg or (65536 if direct else 131072)
    batch = make_batch(wl, n_seg, rank)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    numa_old, numa_note = numa_bind(local)                                # until the pinned buffers below exist

    if direct:
        ns = 7 if wl.startswith("direct7") else 6
        nv = 2 * (ns + 3)
        p = capi.direct_params(mode=capi.LTO_ADAPTIVE if wl.endswith("adaptive") else capi.LTO_FIXED, tol=1e-13, kernel=kern)
        din = {k: torch.from_numpy(v).to(dev) for k, v in batch.items()}
        d_def = torch.empty((n_seg, ns), dtype=torch.float64, device=dev)
        d_err = torch.empty(n_seg, dtype=torch.float64, device=dev)
        d_st = torch.empty(n_seg, dtype=torch.int32, device=dev)
        d_jac = torch.empty((n_seg, nv, ns), dtype=torch.float64, device=dev)

        def step_dev():
            h.direct_dev(p, n_seg, 0, ns, 10, din["Xa"].data_ptr(), din["Xb"].data_ptr(), din["ua"].data_ptr(), din["ub"].data_ptr(),
                         din["ta"].data_ptr(), din["tb"].data_ptr(), d_def.data_ptr(), d_err.data_ptr(), d_st.data_ptr(), d_jac.data_ptr())
        # e2e: pinned host buffers through the host-pointer C ABI
        pin_in = {k: capi.PinnedBuffer(v.shape) for k, v in batch.items()}
        for k, v in batch.items():
            pin_in[k].array[...] = v
        pin_out = {"defect": capi.PinnedBuffer((n_seg, ns)), "errors": capi.PinnedBuffer((n_seg,)),
                   "status": capi.PinnedBuffer((n_seg,), np.int32), "jac": capi.PinnedBuffer((n_seg, nv, ns))}
        out_arrays = {k: b.array for k, b in pin_out.items()}
        a_in = {k: b.array for k, b in pin_in.items()}

        def step_e2e():
            r = h.direct(a_in["Xa"], a_in["Xb"], a_in["ua"], a_in["ub"], a_in["ta"], a_in["tb"], nsteps=10, params=p, jac=True, out=out_arrays)
            return float(r["defect"][0, 0])
        h2d = sum(v.nbytes for v in batch.values())
        d2h = sum(b.array.nbytes for b in pin_out.values())
        flops_unit = FLOPS_PER_SEG["direct7" if ns == 7 else "direct6"]
        flops_counted = FLOPS_COUNTED["direct7" if ns == 7 else "direct6"]
        bytes_unit = BYTES_PER_SEG["direct7" if ns == 7 else "direct6"]
        attempted = None
    else:
        nd = 12 if wl == "indirect12" else 14
        p = capi.indirect_params(p=1.0, rho=1.0, thrustLimit=0.05, kernel=kern,
                                 err_norm=capi.LTO_NORM_STATE_SENS if args.err_norm == "joint" else capi.LTO_NORM_STATE)
        dx0 = torch.from_numpy(batch["x0"]).to(dev); dt0 = torch.from_numpy(batch["t0"]).to(dev); dt1 = torch.from_numpy(batch["t1"]).to(dev)
        d_def = torch.empty((n_seg, nd), dtype=torch.float64, device=dev)
        d_st = torch.empty(n_seg, dtype=torch.int32, device=dev)
        d_ns = torch.empty((n_seg, 2), dtype=torch.int32, device=dev)
        d_phi = torch.empty((n_seg, nd, nd), dtype=torch.float64, device=dev)

        def step_dev():
            h.indirect_dev(p, n_seg, 0, nd, dx0.data_ptr(), dt0.data_ptr(), dt1.data_ptr(), None, None, None, d_def.data_ptr(),
                           d_st.data_ptr(), d_ns.data_ptr(), d_phi.data_ptr())
        pin_in = {k: capi.PinnedBuffer(v.shape) for k, v in batch.items()}
        for k, v in batch.items():
            pin_in[k].array[...] = v
        a_in = {k: b.array for k, b in pin_in.items()}
        pin_out = {"defect": capi.PinnedBuffer((n_seg, nd)), "status": capi.PinnedBuffer((n_seg,), np.int32),
                   "nsteps": capi.PinnedBuffer((n_seg, 2), np.int32), "phi": capi.PinnedBuffer((n_seg, nd, nd))}
        out_arrays = {k: b.array for k, b in pin_out.items()}

        def step_e2e():
            r = h.indirect(a_in["x0"], a_in["t0"], a_in["t1"], params=p, jac=True, out=out_arrays)
            return float(r["defect"][0, 0])
        h2d = sum(v.nbytes for v in batch.values())
        d2h = n_seg * (nd * 8 + 4 + 8 + nd * nd * 8)
        flops_unit = None
        flops_counted = None
        bytes_unit = BYTES_PER_SEG[nd]
        attempted = None
    numa_restore(numa_old)                                               # the CPU baseline below uses every host thread again

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up
    for _ in range(max(args.warmup, 3)):
        step_dev()
    h.sync()
    barrier()
    sampler = ClockSampler(local); sampler.start()
    time.sleep(0.3)
    # ---- device-resident timing: per-iteration event pairs on the launching stream, L2 flushed in between
    l0 = h.launches
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    with torch.cuda.stream(stream):
        for i in range(args.steps):
            flush.fill_(i & 0xFF)
            evs[i][0].record()
            step_dev()
            evs[i][1].record()
    h.sync()
    barrier()
    launches = h.launches - l0
    times = [a.elapsed_time(b) for a, b in evs]
    t_total = torch.tensor([sum(times)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_total, op=dist.ReduceOp.MAX)
    ms_per_step = float(t_total.item()) / args.steps
    value = n_seg * world / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(defect=d_def, errors=d_err, status=d_st, jac=d_jac) if direct else
                     dict(defect=d_def, status=d_st, nsteps=d_ns, phi=d_phi))
    if not direct:
        nst = d_ns.cpu().numpy()
        attempted = float(nst[:, 1].mean()); accepted = float(nst[:, 0].mean())
        flops_unit = FLOPS_PER_STEP_INDIRECT[nd] * attempted
        flops_counted = FLOPS_COUNTED[nd] * attempted
    # ---- e2e through the host-buffer C ABI
    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    chk = 0.0
    for _ in range(args.steps):
        chk += step_e2e()
    t_e2e = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    barrier()
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    e2e_value = n_seg * world * args.steps / float(t_e2e.item())
    clocks = sampler.stop()
    # ---- the same call with PAGEABLE caller memory (what a Julia / numpy caller holds; VERDICT r1 #6).  (a) inputs pageable, results in
    # the arrays the binding allocates itself -- pinned, from its pool (capi.PinnedPool; julia/lto_b200.jl `pinned_array`): the documented
    # way;  (b) results into caller-supplied pageable arrays as well: the driver stages every copy and the pipeline serialises.
    pageable = None
    if rank == 0 or world > 1:
        pg_in = {k: np.array(v, copy=True) for k, v in batch.items()}
        if direct:
            def call(out):
                return h.direct(pg_in["Xa"], pg_in["Xb"], pg_in["ua"], pg_in["ub"], pg_in["ta"], pg_in["tb"], nsteps=10, params=p, jac=True, out=out)
            pg_out = {"defect": np.empty((n_seg, ns)), "errors": np.empty(n_seg), "status": np.empty(n_seg, dtype=np.int32), "jac": np.empty((n_seg, nv, ns))}
        else:
            def call(out):
                return h.indirect(pg_in["x0"], pg_in["t0"], pg_in["t1"], params=p, jac=True, out=out)
            pg_out = {"defect": np.empty((n_seg, nd)), "status": np.empty(n_seg, dtype=np.int32), "nsteps": np.empty((n_seg, 2), dtype=np.int32),
                      "phi": np.empty((n_seg, nd, nd))}
        for v in pg_out.values():
            v.fill(0)                                                   # touch the pages: no first-touch faults inside the timed region
        res = {}
        for name, out in (("pinned_results", None), ("pageable_results", pg_out)):
            r = None
            for _ in range(2):
                r = call(out)
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                r = call(out)
            tt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
            barrier()
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            res[name] = n_seg * world * args.steps / float(tt.item())
            del r
        pageable = {"inputs": "pageable numpy arrays (what a Julia / numpy caller holds)",
                    "pinned_results": {"value": res["pinned_results"], "what": "results in the arrays the binding allocates itself (pinned, pooled) -- the documented "
                                       "way, what julia/lto_b200.jl does"},
                    "pageable_results": {"value": res["pageable_results"], "what": "results copied into caller-supplied pageable arrays as well"},
                    "unit": "segment-propagations/s"}
    # ---- FP64 peak, measured in the same run on the same device (MEASURED_PEAKS.json has no FP64 figure)
    per_gpu_ms = float(np.mean(times))
    roof = fp64_roofline(h, flops_unit, n_seg, per_gpu_ms, bytes_unit, wl, flops_counted, attempted)
    if wl.endswith("adaptive"):
        # the direct entry points do not return step counts, so the algorithmic FLOPs of an ADAPTIVE pass are not known here
        roof["achieved"] = None; roof["frac"] = None; roof["flops_per_unit"] = None
        roof["note"] = "ode78 controller: steps per leg vary (4+ at tol 1e-13 vs the fixed grid's 9); no FLOP count is claimed for this workload"
    if attempted is not None:
        roof["attempted_steps_per_segment"] = attempted
        roof["accepted_steps_per_segment"] = accepted
    line = {"metric": "segment-propagations/s (fp64 state+STM)", "value": value, "unit": "segment-propagations/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(wl, n_seg, world),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "segment-propagations/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "timing": "host wall clock around the blocking lto_*_defect_jac call, pinned host buffers, max over ranks",
                    "host_buffers": numa_note, "pageable": pageable},
            "gpu_launches": int(launches), "roofline": roof, "kernel": args.kernel}
    if world > 1:
        # N > 1: `value` is the rate at which results ARRIVE ON THE SOLVER RANK (north_star: defects + Jacobian blocks delivered to the
        # rank that runs the Newton step) -- every rank's kernel stores its slab into the solver rank's HBM over NVLink peer memory,
        # timed to the solver rank's last completion flag.  The figure with every rank keeping its own outputs (no delivery) and the
        # NCCL all-gather (8 x the bytes: every rank receives everything) are reported beside it.
        ag = allgather_leg(args, h, dev, wl, n_seg, world, rank, batch, p)
        pg = ag.pop("peer_gather")
        line["no_delivery"] = {"value": value, "unit": "segment-propagations/s", "ms_per_step": ms_per_step,
                               "what": "every rank keeps its own outputs: no data-path communication at all (round 1's headline)"}
        line["value"] = pg["value"]; line["ms_per_step"] = pg["ms_per_step"]
        gbs = pg["bytes_into_solver_rank_per_step"] / (pg["ms_per_step"] * 1e-3) / 1e9
        line["delivery"] = {"how": "peer stores (fused into the kernels' epilogue: TMA bulk stores / vector stores into the solver rank's mapped HBM)",
                            "bytes_into_solver_rank_per_step": pg["bytes_into_solver_rank_per_step"], "solver_rank_ingest_gbs": gbs,
                            "nvlink_ingest_nominal_gbs": 900.0,
                            "ingest_bound_ms": pg["bytes_into_solver_rank_per_step"] / 900e9 * 1e3,
                            "matches_allgather": pg["matches_allgather"], "what": pg["what"]}
        line["config"]["parallelism"] = ("segments sharded across %d GPU(s); every rank's defects + Jacobian blocks are stored into the solver rank's "
                                         "HBM over NVLink peer memory by the propagation kernels themselves; no other collective" % world)
        line["allgather_nccl"] = ag
    if rank == 0 and not args.no_cpu_baseline:
        sample = args.cpu_sample or (8192 if direct else 2048)
        line["cpu_baseline"] = cpu_baseline(wl, batch, sample, args.cpu_seconds)
    if rank == 0:
        print(json.dumps(line), flush=True)
    h.close()
    if world > 1:
        dist.destroy_process_group()


def run_single_process(args):
    """One process, N devices, host buffers: lto_init_devices splits every call into contiguous unit ranges, one worker thread and one
    H2D -> kernel -> D2H pipeline per device, each device copying its slab straight into the caller's arrays (no collective).  This is
    what `julia/lto_b200.jl` gets when LowThrustOpt is started with several GPUs visible."""
    from lowthrustopt_b200 import capi
    wl = args.workload
    direct = wl.startswith("direct")
    n_dev = args.gpus
    n_seg = (args.n_seg or (65536 if direct else 131072)) * n_dev         # weak scaling, like the multi-process default
    batch = make_batch(wl, n_seg, 0)
    res = {}
    for last, devs in ((False, [0]), (True, list(range(n_dev)))):
        h = capi.Handle(devs)
        pin_in = {k: capi.PinnedBuffer(v.shape) for k, v in batch.items()}
        for k, v in batch.items():
            pin_in[k].array[...] = v
        a_in = {k: b.array for k, b in pin_in.items()}
        if direct:
            ns = 7 if wl.startswith("direct7") else 6
            p = capi.direct_params(mode=capi.LTO_ADAPTIVE if wl.endswith("adaptive") else capi.LTO_FIXED)
            pin_out = {"defect": capi.PinnedBuffer((n_seg, ns)), "errors": capi.PinnedBuffer((n_seg,)), "status": capi.PinnedBuffer((n_seg,), np.int32),
                       "jac": capi.PinnedBuffer((n_seg, 2 * (ns + 3), ns))}
            out = {k: b.array for k, b in pin_out.items()}
            call = lambda: h.direct(a_in["Xa"], a_in["Xb"], a_in["ua"], a_in["ub"], a_in["ta"], a_in["tb"], nsteps=10, params=p, jac=True, out=out)
        else:
            nd = 12 if wl == "indirect12" else 14
            p = capi.indirect_params(p=1.0, rho=1.0, thrustLimit=0.05)
            pin_out = {"defect": capi.PinnedBuffer((n_seg, nd)), "status": capi.PinnedBuffer((n_seg,), np.int32), "nsteps": capi.PinnedBuffer((n_seg, 2), np.int32),
                       "phi": capi.PinnedBuffer((n_seg, nd, nd))}
            out = {k: b.array for k, b in pin_out.items()}
            call = lambda: h.indirect(a_in["x0"], a_in["t0"], a_in["t1"], params=p, jac=True, out=out)
        for _ in range(max(args.warmup, 3)):
            call()
        l0 = h.launches
        t0 = time.perf_counter()
        for _ in range(args.steps):
            r = call()
        dt = time.perf_counter() - t0
        if args.dump_outputs and last:
            dump_outputs(args.dump_outputs, r)
        res[len(devs)] = {"value": n_seg * args.steps / dt, "ms_per_step": 1e3 * dt / args.steps, "launches": int(h.launches - l0),
                          "checksum": float(np.asarray(r["defect"]).sum())}
        h.close()
        for b in list(pin_in.values()) + list(pin_out.values()):
            b.free()
    one, many = res[1], res[n_dev]
    line = {"metric": "segment-propagations/s (fp64 state+STM)", "value": many["value"], "unit": "segment-propagations/s", "n_gpus": n_dev,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": many["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl, "segments_total": n_seg, "parallelism": "ONE process, %d devices through lto_init_devices (host buffers, a worker thread "
                       "and a copy/compute pipeline per device)" % n_dev},
            "e2e": {"value": many["value"], "unit": "segment-propagations/s", "timing": "host wall clock around the blocking host-buffer call, pinned buffers"},
            "same_batch_on_one_device": one, "speedup_over_one_device": many["value"] / one["value"],
            "identical_results": one["checksum"] == many["checksum"], "gpu_launches": many["launches"], "single_process": True}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    elif a.single_process:
        run_single_process(a)
    else:
        run_ours(a)
