"""Per-warp phase clocks of the direct throughput kernels K1 / K2 (k_direct_cw, lto_direct_cw.cu).

    python tools/k1_phase_clocks.py [--workload direct7_fixed|direct6_fixed|direct7_adaptive] [--n-seg 65536] [--lib PATH]

Builds the -DLTO_K1_PROF variant of the library into tools/experiments/lib/liblto_k1prof.so (the product library is never
built with the switch), runs the bench batch a few times and prints, per role, where a warp's cycles of the last launch went:
  work   inside col_step (column warps) / x_step and the record hand-over (state warps)
  bar    waiting on the ring's mbarriers (columns: `full`, state: `empty`)
  pace   in the per-step pace barrier `bar.sync 3` (column warps)
  store  tile-end staging of the Jacobian blocks and its bulk-store barriers (column warps)
  other  the rest of the warp's lifetime (leg loads, defects, loop overhead)
Warp w sits on SM sub-partition w % 4; warps 2 and 3 are the state warps.  --lib runs an already built profiled library
instead (e.g. one of another commit).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.normpath(os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, ROOT)

K1P = ["work", "bar", "pace", "store", "total", "steps"]
MAX_BLOCKS, MAX_WARPS = 1024, 16


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="direct7_fixed", choices=["direct7_fixed", "direct6_fixed", "direct7_adaptive", "direct6_adaptive"])
    ap.add_argument("--n-seg", type=int, default=65536)
    ap.add_argument("--lib", default=None, help="profiled library to run (default: build it from this tree)")
    ap.add_argument("--json", default=None, help="also write the summary as JSON here")
    args = ap.parse_args()

    if args.lib is None:
        from lowthrustopt_b200 import build as B
        out = os.path.join(B.EXPERIMENTS, "lib")
        args.lib = B.build_lib(lib=os.path.join(out, "liblto_k1prof.so"), obj_dir=os.path.join(out, "_build_k1prof"),
                               extra_flags=["-DLTO_K1_PROF"])
    os.environ["LTO_B200_LIB"] = os.path.abspath(args.lib)
    import numpy as np
    import torch
    from lowthrustopt_b200 import capi, synthetic as S
    L = capi.lib()
    if not hasattr(L, "lto_k1_prof_read"):
        raise SystemExit("%s was not built with -DLTO_K1_PROF" % args.lib)

    ns = 7 if args.workload.startswith("direct7") else 6
    nv = 2 * (ns + 3)
    n = args.n_seg
    mode = capi.LTO_ADAPTIVE if args.workload.endswith("adaptive") else capi.LTO_FIXED
    dev = torch.device("cuda", 0)
    h = capi.Handle(0)
    b = S.direct_batch(n, nstate=ns)
    p = capi.direct_params(mode=mode, tol=1e-13)
    d = {k: torch.from_numpy(v).to(dev) for k, v in b.items()}
    d_def = torch.empty((n, ns), dtype=torch.float64, device=dev)
    d_err = torch.empty(n, dtype=torch.float64, device=dev)
    d_st = torch.empty(n, dtype=torch.int32, device=dev)
    d_jac = torch.empty((n, nv, ns), dtype=torch.float64, device=dev)
    st = torch.cuda.ExternalStream(h.stream, device=dev)
    times = []
    for _ in range(5):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(st):
            e0.record()
            h.direct_dev(p, n, 0, ns, 10, d["Xa"].data_ptr(), d["Xb"].data_ptr(), d["ua"].data_ptr(), d["ub"].data_ptr(),
                         d["ta"].data_ptr(), d["tb"].data_ptr(), d_def.data_ptr(), d_err.data_ptr(), d_st.data_ptr(), d_jac.data_ptr())
            e1.record()
        h.sync()
        times.append(e0.elapsed_time(e1))
    words = MAX_BLOCKS * MAX_WARPS * len(K1P)
    buf = (C.c_ulonglong * words)()
    rc = L.lto_k1_prof_read(buf, words)
    if rc != 0:
        raise SystemExit("lto_k1_prof_read failed: %d" % rc)
    w = np.frombuffer(buf, dtype=np.uint64).astype(np.float64).reshape(MAX_BLOCKS, MAX_WARPS, len(K1P))
    nw = 2 + ns + 3
    grid = int((w[:, 0, 4] > 0).sum())
    w = w[:grid, :nw]

    props = torch.cuda.get_device_properties(0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    print("device: %s  (nvidia-smi: %s)" % (props.name, q))
    print("library: %s" % args.lib)
    print("%s, %d segments: kernel incl. launch %.3f ms (median of %d, profiled build); grid %d" % (
        args.workload, n, float(np.median(times)), len(times), grid))
    print("%-22s %9s %7s %6s %6s %6s %6s %6s %10s" % ("role (warp: sub-part.)", "cycles", "steps", "work", "bar", "pace", "store", "other",
                                                    "work/step"))
    out = {"workload": args.workload, "n_seg": n, "device": props.name, "nvidia_smi": q, "ms_median": float(np.median(times)), "roles": {}}
    for wi in range(nw):
        c = w[:, wi].mean(axis=0)
        tot = c[4]
        other = tot - c[0] - c[1] - c[2] - c[3]
        role = ("state t%d" % (wi - 2)) if wi in (2, 3) else ("col %d" % (wi if wi < 2 else wi - 2))
        label = "%s (w%d: sp%d)" % (role, wi, wi % 4)
        pct = [100 * x / tot for x in (c[0], c[1], c[2], c[3], other)]
        print("%-22s %9.0f %7.0f %5.1f%% %5.1f%% %5.1f%% %5.1f%% %5.1f%% %10.0f" % ((label, tot, c[5]) + tuple(pct) + (c[0] / max(c[5], 1),)))
        out["roles"][label] = {"cycles": tot, "steps": c[5], "work": c[0], "bar": c[1], "pace": c[2], "store": c[3], "other": other}
    cols = [wi for wi in range(nw) if wi not in (2, 3)]
    cw = w[:, cols].mean(axis=(0, 1))
    print("all column warps: work %.1f%%  bar %.1f%%  pace %.1f%%  store %.1f%%; %.0f cycles of work per column step" % (
        100 * cw[0] / cw[4], 100 * cw[1] / cw[4], 100 * cw[2] / cw[4], 100 * cw[3] / cw[4], cw[0] / cw[5]))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
