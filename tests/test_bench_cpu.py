"""CPU: the parts of bench.py that run without a GPU -- the reference arm (`--impl reference`, the reference ALGORITHM restated in
oracle/ timed on the host cores) prints one well-formed JSON line, and the bookkeeping of the batched-solver workload."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.normpath(os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, ROOT)


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-sample", "256"],
                         capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert out.returncode == 0, out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "segment-propagations/s" and line["value"] > 0
    assert line["config"]["workload"] == "direct7_fixed" and line["higher_is_better"] is True and line["dtype"] == "f64"
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0 and line["gpu_launches"] == 0


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, cwd=ROOT, env=env, timeout=600)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_samples_the_same_units_of_every_array(tmp_path):
    """--dump-outputs: float64 files, under 64 MB in all; a larger output (the default workload's 65,536 x 20 x 7 Jacobian blocks) keeps
    the same seeded sample of segments in every array, so two runs write identical files."""
    import bench
    n = 65536
    rng = np.random.default_rng(0)
    out = {"defect": rng.standard_normal((n, 7)), "status": np.arange(n, dtype=np.int32), "jac": rng.standard_normal((n, 20, 7))}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), out)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["defect.npy", "jac.npy", "sample_index.npy", "status.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 << 20
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    assert all(a.dtype == np.float64 for a in got.values())
    keep = got["sample_index"].astype(np.int64)
    assert len(keep) > n // 2 and np.all(np.diff(keep) > 0)
    assert np.array_equal(got["status"], keep) and np.array_equal(got["defect"], out["defect"][keep]) and np.array_equal(got["jac"], out["jac"][keep])
    assert all(np.array_equal(got[f[:-4]], np.load(tmp_path / "b" / f)) for f in files)
    small = tmp_path / "small"
    bench.dump_outputs(str(small), {"defect": out["defect"][:10]})
    assert os.listdir(small) == ["defect.npy"] and np.array_equal(np.load(small / "defect.npy"), out["defect"][:10])


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert out.returncode == 2 and "--steps must be at least 1" in out.stderr


def test_solver_workload_bookkeeping():
    import bench
    from lowthrustopt_b200 import synthetic as S
    assert bench.solve_passes(0) == 1 and bench.solve_passes(3) == 10 and bench.solve_passes(4) == 33      # 20 line-search trials from iteration 4
    c = S.continuation_batch(n_traj=2, n_seg_per_traj=40, ndim=12)
    XC = c["XC_all"].copy(); XC[:, :, 6:] *= 0.1
    cb = bench.cpu_solve_baseline(XC, c["t_TU"], 2, 0.0)
    assert cb["kind"] == "port" and cb["value"] > 0 and cb["trajectories_per_s"] > 0 and "first 1 trajectories" in cb["sample"]
