"""The direct throughput kernels K1 / K2 (k_direct_cw<6|7, fixed|adaptive>) compile for sm_100a without local memory: no spills
at the 168 registers that 384 threads per CTA leave them (no GPU needed)."""
import os
import re
import shutil
import subprocess

import pytest


def test_direct_cw_kernels_have_no_local_memory(tmp_path):
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    from lowthrustopt_b200 import build
    obj = str(tmp_path / "lto_direct_cw.o")
    cmd = [build._nvcc()] + build.ARCH + build.NVCC_FLAGS + ["-I", build.INC, "-I", build.CSRC, "-c",
                                                             os.path.join(build.CSRC, "lto_direct_cw.cu"), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    usage = subprocess.run([cuobjdump, "-res-usage", obj], capture_output=True, text=True).stdout
    found = dict(re.findall(r"Function (_ZN3lto2cw11k_direct_cw\w+):\s*\n\s*(REG:.*)", usage))
    for kern in ("ILi7ELb0E", "ILi6ELb0E", "ILi7ELb1E", "ILi6ELb1E"):
        hits = [v for k, v in found.items() if kern in k]
        assert len(hits) == 1, (kern, sorted(found))
        assert "STACK:0 " in hits[0] and "LOCAL:0 " in hits[0], (kern, hits[0])
        assert int(re.search(r"REG:(\d+)", hits[0]).group(1)) <= 168, (kern, hits[0])
