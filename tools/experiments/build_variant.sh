#!/bin/bash
# tools/experiments/build_variant.sh <name> [-D flags...] : tools/experiments/lib/liblto_<name>.so = the product library PLUS the measured-and-
# not-adopted layouts of the 12-dim STM kernel (lto_indirect_hc.cu, lto_indirect_wl.cu, lto_indirect_hc2.cu), selected at run time with
# LTO_K3=hc|wl|hc2 and loaded with LTO_B200_LIB=tools/experiments/lib/liblto_<name>.so.  The product library (lowthrustopt_b200/liblto_b200.so)
# never contains them.  build() of __graft_entry__.py builds liblto_k3x.so without extra flags (lowthrustopt_b200.build.build_experiments).
set -e
cd "$(dirname "$0")/../.."
python -c "import sys; from lowthrustopt_b200 import build; print(build.build_experiments(sys.argv[1], sys.argv[2:], force=True))" "$@"
