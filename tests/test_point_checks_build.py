"""CPU: the sm_100a build of the point-check kernels.  k_check_points and the checked ingestion kernel must not spill at
their launch bounds (k_check_points: 128 threads, 3 blocks per SM, i.e. 3 resident warps per scheduler), on every curve:
the chains are throughput-bound field products, and local-memory traffic would compete with them."""
import os
import re
import shutil

import pytest

from montgomery_b200 import build

CURVE_TAGS = {"bls12-377": "Fp377", "pallas": "FpPallas", "ed-on-bls12-377": "Fr377", "bls12-381": "Fp381"}


@pytest.mark.skipif(shutil.which(build._nvcc()) is None and not os.path.exists(build._nvcc()), reason="no nvcc")
def test_point_check_kernels_do_not_spill():
    build.build()                                          # -Xptxas -v; the log of the last compile of msm.cu
    log = open(os.path.join(build.OBJDIR, "msm.cu.ptxas.log")).read()
    entries = re.findall(r"Compiling entry function '(_ZN3mgb[^']*)' for 'sm_100a'\n.*?\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads\n"
                         r"ptxas info\s*: Used (\d+) registers", log)
    found = {}
    for name, _stack, stores, loads, regs in entries:
        for kernel in ("k_check_points", "k_set_points"):
            if ("%d%s" % (len(kernel), kernel)) not in name:
                continue
            if kernel == "k_set_points" and "Lb1E" not in name:       # the checked variant: template flag true
                continue
            for label, tag in CURVE_TAGS.items():
                if "%d%s" % (len(tag), tag) in name:
                    found[(kernel, label)] = (int(stores), int(loads), int(regs))
    assert len(found) == 8, sorted(found)
    for (kernel, label), (stores, loads, regs) in found.items():
        assert stores == 0 and loads == 0, (kernel, label, stores, loads)
        if kernel == "k_check_points":
            assert regs * 128 * 3 <= 65536, (label, regs)      # 3 blocks of 128 threads fit the register file
