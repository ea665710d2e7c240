"""CPU test: the GPU unit-test harness (tests/gpu_units/units.cu) still compiles for sm_100a with the product's flags, so
that a change to csrc/ that breaks it is caught on a machine without a GPU (test_gpu_units.py runs it on the device)."""
import os
import re
import shutil

import pytest

from montgomery_b200 import build as b
from tests.helpers import GPU_UNITS_SRC, compile_gpu_units

pytestmark = pytest.mark.timeout(900)


def _defaults(path):
    with open(path) as fh:
        src = fh.read()
    return {k: int(v) for k, v in re.findall(r"#ifndef (MGB_EMAX|MGB_MINB)\s*\n#define \1 (\d+)", src)}


def test_harness_uses_production_tile_bounds():
    """k_batch_add is instantiated in the harness with the same MGB_EMAX / MGB_MINB defaults as in msm.cu."""
    prod = _defaults(os.path.join(b.CSRC, "msm.cu"))
    assert set(prod) == {"MGB_EMAX", "MGB_MINB"} and _defaults(GPU_UNITS_SRC) == prod


@pytest.mark.skipif(not (shutil.which(b._nvcc()) or os.path.exists(b._nvcc())), reason="nvcc not available")
def test_harness_cross_compiles_for_sm100a(tmp_path):
    log = compile_gpu_units(str(tmp_path / "units.so"))
    assert os.path.getsize(tmp_path / "units.so") > 0
    assert "error" not in log.lower()
