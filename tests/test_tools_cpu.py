"""The SASS analysis tools behind DESIGN.md section 4 keep working on the built object (no GPU needed: cuobjdump only)."""
import os
import re
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "temp_fhe_transciphering_b200", "csrc")
OBJ = os.path.join(CSRC, "build", "cbs_kernels.o")
BR = "_ZN3cbs17k_blind_rotate_v4EPKmPmiPKdS4_"
# cuobjdump comes with the toolkit the Makefile compiles with (NVCC ?= /usr/local/cuda/bin/nvcc), which need not be on PATH
CUOBJDUMP = shutil.which("cuobjdump") or shutil.which("cuobjdump", path=os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin"))
TOOL_ENV = dict(os.environ, PATH=os.pathsep.join([os.path.dirname(CUOBJDUMP or ""), os.environ.get("PATH", "")]))

needs_obj = pytest.mark.skipif(not os.path.exists(OBJ) or CUOBJDUMP is None, reason="needs the built kernel object and cuobjdump")


@needs_obj
def test_register_file_model_of_the_blind_rotation():
    out = subprocess.run([sys.executable, os.path.join(CSRC, "tools", "sass_rf_model.py"), OBJ, BR],
                         capture_output=True, text=True, check=True, env=TOOL_ENV).stdout
    m = re.search(r"per warp-step: (\d+) instructions, (\d+) register source words", out)
    assert m, out
    instr, words = int(m.group(1)), int(m.group(2))
    # 768 steps x 2 warps of these are what bench.py's roofline.register_file is computed from (RF_WORDS_PER_WARP_STEP)
    assert 3000 < instr < 4500 and 9000 < words < 12000, out
    lb = re.search(r"register file (\d+), issue slots (\d+), FP64 pipe (\d+)", out)
    assert lb and int(lb.group(3)) == 2 * 1962, out  # 1,962 FP64 instructions per warp and step (DESIGN.md section 4)


@needs_obj
def test_loop_counter_agrees_with_the_model():
    out = subprocess.run([sys.executable, os.path.join(CSRC, "tools", "sass_loop_count.py"), OBJ, BR],
                         capture_output=True, text=True, check=True, env=TOOL_ENV).stdout
    m = re.search(r"per warp-step: (\d+) instructions, (\d+) FP64", out)
    assert m and int(m.group(2)) == 1962, out


def test_bench_constant_matches_the_model_when_the_object_is_there():
    sys.path.insert(0, ROOT)
    import bench
    assert bench.RF_WORDS_PER_WARP_STEP == 10_555
    if os.path.exists(OBJ) and CUOBJDUMP:
        out = subprocess.run([sys.executable, os.path.join(CSRC, "tools", "sass_rf_model.py"), OBJ, BR],
                             capture_output=True, text=True, check=True, env=TOOL_ENV).stdout
        words = int(re.search(r"(\d+) register source words", out).group(1))
        assert abs(words - bench.RF_WORDS_PER_WARP_STEP) <= 0.02 * bench.RF_WORDS_PER_WARP_STEP, out
