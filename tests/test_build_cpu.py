"""CPU checks of what nvcc built for sm_100a (no GPU needed): the sweep loops really are packed DPX code, and the hot
flavors do not spill.  Reads the objects and ptxas logs that opal_b200/csrc/Makefile leaves under build/."""
import glob
import os
import re
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "opal_b200", "csrc", "build")
# cuobjdump of the toolkit whose nvcc opal_b200/csrc/Makefile compiles with (NVCC ?= /usr/local/cuda/bin/nvcc), else
# from PATH; the tools below call it by name
CUOBJDUMP = os.path.join(os.path.dirname(os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")), "cuobjdump")
if not os.path.exists(CUOBJDUMP):
    CUOBJDUMP = shutil.which("cuobjdump") or CUOBJDUMP
TOOL_ENV = dict(os.environ, PATH=os.path.dirname(CUOBJDUMP) + os.pathsep + os.environ.get("PATH", ""))


def _objects():
    objs = sorted(glob.glob(os.path.join(BUILD, "kernels_R*.o")))
    if not objs or not os.path.exists(CUOBJDUMP):
        pytest.skip("no built kernel objects / cuobjdump (run __graft_entry__.build() first)")
    return objs


def test_kernel_objects_are_sm_100a_packed_dpx_code():
    obj = os.path.join(BUILD, "kernels_R17.o")
    if obj not in _objects():
        pytest.skip("R = 17 not built")
    sass = subprocess.run([CUOBJDUMP, "-sass", obj], capture_output=True, text=True, check=True).stdout
    assert "sm_100a" in sass or "SM100a" in sass or "EF_CUDA_SM100" in sass
    for mnemonic in ("VIADDMNMX.S16x2", "VIADDMNMX.S16x2.RELU", "VIMNMX3.S16x2", "VIADD.16x2", "LDS.128", "SHFL.IDX"):
        assert mnemonic in sass, mnemonic
    # the 32-bit re-run uses the scalar forms of the same instructions
    assert re.search(r"VIADDMNMX(\.RELU)? R", sass)


def test_sweep_loop_instruction_mix_matches_the_design():
    """tools/sass_loop.py on the SW score + end flavor at R = 17: 68 VIADDMNMX + 9 VIMNMX per 34 cells (4.5 integer-pipe
    instructions per cell pair) and at most a dozen other integer-pipe instructions in the loop body (DESIGN.md section 3)."""
    obj = os.path.join(BUILD, "kernels_R17.o")
    if obj not in _objects():
        pytest.skip("R = 17 not built")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "sass_loop.py"), obj, "3"], capture_output=True, text=True,
                         check=True, env=TOOL_ENV).stdout
    first = out.split("  loop ")[1]
    counts = {m.group(1): int(m.group(2)) for m in re.finditer(r"ALU\s+(\S+)\s+(\d+)", first)}
    assert counts.get("VIADDMNMX.16x2") == 68
    assert counts.get("VIMNMX3.16x2", 0) + counts.get("VIMNMX.16x2", 0) == 9
    alu = int(re.search(r"ALU=(\d+)", first).group(1))
    assert alu - 77 <= 14, out


def test_hot_flavors_do_not_spill():
    logs = sorted(glob.glob(os.path.join(BUILD, "kernels_R*.ptxas.log")))
    if not logs:
        pytest.skip("no ptxas logs")
    for log in logs:
        text = open(log).read()
        for m in re.finditer(r"Function properties for (\S+)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", text):
            name, _, stores, loads = m.group(1), int(m.group(2)), int(m.group(3)), int(m.group(4))
            if "Packed16" not in name:
                continue
            # SW flavors (0, 1, 3) never spill; the NW/HW/OV flavor capped at 170 registers may park a few words at R >= 32
            if re.search(r"ELi[013]ENS_8Packed16", name):
                assert stores == 0 and loads == 0, (log, name, stores, loads)
            else:
                assert stores <= 64, (log, name, stores)


def test_tall_global_strips_keep_their_loop_invariants_in_registers():
    """tools/sass_hot_path.py on the NW / HW / OV bulk kernel at R = 32 (three warps per partition): the hot path of a
    wavefront step holds the 128 VIADDMNMX of 32 rows, no re-derivation of the profile base address from the CTA id
    (S2UR) or of loop invariants (LEA / LOP3), and at most 258 instructions (267 before the step was tightened;
    DESIGN.md section 3, profiles/README.md)."""
    obj = os.path.join(BUILD, "kernels_R32.o")
    if obj not in _objects():
        pytest.skip("R = 32 not built")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "sass_hot_path.py"), obj, "2", "Packed16", "384"], capture_output=True,
                         text=True, check=True, env=TOOL_ENV).stdout
    loops = re.findall(r"hot path (\d+): ALU=(\d+).*\n\s+(.*)", out)
    # (the tool also lists the task loop around them, which holds the epilogue and several hundred instructions more)
    sweeps = [(int(n), int(alu), ops) for n, alu, ops in loops if "VIADDMNMX=128" in ops and int(n) < 320]
    assert len(sweeps) == 2, out  # first pass and later passes, as two loops
    for n, alu, ops in sweeps:
        assert n <= 258 and alu <= 141, out
        assert "S2UR" not in ops and "LEA" not in ops and "LOP3" not in ops, out
