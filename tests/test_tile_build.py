"""Compiler output of the tiled sweep kernel (csrc/sm_tile.cu): every k_sweep_tile instantiation keeps its registers (0 spill
bytes at the 64 registers that 1024 threads per SM leave) and runs its FAST-beam loop on the integer tensor cores
(IMMA.16832.U8.U8).  The chunk reduction re-reads %tid.x only to stop ptxas from keeping a product live across the beam loop; a
compiler that spills again fails here instead of silently slowing the sweep."""
from __future__ import annotations

import os
import re
import shutil
import subprocess

import pytest

from slam_toolbox_b200 import build as B


def test_sweep_tile_no_spills_and_imma(tmp_path):
    nvcc = os.environ.get("NVCC", "nvcc")
    if shutil.which(nvcc) is None or shutil.which("cuobjdump") is None:
        pytest.skip("CUDA toolkit not on PATH")
    obj = str(tmp_path / "sm_tile.o")
    cmd = [nvcc] + B.ARCH + B.COMMON + B.UNITS["sm_tile.cu"] + ["-Xptxas", "-v", "-c", os.path.join(B.CSRC, "sm_tile.cu"), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    # ptxas -v: "Function properties for <mangled>" followed by "... N bytes spill stores, M bytes spill loads"
    props = re.findall(r"Function properties for (\S+)\s*\n\s*\d+ bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads",
                       r.stdout + r.stderr)
    tile = [(f, int(s), int(l)) for f, s, l in props if "k_sweep_tile" in f]
    assert len(tile) == 5, props   # pitch 0 (run time), 76, 92, 116, 132
    assert all(s == 0 and l == 0 for _, s, l in tile), tile
    for f, _, _ in tile:
        sass = subprocess.run(["cuobjdump", "-sass", "-fun", f, obj], capture_output=True, text=True).stdout
        assert "IMMA.16832.U8.U8" in sass, f
