"""Register budget of the backward sweep: every backward_kernel instantiation must fit 128 registers per thread with
no spill, so that 8 CTAs of 64 threads (16 warps) stay resident per SM (DESIGN.md section 4).  Compiles
csrc/backward.cu alone for sm_100a with `-Xptxas -v`; no GPU needed."""
import os
import re
import shutil
import subprocess
import tempfile

import pytest

from conftest import ROOT

CSRC = os.path.join(ROOT, "steered-mixture-of-experts_b200", "csrc")


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    return None


@pytest.fixture(scope="module")
def ptxas_report():
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("nvcc not found")
    with tempfile.TemporaryDirectory() as tmp:
        cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-c",
               "-o", os.path.join(tmp, "backward.o"), os.path.join(CSRC, "backward.cu")]
        r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    out = {}
    for block in r.stderr.split("Compiling entry function '")[1:]:
        name = block.split("'", 1)[0]
        m = re.search(r"backward_kernelILi(\d)ELi(\d)ELb([01])ELb([01])E", name)
        if not m:
            continue
        regs = re.search(r"Used (\d+) registers", block)
        spill = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", block)
        assert regs and spill, block
        out[tuple(int(g) for g in m.groups())] = (int(regs.group(1)), int(spill.group(1)), int(spill.group(2)))
    return out


def test_every_backward_instantiation_is_compiled(ptxas_report):
    # (d, C) in {2, 3} x {1, 3}, with and without the pair counters, culled/skipping and dense
    assert sorted(ptxas_report) == sorted((d, c, n, e) for d in (2, 3) for c in (1, 3) for n in (0, 1) for e in (0, 1))


def test_backward_fits_128_registers_without_spills(ptxas_report):
    over = {k: v for k, v in ptxas_report.items() if v[0] > 128 or v[1] or v[2]}
    assert not over, f"(d, C, COUNT, DENSE) -> (registers, spill stores, spill loads): {over}"
