"""The grid kernel's time loop keeps its per-thread state out of local memory (CPU only: ptxas's own report).

The headline instantiation runs 1024 threads at a 64-register cap with 208 KB of dynamic shared memory, so a stack
slot is an L2 round trip on the critical path of a latency-bound step.  Compiles csrc/sv_grid.cu with -Xptxas -v
(the library's flags) and checks the stack frame and spill bytes of the SV gradient smoother, one problem and team.
"""
import importlib.util
import os
import shutil

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (stack frame, spill stores, spill loads) in bytes, at most
LIMITS = {
    "sv_grid_kernelILi1024ELb0ENS_15SvLeverageModelELb1ELb0E": (32, 96, 112),
    "sv_grid_kernelILi1024ELb0ENS_15SvLeverageModelELb1ELb1E": (80, 316, 492),
}


def _nvcc():
    nvcc = os.environ.get("NVCC") or shutil.which("nvcc")
    if nvcc is None and os.path.exists("/usr/local/cuda/bin/nvcc"):
        nvcc = "/usr/local/cuda/bin/nvcc"
    return nvcc


@pytest.mark.skipif(_nvcc() is None, reason="needs nvcc")
def test_headline_grid_kernel_stack_and_spills(tmp_path, monkeypatch):
    monkeypatch.setenv("NVCC", _nvcc())
    spec = importlib.util.spec_from_file_location("grid_local_memory",
                                                  os.path.join(ROOT, "tools", "grid_local_memory.py"))
    glm = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(glm)
    table = glm.ptxas_table(glm.compile_cubin(str(tmp_path / "sv_grid.cubin")))
    for key, limit in LIMITS.items():
        found = [v for name, v in table.items() if key in name]
        assert len(found) == 1, key
        _regs, stack, stores, loads = found[0]
        assert stack <= limit[0] and stores <= limit[1] and loads <= limit[2], (key, (stack, stores, loads), limit)
