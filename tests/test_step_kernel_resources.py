"""Every step kernel runs without a stack frame or local memory.

The step kernels are built from shared inlined helpers (the per-env prologue and epilogue, the server pass loop, the
tile search); a change to one of them can make ptxas spill or keep a local copy in one instantiation only.  This reads
the resource usage of the built library and fails on any step kernel with a stack frame or local memory."""
import os
import re
import shutil
import subprocess

import pytest

from colosseum_b200 import build


def _cuobjdump():
    for cand in (shutil.which("cuobjdump"), os.path.join(os.path.dirname(build._nvcc()), "cuobjdump")):
        if cand and os.path.isfile(cand):
            return cand
    pytest.fail("cuobjdump not found next to nvcc")


def test_step_kernels_have_no_stack_or_local_memory():
    lib = build.build_library()
    out = subprocess.run([_cuobjdump(), "-res-usage", lib], capture_output=True, text=True, check=True).stdout
    usage = dict(re.findall(r"Function (\S+):\s*\n\s*(REG:\d+ STACK:\d+ SHARED:\d+ LOCAL:\d+)", out))
    step = {k: v for k, v in usage.items() if "env_step" in k}
    assert len(step) >= 73, sorted(step)  # the dense, k-ary, lean, breakpoint, successor and mixed step kernels
    bad = {k: v for k, v in step.items() if not re.search(r"STACK:0 SHARED:\d+ LOCAL:0$", v)}
    assert not bad, bad
