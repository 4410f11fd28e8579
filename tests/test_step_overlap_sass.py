"""The lean step kernels read and write global memory only after their griddepcontrol.wait.

They are launched with programmatic dependent launch (DESIGN 4.2): a step's grid may start while the grid ahead of it
on the stream still runs, so anything it loads, stores or updates atomically before the wait can see or clobber a
state the grid ahead has not finished with.  Only L2 prefetches may come first.  This reads the SASS of the built
library (runs without a GPU): every env_step_*_lean_kernel holds exactly one ACQBULK (griddepcontrol.wait), and it
comes before every global load, store, atomic and reduction, and the L2 prefetches (UBLKPF) of the prefetching
instantiations (template argument PF = true) come before it; no other kernel of the library waits on a grid ahead."""
import os
import re
import shutil
import subprocess

import pytest

from colosseum_b200 import build

MEMORY_OPS = {"LDG", "STG", "LD", "ST", "ATOM", "ATOMG", "RED", "REDG", "LDGSTS"}


def _cuobjdump():
    for cand in (shutil.which("cuobjdump"), os.path.join(os.path.dirname(build._nvcc()), "cuobjdump")):
        if cand and os.path.isfile(cand):
            return cand
    pytest.fail("cuobjdump not found next to nvcc")


def _opcodes():
    """{mangled kernel name: [opcode without modifiers, in address order]}"""
    out = subprocess.run([_cuobjdump(), "-sass", build.build_library()], capture_output=True, text=True, check=True).stdout
    ops, fn = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            fn = m.group(1)
            ops[fn] = []
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(@!?U?P\w+\s+)?([A-Z0-9_.]+)", line)
        if m and fn:
            ops[fn].append(m.group(2).split(".")[0])
    return ops


def test_lean_step_kernels_wait_before_any_global_access():
    ops = _opcodes()
    lean = {k: v for k, v in ops.items() if re.search(r"env_step_(kary|breaks)_lean_kernel", k)}
    # k-ary: 8 widths, breakpoint: K = 2, 4, 8, 16; x 2 I/O layouts x with and without the prefetch
    assert len(lean) == 48, sorted(lean)
    for name, seq in lean.items():
        assert seq.count("ACQBULK") == 1, name
        first_mem = min((i for i, op in enumerate(seq) if op in MEMORY_OPS), default=len(seq))
        assert seq.index("ACQBULK") < first_mem, (name, seq[: first_mem + 1])
        prefetching = re.search(r"lean_kernelILi\d+ELb[01]ELb([01])E", name).group(1) == "1"
        assert ("UBLKPF" in seq[: seq.index("ACQBULK")]) == prefetching, name
        assert "UBLKPF" not in seq[seq.index("ACQBULK"):], name


def test_only_lean_step_kernels_wait_on_the_grid_ahead():
    waiting = [k for k, v in _opcodes().items() if "ACQBULK" in v and not re.search(r"env_step_(kary|breaks)_lean_kernel", k)]
    assert not waiting, waiting
