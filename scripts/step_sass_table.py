"""Per-kernel code size of env_step.cu at a git revision and in the working tree (runs without a GPU).

    python scripts/step_sass_table.py [REV]     (REV defaults to HEAD)

Both sources are compiled with build.py's flags.  For every kernel the table lists the SASS instructions other than NOP,
the registers, the stack frame and the local memory, from `cuobjdump -sass` and `cuobjdump -res-usage`, and the change
from REV to the working tree.  A kernel whose count moves shows the change; an unchanged one shows "=".
"""
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from colosseum_b200 import build  # noqa: E402

SRC = "colosseum_b200/csrc/env_step.cu"


def compile_obj(src_path, obj_path):
    cmd = [build._nvcc()] + build.NVCC_FLAGS + ["-I", build.INCLUDE, "-I", build.CSRC, "-c", src_path, "-o", obj_path]
    return subprocess.Popen(cmd)


def kernels(obj):
    """{mangled name: (non-NOP instructions, all instructions, registers, stack, local)}"""
    res = {}
    fn = None
    for line in subprocess.run(["cuobjdump", "-res-usage", obj], capture_output=True, text=True, check=True).stdout.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            fn = m.group(1)
            continue
        m = re.match(r"\s*REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", line)
        if m and fn:
            res[fn] = tuple(int(g) for g in m.groups())
            fn = None
    counts = {}
    fn = None
    for line in subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            fn = m.group(1)
            counts[fn] = [0, 0]
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(@!?U?P\w+\s+)?([A-Z0-9_.]+)", line)
        if m and fn:
            counts[fn][1] += 1
            counts[fn][0] += m.group(2).split(".")[0] != "NOP"
    return {k: (c[0], c[1]) + res[k] for k, c in counts.items() if k in res}


def demangle(name):
    d = subprocess.run(["cu++filt", name], capture_output=True, text=True).stdout.strip()
    d = d[: d.rfind(">") + 1] if "<" in d else d.split("(")[0]  # drop the parameter list
    return re.sub(r"^void |colo::|\((int|bool)\)", "", d).replace("(float)0", "float").replace("(double)0", "double")


def main():
    rev = sys.argv[1] if len(sys.argv) > 1 else "HEAD"
    base_text = subprocess.run(["git", "-C", ROOT, "show", f"{rev}:{SRC}"], capture_output=True, text=True, check=True).stdout
    with open(os.path.join(ROOT, SRC)) as f:
        tree_lines = f.read().count("\n")
    with tempfile.TemporaryDirectory() as tmp:
        base_src = os.path.join(tmp, "env_step.cu")
        with open(base_src, "w") as f:
            f.write(base_text)
        procs = [compile_obj(base_src, os.path.join(tmp, "base.o")), compile_obj(os.path.join(ROOT, SRC), os.path.join(tmp, "tree.o"))]
        if any(p.wait() for p in procs):
            sys.exit("nvcc failed")
        base, tree = kernels(os.path.join(tmp, "base.o")), kernels(os.path.join(tmp, "tree.o"))
    rows = sorted((demangle(n), base.get(n), tree.get(n)) for n in set(base) | set(tree))
    w = max(len(r[0]) for r in rows)
    print(f"# {SRC}: {base_text.count(chr(10))} lines at {rev}, {tree_lines} in the working tree")
    print(f"# {len(base)} kernels at {rev}, {len(tree)} in the working tree; SASS instructions (NOPs included): "
          f"{sum(v[1] for v in base.values())} -> {sum(v[1] for v in tree.values())}; "
          f"non-NOP: {sum(v[0] for v in base.values())} -> {sum(v[0] for v in tree.values())}")
    print(f"# per kernel: non-NOP SASS instructions, registers, stack bytes, local bytes at {rev} -> working tree")
    print(f"{'kernel':{w}}  {'sass':>11}  {'reg':>9}  {'stack':>6}  {'local':>6}")
    for name, b, t in rows:
        if b is None or t is None:
            print(f"{name:{w}}  {'new' if b is None else 'removed'}")
            continue
        cols = [f"{b[i]:>{k}}" if b[i] == t[i] else f"{b[i]}->{t[i]}".rjust(2 * k + 2) for i, k in ((0, 5), (2, 4), (3, 2), (4, 2))]
        print(f"{name:{w}}  {cols[0]:>11}  {cols[1]:>9}  {cols[2]:>6}  {cols[3]:>6}")


if __name__ == "__main__":
    main()
