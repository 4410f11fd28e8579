"""Builds libcolosseum_b200.so (hand-written CUDA for sm_100a + the C ABI of include/colosseum_b200.h) in-tree.

    python -m colosseum_b200.build [--force]

nvcc cross-compiles without a GPU; the .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
INCLUDE = os.path.join(os.path.dirname(PKG), "include")
LIB_DIR = os.path.join(PKG, "_lib")
LIB_PATH = os.path.join(LIB_DIR, "libcolosseum_b200.so")
SOURCES = ["lib.cu", "backup.cu", "resident.cu", "gauss_seidel.cu", "sparse_hitting.cu", "env_step.cu", "agents.cu", "continuous_agents.cu", "builders.cu", "extended_vi.cu", "posterior.cu", "markov.cu", "synth.cu", "hitting_umma.cu", "suite_runner.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found: libcolosseum_b200.so cannot be built (there is no CPU fallback)")


def _stale():
    if not os.path.isfile(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, "colosseum_b200.h"), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force=False, verbose=False, defines=None, out=None):
    """Compile every CUDA source for sm_100a and link the shared library.  Returns its path.

    defines: {name: value} passed as -D to every source, for kernel-variant probes; out: path of the library to link
    (its objects go to a directory beside it).  A variant (either argument given) is always rebuilt."""
    lib_path = os.path.abspath(out) if out else LIB_PATH
    variant = bool(defines) or out is not None
    if not force and not variant and not _stale():
        return LIB_PATH
    lib_dir = os.path.dirname(lib_path)
    os.makedirs(lib_dir, exist_ok=True)
    obj_dir = os.path.join(lib_dir, "obj" if not variant else os.path.basename(lib_path) + ".obj")
    os.makedirs(obj_dir, exist_ok=True)
    nvcc = _nvcc()
    env = dict(os.environ)
    dflags = [f"-D{k}={v}" for k, v in (defines or {}).items()]
    procs = []
    for src in SOURCES:
        obj = os.path.join(obj_dir, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + dflags + ["-I", INCLUDE, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, obj, subprocess.Popen(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
    objs = []
    for src, obj, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out.decode())
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}")
        objs.append(obj)
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib_path] + objs
    subprocess.check_call(cmd, env=env)
    return lib_path


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
