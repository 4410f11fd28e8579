"""GPU probe (not part of the product): per-step time of general dense step kernels under two builds of the library.

    python scripts/step_variant_probe.py PARENT_LIB BRANCH_LIB [ROUNDS]

Random dense MDPs (every row has S successors, so no breakpoint table is built) at row widths that select the general
k-ary kernel (S <= 1024, NCH = ld / 128) and the long-row kernel (S > 1024), 65,536 envs, A = 4.  For each: the
persistent step server (`serve` / `step_served`, the SERVER kernels; host wall time per step) and random-action steps
launched back to back (the non-server kernels; CUDA events).  Each library runs in a child process (COLO_B200_LIB);
the driver alternates them for ROUNDS rounds in one call, so both see the same card, and prints the range per library.
"""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from colosseum_b200.batched_mdp import BatchedMDP  # noqa: E402
from colosseum_b200.tables import MDPTables  # noqa: E402

N, A = 65536, 4


def tables(S, seed):
    rng = np.random.default_rng(seed)
    T = rng.random((S, A, S), dtype=np.float32) + 0.01
    T /= T.sum(-1, keepdims=True)
    return MDPTables.from_dense(T, rew_kinds=[("deterministic", (0.5,)), ("beta", (2.0, 3.0))],
                                rew_cls_sa=rng.integers(0, 2, (S, A)).astype(np.int32))


def served_us(tb, mode, steps=400):
    env = BatchedMDP(tb, N, mode=mode, seed=1, host_io=True)
    env.reset()
    buf = torch.randint(0, A, (N,), dtype=torch.int32).pin_memory()
    env.serve(buf)
    for _ in range(50):
        env.step_served()
    t0 = time.perf_counter()
    for _ in range(steps):
        env.step_served()
    t = (time.perf_counter() - t0) / steps * 1e6
    env.stop_serving()
    return t


def launched_us(tb, mode, steps=400):
    env = BatchedMDP(tb, N, mode=mode, seed=1)
    env.reset()
    for _ in range(20):
        env.step_async(None, auto_reset=True)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        env.step_async(None, auto_reset=True)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps * 1e3


CONFIGS = (("dense_f32", 1024), ("dense_f64", 512), ("dense_f64", 896), ("dense_f32", 2048), ("dense_f64", 2048))


def child(label):
    for mode, S in CONFIGS:
        tb = tables(S, S)
        print(json.dumps({"lib": label, "mode": mode, "S": S, "served_us": round(served_us(tb, mode), 3),
                          "launched_us": round(launched_us(tb, mode), 3)}), flush=True)


def main():
    if sys.argv[1] == "--child":
        return child(sys.argv[2])
    libs = {"parent": os.path.abspath(sys.argv[1]), "branch": os.path.abspath(sys.argv[2])}
    rounds = int(sys.argv[3]) if len(sys.argv) > 3 else 3
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip(), flush=True)
    rows = []
    for _ in range(rounds):
        for label, lib in libs.items():
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", label], capture_output=True,
                                 text=True, env=dict(os.environ, COLO_B200_LIB=lib), check=True).stdout
            for line in out.splitlines():
                print(line, flush=True)
                rows.append(json.loads(line))
    for mode, S in CONFIGS:
        for key in ("served_us", "launched_us"):
            rng = {lb: [r[key] for r in rows if r["lib"] == lb and r["mode"] == mode and r["S"] == S] for lb in libs}
            print(f"{mode} S={S:5d} {key:11s} " + "   ".join(f"{lb} {min(v):8.2f}-{max(v):8.2f}" for lb, v in rng.items()))


if __name__ == "__main__":
    main()
