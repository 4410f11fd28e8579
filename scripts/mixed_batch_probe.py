"""Mixed batches (MixedBatchedMDP) against one BatchedMDP per instance.

    python scripts/mixed_batch_probe.py [--out FILE]

1. The C3 step phase of 128 suite instances (1,024 envs x 1,000 random auto-resetting steps each, seed 0, tables
   uploaded beforehand, one warm-up pass): (a) 128 x (BatchedMDP.reset + random_steps_fused) on one stream against
   (b) one MixedBatchedMDP reset + one random_steps_fused.  Wall time to a device synchronise; the per-instance
   visitation counts of (a) and (b) are compared.
2. One launch per step, succ mode, random actions: 65,536 envs spread over the 94 seed-0 parameter sets of the suite
   against 65,536 envs of one instance (c2_deepsea30_prand), 1,000 step launches captured in a CUDA graph and timed
   with CUDA events over one replay.  Two more rows tell apart where a difference comes from: a mixed batch holding
   that one instance only (the per-env descriptor and instance-map loads) and one holding 94 copies of it (the same
   loads, with the warps still reading one MDP's tables).  The graph replay leaves the host's launch cost out of both
   sides: it compares the kernels.  What a caller of step_async() pays per call is timed as well: the same 1,000 steps
   launched one Python call at a time, wall time to a device synchronise.
3. The same for the dense f32 rows: the mixed batch's warp-per-env search against the single-MDP k-ary kernel (the
   kernel a random-action dense f32 step takes).
Prints the GPU's name and power limit with the numbers."""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from colosseum_b200 import suite  # noqa: E402
from colosseum_b200.batched_mdp import BatchedMDP, MixedBatchedMDP, split_sizes  # noqa: E402
from colosseum_b200.tables import MDPTables  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
LINES = []


def say(s=""):
    print(s, flush=True)
    LINES.append(s)


def gpu_line():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # the numbers stand without it, but say so
        q = f"{torch.cuda.get_device_name(0)} (nvidia-smi unavailable: {e})"
    return q


def c3_step_phase(n_inst, n_envs, n_steps, passes):
    insts = suite.load_suite_all(GOLDEN, indices=range(n_inst))
    singles = [BatchedMDP(x.tables, n_envs, mode="succ", seed=0) for x in insts]
    mixed = MixedBatchedMDP([x.tables for x in insts], n_envs, mode="succ", seed=0)
    torch.cuda.synchronize()

    def run_singles():
        for env in singles:
            env.reset()
            env.random_steps_fused(n_steps, auto_reset=True)

    def run_mixed():
        mixed.reset()
        mixed.random_steps_fused(n_steps, auto_reset=True)

    res = {}
    for name, fn in (("a", run_singles), ("b", run_mixed)):
        fn()  # warm-up pass
        torch.cuda.synchronize()
    for env in singles:
        env.reset_visitation_counts()
    mixed.reset_visitation_counts()
    for name, fn in (("a", run_singles), ("b", run_mixed)) * passes:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        res.setdefault(name, []).append(time.perf_counter() - t0)
    same = all(torch.equal(mixed.get_visitation_counts(i), env.visits_s)
               and torch.equal(mixed.get_visitation_counts(i, False), env.visits_sa) for i, env in enumerate(singles))
    same_state = all(torch.equal(mixed.state[mixed.segment(i)], env.state) for i, env in enumerate(singles))
    return res, same and same_state


def graph_rate(env, n_steps, reps):
    """env-steps/s of n_steps single-step launches (random actions, auto-reset) replayed from one CUDA graph"""
    env.reset()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            env.step_async(None, auto_reset=True)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(n_steps):
            env.step_async(None, auto_reset=True)
    g.replay()  # warm-up replay
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1) / 1e3)
    return [env.n_envs * n_steps / t for t in times], times


def eager_rate(env, n_steps, reps):
    """the same n_steps launches, one step_async() call each from Python: wall time to a device synchronise"""
    for _ in range(3):
        env.step_async(None, auto_reset=True)
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        for _ in range(n_steps):
            env.step_async(None, auto_reset=True)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    return [env.n_envs * n_steps / t for t in times], times


def compare(rows, n_steps):
    """one line per row: graph replay (kernels only) and one Python call per step; returns the best graph rates"""
    best = {}
    for label, make in rows:
        env = make()
        rates, times = graph_rate(env, n_steps, 3)
        erates, etimes = eager_rate(env, n_steps, 3)
        best[label] = max(rates)
        say(f"{label}: graph best {max(rates) / 1e9:.3f} G env-steps/s ({min(times) * 1e6 / n_steps:.2f} us per step), "
            f"replays {[round(r / 1e9, 3) for r in rates]} G; one step_async() call per step: best "
            f"{max(erates) / 1e9:.3f} G ({min(etimes) * 1e6 / n_steps:.2f} us per step)")
        del env
        torch.cuda.synchronize()
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--c3-instances", type=int, default=128)
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--passes", type=int, default=3)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    say(f"# python scripts/mixed_batch_probe.py  GPU: {gpu_line()}  (name, power limit, max SM clock)")

    res, same = c3_step_phase(args.c3_instances, 1024, 1000, args.passes)
    say(f"## 1. C3 step phase, {args.c3_instances} suite instances x 1,024 envs x 1,000 random steps (succ, seed 0), "
        f"wall time to a device synchronise, {args.passes} timed passes after one warm-up pass")
    for name, label in (("a", f"(a) {args.c3_instances} x BatchedMDP reset + random_steps_fused, one stream"),
                        ("b", "(b) one MixedBatchedMDP reset + random_steps_fused")):
        ts = res[name]
        say(f"{label}: best {min(ts) * 1e3:.2f} ms, median {np.median(ts) * 1e3:.2f} ms, passes "
            f"{[round(t * 1e3, 2) for t in ts]} ms")
    say(f"(a) / (b), best passes: {min(res['a']) / min(res['b']):.2f}x; per-instance visitation counts and states "
        f"equal: {same}")

    N, n_steps = args.envs, args.steps
    say(f"## 2. one launch per step, succ, random actions, auto-reset, {N:,} envs, {n_steps:,} step launches in one "
        f"CUDA graph, CUDA events around a replay (3 replays after a warm-up replay); then 3 x {n_steps:,} "
        f"step_async() calls, wall time to a device synchronise")
    insts = suite.load_suite_all(GOLDEN, indices=range(94))
    sizes, _ = split_sizes(N, len(insts))
    one = MDPTables.from_golden(np.load(os.path.join(GOLDEN, "inst_c2_deepsea30_prand.npz")))
    rows = [("mixed, the 94 seed-0 parameter sets", lambda: MixedBatchedMDP([x.tables for x in insts], sizes, "succ", 0)),
            ("single BatchedMDP, c2_deepsea30_prand", lambda: BatchedMDP(one, N, mode="succ", seed=0)),
            ("mixed, c2_deepsea30_prand alone", lambda: MixedBatchedMDP([one], N, "succ", 0)),
            ("mixed, 94 copies of c2_deepsea30_prand", lambda: MixedBatchedMDP([one] * 94, sizes, "succ", 0))]
    best = compare(rows, n_steps)
    a, b = best[rows[0][0]], best[rows[1][0]]
    say(f"single / mixed (94 sets), per env-step, graph: {b / a:.2f}x")

    say(f"## 3. the same for dense f32 rows (random actions, auto-reset, {N:,} envs, {n_steps:,} steps): the mixed "
        f"batch's warp-per-env search against the single-MDP k-ary kernel")
    rows = [("mixed dense_f32, the 94 seed-0 parameter sets",
             lambda: MixedBatchedMDP([x.tables for x in insts], sizes, "dense_f32", 0)),
            ("single BatchedMDP dense_f32, c2_deepsea30_prand", lambda: BatchedMDP(one, N, mode="dense_f32", seed=0)),
            ("mixed dense_f32, c2_deepsea30_prand alone", lambda: MixedBatchedMDP([one], N, "dense_f32", 0))]
    best = compare(rows, n_steps)
    a, b = best[rows[0][0]], best[rows[1][0]]
    say(f"single / mixed (94 sets), per env-step, graph: {b / a:.2f}x")
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
