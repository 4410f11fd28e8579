"""The C2 step with and without the breakpoint table (colo_mdp_tables.cdf_breaks), in one process and one build.

    python scripts/step_breaks_probe.py [--out FILE]

A side: the table nulled on every batch (`env.dev.c.cdf_breaks = None`), so the lean-shaped call takes the k-ary lean
kernel (two-level index, four dependent load rounds after the env scalars) and the fused walk the k-ary general kernel.
B side: the table as DeviceTables builds it (K = 2 for C2): one breakpoint round.

1. One step per launch, the bench's `value` protocol: NB env batches of N envs, each with its own tables, stepped in
   rotation (step i on batch i % NB) from ONE CUDA graph, replayed until the region lasts >= 30 ms, CUDA events around
   it.  NB is chosen so that the bytes the B side touches per pass over the batches (env state and counters, 38 bytes
   per env, plus the rows read) exceed 1.5 x the 126 MB L2 (at most 96), and both sides use the same NB.  N = 128 (the
   launch and drain floor of the kernel; its batches stay in L2), 65,536 (the headline), 1 Mi and 16 Mi.  A and B
   alternate, 3 regions each; medians.
2. The fused random walk: 1,000 random-action steps of 65,536 envs in one launch (random_steps_fused), A against B.
3. Outputs: after the same steps, A and B hold identical state, h, obs, reward bits and visitation counts.
Prints the GPU's name, power limit and SM clock, read in the same run."""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from colosseum_b200 import _cabi  # noqa: E402
from colosseum_b200.batched_mdp import BatchedMDP  # noqa: E402
from colosseum_b200.tables import MDPTables  # noqa: E402

L2 = 126 << 20
LINES = []


def say(s=""):
    print(s, flush=True)
    LINES.append(s)


def gpu_line():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                               "--format=csv,noheader"], capture_output=True, text=True,
                              timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # the numbers stand without it, but say so
        return f"{torch.cuda.get_device_name(0)} (nvidia-smi unavailable: {e})"


def launches():
    return np.array([_cabi.lib().colo_step_kernel_launches(k) for k in range(9)], np.int64)


def strip(env):
    env.dev.c.cdf_breaks, env.dev.c.cdf_breaks_k = None, 0


def rotating(tb, N, NB, side, min_ms=30.0):
    """ms per step of one graph of rotating steps over NB batches, replayed to >= min_ms; the graph is built once and
    the regions alternate between the sides by the caller"""
    gen = torch.Generator(device="cuda").manual_seed(1234)
    acts = [torch.randint(0, tb.A, (N,), dtype=torch.int32, device="cuda", generator=gen) for _ in range(2)]
    batches = [BatchedMDP(tb, N, mode="dense_f32", seed=99 + i) for i in range(NB)]
    for b in batches:
        if side == "A":
            strip(b)
        b.reset()
        b.step_async(acts[0], auto_reset=True)
    torch.cuda.synchronize()
    per_graph = max(NB, 64 // NB * NB)
    before = launches()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for i in range(per_graph):
            batches[i % NB].step_async(acts[i % 2], auto_reset=True)
    kind = int(np.argmax(launches() - before))
    graph.replay()
    torch.cuda.synchronize()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    graph.replay()
    g1.record()
    g1.synchronize()
    reps = max(1, int(np.ceil(min_ms / max(g0.elapsed_time(g1), 1e-3))))

    def region():
        g0.record()
        for _ in range(reps):
            graph.replay()
        g1.record()
        g1.synchronize()
        return g0.elapsed_time(g1) / (reps * per_graph)

    assert all(int(b.status.item()) == 0 for b in batches)
    return region, kind, (graph, batches)


def step_ab(tb, N):
    touched = 38 * N + 32 * tb.S * tb.A  # B side: env state and counters, and the breakpoint rows at most
    NB = min(96, max(2, int(1.5 * L2 / touched) + 1))  # (N = 128: the floor, its NB batches stay in L2)
    ra, ka, keep_a = rotating(tb, N, NB, "A")
    rb, kb, keep_b = rotating(tb, N, NB, "B")
    ta, tb_ = [], []
    for _ in range(3):
        ta.append(ra())
        tb_.append(rb())
    a, b = float(np.median(ta)), float(np.median(tb_))
    say(f"N={N:>9,} NB={NB:>3}  A kind {ka}: {a * 1e3:8.2f} us/step ({N / a / 1e6:6.2f} G env-steps/s)  "
        f"B kind {kb}: {b * 1e3:8.2f} us/step ({N / b / 1e6:6.2f} G)  A/B {a / b:5.3f}  "
        f"[A {' '.join(f'{x * 1e3:.2f}' for x in ta)}; B {' '.join(f'{x * 1e3:.2f}' for x in tb_)}]")
    del keep_a, keep_b
    torch.cuda.empty_cache()


def fused_ab(tb, N=65536, K=1000):
    envs = {}
    for side in "AB":
        env = BatchedMDP(tb, N, mode="dense_f32", seed=4321)
        if side == "A":
            strip(env)
        env.reset()
        env.random_steps_fused(50)
        envs[side] = env
    torch.cuda.synchronize()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    res = {"A": [], "B": []}
    for _ in range(3):
        for side in "AB":
            before = launches()
            g0.record()
            envs[side].random_steps_fused(K)
            g1.record()
            g1.synchronize()
            res[side].append(g0.elapsed_time(g1) / K)
            kind = int(np.argmax(launches() - before))
            res.setdefault(side + "kind", kind)
    a, b = float(np.median(res["A"])), float(np.median(res["B"]))
    say(f"fused walk {K} steps x {N:,} envs: A kind {res['Akind']}: {a * 1e3:.3f} us/step  "
        f"B kind {res['Bkind']}: {b * 1e3:.3f} us/step  A/B {a / b:.3f}")
    same = all(torch.equal(getattr(envs["A"], f), getattr(envs["B"], f)) for f in ("state", "h", "obs", "step_type"))
    same &= torch.equal(envs["A"].reward.view(torch.int32), envs["B"].reward.view(torch.int32))
    same &= torch.equal(envs["A"].visits_sa, envs["B"].visits_sa)
    say(f"fused walk outputs identical A vs B: {same}")


def outputs_ab(tb, N=65536, steps=200):
    gen = torch.Generator(device="cuda").manual_seed(7)
    acts = [torch.randint(0, tb.A, (N,), dtype=torch.int32, device="cuda", generator=gen) for _ in range(steps)]
    out = {}
    for side in "AB":
        env = BatchedMDP(tb, N, mode="dense_f32", seed=5)
        if side == "A":
            strip(env)
        env.reset()
        for a in acts:
            env.step_async(a, auto_reset=True)
        out[side] = [env.state, env.h, env.obs, env.step_type, env.reward.view(torch.int32), env.visits_s, env.visits_sa]
    same = all(torch.equal(x, y) for x, y in zip(out["A"], out["B"]))
    say(f"{steps} lean-shaped steps x {N:,} envs, outputs identical A vs B: {same}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="128,65536,1048576,16777216")
    args = ap.parse_args()
    torch.cuda.set_device(0)
    tb = MDPTables.from_golden(np.load(os.path.join(ROOT, "tests", "golden", "inst_c2_deepsea30_prand.npz")))
    say(f"GPU: {gpu_line()}")
    say(f"C2 = DeepSeaContinuous(size=30, p_rand=0.1): S={tb.S} A={tb.A} ld={tb.ld}; "
        f"breakpoint table K={BatchedMDP(tb, 1).dev.breaks_k}")
    say("A = table nulled (k-ary kernels), B = breakpoint table; kinds: 0 k-ary lean, 1 k-ary general, 7 breakpoint "
        "lean, 8 breakpoint general")
    for N in [int(x) for x in args.sizes.split(",")]:
        step_ab(tb, N)
    fused_ab(tb)
    outputs_ab(tb)
    say(f"GPU after the runs: {gpu_line()}")
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
