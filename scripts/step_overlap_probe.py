"""Where the launch overlap of the lean step kernels gains (DESIGN 4.2): the parent library against builds of the branch.

    python scripts/step_overlap_probe.py --build                     (CPU: builds the variant libraries)
    python scripts/step_overlap_probe.py --parent-root DIR [--rounds 3] [--sizes ...] [--out FILE]

Variants, each run in a child process (the branch ones load their library through COLO_B200_LIB; the parent one
imports the package from DIR, a built checkout of the parent commit):
  parent        the parent commit: plain launches, no prefetch
  off           the branch with the switch off (COLO_STEP_OVERLAP=0): plain launches of the kernels without the
                prefetch (only ACQBULK and PREEXIT differ from the parent)
  pdl           the branch built with COLO_STEP_PREFETCH=0: launch overlap without the prefetches
  trigger0/1/2  the branch built with COLO_STEP_PDL_TRIGGER=0 (launch_dependents before the wait, the round-1 form),
                1 (after the wait: the shipped build) and 2 (after the stores)
  prefetch_all  an earlier form of trigger1 (variants/prefetch_all, a library built from that revision; skipped when
                absent): one kernel, prefetching at every grid size, and one CTA prefetching up to 64 chunks of 4 KiB
                per batch-wide array when the grid is too small to share them
Protocol (scripts/step_breaks_probe.py): C2, NB batches of N envs with their own tables, stepped in rotation (step i on
batch i % NB) from one CUDA graph, replayed until a region lasts >= 30 ms, CUDA events around it; NB so that a pass over
the batches touches more than 1.5 x the 126 MB L2 (N = 128: the launch and drain floor, its batches stay in L2).  Every
child builds the same NB batches and times three regions per N; the variants alternate, `--rounds` rounds, and the table
gives the median and range over rounds of the per-child medians.  Each child also runs the same 200 steps of 65,536
envs on one batch and prints a digest of state, h, obs, reward bits, step_type and both counter tables: all variants
must agree.  Prints the GPU's name, power limit and SM clock, read in the same run."""
import argparse
import hashlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VARIANT_DIR = os.path.join(ROOT, "colosseum_b200", "_lib", "variants")
BUILDS = {"pdl": {"COLO_STEP_PREFETCH": 0}, "trigger0": {"COLO_STEP_PDL_TRIGGER": 0},
          "trigger2": {"COLO_STEP_PDL_TRIGGER": 2}}
L2 = 126 << 20


def variant_lib(name):
    return os.path.join(VARIANT_DIR, name, "libcolosseum_b200.so")


def gpu_line():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                               "--format=csv,noheader"], capture_output=True, text=True,
                              timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # the numbers stand without it, but say so
        return f"(nvidia-smi unavailable: {e})"


def child(sizes):
    import numpy as np
    import torch

    from colosseum_b200 import _cabi
    from colosseum_b200.batched_mdp import BatchedMDP
    from colosseum_b200.tables import MDPTables

    lib = _cabi.lib()
    tb = MDPTables.from_golden(np.load(os.path.join(ROOT, "tests", "golden", "inst_c2_deepsea30_prand.npz")))

    def kinds():
        return np.array([lib.colo_step_kernel_launches(k) for k in range(9)], np.int64)

    def overlapped():
        return int(lib.colo_step_overlap_launches()) if hasattr(lib, "colo_step_overlap_launches") else 0

    for N in sizes:
        NB = min(96, max(2, int(1.5 * L2 / (38 * N + 32 * tb.S * tb.A)) + 1))
        gen = torch.Generator(device="cuda").manual_seed(1234)
        acts = [torch.randint(0, tb.A, (N,), dtype=torch.int32, device="cuda", generator=gen) for _ in range(2)]
        batches = [BatchedMDP(tb, N, mode="dense_f32", seed=99 + i) for i in range(NB)]
        for b in batches:
            b.reset()
            b.step_async(acts[0], auto_reset=True)
        torch.cuda.synchronize()
        per_graph = max(NB, 64 // NB * NB)
        k0, o0 = kinds(), overlapped()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for i in range(per_graph):
                batches[i % NB].step_async(acts[i % 2], auto_reset=True)
        kind, n_over = int(np.argmax(kinds() - k0)), overlapped() - o0
        graph.replay()
        torch.cuda.synchronize()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        graph.replay()
        g1.record()
        g1.synchronize()
        reps = max(1, int(np.ceil(30.0 / max(g0.elapsed_time(g1), 1e-3))))
        regions = []
        for _ in range(3):
            g0.record()
            for _ in range(reps):
                graph.replay()
            g1.record()
            g1.synchronize()
            regions.append(g0.elapsed_time(g1) * 1e3 / (reps * per_graph))
        assert all(int(b.status.item()) == 0 for b in batches)
        print(json.dumps({"N": N, "NB": NB, "kind": kind, "overlapped": n_over, "per_graph": per_graph,
                          "us": float(np.median(regions))}), flush=True)
        del graph, batches
        torch.cuda.empty_cache()

    N = 65536
    gen = torch.Generator(device="cuda").manual_seed(7)
    acts = [torch.randint(0, tb.A, (N,), dtype=torch.int32, device="cuda", generator=gen) for _ in range(200)]
    env = BatchedMDP(tb, N, mode="dense_f32", seed=5)
    env.reset()
    for a in acts:
        env.step_async(a, auto_reset=True)
    torch.cuda.synchronize()
    h = hashlib.sha256()
    for x in (env.state, env.h, env.obs, env.step_type, env.reward.view(torch.int32), env.visits_s, env.visits_sa):
        h.update(x.cpu().numpy().tobytes())
    print(json.dumps({"digest": h.hexdigest()}), flush=True)


def build():
    sys.path.insert(0, ROOT)
    from colosseum_b200 import build as b

    print(b.build_library())
    for name, defines in BUILDS.items():
        print(b.build_library(defines=defines, out=variant_lib(name)), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--build", action="store_true")
    ap.add_argument("--child", action="store_true")
    ap.add_argument("--parent-root")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--sizes", default="128,65536,1048576,16777216")
    ap.add_argument("--out")
    args = ap.parse_args()
    sizes = [int(x) for x in args.sizes.split(",")]
    if args.build:
        return build()
    if args.child:
        sys.path.insert(0, os.environ["COLO_PROBE_ROOT"])
        return child(sizes)
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    branch_lib = os.path.join(ROOT, "colosseum_b200", "_lib", "libcolosseum_b200.so")
    parent_root = os.path.abspath(args.parent_root)
    variants = {"parent": (parent_root, {}),
                "off": (ROOT, {"COLO_B200_LIB": branch_lib, "COLO_STEP_OVERLAP": "0"}),
                "pdl": (ROOT, {"COLO_B200_LIB": variant_lib("pdl")}),
                "trigger0": (ROOT, {"COLO_B200_LIB": variant_lib("trigger0")}),
                "trigger1": (ROOT, {"COLO_B200_LIB": branch_lib}),
                "trigger2": (ROOT, {"COLO_B200_LIB": variant_lib("trigger2")}),
                "prefetch_all": (ROOT, {"COLO_B200_LIB": variant_lib("prefetch_all")})}
    if not os.path.isfile(variant_lib("prefetch_all")):
        del variants["prefetch_all"]
    say(f"GPU: {gpu_line()}")
    say("C2 = DeepSeaContinuous(size=30, p_rand=0.1), S=465 A=2, breakpoint table K=2 (env_step_breaks_lean_kernel<2>)")
    rows = {v: {} for v in variants}
    digests = {v: set() for v in variants}
    for r in range(args.rounds):
        for name, (root, env) in variants.items():
            environ = dict(os.environ, COLO_PROBE_ROOT=root)
            environ.pop("COLO_B200_LIB", None)
            environ.pop("COLO_STEP_OVERLAP", None)
            environ.update(env)
            out =subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--sizes", args.sizes],
                                 capture_output=True, text=True, env=environ)
            if out.returncode != 0:
                sys.exit(f"{name}: child failed\n{out.stdout}\n{out.stderr}")
            for line in out.stdout.splitlines():
                d = json.loads(line)
                if "digest" in d:
                    digests[name].add(d["digest"])
                else:
                    rows[name].setdefault(d["N"], []).append(d)
            say(f"round {r + 1} {name:12s} " + "  ".join(f"N={n}: {ds[-1]['us']:.3f} us" for n, ds in rows[name].items()))
    say("")
    say("per step, median over rounds [range]; kind 7 = env_step_breaks_lean_kernel; overlapped = graph launches that "
        "carried the PDL attribute (of per_graph)")
    for N in sizes:
        base = float(sorted(d["us"] for d in rows["parent"][N])[len(rows["parent"][N]) // 2])
        for name in variants:
            ds = rows[name][N]
            us = sorted(d["us"] for d in ds)
            med = us[len(us) // 2]
            say(f"N={N:>9,} NB={ds[0]['NB']:>3}  {name:12s} kind {ds[0]['kind']}  overlapped {ds[0]['overlapped']:>3}/"
                f"{ds[0]['per_graph']}  {med:8.3f} us/step [{us[0]:.3f}-{us[-1]:.3f}]  {N / med / 1e3:7.2f} G env-steps/s"
                f"  parent/this {base / med:5.3f}")
    same = len(set().union(*digests.values())) == 1 and all(len(d) == 1 for d in digests.values())
    say(f"200 steps x 65,536 envs: state, h, obs, reward bits, step_type and counters identical across all variants "
        f"and rounds: {same}")
    say(f"GPU after the runs: {gpu_line()}")
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    if not same:
        sys.exit("outputs differ between variants")


if __name__ == "__main__":
    main()
