"""Mixed agent batches against one single-MDP agent batch per instance, on the C3 suite (profiles/r3_mixed_agents_probe.txt).

For the episodic and the continuous C3 subsets (517 instances each) and L loops per instance: Q-learning (episodic:
UCB-Bernstein, continuous: the reference's defaults) with Colosseum's 500,000-step optimization horizon, advanced by
steps(1000) per launch in two ways that do the same work --
  mixed   one MixedQLearningEpisodic / MixedQLearningContinuous over every instance: one launch per steps()
  singles one QLearningEpisodic / QLearningContinuous per instance, stepped in a host loop on one stream
Both are warmed up with one steps(1000), then timed over one steps(1000) each (host clock around a device
synchronise).  Afterwards every loop's cumulative reward, episode count and Q table must agree between the two.

    python scripts/mixed_agents_probe.py [--loops 1 20] [--steps 1000] [--out FILE]
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

KW = {True: dict(p=0.05, c_1=0.4, c_2=0.9, min_at=0.0, UCB_type="bernstein"), False: dict()}
HORIZON = 500_000


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def run(al, torch, tbs, episodic, L, steps):
    mixed_cls = al.MixedQLearningEpisodic if episodic else al.MixedQLearningContinuous
    one_cls = al.QLearningEpisodic if episodic else al.QLearningContinuous
    seeds = list(range(len(tbs)))
    mixed = mixed_cls(seeds, tbs, HORIZON, n_loops=L, **KW[episodic])
    singles = [one_cls(s, tb, HORIZON, n_loops=L, **KW[episodic]) for s, tb in zip(seeds, tbs)]

    def timed(fn):
        torch.cuda.synchronize()
        t = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t

    def step_singles():
        for one in singles:
            one.steps(steps)

    timed(lambda: mixed.steps(steps))  # warm-up of both shapes
    timed(step_singles)
    t_mixed = timed(lambda: mixed.steps(steps))
    t_singles = timed(step_singles)
    ok = True
    cum, ep = mixed.cumulative_reward.cpu().numpy(), mixed.n_episodes.cpu().numpy()
    for i, one in enumerate(singles):
        sl = mixed.segment(i)
        ok &= np.array_equal(cum[sl], one.cumulative_reward.cpu().numpy())
        ok &= np.array_equal(ep[sl], one.n_episodes.cpu().numpy())
        ok &= torch.equal(mixed.table("Q", i), one.Q)
    n = mixed.n_loops
    q_mb = int(mixed.Q.numel()) * 4 / 2 ** 20
    del singles, mixed
    torch.cuda.empty_cache()
    return n, q_mb, t_mixed, t_singles, bool(ok)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--loops", type=int, nargs="+", default=[1, 20])
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    import colosseum_b200.agent_loop as al
    from colosseum_b200 import suite

    assert torch.cuda.is_available(), "the probe measures on the GPU"
    insts = suite.load_suite_all(os.path.join(ROOT, "tests", "golden"))
    lines = [f"card: {card()}", f"C3 suite: {len(insts)} instances; steps({args.steps}) per launch, horizon {HORIZON}"]
    print(lines[0], flush=True)
    all_ok = True
    for episodic in (True, False):
        tbs = [x.tables for x in insts if (x.tables.H > 0) == episodic]
        for L in args.loops:
            n, q_mb, tm, ts, ok = run(al, torch, tbs, episodic, L, args.steps)
            all_ok &= ok
            steps = n * args.steps
            line = (f"{'episodic' if episodic else 'continuous':10s} instances {len(tbs):4d}  L {L:3d}  loops {n:6d}  "
                    f"Q {q_mb:8.1f} MB  mixed {tm * 1e3:9.2f} ms {steps / tm / 1e6:9.2f} M agent-steps/s  "
                    f"singles {ts * 1e3:9.2f} ms {steps / ts / 1e6:9.2f} M agent-steps/s  "
                    f"speed-up {ts / tm:6.1f}x  parity {'ok' if ok else 'FAILED'}")
            print(line, flush=True)
            lines.append(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    return 0 if all_ok else 1


if __name__ == "__main__":
    sys.exit(main())
