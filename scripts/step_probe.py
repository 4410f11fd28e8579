"""GPU probe (not part of the product): step-kernel timing under different conditions."""
import os, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from colosseum_b200.batched_mdp import BatchedMDP
from colosseum_b200.tables import MDPTables

g = np.load("tests/golden/inst_c2_deepsea30_prand.npz")
tb = MDPTables.from_golden(g)
N = 65536
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

def timeit(env, steps=200, do_flush=False, random_actions=False, acts=None):
    for i in range(10):
        env.step_async(None if random_actions else acts[i % 8], auto_reset=True)
    torch.cuda.synchronize()
    if do_flush:
        tot = 0.0
        for i in range(steps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); env.step_async(None if random_actions else acts[i % 8], auto_reset=True); b.record()
            torch.cuda.synchronize()
            tot += a.elapsed_time(b)
        return tot / steps * 1e3
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(steps):
        env.step_async(None if random_actions else acts[i % 8], auto_reset=True)
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / steps * 1e3

for mode in ("dense_f32", "dense_f64", "succ"):
    for visits in (True, False):
        env = BatchedMDP(tb, N, mode=mode, seed=1, track_visits=visits)
        env.reset()
        acts = [torch.randint(0, tb.A, (N,), dtype=torch.int32, device="cuda") for _ in range(8)]
        t_warm = timeit(env, acts=acts)
        t_cold = timeit(env, acts=acts, do_flush=True)
        t_rand = timeit(env, random_actions=True)
        print(f"{mode:10s} visits={visits!s:5s}  back-to-back {t_warm:7.2f} us   flushed {t_cold:7.2f} us   random-actions b2b {t_rand:7.2f} us")
# spread states: uniform start over all states (less atomic contention, more distinct rows)
env = BatchedMDP(tb, N, mode="dense_f32", seed=1)
env.reset()
env.state.copy_(torch.randint(0, tb.S, (N,), dtype=torch.int32, device="cuda"))
acts = [torch.randint(0, tb.A, (N,), dtype=torch.int32, device="cuda") for _ in range(8)]
env.step_async(acts[0]); torch.cuda.synchronize()
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
env.state.copy_(torch.randint(0, tb.S, (N,), dtype=torch.int32, device="cuda"))
a.record(); env.step_async(acts[1]); b.record(); torch.cuda.synchronize()
print("dense_f32 uniformly spread states, single launch:", a.elapsed_time(b) * 1e3, "us")
# empty-ish launch overhead reference
x = torch.zeros(1, device="cuda")
a.record()
for _ in range(200): x.add_(1)
b.record(); torch.cuda.synchronize()
print("torch tiny kernel back-to-back:", a.elapsed_time(b) / 200 * 1e3, "us")
