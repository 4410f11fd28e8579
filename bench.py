#!/usr/bin/env python
"""bench.py -- the driver's measurement contract for colosseum_b200.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload step|vi|all] [--dump-outputs DIR]

Headline workload (BASELINE.json configs[1], "C2"): DeepSeaContinuous(size=30, p_rand=0.1) -- S=465, A=2 -- with
65,536 parallel envs PER GPU advanced by the batched step kernel; metric = batched env-steps/sec over all GPUs.
One "step" = one launch of the step kernel over every env of the rank (inputs resident in HBM).  The JSON line also
carries, under "vi", value-iteration MDP-sweeps/sec on config C4's shape (B x (S=512, A=4) synthetic Dirichlet
MDPs, one sweep = one launch of the backup kernel over the whole batch) with its own roofline.

`--impl reference` times the reference's CPU algorithm for the same workload on the host cores (the C oracle port
under oracle/, all threads) -- the only other place this file touches oracle/.  /root/reference does not exist on
the GPU box and is never read here.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C2_INSTANCE = "c2_deepsea30_prand"
C2_ENVS_PER_GPU = 65536
STEP_BYTES = lambda S: 4 * S + 28  # SURVEY.md section 8d: dense CDF row + 28 B of state I/O per env-step (nominal)
# what one env-step MUST move to and from HBM once the 2.9 MB of tables are on chip: read state 4 + h 4 + step_type 1 +
# action 4, write state 4 + h 4 + obs 4 + reward 4 + discount 4 + step_type 1
STEP_IO_BYTES = 34


def c2_workload(S, A, N):
    """the one description of the headline workload both arms put in config.workload"""
    return (f"C2 DeepSeaContinuous(size=30,p_rand=0.1) S={S} A={A}, {N} envs per GPU, batched step by inverse-CDF over the "
            "dense CDF row, auto-reset, visitation counts on")
L2_FLUSH_BYTES = 256 << 20
# untimed steps enqueued right before the headline's timed replay (about 70 ms at the ~15 G env-steps/s this bench
# measures for the headline on a B200 at 1,000 W): the GPU is busy and at its steady clocks when the timed steps start,
# and the count is fixed, so the final env state depends on the arguments only
LEAD_IN_STEPS = 16384


def vi_sweep_bytes(S, A, store_q=True):
    """SURVEY.md section 8d: 4*S*A*S (T) + 4*S*A (R) + 4*S (V read) + 4*S (V write) [+ 4*S*A Q] per MDP-sweep"""
    return 4 * S * A * S + 4 * S * A + 8 * S + (4 * S * A if store_q else 0)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def step_ncu_evidence():
    """what ncu measured on the shipped step kernel at 4 Mi envs (profiles/r2_ncu_summary.json, written by
    scripts/summarize_ncu_r2.py from the `ncu --set full` capture of scripts/profile_r2.sh)"""
    p = os.path.join(ROOT, "profiles", "r2_ncu_summary.json")
    if os.path.isfile(p):
        e = json.load(open(p)).get("step_4194304")
        if e:
            return e
    return None


def ncu_traffic(key, units):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture
    (profiles/ncu_traffic.json, written by scripts/summarize_ncu.py), scaled to this run's units per launch"""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.isfile(p):
        e = json.load(open(p)).get(key)
        if e:
            return e["dram_bytes_per_unit"] * units
    return None


class ClockSampler:
    """samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)"""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def load_c2_tables(instance=C2_INSTANCE):
    from colosseum_b200.tables import MDPTables

    g = np.load(os.path.join(ROOT, "tests", "golden", f"inst_{instance}.npz"))
    return MDPTables.from_golden(g)


# ------------------------------------------------------------------------------------------------ GPU arm
def dist_setup(n_gpus):
    import torch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # stdout carries exactly ONE JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local


def barrier_sync(world):
    import torch

    if world > 1:
        import torch.distributed as dist

        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(x, world):
    import torch

    if world == 1:
        return x
    import torch.distributed as dist

    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def _rotating_graph(torch, tb, N, rank, actions, n_steps, seed0, min_ms, world, track_visits=True, outputs=False):
    """`value` protocol: inputs larger than L2 instead of a flush.  NB independent env batches of N envs (each with its
    own tables; together > 1.5 x the 126 MB L2) are stepped in rotation (step i on batch i % NB) from ONE CUDA graph.
    min_ms=None: the graph holds exactly `n_steps` launches and the timed region is one replay of it, enqueued right
    behind at least LEAD_IN_STEPS untimed steps from a second graph that steps every batch once, in order, so that
    whatever `n_steps` is, each timed step's batch was last stepped NB - 1 batches (more than L2) earlier.  Otherwise
    the graph holds max(n_steps, NB) launches and is replayed until the timed region is at least `min_ms`.  Returns ms
    per step (device time, CUDA events on the launching stream, max over ranks), the number of timed steps, the region
    length and the bytes it touched; outputs=True adds what the last timed step left in its batch (the TimeStep
    fields, env state and visitation counts) as host arrays."""
    from colosseum_b200.batched_mdp import BatchedMDP

    per_batch = 38 * N + 4 * tb.S * tb.A * (tb.ld + tb.ld // 4 + tb.ld // 32) + 2 * tb.S * tb.A * tb.ld
    NB = int(1.5 * (126 << 20) / per_batch) + 1
    batches = [BatchedMDP(tb, N, mode="dense_f32", seed=seed0 + i, env_offset=rank * N, track_visits=track_visits)
               for i in range(NB)]
    n_act = len(actions)
    for b in batches:
        b.reset()
        b.step_async(actions[0], auto_reset=True)
    torch.cuda.synchronize()
    for i in range(max(3, min(NB, 8))):  # untimed warm-up steps, same rotation
        batches[i % NB].step_async(actions[i % n_act], auto_reset=True)
    torch.cuda.synchronize()
    per_graph = n_steps if min_ms is None else max(n_steps, NB)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):  # step i runs on env batch i % NB
        for i in range(per_graph):
            batches[i % NB].step_async(actions[i % n_act], auto_reset=True)
    graph.replay()
    torch.cuda.synchronize()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if min_ms is None:
        reps, lead_in = 1, -(-LEAD_IN_STEPS // NB)
        lead = torch.cuda.CUDAGraph()
        with torch.cuda.graph(lead):  # step j on env batch j: each pass ends on batch NB - 1, right before timed step 0
            for j in range(NB):
                batches[j].step_async(actions[j % n_act], auto_reset=True)
        lead.replay()
        torch.cuda.synchronize()
    else:
        g0.record()
        graph.replay()
        g1.record()
        g1.synchronize()
        reps = max(1, int(np.ceil(1.3 * min_ms / max(g0.elapsed_time(g1), 1e-3))))  # 30 % margin over the calibration replay
        lead_in = 0
    barrier_sync(world)
    for _ in range(lead_in):
        lead.replay()
    g0.record()
    for _ in range(reps):
        graph.replay()
    g1.record()
    barrier_sync(world)
    ms = max_over_ranks(g0.elapsed_time(g1), world)
    assert all(int(b.status.item()) == 0 for b in batches)
    out = dict(ms_per_step=ms / (reps * per_graph), timed_steps=reps * per_graph, region_ms=ms, batches=NB,
               batch_bytes=per_batch, bytes_touched=NB * per_batch, timed_bytes=min(reps * per_graph, NB) * per_batch,
               steps_per_graph=per_graph, replays=reps, lead_in_steps=lead_in * NB)
    if outputs:
        last = batches[(per_graph - 1) % NB]
        ts = last._timestep()
        out["outputs"] = {name: t.cpu().numpy() for name, t in (
            ("step_type", ts.step_type), ("reward", ts.reward), ("discount", ts.discount), ("observation", ts.observation),
            ("state", last.state), ("h", last.h), ("visits_s", last.visits_s), ("visits_sa", last.visits_sa))}
    del graph, batches
    if min_ms is None:
        del lead
    torch.cuda.empty_cache()
    return out


def bench_step_gpu(args, rank, world):
    """kernel-resident number (`value`), the env-count sweep that names the step kernel's bound, and the end-to-end
    number (`e2e`) for the batched step"""
    import torch

    from colosseum_b200 import _cabi
    from colosseum_b200.batched_mdp import BatchedMDP

    tb = load_c2_tables()
    N = C2_ENVS_PER_GPU
    env = BatchedMDP(tb, N, mode="dense_f32", seed=1234, env_offset=rank * N)
    env.reset()
    gen = torch.Generator(device="cuda").manual_seed(1234 + rank)
    n_act = 8
    actions = [torch.randint(0, tb.A, (N,), dtype=torch.int32, device="cuda", generator=gen) for _ in range(n_act)]
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device="cuda")
    lib = _cabi.lib()

    def one_step(i):
        env.step_async(actions[i % n_act], auto_reset=True)

    for i in range(args.warmup):
        flush.zero_()
        one_step(i)
    barrier_sync(world)
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    lib.colo_reset_launch_count()
    for i in range(args.steps):
        flush.zero_()  # L2 flush between timed iterations (256 MiB write > 126 MB L2); not timed
        starts[i].record()
        one_step(i)
        stops[i].record()
    barrier_sync(world)
    launches = int(lib.colo_launch_count())
    ms = sum(s.elapsed_time(e) for s, e in zip(starts, stops))
    ms = max_over_ranks(ms, world)
    assert int(env.status.item()) == 0

    # ---- secondary: SURVEY section 8d asks for C2 with p_rand=None too (deterministic rows, 1 non-zero): same kernel,
    # same protocol, fewer steps
    det = None
    try:
        tbd = load_c2_tables("c2_deepsea30")
        envd = BatchedMDP(tbd, N, mode="dense_f32", seed=1234, env_offset=rank * N)
        envd.reset()
        nd = max(20, min(args.steps, 100))
        for i in range(5):
            flush.zero_()
            envd.step_async(actions[i % n_act], auto_reset=True)
        barrier_sync(world)
        ds = [torch.cuda.Event(enable_timing=True) for _ in range(nd)]
        de = [torch.cuda.Event(enable_timing=True) for _ in range(nd)]
        for i in range(nd):
            flush.zero_()
            ds[i].record()
            envd.step_async(actions[i % n_act], auto_reset=True)
            de[i].record()
        barrier_sync(world)
        det = dict(ms=max_over_ranks(sum(a.elapsed_time(b) for a, b in zip(ds, de)), world), steps=nd)
        del envd
    except Exception as e:
        det = dict(error=f"{type(e).__name__}: {e}")
    del flush

    # ---- headline: back-to-back kernel throughput.  The per-step event pair above has a floor of ~10 us on B200
    # (measured with a 32-env launch), i.e. most of it is launch + event latency, not the kernel.  Here the --steps
    # steps of NB independent env batches (each with its own tables; together larger than L2, so no flush is needed)
    # are captured in one CUDA graph and timed over one replay: no CPU in the loop.
    b2b = None
    try:
        b2b = _rotating_graph(torch, tb, N, rank, actions, args.steps, 99, None, world,
                              outputs=args.dump_outputs is not None)
    except Exception as e:  # reported, never fatal: the flushed number above does not depend on it
        b2b = dict(error=f"{type(e).__name__}: {e}")

    # ---- env-count sweep: what bounds the step kernel.  Same kernel, same protocol (rotating batches > L2, >= 20 ms
    # regions), N from the headline's 65,536 (0.38 of a wave: one dependency chain) up to 16 Mi envs, where the
    # env-state stream (STEP_IO_BYTES per env-step to and from HBM) is the compulsory traffic.
    sweep = []
    if world == 1 and not args.no_sweep:
        for n_env in (65536, 262144, 1 << 20, 1 << 22, 1 << 24):
            try:
                acts = [torch.randint(0, tb.A, (n_env,), dtype=torch.int32, device="cuda", generator=gen)
                        for _ in range(2)]
                r = _rotating_graph(torch, tb, n_env, rank, acts, 4, 500, 20.0, world)
                sweep.append(dict(n_envs=n_env, ms_per_step=r["ms_per_step"], batches=r["batches"],
                                  timed_steps=r["timed_steps"], region_ms=r["region_ms"]))
                del acts
            except Exception as e:
                sweep.append(dict(n_envs=n_env, error=f"{type(e).__name__}: {e}"))

    # ---- (c) the on-device-agent case: K random-agent steps of every env fused in ONE launch
    # (BaseMDP.random_steps, base.py:1319-1339; bit-identical to K launches)
    fused = None
    try:
        K = 1000
        envf = BatchedMDP(tb, N, mode="dense_f32", seed=4321, env_offset=rank * N)
        envf.reset()
        envf.random_steps_fused(50)
        barrier_sync(world)
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 0
        f0.record()
        while True:
            envf.random_steps_fused(K)
            reps += 1
            f1.record()
            f1.synchronize()
            if f0.elapsed_time(f1) >= 50.0 or reps >= 64:
                break
        barrier_sync(world)
        fused = dict(ms=max_over_ranks(f0.elapsed_time(f1), world), steps=K * reps, per_launch=K)
        assert int(envf.visits_s.sum()) == N * (K * reps + 51)
        del envf
    except Exception as e:
        fused = dict(error=f"{type(e).__name__}: {e}")

    # ---- end to end through the public API: pinned host actions in, TimeStep fields out on the host, every step.
    # host_io=True: the step kernel reads the pinned action buffer and writes obs/reward/step_type into pinned host
    # memory itself (zero-copy over PCIe) -- one launch + one stream sync per step, no copy launches.
    n_e2e = max(args.steps, 4000)  # >= 50 ms of timed region at ~20-30 us per step, whatever --steps says
    env_h = BatchedMDP(tb, N, mode="dense_f32", seed=1234, env_offset=rank * N, host_io=True)
    env_h.reset()
    h_act = [a.cpu().pin_memory() for a in actions]

    def e2e_step(i):
        obs, reward, step_type = env_h.step_host(h_act[i % n_act], auto_reset=True)  # returns after the stream sync:
        # the caller consumes the TimeStep (host views) before choosing the next action

    for i in range(max(3, args.warmup)):
        e2e_step(i)
    barrier_sync(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n_e2e):
        e2e_step(i)
    e1.record()
    barrier_sync(world)
    e2e_ms = max_over_ranks(e0.elapsed_time(e1), world)
    assert int(env_h.status.item()) == 0 and int(env_h.step_type_host.max()) <= 2

    # ---- the same end-to-end step with the batch split into two groups stepped in a software pipeline
    # (PipelinedBatchedMDP): while the host handles group g's TimeStep, the other group's kernel is on PCIe
    pipe = {}
    try:
        from colosseum_b200.batched_mdp import PipelinedBatchedMDP

        G = 2
        env_p = PipelinedBatchedMDP(tb, N, groups=G, mode="dense_f32", seed=1234, env_offset=rank * N)
        env_p.reset()
        p_act = [[a[g * (N // G):(g + 1) * (N // G)].clone().pin_memory() for g in range(G)] for a in h_act]
        for g in range(G):
            env_p.send(g, p_act[0][g])
        for i in range(1, max(3, args.warmup)):
            for g in range(G):
                env_p.recv(g)                       # group g's TimeStep is on the host ...
                env_p.send(g, p_act[i % n_act][g])  # ... its next actions go out
        barrier_sync(world)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.perf_counter()
        e0.record()
        for i in range(n_e2e):                 # K steps of every env: K recv/send rounds per group
            for g in range(G):
                env_p.recv(g)
                env_p.send(g, p_act[i % n_act][g])
        for g in range(G):
            env_p.recv(g)
        e1.record()
        e1.synchronize()
        wall_ms = (time.perf_counter() - w0) * 1e3
        barrier_sync(world)
        # the pipeline lives on two side streams: the events on the default stream bracket the same host interval
        pipe = {"ms": max_over_ranks(max(e0.elapsed_time(e1), wall_ms), world), "groups": G}
        assert all(int(sh.status.item()) == 0 for sh in env_p.shards)
    except Exception as exc:  # keep the single-batch number if the pipelined variant cannot run
        pipe = {"error": repr(exc)[:200]}

    # ---- the same pipeline with the recv/send loop run by the library (colo_env_pipeline_run): what a host agent
    # written against the C ABI gets -- no interpreter between the per-group calls
    native = {}
    try:
        env_n = PipelinedBatchedMDP(tb, N, groups=2, mode="dense_f32", seed=1234, env_offset=rank * N)
        env_n.reset()
        env_n.run_native(p_act, max(3, args.warmup))
        barrier_sync(world)
        w0 = time.perf_counter()
        env_n.run_native(p_act, n_e2e)
        wall_ms = (time.perf_counter() - w0) * 1e3
        barrier_sync(world)
        native = {"ms": max_over_ranks(wall_ms, world), "groups": 2}
        assert all(int(sh.status.item()) == 0 for sh in env_n.shards)
        del env_n
    except Exception as exc:
        native = {"error": repr(exc)[:200]}

    # ---- the two-group pipeline with COMPACT host I/O: actions cross PCIe as uint8 and observations as int16 (the
    # same information in 8 instead of 13 bytes per env-step; BatchedMDP(compact_io=True)), Python loop and native loop
    compact = {}
    try:
        env_c = PipelinedBatchedMDP(tb, N, groups=2, mode="dense_f32", seed=1234, env_offset=rank * N, compact_io=True)
        env_c.reset()
        c_act = [[a.to(torch.uint8).pin_memory() for a in acts] for acts in p_act]
        for g in range(2):
            env_c.send(g, c_act[0][g])
        for i in range(1, max(3, args.warmup)):
            for g in range(2):
                env_c.recv(g)
                env_c.send(g, c_act[i % n_act][g])
        barrier_sync(world)
        w0 = time.perf_counter()
        for i in range(n_e2e):
            for g in range(2):
                env_c.recv(g)
                env_c.send(g, c_act[i % n_act][g])
        for g in range(2):
            env_c.recv(g)
        py_ms = (time.perf_counter() - w0) * 1e3
        barrier_sync(world)
        env_c.run_native(c_act, max(3, args.warmup))
        barrier_sync(world)
        w0 = time.perf_counter()
        env_c.run_native(c_act, n_e2e)
        nat_ms = (time.perf_counter() - w0) * 1e3
        barrier_sync(world)
        assert all(int(sh.status.item()) == 0 for sh in env_c.shards)
        # same trajectories as the int32 pipeline (same seed, same actions, same number of steps so far)
        compact = {"py_ms": max_over_ranks(py_ms, world), "native_ms": max_over_ranks(nat_ms, world), "groups": 2,
                   "h2d": N, "d2h": 7 * N}
        # measured alternatives of the host loop (DESIGN 4.2): stream memory operations instead of sync + launch
        # (one triple at a time / CUDA-graph replays), and one host thread per group
        for key, run in (("queued_stream_memops", lambda k: env_c.run_queued(c_act, k, graph=False)),
                         ("queued_graph_replays", lambda k: env_c.run_queued(c_act, k, graph=True)),
                         ("thread_per_group", lambda k: env_c.run_native(c_act, k, threads=True))):
            try:
                run(max(3, args.warmup))
                barrier_sync(world)
                w0 = time.perf_counter()
                run(n_e2e)
                v_ms = (time.perf_counter() - w0) * 1e3
                barrier_sync(world)
                compact.setdefault("variants", {})[key] = max_over_ranks(v_ms, world)
            except Exception as exc:
                compact.setdefault("variants", {})[key] = repr(exc)[:160]
        assert all(int(sh.status.item()) == 0 for sh in env_c.shards)
        del env_c
    except Exception as exc:
        compact = {"error": repr(exc)[:200]}

    # ---- and through the persistent step server (no launch, no stream sync per step)
    served = {}
    try:
        env_s = BatchedMDP(tb, N, mode="dense_f32", seed=1234, env_offset=rank * N, host_io=True)
        env_s.reset()
        s_buf = h_act[0].clone().pin_memory()
        env_s.serve(s_buf)
        for i in range(max(3, args.warmup)):
            env_s.step_served()
        barrier_sync(world)
        w0 = time.perf_counter()
        for i in range(n_e2e):
            env_s.step_served()
        wall_ms = (time.perf_counter() - w0) * 1e3
        env_s.stop_serving()
        barrier_sync(world)
        served = {"ms": max_over_ranks(wall_ms, world)}
    except Exception as exc:
        served = {"error": repr(exc)[:200]}
    return dict(tb=tb, N=N, ms=ms, launches=launches, e2e_ms=e2e_ms, h2d=4 * N, d2h=9 * N, b2b=b2b, det=det,
                pipe=pipe, served=served, native=native, sweep=sweep, fused=fused, n_e2e=n_e2e, compact=compact)


def bench_agents_gpu(args, rank, world):
    """SURVEY 8(f)-4: N independent (QLearningContinuous agent, env) loops on the C2 MDP, 500 steps per launch"""
    import torch

    import colosseum_b200.agent_loop as al

    try:
        tb = load_c2_tables()
        n_loops, K = 65536, 500
        ag = al.QLearningContinuous(1234, tb, 10 ** 6, n_loops=n_loops, env_offset=rank * n_loops)
        ag.steps(50)
        barrier_sync(world)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ag.steps(K)
        e1.record()
        barrier_sync(world)
        ms = max_over_ranks(e0.elapsed_time(e1), world)
        assert float(ag.cumulative_reward.min()) >= 0.0 and int(ag.N.sum()) == n_loops * (K + 50)
        return {"value": world * n_loops * K / (ms / 1e3), "unit": "agent-steps/s", "loops_per_gpu": n_loops,
                "steps_per_launch": K, "gpu_launches": 1,
                "what": "QLearningContinuous (select action, env step on the reference's sampler tables, model update) "
                        f"for {n_loops} independent loops per GPU on the C2 MDP, one thread per loop, agent tables "
                        f"{n_loops * tb.S * tb.A * 12 / 2**20:.0f} MiB per GPU"}
    except Exception as exc:
        return {"error": repr(exc)[:200]}


def bench_model_based_agents_gpu(args, rank, world):
    """SURVEY 8(f)-1/-4: the model-based continuous agents as device loops, planners included (UCRL2Continuous: batched
    extended VI over the loops whose artificial episode ended; PSRLContinuous: optimistic sampling + batched discounted
    VI) -- 256 loops per GPU on RiverSwimContinuous (tests/golden), wall clock around a synchronised region"""
    import time

    import torch

    import colosseum_b200.agent_loop as al
    from colosseum_b200.tables import MDPTables

    out = {}
    try:
        tb = MDPTables.from_golden(np.load(os.path.join(ROOT, "tests", "golden", "inst_riverswimcontinuous_ergo0.npz")))
        n_loops, T = 256, 10000
        for name, make in (("ucrl2_continuous", lambda: al.UCRL2Continuous(7, tb, 2 * T + 1, alpha_r=0.1, alpha_p=0.05,
                                                                           n_loops=n_loops, env_offset=rank * n_loops)),
                           ("psrl_continuous", lambda: al.PSRLContinuous(7, tb, 2 * T + 1, psi_weight=0.015, eta_weight=1e-9,
                                                                         n_loops=n_loops, env_offset=rank * n_loops))):
            ag = make()
            ag.steps(T)  # the early, planning-heavy phase is the warm-up
            barrier_sync(world)
            t0 = time.perf_counter()
            c0 = float(ag.cumulative_reward.mean())
            ag.steps(T)
            torch.cuda.synchronize()
            dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
            barrier_sync(world)
            secs = max_over_ranks(float(dt.item()), world)
            out[name] = {"value": world * n_loops * T / secs, "unit": "agent-steps/s", "loops_per_gpu": n_loops,
                         "steps": T, "rounds": int(ag.rounds),
                         "reward_rate": (float(ag.cumulative_reward.mean()) - c0) / T,
                         "replannings_per_loop": float(ag.episode.double().mean())}
        out["what"] = ("N independent agent loops on RiverSwimContinuous (S=30, A=2; optimal average reward 0.889), steps "
                       "10,001..20,000 of each loop, planners included; the reference runs ~1e4 agent-steps/s per process")
    except Exception as exc:
        out["error"] = repr(exc)[:200]
    return out


C1_V0 = [0.45454547, 0.36414355, 0.2737823, 0.3346822, 0.4166667]  # SURVEY section 8d, the parity anchor


def bench_c1(args):
    """C1 (BASELINE.json configs[0], the reference's own CPU-runnable case): RiverSwimEpisodic size 5, 10,000
    random-agent steps with auto-reset + episodic_value_iteration(5, T, R).  CPU: the oracle port on ONE host thread
    (the reference is a single Python thread) with the measured Python-reference numbers quoted beside it; GPU: the
    same two calls through the drop-in surface (a single env is the GPU's worst case -- reported, not hidden)."""
    import torch

    import colosseum_b200.dynamic_programming as dp
    from colosseum_b200.batched_mdp import BatchedMDP
    from colosseum_b200.tables import MDPTables
    from oracle import oracle as orc

    g = np.load(os.path.join(ROOT, "tests", "golden", "inst_c1_riverswim_epi.npz"))
    tb = MDPTables.from_golden(g)
    T, R, H = g["T"], g["R"], int(g["H"])
    out = {"workload": "C1 RiverSwimEpisodic(seed=0,size=5,p_lazy=0.1, Beta rewards of the quick-test gin): 10,000 "
                       "random-agent steps with auto-reset (BaseMDP.random_steps) + episodic_value_iteration(5,T,R)"}
    # -- GPU, scalar drop-in: per-call steps (launch + sync per step) and the fused random walk (one launch)
    env = BatchedMDP(tb, 1, mode="succ", seed=0, scalar_api=True)
    env.reset()
    for _ in range(200):
        env.random_step(auto_reset=True)
    t0 = time.perf_counter()
    for _ in range(2000):
        ts, a = env.random_step(auto_reset=True)
    out["gpu_scalar_steps_per_s"] = 2000 / (time.perf_counter() - t0)
    envb = BatchedMDP(tb, 1, mode="succ", seed=0)
    envb.reset()
    envb.random_steps_fused(100)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    envb.random_steps_fused(10000)
    torch.cuda.synchronize()
    out["gpu_fused_10k_steps_per_s"] = 10000 / (time.perf_counter() - t0)
    Q, V = dp.episodic_value_iteration(H, T, R)
    assert np.allclose(V[0], C1_V0, rtol=2e-5), V[0]
    t0 = time.perf_counter()
    for _ in range(200):
        dp.episodic_value_iteration(H, T, R)
    out["gpu_episodic_vi_us"] = (time.perf_counter() - t0) / 200 * 1e6
    out["V0_matches_anchor"] = True
    # -- CPU port, one thread
    orc.set_threads(1)
    ht = orc.HostTables(tb.S, tb.A, H=tb.H, succ_cum=tb.succ_cum, succ_idx=tb.succ_idx, succ_len=tb.succ_len,
                        rew_cls_succ=tb.rew_cls_succ, rew_q=tb.rew_q, rmin=tb.rmin, rmax=tb.rmax,
                        start_cum=tb.start_cum, start_idx=tb.start_idx)
    state, h, st, obs = orc.env_reset(ht, 1, seed=0, t=0)
    t0 = time.perf_counter()
    for t in range(1, 10001):
        orc.env_step(ht, 2, state, h, st, action=None, seed=0, t=t, auto_reset=True)
    out["cpu_port_steps_per_s"] = 10000 / (time.perf_counter() - t0)
    orc.episodic_f32(H, T, R)
    t0 = time.perf_counter()
    for _ in range(2000):
        Qo, Vo = orc.episodic_f32(H, T, R)
    out["cpu_port_episodic_vi_us"] = (time.perf_counter() - t0) / 2000 * 1e6
    assert np.allclose(Vo[0], C1_V0, rtol=2e-6)
    out["cpu_note"] = ("port = C oracle called through ctypes once per step / per VI, one thread (the call overhead "
                       "dominates at this size)" + measured_reference())
    orc.set_threads()
    return out


def make_c4_batch(B, S, A, seed):
    """C4's generator on the device: T[b,s,a,:] ~ Dirichlet(0.05), rows renormalised in fp32; R ~ U[0,1)"""
    import torch

    gen = torch.Generator(device="cuda").manual_seed(seed)
    T = torch.empty((B, S, A, S), dtype=torch.float32, device="cuda")
    chunk = max(1, min(B, 256))
    for b0 in range(0, B, chunk):
        b1 = min(B, b0 + chunk)
        g = torch._standard_gamma(torch.full((b1 - b0, S, A, S), 0.05, device="cuda"), generator=gen) + 1e-30
        T[b0:b1] = g / g.sum(-1, keepdim=True)
    R = torch.rand((B, S, A), device="cuda", generator=gen)
    return T, R


def bench_vi_gpu(args, rank, world):
    """VI sweeps on C4's shape: one step = one synchronous sweep of the whole resident batch (T > L2: no flush)"""
    import torch

    from colosseum_b200 import _cabi
    from colosseum_b200.dynamic_programming import BatchedValueIteration

    B, S, A = (args.vi_batch or max(1, 4096 // world)), 512, 4
    T, R = make_c4_batch(B, S, A, seed=100 + rank)
    vi = BatchedValueIteration(T, R, gamma=0.99, precision="f32")
    lib = _cabi.lib()
    steps = max(5, min(args.steps, 50))
    for _ in range(max(3, args.warmup)):
        vi.sweep()
    barrier_sync(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    lib.colo_reset_launch_count()
    e0.record()
    vi.sweep(steps)
    e1.record()
    barrier_sync(world)
    launches = int(lib.colo_launch_count())
    ms = max_over_ranks(e0.elapsed_time(e1), world)
    # C4 part (2), SURVEY section 8d: solve the whole batch to the reference's default epsilon = 1e-3 through the
    # public entry point (device tensors in, device tensors out; per-instance stopping on the device)
    import colosseum_b200.dynamic_programming as dp

    del vi
    dp.discounted_value_iteration(T[:8], R[:8], 0.99, 1e-3)  # warm-up of the solver path
    barrier_sync(world)
    e0.record()
    Q, V = dp.discounted_value_iteration(T, R, 0.99, 1e-3)
    e1.record()
    barrier_sync(world)
    solve_ms = max_over_ranks(e0.elapsed_time(e1), world)
    iters = dp.last_iterations()
    assert bool(torch.isfinite(V).all())
    # the same solve with the reference's own in-place (Gauss-Seidel) sweeps: one warp per MDP, one launch
    dp.discounted_value_iteration(T[:8], R[:8], 0.99, 1e-3, sweep_order="gauss_seidel")
    barrier_sync(world)
    e0.record()
    Qg, Vg = dp.discounted_value_iteration(T, R, 0.99, 1e-3, sweep_order="gauss_seidel")
    e1.record()
    barrier_sync(world)
    gs_ms = max_over_ranks(e0.elapsed_time(e1), world)
    gs_iters = dp.last_iterations()
    assert bool(torch.isfinite(Vg).all()) and float((Vg - V).abs().max()) < 0.2  # both within eps*gamma/(1-gamma) of V*
    del T, R, Q, V, Qg, Vg
    torch.cuda.empty_cache()
    return dict(B=B, S=S, A=A, steps=steps, ms=ms, launches=launches, solve_ms=solve_ms, solve_sweeps_max=max(iters),
                solve_sweeps_mean=float(np.mean(iters)), gs_ms=gs_ms, gs_sweeps_max=max(gs_iters),
                gs_sweeps_mean=float(np.mean(gs_iters)))


def bench_c5_gpu(args, rank, world):
    """C5: ONE dense synthetic MDP S=40,000 A=8 fp32 (51.2 GB of T), row-sharded over the ranks; every sweep each
    rank backs up its S/g rows and the new V rows are exchanged (fused peer stores, or NCCL all-gather)."""
    import torch

    from colosseum_b200 import _cabi
    from colosseum_b200.dynamic_programming import BatchedValueIteration
    from colosseum_b200.sharded import RowShardedValueIteration, shard_range
    from colosseum_b200.synth import synth_dense_rows

    S, A = args.c5_states, 8
    r0, r1 = shard_range(S, rank, world)
    T_rows, R_rows = synth_dense_rows(r0, r1 - r0, S, A, seed=7)  # generated on the device, never on the host
    if world == 1:
        vi = BatchedValueIteration(T_rows, R_rows, gamma=0.99, precision="f32")
        transport = "none (1 GPU)"
    else:
        transport = args.c5_transport
        try:
            vi = RowShardedValueIteration(T_rows, R_rows, S, gamma=0.99, transport=transport)
            vi.sweep(1)
        except Exception as e:  # symmetric memory unavailable on this box: the NCCL all-gather does the same exchange
            if transport == "nccl":
                raise
            print(f"[bench] fused V exchange unavailable ({type(e).__name__}: {e}); using nccl", file=sys.stderr)
            transport = "nccl (fused unavailable)"
            vi = RowShardedValueIteration(T_rows, R_rows, S, gamma=0.99, transport="nccl")
    lib = _cabi.lib()
    steps = max(5, min(args.steps, 100))
    vi.sweep(3)
    barrier_sync(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    lib.colo_reset_launch_count()
    e0.record()
    vi.sweep(steps)
    e1.record()
    barrier_sync(world)
    launches = int(lib.colo_launch_count())
    ms = max_over_ranks(e0.elapsed_time(e1), world)
    v = vi.values
    assert bool(torch.isfinite(v).all()) and float(v.max()) > 0
    # automated multi-GPU parity: one more sweep of the sharded solver, then 64 fixed rows of it recomputed by a
    # single-rank BatchedValueIteration on this rank's own rows from the same full V_old (rtol 2e-6: a small shard
    # may use another summation order inside a row, DESIGN section 5); AND-ed over the ranks
    v_old = v.clone()
    vi.sweep(1)
    v_new = vi.values.clone()
    nrows = r1 - r0
    pick = torch.unique(torch.linspace(0, nrows - 1, 64, device="cuda").long())
    # the checker: the picked rows as a row block [0, n) of an S-column problem, fed with the same full V_old
    chk = BatchedValueIteration(T_rows[pick].contiguous(), R_rows[pick].contiguous(), gamma=0.99, precision="f32",
                                row0=0, S_total=S)
    chk.values.view(-1).copy_(v_old.view(-1))
    chk.sweep(1)
    ref_rows = chk.values.view(-1)[: pick.numel()]
    got = v_new.view(-1)[r0 + pick]
    err = float(((got - ref_rows).abs() / ref_rows.abs().clamp_min(1e-30)).max())
    ok = err <= 5e-6
    if world > 1:
        import torch.distributed as dist

        t_ok = torch.tensor([1 if ok else 0], device="cuda")
        dist.all_reduce(t_ok, op=dist.ReduceOp.MIN)
        ok = bool(t_ok.item())
        # every rank must also hold the SAME full V (the exchange delivered every shard everywhere)
        cs = torch.stack([v_new.double().sum(), v_new.double().abs().max()])
        lo, hi = cs.clone(), cs.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        ok = ok and bool((lo == hi).all())
    del vi, T_rows, R_rows, chk
    torch.cuda.empty_cache()
    return dict(S=S, A=A, steps=steps, ms=ms, launches=launches, transport=transport, parity_ok=ok, parity_err=err)


def bench_c3_gpu(args, rank, world):
    """C3: the reference's benchmark MDP instances (gin parameter sets of the seven families x seeds 0..10 in the
    order of SURVEY section 8d, cycled to `--c3-instances`), sharded over the ranks by instance, no communication.  Per
    instance: `--c3-envs` parallel episodes x `--c3-steps` random-agent steps through the step kernel, then diameter +
    value norm + gaps.  Runner: colo_suite_run (C++ worker threads, one stream each) or the Python path."""
    import torch

    from colosseum_b200 import _cabi
    from colosseum_b200.sharded import shard_range
    from colosseum_b200.suite import (load_suite_all, longest_first, run_instance, run_many, run_many_native,
                                       shard_instances, suite_costs, suite_size)

    gdir = os.path.join(ROOT, "tests", "golden")
    n_suite = suite_size(gdir)
    B = args.c3_instances
    # the B instances, sorted by decreasing estimated time (suite.instance_cost: a fit of measured instance times, from the
    # fixtures' metadata), are dealt to the ranks in snake order: same count, nearly the same total cost, longest first (a rank's
    # workers pull from one queue, and the most expensive instance is a large part of a 128-instance region)
    my_ids = shard_instances(B, rank, world, costs=suite_costs(gdir))
    i0, i1 = 0, len(my_ids)
    lib = _cabi.lib()
    mine = load_suite_all(gdir, indices=sorted({i % n_suite for i in my_ids}))
    by_index = dict(zip(sorted({i % n_suite for i in my_ids}), mine))
    work = longest_first([(by_index[i % n_suite], 0) for i in my_ids])
    suite = mine
    # one spinning worker per core this rank may use, at most 8 (colo_suite_run spins in cudaStreamSynchronize when it has
    # a core per worker and blocks otherwise; measured on 4 cores: 4 spinning workers 0.29-0.35 s per 128 instances,
    # 8 blocking ones 0.31-0.45 s; on 32 cores 8 spinning workers 0.25 s)
    workers = args.c3_workers or max(2, min(8, len(os.sched_getaffinity(0))))
    native = args.c3_runner == "native" and args.c3_precision == "f64"
    if native:
        # untimed warm-up: one short pass over every distinct (family, size) of the shard, so that module loading and
        # the growth of the memory pool are not inside the timed region
        seen, warm = set(), []
        for inst, sd in work:
            key = (inst.name.split(".")[0], inst.S, inst.H)
            if key not in seen:
                seen.add(key)
                warm.append((inst, sd))
        run_many_native(warm[:48], n_workers=workers, n_envs=args.c3_envs, n_steps=10)
        # ... and one untimed pass over the whole work list in its real order: the workers' buffer caches and the pool
        # reach their steady state only then (measured on 256 instances: passes of 2.3 / 0.64 / 0.47 s without it)
        run_many_native(work, n_workers=workers, n_envs=args.c3_envs, n_steps=10)
    else:
        run_instance(suite[0], n_envs=args.c3_envs, n_steps=10, seed=0, precision=args.c3_precision)
    # the region is a few hundred ms of many small latency-bound solves driven by host threads: it is sensitive to
    # whatever else runs on the host, so the leg is timed `--c3-passes` times (each pass the whole work list, max over
    # ranks) and the line carries the best pass and the list of all of them
    pass_ms, best = [], None
    for _ in range(max(1, args.c3_passes)):
        barrier_sync(world)
        lib.colo_reset_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.perf_counter()
        e0.record()
        if native:
            res_p = run_many_native(work, n_workers=workers, n_envs=args.c3_envs, n_steps=args.c3_steps)
        else:
            res_p = run_many(work, n_workers=workers, n_envs=args.c3_envs, n_steps=args.c3_steps,
                             precision=args.c3_precision)
        e1.record()
        e1.synchronize()
        wall_ms = (time.perf_counter() - w0) * 1e3
        barrier_sync(world)
        pass_ms.append(max_over_ranks(max(e0.elapsed_time(e1), wall_ms), world))
        if best is None or pass_ms[-1] <= min(pass_ms[:-1]):
            best = (res_p, int(lib.colo_launch_count()))
    results, n_launches = best
    step_s = hard_s = 0.0
    worst = (0.0, "")
    # parity: every instance against the answers the unmodified reference recorded for it (NaN = not recorded): its own
    # diameter / value norm / gaps, or the values of its shipped hardness cache (continuous classes)
    bad, checked = [], 0
    for (inst, _), (res, tm) in zip(work, results):
        step_s += tm["step_s"]
        hard_s += tm["hardness_s"]
        if tm["hardness_s"] > worst[0]:
            worst = (tm["hardness_s"], inst.name)
        assert res["gaps"] > 0 and res["diameter"] > 0 and res["visits_total"] == args.c3_envs * (args.c3_steps + 1)
        # tolerances of tests/test_suite.py: the reference's own numbers are early-stopped iterates (eps = 1e-3)
        for k, ref_k, tol, floor in (("diameter", "diameter", 2e-3, 0.0), ("diameter", "cached_diameter", 2e-3, 0.0),
                                     ("value_norm", "value_norm", 5e-3, 0.2), ("value_norm", "cached_value_norm", 5e-3, 0.2),
                                     ("gaps", "gaps", 1.5e-2, 0.0)):
            ref = inst.ref.get(ref_k, float("nan"))
            if ref == ref and res[k] == res[k]:
                checked += 1
                if abs(res[k] - ref) > tol * max(abs(ref), floor, 1e-9):
                    bad.append((inst.name, ref_k, res[k], ref))
    barrier_sync(world)
    if native:
        from colosseum_b200.suite import release_caches

        release_caches()  # the workers' large buffers go back to the pool before the next leg
    ms = min(pass_ms)
    ok = len(bad) == 0
    if world > 1:
        import torch.distributed as dist

        t_ok = torch.tensor([1 if ok else 0, checked], device="cuda")
        dist.all_reduce(t_ok[:1], op=dist.ReduceOp.MIN)
        dist.all_reduce(t_ok[1:], op=dist.ReduceOp.SUM)
        ok, checked = bool(t_ok[0].item()), int(t_ok[1].item())
    if bad:
        print(f"[bench] C3 parity failures on rank {rank}: {bad[:5]}", file=sys.stderr)
    return dict(B=B, per_rank=i1 - i0, ms=ms, pass_ms=pass_ms, launches=n_launches, step_s=step_s, hard_s=hard_s,
                worst=worst, n_suite=n_suite, workers=workers, runner="native (colo_suite_run)" if native else "python",
                parity_ok=ok,
                parity_what=f"{checked} recorded reference answers (diameter 2e-3, value norm 5e-3 of max(ref, 0.2), gaps "
                            "1.5e-2 relative: the reference stops early at eps = 1e-3, DESIGN section 2) checked over "
                            "all ranks")


# ------------------------------------------------------------------------------------------------ CPU arms
def cpu_step_rate(tb, n_envs, seconds):
    """the reference algorithm for the step (oracle port, C + OpenMP, all host threads), bounded sample"""
    from oracle import oracle as orc

    orc.set_threads()
    cdf = orc.build_dense_cdf(tb.T, ld=tb.ld, f64=False)
    ht = orc.HostTables(tb.S, tb.A, H=tb.H, cdf=cdf, rew_cls_sas=tb.rew_cls_sas, rew_q=tb.rew_q, rmin=tb.rmin,
                        rmax=tb.rmax, start_cum=tb.start_cum, start_idx=tb.start_idx)
    state, h, st, obs = orc.env_reset(ht, n_envs, seed=1234, t=0)
    vs = np.zeros(tb.S, np.uint64)
    vsa = np.zeros((tb.S, tb.A), np.uint64)
    t, n = 1, 0
    for _ in range(3):
        orc.env_step(ht, 0, state, h, st, action=None, seed=1234, t=t, auto_reset=True, visits_s=vs, visits_sa=vsa)
        t += 1
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        orc.env_step(ht, 0, state, h, st, action=None, seed=1234, t=t, auto_reset=True, visits_s=vs, visits_sa=vsa)
        t += 1
        n += 1
    dt = time.perf_counter() - t0
    return n * n_envs / dt, n, dt


def cpu_vi_rate(B, S, A, seconds):
    """reference VI iterate (fp32 in-place sweeps, infinite_horizon.py:121-142) over a batch, all host threads"""
    import ctypes as C

    from oracle import oracle as orc

    orc.set_threads()
    rs = np.random.RandomState(0)
    T = rs.dirichlet(np.ones(S) * 0.05, size=(B, S, A)).astype(np.float32)
    R = rs.uniform(0, 1, size=(B, S, A)).astype(np.float32)
    V = np.zeros((B, S), np.float32)
    lib = orc.lib()
    fn = lib.orc_sweeps_gs_f32_batch
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    fn(p(T), p(R), B, S, A, C.c_float(0.99), 2, p(V))
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        fn(p(T), p(R), B, S, A, C.c_float(0.99), 5, p(V))
        n += 5
    dt = time.perf_counter() - t0
    return n * B / dt, n, dt


def measured_reference():
    """the UNMODIFIED Python reference timed once in the build container (profiles/reference_python_timing.json,
    written by scripts/time_reference.py; /root/reference does not exist on the GPU box) -- quoted, never re-run here"""
    p = os.path.join(ROOT, "profiles", "reference_python_timing.json")
    if not os.path.isfile(p):
        return ""
    d = json.load(open(p))
    return (f"; the Python reference itself, measured in the build container on {d['cores_used']} core of "
            f"{d['cpu']}: C1 mdp.random_steps {d['c1_random_steps_per_s']:.3g} steps/s, C2 mdp.step "
            f"{d['c2_step_per_s']:.3g} steps/s, C1 episodic_value_iteration {d['c1_episodic_vi_us']:.1f} us")


def measured_numba():
    p = os.path.join(ROOT, "profiles", "reference_python_timing.json")
    if not os.path.isfile(p):
        return None
    d = json.load(open(p))
    return {"mdp_sweeps_per_s": d.get("c4_numba_mdp_sweeps_per_s"), "solve_ms": d.get("c4_numba_solve_ms"),
            "sweeps": d.get("c4_numba_sweeps"), "cpu": d["cpu"],
            "what": "the reference's own numba _discounted_value_iteration on one S=512 A=4 MDP, one core, measured in "
                    "the build container (scripts/time_reference.py)"}


def run_reference_arm(args):
    """`--impl reference`: the reference's CPU algorithm (oracle port), all host threads, same config/metric"""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    tb = load_c2_tables()
    N = C2_ENVS_PER_GPU
    from oracle import oracle as orc

    cores = orc.set_threads()  # every host core, also under torchrun (which exports OMP_NUM_THREADS=1)

    cdf = orc.build_dense_cdf(tb.T, ld=tb.ld, f64=False)
    ht = orc.HostTables(tb.S, tb.A, H=tb.H, cdf=cdf, rew_cls_sas=tb.rew_cls_sas, rew_q=tb.rew_q, rmin=tb.rmin,
                        rmax=tb.rmax, start_cum=tb.start_cum, start_idx=tb.start_idx)
    state, h, st, obs = orc.env_reset(ht, N, seed=1234, t=0)
    vs = np.zeros(tb.S, np.uint64)
    vsa = np.zeros((tb.S, tb.A), np.uint64)
    t = 1
    steps = min(args.steps, 2000)
    rs = np.random.RandomState(1234)
    acts = [rs.randint(0, tb.A, size=N).astype(np.int32) for _ in range(8)]  # supplied actions, as in the GPU arm
    for i in range(args.warmup):
        orc.env_step(ht, 0, state, h, st, action=acts[i % 8], seed=1234, t=t, auto_reset=True, visits_s=vs, visits_sa=vsa)
        t += 1
    t0 = time.perf_counter()
    for i in range(steps):
        orc.env_step(ht, 0, state, h, st, action=acts[i % 8], seed=1234, t=t, auto_reset=True, visits_s=vs, visits_sa=vsa)
        t += 1
    dt = time.perf_counter() - t0
    value = steps * N / dt
    measured = measured_reference()
    vi_rate, vi_n, vi_dt = cpu_vi_rate(64, 512, 4, 5.0)
    line = {
        "impl": "reference", "metric": "batched env-steps/sec", "value": value, "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": c2_workload(tb.S, tb.A, N),
                   "implementation": "host CPU cores: the reference algorithm as a C+OpenMP port (the reference is "
                                     "single-env Python and has no batched or GPU path); supplied actions, uniforms "
                                     "from the same Philox stream as the GPU arm",
                   "l2": "n/a (host)"},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port",
                         "sample": f"{steps} batched steps of {N} envs, C+OpenMP oracle port of "
                                   "BaseMDP.step/NextStateSampler.sample, supplied actions" + measured},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "vi": {"metric": "value-iteration MDP-sweeps/sec", "value": vi_rate, "unit": "MDP-sweeps/s",
               "sample": f"{vi_n} in-place fp32 sweeps x 64 MDPs (S=512,A=4) in {vi_dt:.1f}s, {cores} threads"},
    }
    emit(line)


# ------------------------------------------------------------------------------------------------ main
def dump_outputs(directory, b2b, rank):
    """`--dump-outputs`: rank 0 writes the arrays of the last timed headline step as <directory>/<name>.npy, float32
    fields as they are and integer fields as float64 (exact below 2**53).  Actions, seeds and step counts depend only on
    the arguments, so two builds run with the same arguments can be compared output for output."""
    if "outputs" not in b2b:
        raise SystemExit(f"--dump-outputs: the headline step leg failed: {b2b.get('error')}")
    outputs = b2b.pop("outputs")
    if rank != 0:
        return
    os.makedirs(directory, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(directory, f"{name}.npy"), a if a.dtype == np.float32 else a.astype(np.float64))


_RESULT_FD = None


def claim_stdout():
    """stdout must carry exactly ONE JSON line: keep a private copy of fd 1 for it and point fd 1 at stderr, so that
    whatever a library prints on stdout (NCCL's version banner under NCCL_DEBUG=VERSION/WARN, ...) lands on stderr"""
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_RESULT_FD, data)


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="all", choices=["all", "step", "vi", "c5", "c3"])
    ap.add_argument("--c3-instances", type=int, default=0,
                    help="MDP instances of the C3 suite leg over all ranks (default: 128 per GPU inside --workload all, "
                         "1,024 for --workload c3)")
    ap.add_argument("--c3-envs", type=int, default=1024)
    ap.add_argument("--c3-steps", type=int, default=1000)
    ap.add_argument("--c3-precision", default="f64", choices=["f64", "f32"])
    ap.add_argument("--c3-passes", type=int, default=3, help="timed passes over the C3 work list (the best one is reported)")
    ap.add_argument("--c3-workers", type=int, default=0,
                    help="host threads (one CUDA stream each) per GPU for the C3 leg (default min(8, cores / GPUs))")
    ap.add_argument("--c3-runner", default="native", choices=["native", "python"])
    ap.add_argument("--vi-batch", type=int, default=0, help="MDP instances per GPU for the C4 leg (default 4096/g)")
    ap.add_argument("--c5-states", type=int, default=40000, help="S of the row-sharded single MDP (C5: 40,000)")
    ap.add_argument("--c5-transport", default="fused", choices=["fused", "nccl"])
    ap.add_argument("--cpu-seconds", type=float, default=8.0)
    ap.add_argument("--no-sweep", action="store_true", help="skip the env-count sweep of the step leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed headline step left in its env batch (TimeStep fields, env state, "
                         "visitation counts; rank 0) as DIR/<name>.npy, to compare builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.impl != "b200" or args.workload not in ("all", "step")):
        ap.error("--dump-outputs needs the headline step leg (--impl b200, --workload all or step)")
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        run_reference_arm(args)
        return

    if args.gpus > 1 and "RANK" not in os.environ:
        # convenience: re-launch under torchrun, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))

    import torch

    from colosseum_b200 import _cabi

    _cabi.require_cuda()  # fails loudly without the CUDA library / a GPU: there is no fallback
    rank, world, local = dist_setup(args.gpus)
    if world > 1:  # give every rank its own slice of the host cores (the e2e host loops otherwise migrate and collide)
        try:
            cores = sorted(os.sched_getaffinity(0))
            per = max(1, len(cores) // world)
            os.sched_setaffinity(0, set(cores[local * per:(local + 1) * per]) or set(cores))
        except Exception:
            pass
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    step = bench_step_gpu(args, rank, world) if args.workload in ("all", "step") else None
    vi = bench_vi_gpu(args, rank, world) if args.workload in ("all", "vi") else None
    c5 = bench_c5_gpu(args, rank, world) if args.workload in ("all", "c5") else None
    if args.workload == "all":  # bounded C3 leg inside the default run: 128 instances per GPU
        args.c3_instances = args.c3_instances or 128 * world
    elif not args.c3_instances:
        args.c3_instances = 1024
    c3 = bench_c3_gpu(args, rank, world) if args.workload in ("all", "c3") else None
    c1 = bench_c1(args) if args.workload == "all" and world == 1 and rank == 0 else None
    agents = bench_agents_gpu(args, rank, world) if args.workload == "all" else None
    if agents is not None:
        agents["model_based"] = bench_model_based_agents_gpu(args, rank, world)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs is not None:  # after the sampler's nvidia-smi child has been stopped: it may exit here
        dump_outputs(args.dump_outputs, step["b2b"], rank)
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peaks()
    line = {"n_gpus": world, "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "clocks": clocks}
    c3_line = None
    if c3 is not None:
        sec = c3["ms"] / 1e3
        c3_line = {
            "metric": "benchmark-suite MDP instances/sec (batched step + hardness measures)", "value": c3["B"] / sec,
            "unit": "instances/s", "steps": c3["B"], "ms_per_step": 1e3 * sec / c3["B"], "scaling": "strong",
            "gpu_launches": c3["launches"], "dtype": args.c3_precision, "timed_region_s": sec,
            "passes_s": [m / 1e3 for m in c3["pass_ms"]],
            "config": {"workload": f"C3: {c3['B']} MDP instances = the first {c3['B']} of the reference's {c3['n_suite']} "
                                   f"benchmark instances (the gin parameter sets of the 7 families, continuous + episodic, "
                                   f"x seeds 0..10, seed-major; tests/golden/c3_suite*.npz), {c3['per_rank']} per GPU; per "
                                   f"instance {args.c3_envs} envs x {args.c3_steps} random-agent steps, then diameter + "
                                   "value norm + sub-optimality gaps (MiniGrid DoorKey is not in the reference); "
                                   f"runner: {c3['runner']}, {c3['workers']} worker threads per GPU",
                       "rank0_seconds": {"step_phase": c3["step_s"], "hardness_phase": c3["hard_s"],
                                         "slowest_instance": c3["worst"][1], "slowest_hardness_s": c3["worst"][0]}},
            "env_steps_per_s_step_phase": c3["per_rank"] * args.c3_envs * args.c3_steps / max(c3["step_s"], 1e-9) * world,
            "parity_ok": c3.get("parity_ok"), "parity_what": c3.get("parity_what"),
        }
        if args.workload == "c3":
            line.update(c3_line)
            emit(line)
            if world > 1:
                import torch.distributed as dist

                dist.destroy_process_group()
            return
    c5_line = None
    if c5 is not None:
        S5, A5 = c5["S"], c5["A"]
        sec = c5["ms"] / 1e3 / c5["steps"]
        rows = -(-S5 // world)  # rows of the largest shard
        per_rank_bytes = 4 * rows * A5 * S5 + 4 * rows * A5 + 4 * S5 + 4 * rows + 4 * rows * A5
        c5_line = {
            "metric": "row-sharded value-iteration sweeps/sec (one dense MDP)", "value": 1.0 / sec, "unit": "sweeps/s",
            "steps": c5["steps"], "ms_per_step": 1e3 * sec, "gpu_launches": c5["launches"], "scaling": "strong",
            "parity_ok": c5["parity_ok"], "parity_max_rel_err": c5["parity_err"],
            "parity_what": "after the timed sweeps: one more sharded sweep, 64 fixed rows per rank recomputed by a "
                           "single-rank BatchedValueIteration from the same full V_old (rtol 5e-6), AND over ranks; all "
                           "ranks hold the same full V (sum / max equal across ranks)",
            "config": {"workload": f"C5: one synthetic dense MDP S={S5} A={A5} fp32 (T = {4 * S5 * A5 * S5 / 1e9:.1f} GB "
                                   f"generated on device), gamma=0.99, rows sharded over {world} GPU(s), V exchange: "
                                   f"{c5['transport']}", "l2": "T per GPU >> 126 MB L2, no flush"},
            "roofline": {"bound": "hbm", "achieved": per_rank_bytes / sec / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": per_rank_bytes / sec / 1e9 / peak, "traffic": ncu_traffic("backup_c5", rows * A5 * S5),
                         "peak_source": peak_src,
                         "kernel": "backup_kernel<float,MAX,VEC,warp>", "algorithmic_bytes_per_launch": per_rank_bytes,
                         "note": "per-GPU figure: bytes of the largest row shard / sweep time (max over ranks)"},
        }
    if vi is not None:
        per_sweep_bytes = vi_sweep_bytes(vi["S"], vi["A"]) * vi["B"]
        sec = vi["ms"] / 1e3 / vi["steps"]
        vi_line = {
            "metric": "value-iteration MDP-sweeps/sec", "value": world * vi["B"] / sec, "unit": "MDP-sweeps/s",
            "steps": vi["steps"], "ms_per_step": 1e3 * sec, "gpu_launches": vi["launches"],
            "scaling": "strong" if not args.vi_batch else "weak",
            "solve_to_eps": {"epsilon": 1e-3, "seconds": vi["solve_ms"] / 1e3, "sweeps_max": vi["solve_sweeps_max"],
                             "sweeps_mean": vi["solve_sweeps_mean"],
                             "mdp_solves_per_s": world * vi["B"] / (vi["solve_ms"] / 1e3),
                             "what": "dp.discounted_value_iteration(T, R, 0.99, 1e-3) on the whole batch, device "
                                     "tensors in/out, per-instance stopping on the device"},
            "solve_to_eps_gauss_seidel": {
                "epsilon": 1e-3, "seconds": vi["gs_ms"] / 1e3, "sweeps_max": vi["gs_sweeps_max"],
                "sweeps_mean": vi["gs_sweeps_mean"], "mdp_solves_per_s": world * vi["B"] / (vi["gs_ms"] / 1e3),
                "t_stream_gbs": vi["gs_sweeps_mean"] * 4 * vi["S"] * vi["A"] * vi["S"] * vi["B"] / (vi["gs_ms"] / 1e3) / 1e9,
                "what": "the same solve with sweep_order='gauss_seidel': the reference's own in-place iterate "
                        "(infinite_horizon.py:131-135), one warp per MDP, the whole solve in one launch"},
            "config": {"workload": f"C4: {world * vi['B']} synthetic Dirichlet(0.05) MDPs ({vi['B']} per GPU), S=512 A=4 fp32, "
                                   "gamma=0.99, one synchronous sweep of the whole batch per step, Q stored",
                       "l2": f"batch T = {vi['B'] * 4 * 512 * 4 * 512 / 2**30:.1f} GiB per GPU >> 126 MB L2, no flush"},
            "roofline": {"bound": "hbm", "achieved": per_sweep_bytes / sec / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": per_sweep_bytes / sec / 1e9 / peak, "traffic": ncu_traffic("backup_c4", vi["B"]),
                         "peak_source": peak_src, "kernel": "backup_kernel<float,MAX,VEC,warp>",
                         "algorithmic_bytes_per_launch": per_sweep_bytes},
        }
    if step is not None:
        tb, N = step["tb"], step["N"]
        sec_flushed = step["ms"] / 1e3 / args.steps
        b2b = step.get("b2b") or {}
        flushed_note = "L2 flushed between timed steps (256 MiB write), each step timed with its own CUDA-event pair"
        if "ms_per_step" in b2b:
            # headline protocol: inputs larger than L2 instead of a flush -- step i runs on env batch i % NB, every batch
            # with its own tables, the K steps captured in one CUDA graph and timed over one replay
            sec = b2b["ms_per_step"] / 1e3
            nb, mib = b2b["batches"], b2b["batch_bytes"] / 2**20
            l2_note = (f"no flush: step i runs on env batch i % {nb} ({nb} independent batches of {N} envs, each with its "
                       f"own tables, {mib:.1f} MiB each); the {b2b['timed_steps']} steps of --steps captured in one CUDA "
                       f"graph and timed over one replay inside ONE CUDA-event pair, enqueued right behind "
                       f"{b2b['lead_in_steps']} untimed steps that step the {nb} batches in order, so each timed step's "
                       f"batch was last stepped {nb - 1} batches ({(nb - 1) * mib:.0f} MiB > 126 MB L2) earlier; the "
                       f"timed steps touch {b2b['timed_bytes'] / 2**20:.0f} MiB in a {b2b['region_ms']:.3f} ms region "
                       "(one replay: noisier than a long region, a larger --steps gives a steadier number)")
            launches, region_s = b2b["timed_steps"], b2b["region_ms"] / 1e3
        else:
            sec, l2_note, launches, region_s = sec_flushed, flushed_note, step["launches"], step["ms"] / 1e3
        io_bytes = STEP_IO_BYTES * N
        # the sweep names the bound: per N, env-steps/s and the env-state stream in GB/s against the HBM peak
        sweep_out, sat = [], None
        for e in step.get("sweep") or []:
            if "error" in e:
                sweep_out.append(e)
                continue
            t = e["ms_per_step"] / 1e3
            row = {"n_envs": e["n_envs"], "us_per_step": 1e6 * t, "env_steps_per_s": e["n_envs"] / t,
                   "state_stream_gbs": STEP_IO_BYTES * e["n_envs"] / t / 1e9,
                   "frac_of_hbm_peak": STEP_IO_BYTES * e["n_envs"] / t / 1e9 / peak,
                   "waves": e["n_envs"] / (148 * 2048), "timed_steps": e["timed_steps"], "region_ms": e["region_ms"]}
            sweep_out.append(row)
            if sat is None or row["env_steps_per_s"] > sat["env_steps_per_s"]:
                sat = row
        line.update({
            "metric": "batched env-steps/sec", "value": world * N / sec, "unit": "env-steps/s", "steps": args.steps,
            "ms_per_step": 1e3 * sec, "gpu_launches": launches, "timed_region_s": region_s,
            "config": {"workload": c2_workload(tb.S, tb.A, N),
                       "implementation": "B200: one thread per env, three-round k-ary search of the dense CDF row through "
                                         "its two-level index (cdf_coarse / cdf_mid), supplied actions, in-kernel Philox "
                                         "uniforms",
                       "l2": l2_note},
            "flushed_per_step": {"value": world * N / sec_flushed, "unit": "env-steps/s", "ms_per_step": 1e3 * sec_flushed,
                                 "what": flushed_note + " (the event pair alone costs ~10 us on this GPU: a floor, not "
                                         "the kernel)"},
            "e2e": {"value": world * N * step["n_e2e"] / (step["e2e_ms"] / 1e3), "unit": "env-steps/s",
                    "h2d_bytes_per_step": step["h2d"], "d2h_bytes_per_step": step["d2h"], "timed_steps": step["n_e2e"],
                    "timed_region_s": step["e2e_ms"] / 1e3,
                    "what": "BatchedMDP(host_io=True).step_host: pinned host actions read, and obs/reward/step_type "
                            "written to pinned host memory, by the step kernel itself over PCIe (zero-copy), then a "
                            "stream sync, every step"},
            # NOT an HBM achievement at this size: 65,536 envs are a fraction of a wave (ncu: 0.22 waves/SM) of one-thread-per-env work and the
            # 2.9 MB of tables live in L1/L2, so a step is ONE env's dependency chain (env scalars -> coarse index ->
            # mid index + reward classes -> crossing quad -> reward quantiles), not a stream.  `achieved` is the
            # env-state stream the launch really has to move (STEP_IO_BYTES per env-step); `at_saturation` is the same
            # kernel at the env count where that stream is what it waits for.
            "roofline": {"bound": "latency", "achieved": io_bytes / sec / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": io_bytes / sec / 1e9 / peak, "traffic": ncu_traffic("step", N),
                         "peak_source": peak_src, "kernel": "env_step_kary_lean_kernel<4>",
                         "algorithmic_bytes_per_launch": io_bytes,
                         "algorithmic_bytes_per_env_step": STEP_IO_BYTES,
                         "nominal_bytes_per_env_step_survey_8d": STEP_BYTES(tb.S),
                         "limiter": "dependent-load latency of one env's chain (4 L2/L1 round trips) plus the graph-node "
                                    "launch; 0.22 waves per SM at 65,536 envs (ncu) -- see `env_sweep` for the throughput regime",
                         "at_saturation": None if sat is None else {
                             "n_envs": sat["n_envs"], "env_steps_per_s": sat["env_steps_per_s"],
                             "bound": "issue",
                             "hbm_stream": {"achieved": sat["state_stream_gbs"], "peak": peak, "unit": "GB/s",
                                            "frac": sat["frac_of_hbm_peak"]},
                             "evidence": step_ncu_evidence(),
                             "note": "once the batch fills the machine the kernel is bound by instruction issue, not by "
                                     "memory: Philox4x32-10 (~65 instructions per env) plus the 27 comparisons of the "
                                     "k-ary search and the epilogue are ~330 warp instructions per env-step, and the "
                                     "env-state stream (the only compulsory HBM traffic; the 3 table sectors per env "
                                     "come from L1/L2) reaches the fraction of the HBM peak given in `hbm_stream`"}},
            "env_sweep": sweep_out,
        })
        fused = step.get("fused") or {}
        if "ms" in fused:
            line["fused_random_walk"] = {
                "value": world * N * fused["steps"] / (fused["ms"] / 1e3), "unit": "env-steps/s",
                "steps_per_launch": fused["per_launch"], "timed_region_s": fused["ms"] / 1e3,
                "what": "BaseMDP.random_steps(n) for every env in ONE launch per 1000 steps (the on-device-agent case: "
                        "no launch between steps, env state in registers); bit-identical to n single-step launches"}
        elif "error" in fused:
            line["fused_random_walk"] = {"error": fused["error"]}
        single = line["e2e"]
        pipe, served = step.get("pipe") or {}, step.get("served") or {}
        if "ms" in pipe:
            v = world * N * step["n_e2e"] / (pipe["ms"] / 1e3)
            line["e2e_single_batch"] = single
            if v > single["value"]:
                line["e2e"] = {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": step["h2d"],
                               "d2h_bytes_per_step": step["d2h"], "timed_steps": step["n_e2e"],
                               "timed_region_s": pipe["ms"] / 1e3,
                               "what": f"PipelinedBatchedMDP(groups={pipe['groups']}): the same batch as {pipe['groups']} "
                                       "host_io groups on their own streams; per group and step: recv (stream sync, "
                                       "TimeStep in pinned host memory) then send (launch reading the pinned actions); "
                                       "every env steps once per step, all bytes cross PCIe inside the timed region"}
            else:
                line["e2e_pipelined"] = {"value": v, "unit": "env-steps/s", "groups": pipe["groups"]}
        elif "error" in pipe:
            line["e2e_pipelined"] = {"error": pipe["error"]}
        nat = step.get("native") or {}
        if "ms" in nat:
            v = world * N * step["n_e2e"] / (nat["ms"] / 1e3)
            rec = {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": step["h2d"], "d2h_bytes_per_step": step["d2h"],
                   "timed_steps": step["n_e2e"], "timed_region_s": nat["ms"] / 1e3,
                   "what": f"PipelinedBatchedMDP(groups={nat['groups']}).run_native: the same two-group pipeline with the "
                           "recv/send loop inside the library (colo_env_pipeline_run: per group and step one stream "
                           "sync, then one launch reading the pinned actions), wall clock; every env steps once per "
                           "step, all bytes cross PCIe inside the timed region"}
            if v > line["e2e"]["value"]:
                line["e2e_python_loop"] = line["e2e"]
                line["e2e"] = rec
            else:
                line["e2e_native_loop"] = rec
        elif "error" in nat:
            line["e2e_native_loop"] = {"error": nat["error"]}
        cpt = step.get("compact") or {}
        if "py_ms" in cpt:
            best_ms, how = min((cpt["py_ms"], "driven from Python (recv / send per group)"),
                               (cpt["native_ms"], "with the recv/send loop inside the library (colo_env_pipeline_run)"))
            v = world * N * step["n_e2e"] / (best_ms / 1e3)
            rec = {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": cpt["h2d"], "d2h_bytes_per_step": cpt["d2h"],
                   "timed_steps": step["n_e2e"], "timed_region_s": best_ms / 1e3,
                   "python_loop_value": world * N * step["n_e2e"] / (cpt["py_ms"] / 1e3),
                   "native_loop_value": world * N * step["n_e2e"] / (cpt["native_ms"] / 1e3),
                   "what": "PipelinedBatchedMDP(groups=2, compact_io=True) " + how + ": pinned host actions in as uint8, "
                           "TimeStep out into pinned host memory as reward f32 | observation int16 (-1 = terminal) | "
                           "step_type u8 -- the same information in 8 instead of 13 bytes per env-step; every env steps "
                           "once per step, all bytes cross PCIe inside the timed region, wall clock"}
            if cpt.get("variants"):
                rec["host_loop_variants"] = {
                    k: (world * N * step["n_e2e"] / (ms / 1e3) if isinstance(ms, float) else ms)
                    for k, ms in cpt["variants"].items()}
                rec["host_loop_variants"]["what"] = (
                    "env-steps/s of the same compact two-group pipeline with (a) the group-step handshake done by the GPU "
                    "front end (cuStreamWaitValue32 -> kernel -> cuStreamWriteValue32 on pinned flags, enqueued ahead; "
                    "colo_env_pipeline_run_queued), one triple at a time and as replayed CUDA graphs of 64 steps, and (b) "
                    "one host thread per group (colo_env_pipeline_run_threads); bit-identical TimeSteps, reported as "
                    "measured alternatives")
            if v > line["e2e"]["value"]:
                line["e2e_int32_io"] = line["e2e"]
                line["e2e"] = rec
            else:
                line["e2e_compact_io"] = rec
        elif "error" in cpt:
            line["e2e_compact_io"] = {"error": cpt["error"]}
        if "ms" in served:
            line["e2e_served"] = {"value": world * N * step["n_e2e"] / (served["ms"] / 1e3), "unit": "env-steps/s",
                                  "what": "BatchedMDP.serve(): persistent step kernel driven by a doorbell in pinned "
                                          "host memory (no launch / stream sync per step), wall clock"}
        elif "error" in served:
            line["e2e_served"] = {"error": served["error"]}
        det = step.get("det") or {}
        if "ms" in det:
            line["p_rand_none"] = {"value": world * N * det["steps"] / (det["ms"] / 1e3), "unit": "env-steps/s",
                                   "steps": det["steps"],
                                   "what": "same kernel on DeepSeaContinuous(size=30, p_rand=None): deterministic rows; L2-flush protocol, compare with `flushed_per_step`"}
        elif "error" in det:
            line["p_rand_none"] = {"error": det["error"]}
        if "error" in b2b:
            line["back_to_back"] = {"error": b2b["error"]}
        if world == 1:
            rate, n, dt = cpu_step_rate(tb, N, args.cpu_seconds)
            line["cpu_baseline"] = {"value": rate, "unit": "env-steps/s", "cores": os.cpu_count(), "kind": "port",
                                    "sample": f"{n} batched steps of {N} envs in {dt:.1f}s (C+OpenMP oracle port of "
                                              "BaseMDP.step, in-oracle random actions)" + measured_reference()}
        if vi is not None:
            line["vi"] = vi_line
        if c5_line is not None:
            line["vi_c5"] = c5_line
    elif vi is not None:
        line.update(vi_line)
        if c5_line is not None:
            line["vi_c5"] = c5_line
    else:
        line.update(c5_line)
    if vi is not None and world == 1:
        rate, n, dt = cpu_vi_rate(64, 512, 4, args.cpu_seconds)
        tgt = line["vi"] if step is not None else line
        tgt["cpu_baseline"] = {"value": rate, "unit": "MDP-sweeps/s", "cores": os.cpu_count(), "kind": "port",
                               "reference_numba_1core": measured_numba(),
                               "sample": f"{n} in-place fp32 sweeps x 64 MDPs (S=512,A=4) in {dt:.1f}s (C+OpenMP port "
                                         "of _discounted_value_iteration's sweep, row products as SIMD reductions like "
                                         "the BLAS sgemv behind the reference's T[s] @ V)"}
    if agents is not None:
        line["agents"] = agents
    if c3_line is not None:
        line["c3"] = c3_line
    if c1 is not None:
        line["c1"] = c1
    emit(line)
    if world > 1:
        import torch.distributed as dist

        dist.destroy_process_group()


if __name__ == "__main__":
    main()
