"""GPU: the launch overlap of the lean step kernels (colo_set_step_overlap, DESIGN 4.2) changes no result.

With the overlap on, a lean step launches with programmatic dependent launch: its grid may become resident, and
prefetch into L2, while the work ahead of it on the stream still runs.  Every case runs the same steps with the switch
off and on, in one process, and compares every TimeStep field (step_type, reward bits, discount, observation), the
env state (state, h) and both visitation tables bit for bit.  Each case also checks which kernel served the steps
(colo_step_kernel_launches) and how many launches carried the attribute (colo_step_overlap_launches).

(a) back-to-back steps of one batch, eager and captured in one CUDA graph, on the breakpoint table and with it nulled
    (the k-ary lean kernel), at N = 1, 37 (one partial CTA), 4,099 (a partial last CTA), 65,536 and 300,001 (a grid
    above the prefetch's limit: the overlapped launch takes the kernel without the prefetch);
(b) each step preceded on the same stream by PyTorch kernels that rewrite the action tensor in place, and every 7th
    step by in-place writes of state and h: a lean kernel that read any of them before its wait would see stale data;
(c) the benchmark's pattern: one graph stepping 5 batches in rotation, replayed;
(d) host-I/O and compact-I/O steppers through run_native, whose launches follow a host synchronisation and never
    carry the attribute;
(e) the queued pipeline, whose launches follow stream memory operations and never carry the attribute either, against
    the sync + launch pipeline.
"""
import numpy as np
import pytest

from conftest import load_instance
from colosseum_b200 import _cabi
from colosseum_b200.tables import MDPTables

pytestmark = pytest.mark.gpu

LEAN, BREAKS = 0, 7  # COLO_STEP_KIND_* of include/colosseum_b200.h
N_KINDS = 9
STEPS = 300


@pytest.fixture(scope="module")
def c2():
    return MDPTables.from_golden(load_instance("c2_deepsea30_prand"))


def kinds():
    return np.array([_cabi.lib().colo_step_kernel_launches(k) for k in range(N_KINDS)], np.int64)


def counters():
    return kinds(), int(_cabi.lib().colo_step_overlap_launches())


def launched(before):
    k0, o0 = before
    k1, o1 = counters()
    return k1 - k0, o1 - o0


class Overlap:
    """sets the process-wide switch for a block and restores it"""

    def __init__(self, on):
        self.on = on

    def __enter__(self):
        self.prev = _cabi.lib().colo_set_step_overlap(int(self.on))

    def __exit__(self, *exc):
        assert _cabi.lib().colo_set_step_overlap(self.prev) == int(self.on)


def snapshot(env):
    import torch

    torch.cuda.synchronize()
    return {"state": env.state.clone(), "h": env.h.clone(), "step_type": env.step_type.clone(), "obs": env.obs.clone(),
            "reward_bits": env.reward.view(torch.int32).clone(), "discount_bits": env.discount.view(torch.int32).clone(),
            "visits_s": env.visits_s.clone(), "visits_sa": env.visits_sa.clone()}


def assert_same(a, b, what):
    import torch

    for k in a:
        assert torch.equal(a[k], b[k]), (what, k)


def make_env(tb, N, table, seed=17):
    from colosseum_b200.batched_mdp import BatchedMDP

    env = BatchedMDP(tb, N, mode="dense_f32", seed=seed)
    if not table:
        env.dev.c.cdf_breaks, env.dev.c.cdf_breaks_k = None, 0
    env.reset()
    return env


def actions(tb, N, n, seed):
    import torch

    gen = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.randint(0, tb.A, (N,), dtype=torch.int32, device="cuda", generator=gen) for _ in range(n)]


def run_steps(env, steps, graph, before_step=None):
    """steps auto-resetting steps of env with supplied actions; before_step(i) enqueues work ahead of step i"""
    import torch

    def body():
        for i in range(steps):
            a = before_step(i) if before_step else env._acts[i % len(env._acts)]
            env.step_async(a, auto_reset=True)

    if graph:
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            body()
        g.replay()
    else:
        body()
    torch.cuda.synchronize()
    assert int(env.status.item()) == 0


@pytest.mark.parametrize("N", [1, 37, 4099, 65536, 300001])
@pytest.mark.parametrize("table", [True, False], ids=["breaks", "kary"])
@pytest.mark.parametrize("graph", [False, True], ids=["eager", "graph"])
def test_back_to_back_steps(c2, N, table, graph):
    kind = BREAKS if table else LEAN
    out = {}
    for on in (False, True):
        with Overlap(on):
            env = make_env(c2, N, table)
            env._acts = actions(c2, N, 3, seed=N)
            before = counters()
            run_steps(env, STEPS, graph)
            dk, do = launched(before)
            out[on] = snapshot(env)
        assert dk[kind] == STEPS and dk.sum() == STEPS, dk
        assert do == (STEPS if on else 0)
    assert_same(out[False], out[True], (N, table, graph))


@pytest.mark.parametrize("N", [37, 65536])
@pytest.mark.parametrize("graph", [False, True], ids=["eager", "graph"])
def test_steps_behind_writes_of_their_inputs(c2, N, graph):
    import torch

    out = {}
    for on in (False, True):
        with Overlap(on):
            env = make_env(c2, N, True)
            act = actions(c2, N, 1, seed=3)[0]

            def before_step(i, env=env, act=act):
                act.mul_(7).add_(i).remainder_(c2.A)  # rewrites the step's actions in place on the same stream
                if i % 7 == 6:
                    env.state.add_(1).remainder_(c2.S)
                    env.h.add_(1)
                return act

            before = counters()
            run_steps(env, STEPS, graph, before_step)
            dk, do = launched(before)
            out[on] = snapshot(env)
            out[on]["act"] = act.clone()
        assert dk[BREAKS] == STEPS and dk.sum() == STEPS, dk
        assert do == (STEPS if on else 0)
    torch.cuda.synchronize()
    assert_same(out[False], out[True], (N, graph))


def test_rotating_batches_in_one_graph(c2):
    import torch

    NB, per_graph, N = 5, 40, 4099
    out = {}
    for on in (False, True):
        with Overlap(on):
            envs = [make_env(c2, N, True, seed=99 + i) for i in range(NB)]
            acts = actions(c2, N, 2, seed=5)
            torch.cuda.synchronize()
            before = counters()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for i in range(per_graph):
                    envs[i % NB].step_async(acts[i % 2], auto_reset=True)
            for _ in range(3):
                g.replay()
            torch.cuda.synchronize()
            dk, do = launched(before)
            out[on] = [snapshot(e) for e in envs]
        assert dk[BREAKS] == per_graph and dk.sum() == per_graph, dk
        assert do == (per_graph if on else 0)
    for i in range(NB):
        assert_same(out[False][i], out[True][i], i)


def _pipelined(tb, N, G, compact, seed=21):
    from colosseum_b200.batched_mdp import PipelinedBatchedMDP

    env = PipelinedBatchedMDP(tb, N, groups=G, seed=seed, compact_io=compact)
    env.reset()
    return env


def _ring(env, tb, n=4, seed=5):
    import torch

    gen = torch.Generator().manual_seed(seed)
    return [[torch.randint(0, tb.A, (k,), dtype=torch.int32, generator=gen).to(env.shards[0].action_dtype).pin_memory()
             for k in env.sizes] for _ in range(n)]


def _assert_same_pipelines(a, b, outs_a, outs_b, what):
    import torch

    for k in range(len(outs_a)):
        for x, y in zip(outs_a[k], outs_b[k]):
            assert np.array_equal(x.numpy(), y.numpy(), equal_nan=True), (what, k)
        assert torch.equal(a.shards[k].state, b.shards[k].state) and torch.equal(a.shards[k].h, b.shards[k].h), (what, k)
    assert torch.equal(a.get_visitation_counts(False), b.get_visitation_counts(False)), what


@pytest.mark.parametrize("compact", [False, True], ids=["host_io", "compact_io"])
def test_native_host_loop_never_overlaps(c2, compact):
    N, G, K = 6000 + 5, 3, 50
    envs, outs = {}, {}
    for on in (False, True):
        with Overlap(on):
            envs[on] = _pipelined(c2, N, G, compact)
            ring = _ring(envs[on], c2)
            before = counters()
            outs[on] = envs[on].run_native(ring, K)
            dk, do = launched(before)
        assert dk[BREAKS] == K * G and dk.sum() == K * G, dk
        assert do == 0
    _assert_same_pipelines(envs[False], envs[True], outs[False], outs[True], compact)


@pytest.mark.parametrize("graph", [False, True], ids=["queued", "queued_graphs"])
def test_queued_pipeline_never_overlaps(c2, graph):
    from colosseum_b200._cabi import ColosseumB200Error

    N, G, K = 6000 + 5, 3, 64 + 17
    ref = _pipelined(c2, N, G, False)
    ring = _ring(ref, c2)
    with Overlap(True):
        outs_ref = ref.run_native(ring, K)
        env = _pipelined(c2, N, G, False)
        before = counters()
        try:
            outs = env.run_queued(ring, K, graph=graph)
        except ColosseumB200Error as exc:
            # the library's watchdog: the driver mapped the groups' streams onto one hardware queue (see
            # test_gpu_step.test_queued_pipeline_is_identical) -- a property of the box, not of the overlap
            if "no progress" in str(exc):
                pytest.skip(str(exc))
            raise
        dk, do = launched(before)
    assert dk[BREAKS] > 0 and dk.sum() == dk[BREAKS], dk
    assert do == 0
    _assert_same_pipelines(ref, env, outs_ref, outs, graph)
