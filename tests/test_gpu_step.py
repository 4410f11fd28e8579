"""GPU parity: the batched interaction step (BaseMDP.reset/step, colosseum/mdp/base.py:1268-1317).

Bit-exact bar (BASELINE.json north_star): next-state / observation / step-type / h / visitation results are
identical to the reference's inverse-CDF given identical supplied uniforms -- checked (i) against trajectories
recorded from the reference itself (successor-order tables), (ii) against CPython random.choices draws, and
(iii) against the CPU oracle for the dense kernels and the built-in Philox stream; plus a chi-square test of the
sampled frequencies against T."""
import numpy as np
import pytest

from conftest import CONTINUOUS, EPISODIC, load_instance
from colosseum_b200.tables import MDPTables
from oracle import oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def bm():
    import colosseum_b200.batched_mdp as bm

    return bm


def host_tables(tb, mode, cdf=None):
    if mode == 2:
        return orc.HostTables(tb.S, tb.A, H=tb.H, succ_cum=tb.succ_cum, succ_idx=tb.succ_idx, succ_len=tb.succ_len,
                              rew_cls_succ=tb.rew_cls_succ, rew_q=tb.rew_q, rmin=tb.rmin, rmax=tb.rmax,
                              start_cum=tb.start_cum, start_idx=tb.start_idx)
    return orc.HostTables(tb.S, tb.A, H=tb.H, cdf=cdf, rew_cls_sas=tb.rew_cls_sas, rew_cls_sa=tb.rew_cls_sa,
                          rew_q=tb.rew_q, rmin=tb.rmin, rmax=tb.rmax, start_cum=tb.start_cum, start_idx=tb.start_idx)


@pytest.mark.parametrize("name", CONTINUOUS + EPISODIC)
def test_reference_trajectory_replay(bm, name):
    """the reference's own reset/step trajectory (auto_reset=True), replayed with the uniforms its samplers
    consumed, 3 identical envs in parallel: every TimeStep field and the visitation counts are identical."""
    g = load_instance(name)
    tb = MDPTables.from_golden(g)
    N = 3
    env = bm.BatchedMDP(tb, N, mode="succ")
    acts, us = g["traj_action"], np.nan_to_num(g["traj_u"], nan=0.5)
    ts = env.reset(u_next=np.full(N, us[0]))
    assert (ts.step_type.cpu().numpy() == g["traj_step_type"][0]).all()
    assert (ts.observation.cpu().numpy() == g["traj_obs"][0]).all()
    assert ts.scalar(0).reward is None and ts.scalar(0).discount is None and ts.scalar(0).first()
    det = all(k == "deterministic" for k, _ in tb.rew_kinds)
    for t in range(1, len(acts)):
        ts = env.step(np.full(N, acts[t], np.int32), auto_reset=True, u_next=np.full(N, us[t]),
                      u_reward=np.zeros(N, np.float32))
        st = ts.step_type.cpu().numpy()
        assert (st == g["traj_step_type"][t]).all(), f"step {t}"
        assert (ts.observation.cpu().numpy() == g["traj_obs"][t]).all(), f"step {t}"
        one = ts.scalar(1)
        if st[0] != 0:
            assert one.discount == float(g["traj_discount"][t])
            if det:
                assert abs(one.reward - float(g["traj_reward"][t])) < 1e-6
        else:
            assert one.reward is None and one.discount is None
    assert (env.get_visitation_counts().cpu().numpy() == N * g["traj_visits_s"]).all()
    assert (env.get_visitation_counts(False).cpu().numpy() == N * g["traj_visits_sa"]).all()


def test_cpython_choices_kat(bm, sampler_kat):
    """5 x 5000 draws of random.Random(seed).choices (custom_samplers.py:49-72), succ and dense-f64 kernels"""
    for i in range(5):
        probs, us, chosen = sampler_kat[f"probs_{i}"], sampler_kat[f"u_{i}"], sampler_kat[f"chosen_{i}"]
        n = len(probs)
        tb = MDPTables.from_successors(n, 1, np.tile(np.arange(n, dtype=np.int32), (n, 1, 1)),
                                       np.tile(probs, (n, 1, 1)), np.full((n, 1), n), np.zeros((n, 1, n), np.int32),
                                       [("deterministic", (0.0,))], [0], [1.0])
        N = len(us)
        env = bm.BatchedMDP(tb, N, mode="succ")
        env.reset()
        env.state.zero_()
        env.step(np.zeros(N, np.int32), u_next=us, u_reward=np.zeros(N, np.float32))
        assert (env.state.cpu().numpy() == chosen).all(), f"kat {i}"


MODES = [("dense_f32", 0), ("dense_f64", 1), ("succ", 2)]


@pytest.mark.parametrize("name", ["taxicontinuous_ergo0", "c1_riverswim_epi", "frozenlakecontinuous_ergo0",
                                  "minigridempty5_epi", "c2_deepsea30_prand"])
@pytest.mark.parametrize("mode,omode", MODES)
def test_kernels_match_oracle_bit_exact(bm, name, mode, omode):
    """N ragged (not a multiple of 32), supplied uniforms for 6 steps then the built-in Philox stream with random
    actions for 30 more, auto-reset on: every output array equals the oracle's, bit for bit"""
    import torch

    g = load_instance(name)
    tb = MDPTables.from_golden(g)
    N = 1000 + 37
    env = bm.BatchedMDP(tb, N, mode=mode, seed=1234)
    cdf = None
    if omode != 2:
        cdf = env.dev.keep["cdf"].cpu().numpy()
        # the device-built dense CDF equals the oracle's definition (sequential fp64 sum rounded to storage type)
        assert np.array_equal(cdf, orc.build_dense_cdf(tb.T, ld=tb.ld, f64=(omode == 1)))
    ht = host_tables(tb, omode, cdf)
    rs = np.random.RandomState(5)
    vis_s = np.zeros(tb.S, np.uint64)
    vis_sa = np.zeros((tb.S, tb.A), np.uint64)
    u0 = rs.random_sample(N)
    ts = env.reset(u_next=u0)
    state, h, st, obs = orc.env_reset(ht, N, u_next=u0, visits_s=vis_s)
    assert np.array_equal(env.state.cpu().numpy(), state)
    for t in range(36):
        if t < 6:
            a = rs.randint(tb.A, size=N).astype(np.int32)
            un = rs.random_sample(N)
            if omode == 0:
                un = un.astype(np.float32)
            ur = rs.random_sample(N).astype(np.float32)
            ts = env.step(a, auto_reset=True, u_next=un, u_reward=ur)
            r, obs, rc, _ = orc.env_step(ht, omode, state, h, st, action=a.copy(), u_next=un, u_rew=ur,
                                         auto_reset=True, visits_s=vis_s, visits_sa=vis_sa)
        else:
            tcount = env.t
            ts, acts = env.random_step(auto_reset=True)
            r, obs, rc, a_o = orc.env_step(ht, omode, state, h, st, action=None, seed=1234, t=tcount,
                                           auto_reset=True, visits_s=vis_s, visits_sa=vis_sa)
            stepping = st != 0
            assert np.array_equal(acts.cpu().numpy()[stepping], a_o[stepping])
        assert rc == 0
        assert np.array_equal(env.state.cpu().numpy(), state), f"t={t}"
        assert np.array_equal(env.h.cpu().numpy(), h)
        assert np.array_equal(ts.step_type.cpu().numpy(), st)
        assert np.array_equal(ts.observation.cpu().numpy(), obs)
        rg = ts.reward.cpu().numpy()
        assert np.array_equal(np.isnan(rg), np.isnan(r)) and np.array_equal(rg[~np.isnan(r)], r[~np.isnan(r)])
        d = ts.discount.cpu().numpy()
        assert ((d == 1.0) == (st == 1)).all() and ((d == 0.0) == (st == 2)).all()
    assert np.array_equal(env.visits_s.cpu().numpy(), vis_s.astype(np.int64))
    assert np.array_equal(env.visits_sa.cpu().numpy(), vis_sa.astype(np.int64))
    assert int(env.visits_s.sum()) == N * 37 and int(env.visits_sa.sum()) == N * 36 - int((vis_s.sum() - N) - vis_sa.sum())


@pytest.mark.parametrize("mode", ["dense_f32", "dense_f64", "succ"])
def test_chi_square_against_T(bm, mode):
    """sampled next-state frequencies vs T[s,a,:] (Taxi: up to 10 successors), built-in Philox stream"""
    import scipy.stats
    import torch

    g = load_instance("taxicontinuous_ergo0")
    tb = MDPTables.from_golden(g)
    N = 1 << 16
    env = bm.BatchedMDP(tb, N, mode=mode, seed=99)
    env.reset()
    s, a = int(np.argmax((g["succ_len"] >= 8).any(-1))), int(np.argmax(g["succ_len"].max(0) >= 8))
    s, a = [(i, j) for i in range(tb.S) for j in range(tb.A) if g["succ_len"][i, j] >= 8][0]
    env.state.fill_(s)
    env.step(np.full(N, a, np.int32))
    counts = np.bincount(env.state.cpu().numpy(), minlength=tb.S).astype(np.float64)
    p = tb.T[s, a].astype(np.float64)
    assert counts[p == 0].sum() == 0  # zero-probability states are never produced
    sel = p > 0
    chi2 = ((counts[sel] - N * p[sel]) ** 2 / (N * p[sel])).sum()
    pval = scipy.stats.chi2.sf(chi2, sel.sum() - 1)
    assert pval > 1e-4, (chi2, pval)


def test_episodic_termination_and_reset_contract(bm):
    g = load_instance("c1_riverswim_epi")
    tb = MDPTables.from_golden(g)
    env = bm.BatchedMDP(tb, 5, mode="succ")
    with pytest.raises(AttributeError):  # step before reset (reference: necessary_reset unset, base.py:405 vs :1272)
        env.step(np.zeros(5, np.int32))
    env.reset()
    for t in range(tb.H):
        ts = env.step(np.ones(5, np.int32))
    assert bool(ts.last().all()) and bool((ts.observation == -1).all()) and bool((ts.discount == 0).all())
    with pytest.raises(AssertionError):  # base.py:1291
        env.step(np.zeros(5, np.int32))
    ts = env.step(np.zeros(5, np.int32), auto_reset=True)
    assert bool(ts.first().all()) and bool((env.h == 0).all())
    assert env.H == tb.H and env.is_episodic() and env.n_states == 5 and env.n_actions == 2


def test_reward_distribution_on_device(bm):
    """rewards drawn on the GPU from the heavy-tailed C1 distributions vs scipy (base.py:1196-1207's rescale incl.)"""
    import scipy.stats

    g = load_instance("c1_riverswim_epi")
    tb = MDPTables.from_golden(g)
    N = 1 << 17
    env = bm.BatchedMDP(tb, N, mode="succ", seed=3)
    env.reset()
    # state 4 (rightmost), action RIGHT=1 -> the "optimal" Beta(0.01, 0.11) class on the self-loop
    env.state.fill_(4)
    env.step(np.ones(N, np.int32))
    r = env.reward.cpu().numpy().astype(np.float64)
    nxt = env.state.cpu().numpy()
    cls = tb.rew_cls_succ[4, 1]
    for k in range(int(tb.succ_len[4, 1])):
        sel = nxt == tb.succ_idx[4, 1, k]
        kind, args = tb.rew_kinds[cls[k]]
        dist = getattr(scipy.stats, kind)(*args)
        x = (r[sel] + tb.rmin) / (tb.rmax - tb.rmin)  # undo r*(max-min) - min
        assert abs(x.mean() - dist.mean()) < 5 * dist.std() / np.sqrt(sel.sum()) + 1e-4
        xs = np.concatenate([np.logspace(-30, -1, 200), np.linspace(0.1, 1.0, 200)])
        emp = np.searchsorted(np.sort(x), xs, side="right") / sel.sum()
        assert np.abs(emp - dist.cdf(xs)).max() < 0.01


def test_c2_full_size_properties(bm):
    """BASELINE.json configs[1]: DeepSeaContinuous size 30, 65,536 envs.  Size-independent properties: the depth
    coordinate is deterministic in DeepSea, so all envs share h-dependent state sets; sharding the batch over two
    env_offset halves reproduces the unsharded run exactly; visitation totals are conserved."""
    g = load_instance("c2_deepsea30_prand")
    tb = MDPTables.from_golden(g)
    N = 65536
    full = bm.BatchedMDP(tb, N, mode="dense_f32", seed=1234)
    lo = bm.BatchedMDP(tb, N // 2, mode="dense_f32", seed=1234, env_offset=0)
    hi = bm.BatchedMDP(tb, N // 2, mode="dense_f32", seed=1234, env_offset=N // 2)
    for e in (full, lo, hi):
        e.reset()
    for _ in range(40):
        for e in (full, lo, hi):
            e.random_step()
    import torch

    assert torch.equal(full.state, torch.cat([lo.state, hi.state]))
    assert torch.equal(full.reward, torch.cat([lo.reward, hi.reward]))
    assert torch.equal(full.visits_sa, lo.visits_sa + hi.visits_sa)
    assert int(full.visits_s.sum()) == N * 41
    # oracle on a prefix of the batch (same Philox stream)
    cdf = full.dev.keep["cdf"].cpu().numpy()
    ht = host_tables(tb, 0, cdf)
    M = 2048
    state, h, st, obs = orc.env_reset(ht, M, seed=1234, t=0)
    for t in range(1, 41):
        orc.env_step(ht, 0, state, h, st, action=None, seed=1234, t=t)
    assert np.array_equal(full.state[:M].cpu().numpy(), state)


@pytest.mark.parametrize("S,mode,omode", [(1300, "dense_f32", 0), (1300, "dense_f64", 1), (2500, "dense_f32", 0),
                                          (129, "dense_f32", 0), (700, "dense_f64", 1), (3, "dense_f32", 0)])
def test_dense_rows_of_any_length(bm, S, mode, omode):
    """synthetic dense MDPs (CustomMDP-like): long rows (> 1024 states, generic kernel with early exit), rows that
    fill 2..8 chunks, a 3-state MDP; sparse rows with zero-probability states that must never be produced"""
    rs = np.random.RandomState(S)
    A = 2
    T = rs.dirichlet(np.ones(S) * 0.02, size=(S, A)).astype(np.float32)
    T[T < 1e-4] = 0
    T[0, 0] = 0
    T[0, 0, S - 1] = 1.0  # deterministic row hitting the last state
    T[1, 1] = 0
    T[1, 1, 0] = 1.0  # deterministic row hitting the first state
    T = (T / T.sum(-1, keepdims=True)).astype(np.float32)
    tb = MDPTables.from_dense(T, rew_kinds=[("deterministic", (0.5,)), ("beta", (2.0, 3.0))],
                              rew_cls_sa=rs.randint(2, size=(S, A)), start_idx=np.arange(S), start_prob=np.ones(S) / S)
    N = 777
    env = bm.BatchedMDP(tb, N, mode=mode, seed=11)
    cdf = env.dev.keep["cdf"].cpu().numpy()
    assert np.array_equal(cdf, orc.build_dense_cdf(T, ld=tb.ld, f64=(omode == 1)))
    ht = host_tables(tb, omode, cdf)
    env.reset()
    state, h, st, obs = orc.env_reset(ht, N, seed=11, t=0)
    assert np.array_equal(env.state.cpu().numpy(), state)
    for t in range(1, 13):
        # uniforms at the edges of [0,1) exercise the clamp to the last positive-probability state
        un = rs.random_sample(N)
        un[:5] = [0.0, 1.0 - 2.0 ** -24, 1.0 - 2.0 ** -53 if omode else 1.0 - 2.0 ** -24, 0.5, 2.0 ** -30]
        if omode == 0:
            un = un.astype(np.float32)
        a = rs.randint(A, size=N).astype(np.int32)
        ts = env.step(a, u_next=un)
        r, obs, rc, _ = orc.env_step(ht, omode, state, h, st, action=a.copy(), u_next=un, seed=11, t=t)
        nxt = env.state.cpu().numpy()
        assert np.array_equal(nxt, state), f"t={t}"
        assert np.array_equal(ts.reward.cpu().numpy(), r)
        prev = ts.observation  # noqa: F841
    # zero-probability states are never produced
    env2 = bm.BatchedMDP(tb, 4096, mode=mode, seed=5)
    env2.reset()
    env2.state.fill_(2)
    env2.step(np.zeros(4096, np.int32))
    assert (T[2, 0][env2.state.cpu().numpy()] > 0).all()


@pytest.mark.parametrize("name,mode", [("c2_deepsea30_prand", "dense_f32"), ("taxi_epi", "succ"),
                                       ("c1_riverswim_epi", "dense_f64")])
def test_zero_copy_host_io_is_identical(bm, name, mode):
    """host_io=True (the kernel reads pinned host actions and writes the TimeStep fields into pinned host memory
    itself) must emit exactly what the device-resident batch emits, step by step, incl. auto-reset and the oracle."""
    import torch

    g = load_instance(name)
    tb = MDPTables.from_golden(g)
    N = 3000  # ragged last warp
    dev = bm.BatchedMDP(tb, N, mode=mode, seed=11)
    host = bm.BatchedMDP(tb, N, mode=mode, seed=11, host_io=True)
    ts_d, ts_h = dev.reset(), host.reset()
    assert torch.equal(ts_d.observation.cpu(), ts_h.observation) and bool(ts_h.first().all())
    omode = {"dense_f32": 0, "dense_f64": 1, "succ": 2}[mode]
    ht = host_tables(tb, omode, None if omode == 2 else dev.dev.keep["cdf"].cpu().numpy())
    state, h, st, obs = orc.env_reset(ht, N, seed=11, t=0)
    gen = torch.Generator().manual_seed(3)
    for t in range(1, 2 * max(tb.H, 10) + 3):
        a = torch.randint(0, tb.A, (N,), dtype=torch.int32, generator=gen).pin_memory()
        dev.step_async(a, auto_reset=True)
        o, r, stp = host.step_host(a, auto_reset=True)
        ro, oo, rc, _ = orc.env_step(ht, omode, state, h, st, action=a.numpy(), seed=11, t=t, auto_reset=True)
        assert torch.equal(dev.obs.cpu(), o) and torch.equal(dev.step_type.cpu(), stp)
        assert np.array_equal(dev.reward.cpu().numpy(), r.numpy(), equal_nan=True)
        assert np.array_equal(o.numpy(), oo) and np.array_equal(stp.numpy(), st)
        assert np.array_equal(r.numpy(), ro, equal_nan=True)
    assert torch.equal(dev.visits_sa, host.visits_sa) and torch.equal(dev.state, host.state)
    # the general (non-lean) path of step_host: numpy actions, no auto-reset on a continuous MDP
    if tb.H == 0:
        o, r, stp = host.step_host(np.zeros(N, np.int32))
        dev.step_async(np.zeros(N, np.int32))
        assert torch.equal(dev.obs.cpu(), o) and bool((stp == 1).all())


@pytest.mark.parametrize("name,mode", [("c2_deepsea30_prand", "dense_f32"), ("taxi_epi", "succ"),
                                       ("frozenlake4_epi", "dense_f64"), ("minigridempty5_epi", "dense_f32")])
def test_fused_random_steps_equal_single_steps(bm, name, mode):
    """colo_env_random_steps: n random-agent steps in one launch == n launches (same Philox counters)"""
    import torch

    tb = MDPTables.from_golden(load_instance(name))
    N, n = 3000, 75
    a = bm.BatchedMDP(tb, N, mode=mode, seed=21)
    b = bm.BatchedMDP(tb, N, mode=mode, seed=21)
    a.reset(); b.reset()
    for _ in range(n):
        a.step_async(None, auto_reset=True)
    ts = b.random_steps_fused(n, auto_reset=True)
    for x, y in ((a.state, b.state), (a.h, b.h), (a.step_type, b.step_type), (a.obs, b.obs), (a.action, b.action),
                 (a.visits_s, b.visits_s), (a.visits_sa, b.visits_sa)):
        assert torch.equal(x, y)
    assert torch.equal(torch.nan_to_num(a.reward, nan=-7.0), torch.nan_to_num(b.reward, nan=-7.0))
    assert a.t == b.t and ts.observation.shape == (N,)
    if tb.H > 0:
        with pytest.raises(AssertionError):
            b.random_steps_fused(tb.H + 2, auto_reset=False)


@pytest.mark.parametrize("name", ["c1_riverswim_epi", "doc_simplegrid4"])
def test_emission_table_gather(bm, name):
    """non-tabular observations: rows of all_observations[h, s] (emission_maps/base.py:56-76,110-140), zeros at LAST"""
    tb = MDPTables.from_golden(load_instance(name))
    N = 777
    env = bm.BatchedMDP(tb, N, mode="succ", seed=2)
    rs = np.random.RandomState(0)
    shape = (3, 5)
    table = rs.normal(size=((tb.H, tb.S) if tb.H else (tb.S,)) + shape).astype(np.float32)
    env.set_emission_table(table)
    env.reset()
    for _ in range(2 * max(tb.H, 3)):
        env.step_async(None, auto_reset=True)
        obs = env.emit_observations().cpu().numpy()
        s, h, st = env.state.cpu().numpy(), env.h.cpu().numpy(), env.step_type.cpu().numpy()
        exp = table[h.clip(max=max(tb.H - 1, 0)), s] if tb.H else table[s]
        if tb.H:
            exp = np.where((st == 2)[:, None, None], 0.0, exp)
        assert obs.shape == (N,) + shape and np.array_equal(obs, exp.astype(np.float32))


@pytest.mark.parametrize("name,mode", [("c2_deepsea30_prand", "dense_f32"), ("taxi_epi", "succ"),
                                       ("c1_riverswim_epi", "dense_f64")])
def test_step_server_is_identical(bm, name, mode):
    """BatchedMDP.serve(): the persistent step kernel driven by the host doorbell emits, step by step, exactly what
    one launch per step emits and what the oracle emits -- across an idle lapse (the kernel retires by itself and is
    restarted) and across stop/serve."""
    import time

    import torch

    g = load_instance(name)
    tb = MDPTables.from_golden(g)
    N = 3000
    ref = bm.BatchedMDP(tb, N, mode=mode, seed=5, host_io=True)
    srv = bm.BatchedMDP(tb, N, mode=mode, seed=5, host_io=True)
    ref.reset(), srv.reset()
    omode = {"dense_f32": 0, "dense_f64": 1, "succ": 2}[mode]
    ht = host_tables(tb, omode, None if omode == 2 else ref.dev.keep["cdf"].cpu().numpy())
    state, h, st, obs = orc.env_reset(ht, N, seed=5, t=0)
    buf = torch.zeros(N, dtype=torch.int32).pin_memory()
    srv.serve(buf, idle_timeout_ms=50)
    gen = torch.Generator().manual_seed(9)
    n_steps = 2 * max(tb.H, 10) + 3
    try:
        for t in range(1, n_steps):
            a = torch.randint(0, tb.A, (N,), dtype=torch.int32, generator=gen).pin_memory()
            o1, r1, s1 = [x.clone() for x in ref.step_host(a, auto_reset=True)]
            buf.copy_(a)
            o2, r2, s2 = srv.step_served()
            ro, oo, rc, _ = orc.env_step(ht, omode, state, h, st, action=a.numpy(), seed=5, t=t, auto_reset=True)
            assert torch.equal(o1, o2) and torch.equal(s1, s2)
            assert np.array_equal(r1.numpy(), r2.numpy(), equal_nan=True)
            assert np.array_equal(o2.numpy(), oo) and np.array_equal(r2.numpy(), ro, equal_nan=True)
            if t == 4:
                time.sleep(0.25)  # > idle timeout: the server lapses, the next step restarts it
            if t == 8:
                srv.stop_serving()
                srv.serve(buf, idle_timeout_ms=50)
    finally:
        srv.stop_serving()
    assert srv.t == ref.t
    assert torch.equal(ref.visits_sa, srv.visits_sa) and torch.equal(ref.state, srv.state)


def test_pipelined_groups_equal_the_unsplit_batch(bm):
    """PipelinedBatchedMDP: G groups on their own streams, stepped recv/send in a pipeline, walk the trajectories of
    the single batch (env_offset keeps the Philox counters); launch-per-step and served modes."""
    import torch

    tb = MDPTables.from_golden(load_instance("c2_deepsea30_prand"))
    # uneven split: N need not be a multiple of the number of groups
    odd = bm.PipelinedBatchedMDP(tb, 1001, groups=3, seed=3)
    assert odd.sizes == [334, 334, 333] and odd.offsets == [0, 334, 668]
    whole = bm.BatchedMDP(tb, 1001, seed=3, host_io=True)
    odd.reset(), whole.reset()
    a_odd = torch.randint(0, tb.A, (1001,), dtype=torch.int32).pin_memory()
    want_o = [x.clone() for x in whole.step_host(a_odd, auto_reset=True)]
    got_o = odd.step_all([a_odd[o:o + n].clone().pin_memory() for o, n in zip(odd.offsets, odd.sizes)])
    for j in range(3):
        assert np.array_equal(torch.cat([p[j] for p in got_o]).numpy(), want_o[j].numpy(), equal_nan=True)
    N, G = 4096, 2
    gen = torch.Generator().manual_seed(1)
    acts = [torch.randint(0, tb.A, (N,), dtype=torch.int32, generator=gen).pin_memory() for _ in range(12)]
    one = bm.BatchedMDP(tb, N, seed=3, host_io=True)
    one.reset()
    want = [[x.clone() for x in one.step_host(a, auto_reset=True)] for a in acts]
    for serving in (False, True):
        env = bm.PipelinedBatchedMDP(tb, N, groups=G, seed=3)
        env.reset()
        bufs = [torch.zeros(N // G, dtype=torch.int32).pin_memory() for _ in range(G)]
        if serving:
            env.serve(bufs, idle_timeout_ms=100)
        try:
            for k, a in enumerate(acts):
                parts = []
                for g in range(G):
                    bufs[g].copy_(a[g * (N // G):(g + 1) * (N // G)])
                    env.send(g, None if serving else bufs[g])
                for g in range(G):
                    parts.append([x.clone() for x in env.recv(g)])
                for j in range(3):
                    got = torch.cat([p[j] for p in parts])
                    assert np.array_equal(got.numpy(), want[k][j].numpy(), equal_nan=True), (serving, k, j)
        finally:
            if serving:
                env.stop_serving()
        assert torch.equal(env.get_visitation_counts(False), one.visits_sa)


@pytest.mark.parametrize("mode,host_io", [("dense_f32", False), ("succ", True)])
def test_checkpoint_resume_is_bit_exact(bm, mode, host_io):
    """state_dict / load_state_dict: a batch restored from a checkpoint (into a fresh object) continues the very same
    trajectories, rewards and visitation counts"""
    import torch

    tb = MDPTables.from_golden(load_instance("taxi_epi"))
    N = 2000
    gen = torch.Generator().manual_seed(0)
    acts = [torch.randint(0, tb.A, (N,), dtype=torch.int32, generator=gen) for _ in range(30)]
    a = bm.BatchedMDP(tb, N, mode=mode, seed=4, host_io=host_io)
    a.reset()
    for k in range(10):
        a.step_async(acts[k].cuda(), auto_reset=True)
    ck = a.state_dict()
    tail_a = []
    for k in range(10, 30):
        a.step_async(acts[k].cuda(), auto_reset=True)
        torch.cuda.synchronize()
        tail_a.append((a.obs.clone().cpu(), a.reward.clone().cpu()))
    b = bm.BatchedMDP(tb, N, mode=mode, seed=999, host_io=host_io)
    b.load_state_dict(ck)
    for k in range(10, 30):
        b.step_async(acts[k].cuda(), auto_reset=True)
        torch.cuda.synchronize()
        o, r = tail_a[k - 10]
        assert torch.equal(b.obs.cpu(), o) and np.array_equal(b.reward.cpu().numpy(), r.numpy(), equal_nan=True)
    assert torch.equal(a.visits_sa, b.visits_sa) and torch.equal(a.visits_s, b.visits_s) and a.t == b.t


def test_emission_noise_distributions(bm):
    """EmissionMap noise (emission_maps/base.py:136-138): Gaussian per element, Student-t with the reference's
    one-draw-per-first-axis-slice broadcast; terminal (all-zero) observations stay zero; draws change every call"""
    import scipy.stats

    tb = MDPTables.from_golden(load_instance("c1_riverswim_epi"))
    N = 20000
    env = bm.BatchedMDP(tb, N, mode="succ", seed=2)
    table = np.zeros((tb.H, tb.S, 4, 6), np.float32)
    env.set_emission_table(table)
    env.reset()
    for _ in range(tb.H - 1):
        env.step_async(None, auto_reset=True)
    env.set_emission_noise("GaussianUncorrelated", seed=3, scale=0.25)
    a = env.emit_observations().cpu().numpy().astype(np.float64)
    b = env.emit_observations().cpu().numpy().astype(np.float64)
    assert not np.array_equal(a, b)
    assert scipy.stats.kstest(a.ravel()[:200000], scipy.stats.norm(0, 0.25).cdf).pvalue > 1e-3
    assert abs(np.corrcoef(a[:, 0, 0], a[:, 0, 1])[0, 1]) < 0.03  # uncorrelated features
    env.set_emission_noise("StudentTUncorrelated", seed=3, df=5)
    c = env.emit_observations().cpu().numpy().astype(np.float64)
    assert np.array_equal(c[:, 0, :], c[:, 3, :])  # sic: one row of draws broadcast over the first axis
    assert scipy.stats.kstest(c[:, 0, :].ravel(), scipy.stats.t(5).cdf).pvalue > 1e-3
    env.step_async(None, auto_reset=True)  # the last step of the episode: terminal observation, no noise
    d = env.emit_observations().cpu().numpy()
    assert bool((env.step_type == 2).all()) and float(np.abs(d).max()) == 0.0
    env.set_emission_noise(None)
    with pytest.raises(NotImplementedError):
        env.set_emission_noise("NoSuchNoise")


def test_correlated_emission_noises(bm):
    """GaussianCorrelated / StudentTCorrelated (noises/gaussian_correlated.py:9-17, student_t_correlated.py:9-17): the
    covariance W is the reference's own Wishart draw (same scipy call, same RandomState(seed)); the device samples
    x = L z [/ sqrt(chi2_df / df)].  Checked: W equals scipy's draw; the empirical covariance of 200k Gaussian samples
    equals W; every marginal of the Gaussian is N(0, W_ii) and of the Student-t (df = 3) is sqrt(W_ii) * t_3; terminal
    observations stay zero."""
    import scipy.stats

    tb = MDPTables.from_golden(load_instance("c1_riverswim_epi"))
    N, D = 200000, 5
    env = bm.BatchedMDP(tb, N, mode="succ", seed=2)
    env.set_emission_table(np.zeros((tb.H, tb.S, D), np.float32))
    env.reset()
    env.set_emission_noise("GaussianCorrelated", seed=7, scale=0.1)
    W = np.atleast_2d(scipy.stats.wishart(scale=[0.1] * D).rvs(1, np.random.RandomState(7)))
    assert np.array_equal(env._emit_cov, W)
    x = env.emit_observations().cpu().numpy().astype(np.float64)
    y = env.emit_observations().cpu().numpy().astype(np.float64)
    assert not np.array_equal(x, y)
    C_ = np.cov(x.T)
    assert np.abs(C_ - W).max() < 0.02 * np.abs(W).max(), (C_, W)
    for i in range(D):
        assert scipy.stats.kstest(x[:, i], scipy.stats.norm(0, np.sqrt(W[i, i])).cdf).pvalue > 1e-4, i
    env.set_emission_noise("StudentTCorrelated", seed=7, scale=0.1, df=3)
    z = env.emit_observations().cpu().numpy().astype(np.float64)
    for i in range(D):
        assert scipy.stats.kstest(z[:, i] / np.sqrt(W[i, i]), scipy.stats.t(3).cdf).pvalue > 1e-4, i
    # dependence through the shared chi-square and through L: |corr| of the first two features follows W
    r_w = W[0, 1] / np.sqrt(W[0, 0] * W[1, 1])
    assert abs(np.corrcoef(x[:, 0], x[:, 1])[0, 1] - r_w) < 0.02
    for _ in range(tb.H):
        env.step_async(None, auto_reset=True)
    d = env.emit_observations().cpu().numpy()
    last = (env.step_type == 2).cpu().numpy()
    assert last.any() and float(np.abs(d[last]).max()) == 0.0


@pytest.mark.parametrize("mode", ["dense_f32", "dense_f64"])
def test_step_without_search_index_is_identical(bm, mode):
    """colo_mdp_tables.cdf_mid / cdf_coarse / rew_cls_pad are optional: with NULL pointers the k-ary kernel samples the
    same entries from the row itself -- bit-identical to the indexed default."""
    import torch

    tb = MDPTables.from_golden(load_instance("c2_deepsea30_prand"))
    N = 5000
    gen = torch.Generator().manual_seed(5)
    acts = [torch.randint(0, tb.A, (N,), dtype=torch.int32, generator=gen).cuda() for _ in range(25)]

    def run(strip_index):
        env = bm.BatchedMDP(tb, N, mode=mode, seed=8)
        if strip_index:
            env.dev.c.cdf_mid = None
            env.dev.c.cdf_coarse = None
            env.dev.c.rew_cls_pad = None
        env.reset()
        out = []
        for a in acts:
            env.step_async(a, auto_reset=True)
            out.append((env.obs.clone(), env.reward.clone(), env.step_type.clone()))
        return out, env.visits_sa.clone()

    ref, vref = run(False)
    got, vgot = run(True)
    for (o1, r1, s1), (o2, r2, s2) in zip(ref, got):
        assert torch.equal(o1, o2) and torch.equal(s1, s2) and torch.equal(r1.view(torch.int32), r2.view(torch.int32))
    assert torch.equal(vref, vgot)


@pytest.mark.parametrize("name", ["c1_riverswim_epi", "doc_simplegrid4"])
def test_scalar_dropin_surface(bm, name):
    """n_envs=1, scalar_api=True: reset()/step(int) return the reference's SCALAR dm_env.TimeStep (mdp/base.py:1277,
    1316-1317) and the object carries BaseMDP's attribute surface (:463-503, :1233-1252).  Replays the reference's own
    recorded trajectory field by field."""
    from colosseum_b200.timestep import StepType

    g = load_instance(name)
    tb = MDPTables.from_golden(g)
    env = bm.BatchedMDP(tb, 1, mode="succ", scalar_api=True)
    a_spec, o_spec = env.action_spec(), env.observation_spec()
    assert a_spec.num_values == tb.A and a_spec.name == "action" and a_spec.shape == ()
    assert o_spec.num_values == tb.S and o_spec.name == "observation"
    assert env.n_states == tb.S and env.n_actions == tb.A and env.T.shape == (tb.S, tb.A, tb.S)
    assert np.allclose(env.R, g["R"]) and abs(env.starting_state_distribution.sum() - 1.0) < 1e-12
    assert np.array_equal(np.nonzero(env.starting_state_distribution)[0], np.sort(np.unique(tb.start_idx)))
    assert (env.H == int(g["H"])) if int(g["H"]) > 0 else env.H is None
    acts, us = g["traj_action"], np.nan_to_num(g["traj_u"], nan=0.5)
    ts = env.reset(u_next=us[:1])
    assert ts.step_type == StepType.FIRST and ts.reward is None and ts.discount is None
    assert ts.observation == int(g["traj_obs"][0]) and isinstance(ts.observation, int)
    for t in range(1, 60):
        ts = env.step(int(acts[t]), auto_reset=True, u_next=us[t:t + 1], u_reward=np.zeros(1, np.float32))
        assert int(ts.step_type) == int(g["traj_step_type"][t]) and ts.observation == int(g["traj_obs"][t])
        if ts.step_type == StepType.FIRST:
            assert ts.reward is None and ts.discount is None
        else:
            assert ts.discount == float(g["traj_discount"][t]) and isinstance(ts.reward, float)
    ts, a = env.random_step(auto_reset=True)
    assert isinstance(a, int) and 0 <= a < tb.A


def test_discount_written_by_the_kernel(bm):
    """dm_env's discount comes out of the step kernel's epilogue (1.0 MID, 0.0 LAST, NaN FIRST): no eager-PyTorch
    tail after a step; the host_io variant derives it from step_type on the host"""
    g = load_instance("c1_riverswim_epi")
    tb = MDPTables.from_golden(g)
    for host_io in (False, True):
        env = bm.BatchedMDP(tb, 257, mode="succ", seed=3, host_io=host_io)
        ts = env.reset()
        assert bool(np.isnan(ts.discount.cpu().numpy()).all()) and bool(np.isnan(ts.reward.cpu().numpy()).all())
        seen = set()
        for _ in range(2 * tb.H + 2):
            ts, _ = env.random_step(auto_reset=True)
            st, d = ts.step_type.cpu().numpy(), ts.discount.cpu().numpy()
            assert (d[st == 1] == 1.0).all() and (d[st == 2] == 0.0).all() and np.isnan(d[st == 0]).all()
            seen |= set(st.tolist())
        assert seen == {0, 1, 2}


@pytest.mark.parametrize("mode", ["dense_f32", "succ"])
def test_out_of_range_action_is_flagged(bm, mode):
    """the reference raises on an unknown action; the batched step flags COLO_BAD_ACTION, leaves that env untouched
    and steps the others"""
    g = load_instance("doc_simplegrid4")
    tb = MDPTables.from_golden(g)
    env = bm.BatchedMDP(tb, 64, mode=mode, seed=1)
    env.reset()
    before = env.state.cpu().numpy().copy()
    a = np.zeros(64, np.int32)
    a[5], a[40] = tb.A, -1
    with pytest.raises(ValueError):
        env.step(a)
    after = env.state.cpu().numpy()
    assert after[5] == before[5] and after[40] == before[40] and int(env.h[5]) == 0 and int(env.h[6]) == 1
    env.step(np.zeros(64, np.int32))  # the flag was cleared: the batch goes on


def test_native_pipeline_loop_is_identical(bm):
    """colo_env_pipeline_run (the recv/send loop inside the library) == the same loop from Python, bit for bit"""
    import torch

    g = load_instance("c2_deepsea30_prand")
    tb = MDPTables.from_golden(g)
    N, G, K = 4096 + 7, 2, 9
    gen = torch.Generator().manual_seed(3)
    a = bm.PipelinedBatchedMDP(tb, N, groups=G, seed=11)
    b = bm.PipelinedBatchedMDP(tb, N, groups=G, seed=11)
    a.reset(); b.reset()
    ring = [[torch.randint(0, tb.A, (a.sizes[k],), dtype=torch.int32, generator=gen).pin_memory() for k in range(G)]
            for _ in range(4)]
    for k in range(G):
        a.send(k, ring[0][k])
    for i in range(1, K):
        for k in range(G):
            a.recv(k)
            a.send(k, ring[i % 4][k])
    outs_a = [tuple(x.clone() for x in a.recv(k)) for k in range(G)]
    outs_b = b.run_native(ring, K)
    for k in range(G):
        for x, y in zip(outs_a[k], outs_b[k]):
            assert torch.equal(x, y) or (torch.isnan(x) == torch.isnan(y)).all() and torch.equal(torch.nan_to_num(x), torch.nan_to_num(y))
        assert torch.equal(a.shards[k].state, b.shards[k].state) and a.shards[k].t == b.shards[k].t
    assert torch.equal(a.get_visitation_counts(), b.get_visitation_counts())


def test_queued_pipeline_is_identical(bm):
    """colo_env_pipeline_run_queued (stream memory operations instead of a stream sync + launch per group-step; one at a
    time and as replayed CUDA graphs of 64 steps) == colo_env_pipeline_run, bit for bit -- int32 and compact I/O, three
    groups of uneven sizes, step counts that are not multiples of the graph length, two calls in a row, the variant with
    one host thread per group (colo_env_pipeline_run_threads), and a host agent (ctypes callback) that derives every action from the TimeStep it has just been handed."""
    import ctypes as C

    import torch

    from colosseum_b200._cabi import ColosseumB200Error

    def queued(env, *a, **kw):
        try:
            return env.run_queued(*a, **kw)
        except ColosseumB200Error as exc:
            # the library's watchdog: the groups' streams were mapped onto one hardware queue by the driver and a queued
            # wait blocked another group (the call drained its streams and reported it) -- a property of the box
            if "no progress" in str(exc):
                pytest.skip(str(exc))
            raise

    tb = MDPTables.from_golden(load_instance("c2_deepsea30_prand"))
    N, G = 6000 + 5, 3
    for compact in (False, True):
        gen = torch.Generator().manual_seed(5)
        envs = [bm.PipelinedBatchedMDP(tb, N, groups=G, seed=21, compact_io=compact) for _ in range(4)]
        for e in envs:
            e.reset()
        ring = [[torch.randint(0, tb.A, (n,), dtype=torch.int32, generator=gen).to(envs[0].shards[0].action_dtype).pin_memory()
                 for n in envs[0].sizes] for _ in range(8)]
        for K in (5, 64 * 3 + 17, 130):
            ref = envs[0].run_native(ring, K)
            for e, graph in ((envs[1], False), (envs[2], True), (envs[3], "threads")):
                out = e.run_native(ring, K, threads=True) if graph == "threads" else queued(e, ring, K, graph=graph)
                for k in range(G):
                    for x, y in zip(ref[k], out[k]):
                        assert np.array_equal(x.numpy(), y.numpy(), equal_nan=True), (compact, K, graph, k)
                    assert torch.equal(envs[0].shards[k].state, e.shards[k].state) and envs[0].shards[k].t == e.shards[k].t
                assert torch.equal(envs[0].get_visitation_counts(), e.get_visitation_counts())

    # a host agent in the loop: the action of step i+1 is a function of the observation of step i
    cb_t = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.c_int)
    finals = []
    for runner in ("native", "queued", "graph", "threads"):
        env = bm.PipelinedBatchedMDP(tb, 2048, groups=2, seed=9)
        env.reset()
        acts = [torch.zeros(n, dtype=torch.int32).pin_memory() for n in env.sizes]
        seen = []

        def agent(user, g, step, env=env, acts=acts, seen=seen):
            obs = env.shards[g].obs.numpy()
            seen.append((g, step, int(obs.sum())))
            acts[g].numpy()[:] = (obs + step) % tb.A

        cb = cb_t(agent)
        K = 200
        if runner in ("native", "threads"):
            env.run_native([acts], K, on_timestep=cb, threads=runner == "threads")
        else:
            queued(env, [acts], K, on_timestep=cb, graph=runner == "graph")
        if runner == "threads":  # one host thread per group: only the order within a group is defined
            seen.sort(key=lambda x: (x[1], x[0]))
        else:
            assert [x[:2] for x in seen[:4]] == [(0, 0), (1, 0), (0, 1), (1, 1)]
        finals.append((list(seen), [sh.state.cpu().numpy().copy() for sh in env.shards]))
        assert len(seen) == 2 * K
    for other in finals[1:]:
        assert other[0] == finals[0][0]
        assert all(np.array_equal(a, b) for a, b in zip(other[1], finals[0][1]))


def test_compact_host_io_is_identical(bm):
    """compact_io=True (uint8 actions in, int16 observations out: 8 instead of 13 bytes per env-step over PCIe) emits
    exactly the TimeSteps of the int32 host_io batch -- single batch, pipelined groups and the native loop -- on a
    continuous and an episodic MDP (terminal observation -1, auto-reset); calls the compact layout cannot serve fail
    loudly."""
    import torch

    from colosseum_b200._cabi import ColosseumB200Error

    for name in ("c2_deepsea30_prand", "minigridempty5_epi"):
        tb = MDPTables.from_golden(load_instance(name))
        N = 3001
        ref = bm.BatchedMDP(tb, N, seed=11, host_io=True)
        cpt = bm.BatchedMDP(tb, N, seed=11, host_io=True, compact_io=True)
        pipe = bm.PipelinedBatchedMDP(tb, N, groups=2, seed=11, compact_io=True)
        a0, b0 = ref.reset(), cpt.reset()
        pipe.reset()
        assert cpt.obs.dtype == torch.int16 and torch.equal(a0.observation, b0.observation.to(torch.int32))
        gen = torch.Generator().manual_seed(3)
        n0 = pipe.sizes[0]
        for t in range(3 * max(tb.H, 10)):
            a = torch.randint(0, tb.A, (N,), dtype=torch.int32, generator=gen).pin_memory()
            a8 = a.to(torch.uint8).pin_memory()
            o, r, st = ref.step_host(a, auto_reset=True)
            o2, r2, st2 = cpt.step_host(a8, auto_reset=True)
            parts = pipe.step_all([a8[:n0].clone().pin_memory(), a8[n0:].clone().pin_memory()])
            assert torch.equal(o, o2.to(torch.int32)) and torch.equal(st, st2)
            assert np.array_equal(r.numpy(), r2.numpy(), equal_nan=True)
            assert torch.equal(o, torch.cat([p[0] for p in parts]).to(torch.int32))
            assert np.array_equal(r.numpy(), torch.cat([p[1] for p in parts]).numpy(), equal_nan=True)
            if tb.H > 0:
                assert bool(((o2 == -1) == (st2 == 2)).all())
        assert torch.equal(ref.visits_sa, cpt.visits_sa) and torch.equal(ref.state, cpt.state)
        # the native loop continues the same trajectories
        ring = [[torch.randint(0, tb.A, (n,), dtype=torch.int32, generator=gen).to(torch.uint8).pin_memory()
                 for n in pipe.sizes] for _ in range(3)]
        pipe.run_native(ring, 7)
        for i in range(7):
            a8 = torch.cat(ring[i % 3]).pin_memory()
            o2, r2, st2 = cpt.step_host(a8, auto_reset=True)
        assert torch.equal(o2, torch.cat([sh.obs for sh in pipe.shards]))
        assert np.array_equal(r2.numpy(), torch.cat([sh.reward for sh in pipe.shards]).numpy(), equal_nan=True)
        with pytest.raises(ColosseumB200Error):  # no auto-reset: not the lean call
            cpt.step_async(a8, auto_reset=False)
            torch.cuda.synchronize()
    with pytest.raises(AssertionError):
        bm.BatchedMDP(tb, 8, mode="succ", host_io=True, compact_io=True)
