"""GPU: MixedBatchedMDP -- envs of different MDP instances in one batch, one launch per step.

Segment i of a mixed batch must be bit-identical to `BatchedMDP(tables[i], n_i, mode, seed=seed_i)` driven by the same
calls (Philox key seed_i, counter (e - start_i, t)); checked against the reference's own recorded trajectories, against
single-MDP batches and the C oracle (ragged segments so that warps straddle instances), and at the C3 suite's scale."""
import numpy as np
import pytest

from conftest import GOLDEN, golden_instances, load_instance
from colosseum_b200 import _cabi
from colosseum_b200.tables import MDPTables
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

NAMES = golden_instances()  # 17 instances: S 5-465, A 2-6, H 0-24, K 1-13, up to 72 start states


@pytest.fixture(scope="module")
def bm():
    import colosseum_b200.batched_mdp as bm

    return bm


@pytest.fixture(scope="module")
def goldens():
    return {n: load_instance(n) for n in NAMES}


@pytest.fixture(scope="module")
def tables(goldens):
    return {n: MDPTables.from_golden(g) for n, g in goldens.items()}


def _np(t):
    return t.cpu().numpy()


def _same_reward(a, b):
    return np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a[~np.isnan(a)], b[~np.isnan(b)])


def _host_tables(tb, omode, cdf=None):
    if omode == 2:
        return orc.HostTables(tb.S, tb.A, H=tb.H, succ_cum=tb.succ_cum, succ_idx=tb.succ_idx, succ_len=tb.succ_len,
                              rew_cls_succ=tb.rew_cls_succ, rew_q=tb.rew_q, rmin=tb.rmin, rmax=tb.rmax,
                              start_cum=tb.start_cum, start_idx=tb.start_idx)
    return orc.HostTables(tb.S, tb.A, H=tb.H, cdf=cdf, rew_cls_sas=tb.rew_cls_sas, rew_cls_sa=tb.rew_cls_sa,
                          rew_q=tb.rew_q, rmin=tb.rmin, rmax=tb.rmax, start_cum=tb.start_cum, start_idx=tb.start_idx)


def test_reference_trajectories_replayed_in_one_batch(bm, goldens, tables):
    """all 17 recorded reference trajectories (401 steps, auto_reset, the uniforms the reference's samplers consumed),
    3 envs per instance, every instance stepping in the same launches"""
    n = 3
    env = bm.MixedBatchedMDP([tables[k] for k in NAMES], n, mode="succ")
    gs = [goldens[k] for k in NAMES]
    acts = np.stack([g["traj_action"] for g in gs])            # [I, T]
    us = np.stack([np.nan_to_num(g["traj_u"], nan=0.5) for g in gs])
    sts, obss = np.stack([g["traj_step_type"] for g in gs]), np.stack([g["traj_obs"] for g in gs])
    rewards, discounts = np.stack([g["traj_reward"] for g in gs]), np.stack([g["traj_discount"] for g in gs])
    det = np.array([all(k == "deterministic" for k, _ in tables[k].rew_kinds) for k in NAMES])
    rep = lambda x: np.repeat(x, n)  # noqa: E731  per-instance value -> per-env
    ts = env.reset(u_next=rep(us[:, 0]))
    assert np.array_equal(_np(ts.step_type), rep(sts[:, 0])) and np.array_equal(_np(ts.observation), rep(obss[:, 0]))
    N = env.n_envs
    for t in range(1, acts.shape[1]):
        ts = env.step(rep(acts[:, t]).astype(np.int32), auto_reset=True, u_next=rep(us[:, t]),
                      u_reward=np.zeros(N, np.float32))
        st, ob = _np(ts.step_type), _np(ts.observation)
        assert np.array_equal(st, rep(sts[:, t])), f"step {t}"
        assert np.array_equal(ob, rep(obss[:, t])), f"step {t}"
        d, r = _np(ts.discount), _np(ts.reward)
        mid = st != 0
        assert np.array_equal(d[mid], rep(discounts[:, t])[mid]) and np.isnan(d[~mid]).all() and np.isnan(r[~mid]).all()
        ok = mid & rep(det)
        assert (np.abs(r[ok] - rep(rewards[:, t])[ok]) < 1e-6).all(), f"step {t}"
    for i, k in enumerate(NAMES):
        assert np.array_equal(_np(env.get_visitation_counts(i)), n * goldens[k]["traj_visits_s"]), k
        assert np.array_equal(_np(env.get_visitation_counts(i, state_only=False)), n * goldens[k]["traj_visits_sa"]), k


MODES = [("dense_f32", 0), ("dense_f64", 1), ("succ", 2)]
# (instance names, envs per instance, seeds): ragged segments so that warps and CTAs straddle instances
MIXES = {
    "ragged": (["c1_riverswim_epi", "taxi_epi", "frozenlakecontinuous_ergo0", "c2_deepsea30_prand", "deepsea8_epi",
                "doc_simplegrid4", "minigridempty5_epi", "taxicontinuous_ergo0"],
               [1, 3, 31, 33, 1000 + 37, 5, 64, 70], [7, 7, 11, 0, 12345, 7, 3, 2**40 + 5]),
    "all17": (NAMES, [1 + (13 * i) % 40 for i in range(len(NAMES))], list(range(len(NAMES)))),
    "alone": (["simplegrid5_epi"], [45], [99]),
}


@pytest.mark.parametrize("mix", sorted(MIXES))
@pytest.mark.parametrize("mode,omode", MODES)
def test_segments_equal_single_mdp_batches(bm, tables, mix, mode, omode):
    """reset, 6 steps with supplied actions / uniforms, 30 random auto-resetting steps: every segment equals its own
    BatchedMDP bit for bit (state, h, step_type, obs, reward, discount, random actions, visitation counts), and for succ
    and dense_f32 the C oracle with the instance's seed and env0 = 0"""
    names, sizes, seeds = MIXES[mix]
    tbs = [tables[k] for k in names]
    env = bm.MixedBatchedMDP(tbs, sizes, mode=mode, seed=seeds)
    singles = [bm.BatchedMDP(tb, n, mode=mode, seed=s) for tb, n, s in zip(tbs, sizes, seeds)]
    use_oracle = omode in (0, 2)
    if use_oracle:
        hts = [_host_tables(tb, omode, None if omode == 2 else _np(env.dev[i].keep["cdf"])) for i, tb in enumerate(tbs)]
        orcs = []
        vis = [(np.zeros(tb.S, np.uint64), np.zeros((tb.S, tb.A), np.uint64)) for tb in tbs]
    N = env.n_envs
    rs = np.random.RandomState(17)
    u0 = rs.random_sample(N)
    ts = env.reset(u_next=u0)
    for i, b in enumerate(singles):
        b.reset(u_next=u0[env.segment(i)])
        if use_oracle:
            orcs.append(list(orc.env_reset(hts[i], sizes[i], u_next=u0[env.segment(i)], seed=seeds[i], visits_s=vis[i][0])))
    for t in range(37):
        if t == 0:
            pass  # the reset's TimeStep
        elif t <= 6:
            a = np.concatenate([rs.randint(tb.A, size=n) for tb, n in zip(tbs, sizes)]).astype(np.int32)
            un = rs.random_sample(N)
            if omode == 0:
                un = un.astype(np.float32)
            ur = rs.random_sample(N).astype(np.float32)
            ts = env.step(a, auto_reset=True, u_next=un, u_reward=ur)
            acts = None
        else:
            tcount = env.t
            ts, acts = env.random_step(auto_reset=True)
            acts = _np(acts)
        outs = {"state": _np(env.state), "h": _np(env.h), "st": _np(ts.step_type), "obs": _np(ts.observation),
                "rew": _np(ts.reward), "disc": _np(ts.discount)}
        for i, b in enumerate(singles):
            sl = env.segment(i)
            if 1 <= t <= 6:
                bts = b.step(a[sl], auto_reset=True, u_next=un[sl], u_reward=ur[sl])
            elif t > 6:
                bts, bacts = b.random_step(auto_reset=True)
                stepping = _np(bts.step_type) != 0
                assert np.array_equal(acts[sl][stepping], _np(bacts)[stepping]), (names[i], t)
            else:
                bts = b._timestep()
            assert np.array_equal(outs["state"][sl], _np(b.state)), (names[i], t)
            assert np.array_equal(outs["h"][sl], _np(b.h)), (names[i], t)
            assert np.array_equal(outs["st"][sl], _np(bts.step_type)), (names[i], t)
            assert np.array_equal(outs["obs"][sl], _np(bts.observation)), (names[i], t)
            assert _same_reward(outs["rew"][sl], _np(bts.reward)), (names[i], t)
            assert _same_reward(outs["disc"][sl], _np(bts.discount)), (names[i], t)
            if use_oracle and t >= 1:
                state, h, st, _ = orcs[i]
                if t <= 6:
                    r, ob, rc, _ = orc.env_step(hts[i], omode, state, h, st, action=a[sl].copy(), u_next=un[sl],
                                                u_rew=ur[sl], auto_reset=True, visits_s=vis[i][0], visits_sa=vis[i][1])
                else:
                    r, ob, rc, _ = orc.env_step(hts[i], omode, state, h, st, action=None, seed=seeds[i], t=tcount,
                                                auto_reset=True, visits_s=vis[i][0], visits_sa=vis[i][1])
                assert rc == 0
                assert np.array_equal(outs["state"][sl], state) and np.array_equal(outs["h"][sl], h), (names[i], t)
                assert np.array_equal(outs["st"][sl], st) and np.array_equal(outs["obs"][sl], ob), (names[i], t)
                assert _same_reward(outs["rew"][sl], r), (names[i], t)
    for i, b in enumerate(singles):
        assert np.array_equal(_np(env.get_visitation_counts(i)), _np(b.visits_s)), names[i]
        assert np.array_equal(_np(env.get_visitation_counts(i, state_only=False)), _np(b.visits_sa)), names[i]
        if use_oracle:
            assert np.array_equal(_np(env.get_visitation_counts(i)), vis[i][0].astype(np.int64)), names[i]
            assert np.array_equal(_np(env.get_visitation_counts(i, False)), vis[i][1].astype(np.int64)), names[i]


def _snapshot(env):
    return [_np(x).copy() for x in (env.state, env.h, env.step_type, env.obs, env.reward, env.discount,
                                    env._visits_s.sum(0), env._visits_sa.sum(0))]


@pytest.mark.parametrize("mode", ["succ", "dense_f32"])
def test_fused_random_steps_equal_single_steps(bm, tables, mode):
    names = ["deepsea8_epi", "taxicontinuous_ergo0", "c1_riverswim_epi", "frozenlake4_epi", "c2_deepsea30_prand"]
    sizes, seeds = [33, 65, 7, 100, 31], [1, 2, 3, 3, 5]
    tbs = [tables[k] for k in names]
    a = bm.MixedBatchedMDP(tbs, sizes, mode=mode, seed=seeds)
    b = bm.MixedBatchedMDP(tbs, sizes, mode=mode, seed=seeds)
    a.reset()
    b.reset()
    a.random_steps_fused(25, auto_reset=True)
    for _ in range(25):
        b.random_step(auto_reset=True)
    assert a.t == b.t
    for x, y in zip(_snapshot(a), _snapshot(b)):
        assert np.array_equal(x, y, equal_nan=x.dtype.kind == "f")
    # without auto-reset the episodic envs stop at LAST: the fused call raises once, single steps raise along the way
    with pytest.raises(AssertionError):
        a.random_steps_fused(12, auto_reset=False)
    raised = 0
    for _ in range(12):
        try:
            b.random_step(auto_reset=False)
        except AssertionError:
            raised += 1
    assert raised >= 1 and a.t == b.t
    for x, y in zip(_snapshot(a), _snapshot(b)):
        assert np.array_equal(x, y, equal_nan=x.dtype.kind == "f")


def _kinds():
    return np.array([_cabi.lib().colo_step_kernel_launches(k) for k in range(7)], np.int64)


@pytest.mark.parametrize("mode", ["succ", "dense_f32", "dense_f64"])
@pytest.mark.parametrize("n_inst", [1, 94])
def test_one_launch_per_call(bm, tables, n_inst, mode):
    """reset, a step and the fused random steps are one kernel launch each, whatever the number of instances, and
    every step launch is counted against its mixed kernel variant"""
    import torch

    tbs = [tables[NAMES[i % len(NAMES)]] for i in range(n_inst)]
    env = bm.MixedBatchedMDP(tbs, [1 + i % 5 for i in range(n_inst)], mode=mode, seed=list(range(n_inst)))
    lib = _cabi.lib()
    kind = _cabi.STEP_KIND_MIXED_SUCC if mode == "succ" else _cabi.STEP_KIND_MIXED_DENSE
    k0 = _kinds()
    c0 = lib.colo_launch_count()
    env.reset()
    c1 = lib.colo_launch_count()
    env.step(torch.zeros(env.n_envs, dtype=torch.int32, device="cuda"), auto_reset=True)
    c2 = lib.colo_launch_count()
    env.random_steps_fused(50)
    c3 = lib.colo_launch_count()
    env.random_step(auto_reset=True)
    c4 = lib.colo_launch_count()
    assert (c1 - c0, c2 - c1, c3 - c2, c4 - c3) == (1, 1, 1, 1)
    want = np.zeros(7, np.int64)
    want[kind] = 3  # the reset is not a step launch
    assert np.array_equal(_kinds() - k0, want)


def test_action_range_is_per_instance(bm, tables):
    """action 3 is valid in an A = 4 instance and invalid in an A = 2 one of the same batch"""
    import torch

    tbs = [tables["frozenlakecontinuous_ergo0"], tables["riverswimcontinuous_ergo0"], tables["taxicontinuous_ergo0"]]
    assert [tb.A for tb in tbs] == [4, 2, 6]
    env = bm.MixedBatchedMDP(tbs, [40, 24, 9], mode="succ", seed=[1, 2, 3])
    with pytest.raises(AttributeError):
        env.step(np.zeros(env.n_envs, np.int32))  # before reset()
    env.reset()
    before = [_np(x).copy() for x in (env.state, env.h, env.step_type)]
    with pytest.raises(ValueError):
        env.step(np.full(env.n_envs, 3, np.int32))
    bad = env.segment(1)
    for x, y in zip(before, (env.state, env.h, env.step_type)):
        assert np.array_equal(_np(y)[bad], x[bad])  # the A = 2 instance's envs were left untouched
    h = _np(env.h)
    assert (h[env.segment(0)] == 1).all() and (h[env.segment(2)] == 1).all()  # the others stepped
    assert (_np(env.action) == 3).all()
    ts = env.step(np.zeros(env.n_envs, np.int32))  # the next call goes on
    assert (_np(env.h)[bad] == 1).all() and (_np(ts.step_type) == _cabi.STEP_MID).all()
    assert int(env.status.item()) == 0
    # a terminated episode of an episodic instance raises without auto-reset
    epi = bm.MixedBatchedMDP([tables["c1_riverswim_epi"], tables["deepsea10"]], [4, 4], mode="succ")
    epi.reset()
    for _ in range(int(tables["c1_riverswim_epi"].H)):
        epi.step(torch.zeros(8, dtype=torch.int32, device="cuda"))
    assert (_np(epi.step_type)[epi.segment(0)] == _cabi.STEP_LAST).all()
    assert (_np(epi.obs)[epi.segment(0)] == -1).all()
    with pytest.raises(AssertionError):
        epi.step(np.zeros(8, np.int32))


def test_c3_scale_equals_the_suite_step_phase(bm):
    """128 suite instances x 1,024 envs, reset + 1,000 fused random steps with seed 0 in one mixed batch: state, h and
    every instance's visitation counts equal suite.run_instance's step phase (BatchedMDP(inst.tables, 1024, "succ",
    seed=0) + random_steps_fused(1000))"""
    from colosseum_b200 import suite

    insts = suite.load_suite_all(GOLDEN, indices=range(128))
    n, steps = 1024, 1000
    env = bm.MixedBatchedMDP([x.tables for x in insts], n, mode="succ", seed=0)
    env.reset()
    env.random_steps_fused(steps, auto_reset=True)
    state, h = _np(env.state), _np(env.h)
    for i, inst in enumerate(insts):
        one = bm.BatchedMDP(inst.tables, n, mode="succ", seed=0)
        one.reset()
        one.random_steps_fused(steps, auto_reset=True)
        sl = env.segment(i)
        assert np.array_equal(state[sl], _np(one.state)), inst.name
        assert np.array_equal(h[sl], _np(one.h)), inst.name
        assert np.array_equal(_np(env.get_visitation_counts(i)), _np(one.visits_s)), inst.name
        assert np.array_equal(_np(env.get_visitation_counts(i, False)), _np(one.visits_sa)), inst.name
        del one


@pytest.mark.parametrize("mode", ["succ", "dense_f64"])
def test_checkpoint_resume_is_bit_exact(bm, tables, mode):
    names = ["taxi_epi", "riverswimcontinuous_ergo1", "deepsea8_epi"]
    tbs = [tables[k] for k in names]
    a = bm.MixedBatchedMDP(tbs, [50, 3, 77], mode=mode, seed=[4, 5, 6])
    a.reset()
    a.random_steps(7, auto_reset=True)
    ck = a.state_dict()
    b = bm.MixedBatchedMDP(tbs, [50, 3, 77], mode=mode, seed=0)  # other seeds: the checkpoint's are restored
    b.load_state_dict(ck)
    a.random_steps_fused(40, auto_reset=True)
    b.random_steps_fused(40, auto_reset=True)
    for x, y in zip(_snapshot(a), _snapshot(b)):
        assert np.array_equal(x, y, equal_nan=x.dtype.kind == "f")
