"""GPU: mixed agent batches -- Q-learning loops on many MDP instances advanced by one launch (MixedQLearningEpisodic,
MixedQLearningContinuous, MixedBatchedMDPLoop).

Segment i must be bit-identical to the single-MDP class built with tables[i], seed[i] and n_loops = n_i: trace, every
agent table, state, h, cumulative reward and episode count.  Ragged loop counts make warps and 128-thread CTAs straddle
instances; seeds reach past 2**40."""
import ctypes as C
import sys

import numpy as np
import pytest

from conftest import CONTINUOUS, EPISODIC, GOLDEN, load_instance
from colosseum_b200 import _cabi
from colosseum_b200.tables import MDPTables

sys.path.insert(0, GOLDEN)
from make_qlearning_golden import CASES  # noqa: E402

pytestmark = pytest.mark.gpu

RAGGED = [1, 3, 31, 33, 1037, 2, 129, 5, 64, 17, 96, 7]
TABLE_FIELDS = ("N", "Q", "V", "Q_main", "mu", "sigma", "beta")


@pytest.fixture(scope="module")
def al():
    import colosseum_b200.agent_loop as al

    return al


@pytest.fixture(scope="module")
def goldens():
    return {n: load_instance(n) for n in EPISODIC + CONTINUOUS}


def _synthetic_a9():
    """a continuous instance with A = 9: the kernel's long-row (A > 8) path next to the register path"""
    rng = np.random.default_rng(9)
    S, A = 7, 9
    prob = rng.random((S, A, S)) * (rng.random((S, A, S)) < 0.5) + 1e-3
    prob /= prob.sum(-1, keepdims=True)
    idx = np.broadcast_to(np.arange(S, dtype=np.int32), (S, A, S))
    return MDPTables.from_successors(S, A, idx, prob, np.full((S, A), S, np.int32), rng.integers(0, 2, (S, A, S)),
                                     [("deterministic", (0.25,)), ("beta", (2.0, 3.0))], [0, 3], [0.5, 0.5])


def _tables(goldens, episodic):
    tbs = [MDPTables.from_golden(goldens[n]) for n in (EPISODIC if episodic else CONTINUOUS)]
    return tbs if episodic else tbs + [_synthetic_a9()]


def _loops_and_seeds(n):
    return [RAGGED[k % len(RAGGED)] for k in range(n)], [2 ** 40 + 5 - 7919 * k for k in range(n)]


def _mixed(al, tbs, kw, n_loops, seeds):
    kw = dict(kw)
    T = kw.pop("optimization_horizon")
    cls = al.MixedQLearningEpisodic if tbs[0].H > 0 else al.MixedQLearningContinuous
    return cls(seeds, tbs, T, n_loops=n_loops, **kw)


def _single(al, tb, kw, n, seed):
    kw = dict(kw)
    T = kw.pop("optimization_horizon")
    cls = al.QLearningEpisodic if tb.H > 0 else al.QLearningContinuous
    return cls(seed, tb, T, n_loops=n, **kw)


def _np(t):
    return t.cpu().numpy()


def _assert_segments_equal_singles(al, mixed, tbs, kw, n_loops, seeds, steps=(40, 70)):
    tr_m = [_np(mixed.steps(n, trace=True)) for n in steps]
    for i, tb in enumerate(tbs):
        one = _single(al, tb, kw, n_loops[i], seeds[i])
        tr_s = [_np(one.steps(n, trace=True)) for n in steps]
        sl = mixed.segment(i)
        for a, b in zip(tr_m, tr_s):
            assert np.array_equal(a[:, sl], b), f"instance {i}: trace"
        for f in TABLE_FIELDS:
            assert hasattr(mixed, f) == hasattr(one, f), f
            if hasattr(one, f):
                assert np.array_equal(_np(mixed.table(f, i)), _np(getattr(one, f))), f"instance {i}: {f}"
        for f in ("state", "h", "cumulative_reward", "n_episodes"):
            assert np.array_equal(_np(getattr(mixed, f)[sl]), _np(getattr(one, f))), f"instance {i}: {f}"
        del one


@pytest.mark.parametrize("name,inst,kw", CASES, ids=[c[0] for c in CASES])
def test_segments_equal_single_mdp_batches(al, goldens, name, inst, kw):
    """every golden instance of the case's kind in one batch (episodic: different H; continuous: with an A = 9
    instance), the case's hyper-parameters"""
    tbs = _tables(goldens, kw.get("UCB_type") is not None)
    n_loops, seeds = _loops_and_seeds(len(tbs))
    mixed = _mixed(al, tbs, kw, n_loops, seeds)
    assert mixed.n_loops == sum(n_loops)
    _assert_segments_equal_singles(al, mixed, tbs, kw, n_loops, seeds)


ACTORS = {
    "eps_schedule": dict(epsilon_greedy=lambda t: 0.5 / (1.0 + 0.01 * t)),
    "boltzmann_const": dict(boltzmann_temperature=3.0),
    "boltzmann_schedule": dict(epsilon_greedy=0.05, boltzmann_temperature=lambda t: 0.5 + 0.02 * t),
}


@pytest.mark.parametrize("actor", list(ACTORS))
@pytest.mark.parametrize("case", ["epi_bernstein", "cont"])
def test_exploration_segments_equal_single_mdp_batches(al, goldens, actor, case):
    kw = dict(next(c[2] for c in CASES if c[0] == case), **ACTORS[actor])
    tbs = _tables(goldens, case.startswith("epi"))
    n_loops, seeds = _loops_and_seeds(len(tbs))
    n_loops = [min(n, 200) for n in n_loops]
    mixed = _mixed(al, tbs, kw, n_loops, seeds)
    _assert_segments_equal_singles(al, mixed, tbs, kw, n_loops, seeds, steps=(30, 45))


def test_one_launch_per_steps_on_17_instances(al, goldens):
    tbs = [MDPTables.from_golden(goldens[CONTINUOUS[k % len(CONTINUOUS)]]) for k in range(17)]
    kw = next(c[2] for c in CASES if c[0] == "cont")
    mixed = _mixed(al, tbs, kw, RAGGED[:12] + [4] * 5, list(range(17)))
    lib = _cabi.lib()
    for _ in range(3):
        before = lib.colo_launch_count()
        mixed.steps(25)
        assert lib.colo_launch_count() == before + 1


@pytest.mark.parametrize("case", ["epi_bernstein_minat", "cont_taxi"])
def test_checkpoint_resume_is_bit_exact(al, goldens, case):
    kw = next(c[2] for c in CASES if c[0] == case)
    tbs = _tables(goldens, case.startswith("epi"))
    n_loops, seeds = _loops_and_seeds(len(tbs))
    a = _mixed(al, tbs, kw, n_loops, seeds)
    a.steps(60)
    ck = al.agents_state_dict(a)
    b = _mixed(al, tbs, kw, n_loops, seeds)
    al.agents_load_state_dict(b, ck)
    ta, tb_ = _np(a.steps(80, trace=True)), _np(b.steps(80, trace=True))
    assert np.array_equal(ta, tb_)
    for f in TABLE_FIELDS + ("state", "h", "cumulative_reward", "n_episodes"):
        if hasattr(a, f):
            assert np.array_equal(_np(getattr(a, f)), _np(getattr(b, f))), f


REGRET_NAMES = {True: ["c1_riverswim_epi", "frozenlake4_epi", "deepsea8_epi"],
                False: ["riverswimcontinuous_ergo0", "frozenlakecontinuous_ergo0", "riverswimcontinuous_ergo1"]}


@pytest.mark.parametrize("episodic", [True, False], ids=["episodic", "continuous"])
def test_mixed_loop_regret_equals_batched_loop(al, goldens, episodic):
    names = REGRET_NAMES[episodic]
    gs = [goldens[n] for n in names]
    tbs = [MDPTables.from_golden(g) for g in gs]
    T = [np.asarray(g["T"], np.float32) for g in gs]
    R = [np.asarray(g["R"], np.float32) for g in gs]
    kw = next(c[2] for c in CASES if c[0] == ("epi_hoeffding" if episodic else "cont"))
    n_loops, seeds = [5, 33, 2], [3, 2 ** 40 + 5, 11]
    logs = al.MixedBatchedMDPLoop(_mixed(al, tbs, kw, n_loops, seeds), T=T, R=R).run(600, log_every=200,
                                                                                    regret_for="all")
    assert [r["steps"] for r in logs] == [200, 400, 600]
    off = np.concatenate([[0], np.cumsum(n_loops)])
    for i in range(len(tbs)):
        one = _single(al, tbs[i], kw, n_loops[i], seeds[i])
        ref = al.BatchedMDPLoop(one, T=T[i], R=R[i]).run(600, log_every=200, regret_for="all")
        sl = slice(off[i], off[i + 1])
        for rm, rs in zip(logs, ref):
            assert set(rm) == set(rs)
            for k, v in rs.items():
                if k in ("steps", "steps_per_second"):
                    continue
                got = rm[k][sl]
                want = np.broadcast_to(v, got.shape)
                assert np.array_equal(got, want), f"instance {i}: {k}"


def test_c3_smoke_first_128_of_each_kind(al):
    """the first 128 C3 instances of each kind, 2 loops each, one launch per steps(): every episode of an episodic
    loop lasts H steps, cumulative rewards are finite, and sampled segments equal single-MDP batches"""
    from colosseum_b200 import suite

    insts = suite.load_suite_all(GOLDEN)
    for episodic in (True, False):
        tbs = [x.tables for x in insts if (x.tables.H > 0) == episodic][:128]
        kw = next(c[2] for c in CASES if c[0] == ("epi_hoeffding" if episodic else "cont"))
        mixed = _mixed(al, tbs, kw, 2, 0)
        steps = 300
        mixed.steps(steps)
        cum, ep = _np(mixed.cumulative_reward), _np(mixed.n_episodes)
        for i, tb in enumerate(tbs):
            sl = mixed.segment(i)
            assert np.all(np.isfinite(cum[sl])), i
            assert np.all(ep[sl] == (steps // tb.H if episodic else 0)), i
        for i in (0, 77, 127):
            one = _single(al, tbs[i], kw, 2, 0)
            one.steps(steps)
            sl = mixed.segment(i)
            assert np.array_equal(_np(mixed.table("Q", i)), _np(one.Q)), i
            assert np.array_equal(_np(mixed.cumulative_reward[sl]), _np(one.cumulative_reward)), i


def _create(handle, episodic, insts):
    lib = _cabi.lib()
    arr = (_cabi.QLearningInst * len(insts))(*insts)
    out = C.c_void_p()
    before = lib.colo_launch_count()
    rc = lib.colo_mixed_qlearning_create(handle, episodic, arr, None, C.byref(out))
    assert lib.colo_launch_count() == before
    if out.value:
        lib.colo_mixed_qlearning_destroy(out.value)
    return rc, _cabi.last_error(), out.value


def test_create_rejections_name_the_instance(goldens):
    from colosseum_b200.batched_mdp import MixedBatchedMDP

    epi, cont = (MDPTables.from_golden(goldens[n]) for n in ("c1_riverswim_epi", "riverswimcontinuous_ergo0"))
    good = _cabi.QLearningInst(log_term=2.0, sqrt_h7sa=3.0, H_eff=5.0, gamma=0.8, span_approx=1.0)

    dense = MixedBatchedMDP([epi, epi], 2, mode="dense_f32", track_visits=False)
    rc, err, h = _create(dense._handle, 1, [good, good])
    assert rc == -2 and h is None and "successor" in err

    env = MixedBatchedMDP([epi, epi, cont], 2, mode="succ", track_visits=False)
    rc, err, h = _create(env._handle, 1, [good] * 3)
    assert rc == -2 and h is None and "instance 2" in err and "H > 0" in err
    env = MixedBatchedMDP([cont, epi], 2, mode="succ", track_visits=False)
    rc, err, h = _create(env._handle, 0, [good] * 2)
    assert rc == -2 and h is None and "instance 1" in err and "H == 0" in err

    env = MixedBatchedMDP([cont, cont, cont], [1, 2, 3], mode="succ", track_visits=False)
    bad = _cabi.QLearningInst(log_term=float("nan"), sqrt_h7sa=0.0, H_eff=5.0, gamma=0.8, span_approx=1.0)
    rc, err, h = _create(env._handle, 0, [good, bad, good])
    assert rc == -2 and h is None and "instance 1" in err and "finite" in err
    bad = _cabi.QLearningInst(log_term=2.0, sqrt_h7sa=0.0, H_eff=0.0, gamma=0.8, span_approx=1.0)
    rc, err, h = _create(env._handle, 0, [good, good, bad])
    assert rc == -2 and h is None and "instance 2" in err and "H_eff" in err
    rc, err, h = _create(env._handle, 0, [good] * 3)
    assert rc == 0 and h is not None
