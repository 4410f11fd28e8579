"""GPU: the model-based continuous agents as device loops (csrc/continuous_agents.cu, csrc/extended_vi.cu through
colosseum_b200.agent_loop) against the oracle -- itself pinned to the reference's agent classes by
tests/golden/make_ucrl2_golden.py / make_psrlc_golden.py -- and, where the reference package is staged, against the
unmodified reference class directly."""
import importlib
import os
import sys

import numpy as np
import pytest

from conftest import GOLDEN, load_instance
from colosseum_b200.tables import MDPTables
from oracle import oracle as orc

sys.path.insert(0, GOLDEN)
from make_qlearning_golden import host_tables  # noqa: E402
from make_ucrl2_golden import CASES as UCASES, N_LOOPS as UN, N_STEPS as UT, SEED as USEED  # noqa: E402

pytestmark = pytest.mark.gpu


def _ucrl2_pairs(dev, cpu):
    return [("N", dev.N, cpu.Nsas), ("Nsa", dev.Nsa, cpu.Nsa), ("P", dev.P, cpu.P),
            ("est_r", dev.estimated_rewards, cpu.est_r), ("var_r", dev.variance_proxy_reward, cpu.var_r),
            ("hold", dev.estimated_holding_times, cpu.hold), ("iteration", dev.iteration, cpu.iteration),
            ("episode", dev.episode, cpu.episode), ("delta", dev.delta, cpu.delta), ("state", dev.state, cpu.state),
            ("time", dev.time, cpu.t), ("cum_reward", dev.cumulative_reward, cpu.cum_reward), ("nu", dev.nu, cpu.nu),
            ("ep_len", dev.ep_len, cpu.ep_len)]


@pytest.mark.parametrize("name,inst,kw", UCASES, ids=[c[0] for c in UCASES])
def test_ucrl2_kernels_equal_oracle_bit_for_bit(name, inst, kw):
    """Steps, artificial-episode ends, bounds and model updates of N loops: kernel == oracle bit for bit.  Both sides act
    on the SAME Q after every episode end (the oracle's extended VI, looked up by (loop, episode)), so one flipped
    near-tie cannot hide behind a diverged trajectory; the device planner is checked against that Q at every call."""
    import torch

    import colosseum_b200.agent_loop as al

    tb = MDPTables.from_golden(load_instance(inst))
    N, n_steps, seed = 37, 1500, 11
    cpu = orc.UCRL2Loops(host_tables(tb), N, n_steps + 1, seed=seed, record=True, **kw)
    tr_c = cpu.steps(n_steps, trace=True)
    worst = {"beta": 0.0, "Q": 0.0, "calls": 0}

    def planner(ag, idx, br, bp):
        ids = idx.cpu().numpy()
        ep = ag.episode.cpu().numpy()
        want = [cpu.history[(int(i), int(ep[i]))] for i in ids]
        for k, (_, br_c, bp_c) in enumerate(want):
            worst["beta"] = max(worst["beta"], float(np.abs(br[k].cpu().numpy() / br_c - 1).max()),
                                float(np.abs(bp[k].cpu().numpy() / bp_c - 1).max()))
        # the device planner on the same model, into scratch tables
        Qs, Vs = torch.zeros_like(ag.Q), torch.zeros_like(ag.V)
        span, iters, status = ag.solve_optimistic_model(idx, br, bp, Qs, Vs)
        assert int(status.max()) == 0
        Qd = Qs[idx.long()].cpu().numpy()
        Qc = np.stack([w[0] for w in want])
        worst["Q"] = max(worst["Q"], float(np.abs(Qd - Qc).max()))
        worst["calls"] += len(ids)
        ag.Q[idx.long()] = torch.from_numpy(Qc).cuda()

    dev = al.UCRL2Continuous(seed, tb, n_steps + 1, n_loops=N, planner=planner, **kw)
    tr_d = torch.cat([dev.steps(400, trace=True), dev.steps(n_steps - 400, trace=True)]).cpu().numpy()
    assert np.array_equal(tr_d, tr_c)
    for f, d, c in _ucrl2_pairs(dev, cpu):
        assert np.array_equal(d.cpu().numpy(), c), f
    assert worst["calls"] > 10 * N
    assert worst["beta"] < 1e-14, worst  # log() is the one operation that is not correctly rounded on both sides
    assert worst["Q"] < 2e-3, worst      # the extended VI stops at eps = 1e-3 (infinite_horizon.py:111)


def test_ucrl2_golden_trace_and_reference_tables():
    """the complete device agent (its own batched extended VI as the planner): every loop's trajectory is replayed by
    the oracle acting on the DEVICE's Q of each episode -- same trajectory, same episode ends, bit-identical model tables
    -- i.e. the device loop is a valid run of the agent the golden file pins to the reference class."""
    import torch

    import colosseum_b200.agent_loop as al

    name, inst, kw = UCASES[1]
    tb = MDPTables.from_golden(load_instance(inst))
    N, n_steps, seed = 64, 3000, 5
    hist = {}

    class Recording(al.UCRL2Continuous):
        def episode_end_update(self, idx, update_model=True):
            super().episode_end_update(idx, update_model)
            ep = self.episode.cpu().numpy()
            Q = self.Q[idx.long()].cpu().numpy()
            for k, i in enumerate(idx.cpu().numpy()):
                hist[(int(i), int(ep[i]))] = Q[k]

    dev = Recording(seed, tb, n_steps + 1, n_loops=N, **kw)
    tr_d = dev.steps(n_steps, trace=True).cpu().numpy()
    assert dev.rounds > 20 and dev.evi_iterations > 0

    def planner(i, episode, P, est, br, bp, r_max):
        return 0.0, hist[(i, episode)], np.zeros(tb.S, np.float32)

    cpu = orc.UCRL2Loops(host_tables(tb), N, n_steps + 1, seed=seed, planner=planner, **kw)
    tr_c = cpu.steps(n_steps, trace=True)
    assert np.array_equal(tr_d, tr_c)
    for f, d, c in _ucrl2_pairs(dev, cpu):
        assert np.array_equal(d.cpu().numpy(), c), f


def test_ucrl2_device_loop_through_the_reference_class():
    """where the reference package is staged (oracle/reference_import.py): the device loops' trajectories through the
    UNMODIFIED UCRL2Continuous -- its episode ends and model tables must be the device's, bit for bit, and its numba
    extended VI must land within the stopping tolerance of the device's Q."""
    from oracle.reference_import import reference_available

    if not reference_available():
        pytest.skip("the unmodified Colosseum package is not staged (oracle/_ref or $COLOSSEUM_REFERENCE_ROOT)")
    import colosseum_b200.agent_loop as al
    from make_qlearning_golden import reference_models
    from make_ucrl2_golden import mdp_spec, replay_reference

    reference_models()
    ucrl2 = importlib.import_module("colosseum.agent.agents.infinite_horizon.ucrl2")
    for name, inst, kw in UCASES[:2]:
        tb = MDPTables.from_golden(load_instance(inst))
        N, n_steps, seed = 4, 2500, USEED
        dev = al.UCRL2Continuous(seed, tb, n_steps + 1, n_loops=N, **kw)
        tr = dev.steps(n_steps, trace=True).cpu().numpy()
        for i in (0, N - 1):
            ag, ends = replay_reference(ucrl2, mdp_spec(tb), tr[:, i], n_steps + 1, kw, seed=seed)
            assert int(dev.episode[i]) == ag.episode and int(dev.iteration[i]) == ag.iteration, name
            assert float(dev.delta[i]) == ag.delta
            for d, r in ((dev.N[i], ag.N), (dev.P[i], ag.P), (dev.estimated_rewards[i], ag.estimated_rewards),
                         (dev.variance_proxy_reward[i], ag.variance_proxy_reward),
                         (dev.estimated_holding_times[i], ag.estimated_holding_times)):
                assert np.array_equal(d.cpu().numpy(), r), name
            assert np.abs(dev.Q[i].cpu().numpy() - ag.Q).max() < 2e-3, name


def test_extended_vi_batched_equals_single_instance():
    """colo_extended_vi_batched_f32 (one CTA per listed instance) == colo_extended_vi_f32 (one launch per iteration),
    bit for bit, on the reference's numba goldens (tests/golden/evi.npz) -- listed out of order, with an unlisted
    instance left untouched."""
    import ctypes as C

    import torch

    from colosseum_b200 import _cabi

    gold = np.load(os.path.join(GOLDEN, "evi.npz"))
    lib = _cabi.lib()
    for nm in range(int(gold["n_cases"])):
        T, est = gold[f"P_{nm}"], gold[f"est_{nm}"]
        br, bp = gold[f"beta_r_{nm}"], gold[f"beta_p_{nm}"]
        r_max = 1.0
        S, A, _ = T.shape
        bp = np.ascontiguousarray(bp[..., 0] if bp.ndim == 3 else bp).reshape(S, A)
        # three instances: the golden model, a perturbed one, and one that is not listed
        Ts = torch.from_numpy(np.stack([T, T, T])).cuda()
        ests = torch.from_numpy(np.stack([est, est * 0.5, est])).cuda().float()
        idx = torch.tensor([1, 0], dtype=torch.int32, device="cuda")
        brd = torch.from_numpy(np.stack([br, br])).cuda().double().contiguous()
        bpd = torch.from_numpy(np.stack([bp * 2.0, bp])).cuda().double().contiguous()
        Q = torch.full((3, S, A), -7.0, dtype=torch.float32, device="cuda")
        V = torch.full((3, S), -7.0, dtype=torch.float32, device="cuda")
        span = torch.zeros(2, dtype=torch.float64, device="cuda")
        iters = torch.zeros(2, dtype=torch.int64, device="cuda")
        status = torch.zeros(2, dtype=torch.int32, device="cuda")
        rc = lib.colo_extended_vi_batched_f32(Ts.data_ptr(), ests.data_ptr(), brd.data_ptr(), bpd.data_ptr(),
                                              idx.data_ptr(), 2, S, A, r_max, 1e-3, int(1e6), Q.data_ptr(), V.data_ptr(),
                                              span.data_ptr(), iters.data_ptr(), status.data_ptr(), _cabi.current_stream())
        _cabi.check(rc, "colo_extended_vi_batched_f32")
        assert status.cpu().tolist() == [0, 0]
        assert float(Q[2].max()) == -7.0 and float(V[2].max()) == -7.0
        work = torch.empty(lib.colo_extended_vi_work_bytes(S, 0), dtype=torch.uint8, device="cuda")
        for k, inst in enumerate((1, 0)):
            Q1 = torch.empty((S, A), dtype=torch.float32, device="cuda")
            V1 = torch.empty(S, dtype=torch.float32, device="cuda")
            out = (C.c_double * 2)()
            rc = lib.colo_extended_vi_f32(Ts[inst].data_ptr(), ests[inst].data_ptr(), brd[k].data_ptr(), bpd[k].data_ptr(),
                                          S, A, r_max, 1e-3, int(1e6), Q1.data_ptr(), V1.data_ptr(), out, work.data_ptr(),
                                          _cabi.current_stream())
            _cabi.check(rc, "colo_extended_vi_f32")
            assert torch.equal(Q1, Q[inst]) and torch.equal(V1, V[inst]), nm
            assert out[0] == float(span[k]) and int(out[1]) == int(iters[k]), nm
        # and the golden of the reference's numba run, within the stopping tolerance
        assert np.abs(Q[0].cpu().numpy() - gold[f"Q_{nm}_loose"]).max() < 2e-3 + 3e-6, nm


def test_ucrl2_learns_river_swim():
    """256 loops on RiverSwimContinuous (optimal average reward 0.889, uniformly random policy 0.017): the batch's
    reward rate over the last fifth of 30,000 steps is above 0.7 (measured 0.85; first fifth 0.61)."""
    import colosseum_b200.agent_loop as al

    tb = MDPTables.from_golden(load_instance("riverswimcontinuous_ergo0"))
    T = 30000
    ag = al.UCRL2Continuous(0, tb, T + 1, alpha_r=0.1, alpha_p=0.05, n_loops=256)
    ag.steps(T * 4 // 5)
    before = float(ag.cumulative_reward.mean())
    ag.steps(T // 5)
    rate = (float(ag.cumulative_reward.mean()) - before) / (T // 5)
    assert rate > 0.7, rate
    assert int(ag.time.min()) == int(ag.time.max()) == T + 1 and int(ag.ended.max()) == 0


# ------------------------------------------------------------------------------------------------- PSRLContinuous
import make_psrlc_golden as pmk  # noqa: E402


def _psrlc_pairs(dev, cpu):
    return [("N", dev.N, cpu.Nsas), ("Nsa", dev.Nsa, cpu.Nsa), ("dir", dev.dir_hyper, cpu.dir_hyper),
            ("nig", dev.nig_hyper, cpu.nig_hyper), ("episode", dev.episode, cpu.episode), ("state", dev.state, cpu.state),
            ("time", dev.time, cpu.t), ("cum_reward", dev.cumulative_reward, cpu.cum_reward), ("nu", dev.nu, cpu.nu),
            ("Q", dev.Q, cpu.Q)]


def _agent_kwargs(kw):
    return {k: v for k, v in kw.items() if k != "reward_prior_model"} | (
        {"reward_prior_model": kw["reward_prior_model"]} if "reward_prior_model" in kw else {})


@pytest.mark.parametrize("name,inst,kw", pmk.CASES, ids=[c[0] for c in pmk.CASES])
def test_psrl_continuous_kernels_equal_oracle_bit_for_bit(name, inst, kw):
    """steps, extended-action decoding, posterior updates and artificial-episode ends of N loops: kernel == oracle bit
    for bit, both sides acting on the same extended q-values after every re-planning (the oracle's deterministic
    planner, looked up by (loop, episode)).  At every re-planning the device's optimistic sampling is checked on the same
    posterior: the under-visited rows against the reference's own expressions with the same z, the Dirichlet rows and
    the reward layout structurally."""
    import torch

    import colosseum_b200.agent_loop as al

    tb = MDPTables.from_golden(load_instance(inst))
    N, n_steps, seed = 29, 1200, 7
    prm = pmk.parameters(tb, kw, n_steps + 1)
    hist = {}
    base = pmk.make_planner(prm)

    def cpu_planner(loops, idx):
        base(loops, idx)
        for i in idx:
            hist[(int(i), int(loops.episode[i]))] = loops.Q[i].copy()

    cpu = orc.PSRLCLoops(host_tables(tb), N, prm["psi"], seed=seed, planner=cpu_planner, **pmk.loop_kwargs(kw))
    tr_c = cpu.steps(n_steps, trace=True)
    seen = {"simple_rows": 0, "posterior_rows": 0, "worst_simple": 0.0, "worst_rowsum": 0.0}
    S, A = tb.S, tb.A

    def planner(ag, idx):
        ids = idx.cpu().numpy()
        ep = ag.episode.cpu().numpy()
        T_ext, R_ext = ag.sample_models(idx)
        psi = ag._psi
        Tn = T_ext.cpu().numpy().reshape(len(ids), S, A, psi, S)
        Rn = R_ext.cpu().numpy()
        assert np.isfinite(Tn).all() and np.isfinite(Rn).all() and (Tn >= 0).all()
        assert np.array_equal(Rn, np.tile(Rn[:, :, :A], (1, 1, psi)))  # np.tile(R, (1, psi)), :371-372
        Nn = ag.N[idx.long()].cpu().numpy()
        for k, i in enumerate(ids):
            cond = Nn[k].sum(-1) < ag._eta
            for q in range(psi):
                if cond.any():
                    z = orc.psrlc_z(seed, int(i), int(ep[i]), q, S)
                    want = orc.psrlc_simple_rows(Nn[k], z)
                    seen["worst_simple"] = max(seen["worst_simple"], float(np.abs(Tn[k][:, :, q][cond] - want[cond]).max()))
                if (~cond).any():
                    seen["worst_rowsum"] = max(seen["worst_rowsum"], float(np.abs(Tn[k][:, :, q][~cond].sum(-1) - 1).max()))
            seen["simple_rows"] += int(cond.sum())
            seen["posterior_rows"] += int((~cond).sum())
        ag.Q[idx.long()] = torch.from_numpy(np.stack([hist[(int(i), int(ep[i]))] for i in ids])).cuda()

    akw = {k: v for k, v in kw.items()}
    dev = al.PSRLContinuous(seed, tb, n_steps + 1, n_loops=N, planner=planner, **akw)
    assert (dev._psi, dev.omega, dev.kappa, dev._eta) == (prm["psi"], prm["omega"], prm["kappa"], prm["eta"])
    tr_d = torch.cat([dev.steps(500, trace=True), dev.steps(n_steps - 500, trace=True)]).cpu().numpy()
    assert np.array_equal(tr_d, tr_c)
    for f, d, c in _psrlc_pairs(dev, cpu):
        assert np.array_equal(d.cpu().numpy(), c), f
    assert seen["posterior_rows"] > 0
    assert seen["worst_simple"] < 1e-7 and seen["worst_rowsum"] < 1e-4, seen
    if not prm["no_optimistic_sampling"]:
        assert seen["simple_rows"] > 0


def test_psrl_continuous_sampled_models_follow_the_posterior():
    """moments of the device's model samples against the posterior they are drawn from: Dirichlet rows (mean alpha /
    alpha_0, variance alpha_j (alpha_0 - alpha_j) / (alpha_0^2 (alpha_0 + 1))) and the N_NIG reward marginal (mean mu),
    over 600 re-plannings of one fixed posterior, for both samplers."""
    import torch

    import colosseum_b200.agent_loop as al

    tb = MDPTables.from_golden(load_instance("riverswimcontinuous_ergo0"))
    S, A = tb.S, tb.A
    for sampler in ("fast", "f64"):
        ag = al.PSRLContinuous(3, tb, 10_000, psi_weight=0.02, eta_weight=1e-9, n_loops=2, sampler=sampler)
        ag.steps(3000)
        idx = torch.tensor([1], dtype=torch.int32, device="cuda")
        alpha = ag.dir_hyper[1].double().cpu().numpy()
        visited = (ag.Nsa[1].cpu().numpy() >= ag._eta)
        assert visited.sum() >= 4
        acc, acc2, racc, n = 0.0, 0.0, 0.0, 0
        for rep in range(600):
            ag.episode[1] = 10_000 + rep  # a fresh draw counter, the posterior untouched
            T_ext, R_ext = ag.sample_models(idx)
            t = T_ext[0].double().cpu().numpy().reshape(S, A, ag._psi, S)
            acc, acc2 = acc + t.sum(2), acc2 + (t ** 2).sum(2)
            racc = racc + R_ext[0, :, :A].double().cpu().numpy()
            n += ag._psi
        mean, var = acc / n, acc2 / n - (acc / n) ** 2
        a0 = alpha.sum(-1, keepdims=True)
        want_mean, want_var = alpha / a0, alpha * (a0 - alpha) / (a0 ** 2 * (a0 + 1))
        se = np.sqrt(want_var / n) + 1e-4
        assert (np.abs(mean - want_mean)[visited] < 6 * se[visited]).all(), sampler
        big = visited[..., None] & (want_var > 1e-4)
        ratio = var[big] / want_var[big]  # sample variances of skewed marginals from 600 * psi draws: noisy one by one
        assert big.sum() > 4 and abs(np.median(ratio) - 1) < 0.1 and (np.abs(ratio - 1) < 0.6).mean() > 0.98, sampler
        hp = ag.nig_hyper[1].double().cpu().numpy()
        # marginal of the mean: Student-t centred at mu with scale sqrt(beta / (alpha lambda)); alpha > 1 after visits
        ok = visited & (hp[..., 2] > 2)
        sd = np.sqrt(hp[..., 3] / ((hp[..., 2] - 1) * hp[..., 1]))
        assert ok.sum() >= 4 and (np.abs(racc / 600 - hp[..., 0])[ok] < 6 * sd[ok] / np.sqrt(600) + 1e-4).all(), sampler


def test_psrl_continuous_device_loop_replays_and_learns():
    """the complete device agent (its own sampling and batched value iteration): the oracle, acting on the DEVICE's
    extended q-values of each re-planning, reproduces every trajectory and posterior bit for bit; and the batch learns
    RiverSwim (optimal average reward 0.889, random policy 0.017)."""
    import colosseum_b200.agent_loop as al

    tb = MDPTables.from_golden(load_instance("riverswimcontinuous_ergo0"))
    N, n_steps, seed = 48, 6000, 9
    kw = dict(psi_weight=0.015, eta_weight=1e-9)
    prm = pmk.parameters(tb, kw, n_steps + 1)
    hist = {}

    class Recording(al.PSRLContinuous):
        def episode_end_update(self, idx):
            ep = self.episode.cpu().numpy().copy()
            super().episode_end_update(idx)
            Q = self.Q[idx.long()].cpu().numpy()
            for k, i in enumerate(idx.cpu().numpy()):
                hist[(int(i), int(ep[i]))] = Q[k]

    dev = Recording(seed, tb, n_steps + 1, n_loops=N, **kw)
    tr_d = dev.steps(n_steps, trace=True).cpu().numpy()
    assert dev.rounds > 20 and dev.vi_sweeps > 0

    def planner(loops, idx):
        for i in idx:
            loops.Q[i] = hist[(int(i), int(loops.episode[i]))]

    cpu = orc.PSRLCLoops(host_tables(tb), N, prm["psi"], seed=seed, planner=planner)
    tr_c = cpu.steps(n_steps, trace=True)
    assert np.array_equal(tr_d, tr_c)
    for f, d, c in _psrlc_pairs(dev, cpu):
        assert np.array_equal(d.cpu().numpy(), c), f
    r = tr_d[..., 3].view(np.float32)
    assert r[-n_steps // 4:].mean() > 0.5, r[-n_steps // 4:].mean()


def test_psrl_continuous_device_loop_through_the_reference_class():
    """where the reference package is staged: the device loops' trajectories through the UNMODIFIED PSRLContinuous -- its
    episode ends, visit counts and posteriors must be the device's, bit for bit."""
    from oracle.reference_import import reference_available

    if not reference_available():
        pytest.skip("the unmodified Colosseum package is not staged (oracle/_ref or $COLOSSEUM_REFERENCE_ROOT)")
    import colosseum_b200.agent_loop as al
    from make_qlearning_golden import reference_models
    from make_ucrl2_golden import mdp_spec

    reference_models()
    psrl = importlib.import_module("colosseum.agent.agents.infinite_horizon.posterior_sampling")
    for name, inst, kw in pmk.CASES[:2]:
        tb = MDPTables.from_golden(load_instance(inst))
        N, n_steps, seed = 3, 1500, pmk.SEED
        dev = al.PSRLContinuous(seed, tb, n_steps + 1, n_loops=N, **kw)
        tr = dev.steps(n_steps, trace=True).cpu().numpy()
        for i in (0, N - 1):
            ag, ends = pmk.replay_reference(psrl, mdp_spec(tb), tr[:, i], dev._psi, n_steps + 1, kw, seed=seed)
            assert int(dev.episode[i]) == len(ends) + 1, name  # + the plan of before_start_interacting
            assert (ag.psi, ag.omega, ag.kappa, ag.eta) == (dev.psi, dev.omega, dev.kappa, dev.eta)
            assert np.array_equal(dev.N[i].cpu().numpy(), ag.N), name
            assert np.array_equal(dev.dir_hyper[i].cpu().numpy(), ag._mdp_model._transitions_model.hyper_params), name
            k = ag._mdp_model._rewards_model.hyper_params.shape[-1]
            assert np.array_equal(dev.nig_hyper[i, ..., :k].cpu().numpy(), ag._mdp_model._rewards_model.hyper_params), name
