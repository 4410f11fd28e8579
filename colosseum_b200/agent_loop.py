"""N independent agent/MDP interaction loops on the device (SURVEY.md section 8(f)-4).

The reference runs one `MDPLoop` (colosseum/experiment/agent_mdp_interaction.py:160-298) per (agent, MDP, seed) and
spreads the seeds over processes.  Here the N loops of one (agent class, MDP) pair -- N seeds -- are the lanes of one
kernel (`csrc/agents.cu`): every loop owns its env and its agent tables, and `log_every` iterations of MDPLoop.run's
body execute per launch.  Classes keep the reference's names and constructor arguments:

    QLearningEpisodic   colosseum/agent/agents/episodic/q_learning.py:106-240   (Jin et al. 2018; Hoeffding / Bernstein)
    QLearningContinuous colosseum/agent/agents/infinite_horizon/q_learning.py:114-255 (Wei et al. 2020)
    BatchedMDPLoop.run(T, log_every)  MDPLoop.run: cumulative reward per loop, and at every log tick the expected
                        regret of each loop's greedy policy (experiment/indicators.py:29-45 / markov_chain.py:12-31)
    MixedQLearningEpisodic, MixedQLearningContinuous, MixedBatchedMDPLoop
                        the same loops on many MDP instances at once (a benchmark's instances x seeds), one launch

`mdp_specs` is replaced by the `MDPTables` of the MDP (the kernel needs the sampler tables, not only the sizes).
`epsilon_greedy` and `boltzmann_temperature` are constants or, as in the reference, functions of the actor's interaction
counter (tabulated per launch, `_set_actor`).
"""
import ctypes as C
import time

import numpy as np

from . import _cabi
from .batched_mdp import DeviceTables
from .tables import MDPTables


def get_H(n_states, n_actions, T, span_approx, confidence):
    """infinite_horizon/q_learning.py:21-45"""
    return min(np.sqrt(span_approx * T / n_states / n_actions),
               (T / n_states / n_actions / np.log(4 * T / confidence)) ** 0.333)


def _set_actor(agents, t0, n):
    """QValuesActor's exploration for the interaction counts t0 .. t0 + n - 1 (Q_values_actor.py:20-82) into the
    argument struct of `agents`: constants as they are; functions of the actor's interaction counter -- the only form the
    reference itself can run, its float branch wraps the number into a lambda that returns itself (:44-49) -- are
    tabulated on the host and uploaded (f64 [n])."""
    import torch

    args, a = agents._args, agents._args.actor
    eps, temp = agents._explore
    a.t0, a.len = int(t0), int(n)
    a.epsilon_schedule = a.temperature_schedule = None
    args.epsilon_greedy = -1.0
    agents._schedules = keep = {}
    if callable(eps):
        keep["eps"] = torch.tensor([float(eps(t0 + k)) for k in range(n)], dtype=torch.float64).cuda()
        a.epsilon_schedule = keep["eps"].data_ptr()
        args.epsilon_greedy = 0.0
    elif eps is not None:
        args.epsilon_greedy = float(eps)
    a.boltzmann = int(temp is not None)
    if callable(temp):
        keep["temp"] = torch.tensor([float(temp(t0 + k)) for k in range(n)], dtype=torch.float64).cuda()
        a.temperature_schedule = keep["temp"].data_ptr()
    elif temp is not None:
        a.boltzmann_temperature = float(temp)


class _QLearningBatch:
    episodic = None

    def _alloc(self, tables: MDPTables, n_loops: int, seed: int, env_offset: int, epsilon_greedy, boltzmann_temperature):
        import torch

        _cabi.require_cuda()
        self._explore = (epsilon_greedy, boltzmann_temperature)
        assert (tables.H > 0) == self.episodic, "episodic agents need an episodic MDP and vice versa"
        self.torch = torch
        self.tables = tables
        self.dev = DeviceTables(tables, "succ")
        self.n_loops = N = int(n_loops)
        self.seed, self.env_offset = int(seed), int(env_offset)
        self.t = 0
        S, A = tables.S, tables.A
        self.state = torch.zeros(N, dtype=torch.int32, device="cuda")
        self.h = torch.zeros(N, dtype=torch.int32, device="cuda")
        self.cumulative_reward = torch.zeros(N, dtype=torch.float64, device="cuda")
        self.n_episodes = torch.zeros(N, dtype=torch.int64, device="cuda")
        a = _cabi.QLearningArgs()
        a.N, a.seed, a.env0 = N, self.seed, self.env_offset
        a.state, a.h = self.state.data_ptr(), self.h.data_ptr()
        a.cum_reward, a.n_episodes = self.cumulative_reward.data_ptr(), self.n_episodes.data_ptr()
        self._args = a
        self._fn = (_cabi.lib().colo_qlearning_episodic_steps if self.episodic
                    else _cabi.lib().colo_qlearning_continuous_steps)
        self.reset_envs()
        return S, A

    def reset_envs(self):
        """mdp.reset() for every loop: start states drawn with the env Philox stream at counter t (as colo_env_reset)"""
        torch = self.torch
        tb = self.tables
        if tb.n_start == 1:
            self.state.fill_(int(tb.start_idx[0]))
        else:
            from .batched_mdp import BatchedMDP

            env = BatchedMDP(tb, self.n_loops, mode="succ", seed=self.seed, env_offset=self.env_offset,
                             track_visits=False)
            env.t = self.t
            env.reset()
            self.state.copy_(env.state)
        self.h.zero_()
        self.t += 1
        torch.cuda.current_stream().synchronize()

    def steps(self, n_steps: int, trace: bool = False):
        """n_steps iterations of the interaction loop for every loop, one launch.  trace=True returns
        i32 [n_steps, N, 4] = (s_t, a_t, obs_tp1, reward bits)."""
        torch = self.torch
        tr = torch.empty((n_steps, self.n_loops, 4), dtype=torch.int32, device="cuda") if trace else None
        self._args.trace = None if tr is None else tr.data_ptr()
        _set_actor(self, self.t, n_steps)
        rc = self._fn(C.byref(self.dev.c), C.byref(self._args), int(n_steps), self.t, _cabi.current_stream())
        _cabi.check(rc, "colo_qlearning_steps")
        self.t += int(n_steps)
        return tr

    def current_optimal_stochastic_policy(self, i: int) -> np.ndarray:
        """get_policy_from_q_values(Q, True) of loop i (q_learning.py:164-166)"""
        from .dynamic_programming import get_policy_from_q_values

        return get_policy_from_q_values(self.Q[i].cpu().numpy(), True)


class QLearningEpisodic(_QLearningBatch):
    episodic = True

    def __init__(self, seed: int, tables: MDPTables, optimization_horizon: int, p: float, c_1: float,
                 c_2: float = None, min_at: float = 0, UCB_type="hoeffding", epsilon_greedy=None,
                 boltzmann_temperature=None, *, n_loops: int = 1, env_offset: int = 0):
        UCB_type = UCB_type.lower()
        assert 0 <= min_at < 0.99 and 0 < p < 1 and c_1 > 0 and UCB_type in ("hoeffding", "bernstein")
        if UCB_type == "bernstein":
            assert c_2 is not None and c_2 > 0
        S, A = self._alloc(tables, n_loops, seed, env_offset, epsilon_greedy, boltzmann_temperature)
        torch, N, H = self.torch, self.n_loops, tables.H
        self.N = torch.ones((N, H, S, A), dtype=torch.int32, device="cuda")          # q_learning.py:44
        self.Q = torch.full((N, H, S, A), float(H), dtype=torch.float32, device="cuda")  # :45-47
        self.V = torch.zeros((N, H + 1, S), dtype=torch.float32, device="cuda")      # :48
        a = self._args
        a.cnt, a.Q, a.V = self.N.data_ptr(), self.Q.data_ptr(), self.V.data_ptr()
        a.ucb_type = 0
        if UCB_type == "bernstein":
            self.mu = torch.zeros((N, H, S, A), dtype=torch.float32, device="cuda")
            self.sigma = torch.zeros_like(self.mu)
            self.beta = torch.zeros_like(self.mu)
            a.mu, a.sigma, a.beta = self.mu.data_ptr(), self.sigma.data_ptr(), self.beta.data_ptr()
            a.ucb_type = 1
            a.c_2 = float(c_2)
        a.c_1, a.min_at = float(c_1), float(min_at)
        a.log_term = float(np.log(S * A * optimization_horizon / p))                 # :43
        a.sqrt_h7sa = float(np.sqrt(H ** 7 * S * A))
        self.i = a.log_term


class QLearningContinuous(_QLearningBatch):
    episodic = False

    def __init__(self, seed: int, tables: MDPTables, optimization_horizon: int, min_at: float = 0,
                 confidence: float = 0.95, span_approx_weight: float = 1, get_span_approx=None, h_weight: float = 1,
                 get_H=get_H, epsilon_greedy=None, boltzmann_temperature=None, *, n_loops: int = 1,
                 env_offset: int = 0):
        assert 0 <= min_at < 0.99 and 0 < confidence < 1 and span_approx_weight > 0 and h_weight > 0
        S, A = self._alloc(tables, n_loops, seed, env_offset, epsilon_greedy, boltzmann_temperature)
        torch, N = self.torch, self.n_loops
        self.min_at = min_at if min_at > 0.009 else 0                                # :62
        self.span_approx = span_approx_weight
        if get_span_approx is not None:
            self.span_approx *= get_span_approx(S, A)
        self.H = float(h_weight * get_H(S, A, optimization_horizon, self.span_approx, confidence))
        self.gamma = 1 - 1 / self.H
        self.N = torch.zeros((N, S, A), dtype=torch.int32, device="cuda")
        self.Q = torch.full((N, S, A), self.H, dtype=torch.float32, device="cuda")
        self.Q_main = torch.full((N, S, A), self.H, dtype=torch.float32, device="cuda")
        self.V = torch.full((N, S), self.H, dtype=torch.float32, device="cuda")
        a = self._args
        a.cnt, a.Q, a.Q_main, a.V = self.N.data_ptr(), self.Q.data_ptr(), self.Q_main.data_ptr(), self.V.data_ptr()
        a.min_at, a.H_eff, a.gamma, a.span_approx = float(self.min_at), self.H, float(self.gamma), float(self.span_approx)
        a.log_term = float(np.log(2 * optimization_horizon / confidence))


class PSRLEpisodic:
    """N PSRLEpisodic loops (colosseum/agent/agents/episodic/posterior_sampling.py:20-147; Osband et al. 2013) with
    the N_NIG reward model and the M_DIR transition model (the agent's defaults,
    agent/mdp_models/bayesian_model.py:44-57).  Every H steps: one Dirichlet sample of all N*S*A rows
    (colo_sample_dirichlet_rows), one Normal-Inverse-Gamma sample (colo_sample_nig_rewards), one batched episodic value
    iteration (colo_episodic_f32, B = N); in between, `colo_psrl_episodic_steps` acts and updates the posteriors.
    The sampled models never leave HBM."""

    episodic = True

    def __init__(self, seed: int, tables: MDPTables, optimization_horizon: int, reward_prior_model=None,
                 transitions_prior_model=None, rewards_prior_prms=None, transitions_prior_prms=None,
                 epsilon_greedy=None, boltzmann_temperature=None, *, n_loops: int = 1, env_offset: int = 0,
                 sampler: str = "fast"):
        import torch

        _cabi.require_cuda()
        assert sampler in ("fast", "f64")
        self._dirichlet = (_cabi.lib().colo_sample_dirichlet_rows_fast if sampler == "fast"
                           else _cabi.lib().colo_sample_dirichlet_rows)
        rname = getattr(reward_prior_model, "name", reward_prior_model)   # the reference's IntEnum or its name
        tname = getattr(transitions_prior_model, "name", transitions_prior_model)
        assert rname in (None, "N_NIG", "N_N") and tname in (None, "M_DIR"), \
            "the batched PSRL offers the N_NIG / N_N reward models and the M_DIR transition model"
        self.reward_model = 1 if rname == "N_N" else 0
        self._explore = (epsilon_greedy, boltzmann_temperature)
        assert tables.H > 0, "PSRLEpisodic needs an episodic MDP"
        self.torch, self.tables = torch, tables
        self.dev = DeviceTables(tables, "succ")
        self.n_loops = N = int(n_loops)
        self.seed, self.env_offset = int(seed), int(env_offset)
        S, A, H = tables.S, tables.A, tables.H
        rp = [tables.rmax, 1, 1, 1] if rewards_prior_prms is None else rewards_prior_prms       # bayesian_model.py:46-48
        tp = [1.0 / S] if transitions_prior_prms is None else transitions_prior_prms              # :49-51
        if self.reward_model == 1:  # N_N: (mu, tau) in the first two of the four slots (conjugate_rewards.py:95-110)
            hp = np.zeros((S, A, 4), np.float32)
            hp[..., :2] = np.tile(rp, (S, A, 1)).astype(np.float32)
        else:
            hp = np.tile(rp, (S, A, 1)).astype(np.float32)                                        # base_conjugate.py:44-47
            mu, n_mu, tau, n_tau = (hp[..., k].copy() for k in range(4))
            hp[..., 2], hp[..., 3] = n_tau * 0.5, (0.5 * n_tau) / tau                            # conjugate_rewards.py:45-54
        self.nig_hyper = torch.from_numpy(np.tile(hp, (N, 1, 1, 1))).cuda()
        self.dir_hyper = torch.full((N, S, A, S), float(np.float32(tp[0])), dtype=torch.float32, device="cuda")
        self.T_sample = torch.empty((N, S, A, S), dtype=torch.float32, device="cuda")
        self.R_sample = torch.empty((N, S, A), dtype=torch.float32, device="cuda")
        self.Q = torch.zeros((N, H + 1, S, A), dtype=torch.float32, device="cuda")
        self.state = torch.zeros(N, dtype=torch.int32, device="cuda")
        self.h = torch.zeros(N, dtype=torch.int32, device="cuda")
        self.cumulative_reward = torch.zeros(N, dtype=torch.float64, device="cuda")
        self.n_episodes = torch.zeros(N, dtype=torch.int64, device="cuda")
        self.t = 0          # Philox counter of the interaction steps
        self.n_samples = 0  # Philox counter of the posterior samples
        self._h_episode = 0
        a = _cabi.PsrlArgs()
        a.N, a.seed, a.env0 = N, self.seed, self.env_offset
        a.state, a.h, a.Q = self.state.data_ptr(), self.h.data_ptr(), self.Q.data_ptr()
        a.dir_hyper, a.nig_hyper = self.dir_hyper.data_ptr(), self.nig_hyper.data_ptr()
        a.cum_reward, a.n_episodes = self.cumulative_reward.data_ptr(), self.n_episodes.data_ptr()
        a.reward_model = self.reward_model
        self._args = a
        _QLearningBatch.reset_envs(self)
        self.episode_end_update()  # before_start_interacting (:146-147)

    def sample(self):
        """BayesianMDPModel.sample for every loop (bayesian_model.py:59-63): fills T_sample, R_sample"""
        lib = _cabi.lib()
        N, S, A = self.n_loops, self.tables.S, self.tables.A
        rows, row0 = N * S * A, self.env_offset * S * A
        st = _cabi.current_stream()
        rc = self._dirichlet(self.dir_hyper.data_ptr(), rows, S, row0, self.seed, self.n_samples,
                             self.T_sample.data_ptr(), st)
        _cabi.check(rc, "colo_sample_dirichlet_rows")
        sample_r = lib.colo_sample_nn_rewards if self.reward_model == 1 else lib.colo_sample_nig_rewards
        rc = sample_r(self.nig_hyper.data_ptr(), rows, row0, self.seed, self.n_samples, self.R_sample.data_ptr(), st)
        _cabi.check(rc, "colo_sample_rewards")
        self.n_samples += 1
        return self.T_sample, self.R_sample

    def episode_end_update(self):
        """posterior_sampling.py:142-144: Q = episodic_value_iteration(H, *model.sample())"""
        from .dynamic_programming import episodic_value_iteration

        T, R = self.sample()
        Q, _ = episodic_value_iteration(self.tables.H, T, R, precision="f32")
        self.Q.copy_(Q)

    def steps(self, n_steps: int, trace: bool = False):
        """n_steps interaction steps for every loop; the posterior is resampled at every episode end"""
        torch, H = self.torch, self.tables.H
        tr = torch.empty((n_steps, self.n_loops, 4), dtype=torch.int32, device="cuda") if trace else None
        done = 0
        while done < n_steps:
            n = min(H - self._h_episode, n_steps - done)
            self._args.trace = None if tr is None else tr[done:].data_ptr()
            _set_actor(self, self.t, n)
            rc = _cabi.lib().colo_psrl_episodic_steps(C.byref(self.dev.c), C.byref(self._args), n, self.t,
                                                      _cabi.current_stream())
            _cabi.check(rc, "colo_psrl_episodic_steps")
            self.t += n
            done += n
            self._h_episode = (self._h_episode + n) % H
            if self._h_episode == 0:
                self.episode_end_update()
        return tr

    def get_map_estimate(self):
        """BayesianMDPModel.get_map_estimate (bayesian_model.py:71-76) for every loop"""
        return self.dir_hyper / self.dir_hyper.sum(-1, keepdim=True), self.nig_hyper[..., 0]

    def current_optimal_stochastic_policy(self, i: int) -> np.ndarray:
        """posterior_sampling.py:76-80: greedy policy of the MAP model"""
        from .dynamic_programming import episodic_value_iteration, get_policy_from_q_values

        T_map, R_map = self.get_map_estimate()
        Q, _ = episodic_value_iteration(self.tables.H, T_map[i].contiguous(), R_map[i].contiguous(), precision="f32")
        return get_policy_from_q_values(Q.cpu().numpy(), True)


class UCRL2Continuous:
    """N UCRL2Continuous loops (colosseum/agent/agents/infinite_horizon/ucrl2.py:34-357; Auer et al. 2008, Fruit et al.
    2020) on one continuous MDP.  Artificial episodes end at loop-dependent times, so `steps` advances the batch in
    rounds: `colo_ucrl2_steps` runs every loop to its episode end or the target time; the loops that wait are listed and
    re-planned together -- `colo_ucrl2_bounds` (delta, beta_r, beta_p), `colo_extended_vi_batched_f32` (one CTA per
    listed loop, the whole optimistic value iteration in one launch), `colo_ucrl2_model_update` -- in the reference's
    order (plan on the old model, then update it, :183-192).  The models never leave HBM.

    Constructor arguments are the reference's (`mdp_specs` -> the MDP's tables).  bound_type_rew="bernstein" is refused:
    the reference's own branch reads `self.r_max`, which the class never defines (ucrl2.py:268)."""

    episodic = False

    def __init__(self, seed: int, tables: MDPTables, optimization_horizon: int, alpha_r=1.0, alpha_p=1.0,
                 bound_type_p="_chernoff", bound_type_rew="_chernoff", epsilon_greedy=None, boltzmann_temperature=None,
                 *, n_loops: int = 1, env_offset: int = 0, planner=None):
        import torch

        _cabi.require_cuda()
        assert bound_type_p in ("_chernoff", "bernstein") and bound_type_rew in ("_chernoff", "bernstein")
        if bound_type_rew == "bernstein":
            raise NotImplementedError("bound_type_rew='bernstein' raises AttributeError in the reference (self.r_max, "
                                      "ucrl2.py:268); only '_chernoff' is defined")
        self._explore = (epsilon_greedy, boltzmann_temperature)
        assert tables.H == 0, "UCRL2Continuous needs a continuous MDP"
        self.torch, self.tables = torch, tables
        self.dev = DeviceTables(tables, "succ")
        self.n_loops = N = int(n_loops)
        self.seed, self.env_offset = int(seed), int(env_offset)
        self.alpha_r, self.alpha_p = float(alpha_r), float(alpha_p)
        self.bernstein_p = int(bound_type_p == "bernstein")
        self.r_max = float(tables.rmax)
        self._planner = planner
        S, A = tables.S, tables.A
        dev = "cuda"
        self.state = torch.zeros(N, dtype=torch.int32, device=dev)
        self.h = torch.zeros(N, dtype=torch.int32, device=dev)  # (reset helper)
        self.t = 0
        _QLearningBatch.reset_envs(self)                        # Philox counter 0 = the reset draw
        self.time = torch.full((N,), self.t, dtype=torch.int64, device=dev)
        self.cumulative_reward = torch.zeros(N, dtype=torch.float64, device=dev)
        self.n_episodes = torch.zeros(N, dtype=torch.int64, device=dev)  # MDP episodes: none in a continuous MDP
        self.Q = torch.zeros((N, S, A), dtype=torch.float32, device=dev)
        self.V = torch.zeros((N, S), dtype=torch.float32, device=dev)
        self.N = torch.zeros((N, S, A, S), dtype=torch.int32, device=dev)                        # ucrl2.py:155
        self.Nsa = torch.zeros((N, S, A), dtype=torch.int32, device=dev)
        self.P = torch.full((N, S, A, S), float(np.float32(1.0) / np.float32(S)), dtype=torch.float32, device=dev)  # :148
        self.estimated_rewards = torch.full((N, S, A), float(np.float32(tables.rmax)), dtype=torch.float32, device=dev)
        self.variance_proxy_reward = torch.zeros((N, S, A), dtype=torch.float32, device=dev)
        self.estimated_holding_times = torch.ones((N, S, A), dtype=torch.float32, device=dev)
        self.nu = torch.zeros((N, S, A), dtype=torch.int32, device=dev)
        self._seen = torch.zeros((N, S, A), dtype=torch.int32, device=dev)
        # an artificial episode that starts at time t0 holds at most S*A + t0 steps and at most T - t0 of the run
        self.log_cap = (int(optimization_horizon) + S * A) // 2 + 2
        self.ep_len = torch.zeros(N, dtype=torch.int32, device=dev)
        self._ep_log = torch.zeros((N, self.log_cap, 2), dtype=torch.int32, device=dev)
        self.ended = torch.zeros(N, dtype=torch.int32, device=dev)
        self.iteration = torch.zeros(N, dtype=torch.int64, device=dev)
        self.episode = torch.zeros(N, dtype=torch.int64, device=dev)
        self.delta = torch.ones(N, dtype=torch.float64, device=dev)
        self.span_value = torch.zeros(N, dtype=torch.float64, device=dev)
        self.evi_iterations = 0
        a = _cabi.Ucrl2Args()
        a.N, a.seed, a.env0 = N, self.seed, self.env_offset
        a.state, a.t, a.cum_reward, a.Q = (self.state.data_ptr(), self.time.data_ptr(),
                                           self.cumulative_reward.data_ptr(), self.Q.data_ptr())
        a.Nsas, a.Nsa, a.P = self.N.data_ptr(), self.Nsa.data_ptr(), self.P.data_ptr()
        a.est_r, a.var_r, a.hold = (self.estimated_rewards.data_ptr(), self.variance_proxy_reward.data_ptr(),
                                    self.estimated_holding_times.data_ptr())
        a.nu, a.seen, a.ep_len, a.ep_log = (self.nu.data_ptr(), self._seen.data_ptr(), self.ep_len.data_ptr(),
                                            self._ep_log.data_ptr())
        a.log_cap = self.log_cap
        a.ended, a.iteration, a.episode, a.delta = (self.ended.data_ptr(), self.iteration.data_ptr(),
                                                    self.episode.data_ptr(), self.delta.data_ptr())
        self._args = a
        self.episode_end_update(torch.arange(N, dtype=torch.int32, device=dev), update_model=False)  # :194-195

    def bounds(self, idx):
        """episode += 1, delta and the confidence bounds (beta_r, beta_p f64 [m,S,A]) of the loops in idx (:183-186, :223-311)"""
        torch, S, A = self.torch, self.tables.S, self.tables.A
        m = int(idx.numel())
        br = torch.empty((m, S, A), dtype=torch.float64, device="cuda")
        bp = torch.empty((m, S, A), dtype=torch.float64, device="cuda")
        rc = _cabi.lib().colo_ucrl2_bounds(C.byref(self._args), S, A, idx.data_ptr(), m, self.alpha_r, self.alpha_p,
                                           self.r_max, self.bernstein_p, br.data_ptr(), bp.data_ptr(),
                                           _cabi.current_stream())
        _cabi.check(rc, "colo_ucrl2_bounds")
        return br, bp

    def solve_optimistic_model(self, idx, beta_r, beta_p, Q=None, V=None):
        """extended_value_iteration for the loops in idx, one launch (:313-357).  Q, V default to the loops' own."""
        torch, S, A = self.torch, self.tables.S, self.tables.A
        m = int(idx.numel())
        span = torch.empty(m, dtype=torch.float64, device="cuda")
        iters = torch.empty(m, dtype=torch.int64, device="cuda")
        status = torch.empty(m, dtype=torch.int32, device="cuda")
        Q = self.Q if Q is None else Q
        V = self.V if V is None else V
        rc = _cabi.lib().colo_extended_vi_batched_f32(
            self.P.data_ptr(), self.estimated_rewards.data_ptr(), beta_r.data_ptr(), beta_p.data_ptr(), idx.data_ptr(), m,
            S, A, self.r_max, 1e-3, int(1e6), Q.data_ptr(), V.data_ptr(), span.data_ptr(), iters.data_ptr(),
            status.data_ptr(), _cabi.current_stream())
        _cabi.check(rc, "colo_extended_vi_batched_f32")
        return span, iters, status

    def episode_end_update(self, idx, update_model=True):
        """ucrl2.py:183-192 for the loops listed in idx (i32 device tensor)"""
        S, A = self.tables.S, self.tables.A
        br, bp = self.bounds(idx)
        if self._planner is not None:
            self._planner(self, idx, br, bp)
        else:
            span, iters, status = self.solve_optimistic_model(idx, br, bp)
            self.span_value[idx.long()] = span / self.r_max
            self.evi_iterations += int(iters.sum())
            if int(status.max()) != 0:
                from .dynamic_programming import DynamicProgrammingMaxIterationExceeded

                raise DynamicProgrammingMaxIterationExceeded()
        if update_model:
            rc = _cabi.lib().colo_ucrl2_model_update(C.byref(self._args), S, A, idx.data_ptr(), int(idx.numel()),
                                                     _cabi.current_stream())
            _cabi.check(rc, "colo_ucrl2_model_update")
        else:
            self.ended.zero_()

    def steps(self, n_steps: int, trace: bool = False):
        """n_steps interactions for every loop.  trace=True returns i32 [n_steps, N, 4] = (s_t, a_t, s_tp1, reward bits)."""
        torch = self.torch
        tr = torch.zeros((n_steps, self.n_loops, 4), dtype=torch.int32, device="cuda") if trace else None
        a = self._args
        a.trace, a.trace_t0, a.trace_steps = (None if tr is None else tr.data_ptr()), self.t, int(n_steps)
        target = self.t + int(n_steps)
        _set_actor(self, self.t, n_steps)
        self.rounds = 0
        while True:
            rc = _cabi.lib().colo_ucrl2_steps(C.byref(self.dev.c), C.byref(a), target, _cabi.current_stream())
            _cabi.check(rc, "colo_ucrl2_steps")
            ended = self.ended.cpu()
            if int(ended.max()) == 2:
                raise RuntimeError("an artificial episode outgrew its log: optimization_horizon is smaller than the run")
            idx = torch.nonzero(ended).flatten().to(torch.int32).cuda()
            if idx.numel() == 0:
                break
            self.rounds += 1
            self.episode_end_update(idx)
        a.trace = None
        self.t = target
        return tr

    def current_optimal_stochastic_policy(self, i: int) -> np.ndarray:
        """ucrl2.py:77-80: greedy policy of the discounted VI on the empirical model"""
        from .dynamic_programming import discounted_value_iteration, get_policy_from_q_values

        Q, _ = discounted_value_iteration(self.P[i].contiguous(), self.estimated_rewards[i].contiguous())
        return get_policy_from_q_values(Q.cpu().numpy(), True)


def get_psi(n_states, n_actions, T, p):
    """infinite_horizon/posterior_sampling.py:20-42"""
    return n_states * np.log(n_states * n_actions / p)


def get_omega(n_states, n_actions, T, p):
    """:45-66"""
    return np.log(T / p)


def get_kappa(n_states, n_actions, T, p):
    """:69-90"""
    return np.log(T / p)


def get_eta(n_states, n_actions, T, p, omega):
    """:93-115"""
    return np.sqrt(T * n_states / n_actions) + 12 * omega * n_states ** 4


class PSRLContinuous:
    """N PSRLContinuous loops (colosseum/agent/agents/infinite_horizon/posterior_sampling.py:117-452; Agrawal & Jia 2017)
    on one continuous MDP, advanced in rounds like UCRL2Continuous: `colo_psrlc_steps` to each loop's artificial-episode
    end; for the loops that wait, `colo_psrlc_sample_models` (optimistic sampling: psi transition samples per (s, a) --
    Dirichlet posterior rows for visited pairs, the confidence-set rows for under-visited ones -- and one reward sample,
    laid out as the reference's extended MDP with A * psi actions), one batched `discounted_value_iteration` (the
    reference's gamma = 0.99, epsilon = 1e-3) and the q-values written back.  The sampled models never leave HBM.
    Constructor arguments are the reference's (`mdp_specs` -> the MDP's tables).

    sweep_order: "jacobi" (default) plans with synchronous sweeps stopped by the reference's rule -- the planner's input
    is a random posterior sample, so no bit-level parity exists to keep, and the early-stopped iterate differs from the
    reference's in-place one by less than the sampling noise (error bound eps gamma / (1 - gamma) for both);
    "gauss_seidel" runs the reference's own in-place iterate (one warp per model: 5-90x slower for the few models a
    round re-plans -- measured: RiverSwim 256 loops 18.6 s vs 2.1 s, DeepSea-30 32 loops 235 s vs 2.7 s)."""

    episodic = False

    def __init__(self, seed: int, tables: MDPTables, optimization_horizon: int, reward_prior_model=None,
                 transitions_prior_model=None, rewards_prior_prms=None, transitions_prior_prms=None,
                 epsilon_greedy=None, boltzmann_temperature=None, psi_weight=1.0, omega_weight=1.0, kappa_weight=1.0,
                 eta_weight=1.0, get_psi=get_psi, get_omega=get_omega, get_kappa=get_kappa, get_eta=get_eta, p=0.05,
                 no_optimistic_sampling=False, truncate_reward_with_max=False, min_steps_before_new_episode=0,
                 max_psi=60, *, n_loops: int = 1, env_offset: int = 0, sampler: str = "fast",
                 sweep_order: str = "jacobi", planner=None, max_plan_bytes: int = 8 << 30):
        import torch

        _cabi.require_cuda()
        assert sampler in ("fast", "f64")
        rname = getattr(reward_prior_model, "name", reward_prior_model)
        tname = getattr(transitions_prior_model, "name", transitions_prior_model)
        assert rname in (None, "N_NIG", "N_N") and tname in (None, "M_DIR")
        self._explore = (epsilon_greedy, boltzmann_temperature)
        if min_steps_before_new_episode != 0:
            raise NotImplementedError("min_steps_before_new_episode > 0 is not offered by the batched agent")
        assert tables.H == 0, "PSRLContinuous needs a continuous MDP"
        self.torch, self.tables = torch, tables
        self.dev = DeviceTables(tables, "succ")
        self.n_loops = N = int(n_loops)
        self.seed, self.env_offset = int(seed), int(env_offset)
        S, A = tables.S, tables.A
        T = optimization_horizon
        # posterior_sampling.py:268-303, in the reference's expressions
        self.truncate_reward_with_max = bool(truncate_reward_with_max)
        self.no_optimistic_sampling = bool(no_optimistic_sampling or (S ** 2 * A) > 6_000_000)
        self.p = p
        self.psi = min(max_psi, max(2, int(psi_weight * get_psi(S, A, T, p))))
        self.omega = omega_weight * get_omega(S, A, T, p)
        self.kappa = kappa_weight * get_kappa(S, A, T, p)
        self.eta = max(5, min(10 * S, eta_weight * get_eta(S, A, T, p, self.omega)))
        self._psi = 1 if self.no_optimistic_sampling else self.psi        # columns per real action on the device
        self._eta = 0.0 if self.no_optimistic_sampling else float(self.eta)
        self.reward_model = 1 if rname == "N_N" else 0
        self._fast = int(sampler == "fast")
        self._sweep_order = sweep_order
        self._planner = planner
        self._max_plan_bytes = int(max_plan_bytes)
        rp = [tables.rmax, 1, 1, 1] if rewards_prior_prms is None else rewards_prior_prms       # bayesian_model.py:46-48
        tp = [1.0 / S] if transitions_prior_prms is None else transitions_prior_prms              # :49-51
        if self.reward_model == 1:
            hp = np.zeros((S, A, 4), np.float32)
            hp[..., :2] = np.tile(rp, (S, A, 1)).astype(np.float32)
        else:
            hp = np.tile(rp, (S, A, 1)).astype(np.float32)                                        # base_conjugate.py:44-47
            mu, n_mu, tau, n_tau = (hp[..., k].copy() for k in range(4))
            hp[..., 2], hp[..., 3] = n_tau * 0.5, (0.5 * n_tau) / tau                            # conjugate_rewards.py:45-54
        dev = "cuda"
        self.nig_hyper = torch.from_numpy(np.tile(hp, (N, 1, 1, 1))).cuda()
        self.dir_hyper = torch.full((N, S, A, S), float(np.float32(tp[0])), dtype=torch.float32, device=dev)
        self.N = torch.zeros((N, S, A, S), dtype=torch.int32, device=dev)                        # :309-311
        self.Nsa = torch.zeros((N, S, A), dtype=torch.int32, device=dev)
        self.nu = torch.zeros((N, S, A), dtype=torch.int32, device=dev)
        self.Q = torch.zeros((N, S, A * self._psi), dtype=torch.float32, device=dev)
        self.state = torch.zeros(N, dtype=torch.int32, device=dev)
        self.h = torch.zeros(N, dtype=torch.int32, device=dev)
        self.t = 0
        _QLearningBatch.reset_envs(self)
        self.time = torch.full((N,), self.t, dtype=torch.int64, device=dev)
        self.cumulative_reward = torch.zeros(N, dtype=torch.float64, device=dev)
        self.n_episodes = torch.zeros(N, dtype=torch.int64, device=dev)
        self.ended = torch.zeros(N, dtype=torch.int32, device=dev)
        self.episode = torch.zeros(N, dtype=torch.int64, device=dev)
        self.vi_sweeps = 0
        a = _cabi.PsrlcArgs()
        a.N, a.seed, a.env0, a.psi, a.reward_model = N, self.seed, self.env_offset, self._psi, self.reward_model
        a.state, a.t, a.cum_reward, a.Q = (self.state.data_ptr(), self.time.data_ptr(),
                                           self.cumulative_reward.data_ptr(), self.Q.data_ptr())
        a.dir_hyper, a.nig_hyper = self.dir_hyper.data_ptr(), self.nig_hyper.data_ptr()
        a.Nsas, a.Nsa, a.nu = self.N.data_ptr(), self.Nsa.data_ptr(), self.nu.data_ptr()
        a.ended, a.episode = self.ended.data_ptr(), self.episode.data_ptr()
        self._args = a
        # before_start_interacting (:378-382): the random q-values it sets are replaced by the first plan at once
        self.episode_end_update(torch.arange(N, dtype=torch.int32, device=dev))

    def sample_models(self, idx):
        """optimistic_sampling + sample_R for the loops in idx: (T_ext f32[m,S,A*psi,S], R_ext f32[m,S,A*psi])"""
        torch, S, A = self.torch, self.tables.S, self.tables.A
        m = int(idx.numel())
        T_ext = torch.empty((m, S, A * self._psi, S), dtype=torch.float32, device="cuda")
        R_ext = torch.empty((m, S, A * self._psi), dtype=torch.float32, device="cuda")
        rc = _cabi.lib().colo_psrlc_sample_models(C.byref(self._args), S, A, idx.data_ptr(), m, self._eta,
                                                  int(self.truncate_reward_with_max), float(self.tables.rmax),
                                                  self._fast, T_ext.data_ptr(), R_ext.data_ptr(), _cabi.current_stream())
        _cabi.check(rc, "colo_psrlc_sample_models")
        return T_ext, R_ext

    def episode_end_update(self, idx):
        """posterior_sampling.py:347-376 for the loops listed in idx (i32 device tensor), in chunks that keep the sampled
        extended models under max_plan_bytes"""
        from . import dynamic_programming as dp

        S, A = self.tables.S, self.tables.A
        per = S * A * self._psi * S * 4
        chunk = max(1, self._max_plan_bytes // per)
        for lo in range(0, int(idx.numel()), chunk):
            sub = idx[lo:lo + chunk].contiguous()
            if self._planner is not None:
                self._planner(self, sub)
            else:
                T_ext, R_ext = self.sample_models(sub)
                Q, _ = dp.discounted_value_iteration(T_ext, R_ext, precision="f32", sweep_order=self._sweep_order)
                self.vi_sweeps += int(sum(dp.last_iterations()))
                self.Q[sub.long()] = Q
            rc = _cabi.lib().colo_psrlc_finish_episode(C.byref(self._args), S, A, sub.data_ptr(), int(sub.numel()),
                                                       _cabi.current_stream())
            _cabi.check(rc, "colo_psrlc_finish_episode")

    def steps(self, n_steps: int, trace: bool = False):
        """n_steps interactions for every loop.  trace=True returns i32 [n_steps, N, 4] = (s_t, EXTENDED action, s_tp1,
        reward bits); the real action is column 1 // psi."""
        torch = self.torch
        tr = torch.zeros((n_steps, self.n_loops, 4), dtype=torch.int32, device="cuda") if trace else None
        a = self._args
        a.trace, a.trace_t0, a.trace_steps = (None if tr is None else tr.data_ptr()), self.t, int(n_steps)
        target = self.t + int(n_steps)
        _set_actor(self, self.t, n_steps)
        self.rounds = 0
        while True:
            rc = _cabi.lib().colo_psrlc_steps(C.byref(self.dev.c), C.byref(a), target, _cabi.current_stream())
            _cabi.check(rc, "colo_psrlc_steps")
            idx = torch.nonzero(self.ended).flatten().to(torch.int32)
            if idx.numel() == 0:
                break
            self.rounds += 1
            self.episode_end_update(idx)
        a.trace = None
        self.t = target
        return tr

    def get_map_estimate(self):
        """BayesianMDPModel.get_map_estimate (bayesian_model.py:71-76) for every loop"""
        return self.dir_hyper / self.dir_hyper.sum(-1, keepdim=True), self.nig_hyper[..., 0]

    def current_optimal_stochastic_policy(self, i: int) -> np.ndarray:
        """posterior_sampling.py:176-180: greedy policy of the discounted VI on the MAP model"""
        from .dynamic_programming import discounted_value_iteration, get_policy_from_q_values

        T_map, R_map = self.get_map_estimate()
        Q, _ = discounted_value_iteration(T_map[i].contiguous(), R_map[i].contiguous())
        return get_policy_from_q_values(Q.cpu().numpy(), True)


_CKPT_FIELDS = ("state", "h", "cumulative_reward", "n_episodes", "N", "Q", "Q_main", "V", "mu", "sigma", "beta",
                "dir_hyper", "nig_hyper", "T_sample", "R_sample",
                # UCRL2Continuous / PSRLContinuous
                "time", "Nsa", "P", "estimated_rewards", "variance_proxy_reward", "estimated_holding_times", "nu",
                "ep_len", "_ep_log", "ended", "iteration", "episode", "delta", "span_value")


def agents_state_dict(agents):
    """checkpoint of a batch of loops (env state, agent tables, Philox counters): resuming reproduces the run bit for
    bit"""
    agents.torch.cuda.current_stream().synchronize()
    d = {k: getattr(agents, k).cpu() for k in _CKPT_FIELDS if hasattr(agents, k)}
    d["t"] = agents.t
    for k in ("n_samples", "_h_episode"):
        if hasattr(agents, k):
            d[k] = getattr(agents, k)
    return d


def agents_load_state_dict(agents, d):
    for k in _CKPT_FIELDS:
        if k in d:
            getattr(agents, k).copy_(d[k])
    agents.t = int(d["t"])
    for k in ("n_samples", "_h_episode"):
        if k in d:
            setattr(agents, k, int(d[k]))
    agents.torch.cuda.current_stream().synchronize()


def _normalised_indicators(rec, cum_regret, base, done):
    """the normalised indicators of MDPLoop._update_performance_logs (agent_mdp_interaction.py:395-428) from the
    episodic baselines `base` (scalars, or one value per loop)"""
    span = base["optimal"] - base["worst"]
    rec["normalized_cumulative_regret"] = cum_regret / span
    rec["normalized_cumulative_reward"] = (rec["cumulative_reward"] - done * base["worst"]) / span
    for k in ("optimal", "worst", "random"):
        rec[f"{k}_cumulative_expected_reward"] = base[k] * done
    rec["random_cumulative_regret"] = (base["optimal"] - base["random"]) * done
    rec["worst_cumulative_regret"] = span * done


class BatchedMDPLoop:
    """MDPLoop for N loops at once.  `T`, `R` (numpy float32) are only needed for the regret indicators."""

    def __init__(self, agents: _QLearningBatch, T=None, R=None):
        self.agents = agents
        self.T, self.R = T, R
        self.logs = []

    def _expected_regret(self, loops):
        """per-step expected regret of the greedy policy of each loop in `loops`
        (agent_mdp_interaction.py:520-578: episodic -> regret at time zero / H; continuous -> optimal minus the
        policy's average reward)."""
        from . import dynamic_programming as dp
        from . import indicators, markov_chain

        ag, tb = self.agents, self.agents.tables
        out = np.zeros(len(loops))
        if ag.episodic:
            start = np.zeros(tb.S, np.float64)
            prob = np.diff(np.concatenate([[0.0], np.asarray(tb.start_cum, np.float64)]))
            np.add.at(start, np.asarray(tb.start_idx), prob / prob.sum())
            if not hasattr(self, "_opt_V"):
                self._opt_V = dp.episodic_value_iteration(tb.H, self.T, self.R)[1]
            for k, i in enumerate(loops):
                pi = ag.current_optimal_stochastic_policy(i)
                Rs, _ = indicators.get_episodic_regrets_and_average_reward_at_time_zero(
                    tb.H, self.T, self.R, pi, start, self._opt_V)
                out[k] = float((np.asarray(Rs) * start).sum()) / tb.H
        else:
            if not hasattr(self, "_opt_ar"):
                Q, _ = dp.discounted_value_iteration(self.T, self.R)
                self._opt_ar = markov_chain.get_average_reward(self.T, self.R, dp.get_policy_from_q_values(Q, True))
            states = ag.state.cpu().numpy()
            cache = self.__dict__.setdefault("_ar_cache", {})  # greedy policies repeat from tick to tick and loop to loop
            for k, i in enumerate(loops):
                pi = ag.current_optimal_stochastic_policy(i)
                pin = np.ascontiguousarray(pi.cpu().numpy() if hasattr(pi, "cpu") else pi)
                # the start state matters only for multichain policies (markov_chain.recurrent_class_weights); a
                # unichain entry is stored under start -1 and serves every start state
                key = pin.tobytes()
                ar = cache.get((key, -1), cache.get((key, int(states[i]))))
                if ar is None:
                    ar = markov_chain.get_average_reward(self.T, self.R, pi, [(int(states[i]), 1.0)])
                    one = markov_chain.get_stationary_distribution.last_classes == 1
                    if len(cache) > 4096:
                        cache.clear()
                    cache[(key, -1 if one else int(states[i]))] = ar
                r = self._opt_ar - ar
                out[k] = 0.0 if (np.isclose(r, 0.0, atol=1e-3) or r < 0) else r
        return out

    def _expected_regret_all(self, chunk: int = 4096):
        """episodic: the per-step expected regret of EVERY loop's greedy policy, on the device: one-hot greedy policies
        (uniformly random among argmax ties under the reference's fixed seed 42, dynamic_programming/utils.py:4,30-38 --
        the draws themselves differ from numba's stream), all evaluated on the true MDP by one launch of
        colo_episodic_policies_f32 per chunk of loops, then max(V*[0] - V[0], 0) averaged over the start distribution
        and divided by H (indicators.py:29-45, agent_mdp_interaction.py:549-566)."""
        import torch

        from . import dynamic_programming as dp

        ag, tb = self.agents, self.agents.tables
        assert self.T is not None
        if not ag.episodic:
            return self._expected_regret_all_continuous(chunk)
        S, A, H = tb.S, tb.A, tb.H
        if not hasattr(self, "_dev_TR"):
            Td, Rd = dp.to_device(self.T), dp.to_device(self.R)
            v_star = dp.episodic_value_iteration(H, Td, Rd, precision="f32")[1][0]
            start = torch.zeros(S, dtype=torch.float64, device="cuda")
            prob = np.diff(np.concatenate([[0.0], np.asarray(tb.start_cum, np.float64)]))
            start.index_add_(0, torch.from_numpy(np.asarray(tb.start_idx, np.int64)).cuda(),
                             torch.from_numpy(prob / prob.sum()).cuda())
            self._dev_TR = (Td, Rd, v_star.double(), start)
        Td, Rd, v_star, start = self._dev_TR
        if isinstance(ag, PSRLEpisodic):  # greedy policy of the MAP model (posterior_sampling.py:76-80)
            T_map, R_map = ag.get_map_estimate()
            Qall = dp.episodic_value_iteration(H, T_map.contiguous(), R_map.contiguous(), precision="f32")[0][:, :H]
        else:
            Qall = ag.Q
        out = torch.empty(ag.n_loops, dtype=torch.float64, device="cuda")
        avg = torch.empty_like(out)
        gen = torch.Generator(device="cuda").manual_seed(dp.ARGMAX_SEED)
        lib = _cabi.lib()
        for lo in range(0, ag.n_loops, chunk):
            Qc = Qall[lo:lo + chunk]
            n = Qc.shape[0]
            tie = torch.rand(Qc.shape, generator=gen, device="cuda")
            idx = torch.where(Qc == Qc.max(-1, keepdim=True).values, tie, torch.full_like(tie, -1.0)).argmax(-1)
            pi = torch.nn.functional.one_hot(idx, A).to(torch.float32).contiguous()
            Qp = torch.empty((n, H + 1, S, A), dtype=torch.float32, device="cuda")
            Vp = torch.empty((n, H + 1, S), dtype=torch.float32, device="cuda")
            rc = lib.colo_episodic_policies_f32(Td.data_ptr(), Rd.data_ptr(), pi.data_ptr(), n, S, A, H, Qp.data_ptr(),
                                                Vp.data_ptr(), _cabi.current_stream())
            _cabi.check(rc, "colo_episodic_policies_f32")
            reg = (v_star[None, :] - Vp[:, 0].double()).clamp_min(0.0)
            out[lo:lo + n] = (reg * start[None, :]).sum(-1) / H
            avg[lo:lo + n] = (Vp[:, 0].double() * start[None, :]).sum(-1) / H
        self._agent_average_reward = avg.cpu().numpy()  # agent_mdp_interaction.py:514-518
        return out.cpu().numpy()

    def _greedy_q_continuous(self):
        """the q-values whose greedy policy is `current_optimal_stochastic_policy` of every loop, f32 [N,S,A] on the
        device: the agent's own table (Q-learning, q_learning.py:164-166), or the discounted value iteration on each
        loop's empirical (ucrl2.py:77-80) / MAP (posterior_sampling.py:176-180) model, all loops in one batched solve"""
        from . import dynamic_programming as dp

        ag = self.agents
        if isinstance(ag, UCRL2Continuous):
            return dp.discounted_value_iteration(ag.P, ag.estimated_rewards, precision="f32")[0]
        if isinstance(ag, PSRLContinuous):
            T_map, R_map = ag.get_map_estimate()
            return dp.discounted_value_iteration(T_map.contiguous(), R_map.contiguous(), precision="f32")[0]
        return ag.Q

    def _expected_regret_all_continuous(self, chunk: int = 4096):
        """continuous: the expected per-step regret of EVERY loop's greedy policy (agent_mdp_interaction.py:567-578:
        optimal average reward minus the policy's, zero when within 1e-3), all policies through one batched
        stationary-distribution solve per chunk (markov_chain.get_average_reward_batched)."""
        import torch

        from . import dynamic_programming as dp
        from . import markov_chain

        ag, tb = self.agents, self.agents.tables
        A = tb.A
        if not hasattr(self, "_opt_ar"):
            Q, _ = dp.discounted_value_iteration(self.T, self.R)
            self._opt_ar = markov_chain.get_average_reward(self.T, self.R, dp.get_policy_from_q_values(Q, True))
        if not hasattr(self, "_dev_TR_c"):
            self._dev_TR_c = (dp.to_device(self.T), dp.to_device(self.R))
        Td, Rd = self._dev_TR_c
        Qall = self._greedy_q_continuous()
        states = ag.state.cpu().numpy()
        gen = torch.Generator(device="cuda").manual_seed(dp.ARGMAX_SEED)
        out = np.empty(ag.n_loops)
        avg = np.empty(ag.n_loops)
        self._greedy_actions = torch.empty(Qall.shape[:2], dtype=torch.int64, device="cuda")  # the policies evaluated
        for lo in range(0, ag.n_loops, chunk):
            Qc = Qall[lo:lo + chunk]
            tie = torch.rand(Qc.shape, generator=gen, device="cuda")
            idx = torch.where(Qc == Qc.max(-1, keepdim=True).values, tie, torch.full_like(tie, -1.0)).argmax(-1)
            self._greedy_actions[lo:lo + chunk] = idx
            pi = torch.nn.functional.one_hot(idx, A).to(torch.float32).contiguous()
            ar = markov_chain.get_average_reward_batched(Td, Rd, pi, states[lo:lo + chunk])
            r = self._opt_ar - ar
            out[lo:lo + len(ar)] = np.where(np.isclose(r, 0.0, atol=1e-3) | (r < 0), 0.0, r)
            avg[lo:lo + len(ar)] = ar
        self._agent_average_reward = avg
        return out

    def episodic_baselines(self):
        """per-step average rewards of the optimal, worst and uniformly random policies of an episodic MDP
        (mdp/base_finite.py:211-253: start-distribution average of V[0] divided by H; the worst policy is the optimal one
        of -R, mdp/base.py:649-664) -- the normalisers of MDPLoop's indicators"""
        import torch

        from . import dynamic_programming as dp

        if not hasattr(self, "_baselines"):
            tb = self.agents.tables
            H, S, A = tb.H, tb.S, tb.A
            Td, Rd = dp.to_device(self.T), dp.to_device(self.R)
            prob = np.diff(np.concatenate([[0.0], np.asarray(tb.start_cum, np.float64)]))
            start = np.zeros(S)
            np.add.at(start, np.asarray(tb.start_idx), prob / prob.sum())
            v_opt = dp.episodic_value_iteration(H, Td, Rd, precision="f64")[1][0].cpu().numpy()
            v_worst = -dp.episodic_value_iteration(H, Td, -Rd, precision="f64")[1][0].cpu().numpy()
            uni = torch.full((H, S, A), 1.0 / A, dtype=torch.float32, device="cuda")
            v_rand = dp.episodic_policy_evaluation(H, Td, Rd, uni, precision="f64")[1][0].cpu().numpy()
            self._baselines = {k: float((v * start).sum()) / H for k, v in
                               (("optimal", v_opt), ("worst", v_worst), ("random", v_rand))}
        return self._baselines

    def run(self, T: int, log_every: int = -1, regret_for=None):
        """T interaction steps for every loop, `log_every` steps per launch.  Returns the list of log records
        (steps, cumulative_reward f64[N], n_episodes i64[N], and -- for the loops listed in `regret_for`, when T/R were
        given -- regret and cumulative_regret).  regret_for="all": every loop, evaluated on the device in one batched
        solve per tick (episodic: colo_episodic_policies_f32; continuous: colo_average_rewards_f64)."""
        ag = self.agents
        log_every = T if log_every in (0, -1, None) else int(log_every)
        all_loops = isinstance(regret_for, str) and regret_for == "all"
        if all_loops:
            assert self.T is not None, "regret_for='all' needs T, R"
            regret_for = list(range(ag.n_loops))
        regret_for = [] if (regret_for is None or self.T is None) else list(regret_for)
        cum_regret = np.zeros(len(regret_for))
        cum_expected = np.zeros(len(regret_for))
        base = self.episodic_baselines() if (ag.episodic and (all_loops or regret_for)) else None
        t_start = time.perf_counter()
        done = 0
        while done < T:
            n = min(log_every, T - done)
            ag.steps(n)
            done += n
            rec = {"steps": done, "cumulative_reward": ag.cumulative_reward.cpu().numpy(),
                   "n_episodes": ag.n_episodes.cpu().numpy()}
            if regret_for:
                reg = self._expected_regret_all() if all_loops else self._expected_regret(regret_for)
                cum_regret = cum_regret + reg * n  # agent_mdp_interaction.py:503-506
                rec["regret"], rec["cumulative_regret"] = reg, cum_regret.copy()
                if base is not None:
                    _normalised_indicators(rec, cum_regret, base, done)
                if all_loops:
                    cum_expected = cum_expected + self._agent_average_reward * n
                    rec["cumulative_expected_reward"] = cum_expected.copy()
            rec["steps_per_second"] = done * ag.n_loops / (time.perf_counter() - t_start)
            self.logs.append(rec)
        return self.logs


class _MixedQLearningBatch:
    """Q-learning loops on many MDP instances, all advanced by one launch per `steps` (colo_mixed_qlearning_*).
    Instance i owns the contiguous loops `segment(i)`; they are bit-identical to the single-MDP class built with
    tables[i], seed[i] and n_loops[i].  The flat tables keep the single-MDP names (N, Q, V, ...; state, h,
    cumulative_reward, n_episodes are flat [n_loops]); `table(name, i)` is instance i's view, shaped as the single-MDP
    class's table ([n_i, H_i, S_i, A_i], V [n_i, H_i + 1, S_i]; continuous [n_i, S_i, A_i], V [n_i, S_i])."""
    episodic = None

    def _alloc(self, tables, n_loops, seed, epsilon_greedy, boltzmann_temperature):
        import torch

        from .batched_mdp import MixedBatchedMDP

        _cabi.require_cuda()
        self._explore = (epsilon_greedy, boltzmann_temperature)
        tables = list(tables)
        for i, tb in enumerate(tables):
            assert (tb.H > 0) == self.episodic, f"instance {i}: episodic agents need an episodic MDP and vice versa"
        self.torch = torch
        self._handle = None
        # the env handle (successor tables, per-instance seeds and segments) and the resets
        self.env = MixedBatchedMDP(tables, n_loops, "succ", seed, track_visits=False)
        self.tables = self.env.tables
        self.sizes, self.seeds = self.env.sizes, self.env.seeds
        self.n_loops = N = self.env.n_envs
        self.t = 0
        self.state, self.h = self.env.state, self.env.h
        self.cumulative_reward = torch.zeros(N, dtype=torch.float64, device="cuda")
        self.n_episodes = torch.zeros(N, dtype=torch.int64, device="cuda")
        a = _cabi.QLearningArgs()
        a.N = N  # seed, env0 and the per-instance constants live in the handle
        a.state, a.h = self.state.data_ptr(), self.h.data_ptr()
        a.cum_reward, a.n_episodes = self.cumulative_reward.data_ptr(), self.n_episodes.data_ptr()
        self._args = a
        self.reset_envs()

    def _make_handle(self, insts):
        """uploads the per-instance constants; returns the element counts of the Q-shaped and V-shaped flat tables"""
        n = len(self.tables)
        lib = _cabi.lib()
        out = C.c_void_p()
        rc = lib.colo_mixed_qlearning_create(self.env._handle, int(self.episodic), (_cabi.QLearningInst * n)(*insts),
                                             _cabi.current_stream(), C.byref(out))
        _cabi.check(rc, "colo_mixed_qlearning_create")
        self._handle = out.value
        nq, nv = C.c_longlong(), C.c_longlong()
        _cabi.check(lib.colo_mixed_qlearning_sizes(self._handle, C.byref(nq), C.byref(nv)), "colo_mixed_qlearning_sizes")
        ep = self.episodic
        self._shapes = {"q": [(int(m), tb.H, tb.S, tb.A) if ep else (int(m), tb.S, tb.A) for m, tb in zip(self.sizes, self.tables)],
                        "v": [(int(m), tb.H + 1, tb.S) if ep else (int(m), tb.S) for m, tb in zip(self.sizes, self.tables)]}
        self._region = {k: [int(np.prod(sh)) for sh in v] for k, v in self._shapes.items()}
        self._off = {k: np.concatenate([[0], np.cumsum(v)]).astype(np.int64) for k, v in self._region.items()}
        assert (self._off["q"][-1], self._off["v"][-1]) == (nq.value, nv.value), "table layout of the library"
        return nq.value, nv.value

    def _per_instance(self, kind, dtype, values):
        """a flat table whose region of instance i is filled with values[i]"""
        torch = self.torch
        counts = torch.tensor(self._region[kind], dtype=torch.int64, device="cuda")
        return torch.repeat_interleave(torch.tensor(values, dtype=dtype, device="cuda"), counts,
                                       output_size=int(self._off[kind][-1]))

    def __del__(self):
        try:
            if getattr(self, "_handle", None):
                _cabi.lib().colo_mixed_qlearning_destroy(self._handle)
                self._handle = None
        except Exception:
            pass

    @property
    def n_instances(self):
        return len(self.tables)

    def segment(self, i: int) -> slice:
        """the loops of instance i"""
        return self.env.segment(i)

    def table(self, name: str, i: int):
        """instance i's view of the flat table `name`, shaped as the single-MDP class's"""
        kind = "v" if name == "V" else "q"
        lo, hi = int(self._off[kind][i]), int(self._off[kind][i + 1])
        return getattr(self, name)[lo:hi].view(self._shapes[kind][i])

    def reset_envs(self):
        """mdp.reset() for every loop, as the single-MDP classes: start states drawn at counter t, then t += 1"""
        self.env.t = self.t
        self.env.reset()
        self.t += 1
        self.torch.cuda.current_stream().synchronize()

    def steps(self, n_steps: int, trace: bool = False):
        """n_steps iterations of the interaction loop for every loop of every instance, one launch.  trace=True returns
        i32 [n_steps, n_loops, 4] = (s_t, a_t, obs_tp1, reward bits)."""
        torch = self.torch
        tr = torch.empty((n_steps, self.n_loops, 4), dtype=torch.int32, device="cuda") if trace else None
        self._args.trace = None if tr is None else tr.data_ptr()
        _set_actor(self, self.t, n_steps)
        rc = _cabi.lib().colo_mixed_qlearning_steps(self._handle, C.byref(self._args), int(n_steps), self.t,
                                                    _cabi.current_stream())
        _cabi.check(rc, "colo_mixed_qlearning_steps")
        self.t += int(n_steps)
        return tr


class MixedQLearningEpisodic(_MixedQLearningBatch):
    """QLearningEpisodic's loops on many episodic MDPs: `tables` a list, `seed` and `n_loops` one value or one per
    instance"""
    episodic = True

    def __init__(self, seed, tables, optimization_horizon: int, p: float, c_1: float, c_2: float = None,
                 min_at: float = 0, UCB_type="hoeffding", epsilon_greedy=None, boltzmann_temperature=None, *,
                 n_loops=1):
        UCB_type = UCB_type.lower()
        assert 0 <= min_at < 0.99 and 0 < p < 1 and c_1 > 0 and UCB_type in ("hoeffding", "bernstein")
        if UCB_type == "bernstein":
            assert c_2 is not None and c_2 > 0
        self._alloc(tables, n_loops, seed, epsilon_greedy, boltzmann_temperature)
        torch = self.torch
        insts = [_cabi.QLearningInst(log_term=float(np.log(tb.S * tb.A * optimization_horizon / p)),  # q_learning.py:43
                                     sqrt_h7sa=float(np.sqrt(tb.H ** 7 * tb.S * tb.A))) for tb in self.tables]
        nq, nv = self._make_handle(insts)
        self.N = torch.ones(nq, dtype=torch.int32, device="cuda")                              # q_learning.py:44
        self.Q = self._per_instance("q", torch.float32, [float(tb.H) for tb in self.tables])   # :45-47
        self.V = torch.zeros(nv, dtype=torch.float32, device="cuda")                          # :48
        a = self._args
        a.cnt, a.Q, a.V = self.N.data_ptr(), self.Q.data_ptr(), self.V.data_ptr()
        a.ucb_type = 0
        if UCB_type == "bernstein":
            self.mu = torch.zeros(nq, dtype=torch.float32, device="cuda")
            self.sigma = torch.zeros_like(self.mu)
            self.beta = torch.zeros_like(self.mu)
            a.mu, a.sigma, a.beta = self.mu.data_ptr(), self.sigma.data_ptr(), self.beta.data_ptr()
            a.ucb_type = 1
            a.c_2 = float(c_2)
        a.c_1, a.min_at = float(c_1), float(min_at)


class MixedQLearningContinuous(_MixedQLearningBatch):
    """QLearningContinuous's loops on many continuous MDPs: `tables` a list, `seed` and `n_loops` one value or one per
    instance; H, gamma and span_approx are lists, one value per instance"""
    episodic = False

    def __init__(self, seed, tables, optimization_horizon: int, min_at: float = 0, confidence: float = 0.95,
                 span_approx_weight: float = 1, get_span_approx=None, h_weight: float = 1, get_H=get_H,
                 epsilon_greedy=None, boltzmann_temperature=None, *, n_loops=1):
        assert 0 <= min_at < 0.99 and 0 < confidence < 1 and span_approx_weight > 0 and h_weight > 0
        self._alloc(tables, n_loops, seed, epsilon_greedy, boltzmann_temperature)
        torch = self.torch
        self.min_at = min_at if min_at > 0.009 else 0                                # q_learning.py:62
        log_term = float(np.log(2 * optimization_horizon / confidence))
        self.span_approx, self.H, self.gamma, insts = [], [], [], []
        for tb in self.tables:
            span = span_approx_weight
            if get_span_approx is not None:
                span *= get_span_approx(tb.S, tb.A)
            H = float(h_weight * get_H(tb.S, tb.A, optimization_horizon, span, confidence))
            self.span_approx.append(span)
            self.H.append(H)
            self.gamma.append(1 - 1 / H)
            insts.append(_cabi.QLearningInst(log_term=log_term, H_eff=H, gamma=float(1 - 1 / H), span_approx=float(span)))
        nq, nv = self._make_handle(insts)
        self.N = torch.zeros(nq, dtype=torch.int32, device="cuda")
        self.Q = self._per_instance("q", torch.float32, self.H)
        self.Q_main = self.Q.clone()
        self.V = self._per_instance("v", torch.float32, self.H)
        a = self._args
        a.cnt, a.Q, a.Q_main, a.V = self.N.data_ptr(), self.Q.data_ptr(), self.Q_main.data_ptr(), self.V.data_ptr()
        a.min_at = float(self.min_at)


class _SegmentView:
    """instance i of a mixed agent batch, with the attributes BatchedMDPLoop's regret evaluation reads"""

    def __init__(self, agents, i):
        self.torch, self.episodic = agents.torch, agents.episodic
        self.tables = agents.tables[i]
        self.n_loops = int(agents.sizes[i])
        self.Q = agents.table("Q", i)
        self.state = agents.state[agents.segment(i)]


class MixedBatchedMDPLoop:
    """BatchedMDPLoop for a mixed agent batch.  `T`, `R` (lists, one numpy float32 pair per instance) are only needed
    for the regret indicators.  The record has BatchedMDPLoop.run's fields, each as a flat per-loop array.
    regret_for="all" evaluates the greedy policies instance by instance, through one BatchedMDPLoop per instance over a
    view of its segment: a log tick costs a few launches and a host synchronisation per instance (one ragged launch
    over every instance is not offered)."""

    def __init__(self, agents: _MixedQLearningBatch, T=None, R=None):
        self.agents = agents
        self.T, self.R = T, R
        self.loops = None if T is None else [BatchedMDPLoop(_SegmentView(agents, i), T[i], R[i])
                                             for i in range(agents.n_instances)]
        self.logs = []

    def run(self, T: int, log_every: int = -1, regret_for=None):
        """T interaction steps for every loop, `log_every` steps per launch; regret_for None or "all"."""
        assert regret_for in (None, "all"), "a mixed batch evaluates the regret of every loop or of none"
        ag = self.agents
        log_every = T if log_every in (0, -1, None) else int(log_every)
        regret = regret_for == "all"
        assert not regret or self.loops is not None, "regret_for='all' needs T, R"
        cum_regret = np.zeros(ag.n_loops)
        cum_expected = np.zeros(ag.n_loops)
        base = None
        if regret and ag.episodic:
            per = [lp.episodic_baselines() for lp in self.loops]
            base = {k: np.repeat([b[k] for b in per], ag.sizes) for k in ("optimal", "worst", "random")}
        t_start = time.perf_counter()
        done = 0
        while done < T:
            n = min(log_every, T - done)
            ag.steps(n)
            done += n
            rec = {"steps": done, "cumulative_reward": ag.cumulative_reward.cpu().numpy(),
                   "n_episodes": ag.n_episodes.cpu().numpy()}
            if regret:
                reg = np.concatenate([lp._expected_regret_all() for lp in self.loops])
                cum_regret = cum_regret + reg * n
                rec["regret"], rec["cumulative_regret"] = reg, cum_regret.copy()
                if base is not None:
                    _normalised_indicators(rec, cum_regret, base, done)
                cum_expected = cum_expected + np.concatenate([lp._agent_average_reward for lp in self.loops]) * n
                rec["cumulative_expected_reward"] = cum_expected.copy()
            rec["steps_per_second"] = done * ag.n_loops / (time.perf_counter() - t_start)
            self.logs.append(rec)
        return self.logs
