"""GPU: the drop-in exercised behind LIVE reference MDP objects.  `patch.install()` rebinds the reference's hot-path
names (colosseum_b200/patch.py); the reference's own property layer (colosseum/mdp/base.py:592-679, :996-1114,
mdp/base_finite.py:167-208) then decides which DP runs on which tensor, and every number it returns is compared with
the value the UNPATCHED reference produced for the same constructor arguments (tests/golden/inst_*.npz).

The reference package is the unmodified one, staged outside git (oracle/reference_import.py says where it is looked
for).  Skipped when it is not staged."""
import numpy as np
import pytest

from conftest import load_instance

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ref():
    from oracle.reference_import import import_reference, reference_available

    if not reference_available():
        pytest.skip("the unmodified Colosseum package is not staged (oracle/_ref or $COLOSSEUM_REFERENCE_ROOT)")
    import_reference()
    import colosseum.mdp  # noqa: F401

    import colosseum_b200.patch as patch

    n = patch.install()  # BEFORE constructing MDPs (an MDP binds its DP functions at construction, base.py:476-480)
    assert n >= 12
    yield patch
    patch.uninstall()


def _make(name):
    from colosseum.mdp.deep_sea import DeepSeaContinuous
    from colosseum.mdp.frozen_lake import FrozenLakeEpisodic
    from colosseum.mdp.river_swim import RiverSwimEpisodic
    from colosseum.mdp.simple_grid import SimpleGridContinuous, SimpleGridEpisodic

    return {
        "doc_simplegrid4": lambda: SimpleGridContinuous(seed=0, size=4, p_rand=0.01, n_starting_states=3),
        "deepsea10": lambda: DeepSeaContinuous(seed=0, size=10, p_rand=None),
        "frozenlake4_epi": lambda: FrozenLakeEpisodic(seed=1, size=4, p_frozen=0.8),
        "simplegrid5_epi": lambda: SimpleGridEpisodic(seed=2, size=5, p_lazy=0.1, p_rand=0.1),
        "c1_riverswim_epi": lambda: RiverSwimEpisodic(
            seed=0, size=5, p_lazy=0.1, make_reward_stochastic=True, randomize_actions=False,
            sub_optimal_distribution=("beta", (2.4, 24.0)), optimal_distribution=("beta", (0.01, 0.11)),
            other_distribution=("beta", (2.4, 249.0))),
    }[name]()


@pytest.mark.parametrize("name", ["doc_simplegrid4", "deepsea10", "frozenlake4_epi", "simplegrid5_epi", "c1_riverswim_epi"])
def test_reference_properties_run_on_the_gpu(ref, name):
    from colosseum_b200 import _cabi

    g = load_instance(name)
    mdp = _make(name)
    assert np.array_equal(mdp.T, g["T"]) and np.allclose(mdp.R, g["R"])  # same instance as the golden
    n0 = _cabi.lib().colo_launch_count()
    Q, V = mdp.optimal_value_functions
    assert _cabi.lib().colo_launch_count() > n0, "the reference's property did not reach the GPU library"
    # install() defaults to the reference's own early-stopped iterates (in-place sweeps, its epsilon): same numbers
    # up to the stopping tolerance (continuous) / fp32 rounding (episodic: exact recurrence)
    tol = 2e-5 if mdp.is_episodic() else 2e-3
    np.testing.assert_allclose(V, g["vi_V"], atol=tol)
    np.testing.assert_allclose(Q, g["vi_Q"], atol=tol)
    Qr, Vr = mdp.random_value_functions
    np.testing.assert_allclose(Vr, g["pe_V"], atol=2e-4)
    d = mdp.diameter
    assert abs(d - float(g["diameter"])) < 2e-3 * max(1.0, float(g["diameter"])), (d, float(g["diameter"]))
    gaps = mdp.sum_reciprocals_suboptimality_gaps
    assert abs(gaps - float(g["gaps"])) < 6e-3 * float(g["gaps"]), (gaps, float(g["gaps"]))
    vn = mdp.value_norm
    assert abs(vn - float(g["value_norm"])) < 3e-3 * max(float(g["value_norm"]), 1e-3), (vn, float(g["value_norm"]))
    moh = mdp.measures_of_hardness
    assert set(moh) == {"diameter", "suboptimal_gaps", "value_norm"} and moh["diameter"] == d
    # the policy layer on top of the GPU value functions
    pi = mdp.get_optimal_policy(False)
    assert pi.shape == Q.shape[:-1]
    Qw, Vw = mdp.worst_value_functions
    assert float(np.max(Vw - V)) <= 1e-3  # the worst policy is never better than the optimal one


def test_notebook_values_through_the_live_reference(ref):
    """docs/_sources/mds/hardness-analysis.ipynb:83-193 through the patched reference object"""
    mdp = _make("doc_simplegrid4")
    assert abs(mdp.diameter - 6.0545096) < 2e-3
    assert abs(mdp.value_norm - 0.49540126) < 3e-3 * 0.4954
    assert abs(mdp.sum_reciprocals_suboptimality_gaps - 361.29538) < 6e-3 * 361.3


def test_batched_mdp_from_a_live_reference_mdp(ref):
    """MDPTables.from_mdp on a live object: the attribute surface of BatchedMDP equals the reference's own"""
    import colosseum_b200.batched_mdp as bm
    from colosseum_b200.tables import MDPTables

    mdp = _make("frozenlake4_epi")
    env = bm.BatchedMDP(MDPTables.from_mdp(mdp), 1, mode="succ", scalar_api=True)
    assert env.n_states == mdp.n_states and env.n_actions == mdp.n_actions and env.H == mdp.H
    assert np.array_equal(env.T, mdp.T) and np.array_equal(env.R, mdp.R)
    assert np.allclose(env.starting_state_distribution, mdp.starting_state_distribution)
    assert env.node_to_index == mdp.node_to_index and env.index_to_node == mdp.index_to_node
    assert env.action_spec().num_values == mdp.action_spec().num_values
    assert env.observation_spec().num_values == mdp.observation_spec().num_values
    ts_ref, ts = mdp.reset(), env.reset()
    assert ts.step_type == ts_ref.step_type and ts.reward is None and ts.observation == ts_ref.observation
    for _ in range(3 * mdp.H):
        ts, a = env.random_step(auto_reset=True)
        assert ts.observation == -1 or 0 <= ts.observation < mdp.n_states
