"""CPU: host-side table extraction (colosseum_b200/tables.py) against the arrays recorded from the reference."""
import numpy as np
import pytest

from conftest import CONTINUOUS, EPISODIC, load_instance
from colosseum_b200.tables import MDPTables, quantile_table, running_sum


@pytest.mark.parametrize("name", CONTINUOUS + EPISODIC)
def test_tables_from_golden(name):
    g = load_instance(name)
    tb = MDPTables.from_golden(g)
    S, A = tb.S, tb.A
    # dense T rebuilt from the successor lists (duplicates summed) == the reference's T (mdp_creation.py:80)
    tb2 = MDPTables.from_successors(S, A, g["succ_idx"], g["succ_prob"], g["succ_len"], g["rew_cls"],
                                    tb.rew_kinds, g["start_idx"], g["start_prob"], H=tb.H)
    np.testing.assert_allclose(tb2.T, g["T"], rtol=0, atol=2e-7)  # the reference sums duplicates in fp32
    # expected rewards from (p, reward class means) == the reference's R (mdp_creation.py:71-81)
    np.testing.assert_allclose(tb.expected_rewards(), g["R"], rtol=1e-5, atol=1e-6)
    # running sums: last finite entry is the row total ~ 1, padding is +inf, indices padded with the last successor
    last = np.take_along_axis(tb.succ_cum, (tb.succ_len - 1)[..., None].astype(np.int64), -1)[..., 0]
    np.testing.assert_allclose(last, 1.0, atol=1e-9)
    K = tb.succ_cum.shape[-1]
    pad = np.arange(K)[None, None, :] >= tb.succ_len[..., None]
    assert np.isinf(tb.succ_cum[pad]).all()
    assert (tb.succ_cum[..., 1:] >= tb.succ_cum[..., :-1]).all()  # non-decreasing, +inf padding included
    assert tb.rew_cls_sas.shape == (S, A, S) and tb.rew_q.shape[0] == len(tb.rew_kinds)
    assert tb.ld % 32 == 0 and tb.ld >= S
    assert abs(tb.start_cum[-1] - 1.0) < 1e-9 and tb.n_start == len(g["start_idx"])


def test_running_sum_is_sequential():
    p = np.random.RandomState(0).dirichlet(np.ones(13))
    acc, ref = 0.0, []
    for x in p:
        acc = acc + x
        ref.append(acc)
    assert (running_sum(p) == np.asarray(ref)).all()  # bit-for-bit itertools.accumulate


def test_quantile_tables():
    q = quantile_table("deterministic", (0.25,), 17)
    assert (q == np.float32(0.25)).all()
    q = quantile_table("beta", (2.4, 24.0), 1025)
    assert q[0] == 0.0 and q[-1] == 1.0 and (np.diff(q) >= 0).all()
    q = quantile_table("norm", (0.0, 1.0), 1025)
    assert np.isfinite(q).all() and (np.diff(q) > 0).all()


@pytest.mark.reference
def test_from_mdp_matches_golden_recording():
    """the duck-typed extractor on a live reference object == what make_golden.py recorded (build container only)"""
    from oracle.reference_import import import_reference, reference_available

    if not reference_available():
        pytest.skip("the unmodified Colosseum package is not staged (oracle/_ref or $COLOSSEUM_REFERENCE_ROOT)")
    import_reference()
    import colosseum.mdp  # noqa: F401
    from colosseum.mdp.simple_grid import SimpleGridContinuous

    mdp = SimpleGridContinuous(seed=0, size=4, p_rand=0.01, n_starting_states=3)
    tb = MDPTables.from_mdp(mdp)
    g = load_instance("doc_simplegrid4")
    ref = MDPTables.from_golden(g)
    for f in ("succ_idx", "succ_cum", "succ_len", "rew_cls_succ", "T", "rew_cls_sas", "start_idx", "start_cum", "rew_q"):
        assert np.array_equal(getattr(tb, f), getattr(ref, f)), f
    assert tb.rew_kinds == ref.rew_kinds and (tb.S, tb.A, tb.H) == (ref.S, ref.A, ref.H)


@pytest.mark.reference
def test_patch_rebinds_reference_names():
    """colosseum_b200.patch.install() replaces every by-name binding of the hot-path entry points inside the imported
    reference package, and uninstall() restores them (mechanics only: no GPU call is made here)"""
    from oracle.reference_import import import_reference, reference_available

    if not reference_available():
        pytest.skip("the unmodified Colosseum package is not staged (oracle/_ref or $COLOSSEUM_REFERENCE_ROOT)")
    import_reference()
    import colosseum.mdp  # noqa: F401
    import colosseum.hardness.measures.diameter as ref_diam
    import colosseum.mdp.base as ref_base
    import colosseum.mdp.base_finite as ref_fin
    import colosseum_b200.dynamic_programming as dp
    import colosseum_b200.hardness as hd
    import colosseum_b200.patch as patch

    orig = ref_base.get_diameter
    n = patch.install()
    try:
        assert n >= 12
        assert ref_base.get_diameter is hd.get_diameter and ref_base.calculate_norm_discounted is hd.calculate_norm_discounted
        assert ref_fin.episodic_value_iteration is dp.episodic_value_iteration
        assert ref_fin.discounted_value_iteration is dp.discounted_value_iteration
        assert ref_diam.discounted_value_iteration is dp.discounted_value_iteration
    finally:
        assert patch.uninstall() == n
    assert ref_base.get_diameter is orig


@pytest.mark.reference
def test_patched_reference_fails_loudly_without_gpu():
    """with the GPU path installed behind the reference's names there is NO fallback: on a box without a CUDA device
    the reference's own properties raise instead of silently running numba"""
    import torch

    from oracle.reference_import import import_reference, reference_available

    if not reference_available():
        pytest.skip("the unmodified Colosseum package is not staged (oracle/_ref or $COLOSSEUM_REFERENCE_ROOT)")
    if torch.cuda.is_available():
        pytest.skip("needs a box without a GPU")
    import_reference()
    from colosseum.mdp.river_swim import RiverSwimContinuous

    import colosseum_b200.patch as patch
    from colosseum_b200._cabi import ColosseumB200Error

    n = patch.install()  # BEFORE constructing MDPs: an MDP object binds its DP function at construction (base.py:476-480)
    try:
        assert n > 0
        mdp = RiverSwimContinuous(seed=0, size=6)
        with pytest.raises(ColosseumB200Error):
            mdp.optimal_value_functions
        with pytest.raises(ColosseumB200Error):
            mdp.diameter
    finally:
        patch.uninstall()
    mdp = RiverSwimContinuous(seed=0, size=6)
    assert mdp.optimal_value_functions[1].shape == (6,)  # restored: the reference's numba path again


def test_split_sizes_cover_the_batch_contiguously():
    """the shards of PipelinedBatchedMDP: contiguous, covering, sizes differing by at most one"""
    from colosseum_b200.batched_mdp import split_sizes

    for n, g in ((65536, 2), (65536, 3), (1001, 3), (7, 7), (5, 1)):
        sizes, offsets = split_sizes(n, g)
        assert sum(sizes) == n and len(sizes) == g and max(sizes) - min(sizes) <= 1
        assert offsets[0] == 0 and all(offsets[i + 1] == offsets[i] + sizes[i] for i in range(g - 1))
    assert split_sizes(1001, 3) == ([334, 334, 333], [0, 334, 668])


def test_batched_apis_fail_loudly_without_gpu():
    """no CPU fallback anywhere: the batched env, the pipelined groups and the agent loops raise on a box without a
    CUDA device instead of computing on the host"""
    import torch

    if torch.cuda.is_available():
        pytest.skip("needs a box without a GPU")
    from conftest import load_instance
    from colosseum_b200._cabi import ColosseumB200Error
    from colosseum_b200.tables import MDPTables
    import colosseum_b200.agent_loop as al
    import colosseum_b200.batched_mdp as bm

    tb = MDPTables.from_golden(load_instance("c1_riverswim_epi"))
    for make in (lambda: bm.BatchedMDP(tb, 8), lambda: bm.PipelinedBatchedMDP(tb, 8, groups=2),
                 lambda: al.QLearningEpisodic(0, tb, 100, p=0.05, c_1=0.5, n_loops=4),
                 lambda: al.PSRLEpisodic(0, tb, 100, n_loops=4)):
        with pytest.raises(ColosseumB200Error):
            make()
