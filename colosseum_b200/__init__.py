"""colosseum_b200 -- B200-native (sm_100a) implementation of Colosseum's data-parallel hot path:
the batched agent/MDP interaction step and the dynamic-programming Bellman backups behind the hardness measures.

    colosseum_b200.dynamic_programming   twin of colosseum.dynamic_programming
    colosseum_b200.hardness              twin of colosseum.hardness.measures
    colosseum_b200.batched_mdp           BatchedMDP: N parallel BaseMDP.reset/step
                                         MixedBatchedMDP: envs of many MDP instances in one batch, one launch per step
    colosseum_b200.tables                host-side table extraction from reference MDP objects
    colosseum_b200.patch                 install the GPU path behind the reference's own module attributes

Everything computes in hand-written CUDA kernels behind the C ABI of include/colosseum_b200.h.
There is no CPU, PyTorch-eager or Triton fallback: without the built library or a GPU the calls raise.
"""
__version__ = "0.1.0"
