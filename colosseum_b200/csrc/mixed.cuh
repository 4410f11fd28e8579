// mixed.cuh -- the mixed-batch handle (colo_mixed_tables), shared by the env kernels of env_step.cu that create and step
// it and by the agent-loop kernels of agents.cu that run agents on its instances.
#pragma once
#include "common.cuh"

namespace colo {

// Instance i owns the contiguous envs [start, start + n_i).  Env e looks up its instance in inst_of[e] and then runs the
// per-env code on that instance's tables, Philox key and counter (seed_i; e - start), and counter offsets.  Envs of
// one instance are contiguous, so the lanes of a warp almost always read the same descriptor (one broadcast load).
struct MixedInst {
  colo_mdp_tables tb;
  unsigned long long seed;
  long long start;          // first env of the instance
  long long off_s, off_sa;  // sum of S, of S*A over the instances before it: its columns in the counter rows
};

}  // namespace colo

struct colo_mixed_tables {
  int n_inst, mode;
  long long N, sum_s, sum_sa;
  colo::MixedInst* insts;       // device [n_inst]
  int* inst_of;                 // device [N]: instance of every env
  colo::MixedInst* host_insts;  // host copy of insts: callers check their arguments against it before any CUDA call
};
