/*
 * colosseum_b200.h -- C ABI of libcolosseum_b200.so (sm_100a).
 *
 * Drop-in boundary for the ONE data-parallel hot path of MichelangeloConserva/Colosseum (SURVEY.md section 8):
 *   (A) the batched agent/MDP interaction step       -- colosseum/mdp/base.py:1268-1317
 *   (B) the Bellman backups behind the hardness       -- colosseum/dynamic_programming/{finite,infinite}_horizon.py,
 *       measures and model-based agents                  colosseum/hardness/measures/*.py
 *
 * The reference has no FFI of its own (it is pure Python + numba); these are the entry points a ctypes binding
 * placed behind the reference's Python signatures would call (INTEGRATION.md shows that binding).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (torch tensors on the host side), unless the
 *     parameter name ends in `_host`;
 *   - arrays are C-contiguous with the layouts of the reference (T[S,A,S], R[S,A], Q[S,A], V[S], episodic
 *     Q[H+1,S,A] / V[H+1,S]); batched variants add a leading B;
 *   - every call takes the cudaStream_t (as void*) it enqueues on and does NOT synchronise unless stated;
 *   - return value: COLO_OK (0); COLO_OVERFLOW (1) = the reference's `return None` on max_value/max_abs_value;
 *     COLO_MAX_ITER (2) = the reference's DynamicProgrammingMaxIterationExceeded; COLO_NEEDS_RESET (3) = the
 *     reference's `assert not self.necessary_reset`; < 0 = CUDA error / bad argument, text in colo_last_error().
 */
#ifndef COLOSSEUM_B200_H_
#define COLOSSEUM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define COLO_OK 0
#define COLO_OVERFLOW 1
#define COLO_MAX_ITER 2
#define COLO_NEEDS_RESET 3
#define COLO_SERVER_LAPSED 4
#define COLO_BAD_ACTION 5 /* a supplied action outside [0, A): flagged in colo_env_batch.status, the env is not stepped */
#define COLO_ERR_CUDA (-1)
#define COLO_ERR_ARG (-2)

/* backup modes: how Q[s,:] is folded into V[s] */
#define COLO_FOLD_MAX 0 /* value iteration            V[s] = max_a Q[s,a]            */
#define COLO_FOLD_PI 1  /* policy evaluation          V[s] = sum_a pi[s,a] Q[s,a]    */
#define COLO_FOLD_MIN 2 /* hitting times (diameter)   V[s] = min_a Q[s,a]            */

/* dm_env.StepType */
#define COLO_STEP_FIRST 0
#define COLO_STEP_MID 1
#define COLO_STEP_LAST 2

/* ---------------------------------------------------------------- library ------------------------------- */
const char* colo_last_error(void);
int colo_version(void);
/* number of kernels this library has launched since load / since the last reset (bench.py's gpu_launches) */
unsigned long long colo_launch_count(void);
/* cudaStreamSynchronize(stream): the host-side wait of a zero-copy env step (one ctypes call, no Python layers) */
int colo_stream_synchronize(void* stream);
void colo_reset_launch_count(void);
/* sweeps taken by the TMA-staged variant of the streaming backup kernel (COLO_BACKUP_TMA=1, DESIGN 4.1) since load */
unsigned long long colo_backup_tma_sweeps(void);
/* step launches since load that went to each step-kernel variant (`kind`: COLO_STEP_KIND_*; 0 for any other value).
 * Counted on the host when the launch is enqueued: a launch captured into a CUDA graph counts once. */
#define COLO_STEP_KIND_LEAN 0  /* env_step_kary_lean_kernel: the common dense f32 call                         */
#define COLO_STEP_KIND_KARY 1  /* env_step_dense_kary_kernel: rows of <= 1024 states, every other dense call    */
#define COLO_STEP_KIND_SHORT 2 /* env_step_dense_short_kernel: the warp-cooperative kernel (COLO_STEP_KERNEL=coop) */
#define COLO_STEP_KIND_LONG 3  /* env_step_dense_kernel: rows of more than 1024 states (or ld % 128 != 0)      */
#define COLO_STEP_KIND_SUCC 4  /* env_step_succ_kernel: successor-list tables                                  */
#define COLO_STEP_KIND_MIXED_SUCC 5  /* env_step_succ_mixed_kernel: a mixed batch, successor-list tables       */
#define COLO_STEP_KIND_MIXED_DENSE 6 /* env_step_dense_mixed_kernel: a mixed batch, dense rows (f32 or f64)   */
#define COLO_STEP_KIND_BREAKS 7 /* env_step_breaks_lean_kernel: the common dense f32 call, breakpoint table set     */
#define COLO_STEP_KIND_BREAKS_GENERAL 8 /* env_step_dense_kary_kernel searching the breakpoint table (other f32 calls) */
#define COLO_STEP_KINDS 9
unsigned long long colo_step_kernel_launches(int kind);

/* ---------------------------------------------------------------- (B) Bellman backups ------------------- */
/*
 * One synchronous (Jacobi) backup of B independent MDPs (one kernel launch, T is read once):
 *     Q[b,s,a] = R[b,s,a] + gamma * sum_j T[b,s,a,j] * V_in[b,j];   V_out[b,s] = fold_a Q[b,s,a]
 * Restates the sweep body of  colosseum/dynamic_programming/infinite_horizon.py:131-135 (VI), :176-179 (PE),
 * colosseum/dynamic_programming/finite_horizon.py:21-23, :38-40 (one horizon layer) and the hitting-time sweep of
 * colosseum/hardness/measures/diameter.py:330-339 as one parallel sweep.  All strides are in ELEMENTS between
 * consecutive instances b (t_stride = 0 shares one T between all instances, e.g. the K targets of a diameter).
 *   _f32    : T,R,pi float; V,Q float;  fp32 accumulation (the reference's arithmetic type)
 *   _f64acc : T,R,pi float; V,Q double; fp64 accumulation (the 1e-6 parity mode of BASELINE.json)
 */
typedef struct {
  const float* T;        /* [B][nrows,A,S] rows row0..row0+nrows of each instance (nrows = S unless row-sharded) */
  const float* R;        /* [B][nrows,A] or NULL (then r_const is used)                                          */
  const float* pi;       /* [B][nrows,A], COLO_FOLD_PI only                                                      */
  const void* V_in;      /* [B][S] (float | double); with v_action_stride != 0: [B][A][S], one vector per action */
  void* V_out;           /* [B][S] or NULL; only entries row0..row0+nrows are written                            */
  void* Q;               /* [B][nrows,A] or NULL                                                                 */
  long long t_stride, r_stride, pi_stride, v_in_stride, v_out_stride, q_stride, v_action_stride;
  int B, S, A, fold;
  double gamma, r_const;
  void* resid;           /* per instance max|V_out - V_in| as the bits of a non-negative float (u32) | double
                            (u64), accumulated with atomicMax; zero it before the sweep; or NULL                 */
  int resid_vs_out;      /* != 0: the residual compares with the previous content of V_out instead of V_in      */
  const unsigned char* active; /* per instance; 0 = converged: V is carried forward, nothing else is touched    */
  double max_abs;        /* > 0: set *overflow_flag = 1 when |V_out| exceeds it (the reference's `return None`);
                            with overflow_signed != 0 the test is V_out > max_abs (finite_horizon.py:24-25)      */
  int overflow_signed;
  int* overflow_flag;
  int row0, nrows;       /* nrows == 0 && row0 == 0 means all S rows                                             */
  const int* pin_index;  /* per instance or NULL: V_out[b, pin_index[b]] = pin_value (absorbing target)          */
  double pin_value;
  const int* exclude_index; /* per instance or NULL: V_in[b, exclude_index[b]] is read as exclude_value          */
  double exclude_value;
  void* const* V_out_peers; /* device array of n_peers pointers or NULL: V_out rows are ALSO stored into every
                               listed [B][S] buffer (peer GPUs' V over NVLink: the all-gather of a row-sharded
                               sweep fused into the backup's epilogue, SURVEY.md section 8e-3)                    */
  int n_peers;
} colo_backup_args;

int colo_backup_f32(const colo_backup_args* args, void* stream);
int colo_backup_f64acc(const colo_backup_args* args, void* stream);

/*
 * On-chip resident solver: ONE launch runs a whole solve for problems whose T fits the shared memory of a
 * thread-block cluster (<= 16 CTAs x 227 KB).  Problem b is iterated by cluster b: every CTA keeps its slice of T
 * rows in shared memory for the entire solve, the value vectors are exchanged through distributed shared memory
 * with one cluster barrier per sweep, and the stopping rule (max|dV| < eps after a sweep, the reference's
 * infinite_horizon.py:140-141), the overflow test and the max_iter cap are evaluated on the device.
 *   NV = 1: B independent MDPs (t_stride/r_stride = elements between their T/R; V [B][S], Q [B][S,A] or NULL).
 *   NV = 4: tiles of 4 value vectors sharing one T (t_stride = 0): the multi-target hitting-time iteration of the
 *           diameter (diameter.py:76-106) -- V [B*4][S], pin_index [B*4] = targets, fold MIN, gamma 1, r_const 1.
 *   episodic_H > 0: exactly H sweeps without a stopping rule; sweep i stores layer H-1-i of V [B][H+1][S] and
 *           Q [B][H+1][S,A] (finite_horizon.py:11-42; the caller zeroes layer H); pi is then [B][H][S,A].
 * status_out[b] (device): COLO_OK / COLO_OVERFLOW / COLO_MAX_ITER; iters_out[B*NV] (device, may be NULL).
 * colo_resident_fits returns 1 (and the cluster size) when (S, A, NV) fits.  Does not synchronise.
 */
typedef struct {
  const float* T;
  const float* R;      /* or NULL: r_const */
  const float* pi;     /* COLO_FOLD_PI only */
  void* V;
  void* Q;             /* or NULL */
  long long t_stride, r_stride;
  int B, S, A, NV, fold;
  double gamma, r_const, eps;
  double max_abs;      /* > 0 enables the overflow test: |V| > max_abs, or V > max_abs when overflow_signed != 0 */
  int overflow_signed;
  long long max_iter;
  int episodic_H;
  const int* pin_index; /* [B*NV] or NULL */
  double pin_value;
  long long* iters_out;
  int* status_out;
} colo_resident_args;

int colo_resident_fits(int S, int A, int NV, int f64, int* cluster_size_out);
int colo_resident_solve_f32(const colo_resident_args* args, void* stream);
int colo_resident_solve_f64acc(const colo_resident_args* args, void* stream);

/*
 * Discounted value iteration / policy evaluation to convergence for B independent MDPs
 * (colosseum/dynamic_programming/infinite_horizon.py:14-64,121-184).  V starts at 0.  Sweeps are synchronous
 * (Jacobi); an instance stops after the sweep in which max_s|dV| < eps (the reference's test, :140-141) and its
 * Q is the Q of that sweep; returns COLO_OVERFLOW if any |V| > max_abs (pass max_abs <= 0 to disable; :136-138),
 * COLO_MAX_ITER after max_iter sweeps (:142).  fold = COLO_FOLD_MAX (VI) or COLO_FOLD_PI (PE, pi [B,S,A]).
 * Synchronises the stream (the host needs the convergence flags).  iters_out_host[b] = sweeps run by b (or NULL).
 * work: device scratch of colo_solve_work_bytes(B,S,f64) bytes.  Q may be NULL.
 * The kernel is chosen from the tensor itself, never by a flag: T with sparse rows (<= 256 non-zeros and <= 1/8 of a
 * row: the benchmark families, continuous forms) is compressed on the device and solved on chip in one launch
 * (S <= 2048) or with one compressed-row launch per sweep; small dense MDPs (colo_resident_fits) go to the resident
 * cluster solver in one launch; everything else streams T from HBM, one backup launch per sweep.  Same algorithm
 * (synchronous sweeps), same stopping rule, same results up to the summation order inside a row.
 */
size_t colo_solve_work_bytes(long long B, long long S, int f64);
int colo_solve_discounted_f32(const float* T, const float* R, const float* pi, int B, int S, int A, float gamma,
                              float eps, float max_abs, long long max_iter, int fold, float* Q, float* V,
                              long long* iters_out_host, void* work, void* stream);
int colo_solve_discounted_f64acc(const float* T, const float* R, const float* pi, int B, int S, int A,
                                 double gamma, double eps, double max_abs, long long max_iter, int fold, double* Q,
                                 double* V, long long* iters_out_host, void* work, void* stream);

/*
 * The reference's OWN iterate: in-place (Gauss-Seidel) sweeps, infinite_horizon.py:121-142 / :167-184 -- for s in
 * range(S): Q[s] = R[s] + gamma T[s] @ V; V[s] = fold(Q[s]) with V updated in place; stop when max|V_old - V| < eps
 * after a sweep; COLO_OVERFLOW as soon as |V[s]| > max_abs (> 0).  One warp per instance, V in shared memory, the
 * whole solve in one launch (does not synchronise): status_dev[b] = COLO_OK / COLO_OVERFLOW / COLO_MAX_ITER and
 * iters_dev[b] are DEVICE arrays.  Returns the reference's early-stopped (Q, V) up to the summation order of the
 * row dot products (the colo_solve_discounted_* entry points sweep synchronously: same fixed point, other iterates).
 */
int colo_solve_discounted_gs_f32(const float* T, const float* R, const float* pi, int B, int S, int A, float gamma,
                                 float eps, float max_abs, long long max_iter, int fold, float* Q, float* V,
                                 long long* iters_dev, int* status_dev, void* stream);
int colo_solve_discounted_gs_f64acc(const float* T, const float* R, const float* pi, int B, int S, int A, double gamma,
                                    double eps, double max_abs, long long max_iter, int fold, double* Q, double* V,
                                    long long* iters_dev, int* status_dev, void* stream);

/*
 * Episodic backward induction for B MDPs (colosseum/dynamic_programming/finite_horizon.py:11-42):
 * Q[b,H]=0, V[b,H]=0; for h=H-1..0: Q[b,h]=R+T@V[b,h+1]; V[b,h]=fold(Q[b,h]) with pi[b,h] for PE
 * (pi is [B,H,S,A]).  Q is [B,H+1,S,A], V is [B,H+1,S].  max_value<=0 disables the overflow test (:24-25);
 * with it enabled the call synchronises and may return COLO_OVERFLOW.
 */
int colo_episodic_f32(const float* T, const float* R, const float* pi, int B, int S, int A, int H, int fold,
                      float max_value, float* Q, float* V, void* stream);
int colo_episodic_f64acc(const float* T, const float* R, const float* pi, int B, int S, int A, int H, int fold,
                         double max_value, double* Q, double* V, void* stream);
/*
 * B policies pi f32[B,H,S,A] evaluated on ONE episodic MDP (T f32[S,A,S], R f32[S,A]) in one launch: the regret
 * indicator of every loop of a batched agent run per log tick (colosseum/experiment/indicators.py:29-45 calls
 * episodic_policy_evaluation once per agent).  Q [B,H+1,S,A], V [B,H+1,S].  Does not synchronise.
 */
int colo_episodic_policies_f32(const float* T, const float* R, const float* pi, int B, int S, int A, int H, float* Q,
                               float* V, void* stream);
int colo_episodic_policies_f64acc(const float* T, const float* R, const float* pi, int B, int S, int A, int H,
                                  double* Q, double* V, void* stream);

/*
 * Optimal values of the CONTINUOUS FORM of an episodic MDP (mdp/utils/mdp_creation.py:131-176 +
 * mdp/base_finite.py:167-178: discounted_value_iteration on the n x A x n tensor over the reachable (h, s) nodes) from
 * the structure of that tensor, without building it: the fixed point depends on ONE scalar c = sum_k p[k] *
 * V[pos_h[k], pos_s[k]] (the value the last layer jumps to; pos = the node sitting at list position start_k, sic
 * :168), one backward induction over the original T maps c to F(c), and c* = F(c*) is found by safeguarded secant
 * steps.  V [H][S] (device) receives the values of EVERY (h, s) pair at c*, to |error| <= eps; the caller gathers the
 * reachable nodes in the reference's order.  pos_h, pos_s, p (float32 start probabilities as stored in T_cf): device
 * arrays of n_start entries.  out_host[0] = c*, out_host[1] = backward inductions run.  COLO_MAX_ITER after max_eval.
 * Synchronises.
 */
int colo_continuous_form_values_f32(const float* T, const float* R, int S, int A, int H, double gamma, const int* pos_h,
                                    const int* pos_s, const float* p, int n_start, double eps, int max_eval, float* V,
                                    double* out_host, void* stream);
int colo_continuous_form_values_f64acc(const float* T, const float* R, int S, int A, int H, double gamma, const int* pos_h,
                                       const int* pos_s, const float* p, int n_start, double eps, int max_eval, double* V,
                                       double* out_host, void* stream);

/*
 * Continuous diameter (colosseum/hardness/measures/diameter.py:20-39,76-106; == :321-346 at the fixed point):
 * multi-target hitting-time iteration  E[k,s] = (s == target[k]) ? 0 : min_a(1 + sum_j T[s,a,j] E[k,j])  over the
 * K given targets at once (all S for the full diameter), every target (tile of targets) iterated until its own
 * max|dE| < eps.  Sparse rows: compressed rows, a few targets per CTA with E in shared memory, the whole solve in one
 * launch; dense T that fits a cluster's shared memory: resident solver, 4 targets per cluster; otherwise one tiled
 * GEMM launch per sweep (>= 128^2 (target, state) pairs) or one streaming backup launch per sweep.  In f32 mode with
 * S >= 128 and K >= 64 that GEMM runs on the tensor cores (hitting_umma.cu: tcgen05.mma kind::tf32 with both
 * operands split hi + lo, three products per k-step into fp32 TMEM accumulators, TMA-fed through an mbarrier ring).
 * out_host[0] = max_k max_s E, out_host[1] = sweeps run (max over targets).  COLO_OVERFLOW if a hitting time
 * exceeds max_value (>0).  Synchronises.  work: colo_diameter_continuous_work_bytes(K,S,f64) device bytes.
 */
size_t colo_diameter_continuous_work_bytes(int K, int S, int f64);
int colo_diameter_continuous_f32(const float* T, const int* targets, int K, int S, int A, float eps,
                                 float max_value, long long max_iter, void* work, double* out_host, void* stream);
int colo_diameter_continuous_f64acc(const float* T, const int* targets, int K, int S, int A, double eps,
                                    double max_value, long long max_iter, void* work, double* out_host,
                                    void* stream);
/*
 * Episodic diameter in the augmented (h,s) space (colosseum/hardness/measures/diameter.py:193-234,285-318) on
 * T_epi[H,S,A,S] (colosseum/mdp/utils/mdp_creation.py:98-128), iterated to max|dE| < eps for all K targets at once.
 */
/*
 * The reference's continuous diameter ITERATE FOR ITERATE (diameter.py:76-106): per target es a discounted VI with
 * gamma = 1 on T_es (es absorbing) and R_es = -1 (0 at es), in-place (Gauss-Seidel) sweeps stopped at max|dV| < eps
 * (the reference's default 1e-3), diameter = max_es (-min_s V_es).  One warp per target, all targets share T; the whole
 * computation is one launch + one reduction.  Reproduces the reference's own early-stopped value (which sits up to
 * ~5e-4 below the fixed point that colo_diameter_continuous_* returns).  Synchronises.
 */
/*
 * colo_hitting_umma_sweeps_f32 -- n_sweeps synchronous sweeps of the multi-target hitting-time iteration above through
 * the tcgen05 kernel alone (parity and throughput probe of that kernel): E f32 [K][S] is iterated in place (zeroed first
 * when zero_start != 0), E_work is a second [K][S] buffer.  COLO_ERR_ARG when the shape is outside the kernel's range
 * (S >= 128, K >= 64).  Does not synchronise.
 */
int colo_hitting_umma_sweeps_f32(const float* T, const int* targets, int K, int S, int A, int n_sweeps, int zero_start,
                                 float* E, float* E_work, void* stream);

size_t colo_diameter_continuous_gs_work_bytes(int K, int S, int f64);
int colo_diameter_continuous_gs_f32(const float* T, const int* targets, int K, int S, int A, float eps, float max_value,
                                    long long max_iter, void* work, double* out_host, void* stream);
int colo_diameter_continuous_gs_f64acc(const float* T, const int* targets, int K, int S, int A, double eps,
                                       double max_value, long long max_iter, void* work, double* out_host, void* stream);
size_t colo_diameter_episodic_work_bytes(int K, int H, int S, int A, int f64);
int colo_diameter_episodic_f32(const float* T_epi, const int* targets, int K, int H, int S, int A, float eps,
                               float max_value, long long max_iter, void* work, double* out_host, void* stream);
int colo_diameter_episodic_f64acc(const float* T_epi, const int* targets, int K, int H, int S, int A, double eps,
                                  double max_value, long long max_iter, void* work, double* out_host, void* stream);

/*
 * Environmental value norm (colosseum/hardness/measures/value_norm.py:55-61,85-87), two passes over T:
 *   Ev[i,a] = sum_j T[i,a,j] V[j];   out[0] = max_{i,a} sqrt( sum_j T[i,a,j] * (V[j] - Ev[j,a])^2 )
 * (sic: Ev is indexed by the NEXT state j, reference behaviour).  out: 1 element (device).  Does not synchronise.
 * work: colo_value_norm_work_bytes(S,A,f64) device bytes.
 */
size_t colo_value_norm_work_bytes(int S, int A, int f64);
int colo_value_norm_f32(const float* T, const float* V, int S, int A, void* work, float* out, void* stream);
int colo_value_norm_f64acc(const float* T, const double* V, int S, int A, void* work, double* out, void* stream);

/*
 * Sum of reciprocals of the sub-optimality gaps
 * (colosseum/hardness/measures/sum_reciprocals_suboptimality_gaps.py:6-28):
 *   out[0] = sum_{n<NS, a<A, mask[n]} 1 / (V[n] - Q[n,a] + reg)     (mask may be NULL = all; episodic callers
 * pass NS=(H+1)*S rows and the reachable (h,s) mask).  Deterministic fp64 reduction (fixed order).
 */
/*
 * colo_bias_series_f64 -- _calculate_gain / _calculate_bias (colosseum/hardness/measures/value_norm.py:64-82), the
 * vector the UNDISCOUNTED value norm (calculate_norm_average, :90-93) is taken of:  gain = P^steps r,
 * h = sum_{i < steps} P^i (r - gain), P f32 [S,S] the chain of the policy (colo_policy_chain), r f32 [S] its average
 * rewards.  fp64 accumulation (the reference mixes float32 matrix_power and float64 sums; its 60 s wall-clock cut-off of
 * the series is not reproduced).  The norm itself is colo_value_norm_f64acc(T, h).  Does not synchronise.
 */
size_t colo_bias_series_work_bytes(int S);
int colo_bias_series_f64(const float* P, const float* avg_rewards, int S, int steps, double* h_out, void* work,
                         void* stream);
int colo_gaps_f64(const double* Q, const double* V, const unsigned char* mask, long long NS, int A, double reg,
                  double* out, void* stream);

/* ---------------------------------------------------------------- extended value iteration (UCRL2) --------- */
/*
 * extended_value_iteration + _max_proba (colosseum/dynamic_programming/infinite_horizon.py:67-118, :222-251; called by
 * colosseum/agent/agents/infinite_horizon/ucrl2.py:330).  T f32[S,A,S] (the empirical model), est_rewards f32[S,A],
 * beta_r f64[S,A], beta_p f64[S,A] (the reference passes [S,A,1] -- or [S,A,S] of which it reads element 0 only,
 * :230).  Synchronous iterations u1 -> u2 from u = 0 until ptp(u2 - u1) < eps; outputs Q [S,A], V [S] of the stopping
 * iteration, out_host[0] = ptp(u1) (the span the reference returns), out_host[1] = iterations.  Returns COLO_OK, or
 * COLO_MAX_ITER after max_iter iterations (the reference then returns None).  Synchronises.  S <= 8192.
 * work: colo_extended_vi_work_bytes(S, f64) bytes of device scratch.
 */
size_t colo_extended_vi_work_bytes(int S, int f64);
int colo_extended_vi_f32(const float* T, const float* est_rewards, const double* beta_r, const double* beta_p, int S,
                         int A, double r_max, double eps, long long max_iter, float* Q, float* V, double* out_host,
                         void* work, void* stream);
int colo_extended_vi_f64acc(const float* T, const float* est_rewards, const double* beta_r, const double* beta_p, int S,
                            int A, double r_max, double eps, long long max_iter, double* Q, double* V, double* out_host,
                            void* work, void* stream);
/*
 * colo_extended_vi_batched_* -- the same solve for a SUBSET of a batch of models in ONE launch (one CTA per listed
 * instance, u1 / u2 / argsort in shared memory; S <= 8192): UCRL2's artificial episodes end at loop-dependent times
 * (agent/agents/infinite_horizon/ucrl2.py:173-192), so every round of a batch of loops re-plans the loops in `index`.
 * T f32[*,S,A,S], est_rewards f32[*,S,A], Q [*,S,A], V [*,S] are addressed by instance index[k] (index NULL: k);
 * beta_r, beta_p f64[m,S,A] and the outputs span f64[m], iters i64[m], status i32[m] (COLO_OK / COLO_MAX_ITER) are
 * compact, all on the device.  Same operations in the same order as colo_extended_vi_* (bit-identical Q, V, span).
 * Does not synchronise.
 */
int colo_extended_vi_batched_f32(const float* T, const float* est_rewards, const double* beta_r, const double* beta_p,
                                 const int* index, int m, int S, int A, double r_max, double eps, long long max_iter,
                                 float* Q, float* V, double* span, long long* iters, int* status, void* stream);
int colo_extended_vi_batched_f64acc(const float* T, const float* est_rewards, const double* beta_r, const double* beta_p,
                                    const int* index, int m, int S, int A, double r_max, double eps, long long max_iter,
                                    double* Q, double* V, double* span, long long* iters, int* status, void* stream);

/* ---------------------------------------------------------------- posterior sampling (PSRL) ---------------- */
/*
 * colo_sample_dirichlet_rows -- M_DIR._sample (colosseum/agent/mdp_models/bayesian_models/conjugate_transitions.py:
 * 48-60): T_out[r, :] = g / (1e-5 + sum(g)), g[j] ~ Gamma(hyper[r, j]) rounded to float32; rows = S*A for a whole
 * model.  Philox counter = ((row0 + r)*S + j, t): row0 is the global index of the first row (row sharding), t the
 * caller's draw counter.  Distributional parity with numpy's standard_gamma.  Does not synchronise.
 */
/*
 * colo_sample_nig_rewards -- N_NIG.sample (bayesian_models/conjugate_rewards.py:76-92): for each row (mu, lambda,
 * alpha, beta) f32[rows,4]: tau ~ Gamma(alpha, scale 1/beta) -> float32, R_out[r] ~ Normal(mu, sqrt(1/(lambda*tau)))
 * -> float32.  Philox counter (row0 + r, t).  Distributional parity.  Does not synchronise.
 */
int colo_sample_nig_rewards(const float* hyper, long long rows, long long row0, unsigned long long seed,
                            unsigned long long t, float* R_out, void* stream);
/* N_N.sample (conjugate_rewards.py:119-127) on the same [rows,4] layout: R_out[r] ~ Normal(mu, scale = tau) (sic: the
 * reference passes its precision-like second parameter as the scale) -> float32. */
int colo_sample_nn_rewards(const float* hyper, long long rows, long long row0, unsigned long long seed,
                           unsigned long long t, float* R_out, void* stream);
int colo_sample_dirichlet_rows(const float* hyper, long long rows, int S, long long row0, unsigned long long seed,
                               unsigned long long t, float* T_out, void* stream);
/* The same sample with single-precision arithmetic (SFU log / pow / cos, normal truncated at 5.8 sigma): another
 * stream of numbers with the same distribution up to ~1e-6, ~20x the throughput; used by the batched PSRL loops. */
int colo_sample_dirichlet_rows_fast(const float* hyper, long long rows, int S, long long row0, unsigned long long seed,
                               unsigned long long t, float* T_out, void* stream);

/* ---------------------------------------------------------------- policy-induced Markov chain -------------- */
/*
 * colo_policy_chain -- get_transition_probabilities / get_average_rewards (colosseum/mdp/utils/markov_chain.py:34-51):
 *   P_out[s,j] = min(1, sum_a T[s,a,j] pi[s,a]) f32 [S,S];  r_out[s] = sum_a R[s,a] pi[s,a] f32 [S] (or NULL).
 * colo_lazy_transpose -- M_out[j,s] = (P[s,j] + (s == j)) / 2: the matrix of the lazy chain, transposed so that the
 *   distribution update x <- M x is a row-times-vector product.
 * colo_power_iteration_f64 -- x <- M x / |M x|_1 from x0 until max|dx| < eps (fp64 accumulation; runs on the backup
 *   kernels: compressed rows on chip when M is sparse).  A building block for WELL-MIXING chains only: on nearly
 *   reducible chains the per-step change falls below any eps long before the limit is reached -- use
 *   colo_stationary_distribution_f64.  Synchronises.  Returns COLO_MAX_ITER after max_iter sweeps.
 *   work: colo_power_iteration_work_bytes(S).
 */
int colo_policy_chain(const float* T, const float* R, const float* pi, int S, int A, float* P_out, float* r_out,
                      void* stream);
/*
 * colo_average_rewards_f64 -- get_average_reward (colosseum/mdp/utils/markov_chain.py:12-31) for a BATCH of B policies on
 * one MDP: the continuous-MDP regret tick of N agent loops (experiment/agent_mdp_interaction.py:518-578) in a handful of
 * launches.  T f32[S,A,S], R f32[S,A] shared; pi f32[B,S,A].  Per policy: the chain P = min(1, sum_a T pi), its lazy
 * version (I + P)/2 squared repeatedly in fp64 (batched 64x64-tile GEMM; a chain freezes once a squaring moves it by
 * less than tol), and ar_out[b] = row 0 of the limit . r.  multichain_out[b] = 1 when the rows of the limit disagree
 * (several recurrent classes): the reference then weighs the classes by its first-reachable-class rule (:113-126), which
 * the caller resolves per policy (colo_stationary_distribution_f64 with the rule's start vector).  squarings_out i32[B]
 * (device, may be NULL).  Synchronises.  Returns COLO_MAX_ITER if a chain is still moving after max_squarings.
 * work: colo_average_rewards_work_bytes(B, S) device bytes.  B <= 65535.
 */
size_t colo_average_rewards_work_bytes(int B, int S);
int colo_average_rewards_f64(const float* T, const float* R, const float* pi, int B, int S, int A, double tol,
                             int max_squarings, double* ar_out, int* multichain_out, int* squarings_out, void* work,
                             void* stream);
/*
 * colo_stationary_distribution_f64 -- get_stationary_distribution (markov_chain.py:64-137): x_out = x0 * lim L^(2^k),
 * L = (I + P)/2, by repeated squaring in fp64 (rows rescaled to unit sum after every product) until max|L^(2^(k+1)) -
 * L^(2^k)| < tol or max_squarings products.  Exact limit of the start distribution x0 for every chain: with one
 * recurrent class THE stationary distribution; with several, their mixture by absorption probabilities (the reference
 * assigns each start state to the first class it can reach).  Synchronises.  work: colo_stationary_distribution_
 * work_bytes(S) (two S x S fp64 matrices).
 */
size_t colo_stationary_distribution_work_bytes(int S);
int colo_stationary_distribution_f64(const float* P, int S, const double* x0, double tol, int max_squarings,
                                     double* x_out, int* squarings_out_host, void* work, void* stream);
int colo_lazy_transpose(const float* P, int S, float* M_out, void* stream);
size_t colo_power_iteration_work_bytes(int S);
int colo_power_iteration_f64(const float* M, int S, const double* x0, double eps, long long max_iter, double* x,
                             long long* iters_out_host, void* work, void* stream);

/* ---------------------------------------------------------------- episodic tensor builders --------------- */
/*
 * colo_build_episodic_tensor -- get_episodic_transition_matrix_and_rewards (colosseum/mdp/utils/mdp_creation.py:98-128):
 *   T_epi[0, sn] = T[sn] and T_epi[H-1, :, :, sn] = p for every start state (sn, p); for 0 < h < H-1,
 *   T_epi[h, s] = T[s] iff s is reachable at step h (some T_epi[h-1, :, :, s] > 0); R_epi = tile(R, H), last layer 0.
 *   Outputs: T_epi f32[H,S,A,S], R_epi f32[H,S,A] (or NULL), reach u8[H,S] (1 = state reachable at step h; the set
 *   of (h,s) pairs of EpisodicMDP.reachable_states, base_finite.py:138-150).  H >= 2.  Does not synchronise.
 * colo_build_continuous_form -- get_continuous_form_episodic_transition_matrix_and_rewards (:131-176): the MDP over
 *   the n reachable (h,s) nodes, listed by the caller in node_h/node_s (any order; the reference's is its DFS
 *   order) with pos[h*S+s] = node index or -1: T_cf f32[n,A,n], R_cf f32[n,A].  Reference quirk kept: the rows of
 *   the last layer put the start probabilities in column start_idx[k] (the start state's ORIGINAL index, :168), not in
 *   the column of node (0, start_idx[k]).  *lost_mass_flag (device int) is set
 *   to 1 if a positive-probability successor is missing from the node list (the reference asserts row sums == 1).
 */
int colo_build_episodic_tensor(const float* T, const float* R, const int* start_idx, const double* start_prob, int n_start,
                          int H, int S, int A, float* T_epi, float* R_epi, unsigned char* reach, void* stream);
int colo_build_continuous_form(const float* T, const float* R, const int* node_h, const int* node_s, int n,
                               const int* pos, const int* start_idx, const double* start_prob, int n_start, int H,
                               int S, int A, float* T_cf, float* R_cf, int* lost_mass_flag, void* stream);

/* ---------------------------------------------------------------- (A) interaction step ------------------ */
/*
 * Tables of one MDP for the step kernels (built once per MDP by the host, colosseum_b200/tables.py).
 *
 * DENSE form (the north-star kernel; any dense T, CustomMDP, synthetic MDPs):
 *   cdf [S,A,ld]   sequential cumulative sum of T[s,a,:] over the next-state INDEX (fp64 running sum rounded
 *                  to the storage type), rows padded to ld (multiple of 32 elements) with the row total.
 *   Sampling restates CPython random.choices as used by NextStateSampler.sample
 *   (colosseum/mdp/utils/custom_samplers.py:49-72):  x = u*total;  next = first j with cdf[j] > x, clamped to
 *   the last positive-probability index (bisect_right(cum, x, 0, n-1)).
 * SUCCESSOR form (the seven benchmark families, <= ~13 successors per (s,a)):
 *   succ_cum f64 [S,A,Ksucc]  running sum of the sampler's probs IN ITS OWN ORDER (mdp_creation.py:276-310),
 *                             padded with +inf;  succ_idx i32 [S,A,Ksucc] next-state indices (padded with the
 *                             last real successor);  succ_len i32 [S,A].
 *   Bit-exact with the reference's sampler for the same fp64 uniform, including its successor order.
 *
 * Rewards (colosseum/mdp/base.py:1187-1207): reward class c = rew_cls[...] selects an inverse-CDF (quantile)
 * table rew_q[c, 0..nq-1] of the scipy frozen distribution on a uniform grid; a draw is the linear interpolation
 * at u_rew, then the reference's rescale  r*(rmax-rmin) - rmin  (sic).
 *   dense:      rew_cls_sas u8 [S,A,S] (or NULL) else rew_cls_sa i32 [S,A] (or NULL -> class 0)
 *   successor:  rew_cls_succ i32 [S,A,Ksucc]
 */
typedef struct {
  int S, A;
  int H;                 /* episode length; 0 = continuous (infinite horizon) */
  int ld;                /* dense row stride in elements */
  const void* cdf;       /* dense: float or double [S,A,ld] */
  const double* succ_cum;
  const int* succ_idx;
  const int* succ_len;
  int Ksucc;
  const unsigned char* rew_cls_sas;
  const int* rew_cls_sa;
  const int* rew_cls_succ;
  const float* rew_q;    /* [n_cls, nq] */
  int n_cls, nq;
  float rmin, rmax;      /* rewards_range */
  const double* start_cum; /* [n_start] running sum of the start distribution (sampler order) */
  const int* start_idx;    /* [n_start] */
  int n_start;
  /* optional two-level search index over rows of up to 1024 entries (ld % 128 == 0), built by colo_build_cdf_index:
   * cdf_mid [S,A,ld/4] = the last entry of every quad of the row, cdf_coarse [S,A,ld/32] = the last entry of every
   * 8th quad; same element type as cdf.  NULL: the step kernel samples those entries from the row itself.
   * rew_cls_pad u8 [S,A,ld] (optional, used with the index): rew_cls_sas with its rows padded to ld, so that the
   * classes of a 32-entry block's candidate next states are one aligned 32-byte read issued with the cdf_mid read. */
  const void* cdf_mid;
  const void* cdf_coarse;
  const unsigned char* rew_cls_pad;
  /* optional breakpoint table of an f32 cdf with short rows (ld % 128 == 0, ld <= 1024), built by colo_build_cdf_breaks:
   * [S,A,cdf_breaks_k] 16-byte entries {float v; int p; unsigned cls_flags; float r}, cdf_breaks_k in {2, 4, 8, 16}.
   * The breakpoints of row c[0..S) (c[-1] := 0) are the p with c[p] > c[p-1], in order, v = c[p]; entries past the
   * row's last breakpoint repeat it (a row without one holds {0, 0}).  cls_flags: bits 0-30 the reward class of
   * (s, a, p) (rew_cls_sas, else rew_cls_sa, else 0); bit 31 set when that class's quantile row is bitwise constant
   * and finite, r then being its reward.  Searching it returns exactly what searching the row returns; the dense f32
   * steps use it in place of the row and the index.  NULL: not used. */
  const void* cdf_breaks;
  int cdf_breaks_k;
} colo_mdp_tables;

/*
 * One batch of N parallel episodes (all device pointers): state i32[N], h i32[N], step_type u8[N] (the type of the
 * LAST emitted TimeStep; initialise to COLO_STEP_LAST so that stepping before reset is flagged), action i32[N]
 * (read, or -- with random_actions -- written with the uniformly random action taken, BaseMDP.random_step,
 * base.py:1341-1355), outputs reward f32[N] (NaN where the reference has None) and obs i32[N].
 * Visitation counters (u64, or NULL): `visits_copies` (a power of two >= 1) privatised copies laid out as
 * visits_s[copy][S] and visits_sa[copy][S*A]; a block adds to copy (blockIdx & (copies-1)) so that 65,536 envs
 * sitting on a handful of states do not serialise on a handful of L2 atomics -- the count is the sum over copies.
 * status: device int (may be NULL), set to COLO_NEEDS_RESET if an env needed a reset without auto_reset, to
 * COLO_BAD_ACTION if a supplied action was outside [0, A) (that env keeps its state: the reference raises there).
 * Zero-copy host I/O: `action` is only read and `reward` / `obs` are only written by the kernels, so each of them may
 * be a PINNED HOST buffer (cudaHostAlloc memory is mapped into the device's address space under unified addressing):
 * the kernel then pulls the actions and pushes the TimeStep fields over PCIe itself, lane-coalesced, and an
 * agent on the host needs no copy launches around the step.  step_type is also an INPUT of the next step and
 * therefore stays in device memory; `step_type_mirror` (may be NULL) is a second, write-only target for it.
 * Philox: when u_next / u_rew are NULL (or random_actions is set) the numbers come from Philox4x32-10 with
 * counter (env0 + i, t) and key seed -- env0 is the global index of the batch's first env, so a batch sharded
 * over GPUs draws exactly the numbers of the unsharded batch; t is the caller's step counter.
 */
typedef struct {
  long long N;
  unsigned long long seed, env0;
  int* state;
  int* h;
  unsigned char* step_type;
  int* action;
  float* reward;
  int* obs;
  unsigned long long* visits_s;
  unsigned long long* visits_sa;
  int visits_copies;
  int* status;
  unsigned char* step_type_mirror;
  float* discount; /* f32[N] or NULL: dm_env's discount of the emitted TimeStep (base.py:1316-1317): 1.0 MID,
                      0.0 LAST, NaN where the reference has None (FIRST) -- written by the step / reset epilogue */
  int io_compact;  /* != 0: compact host I/O -- `action` is read as u8[N] and `obs` written as i16[N] (-1 = the terminal
                      observation), 8 instead of 13 bytes per env-step over PCIe (reward f32, step_type u8 unchanged).
                      Needs S <= 32767, A <= 256 and the common call of the dense f32 step (supplied actions, in-kernel
                      uniforms, auto_reset, CDF index or breakpoint table present, counters on); COLO_ERR_ARG
                      otherwise. */
} colo_env_batch;

/*
 * colo_env_reset  -- BaseMDP.reset (base.py:1268-1277): h=0, state ~ start distribution, step_type=FIRST,
 *                    obs=state, visits_s[state]++.  u_next: double[N] or NULL (Philox).
 * colo_env_step_* -- BaseMDP.step (base.py:1279-1317).  Per env: if step_type==LAST: auto_reset ? reset path
 *                    (reward NaN for None, the action is ignored) : flag COLO_NEEDS_RESET; else h++, sample next,
 *                    visits_s[next]++, visits_sa[next,a]++ (sic: counted on the NEXT node), reward, and
 *                    LAST/obs=-1 if episodic and h>=H else MID/obs=next.
 *                    u_next: float[N] for _dense_f32, double[N] otherwise, or NULL; u_rew: float[N] or NULL.
 */
int colo_env_reset(const colo_mdp_tables* tb, const colo_env_batch* batch, const double* u_next,
                   unsigned long long t, void* stream);
int colo_env_step_dense_f32(const colo_mdp_tables* tb, const colo_env_batch* batch, int random_actions,
                            const float* u_next, const float* u_rew, unsigned long long t, int auto_reset,
                            void* stream);
int colo_env_step_dense_f64(const colo_mdp_tables* tb, const colo_env_batch* batch, int random_actions,
                            const double* u_next, const float* u_rew, unsigned long long t, int auto_reset,
                            void* stream);
/*
 * colo_env_random_steps -- BaseMDP.random_steps(n, auto_reset) (base.py:1319-1339) for every env in ONE launch: each
 * env is advanced n_steps times with uniformly random actions drawn from the Philox stream at counters t0, t0+1, ...
 * Bit-identical to n_steps calls of colo_env_step_* with random_actions = 1 and t = t0 .. t0+n_steps-1 (state, h,
 * step_type, visitation counters; reward / obs / action hold the LAST step's values).  mode: 0 dense f32 rows,
 * 1 dense f64 rows, 2 successor tables.  The caller advances its step counter by n_steps.
 */
int colo_env_random_steps(const colo_mdp_tables* tb, const colo_env_batch* batch, int mode, int n_steps,
                          unsigned long long t0, int auto_reset, void* stream);
/*
 * colo_emit_observations -- EmissionMap.get_observation (colosseum/emission_maps/base.py:110-140) for every env: the
 * row of the precomputed table all_observations (:56-76; f32 [H,S,D] episodic, [S,D] continuous with H = 0) at
 * (h[e], state[e]); zeros for an env whose last TimeStep was LAST (in_episode_time >= H, :131-132).  out f32 [N,D].
 */
int colo_emit_observations(const float* table, const int* state, const int* h, const unsigned char* step_type,
                           long long N, int H, int S, int D, float* out, void* stream);
/*
 * colo_emit_noise -- the noise EmissionMap.get_observation adds (emission_maps/base.py:136-138) on top of the rows
 * written by colo_emit_observations, in place; all-zero terminal observations stay zero (:131-132).  kind 1:
 * GaussianUncorrelated(scale = param) (colosseum/noises/gaussian_uncorrelated.py), period = D; kind 2:
 * StudentTUncorrelated(df = param) (noises/student_t_uncorrelated.py -- sic: one draw per slice along the first axis of
 * the observation, i.e. period = prod(shape[1:]), 1 for vector observations).  Element j of env e uses Philox counter
 * ((env0 + e) * period + j % period, t).  Distributional parity.  Correlated variants: colo_emit_noise_correlated.
 */
int colo_emit_noise(float* out, const unsigned char* step_type, const int* h, long long N, int H, int D, int period,
                    int kind, double param, unsigned long long seed, unsigned long long t, unsigned long long env0,
                    void* stream);
/*
 * colo_emit_noise_correlated -- the correlated noises (colosseum/noises/gaussian_correlated.py:9-17,
 * student_t_correlated.py:9-17) on top of colo_emit_observations' rows, in place: chol f32 [D,D] is the lower Cholesky
 * factor of the covariance W the reference draws once per emission map from Wishart(df = D, scale * I) (drawn by the
 * caller with the reference's own scipy call and RandomState(seed): the SAME W); kind 1: x ~ N(0, W); kind 2:
 * multivariate Student-t with shape W and `df` degrees of freedom (scipy's default df = 1).  Philox counter
 * ((env0 + e) * D + j, t) for the normals, (env0 + e, t) for the chi-square.  All-zero terminal observations stay zero.
 * Distributional parity.
 */
int colo_emit_noise_correlated(float* out, const unsigned char* step_type, const int* h, long long N, int H, int D,
                               const float* chol, int kind, double df, unsigned long long seed, unsigned long long t,
                               unsigned long long env0, void* stream);
int colo_env_step_succ(const colo_mdp_tables* tb, const colo_env_batch* batch, int random_actions,
                       const double* u_next, const float* u_rew, unsigned long long t, int auto_reset,
                       void* stream);

/*
 * Mixed batches -- one batch whose envs belong to different MDP instances (e.g. a benchmark's parameter sets x seeds),
 * advanced by ONE launch per reset / step / fused random steps whatever the number of instances.
 *   Layout: instance i owns the contiguous envs [start_i, start_i + n_envs[i]), in instance order; N = sum n_envs[i].
 *   Semantics: per env, those of colo_env_reset / colo_env_step_* / colo_env_random_steps on the env's OWN instance
 *   (start distribution, sampler, reward classes and quantiles, rewards_range, H -- episodic and continuous instances
 *   may share a batch --, auto-reset, obs = state index within the instance, random actions in [0, A_i)).
 *   Philox: env e of instance i uses key seeds[i] and counter (e - start_i, t): segment i is bit-identical to a
 *   single-MDP batch of instance i with seed = seeds[i], env0 = 0, driven by the same calls.
 *   colo_env_batch is reused as is: N must equal sum n_envs[i] (COLO_ERR_ARG otherwise); its `seed` and `env0` are NOT
 *   used (the seeds live in the handle); io_compact must be 0.  Visitation counters: visits_s [copies][sum S] and
 *   visits_sa [copies][sum S*A], instance i's columns starting at sum_{j<i} S_j (sum_{j<i} S_j*A_j) --
 *   colo_mixed_visits_size gives one copy's length (pairs = 0: sum S, pairs != 0: sum S*A).
 *   An action outside [0, A_i) sets COLO_BAD_ACTION in `status` and leaves that env untouched.
 * colo_mixed_tables_create -- host_tables[n_inst]: each instance's tables (device pointers inside, as for the
 *   single-MDP calls; they must outlive the handle); n_envs[n_inst] >= 1; seeds[n_inst]; mode 0 dense f32 rows, 1 dense
 *   f64 rows (rows may have a different ld per instance), 2 successor tables (every instance needs the mode's tables).
 *   Validates every instance before touching the device (COLO_ERR_ARG, colo_last_error names the instance), then
 *   uploads the per-instance descriptors and an env -> instance map on `stream` and synchronises it.
 * colo_mixed_env_step -- u_next: float[N] for mode 0, double[N] otherwise, or NULL; u_rew float[N] or NULL.
 * Dense mixed batches use the general warp-per-env search (the short-row specialisations are single-MDP); host I/O,
 * the pipelines, the step server and emission maps are single-MDP only.
 */
typedef struct colo_mixed_tables colo_mixed_tables;
int colo_mixed_tables_create(const colo_mdp_tables* host_tables, int n_inst, const long long* n_envs,
                             const unsigned long long* seeds, int mode, void* stream, colo_mixed_tables** out);
void colo_mixed_tables_destroy(colo_mixed_tables* h);
long long colo_mixed_visits_size(const colo_mixed_tables* h, int pairs);
int colo_mixed_env_reset(const colo_mixed_tables* h, const colo_env_batch* batch, const double* u_next,
                         unsigned long long t, void* stream);
int colo_mixed_env_step(const colo_mixed_tables* h, const colo_env_batch* batch, int random_actions,
                        const void* u_next, const float* u_rew, unsigned long long t, int auto_reset, void* stream);
int colo_mixed_env_random_steps(const colo_mixed_tables* h, const colo_env_batch* batch, int n_steps,
                                unsigned long long t0, int auto_reset, void* stream);

/*
 * Prepared step -- the same launch as colo_env_step_* (auto_reset on, in-kernel Philox uniforms, supplied actions) with
 * everything but the action pointer and the step counter resolved once: a host loop that steps several env groups in
 * a pipeline pays for argument marshalling on every call (measured from Python: 6.4 us per colo_env_step_dense_f32
 * call, of which ~3 us are the launch).  mode: 0 dense f32 rows, 1 dense f64 rows, 2 successor tables.  The tables and
 * batch structs are copied; the buffers they point to must outlive the stepper.  Bit-identical to colo_env_step_*.
 */
typedef struct colo_env_stepper colo_env_stepper;
int colo_env_stepper_create(const colo_mdp_tables* tb, const colo_env_batch* batch, int mode, void* stream,
                            colo_env_stepper** out);
int colo_env_stepper_launch(colo_env_stepper* h, const int* action, unsigned long long t);
void colo_env_stepper_destroy(colo_env_stepper* h);
/*
 * colo_env_pipeline_run -- n_steps steps of every env of n_groups prepared steppers (host_io groups of one batch, each on
 * its own stream) as a software pipeline run by the library: prime every group, then per step and group: wait for the
 * group's stream (its TimeStep of the previous step is in the pinned buffers), call on_timestep(user, group, step) if
 * given -- the host agent reads the TimeStep and writes the next actions there -- and launch the next step reading
 * action_ring[(step % ring) * n_groups + group] (pinned int32 buffers).  The same recv/send order as the Python loop
 * over colo_env_stepper_launch + colo_stream_synchronize, without an interpreter between the calls (measured from
 * Python: ~9 us per group-step, which bounds a 25 us step).  Philox counters t0, t0 + 1, ...; bit-identical to
 * stepping the groups one call at a time.  Synchronises every group before it returns.
 */
typedef void (*colo_env_pipeline_callback)(void* user, int group, int step);
int colo_env_pipeline_run(colo_env_stepper* const* steppers, int n_groups, const int* const* action_ring, int ring,
                          unsigned long long t0, int n_steps, colo_env_pipeline_callback on_timestep, void* user);

/*
 * colo_env_pipeline_run_threads -- colo_env_pipeline_run with one host thread per group (the caller's thread runs group 0):
 * a group's cycle (launch latency, the kernel's PCIe reads and writes, completion latency, on_timestep) overlaps with
 * every other group's.  Same per-group order of events, same Philox counters, bit-identical TimeSteps; on_timestep is
 * called on the group's own thread, concurrently for different groups (a host agent with per-group state).
 */
int colo_env_pipeline_run_threads(colo_env_stepper* const* steppers, int n_groups, const int* const* action_ring, int ring,
                                  unsigned long long t0, int n_steps, colo_env_pipeline_callback on_timestep, void* user);

/*
 * Queued pipeline -- the same n_steps steps of every env of the groups as colo_env_pipeline_run (same recv / send order,
 * same Philox counters, bit-identical TimeSteps), without a stream synchronisation and a launch on the host per
 * group-step.  The handshake of a group-step is two 32-bit words in pinned host memory: on the group's (library-owned,
 * non-blocking) stream step i is   wait (go[g] == i % L + 1) -> step kernel -> write (done[g] = i % L + 1)   with the
 * wait and the write done by the GPU front end (stream memory operations, cuStreamWaitValue32 / cuStreamWriteValue32,
 * resolved at run time: no link dependency on libcuda), enqueued ahead of time.  The host loop per group-step is: spin
 * on done[g], on_timestep(user, group, step) -- the host agent reads the TimeStep and writes the next actions --, store
 * go[g].  use_graph != 0: the triples of L consecutive steps (L a multiple of `ring`, >= 64) are one instantiated CUDA
 * graph per group, replayed every L steps (the kernels then read the Philox counter as node index + a device word the
 * library rewrites in stream order before each replay); otherwise, and for the last n_steps % L steps, the triples
 * are enqueued one at a time, three group-steps ahead.  The action ring must hold pinned buffers (read over PCIe by
 * the kernels) and, with graphs, stay the same between calls for the graphs to be reused.  Fails with COLO_ERR_CUDA --
 * after feeding the queued waits so that no stream stays blocked -- if no step finishes for 10 s.
 * Reference path: BaseMDP.step (colosseum/mdp/base.py:1279-1317) driven by a host agent (MDPLoop,
 * colosseum/experiment/agent_mdp_interaction.py:236-298).
 */
typedef struct colo_env_pipeline colo_env_pipeline;
int colo_env_pipeline_create(colo_env_stepper* const* steppers, int n_groups, colo_env_pipeline** out);
int colo_env_pipeline_run_queued(colo_env_pipeline* p, const int* const* action_ring, int ring, unsigned long long t0,
                                 int n_steps, colo_env_pipeline_callback on_timestep, void* user, int use_graph);
void colo_env_pipeline_destroy(colo_env_pipeline* p);

/*
 * Step server -- BaseMDP.step (base.py:1279-1317) for an agent living on the host, without a launch and a stream
 * synchronisation per step.  colo_env_server_start launches the step kernel of `mode` (0 dense f32 rows, 1 dense f64
 * rows, 2 successor tables; auto_reset on, Philox uniforms) as a PERSISTENT kernel on `stream` (which must be a
 * non-blocking stream of its own).  batch->action / reward / obs / step_type_mirror are pinned host buffers, fixed
 * for the life of the server.  One step = the host writes the actions, colo_env_server_post() rings the doorbell,
 * the resident kernel reads the actions over PCIe, steps every env with Philox counter t + (step index - served - 1)
 * and writes the TimeStep fields into the pinned buffers, the last CTA publishes the step index in done_host, and
 * colo_env_server_wait() returns once it sees it (it spins on host memory; no CUDA call).  Bit-identical to the same
 * steps through colo_env_step_*.
 *   doorbell_host, done_host : one pinned u64 each (own cache lines);  ctl_dev : two device u64
 *   share          : the kernel takes at most 1/share of the CTAs the device can hold at once (servers running side
 *                    by side must not starve each other: their CTAs meet at a counter and must all be resident)
 *   idle_timeout_ms: the kernel retires by itself after this long without a doorbell (a forgotten server must not
 *                    hold the GPU); a wait that meets a retired server returns COLO_SERVER_LAPSED and the caller
 *                    restarts it with served = steps finished so far (the doorbell may already hold served + 1)
 * colo_env_server_stop retires the kernel and synchronises `stream`.  Nothing else may be enqueued on `stream` while
 * the server runs; a device-wide synchronisation blocks until it retires.
 */
typedef struct {
  unsigned long long* doorbell_host;
  unsigned long long* done_host;
  unsigned long long* ctl_dev;
  int share;
  unsigned idle_timeout_ms;
} colo_env_server;
int colo_env_server_start(const colo_mdp_tables* tb, const colo_env_batch* batch, const colo_env_server* srv, int mode,
                          unsigned long long t, unsigned long long served, void* stream);
unsigned long long colo_env_server_post(const colo_env_server* srv);
int colo_env_server_wait(const colo_env_server* srv, unsigned long long step_index, unsigned timeout_ms);
int colo_env_server_stop(const colo_env_server* srv, void* stream);

/*
 * The actor's exploration (QValuesActor, colosseum/agent/actors/Q_values_actor.py:20-82), shared by every agent-loop entry
 * point below as the LAST field of its argument struct.  The reference takes `epsilon_greedy` and `boltzmann_temperature`
 * as functions of the actor's interaction counter (its float forms are wrapped into a lambda that returns itself, :44-49,
 * and cannot be called); here a CONSTANT goes into the struct's `epsilon_greedy` / `boltzmann_temperature`, a FUNCTION is
 * tabulated by the caller for the interaction counts a launch covers: schedule[k] = f(t0 + k), k < len (device f64; the
 * counter of a step is the loop's time t, 1 at its first action).
 * Order as in select_action (:58-82): with probability epsilon a uniformly random action; else, boltzmann != 0: an action
 * drawn from softmax(temperature * q) -- exp in float32, p = e / e.sum() in float32, then numpy's choice: the first index
 * whose normalised float64 running sum exceeds a uniform (draw keyed seed ^ 0x94D049BB133111EB); else greedy with uniform
 * tie-breaking.  All zero / NULL = the constant-epsilon greedy actor.
 */
typedef struct {
  const double* epsilon_schedule;
  const double* temperature_schedule;
  long long t0;
  int len;
  int boltzmann;
  double boltzmann_temperature;
} colo_actor_args;

/*
 * Batched agent/MDP interaction loops (SURVEY.md section 8(f)-4): N independent (Q-learning agent, env) pairs on one
 * MDP, one thread per loop, n_steps iterations of MDPLoop.run's body (experiment/agent_mdp_interaction.py:238-298)
 * per launch: QValuesActor.select_action (agent/actors/Q_values_actor.py:58-82; epsilon-greedy or uniform among the
 * argmax ties), BaseMDP.step on the successor tables, the model update, cumulative reward, reset after LAST.
 *   colo_qlearning_episodic_steps   QValuesModel.step_update (agent/agents/episodic/q_learning.py:53-103):
 *       cnt i32[N,H,S,A] (init 1), Q f32[N,H,S,A] (init H), V f32[N,H+1,S] (init 0);
 *       ucb_type 0 = Hoeffding bonus c_1*sqrt(H^3*log_term/n); 1 = Bernstein (mu, sigma, beta f32[N,H,S,A], init 0)
 *       log_term = log(S*A*optimization_horizon/p), sqrt_h7sa = sqrt(H^7*S*A)
 *   colo_qlearning_continuous_steps _QValuesModel.step_update (agent/agents/infinite_horizon/q_learning.py:86-111):
 *       cnt i32[N,S,A] (init 0), Q, Q_main f32[N,S,A] (init H_eff), V f32[N,S] (init H_eff);
 *       log_term = log(2*optimization_horizon/confidence), gamma = 1 - 1/H_eff
 * Randomness: env draws from Philox4x32-10 keyed (seed; env0+i, t) exactly as colo_env_step_succ, the agent's from
 * (seed ^ 0x9E3779B97F4A7C15; env0+i, t): word 0 epsilon test, word 1 random action / tie break, words 2-3 the
 * start-state draw of the reset after LAST.  t runs t0 .. t0+n_steps-1; the caller advances its counter.
 * trace (optional) i32[n_steps,N,4] = (s_t, a_t, observation of ts_tp1 (-1 at LAST), reward bits) per step.
 * Does not synchronise.
 */
typedef struct {
  long long N;
  unsigned long long seed, env0;
  int* state;
  int* h;
  int* cnt;
  float* Q;
  float* Q_main;
  float* V;
  float* mu;
  float* sigma;
  float* beta;
  int ucb_type;
  double c_1, c_2, min_at, log_term, sqrt_h7sa;
  double H_eff, gamma, span_approx;
  double epsilon_greedy; /* < 0: greedy */
  double* cum_reward;    /* f64[N], accumulated across calls */
  long long* n_episodes; /* i64[N] or NULL */
  int* trace;
  colo_actor_args actor;
} colo_qlearning_args;
int colo_qlearning_episodic_steps(const colo_mdp_tables* tb, const colo_qlearning_args* a, int n_steps,
                                  unsigned long long t0, void* stream);
int colo_qlearning_continuous_steps(const colo_mdp_tables* tb, const colo_qlearning_args* a, int n_steps,
                                    unsigned long long t0, void* stream);

/*
 * colo_psrl_episodic_steps -- PSRLEpisodic between two posterior samples (agent/agents/episodic/posterior_sampling.py:
 * 142-147) for N independent loops: greedy / epsilon-greedy action on Q f32[N,H+1,S,A] (the episodic value iteration of
 * each loop's sampled model), BaseMDP.step, BayesianMDPModel.step_update (agent/mdp_models/bayesian_model.py:78-92):
 * N_NIG.update_sa with the one reward on nig_hyper f32[N,S,A,4] = (mu, lambda, alpha, beta)
 * (bayesian_models/conjugate_rewards.py:56-74) and, unless the step ended the episode, dir_hyper[N,S,A,S][s,a,s'] += 1
 * (conjugate_transitions.py:43-45).  Randomness, trace and counters as colo_qlearning_*.  The caller resamples the
 * models (colo_sample_dirichlet_rows, colo_sample_nig_rewards) and re-solves (colo_episodic_f32, B = N) every H steps.
 */
typedef struct {
  long long N;
  unsigned long long seed, env0;
  int* state;
  int* h;
  const float* Q;
  float* dir_hyper;
  float* nig_hyper;
  double epsilon_greedy;
  double* cum_reward;
  long long* n_episodes;
  int* trace;
  int reward_model; /* 0 = N_NIG (mu, lambda, alpha, beta); 1 = N_N (mu, tau, -, -): N_N.update_sa, conjugate_rewards.py:112-117 */
  colo_actor_args actor;
} colo_psrl_args;
int colo_psrl_episodic_steps(const colo_mdp_tables* tb, const colo_psrl_args* a, int n_steps, unsigned long long t0,
                             void* stream);

/*
 * UCRL2Continuous (colosseum/agent/agents/infinite_horizon/ucrl2.py:34-357) for N independent loops on one continuous
 * MDP.  The batch advances in rounds because artificial episodes end at loop-dependent times:
 *   colo_ucrl2_steps        every loop that is not waiting runs MDPLoop.run's body (select_action on Q f32[N,S,A],
 *                           BaseMDP.step, step_update :183-199, is_episode_end :173-181) until its own time t[i] reaches
 *                           t_target or its artificial episode ends (ended[i] = 1; 2 = the episode log overflowed);
 *   colo_ucrl2_bounds       for the loops listed in index[m] (device): episode += 1, delta = 1/sqrt(iteration+1) and the
 *                           confidence bounds of solve_optimistic_model (:223-311) into beta_r, beta_p f64[m,S,A]
 *                           (rewards: _chernoff; transitions: _chernoff or, bernstein_p != 0, bernstein; beta_p is the
 *                           [s,a,0] entry of the reference's array, the one _max_proba reads);
 *   colo_extended_vi_batched_f32 on (P, est_r, beta_r, beta_p) -> Q, V of the listed loops;
 *   colo_ucrl2_model_update model_update (:201-221) from the episode log, iteration += episode length, log / nu / ended
 *                           cleared.
 * Tables (device, per loop contiguous): Nsas i32[N,S,A,S] (init 0), Nsa i32[N,S,A] = Nsas.sum(-1), P f32[N,S,A,S]
 * (init 1/S), est_r f32[N,S,A] (init r_max), var_r, hold f32[N,S,A] (init 0 / 1), nu i32[N,S,A] = visits inside the
 * running episode, seen i32[N,S,A] scratch (all zero between calls), ep_log i32[N,log_cap,2] = (s*A+a, reward bits) in
 * time order, ep_len i32[N], iteration / episode i64[N], delta f64[N], t i64[N], state i32[N], cum_reward f64[N].
 * Randomness as colo_qlearning_*: env draws keyed (seed; env0+i, t[i]), agent draws (seed ^ 0x9E3779B97F4A7C15; ...).
 * trace (optional) i32[trace_steps,N,4] = (s_t, a_t, s_tp1, reward bits) at row t - trace_t0.  None synchronises.
 */
typedef struct {
  long long N;
  unsigned long long seed, env0;
  int* state;
  long long* t;
  double* cum_reward;
  const float* Q;
  int* Nsas;
  int* Nsa;
  float* P;
  float* est_r;
  float* var_r;
  float* hold;
  int* nu;
  int* seen;
  int* ep_len;
  int* ep_log;
  int log_cap;
  int* ended;
  long long* iteration;
  long long* episode;
  double* delta;
  double epsilon_greedy; /* < 0: greedy */
  int* trace;
  long long trace_t0;
  int trace_steps;
  colo_actor_args actor;
} colo_ucrl2_args;
int colo_ucrl2_steps(const colo_mdp_tables* tb, const colo_ucrl2_args* a, long long t_target, void* stream);
int colo_ucrl2_bounds(const colo_ucrl2_args* a, int S, int A, const int* index, int m, double alpha_r, double alpha_p,
                      double r_max, int bernstein_p, double* beta_r, double* beta_p, void* stream);
int colo_ucrl2_model_update(const colo_ucrl2_args* a, int S, int A, const int* index, int m, void* stream);

/*
 * PSRLContinuous (colosseum/agent/agents/infinite_horizon/posterior_sampling.py:117-452; Agrawal & Jia 2017) for N
 * independent loops on one continuous MDP, in the same rounds as UCRL2Continuous:
 *   colo_psrlc_steps          select_action on the extended q-values Q f32[N,S,A*psi] (real action = extended / psi,
 *                             :449-452), BaseMDP.step, step_update (:394-412: BayesianMDPModel.step_update on nig_hyper
 *                             f32[N,S,A,4] / dir_hyper f32[N,S,A,S], N[s,a,s'] += 1), is_episode_end (:333-345:
 *                             N_tau >= 2 (N_tau - nu_k)) until t[i] reaches t_target or the artificial episode ends;
 *   colo_psrlc_sample_models  for the loops in index[m]: optimistic_sampling (:414-447) into T_ext f32[m,S,A*psi,S]
 *                             (rows with N[s,a].sum() >= eta: psi Dirichlet posterior samples; the others: the
 *                             "simple sampling" rows P_minus + the missing mass on one random state per sample) and the
 *                             reward sample tiled psi times into R_ext f32[m,S,A*psi] (:368-372; truncate != 0:
 *                             maximum(r_max, R) first).  fast != 0: single-precision gamma draws.  The caller solves
 *                             (T_ext, R_ext) with colo_solve_discounted_* (B = m) and writes the q-values back;
 *   colo_psrlc_finish_episode the episode's visit counts nu are dropped, ended cleared, episode += 1.
 * psi = 1 and eta = 0 give no_optimistic_sampling (T = sample_T()).  Tables per loop contiguous; Nsas i32[N,S,A,S],
 * Nsa i32[N,S,A], nu i32[N,S,A], t / episode i64[N], ended i32[N].  Randomness and trace as colo_ucrl2_* (trace column
 * 1 is the EXTENDED action).  None synchronises.
 */
typedef struct {
  long long N;
  unsigned long long seed, env0;
  int* state;
  long long* t;
  double* cum_reward;
  const float* Q;
  int psi;
  float* dir_hyper;
  float* nig_hyper;
  int reward_model; /* 0 = N_NIG, 1 = N_N */
  int* Nsas;
  int* Nsa;
  int* nu;
  int* ended;
  long long* episode;
  double epsilon_greedy; /* < 0: greedy */
  int* trace;
  long long trace_t0;
  int trace_steps;
  colo_actor_args actor;
} colo_psrlc_args;
int colo_psrlc_steps(const colo_mdp_tables* tb, const colo_psrlc_args* a, long long t_target, void* stream);
int colo_psrlc_sample_models(const colo_psrlc_args* a, int S, int A, const int* index, int m, double eta, int truncate,
                             float r_max, int fast, float* T_ext, float* R_ext, void* stream);
int colo_psrlc_finish_episode(const colo_psrlc_args* a, int S, int A, const int* index, int m, void* stream);

/* Dense CDF builder on device: cdf[s,a,0..ld) from T[s,a,0..S) (sequential fp64 running sum per row, one thread
 * per row -- the DEFINED summation order the oracle shares).  out_is_f64: 0 float, 1 double. */
int colo_build_dense_cdf(const float* T, int S, int A, int ld, void* cdf, int out_is_f64, void* stream);
/* The search index of colo_mdp_tables (cdf_mid [S,A,ld/4], cdf_coarse [S,A,ld/32]) from a dense cdf with ld % 128 == 0:
 * plain copies of entries of the row, so searching through the index returns exactly what searching the row returns. */
int colo_build_cdf_index(const void* cdf, int S, int A, int ld, int is_f64, void* cdf_mid, void* cdf_coarse,
                         void* stream);
/* The largest number of breakpoints (entries c[j] > c[j-1], c[-1] := 0) over the rows of an f32 cdf [S,A,ld], into
 * *max_breaks (host).  A row that decreases somewhere or holds a NaN counts as S + 1.  Synchronises `stream`. */
int colo_count_cdf_breaks(const float* cdf, int S, int A, int ld, int* max_breaks, void* stream);
/* The breakpoint table of colo_mdp_tables (cdf_breaks [S,A,k], see there) from tb->cdf (f32) and tb's reward classes
 * and quantiles; k in {2, 4, 8, 16} must be at least colo_count_cdf_breaks of the cdf (rows with more are refused
 * with COLO_ERR_ARG after the build, the table then being unusable).  Synchronises `stream`. */
int colo_build_cdf_breaks(const colo_mdp_tables* tb, int k, void* cdf_breaks, void* stream);

/* ---------------------------------------------------------------- multi-GPU ---------------------------- */
/*
 * Row-sharded value iteration of ONE large MDP (SURVEY.md section 8e-3) uses colo_backup_* with row0/nrows set to
 * the rank's row range, T/R/pi/Q pointing at the local shard, V_in the full [S] vector and V_out_peers listing
 * every rank's next-V buffer (peer-mapped through torch symmetric memory / CUDA IPC).  Independent MDP instances
 * and parallel envs shard with no communication at all.
 *
 * colo_synth_dense_rows fills T_rows[nrows,A,S] / R_rows[nrows,A] with the synthetic dense MDP of config C5
 * directly on the device (51 GB is never materialised on the host): weights u^8 + 1e-12 from Philox4x32-10 keyed
 * by (seed; global row index*A+a, column/4), each row normalised in fp32; R ~ U[0,1).  Deterministic in
 * (seed, global row), hence independent of the sharding.
 */
int colo_synth_dense_rows(float* T_rows, float* R_rows, int row0, int nrows, int S, int A, unsigned long long seed,
                          void* stream);

/* ---------------------------------------------------------------- benchmark-suite work items (C3) ------------ */
/*
 * colo_suite_run -- BASELINE.json configs[2]: for every MDP instance, cfg->n_envs parallel episodes x cfg->n_steps
 * random-agent steps (BaseMDP.random_steps with auto_reset, mdp/base.py:1319-1355; successor-table sampler, Philox
 * seed cfg->seed, reset at t = 0, steps at t = 1..), then the hardness measures with the reference's property layer's
 * choices (mdp/base.py:996-1114): continuous MDPs -- discounted VI on T, R (gamma = float32(0.99)), gaps, value norm
 * (0 when deterministic), diameter over all S targets; episodic ones -- backward induction + the reachable (h, s)
 * pairs for the gaps, the episodic tensor for the diameter, the continuous form for the value norm (skipped, NaN,
 * when 4 n^2 A > cfg->max_cf_bytes).  f64acc arithmetic, every iteration to cfg->eps.  Each step is the public entry
 * point of this header that colosseum_b200/suite.py calls from Python; what this call adds is the scheduling:
 * n_workers host threads, one CUDA stream each, pull instances from a shared counter, so that many small latency-bound
 * solves are in flight at once without an interpreter in between.  ALL pointers of colo_suite_instance are HOST
 * pointers (numpy arrays of the caller); out[i] receives instance i's results.  Runs on the current device.
 * Synchronises.  Returns the first non-zero status (out[i].status / out[i].error say which instance and why).
 * The workers spin in their stream synchronisations when the process may run on at least n_workers cores
 * (sched_getaffinity) and block otherwise (environment: COLO_SUITE_SPIN / COLO_SUITE_BLOCK force either;
 * COLO_SUITE_VERBOSE prints the wall time of every phase of every instance on stderr); they keep their large device
 * buffers between instances and calls (colo_suite_release_caches), and one call runs at a time per process.
 */
typedef struct {
  int S, A, H, K;                /* H = 0: continuous; K = successor slots per (s, a) */
  const float* T;                /* f32 [S,A,S] */
  const float* R;                /* f32 [S,A], the reference's mdp.R */
  const double* succ_cum;        /* f64 [S,A,K] running sums in sampler order, +inf padded */
  const int* succ_idx;           /* i32 [S,A,K] */
  const int* succ_len;           /* i32 [S,A] */
  const int* rew_cls_succ;       /* i32 [S,A,K] */
  const float* rew_q;            /* f32 [n_cls, nq] */
  int n_cls, nq;
  float rmin, rmax;
  const int* start_idx;          /* i32 [n_start] */
  const double* start_cum;       /* f64 [n_start] */
  const double* start_prob;      /* f64 [n_start] */
  int n_start;
  const int* node_h;             /* episodic: the reachable (h, s) pairs in the reference's node order */
  const int* node_s;
  int n_nodes;
  int deterministic;             /* all transitions and rewards deterministic: value norm = 0 (base.py:1069-1074) */
} colo_suite_instance;
typedef struct {
  long long n_envs;
  int n_steps;
  unsigned long long seed;
  double eps;                    /* stopping tolerance of every iteration (1e-9: the fixed point in fp64) */
  size_t max_cf_bytes;
  int diameter;                  /* 0: skip the diameter */
} colo_suite_config;
typedef struct {
  int status;
  double visits_total, mean_reward_last_step;
  double gaps, value_norm, diameter, diameter_sweeps;
  double step_s, hardness_s;     /* wall-clock seconds of the two phases of this instance (its worker thread) */
  char error[160];
} colo_suite_result;
int colo_suite_run(const colo_suite_instance* inst, int n, const colo_suite_config* cfg, colo_suite_result* out,
                   int n_workers);
/*
 * colo_suite_release_caches -- colo_suite_run's workers keep their large device buffers (episodic tensor, continuous form,
 * diameter work space) from one instance and one call to the next; this frees them (to the stream-ordered pool).
 */
int colo_suite_release_caches(void);

#ifdef __cplusplus
}
#endif
#endif /* COLOSSEUM_B200_H_ */
