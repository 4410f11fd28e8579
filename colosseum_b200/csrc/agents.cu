// agents.cu -- N independent agent/MDP interaction loops on the device (SURVEY.md section 8(f)-4: "a batched MDPLoop
// that drives N envs with vectorised tabular agents").
//
// One thread owns one loop: its env (state, h), its agent model (count / Q / V tables) and its Philox streams, and
// runs n_steps iterations of MDPLoop.run's body (colosseum/experiment/agent_mdp_interaction.py:238-298) in ONE
// launch:  a = actor.select_action(ts, h);  new_ts = mdp.step(a);  agent.step_update(ts, a, new_ts, h);
//          cumulative_reward += r;  if new_ts.last(): ts = mdp.reset().
//   actor   QValuesActor.select_action (colosseum/agent/actors/Q_values_actor.py:58-82): epsilon-greedy, else uniform
//           among the argmax ties of q[time, s].  (Boltzmann exploration is not offered.)
//   model   episodic  QValuesModel.step_update  (colosseum/agent/agents/episodic/q_learning.py:53-103), UCB-Hoeffding
//                     and UCB-Bernstein bonuses, including numpy's type promotion in each sub-expression
//           continuous _QValuesModel.step_update (colosseum/agent/agents/infinite_horizon/q_learning.py:86-111)
//   env     BaseMDP.step / reset as in env_step.cu (successor tables == the reference's own sampler)
// Every floating-point operation is written with round-to-nearest intrinsics (no FMA contraction): the CPU oracle
// computes the same IEEE operations in the same order, so whole trajectories are compared bit for bit.
//
// Memory: the tables of a loop are contiguous ([N][H,S,A]); accesses are 4-byte gathers at (h, s, a) -- latency
// bound, hidden by running one thread per loop with as many loops as the caller has seeds.
#include <cmath>
#include <vector>

#include "agent_device.cuh"
#include "mixed.cuh"

namespace colo {

// Loop i of a batch: it is loop j of the region of the flat tables that starts base_q (Q-shaped tables) / base_v (V)
// elements in; it draws with Philox key `seed` (agent: seed ^ kAgentKey) and counter (ctr, t), and its MDP's constants
// are `c`.  The flat per-loop arrays of p (state, h, cum_reward, n_episodes, trace) are indexed by i.
template <bool EPISODIC>
__device__ __forceinline__ void qlearning_loop(const colo_mdp_tables& tb, const colo_qlearning_args& p,
                                               const colo_qlearning_inst& c, size_t base_q, size_t base_v, long long j,
                                               unsigned long long seed, unsigned long long ctr, long long i,
                                               int n_steps, unsigned long long t0) {
  const int S = tb.S, A = tb.A, H = tb.H;
  const size_t per_q = (size_t)(EPISODIC ? H : 1) * S * A, per_v = (size_t)(EPISODIC ? H + 1 : 1) * S;
  const size_t off_q = base_q + j * per_q, off_v = base_v + j * per_v;
  int* cnt = p.cnt + off_q;
  float* Q = p.Q + off_q;
  float* V = p.V + off_v;
  float* Qm = EPISODIC ? nullptr : p.Q_main + off_q;
  float* mu = p.mu ? p.mu + off_q : nullptr;
  float* sg = p.sigma ? p.sigma + off_q : nullptr;
  float* be = p.beta ? p.beta + off_q : nullptr;
  int s = p.state[i], h = p.h[i];
  double cum = p.cum_reward[i];
  long long episodes = p.n_episodes ? p.n_episodes[i] : 0;
  const double Hd = EPISODIC ? (double)H : c.H_eff;
  const double H3 = (double)H * H * H;  // exact: H**3 is a python int in the reference

  for (int step = 0; step < n_steps; ++step) {
    const unsigned long long t = t0 + step;
    const Philox4 we = philox4x32_10(seed, ctr, t);
    const Philox4 wa = philox4x32_10(seed ^ kAgentKey, ctr, t);
    const size_t row = ((size_t)(EPISODIC ? h : 0) * S + s) * A;
    const int a = actor_select(Q + row, A, A, p.epsilon_greedy, p.actor, (long long)t, wa, seed, ctr);
    const size_t idx = row + a;
    // every table entry the update needs is requested as soon as its address is known, and consumed only after the
    // sampler's own (dependent) table walk: the loop body is a chain of cold gathers, the fewer in series the better
    const int n0 = cnt[idx];
    const float q_old = Q[idx];
    float mu0 = 0.f, sg0 = 0.f, be0 = 0.f;
    if (EPISODIC && p.ucb_type != 0) {
      mu0 = mu[idx];
      sg0 = sg[idx];
      be0 = be[idx];
    }
    const Step st = env_succ(tb, s, a, u53(we.w[0], we.w[1]));
    const int hh = h + 1;
    const bool last = EPISODIC && hh >= H;
    const int obs = last ? -1 : st.nxt;
    const int sp = obs < 0 ? S - 1 : obs;  // numpy's negative index: the terminal observation -1 reads state S-1
    const float v_sp = V[EPISODIC ? (size_t)hh * S + sp : (size_t)sp];
    constexpr int kRowRegs = 8;
    float qsp[kRowRegs];
    const size_t rp = (size_t)sp * A;
    if (!EPISODIC && A <= kRowRegs) {
#pragma unroll
      for (int k = 0; k < kRowRegs; ++k) qsp[k] = k < A ? Q[rp + k] : -INFINITY;
    }
    const float r = reward_from_class(tb, st.cls, u24(we.w[2]));
    const int n = n0 + 1;
    cnt[idx] = n;
    // python's max(min_at, ratio) returns min_at -- a PYTHON float -- unless ratio > min_at; a python float is a weak
    // scalar under NEP 50: times a float32 table entry it is a float32 product, where the np.float64 ratio promotes
    const double ratio = __ddiv_rn(__dadd_rn(Hd, 1.0), __dadd_rn(Hd, (double)n));
    const bool py_alpha = !(ratio > p.min_at);
    const double alpha = py_alpha ? p.min_at : ratio;
    const double om = __dsub_rn(1.0, alpha);
    if (EPISODIC) {
      const float vnext = v_sp;
      double b = 0.0;
      float b32 = 0.f;
      bool b_is_f32 = false;
      if (p.ucb_type == 0) {
        b = __dmul_rn(p.c_1, __dsqrt_rn(__ddiv_rn(__dmul_rn(H3, c.log_term), (double)n)));
      } else {
        const float m = __fadd_rn(mu0, vnext);
        const float g = __fadd_rn(sg0, __fmul_rn(vnext, vnext));
        mu[idx] = m;
        sg[idx] = g;
        const float old_beta = be0;
        const float d = __fsub_rn(g, m);
        const float hd2 = __fmul_rn((float)H, __fmul_rn(d, d));
        const int n2 = (int)((unsigned)n * (unsigned)n);  // np.int32 ** 2 wraps
        const double x = __dadd_rn(__ddiv_rn((double)hd2, (double)n2), (double)H);
        const double first = __dsqrt_rn(__dmul_rn(x, c.log_term));
        const double second = __ddiv_rn(__dmul_rn(c.sqrt_h7sa, c.log_term), (double)n);
        const double v1 = __dmul_rn(p.c_1, __dadd_rn(first, second));
        const double v2 = __dmul_rn(p.c_2, __dsqrt_rn(__ddiv_rn(__dmul_rn(H3, c.log_term), (double)n)));
        const float nb = (float)(v2 < v1 ? v2 : v1);  // python min(v1, v2)
        be[idx] = nb;
        if (py_alpha) {  // every operand is float32 or a python scalar: the whole bonus is float32 arithmetic
          b32 = __fdiv_rn(__fdiv_rn(__fsub_rn(nb, __fmul_rn((float)om, old_beta)), 2.0f), (float)alpha);
          b_is_f32 = true;
        } else {
          b = __ddiv_rn(__ddiv_rn(__dsub_rn((double)nb, __dmul_rn(om, (double)old_beta)), 2.0), alpha);
        }
      }
      // python float + np.float32 is a float32 sum (NEP 50); the np.float64 bonus then promotes
      const float rv = __fadd_rn(r, vnext);
      // sic: the reference weighs the OLD estimate with alpha_t (q_learning.py:100-102)
      if (b_is_f32) {  // float32 bonus, python-float alpha: the update never leaves float32
        Q[idx] = __fadd_rn(__fmul_rn((float)alpha, q_old), __fmul_rn((float)om, __fadd_rn(rv, b32)));
      } else {
        const double target = __dadd_rn((double)rv, b);
        const double lhs = py_alpha ? (double)__fmul_rn((float)alpha, q_old) : __dmul_rn(alpha, (double)q_old);
        Q[idx] = (float)__dadd_rn(lhs, __dmul_rn(om, target));
      }
      float mx = Q[row];
      for (int k = 1; k < A; ++k) mx = fmaxf(mx, Q[row + k]);
      V[(size_t)h * S + s] = fminf((float)H, mx);
    } else {
      const double b = __dmul_rn(__dmul_rn(4.0, c.span_approx),
                                 __dsqrt_rn(__dmul_rn(__ddiv_rn(Hd, (double)n), c.log_term)));
      const double target = __dadd_rn(__dadd_rn((double)r, __dmul_rn(c.gamma, (double)v_sp)), b);
      const float qm = (float)__dadd_rn(__dmul_rn(om, (double)q_old), __dmul_rn(alpha, target));
      Qm[idx] = qm;
      const float q_new = fminf(q_old, qm);
      Q[idx] = q_new;
      float mx;
      if (A <= kRowRegs) {  // the row of the next state was fetched before the update: patch it if it is this row
        mx = -INFINITY;
#pragma unroll
        for (int k = 0; k < kRowRegs; ++k) mx = fmaxf(mx, (sp == s && k == a) ? q_new : qsp[k]);
      } else {
        mx = Q[rp];
        for (int k = 1; k < A; ++k) mx = fmaxf(mx, Q[rp + k]);
      }
      V[sp] = mx;
    }
    cum = __dadd_rn(cum, (double)r);
    if (p.trace) {
      int* tr = p.trace + ((size_t)step * p.N + i) * 4;
      tr[0] = s; tr[1] = a; tr[2] = obs; tr[3] = __float_as_int(r);
    }
    if (last) {
      ++episodes;
      h = 0;
      s = start_state(tb, u53(wa.w[2], wa.w[3]));
    } else {
      h = hh;
      s = st.nxt;
    }
  }
  p.state[i] = s;
  p.h[i] = h;
  p.cum_reward[i] = cum;
  if (p.n_episodes) p.n_episodes[i] = episodes;
}

template <bool EPISODIC>
__global__ void __launch_bounds__(128) qlearning_steps_kernel(const colo_mdp_tables tb, const colo_qlearning_args p,
                                                              int n_steps, unsigned long long t0) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.N) return;
  const colo_qlearning_inst c = {p.log_term, p.sqrt_h7sa, p.H_eff, p.gamma, p.span_approx};
  qlearning_loop<EPISODIC>(tb, p, c, 0, 0, i, p.seed, p.env0 + (uint64_t)i, i, n_steps, t0);
}

// a mixed agent batch's instance: its constants and where its region of the flat tables starts
struct MixedQInst {
  colo_qlearning_inst c;
  long long off_q, off_v;
};

// one loop per thread over the instances of a mixed batch: loop i is env i of the batch, on its instance's tables,
// keys and constants, with counter i - start (bit-identical to the instance's single-MDP batch)
template <bool EPISODIC>
__global__ void __launch_bounds__(128) qlearning_mixed_steps_kernel(const MixedInst* __restrict__ insts,
                                                                    const MixedQInst* __restrict__ qinsts,
                                                                    const int* __restrict__ inst_of,
                                                                    const colo_qlearning_args p, int n_steps,
                                                                    unsigned long long t0) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.N) return;
  const int k = __ldg(inst_of + i);
  const MixedInst& d = insts[k];
  const MixedQInst& q = qinsts[k];
  const long long j = i - d.start;
  qlearning_loop<EPISODIC>(d.tb, p, q.c, (size_t)q.off_q, (size_t)q.off_v, j, d.seed, (unsigned long long)j, i, n_steps,
                           t0);
}

// PSRLEpisodic between two posterior samples (colosseum/agent/agents/episodic/posterior_sampling.py:142-147): act
// greedily on the Q of the sampled model, BayesianMDPModel.step_update (agent/mdp_models/bayesian_model.py:78-92):
// N_NIG.update_sa with one reward (bayesian_models/conjugate_rewards.py:56-74) and, unless the step was the last of the
// episode, M_DIR.update_sa (conjugate_transitions.py:43-45).  Same numpy type promotion rules as above.
__global__ void __launch_bounds__(128) psrl_steps_kernel(const colo_mdp_tables tb, const colo_psrl_args p, int n_steps,
                                                         unsigned long long t0) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.N) return;
  const int S = tb.S, A = tb.A, H = tb.H;
  const float* Q = p.Q + (size_t)i * (H + 1) * S * A;
  float* dir = p.dir_hyper + (size_t)i * S * A * S;
  float* nig = p.nig_hyper + (size_t)i * S * A * 4;
  int s = p.state[i], h = p.h[i];
  double cum = p.cum_reward[i];
  long long episodes = p.n_episodes ? p.n_episodes[i] : 0;
  for (int step = 0; step < n_steps; ++step) {
    const unsigned long long t = t0 + step;
    const Philox4 we = philox4x32_10(p.seed, p.env0 + (uint64_t)i, t);
    const Philox4 wa = philox4x32_10(p.seed ^ kAgentKey, p.env0 + (uint64_t)i, t);
    const int a = actor_select(Q + ((size_t)h * S + s) * A, A, A, p.epsilon_greedy, p.actor, (long long)t, wa, p.seed,
                               p.env0 + (uint64_t)i);
    float* hp = nig + ((size_t)s * A + a) * 4;
    const float4 hp0 = *reinterpret_cast<const float4*>(hp);  // requested before the sampler's dependent table walk
    const Step st = env_succ(tb, s, a, u53(we.w[0], we.w[1]));
    const int hh = h + 1;
    const bool last = hh >= H;
    float* dc = dir + ((size_t)s * A + a) * S + st.nxt;
    const float d0 = last ? 0.f : *dc;
    const float r = reward_from_class(tb, st.cls, u24(we.w[2]));
    const float mu0 = hp0.x, l0 = hp0.y, a0 = hp0.z, b0 = hp0.w;
    if (p.reward_model == 1) {
      // N_N.update_sa: mu1 = (mu0*tau0 + r*1) / tau1, every operand float32 or a weak python scalar -> float32 ops
      const float t1 = __fadd_rn(l0, 1.0f);
      hp[0] = __fdiv_rn(__fadd_rn(__fmul_rn(mu0, l0), r), t1);
      hp[1] = t1;
    } else {
      const double y = (double)r;
      const float l1 = __fadd_rn(l0, 1.0f);
      const double mu1 = __ddiv_rn(__dadd_rn((double)__fmul_rn(l0, mu0), y), (double)l1);
      const double dy = __dsub_rn(y, (double)mu0);
      const double disc = __ddiv_rn(__dmul_rn((double)l0, __dmul_rn(dy, dy)), (double)l1);
      hp[0] = (float)mu1;
      hp[1] = l1;
      hp[2] = __fadd_rn(a0, 0.5f);
      hp[3] = (float)__dadd_rn((double)b0, __dmul_rn(0.5, __dadd_rn(0.0, disc)));
    }
    if (!last) *dc = __fadd_rn(d0, 1.0f);
    cum = __dadd_rn(cum, (double)r);
    if (p.trace) {
      int* tr = p.trace + ((size_t)step * p.N + i) * 4;
      tr[0] = s; tr[1] = a; tr[2] = last ? -1 : st.nxt; tr[3] = __float_as_int(r);
    }
    if (last) {
      ++episodes;
      h = 0;
      s = start_state(tb, u53(wa.w[2], wa.w[3]));
    } else {
      h = hh;
      s = st.nxt;
    }
  }
  p.state[i] = s;
  p.h[i] = h;
  p.cum_reward[i] = cum;
  if (p.n_episodes) p.n_episodes[i] = episodes;
}

// the buffers and shared hyper-parameters of a non-empty batch (single-MDP and mixed)
static int check_loop_args(const colo_qlearning_args* a, bool episodic) {
  COLO_ARG_CHECK(a->state && a->h && a->cnt && a->Q && a->V && a->cum_reward, "state, h, cnt, Q, V, cum_reward");
  if (episodic) {
    COLO_ARG_CHECK(a->ucb_type == 0 || (a->ucb_type == 1 && a->mu && a->sigma && a->beta && a->c_2 > 0),
                   "ucb_type 0 (hoeffding) or 1 (bernstein with mu, sigma, beta, c_2)");
    COLO_ARG_CHECK(a->c_1 > 0, "c_1 > 0");
  } else {
    COLO_ARG_CHECK(a->Q_main, "Q_main");
  }
  return COLO_OK;
}

static int check_args(const colo_mdp_tables* tb, const colo_qlearning_args* a, int n_steps, bool episodic) {
  COLO_ARG_CHECK(tb && a, "tables / args are NULL");
  COLO_ARG_CHECK(tb->S > 0 && tb->A > 0 && tb->rew_q && tb->n_cls > 0 && tb->nq >= 2, "tables");
  COLO_ARG_CHECK(tb->succ_cum && tb->succ_idx && tb->succ_len && tb->Ksucc > 0, "successor tables");
  COLO_ARG_CHECK(tb->start_cum && tb->start_idx && tb->n_start > 0, "start distribution");
  COLO_ARG_CHECK(episodic ? tb->H > 0 : tb->H == 0, "episodic agents need H > 0, continuous agents H == 0");
  COLO_ARG_CHECK(a->N >= 0 && n_steps >= 1, "N >= 0, n_steps >= 1");
  if (a->N == 0) return COLO_OK;
  const int r = check_loop_args(a, episodic);
  if (r != COLO_OK) return r;
  if (!episodic) COLO_ARG_CHECK(a->H_eff > 0, "Q_main, H_eff");
  return COLO_OK;
}

}  // namespace colo

extern "C" {

int colo_qlearning_episodic_steps(const colo_mdp_tables* tb, const colo_qlearning_args* a, int n_steps,
                                  unsigned long long t0, void* stream) {
  int r = colo::check_args(tb, a, n_steps, true);
  if (r != COLO_OK || a->N == 0) return r;
  const int grid = (int)((a->N + 127) / 128);
  colo::qlearning_steps_kernel<true><<<grid, 128, 0, (cudaStream_t)stream>>>(*tb, *a, n_steps, t0);
  return colo::check_launch("qlearning_steps_kernel<episodic>");
}

int colo_qlearning_continuous_steps(const colo_mdp_tables* tb, const colo_qlearning_args* a, int n_steps,
                                    unsigned long long t0, void* stream) {
  int r = colo::check_args(tb, a, n_steps, false);
  if (r != COLO_OK || a->N == 0) return r;
  const int grid = (int)((a->N + 127) / 128);
  colo::qlearning_steps_kernel<false><<<grid, 128, 0, (cudaStream_t)stream>>>(*tb, *a, n_steps, t0);
  return colo::check_launch("qlearning_steps_kernel<continuous>");
}

int colo_psrl_episodic_steps(const colo_mdp_tables* tb, const colo_psrl_args* a, int n_steps, unsigned long long t0,
                             void* stream) {
  COLO_ARG_CHECK(tb && a, "tables / args are NULL");
  COLO_ARG_CHECK(tb->S > 0 && tb->A > 0 && tb->H > 0 && tb->rew_q && tb->n_cls > 0 && tb->nq >= 2, "episodic tables");
  COLO_ARG_CHECK(tb->succ_cum && tb->succ_idx && tb->succ_len && tb->Ksucc > 0, "successor tables");
  COLO_ARG_CHECK(tb->start_cum && tb->start_idx && tb->n_start > 0, "start distribution");
  COLO_ARG_CHECK(a->N >= 0 && n_steps >= 1, "N >= 0, n_steps >= 1");
  if (a->N == 0) return COLO_OK;
  COLO_ARG_CHECK(a->state && a->h && a->Q && a->dir_hyper && a->nig_hyper && a->cum_reward,
                 "state, h, Q, dir_hyper, nig_hyper, cum_reward");
  COLO_ARG_CHECK((uintptr_t)a->nig_hyper % 16 == 0, "nig_hyper must be 16-byte aligned (rows are read as one float4)");
  const int grid = (int)((a->N + 127) / 128);
  colo::psrl_steps_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(*tb, *a, n_steps, t0);
  return colo::check_launch("psrl_steps_kernel");
}

// ---- mixed agent batches ------------------------------------------------------------------------------------------------
struct colo_mixed_qlearning {
  const colo_mixed_tables* tables;
  int episodic;
  long long q_elems, v_elems;
  colo::MixedQInst* insts;  // device [n_inst]
};

void colo_mixed_qlearning_destroy(colo_mixed_qlearning* q) {
  if (!q) return;
  if (q->insts) cudaFree(q->insts);
  free(q);
}

int colo_mixed_qlearning_create(const colo_mixed_tables* tables, int episodic, const colo_qlearning_inst* host_insts,
                                void* stream, colo_mixed_qlearning** out) {
  COLO_ARG_CHECK(out && tables && host_insts, "tables, host_insts, out");
  COLO_ARG_CHECK(episodic == 0 || episodic == 1, "episodic 0 or 1");
  COLO_ARG_CHECK(tables->mode == 2, "colo_mixed_qlearning_create: the mixed tables must be made in successor mode (2)");
  const int n_inst = tables->n_inst;
  std::vector<colo::MixedQInst> insts((size_t)n_inst);
  long long q_elems = 0, v_elems = 0;
  for (int k = 0; k < n_inst; ++k) {
    const colo::MixedInst& d = tables->host_insts[k];
    const colo_qlearning_inst& c = host_insts[k];
    const char* why = nullptr;
    if (episodic ? d.tb.H <= 0 : d.tb.H != 0)
      why = episodic ? "episodic agents need H > 0" : "continuous agents need H == 0";
    else if (!(std::isfinite(c.log_term) && std::isfinite(c.sqrt_h7sa) && std::isfinite(c.H_eff) &&
               std::isfinite(c.gamma) && std::isfinite(c.span_approx)))
      why = "non-finite constant";
    else if (!(c.sqrt_h7sa >= 0))
      why = "sqrt_h7sa < 0";
    else if (!episodic && !(c.H_eff > 0 && c.span_approx >= 0))
      why = "continuous agents need H_eff > 0 and span_approx >= 0";
    if (why) {
      colo::set_error("colo_mixed_qlearning_create: instance %d: %s", k, why);
      return COLO_ERR_ARG;
    }
    const long long n = (k + 1 < n_inst ? tables->host_insts[k + 1].start : tables->N) - d.start;
    const long long S = d.tb.S, A = d.tb.A, H = d.tb.H;
    insts[(size_t)k].c = c;
    insts[(size_t)k].off_q = q_elems;
    insts[(size_t)k].off_v = v_elems;
    q_elems += n * (episodic ? H : 1) * S * A;
    v_elems += n * (episodic ? H + 1 : 1) * S;
  }
  colo_mixed_qlearning* q = (colo_mixed_qlearning*)calloc(1, sizeof(colo_mixed_qlearning));
  COLO_ARG_CHECK(q != nullptr, "out of host memory");
  q->tables = tables;
  q->episodic = episodic;
  q->q_elems = q_elems;
  q->v_elems = v_elems;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMalloc((void**)&q->insts, sizeof(colo::MixedQInst) * (size_t)n_inst);
  if (e == cudaSuccess)
    e = cudaMemcpyAsync(q->insts, insts.data(), sizeof(colo::MixedQInst) * (size_t)n_inst, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);  // the host staging vector dies with this call
  if (e != cudaSuccess) {
    colo::set_error("colo_mixed_qlearning_create: %s", cudaGetErrorString(e));
    colo_mixed_qlearning_destroy(q);
    return COLO_ERR_CUDA;
  }
  *out = q;
  return COLO_OK;
}

int colo_mixed_qlearning_sizes(const colo_mixed_qlearning* q, long long* q_elems, long long* v_elems) {
  COLO_ARG_CHECK(q && q_elems && v_elems, "handle, q_elems, v_elems");
  *q_elems = q->q_elems;
  *v_elems = q->v_elems;
  return COLO_OK;
}

int colo_mixed_qlearning_steps(const colo_mixed_qlearning* q, const colo_qlearning_args* a, int n_steps,
                               unsigned long long t0, void* stream) {
  COLO_ARG_CHECK(q && a, "handle / args are NULL");
  COLO_ARG_CHECK(n_steps >= 1, "n_steps >= 1");
  if (a->N != q->tables->N) {
    colo::set_error("bad argument: args N = %lld, the mixed tables hold %lld loops", a->N, q->tables->N);
    return COLO_ERR_ARG;
  }
  const int r = colo::check_loop_args(a, q->episodic);
  if (r != COLO_OK) return r;
  const int grid = (int)((a->N + 127) / 128);
  const colo_mixed_tables* m = q->tables;
  if (q->episodic) {
    colo::qlearning_mixed_steps_kernel<true><<<grid, 128, 0, (cudaStream_t)stream>>>(m->insts, q->insts, m->inst_of,
                                                                                     *a, n_steps, t0);
    return colo::check_launch("qlearning_mixed_steps_kernel<episodic>");
  }
  colo::qlearning_mixed_steps_kernel<false><<<grid, 128, 0, (cudaStream_t)stream>>>(m->insts, q->insts, m->inst_of,
                                                                                    *a, n_steps, t0);
  return colo::check_launch("qlearning_mixed_steps_kernel<continuous>");
}

}  // extern "C"
