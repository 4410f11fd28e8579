// env_step.cu -- the batched agent/MDP interaction step (hot path A) for sm_100a.
//
// Restates BaseMDP.reset / BaseMDP.step (colosseum/mdp/base.py:1268-1317) for N independent episodes:
//   next state  : inverse-CDF sampling == NextStateSampler.sample == CPython random.choices
//                 (colosseum/mdp/utils/custom_samplers.py:49-72): bisect_right(cum, u*total, 0, n-1)
//   reward      : BaseMDP.sample_reward (base.py:1187-1207): a draw of the per-(s,a,s') distribution through its
//                 tabulated quantile function, then the reference's rescale r*(max-min) - min (sic)
//   bookkeeping : h, episodic termination (LAST, obs -1), auto-reset, visitation counts on the NEXT node (sic).
//
// Dense kernel: a warp owns a tile of 32 consecutive envs.  Env scalars are loaded / stored coalesced (lane i <->
// env i); the search over the dense CDF row T[s,a,:] is warp-cooperative: the row is read with 128-bit coalesced
// loads, all issued before any is consumed, and because the row is monotone the bisect position is simply the
// COUNT of entries <= x, i.e. one integer warp reduction, no branches and no early exit.
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <cuda.h>

#include <atomic>
#include <thread>
#include <vector>

#include "common.cuh"
#include "mixed.cuh"

namespace colo {

constexpr int kStepThreads = 64;  // small CTAs: 2048 warp-tiles at N=65,536 spread evenly over 148 SMs

// step launches per kernel variant (colo_step_kernel_launches), counted on the host where the variant is chosen, so a
// caller can tell which kernel served a call; a launch captured into a CUDA graph counts once, at capture
static std::atomic<unsigned long long> g_step_launches[COLO_STEP_KINDS];
static void count_step_launch(int kind) { g_step_launches[kind].fetch_add(1, std::memory_order_relaxed); }

struct StepIO {
  long long N;
  int* action;
  int random_actions;
  const void* u_next;
  const float* u_rew;
  unsigned long long seed, t, env0;
  int auto_reset;
  int* state;
  int* h;
  unsigned char* step_type;
  float* reward;
  int* obs;
  unsigned long long* visits_s;
  unsigned long long* visits_sa;
  int visits_mask;       // copies - 1
  long long n_s, n_sa;   // S, S*A: stride between privatised counter copies
  int* status;
  unsigned char* step_type_mirror;  // write-only second target of step_type (pinned host memory) or null
  float* discount;                  // dm_env discount of the emitted TimeStep (1 MID, 0 LAST, NaN FIRST) or null
  int n_steps;  // > 1: that many consecutive steps in ONE launch (random actions; Philox counter t, t+1, ...)
  int io_compact;  // action u8[N] in, obs i16[N] out (colo_env_batch.io_compact)
  // queued pipeline (colo_env_pipeline_run_queued): the launch is a node of a replayed CUDA graph, so the Philox step
  // counter cannot be a baked kernel argument: t = t + *t_dev (device word rewritten in stream order before each replay)
  const unsigned long long* t_dev;
  // persistent step server (colo_env_server_*; SERVER kernels only): the kernel stays resident and runs one pass per
  // doorbell value posted by the host instead of one pass per launch
  const unsigned long long* srv_doorbell;  // pinned host, written by the host: index of the newest requested step
  unsigned long long* srv_done;            // pinned host, written by the kernel: index of the newest finished step
  unsigned long long* srv_go;              // device: the doorbell as relayed by CTA 0
  unsigned long long* srv_arrive;          // device: CTA passes finished, monotonic
  unsigned long long srv_seq0;             // steps served before this launch
  unsigned long long srv_idle_ns;          // the server retires after this long without a doorbell
};

__device__ __forceinline__ unsigned long long step_t0(const StepIO& io) { return io.t_dev ? io.t + *io.t_dev : io.t; }

constexpr unsigned long long kSrvExit = ~0ULL, kSrvLapsed = ~0ULL - 1;
#ifndef COLO_SRV_POLL_NS
#define COLO_SRV_POLL_NS 400
#endif
constexpr unsigned kSrvPollNs = COLO_SRV_POLL_NS;  // back-off of the CTAs waiting for the relayed doorbell

__device__ __forceinline__ unsigned long long ld_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_sys_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_gpu_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

// Server side of the doorbell protocol.  CTA 0 alone polls the host word (one PCIe read per poll) and relays it
// through a device word the other CTAs poll in L2.  Returns false when the server has to retire (host asked, or no
// doorbell for srv_idle_ns: a forgotten server must not hold the GPU).
__device__ __forceinline__ bool server_wait(const StepIO& io, unsigned long long want) {
  __shared__ unsigned long long s_cmd;
  if (threadIdx.x == 0) {
    unsigned long long v;
    if (blockIdx.x == 0) {
      const unsigned long long t0 = global_ns();
      for (;;) {
        v = ld_sys_u64(io.srv_doorbell);
        if (v == want || v == kSrvExit) break;
        if (global_ns() - t0 > io.srv_idle_ns) {
          v = kSrvExit;
          st_sys_u64(io.srv_done, kSrvLapsed);
          break;
        }
      }
      __threadfence_system();  // the host wrote the actions before the doorbell: order our reads after it
      st_release_gpu_u64(io.srv_go, v);
    } else {
      for (;;) {
        v = ld_acquire_gpu_u64(io.srv_go);
        if (v == want || v == kSrvExit) break;
        __nanosleep(kSrvPollNs);
      }
    }
    s_cmd = v;
  }
  __syncthreads();
  const bool run = s_cmd != kSrvExit;
  __syncthreads();
  return run;
}

// every thread's host writes are fenced to system scope before its CTA arrives; the last CTA publishes the step
__device__ __forceinline__ void server_done(const StepIO& io, unsigned long long step_index) {
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned long long passes = step_index - io.srv_seq0;  // passes finished by every CTA once all arrive
    const unsigned long long prev = atomicAdd(io.srv_arrive, 1ULL);
    if (prev + 1 == passes * gridDim.x) {
      __threadfence_system();
      st_sys_u64(io.srv_done, step_index);
    }
  }
}

__device__ __forceinline__ float reward_draw(const colo_mdp_tables& tb, int cls, float u) {
  const float* q = tb.rew_q + (size_t)cls * tb.nq;
  const float t = u * (float)(tb.nq - 1);
  int i = (int)t;
  i = i > tb.nq - 2 ? tb.nq - 2 : i;
  const float f = t - (float)i;
  const float q0 = __ldg(q + i), q1 = __ldg(q + i + 1);
  const float r0 = fmaf(f, q1 - q0, q0);
  return fmaf(r0, tb.rmax - tb.rmin, -tb.rmin);
}

// bisect_right(cum, x, 0, n-1) == number of k in [0, n-2] with cum[k] <= x   (cum is non-decreasing)
__device__ __forceinline__ int bisect_count(const double* __restrict__ cum, int n, double x) {
  int pos = 0;
  for (int k = 0; k < n - 1; ++k) pos += (__ldg(cum + k) <= x) ? 1 : 0;
  return pos;
}

__device__ __forceinline__ int sample_start(const colo_mdp_tables& tb, double u) {
  if (tb.n_start == 1) return __ldg(tb.start_idx);
  const double total = __ldg(tb.start_cum + tb.n_start - 1) + 0.0;
  return __ldg(tb.start_idx + bisect_count(tb.start_cum, tb.n_start, u * total));
}

// warp-aggregated counter increment: lanes with equal keys elect one leader that adds the group size
__device__ __forceinline__ void aggregated_inc(unsigned long long* base, long long key, bool valid) {
  const unsigned act = __ballot_sync(FULL, valid);
  if (!valid) return;
  const unsigned peers = __match_any_sync(act, key);
  const int leader = __ffs(peers) - 1;
  if ((int)(threadIdx.x & 31) == leader) atomicAdd(base + key, (unsigned long long)__popc(peers));
}

template <typename TC>
struct Quad;
template <>
struct Quad<float> {
  float v[4];
  __device__ __forceinline__ void load(const float* p) {
    float4 t = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
};
template <>
struct Quad<double> {
  double v[4];
  __device__ __forceinline__ void load(const double* p) {
    double2 a = __ldg(reinterpret_cast<const double2*>(p));
    double2 b = __ldg(reinterpret_cast<const double2*>(p) + 1);
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
  }
};

// per-env prologue shared by all step kernels: resolves uniforms/actions, handles the reset path.
// returns true when the env takes a regular step.
struct EnvIn {
  int s, a, st, h, bad;
  double un64;
  float un32, ur;
};

// `seed` / `ctr`: the env's Philox key and counter -- (io.seed, io.env0 + e) in a single-MDP batch, (the instance's
// seed, e - the instance's first env) in a mixed batch
template <bool F32U>
__device__ __forceinline__ EnvIn load_env(const StepIO& io, const colo_mdp_tables& tb, long long e,
                                           unsigned long long t, unsigned long long seed, unsigned long long ctr) {
  EnvIn in;
  in.bad = 0;
  in.st = io.step_type[e];
  in.s = io.state[e];
  in.h = io.h[e];  // needed only by the epilogue: issued here so that its (cold) latency overlaps the search
  Philox4 w;
  const bool need_rng = io.u_next == nullptr || io.u_rew == nullptr || io.random_actions;
  if (need_rng) w = philox4x32_10(seed, ctr, t);
  if (io.u_next) {
    if (F32U) {
      in.un32 = reinterpret_cast<const float*>(io.u_next)[e];
      in.un64 = (double)in.un32;
    } else {
      in.un64 = reinterpret_cast<const double*>(io.u_next)[e];
      in.un32 = 0.f;
    }
  } else {
    in.un64 = u53(w.w[0], w.w[1]);
    in.un32 = u24(w.w[0]);
  }
  in.ur = io.u_rew ? io.u_rew[e] : u24(w.w[2]);
  in.a = io.random_actions ? act_from_word(w.w[3], tb.A) : (io.srv_go ? __ldcv(io.action + e) : io.action[e]);
  if ((unsigned)in.a >= (unsigned)tb.A) {  // the reference raises on an unknown action: flag it, touch no table
    if (io.status) *io.status = COLO_BAD_ACTION;
    in.a = 0;
    in.bad = 1;
  }
  return in;
}

template <bool F32U>
__device__ __forceinline__ EnvIn load_env(const StepIO& io, const colo_mdp_tables& tb, long long e,
                                           unsigned long long t) {
  return load_env<F32U>(io, tb, e, t, io.seed, io.env0 + (uint64_t)e);
}

// epilogue of a regular step for one env held by this thread.  off_s / off_sa: where the env's MDP starts in the
// counter rows (non-zero in a mixed batch, whose instances share one concatenated [copies][sum S] / [copies][sum S*A])
// have_rew: `rew` is the reward of the step (a constant class resolved by the breakpoint table), no draw needed
__device__ __forceinline__ void finish_env(const StepIO& io, const colo_mdp_tables& tb, long long e, const EnvIn& in,
                                           int nxt, int cls, bool stepping, bool resetting, long long off_s = 0,
                                           long long off_sa = 0, bool have_rew = false, float rew = 0.f) {
  if (resetting) {  // auto_reset path == BaseMDP.reset(): the action is ignored, reward is None (NaN here)
    nxt = sample_start(tb, in.un64);
    io.state[e] = nxt;
    io.h[e] = 0;
    io.step_type[e] = COLO_STEP_FIRST;
    if (io.step_type_mirror) io.step_type_mirror[e] = COLO_STEP_FIRST;
    io.reward[e] = __int_as_float(0x7fc00000);
    if (io.discount) io.discount[e] = __int_as_float(0x7fc00000);
    io.obs[e] = nxt;
  } else if (stepping) {
    const int hh = in.h + 1;
    io.h[e] = hh;
    io.state[e] = nxt;
    io.reward[e] = have_rew ? rew : reward_draw(tb, cls, in.ur);
    if (io.random_actions) io.action[e] = in.a;
    const bool last = tb.H > 0 && hh >= tb.H;
    const unsigned char st = last ? COLO_STEP_LAST : COLO_STEP_MID;
    io.step_type[e] = st;
    if (io.step_type_mirror) io.step_type_mirror[e] = st;
    if (io.discount) io.discount[e] = last ? 0.f : 1.f;
    io.obs[e] = last ? -1 : nxt;
  }
  const long long copy = blockIdx.x & io.visits_mask;  // privatised counters: spread same-state atomics over L2
  if (io.visits_s) aggregated_inc(io.visits_s + copy * io.n_s, off_s + nxt, stepping || resetting);
  if (io.visits_sa) aggregated_inc(io.visits_sa + copy * io.n_sa, off_sa + (long long)nxt * tb.A + in.a, stepping);
}

// the dense reward class of a step s --a--> nxt
__device__ __forceinline__ int dense_cls(const colo_mdp_tables& tb, const EnvIn& in, int nxt) {
  if (tb.rew_cls_sas) return tb.rew_cls_sas[((size_t)in.s * tb.A + in.a) * tb.S + nxt];
  if (tb.rew_cls_sa) return tb.rew_cls_sa[(size_t)in.s * tb.A + in.a];
  return 0;
}

// Position of x in one monotone dense row, warp-cooperative.  The row is read as quads (4 consecutive entries per
// lane per 128-entry chunk), every load issued before any is consumed.  Because the row is non-decreasing, the
// number of entries <= x (STRICT: < x) is found hierarchically: one ballot per chunk on each quad's LAST entry
// counts the quads lying entirely at or below x; only the lane owning the crossing quad then looks at its other
// three entries.  ~3 instructions per chunk instead of a compare+add per entry and a 5-step shuffle reduction.
template <typename TC, int NCH, bool STRICT>
__device__ __forceinline__ int row_count_below(const TC* __restrict__ row, int ld, TC x, int lane) {
  for (int g = 0; g < ld; g += 128 * NCH) {
    Quad<TC> q[NCH];
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      const int c = g + k * 128 + lane * 4;
      if (c < ld) q[k].load(row + c);
    }
    int quads = 0;
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      const int c = g + k * 128 + lane * 4;
      const bool below = (c < ld) && (STRICT ? (q[k].v[3] < x) : (q[k].v[3] <= x));
      quads += __popc(__ballot_sync(FULL, below));
    }
    const int in_group = min(32 * NCH, (ld - g) >> 2);
    if (quads < in_group) {  // warp-uniform: the crossing quad is in this group
      const int kq = quads >> 5, lq = quads & 31;
      int part = 0;
#pragma unroll
      for (int k = 0; k < NCH; ++k)
        if (k == kq)
          part = STRICT ? ((q[k].v[0] < x) + (q[k].v[1] < x) + (q[k].v[2] < x))
                        : ((q[k].v[0] <= x) + (q[k].v[1] <= x) + (q[k].v[2] <= x));
      return g + 4 * quads + __shfl_sync(FULL, part, lq);
    }
  }
  return ld;
}

// next state of one env from its dense row, searched by the whole warp (row, S, ld, u warp-uniform):
// first j with cdf[j] > u * total  ==  number of entries <= x
template <typename TC, int NCH>
__device__ __forceinline__ int warp_row_next(const TC* __restrict__ row, int S, int ld, TC u, int lane) {
  const TC total = __ldg(row + S - 1);
  const TC x = u * total;
  int nxt = row_count_below<TC, NCH, false>(row, ld, x, lane);
  if (nxt >= S)  // x >= total (rounding): bisect's hi = n-1 clamp == first index where the row reaches total
    nxt = row_count_below<TC, NCH, true>(row, ld, total, lane);
  return nxt;
}

constexpr int kEnvUnroll = 4;  // independent row searches in flight per warp

template <typename TC, int NCH, bool SERVER>
__global__ void __launch_bounds__(kStepThreads) env_step_dense_kernel(const colo_mdp_tables tb, const StepIO io) {
  const int lane = threadIdx.x & 31;
  const long long warp_global = ((long long)blockIdx.x * kStepThreads + threadIdx.x) >> 5;
  const long long n_warps = ((long long)gridDim.x * kStepThreads) >> 5;
  const long long n_tiles = (io.N + 31) >> 5;
  const int S = tb.S, A = tb.A, ld = tb.ld;
  const TC* __restrict__ cdf = reinterpret_cast<const TC*>(tb.cdf);
  constexpr bool F32U = sizeof(TC) == 4;

  for (unsigned long long pass = io.srv_seq0 + 1;; ++pass) {  // SERVER: one pass per doorbell; else exactly one pass
  unsigned long long t_pass = step_t0(io);
  if (SERVER) {
    if (!server_wait(io, pass)) return;
    t_pass += pass - io.srv_seq0 - 1;
  }
  for (long long tile = warp_global; tile < n_tiles; tile += n_warps)
  for (int step = 0; step < io.n_steps; ++step) {  // an env is owned by the same lane for every step of the launch
    const long long e = tile * 32 + lane;
    const bool valid = e < io.N;
    EnvIn in;
    in.s = 0; in.a = 0; in.st = COLO_STEP_MID; in.h = 0; in.bad = 0; in.un64 = 0.0; in.un32 = 0.f; in.ur = 0.f;
    if (valid) in = load_env<F32U>(io, tb, e, t_pass + step);
    const bool is_last = valid && in.st == COLO_STEP_LAST;
    const bool resetting = is_last && io.auto_reset;
    const bool stepping = valid && !is_last && !in.bad;
    if (is_last && !io.auto_reset && io.status) *io.status = COLO_NEEDS_RESET;
    // lanes that do not step still take part in the searches with a harmless row (keeps the loop branch-free)
    const int s_l = stepping ? in.s : 0, a_l = stepping ? in.a : 0;
    const TC u_l = F32U ? (TC)in.un32 : (TC)in.un64;

    int my_next = 0;
    // the warp walks over the 32 envs of its tile; every lane helps searching env i's row
    for (int i0 = 0; i0 < 32; i0 += kEnvUnroll) {
#pragma unroll
      for (int k = 0; k < kEnvUnroll; ++k) {
        const int i = i0 + k;
        const int s_i = __shfl_sync(FULL, s_l, i);
        const int a_i = __shfl_sync(FULL, a_l, i);
        const TC u_i = __shfl_sync(FULL, u_l, i);
        const TC* row = cdf + ((size_t)s_i * A + a_i) * ld;
        const int nxt = warp_row_next<TC, NCH>(row, S, ld, u_i, lane);
        if (lane == i) my_next = nxt;
      }
    }
    const int cls = stepping ? dense_cls(tb, in, my_next) : 0;
    finish_env(io, tb, valid ? e : 0, in, my_next, cls, stepping, resetting);
  }
  if (!SERVER) return;
  server_done(io, pass);
  }
}

// SHORT rows (ld == 128 * NCH, NCH <= 8; the host pads rows of S <= 1024 to whole 128-entry chunks):
// branch-free, software-pipelined variant.  For U envs at a time the warp issues every row load (U * NCH 128-bit
// loads per lane in flight), then finds for each env the number G of quads lying entirely at or below x with one
// ballot + popc per chunk.  The within-quad step is deferred to the epilogue, where lane i finishes env i on its
// own (one 16-byte gather of quad G, which the warp has just pulled into L1), i.e. it is vectorised over the 32
// envs of the tile instead of costing shuffles and selects inside the per-env loop.
template <typename TC, int NCH, int U, int TILE, bool SERVER>
__global__ void __launch_bounds__(kStepThreads) env_step_dense_short_kernel(const colo_mdp_tables tb, const StepIO io) {
  // TILE envs per warp (lanes >= TILE idle in the per-lane phases): smaller tiles = more warps in flight when the
  // batch alone cannot fill the machine (65,536 envs / 32 = 14 warps per SM)
  const int lane = threadIdx.x & 31;
  const long long warp_global = ((long long)blockIdx.x * kStepThreads + threadIdx.x) >> 5;
  const long long n_warps = ((long long)gridDim.x * kStepThreads) >> 5;
  const long long n_tiles = (io.N + TILE - 1) / TILE;
  const int S = tb.S, A = tb.A;
  constexpr int ld = 128 * NCH;
  const TC* __restrict__ cdf = reinterpret_cast<const TC*>(tb.cdf);
  constexpr bool F32U = sizeof(TC) == 4;

  for (unsigned long long pass = io.srv_seq0 + 1;; ++pass) {  // SERVER: one pass per doorbell; else exactly one pass
  unsigned long long t_pass = step_t0(io);
  if (SERVER) {
    if (!server_wait(io, pass)) return;
    t_pass += pass - io.srv_seq0 - 1;
  }
  for (long long tile = warp_global; tile < n_tiles; tile += n_warps)
  for (int step = 0; step < io.n_steps; ++step) {  // an env is owned by the same lane for every step of the launch
    const long long e = tile * TILE + lane;
    const bool valid = lane < TILE && e < io.N;
    EnvIn in;
    in.s = 0; in.a = 0; in.st = COLO_STEP_MID; in.h = 0; in.bad = 0; in.un64 = 0.0; in.un32 = 0.f; in.ur = 0.f;
    if (valid) in = load_env<F32U>(io, tb, e, t_pass + step);
    const bool is_last = valid && in.st == COLO_STEP_LAST;
    const bool resetting = is_last && io.auto_reset;
    const bool stepping = valid && !is_last && !in.bad;
    if (is_last && !io.auto_reset && io.status) *io.status = COLO_NEEDS_RESET;
    // lanes that do not step take part with row 0 (keeps the loop branch-free); 32-bit element offsets
    // (the host checks S*A*ld < 2^31)
    const unsigned off_l = stepping ? (unsigned)(in.s * A + in.a) * (unsigned)ld : 0u;
    const TC u_l = F32U ? (TC)in.un32 : (TC)in.un64;

    int my_G = 0;
    for (int i0 = 0; i0 < TILE; i0 += U) {
      Quad<TC> q[U][NCH];
      TC x[U];
#pragma unroll
      for (int k = 0; k < U; ++k) {
        const unsigned off = __shfl_sync(FULL, off_l, i0 + k);
        const TC u = __shfl_sync(FULL, u_l, i0 + k);
        const TC* row = cdf + off;
        x[k] = u * __ldg(row + S - 1);
#pragma unroll
        for (int c = 0; c < NCH; ++c) q[k][c].load(row + c * 128 + lane * 4);
      }
#pragma unroll
      for (int k = 0; k < U; ++k) {
        int G = 0;
#pragma unroll
        for (int c = 0; c < NCH; ++c) G += __popc(__ballot_sync(FULL, q[k][c].v[3] <= x[k]));
        my_G = (lane == i0 + k) ? G : my_G;
      }
    }
    // per-lane finish: env `lane` of the tile
    int nxt = 0, cls = 0;
    if (stepping) {
      const TC* row = cdf + off_l;
      const TC total = __ldg(row + S - 1);
      const TC xl = u_l * total;  // same operands, same product as in the search above
      nxt = ld;
      if (my_G < 32 * NCH) {
        Quad<TC> qq;
        qq.load(row + 4 * my_G);  // the crossing quad: its last entry is > x, its first three decide
        nxt = 4 * my_G + (qq.v[0] <= xl) + (qq.v[1] <= xl) + (qq.v[2] <= xl);
      }
      if (nxt >= S) {  // x >= total (rounding): bisect's hi = n-1 clamp == first index where the row reaches total
        nxt = 0;
        while (nxt < S - 1 && __ldg(row + nxt) < total) ++nxt;
      }
      if (tb.rew_cls_sas)
        cls = tb.rew_cls_sas[((size_t)in.s * A + in.a) * S + nxt];
      else if (tb.rew_cls_sa)
        cls = tb.rew_cls_sa[(size_t)in.s * A + in.a];
    }
    finish_env(io, tb, valid ? e : 0, in, nxt, cls, stepping, resetting);
  }
  if (!SERVER) return;
  server_done(io, pass);
  }
}

// ---- breakpoint table (colo_mdp_tables.cdf_breaks) ----------------------------------------------------------------------
// Most benchmark rows have a handful of successors, so the CDF row is a step function with a few breakpoints p_k (where
// c[p_k] > c[p_k - 1]).  For x >= 0 the count of entries <= x over the whole padded row, with the clamp to the first
// index reaching the total, is p_min(k*, m-1), k* = #{k : v_k <= x}: one 16-byte entry per breakpoint carries the whole
// step (next state, its reward class, and the reward itself when the class's quantile row is constant).  A row of K
// entries is read in ONE round of K independent loads (K = 2: one 32-byte sector), instead of the three dependent rounds
// of the two-level index plus a fourth for the reward quantiles.
struct CdfBreak {
  float v;             // c[p]
  int p;               // the breakpoint: the next state
  unsigned cls_flags;  // reward class of (s, a, p) | kBreakInline
  float r;             // the reward, when kBreakInline
};
constexpr unsigned kBreakInline = 0x80000000u;

struct BreakStep {
  int nxt, cls;
  float rew;
  bool have_cls, have_rew;
};

// the step of row r for uniform u (x = u * total, total = v of the last entry), from its K breakpoint entries; x not >= 0
// (supplied uniforms: negative, NaN) finds no entry <= x, i.e. state 0, whose class the caller looks up (have_cls false)
template <int K>
__device__ __forceinline__ BreakStep breaks_step(const void* table, unsigned r, float u) {
  const int4* __restrict__ row = reinterpret_cast<const int4*>(table) + (size_t)r * K;
  int4 e[K];
#pragma unroll
  for (int k = 0; k < K; ++k) e[k] = __ldg(row + k);
  const float x = u * __int_as_float(e[K - 1].x);
  BreakStep b;
  b.nxt = 0; b.cls = 0; b.rew = 0.f; b.have_cls = false; b.have_rew = false;
  if (!(x >= 0.f)) return b;
  int ks = 0;
#pragma unroll
  for (int k = 0; k < K; ++k) ks += __int_as_float(e[k].x) <= x;
  ks = min(ks, K - 1);  // x >= total: the last breakpoint (the padding repeats it)
  int4 sel = e[0];
#pragma unroll
  for (int k = 1; k < K; ++k) sel = k == ks ? e[k] : sel;
  b.nxt = sel.y;
  b.cls = (int)((unsigned)sel.z & ~kBreakInline);
  b.have_cls = true;
  b.have_rew = ((unsigned)sel.z & kBreakInline) != 0u;
  b.rew = __int_as_float(sel.w);
  return b;
}

// SHORT rows, one THREAD per env: a three-round k-ary search instead of reading the whole row.  The last entries of
// the row's quads are monotone, so the number G of quads lying entirely at or below x is found from (1) the last entry
// of every 8th quad (4*NCH independent 4-byte loads, all issued before any is consumed), (2) the last entries of the 8
// quads of the block that holds the crossing, (3) the crossing quad itself (the same 16-byte gather the warp-
// cooperative kernel ends with).  With the two-level index of colo_mdp_tables (cdf_coarse / cdf_mid: copies of exactly
// those entries, contiguous) round 1 is NCH 128-bit loads of a 60 KB table and also yields the row total; round 2 is
// one 32-byte sector of cdf_mid plus, in the same round, the 32-byte sector of reward classes of the block's candidate
// next states (rew_cls_pad); round 3 the crossing quad.  Three dependent rounds per env after the env scalars, instead
// of 32/U per tile plus two.  (Tried on one box each: reading the whole 128-byte block in round 2 and skipping round 3
// -- 5.58 us per step instead of 5.17: four sectors cost more than one extra round; fetching the reward quantiles of
// every class before the search -- 5.50 us instead of 5.26.)  With 65,536 envs every warp is resident at once, so the step time IS the length of
// that dependency chain.  Same comparisons against the same x => the same index, bit for bit.
// KB > 0 (f32): the search is one round over the KB-entry breakpoint row instead (NCH is then unused).
template <typename TC, int NCH, bool SERVER, int KB = 0>
__global__ void __launch_bounds__(kStepThreads) env_step_dense_kary_kernel(const colo_mdp_tables tb, const StepIO io) {
  const long long n_thr = (long long)gridDim.x * kStepThreads;
  const long long n_pad = (io.N + 31) & ~31LL;  // whole warps: finish_env uses warp collectives
  const int S = tb.S, A = tb.A;
  constexpr int ld = 128 * NCH, NB = 4 * NCH;  // NB blocks of 8 quads
  const TC* __restrict__ cdf = reinterpret_cast<const TC*>(tb.cdf);
  const TC* __restrict__ mid = reinterpret_cast<const TC*>(tb.cdf_mid);
  const TC* __restrict__ coarse = tb.cdf_mid ? reinterpret_cast<const TC*>(tb.cdf_coarse) : nullptr;
  constexpr bool F32U = sizeof(TC) == 4;
  for (unsigned long long pass = io.srv_seq0 + 1;; ++pass) {  // SERVER: one pass per doorbell; else exactly one pass
  unsigned long long t_pass = step_t0(io);
  if (SERVER) {
    if (!server_wait(io, pass)) return;
    t_pass += pass - io.srv_seq0 - 1;
  }
  for (long long e = (long long)blockIdx.x * kStepThreads + threadIdx.x; e < n_pad; e += n_thr)
  for (int step = 0; step < io.n_steps; ++step) {  // an env is owned by the same thread for every step of the launch
    const bool valid = e < io.N;
    EnvIn in;
    in.s = 0; in.a = 0; in.st = COLO_STEP_MID; in.h = 0; in.bad = 0; in.un64 = 0.0; in.un32 = 0.f; in.ur = 0.f;
    if (valid) in = load_env<F32U>(io, tb, e, t_pass + step);
    const bool is_last = valid && in.st == COLO_STEP_LAST;
    const bool resetting = is_last && io.auto_reset;
    const bool stepping = valid && !is_last && !in.bad;
    if (is_last && !io.auto_reset && io.status) *io.status = COLO_NEEDS_RESET;
    int nxt = 0, cls = 0;
    bool have_rew = false;
    float rew = 0.f;
    if (stepping) {
      bool have_cls = false;
      if constexpr (KB > 0) {
        const BreakStep b = breaks_step<KB>(tb.cdf_breaks, (unsigned)(in.s * A + in.a), in.un32);
        nxt = b.nxt;
        cls = b.cls;
        have_cls = b.have_cls;
        // a constant class gives its reward at every uniform in [0, 1] (supplied ones may lie outside)
        have_rew = b.have_rew && in.ur >= 0.f && in.ur <= 1.f;
        rew = b.rew;
      } else {
        const TC* row = cdf + (size_t)(unsigned)(in.s * A + in.a) * (unsigned)ld;
        TC total, x;
        int blk = 0, G = 0;
        uint4 c0 = make_uint4(0, 0, 0, 0), c1 = c0;
        nxt = ld;
        if (coarse) {  // two-level index: NCH 128-bit loads of a small hot table, then the 8 quad ends of one block
          const unsigned r = (unsigned)(in.s * A + in.a);
          Quad<TC> cq[NCH];
#pragma unroll
          for (int k = 0; k < NCH; ++k) cq[k].load(coarse + (size_t)r * NB + 4 * k);
          total = cq[NCH - 1].v[3];  // row[ld-1]: the padding [S, ld) holds the row total, i.e. the value of row[S-1]
          x = (F32U ? (TC)in.un32 : (TC)in.un64) * total;
#pragma unroll
          for (int k = 0; k < NCH; ++k) blk += (cq[k].v[0] <= x) + (cq[k].v[1] <= x) + (cq[k].v[2] <= x) + (cq[k].v[3] <= x);
          if (blk < NB) {
            // round 2: the 8 quad ends of the block (one 32-byte sector of cdf_mid) and, in the same round, the reward
            // classes of the block's 32 candidate next states (rew_cls_pad: rew_cls_sas with rows padded to ld, so the
            // slice is one aligned 32-byte sector): the class lookup no longer waits for the search to finish
            Quad<TC> m0, m1;
            const TC* mp = mid + (size_t)r * (32 * NCH) + 8 * blk;
            m0.load(mp);
            m1.load(mp + 4);
            if (tb.rew_cls_pad) {
              const uint4* cp = reinterpret_cast<const uint4*>(tb.rew_cls_pad + (size_t)r * ld + 32 * blk);
              c0 = __ldg(cp);
              c1 = __ldg(cp + 1);
            }
            G = 8 * blk + (m0.v[0] <= x) + (m0.v[1] <= x) + (m0.v[2] <= x) + (m0.v[3] <= x) + (m1.v[0] <= x) +
                (m1.v[1] <= x) + (m1.v[2] <= x) + (m1.v[3] <= x);
          }
        } else {
          total = __ldg(row + S - 1);
          x = (F32U ? (TC)in.un32 : (TC)in.un64) * total;
          TC c[NB];
#pragma unroll
          for (int k = 0; k < NB; ++k) c[k] = __ldg(row + 32 * k + 31);  // last entry of quad 8k+7
#pragma unroll
          for (int k = 0; k < NB; ++k) blk += c[k] <= x ? 1 : 0;
          if (blk < NB) {
            const TC* b = row + 32 * blk;
            TC q[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) q[k] = __ldg(b + 4 * k + 3);
            G = 8 * blk;
#pragma unroll
            for (int k = 0; k < 8; ++k) G += q[k] <= x ? 1 : 0;
          }
        }
        if (blk < NB) {
          Quad<TC> qq;
          qq.load(row + 4 * G);  // the crossing quad: its last entry is > x, its first three decide
          nxt = 4 * G + (qq.v[0] <= x) + (qq.v[1] <= x) + (qq.v[2] <= x);
          if (coarse && tb.rew_cls_pad && nxt < S) {
            const int pos = nxt - 32 * blk;
            const unsigned w = pos < 16 ? (pos < 8 ? (pos < 4 ? c0.x : c0.y) : (pos < 12 ? c0.z : c0.w))
                                        : (pos < 24 ? (pos < 20 ? c1.x : c1.y) : (pos < 28 ? c1.z : c1.w));
            cls = (int)((w >> (8 * (pos & 3))) & 0xffu);
            have_cls = true;
          }
        }
        if (nxt >= S) {  // x >= total (rounding): bisect's hi = n-1 clamp == first index where the row reaches total
          nxt = 0;
          while (nxt < S - 1 && __ldg(row + nxt) < total) ++nxt;
          have_cls = false;
        }
      }
      if (!have_cls) {
        if (tb.rew_cls_sas)
          cls = tb.rew_cls_sas[((size_t)in.s * A + in.a) * S + nxt];
        else if (tb.rew_cls_sa)
          cls = tb.rew_cls_sa[(size_t)in.s * A + in.a];
      }
    }
    finish_env(io, tb, valid ? e : 0, in, nxt, cls, stepping, resetting, 0, 0, have_rew, rew);
  }
  if (!SERVER) return;
  server_done(io, pass);
  }
}

// The LEAN form of the k-ary step for the common call: one step per launch, supplied actions, in-kernel Philox uniforms,
// auto-reset, visitation counters on, two-level index present, fewer than 2^31 envs.  Same loads, same comparisons
// against the same x, same Philox counters as env_step_dense_kary_kernel -- bit-identical results -- but none of the
// generality is paid for at run time: no grid-stride / n_steps / server loops, 32-bit env indices, the fp64 start
// uniform only on the (rare) reset path, no optional-pointer tests on the hot path.  ncu of the general kernel at
// 4 Mi envs: 505 warp instructions per env-step, issue slots 68 % busy, DRAM 11 % -- the kernel is ISSUE bound once
// the batch fills the machine, so instructions are what the asymptotic env-steps/s is made of.
constexpr int kLeanThreads = 128;

// prologue and epilogue of the lean kernels: env scalars in, Philox words, the action check; stores and counters out
struct LeanEnv {
  int st, s, h, a;
  bool resetting, stepping;
  Philox4 w;
};

template <bool COMPACT>
__device__ __forceinline__ LeanEnv lean_load(const colo_mdp_tables& tb, const StepIO& io, unsigned e) {
  LeanEnv v;
  const bool valid = e < (unsigned)io.N;
  v.st = COLO_STEP_MID; v.s = 0; v.h = 0; v.a = 0;
  if (valid) {
    v.st = io.step_type[e];
    v.s = io.state[e];
    v.h = io.h[e];
    if (COMPACT)
      v.a = reinterpret_cast<const unsigned char*>(io.action)[e];
    else
      v.a = io.srv_go ? __ldcv(io.action + e) : io.action[e];
  }
  v.w = philox4x32_10(io.seed, io.env0 + (uint64_t)e, step_t0(io));
  bool bad = false;
  if ((unsigned)v.a >= (unsigned)tb.A) {
    if (io.status) *io.status = COLO_BAD_ACTION;
    v.a = 0;
    bad = true;
  }
  v.resetting = valid && v.st == COLO_STEP_LAST;
  v.stepping = valid && v.st != COLO_STEP_LAST && !bad;
  return v;
}

// have_rew: `rew` is the step's reward (no draw from class `cls`)
template <bool COMPACT>
__device__ __forceinline__ void lean_store(const colo_mdp_tables& tb, const StepIO& io, unsigned e, const LeanEnv& v,
                                           int nxt, int cls, bool have_rew, float rew) {
  if (v.resetting) {  // auto_reset path == BaseMDP.reset(): the action is ignored, reward is None (NaN here)
    nxt = sample_start(tb, u53(v.w.w[0], v.w.w[1]));
    io.state[e] = nxt;
    io.h[e] = 0;
    io.step_type[e] = COLO_STEP_FIRST;
    if (io.step_type_mirror) io.step_type_mirror[e] = COLO_STEP_FIRST;
    io.reward[e] = __int_as_float(0x7fc00000);
    if (io.discount) io.discount[e] = __int_as_float(0x7fc00000);
    if (COMPACT)
      reinterpret_cast<short*>(io.obs)[e] = (short)nxt;
    else
      io.obs[e] = nxt;
  } else if (v.stepping) {
    const int hh = v.h + 1;
    const bool last = tb.H > 0 && hh >= tb.H;
    const unsigned char nst = last ? COLO_STEP_LAST : COLO_STEP_MID;
    io.h[e] = hh;
    io.state[e] = nxt;
    io.reward[e] = have_rew ? rew : reward_draw(tb, cls, u24(v.w.w[2]));
    io.step_type[e] = nst;
    if (io.step_type_mirror) io.step_type_mirror[e] = nst;
    if (io.discount) io.discount[e] = last ? 0.f : 1.f;
    if (COMPACT)
      reinterpret_cast<short*>(io.obs)[e] = last ? (short)-1 : (short)nxt;
    else
      io.obs[e] = last ? -1 : nxt;
  }
  const unsigned copy = blockIdx.x & (unsigned)io.visits_mask;
  aggregated_inc(io.visits_s + (size_t)copy * io.n_s, nxt, v.stepping || v.resetting);
  aggregated_inc(io.visits_sa + (size_t)copy * io.n_sa, (long long)nxt * tb.A + v.a, v.stepping);
}

template <int NCH, bool COMPACT>
__global__ void __launch_bounds__(kLeanThreads) env_step_kary_lean_kernel(const colo_mdp_tables tb, const StepIO io) {
  constexpr int ld = 128 * NCH, NB = 4 * NCH;
  const unsigned e = blockIdx.x * kLeanThreads + threadIdx.x;
  const int S = tb.S, A = tb.A;
  const LeanEnv v = lean_load<COMPACT>(tb, io, e);
  const int s = v.s, a = v.a;
  int nxt = 0, cls = 0;
  if (v.stepping) {
    const unsigned r = (unsigned)(s * A + a);
    const float* __restrict__ coarse = reinterpret_cast<const float*>(tb.cdf_coarse) + (size_t)r * NB;
    const float* __restrict__ row = reinterpret_cast<const float*>(tb.cdf) + (size_t)r * ld;
    float4 cq[NCH];
#pragma unroll
    for (int k = 0; k < NCH; ++k) cq[k] = __ldg(reinterpret_cast<const float4*>(coarse) + k);
    const float total = cq[NCH - 1].w;
    const float x = u24(v.w.w[0]) * total;
    int blk = 0;
#pragma unroll
    for (int k = 0; k < NCH; ++k) blk += (cq[k].x <= x) + (cq[k].y <= x) + (cq[k].z <= x) + (cq[k].w <= x);
    bool have_cls = false;
    nxt = ld;
    if (blk < NB) {
      const float4* mp = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(tb.cdf_mid) + (size_t)r * (32 * NCH) + 8 * blk);
      const uint4* cp = reinterpret_cast<const uint4*>(tb.rew_cls_pad + (size_t)r * ld + 32 * blk);
      const float4 m0 = __ldg(mp), m1 = __ldg(mp + 1);
      const uint4 c0 = __ldg(cp), c1 = __ldg(cp + 1);
      const int G = 8 * blk + (m0.x <= x) + (m0.y <= x) + (m0.z <= x) + (m0.w <= x) + (m1.x <= x) + (m1.y <= x) +
                    (m1.z <= x) + (m1.w <= x);
      const float4 qq = __ldg(reinterpret_cast<const float4*>(row) + G);
      nxt = 4 * G + (qq.x <= x) + (qq.y <= x) + (qq.z <= x);
      if (nxt < S) {
        const int pos = nxt - 32 * blk;
        const unsigned wsel = pos < 16 ? (pos < 8 ? (pos < 4 ? c0.x : c0.y) : (pos < 12 ? c0.z : c0.w))
                                       : (pos < 24 ? (pos < 20 ? c1.x : c1.y) : (pos < 28 ? c1.z : c1.w));
        cls = (int)((wsel >> (8 * (pos & 3))) & 0xffu);
        have_cls = true;
      }
    }
    if (nxt >= S) {  // x >= total (rounding): bisect's hi = n-1 clamp == first index where the row reaches total
      nxt = 0;
      while (nxt < S - 1 && __ldg(row + nxt) < total) ++nxt;
    }
    if (!have_cls) cls = tb.rew_cls_sas ? tb.rew_cls_sas[((size_t)s * A + a) * S + nxt] : (tb.rew_cls_sa ? tb.rew_cls_sa[(size_t)s * A + a] : 0);
  }
  lean_store<COMPACT>(tb, io, e, v, nxt, cls, false, 0.f);
}

// The lean call on the breakpoint table: env scalars -> one K-entry breakpoint row (one round of K independent 16-byte
// loads) -> stores, plus a reward-quantile round only where the class is not constant.  Same Philox words, same x, same
// result and reward bits as env_step_kary_lean_kernel.
template <int K, bool COMPACT>
__global__ void __launch_bounds__(kLeanThreads) env_step_breaks_lean_kernel(const colo_mdp_tables tb, const StepIO io) {
  const unsigned e = blockIdx.x * kLeanThreads + threadIdx.x;
  const LeanEnv v = lean_load<COMPACT>(tb, io, e);
  int nxt = 0, cls = 0;
  bool have_rew = false;
  float rew = 0.f;
  if (v.stepping) {
    // x = u24 * total >= 0 (the builder refuses negative and NaN rows): the entry always carries the class
    const BreakStep b = breaks_step<K>(tb.cdf_breaks, (unsigned)(v.s * tb.A + v.a), u24(v.w.w[0]));
    nxt = b.nxt;
    cls = b.cls;
    have_rew = b.have_rew;
    rew = b.rew;
  }
  lean_store<COMPACT>(tb, io, e, v, nxt, cls, have_rew, rew);
}

// one step of one env from successor-list tables (every lane of the warp calls it: finish_env uses warp collectives);
// seed / ctr / off_s / off_sa as in load_env and finish_env
__device__ __forceinline__ void succ_env_step(const StepIO& io, const colo_mdp_tables& tb, long long e, bool valid,
                                              unsigned long long t, unsigned long long seed, unsigned long long ctr,
                                              long long off_s, long long off_sa) {
  EnvIn in;
  in.s = 0; in.a = 0; in.st = COLO_STEP_MID; in.h = 0; in.bad = 0; in.un64 = 0.0; in.un32 = 0.f; in.ur = 0.f;
  if (valid) in = load_env<false>(io, tb, e, t, seed, ctr);
  const bool is_last = valid && in.st == COLO_STEP_LAST;
  const bool resetting = is_last && io.auto_reset;
  const bool stepping = valid && !is_last && !in.bad;
  if (is_last && !io.auto_reset && io.status) *io.status = COLO_NEEDS_RESET;
  int nxt = 0, cls = 0;
  if (stepping) {
    const size_t sa = (size_t)in.s * tb.A + in.a;
    const size_t base = sa * tb.Ksucc;
    const int n = __ldg(tb.succ_len + sa);
    int pos = 0;
    if (n > 1) {
      const double total = __ldg(tb.succ_cum + base + n - 1) + 0.0;
      pos = bisect_count(tb.succ_cum + base, n, in.un64 * total);
    }
    nxt = __ldg(tb.succ_idx + base + pos);
    cls = tb.rew_cls_succ ? __ldg(tb.rew_cls_succ + base + pos) : 0;
  }
  finish_env(io, tb, valid ? e : 0, in, nxt, cls, stepping, resetting, off_s, off_sa);
}

template <bool SERVER>
__global__ void __launch_bounds__(kStepThreads) env_step_succ_kernel(const colo_mdp_tables tb, const StepIO io) {
  const long long n_thr = (long long)gridDim.x * kStepThreads;
  // round the loop bound up to whole warps: finish_env uses warp collectives
  const long long n_pad = (io.N + 31) & ~31LL;
  for (unsigned long long pass = io.srv_seq0 + 1;; ++pass) {  // SERVER: one pass per doorbell; else exactly one pass
  unsigned long long t_pass = step_t0(io);
  if (SERVER) {
    if (!server_wait(io, pass)) return;
    t_pass += pass - io.srv_seq0 - 1;
  }
  for (long long e = (long long)blockIdx.x * kStepThreads + threadIdx.x; e < n_pad; e += n_thr)
  for (int step = 0; step < io.n_steps; ++step)  // an env is owned by the same thread for every step of the launch
    succ_env_step(io, tb, e, e < io.N, t_pass + step, io.seed, io.env0 + (uint64_t)e, 0, 0);
  if (!SERVER) return;
  server_done(io, pass);
  }
}

// BaseMDP.reset of one env (valid); returns its start state
__device__ __forceinline__ int reset_env(const StepIO& io, const colo_mdp_tables& tb, long long e,
                                         unsigned long long seed, unsigned long long ctr) {
  const double* u_next = reinterpret_cast<const double*>(io.u_next);
  double u;
  if (u_next)
    u = u_next[e];
  else {
    Philox4 w = philox4x32_10(seed, ctr, io.t);
    u = u53(w.w[0], w.w[1]);
  }
  const int s0 = sample_start(tb, u);
  io.state[e] = s0;
  io.h[e] = 0;
  io.step_type[e] = COLO_STEP_FIRST;
  if (io.step_type_mirror) io.step_type_mirror[e] = COLO_STEP_FIRST;
  if (io.discount) io.discount[e] = __int_as_float(0x7fc00000);
  if (io.reward) io.reward[e] = __int_as_float(0x7fc00000);  // the reference's reward of a FIRST TimeStep is None
  if (io.io_compact)
    reinterpret_cast<short*>(io.obs)[e] = (short)s0;
  else
    io.obs[e] = s0;
  return s0;
}

__global__ void __launch_bounds__(kStepThreads) env_reset_kernel(const colo_mdp_tables tb, const StepIO io) {
  const long long n_thr = (long long)gridDim.x * kStepThreads;
  const long long n_pad = (io.N + 31) & ~31LL;
  for (long long e = (long long)blockIdx.x * kStepThreads + threadIdx.x; e < n_pad; e += n_thr) {
    const bool valid = e < io.N;
    const int s0 = valid ? reset_env(io, tb, e, io.seed, io.env0 + (uint64_t)e) : 0;
    const long long copy = blockIdx.x & io.visits_mask;
    if (io.visits_s) aggregated_inc(io.visits_s + copy * io.n_s, s0, valid);
  }
}

// ---- mixed batches (colo_mixed_tables, mixed.cuh): envs of different MDP instances in one launch -----------------------
__device__ __forceinline__ int mixed_inst_of(const int* __restrict__ inst_of, long long e, bool valid) {
  return valid ? __ldg(inst_of + e) : 0;  // lanes past the batch take part in the warp collectives as instance 0
}

__global__ void __launch_bounds__(kStepThreads) env_reset_mixed_kernel(const MixedInst* __restrict__ insts,
                                                                      const int* __restrict__ inst_of, const StepIO io) {
  const long long n_thr = (long long)gridDim.x * kStepThreads;
  const long long n_pad = (io.N + 31) & ~31LL;
  for (long long e = (long long)blockIdx.x * kStepThreads + threadIdx.x; e < n_pad; e += n_thr) {
    const bool valid = e < io.N;
    const MixedInst d = insts[mixed_inst_of(inst_of, e, valid)];
    const int s0 = valid ? reset_env(io, d.tb, e, d.seed, (unsigned long long)(e - d.start)) : 0;
    const long long copy = blockIdx.x & io.visits_mask;
    if (io.visits_s) aggregated_inc(io.visits_s + copy * io.n_s, d.off_s + s0, valid);
  }
}

__global__ void __launch_bounds__(kStepThreads) env_step_succ_mixed_kernel(const MixedInst* __restrict__ insts,
                                                                          const int* __restrict__ inst_of, const StepIO io) {
  const long long n_thr = (long long)gridDim.x * kStepThreads;
  const long long n_pad = (io.N + 31) & ~31LL;
  for (long long e = (long long)blockIdx.x * kStepThreads + threadIdx.x; e < n_pad; e += n_thr) {
    const bool valid = e < io.N;
    const MixedInst d = insts[mixed_inst_of(inst_of, e, valid)];
    for (int step = 0; step < io.n_steps; ++step)
      succ_env_step(io, d.tb, e, valid, io.t + step, d.seed, (unsigned long long)(e - d.start), d.off_s, d.off_sa);
  }
}

// the warp-per-env dense search of env_step_dense_kernel, every env searching its own instance's row
template <typename TC, int NCH>
__global__ void __launch_bounds__(kStepThreads) env_step_dense_mixed_kernel(const MixedInst* __restrict__ insts,
                                                                           const int* __restrict__ inst_of, const StepIO io) {
  const int lane = threadIdx.x & 31;
  const long long warp_global = ((long long)blockIdx.x * kStepThreads + threadIdx.x) >> 5;
  const long long n_warps = ((long long)gridDim.x * kStepThreads) >> 5;
  const long long n_tiles = (io.N + 31) >> 5;
  constexpr bool F32U = sizeof(TC) == 4;
  for (long long tile = warp_global; tile < n_tiles; tile += n_warps) {
    const long long e = tile * 32 + lane;
    const bool valid = e < io.N;
    const MixedInst d = insts[mixed_inst_of(inst_of, e, valid)];
    const TC* __restrict__ cdf = reinterpret_cast<const TC*>(d.tb.cdf);
    for (int step = 0; step < io.n_steps; ++step) {
      EnvIn in;
      in.s = 0; in.a = 0; in.st = COLO_STEP_MID; in.h = 0; in.bad = 0; in.un64 = 0.0; in.un32 = 0.f; in.ur = 0.f;
      if (valid) in = load_env<F32U>(io, d.tb, e, io.t + step, d.seed, (unsigned long long)(e - d.start));
      const bool is_last = valid && in.st == COLO_STEP_LAST;
      const bool resetting = is_last && io.auto_reset;
      const bool stepping = valid && !is_last && !in.bad;
      if (is_last && !io.auto_reset && io.status) *io.status = COLO_NEEDS_RESET;
      // lanes that do not step search row 0 of their instance; every lane hands the warp its own row and shape
      const TC* row_l = cdf + (stepping ? ((size_t)in.s * d.tb.A + in.a) * d.tb.ld : 0);
      const TC u_l = F32U ? (TC)in.un32 : (TC)in.un64;
      int my_next = 0;
      for (int i0 = 0; i0 < 32; i0 += kEnvUnroll) {
#pragma unroll
        for (int k = 0; k < kEnvUnroll; ++k) {
          const int i = i0 + k;
          const TC* row = reinterpret_cast<const TC*>(__shfl_sync(FULL, (unsigned long long)row_l, i));
          const int S_i = __shfl_sync(FULL, d.tb.S, i), ld_i = __shfl_sync(FULL, d.tb.ld, i);
          const TC u_i = __shfl_sync(FULL, u_l, i);
          const int nxt = warp_row_next<TC, NCH>(row, S_i, ld_i, u_i, lane);
          if (lane == i) my_next = nxt;
        }
      }
      const int cls = stepping ? dense_cls(d.tb, in, my_next) : 0;
      finish_env(io, d.tb, valid ? e : 0, in, my_next, cls, stepping, resetting, d.off_s, d.off_sa);
    }
  }
}

template <typename TC>
__global__ void build_dense_cdf_kernel(const float* __restrict__ T, int S, int A, int ld, TC* __restrict__ cdf) {
  // one thread per (s,a) row: sequential fp64 running sum -- the DEFINED summation order of the dense CDF
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= (long long)S * A) return;
  const float* row = T + r * S;
  TC* out = cdf + r * ld;
  double acc = 0.0;
  for (int j = 0; j < ld; ++j) {
    if (j < S) acc += (double)row[j];
    out[j] = (TC)acc;
  }
}

template <typename TC>
__global__ void build_cdf_index_kernel(const TC* __restrict__ cdf, long long rows, int ld, TC* __restrict__ mid,
                                       TC* __restrict__ coarse) {
  const int nq = ld / 4, nb = ld / 32;
  const long long total = rows * nq;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / nq;
    const int q = (int)(i - r * nq);
    const TC v = cdf[r * ld + 4 * q + 3];
    mid[i] = v;
    if ((q & 7) == 7) coarse[r * nb + (q >> 3)] = v;
  }
}

// the breakpoints of one f32 cdf row c[0..S) (c[-1] := 0): calls at(k, p_k, v_k) for each, returns their number, or -1 when
// the row decreases somewhere or holds a NaN (no step function to tabulate)
template <typename F>
__device__ __forceinline__ int row_breaks(const float* __restrict__ row, int S, F at) {
  float prev = 0.f;
  int m = 0;
  for (int j = 0; j < S; ++j) {
    const float c = row[j];
    if (!(c >= prev)) return -1;
    if (c > prev) at(m++, j, c);
    prev = c;
  }
  return m;
}

__global__ void count_cdf_breaks_kernel(const float* __restrict__ cdf, long long rows, int S, int ld, int* __restrict__ out) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const int m = row_breaks(cdf + r * ld, S, [](int, int, float) {});
  atomicMax(out, m < 0 ? S + 1 : m);
}

// one thread per (s, a) row: the row's breakpoints, padded with copies of the last, then every entry's reward class and,
// for a class whose quantile row is bitwise constant and finite, its reward as reward_draw computes it (the same bits at
// every uniform in [0, 1]: fmaf(f, +0, q0) == q0 + 0)
__global__ void build_cdf_breaks_kernel(const colo_mdp_tables tb, int K, CdfBreak* __restrict__ out, int* __restrict__ err) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= (long long)tb.S * tb.A) return;
  CdfBreak* b = out + r * K;
  int m = row_breaks(reinterpret_cast<const float*>(tb.cdf) + r * tb.ld, tb.S, [&](int k, int p, float v) {
    if (k < K) {
      b[k].v = v;
      b[k].p = p;
    }
  });
  if (m < 0 || m > K) {
    atomicExch(err, 1);
    m = m < 0 ? 0 : K;
  }
  if (m == 0) {  // an all-zero row: its search returns state 0
    b[0].v = 0.f;
    b[0].p = 0;
    m = 1;
  }
  for (int k = m; k < K; ++k) {
    b[k].v = b[m - 1].v;
    b[k].p = b[m - 1].p;
  }
  for (int k = 0; k < K; ++k) {
    const int p = b[k].p;
    const int cls = tb.rew_cls_sas ? tb.rew_cls_sas[r * tb.S + p] : (tb.rew_cls_sa ? tb.rew_cls_sa[r] : 0);
    const float* q = tb.rew_q + (size_t)cls * tb.nq;
    bool constant = isfinite(q[0]);
    for (int i = 1; i < tb.nq && constant; ++i) constant = __float_as_uint(q[i]) == __float_as_uint(q[0]);
    b[k].cls_flags = (unsigned)cls | (constant ? kBreakInline : 0u);
    b[k].r = constant ? reward_draw(tb, cls, 0.f) : 0.f;
  }
}

// Non-tabular observations: EmissionMap.get_observation (colosseum/emission_maps/base.py:110-140) is a row gather from
// the precomputed table all_observations[h, s, ...] (:56-76); past the horizon (in_episode_time >= H, i.e. the LAST
// step of an episode) the reference returns zeros (:131-132).  One warp per env copies the D floats of its row.
__global__ void __launch_bounds__(256) emit_observations_kernel(const float* __restrict__ table, const int* __restrict__ state,
                                                                const int* __restrict__ h,
                                                                const unsigned char* __restrict__ step_type, long long N,
                                                                int H, int S, int D, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long e = warp; e < N; e += n_warps) {
    const int s = state[e];
    const int hh = H > 0 ? h[e] : 0;
    const bool zero = H > 0 && (hh >= H || step_type[e] == COLO_STEP_LAST);
    const float* row = table + ((size_t)(H > 0 ? hh : 0) * S + s) * D;
    float* o = out + (size_t)e * D;
    for (int j = lane; j < D; j += 32) o[j] = zero ? 0.f : row[j];
  }
}

static int grid_for(long long work_items_per_thread_block, long long total) {
  long long blocks = (total + work_items_per_thread_block - 1) / work_items_per_thread_block;
  long long cap = (long long)sm_count() * 32;  // 64-thread CTAs: up to 32 resident per SM
  if (blocks < 1) blocks = 1;
  return (int)(blocks < cap ? blocks : cap);
}

static int check_tables_common(const colo_mdp_tables* tb) {
  COLO_ARG_CHECK(tb != nullptr, "tables is NULL");
  COLO_ARG_CHECK(tb->S > 0 && tb->A > 0 && tb->H >= 0, "S, A, H");
  COLO_ARG_CHECK(tb->rew_q && tb->n_cls > 0 && tb->nq >= 2, "reward quantile table");
  COLO_ARG_CHECK(tb->start_cum && tb->start_idx && tb->n_start > 0, "start distribution");
  return COLO_OK;
}

// SERVER launches must be wholly co-resident (the CTAs of a pass meet at a counter): the grid is capped at
// 1/share of what the device holds at once
template <typename K>
static int resident_cap(K kernel, int share) {
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kStepThreads, 0) != cudaSuccess || per_sm < 1) per_sm = 1;
  const int cap = per_sm * sm_count() / (share < 1 ? 1 : share);
  return cap < 1 ? 1 : cap;
}

template <typename K>
static void launch_step(K kernel, int grid, bool server, int share, const colo_mdp_tables* tb, const StepIO& io,
                        cudaStream_t st) {
  if (server) {
    const int cap = resident_cap(kernel, share);
    grid = grid < cap ? grid : cap;
  }
  kernel<<<grid, kStepThreads, 0, st>>>(*tb, io);
}

template <typename TC, bool SERVER>
static int launch_dense(const colo_mdp_tables* tb, const StepIO& io, void* stream, int share = 1) {
  int r = check_tables_common(tb);
  if (r != COLO_OK) return r;
  COLO_ARG_CHECK(tb->cdf && tb->ld >= tb->S && tb->ld % 4 == 0, "dense cdf with ld % 4 == 0 is required");
  COLO_ARG_CHECK((uintptr_t)tb->cdf % 16 == 0, "cdf must be 16-byte aligned");
  COLO_ARG_CHECK(io.reward && io.action, "env buffers");
  if (io.N == 0) return COLO_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int ld = tb->ld;
  const bool short_rows = ld % 128 == 0 && ld <= 1024 && (long long)tb->S * tb->A * ld < (1LL << 31);
  if (short_rows) {
    // envs per warp: 32 when the batch alone fills the machine, fewer (more warps in flight) otherwise
    static const int forced = getenv("COLO_STEP_TILE") ? atoi(getenv("COLO_STEP_TILE")) : 0;
    const long long warps32 = (io.N + 31) / 32;
    // measured on B200 at N=65,536 (14 warps/SM with 32-env tiles): 32 -> 14.1 us, 16 -> 14.4 us, 8 -> 16.6 us
    int tile = warps32 >= (long long)sm_count() * 8 ? 32 : (warps32 >= (long long)sm_count() * 4 ? 16 : 8);
    if (forced == 8 || forced == 16 || forced == 32) tile = forced;
    // thread-per-env k-ary search (default) or the warp-cooperative full-row count (COLO_STEP_KERNEL=coop)
    static const bool coop = getenv("COLO_STEP_KERNEL") && !strcmp(getenv("COLO_STEP_KERNEL"), "coop");
    static const bool no_lean = getenv("COLO_STEP_KERNEL") && !strcmp(getenv("COLO_STEP_KERNEL"), "general");
    // the breakpoint table (f32 only) replaces the row search and the index in both thread-per-env kernels
    const int kb = sizeof(TC) == 4 && tb->cdf_breaks ? tb->cdf_breaks_k : 0;
    COLO_ARG_CHECK(kb == 0 || kb == 2 || kb == 4 || kb == 8 || kb == 16, "cdf_breaks_k must be 2, 4, 8 or 16");
    COLO_ARG_CHECK(kb == 0 || (uintptr_t)tb->cdf_breaks % 16 == 0, "cdf_breaks must be 16-byte aligned");
    if (!coop && !no_lean && !SERVER && sizeof(TC) == 4 && io.n_steps == 1 && !io.random_actions && io.u_next == nullptr &&
        io.u_rew == nullptr && io.auto_reset && (kb || (tb->cdf_mid && tb->cdf_coarse && tb->rew_cls_pad)) && io.visits_s &&
        io.visits_sa && io.N < (1LL << 31) - kLeanThreads) {
      const int gl = (int)((io.N + kLeanThreads - 1) / kLeanThreads);
      if (kb) {
#define COLO_BREAKS_LEAN(K)                                                                          \
  case K:                                                                                            \
    if (io.io_compact) env_step_breaks_lean_kernel<K, true><<<gl, kLeanThreads, 0, st>>>(*tb, io);   \
    else env_step_breaks_lean_kernel<K, false><<<gl, kLeanThreads, 0, st>>>(*tb, io);                 \
    break
        switch (kb) {
          COLO_BREAKS_LEAN(2);
          COLO_BREAKS_LEAN(4);
          COLO_BREAKS_LEAN(8);
          COLO_BREAKS_LEAN(16);
        }
#undef COLO_BREAKS_LEAN
        count_step_launch(COLO_STEP_KIND_BREAKS);
        return check_launch("env_step_breaks_lean_kernel");
      }
#define COLO_LEAN(NCH)                                                              \
  case NCH:                                                                         \
    if (io.io_compact) env_step_kary_lean_kernel<NCH, true><<<gl, kLeanThreads, 0, st>>>(*tb, io);   \
    else env_step_kary_lean_kernel<NCH, false><<<gl, kLeanThreads, 0, st>>>(*tb, io);                 \
    break
      switch (ld / 128) {
        COLO_LEAN(1);
        COLO_LEAN(2);
        COLO_LEAN(3);
        COLO_LEAN(4);
        COLO_LEAN(5);
        COLO_LEAN(6);
        COLO_LEAN(7);
        COLO_LEAN(8);
      }
#undef COLO_LEAN
      count_step_launch(COLO_STEP_KIND_LEAN);
      return check_launch("env_step_kary_lean_kernel");
    }
    COLO_ARG_CHECK(!io.io_compact, "io_compact is offered by the common call of the dense f32 step only (supplied actions, "
                                   "in-kernel uniforms, auto_reset, CDF index present, counters on, no server)");
    if (!coop) {
      const int gk = grid_for(kStepThreads, io.N);
      if (kb) {
        switch (kb) {
          case 2: launch_step(env_step_dense_kary_kernel<float, 1, SERVER, 2>, gk, SERVER, share, tb, io, st); break;
          case 4: launch_step(env_step_dense_kary_kernel<float, 1, SERVER, 4>, gk, SERVER, share, tb, io, st); break;
          case 8: launch_step(env_step_dense_kary_kernel<float, 1, SERVER, 8>, gk, SERVER, share, tb, io, st); break;
          case 16: launch_step(env_step_dense_kary_kernel<float, 1, SERVER, 16>, gk, SERVER, share, tb, io, st); break;
        }
        count_step_launch(COLO_STEP_KIND_BREAKS_GENERAL);
        return check_launch("env_step_dense_kary_kernel");
      }
#define COLO_KARY(NCH)                                                                              \
  case NCH:                                                                                         \
    launch_step(env_step_dense_kary_kernel<TC, NCH, SERVER>, gk, SERVER, share, tb, io, st);        \
    break
      switch (ld / 128) {
        COLO_KARY(1);
        COLO_KARY(2);
        COLO_KARY(3);
        COLO_KARY(4);
        COLO_KARY(5);
        COLO_KARY(6);
        COLO_KARY(7);
        COLO_KARY(8);
      }
#undef COLO_KARY
      count_step_launch(COLO_STEP_KIND_KARY);
      return check_launch("env_step_dense_kary_kernel");
    }
    const int grid = grid_for(kStepThreads / 32, (io.N + tile - 1) / tile);
#define COLO_SHORT(NCH, U)                                                                                        \
  case NCH:                                                                                                       \
    if (tile == 32) launch_step(env_step_dense_short_kernel<TC, NCH, U, 32, SERVER>, grid, SERVER, share, tb, io, st);      \
    else if (tile == 16) launch_step(env_step_dense_short_kernel<TC, NCH, U, 16, SERVER>, grid, SERVER, share, tb, io, st); \
    else launch_step(env_step_dense_short_kernel<TC, NCH, U, 8, SERVER>, grid, SERVER, share, tb, io, st);                  \
    break
    switch (ld / 128) {
      COLO_SHORT(1, 4);
      COLO_SHORT(2, 4);
      COLO_SHORT(3, 4);
      COLO_SHORT(4, 4);
      COLO_SHORT(5, 2);
      COLO_SHORT(6, 2);
      COLO_SHORT(7, 2);
      COLO_SHORT(8, 2);
    }
#undef COLO_SHORT
    count_step_launch(COLO_STEP_KIND_SHORT);
  } else {
    COLO_ARG_CHECK(!io.io_compact, "io_compact needs rows of at most 1024 states");
    const int grid = grid_for(kStepThreads / 32, (io.N + 31) / 32);
    launch_step(env_step_dense_kernel<TC, 8, SERVER>, grid, SERVER, share, tb, io, st);
    count_step_launch(COLO_STEP_KIND_LONG);
  }
  return check_launch("env_step_dense_kernel");
}

template <bool SERVER>
static int launch_succ(const colo_mdp_tables* tb, const StepIO& io, void* stream, int share = 1) {
  COLO_ARG_CHECK(tb->succ_cum && tb->succ_idx && tb->succ_len && tb->Ksucc > 0, "successor tables");
  COLO_ARG_CHECK(io.reward && io.action, "env buffers");
  COLO_ARG_CHECK(!io.io_compact, "io_compact is offered by the dense f32 step only");
  if (io.N == 0) return COLO_OK;
  launch_step(env_step_succ_kernel<SERVER>, grid_for(kStepThreads, io.N), SERVER, share, tb, io, (cudaStream_t)stream);
  count_step_launch(COLO_STEP_KIND_SUCC);
  return check_launch("env_step_succ_kernel");
}

}  // namespace colo

static int make_io(const colo_mdp_tables* tb, const colo_env_batch* b, int random_actions, const void* u_next,
                   const float* u_rew, unsigned long long t, int auto_reset, colo::StepIO* io) {
  COLO_ARG_CHECK(b != nullptr, "batch is NULL");
  memset(io, 0, sizeof(*io));
  if (b->N == 0) return COLO_OK;  // an empty batch has no buffers to check: every entry point returns COLO_OK
  COLO_ARG_CHECK(b->N >= 0 && b->state && b->h && b->step_type && b->obs, "env buffers");
  const int copies = b->visits_copies <= 0 ? 1 : b->visits_copies;
  COLO_ARG_CHECK((copies & (copies - 1)) == 0, "visits_copies must be a power of two");
  io->N = b->N; io->action = b->action; io->random_actions = random_actions; io->u_next = u_next; io->u_rew = u_rew;
  io->seed = b->seed; io->t = t; io->env0 = b->env0; io->auto_reset = auto_reset; io->state = b->state; io->h = b->h;
  io->step_type = b->step_type; io->reward = b->reward; io->obs = b->obs; io->visits_s = b->visits_s;
  io->visits_sa = b->visits_sa; io->visits_mask = copies - 1; io->n_s = tb->S; io->n_sa = (long long)tb->S * tb->A;
  io->status = b->status;
  io->step_type_mirror = b->step_type_mirror;
  io->discount = b->discount;
  io->n_steps = 1;
  io->io_compact = b->io_compact;
  COLO_ARG_CHECK(!b->io_compact || (tb->S <= 32767 && tb->A <= 256), "io_compact needs S <= 32767 and A <= 256");
  return COLO_OK;
}

extern "C" {

int colo_env_reset(const colo_mdp_tables* tb, const colo_env_batch* batch, const double* u_next,
                   unsigned long long t, void* stream) {
  int r = colo::check_tables_common(tb);
  if (r != COLO_OK) return r;
  colo::StepIO io;
  r = make_io(tb, batch, 0, u_next, nullptr, t, 0, &io);
  if (r != COLO_OK || io.N == 0) return r;
  const int grid = colo::grid_for(colo::kStepThreads, io.N);
  colo::env_reset_kernel<<<grid, colo::kStepThreads, 0, (cudaStream_t)stream>>>(*tb, io);
  return colo::check_launch("env_reset_kernel");
}

int colo_env_step_dense_f32(const colo_mdp_tables* tb, const colo_env_batch* batch, int random_actions,
                            const float* u_next, const float* u_rew, unsigned long long t, int auto_reset,
                            void* stream) {
  int r = colo::check_tables_common(tb);
  if (r != COLO_OK) return r;
  colo::StepIO io;
  r = make_io(tb, batch, random_actions, u_next, u_rew, t, auto_reset, &io);
  if (r != COLO_OK || io.N == 0) return r;
  return colo::launch_dense<float, false>(tb, io, stream);
}

int colo_env_step_dense_f64(const colo_mdp_tables* tb, const colo_env_batch* batch, int random_actions,
                            const double* u_next, const float* u_rew, unsigned long long t, int auto_reset,
                            void* stream) {
  int r = colo::check_tables_common(tb);
  if (r != COLO_OK) return r;
  colo::StepIO io;
  r = make_io(tb, batch, random_actions, u_next, u_rew, t, auto_reset, &io);
  if (r != COLO_OK || io.N == 0) return r;
  return colo::launch_dense<double, false>(tb, io, stream);
}

int colo_env_step_succ(const colo_mdp_tables* tb, const colo_env_batch* batch, int random_actions,
                       const double* u_next, const float* u_rew, unsigned long long t, int auto_reset,
                       void* stream) {
  int r = colo::check_tables_common(tb);
  if (r != COLO_OK) return r;
  colo::StepIO io;
  r = make_io(tb, batch, random_actions, u_next, u_rew, t, auto_reset, &io);
  if (r != COLO_OK || io.N == 0) return r;
  return colo::launch_succ<false>(tb, io, stream);
}

int colo_env_random_steps(const colo_mdp_tables* tb, const colo_env_batch* batch, int mode, int n_steps,
                          unsigned long long t0, int auto_reset, void* stream) {
  int r = colo::check_tables_common(tb);
  if (r != COLO_OK) return r;
  COLO_ARG_CHECK(n_steps >= 1 && mode >= 0 && mode <= 2, "n_steps >= 1, mode in {0,1,2}");
  colo::StepIO io;
  r = make_io(tb, batch, 1, nullptr, nullptr, t0, auto_reset, &io);
  if (r != COLO_OK || io.N == 0) return r;
  io.n_steps = n_steps;
  if (mode == 0) return colo::launch_dense<float, false>(tb, io, stream);
  if (mode == 1) return colo::launch_dense<double, false>(tb, io, stream);
  return colo::launch_succ<false>(tb, io, stream);
}

// ---- mixed batches ------------------------------------------------------------------------------------------------------
static int mixed_check_instance(const colo_mdp_tables* tb, int mode) {
  int r = colo::check_tables_common(tb);
  if (r != COLO_OK) return r;
  if (mode == 2) {
    COLO_ARG_CHECK(tb->succ_cum && tb->succ_idx && tb->succ_len && tb->Ksucc > 0, "successor tables");
  } else {
    COLO_ARG_CHECK(tb->cdf && tb->ld >= tb->S && tb->ld % 4 == 0, "dense cdf with ld % 4 == 0 is required");
    COLO_ARG_CHECK((uintptr_t)tb->cdf % 16 == 0, "cdf must be 16-byte aligned");
  }
  return COLO_OK;
}

void colo_mixed_tables_destroy(colo_mixed_tables* h) {
  if (!h) return;
  if (h->insts) cudaFree(h->insts);
  if (h->inst_of) cudaFree(h->inst_of);
  free(h->host_insts);
  free(h);
}

int colo_mixed_tables_create(const colo_mdp_tables* host_tables, int n_inst, const long long* n_envs,
                             const unsigned long long* seeds, int mode, void* stream, colo_mixed_tables** out) {
  COLO_ARG_CHECK(out && host_tables && n_envs && seeds, "host_tables, n_envs, seeds, out");
  COLO_ARG_CHECK(n_inst >= 1, "colo_mixed_tables_create: n_inst >= 1");
  COLO_ARG_CHECK(mode >= 0 && mode <= 2, "mode in {0,1,2}");
  // every instance is validated before anything touches the device
  std::vector<colo::MixedInst> insts((size_t)n_inst);
  long long N = 0, sum_s = 0, sum_sa = 0;
  for (int i = 0; i < n_inst; ++i) {
    if (mixed_check_instance(&host_tables[i], mode) != COLO_OK) {
      char why[256];
      snprintf(why, sizeof(why), "%s", colo_last_error());
      colo::set_error("colo_mixed_tables_create: instance %d: %s", i, why);
      return COLO_ERR_ARG;
    }
    if (n_envs[i] < 1) {
      colo::set_error("colo_mixed_tables_create: instance %d: n_envs %lld < 1", i, n_envs[i]);
      return COLO_ERR_ARG;
    }
    colo::MixedInst& d = insts[(size_t)i];
    d.tb = host_tables[i];
    d.seed = seeds[i];
    d.start = N;
    d.off_s = sum_s;
    d.off_sa = sum_sa;
    N += n_envs[i];
    sum_s += host_tables[i].S;
    sum_sa += (long long)host_tables[i].S * host_tables[i].A;
  }
  COLO_ARG_CHECK(N < (1LL << 31), "colo_mixed_tables_create: fewer than 2^31 envs in all");
  std::vector<int> inst_of((size_t)N);
  for (int i = 0; i < n_inst; ++i)
    for (long long e = insts[(size_t)i].start; e < insts[(size_t)i].start + n_envs[i]; ++e) inst_of[(size_t)e] = i;
  colo_mixed_tables* h = (colo_mixed_tables*)calloc(1, sizeof(colo_mixed_tables));
  COLO_ARG_CHECK(h != nullptr, "out of host memory");
  h->n_inst = n_inst;
  h->mode = mode;
  h->N = N;
  h->sum_s = sum_s;
  h->sum_sa = sum_sa;
  h->host_insts = (colo::MixedInst*)malloc(sizeof(colo::MixedInst) * (size_t)n_inst);
  if (h->host_insts == nullptr) {
    colo_mixed_tables_destroy(h);
    COLO_ARG_CHECK(false, "out of host memory");
  }
  memcpy(h->host_insts, insts.data(), sizeof(colo::MixedInst) * (size_t)n_inst);
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMalloc((void**)&h->insts, sizeof(colo::MixedInst) * (size_t)n_inst);
  if (e == cudaSuccess) e = cudaMalloc((void**)&h->inst_of, sizeof(int) * (size_t)N);
  if (e == cudaSuccess)
    e = cudaMemcpyAsync(h->insts, insts.data(), sizeof(colo::MixedInst) * (size_t)n_inst, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(h->inst_of, inst_of.data(), sizeof(int) * (size_t)N, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);  // the host staging vectors die with this call
  if (e != cudaSuccess) {
    colo::set_error("colo_mixed_tables_create: %s", cudaGetErrorString(e));
    colo_mixed_tables_destroy(h);
    return COLO_ERR_CUDA;
  }
  *out = h;
  return COLO_OK;
}

long long colo_mixed_visits_size(const colo_mixed_tables* h, int pairs) {
  return h == nullptr ? 0 : (pairs ? h->sum_sa : h->sum_s);
}

static int make_mixed_io(const colo_mixed_tables* h, const colo_env_batch* b, int random_actions, const void* u_next,
                         const float* u_rew, unsigned long long t, int auto_reset, colo::StepIO* io) {
  COLO_ARG_CHECK(h != nullptr && b != nullptr, "mixed tables, batch");
  if (b->N != h->N) {
    colo::set_error("bad argument: batch N = %lld, the mixed tables hold %lld envs", b->N, h->N);
    return COLO_ERR_ARG;
  }
  COLO_ARG_CHECK(!b->io_compact, "mixed batches have no compact I/O");
  colo_mdp_tables shape;
  memset(&shape, 0, sizeof(shape));
  shape.S = shape.A = 1;
  const int r = make_io(&shape, b, random_actions, u_next, u_rew, t, auto_reset, io);
  if (r != COLO_OK) return r;
  io->n_s = h->sum_s;  // counter rows are the concatenation of the instances' rows
  io->n_sa = h->sum_sa;
  io->seed = io->env0 = 0;  // every env takes its key and counter from its instance
  return COLO_OK;
}

int colo_mixed_env_reset(const colo_mixed_tables* h, const colo_env_batch* batch, const double* u_next,
                         unsigned long long t, void* stream) {
  colo::StepIO io;
  const int r = make_mixed_io(h, batch, 0, u_next, nullptr, t, 0, &io);
  if (r != COLO_OK) return r;
  colo::env_reset_mixed_kernel<<<colo::grid_for(colo::kStepThreads, io.N), colo::kStepThreads, 0, (cudaStream_t)stream>>>(
      h->insts, h->inst_of, io);
  return colo::check_launch("env_reset_mixed_kernel");
}

static int launch_mixed(const colo_mixed_tables* h, const colo::StepIO& io, void* stream) {
  COLO_ARG_CHECK(io.reward && io.action, "env buffers");
  cudaStream_t st = (cudaStream_t)stream;
  if (h->mode == 2) {
    colo::env_step_succ_mixed_kernel<<<colo::grid_for(colo::kStepThreads, io.N), colo::kStepThreads, 0, st>>>(
        h->insts, h->inst_of, io);
    colo::count_step_launch(COLO_STEP_KIND_MIXED_SUCC);
    return colo::check_launch("env_step_succ_mixed_kernel");
  }
  const int grid = colo::grid_for(colo::kStepThreads / 32, (io.N + 31) / 32);
  if (h->mode == 0)
    colo::env_step_dense_mixed_kernel<float, 8><<<grid, colo::kStepThreads, 0, st>>>(h->insts, h->inst_of, io);
  else
    colo::env_step_dense_mixed_kernel<double, 8><<<grid, colo::kStepThreads, 0, st>>>(h->insts, h->inst_of, io);
  colo::count_step_launch(COLO_STEP_KIND_MIXED_DENSE);
  return colo::check_launch("env_step_dense_mixed_kernel");
}

int colo_mixed_env_step(const colo_mixed_tables* h, const colo_env_batch* batch, int random_actions,
                        const void* u_next, const float* u_rew, unsigned long long t, int auto_reset, void* stream) {
  colo::StepIO io;
  const int r = make_mixed_io(h, batch, random_actions, u_next, u_rew, t, auto_reset, &io);
  if (r != COLO_OK) return r;
  return launch_mixed(h, io, stream);
}

int colo_mixed_env_random_steps(const colo_mixed_tables* h, const colo_env_batch* batch, int n_steps,
                                unsigned long long t0, int auto_reset, void* stream) {
  COLO_ARG_CHECK(n_steps >= 1, "n_steps >= 1");
  colo::StepIO io;
  const int r = make_mixed_io(h, batch, 1, nullptr, nullptr, t0, auto_reset, &io);
  if (r != COLO_OK) return r;
  io.n_steps = n_steps;
  return launch_mixed(h, io, stream);
}

struct colo_env_stepper {
  colo_mdp_tables tb;
  colo::StepIO io;
  int mode;
  void* stream;
};

int colo_env_stepper_create(const colo_mdp_tables* tb, const colo_env_batch* batch, int mode, void* stream,
                            colo_env_stepper** out) {
  int r = colo::check_tables_common(tb);
  if (r != COLO_OK) return r;
  COLO_ARG_CHECK(out && mode >= 0 && mode <= 2, "out, mode in {0,1,2}");
  colo_env_stepper* h = (colo_env_stepper*)malloc(sizeof(colo_env_stepper));
  COLO_ARG_CHECK(h != nullptr, "out of host memory");
  h->tb = *tb;
  r = make_io(tb, batch, 0, nullptr, nullptr, 0, 1, &h->io);
  if (r != COLO_OK) {
    free(h);
    return r;
  }
  h->mode = mode;
  h->stream = stream;
  *out = h;
  return COLO_OK;
}

int colo_env_stepper_launch(colo_env_stepper* h, const int* action, unsigned long long t) {
  if (h->io.N == 0) return COLO_OK;
  h->io.action = const_cast<int*>(action);
  h->io.t = t;
  if (h->mode == 0) return colo::launch_dense<float, false>(&h->tb, h->io, h->stream);
  if (h->mode == 1) return colo::launch_dense<double, false>(&h->tb, h->io, h->stream);
  return colo::launch_succ<false>(&h->tb, h->io, h->stream);
}

void colo_env_stepper_destroy(colo_env_stepper* h) { free(h); }

int colo_env_pipeline_run(colo_env_stepper* const* steppers, int n_groups, const int* const* action_ring, int ring,
                          unsigned long long t0, int n_steps, colo_env_pipeline_callback on_timestep, void* user) {
  COLO_ARG_CHECK(steppers && action_ring && n_groups >= 1 && ring >= 1 && n_steps >= 1, "steppers, action_ring, n_groups, ring, n_steps");
  // software pipeline over the groups: while the host handles group g's TimeStep the other groups' kernels are on PCIe
  for (int g = 0; g < n_groups; ++g) {
    const int r = colo_env_stepper_launch(steppers[g], action_ring[(size_t)0 * n_groups + g], t0);
    if (r != COLO_OK) return r;
  }
  for (int i = 1; i <= n_steps; ++i)
    for (int g = 0; g < n_groups; ++g) {
      COLO_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)steppers[g]->stream));  // step i-1 of group g is in host memory
      if (on_timestep) on_timestep(user, g, i - 1);
      if (i < n_steps) {
        const int r = colo_env_stepper_launch(steppers[g], action_ring[(size_t)(i % ring) * n_groups + g], t0 + (unsigned long long)i);
        if (r != COLO_OK) return r;
      }
    }
  return COLO_OK;
}


// One host thread per group: every group runs its own recv / send loop (stream sync, on_timestep, launch), so a group's
// cycle -- launch latency, PCIe reads and writes of the kernel, completion latency -- overlaps with every other group's
// instead of being stepped through by one thread.  Per-group order of events and TimeSteps are those of
// colo_env_pipeline_run; on_timestep is called on the group's own thread, concurrently for different groups.
int colo_env_pipeline_run_threads(colo_env_stepper* const* steppers, int n_groups, const int* const* action_ring, int ring,
                                  unsigned long long t0, int n_steps, colo_env_pipeline_callback on_timestep, void* user) {
  COLO_ARG_CHECK(steppers && action_ring && n_groups >= 1 && ring >= 1 && n_steps >= 1, "steppers, action_ring, n_groups, ring, n_steps");
  int dev = 0;
  COLO_CUDA_TRY(cudaGetDevice(&dev));
  std::vector<int> rcs((size_t)n_groups, COLO_OK);
  auto group_loop = [&](int g) {
    if (cudaSetDevice(dev) != cudaSuccess) {
      rcs[g] = COLO_ERR_CUDA;
      return;
    }
    int r = colo_env_stepper_launch(steppers[g], action_ring[g], t0);
    for (int i = 1; i <= n_steps && r == COLO_OK; ++i) {
      if (cudaStreamSynchronize((cudaStream_t)steppers[g]->stream) != cudaSuccess) {
        r = COLO_ERR_CUDA;
        break;
      }
      if (on_timestep) on_timestep(user, g, i - 1);
      if (i < n_steps) r = colo_env_stepper_launch(steppers[g], action_ring[(size_t)(i % ring) * n_groups + g], t0 + (unsigned long long)i);
    }
    rcs[g] = r;
  };
  std::vector<std::thread> workers;
  for (int g = 1; g < n_groups; ++g) workers.emplace_back(group_loop, g);
  group_loop(0);
  for (auto& w : workers) w.join();
  for (int g = 0; g < n_groups; ++g)
    if (rcs[g] != COLO_OK) {
      colo::set_error("colo_env_pipeline_run_threads: group %d failed (status %d)", g, rcs[g]);
      return rcs[g];
    }
  return COLO_OK;
}

// ---- queued pipeline ---------------------------------------------------------------------------------------------------
// colo_env_pipeline_run pays a stream synchronisation and a launch on the host for every group-step (~10 us per
// group-step: the measured bound of the end-to-end step).  Here the per-step handshake is two words in pinned host memory
// and the GPU's own front end does the waiting: every group's stream holds, for step i,
//     wait32(go[g] == i % L + 1)  ->  step kernel  ->  write32(done[g] = i % L + 1)
// (stream memory operations, cuStreamWaitValue32 / cuStreamWriteValue32), enqueued AHEAD of time -- as replays of one
// CUDA graph of L steps per group when graphs are on, or one triple at a time during the host's waits.  In the steady
// state a group-step costs the host one flag store and one flag poll; no CUDA call is on the critical path.
constexpr int kMaxPipelineGroups = 8;
constexpr int kFlagStride = 32;  // u32 words between flags: go[g] and done[g] on their own 128-byte lines

typedef CUresult (*colo_stream_value32_fn)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
struct StreamMemOps {
  colo_stream_value32_fn wait32 = nullptr, write32 = nullptr;
};
static const StreamMemOps& stream_mem_ops() {
  // resolved through the runtime: the library carries no link dependency on libcuda (it must load on a CPU-only box)
  static const StreamMemOps ops = [] {
    StreamMemOps r;
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuStreamWaitValue32", &f, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      r.wait32 = (colo_stream_value32_fn)f;
    f = nullptr;
    if (cudaGetDriverEntryPoint("cuStreamWriteValue32", &f, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      r.write32 = (colo_stream_value32_fn)f;
    (void)cudaGetLastError();
    return r;
  }();
  return ops;
}

struct colo_env_pipeline {
  int G;
  colo_env_stepper* steppers[kMaxPipelineGroups];  // borrowed
  cudaStream_t streams[kMaxPipelineGroups];        // own non-blocking streams: nothing else may ever wait behind a flag
  unsigned* flags;                                 // pinned host: go[g] = flags[(2g) * kFlagStride], done[g] = flags[(2g+1) * kFlagStride]
  unsigned long long* t_dev;                       // device: one Philox step-counter base per group (graph replays)
  // one instantiated graph of L steps per group, valid for one action ring
  int L, ring;
  const int** ring_ptrs;
  cudaGraphExec_t exec[kMaxPipelineGroups];
  int graphs_failed;
};

static volatile unsigned* pl_go(colo_env_pipeline* p, int g) { return p->flags + (size_t)(2 * g) * kFlagStride; }
static volatile unsigned* pl_done(colo_env_pipeline* p, int g) { return p->flags + (size_t)(2 * g + 1) * kFlagStride; }

static int pl_launch(colo_env_pipeline* p, int g, const int* action, unsigned long long t, const unsigned long long* t_dev) {
  colo_env_stepper* h = p->steppers[g];
  colo::StepIO io = h->io;
  io.action = const_cast<int*>(action);
  io.t = t;
  io.t_dev = t_dev;
  if (h->mode == 0) return colo::launch_dense<float, false>(&h->tb, io, p->streams[g]);
  if (h->mode == 1) return colo::launch_dense<double, false>(&h->tb, io, p->streams[g]);
  return colo::launch_succ<false>(&h->tb, io, p->streams[g]);
}

#define COLO_CU_TRY(expr)                                                               \
  do {                                                                                  \
    CUresult _r = (expr);                                                               \
    if (_r != CUDA_SUCCESS) {                                                           \
      colo::set_error("%s failed: CUresult %d (%s:%d)", #expr, (int)_r, __FILE__, __LINE__); \
      return COLO_ERR_CUDA;                                                             \
    }                                                                                   \
  } while (0)

// wait(go == v) -> step kernel -> write(done = v) on group g's stream
static int pl_enqueue_step(colo_env_pipeline* p, int g, unsigned v, const int* action, unsigned long long t,
                           const unsigned long long* t_dev) {
  const StreamMemOps& mo = stream_mem_ops();
  COLO_CU_TRY(mo.wait32((CUstream)p->streams[g], (CUdeviceptr)(uintptr_t)pl_go(p, g), v, CU_STREAM_WAIT_VALUE_EQ));
  const int r = pl_launch(p, g, action, t, t_dev);
  if (r != COLO_OK) return r;
  COLO_CU_TRY(mo.write32((CUstream)p->streams[g], (CUdeviceptr)(uintptr_t)pl_done(p, g), v, CU_STREAM_WRITE_VALUE_DEFAULT));
  return COLO_OK;
}

static void pl_drop_graphs(colo_env_pipeline* p) {
  for (int g = 0; g < p->G; ++g)
    if (p->exec[g]) {
      cudaGraphExecDestroy(p->exec[g]);
      p->exec[g] = nullptr;
    }
  free(p->ring_ptrs);
  p->ring_ptrs = nullptr;
  p->L = p->ring = 0;
}

// L steps of every group as one graph per group (stream capture of the same triples); the kernels read the step counter
// as j + *t_dev, the action pointers repeat with period `ring` (L is a multiple of it)
static int pl_build_graphs(colo_env_pipeline* p, const int* const* action_ring, int ring) {
  const size_t n = (size_t)ring * p->G;
  if (p->exec[0] && p->ring == ring && memcmp(p->ring_ptrs, action_ring, n * sizeof(int*)) == 0) return COLO_OK;
  pl_drop_graphs(p);
  if (ring > 256) return COLO_ERR_ARG;  // a graph of a multiple of `ring` steps would be unreasonably long
  const int L = ring * ((64 + ring - 1) / ring) < 2 ? 2 : ring * ((64 + ring - 1) / ring);
  for (int g = 0; g < p->G; ++g) {
    COLO_CUDA_TRY(cudaStreamBeginCapture(p->streams[g], cudaStreamCaptureModeRelaxed));
    int r = COLO_OK;
    for (int j = 0; j < L && r == COLO_OK; ++j)
      r = pl_enqueue_step(p, g, (unsigned)j + 1, action_ring[(size_t)(j % ring) * p->G + g], (unsigned long long)j, p->t_dev + g);
    cudaGraph_t graph = nullptr;
    const cudaError_t e = cudaStreamEndCapture(p->streams[g], &graph);
    if (r == COLO_OK && e == cudaSuccess && graph) {
      if (cudaGraphInstantiate(&p->exec[g], graph, 0) != cudaSuccess) r = COLO_ERR_CUDA;
    } else if (r == COLO_OK) {
      r = COLO_ERR_CUDA;
    }
    if (graph) cudaGraphDestroy(graph);
    if (r != COLO_OK) {
      (void)cudaGetLastError();
      pl_drop_graphs(p);
      return r;
    }
  }
  p->ring_ptrs = (const int**)malloc(n * sizeof(int*));
  memcpy(p->ring_ptrs, action_ring, n * sizeof(int*));
  p->L = L;
  p->ring = ring;
  return COLO_OK;
}

int colo_env_pipeline_create(colo_env_stepper* const* steppers, int n_groups, colo_env_pipeline** out) {
  COLO_ARG_CHECK(steppers && out && n_groups >= 1 && n_groups <= kMaxPipelineGroups, "steppers, out, 1 <= n_groups <= 8");
  const StreamMemOps& mo = stream_mem_ops();
  if (!mo.wait32 || !mo.write32) {
    colo::set_error("colo_env_pipeline_create: the driver does not offer cuStreamWaitValue32 / cuStreamWriteValue32");
    return COLO_ERR_CUDA;
  }
  colo_env_pipeline* p = (colo_env_pipeline*)calloc(1, sizeof(colo_env_pipeline));
  COLO_ARG_CHECK(p != nullptr, "out of host memory");
  p->G = n_groups;
  for (int g = 0; g < n_groups; ++g) p->steppers[g] = steppers[g];
  cudaError_t e = cudaHostAlloc((void**)&p->flags, (size_t)2 * n_groups * kFlagStride * sizeof(unsigned), cudaHostAllocPortable);
  if (e == cudaSuccess) e = cudaMalloc((void**)&p->t_dev, sizeof(unsigned long long) * 2 * n_groups);
  for (int g = 0; g < n_groups && e == cudaSuccess; ++g) e = cudaStreamCreateWithFlags(&p->streams[g], cudaStreamNonBlocking);
  if (e != cudaSuccess) {
    colo::set_error("colo_env_pipeline_create: %s", cudaGetErrorString(e));
    colo_env_pipeline_destroy(p);
    return COLO_ERR_CUDA;
  }
  memset(p->flags, 0, (size_t)2 * n_groups * kFlagStride * sizeof(unsigned));
  *out = p;
  return COLO_OK;
}

void colo_env_pipeline_destroy(colo_env_pipeline* p) {
  if (!p) return;
  pl_drop_graphs(p);
  for (int g = 0; g < p->G; ++g)
    if (p->streams[g]) cudaStreamDestroy(p->streams[g]);
  if (p->t_dev) cudaFree(p->t_dev);
  if (p->flags) cudaFreeHost(p->flags);
  free(p);
}

int colo_env_pipeline_run_queued(colo_env_pipeline* p, const int* const* action_ring, int ring, unsigned long long t0,
                                 int n_steps, colo_env_pipeline_callback on_timestep, void* user, int use_graph) {
  COLO_ARG_CHECK(p && action_ring && ring >= 1 && n_steps >= 1, "pipeline, action_ring, ring, n_steps");
  const int G = p->G;
  const StreamMemOps& mo = stream_mem_ops();
  // whatever was enqueued on the groups' own streams (reset, earlier steps) comes first
  for (int g = 0; g < G; ++g) COLO_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)p->steppers[g]->stream));
  if (use_graph && !p->graphs_failed && n_steps >= 2 * 64) {
    if (pl_build_graphs(p, action_ring, ring) != COLO_OK) p->graphs_failed = 1;  // the triples still work one at a time
  }
  const bool graphs = use_graph && !p->graphs_failed && p->exec[0] != nullptr && n_steps >= p->L;
  const int L = graphs ? p->L : (1 << 30);  // flag values are i % L + 1
  const int lead = graphs ? L / 2 + 1 : 3;  // group-steps kept enqueued ahead of the newest finished one
  for (int g = 0; g < G; ++g) {
    *pl_go(p, g) = 0;
    *pl_done(p, g) = 0;
  }
  __atomic_thread_fence(__ATOMIC_SEQ_CST);
  int enq[kMaxPipelineGroups] = {0}, fin[kMaxPipelineGroups] = {0};
  int rc = COLO_OK;
  auto top_up = [&](int g) -> int {
    while (enq[g] < n_steps && enq[g] - fin[g] < lead) {
      const int i = enq[g];
      if (graphs && i % L == 0 && n_steps - i >= L) {
        const unsigned long long base = t0 + (unsigned long long)i;
        unsigned* td = reinterpret_cast<unsigned*>(p->t_dev + g);
        COLO_CU_TRY(mo.write32((CUstream)p->streams[g], (CUdeviceptr)(uintptr_t)td, (unsigned)base, CU_STREAM_WRITE_VALUE_DEFAULT));
        COLO_CU_TRY(mo.write32((CUstream)p->streams[g], (CUdeviceptr)(uintptr_t)(td + 1), (unsigned)(base >> 32), CU_STREAM_WRITE_VALUE_DEFAULT));
        COLO_CUDA_TRY(cudaGraphLaunch(p->exec[g], p->streams[g]));
        colo::count_launch((unsigned long long)L);
        enq[g] += L;
      } else {
        const int r = pl_enqueue_step(p, g, (unsigned)(i % L) + 1, action_ring[(size_t)(i % ring) * G + g],
                                      t0 + (unsigned long long)i, nullptr);
        if (r != COLO_OK) return r;
        enq[g] += 1;
      }
    }
    return COLO_OK;
  };
  for (int g = 0; g < G && rc == COLO_OK; ++g) rc = top_up(g);
  if (rc == COLO_OK)
    for (int g = 0; g < G; ++g) __atomic_store_n(const_cast<unsigned*>(pl_go(p, g)), 1u, __ATOMIC_RELEASE);  // step 0's actions are in place
  bool stuck = false;
  for (int i = 1; i <= n_steps && rc == COLO_OK && !stuck; ++i)
    for (int g = 0; g < G; ++g) {
      const unsigned want = (unsigned)((i - 1) % L) + 1;
      unsigned long long spins = 0;
      struct timespec w0 = {0, 0};
      while (__atomic_load_n(const_cast<unsigned*>(pl_done(p, g)), __ATOMIC_ACQUIRE) != want) {
        if ((++spins & 0xffff) == 0) {  // look at the clock every 65,536 polls only
          struct timespec now;
          clock_gettime(CLOCK_MONOTONIC, &now);
          if (w0.tv_sec == 0 && w0.tv_nsec == 0) w0 = now;
          if ((now.tv_sec - w0.tv_sec) + (now.tv_nsec - w0.tv_nsec) * 1e-9 > 10.0) {
            stuck = true;
            break;
          }
        }
      }
      if (stuck) break;
      fin[g] = i;  // step i-1 of group g is in host memory
      if ((rc = top_up(g)) != COLO_OK) break;
      if (on_timestep) on_timestep(user, g, i - 1);
      if (i < n_steps) __atomic_store_n(const_cast<unsigned*>(pl_go(p, g)), (unsigned)(i % L) + 1, __ATOMIC_RELEASE);
    }
  if (stuck || rc != COLO_OK) {
    // never leave a stream blocked behind a flag: feed every group the values it waits for until the queues are empty
    // (the steps run with whatever actions are in the ring; the call reports the failure)
    struct timespec d0;
    clock_gettime(CLOCK_MONOTONIC, &d0);
    for (;;) {
      bool idle = true;
      for (int g = 0; g < G; ++g) {
        if (cudaStreamQuery(p->streams[g]) == cudaSuccess) continue;
        idle = false;
        const unsigned v = __atomic_load_n(const_cast<unsigned*>(pl_done(p, g)), __ATOMIC_ACQUIRE);
        __atomic_store_n(const_cast<unsigned*>(pl_go(p, g)), v % (unsigned)L + 1, __ATOMIC_RELEASE);
      }
      struct timespec now;
      clock_gettime(CLOCK_MONOTONIC, &now);
      if (idle || (now.tv_sec - d0.tv_sec) > 20) break;
    }
    (void)cudaGetLastError();
    if (stuck) {
      colo::set_error("colo_env_pipeline_run_queued: no progress for 10 s (streams sharing a hardware queue?); drained");
      return COLO_ERR_CUDA;
    }
    return rc;
  }
  for (int g = 0; g < G; ++g) COLO_CUDA_TRY(cudaStreamSynchronize(p->streams[g]));
  return COLO_OK;
}

int colo_env_server_start(const colo_mdp_tables* tb, const colo_env_batch* batch, const colo_env_server* srv, int mode,
                          unsigned long long t, unsigned long long served, void* stream) {
  int r = colo::check_tables_common(tb);
  if (r != COLO_OK) return r;
  COLO_ARG_CHECK(srv && srv->doorbell_host && srv->done_host && srv->ctl_dev, "server control words");
  COLO_ARG_CHECK(mode >= 0 && mode <= 2 && srv->share >= 1 && srv->idle_timeout_ms > 0, "mode, share, idle_timeout_ms");
  colo::StepIO io;
  r = make_io(tb, batch, 0, nullptr, nullptr, t, 1, &io);
  if (r != COLO_OK) return r;
  COLO_ARG_CHECK(io.N > 0, "a served batch cannot be empty");
  // `served` steps are finished; the doorbell may already hold served + 1 (a step posted while the last server lapsed)
  const unsigned long long seq = served;
  const unsigned long long bell = *(volatile unsigned long long*)srv->doorbell_host;
  COLO_ARG_CHECK(bell == seq || bell == seq + 1, "doorbell must hold `served` or `served + 1`");
  __atomic_store_n(srv->done_host, seq, __ATOMIC_SEQ_CST);
  io.srv_doorbell = srv->doorbell_host;
  io.srv_done = srv->done_host;
  io.srv_go = srv->ctl_dev;
  io.srv_arrive = srv->ctl_dev + 1;
  io.srv_seq0 = seq;
  io.srv_idle_ns = (unsigned long long)srv->idle_timeout_ms * 1000000ULL;
  cudaStream_t st = (cudaStream_t)stream;
  // go = seq (nothing pending), arrive = 0: written on the launch stream ahead of the kernel
  const unsigned long long init[2] = {seq, 0ULL};
  COLO_CUDA_TRY(cudaMemcpyAsync(srv->ctl_dev, init, sizeof(init), cudaMemcpyHostToDevice, st));
  if (mode == 0) return colo::launch_dense<float, true>(tb, io, stream, srv->share);
  if (mode == 1) return colo::launch_dense<double, true>(tb, io, stream, srv->share);
  return colo::launch_succ<true>(tb, io, stream, srv->share);
}

unsigned long long colo_env_server_post(const colo_env_server* srv) {
  // the caller finished writing the actions: publish them with the doorbell
  unsigned long long* d = srv->doorbell_host;
  const unsigned long long next = *d + 1;
  __atomic_store_n(d, next, __ATOMIC_SEQ_CST);
  return next;
}

int colo_env_server_wait(const colo_env_server* srv, unsigned long long step_index, unsigned timeout_ms) {
  const unsigned long long* done = srv->done_host;
  unsigned long long spins = 0;
  struct timespec t0 = {0, 0};
  for (;;) {
    const unsigned long long v = __atomic_load_n(done, __ATOMIC_ACQUIRE);
    if (v == colo::kSrvLapsed) return COLO_SERVER_LAPSED;
    if (v >= step_index) return COLO_OK;
    if ((++spins & 0xfff) == 0) {  // look at the clock every 4096 polls only
      struct timespec now;
      clock_gettime(CLOCK_MONOTONIC, &now);
      if (t0.tv_sec == 0 && t0.tv_nsec == 0) t0 = now;
      const double ms = (now.tv_sec - t0.tv_sec) * 1e3 + (now.tv_nsec - t0.tv_nsec) * 1e-6;
      if (ms > (double)timeout_ms) {
        colo::set_error("colo_env_server_wait: step %llu not finished after %u ms (done = %llu)", step_index, timeout_ms, v);
        return COLO_ERR_CUDA;
      }
    }
  }
}

int colo_env_server_stop(const colo_env_server* srv, void* stream) {
  COLO_ARG_CHECK(srv && srv->doorbell_host, "server control words");
  unsigned long long* d = srv->doorbell_host;
  const unsigned long long seq = *d;
  __atomic_store_n(d, colo::kSrvExit, __ATOMIC_SEQ_CST);
  const cudaError_t e = cudaStreamSynchronize((cudaStream_t)stream);
  __atomic_store_n(d, seq, __ATOMIC_SEQ_CST);  // the step count survives for the next start
  if (e != cudaSuccess) {
    colo::set_error("colo_env_server_stop: %s", cudaGetErrorString(e));
    return COLO_ERR_CUDA;
  }
  return COLO_OK;
}

unsigned long long colo_step_kernel_launches(int kind) {
  return kind >= 0 && kind < COLO_STEP_KINDS ? colo::g_step_launches[kind].load(std::memory_order_relaxed) : 0ULL;
}

int colo_emit_observations(const float* table, const int* state, const int* h, const unsigned char* step_type,
                           long long N, int H, int S, int D, float* out, void* stream) {
  COLO_ARG_CHECK(table && state && h && step_type && out && N >= 0 && H >= 0 && S > 0 && D > 0, "emit_observations");
  if (N == 0) return COLO_OK;
  const long long blocks = (N + 7) / 8;
  const long long cap = (long long)colo::sm_count() * 16;
  colo::emit_observations_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, (cudaStream_t)stream>>>(table, state, h, step_type,
                                                                                                       N, H, S, D, out);
  return colo::check_launch("emit_observations_kernel");
}

int colo_build_cdf_index(const void* cdf, int S, int A, int ld, int is_f64, void* cdf_mid, void* cdf_coarse,
                         void* stream) {
  COLO_ARG_CHECK(cdf && cdf_mid && cdf_coarse && S > 0 && A > 0 && ld >= S && ld % 128 == 0 && ld <= 1024,
                 "cdf, cdf_mid, cdf_coarse, ld % 128 == 0, ld <= 1024");
  const long long rows = (long long)S * A;
  const long long blocks = (rows * (ld / 4) + 255) / 256;
  const int grid = (int)(blocks < 65535 ? blocks : 65535);
  if (is_f64)
    colo::build_cdf_index_kernel<double><<<grid, 256, 0, (cudaStream_t)stream>>>((const double*)cdf, rows, ld, (double*)cdf_mid,
                                                                              (double*)cdf_coarse);
  else
    colo::build_cdf_index_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>((const float*)cdf, rows, ld, (float*)cdf_mid,
                                                                             (float*)cdf_coarse);
  return colo::check_launch("build_cdf_index_kernel");
}

int colo_count_cdf_breaks(const float* cdf, int S, int A, int ld, int* max_breaks, void* stream) {
  COLO_ARG_CHECK(cdf && max_breaks && S > 0 && A > 0 && ld >= S, "cdf, max_breaks, S, A, ld");
  cudaStream_t st = (cudaStream_t)stream;
  const long long rows = (long long)S * A;
  int* d = nullptr;
  COLO_CUDA_TRY(cudaMalloc((void**)&d, sizeof(int)));
  cudaError_t e = cudaMemsetAsync(d, 0, sizeof(int), st);
  if (e == cudaSuccess) {
    colo::count_cdf_breaks_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, st>>>(cdf, rows, S, ld, d);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(max_breaks, d, sizeof(int), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaFree(d);
  if (e != cudaSuccess) {
    colo::set_error("colo_count_cdf_breaks: %s", cudaGetErrorString(e));
    return COLO_ERR_CUDA;
  }
  return COLO_OK;
}

int colo_build_cdf_breaks(const colo_mdp_tables* tb, int k, void* cdf_breaks, void* stream) {
  int r = colo::check_tables_common(tb);
  if (r != COLO_OK) return r;
  COLO_ARG_CHECK(tb->cdf && tb->ld >= tb->S && cdf_breaks && (uintptr_t)cdf_breaks % 16 == 0,
                 "f32 cdf and a 16-byte aligned cdf_breaks");
  COLO_ARG_CHECK(k == 2 || k == 4 || k == 8 || k == 16, "k must be 2, 4, 8 or 16");
  cudaStream_t st = (cudaStream_t)stream;
  const long long rows = (long long)tb->S * tb->A;
  int* d = nullptr;
  int err = 0;
  COLO_CUDA_TRY(cudaMalloc((void**)&d, sizeof(int)));
  cudaError_t e = cudaMemsetAsync(d, 0, sizeof(int), st);
  if (e == cudaSuccess) {
    colo::build_cdf_breaks_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, st>>>(*tb, k, (colo::CdfBreak*)cdf_breaks, d);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(&err, d, sizeof(int), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaFree(d);
  if (e != cudaSuccess) {
    colo::set_error("colo_build_cdf_breaks: %s", cudaGetErrorString(e));
    return COLO_ERR_CUDA;
  }
  if (err) {
    colo::set_error("colo_build_cdf_breaks: a row has more than %d breakpoints, decreases or holds a NaN", k);
    return COLO_ERR_ARG;
  }
  return COLO_OK;
}

int colo_build_dense_cdf(const float* T, int S, int A, int ld, void* cdf, int out_is_f64, void* stream) {
  COLO_ARG_CHECK(T && cdf && S > 0 && A > 0 && ld >= S, "T, cdf, S, A, ld");
  const long long rows = (long long)S * A;
  const int grid = (int)((rows + 127) / 128);
  if (out_is_f64)
    colo::build_dense_cdf_kernel<double><<<grid, 128, 0, (cudaStream_t)stream>>>(T, S, A, ld, (double*)cdf);
  else
    colo::build_dense_cdf_kernel<float><<<grid, 128, 0, (cudaStream_t)stream>>>(T, S, A, ld, (float*)cdf);
  return colo::check_launch("build_dense_cdf_kernel");
}

}  // extern "C"
