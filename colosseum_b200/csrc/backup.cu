// backup.cu -- the Bellman backup family (hot path B) for sm_100a.
//
// One streaming kernel template covers every S x A x S contraction of the path:
//   value iteration / policy evaluation sweeps   colosseum/dynamic_programming/infinite_horizon.py:121-184
//   episodic backward-induction layers           colosseum/dynamic_programming/finite_horizon.py:11-42
//   hitting-time (diameter) sweeps, multi-target  colosseum/hardness/measures/diameter.py:76-106, :285-346
//   the two passes of the environmental value norm colosseum/hardness/measures/value_norm.py:55-61,85-87
//
// It is a memory-bound batched GEMV: T is streamed from HBM exactly once per sweep with 128-bit
// no-L1-allocate loads; the V vector is re-read through L1 (it is S*4 bytes, shared by every row of the MDP) and
// each V element loaded is reused across the actions held in registers; the per-state fold over actions
// (max / pi-weighted sum / min) is a warp-shuffle reduction fused into the same kernel together with the
// residual max|dV|, the overflow test and the Q store, so a sweep is ONE launch and touches T once.
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <vector>

#include "tma_device.cuh"

extern "C" size_t colo_diameter_continuous_work_bytes(int K, int S, int f64);

namespace colo {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kAT = 4;  // actions held in registers at once

template <typename TV>
struct VecOf;
template <>
struct VecOf<float> {
  using resid_t = unsigned int;
};
template <>
struct VecOf<double> {
  using resid_t = unsigned long long;
};

}  // namespace colo
#include "multirhs.cuh"
namespace colo {

template <typename TV>
__device__ __forceinline__ void load_v4(const TV* p, TV (&v)[4]);
template <>
__device__ __forceinline__ void load_v4<float>(const float* p, float (&v)[4]) {
  float4 t = __ldg(reinterpret_cast<const float4*>(p));
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
template <>
__device__ __forceinline__ void load_v4<double>(const double* p, double (&v)[4]) {
  double2 a = __ldg(reinterpret_cast<const double2*>(p));
  double2 b = __ldg(reinterpret_cast<const double2*>(p) + 1);
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}

// Partial dot products of up to kAT action rows of one state against V, over the j-range owned by this thread.
// VEC: rows are 16-byte aligned and S % 4 == 0 -> 128-bit streaming loads, two row-quads in flight per action.
template <typename TV, bool VEC>
__device__ __forceinline__ void rows_dot(const float* __restrict__ Trow, const TV* __restrict__ Vb,
                                         long long v_action_stride, int a0, int na, int S, int tid, int nthr,
                                         TV (&acc)[kAT]) {
#pragma unroll
  for (int i = 0; i < kAT; ++i) acc[i] = TV(0);
  if (VEC) {
    const int S4 = S >> 2;
    const float4* T4 = reinterpret_cast<const float4*>(Trow);
    int j4 = tid;
    // main loop: two independent column quads per iteration -> 2*na 128-bit loads in flight per thread
    for (; j4 + nthr < S4; j4 += 2 * nthr) {
      float4 t0[kAT], t1[kAT];
#pragma unroll
      for (int i = 0; i < kAT; ++i)
        if (i < na) {
          t0[i] = ldg_stream4(T4 + (size_t)(a0 + i) * S4 + j4);
          t1[i] = ldg_stream4(T4 + (size_t)(a0 + i) * S4 + j4 + nthr);
        }
      if (v_action_stride == 0) {
        TV v0[4], v1[4];
        load_v4<TV>(Vb + 4 * (size_t)j4, v0);
        load_v4<TV>(Vb + 4 * (size_t)(j4 + nthr), v1);
#pragma unroll
        for (int i = 0; i < kAT; ++i)
          if (i < na) {
            acc[i] += (TV)t0[i].x * v0[0] + (TV)t0[i].y * v0[1] + (TV)t0[i].z * v0[2] + (TV)t0[i].w * v0[3];
            acc[i] += (TV)t1[i].x * v1[0] + (TV)t1[i].y * v1[1] + (TV)t1[i].z * v1[2] + (TV)t1[i].w * v1[3];
          }
      } else {
#pragma unroll
        for (int i = 0; i < kAT; ++i)
          if (i < na) {
            TV v0[4], v1[4];
            const TV* Va = Vb + (size_t)(a0 + i) * v_action_stride;
            load_v4<TV>(Va + 4 * (size_t)j4, v0);
            load_v4<TV>(Va + 4 * (size_t)(j4 + nthr), v1);
            acc[i] += (TV)t0[i].x * v0[0] + (TV)t0[i].y * v0[1] + (TV)t0[i].z * v0[2] + (TV)t0[i].w * v0[3];
            acc[i] += (TV)t1[i].x * v1[0] + (TV)t1[i].y * v1[1] + (TV)t1[i].z * v1[2] + (TV)t1[i].w * v1[3];
          }
      }
    }
    for (; j4 < S4; j4 += nthr) {
      float4 t0[kAT];
#pragma unroll
      for (int i = 0; i < kAT; ++i)
        if (i < na) t0[i] = ldg_stream4(T4 + (size_t)(a0 + i) * S4 + j4);
#pragma unroll
      for (int i = 0; i < kAT; ++i)
        if (i < na) {
          TV v0[4];
          load_v4<TV>(Vb + (size_t)(a0 + i) * v_action_stride + 4 * (size_t)j4, v0);
          acc[i] += (TV)t0[i].x * v0[0] + (TV)t0[i].y * v0[1] + (TV)t0[i].z * v0[2] + (TV)t0[i].w * v0[3];
        }
    }
  } else {
    // unaligned / odd-S rows: coalesced 32-bit streaming loads
    for (int j = tid; j < S; j += nthr) {
#pragma unroll
      for (int i = 0; i < kAT; ++i)
        if (i < na) {
          float t = ldg_stream1(Trow + (size_t)(a0 + i) * S + j);
          acc[i] += (TV)t * __ldg(Vb + (size_t)(a0 + i) * v_action_stride + j);
        }
    }
  }
}

// GROUP_CTA == false: one warp per (instance, state); GROUP_CTA == true: one CTA per (instance, state).
template <typename TV, int FOLD, bool VEC, bool GROUP_CTA>
#ifndef COLO_BACKUP_MIN_BLOCKS
#define COLO_BACKUP_MIN_BLOCKS 3  // measured on B200 (C4): 2 -> 90.6 %, 3 -> 99.5 %, 4 -> 95.6 % of the HBM peak (85 regs, 24 warps/SM)
#endif
__global__ void __launch_bounds__(kThreads, COLO_BACKUP_MIN_BLOCKS) backup_kernel(const colo_backup_args p) {
  using resid_t = typename VecOf<TV>::resid_t;
  __shared__ TV s_part[kWarps][kAT];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int S = p.S, A = p.A, nrows = p.nrows;
  const long long items = (long long)p.B * nrows;
  const long long first = GROUP_CTA ? blockIdx.x : (long long)blockIdx.x * kWarps + warp;
  const long long step = GROUP_CTA ? gridDim.x : (long long)gridDim.x * kWarps;
  const int tid = GROUP_CTA ? threadIdx.x : lane;
  const int nthr = GROUP_CTA ? kThreads : 32;
  const bool leader = GROUP_CTA ? threadIdx.x == 0 : lane == 0;
  const TV* V_in = reinterpret_cast<const TV*>(p.V_in);
  TV* V_out = reinterpret_cast<TV*>(p.V_out);
  TV* Q = reinterpret_cast<TV*>(p.Q);
  const TV gamma = (TV)p.gamma;

  for (long long it = first; it < items; it += step) {
    const int b = (int)(it / nrows);
    const int sl = (int)(it - (long long)b * nrows);  // shard-local state index
    const int s = p.row0 + sl;                        // global state index
    const TV* Vb = V_in + (size_t)b * p.v_in_stride;
    if (p.active != nullptr && p.active[b] == 0) {
      // converged instance of a batch: carry V forward so the ping-pong buffers stay consistent
      if (leader && V_out != nullptr && p.v_action_stride == 0) V_out[(size_t)b * p.v_out_stride + s] = Vb[s];
      continue;
    }
    const float* Trow = p.T + (size_t)b * p.t_stride + (size_t)sl * A * S;
    const int excl = p.exclude_index ? p.exclude_index[b] : -1;
    TV folded = FOLD == COLO_FOLD_MIN ? (TV)INFINITY : (FOLD == COLO_FOLD_MAX ? (TV)-INFINITY : (TV)0);
    for (int a0 = 0; a0 < A; a0 += kAT) {
      const int na = min(kAT, A - a0);
      TV acc[kAT];
      rows_dot<TV, VEC>(Trow, Vb, p.v_action_stride, a0, na, S, tid, nthr, acc);
#pragma unroll
      for (int i = 0; i < kAT; ++i) acc[i] = warp_sum(acc[i]);
      if (GROUP_CTA) {
        if (lane == 0) {
#pragma unroll
          for (int i = 0; i < kAT; ++i) s_part[warp][i] = acc[i];
        }
        __syncthreads();
        if (threadIdx.x == 0) {
#pragma unroll
          for (int i = 0; i < kAT; ++i) {
            TV t = 0;
            for (int w = 0; w < kWarps; ++w) t += s_part[w][i];
            acc[i] = t;
          }
        }
        __syncthreads();
      }
      if (leader) {
#pragma unroll
        for (int i = 0; i < kAT; ++i)
          if (i < na) {
            const int a = a0 + i;
            TV dot = acc[i];
            if (excl >= 0)  // one next state's V is replaced by a constant (episodic diameter: the ns == es term)
              dot += (TV)Trow[(size_t)a * S + excl] * ((TV)p.exclude_value - Vb[(size_t)a * p.v_action_stride + excl]);
            const TV r = p.R ? (TV)p.R[(size_t)b * p.r_stride + (size_t)sl * A + a] : (TV)p.r_const;
            const TV q = r + gamma * dot;
            if (Q) Q[(size_t)b * p.q_stride + (size_t)sl * A + a] = q;
            if (FOLD == COLO_FOLD_MAX) folded = q > folded ? q : folded;
            if (FOLD == COLO_FOLD_MIN) folded = q < folded ? q : folded;
            if (FOLD == COLO_FOLD_PI) folded += q * (TV)p.pi[(size_t)b * p.pi_stride + (size_t)sl * A + a];
          }
      }
    }
    if (leader && V_out != nullptr) {
      if (p.pin_index != nullptr && p.pin_index[b] == s) folded = (TV)p.pin_value;
      TV* vo = V_out + (size_t)b * p.v_out_stride + s;
      const TV old = p.resid_vs_out ? *vo : Vb[s];
      *vo = folded;
      for (int r = 0; r < p.n_peers; ++r)  // fused all-gather: the row also lands in every peer GPU's V
        reinterpret_cast<TV*>(p.V_out_peers[r])[(size_t)b * p.v_out_stride + s] = folded;
      if (p.resid != nullptr) {
        const TV d = fabs(folded - old);
        if (d > (TV)0) atomic_max_nonneg(reinterpret_cast<resid_t*>(p.resid) + b, d);
      }
      if (p.max_abs > 0.0 && p.overflow_flag &&
          (p.overflow_signed ? (double)folded : fabs((double)folded)) > p.max_abs)
        *p.overflow_flag = 1;
    }
  }
}

// ---- the same sweep with the rows of T staged in shared memory by the TMA (BASELINE north star: "TMA-staged T tiles") --
// One persistent CTA per SM slot: a producer thread keeps a ring of NST stages full -- one cp.async.bulk per state (its A
// rows are A*S*4 contiguous bytes), completion signalled on the stage's `full` mbarrier -- and 8 consumer warps each take
// every 8th stage: dot products from shared memory against V (L1), warp-shuffle fold over the actions, the same epilogue
// as backup_kernel, then an arrive on the stage's `empty` mbarrier.  States are dealt to CTAs round-robin, so consecutive
// CTAs stream consecutive 8 KB chunks.  Built to MEASURE the north star's suggestion against the LDG path (DESIGN 4.1):
// selected with COLO_BACKUP_TMA=1 (COLO_BACKUP_TMA_{STAGES,CTAS,WARPS} size the ring, the CTAs per SM and the consumer
// warps per CTA), f32 / contiguous rows / no exclude, pin or peer options.
constexpr int kTmaProducers = 8;
template <int FOLD, int kTmaConsumers>
__global__ void __launch_bounds__((kTmaConsumers + 1) * 32) backup_tma_kernel(const colo_backup_args p, int n_stages,
                                                                             uint32_t stage_bytes) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int S = p.S, A = p.A, nrows = p.nrows;
  const uint32_t row_bytes = (uint32_t)A * S * 4;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)n_stages * stage_bytes);
  uint64_t* empty = full + n_stages;
  if (threadIdx.x == 0) {
    for (int k = 0; k < n_stages; ++k) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(gs_smem_u32(full + k)) : "memory");
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(gs_smem_u32(empty + k)) : "memory");
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const long long items = (long long)p.B * nrows;
  const long long mine = (items - blockIdx.x + gridDim.x - 1) / gridDim.x;  // items blockIdx.x, + gridDim.x, ...
  if (warp == kTmaConsumers) {  // producer warp: kTmaProducers lanes, lane l re-arms the stages k = l (mod kTmaProducers)
    // (one lane alone -- wait on `empty`, proxy fence, expect_tx, bulk copy -- re-arms a stage every ~0.45 us: measured,
    // 2.6 TB/s with one CTA per SM; the lanes issue independently)
    if (lane < kTmaProducers) {
      for (long long k = lane; k < mine; k += kTmaProducers) {
        const int slot = (int)(k % n_stages);
        if (k >= n_stages) {
          gs_bar_wait(empty + slot, (uint32_t)(((k / n_stages) - 1) & 1));
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic reads of the stage before the async write
        }
        const long long it = blockIdx.x + k * gridDim.x;
        const int b = (int)(it / nrows);
        const int sl = (int)(it - (long long)b * nrows);
        if (p.active != nullptr && p.active[b] == 0) {  // nothing to stage: the consumer only carries V forward
          asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(gs_smem_u32(full + slot)) : "memory");
          continue;
        }
        gs_bulk_load(smem_raw + (size_t)slot * stage_bytes, p.T + (size_t)b * p.t_stride + (size_t)sl * A * S, row_bytes,
                     full + slot);
      }
    }
    return;
  }
  const float* V_in = reinterpret_cast<const float*>(p.V_in);
  float* V_out = reinterpret_cast<float*>(p.V_out);
  float* Q = reinterpret_cast<float*>(p.Q);
  const float gamma = (float)p.gamma;
  const int S4 = S >> 2;
  for (long long k = warp; k < mine; k += kTmaConsumers) {
    const int slot = (int)(k % n_stages);
    const long long it = blockIdx.x + k * gridDim.x;
    const int b = (int)(it / nrows);
    const int sl = (int)(it - (long long)b * nrows);
    const int s = p.row0 + sl;
    const float* Vb = V_in + (size_t)b * p.v_in_stride;
    gs_bar_wait(full + slot, (uint32_t)((k / n_stages) & 1));
    if (p.active != nullptr && p.active[b] == 0) {
      if (lane == 0 && V_out != nullptr) V_out[(size_t)b * p.v_out_stride + s] = Vb[s];
    } else {
      const float* Ts = reinterpret_cast<const float*>(smem_raw + (size_t)slot * stage_bytes);
      float folded = FOLD == COLO_FOLD_MIN ? INFINITY : (FOLD == COLO_FOLD_MAX ? -INFINITY : 0.f);
      for (int a0 = 0; a0 < A; a0 += kAT) {
        const int na = min(kAT, A - a0);
        float acc[kAT];
#pragma unroll
        for (int i = 0; i < kAT; ++i) acc[i] = 0.f;
        for (int j4 = lane; j4 < S4; j4 += 32) {
          const float4 v = __ldg(reinterpret_cast<const float4*>(Vb) + j4);
#pragma unroll
          for (int i = 0; i < kAT; ++i)
            if (i < na) {
              const float4 t = *reinterpret_cast<const float4*>(Ts + (size_t)(a0 + i) * S + 4 * j4);
              acc[i] += t.x * v.x + t.y * v.y + t.z * v.z + t.w * v.w;
            }
        }
#pragma unroll
        for (int i = 0; i < kAT; ++i) acc[i] = warp_sum(acc[i]);
        if (lane == 0) {
#pragma unroll
          for (int i = 0; i < kAT; ++i)
            if (i < na) {
              const int a = a0 + i;
              const float r = p.R ? p.R[(size_t)b * p.r_stride + (size_t)sl * A + a] : (float)p.r_const;
              const float q = r + gamma * acc[i];
              if (Q) Q[(size_t)b * p.q_stride + (size_t)sl * A + a] = q;
              if (FOLD == COLO_FOLD_MAX) folded = q > folded ? q : folded;
              if (FOLD == COLO_FOLD_MIN) folded = q < folded ? q : folded;
              if (FOLD == COLO_FOLD_PI) folded += q * p.pi[(size_t)b * p.pi_stride + (size_t)sl * A + a];
            }
        }
      }
      if (lane == 0 && V_out != nullptr) {
        float* vo = V_out + (size_t)b * p.v_out_stride + s;
        const float old = p.resid_vs_out ? *vo : Vb[s];
        *vo = folded;
        if (p.resid != nullptr) {
          const float d = fabsf(folded - old);
          if (d > 0.f) atomic_max_nonneg(reinterpret_cast<unsigned int*>(p.resid) + b, d);
        }
        if (p.max_abs > 0.0 && p.overflow_flag &&
            (p.overflow_signed ? (double)folded : fabs((double)folded)) > p.max_abs)
          *p.overflow_flag = 1;
      }
    }
    __syncwarp();  // every lane is done with the stage
    if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(gs_smem_u32(empty + slot)) : "memory");
  }
}

static std::atomic<unsigned long long> g_tma_sweeps{0};
// returns COLO_OK and *handled = 1 when the TMA-staged variant took the sweep
static int launch_backup_tma(const colo_backup_args& p, cudaStream_t st, int* handled) {
  *handled = 0;
  static const char* env = getenv("COLO_BACKUP_TMA");
  if (!env || env[0] == '0') return COLO_OK;
  const size_t row_bytes = (size_t)p.A * p.S * 4;
  if (p.exclude_index || p.pin_index || p.n_peers || p.v_action_stride != 0 || row_bytes % 16 || row_bytes > 32768 ||
      p.S % 4 || (uintptr_t)p.T % 16 || p.t_stride % 4 || (uintptr_t)p.V_in % 16 || p.v_in_stride % 4)
    return COLO_OK;
  const long long items = (long long)p.B * p.nrows;
  if (items < (long long)sm_count() * 64) return COLO_OK;
  const uint32_t stage_bytes = (uint32_t)((row_bytes + 127) & ~(size_t)127);
  static const int want = getenv("COLO_BACKUP_TMA_STAGES") ? atoi(getenv("COLO_BACKUP_TMA_STAGES")) : 24;
  static const int ctas_per_sm = getenv("COLO_BACKUP_TMA_CTAS") ? atoi(getenv("COLO_BACKUP_TMA_CTAS")) : 1;
  const size_t budget = (size_t)(227 * 1024) / ctas_per_sm - 2048;
  int n_stages = (int)((budget - 1024) / stage_bytes);
  if (n_stages > want) n_stages = want;
  // every stage must belong to ONE producer lane (slot = k % n_stages, lane = k % kTmaProducers): a parity wait only
  // tells the current phase from the previous one, so two lanes sharing a slot could run a whole phase apart
  n_stages -= n_stages % kTmaProducers;
  if (n_stages < 2) return COLO_OK;
  const size_t smem = (size_t)n_stages * stage_bytes + (size_t)n_stages * 16 + 128;
  const int grid = sm_count() * ctas_per_sm;
  static const int ncons_env = getenv("COLO_BACKUP_TMA_WARPS") ? atoi(getenv("COLO_BACKUP_TMA_WARPS")) : 8;
  // a consumer warp owns every ncons-th stage: more consumers than stages would wait on a stage that was never filled
  const int ncons = n_stages >= 16 ? ncons_env : 8;
  if (n_stages < 8) return COLO_OK;
#define COLO_TMA(FOLD)                                                                                   \
  if (ncons >= 16) {                                                                                     \
    auto k = backup_tma_kernel<FOLD, 16>;                                                                \
    const int es = ensure_dynamic_smem((const void*)k, smem);                                            \
    if (es != COLO_OK) return es;                                                                        \
    k<<<grid, 17 * 32, smem, st>>>(p, n_stages, stage_bytes);                                            \
  } else {                                                                                               \
    auto k = backup_tma_kernel<FOLD, 8>;                                                                 \
    const int es = ensure_dynamic_smem((const void*)k, smem);                                            \
    if (es != COLO_OK) return es;                                                                        \
    k<<<grid, 9 * 32, smem, st>>>(p, n_stages, stage_bytes);                                             \
  }
  switch (p.fold) {
    case COLO_FOLD_MAX: COLO_TMA(COLO_FOLD_MAX); break;
    case COLO_FOLD_PI: COLO_TMA(COLO_FOLD_PI); break;
    default: COLO_TMA(COLO_FOLD_MIN); break;
  }
#undef COLO_TMA
  *handled = 1;
  g_tma_sweeps.fetch_add(1);
  return check_launch("backup_tma_kernel");
}

template <typename TV, int FOLD, bool VEC>
static int launch_backup_2(const colo_backup_args& p, bool group_cta, cudaStream_t st) {
  const long long items = (long long)p.B * p.nrows;
  if (items == 0) return COLO_OK;
  const int cap = sm_count() * 32;
  if (group_cta) {
    int grid = (int)(items < cap ? items : cap);
    count_solver_path(COLO_PATH_BACKUP_CTA);
    backup_kernel<TV, FOLD, VEC, true><<<grid, kThreads, 0, st>>>(p);
  } else {
    long long blocks = (items + kWarps - 1) / kWarps;
    int grid = (int)(blocks < cap ? blocks : cap);
    count_solver_path(COLO_PATH_BACKUP_WARP);
    backup_kernel<TV, FOLD, VEC, false><<<grid, kThreads, 0, st>>>(p);
  }
  return check_launch("backup_kernel");
}

template <typename TV>
int launch_backup(const colo_backup_args* pp, void* stream) {
  COLO_ARG_CHECK(pp != nullptr, "args is NULL");
  colo_backup_args p = *pp;
  COLO_ARG_CHECK(p.T && p.V_in, "T and V_in are required");
  COLO_ARG_CHECK(p.B >= 0 && p.S > 0 && p.A > 0, "B,S,A");
  COLO_ARG_CHECK(p.fold >= 0 && p.fold <= 2, "fold");
  COLO_ARG_CHECK(p.fold != COLO_FOLD_PI || p.pi, "pi is required for COLO_FOLD_PI");
  if (p.nrows == 0 && p.row0 == 0) p.nrows = p.S;
  COLO_ARG_CHECK(p.row0 >= 0 && p.nrows >= 0 && p.row0 + p.nrows <= p.S, "row0/nrows");
  cudaStream_t st = (cudaStream_t)stream;
  const bool vec = (p.S % 4 == 0) && ((uintptr_t)p.T % 16 == 0) && ((uintptr_t)p.V_in % 16 == 0) &&
                   (p.t_stride % 4 == 0) && (p.v_in_stride % 4 == 0) && (p.v_action_stride % 4 == 0);
  // one warp per state while that still fills the machine; one CTA per state for few, long rows
  const long long items = (long long)p.B * p.nrows;
  const bool group_cta = (items < (long long)sm_count() * 64) && ((long long)p.S * p.A >= 4096);
  if (sizeof(TV) == 4 && vec && !group_cta) {
    int handled = 0;
    const int r = launch_backup_tma(p, st, &handled);
    if (r != COLO_OK || handled) return r;
  }
#define COLO_DISPATCH(FOLD)                                                            \
  return vec ? launch_backup_2<TV, FOLD, true>(p, group_cta, st) : launch_backup_2<TV, FOLD, false>(p, group_cta, st)
  switch (p.fold) {
    case COLO_FOLD_MAX: COLO_DISPATCH(COLO_FOLD_MAX);
    case COLO_FOLD_PI: COLO_DISPATCH(COLO_FOLD_PI);
    default: COLO_DISPATCH(COLO_FOLD_MIN);
  }
#undef COLO_DISPATCH
}

// ---- small helper kernels -----------------------------------------------------------------------------------
template <typename TV>
__global__ void finish_sweep_kernel(typename VecOf<TV>::resid_t* resid, unsigned char* active, long long* iters,
                                    int B, TV eps, int* flags) {
  // after one sweep: iters++ for the instances that ran it; an instance whose max|dV| < eps stops
  // (infinite_horizon.py:140-141); flags[0] counts the instances still running.
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  int still = 0;
  if (b < B && active[b]) {
    TV r;
    if (sizeof(TV) == 4)
      r = (TV)__uint_as_float((unsigned int)resid[b]);
    else
      r = (TV)__longlong_as_double((long long)resid[b]);
    iters[b] += 1;
    if (r < eps)
      active[b] = 0;
    else
      still = 1;
    resid[b] = 0;
  }
  still = __syncthreads_count(still);
  if (threadIdx.x == 0 && still) atomicAdd(&flags[0], still);
}

template <typename TV>
__global__ void fill_kernel(TV* x, long long n, TV v) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] = v;
}

__global__ void cast_f32_f64_kernel(const float* __restrict__ x, double* __restrict__ y, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] = (double)x[i];
}
__global__ void bias_init_kernel(const float* __restrict__ r, const double* __restrict__ gain, double* __restrict__ v,
                                 double* __restrict__ h, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    const double d = (double)r[i] - gain[i];
    v[i] = d;
    h[i] = d;  // the i = 0 term: P^0 (r - gain)
  }
}
__global__ void axpy_kernel(const double* __restrict__ x, double* __restrict__ y, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] += x[i];
}

template <typename TV>
__global__ void normalize_resid_kernel(TV* __restrict__ x_new, const TV* __restrict__ x_old, int S,
                                       typename VecOf<TV>::resid_t* __restrict__ resid) {
  // single CTA: x_new /= sum(x_new); resid[0] = max|x_new - x_old| (power iteration on a distribution)
  using resid_t = typename VecOf<TV>::resid_t;
  __shared__ double sm[32];
  __shared__ double s_tot;
  double part = 0.0;
  for (int i = threadIdx.x; i < S; i += blockDim.x) part += (double)x_new[i];
  part = warp_sum(part);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = part;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sm[w];
    s_tot = t;
  }
  __syncthreads();
  const TV inv = (TV)(1.0 / s_tot);
  TV d = 0;
  for (int i = threadIdx.x; i < S; i += blockDim.x) {
    const TV v = x_new[i] * inv;
    x_new[i] = v;
    const TV dd = fabs(v - x_old[i]);
    d = dd > d ? dd : d;
  }
  d = warp_max(d);
  if ((threadIdx.x & 31) == 0 && d > (TV)0) atomic_max_nonneg(reinterpret_cast<resid_t*>(resid), d);
}

template <typename TV>
__global__ void max_reduce_kernel(const TV* x, long long n, TV* out, int take_sqrt) {
  // single-CTA deterministic max (n is small: S or K*S)
  __shared__ TV sm[32];
  TV m = -INFINITY;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) m = x[i] > m ? x[i] : m;
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x < 32) {
    m = threadIdx.x < (blockDim.x >> 5) ? sm[threadIdx.x] : (TV)-INFINITY;
    m = warp_max(m);
    if (threadIdx.x == 0) out[0] = take_sqrt ? (TV)sqrt((double)(m > 0 ? m : 0)) : m;
  }
}

template <typename TV>
__global__ void sqdev_kernel(const TV* V, const TV* Ev, int S, int A, TV* W) {
  // W[a,j] = (V[j] - Ev[j,a])^2   (value_norm.py:87: Ev indexed by the NEXT state j, sic)
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < S * A) {
    int a = i / S, j = i - a * S;
    TV d = V[j] - Ev[(size_t)j * A + a];
    W[i] = d * d;
  }
}

__global__ void gaps_kernel(const double* Q, const double* V, const unsigned char* mask, long long NS, int A,
                            double reg, double* out) {
  // sum_{n,a} 1/(V[n]-Q[n,a]+reg): fixed thread-strided order + fixed tree -> deterministic
  __shared__ double sm[1024];
  double acc = 0.0;
  for (long long n = threadIdx.x; n < NS; n += blockDim.x) {
    if (mask && !mask[n]) continue;
    const double v = V[n];
    for (int a = 0; a < A; ++a) acc += 1.0 / (v - Q[n * A + a] + reg);
  }
  sm[threadIdx.x] = acc;
  __syncthreads();
  for (int o = blockDim.x >> 1; o > 0; o >>= 1) {
    if (threadIdx.x < o) sm[threadIdx.x] += sm[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = sm[0];
}

template <typename TV>
__global__ void episodic_last_layer_kernel(const float* start_row, const TV* E, long long e_stride, int S, int H,
                                           typename VecOf<TV>::resid_t* resid) {
  // diameter.py:293  ETs[-1] = T[-1,0,0] @ (1 + ETs[0])  for target k = blockIdx.x (every state gets the value);
  // stored form F = 1 + ETs:  F[H-1,:] = 1 + start . F[0,:]
  using resid_t = typename VecOf<TV>::resid_t;
  __shared__ TV sm[32];
  __shared__ TV s_val;
  TV* Ek = const_cast<TV*>(E) + (size_t)blockIdx.x * e_stride;
  TV acc = 0;
  for (int ns = threadIdx.x; ns < S; ns += blockDim.x) acc += (TV)start_row[ns] * Ek[ns];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    TV t = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += sm[w];
    s_val = (TV)1 + t;
  }
  __syncthreads();
  const TV v = s_val;
  TV* last = Ek + (size_t)(H - 1) * S;
  TV d = 0;
  for (int j = threadIdx.x; j < S; j += blockDim.x) {
    TV dd = fabs(v - last[j]);
    d = dd > d ? dd : d;
    last[j] = v;
  }
  d = warp_max(d);
  if ((threadIdx.x & 31) == 0 && d > 0 && resid) atomic_max_nonneg(reinterpret_cast<resid_t*>(resid) + blockIdx.x, d);
}

template <typename TV>
__global__ void episodic_diam_reduce_kernel(const TV* E, int K, int H, int S, TV* out) {
  // diameter.py:311-314: per state the min over h of the POSITIVE entries, max over states, max over targets
  __shared__ TV sm[32];
  TV best = -INFINITY;
  for (long long i = threadIdx.x; i < (long long)K * S; i += blockDim.x) {
    const int k = (int)(i / S), s = (int)(i - (long long)k * S);
    TV mn = INFINITY;
    for (int h = 0; h < H; ++h) {
      TV v = E[((size_t)k * H + h) * S + s] - (TV)1;  // stored F = 1 + ETs
      if (v > 0 && v < mn) mn = v;
    }
    best = mn > best ? mn : best;
  }
  best = warp_max(best);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = best;
  __syncthreads();
  if (threadIdx.x < 32) {
    best = threadIdx.x < (blockDim.x >> 5) ? sm[threadIdx.x] : (TV)-INFINITY;
    best = warp_max(best);
    if (threadIdx.x == 0) out[0] = best;
  }
}

// ---- host-side solvers ----------------------------------------------------------------------------------------
struct SolveWork {  // carved from the caller's `work` buffer
  void* v_alt;
  void* resid;
  unsigned char* active;
  long long* iters;
  int* flags;  // [0] still-running count, [1] overflow
};

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

template <typename TV>
static size_t solve_work_bytes(long long B, long long S) {
  size_t n = 0;
  n += align_up((size_t)B * S * sizeof(TV), 256);
  n += align_up((size_t)B * sizeof(typename VecOf<TV>::resid_t), 256);
  n += align_up((size_t)B, 256);
  n += align_up((size_t)B * sizeof(long long), 256);
  n += 256;
  return n;
}

template <typename TV>
static SolveWork carve(void* work, long long B, long long S) {
  char* p = (char*)work;
  SolveWork w;
  w.v_alt = p;
  p += align_up((size_t)B * S * sizeof(TV), 256);
  w.resid = p;
  p += align_up((size_t)B * sizeof(typename VecOf<TV>::resid_t), 256);
  w.active = (unsigned char*)p;
  p += align_up((size_t)B, 256);
  w.iters = (long long*)p;
  p += align_up((size_t)B * sizeof(long long), 256);
  w.flags = (int*)p;
  return w;
}

// Iterate `sweep(V_cur, V_nxt)` until every instance has max|dV| < eps.  The host only looks at two ints every
// `check` sweeps; instance-level stopping happens on the device (active mask), so late checks cost nothing but
// idle sweeps of already-frozen instances.
template <typename TV, typename SweepFn>
static int iterate_to_convergence(SweepFn sweep, TV* V_user, SolveWork& w, long long B, long long S, TV eps,
                                  long long max_iter, long long* iters_out_host, long long* sweeps_run,
                                  cudaStream_t st, const TV* V0 = nullptr) {
  using resid_t = typename VecOf<TV>::resid_t;
  if (V0 != nullptr && V0 != V_user)
    COLO_CUDA_TRY(cudaMemcpyAsync(V_user, V0, (size_t)B * S * sizeof(TV), cudaMemcpyDeviceToDevice, st));
  else if (V0 == nullptr)
    COLO_CUDA_TRY(cudaMemsetAsync(V_user, 0, (size_t)B * S * sizeof(TV), st));
  COLO_CUDA_TRY(cudaMemsetAsync(w.resid, 0, (size_t)B * sizeof(resid_t), st));
  COLO_CUDA_TRY(cudaMemsetAsync(w.active, 1, (size_t)B, st));
  COLO_CUDA_TRY(cudaMemsetAsync(w.iters, 0, (size_t)B * sizeof(long long), st));
  COLO_CUDA_TRY(cudaMemsetAsync(w.flags, 0, 2 * sizeof(int), st));
  TV* cur = V_user;
  TV* nxt = (TV*)w.v_alt;
  int rc = COLO_MAX_ITER;
  long long it = 0;
  int check = 1;
  int h_flags[2] = {0, 0};
  while (it < max_iter) {
    long long burst = check;
    if (it + burst > max_iter) burst = max_iter - it;
    for (long long i = 0; i < burst; ++i) {
      if (i == burst - 1) COLO_CUDA_TRY(cudaMemsetAsync(w.flags, 0, sizeof(int), st));
      int r = sweep(cur, nxt);
      if (r != COLO_OK) return r;
      finish_sweep_kernel<TV><<<(int)((B + 255) / 256), 256, 0, st>>>((resid_t*)w.resid, w.active, w.iters, (int)B,
                                                                    eps, w.flags);
      r = check_launch("finish_sweep_kernel");
      if (r != COLO_OK) return r;
      TV* t = cur;
      cur = nxt;
      nxt = t;
    }
    it += burst;
    COLO_CUDA_TRY(cudaMemcpyAsync(h_flags, w.flags, 2 * sizeof(int), cudaMemcpyDeviceToHost, st));
    COLO_CUDA_TRY(cudaStreamSynchronize(st));
    if (h_flags[1]) {
      rc = COLO_OVERFLOW;
      break;
    }
    if (h_flags[0] == 0) {
      rc = COLO_OK;
      break;
    }
    if (check < 64) check *= 2;
  }
  if (cur != V_user) COLO_CUDA_TRY(cudaMemcpyAsync(V_user, cur, (size_t)B * S * sizeof(TV), cudaMemcpyDeviceToDevice, st));
  if (iters_out_host)
    COLO_CUDA_TRY(cudaMemcpyAsync(iters_out_host, w.iters, (size_t)B * sizeof(long long), cudaMemcpyDeviceToHost, st));
  COLO_CUDA_TRY(cudaStreamSynchronize(st));
  if (sweeps_run) *sweeps_run = it;
  return rc;
}

template <typename TV>
int solve_discounted(const float* T, const float* R, const float* pi, int B, int S, int A, double gamma, double eps,
                     double max_abs, long long max_iter, int fold, TV* Q, TV* V, long long* iters_out_host,
                     void* work, void* stream, const TV* V0 = nullptr, bool normalize = false) {
  COLO_ARG_CHECK(T && R && V && work, "T, R, V, work are required");
  cudaStream_t st = (cudaStream_t)stream;
  SolveWork w = carve<TV>(work, B, S);
  static const bool no_sparse = getenv("COLO_NO_SPARSE") != nullptr;
  SparseRows sp;
  if (!no_sparse && (long long)B * S * A < (1LL << 31)) {
    // sparse rows (benchmark families, continuous forms): compressed once, then either the whole solve in one launch
    // with V in shared memory (S <= 2048) or one compressed-row launch per sweep under the host loop below
    int rs = sparse_rows_build(T, (long long)B * S * A, S, A, &sp, stream);
    if (rs != COLO_OK) return rs;
    if (sp.kmax > 0 && sparse_vi_fits_one_cta(S, sizeof(TV) == 8)) {
      rs = sparse_solve_resident<TV>(sp, R, pi, B, S, A, gamma, eps, max_abs, max_iter, fold, Q, V, iters_out_host, stream,
                                     V0, normalize);
      sparse_rows_free(&sp, stream);
      return rs;
    }
  }
  if (sp.kmax > 0) {
    auto sweep = [&](TV* cur, TV* nxt) {
      int r = sparse_sweep_launch<TV>(sp, R, pi, B, S, A, fold, gamma, cur, nxt, Q, normalize ? nullptr : w.resid, w.active,
                                      max_abs, w.flags + 1, stream);
      if (r == COLO_OK && normalize) {
        normalize_resid_kernel<TV><<<1, 1024, 0, st>>>(nxt, cur, S, (typename VecOf<TV>::resid_t*)w.resid);
        r = check_launch("normalize_resid_kernel");
      }
      return r;
    };
    const int rc = iterate_to_convergence<TV>(sweep, V, w, B, S, (TV)eps, max_iter, iters_out_host, nullptr, st, V0);
    sparse_rows_free(&sp, stream);
    return rc;
  }
  COLO_ARG_CHECK(!normalize || B == 1, "normalize needs B == 1");
  if (V0 == nullptr && !normalize && resident_enabled() && resident_fits_any(S, A, 1, sizeof(TV) == 8, nullptr)) {
    // small MDPs: the whole solve is ONE launch of the on-chip resident solver (resident.cu)
    colo_resident_args ra = {};
    ra.T = T; ra.R = R; ra.pi = pi; ra.V = V; ra.Q = Q;
    ra.t_stride = (long long)S * A * S; ra.r_stride = (long long)S * A;
    ra.B = B; ra.S = S; ra.A = A; ra.NV = 1; ra.fold = fold;
    ra.gamma = gamma; ra.eps = eps; ra.max_abs = max_abs; ra.max_iter = max_iter;
    ra.iters_out = w.iters; ra.status_out = (int*)w.resid;
    int r = resident_solve_any(&ra, sizeof(TV) == 8, stream);
    if (r != COLO_OK) return r;
    std::vector<int> h_status((size_t)B);
    COLO_CUDA_TRY(cudaMemcpyAsync(h_status.data(), w.resid, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st));
    if (iters_out_host)
      COLO_CUDA_TRY(cudaMemcpyAsync(iters_out_host, w.iters, (size_t)B * sizeof(long long), cudaMemcpyDeviceToHost, st));
    COLO_CUDA_TRY(cudaStreamSynchronize(st));
    int rc = COLO_OK;
    for (int b = 0; b < B; ++b) {
      if (h_status[b] == COLO_OVERFLOW) return COLO_OVERFLOW;
      if (h_status[b] == COLO_MAX_ITER) rc = COLO_MAX_ITER;
    }
    return rc;
  }
  colo_backup_args a = {};
  a.T = T; a.R = R; a.pi = pi; a.Q = Q;
  a.B = B; a.S = S; a.A = A; a.fold = fold; a.gamma = gamma;
  a.t_stride = (long long)S * A * S; a.r_stride = (long long)S * A; a.pi_stride = (long long)S * A;
  a.v_in_stride = S; a.v_out_stride = S; a.q_stride = (long long)S * A;
  a.resid = normalize ? nullptr : w.resid; a.active = w.active; a.max_abs = max_abs; a.overflow_flag = w.flags + 1;
  a.row0 = 0; a.nrows = S;
  auto sweep = [&](TV* cur, TV* nxt) {
    a.V_in = cur;
    a.V_out = nxt;
    int r = launch_backup<TV>(&a, stream);
    if (r == COLO_OK && normalize) {
      normalize_resid_kernel<TV><<<1, 1024, 0, st>>>(nxt, cur, S, (typename VecOf<TV>::resid_t*)w.resid);
      r = check_launch("normalize_resid_kernel");
    }
    return r;
  };
  return iterate_to_convergence<TV>(sweep, V, w, B, S, (TV)eps, max_iter, iters_out_host, nullptr, st, V0);
}

// Many small MDPs (the batched PSRL agents re-solve N sampled models every episode): one CTA walks one MDP through all
// H layers of backward induction in a single launch.  L lanes (a power of two <= 32) share a row T[s,a,:] -- short
// rows do not pay a 32-lane reduction each -- with up to four 128-bit loads in flight per lane; V[h+1] and Q[h] live
// in shared memory, T is re-read from L2 for every layer (only the first layer touches HBM).
template <typename TV, int L, bool VEC4>
__global__ void __launch_bounds__(256) episodic_batched_kernel(const float* __restrict__ T, const float* __restrict__ R,
                                                               const float* __restrict__ pi, int B, int S, int A, int H,
                                                               int fold, TV* __restrict__ Q, TV* __restrict__ V,
                                                               long long t_stride, long long r_stride) {
  extern __shared__ __align__(16) unsigned char smem_eb[];
  TV* Vn = reinterpret_cast<TV*>(smem_eb);           // V[h+1], padded to a multiple of 4
  TV* Qs = Vn + ((S + 3) & ~3);                      // Q[h]
  const int tid = threadIdx.x, sub = tid % L, grp = tid / L, groups = blockDim.x / L;
  const int SA = S * A;
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    const float* Tb = T + (size_t)b * t_stride;  // stride 0: every instance evaluates its policy on the same MDP
    const float* Rb = R + (size_t)b * r_stride;
    TV* Qb = Q + (size_t)b * (H + 1) * SA;
    TV* Vb = V + (size_t)b * (H + 1) * S;
    for (int i = tid; i < SA; i += blockDim.x) Qb[(size_t)H * SA + i] = TV(0);
    for (int i = tid; i < S; i += blockDim.x) {
      Vb[(size_t)H * S + i] = TV(0);
      Vn[i] = TV(0);
    }
    __syncthreads();
    for (int h = H - 1; h >= 0; --h) {
      for (int base = 0; base < SA; base += groups) {  // warp-uniform trip count: the shuffles below use the full mask
        const int row = base + grp;
        TV acc = TV(0);
        if (row < SA) {
          const float* t = Tb + (size_t)row * S;
          if (VEC4) {
            const float4* t4 = reinterpret_cast<const float4*>(t);
            const int n4 = S >> 2;
            for (int j0 = sub; j0 < n4; j0 += 4 * L) {
              float4 x[4];
#pragma unroll
              for (int u = 0; u < 4; ++u)
                if (j0 + u * L < n4) x[u] = __ldg(t4 + j0 + u * L);
#pragma unroll
              for (int u = 0; u < 4; ++u)
                if (j0 + u * L < n4) {
                  const int j = (j0 + u * L) << 2;
                  acc += (TV)x[u].x * Vn[j] + (TV)x[u].y * Vn[j + 1] + (TV)x[u].z * Vn[j + 2] + (TV)x[u].w * Vn[j + 3];
                }
            }
          } else {
            for (int j = sub; j < S; j += L) acc += (TV)__ldg(t + j) * Vn[j];
          }
        }
#pragma unroll
        for (int o = L >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(FULL, acc, o);
        if (row < SA && sub == 0) {
          const TV q = (TV)__ldg(Rb + row) + acc;
          Qs[row] = q;
          Qb[(size_t)h * SA + row] = q;
        }
      }
      __syncthreads();
      for (int s0 = tid; s0 < S; s0 += blockDim.x) {
        TV v;
        if (fold == COLO_FOLD_PI) {
          const float* p = pi + ((size_t)b * H + h) * SA + (size_t)s0 * A;
          v = TV(0);
          for (int a = 0; a < A; ++a) v += Qs[s0 * A + a] * (TV)__ldg(p + a);
        } else {
          v = Qs[s0 * A];
          for (int a = 1; a < A; ++a) {
            const TV q = Qs[s0 * A + a];
            v = fold == COLO_FOLD_MAX ? (q > v ? q : v) : (q < v ? q : v);
          }
        }
        Vn[s0] = v;
        Vb[(size_t)h * S + s0] = v;
      }
      __syncthreads();
    }
  }
}

template <typename TV, int L>
static int episodic_batched_launch(const float* T, const float* R, const float* pi, int B, int S, int A, int H, int fold,
                                   TV* Q, TV* V, bool vec4, size_t smem, cudaStream_t st, bool shared_mdp) {
  // up to 8 CTAs per SM in flight.  (Measured on 1,024 Taxi models: capping the CTAs in flight so that their T stays
  // L2-resident between layers -- 24/48/64/96/160 MB -- costs 2.71/2.37/1.99/1.60/1.44 ms against 1.31 ms uncapped:
  // parallelism beats residency.)
  // CTA size from the lanes one layer can use (rows x L).  Measured, us per solve of the whole batch at 64/128/256
  // threads: 8,192 C1 models (40 lanes) 26/32/54, 8,192 DeepSea-8 models (288 lanes) 128/137/186, 1,024 Taxi models
  // (5,184 lanes) 2366/1391/1287.
  static const int forced = getenv("COLO_EPI_THREADS") ? atoi(getenv("COLO_EPI_THREADS")) : 0;
  const long long lanes = (long long)S * A * L;
  const int threads = forced ? forced : (lanes <= 512 ? 64 : (lanes <= 2048 ? 128 : 256));
  const long long cap = (long long)sm_count() * (2048 / threads);
  const int grid = (int)(B < cap ? B : cap);
  (void)shared_mdp;
  const long long ts = shared_mdp ? 0 : (long long)S * A * S, rs = shared_mdp ? 0 : (long long)S * A;
  count_solver_path(COLO_PATH_EPI_BATCHED);
  if (vec4) {
    auto k = episodic_batched_kernel<TV, L, true>;
    { const int _es = ensure_dynamic_smem((const void*)k, smem); if (_es != COLO_OK) return _es; }
    k<<<grid, threads, smem, st>>>(T, R, pi, B, S, A, H, fold, Q, V, ts, rs);
  } else {
    auto k = episodic_batched_kernel<TV, L, false>;
    { const int _es = ensure_dynamic_smem((const void*)k, smem); if (_es != COLO_OK) return _es; }
    k<<<grid, threads, smem, st>>>(T, R, pi, B, S, A, H, fold, Q, V, ts, rs);
  }
  return check_launch("episodic_batched_kernel");
}

// returns COLO_OK with *handled = 1 when the batched kernel took the solve
template <typename TV>
static int episodic_batched(const float* T, const float* R, const float* pi, int B, int S, int A, int H, int fold,
                            TV* Q, TV* V, int* handled, cudaStream_t st, bool shared_mdp = false) {
  *handled = 0;
  const size_t smem = ((size_t)((S + 3) & ~3) + (size_t)S * A) * sizeof(TV);
  static const bool off = getenv("COLO_EPISODIC_BATCHED") && atoi(getenv("COLO_EPISODIC_BATCHED")) == 0;
  if (!shared_mdp &&
      (off || B < 16 || H < 1 || smem > (size_t)96 * 1024 || (size_t)S * A * S * sizeof(float) > ((size_t)8 << 20)))
    return COLO_OK;
  if (shared_mdp && (H < 1 || smem > (size_t)200 * 1024)) {
    set_error("colo_episodic_policies: S*(A+1) = %d values do not fit shared memory", S * (A + 1));
    return COLO_ERR_ARG;
  }
  const bool vec4 = (S % 4 == 0) && ((uintptr_t)T % 16 == 0);
  const int units = vec4 ? S / 4 : S;  // loads per row
  int r;
  if (units <= 16) r = episodic_batched_launch<TV, 4>(T, R, pi, B, S, A, H, fold, Q, V, vec4, smem, st, shared_mdp);
  else if (units <= 32) r = episodic_batched_launch<TV, 8>(T, R, pi, B, S, A, H, fold, Q, V, vec4, smem, st, shared_mdp);
  else if (units <= 64) r = episodic_batched_launch<TV, 16>(T, R, pi, B, S, A, H, fold, Q, V, vec4, smem, st, shared_mdp);
  else r = episodic_batched_launch<TV, 32>(T, R, pi, B, S, A, H, fold, Q, V, vec4, smem, st, shared_mdp);
  if (r == COLO_OK) *handled = 1;
  return r;
}

template <typename TV>
int episodic(const float* T, const float* R, const float* pi, int B, int S, int A, int H, int fold, double max_value,
             TV* Q, TV* V, void* stream) {
  COLO_ARG_CHECK(T && R && V && Q, "T, R, Q, V are required");
  COLO_ARG_CHECK(H >= 0, "H");
  cudaStream_t st = (cudaStream_t)stream;
  const long long qs = (long long)(H + 1) * S * A, vs = (long long)(H + 1) * S;
  if (!(max_value > 0)) {  // many small instances, no overflow test: one CTA per instance, all layers in one launch
    int handled = 0;
    const int r = episodic_batched<TV>(T, R, pi, B, S, A, H, fold, Q, V, &handled, st);
    if (r != COLO_OK || handled) return r;
  }
  int* flag = nullptr;
  if (max_value > 0) {
    COLO_CUDA_TRY(cudaMallocAsync(&flag, sizeof(int), st));
    COLO_CUDA_TRY(cudaMemsetAsync(flag, 0, sizeof(int), st));
  }
  // rows H are zero (finite_horizon.py:17-18); cudaMemset2D clears the last layer of every instance
  COLO_CUDA_TRY(cudaMemset2DAsync(V + (size_t)H * S, vs * sizeof(TV), 0, (size_t)S * sizeof(TV), B, st));
  COLO_CUDA_TRY(cudaMemset2DAsync(Q + (size_t)H * S * A, qs * sizeof(TV), 0, (size_t)S * A * sizeof(TV), B, st));
  if (H > 0 && resident_enabled() && resident_fits_any(S, A, 1, sizeof(TV) == 8, nullptr)) {
    // small MDPs: all H layers in one launch, T resident in shared memory
    int* status = nullptr;
    COLO_CUDA_TRY(cudaMallocAsync(&status, (size_t)B * sizeof(int), st));
    colo_resident_args ra = {};
    ra.T = T; ra.R = R; ra.pi = pi; ra.V = V; ra.Q = Q;
    ra.t_stride = (long long)S * A * S; ra.r_stride = (long long)S * A;
    ra.B = B; ra.S = S; ra.A = A; ra.NV = 1; ra.fold = fold; ra.gamma = 1.0;
    ra.max_abs = fold == COLO_FOLD_MAX ? max_value : 0.0; ra.overflow_signed = 1;
    ra.max_iter = H; ra.episodic_H = H; ra.status_out = status;
    int r = resident_solve_any(&ra, sizeof(TV) == 8, stream);
    int rc = COLO_OK;
    if (r == COLO_OK && max_value > 0) {
      std::vector<int> h_status((size_t)B);
      COLO_CUDA_TRY(cudaMemcpyAsync(h_status.data(), status, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st));
      COLO_CUDA_TRY(cudaStreamSynchronize(st));
      for (int b = 0; b < B; ++b)
        if (h_status[b] == COLO_OVERFLOW) rc = COLO_OVERFLOW;
    }
    COLO_CUDA_TRY(cudaFreeAsync(status, st));
    if (flag) COLO_CUDA_TRY(cudaFreeAsync(flag, st));
    return r != COLO_OK ? r : rc;
  }
  colo_backup_args a = {};
  a.T = T; a.R = R;
  a.B = B; a.S = S; a.A = A; a.fold = fold; a.gamma = 1.0;
  a.t_stride = (long long)S * A * S; a.r_stride = (long long)S * A; a.pi_stride = (long long)H * S * A;
  a.v_in_stride = vs; a.v_out_stride = vs; a.q_stride = qs;
  a.max_abs = fold == COLO_FOLD_MAX ? max_value : 0.0; a.overflow_signed = 1; a.overflow_flag = flag;
  a.row0 = 0; a.nrows = S;
  for (int h = H - 1; h >= 0; --h) {
    a.V_in = V + (size_t)(h + 1) * S;
    a.V_out = V + (size_t)h * S;
    a.Q = Q + (size_t)h * S * A;
    a.pi = pi ? pi + (size_t)h * S * A : nullptr;
    int r = launch_backup<TV>(&a, stream);
    if (r != COLO_OK) return r;
  }
  if (flag) {
    int hflag = 0;
    COLO_CUDA_TRY(cudaMemcpyAsync(&hflag, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
    COLO_CUDA_TRY(cudaStreamSynchronize(st));
    COLO_CUDA_TRY(cudaFreeAsync(flag, st));
    if (hflag) return COLO_OVERFLOW;
  }
  return COLO_OK;
}

// ---- optimal values of the CONTINUOUS FORM of an episodic MDP, from its structure ----------------------------------
// mdp/utils/mdp_creation.py:131-176 builds, over the reachable (h, s) nodes, the chain  (h,s) --T[s,a,:]--> (h+1,.)  for
// h < H-1, and for the last layer ONE row for every action: probability p_k on the column whose INDEX is the original
// state index of start state k (sic, :168 -- i.e. the node that happens to sit at that position of the node list).
// mdp/base_finite.py:167-178 then runs discounted_value_iteration on that n x A x n tensor: thousands of sweeps over
// thousands of nodes (gamma = 0.99 -> 2,062 sweeps to 1e-9), the largest single cost of the C3 hardness phase.
// The structure makes the fixed point a SCALAR one.  With c = sum_k p_k V[node at position start_k]:
//     V[H-1, s] = max_a R[s,a] + gamma * c              V[h, s] = max_a R[s,a] + gamma * sum_j T[s,a,j] V[h+1, j]
// so one backward induction over the ORIGINAL T (H launches of the backup kernel, never the n x A x n tensor) maps c to
// F(c) = sum_k p_k V[pos_k]; F is increasing, convex, piecewise linear and a contraction (every path back to a start
// position takes at least one step: slope <= gamma).  c* = F(c*) by safeguarded secant steps; the values at c* are the
// fixed point of the reference's iteration (same equations, rows of T_cf = rows of T).  Unreachable (h, s) pairs are
// computed too and ignored: reachable nodes only lead to reachable nodes.
template <typename TV>
__global__ void cf_last_layer_kernel(const float* __restrict__ R, int S, int A, double gamma_c, TV* __restrict__ V_last) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  TV best = (TV)__ldg(R + (size_t)s * A);
  for (int a = 1; a < A; ++a) {
    const TV r = (TV)__ldg(R + (size_t)s * A + a);
    best = r > best ? r : best;
  }
  V_last[s] = best + (TV)gamma_c;
}

template <typename TV>
__global__ void cf_start_value_kernel(const TV* __restrict__ V, const int* __restrict__ pos_h, const int* __restrict__ pos_s,
                                      const float* __restrict__ p, int n, int S, double* __restrict__ c_out) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double c = 0.0;  // fixed order, float32 probabilities as stored in the reference's T_cf row
  for (int k = 0; k < n; ++k) c += (double)p[k] * (double)V[(size_t)pos_h[k] * S + pos_s[k]];
  *c_out = c;
}

template <typename TV>
int continuous_form_values(const float* T, const float* R, int S, int A, int H, double gamma, const int* pos_h,
                           const int* pos_s, const float* p, int n_start, double eps, int max_eval, TV* V,
                           double* out_host, void* stream) {
  COLO_ARG_CHECK(T && R && V && pos_h && pos_s && p && out_host, "T, R, V, start positions, out_host are required");
  COLO_ARG_CHECK(H >= 1 && n_start >= 1 && gamma > 0.0 && gamma < 1.0 && eps > 0.0, "H >= 1, n_start >= 1, 0 < gamma < 1");
  cudaStream_t st = (cudaStream_t)stream;
  double* d_c = nullptr;
  COLO_CUDA_TRY(cudaMallocAsync(&d_c, sizeof(double), st));
  colo_backup_args a = {};
  a.T = T; a.R = R; a.B = 1; a.S = S; a.A = A; a.fold = COLO_FOLD_MAX; a.gamma = gamma;
  a.t_stride = 0; a.r_stride = 0; a.v_in_stride = S; a.v_out_stride = S; a.row0 = 0; a.nrows = S;
  auto F = [&](double c, double* fc) -> int {
    cf_last_layer_kernel<TV><<<(S + 127) / 128, 128, 0, st>>>(R, S, A, gamma * c, V + (size_t)(H - 1) * S);
    int r = check_launch("cf_last_layer_kernel");
    for (int h = H - 2; h >= 0 && r == COLO_OK; --h) {
      a.V_in = V + (size_t)(h + 1) * S;
      a.V_out = V + (size_t)h * S;
      r = launch_backup<TV>(&a, stream);
    }
    if (r != COLO_OK) return r;
    cf_start_value_kernel<TV><<<1, 32, 0, st>>>(V, pos_h, pos_s, p, n_start, S, d_c);
    r = check_launch("cf_start_value_kernel");
    if (r != COLO_OK) return r;
    COLO_CUDA_TRY(cudaMemcpyAsync(fc, d_c, sizeof(double), cudaMemcpyDeviceToHost, st));
    COLO_CUDA_TRY(cudaStreamSynchronize(st));
    return COLO_OK;
  };
  // |c - c*| <= |F(c) - c| / (1 - gamma), and the values move by at most gamma * |c - c*|
  const double tol = eps * (1.0 - gamma);
  double c = 0.0, fc = 0.0, c_prev = 0.0, g_prev = 0.0;
  bool have_prev = false;
  int evals = 0, rc = COLO_MAX_ITER;
  while (evals < max_eval) {
    const int r = F(c, &fc);
    ++evals;
    if (r != COLO_OK) {
      cudaFreeAsync(d_c, st);
      return r;
    }
    const double g = fc - c;
    if (fabs(g) <= tol) {
      rc = COLO_OK;
      break;
    }
    // secant step on g(c) = F(c) - c (g is decreasing: slope of F < 1), kept inside the bracket the contraction gives:
    // c* lies between F(c) and c + g / (1 - gamma)
    double next = fc;
    if (have_prev && g != g_prev) {
      const double sec = c - g * (c - c_prev) / (g - g_prev);
      const double lo = g > 0 ? fc : c + g / (1.0 - gamma), hi = g > 0 ? c + g / (1.0 - gamma) : fc;
      if (sec >= lo && sec <= hi) next = sec;
    }
    c_prev = c; g_prev = g; have_prev = true;
    c = next;
  }
  COLO_CUDA_TRY(cudaFreeAsync(d_c, st));
  out_host[0] = c;
  out_host[1] = (double)evals;
  return rc;
}

template <typename TV>
int diameter_continuous(const float* T, const int* targets, int K, int S, int A, double eps, double max_value,
                        long long max_iter, void* work, double* out_host, void* stream) {
  COLO_ARG_CHECK(T && targets && work && out_host, "T, targets, work, out_host are required");
  cudaStream_t st = (cudaStream_t)stream;
  // work = E ping [K*S] | solver work (E pong, resid, active, iters, flags) | 1 TV result
  TV* E = (TV*)work;
  char* rest = (char*)work + align_up((size_t)K * S * sizeof(TV), 256);
  SolveWork w = carve<TV>(rest, K, S);
  TV* d_out = (TV*)(rest + solve_work_bytes<TV>(K, S));
  // COLO_DIAM_PATH = resident | gemm | stream forces one of the three implementations (probing); default: automatic
  static const int diam_path = [] {
    const char* e = getenv("COLO_DIAM_PATH");
    if (!e) return 0;
    return !strcmp(e, "resident") ? 1 : (!strcmp(e, "gemm") ? 2 : (!strcmp(e, "stream") ? 3 : (!strcmp(e, "sparse") ? 4 : (!strcmp(e, "umma") ? 5 : 0))));
  }();
  if (diam_path == 0 || diam_path == 4) {
    // benchmark-family MDPs (<= 32 successors per row): compressed rows, the whole solve in one launch
    int handled = 0;
    const int r = sparse_diameter_continuous<TV>(T, targets, K, S, A, eps, max_value, max_iter, out_host, &handled, stream);
    if (r < 0 || handled) return r;
  }
  const bool fits = resident_fits_any(S, A, 4, sizeof(TV) == 8, nullptr) != 0;
  if ((diam_path == 1 || (diam_path == 0 && resident_enabled())) && fits) {
    // T fits a cluster's shared memory: tiles of 4 targets, each tile iterated to convergence on chip by its own
    // cluster in ONE launch (every T quad read from shared memory serves 4 targets)
    const int K4 = (K + 3) & ~3, tiles = K4 / 4;
    // carve: E4 [K4][S] | targets4 [K4] | status [tiles] | iters [K4]   (fits: the work buffer holds 2*K*S + extras)
    char* q = (char*)work;
    TV* E4 = (TV*)q;
    q += align_up((size_t)K4 * S * sizeof(TV), 256);
    int* tg4 = (int*)q;
    q += align_up((size_t)K4 * sizeof(int), 256);
    int* status = (int*)q;
    q += align_up((size_t)tiles * sizeof(int), 256);
    long long* iters = (long long*)q;
    q += align_up((size_t)K4 * sizeof(long long), 256);
    TV* res_out = (TV*)q;
    COLO_ARG_CHECK((size_t)(q + 256 - (char*)work) <= colo_diameter_continuous_work_bytes(K, S, sizeof(TV) == 8),
                   "work buffer too small");
    COLO_CUDA_TRY(cudaMemcpyAsync(tg4, targets, (size_t)K * sizeof(int), cudaMemcpyDeviceToDevice, st));
    for (int k = K; k < K4; ++k)  // pad the last tile with copies of the last target
      COLO_CUDA_TRY(cudaMemcpyAsync(tg4 + k, targets + (K - 1), sizeof(int), cudaMemcpyDeviceToDevice, st));
    colo_resident_args ra = {};
    ra.T = T; ra.V = E4; ra.t_stride = 0; ra.r_stride = 0;
    ra.B = tiles; ra.S = S; ra.A = A; ra.NV = 4; ra.fold = COLO_FOLD_MIN;
    ra.gamma = 1.0; ra.r_const = 1.0; ra.eps = eps; ra.max_abs = max_value; ra.max_iter = max_iter;
    ra.pin_index = tg4; ra.pin_value = 0.0; ra.iters_out = iters; ra.status_out = status;
    int r = resident_solve_any(&ra, sizeof(TV) == 8, stream);
    if (r != COLO_OK) return r;
    max_reduce_kernel<TV><<<1, 1024, 0, st>>>(E4, (long long)K * S, res_out, 0);
    r = check_launch("max_reduce_kernel");
    if (r != COLO_OK) return r;
    std::vector<int> h_status((size_t)tiles);
    std::vector<long long> h_iters((size_t)K4);
    TV h = 0;
    COLO_CUDA_TRY(cudaMemcpyAsync(h_status.data(), status, (size_t)tiles * sizeof(int), cudaMemcpyDeviceToHost, st));
    COLO_CUDA_TRY(cudaMemcpyAsync(h_iters.data(), iters, (size_t)K4 * sizeof(long long), cudaMemcpyDeviceToHost, st));
    COLO_CUDA_TRY(cudaMemcpyAsync(&h, res_out, sizeof(TV), cudaMemcpyDeviceToHost, st));
    COLO_CUDA_TRY(cudaStreamSynchronize(st));
    int rc = COLO_OK;
    long long mx = 0;
    for (int t = 0; t < tiles; ++t) {
      if (h_status[t] == COLO_OVERFLOW) return COLO_OVERFLOW;
      if (h_status[t] == COLO_MAX_ITER) rc = COLO_MAX_ITER;
    }
    for (auto v : h_iters) mx = v > mx ? v : mx;
    out_host[0] = (double)h;
    out_host[1] = (double)mx;
    return rc;
  }
  const bool use_gemm = diam_path == 2 || diam_path == 5 || (diam_path == 0 && (long long)K * S >= 128LL * 128);
  // f32 mode: the GEMM sweep runs on the tensor cores (hitting_umma.cu); f64acc mode keeps the fp64 SIMT tile
  UmmaPlan* umma = nullptr;
  if (sizeof(TV) == 4 && use_gemm && diam_path != 2 && hitting_umma_supported(S, A, K)) {
    const int r = hitting_umma_plan(T, S, A, K, &umma, st);
    if (r != COLO_OK) return r;
  }
  COLO_ARG_CHECK(diam_path != 5 || umma != nullptr, "COLO_DIAM_PATH=umma: f32 mode, S >= 128, K >= 64");
  HittingGemmArgs ga = {};
  ga.T = T; ga.e_stride = S; ga.targets = targets; ga.active = w.active; ga.resid = w.resid;
  ga.S = S; ga.A = A; ga.K = K; ga.max_value = max_value; ga.overflow_flag = w.flags + 1;
  colo_backup_args a = {};
  a.T = T; a.R = nullptr; a.r_const = 1.0;
  a.B = K; a.S = S; a.A = A; a.fold = COLO_FOLD_MIN; a.gamma = 1.0;
  a.t_stride = 0;  // every target shares T: row tiles are re-served from L2 across targets
  a.v_in_stride = S; a.v_out_stride = S;
  a.pin_index = targets; a.pin_value = 0.0;
  a.resid = w.resid; a.active = w.active; a.max_abs = max_value; a.overflow_flag = w.flags + 1;
  a.row0 = 0; a.nrows = S;
  auto sweep = [&](TV* cur, TV* nxt) {
    if (umma)
      return hitting_umma_sweep(umma, (const float*)cur, (float*)nxt, S, targets, w.active, (unsigned*)w.resid, max_value,
                                w.flags + 1, st);
    if (use_gemm) {  // many targets: one tiled GEMM per sweep (multirhs.cuh)
      ga.E_in = cur;
      ga.E_out = nxt;
      return launch_hitting_gemm<TV>(ga, st);
    }
    a.V_in = cur;
    a.V_out = nxt;
    return launch_backup<TV>(&a, stream);
  };
  long long sweeps = 0;
  int rc = iterate_to_convergence<TV>(sweep, E, w, K, S, (TV)eps, max_iter, nullptr, &sweeps, st);
  hitting_umma_free(umma, st);
  if (rc != COLO_OK && rc != COLO_MAX_ITER) return rc;
  max_reduce_kernel<TV><<<1, 1024, 0, st>>>(E, (long long)K * S, d_out, 0);
  int r = check_launch("max_reduce_kernel");
  if (r != COLO_OK) return r;
  TV h = 0;
  COLO_CUDA_TRY(cudaMemcpyAsync(&h, d_out, sizeof(TV), cudaMemcpyDeviceToHost, st));
  COLO_CUDA_TRY(cudaStreamSynchronize(st));
  out_host[0] = (double)h;
  out_host[1] = (double)sweeps;
  return rc;
}

template <typename TV>
int diameter_episodic(const float* T_epi, const int* targets, int K, int H, int S, int A, double eps, double max_value,
                      long long max_iter, void* work, double* out_host, void* stream) {
  using resid_t = typename VecOf<TV>::resid_t;
  COLO_ARG_CHECK(T_epi && targets && work && out_host, "T_epi, targets, work, out_host are required");
  COLO_ARG_CHECK(H >= 2, "H >= 2");
  cudaStream_t st = (cudaStream_t)stream;
  // work = F [K,H,S] | resid [K] | flags [2] | result        (F = 1 + ETs of diameter.py:285-318)
  char* p = (char*)work;
  TV* E = (TV*)p;
  p += align_up((size_t)K * H * S * sizeof(TV), 256);
  resid_t* resid = (resid_t*)p;
  p += align_up((size_t)K * sizeof(resid_t), 256);
  int* flags = (int*)p;
  p += 256;
  TV* d_out = (TV*)p;
  COLO_CUDA_TRY(cudaMemsetAsync(flags, 0, 2 * sizeof(int), st));
  // F = 1 + ETs is what is stored (ETs = 0 everywhere at the start, diameter.py:289)
  fill_kernel<TV><<<(int)(((long long)K * H * S + 255) / 256), 256, 0, st>>>(E, (long long)K * H * S, (TV)1);
  int r = check_launch("fill_kernel");
  if (r != COLO_OK) return r;
  colo_backup_args a = {};
  a.B = K; a.S = S; a.A = A; a.fold = COLO_FOLD_MIN; a.gamma = 1.0;
  a.t_stride = 0; a.r_stride = 0;
  a.v_in_stride = (long long)H * S; a.v_out_stride = (long long)H * S;
  // F[h-1,j] = min_a( 1 + sum_ns T[h-1,j,a,ns] * (ns == es ? 1 : F[h,ns]) );  F[h-1,es] = 1
  a.r_const = 1.0;
  a.pin_index = targets; a.pin_value = 1.0; a.exclude_index = targets; a.exclude_value = 1.0;
  a.resid = resid; a.resid_vs_out = 1; a.max_abs = max_value > 0 ? max_value + 1.0 : 0.0; a.overflow_flag = flags + 1;
  a.row0 = 0; a.nrows = S;
  static const int epi_path = [] {
    const char* e = getenv("COLO_DIAM_PATH");
    return !e ? 0 : (!strcmp(e, "gemm") ? 2 : (!strcmp(e, "stream") ? 3 : (!strcmp(e, "sparse") ? 4 : 0)));
  }();
  if (epi_path == 0 || epi_path == 4) {
    int handled = 0;
    const int rs = sparse_diameter_episodic<TV>(T_epi, targets, K, H, S, A, eps, max_value, max_iter, out_host, &handled,
                                               stream);
    if (rs < 0 || handled) return rs;
  }
  const bool use_gemm = epi_path == 2 || (epi_path == 0 && (long long)K * S >= 64LL * 64);
  HittingGemmArgs ga = {};
  ga.e_stride = (long long)H * S; ga.targets = targets; ga.resid = resid; ga.S = S; ga.A = A; ga.K = K;
  ga.max_value = a.max_abs; ga.overflow_flag = flags + 1;
  ga.pin_value = 1.0; ga.exclude_value = 1.0; ga.resid_vs_out = 1;
  int rc = COLO_MAX_ITER;
  long long it = 0;
  int check = 1, since = 0;
  std::vector<resid_t> h_res((size_t)K);
  int h_flags[2];
  for (; it < max_iter;) {
    COLO_CUDA_TRY(cudaMemsetAsync(resid, 0, (size_t)K * sizeof(resid_t), st));
    episodic_last_layer_kernel<TV><<<K, 128, 0, st>>>(T_epi + (size_t)(H - 1) * S * A * S, E, (long long)H * S, S, H,
                                                     resid);
    r = check_launch("episodic_last_layer_kernel");
    if (r != COLO_OK) return r;
    for (int h = H - 1; h >= 1; --h) {
      if (use_gemm) {  // many targets: the layer is one tiled GEMM (multirhs.cuh)
        ga.T = T_epi + (size_t)(h - 1) * S * A * S;
        ga.E_in = E + (size_t)h * S;
        ga.E_out = E + (size_t)(h - 1) * S;
        ga.exclude = h == H - 1;  // below the last layer F[h, es] is pinned to 1 already: no correction needed
        r = launch_hitting_gemm<TV>(ga, st);
      } else {
        a.T = T_epi + (size_t)(h - 1) * S * A * S;
        a.V_in = E + (size_t)h * S;
        a.V_out = E + (size_t)(h - 1) * S;
        r = launch_backup<TV>(&a, stream);
      }
      if (r != COLO_OK) return r;
    }
    ++it;
    if (++since >= check) {
      since = 0;
      COLO_CUDA_TRY(cudaMemcpyAsync(h_res.data(), resid, (size_t)K * sizeof(resid_t), cudaMemcpyDeviceToHost, st));
      COLO_CUDA_TRY(cudaMemcpyAsync(h_flags, flags, 2 * sizeof(int), cudaMemcpyDeviceToHost, st));
      COLO_CUDA_TRY(cudaStreamSynchronize(st));
      if (h_flags[1]) {
        rc = COLO_OVERFLOW;
        break;
      }
      resid_t mx = 0;
      for (auto v : h_res) mx = v > mx ? v : mx;
      TV res;
      if (sizeof(TV) == 4) {
        unsigned int u = (unsigned int)mx;
        float f;
        memcpy(&f, &u, 4);
        res = (TV)f;
      } else {
        unsigned long long u = (unsigned long long)mx;
        double f;
        memcpy(&f, &u, 8);
        res = (TV)f;
      }
      if (res < (TV)eps) {
        rc = COLO_OK;
        break;
      }
      if (check < 8) check *= 2;
    }
  }
  if (rc == COLO_OVERFLOW) return rc;
  episodic_diam_reduce_kernel<TV><<<1, 1024, 0, st>>>(E, K, H, S, d_out);
  r = check_launch("episodic_diam_reduce_kernel");
  if (r != COLO_OK) return r;
  TV hval = 0;
  COLO_CUDA_TRY(cudaMemcpyAsync(&hval, d_out, sizeof(TV), cudaMemcpyDeviceToHost, st));
  COLO_CUDA_TRY(cudaStreamSynchronize(st));
  out_host[0] = (double)hval;
  out_host[1] = (double)it;
  return rc;
}

template <typename TV>
int value_norm(const float* T, const TV* V, int S, int A, void* work, TV* out, void* stream) {
  COLO_ARG_CHECK(T && V && work && out, "T, V, work, out are required");
  cudaStream_t st = (cudaStream_t)stream;
  TV* Ev = (TV*)work;                                 // [S,A]
  TV* W = Ev + align_up((size_t)S * A, 64);           // [A,S]
  TV* rowmax = W + align_up((size_t)S * A, 64);       // [S]
  colo_backup_args a = {};
  a.T = T; a.B = 1; a.S = S; a.A = A; a.fold = COLO_FOLD_MAX; a.gamma = 1.0; a.r_const = 0.0;
  a.v_in_stride = S; a.q_stride = (long long)S * A; a.row0 = 0; a.nrows = S;
  a.V_in = V; a.V_out = nullptr; a.Q = Ev;  // pass 1: Ev[i,a] = sum_j T[i,a,j] V[j]
  int r = launch_backup<TV>(&a, stream);
  if (r != COLO_OK) return r;
  sqdev_kernel<TV><<<(S * A + 255) / 256, 256, 0, st>>>(V, Ev, S, A, W);
  r = check_launch("sqdev_kernel");
  if (r != COLO_OK) return r;
  // pass 2: sum_j T[i,a,j] * W[a,j], max over a into rowmax[i]
  a.V_in = W; a.v_action_stride = S; a.V_out = rowmax; a.v_out_stride = S; a.Q = nullptr;
  r = launch_backup<TV>(&a, stream);
  if (r != COLO_OK) return r;
  max_reduce_kernel<TV><<<1, 1024, 0, st>>>(rowmax, S, out, 1);
  return check_launch("max_reduce_kernel");
}

}  // namespace colo

// ---- C ABI --------------------------------------------------------------------------------------------------
extern "C" {

int colo_backup_f32(const colo_backup_args* args, void* stream) { return colo::launch_backup<float>(args, stream); }
int colo_backup_f64acc(const colo_backup_args* args, void* stream) { return colo::launch_backup<double>(args, stream); }

size_t colo_solve_work_bytes(long long B, long long S, int f64) {
  return f64 ? colo::solve_work_bytes<double>(B, S) : colo::solve_work_bytes<float>(B, S);
}

int colo_solve_discounted_f32(const float* T, const float* R, const float* pi, int B, int S, int A, float gamma,
                              float eps, float max_abs, long long max_iter, int fold, float* Q, float* V,
                              long long* iters_out_host, void* work, void* stream) {
  return colo::solve_discounted<float>(T, R, pi, B, S, A, gamma, eps, max_abs, max_iter, fold, Q, V, iters_out_host,
                                       work, stream);
}
int colo_solve_discounted_f64acc(const float* T, const float* R, const float* pi, int B, int S, int A, double gamma,
                                 double eps, double max_abs, long long max_iter, int fold, double* Q, double* V,
                                 long long* iters_out_host, void* work, void* stream) {
  return colo::solve_discounted<double>(T, R, pi, B, S, A, gamma, eps, max_abs, max_iter, fold, Q, V, iters_out_host,
                                        work, stream);
}

size_t colo_power_iteration_work_bytes(int S) {
  return colo::solve_work_bytes<double>(1, S) + colo::align_up((size_t)S * sizeof(float), 256) + 256;
}
int colo_power_iteration_f64(const float* M, int S, const double* x0, double eps, long long max_iter, double* x,
                             long long* iters_out_host, void* work, void* stream) {
  // x <- M x from x0 until max|dx| < eps: the synchronous sweep of the backup family with one action, no reward and
  // gamma = 1, so it runs on the same kernels (compressed rows on chip when M is sparse, streaming otherwise)
  COLO_ARG_CHECK(M && x0 && x && work && S > 0, "M, x0, x, work, S");
  float* zeros = (float*)work;
  COLO_CUDA_TRY(cudaMemsetAsync(zeros, 0, (size_t)S * sizeof(float), (cudaStream_t)stream));
  void* rest = (char*)work + colo::align_up((size_t)S * sizeof(float), 256);
  return colo::solve_discounted<double>(M, zeros, nullptr, 1, S, 1, 1.0, eps, 0.0, max_iter, COLO_FOLD_MAX, nullptr, x,
                                        iters_out_host, rest, stream, x0, true);
}

size_t colo_bias_series_work_bytes(int S) { return (size_t)4 * colo::align_up((size_t)S * sizeof(double), 256) + 256; }
int colo_bias_series_f64(const float* P, const float* avg_rewards, int S, int steps, double* h_out, void* work,
                         void* stream) {
  // _calculate_gain / _calculate_bias (colosseum/hardness/measures/value_norm.py:64-82):
  //   gain = P^steps r;  h = sum_{i < steps} P^i (r - gain)  -- 2*steps matrix-vector products on the backup kernel
  COLO_ARG_CHECK(P && avg_rewards && h_out && work && S > 0 && steps > 0, "P, avg_rewards, h_out, work, S, steps");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t stride = colo::align_up((size_t)S * sizeof(double), 256) / sizeof(double);
  double* a = (double*)work;
  double* b = a + stride;
  double* gain = b + stride;
  double* c = gain + stride;
  colo_backup_args g = {};
  g.T = P; g.B = 1; g.S = S; g.A = 1; g.fold = COLO_FOLD_MAX; g.gamma = 1.0; g.r_const = 0.0;
  g.t_stride = (long long)S * S; g.v_in_stride = S; g.v_out_stride = S; g.row0 = 0; g.nrows = S;
  colo::cast_f32_f64_kernel<<<(S + 255) / 256, 256, 0, st>>>(avg_rewards, a, S);
  int r = colo::check_launch("cast_f32_f64_kernel");
  if (r != COLO_OK) return r;
  double* cur = a;
  double* nxt = b;
  for (int i = 0; i < steps; ++i) {  // gain = P^steps r
    g.V_in = cur; g.V_out = nxt;
    r = colo::launch_backup<double>(&g, stream);
    if (r != COLO_OK) return r;
    double* t = cur; cur = nxt; nxt = t;
  }
  COLO_CUDA_TRY(cudaMemcpyAsync(gain, cur, (size_t)S * sizeof(double), cudaMemcpyDeviceToDevice, st));
  // v_0 = r - gain; h = sum_i v_i; v_{i+1} = P v_i
  colo::bias_init_kernel<<<(S + 255) / 256, 256, 0, st>>>(avg_rewards, gain, a, h_out, S);
  r = colo::check_launch("bias_init_kernel");
  if (r != COLO_OK) return r;
  cur = a; nxt = b;
  for (int i = 1; i < steps; ++i) {
    g.V_in = cur; g.V_out = nxt;
    r = colo::launch_backup<double>(&g, stream);
    if (r != COLO_OK) return r;
    colo::axpy_kernel<<<(S + 255) / 256, 256, 0, st>>>(nxt, h_out, S);
    r = colo::check_launch("axpy_kernel");
    if (r != COLO_OK) return r;
    double* t = cur; cur = nxt; nxt = t;
  }
  (void)c;
  return COLO_OK;
}

int colo_episodic_f32(const float* T, const float* R, const float* pi, int B, int S, int A, int H, int fold,
                      float max_value, float* Q, float* V, void* stream) {
  return colo::episodic<float>(T, R, pi, B, S, A, H, fold, max_value, Q, V, stream);
}
int colo_episodic_policies_f32(const float* T, const float* R, const float* pi, int B, int S, int A, int H, float* Q,
                               float* V, void* stream) {
  COLO_ARG_CHECK(T && R && pi && Q && V && B >= 0 && S > 0 && A > 0 && H >= 1, "T, R, pi, Q, V, B, S, A, H");
  if (B == 0) return COLO_OK;
  int handled = 0;
  return colo::episodic_batched<float>(T, R, pi, B, S, A, H, COLO_FOLD_PI, Q, V, &handled, (cudaStream_t)stream, true);
}

int colo_episodic_policies_f64acc(const float* T, const float* R, const float* pi, int B, int S, int A, int H,
                                  double* Q, double* V, void* stream) {
  COLO_ARG_CHECK(T && R && pi && Q && V && B >= 0 && S > 0 && A > 0 && H >= 1, "T, R, pi, Q, V, B, S, A, H");
  if (B == 0) return COLO_OK;
  int handled = 0;
  return colo::episodic_batched<double>(T, R, pi, B, S, A, H, COLO_FOLD_PI, Q, V, &handled, (cudaStream_t)stream, true);
}

int colo_episodic_f64acc(const float* T, const float* R, const float* pi, int B, int S, int A, int H, int fold,
                         double max_value, double* Q, double* V, void* stream) {
  return colo::episodic<double>(T, R, pi, B, S, A, H, fold, max_value, Q, V, stream);
}

int colo_continuous_form_values_f32(const float* T, const float* R, int S, int A, int H, double gamma, const int* pos_h,
                                    const int* pos_s, const float* p, int n_start, double eps, int max_eval, float* V,
                                    double* out_host, void* stream) {
  return colo::continuous_form_values<float>(T, R, S, A, H, gamma, pos_h, pos_s, p, n_start, eps, max_eval, V, out_host, stream);
}
int colo_continuous_form_values_f64acc(const float* T, const float* R, int S, int A, int H, double gamma, const int* pos_h,
                                       const int* pos_s, const float* p, int n_start, double eps, int max_eval, double* V,
                                       double* out_host, void* stream) {
  return colo::continuous_form_values<double>(T, R, S, A, H, gamma, pos_h, pos_s, p, n_start, eps, max_eval, V, out_host, stream);
}

size_t colo_diameter_continuous_work_bytes(int K, int S, int f64) {
  size_t e = f64 ? 8 : 4;
  const int K4 = (K + 3) & ~3;  // the resident path pads the targets to whole tiles of 4
  return colo::align_up((size_t)K4 * S * e, 256) +
         (f64 ? colo::solve_work_bytes<double>(K4, S) : colo::solve_work_bytes<float>(K4, S)) + 1024;
}
int colo_diameter_continuous_f32(const float* T, const int* targets, int K, int S, int A, float eps, float max_value,
                                 long long max_iter, void* work, double* out_host, void* stream) {
  return colo::diameter_continuous<float>(T, targets, K, S, A, eps, max_value, max_iter, work, out_host, stream);
}
int colo_diameter_continuous_f64acc(const float* T, const int* targets, int K, int S, int A, double eps,
                                    double max_value, long long max_iter, void* work, double* out_host,
                                    void* stream) {
  return colo::diameter_continuous<double>(T, targets, K, S, A, eps, max_value, max_iter, work, out_host, stream);
}

size_t colo_diameter_episodic_work_bytes(int K, int H, int S, int A, int f64) {
  size_t e = f64 ? 8 : 4;
  (void)A;
  return colo::align_up((size_t)K * H * S * e, 256) + colo::align_up((size_t)K * 8, 256) + 512;
}
int colo_diameter_episodic_f32(const float* T_epi, const int* targets, int K, int H, int S, int A, float eps,
                               float max_value, long long max_iter, void* work, double* out_host, void* stream) {
  return colo::diameter_episodic<float>(T_epi, targets, K, H, S, A, eps, max_value, max_iter, work, out_host, stream);
}
int colo_diameter_episodic_f64acc(const float* T_epi, const int* targets, int K, int H, int S, int A, double eps,
                                  double max_value, long long max_iter, void* work, double* out_host, void* stream) {
  return colo::diameter_episodic<double>(T_epi, targets, K, H, S, A, eps, max_value, max_iter, work, out_host, stream);
}

size_t colo_value_norm_work_bytes(int S, int A, int f64) {
  size_t e = f64 ? 8 : 4;
  return (2 * colo::align_up((size_t)S * A, 64) + colo::align_up((size_t)S, 64)) * e;
}
int colo_value_norm_f32(const float* T, const float* V, int S, int A, void* work, float* out, void* stream) {
  return colo::value_norm<float>(T, V, S, A, work, out, stream);
}
int colo_value_norm_f64acc(const float* T, const double* V, int S, int A, void* work, double* out, void* stream) {
  return colo::value_norm<double>(T, V, S, A, work, out, stream);
}

int colo_gaps_f64(const double* Q, const double* V, const unsigned char* mask, long long NS, int A, double reg,
                  double* out, void* stream) {
  COLO_ARG_CHECK(Q && V && out, "Q, V, out are required");
  colo::gaps_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(Q, V, mask, NS, A, reg, out);
  return colo::check_launch("gaps_kernel");
}

}  // extern "C"

extern "C" unsigned long long colo_backup_tma_sweeps(void) { return colo::g_tma_sweeps.load(); }
