// gauss_seidel.cu -- the reference's own iterate of discounted VI / PE: in-place (Gauss-Seidel) sweeps.
//
//   colosseum/dynamic_programming/infinite_horizon.py:121-142   _discounted_value_iteration
//   colosseum/dynamic_programming/infinite_horizon.py:167-184   _discounted_policy_evaluation
//       for s in range(S):  Q[s] = R[s] + gamma * T[s] @ V;  V[s] = max(Q[s])  (or sum(Q[s] * pi[s]))   -- V updated IN PLACE
//       stop when max|V_old - V| < epsilon after a sweep; return None as soon as |V[s]| > max_abs_value
//
// The streaming / resident / compressed-row solvers sweep synchronously (Jacobi): same fixed point, different
// early-stopped iterates (SURVEY.md section 7: 0.05 absolute at the reference's default epsilon = 1e-3).  This kernel
// reproduces the reference's iterate itself, for callers that want the numbers the reference returns at ITS stopping
// sweep: the state loop is sequential by definition, so ONE WARP owns one MDP instance -- V lives in the warp's slice
// of shared memory and is updated in place, the A row dot products of a state are lane-parallel (128-bit streaming
// loads of T, V quads from shared memory) and folded with shuffles, and the whole solve (all sweeps, stopping rule,
// overflow test) is one launch.  A batch of B instances runs B warps side by side: for large batches the kernel is
// HBM bound like the Jacobi sweep (T is streamed once per sweep) and needs about half the sweeps.
#include <vector>

#include <stdlib.h>

#include "tma_device.cuh"

namespace colo {

struct GsArgs {
  const float* T;   // [B][S,A,S]  (t_stride = 0: one T shared by all instances)
  const float* R;   // [B][S,A] or null: r_const
  const float* pi;  // [B][S,A] or null
  long long t_stride, r_stride;
  double r_const;
  const int* pin_index;  // per instance or null: V[pin] is held at pin_value (absorbing target of the diameter)
  double pin_value;
  // compressed rows (sparse T): row-major ELL, row (s*A + a) holds KMp slots of int2 (column, value bits), column -1 =
  // padding; KMp is a power of two.  cv_stride = slots between instances (0 = shared T)
  const int2* cv_rm;
  int KMp;
  long long cv_stride;
  int B, S, A, fold, warps_per_cta;
  double gamma, eps, max_abs;
  long long max_iter;
  void* V;          // out [B][S]
  void* Q;          // out [B][S,A]
  long long* iters; // [B]
  int* status;      // [B]
};

template <typename TV>
__device__ __forceinline__ void lds_v4(const TV* p, TV (&v)[4]);
template <>
__device__ __forceinline__ void lds_v4<float>(const float* p, float (&v)[4]) {
  const float4 t = *reinterpret_cast<const float4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
template <>
__device__ __forceinline__ void lds_v4<double>(const double* p, double (&v)[4]) {
  const double2 a = *reinterpret_cast<const double2*>(p);
  const double2 b = *reinterpret_cast<const double2*>(p + 2);
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}

constexpr int kGsAT = 4;  // actions held in registers at once

template <typename TV, bool VEC>
__global__ void __launch_bounds__(256) gs_solve_kernel(const GsArgs p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int S = p.S, A = p.A;
  const int Sp = (S + 3) & ~3;
  const long long b = (long long)blockIdx.x * p.warps_per_cta + warp;
  if (warp >= p.warps_per_cta || b >= p.B) return;  // warps are independent: no block-level barrier below
  TV* Vs = reinterpret_cast<TV*>(smem_raw) + (size_t)warp * Sp;
  for (int i = lane; i < Sp; i += 32) Vs[i] = TV(0);
  __syncwarp();
  const float* T = p.T + (size_t)b * p.t_stride;
  const float* R = p.R ? p.R + (size_t)b * p.r_stride : nullptr;
  const float* pi = p.pi ? p.pi + (size_t)b * S * A : nullptr;
  TV* Qg = p.Q ? reinterpret_cast<TV*>(p.Q) + (size_t)b * S * A : nullptr;
  const int pin = p.pin_index ? p.pin_index[b] : -1;
  const TV gamma = (TV)p.gamma;
  int status = COLO_MAX_ITER;
  long long it = 0;
  while (it < p.max_iter) {
    TV res = 0;
    bool overflow = false;
    for (int s = 0; s < S && !overflow; ++s) {
      if (s == pin) {  // absorbing target: T_es[es,:,es] = 1, R_es[es] = 0 -> V[es] stays at its value (diameter.py:85-90)
        const TV d0 = fabs((TV)p.pin_value - Vs[s]);
        res = d0 > res ? d0 : res;
        __syncwarp();
        if (lane == 0) Vs[s] = (TV)p.pin_value;
        __syncwarp();
        continue;
      }
      const float* Trow = T + (size_t)s * A * S;
      TV folded = p.fold == COLO_FOLD_MIN ? (TV)INFINITY : (p.fold == COLO_FOLD_MAX ? (TV)-INFINITY : (TV)0);
      for (int a0 = 0; a0 < A; a0 += kGsAT) {
        const int na = min(kGsAT, A - a0);
        TV acc[kGsAT];
#pragma unroll
        for (int i = 0; i < kGsAT; ++i) acc[i] = TV(0);
        if (VEC) {
          const int S4 = S >> 2;
          const float4* T4 = reinterpret_cast<const float4*>(Trow);
          for (int j4 = lane; j4 < S4; j4 += 32) {
            TV v[4];
            lds_v4<TV>(Vs + 4 * j4, v);
#pragma unroll
            for (int i = 0; i < kGsAT; ++i)
              if (i < na) {
                const float4 t = ldg_stream4(T4 + (size_t)(a0 + i) * S4 + j4);
                acc[i] += (TV)t.x * v[0] + (TV)t.y * v[1] + (TV)t.z * v[2] + (TV)t.w * v[3];
              }
          }
        } else {
          for (int j = lane; j < S; j += 32) {
            const TV v = Vs[j];
#pragma unroll
            for (int i = 0; i < kGsAT; ++i)
              if (i < na) acc[i] += (TV)ldg_stream1(Trow + (size_t)(a0 + i) * S + j) * v;
          }
        }
#pragma unroll
        for (int i = 0; i < kGsAT; ++i) acc[i] = warp_sum(acc[i]);  // every lane holds the full sums
#pragma unroll
        for (int i = 0; i < kGsAT; ++i)
          if (i < na) {
            const int a = a0 + i;
            const TV q = (R ? (TV)__ldg(R + (size_t)s * A + a) : (TV)p.r_const) + gamma * acc[i];
            if (lane == 0 && Qg) Qg[(size_t)s * A + a] = q;  // the reference returns the Q rows of the stopping sweep
            if (p.fold == COLO_FOLD_MAX) folded = q > folded ? q : folded;
            if (p.fold == COLO_FOLD_MIN) folded = q < folded ? q : folded;
            if (p.fold == COLO_FOLD_PI) folded += q * (TV)__ldg(pi + (size_t)s * A + a);
          }
      }
      const TV d = fabs(folded - Vs[s]);
      res = d > res ? d : res;
      __syncwarp();  // all lanes have read V[s] of the previous sweep
      if (lane == 0) Vs[s] = folded;  // in place: the following states of THIS sweep see it
      __syncwarp();
      if (p.max_abs > 0.0 && fabs((double)folded) > p.max_abs) overflow = true;  // infinite_horizon.py:136-138
    }
    ++it;
    if (overflow) { status = COLO_OVERFLOW; break; }
    if (res < (TV)p.eps) { status = COLO_OK; break; }  // :139-141
  }
  TV* Vg = reinterpret_cast<TV*>(p.V) + (size_t)b * S;
  for (int i = lane; i < S; i += 32) Vg[i] = Vs[i];
  if (lane == 0) {
    p.iters[b] = it;
    p.status[b] = status;
  }
}

// ---- the same in-place sweep with the rows of T prefetched by the TMA (cp.async.bulk, 1-D) ------------------------
// T does not depend on V: while the warp reduces state s, the A rows of the next states (A*S*4 contiguous bytes each)
// are already on their way into a ring of NST shared-memory stages, one bulk copy per state issued by lane 0 and
// signalled on an mbarrier.  The LDG version above waits for DRAM once per 128-column chunk of every state (the loop
// over j4 cannot issue past the accumulator dependence), which with one warp per MDP leaves the HBM pipe 2/3 full
// (measured on C4: 4.4 TB/s); here the warp only ever waits for a stage that was requested NST-1 states ago.
// Warps take MDP instances from a device counter (no wave quantisation when B is not a multiple of the warps in flight).
constexpr int kGsStages = 3;

template <typename TV>
__global__ void __launch_bounds__(256) gs_solve_tma_kernel(const GsArgs p, int* __restrict__ next_instance) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int S = p.S, A = p.A;
  const int Sp = (S + 3) & ~3;
  const uint32_t row_bytes = (uint32_t)A * S * 4;           // the A rows of one state, contiguous in T[s, :, :]
  const size_t stage_bytes = ((size_t)row_bytes + 127) & ~(size_t)127;
  const size_t per_warp = kGsStages * stage_bytes + (((size_t)Sp * sizeof(TV) + 127) & ~(size_t)127) + 128;
  unsigned char* mine = smem_raw + (size_t)warp * per_warp;
  float* stage0 = reinterpret_cast<float*>(mine);
  TV* Vs = reinterpret_cast<TV*>(mine + kGsStages * stage_bytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(mine + per_warp - 128);
  if (lane == 0) {
    for (int k = 0; k < kGsStages; ++k)
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(gs_smem_u32(bars + k)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  const TV gamma = (TV)p.gamma;
  const int S4 = S >> 2;
  unsigned long long seq = 0;  // stages consumed by this warp since the kernel started: slot = seq % NST, parity from seq / NST
  for (;;) {
    int b = 0;
    if (lane == 0) b = atomicAdd(next_instance, 1);
    b = __shfl_sync(FULL, b, 0);
    if (b >= p.B) break;
    for (int i = lane; i < Sp; i += 32) Vs[i] = TV(0);
    __syncwarp();
    const float* T = p.T + (size_t)b * p.t_stride;
    const float* R = p.R ? p.R + (size_t)b * p.r_stride : nullptr;
    const float* pi = p.pi ? p.pi + (size_t)b * S * A : nullptr;
    TV* Qg = p.Q ? reinterpret_cast<TV*>(p.Q) + (size_t)b * S * A : nullptr;
    const int pin = p.pin_index ? p.pin_index[b] : -1;
    // prime the ring with the first NST-1 states (state index runs modulo S across sweeps: T is the same every sweep)
    unsigned long long issued = seq;
    int s_issue = 0;
    if (lane == 0) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      for (int k = 0; k < kGsStages - 1; ++k) {
        gs_bulk_load(reinterpret_cast<unsigned char*>(stage0) + (issued % kGsStages) * stage_bytes,
                     T + (size_t)s_issue * A * S, row_bytes, bars + (issued % kGsStages));
        ++issued;
        s_issue = s_issue + 1 == S ? 0 : s_issue + 1;
      }
    }
    int status = COLO_MAX_ITER;
    long long it = 0;
    while (it < p.max_iter) {
      TV res = 0;
      bool overflow = false;
      for (int s = 0; s < S; ++s) {
        // keep the ring full: the stage consumed one state ago is free again (every lane passed the __syncwarp below)
        if (lane == 0) {
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          gs_bulk_load(reinterpret_cast<unsigned char*>(stage0) + (issued % kGsStages) * stage_bytes,
                       T + (size_t)s_issue * A * S, row_bytes, bars + (issued % kGsStages));
          ++issued;
          s_issue = s_issue + 1 == S ? 0 : s_issue + 1;
        }
        const int slot = (int)(seq % kGsStages);
        gs_bar_wait(bars + slot, (uint32_t)((seq / kGsStages) & 1ULL));
        ++seq;
        const float* Ts = reinterpret_cast<const float*>(reinterpret_cast<const unsigned char*>(stage0) + slot * stage_bytes);
        if (overflow) {  // the sweep is abandoned: keep consuming so that no copy is left in flight
          __syncwarp();
          continue;
        }
        if (s == pin) {  // absorbing target (diameter.py:85-90)
          const TV d0 = fabs((TV)p.pin_value - Vs[s]);
          res = d0 > res ? d0 : res;
          __syncwarp();
          if (lane == 0) Vs[s] = (TV)p.pin_value;
          __syncwarp();
          continue;
        }
        TV folded = p.fold == COLO_FOLD_MIN ? (TV)INFINITY : (p.fold == COLO_FOLD_MAX ? (TV)-INFINITY : (TV)0);
        for (int a0 = 0; a0 < A; a0 += kGsAT) {
          const int na = min(kGsAT, A - a0);
          TV acc[kGsAT];
#pragma unroll
          for (int i = 0; i < kGsAT; ++i) acc[i] = TV(0);
          for (int j4 = lane; j4 < S4; j4 += 32) {
            TV v[4];
            lds_v4<TV>(Vs + 4 * j4, v);
#pragma unroll
            for (int i = 0; i < kGsAT; ++i)
              if (i < na) {
                const float4 t = *reinterpret_cast<const float4*>(Ts + (size_t)(a0 + i) * S + 4 * j4);
                acc[i] += (TV)t.x * v[0] + (TV)t.y * v[1] + (TV)t.z * v[2] + (TV)t.w * v[3];
              }
          }
#pragma unroll
          for (int i = 0; i < kGsAT; ++i) acc[i] = warp_sum(acc[i]);
#pragma unroll
          for (int i = 0; i < kGsAT; ++i)
            if (i < na) {
              const int a = a0 + i;
              const TV q = (R ? (TV)__ldg(R + (size_t)s * A + a) : (TV)p.r_const) + gamma * acc[i];
              if (lane == 0 && Qg) Qg[(size_t)s * A + a] = q;
              if (p.fold == COLO_FOLD_MAX) folded = q > folded ? q : folded;
              if (p.fold == COLO_FOLD_MIN) folded = q < folded ? q : folded;
              if (p.fold == COLO_FOLD_PI) folded += q * (TV)__ldg(pi + (size_t)s * A + a);
            }
        }
        const TV d = fabs(folded - Vs[s]);
        res = d > res ? d : res;
        __syncwarp();  // all lanes have read V[s] of the previous sweep and this state's stage
        if (lane == 0) Vs[s] = folded;
        __syncwarp();
        if (p.max_abs > 0.0 && fabs((double)folded) > p.max_abs) overflow = true;
      }
      ++it;
      if (overflow) { status = COLO_OVERFLOW; break; }
      if (res < (TV)p.eps) { status = COLO_OK; break; }
    }
    // drain: NST-1 copies are still in flight (or landed): consume them before the ring is reused or the warp exits
    for (int k = 0; k < kGsStages - 1; ++k) {
      gs_bar_wait(bars + (int)(seq % kGsStages), (uint32_t)((seq / kGsStages) & 1ULL));
      ++seq;
    }
    __syncwarp();
    TV* Vg = reinterpret_cast<TV*>(p.V) + (size_t)b * S;
    for (int i = lane; i < S; i += 32) Vg[i] = Vs[i];
    if (lane == 0) {
      p.iters[b] = it;
      p.status[b] = status;
    }
    __syncwarp();
  }
}

__global__ void ell_to_row_major_kernel(const int* __restrict__ len, const int2* __restrict__ cv, long long rows, int S,
                                        int A, int kmax, int KMp, int2* __restrict__ cv_rm) {
  // slot-major ELL of sparse_hitting.cu (len[(g*A+a)*S+s], cv[((g*A+a)*kmax+i)*S+s]) -> row-major padded rows
  const long long n = rows * KMp;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (long long)gridDim.x * blockDim.x) {
    const long long r = t / KMp;
    const int i = (int)(t - r * KMp);
    const long long gs = r / A;
    const int a = (int)(r - gs * A);
    const long long g = gs / S;
    const int s = (int)(gs - g * S);
    const long long ga = g * A + a;
    int2 e = make_int2(-1, 0);
    if (i < len[ga * S + s]) e = cv[(ga * kmax + i) * S + s];
    cv_rm[t] = e;
  }
}

// In-place sweeps on compressed rows: the state loop stays sequential, the lanes of the warp take the (action, slot)
// pairs of the current state -- seg = min(KMp, 32) lanes per action, 32/seg actions per pass -- so a state of a
// benchmark MDP (A*kmax <= 32 entries) costs one load round, a segmented shuffle sum and one warp fold.
// ONEPASS (A * KMp <= 32): every lane holds exactly one (action, slot) entry of a state, so the entry and the reward
// of state s+1 -- which do not depend on V -- are fetched while state s is still being reduced.
template <typename TV, bool ONEPASS>
__global__ void __launch_bounds__(256) gs_sparse_kernel(const GsArgs p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int S = p.S, A = p.A, KMp = p.KMp;
  const int Sp = (S + 3) & ~3;
  const long long b = (long long)blockIdx.x * p.warps_per_cta + warp;
  if (warp >= p.warps_per_cta || b >= p.B) return;
  TV* Vs = reinterpret_cast<TV*>(smem_raw) + (size_t)warp * Sp;
  for (int i = lane; i < Sp; i += 32) Vs[i] = TV(0);
  __syncwarp();
  const int2* cv = p.cv_rm + (size_t)b * p.cv_stride;
  const float* R = p.R ? p.R + (size_t)b * p.r_stride : nullptr;
  const float* pi = p.pi ? p.pi + (size_t)b * S * A : nullptr;
  TV* Qg = p.Q ? reinterpret_cast<TV*>(p.Q) + (size_t)b * S * A : nullptr;
  const int pin = p.pin_index ? p.pin_index[b] : -1;
  const TV gamma = (TV)p.gamma;
  const int seg = KMp < 32 ? KMp : 32, chunks = KMp / seg, per_pass = 32 / seg;
  const int il = lane % seg, al = lane / seg;
  const TV ident = p.fold == COLO_FOLD_MIN ? (TV)INFINITY : (p.fold == COLO_FOLD_MAX ? (TV)-INFINITY : (TV)0);
  int status = COLO_MAX_ITER;
  long long it = 0;
  while (it < p.max_iter) {
    TV res = 0;
    bool overflow = false;
    int2 e_nx = make_int2(-1, 0);
    TV r_nx = TV(0);
    if (ONEPASS && al < A) {
      e_nx = __ldg(cv + (size_t)al * KMp + il);
      r_nx = R ? (TV)__ldg(R + al) : (TV)p.r_const;
    }
    for (int s = 0; s < S && !overflow; ++s) {
      TV folded;
      if (ONEPASS) {
        const int2 e = e_nx;
        const TV rr = r_nx;
        if (s + 1 < S && al < A) {  // state s+1's row and rewards: independent of V, in flight during the reduction
          e_nx = __ldg(cv + ((size_t)(s + 1) * A + al) * KMp + il);
          r_nx = R ? (TV)__ldg(R + (size_t)(s + 1) * A + al) : (TV)p.r_const;
        }
        if (s == pin) {
          folded = (TV)p.pin_value;
        } else {
          TV part = e.x >= 0 ? (TV)__int_as_float(e.y) * Vs[e.x] : TV(0);
          for (int o = seg >> 1; o > 0; o >>= 1) part += __shfl_xor_sync(FULL, part, o);
          TV cand = ident;
          if (al < A) {
            const TV q = rr + gamma * part;
            if (il == 0 && Qg) Qg[(size_t)s * A + al] = q;
            if (p.fold == COLO_FOLD_PI) cand = il == 0 ? q * (TV)__ldg(pi + (size_t)s * A + al) : (TV)0;
            else cand = q;
          }
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            const TV w = __shfl_xor_sync(FULL, cand, o);
            if (p.fold == COLO_FOLD_MAX) cand = w > cand ? w : cand;
            else if (p.fold == COLO_FOLD_MIN) cand = w < cand ? w : cand;
            else cand += w;
          }
          folded = cand;
        }
      } else
      if (s == pin) {
        folded = (TV)p.pin_value;
      } else {
        folded = ident;
        for (int a0 = 0; a0 < A; a0 += per_pass) {
          const int a = a0 + al;
          TV part = 0;
          if (a < A) {
            const int2* row = cv + ((size_t)s * A + a) * KMp;
            for (int c = 0; c < chunks; ++c) {
              const int2 e = __ldg(row + c * seg + il);
              if (e.x >= 0) part += (TV)__int_as_float(e.y) * Vs[e.x];
            }
          }
          for (int o = seg >> 1; o > 0; o >>= 1) part += __shfl_xor_sync(FULL, part, o);
          TV cand = ident;
          if (a < A) {
            const TV q = (R ? (TV)__ldg(R + (size_t)s * A + a) : (TV)p.r_const) + gamma * part;
            if (il == 0 && Qg) Qg[(size_t)s * A + a] = q;
            if (p.fold == COLO_FOLD_PI) cand = il == 0 ? q * (TV)__ldg(pi + (size_t)s * A + a) : (TV)0;
            else cand = q;
          }
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            const TV w = __shfl_xor_sync(FULL, cand, o);
            if (p.fold == COLO_FOLD_MAX) cand = w > cand ? w : cand;
            else if (p.fold == COLO_FOLD_MIN) cand = w < cand ? w : cand;
            else cand += w;
          }
          if (p.fold == COLO_FOLD_MAX) folded = cand > folded ? cand : folded;
          else if (p.fold == COLO_FOLD_MIN) folded = cand < folded ? cand : folded;
          else folded += cand;
        }
      }
      const TV d = fabs(folded - Vs[s]);
      res = d > res ? d : res;
      __syncwarp();
      if (lane == 0) Vs[s] = folded;
      __syncwarp();
      if (p.max_abs > 0.0 && fabs((double)folded) > p.max_abs) overflow = true;
    }
    ++it;
    if (overflow) { status = COLO_OVERFLOW; break; }
    if (res < (TV)p.eps) { status = COLO_OK; break; }
  }
  TV* Vg = reinterpret_cast<TV*>(p.V) + (size_t)b * S;
  for (int i = lane; i < S; i += 32) Vg[i] = Vs[i];
  if (lane == 0) {
    p.iters[b] = it;
    p.status[b] = status;
  }
}

// Compress T (groups = instances, or 1 when shared) into the row-major ELL of gs_sparse_kernel.  *cv_rm_out stays null
// when the rows are dense.  The caller frees it with cudaFreeAsync.
static int gs_compress(const float* T, long long groups, int S, int A, int2** cv_rm_out, int* KMp_out, cudaStream_t st) {
  *cv_rm_out = nullptr;
  SparseRows sp;
  int r = sparse_rows_build(T, groups * S * A, S, A, &sp, st);
  if (r != COLO_OK || sp.kmax == 0) return r;
  int KMp = 1;
  while (KMp < sp.kmax) KMp <<= 1;
  const long long rows = groups * S * A;
  int2* cv_rm = nullptr;
  COLO_CUDA_TRY(cudaMallocAsync(&cv_rm, (size_t)rows * KMp * sizeof(int2), st));
  const long long n = rows * KMp;
  const long long blocks = (n + 255) / 256;
  ell_to_row_major_kernel<<<(int)(blocks < 65535 ? blocks : 65535), 256, 0, st>>>(sp.len, (const int2*)sp.cv, rows, S, A,
                                                                                  sp.kmax, KMp, cv_rm);
  r = check_launch("ell_to_row_major_kernel");
  sparse_rows_free(&sp, st);
  if (r != COLO_OK) {
    cudaFreeAsync(cv_rm, st);
    return r;
  }
  *cv_rm_out = cv_rm;
  *KMp_out = KMp;
  return COLO_OK;
}

template <typename TV>
static int gs_launch(GsArgs a, void* stream) {
  int dev = 0, max_smem = 0;
  cudaGetDevice(&dev);
  if (cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess) max_smem = 227 * 1024;
  const size_t per_warp = (size_t)((a.S + 3) & ~3) * sizeof(TV);
  if (per_warp > (size_t)max_smem) {
    set_error("Gauss-Seidel solver: V of %d states does not fit shared memory", a.S);
    return COLO_ERR_ARG;
  }
  int W = (int)((size_t)max_smem / 2 / per_warp);  // two CTAs per SM
  W = W < 1 ? 1 : (W > 8 ? 8 : W);
  if (a.B < W) W = a.B;
  a.warps_per_cta = W;
  const size_t smem = per_warp * W;
  const bool vec = (a.S % 4 == 0) && ((uintptr_t)a.T % 16 == 0) && (a.t_stride % 4 == 0);
  const int grid = (a.B + W - 1) / W;
  cudaStream_t st = (cudaStream_t)stream;
  if (a.cv_rm != nullptr) {
    count_solver_path(COLO_PATH_GS_SPARSE);
    if (a.A * a.KMp <= 32) {
      auto k = gs_sparse_kernel<TV, true>;
      { const int _es = ensure_dynamic_smem((const void*)k, smem); if (_es != COLO_OK) return _es; }
      k<<<grid, W * 32, smem, st>>>(a);
    } else {
      auto k = gs_sparse_kernel<TV, false>;
      { const int _es = ensure_dynamic_smem((const void*)k, smem); if (_es != COLO_OK) return _es; }
      k<<<grid, W * 32, smem, st>>>(a);
    }
    return check_launch("gs_sparse_kernel");
  }
  // dense rows, 16-byte granular: the TMA-prefetch kernel (rows of a state staged by cp.async.bulk, NST-deep ring)
  static const bool no_tma = getenv("COLO_GS_NO_TMA") != nullptr;
  const size_t row_bytes = (size_t)a.A * a.S * 4;
  const size_t stage_bytes = (row_bytes + 127) & ~(size_t)127;
  const size_t tma_per_warp = kGsStages * stage_bytes + ((per_warp + 127) & ~(size_t)127) + 128;
  if (vec && !no_tma && row_bytes % 16 == 0 && tma_per_warp <= (size_t)max_smem - 1024) {
    int Wmax = (int)(((size_t)max_smem - 1024) / tma_per_warp);
    Wmax = Wmax > 8 ? 8 : Wmax;
    // every instance takes about as long as the others, so warps in flight that do not divide B leave the last round
    // partly empty (4,096 instances on 148 x 8 warps: 3.46 rounds -> 86 %): pick the warp count that fills the rounds
    int Wt = Wmax;
    double best_fill = 0.0;
    for (int w = Wmax; w >= (Wmax > 3 ? Wmax / 2 : 1); --w) {
      const long long in_flight = (long long)sm_count() * w;
      const long long rounds = (a.B + in_flight - 1) / in_flight;
      const double fill = (double)a.B / (double)(rounds * in_flight);
      if (fill > best_fill + 0.02) {
        best_fill = fill;
        Wt = w;
      }
    }
    if (a.B < Wt) Wt = a.B;
    a.warps_per_cta = Wt;
    const size_t smem_t = tma_per_warp * Wt;
    int* counter = nullptr;
    COLO_CUDA_TRY(cudaMallocAsync(&counter, sizeof(int), st));
    COLO_CUDA_TRY(cudaMemsetAsync(counter, 0, sizeof(int), st));
    const long long want = ((long long)a.B + Wt - 1) / Wt;
    const int grid_t = (int)(want < (long long)sm_count() ? want : (long long)sm_count());  // one CTA per SM, persistent
    auto k = gs_solve_tma_kernel<TV>;
    { const int _es = ensure_dynamic_smem((const void*)k, smem_t); if (_es != COLO_OK) return _es; }
    count_solver_path(COLO_PATH_GS_TMA);
    k<<<grid_t, Wt * 32, smem_t, st>>>(a, counter);
    const int r = check_launch("gs_solve_tma_kernel");
    cudaFreeAsync(counter, st);
    return r;
  }
  count_solver_path(COLO_PATH_GS_LDG);
  if (vec) {
    auto k = gs_solve_kernel<TV, true>;
    { const int _es = ensure_dynamic_smem((const void*)k, smem); if (_es != COLO_OK) return _es; }
    k<<<grid, W * 32, smem, st>>>(a);
  } else {
    auto k = gs_solve_kernel<TV, false>;
    { const int _es = ensure_dynamic_smem((const void*)k, smem); if (_es != COLO_OK) return _es; }
    k<<<grid, W * 32, smem, st>>>(a);
  }
  return check_launch("gs_solve_kernel");
}

template <typename TV>
int gs_solve(const float* T, const float* R, const float* pi, int B, int S, int A, double gamma, double eps,
             double max_abs, long long max_iter, int fold, TV* Q, TV* V, long long* iters_dev, int* status_dev,
             void* stream) {
  COLO_ARG_CHECK(T && R && Q && V && iters_dev && status_dev, "T, R, Q, V, iters, status are required");
  COLO_ARG_CHECK(B >= 0 && S > 0 && A > 0 && fold >= 0 && fold <= 2 && (fold != COLO_FOLD_PI || pi), "B, S, A, fold, pi");
  if (B == 0) return COLO_OK;
  GsArgs a = {};
  a.T = T; a.R = R; a.pi = pi; a.B = B; a.S = S; a.A = A; a.fold = fold;
  a.t_stride = (long long)S * A * S; a.r_stride = (long long)S * A;
  a.gamma = gamma; a.eps = eps; a.max_abs = max_abs; a.max_iter = max_iter; a.V = V; a.Q = Q;
  a.iters = iters_dev; a.status = status_dev;
  int2* cv_rm = nullptr;
  int r = gs_compress(T, B, S, A, &cv_rm, &a.KMp, (cudaStream_t)stream);
  if (r != COLO_OK) return r;
  a.cv_rm = cv_rm;
  a.cv_stride = (long long)S * A * a.KMp;
  r = gs_launch<TV>(a, stream);
  if (cv_rm) cudaFreeAsync(cv_rm, (cudaStream_t)stream);
  return r;
}

template <typename TV>
__global__ void neg_min_per_row_kernel(const TV* __restrict__ V, int K, int S, TV* __restrict__ out) {
  // out[k] = -min_s V[k,s]   (diameter.py:95); one warp per target
  const int lane = threadIdx.x & 31;
  const int k = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (k >= K) return;
  TV m = INFINITY;
  for (int s = lane; s < S; s += 32) m = V[(size_t)k * S + s] < m ? V[(size_t)k * S + s] : m;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const TV w = __shfl_xor_sync(FULL, m, o);
    m = w < m ? w : m;
  }
  if (lane == 0) out[k] = -m;
}

// The reference's continuous diameter, iterate for iterate (diameter.py:76-106): for every target es a discounted VI
// with gamma = 1 on T_es (es absorbing) and R_es = -1 (0 at es), in-place sweeps, eps = 1e-3; diameter = max_es -min V.
// All K solves share T (t_stride = 0): K warps stream it from L2.
template <typename TV>
int gs_diameter(const float* T, const int* targets, int K, int S, int A, double eps, double max_value,
                long long max_iter, void* work, double* out_host, void* stream) {
  COLO_ARG_CHECK(T && targets && work && out_host && K > 0 && S > 0 && A > 0, "T, targets, work, out_host, K, S, A");
  cudaStream_t st = (cudaStream_t)stream;
  char* w = (char*)work;
  TV* V = (TV*)w;
  w += ((size_t)K * S * sizeof(TV) + 255) / 256 * 256;
  TV* d = (TV*)w;
  w += ((size_t)K * sizeof(TV) + 255) / 256 * 256;
  long long* iters = (long long*)w;
  w += ((size_t)K * sizeof(long long) + 255) / 256 * 256;
  int* status = (int*)w;
  GsArgs a = {};
  a.T = T; a.R = nullptr; a.r_const = -1.0; a.B = K; a.S = S; a.A = A; a.fold = COLO_FOLD_MAX;
  a.t_stride = 0; a.r_stride = 0; a.pin_index = targets; a.pin_value = 0.0;
  a.gamma = 1.0; a.eps = eps; a.max_abs = max_value; a.max_iter = max_iter; a.V = V; a.Q = nullptr;
  a.iters = iters; a.status = status;
  int2* cv_rm = nullptr;
  int r = gs_compress(T, 1, S, A, &cv_rm, &a.KMp, st);
  if (r != COLO_OK) return r;
  a.cv_rm = cv_rm;
  a.cv_stride = 0;  // every target shares T
  r = gs_launch<TV>(a, stream);
  if (cv_rm) cudaFreeAsync(cv_rm, st);
  if (r != COLO_OK) return r;
  neg_min_per_row_kernel<TV><<<(K * 32 + 255) / 256, 256, 0, st>>>(V, K, S, d);
  r = check_launch("neg_min_per_row_kernel");
  if (r != COLO_OK) return r;
  std::vector<TV> hd((size_t)K);
  std::vector<long long> hit((size_t)K);
  std::vector<int> hst((size_t)K);
  COLO_CUDA_TRY(cudaMemcpyAsync(hd.data(), d, (size_t)K * sizeof(TV), cudaMemcpyDeviceToHost, st));
  COLO_CUDA_TRY(cudaMemcpyAsync(hit.data(), iters, (size_t)K * sizeof(long long), cudaMemcpyDeviceToHost, st));
  COLO_CUDA_TRY(cudaMemcpyAsync(hst.data(), status, (size_t)K * sizeof(int), cudaMemcpyDeviceToHost, st));
  COLO_CUDA_TRY(cudaStreamSynchronize(st));
  double best = 0.0;
  long long mx = 0;
  int rc = COLO_OK;
  for (int k = 0; k < K; ++k) {
    if (hst[k] == COLO_OVERFLOW) return COLO_OVERFLOW;
    if (hst[k] == COLO_MAX_ITER) rc = COLO_MAX_ITER;
    if ((double)hd[k] > best) best = (double)hd[k];
    if (hit[k] > mx) mx = hit[k];
  }
  out_host[0] = best;
  out_host[1] = (double)mx;
  return rc;
}

}  // namespace colo

extern "C" {

int colo_solve_discounted_gs_f32(const float* T, const float* R, const float* pi, int B, int S, int A, float gamma,
                                 float eps, float max_abs, long long max_iter, int fold, float* Q, float* V,
                                 long long* iters_dev, int* status_dev, void* stream) {
  return colo::gs_solve<float>(T, R, pi, B, S, A, gamma, eps, max_abs, max_iter, fold, Q, V, iters_dev, status_dev, stream);
}
int colo_solve_discounted_gs_f64acc(const float* T, const float* R, const float* pi, int B, int S, int A, double gamma,
                                    double eps, double max_abs, long long max_iter, int fold, double* Q, double* V,
                                    long long* iters_dev, int* status_dev, void* stream) {
  return colo::gs_solve<double>(T, R, pi, B, S, A, gamma, eps, max_abs, max_iter, fold, Q, V, iters_dev, status_dev, stream);
}

size_t colo_diameter_continuous_gs_work_bytes(int K, int S, int f64) {
  const size_t e = f64 ? 8 : 4;
  return ((size_t)K * S * e + 255) / 256 * 256 + ((size_t)K * e + 255) / 256 * 256 + ((size_t)K * 8 + 255) / 256 * 256 +
         ((size_t)K * 4 + 255) / 256 * 256 + 256;
}
int colo_diameter_continuous_gs_f32(const float* T, const int* targets, int K, int S, int A, float eps, float max_value,
                                    long long max_iter, void* work, double* out_host, void* stream) {
  return colo::gs_diameter<float>(T, targets, K, S, A, eps, max_value, max_iter, work, out_host, stream);
}
int colo_diameter_continuous_gs_f64acc(const float* T, const int* targets, int K, int S, int A, double eps,
                                       double max_value, long long max_iter, void* work, double* out_host, void* stream) {
  return colo::gs_diameter<double>(T, targets, K, S, A, eps, max_value, max_iter, work, out_host, stream);
}

}  // extern "C"
