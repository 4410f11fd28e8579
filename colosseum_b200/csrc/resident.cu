// resident.cu -- on-chip resident Bellman solver for MDPs whose T fits the shared memory of one thread-block cluster.
//
// The streaming backup kernel (backup.cu) is the right tool when one sweep moves megabytes: it runs at the HBM
// roofline.  The benchmark families of the reference are small (S = 16 ... ~950, T = 5 KB ... ~3 MB) and their
// solves need hundreds to thousands of sweeps (colosseum/dynamic_programming/infinite_horizon.py:121-142; the
// diameter, colosseum/hardness/measures/diameter.py:76-106, needs that for each of S targets).  Launching one
// kernel per sweep makes such a solve launch-latency bound (~10 us per sweep, measured), slower than the
// reference's numba loop for the smallest MDPs.  Here ONE launch does the whole solve:
//
//   * a cluster of C CTAs (C = 1..16, 227 KB of shared memory each, up to 3.6 MB per cluster) owns one problem;
//     CTA r keeps the T rows of its slice of states resident in shared memory for the entire solve;
//   * every CTA holds the full value vector(s) in its own shared memory (ping-pong); after a sweep each CTA
//     pushes its new V entries into all C copies through distributed shared memory, together with its partial
//     max|dV| and overflow flag, and ONE cluster barrier per sweep makes them visible -- the barrier is the only
//     synchronisation, no global memory traffic, no host round trip;
//   * NV value vectors (1 or 4) are iterated at once against the same T rows: the 4 targets of a diameter tile
//     reuse every T quad loaded from shared memory (the reuse that turns the GEMV into a small GEMM).
#include <cooperative_groups.h>
#include <stdlib.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace colo {

constexpr int kResThreads = 512;
constexpr int kResWarps = kResThreads / 32;
constexpr int kResAT = 4;  // actions per register tile

struct ResidentArgs {
  const float* T;   // [B or 1][S,A,S]
  const float* R;   // [B or 1][S,A] or null
  const float* pi;  // [B][S,A] or null
  void* V;          // out [B*NV][S]
  void* Q;          // out [B*NV][S,A] or null
  long long t_stride, r_stride;  // elements between problems (0 = shared)
  int B, S, A, fold, C, Sp;      // C = cluster size, Sp = S rounded up to 4
  int rows_per_cta;              // states per CTA
  double gamma, r_const, eps, max_abs;
  int overflow_signed;
  long long max_iter;
  int episodic_H;                // > 0: exactly H sweeps, layer h of V/Q stored every sweep (finite_horizon.py)
  const int* pin_index;          // per value vector or null
  double pin_value;
  long long* iters_out;          // [B*NV] or null
  int* status_out;               // [B] : 0 ok, 1 overflow, 2 max_iter
};

template <typename TV>
__device__ __forceinline__ void lds4(const TV* p, TV (&v)[4]);
template <>
__device__ __forceinline__ void lds4<float>(const float* p, float (&v)[4]) {
  float4 t = *reinterpret_cast<const float4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
template <>
__device__ __forceinline__ void lds4<double>(const double* p, double (&v)[4]) {
  double2 a = *reinterpret_cast<const double2*>(p);
  double2 b = *reinterpret_cast<const double2*>(p + 2);
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}

template <typename TV, int FOLD, int NV>
__global__ void __launch_bounds__(kResThreads, 1) resident_solve_kernel(const ResidentArgs p) {
  cg::cluster_group cluster = cg::this_cluster();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int S = p.S, A = p.A, Sp = p.Sp, C = p.C;
  const int rank = (int)cluster.block_rank();
  const int prob = blockIdx.x / C;  // problem (MDP instance or tile of NV targets)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int s_begin = min(S, rank * p.rows_per_cta), s_end = min(S, s_begin + p.rows_per_cta);
  const int n_local = s_end - s_begin;

  // ---- shared memory carve-up: T slice | R slice | V[2][NV][Sp]
  float* Tsm = reinterpret_cast<float*>(smem_raw);
  size_t off = ((size_t)p.rows_per_cta * A * Sp * sizeof(float) + 15) & ~(size_t)15;
  float* Rsm = reinterpret_cast<float*>(smem_raw + off);  // [rows_per_cta * A]
  off += ((size_t)p.rows_per_cta * A * sizeof(float) + 15) & ~(size_t)15;
  TV* Vsm = reinterpret_cast<TV*>(smem_raw + off);  // [2][NV][Sp]
  // cluster-wide max|dV| of a sweep: every warp pushes its partial into slot (sweep % 3) of EVERY CTA with a
  // distributed-shared-memory atomicMax (float bits; +inf encodes overflow); slot (sweep+2) % 3 is recycled
  __shared__ unsigned int s_res[3];

  // ---- load this CTA's T and R rows once (T zero padded to Sp), zero V
  {
    const float* Tg = p.T + (size_t)prob * p.t_stride + (size_t)s_begin * A * S;
    const int rows = n_local * A;
    for (long long i = threadIdx.x; i < (long long)rows * Sp; i += kResThreads) {
      const int r = (int)(i / Sp), j = (int)(i - (long long)r * Sp);
      Tsm[i] = j < S ? ldg_stream1(Tg + (size_t)r * S + j) : 0.f;
    }
    const float* Rg = p.R ? p.R + (size_t)prob * p.r_stride + (size_t)s_begin * A : nullptr;
    for (int i = threadIdx.x; i < rows; i += kResThreads) Rsm[i] = Rg ? Rg[i] : (float)p.r_const;
    for (int i = threadIdx.x; i < 2 * NV * Sp; i += kResThreads) Vsm[i] = TV(0);
    if (threadIdx.x < 3) s_res[threadIdx.x] = 0u;
  }
  int pins[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) pins[v] = p.pin_index ? p.pin_index[(size_t)prob * NV + v] : -1;
  if (C == 1) __syncthreads(); else cluster.sync();

  const TV gamma = (TV)p.gamma;
  const float* pig = p.pi ? p.pi + (size_t)prob * (p.episodic_H > 0 ? p.episodic_H : 1) * S * A : nullptr;
  TV* Vg = reinterpret_cast<TV*>(p.V);
  TV* Qg = reinterpret_cast<TV*>(p.Q);

  int cur = 0;
  long long it = 0;
  int status = COLO_MAX_ITER;
  const long long n_sweeps = p.episodic_H > 0 ? p.episodic_H : p.max_iter;
  bool final_pass = false;  // one extra pass after convergence re-derives Q (and V) of the last sweep for output

  while (true) {
    const TV* Vin = Vsm + (size_t)cur * NV * Sp;
    TV* Vout = Vsm + (size_t)(cur ^ 1) * NV * Sp;
    float res = 0.f;
    const bool store = final_pass || p.episodic_H > 0;
    const long long layer = p.episodic_H > 0 ? (p.episodic_H - 1 - it) : 0;  // episodic: sweep `it` fills layer H-1-it
    const int slot = (int)(it % 3);

    for (int sl = warp; sl < n_local; sl += kResWarps) {
      const int s = s_begin + sl;
      TV folded[NV];
#pragma unroll
      for (int v = 0; v < NV; ++v)
        folded[v] = FOLD == COLO_FOLD_MIN ? (TV)INFINITY : (FOLD == COLO_FOLD_MAX ? (TV)-INFINITY : (TV)0);
      for (int a0 = 0; a0 < A; a0 += kResAT) {
        const int na = min(kResAT, A - a0);
        TV acc[NV][kResAT];
#pragma unroll
        for (int v = 0; v < NV; ++v)
#pragma unroll
          for (int i = 0; i < kResAT; ++i) acc[v][i] = TV(0);
        const float* Trow = Tsm + ((size_t)sl * A + a0) * Sp;
        for (int j = lane * 4; j < Sp; j += 128) {
          TV vv[NV][4];
#pragma unroll
          for (int v = 0; v < NV; ++v) lds4<TV>(Vin + (size_t)v * Sp + j, vv[v]);
#pragma unroll
          for (int i = 0; i < kResAT; ++i)
            if (i < na) {
              const float4 t = *reinterpret_cast<const float4*>(Trow + (size_t)i * Sp + j);
#pragma unroll
              for (int v = 0; v < NV; ++v)
                acc[v][i] += (TV)t.x * vv[v][0] + (TV)t.y * vv[v][1] + (TV)t.z * vv[v][2] + (TV)t.w * vv[v][3];
            }
        }
        // butterfly reduction: afterwards EVERY lane holds the full sums, so the epilogue below is computed
        // redundantly by all lanes (no broadcast) and the stores are spread over the lanes
#pragma unroll
        for (int v = 0; v < NV; ++v)
#pragma unroll
          for (int i = 0; i < kResAT; ++i) acc[v][i] = warp_sum(acc[v][i]);
#pragma unroll
        for (int i = 0; i < kResAT; ++i)
          if (i < na) {
            const int a = a0 + i;
            const TV r = (TV)Rsm[sl * A + a];
#pragma unroll
            for (int v = 0; v < NV; ++v) {
              const TV q = r + gamma * acc[v][i];
              if (store && Qg && lane == 0) {
                const size_t vec = (size_t)prob * NV + v;
                if (p.episodic_H > 0)
                  Qg[((vec * (p.episodic_H + 1) + layer) * S + s) * A + a] = q;
                else
                  Qg[(vec * S + s) * A + a] = q;
              }
              if (FOLD == COLO_FOLD_MAX) folded[v] = q > folded[v] ? q : folded[v];
              if (FOLD == COLO_FOLD_MIN) folded[v] = q < folded[v] ? q : folded[v];
              if (FOLD == COLO_FOLD_PI)  // episodic PE: pi is [B][H][S,A], one layer per sweep
                folded[v] += q * (TV)__ldg(pig + ((size_t)layer * S + s) * A + a);
            }
          }
      }
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        TV f = folded[v];
        if (pins[v] == s) f = (TV)p.pin_value;
        const float d = (float)fabs(f - Vin[(size_t)v * Sp + s]);
        res = d > res ? d : res;
        if (p.max_abs > 0.0 && (p.overflow_signed ? (double)f : fabs((double)f)) > p.max_abs) res = INFINITY;
        if (store && lane == 0) {
          const size_t vec = (size_t)prob * NV + v;
          if (p.episodic_H > 0)
            Vg[(vec * (p.episodic_H + 1) + layer) * S + s] = f;
          else
            Vg[vec * S + s] = f;
        }
        // lane r pushes the new entry into CTA r's copy of the next V (distributed shared memory)
        if (C == 1) {
          if (lane == 0) Vout[(size_t)v * Sp + s] = f;
        } else if (lane < C) {
          *cluster.map_shared_rank(Vout + (size_t)v * Sp + s, lane) = f;
        }
      }
    }
    // ---- cluster-wide max residual: lane r of every warp pushes the warp's partial to CTA r's slot
    if (!final_pass) {
      if (C == 1) {
        if (lane == 0 && res > 0.f) atomicMax(&s_res[slot], __float_as_uint(res));
      } else if (lane < C && res > 0.f) {
        atomicMax(cluster.map_shared_rank(&s_res[slot], lane), __float_as_uint(res));
      }
    }
    if (C == 1) __syncthreads(); else cluster.sync();  // the one barrier of the sweep
    if (final_pass) break;
    const float gres = __uint_as_float(s_res[slot]);
    if (threadIdx.x == 0) s_res[(slot + 2) % 3] = 0u;  // recycled two sweeps from now; nobody reads or writes it now
    ++it;
    if (isinf(gres)) { status = COLO_OVERFLOW; break; }
    if (p.episodic_H > 0) {
      cur ^= 1;
      if (it >= n_sweeps) { status = COLO_OK; break; }
      continue;
    }
    if (gres < (float)p.eps) {
      // converged: the reference returns the Q and V of THIS sweep; redo it from the same V_in, storing outputs
      status = COLO_OK;
      final_pass = true;
      continue;  // cur unchanged: V_in is still the input of the converged sweep
    }
    if (it >= n_sweeps) {
      status = COLO_MAX_ITER;
      final_pass = true;
      continue;
    }
    cur ^= 1;
  }
  if (threadIdx.x == 0 && rank == 0) {
    if (p.status_out) p.status_out[prob] = status;
    if (p.iters_out)
      for (int v = 0; v < NV; ++v) p.iters_out[(size_t)prob * NV + v] = it;
  }
  if (C > 1) cluster.sync();  // no CTA may exit while peers can still address its shared memory
}

// ---- host side -------------------------------------------------------------------------------------------------
struct ResidentPlan {
  int C, rows_per_cta, Sp;
  size_t smem;
  bool ok;
};

template <typename TV>
static ResidentPlan plan_resident(int S, int A, int NV, int max_smem) {
  ResidentPlan pl{};
  pl.Sp = (S + 3) & ~3;
  pl.ok = false;
  for (int C = 1; C <= 16; C *= 2) {
    const int rows = (S + C - 1) / C;
    size_t need = (((size_t)rows * A * pl.Sp * sizeof(float)) + 15) & ~(size_t)15;
    need += (((size_t)rows * A * sizeof(float)) + 15) & ~(size_t)15;
    need += (size_t)2 * NV * pl.Sp * sizeof(TV) + 64;
    if (need <= (size_t)max_smem) {
      // prefer enough CTAs that a CTA's slice is at most ~64 KB (more SMs, more shared-memory bandwidth), while it fits
      pl.C = C;
      pl.rows_per_cta = rows;
      pl.smem = need;
      pl.ok = true;
      if ((size_t)rows * A * pl.Sp * sizeof(float) <= 64 * 1024 || C == 16) break;
    }
  }
  return pl;
}

template <typename TV, int FOLD, int NV>
static int launch_resident_3(const ResidentArgs& a, size_t smem, cudaStream_t st) {
  auto kern = resident_solve_kernel<TV, FOLD, NV>;
  { const int _es = ensure_dynamic_smem((const void*)kern, smem); if (_es != COLO_OK) return _es; }
  if (a.C > 8) COLO_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(a.B * a.C));
  cfg.blockDim = dim3(kResThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)a.C;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int max_clusters = 0;
  cudaError_t e = cudaOccupancyMaxActiveClusters(&max_clusters, kern, &cfg);
  if (e != cudaSuccess || max_clusters < 1) {
    cudaGetLastError();
    set_error("resident solver: a cluster of %d CTAs with %zu B of shared memory cannot be scheduled", a.C, smem);
    return COLO_ERR_ARG;
  }
  count_solver_path(COLO_PATH_RESIDENT);
  COLO_CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, a));
  return check_launch("resident_solve_kernel");
}

template <typename TV, int NV>
static int launch_resident_2(const ResidentArgs& a, size_t smem, cudaStream_t st) {
  switch (a.fold) {
    case COLO_FOLD_MAX: return launch_resident_3<TV, COLO_FOLD_MAX, NV>(a, smem, st);
    case COLO_FOLD_PI: return launch_resident_3<TV, COLO_FOLD_PI, NV>(a, smem, st);
    default: return launch_resident_3<TV, COLO_FOLD_MIN, NV>(a, smem, st);
  }
}

static int max_optin_smem() {
  static int cached = 0;
  if (!cached) {
    int dev = 0, v = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess || v <= 0) v = 227 * 1024;
    cached = v - 1024;  // room for the kernel's static shared memory
  }
  return cached;
}

// returns 1 if the problem fits the resident solver (and fills *C_out), 0 otherwise
template <typename TV>
int resident_fits(int S, int A, int NV, int* C_out) {
  ResidentPlan pl = plan_resident<TV>(S, A, NV, max_optin_smem());
  if (pl.ok && C_out) *C_out = pl.C;
  return pl.ok ? 1 : 0;
}

template <typename TV>
int resident_solve(const colo_resident_args* u, void* stream) {
  COLO_ARG_CHECK(u && u->T && u->V && u->status_out, "T, V, status_out are required");
  COLO_ARG_CHECK(u->B > 0 && u->S > 0 && u->A > 0, "B, S, A");
  COLO_ARG_CHECK(u->NV == 1 || u->NV == 4, "NV must be 1 or 4");
  COLO_ARG_CHECK(u->fold >= 0 && u->fold <= 2 && (u->fold != COLO_FOLD_PI || u->pi), "fold / pi");
  ResidentPlan pl = plan_resident<TV>(u->S, u->A, u->NV, max_optin_smem());
  if (!pl.ok) {
    set_error("resident solver: S=%d A=%d does not fit the shared memory of a 16-CTA cluster", u->S, u->A);
    return COLO_ERR_ARG;
  }
  ResidentArgs a = {};
  a.T = u->T; a.R = u->R; a.pi = u->pi; a.V = u->V; a.Q = u->Q;
  a.t_stride = u->t_stride; a.r_stride = u->r_stride;
  a.B = u->B; a.S = u->S; a.A = u->A; a.fold = u->fold; a.C = pl.C; a.Sp = pl.Sp; a.rows_per_cta = pl.rows_per_cta;
  a.gamma = u->gamma; a.r_const = u->r_const; a.eps = u->eps; a.max_abs = u->max_abs; a.max_iter = u->max_iter;
  a.overflow_signed = u->overflow_signed;
  a.episodic_H = u->episodic_H; a.pin_index = u->pin_index; a.pin_value = u->pin_value;
  a.iters_out = u->iters_out; a.status_out = u->status_out;
  cudaStream_t st = (cudaStream_t)stream;
  return u->NV == 4 ? launch_resident_2<TV, 4>(a, pl.smem, st) : launch_resident_2<TV, 1>(a, pl.smem, st);
}

int resident_fits_any(int S, int A, int NV, bool f64, int* C_out) {
  return f64 ? resident_fits<double>(S, A, NV, C_out) : resident_fits<float>(S, A, NV, C_out);
}
int resident_solve_any(const colo_resident_args* args, bool f64, void* stream) {
  return f64 ? resident_solve<double>(args, stream) : resident_solve<float>(args, stream);
}
bool resident_enabled() {
  static const bool on = getenv("COLO_NO_RESIDENT") == nullptr;
  return on;
}

}  // namespace colo

extern "C" {
int colo_resident_fits(int S, int A, int NV, int f64, int* cluster_size_out) {
  return f64 ? colo::resident_fits<double>(S, A, NV, cluster_size_out) : colo::resident_fits<float>(S, A, NV, cluster_size_out);
}
int colo_resident_solve_f32(const colo_resident_args* args, void* stream) {
  return colo::resident_solve<float>(args, stream);
}
int colo_resident_solve_f64acc(const colo_resident_args* args, void* stream) {
  return colo::resident_solve<double>(args, stream);
}
}
