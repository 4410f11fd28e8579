// multirhs.cuh -- the multi-target hitting-time sweep of the diameter as a tiled GEMM (included by backup.cu).
//
// colosseum/hardness/measures/diameter.py:76-106 solves, for every target state k, a value iteration with gamma = 1,
// reward -1 and k absorbing.  All K targets share T, so one synchronous sweep over all of them is
//     C[(s,a), k] = sum_j T[s,a,j] * E[k,j]          an (S*A x S) . (S x K) product, 2*S*A*S*K flop
//     E'[k,s]     = (s == target_k) ? 0 : min_a (1 + C[(s,a), k])
// i.e. a genuine GEMM with a min-over-actions epilogue: arithmetic intensity grows with K, and for the benchmark
// families (S = K up to ~950, T up to 11 MB, L2 resident) the sweep is compute bound, not HBM bound.  The GEMV-style
// streaming kernel re-reads T from L2 once per target; this kernel reads each T tile once per BN targets.
//
// Tiling: a CTA owns BM states x BN targets and loops over the actions; for each action it accumulates the
// BM x BN x S product in registers (TM x TN per thread) from k-major shared-memory tiles that are filled through
// registers (global -> register prefetch of the next tile overlaps the FMAs of the current one), then folds
// min(best, 1 + acc).  The epilogue pins the target, carries converged targets forward, stores E' coalesced and
// reduces max|dE| per target (one atomicMax per target per tile).  fp32 or fp64 accumulation (T stays fp32).
#pragma once

namespace colo {

struct HittingGemmArgs {
  const float* T;        // [S,A,S]
  const void* E_in;      // [K][e_stride] TV
  void* E_out;           // [K][e_stride] TV
  long long e_stride;    // elements between targets
  const int* targets;    // [K]
  const unsigned char* active;  // [K] or null
  void* resid;           // [K] float/double bits, atomicMax
  int S, A, K;
  double max_value;      // > 0: overflow test E' > max_value
  int* overflow_flag;
  double pin_value;      // E'[k, target_k]: 0 for the continuous form, 1 for the episodic F = 1 + ETs form
  int exclude;           // != 0: the next-state term j == target_k uses exclude_value instead of E[k, target_k]
  double exclude_value;  //       (episodic diameter, diameter.py:301-306: reaching the target costs exactly one step)
  int resid_vs_out;      // != 0: max|dE| compares with the previous content of E_out (in-place layered iteration)
};

template <typename TV>
__device__ __forceinline__ void lds4(const TV* p, TV (&v)[4]);
template <>
__device__ __forceinline__ void lds4<float>(const float* p, float (&v)[4]) {
  const float4 t = *reinterpret_cast<const float4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
template <>
__device__ __forceinline__ void lds4<double>(const double* p, double (&v)[4]) {
  const double2 a = *reinterpret_cast<const double2*>(p);
  const double2 b = *reinterpret_cast<const double2*>(p + 2);
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}

template <typename TV, int BM, int BN, int BK, int TM, int TN>
__global__ void __launch_bounds__((BM / TM) * (BN / TN))
hitting_gemm_kernel(const HittingGemmArgs p) {
  using resid_t = typename VecOf<TV>::resid_t;
  constexpr int NT = (BM / TM) * (BN / TN);
  constexpr int MT = BM / TM;           // threads along the state axis (fastest): coalesced E' stores
  constexpr int LA = BM * BK / NT;      // T elements each thread stages per tile
  constexpr int LB = BN * BK / NT;      // E elements each thread stages per tile
  // staging map (global -> registers -> k-major shared tiles): a warp covers 4 rows x 8 consecutive j (one 32-byte
  // sector per row); with the row stride of BM + 4 words the transposed stores hit 32 distinct banks
  constexpr int KG = BK / 8;                           // groups of 8 j per tile row
  constexpr int ROWS_PER_PASS = (NT / 32 / KG) * 4;    // rows of a tile covered by one pass of the CTA
  static_assert(BK % 8 == 0 && (NT / 32) % KG == 0 && BM % ROWS_PER_PASS == 0 && BN % ROWS_PER_PASS == 0, "tile shape");
  static_assert(LA * ROWS_PER_PASS == BM && LB * ROWS_PER_PASS == BN && TN == 4 && TM % 4 == 0, "tile shape");
  __shared__ __align__(16) float As[2][BK][BM + 4];
  __shared__ __align__(16) TV Bs[2][BK][BN + 4];
  __shared__ float s_red[NT / 32][BN];
  __shared__ int s_any_active;

  const int S = p.S, A = p.A, K = p.K;
  const int tid = threadIdx.x;
  const int tm = tid % MT, tn = tid / MT;
  const int s0 = blockIdx.y * BM, k0 = blockIdx.x * BN;
  const TV* __restrict__ E_in = reinterpret_cast<const TV*>(p.E_in);
  TV* __restrict__ E_out = reinterpret_cast<TV*>(p.E_out);

  // ---- a tile whose targets have all converged only carries E forward
  if (tid == 0) s_any_active = 0;
  __syncthreads();
  if (p.active) {
    for (int n = tid; n < BN; n += NT)
      if (k0 + n < K && p.active[k0 + n]) s_any_active = 1;
  } else if (tid == 0) {
    s_any_active = 1;
  }
  __syncthreads();
  if (!s_any_active) {
    for (int i = tid; i < BM * BN; i += NT) {
      const int m = i % BM, n = i / BM;
      if (s0 + m < S && k0 + n < K) E_out[(size_t)(k0 + n) * p.e_stride + s0 + m] = E_in[(size_t)(k0 + n) * p.e_stride + s0 + m];
    }
    return;
  }

  const int lane = tid & 31, warp = tid >> 5;
  const int kk_l = (warp % KG) * 8 + (lane & 7), row_l = (warp / KG) * 4 + (lane >> 3);
  TV best[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) best[i][j] = (TV)INFINITY;

  const int n_kt = (S + BK - 1) / BK;
  float ra[LA];
  TV rb[LB];
  auto load_tile = [&](int a, int kt) {
    const int j = kt * BK + kk_l;
#pragma unroll
    for (int r = 0; r < LA; ++r) {
      const int m = row_l + r * ROWS_PER_PASS;
      const int s = s0 + m;
      ra[r] = (s < S && j < S) ? __ldg(p.T + ((size_t)s * A + a) * S + j) : 0.f;
    }
#pragma unroll
    for (int r = 0; r < LB; ++r) {
      const int n = row_l + r * ROWS_PER_PASS;
      const int k = k0 + n;
      rb[r] = (k < K && j < S) ? __ldg(E_in + (size_t)k * p.e_stride + j) : (TV)0;
    }
  };
  auto store_tile = [&](int buf) {
#pragma unroll
    for (int r = 0; r < LA; ++r) As[buf][kk_l][row_l + r * ROWS_PER_PASS] = ra[r];
#pragma unroll
    for (int r = 0; r < LB; ++r) Bs[buf][kk_l][row_l + r * ROWS_PER_PASS] = rb[r];
  };

  const int total = A * n_kt;  // tiles over (action, k-tile), action-major
  load_tile(0, 0);
  store_tile(0);
  __syncthreads();
  TV acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = TV(0);
  for (int t = 0; t < total; ++t) {
    const int buf = t & 1;
    const bool has_next = t + 1 < total;
    if (has_next) load_tile((t + 1) / n_kt, (t + 1) % n_kt);  // global -> registers, overlapped with the FMAs below
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float av[TM];
      TV bv[TN];
#pragma unroll
      for (int i = 0; i < TM; i += 4) {
        const float4 v = *reinterpret_cast<const float4*>(&As[buf][kk][tm * TM + i]);
        av[i] = v.x; av[i + 1] = v.y; av[i + 2] = v.z; av[i + 3] = v.w;
      }
      lds4<TV>(&Bs[buf][kk][tn * TN], bv);
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] += (TV)av[i] * bv[j];
    }
    if ((t + 1) % n_kt == 0) {  // action finished: fold min_a (1 + C) and restart the accumulators
      const int a_done = t / n_kt;
#pragma unroll
      for (int j = 0; j < TN; ++j) {
        int tgt = -1;
        TV e_tgt = 0;
        const int k = k0 + tn * TN + j;
        if (p.exclude && k < K) {
          tgt = p.targets[k];
          e_tgt = (TV)p.exclude_value - E_in[(size_t)k * p.e_stride + tgt];
        }
#pragma unroll
        for (int i = 0; i < TM; ++i) {
          TV q = (TV)1 + acc[i][j];
          const int s = s0 + tm * TM + i;
          if (tgt >= 0 && s < S) q += (TV)__ldg(p.T + ((size_t)s * A + a_done) * S + tgt) * e_tgt;
          best[i][j] = q < best[i][j] ? q : best[i][j];
          acc[i][j] = TV(0);
        }
      }
    }
    if (has_next) store_tile(buf ^ 1);
    __syncthreads();
  }

  // ---- epilogue
  float dmax[TN];
#pragma unroll
  for (int j = 0; j < TN; ++j) {
    dmax[j] = 0.f;
    const int k = k0 + tn * TN + j;
    if (k < K) {
      const int tgt = p.targets[k];
      const bool act = p.active == nullptr || p.active[k] != 0;
#pragma unroll
      for (int i = 0; i < TM; ++i) {
        const int s = s0 + tm * TM + i;
        if (s < S) {
          const TV old = p.resid_vs_out ? E_out[(size_t)k * p.e_stride + s] : E_in[(size_t)k * p.e_stride + s];
          TV v = (s == tgt) ? (TV)p.pin_value : best[i][j];
          if (!act) v = old;
          E_out[(size_t)k * p.e_stride + s] = v;
          const float d = (float)fabs(v - old);
          dmax[j] = d > dmax[j] ? d : dmax[j];
          if (p.max_value > 0.0 && (double)v > p.max_value && p.overflow_flag) *p.overflow_flag = 1;
        }
      }
    }
  }
  // max|dE| per target: lanes that share tn (MT consecutive lanes when MT <= 32) -> shuffle, then across warps
  constexpr int SH = MT < 32 ? MT : 32;
#pragma unroll
  for (int j = 0; j < TN; ++j) {
#pragma unroll
    for (int o = SH / 2; o > 0; o >>= 1) {
      const float w = __shfl_xor_sync(FULL, dmax[j], o);
      dmax[j] = w > dmax[j] ? w : dmax[j];
    }
  }
  static_assert(MT >= 32 ? (MT % 32 == 0) : (32 % MT == 0), "MT");
  // after the shuffle, the first lane of each group of SH lanes holds the partial of (its tn, j)
  for (int n = tid; n < (NT / 32) * BN; n += NT) (&s_red[0][0])[n] = 0.f;
  __syncthreads();
  if ((tid % SH) == 0) {
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      float* slot = &s_red[tid / 32][tn * TN + j];
      // several groups of one warp may share tn only when MT > 32 (then SH = 32 and each warp has one tn): no race
      *slot = dmax[j] > *slot ? dmax[j] : *slot;
    }
  }
  __syncthreads();
  if (p.resid)
    for (int n = tid; n < BN; n += NT) {
      float m = 0.f;
#pragma unroll
      for (int w = 0; w < NT / 32; ++w) m = s_red[w][n] > m ? s_red[w][n] : m;
      if (k0 + n < K && m > 0.f) atomic_max_nonneg(reinterpret_cast<resid_t*>(p.resid) + k0 + n, (TV)m);
    }
}

template <typename TV>
static int launch_hitting_gemm(const HittingGemmArgs& a, cudaStream_t st) {
  // 64 x 64 tile, 4 x 4 per thread, 256 threads; BK = 32 (fp32) / 16 (fp64: the E tile is twice as wide, static
  // shared memory stays under 48 KB).  When that grid has fewer CTAs than SMs, 32 x 64 tiles with 128 threads double
  // the number of CTAs.
  constexpr int BN = 64, TM = 4, TN = 4;
  constexpr int BK = sizeof(TV) == 8 ? 16 : 32;
  const long long tiles64 = (long long)((a.K + BN - 1) / BN) * ((a.S + 63) / 64);
  count_solver_path(COLO_PATH_HIT_GEMM);
  if (tiles64 >= (long long)sm_count()) {  // measured: at 225 tiles (S = 948) the 64 x 64 tile is 15 % faster, at 49 (S = 400) slower
    constexpr int BM = 64;
    dim3 grid((a.K + BN - 1) / BN, (a.S + BM - 1) / BM);
    hitting_gemm_kernel<TV, BM, BN, BK, TM, TN><<<grid, (BM / TM) * (BN / TN), 0, st>>>(a);
  } else {
    constexpr int BM = 32;
    dim3 grid((a.K + BN - 1) / BN, (a.S + BM - 1) / BM);
    hitting_gemm_kernel<TV, BM, BN, BK, TM, TN><<<grid, (BM / TM) * (BN / TN), 0, st>>>(a);
  }
  return check_launch("hitting_gemm_kernel");
}

}  // namespace colo
