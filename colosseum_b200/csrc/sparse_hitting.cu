// sparse_hitting.cu -- Bellman backups on compressed rows: diameter (continuous + episodic) and discounted VI / PE.
//
// The benchmark families of the reference have at most ~13 successors per (state, action) (SURVEY.md appendix A):
// their dense T[S,A,S] is > 98 % zeros, and so are the derived tensors (episodic T_epi, the continuous form T_cf whose
// dense shape reaches a gigabyte).  The reference itself switches to sparse Jacobi iterations for large MDPs
// (`_get_sparse_diameter`, hardness/measures/diameter.py:382-420; `_discounted_value_iteration_sparse`,
// dynamic_programming/infinite_horizon.py:145-164).  Here, whenever every row of the dense tensor has at most kEllMax
// non-zeros, it is compressed once on the device into ELL rows -- (column, value) pairs in increasing column order,
// i.e. the summation order of the dense loop with the zero terms dropped (adding 0*x changes nothing, so the
// arithmetic is the dense recurrence's) -- and the whole solve runs in ONE launch with the value vectors resident in
// shared memory:
//
//   continuous diameter (diameter.py:76-106): a CTA owns a tile of NT targets and keeps E[S][NT] (ping-pong) in
//     shared memory; thread <-> state, the NT targets ride in registers and are gathered with one vector load.
//   episodic diameter (diameter.py:285-318): a CTA owns one target and keeps the layered table F[H][S] = 1 + ETs in
//     shared memory; one iteration = the start-row dot product + H-1 dependent layer updates.
//   discounted VI / PE (infinite_horizon.py:121-184): a CTA owns one MDP (S <= 2048) and keeps V (ping-pong) in shared
//     memory; larger MDPs (continuous forms with thousands of nodes) run one compressed-row launch per sweep over all
//     SMs with V in L2, under the host loop of backup.cu.
//
// Stopping rules (max|dV| < eps after a sweep), overflow tests and iteration caps are evaluated on chip; the only
// host round trip is the final status read.  Work per sweep drops from S*A*S*K multiply-adds to nnz*K (240x less for
// MiniGridRooms S=948).  Dense or very large problems keep using the tiled GEMM / streaming kernels.
#include <stdlib.h>

#include <type_traits>
#include <vector>

#include "common.cuh"

namespace colo {

constexpr int kEllMax = 256;                     // rows with more non-zeros than this are "dense": the caller falls back
constexpr size_t kEllMaxBytes = (size_t)2 << 30;  // ... and so are tables that would not compress below 2 GB
constexpr int kSpThreads = 512;

// ---------------------------------------------------------------- ELL compression of dense rows
// Layout (slot-major, so that threads walking consecutive states read consecutive addresses): dense row r =
// (g*S + s)*A + a of group g (MDP instance or episodic layer) has its length at len[(g*A + a)*S + s] and its i-th
// non-zero, packed as int2 (column, float bits of the value), at cv[((g*A + a)*kmax + i)*S + s].
__global__ void ell_count_kernel(const float* __restrict__ T, long long rows, int S, int A, int* __restrict__ len,
                                 int* __restrict__ max_len) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
  int wmax = 0;
  for (long long r = warp; r < rows; r += n_warps) {
    const float* row = T + (size_t)r * S;
    int n = 0;
    for (int j = lane; j < S; j += 32) n += row[j] != 0.f;
    n = warp_sum(n);
    if (lane == 0) {
      const long long gs = r / A;
      const int a = (int)(r - gs * A);
      const long long g = gs / S;
      const int s = (int)(gs - g * S);
      len[(g * A + a) * S + s] = n;
    }
    wmax = n > wmax ? n : wmax;
  }
  if (lane == 0 && wmax > 0) atomicMax(max_len, wmax);
}

__global__ void ell_fill_kernel(const float* __restrict__ T, long long rows, int S, int A, int kmax,
                                int2* __restrict__ cv) {
  // one warp per row: non-zeros are compacted in increasing column order (ballot + popc prefix)
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long r = warp; r < rows; r += n_warps) {
    const float* row = T + (size_t)r * S;
    const long long gs = r / A;
    const int a = (int)(r - gs * A);
    const long long g = gs / S;
    const int s = (int)(gs - g * S);
    const size_t base = (size_t)(g * A + a) * kmax * S + s;  // + i*S for slot i
    int off = 0;
    for (int j0 = 0; j0 < S; j0 += 32) {
      const int j = j0 + lane;
      const float t = j < S ? row[j] : 0.f;
      const unsigned m = __ballot_sync(FULL, t != 0.f);
      if (t != 0.f) {
        const int pos = off + __popc(m & ((1u << lane) - 1u));
        cv[base + (size_t)pos * S] = make_int2(j, __float_as_int(t));
      }
      off += __popc(m);
    }
  }
}

struct Ell {
  long long rows = 0;
  int kmax = 0;
  int* len = nullptr;
  int2* cv = nullptr;
};

static void ell_free(Ell& e, cudaStream_t st) {
  if (e.len) cudaFreeAsync(e.len, st);
  if (e.cv) cudaFreeAsync(e.cv, st);
  e = Ell();
}

// Compress `rows` dense rows of length S.  Returns COLO_OK and e.kmax > 0 when the rows are sparse; e.kmax = 0 (nothing
// kept) when some row has more than kEllMax non-zeros or the table would be too large.  Synchronises once.
static int ell_build(const float* T, long long rows, int S, int A, Ell& e, cudaStream_t st) {
  e = Ell();
  e.rows = rows;
  int* d_max = nullptr;
  COLO_CUDA_TRY(cudaMallocAsync(&e.len, (size_t)rows * sizeof(int), st));
  COLO_CUDA_TRY(cudaMallocAsync(&d_max, sizeof(int), st));
  COLO_CUDA_TRY(cudaMemsetAsync(d_max, 0, sizeof(int), st));
  const long long blocks = (rows + 7) / 8;
  const int grid = (int)(blocks < (long long)sm_count() * 16 ? blocks : (long long)sm_count() * 16);
  ell_count_kernel<<<grid, 256, 0, st>>>(T, rows, S, A, e.len, d_max);
  int r = check_launch("ell_count_kernel");
  if (r != COLO_OK) return r;
  int h_max = 0;
  COLO_CUDA_TRY(cudaMemcpyAsync(&h_max, d_max, sizeof(int), cudaMemcpyDeviceToHost, st));
  COLO_CUDA_TRY(cudaStreamSynchronize(st));
  COLO_CUDA_TRY(cudaFreeAsync(d_max, st));
  if (h_max < 1) h_max = 1;
  if (h_max > kEllMax || (h_max > 8 && h_max * 8 > S) || (size_t)rows * h_max * sizeof(int2) > kEllMaxBytes ||
      (long long)rows * h_max >= (1LL << 31)) {  // dense (> 1/8 of a row) or too large: kmax stays 0
    ell_free(e, st);
    return COLO_OK;
  }
  e.kmax = h_max;
  COLO_CUDA_TRY(cudaMallocAsync(&e.cv, (size_t)rows * e.kmax * sizeof(int2), st));
  ell_fill_kernel<<<grid, 256, 0, st>>>(T, rows, S, A, e.kmax, e.cv);
  return check_launch("ell_fill_kernel");
}

// ---------------------------------------------------------------- continuous diameter, NT targets per CTA
struct SparseHitArgs {
  const int* len;
  const int2* cv;
  int kmax, S, A, K;
  const int* targets;
  float eps;
  double max_value;
  long long max_iter;
  void* tile_max;     // TV [tiles]: max over the tile's targets and all states of the hitting time
  long long* iters;   // [tiles]
  int* status;        // [tiles]
};

template <typename TV, int NT>
__global__ void __launch_bounds__(kSpThreads) sparse_hitting_kernel(const SparseHitArgs p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ double s_m[kSpThreads / 32];
  __shared__ int s_overflow;
  const int S = p.S, A = p.A, kS = p.kmax * p.S;
  TV* Es = reinterpret_cast<TV*>(smem_raw);  // [2][S][NT]
  const int tile = blockIdx.x;
  int tgt[NT];
#pragma unroll
  for (int t = 0; t < NT; ++t) {
    const int k = tile * NT + t;
    tgt[t] = __ldg(p.targets + (k < p.K ? k : p.K - 1));  // a ragged last tile repeats the last target
  }
  for (int i = threadIdx.x; i < 2 * S * NT; i += blockDim.x) Es[i] = TV(0);
  if (threadIdx.x == 0) s_overflow = 0;
  __syncthreads();

  const int n_out = S * NT;
  const bool check_max = p.max_value > 0.0;
  const TV max_v = (TV)p.max_value;
  int cur = 0, status = COLO_MAX_ITER;
  long long it = 0;
  while (it < p.max_iter) {
    const TV* Ein = Es + cur * n_out;
    TV* Eout = Es + (cur ^ 1) * n_out;
    bool conv = true;
    for (int s = threadIdx.x; s < S; s += blockDim.x) {
      TV best[NT];
#pragma unroll
      for (int t = 0; t < NT; ++t) best[t] = (TV)INFINITY;
      for (int a = 0; a < A; ++a) {
        const int n = __ldg(p.len + a * S + s);
        int idx = a * kS + s;
        TV acc[NT];
#pragma unroll
        for (int t = 0; t < NT; ++t) acc[t] = (TV)1;  // diameter.py:88-90: reward -1 per step, gamma 1
        for (int i = 0; i < n; ++i, idx += S) {
          const int2 e = __ldg(p.cv + idx);
          const TV w = (TV)__int_as_float(e.y);
          const TV* ev = Ein + e.x * NT;
#pragma unroll
          for (int t = 0; t < NT; ++t) acc[t] += w * ev[t];
        }
#pragma unroll
        for (int t = 0; t < NT; ++t) best[t] = acc[t] < best[t] ? acc[t] : best[t];
      }
#pragma unroll
      for (int t = 0; t < NT; ++t) {
        TV bt = best[t];
        if (s == tgt[t]) bt = (TV)0;  // the target is absorbing with reward 0 (diameter.py:85-90)
        // NaN-safe: a NaN difference counts as "not converged"
        conv = conv && ((float)fabs(bt - Ein[s * NT + t]) < p.eps);
        if (check_max && bt > max_v) s_overflow = 1;
        Eout[s * NT + t] = bt;
      }
    }
    const int all_conv = __syncthreads_and(conv);  // the barrier also publishes Eout and s_overflow
    ++it;
    cur ^= 1;
    if (s_overflow) { status = COLO_OVERFLOW; break; }
    if (all_conv) { status = COLO_OK; break; }
  }
  // tile result: max over states and (valid) targets of the converged hitting times
  const TV* E = Es + cur * n_out;
  TV mt = 0;
  for (int s = threadIdx.x; s < S; s += blockDim.x)
#pragma unroll
    for (int t = 0; t < NT; ++t)
      if (tile * NT + t < p.K) mt = E[s * NT + t] > mt ? E[s * NT + t] : mt;
  mt = warp_max(mt);
  if ((threadIdx.x & 31) == 0) s_m[threadIdx.x >> 5] = (double)mt;
  __syncthreads();
  if (threadIdx.x == 0) {
    double mm = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) mm = s_m[w] > mm ? s_m[w] : mm;
    reinterpret_cast<TV*>(p.tile_max)[tile] = (TV)mm;
    p.iters[tile] = it;
    p.status[tile] = status;
  }
}

// ---------------------------------------------------------------- episodic diameter, one target per CTA
struct SparseEpiArgs {
  const int* len;          // ELL over rows ((h*S + s)*A + a), h = 0 .. H-2  (group = layer)
  const int2* cv;
  const float* start_row;  // dense T_epi[H-1, 0, 0, :]  (diameter.py:293)
  int kmax, H, S, A, K;
  const int* targets;
  float eps;
  double max_value;        // in ETs units (0 = off)
  long long max_iter;
  void* out;               // TV [K]: per target max_s min_{h: ETs>0} ETs[h,s]   (diameter.py:311-314)
  long long* iters;        // [K]
  int* status;             // [K]
};

template <typename TV>
__global__ void __launch_bounds__(kSpThreads) sparse_episodic_kernel(const SparseEpiArgs p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ double s_sum[kSpThreads / 32];
  __shared__ int s_overflow;
  const int H = p.H, S = p.S, A = p.A, kS = p.kmax * p.S;
  TV* F = reinterpret_cast<TV*>(smem_raw);  // [H][S], F = 1 + ETs
  const int k = blockIdx.x;
  const int es = p.targets[k];
  for (int i = threadIdx.x; i < H * S; i += blockDim.x) F[i] = (TV)1;
  if (threadIdx.x == 0) s_overflow = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const bool check_max = p.max_value > 0.0;
  const TV max_f = (TV)(p.max_value + 1.0);  // F = 1 + ETs
  int status = COLO_MAX_ITER;
  long long it = 0;
  while (it < p.max_iter) {
    bool conv = true;
    // ETs[-1] = T[-1,0,0] @ (1 + ETs[0])  (diameter.py:293): the same value for every state of the last layer
    TV part = 0;
    for (int ns = threadIdx.x; ns < S; ns += blockDim.x) part += (TV)__ldg(p.start_row + ns) * F[ns];
    part = warp_sum(part);
    if (lane == 0) s_sum[warp] = (double)part;
    __syncthreads();
    TV tot = 0;
    for (int w = 0; w < nw; ++w) tot += (TV)s_sum[w];
    const TV v = (TV)1 + tot;
    TV* last = F + (H - 1) * S;
    for (int j = threadIdx.x; j < S; j += blockDim.x) {
      conv = conv && ((float)fabs(v - last[j]) < p.eps);
      last[j] = v;
    }
    __syncthreads();
    for (int h = H - 1; h >= 1; --h) {  // diameter.py:294-306
      const TV* Fn = F + h * S;
      TV* Fo = F + (h - 1) * S;
      for (int j = threadIdx.x; j < S; j += blockDim.x) {
        if (j == es) continue;  // ETs[h-1, es] is never written: stays 0 (F = 1)
        TV best = (TV)INFINITY;
        for (int a = 0; a < A; ++a) {
          const int ga = (h - 1) * A + a;  // group = layer
          const int n = __ldg(p.len + ga * S + j);
          int idx = ga * kS + j;
          TV acc = (TV)1;
          for (int i = 0; i < n; ++i, idx += S) {
            const int2 e = __ldg(p.cv + idx);
            acc += (TV)__int_as_float(e.y) * (e.x == es ? (TV)1 : Fn[e.x]);  // reaching the target costs one step
          }
          best = acc < best ? acc : best;
        }
        conv = conv && ((float)fabs(best - Fo[j]) < p.eps);
        if (check_max && best > max_f) s_overflow = 1;
        Fo[j] = best;
      }
      __syncthreads();
    }
    const int all_conv = __syncthreads_and(conv);
    ++it;
    if (s_overflow) { status = COLO_OVERFLOW; break; }
    if (all_conv) { status = COLO_OK; break; }
  }
  // per state the min over h of the POSITIVE entries, max over states (diameter.py:311-314)
  TV cur = (TV)-INFINITY;
  for (int s = threadIdx.x; s < S; s += blockDim.x) {
    TV mn = (TV)INFINITY;
    for (int h = 0; h < H; ++h) {
      const TV e = F[h * S + s] - (TV)1;
      if (e > 0 && e < mn) mn = e;
    }
    cur = mn > cur ? mn : cur;
  }
  cur = warp_max(cur);
  __syncthreads();
  if (lane == 0) s_sum[warp] = (double)cur;
  __syncthreads();
  if (threadIdx.x == 0) {
    double mm = -INFINITY;
    for (int w = 0; w < nw; ++w) mm = s_sum[w] > mm ? s_sum[w] : mm;
    reinterpret_cast<TV*>(p.out)[k] = (TV)mm;
    p.iters[k] = it;
    p.status[k] = status;
  }
}

// ---------------------------------------------------------------- discounted VI / PE, one CTA per MDP
struct SparseViArgs {
  const int* len;      // ELL over rows ((b*S + s)*A + a)  (group = instance)
  const int2* cv;
  int kmax;
  const float* R;      // [B][S,A]
  const float* pi;     // [B][S,A] (COLO_FOLD_PI) or null
  int B, S, A;
  double gamma, max_abs;
  float eps;
  long long max_iter;
  void* V;             // out [B][S]
  void* Q;             // out [B][S,A] or null
  const void* V0;      // initial V [B][S] or null (zeros)
  int normalize;       // != 0: V is rescaled to unit sum after every sweep (power iteration on a distribution)
  long long* iters;    // [B]
  int* status;         // [B]
};

template <typename TV, int FOLD>
__device__ __forceinline__ TV sparse_row_fold(const int* __restrict__ len, const int2* __restrict__ cv,
                                              const float* __restrict__ R, const float* __restrict__ pi, int S, int A,
                                              int kS, int s, TV gamma, const TV* __restrict__ Vin, TV* Qrow) {
  // Q[s,a] = R[s,a] + gamma * sum_i val_i * V[col_i];  returns fold_a Q[s,a]
  TV folded = FOLD == COLO_FOLD_MIN ? (TV)INFINITY : (FOLD == COLO_FOLD_MAX ? (TV)-INFINITY : (TV)0);
  for (int a = 0; a < A; ++a) {
    const int n = __ldg(len + a * S + s);
    int idx = a * kS + s;
    TV dot = 0;
    for (int i = 0; i < n; ++i, idx += S) {
      const int2 e = __ldg(cv + idx);
      dot += (TV)__int_as_float(e.y) * Vin[e.x];
    }
    const TV q = (TV)__ldg(R + s * A + a) + gamma * dot;
    if (Qrow) Qrow[a] = q;
    if (FOLD == COLO_FOLD_MAX) folded = q > folded ? q : folded;
    if (FOLD == COLO_FOLD_MIN) folded = q < folded ? q : folded;
    if (FOLD == COLO_FOLD_PI) folded += q * (TV)__ldg(pi + s * A + a);
  }
  return folded;
}

template <typename TV, int FOLD>
__global__ void __launch_bounds__(kSpThreads) sparse_vi_kernel(const SparseViArgs p) {
  // (a thread-block-cluster variant with V replicated through distributed shared memory was measured on B200 and
  // dropped: 10-200x run-to-run spread; large MDPs use the per-sweep kernel below instead)
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int s_overflow;
  const int S = p.S, A = p.A, kS = p.kmax * p.S;
  const int b = blockIdx.x;
  TV* Vs = reinterpret_cast<TV*>(smem_raw);  // [2][S]
  const TV* V0 = p.V0 ? reinterpret_cast<const TV*>(p.V0) + (size_t)b * S : nullptr;
  for (int i = threadIdx.x; i < 2 * S; i += blockDim.x) Vs[i] = (V0 && i < S) ? V0[i] : TV(0);
  if (threadIdx.x == 0) s_overflow = 0;
  __syncthreads();
  const float* R = p.R + (size_t)b * S * A;
  const float* pi = FOLD == COLO_FOLD_PI ? p.pi + (size_t)b * S * A : nullptr;
  const int* len = p.len + (size_t)b * A * S;
  const int2* cv = p.cv + (size_t)b * A * kS;
  const TV gamma = (TV)p.gamma;
  const bool check_max = p.max_abs > 0.0;
  const TV max_abs = (TV)p.max_abs;
  TV* Vg = reinterpret_cast<TV*>(p.V) + (size_t)b * S;
  TV* Qg = p.Q ? reinterpret_cast<TV*>(p.Q) + (size_t)b * S * A : nullptr;
  int cur = 0, status = COLO_MAX_ITER;
  long long it = 0;
  __shared__ double s_part[kSpThreads / 32];
  while (true) {
    const TV* Vin = Vs + cur * S;
    TV* Vout = Vs + (cur ^ 1) * S;
    bool conv = true;
    if (!p.normalize) {
      for (int s = threadIdx.x; s < S; s += blockDim.x) {
        const TV folded = sparse_row_fold<TV, FOLD>(len, cv, R, pi, S, A, kS, s, gamma, Vin, nullptr);
        conv = conv && ((float)fabs(folded - Vin[s]) < p.eps);
        if (check_max && fabs(folded) > max_abs) s_overflow = 1;
        Vout[s] = folded;
      }
    } else {
      // x <- M x / |M x|_1: rows of a float32 matrix sum to 1 +- 1e-7, so the raw iteration drifts; the rescaled one
      // has the Perron vector as its fixed point and the stopping rule compares rescaled iterates
      double part = 0.0;
      for (int s = threadIdx.x; s < S; s += blockDim.x) {
        const TV folded = sparse_row_fold<TV, FOLD>(len, cv, R, pi, S, A, kS, s, gamma, Vin, nullptr);
        Vout[s] = folded;
        part += (double)folded;
      }
      part = warp_sum(part);
      if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = part;
      __syncthreads();
      double tot = 0.0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += s_part[w];
      const TV inv = (TV)(1.0 / tot);
      for (int s = threadIdx.x; s < S; s += blockDim.x) {  // each thread rescales the entries it wrote
        const TV x = Vout[s] * inv;
        conv = conv && ((float)fabs(x - Vin[s]) < p.eps);
        Vout[s] = x;
      }
    }
    const int all_conv = __syncthreads_and(conv);
    ++it;
    if (s_overflow) { status = COLO_OVERFLOW; break; }
    if (all_conv) { status = COLO_OK; break; }
    if (it >= p.max_iter) { status = COLO_MAX_ITER; break; }
    cur ^= 1;
  }
  if (p.normalize) {
    const TV* Vlast = Vs + (cur ^ 1) * S;  // the rescaled iterate of the stopping sweep
    for (int s = threadIdx.x; s < S; s += blockDim.x) Vg[s] = Vlast[s];
  } else if (status != COLO_OVERFLOW) {
    // the stopping sweep is redone from the same V_in, storing the Q and V it produced (the reference returns those)
    const TV* Vin = Vs + cur * S;
    for (int s = threadIdx.x; s < S; s += blockDim.x) {
      const TV folded = sparse_row_fold<TV, FOLD>(len, cv, R, pi, S, A, kS, s, gamma, Vin, Qg ? Qg + (size_t)s * A : nullptr);
      Vg[s] = folded;
    }
  }
  if (threadIdx.x == 0) {
    p.iters[b] = it;
    p.status[b] = status;
  }
}

// ---------------------------------------------------------------- one synchronous sweep on compressed rows
// For MDPs too large for one CTA (continuous forms with thousands of nodes): V lives in global memory (L2 resident),
// one launch per sweep over all SMs, driven by the same host loop as the dense streaming kernel (backup.cu).
struct SparseSweepArgs {
  const int* len;
  const int2* cv;
  int kmax;
  const float* R;
  const float* pi;
  int B, S, A;
  double gamma, max_abs;
  const void* V_in;    // [B][S]
  void* V_out;         // [B][S]
  void* Q;             // [B][S,A] or null
  void* resid;         // [B] float/double bits, atomicMax (or null)
  const unsigned char* active;  // [B] or null
  int* overflow_flag;
};

constexpr int kSweepGroup = 8;  // lanes per state in the per-sweep kernel

template <typename TV, int FOLD>
__global__ void __launch_bounds__(256) sparse_sweep_kernel(const SparseSweepArgs p) {
  // kSweepGroup lanes share one state: they stride over the row's non-zeros and combine with shuffles, so that the
  // long rows of a continuous form (its last layer carries the whole start distribution, > 100 entries) cost a
  // handful of load round trips instead of one per entry; 4 states per warp keep the short rows busy.
  using resid_t = typename std::conditional<sizeof(TV) == 8, unsigned long long, unsigned int>::type;
  const int S = p.S, A = p.A, kS = p.kmax * p.S;
  const int b = blockIdx.y;
  const TV* Vin = reinterpret_cast<const TV*>(p.V_in) + (size_t)b * S;
  TV* Vout = reinterpret_cast<TV*>(p.V_out) + (size_t)b * S;
  const int gtid = blockIdx.x * blockDim.x + threadIdx.x;
  const int s = gtid / kSweepGroup, sub = gtid % kSweepGroup;
  const bool live = s < S;
  const bool frozen = p.active != nullptr && p.active[b] == 0;
  const int* len = p.len + (size_t)b * A * S;
  const int2* cv = p.cv + (size_t)b * A * kS;
  const float* R = p.R + (size_t)b * S * A;
  const float* pi = FOLD == COLO_FOLD_PI ? p.pi + (size_t)b * S * A : nullptr;
  const TV gamma = (TV)p.gamma;
  TV d = 0;
  TV folded = FOLD == COLO_FOLD_MIN ? (TV)INFINITY : (FOLD == COLO_FOLD_MAX ? (TV)-INFINITY : (TV)0);
  if (!frozen) {
    for (int a = 0; a < A; ++a) {  // uniform trip count: the shuffles below are executed by every lane of the warp
      TV dot = 0;
      if (live) {
        const int n = __ldg(len + a * S + s);
        for (int i = sub; i < n; i += kSweepGroup) {
          const int2 e = __ldg(cv + a * kS + i * S + s);
          dot += (TV)__int_as_float(e.y) * __ldg(Vin + e.x);
        }
      }
#pragma unroll
      for (int o = kSweepGroup / 2; o > 0; o >>= 1) dot += __shfl_xor_sync(FULL, dot, o);
      if (live) {
        const TV q = (TV)__ldg(R + s * A + a) + gamma * dot;
        if (p.Q && sub == 0) reinterpret_cast<TV*>(p.Q)[((size_t)b * S + s) * A + a] = q;
        if (FOLD == COLO_FOLD_MAX) folded = q > folded ? q : folded;
        if (FOLD == COLO_FOLD_MIN) folded = q < folded ? q : folded;
        if (FOLD == COLO_FOLD_PI) folded += q * (TV)__ldg(pi + s * A + a);
      }
    }
  }
  if (live && sub == 0) {
    if (frozen) {
      Vout[s] = Vin[s];  // converged instance of a batch: carried forward
    } else {
      d = fabs(folded - Vin[s]);
      Vout[s] = folded;
      if (p.max_abs > 0.0 && p.overflow_flag && fabs((double)folded) > p.max_abs) *p.overflow_flag = 1;
    }
  }
  d = warp_max(d);
  if (p.resid && (threadIdx.x & 31) == 0 && d > (TV)0) atomic_max_nonneg(reinterpret_cast<resid_t*>(p.resid) + b, d);
}

// ---------------------------------------------------------------- host side
static void ensure_pool_keeps_memory();
static int max_optin_smem_sp() {
  static int cached = 0;
  if (!cached) {
    int dev = 0, v = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess || v <= 0) v = 227 * 1024;
    cached = v - 2048;  // room for the kernels' static shared memory
  }
  return cached;
}

template <typename TV>
static int collect(const TV* d_vals, const long long* d_iters, const int* d_status, int n, double* out_host,
                   cudaStream_t st) {
  std::vector<TV> v((size_t)n);
  std::vector<long long> it((size_t)n);
  std::vector<int> stt((size_t)n);
  COLO_CUDA_TRY(cudaMemcpyAsync(v.data(), d_vals, (size_t)n * sizeof(TV), cudaMemcpyDeviceToHost, st));
  COLO_CUDA_TRY(cudaMemcpyAsync(it.data(), d_iters, (size_t)n * sizeof(long long), cudaMemcpyDeviceToHost, st));
  COLO_CUDA_TRY(cudaMemcpyAsync(stt.data(), d_status, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, st));
  COLO_CUDA_TRY(cudaStreamSynchronize(st));
  int rc = COLO_OK;
  double best = -INFINITY;
  long long mx = 0;
  for (int i = 0; i < n; ++i) {
    if (stt[i] == COLO_OVERFLOW) return COLO_OVERFLOW;
    if (stt[i] == COLO_MAX_ITER) rc = COLO_MAX_ITER;
    if ((double)v[i] > best) best = (double)v[i];
    if (it[i] > mx) mx = it[i];
  }
  out_host[0] = best;
  out_host[1] = (double)mx;
  return rc;
}

static int block_threads(int n) {
  int t = n < kSpThreads ? ((n + 31) / 32) * 32 : kSpThreads;
  return t < 64 ? 64 : t;
}

// Returns COLO_OK/OVERFLOW/MAX_ITER with *handled = 1 when the compressed-row path ran; *handled = 0 (and COLO_OK)
// when T is not sparse enough or the tables do not fit shared memory: the caller then uses the dense kernels.
template <typename TV>
int sparse_diameter_continuous(const float* T, const int* targets, int K, int S, int A, double eps, double max_value,
                               long long max_iter, double* out_host, int* handled, void* stream) {
  *handled = 0;
  ensure_pool_keeps_memory();
  cudaStream_t st = (cudaStream_t)stream;
  // NT targets per CTA: a CTA's sweep time is nearly independent of NT (thread <-> state, NT only adds FMAs), so take
  // the largest NT that still leaves >= one CTA per SM, and that fits E[2][S][NT] in shared memory
  int NT = 4;
  static const int forced_nt = getenv("COLO_SPARSE_NT") ? atoi(getenv("COLO_SPARSE_NT")) : 0;
  while (NT > 1 && ((K + NT - 1) / NT < sm_count() || (size_t)2 * S * NT * sizeof(TV) > (size_t)max_optin_smem_sp())) NT >>= 1;
  if (forced_nt == 1 || forced_nt == 2 || forced_nt == 4) NT = forced_nt;
  const size_t smem = (size_t)2 * S * NT * sizeof(TV);
  if (smem > (size_t)max_optin_smem_sp()) return COLO_OK;
  Ell e;
  int r = ell_build(T, (long long)S * A, S, A, e, st);
  if (r != COLO_OK || e.kmax == 0) return r;
  const int tiles = (K + NT - 1) / NT;
  TV* d_max = nullptr;
  long long* d_it = nullptr;
  int* d_st = nullptr;
  COLO_CUDA_TRY(cudaMallocAsync(&d_max, (size_t)tiles * sizeof(TV), st));
  COLO_CUDA_TRY(cudaMallocAsync(&d_it, (size_t)tiles * sizeof(long long), st));
  COLO_CUDA_TRY(cudaMallocAsync(&d_st, (size_t)tiles * sizeof(int), st));
  SparseHitArgs a = {};
  a.len = e.len; a.cv = e.cv; a.kmax = e.kmax; a.S = S; a.A = A; a.K = K;
  a.targets = targets; a.eps = (float)eps; a.max_value = max_value; a.max_iter = max_iter;
  a.tile_max = d_max; a.iters = d_it; a.status = d_st;
  const int threads = block_threads(S);
  count_solver_path(COLO_PATH_SPARSE_HIT);
#define COLO_SPHIT(N)                                                                                     \
  {                                                                                                         \
    auto kern = sparse_hitting_kernel<TV, N>;                                                               \
    { const int _es = ensure_dynamic_smem((const void*)kern, smem); if (_es != COLO_OK) return _es; }      \
    kern<<<tiles, threads, smem, st>>>(a);                                                                  \
  }
  if (NT == 4) COLO_SPHIT(4)
  else if (NT == 2) COLO_SPHIT(2)
  else COLO_SPHIT(1)
#undef COLO_SPHIT
  r = check_launch("sparse_hitting_kernel");
  if (r == COLO_OK) r = collect<TV>(d_max, d_it, d_st, tiles, out_host, st);
  cudaFreeAsync(d_max, st);
  cudaFreeAsync(d_it, st);
  cudaFreeAsync(d_st, st);
  ell_free(e, st);
  if (r >= 0) *handled = 1;
  return r;
}

template <typename TV>
int sparse_diameter_episodic(const float* T_epi, const int* targets, int K, int H, int S, int A, double eps,
                             double max_value, long long max_iter, double* out_host, int* handled, void* stream) {
  *handled = 0;
  ensure_pool_keeps_memory();
  cudaStream_t st = (cudaStream_t)stream;
  const size_t smem = (size_t)H * S * sizeof(TV);
  if (smem > (size_t)max_optin_smem_sp()) return COLO_OK;
  Ell e;
  int r = ell_build(T_epi, (long long)(H - 1) * S * A, S, A, e, st);
  if (r != COLO_OK || e.kmax == 0) return r;
  TV* d_out = nullptr;
  long long* d_it = nullptr;
  int* d_st = nullptr;
  COLO_CUDA_TRY(cudaMallocAsync(&d_out, (size_t)K * sizeof(TV), st));
  COLO_CUDA_TRY(cudaMallocAsync(&d_it, (size_t)K * sizeof(long long), st));
  COLO_CUDA_TRY(cudaMallocAsync(&d_st, (size_t)K * sizeof(int), st));
  SparseEpiArgs a = {};
  a.len = e.len; a.cv = e.cv; a.kmax = e.kmax;
  a.start_row = T_epi + (size_t)(H - 1) * S * A * S;
  a.H = H; a.S = S; a.A = A; a.K = K; a.targets = targets; a.eps = (float)eps; a.max_value = max_value;
  a.max_iter = max_iter; a.out = d_out; a.iters = d_it; a.status = d_st;
  auto kern = sparse_episodic_kernel<TV>;
  { const int _es = ensure_dynamic_smem((const void*)kern, smem); if (_es != COLO_OK) return _es; }
  count_solver_path(COLO_PATH_SPARSE_EPI);
  kern<<<K, block_threads(S), smem, st>>>(a);
  r = check_launch("sparse_episodic_kernel");
  if (r == COLO_OK) r = collect<TV>(d_out, d_it, d_st, K, out_host, st);
  cudaFreeAsync(d_out, st);
  cudaFreeAsync(d_it, st);
  cudaFreeAsync(d_st, st);
  ell_free(e, st);
  if (r >= 0) *handled = 1;
  return r;
}

static void ensure_pool_keeps_memory() {
  // cudaFreeAsync'd blocks go back to the OS at the next synchronisation unless the pool may retain them: every
  // solve allocates its compressed tables with cudaMallocAsync, so let the default pool keep what it has
  static bool done = false;
  if (done) return;
  done = true;
  int dev = 0;
  cudaMemPool_t pool;
  if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
    unsigned long long thr = ~0ULL;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
  }
  cudaGetLastError();
}

int sparse_rows_build(const float* T, long long rows, int S, int A, SparseRows* out, void* stream) {
  ensure_pool_keeps_memory();
  Ell e;
  const int r = ell_build(T, rows, S, A, e, (cudaStream_t)stream);
  out->kmax = e.kmax;
  out->len = e.len;
  out->cv = e.cv;
  return r;
}

void sparse_rows_free(SparseRows* h, void* stream) {
  Ell e;
  e.len = h->len;
  e.cv = (int2*)h->cv;
  ell_free(e, (cudaStream_t)stream);
  h->len = nullptr;
  h->cv = nullptr;
  h->kmax = 0;
}

bool sparse_vi_fits_one_cta(int S, bool f64) {
  return S <= 2048 && (size_t)2 * S * (f64 ? 8 : 4) <= (size_t)max_optin_smem_sp();
}

// whole solve in one launch, one CTA per instance (S <= 2048)
template <typename TV>
int sparse_solve_resident(const SparseRows& h, const float* R, const float* pi, int B, int S, int A, double gamma,
                          double eps, double max_abs, long long max_iter, int fold, TV* Q, TV* V,
                          long long* iters_out_host, void* stream, const TV* V0, bool normalize) {
  cudaStream_t st = (cudaStream_t)stream;
  const size_t smem = (size_t)2 * S * sizeof(TV);
  long long* d_it = nullptr;
  int* d_st = nullptr;
  COLO_CUDA_TRY(cudaMallocAsync(&d_it, (size_t)B * sizeof(long long), st));
  COLO_CUDA_TRY(cudaMallocAsync(&d_st, (size_t)B * sizeof(int), st));
  SparseViArgs a = {};
  a.len = h.len; a.cv = (const int2*)h.cv; a.kmax = h.kmax; a.R = R; a.pi = pi; a.B = B; a.S = S; a.A = A;
  a.gamma = gamma; a.eps = (float)eps; a.max_abs = max_abs; a.max_iter = max_iter; a.V = V; a.Q = Q; a.V0 = V0;
  a.normalize = normalize ? 1 : 0;
  a.iters = d_it; a.status = d_st;
  const int threads = block_threads(S);
  count_solver_path(COLO_PATH_SPARSE_VI);
#define COLO_SPVI(FOLD)                                                                                   \
  {                                                                                                         \
    auto kern = sparse_vi_kernel<TV, FOLD>;                                                                 \
    { const int _es = ensure_dynamic_smem((const void*)kern, smem); if (_es != COLO_OK) return _es; }      \
    kern<<<B, threads, smem, st>>>(a);                                                                      \
  }
  if (fold == COLO_FOLD_MAX) COLO_SPVI(COLO_FOLD_MAX)
  else if (fold == COLO_FOLD_PI) COLO_SPVI(COLO_FOLD_PI)
  else COLO_SPVI(COLO_FOLD_MIN)
#undef COLO_SPVI
  int rc = check_launch("sparse_vi_kernel");
  if (rc == COLO_OK) {
    std::vector<long long> it((size_t)B);
    std::vector<int> stt((size_t)B);
    COLO_CUDA_TRY(cudaMemcpyAsync(it.data(), d_it, (size_t)B * sizeof(long long), cudaMemcpyDeviceToHost, st));
    COLO_CUDA_TRY(cudaMemcpyAsync(stt.data(), d_st, (size_t)B * sizeof(int), cudaMemcpyDeviceToHost, st));
    COLO_CUDA_TRY(cudaStreamSynchronize(st));
    for (int b = 0; b < B; ++b) {
      if (stt[b] == COLO_OVERFLOW) rc = COLO_OVERFLOW;
      else if (stt[b] == COLO_MAX_ITER && rc == COLO_OK) rc = COLO_MAX_ITER;
      if (iters_out_host) iters_out_host[b] = it[b];
    }
  }
  cudaFreeAsync(d_it, st);
  cudaFreeAsync(d_st, st);
  return rc;
}

// one synchronous sweep (any size), for the host-driven loop of backup.cu
template <typename TV>
int sparse_sweep_launch(const SparseRows& h, const float* R, const float* pi, int B, int S, int A, int fold,
                        double gamma, const TV* V_in, TV* V_out, TV* Q, void* resid, const unsigned char* active,
                        double max_abs, int* overflow_flag, void* stream) {
  SparseSweepArgs a = {};
  a.len = h.len; a.cv = (const int2*)h.cv; a.kmax = h.kmax; a.R = R; a.pi = pi; a.B = B; a.S = S; a.A = A;
  a.gamma = gamma; a.max_abs = max_abs; a.V_in = V_in; a.V_out = V_out; a.Q = Q; a.resid = resid; a.active = active;
  a.overflow_flag = overflow_flag;
  // small CTAs so that a few thousand states still spread over all SMs (kSweepGroup lanes per state)
  const long long lanes = (long long)S * kSweepGroup;
  const int threads = lanes >= 148LL * 1024 ? 256 : 128;
  dim3 grid((unsigned)((lanes + threads - 1) / threads), B);
  cudaStream_t st = (cudaStream_t)stream;
  count_solver_path(COLO_PATH_SPARSE_SWEEP);
  if (fold == COLO_FOLD_MAX) sparse_sweep_kernel<TV, COLO_FOLD_MAX><<<grid, threads, 0, st>>>(a);
  else if (fold == COLO_FOLD_PI) sparse_sweep_kernel<TV, COLO_FOLD_PI><<<grid, threads, 0, st>>>(a);
  else sparse_sweep_kernel<TV, COLO_FOLD_MIN><<<grid, threads, 0, st>>>(a);
  return check_launch("sparse_sweep_kernel");
}

template int sparse_solve_resident<float>(const SparseRows&, const float*, const float*, int, int, int, double, double,
                                          double, long long, int, float*, float*, long long*, void*, const float*, bool);
template int sparse_solve_resident<double>(const SparseRows&, const float*, const float*, int, int, int, double, double,
                                           double, long long, int, double*, double*, long long*, void*, const double*, bool);
template int sparse_sweep_launch<float>(const SparseRows&, const float*, const float*, int, int, int, int, double,
                                        const float*, float*, float*, void*, const unsigned char*, double, int*, void*);
template int sparse_sweep_launch<double>(const SparseRows&, const float*, const float*, int, int, int, int, double,
                                         const double*, double*, double*, void*, const unsigned char*, double, int*, void*);
template int sparse_diameter_continuous<float>(const float*, const int*, int, int, int, double, double, long long,
                                               double*, int*, void*);
template int sparse_diameter_continuous<double>(const float*, const int*, int, int, int, double, double, long long,
                                                double*, int*, void*);
template int sparse_diameter_episodic<float>(const float*, const int*, int, int, int, int, double, double, long long,
                                             double*, int*, void*);
template int sparse_diameter_episodic<double>(const float*, const int*, int, int, int, int, double, double, long long,
                                              double*, int*, void*);

}  // namespace colo
