// common.cuh -- shared helpers for libcolosseum_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/colosseum_b200.h"

namespace colo {

// ---- error plumbing -------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
void count_launch(unsigned long long n = 1);
int check_launch(const char* what);  // cudaGetLastError -> COLO_OK / COLO_ERR_CUDA (+ counts one launch)
void count_solver_path(int kind);    // one launch of a Bellman-solver path (COLO_PATH_*, colo_solver_path_launches)

#define COLO_CUDA_TRY(expr)                                                                  \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess) {                                                                 \
      colo::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return COLO_ERR_CUDA;                                                                  \
    }                                                                                        \
  } while (0)

#define COLO_ARG_CHECK(cond, msg)                  \
  do {                                             \
    if (!(cond)) {                                 \
      colo::set_error("bad argument: %s", msg);    \
      return COLO_ERR_ARG;                         \
    }                                              \
  } while (0)

int sm_count();  // SMs of the current device (148 on B200), cached
// grow-only, locked cudaFuncAttributeMaxDynamicSharedMemorySize (the entry points run on several host threads)
int ensure_dynamic_smem(const void* kernel, size_t bytes);

// resident.cu: on-chip resident solver (see there)
int resident_fits_any(int S, int A, int NV, bool f64, int* cluster_size_out);
int resident_solve_any(const colo_resident_args* args, bool f64, void* stream);
bool resident_enabled();  // false when COLO_NO_RESIDENT is set (benchmarking the streaming path)

// sparse_hitting.cu: diameter on ELL-compressed rows (one launch per solve); *handled = 0 when T is not sparse
// enough / does not fit shared memory and the dense kernels must be used
template <typename TV>
int sparse_diameter_continuous(const float* T, const int* targets, int K, int S, int A, double eps, double max_value,
                               long long max_iter, double* out_host, int* handled, void* stream);
template <typename TV>
int sparse_diameter_episodic(const float* T_epi, const int* targets, int K, int H, int S, int A, double eps,
                             double max_value, long long max_iter, double* out_host, int* handled, void* stream);

// compressed rows of a dense tensor (kmax = 0: the rows are dense, nothing was kept); see sparse_hitting.cu
struct SparseRows {
  int kmax = 0;
  int* len = nullptr;
  void* cv = nullptr;  // int2 (column, float bits)
};
int sparse_rows_build(const float* T, long long rows, int S, int A, SparseRows* out, void* stream);
void sparse_rows_free(SparseRows* h, void* stream);
bool sparse_vi_fits_one_cta(int S, bool f64);
template <typename TV>
int sparse_solve_resident(const SparseRows& h, const float* R, const float* pi, int B, int S, int A, double gamma,
                          double eps, double max_abs, long long max_iter, int fold, TV* Q, TV* V,
                          long long* iters_out_host, void* stream, const TV* V0 = nullptr, bool normalize = false);
template <typename TV>
int sparse_sweep_launch(const SparseRows& h, const float* R, const float* pi, int B, int S, int A, int fold,
                        double gamma, const TV* V_in, TV* V_out, TV* Q, void* resid, const unsigned char* active,
                        double max_abs, int* overflow_flag, void* stream);

// hitting_umma.cu: the multi-target hitting-time sweep on the tensor cores (tcgen05 / TMEM / TMA), fp32 iterates
struct UmmaPlan;
bool hitting_umma_supported(int S, int A, int K);
int hitting_umma_plan(const float* T, int S, int A, int K, UmmaPlan** out, cudaStream_t st);
int hitting_umma_sweep(UmmaPlan* pl, const float* E_in, float* E_out, long long e_stride, const int* targets,
                       const unsigned char* active, unsigned* resid, double max_value, int* overflow_flag, cudaStream_t st);
void hitting_umma_free(UmmaPlan* pl, cudaStream_t st);

// ---- device helpers -------------------------------------------------------------------------------------
constexpr unsigned FULL = 0xffffffffu;

// streaming 128-bit load: T tiles are read exactly once per sweep -> bypass L1 allocation, keep L1 for V
__device__ __forceinline__ float4 ldg_stream4(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.L2::128B.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ float ldg_stream1(const float* p) {
  float r;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
  return r;
}

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
  return v;
}
template <typename T>
__device__ __forceinline__ T warp_max(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    T w = __shfl_xor_sync(FULL, v, o);
    v = w > v ? w : v;
  }
  return v;
}

// non-negative float/double max through integer atomics (IEEE ordering == unsigned ordering for x >= 0)
__device__ __forceinline__ void atomic_max_nonneg(unsigned int* addr, float v) { atomicMax(addr, __float_as_uint(v)); }
__device__ __forceinline__ void atomic_max_nonneg(unsigned long long* addr, double v) {
  atomicMax(addr, (unsigned long long)__double_as_longlong(v));
}

// ---- Philox4x32-10 (Salmon et al. SC'11): counter = (env lo, env hi, t lo, t hi), key = seed -------------
struct Philox4 {
  uint32_t w[4];
};
__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint64_t seed, uint64_t env, uint64_t t) {
  uint32_t c0 = (uint32_t)env, c1 = (uint32_t)(env >> 32), c2 = (uint32_t)t, c3 = (uint32_t)(t >> 32);
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    uint32_t n1 = (uint32_t)p1;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    uint32_t n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  Philox4 o;
  o.w[0] = c0; o.w[1] = c1; o.w[2] = c2; o.w[3] = c3;
  return o;
}
// word -> uniform conventions (53-bit double as CPython's random(); 24-bit float)
__host__ __device__ __forceinline__ double u53(uint32_t a, uint32_t b) {  // CPython random(): 53 bits
  return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) * (1.0 / 9007199254740992.0);
}
__host__ __device__ __forceinline__ float u24(uint32_t a) { return (float)(a >> 8) * (1.0f / 16777216.0f); }
__host__ __device__ __forceinline__ int act_from_word(uint32_t w, int A) {
  return (int)(((uint64_t)w * (uint64_t)A) >> 32);
}

}  // namespace colo
