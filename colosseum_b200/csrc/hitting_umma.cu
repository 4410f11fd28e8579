// hitting_umma.cu -- the multi-target hitting-time sweep of the continuous diameter on the 5th-generation tensor cores
// (tcgen05.mma, accumulators in TMEM, operands staged by TMA behind an mbarrier ring).  sm_100a only.
//
// colosseum/hardness/measures/diameter.py:76-106 solves, for every target state k, a value iteration with gamma = 1,
// reward -1 and k absorbing.  All K targets share T, so one synchronous sweep over all of them is the GEMM
//     C[(s,a), k] = sum_j T[s,a,j] * E[k,j]              (S*A x S) . (S x K),  2*S*A*S*K flop
//     E'[k,s]     = (s == target_k) ? 0 : min_a (1 + C[(s,a), k])
// with a min-over-actions epilogue (multirhs.cuh is the SIMT FFMA version of the same sweep).
//
// Precision: the bar is 1e-4 relative in f32 mode (BASELINE.json north_star), which a single TF32 product (10-bit
// mantissa) does not meet.  Both operands are therefore split into two TF32-exact halves, x = hi + lo with
// hi = rn_tf32(x) and lo = rn_tf32(x - hi), and the sweep runs THREE tensor-core products per k-step into fp32 TMEM
// accumulators:  T_hi.E_hi  and  T_hi.E_lo + T_lo.E_hi   (the dropped T_lo.E_lo term is 2^-24 relative).  T is split
// once per solve, E' is split by the epilogue that produces it.  See the kernel for how the accumulators are kept at
// fp32 quality (the tensor core truncates when it accumulates).  Measured (scripts/umma_probe.py, 20 sweeps against
// fp64): 5e-7 max relative error on the S = 948 benchmark instance, 2e-6 on dense S = 2,048; the converged diameter
// of the S = 948 instance is 9e-7 from the fp64 fixed point.
//
// Layout.  T_split f32 [2][A][Sm][Sk] (part, action, state, next state; Sm = S rounded up to 128, Sk to 32, zero
// padded): for a fixed (part, action) the 128 states of a CTA are 128 consecutive rows, so ONE 2-D TMA box {32, 128}
// with SWIZZLE_128B lands a K-major [128][32] fp32 tile exactly as the UMMA shared-memory descriptor wants it.
// E_split f32 [2 ping/pong][2][Kp][Sk] likewise (rows = targets).  D (TMEM): lane = state of the tile, column =
// target of the tile; 4 * BN columns hold two hi-chain and two lo-chain accumulators (double buffering).
//
// Roles (320 threads): warp 0 lane 0 = TMA producer, warp 1 = TMEM allocator + (lane 0) MMA issuer, warps 2-9 =
// epilogue (warp w reads the TMEM lanes 32*(w%4) .. +31; the two warps of a lane quarter split the BN targets).
// One ring of NS stages {T_hi, T_lo, E_hi, E_lo} with full/empty mbarriers (tcgen05.commit frees a stage when the
// MMAs that read it have retired) and an accumulator ring (acc_full by tcgen05.commit, acc_empty by the epilogue warps).
// The epilogue keeps the running sum of the action and the min over actions in registers (64 + 64 per thread), then
// pins the target, carries converged targets forward, writes E' and its split twin and reduces max|dE| per target.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace colo {

constexpr int UM_BM = 128;       // states per CTA == UMMA M (cta_group::1)
constexpr int UM_BK = 32;        // fp32 per k-block == one 128-byte swizzle row; 4 MMAs of K = 8 each
constexpr int UM_EPI_WARPS = 8;   // two per TMEM lane quarter, each owning half of the tile's target columns
constexpr int UM_THREADS = 64 + 32 * UM_EPI_WARPS;  // warp 0 TMA, warp 1 MMA + TMEM, warps 2.. epilogue
constexpr int UM_T_TILE = UM_BM * UM_BK * 4;  // 16 KiB
constexpr int UM_NH = 3;  // hi-chain accumulators in flight: the drain of a group has two groups of MMAs to hide behind

struct UmmaSweepArgs {
  const float* E_in;   // [K][e_stride] fp32 iterate the sweep reads (its split twin is behind mapE, half `in_buf`)
  float* E_out;        // [K][e_stride]
  long long e_stride;
  float* E_split_out;  // [2][Kp][Sk] split twin of E_out
  const int* targets;
  const unsigned char* active;
  unsigned* resid;
  int S, A, K, Sm, Sk, Kp, in_buf;
  int flush;           // k-blocks accumulated in TMEM before the epilogue drains them (see the kernel)
  float max_value;
  int* overflow_flag;
};

// ---- PTX wrappers ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int x, int y, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(x), "r"(y), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_mc(void* dst, const CUtensorMap* map, int x, int y, uint64_t* bar, uint16_t mask) {
  // multicast: the box lands at the same shared-memory offset, and completes on the mbarrier at the same offset, in
  // every CTA of the cluster named by `mask`
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%2, %3}], "
      "[%4], %5;" ::"r"(smem_u32(dst)),
      "l"(map), "r"(x), "r"(y), "r"(smem_u32(bar)), "h"(mask)
      : "memory");
}
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(mask)
               : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// D[tmem] (+)= A[smem] . B[smem]^T, both operands K-major TF32, fp32 accumulate
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,"
      "%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]),
        "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]),
        "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// shared-memory matrix descriptor of a K-major tile whose rows are 128 bytes, SWIZZLE_128B (cute::UMMA::SmemDescriptor):
// start address >> 4 | LBO (ignored for swizzled K-major, 1) << 16 | SBO = 1024 B (8 rows) >> 4 << 32 | version 1 << 46
// | layout type SWIZZLE_128B (2) << 61.  The tile base is 1024-byte aligned (base_offset 0); a k-step of 8 fp32
// advances the start address by 32 bytes inside the swizzle atom.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): D fp32 (1 << 4), A/B TF32 (2 << 7, 2 << 10), both K-major,
// N >> 3 at bit 17, M >> 4 at bit 24
__host__ __device__ constexpr uint32_t umma_idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// x = hi + lo with both halves exactly representable in TF32: hi = x rounded to nearest TF32, lo = the remainder (exact
// in fp32, either sign, |lo| <= 2^-11 |x|) rounded to nearest TF32.  Rounding, not truncation: the tensor core
// truncates whatever low mantissa bits it is given, which for the always-positive operands of this sweep is a
// one-sided error (measured: -3e-7 relative per sweep with hi = x & 0xffffe000); pre-rounded halves have nothing left
// to truncate and their errors are two-sided (2^-24 relative).
__device__ __forceinline__ float tf32_rn(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
__device__ __forceinline__ void tf32_split(float x, float& hi, float& lo) {
  hi = tf32_rn(x);
  lo = tf32_rn(x - hi);
}

template <int BN>
struct UmmaCfg {
  static constexpr int E_TILE = BN * UM_BK * 4;
  static constexpr int STAGE = 2 * UM_T_TILE + 2 * E_TILE;  // 64 KiB (BN = 128) / 48 KiB (BN = 64)
  static constexpr int NS = BN == 128 ? 3 : 4;
  static constexpr int SMEM = NS * STAGE + 1024 /* alignment slack */ + 256 /* barriers, tmem pointer */;
  static constexpr int NCOLS = 4 * BN;  // UM_NH = 3 hi-chain accumulators + 1 lo-chain accumulator, BN columns each
};

// Why the accumulators are flushed.  The tensor core adds into its fp32 accumulator with TRUNCATION (round toward
// zero after aligning the addends), so a chain of n MMAs into one accumulator carries a bias of ~0.4 ulp(acc) per MMA,
// always downwards for the positive sums of this sweep -- measured here: 2.3e-6 relative per sweep at S = 256 with one
// chain of 96 MMAs, and the hitting-time fixed point amplifies a relative bias by ~max E.  Two measures keep the sweep
// at fp32 quality: (1) the two small products (T_hi.E_lo, T_lo.E_hi: 2^-11 of the result) get their own accumulator,
// so only the T_hi.E_hi chain truncates at full magnitude; (2) every `flush` k-blocks (4 MMAs of that chain each) the
// epilogue warps drain the accumulators into registers with round-to-nearest adds and the next chain restarts at zero:
// the bias is then that of `4 * flush` MMAs on a PARTIAL sum, ~1e-7 relative for flush = 1.  The accumulators are
// double buffered in TMEM (4 * BN columns), so the drain of one group overlaps the MMAs of the next.
// MC = true: launched as 2 x 2 thread-block clusters.  The two CTAs of a cluster row (same state tile, neighbouring target
// tiles) need the same T tiles, the two of a cluster column (same target tile) the same E tiles: every CTA loads HALF of
// each (64 T rows, BN/2 E rows, hi and lo) and the TMA multicasts it into both CTAs that need it -- the same 64 KiB land
// in every CTA's stage, but each byte is read from L2 once per pair instead of once per CTA (the L2 feed is what the
// kernel waits for at S >= 2,048).  A stage may be refilled only when all three writers' consumers have released it:
// the MMA issuer's tcgen05.commit is multicast to itself and to its row / column peers (empty barriers count 3).
template <int BN, bool MC>
__global__ void __launch_bounds__(UM_THREADS, 1)
hitting_umma_kernel(const __grid_constant__ CUtensorMap mapT, const __grid_constant__ CUtensorMap mapE,
                    const UmmaSweepArgs p) {
  using Cfg = UmmaCfg<BN>;
  constexpr int NS = Cfg::NS;
  constexpr int NE = UM_EPI_WARPS / 4;   // epilogue warps per TMEM lane quarter: each takes BN / NE target columns
  constexpr int CW = BN / NE;            // columns per epilogue thread
  extern __shared__ unsigned char umma_smem_raw[];
  unsigned char* smem = (unsigned char*)(((uintptr_t)umma_smem_raw + 1023) & ~(uintptr_t)1023);  // SWIZZLE_128B: 1024 B
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + NS * Cfg::STAGE);
  uint64_t* empty = full + NS;
  uint64_t* acc_full = empty + NS;   // [NH] MMA -> epilogue: the group's accumulators are final
  uint64_t* acc_empty = acc_full + UM_NH;  // [NH] epilogue -> MMA: drained
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + UM_NH);
  __shared__ int s_any_active;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int S = p.S, A = p.A, K = p.K;
  const int k0 = blockIdx.x * BN, s0 = blockIdx.y * UM_BM;
  const int nkb = p.Sk / UM_BK;
  const int G = p.flush;                      // k-blocks per accumulator group
  const int gpa = (nkb + G - 1) / G;          // groups per action

  // ---- a tile whose targets have all converged only carries E forward (its split twin is a function of the value)
  if (threadIdx.x == 0) s_any_active = p.active == nullptr;
  __syncthreads();
  if (p.active)
    for (int n = threadIdx.x; n < BN; n += UM_THREADS)
      if (k0 + n < K && p.active[k0 + n]) s_any_active = 1;
  __syncthreads();
  if (!MC && !s_any_active) {  // (a cluster keeps every CTA in the protocol: its peers wait for this CTA's halves)
    for (int i = threadIdx.x; i < UM_BM * BN; i += UM_THREADS) {
      const int m = i % UM_BM, n = i / UM_BM;
      const int s = s0 + m, k = k0 + n;
      if (s < S && k < K) {
        const float v = p.E_in[(size_t)k * p.e_stride + s];
        p.E_out[(size_t)k * p.e_stride + s] = v;
        float hi, lo;
        tf32_split(v, hi, lo);
        p.E_split_out[(size_t)k * p.Sk + s] = hi;
        p.E_split_out[((size_t)p.Kp + k) * p.Sk + s] = lo;
      }
    }
    return;
  }

  // ---- one-time setup: barriers (warp 0), TMEM columns (warp 1)
  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&mapT) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&mapE) : "memory");
    for (int i = 0; i < NS; ++i) {
      mbar_init(full + i, 1);
      mbar_init(empty + i, MC ? 3 : 1);
    }
    for (int i = 0; i < UM_NH; ++i) {
      mbar_init(acc_full + i, 1);
      mbar_init(acc_empty + i, UM_EPI_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  } else if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"((uint32_t)Cfg::NCOLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // cluster geometry (MC): rank = cx + 2 cy; row peer = rank ^ 1 (same states), column peer = rank ^ 2 (same targets)
  const int cx = blockIdx.x & 1, cy = blockIdx.y & 1;
  const uint16_t mask_T = (uint16_t)(0x3u << (2 * cy)), mask_E = (uint16_t)(0x5u << cx);
  const uint16_t mask_release = (uint16_t)((1u << (cx + 2 * cy)) | (1u << ((cx ^ 1) + 2 * cy)) | (1u << (cx + 2 * (cy ^ 1))));
  if (MC) cluster_sync_all();  // every CTA's barriers are initialised before a peer's copy or commit can reach them

  if (warp == 0) {
    if (lane == 0) {  // ===== TMA producer =====
      const int total = A * nkb;
      for (int it = 0; it < total; ++it) {
        const int st = it % NS;
        const uint32_t ph = (uint32_t)(it / NS) & 1u;
        mbar_wait(empty + st, ph ^ 1u);
        mbar_expect_tx(full + st, (uint32_t)Cfg::STAGE);
        const int a = it / nkb, kb = it - a * nkb;
        unsigned char* sb = smem + st * Cfg::STAGE;
        if (MC) {
          // my half of the shared tiles: 64 of the 128 state rows (mapT box {32, 64}), BN/2 of the BN target rows
          // (mapE box {32, BN/2}), each multicast to the two CTAs that use it
          const int tr = 64 * cx, er = (BN / 2) * cy;
          tma_load_2d_mc(sb + tr * 128, &mapT, kb * UM_BK, a * p.Sm + s0 + tr, full + st, mask_T);
          tma_load_2d_mc(sb + UM_T_TILE + tr * 128, &mapT, kb * UM_BK, (A + a) * p.Sm + s0 + tr, full + st, mask_T);
          tma_load_2d_mc(sb + 2 * UM_T_TILE + er * 128, &mapE, kb * UM_BK, (p.in_buf * 2) * p.Kp + k0 + er, full + st, mask_E);
          tma_load_2d_mc(sb + 2 * UM_T_TILE + Cfg::E_TILE + er * 128, &mapE, kb * UM_BK, (p.in_buf * 2 + 1) * p.Kp + k0 + er,
                         full + st, mask_E);
        } else {
          tma_load_2d(sb, &mapT, kb * UM_BK, a * p.Sm + s0, full + st);
          tma_load_2d(sb + UM_T_TILE, &mapT, kb * UM_BK, (A + a) * p.Sm + s0, full + st);
#pragma unroll
          for (int h = 0; h < BN / 64; ++h) {
            tma_load_2d(sb + 2 * UM_T_TILE + h * 8192, &mapE, kb * UM_BK, (p.in_buf * 2) * p.Kp + k0 + 64 * h, full + st);
            tma_load_2d(sb + 2 * UM_T_TILE + Cfg::E_TILE + h * 8192, &mapE, kb * UM_BK,
                        (p.in_buf * 2 + 1) * p.Kp + k0 + 64 * h, full + st);
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {  // ===== MMA issuer =====
      constexpr uint32_t idesc = umma_idesc_tf32(UM_BM, BN);
      int it = 0, f = 0;
      for (int a = 0; a < A; ++a)
        for (int g = 0; g < gpa; ++g, ++f) {
          const int b = f % UM_NH;
          mbar_wait(acc_empty + b, (((uint32_t)(f / UM_NH)) & 1u) ^ 1u);  // the epilogue has drained this buffer
          // the single lo-chain buffer is drained with the LAST group of the previous action: wait for that drain
          // before the first MMA of a new action overwrites it (never more than one completion behind: see NH)
          if (g == 0 && f > 0) mbar_wait(acc_empty + (f - 1) % UM_NH, ((uint32_t)((f - 1) / UM_NH)) & 1u);
          tc_fence_after();
          // TMEM columns: [0, NH*BN) a ring of NH hi-chain accumulators (one per group in flight), [NH*BN, (NH+1)*BN)
          // the lo-chain accumulator of the current action (the small products keep one chain per action, see above)
          const uint32_t d_hi = tmem_base + (uint32_t)(b * BN), d_lo = tmem_base + (uint32_t)(UM_NH * BN);
          const int kb_end = min(nkb, (g + 1) * G);
          for (int kb = g * G; kb < kb_end; ++kb, ++it) {
            const int st = it % NS;
            const uint32_t ph = (uint32_t)(it / NS) & 1u;
            mbar_wait(full + st, ph);
            tc_fence_after();
            const uint32_t sb = smem_u32(smem + st * Cfg::STAGE);
            const uint64_t d_th = umma_desc_sw128(sb), d_tl = umma_desc_sw128(sb + UM_T_TILE);
            const uint64_t d_eh = umma_desc_sw128(sb + 2 * UM_T_TILE),
                           d_el = umma_desc_sw128(sb + 2 * UM_T_TILE + Cfg::E_TILE);
            const bool first = kb == g * G;
#pragma unroll
            for (int k = 0; k < UM_BK / 8; ++k) {
              const uint64_t adv = (uint64_t)(k * 2);  // 8 fp32 = 32 bytes = 2 x 16-byte units of the start address
              umma_tf32(d_hi, d_th + adv, d_eh + adv, idesc, (first && k == 0) ? 0u : 1u);
              umma_tf32(d_lo, d_th + adv, d_el + adv, idesc, (first && g == 0 && k == 0) ? 0u : 1u);
              umma_tf32(d_lo, d_tl + adv, d_eh + adv, idesc, 1u);
            }
            if (MC) umma_commit_mc(empty + st, mask_release);  // ... in this CTA and in the two peers that write into it
            else umma_commit(empty + st);  // the stage is free once these MMAs have read it
          }
          umma_commit(acc_full + b);  // this group's accumulators are final
        }
    }
  } else {
    // ===== epilogue: drain the accumulator groups (round-to-nearest adds), min over actions, pin / carry / residual,
    //       E' and its split twin =====
    const int ew = warp - 2;
    const int q = warp & 3;        // the TMEM lane quarter this warp may read
    const int half = ew / 4;       // which CW columns of the tile
    const int s = s0 + q * 32 + lane;
    const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(half * CW);
    float best[CW];
#pragma unroll
    for (int i = 0; i < CW; ++i) best[i] = INFINITY;
    int f = 0;
    for (int a = 0; a < A; ++a) {
      float acc[CW];
#pragma unroll
      for (int i = 0; i < CW; ++i) acc[i] = 0.f;
      for (int g = 0; g < gpa; ++g, ++f) {
        const int b = f % UM_NH;
        mbar_wait(acc_full + b, ((uint32_t)(f / UM_NH)) & 1u);
        tc_fence_after();
        const uint32_t t_hi = lane_base + (uint32_t)(b * BN);
        {  // the thread's CW columns of the group: CW / 32 loads of 32 columns in flight, ONE wait
          float vh[CW / 32][32];
#pragma unroll
          for (int c = 0; c < CW / 32; ++c) tmem_ld32(t_hi + (uint32_t)(c * 32), vh[c]);
          tmem_ld_wait();
#pragma unroll
          for (int c = 0; c < CW / 32; ++c)
#pragma unroll
            for (int i = 0; i < 32; ++i) acc[c * 32 + i] += vh[c][i];
        }
        if (g == gpa - 1) {  // the action's last group: its lo chain is final too (commits are cumulative)
          const uint32_t t_lo = lane_base + (uint32_t)(UM_NH * BN);
          float vl[CW / 32][32];
#pragma unroll
          for (int c = 0; c < CW / 32; ++c) tmem_ld32(t_lo + (uint32_t)(c * 32), vl[c]);
          tmem_ld_wait();
#pragma unroll
          for (int c = 0; c < CW / 32; ++c)
#pragma unroll
            for (int i = 0; i < 32; ++i) acc[c * 32 + i] += vl[c][i];
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(acc_empty + b);
      }
#pragma unroll
      for (int i = 0; i < CW; ++i) best[i] = fminf(best[i], 1.f + acc[i]);
    }
    // the previous iterate of this thread's CW (target, state) pairs: every load in flight before any is used (one
    // dependent L2 round trip per column would cost more than the tile's MMAs at S ~ 1,000)
    float old[CW];
#pragma unroll
    for (int i = 0; i < CW; ++i) {
      const int k = k0 + half * CW + i;
      old[i] = (k < K && s < S) ? p.E_in[(size_t)k * p.e_stride + s] : 0.f;
    }
#pragma unroll
    for (int i = 0; i < CW; ++i) {
      const int k = k0 + half * CW + i;
      if (k < K) {  // warp-uniform
        const int tgt = __ldg(p.targets + k);
        const bool act = p.active == nullptr || p.active[k] != 0;
        float dlt = 0.f;
        if (s < S) {
          float nv = (s == tgt) ? 0.f : best[i];
          if (!act) nv = old[i];
          p.E_out[(size_t)k * p.e_stride + s] = nv;
          float hi, lo;
          tf32_split(nv, hi, lo);
          p.E_split_out[(size_t)k * p.Sk + s] = hi;
          p.E_split_out[((size_t)p.Kp + k) * p.Sk + s] = lo;
          dlt = fabsf(nv - old[i]);
          if (p.max_value > 0.f && nv > p.max_value && p.overflow_flag) *p.overflow_flag = 1;
        }
        const unsigned m = __reduce_max_sync(FULL, __float_as_uint(dlt));  // dlt >= 0: IEEE order == unsigned order
        if (lane == 0 && m != 0u && p.resid) atomicMax(p.resid + k, m);
      }
    }
  }
  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (MC) cluster_sync_all();  // no CTA leaves while a peer's copy or commit may still be addressed to it
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)Cfg::NCOLS)
                 : "memory");
  }
}

// T f32 [S,A,S] -> T_split f32 [2][A][Sm][Sk] (TF32-exact hi, remainder lo; zero padding)
__global__ void __launch_bounds__(256) umma_split_T_kernel(const float* __restrict__ T, int S, int A, int Sm, int Sk,
                                                           float* __restrict__ out) {
  const long long n = (long long)A * Sm * Sk;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(i % Sk);
    const long long r = i / Sk;
    const int s = (int)(r % Sm), a = (int)(r / Sm);
    float v = 0.f;
    if (s < S && j < S) v = __ldg(T + ((size_t)s * A + a) * S + j);
    float hi, lo;
    tf32_split(v, hi, lo);
    out[i] = hi;
    out[n + i] = lo;
  }
}

// ---- host side ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return (EncodeTiledFn)p;
  }();
  return fn;
}

static int make_map_2d(CUtensorMap* map, float* base, int cols, long long rows, int box_rows) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled is not available from this driver");
    return COLO_ERR_CUDA;
  }
  const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)cols * 4};
  const cuuint32_t box[2] = {(cuuint32_t)UM_BK, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                        CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed: CUresult %d (cols %d rows %lld box %d)", (int)r, cols, rows, box_rows);
    return COLO_ERR_CUDA;
  }
  return COLO_OK;
}

struct UmmaPlan {
  float* T_split = nullptr;  // [2][A][Sm][Sk]
  float* E_split = nullptr;  // [2][2][Kp][Sk]
  CUtensorMap mapT, mapE;
  int S = 0, A = 0, K = 0, Sm = 0, Sk = 0, Kp = 0, BN = 0, cur = 0, flush = 1;
  bool mc = false;  // 2 x 2 clusters with multicast TMA
};

bool hitting_umma_supported(int S, int A, int K) {
  static const bool off = getenv("COLO_NO_UMMA") != nullptr;
  return !off && A >= 1 && S >= 128 && K >= 64 && encode_tiled_fn() != nullptr;
}

int hitting_umma_plan(const float* T, int S, int A, int K, UmmaPlan** out, cudaStream_t st) {
  COLO_ARG_CHECK(T && out && A >= 1 && S >= 1 && K >= 1, "hitting_umma_plan: T, A >= 1");
  UmmaPlan* pl = new UmmaPlan();
  pl->S = S; pl->A = A; pl->K = K;
  // tile width: 128 targets per CTA, 64 when that grid would leave SMs idle
  pl->BN = (long long)((K + 127) / 128) * ((S + UM_BM - 1) / UM_BM) >= (long long)sm_count() ? 128 : 64;
  {
    const char* e = getenv("COLO_UMMA_FLUSH");  // accuracy / speed probe: k-blocks per TMEM accumulator chain
    pl->flush = e && atoi(e) >= 1 ? atoi(e) : 1;
    const char* bn = getenv("COLO_UMMA_BN");
    if (bn && (atoi(bn) == 64 || atoi(bn) == 128)) pl->BN = atoi(bn);
  }
  {
    // 2 x 2 clusters with multicast TMA halve the L2 reads.  Measured (scripts/umma_probe.py, three hi accumulators in
    // flight): S = 2,048 A = 8: 615 us per sweep with clusters, 741 without; no difference at S <= 1,024, where the
    // padding to whole clusters is pure overhead.  On when the grid fills the machine; COLO_UMMA_CLUSTER=0/1 forces it.
    const char* e = getenv("COLO_UMMA_CLUSTER");
    const long long tiles = (long long)((K + pl->BN - 1) / pl->BN) * ((S + UM_BM - 1) / UM_BM);
    pl->mc = e ? atoi(e) == 1 : tiles >= (long long)sm_count();
  }
  const int m_unit = pl->mc ? 2 * UM_BM : UM_BM, n_unit = pl->mc ? 2 * pl->BN : pl->BN;  // whole 2 x 2 clusters
  pl->Sm = (S + m_unit - 1) / m_unit * m_unit;
  pl->Sk = (S + UM_BK - 1) / UM_BK * UM_BK;
  pl->Kp = (K + n_unit - 1) / n_unit * n_unit;
  const size_t t_elems = (size_t)2 * A * pl->Sm * pl->Sk, e_elems = (size_t)4 * pl->Kp * pl->Sk;
  cudaError_t e = cudaMallocAsync((void**)&pl->T_split, t_elems * 4, st);
  if (e == cudaSuccess) e = cudaMallocAsync((void**)&pl->E_split, e_elems * 4, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(pl->E_split, 0, e_elems * 4, st);  // E = 0 and finite padding
  if (e != cudaSuccess) {
    set_error("hitting_umma_plan: %s", cudaGetErrorString(e));
    if (pl->T_split) cudaFreeAsync(pl->T_split, st);
    delete pl;
    return COLO_ERR_CUDA;
  }
  const long long n = (long long)A * pl->Sm * pl->Sk;
  const int grid = (int)((n + 255) / 256 < (long long)sm_count() * 16 ? (n + 255) / 256 : (long long)sm_count() * 16);
  umma_split_T_kernel<<<grid, 256, 0, st>>>(T, S, A, pl->Sm, pl->Sk, pl->T_split);
  int r = check_launch("umma_split_T_kernel");
  if (r == COLO_OK) r = make_map_2d(&pl->mapT, pl->T_split, pl->Sk, (long long)2 * A * pl->Sm, pl->mc ? UM_BM / 2 : UM_BM);
  if (r == COLO_OK) r = make_map_2d(&pl->mapE, pl->E_split, pl->Sk, (long long)4 * pl->Kp, pl->mc ? pl->BN / 2 : 64);
  if (r != COLO_OK) {
    cudaFreeAsync(pl->T_split, st);
    cudaFreeAsync(pl->E_split, st);
    delete pl;
    return r;
  }
  *out = pl;
  return COLO_OK;
}

void hitting_umma_free(UmmaPlan* pl, cudaStream_t st) {
  if (!pl) return;
  cudaFreeAsync(pl->T_split, st);
  cudaFreeAsync(pl->E_split, st);
  delete pl;
}

// overwrite the split twin of the CURRENT iterate from a full fp32 E (a solve that starts from a given E0)
__global__ void __launch_bounds__(256) umma_split_E_kernel(const float* __restrict__ E, long long e_stride, int K, int S,
                                                           int Kp, int Sk, float* __restrict__ out) {
  const long long n = (long long)K * S;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int s = (int)(i % S), k = (int)(i / S);
    const float v = E[(size_t)k * e_stride + s];
    float hi, lo;
    tf32_split(v, hi, lo);
    out[(size_t)k * Sk + s] = hi;
    out[((size_t)Kp + k) * Sk + s] = lo;
  }
}

int hitting_umma_set_iterate(UmmaPlan* pl, const float* E, long long e_stride, cudaStream_t st) {
  const long long n = (long long)pl->K * pl->S;
  const int grid = (int)((n + 255) / 256 < (long long)sm_count() * 16 ? (n + 255) / 256 : (long long)sm_count() * 16);
  umma_split_E_kernel<<<grid, 256, 0, st>>>(E, e_stride, pl->K, pl->S, pl->Kp, pl->Sk,
                                            pl->E_split + (size_t)pl->cur * 2 * pl->Kp * pl->Sk);
  return check_launch("umma_split_E_kernel");
}

// one synchronous sweep E_in -> E_out (fp32, [K][e_stride]); the plan keeps the split twins and flips its ping/pong
int hitting_umma_sweep(UmmaPlan* pl, const float* E_in, float* E_out, long long e_stride, const int* targets,
                       const unsigned char* active, unsigned* resid, double max_value, int* overflow_flag, cudaStream_t st) {
  UmmaSweepArgs a;
  a.E_in = E_in; a.E_out = E_out; a.e_stride = e_stride;
  a.E_split_out = pl->E_split + (size_t)(1 - pl->cur) * 2 * pl->Kp * pl->Sk;
  a.targets = targets; a.active = active; a.resid = resid;
  a.S = pl->S; a.A = pl->A; a.K = pl->K; a.Sm = pl->Sm; a.Sk = pl->Sk; a.Kp = pl->Kp; a.in_buf = pl->cur;
  a.max_value = (float)max_value; a.overflow_flag = overflow_flag;
  a.flush = pl->flush;
  dim3 grid(pl->Kp / pl->BN, pl->Sm / UM_BM);
  auto launch = [&](auto kern, size_t smem) -> int {
    { const int es = ensure_dynamic_smem((const void*)kern, smem); if (es != COLO_OK) return es; }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(UM_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = pl->mc ? 2 : 1;
    attr[0].val.clusterDim.y = pl->mc ? 2 : 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    COLO_CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, pl->mapT, pl->mapE, a));
    return COLO_OK;
  };
  int r;
  count_solver_path(COLO_PATH_HIT_UMMA);
  if (pl->BN == 128) r = pl->mc ? launch(hitting_umma_kernel<128, true>, UmmaCfg<128>::SMEM) : launch(hitting_umma_kernel<128, false>, UmmaCfg<128>::SMEM);
  else r = pl->mc ? launch(hitting_umma_kernel<64, true>, UmmaCfg<64>::SMEM) : launch(hitting_umma_kernel<64, false>, UmmaCfg<64>::SMEM);
  if (r != COLO_OK) return r;
  pl->cur ^= 1;
  return check_launch("hitting_umma_kernel");
}

}  // namespace colo

extern "C" {

// Fixed number of synchronous hitting-time sweeps on the tensor cores (parity / throughput probe of the kernel behind
// colo_diameter_continuous_f32's dense path): E f32 [K][S] in place, E = 0 at the start when `zero_start`.
int colo_hitting_umma_sweeps_f32(const float* T, const int* targets, int K, int S, int A, int n_sweeps, int zero_start,
                                 float* E, float* E_work, void* stream) {
  COLO_ARG_CHECK(T && targets && E && E_work && n_sweeps >= 0, "T, targets, E, E_work");
  COLO_ARG_CHECK(colo::hitting_umma_supported(S, A, K), "shape not supported by the tcgen05 path (S >= 128, K >= 64)");
  cudaStream_t st = (cudaStream_t)stream;
  colo::UmmaPlan* pl = nullptr;
  int r = colo::hitting_umma_plan(T, S, A, K, &pl, st);
  if (r != COLO_OK) return r;
  if (zero_start)
    COLO_CUDA_TRY(cudaMemsetAsync(E, 0, (size_t)K * S * 4, st));
  else
    r = colo::hitting_umma_set_iterate(pl, E, S, st);
  float* cur = E;
  float* nxt = E_work;
  for (int i = 0; i < n_sweeps && r == COLO_OK; ++i) {
    r = colo::hitting_umma_sweep(pl, cur, nxt, S, targets, nullptr, nullptr, 0.0, nullptr, st);
    float* t = cur; cur = nxt; nxt = t;
  }
  if (r == COLO_OK && cur != E) COLO_CUDA_TRY(cudaMemcpyAsync(E, cur, (size_t)K * S * 4, cudaMemcpyDeviceToDevice, st));
  colo::hitting_umma_free(pl, st);
  return r;
}

}  // extern "C"
