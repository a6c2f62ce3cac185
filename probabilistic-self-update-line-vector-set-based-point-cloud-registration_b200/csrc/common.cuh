// common.cuh -- shared device/host helpers of the PSULVSB B200 library (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdio>
#include <string>

#include "../../include/psulvsb.h"

namespace psulvsb {

// ------------------------------------------------------------------------------------------
// error plumbing (thread-local message behind psulvsb_last_error)
// ------------------------------------------------------------------------------------------
void set_error(const std::string& msg);
int fail(int code, const std::string& msg);

#define PSU_CUDA(call)                                                                              \
  do {                                                                                              \
    cudaError_t e__ = (call);                                                                       \
    if (e__ != cudaSuccess) {                                                                       \
      return ::psulvsb::fail(PSULVSB_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); \
    }                                                                                               \
  } while (0)

#define PSU_CHECK_LAUNCH(name)                                                                      \
  do {                                                                                              \
    cudaError_t e__ = cudaGetLastError();                                                           \
    if (e__ != cudaSuccess) {                                                                       \
      return ::psulvsb::fail(PSULVSB_ERR_CUDA, std::string(name) + " launch: " + cudaGetErrorString(e__)); \
    }                                                                                               \
  } while (0)

// PSULVSB_ERR_NO_DEVICE (with its message) when no CUDA device is visible, else PSULVSB_OK
int need_device();

// SMs of the current device (cudaDevAttrMultiProcessorCount, cached per device): every grid is sized from it
int sm_count();

// Debug / test switches (psulvsb_debug_set in include/psulvsb.h).  They never change results, only which of several
// equivalent code paths runs; production callers leave them alone.  No environment variable is read anywhere.
struct DebugKnobs {
  double gnc_deep_margin = 0.0;   // > 0: overrides the remaining-margin threshold (rad) for parking sleeping line vectors
  int gnc_cluster = 0;            // 1, 2, 4, 8: CTAs per registration of the GNC-TLS kernel (512 threads, one CTA per SM)
  int gnc_prefetch = -1;          // >= 0: look-ahead (double-steps) of the L2 prefetch in the streamed GNC pass
  int gnc_grid_lv = 0;            // > 0: line vectors per CTA above which GNC-TLS goes to grid mode (default 4096)
  int gnc_cps = 0;                // 1, 2, 4: CTAs per SM (512 / 256 / 128 threads) of one-CTA-per-registration GNC-TLS launches
  int gnc_park_pct = 0;           // > 0: share (%) of deep sleepers that arms a parking pass of the GNC-TLS kernel
  int sample_list_cap_test = 0;   // > 0: caps the sampler's bucket lists and its on-chip duplicate table (exercises both fallbacks)
  int k1_variant = 0;             // 1..4: rows per thread of the consistency kernel
  int upload_prof = 0;            // 1: print the upload's phase timings to stderr
  int edge_wide = 0;              // 1: the engine keeps the reduced set in EdgeWide format whatever the working-set size
};
DebugKnobs& debug_knobs();

inline unsigned long long ceil_div_ull(unsigned long long a, unsigned long long b) { return (a + b - 1) / b; }
// doubles of sorting scratch block_translation (solve_dev.cuh) needs for n_points points (+ the pseudo-measurement)
inline size_t translation_sort_doubles(int n_points) {
  size_t m = 1;
  while (m < (size_t)n_points + 1) m <<= 1;
  return m;
}

// ------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon, Moraes, Dror, Shaw, SC'11): the replayable sample stream.
//   counter = (block_lo, block_hi, event, domain), key = (seed_lo, seed_hi)
//   rand31(k)    = word[k & 3] of block k>>2, shifted right by one (31 bits, like glibc rand())
//   uniform01(k) = 53-bit fraction from words 0,1 of block k
// ------------------------------------------------------------------------------------------
struct Philox4 {
  uint32_t w[4];
};

__host__ __device__ __forceinline__ uint32_t mulhi32(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}

__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint64_t seed, uint32_t domain, uint32_t event,
                                                          uint64_t block) {
  uint32_t c0 = (uint32_t)block, c1 = (uint32_t)(block >> 32), c2 = event, c3 = domain;
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = mulhi32(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = mulhi32(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0;
    c1 = lo1;
    c2 = n2;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  Philox4 o;
  o.w[0] = c0;
  o.w[1] = c1;
  o.w[2] = c2;
  o.w[3] = c3;
  return o;
}

__host__ __device__ __forceinline__ uint32_t philox_rand31(uint64_t seed, uint32_t domain, uint32_t event,
                                                           uint64_t k) {
  Philox4 o = philox4x32_10(seed, domain, event, k >> 2);
  return o.w[k & 3] >> 1;
}

__host__ __device__ __forceinline__ double philox_uniform01(uint64_t seed, uint32_t domain, uint32_t event,
                                                            uint64_t k) {
  Philox4 o = philox4x32_10(seed, domain, event, k);
  return ((double)(o.w[0] >> 5) * 67108864.0 + (double)(o.w[1] >> 6)) / 9007199254740992.0;
}

// ------------------------------------------------------------------------------------------
// FP64 helpers with the reference's operation order and NO fused multiply-add, so results are
// bit-identical to an x86-64 build without FMA contraction (the reference's default Release
// build, CMakeLists.txt:9-13,21).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }

// (x^2 + y^2) + z^2, as Eigen's 3-element reduction evaluates it (SURVEY.md appendix A.2)
__device__ __forceinline__ double sqnorm3(double x, double y, double z) {
  return dadd(dadd(dmul(x, x), dmul(y, y)), dmul(z, z));
}

// centred FP64 point -> FP32 tile entry (x, y, z, |p|^2); the squared norm is taken of the ROUNDED
// coordinates in FP64 and rounded once (K1 fast path, DESIGN.md)
__device__ __forceinline__ float4 pack_point(double x, double y, double z) {
  const float xf = (float)x, yf = (float)y, zf = (float)z;
  const double n2 = (double)xf * (double)xf + (double)yf * (double)yf + (double)zf * (double)zf;
  return make_float4(xf, yf, zf, (float)n2);
}

// Pair-interleaved tile layout of packed points (K1's column tiles): points 2q and 2q + 1 share two float4 records,
//   il[2q] = (x_2q, x_2q+1, y_2q, y_2q+1),  il[2q + 1] = (z_2q, z_2q+1, n_2q, n_2q+1)      (n = |p|^2),
// so that one LDS.128 hands a thread the SAME coordinate of two neighbouring columns in an aligned register pair -- the
// 64-bit operand of an FFMA2.  An array of n points has (n + 1) & ~1 records (an odd n ends with a zero point).
__host__ __device__ inline size_t il_records(size_t n) { return (n + 1) & ~(size_t)1; }
__device__ __forceinline__ void il_store(float4* __restrict__ il, int i, const float4 p) {
  float* f = reinterpret_cast<float*>(il + (i & ~1)) + (i & 1);
  f[0] = p.x;
  f[2] = p.y;
  f[4] = p.z;
  f[6] = p.w;
}
__device__ __forceinline__ float4 il_load(const float4* __restrict__ il, int i) {
  const float* f = reinterpret_cast<const float*>(il + (i & ~1)) + (i & 1);
  return make_float4(f[0], f[2], f[4], f[6]);
}

// ------------------------------------------------------------------------------------------
// mbarrier / 1-D TMA bulk copy / packed FP32 helpers shared by the tile-streaming kernels (K1, K3, K4)
// ------------------------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// 1-D TMA bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP).  16-byte aligned, size a
// multiple of 16.
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// Packed FP32 (Blackwell FFMA2 / FADD2: two FP32 operations per lane and issue slot).  Each half is an IEEE
// round-to-nearest fma / add; ptxas folds a {x, x} operand into the instruction's .F32 broadcast operand form.
__device__ __forceinline__ float2 fma2(const float2 a, const float2 b, const float2 c) {
  unsigned long long ra, rb, rc, rd;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rc) : "f"(c.x), "f"(c.y));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
  float2 d;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(rd));
  return d;
}
__device__ __forceinline__ float2 add2(const float2 a, const float2 b) {
  unsigned long long ra, rb, rd;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(rd) : "l"(ra), "l"(rb));
  float2 d;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(rd));
  return d;
}
__device__ __forceinline__ float2 bc2(const float x) { return make_float2(x, x); }
#endif  // __CUDACC__

struct Mat3d {
  double m[3][3];  // row-major
};

// ------------------------------------------------------------------------------------------
// warp / block reductions
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ int warp_sum_int(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace psulvsb
