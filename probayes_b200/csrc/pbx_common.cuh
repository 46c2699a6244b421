// pbx_common.cuh -- shared host/device helpers for libpbx (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include "pbx.h"

// ---------------------------------------------------------------------------
// context + error plumbing (host)
// ---------------------------------------------------------------------------
struct pbx_ctx {
  int device;
  cudaStream_t stream;       // compute stream (borrowed or owned)
  cudaStream_t copy_stream;  // owned; D2H of the *_host entry points
  bool own_stream;
  int sm_count;
  int64_t launches;
  cudaEvent_t ev0, ev1;      // bracket the kernels of the most recent *_run call
  void* ws;                  // device workspace
  size_t ws_bytes;
  bool tables_ready;         // K1 math tables uploaded to this context's device
  bool exptab_ready;         // K4 exp table uploaded
  bool ndtab_ready;          // K5 ndtri table uploaded
  unsigned int* ticket;      // K4 last-CTA ticket (device, 256 B, zero between calls)
};

void pbx_set_error(const char* fmt, ...);
int pbx_ws_reserve(pbx_ctx* ctx, size_t bytes);

#define PBX_CUDA(call)                                                          \
  do {                                                                          \
    cudaError_t _e = (call);                                                    \
    if (_e != cudaSuccess) {                                                    \
      pbx_set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #call,          \
                    cudaGetErrorString(_e));                                    \
      return PBX_ERR_CUDA;                                                      \
    }                                                                           \
  } while (0)

#define PBX_REQUIRE(cond, ...)                                                  \
  do {                                                                          \
    if (!(cond)) {                                                              \
      pbx_set_error(__VA_ARGS__);                                               \
      return PBX_ERR_INVALID;                                                   \
    }                                                                           \
  } while (0)

#define PBX_LAUNCH_CHECK(ctx)                                                   \
  do {                                                                          \
    (ctx)->launches++;                                                          \
    PBX_CUDA(cudaGetLastError());                                               \
  } while (0)

// Raises the kernel's dynamic shared-memory limit to smem and launches it on the context's stream
template <class... P, class... A>
static int launch_smem(pbx_ctx* ctx, void (*kernel)(P...), int grid, int threads, size_t smem,
                       const A&... args) {
  PBX_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kernel<<<grid, threads, smem, ctx->stream>>>(args...);
  PBX_LAUNCH_CHECK(ctx);
  return PBX_OK;
}

// centred sufficient statistics of (x, y) observations for the normal likelihoods
// (pbx_mh_normreg.cu, "variant 3"); computed into the context workspace
struct NrStats { double N, cx, cy, Sxx, b1s, RSS, Su, Se, Seu, pad; };
int pbx_ss_compute(pbx_ctx* ctx, const double* x, const double* y, int64_t n, NrStats** out);

// ---------------------------------------------------------------------------
// probayes/constants.py:9-32 (fp64)
// ---------------------------------------------------------------------------
#define PBX_TINY 2.2250738585072014e-308
#define PBX_HUGE 1.7976931348623158e+308
#define PBX_LOG_HUGE 709.782712893384   /* log(PBX_HUGE) */
#define PBX_LOG_SQRT_2PI 0.91893853320467274178

// clamped log / exp of probayes/pscales.py:44-65 (NaN -> +huge, as the reference)
__device__ __forceinline__ double pbx_log_prob(double p) {
  return (p >= PBX_TINY) ? log(p) : -PBX_HUGE;
}
__device__ __forceinline__ double pbx_exp_logp(double l) {
  return (l <= PBX_LOG_HUGE) ? exp(l) : PBX_HUGE;
}

// Variable.apply_delta(bound=True), scalar branch (variable.py:700-727): proposal v of a
// coordinate whose current value is cur, inside [lo, hi]; closed ends clip, beyond an open
// end the proposal bounces back to the current value
__device__ __forceinline__ double pbx_bound(double v, double cur, double lo, double hi,
                                            bool olo, bool ohi) {
  if (!olo && !ohi) return fmax(lo, fmin(hi, v));
  if (olo && ohi) return (v > lo && v < hi) ? v : cur;
  if (olo) return (v < lo) ? cur : fmin(hi, v);
  return (v > hi) ? cur : fmax(lo, v);
}

// ---------------------------------------------------------------------------
// Philox4x32-10 counter RNG.  Stream layout documented in oracle/philox.py:
//   key = (seed lo, seed hi); counter = (step lo, step hi, chain, slot)
//   slot s -> draws for dims 2s, 2s+1:  u52(w0, w1), u32(w2)
//   threshold = t44(w3, w1) of slot 0  => one Philox block per step for D <= 2
// ---------------------------------------------------------------------------
struct pbx_u4 { uint32_t x, y, z, w; };

__host__ __device__ __forceinline__ pbx_u4 pbx_philox(uint32_t c0, uint32_t c1, uint32_t c2,
                                                      uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
#ifdef __CUDA_ARCH__
    uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
#else
    uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0;
    uint32_t hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
#endif
    uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  pbx_u4 o; o.x = c0; o.y = c1; o.z = c2; o.w = c3;
  return o;
}

// Same rounds with the 20 round keys precomputed on the host (they depend on the seed
// only): as constant-bank operands of the XORs they cost no instruction, the key
// schedule above costs two integer adds per round.
struct pbx_round_keys { uint32_t k[20]; };
static inline void pbx_make_round_keys(uint64_t seed, pbx_round_keys& rk) {
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  for (int r = 0; r < 10; ++r) {
    rk.k[2 * r] = k0;
    rk.k[2 * r + 1] = k1;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
}
#ifdef __CUDACC__
__device__ __forceinline__ pbx_u4 pbx_philox_rk(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                const pbx_round_keys& rk) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ rk.k[2 * r], n2 = hi0 ^ c3 ^ rk.k[2 * r + 1];
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
  }
  pbx_u4 o; o.x = c0; o.y = c1; o.z = c2; o.w = c3;
  return o;
}
#endif

__host__ __device__ __forceinline__ pbx_u4 pbx_block(uint64_t seed, uint64_t step, uint32_t chain,
                                                     uint32_t slot) {
  return pbx_philox((uint32_t)step, (uint32_t)(step >> 32), chain, slot, (uint32_t)seed,
                    (uint32_t)(seed >> 32));
}

#ifdef __CUDACC__
// The three uniforms are built by dropping the random bits into the mantissa of a
// double in [1, 2) and subtracting (1 - half ulp of the grid): exact, no I2F.
//   u52 = (2k+1) 2^-53, k = (w0 << 20) | (w1 >> 12)
__device__ __forceinline__ double pbx_u52(uint32_t w0, uint32_t w1) {
  double v = __hiloint2double((int)(0x3FF00000u | (w0 >> 12)), (int)((w0 << 20) | (w1 >> 12)));
  return v - 0.99999999999999988897769753748;       // 1 - 2^-53
}
//   u32 = (2 w2 + 1) 2^-33
__device__ __forceinline__ double pbx_u32(uint32_t w2) {
  double v = __hiloint2double((int)(0x3FF00000u | (w2 >> 12)), (int)(w2 << 20));
  return v - 0.99999999988358467817306518555;       // 1 - 2^-33
}
//   t44 = (2k+1) 2^-45, k = (w3 << 12) | (w1 & 0xfff)
__device__ __forceinline__ double pbx_t44(uint32_t w3, uint32_t w1) {
  double v = __hiloint2double((int)(0x3FF00000u | (w3 >> 12)),
                              (int)((w3 << 20) | ((w1 & 0xFFFu) << 8)));
  return v - 0.99999999999997157829056959599;       // 1 - 2^-45
}

// Box-Muller pair from one Philox block
__device__ __forceinline__ void pbx_normal_pair(pbx_u4 w, double& z0, double& z1) {
  double u1 = pbx_u52(w.x, w.y), u2 = pbx_u32(w.z);
  double r = sqrt(-2.0 * log(u1));
  double s, c;
  sincospi(2.0 * u2, &s, &c);
  z0 = r * c;
  z1 = r * s;
}

// ---- mbarrier helpers (shared::cta, generic-proxy producers/consumers) --------
__device__ __forceinline__ uint32_t pbx_smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void pbx_mbar_init(void* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(pbx_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void pbx_mbar_arrive(void* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(pbx_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void pbx_mbar_expect_tx(void* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(pbx_smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool pbx_mbar_try_wait(void* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(pbx_smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void pbx_mbar_wait(void* bar, uint32_t parity) {
  while (!pbx_mbar_try_wait(bar, parity)) {
  }
}
// 1-D bulk copy global -> shared (TMA engine, no tensor map), completes on mbarrier
__device__ __forceinline__ void pbx_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes,
                                             void* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(pbx_smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(pbx_smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void pbx_fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
#endif
