// pbx_grid.cu -- K3/K4: discrete grid exact inference of a normal (mu, sigma)
// posterior (examples/dgei/dgei_norm1d_improved.py:36-43).
//
// K3  log-joint[m][s] = (logprior_mu[m] + logprior_sigma[s])
//                       + sum_i norm.logpdf(x_i; mu_m, sigma_s)   (or t.logpdf, df nu)
//     The reference materialises the [N, M, S] tensor and np.sum(axis=0)s it
//     (probayes/rf.py:565-581, pd.py:368), then prod_rule adds the priors
//     (pd_utils.py:85-328, pscales.py:160-216).  Here every CTA owns 1 mu x 1024
//     sigma cells, keeps 8 running sums per thread in registers and streams the
//     observations through shared memory (1-D TMA bulk copies, 3-stage mbarrier
//     pipeline, 128-bit broadcast reads): 8 B * N of L2 traffic per 1024 cells, no
//     [N, M, S] temporary.  FP64-pipe bound: 2 instructions per (cell, observation).
// K4  PD.conditionalise (pd.py:285-295): p - max; exp; / max(tiny, sum); clamped log
//     PD.marginalise   (pd.py:162-164): exp (no shift); sum over an axis; clamped log
//     in two deterministic passes over the grid (below); HBM bound.
#include <math.h>
#include "pbx_common.cuh"

#define GR_TILE 1024
#define GR_STAGES 3
#define GR_THREADS 128
#define GR_KS 8                        // sigma cells per thread

// kLik = PBX_LIK_STUDENT_T: t.logpdf with df nu, the sum N logc - N log sigma
// - (nu+1)/2 sum_i log1p((x_i - mu)^2 / (nu sigma^2)) (logc from the host, see pbx.h).  df and
// logc are the last arguments, unread by the normal instantiation, so that its argument
// offsets and SASS are those of the normal-only kernel
template <int kLik>
__global__ void __launch_bounds__(GR_THREADS)
    grid_logjoint_kernel(const double* __restrict__ x, int64_t N, const double* __restrict__ mu,
                         const double* __restrict__ sigma, int S,
                         const double* __restrict__ lp_mu, const double* __restrict__ lp_sigma,
                         double* __restrict__ out, int use_tma, double df, double logc) {
  constexpr bool kT = kLik == PBX_LIK_STUDENT_T;
  __shared__ __align__(128) double sm[GR_STAGES][GR_TILE];
  __shared__ __align__(8) unsigned long long full_bar[GR_STAGES];
  const int m = blockIdx.y;
  const int s_base = blockIdx.x * (GR_THREADS * GR_KS) + threadIdx.x;
  const double mu_m = mu[m];
  double isg[GR_KS], acc[GR_KS];
#pragma unroll
  for (int k = 0; k < GR_KS; ++k) {
    const int s = s_base + k * GR_THREADS;
    // Student-t: isg holds q = 1/(nu sigma^2)
    isg[k] = (s < S) ? (kT ? 1.0 / (df * (sigma[s] * sigma[s])) : 1.0 / sigma[s]) : 0.0;
    acc[k] = 0.0;
  }
  const int64_t n_full = N / GR_TILE;
  constexpr uint32_t kTileBytes = GR_TILE * sizeof(double);
  if (threadIdx.x == 0) {
    for (int s = 0; s < GR_STAGES; ++s) pbx_mbar_init(&full_bar[s], 1);
    pbx_fence_barrier_init();
  }
  __syncthreads();
  auto tile_math = [&](const double* sx, int cnt) {
#pragma unroll 2
    for (int i = 0; i < cnt; i += 2) {
      const double2 xv = *reinterpret_cast<const double2*>(sx + i);
      const double d0 = xv.x - mu_m, d1 = xv.y - mu_m;
#pragma unroll
      for (int k = 0; k < GR_KS; ++k) {
        if (kT) {
          acc[k] += log1p((d0 * d0) * isg[k]);
          acc[k] += log1p((d1 * d1) * isg[k]);
        } else {
          const double z0 = d0 * isg[k], z1 = d1 * isg[k];
          acc[k] = fma(z0, z0, acc[k]);
          acc[k] = fma(z1, z1, acc[k]);
        }
      }
    }
  };
  if (use_tma) {
    auto issue = [&](int64_t t) {
      const int s = (int)(t % GR_STAGES);
      pbx_mbar_expect_tx(&full_bar[s], kTileBytes);
      pbx_bulk_g2s(sm[s], x + t * GR_TILE, kTileBytes, &full_bar[s]);
    };
    if (threadIdx.x == 0)
      for (int64_t t = 0; t < n_full && t < GR_STAGES; ++t) issue(t);
    for (int64_t t = 0; t < n_full; ++t) {
      const int s = (int)(t % GR_STAGES);
      pbx_mbar_wait(&full_bar[s], (uint32_t)(t / GR_STAGES) & 1);
      tile_math(sm[s], GR_TILE);
      __syncthreads();
      if (threadIdx.x == 0 && t + GR_STAGES < n_full) issue(t + GR_STAGES);
    }
  } else {
    for (int64_t t = 0; t < n_full; ++t) {
      for (int i = threadIdx.x; i < GR_TILE; i += GR_THREADS) sm[0][i] = x[t * GR_TILE + i];
      __syncthreads();
      tile_math(sm[0], GR_TILE);
      __syncthreads();
    }
  }
  const int rem = (int)(N - n_full * GR_TILE);
  if (rem > 0) {
    __syncthreads();
    for (int i = threadIdx.x; i < GR_TILE; i += GR_THREADS)
      sm[0][i] = (i < rem) ? x[n_full * GR_TILE + i] : 0.0;
    __syncthreads();
    const int even = rem & ~1;
    tile_math(sm[0], even);
    if (rem & 1) {
      const double d0 = sm[0][even] - mu_m;
#pragma unroll
      for (int k = 0; k < GR_KS; ++k) {
        if (kT) {
          acc[k] += log1p((d0 * d0) * isg[k]);
        } else {
          const double z0 = d0 * isg[k];
          acc[k] = fma(z0, z0, acc[k]);
        }
      }
    }
  }
  const double n = (double)N, lpm = lp_mu[m];
#pragma unroll
  for (int k = 0; k < GR_KS; ++k) {
    const int s = s_base + k * GR_THREADS;
    if (s < S) {
      const double ll = kT ? -(0.5 * (df + 1.0)) * acc[k] + n * (logc - log(sigma[s]))
                           : -acc[k] * 0.5 - n * (PBX_LOG_SQRT_2PI + log(sigma[s]));
      out[(int64_t)m * S + s] = (lpm + lp_sigma[s]) + ll;      // prior first (prod_rule)
    }
  }
}

// ---------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------
template <int kLik>
static int grid_logjoint(pbx_ctx* ctx, const char* who, const double* x_obs, int64_t n_obs,
                         const double* mu, int32_t n_mu, const double* sigma, int32_t n_sigma,
                         const double* logprior_mu, const double* logprior_sigma, double* out,
                         double df, double logc) {
  PBX_REQUIRE(ctx && x_obs && mu && sigma && logprior_mu && logprior_sigma && out,
              "%s: null argument", who);
  PBX_REQUIRE(n_obs >= 1 && n_mu >= 1 && n_sigma >= 1, "%s: sizes must be positive", who);
  PBX_REQUIRE(n_mu <= 65535, "%s: at most 65535 mu rows per call (slab it)", who);
  PBX_CUDA(cudaSetDevice(ctx->device));
  dim3 grid((n_sigma + GR_THREADS * GR_KS - 1) / (GR_THREADS * GR_KS), n_mu);
  const int use_tma = (((uintptr_t)x_obs) % 16 == 0) ? 1 : 0;
  PBX_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
  grid_logjoint_kernel<kLik><<<grid, GR_THREADS, 0, ctx->stream>>>(
      x_obs, n_obs, mu, sigma, n_sigma, logprior_mu, logprior_sigma, out, use_tma, df, logc);
  PBX_LAUNCH_CHECK(ctx);
  PBX_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
  return PBX_OK;
}

extern "C" int pbx_grid_norm_logjoint(pbx_ctx* ctx, const double* x_obs, int64_t n_obs,
                                      const double* mu, int32_t n_mu, const double* sigma,
                                      int32_t n_sigma, const double* logprior_mu,
                                      const double* logprior_sigma, double* out) {
  return grid_logjoint<PBX_LIK_NORMAL>(ctx, "pbx_grid_norm_logjoint", x_obs, n_obs, mu, n_mu,
                                       sigma, n_sigma, logprior_mu, logprior_sigma, out, 0.0,
                                       0.0);
}

extern "C" int pbx_grid_t_logjoint(pbx_ctx* ctx, const double* x_obs, int64_t n_obs,
                                   const double* mu, int32_t n_mu, const double* sigma,
                                   int32_t n_sigma, const double* logprior_mu,
                                   const double* logprior_sigma, double* out, double df,
                                   double logc) {
  PBX_REQUIRE(df > 0.0 && isfinite(df), "pbx_grid_t_logjoint: needs 0 < df < inf (got %g)", df);
  PBX_REQUIRE(isfinite(logc), "pbx_grid_t_logjoint: logc is not finite");
  return grid_logjoint<PBX_LIK_STUDENT_T>(ctx, "pbx_grid_t_logjoint", x_obs, n_obs, mu, n_mu,
                                          sigma, n_sigma, logprior_mu, logprior_sigma, out, df,
                                          logc);
}

// ---------------------------------------------------------------------------
// opt-in: the same log-joint from centred sufficient statistics of the observations
// (see pbx_mh_normreg.cu, variant 3): sum (x - mu)^2 = RSS + N a^2 - 2 a Se with
// a = mu - mean(x), every term non-negative or a rounding residual.  O(M S) instead of
// O(N M S): 4096^2 cells in ~50 us instead of 198 ms, same values to <= 1e-15.
// ---------------------------------------------------------------------------
#define GSS_ROWS 32
__global__ void __launch_bounds__(256) grid_logjoint_ss_kernel(
    const NrStats* __restrict__ stp, const double* __restrict__ mu,
    const double* __restrict__ sigma, int M, int S, const double* __restrict__ lp_mu,
    const double* __restrict__ lp_sigma, double* __restrict__ out) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  const NrStats st = *stp;
  // per-column terms once, then GSS_ROWS cells of the column (log and the reciprocal are
  // the expensive part of a cell)
  const double sg = sigma[s], isg = 1.0 / sg;
  const double colc = st.N * (PBX_LOG_SQRT_2PI + log(sg)), lps = lp_sigma[s];
  const int m1 = min(M, (int)(blockIdx.y + 1) * GSS_ROWS);
  for (int m = blockIdx.y * GSS_ROWS; m < m1; ++m) {
    const double a = mu[m] - st.cy;
    double ssq = fma(st.N * a, a, st.RSS);
    ssq = fma(-2.0 * a, st.Se, ssq);
    const double acc = (ssq * isg) * isg;
    const double ll = -acc * 0.5 - colc;
    __stcs(out + (int64_t)m * S + s, (lp_mu[m] + lps) + ll);
  }
}

extern "C" int pbx_grid_norm_logjoint_ss(pbx_ctx* ctx, const double* x_obs, int64_t n_obs,
                                         const double* mu, int32_t n_mu, const double* sigma,
                                         int32_t n_sigma, const double* logprior_mu,
                                         const double* logprior_sigma, double* out) {
  PBX_REQUIRE(ctx && x_obs && mu && sigma && logprior_mu && logprior_sigma && out,
              "pbx_grid_norm_logjoint_ss: null argument");
  PBX_REQUIRE(n_obs >= 1 && n_mu >= 1 && n_sigma >= 1,
              "pbx_grid_norm_logjoint_ss: sizes must be positive");
  PBX_REQUIRE(n_mu <= 65535, "pbx_grid_norm_logjoint_ss: at most 65535 mu rows per call (slab it)");
  PBX_CUDA(cudaSetDevice(ctx->device));
  PBX_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
  NrStats* st = nullptr;
  int rc = pbx_ss_compute(ctx, nullptr, x_obs, n_obs, &st);
  if (rc) return rc;
  dim3 grid((n_sigma + 255) / 256, (n_mu + GSS_ROWS - 1) / GSS_ROWS);
  grid_logjoint_ss_kernel<<<grid, 256, 0, ctx->stream>>>(st, mu, sigma, n_mu, n_sigma,
                                                         logprior_mu, logprior_sigma, out);
  PBX_LAUNCH_CHECK(ctx);
  PBX_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
  return PBX_OK;
}

// ---------------------------------------------------------------------------
// K4 in two passes over the grid.
//
// Pass A  pbx_grid_max_sumexp: ONE read.  Every thread keeps an online (max, sum-exp)
//         pair: per chunk of 8 entries held in registers, the running maximum is raised
//         first (one rescaling table-exp per chunk, branch-free), then the
//         8 terms exp(v - max) are added.  Pairs are merged (m, s) + (m', s') =
//         (M = max, s exp(m - M) + s' exp(m' - M)) by shuffles and shared memory in a
//         fixed order; the last CTA to finish (ticket) merges the per-CTA pairs in index
//         order.  The result differs from sum exp(v - global max) only by the rounding of
//         the rescaling factors (~1e-16 relative).  Linear-pscale input: plain sum.
// Pass B  pbx_grid_posterior2: one read + one write (or in place), both marginals from
//         the same pass, their clamped logs fused into the finishing kernel.
// ---------------------------------------------------------------------------
// Table-driven exp for the two passes (libm's exp costs ~70 SASS instructions and made pass
// A instruction-bound at 2.2 TB/s): exp(x) = 2^(n/64) 2^k e^r, |r| <= ln2/128, one 8-byte
// table entry + a degree-5 polynomial, <= 2 ulp on [-700, 700] (libm outside: a rare branch).
// The 64-entry table is stored 16 times interleaved (entry j of copy g at 16 j + g) and lane
// l reads copy l % 16, so the per-lane lookups never collide in a shared-memory bank; each
// CTA stages the 8 KB into shared memory.
static __device__ double g_exptab[64 * 16];
// (constants live in the constant bank: FP64 instructions take no 64-bit immediates, and a
// literal costs two MOVs at every use)
__constant__ double kGE[12] = {92.332482616893656877,     // 0: 64 / ln2
                               6755399441055744.0,        // 1: 1.5 * 2^52
                               -0.01083042469326756,      // 2: -ln2/64 hi (32 bits)
                               -2.9815858269852933e-12,   // 3: -ln2/64 lo
                               1.0 / 120.0, 1.0 / 24.0, 1.0 / 6.0, 0.5,   // 4..7
                               -600.0, 100.0, -700.0,     // 8..10
                               3.7200759760208361e-44};   // 11: exp(-100)
// Clamps and range selection are done on the HIGH WORD of the double with integer
// instructions (there is no double min/max instruction:
// fmax/fmin compile to DSETP + 2 FSEL each, and a first version whose clamp + select logic was
// written with them came to more instructions than the exponential itself -- 89 SASS
// instructions per grid cell in the posterior pass, issue-bound at 1.6 TB/s).
//   * for a negative double the unsigned high word grows with the magnitude, so
//     min_u(hi, hi(-L)) clamps x at (just below) -L in ONE instruction and leaves
//     non-negative x alone;
//   * the binary exponent k = n >> 6 of the result is known as an integer before the result
//     is assembled, so the subnormal range is handled by adding 200 to k and multiplying by
//     2^-200 (folded into the normaliser) -- one correctly rounded multiply, as before.
__device__ __forceinline__ double grid_clamp_neg(double x, unsigned hi_limit) {
  return __hiloint2double((int)min((unsigned)__double2hiint(x), hi_limit), __double2loint(x));
}
// mantissa part y = 2^((n & 63)/64) e^r in [1, 2) and n = round(64 x / ln2)
__device__ __forceinline__ double grid_exp_core(double x, const double* tab, int& n) {
  const double fn = fma(x, kGE[0], kGE[1]);
  n = __double2loint(fn);
  const double k = fn - kGE[1];
  double r = fma(k, kGE[2], x);                        // k * hi is exact
  r = fma(k, kGE[3], r);
  double p = fma(r, kGE[4], kGE[5]);
  p = fma(r, p, kGE[6]);
  p = fma(r, p, kGE[7]);
  p = fma(r * r, p, r);                                                    // expm1(r)
  const double tj = tab[((n & 63) << 4) | (threadIdx.x & 15)];
  return fma(tj, p, tj);
}
// exp(x) for x <= 0 (or NaN -> garbage the caller masks), clamped at x = -700: for the
// sum-exp pass, where a term below 1e-304 of a sum >= 1 changes no bit
__device__ __forceinline__ double grid_exp_nonpos(double x, const double* tab) {
  int n;
  const double y = grid_exp_core(grid_clamp_neg(x, 0xC085E000u), tab, n);   // -700 = 0xC085E000..
  return __hiloint2double(__double2hiint(y) + ((n >> 6) << 20), __double2loint(y));
}
// exp_logp(l) * scale over the whole double range, branch-free: scale_lo2 = scale * 2^-200
// (both finite and normal for any realistic normaliser).  l > log(huge) and NaN -> huge * scale.
__device__ __forceinline__ double grid_exp_logp_scaled(double l, const double* tab, double scale,
                                                       double scale_lo2) {
  int n;
  const double y = grid_exp_core(grid_clamp_neg(l, 0xC0890000u), tab, n);   // -800
  int k = n >> 6;
  const bool low = k < -1000;
  k = low ? k + 200 : k;
  const double sc = low ? scale_lo2 : scale;
  const double v = __hiloint2double(__double2hiint(y) + (k << 20), __double2loint(y)) * sc;
  return (l <= PBX_LOG_HUGE) ? v : PBX_HUGE * scale;
}
__device__ __forceinline__ void grid_stage_exptab(double* s_tab, int nthreads) {
  for (int i = threadIdx.x; i < 64 * 16; i += nthreads) s_tab[i] = g_exptab[i];
  __syncthreads();
}
static int grid_init_exptab(pbx_ctx* ctx) {
  if (ctx->exptab_ready) return PBX_OK;
  double* h = new double[64 * 16];
  for (int j = 0; j < 64; ++j)
    for (int g = 0; g < 16; ++g) h[16 * j + g] = (double)exp2l(j / 64.0L);
  cudaError_t e = cudaMemcpyToSymbolAsync(g_exptab, h, sizeof(double) * 64 * 16, 0,
                                          cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  delete[] h;
  PBX_CUDA(e);
  ctx->exptab_ready = true;
  return PBX_OK;
}

struct MsPair { double m, s; };
// (m, s) + (m', s') = (M = max(m, m'), s exp(m - M) + s' exp(m' - M)); an empty pair is
// (-1.797e308, 0): its factor is clamped at exp(-700) and multiplies a zero, so no infinities
// or NaNs arise and the merge is branch-free (table exp, ~45 instructions)
__device__ __forceinline__ MsPair ms_merge(MsPair a, MsPair b, const double* tab) {
  const double M = (a.m > b.m) ? a.m : b.m;
  MsPair r;
  r.m = M;
  r.s = fma(a.s, grid_exp_nonpos(a.m - M, tab), b.s * grid_exp_nonpos(b.m - M, tab));
  return r;
}

#define MS_THREADS 256
#define MS_WARPS (MS_THREADS / 32)
#ifndef MS_CHUNK
#define MS_CHUNK 16           // entries per lane and turn (measured: 4 / 8 / 16 -> 47.8 / 39.9 / 38.0 us)
#endif
// Persistent grid (as many CTAs as are resident at once, each warp takes the 256-entry warp
// chunks w, w + n_warps, ...), the next chunk's four 128-bit loads issued before the current
// chunk is folded.  Per chunk a lane raises its running maximum and rescales its sum by
// exp(m_old - m_new) UNCONDITIONALLY: a lane sees a few dozen entries only, so "rescale only
// when the maximum moves" was a divergent branch taken by 85 % of the warp-chunks (with a libm
// exp behind it) -- 58 SASS instructions per entry, issue-bound at 2.6 TB/s.
template <bool kLinear>
__global__ void __launch_bounds__(MS_THREADS)
    grid_max_sumexp_kernel(const double* __restrict__ v, int64_t n, MsPair* __restrict__ partial,
                           unsigned int* __restrict__ ticket, double* __restrict__ out2) {
  __shared__ double s_tab[64 * 16];
  if (!kLinear) grid_stage_exptab(s_tab, MS_THREADS);
  double m = -PBX_HUGE, s = 0.0;
  // a warp owns 32 * MS_CHUNK consecutive entries per turn: load i of lane l is the double2 at
  // 32 i + l of the block, so every 128-bit load instruction is one fully used 512-byte
  // segment (a per-thread run of 64 bytes leaves half of each sector to the next load)
  constexpr int WCH = 32 * MS_CHUNK;
  const int64_t nwch = n / WCH;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t wstride = (int64_t)gridDim.x * MS_WARPS;
  const bool vec = (((uintptr_t)v) & 15) == 0;
  auto fold = [&](const double (&e)[MS_CHUNK], unsigned mask) {      // bit i: slot i holds an entry
    if (kLinear) {
#pragma unroll
      for (int i = 0; i < MS_CHUNK; ++i) s += ((mask >> i) & 1u) ? e[i] : 0.0;
    } else {
      double cm = m;
#pragma unroll
      for (int i = 0; i < MS_CHUNK; ++i) {
        const double ei = ((mask >> i) & 1u) ? e[i] : -PBX_HUGE;
        cm = (ei > cm) ? ei : cm;
      }
      const double f = grid_exp_nonpos(m - cm, s_tab);
      m = cm;
      double t0 = 0.0, t1 = 0.0;
#pragma unroll
      for (int i = 0; i < MS_CHUNK; i += 2) {
        // e - m <= 0 here; below -700 a term is < 1e-304 of a sum that is >= 1 (the maximum
        // contributes exp(0)): clamping the argument (one integer min on the high word)
        // changes no bit of the result
        t0 += ((mask >> i) & 1u) ? grid_exp_nonpos(e[i] - m, s_tab) : 0.0;
        t1 += ((mask >> (i + 1)) & 1u) ? grid_exp_nonpos(e[i + 1] - m, s_tab) : 0.0;
      }
      s = fma(s, f, t0 + t1);
    }
  };
  auto load = [&](double (&e)[MS_CHUNK], int64_t wc) {
    const double* base = v + wc * WCH;
    if (vec) {
      const double2* v2 = reinterpret_cast<const double2*>(base);
#pragma unroll
      for (int i = 0; i < MS_CHUNK / 2; ++i) {
        const double2 t = __ldcs(v2 + 32 * i + lane);
        e[2 * i] = t.x;
        e[2 * i + 1] = t.y;
      }
    } else {
#pragma unroll
      for (int i = 0; i < MS_CHUNK; ++i) e[i] = base[32 * i + lane];
    }
  };
  {
    int64_t wc = (int64_t)blockIdx.x * MS_WARPS + warp;
    double e[MS_CHUNK], en[MS_CHUNK];
    if (wc < nwch) load(en, wc);
    for (; wc < nwch; wc += wstride) {
#pragma unroll
      for (int i = 0; i < MS_CHUNK; ++i) e[i] = en[i];
      if (wc + wstride < nwch) load(en, wc + wstride);
      fold(e, (1u << MS_CHUNK) - 1u);
    }
  }
  if (blockIdx.x == 0 && threadIdx.x < 32) {               // the n % 256 tail: one warp
    double e[MS_CHUNK];
    unsigned mask = 0;
#pragma unroll
    for (int i = 0; i < MS_CHUNK; ++i) {
      const int64_t idx = nwch * WCH + 32 * i + lane;
      e[i] = (idx < n) ? v[idx] : 0.0;
      mask |= (idx < n) ? (1u << i) : 0u;
    }
    if (mask) fold(e, mask);
  }
  // fixed merge tree: lanes (butterfly: both lanes of a pair get the same bits), the CTA's
  // warps (warp 0), then the CTAs' pairs by the last CTA to finish (ticket) -- deterministic
  // for a given grid size
  MsPair p;
  p.m = kLinear ? 0.0 : m;
  p.s = s;
  auto warp_merge = [&](MsPair a, int from) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      if (o > from) continue;
      MsPair q;
      q.m = __shfl_xor_sync(0xffffffffu, a.m, o);
      q.s = __shfl_xor_sync(0xffffffffu, a.s, o);
      if (kLinear) a.s += q.s;
      else a = ms_merge(a, q, s_tab);
    }
    return a;
  };
  p = warp_merge(p, 16);
  __shared__ MsPair sh[MS_WARPS];
  __shared__ bool last;
  if (lane == 0) sh[warp] = p;
  __syncthreads();
  if (warp == 0) {
    MsPair a = sh[lane & (MS_WARPS - 1)];
    a = warp_merge(a, MS_WARPS / 2);
    if (lane == 0) {
      partial[blockIdx.x] = a;
      __threadfence();
      last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
  }
  __syncthreads();
  if (last) {
    __threadfence();
    const volatile MsPair* pv = partial;
    MsPair a;
    a.m = kLinear ? 0.0 : -PBX_HUGE;
    a.s = 0.0;
    for (unsigned i = threadIdx.x; i < gridDim.x; i += MS_THREADS) {
      MsPair b;
      b.m = pv[i].m;
      b.s = pv[i].s;
      if (kLinear) a.s += b.s;
      else a = ms_merge(a, b, s_tab);
    }
    a = warp_merge(a, 16);
    __syncthreads();                                       // sh[] is free again
    if (lane == 0) sh[warp] = a;
    __syncthreads();
    if (warp == 0) {
      MsPair t = sh[lane & (MS_WARPS - 1)];
      t = warp_merge(t, MS_WARPS / 2);
      if (lane == 0) {
        out2[0] = t.m;
        out2[1] = t.s;
        *ticket = 0;                                       // ready for the next call
      }
    }
  }
}

__global__ void grid_rescale_sumexp_kernel(const double* lmax, const double* gmax, double* sum) {
  sum[0] = (sum[0] == 0.0) ? 0.0 : sum[0] * exp(lmax[0] - gmax[0]);
}

#define P2_CPT 4                        // columns per thread (two 128-bit accesses per row)
#define P2_THREADS 256
#define P2_WARPS (P2_THREADS / 32)
#define P2_COLS (P2_THREADS * P2_CPT)
#ifndef P2_RU
#define P2_RU 4                         // rows per tile = rows in flight per thread
#endif

// kLinear: the input (and the output) are linear-pscale probabilities: post = p / max(tiny,
// sum) (pd.py:285-295 without the log/exp round trip), marginals = plain sums.
//
// Persistent grid: CTA b owns the column block b % n_colblocks (P2_COLS columns: a warp covers
// 128 consecutive columns; thread (warp w, lane l) owns the two column PAIRS at cb + 2 l and
// cb + 64 + 2 l, so each of its two 128-bit accesses per row is, warp-wide, one contiguous
// 512-byte segment) and the 4-row tiles b / n_colblocks, + n_rowctas, + 2 n_rowctas ... of it:
// with 3 CTAs per SM and 4-row tiles the last round of tiles is a few % of the work whatever M
// (32-row tiles on a (4, 128) grid left 14 % of the CTA slots idle at 4096 x 4096).  Column
// sums stay in registers for the whole kernel; each warp writes its own partial row sums
// (no shared memory, no __syncthreads in the loop).
// kFull: every tile is interior and 16-byte aligned -- no bounds predicates in the loop.
template <bool kLinear, bool kFull>
__global__ void __launch_bounds__(P2_THREADS)
    grid_posterior2_kernel(const double* lj, int M, int S, const double* __restrict__ gmax,
                           const double* __restrict__ gsum, double* post,
                           double* __restrict__ row_partial, double* __restrict__ col_partial,
                           int n_colblocks, int n_rowctas, double qmin) {
  __shared__ double s_tab[64 * 16];
  if (!kLinear) {
    grid_stage_exptab(s_tab, P2_THREADS);
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int cblk = blockIdx.x % n_colblocks, rcta = blockIdx.x / n_colblocks;
  const int cb = cblk * P2_COLS + warp * 128 + 2 * lane;
  const double mx = kLinear ? 0.0 : gmax[0];
  const double den = fmax(PBX_TINY, gsum[0]);
  const double lden = kLinear ? 0.0 : log(den);
  const double rden = 1.0 / den;
  const double rden_lo2 = rden * 6.223015277861142e-61;            // 2^-200
  // 128-bit path: even row length, 16-byte aligned bases
  const bool vec = kFull || ((S % 2 == 0) && ((((uintptr_t)lj) & 15) == 0) &&
                             (post == nullptr || (((uintptr_t)post) & 15) == 0));
  int colidx[P2_CPT];
  colidx[0] = cb; colidx[1] = cb + 1; colidx[2] = cb + 64; colidx[3] = cb + 65;
  double col[P2_CPT];
#pragma unroll
  for (int k = 0; k < P2_CPT; ++k) col[k] = 0.0;
  const int rp_stride = n_colblocks * P2_WARPS;
  for (int m0 = rcta * P2_RU; m0 < M; m0 += n_rowctas * P2_RU) {
    double e[P2_RU][P2_CPT];
    // all loads of the tile first (post may alias lj: the compiler cannot hoist them)
#pragma unroll
    for (int u = 0; u < P2_RU; ++u) {
      const int m = m0 + u;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int c0 = colidx[2 * h];
        if (kFull || (m < M && vec && c0 + 1 < S)) {
          const double2 a = __ldcs(reinterpret_cast<const double2*>(lj + (int64_t)m * S + c0));
          e[u][2 * h] = a.x;
          e[u][2 * h + 1] = a.y;
        } else {
#pragma unroll
          for (int k = 0; k < 2; ++k)
            e[u][2 * h + k] = (m < M && c0 + k < S) ? lj[(int64_t)m * S + c0 + k]
                                                    : (kLinear ? 0.0 : -PBX_HUGE);
        }
      }
    }
    double w[P2_RU];
#pragma unroll
    for (int u = 0; u < P2_RU; ++u) {
      const int m = m0 + u;
      double q[P2_CPT], o[P2_CPT];
#pragma unroll
      for (int k = 0; k < P2_CPT; ++k) {
        if (kLinear) {
          // reference: div_prob(p, sum) = p / max(tiny, sum)
          q[k] = e[u][k] / den;
          o[k] = q[k];
        } else {
          // reference: q = exp_logp(lj - max) / max(tiny, sum); post = log_prob(q); the
          // marginal term is exp_logp(post).  log(q) is evaluated as (lj - max) - log(den)
          // and exp(log q) as q itself: the same values to ~1e-16 relative for a third of
          // the transcendental work; the clamp decision (q < tiny -> -1.797e308) is the
          // reference's, taken on q.
          // (qmin = tiny; 0 for PD.marginalise, which sums exp_logp(p) unclamped)
          const double sh = e[u][k] - mx;
          const double qq = grid_exp_logp_scaled(sh, s_tab, rden, rden_lo2);
          const bool keep = qq >= qmin;
          o[k] = keep ? sh - lden : -PBX_HUGE;
          q[k] = keep ? qq : 0.0;                           // exp_logp(-1.797e308) = 0
        }
        if (!kFull && !(m < M && colidx[k] < S)) q[k] = 0.0;
        col[k] += q[k];
      }
      if (post && (kFull || m < M)) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int c0 = colidx[2 * h];
          if (kFull || (vec && c0 + 1 < S)) {
            __stcs(reinterpret_cast<double2*>(post + (int64_t)m * S + c0),
                   make_double2(o[2 * h], o[2 * h + 1]));
          } else {
#pragma unroll
            for (int k = 0; k < 2; ++k)
              if (c0 + k < S) post[(int64_t)m * S + c0 + k] = o[2 * h + k];
          }
        }
      }
      w[u] = (q[0] + q[1]) + (q[2] + q[3]);
    }
    // the row sums of the warp's 128 columns: fold the rows onto lane groups first (4 rows:
    // lanes 16+ keep rows 2, 3; then bit 3 picks the odd row -- 6 exchanges instead of 20),
    // then a butterfly inside each group.  Row u ends up in lane (32 / P2_RU) u.
    {
      const bool up = (lane & 16) != 0;
#if P2_RU == 4
      double k0 = up ? w[2] : w[0], k1 = up ? w[3] : w[1];
      const double a0 = up ? w[0] : w[2], a1 = up ? w[1] : w[3];
      k0 += __shfl_xor_sync(0xffffffffu, a0, 16);
      k1 += __shfl_xor_sync(0xffffffffu, a1, 16);
      const bool up2 = (lane & 8) != 0;
      double kk = up2 ? k1 : k0;
      const double ss = up2 ? k0 : k1;
      kk += __shfl_xor_sync(0xffffffffu, ss, 8);
#elif P2_RU == 2
      double kk = up ? w[1] : w[0];
      const double ss = up ? w[0] : w[1];
      kk += __shfl_xor_sync(0xffffffffu, ss, 16);
      kk += __shfl_xor_sync(0xffffffffu, kk, 8);
#else
#error "P2_RU must be 2 or 4"
#endif
      kk += __shfl_xor_sync(0xffffffffu, kk, 4);
      kk += __shfl_xor_sync(0xffffffffu, kk, 2);
      kk += __shfl_xor_sync(0xffffffffu, kk, 1);
      const int m = m0 + lane / (32 / P2_RU);
      if ((lane & (32 / P2_RU - 1)) == 0 && (kFull || m < M))
        row_partial[(int64_t)m * rp_stride + cblk * P2_WARPS + warp] = kk;
    }
  }
#pragma unroll
  for (int k = 0; k < P2_CPT; ++k)
    if (kFull || colidx[k] < S) col_partial[(int64_t)rcta * S + colidx[k]] = col[k];
}

// log_flags: bit 0 -> marg_mu through the clamped log, bit 1 -> marg_sigma
// blocks [0, row_blocks): a warp per row, the lanes stride over the row's partial sums
// (contiguous) and finish with a butterfly; blocks from row_blocks on: 32 columns x 8 partial
// groups per block (coalesced across the columns), the 8 group sums added in order.  Fixed
// association -> identical bits from run to run.
__global__ void __launch_bounds__(256)
    grid_marginal_finish2(const double* __restrict__ row_partial, int M, int n_per_row,
                          const double* __restrict__ col_partial, int n_rowctas, int S,
                          double* __restrict__ marg_mu, double* __restrict__ marg_sigma,
                          int log_flags, int row_blocks) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if ((int)blockIdx.x < row_blocks) {
    const int i = blockIdx.x * 8 + warp;
    if (i >= M) return;
    double w = 0.0;
    for (int k = lane; k < n_per_row; k += 32) w += row_partial[(int64_t)i * n_per_row + k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) w += __shfl_xor_sync(0xffffffffu, w, o);
    if (lane == 0) marg_mu[i] = (log_flags & 1) ? pbx_log_prob(w) : w;
    return;
  }
  __shared__ double s_w[8][33];
  const int i = (blockIdx.x - row_blocks) * 32 + lane;
  double w0 = 0.0, w1 = 0.0;
  if (i < S) {
    int k = warp;
    for (; k + 8 < n_rowctas; k += 16) {
      w0 += col_partial[(int64_t)k * S + i];
      w1 += col_partial[(int64_t)(k + 8) * S + i];
    }
    if (k < n_rowctas) w0 += col_partial[(int64_t)k * S + i];
  }
  s_w[warp][lane] = w0 + w1;
  __syncthreads();
  if (warp == 0 && i < S) {
    double w = s_w[0][lane];
#pragma unroll
    for (int g = 1; g < 8; ++g) w += s_w[g][lane];
    marg_sigma[i] = (log_flags & 2) ? pbx_log_prob(w) : w;
  }
}

extern "C" int pbx_grid_max_sumexp(pbx_ctx* ctx, const double* v, int64_t n, int32_t linear,
                                   double* out2) {
  PBX_REQUIRE(ctx && v && out2 && n >= 1, "pbx_grid_max_sumexp: bad argument");
  PBX_CUDA(cudaSetDevice(ctx->device));
  {
    int rc0 = grid_init_exptab(ctx);
    if (rc0) return rc0;
  }
  int per_sm = 0;
  PBX_CUDA(linear ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(
                        &per_sm, grid_max_sumexp_kernel<true>, MS_THREADS, 0)
                  : cudaOccupancyMaxActiveBlocksPerMultiprocessor(
                        &per_sm, grid_max_sumexp_kernel<false>, MS_THREADS, 0));
  if (per_sm < 1) per_sm = 1;
  const int64_t cap = (int64_t)ctx->sm_count * per_sm;     // one resident wave
  int64_t want = (n + (int64_t)MS_THREADS * MS_CHUNK * 2 - 1) / ((int64_t)MS_THREADS * MS_CHUNK * 2);
  const int np = (int)(want < 1 ? 1 : (want > cap ? cap : want));
  // the ticket word is the context's own (zeroed once; the last CTA of every call resets it),
  // the per-CTA pairs go to the shared workspace
  if (!ctx->ticket) {
    PBX_CUDA(cudaMalloc(&ctx->ticket, 256));
    PBX_CUDA(cudaMemsetAsync(ctx->ticket, 0, 256, ctx->stream));
  }
  int rc = pbx_ws_reserve(ctx, (size_t)np * sizeof(MsPair));
  if (rc) return rc;
  unsigned int* ticket = ctx->ticket;
  MsPair* partial = (MsPair*)ctx->ws;
  PBX_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
  if (linear)
    grid_max_sumexp_kernel<true><<<np, MS_THREADS, 0, ctx->stream>>>(v, n, partial, ticket, out2);
  else
    grid_max_sumexp_kernel<false><<<np, MS_THREADS, 0, ctx->stream>>>(v, n, partial, ticket, out2);
  PBX_LAUNCH_CHECK(ctx);
  PBX_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
  return PBX_OK;
}

extern "C" int pbx_grid_rescale_sumexp(pbx_ctx* ctx, const double* local_max,
                                       const double* global_max, double* sum_inout) {
  PBX_REQUIRE(ctx && local_max && global_max && sum_inout, "pbx_grid_rescale_sumexp: null argument");
  PBX_CUDA(cudaSetDevice(ctx->device));
  grid_rescale_sumexp_kernel<<<1, 1, 0, ctx->stream>>>(local_max, global_max, sum_inout);
  PBX_LAUNCH_CHECK(ctx);
  return PBX_OK;
}

extern "C" int pbx_grid_posterior2(pbx_ctx* ctx, const double* prob, int32_t n_mu, int32_t n_sigma,
                                   const double* gmax, const double* gsum, int32_t linear,
                                   double* post, double* marg_mu, double* marg_sigma,
                                   int32_t marg_log_flags) {
  PBX_REQUIRE(ctx && prob && gsum && (linear || gmax), "pbx_grid_posterior2: null argument");
  PBX_REQUIRE(n_mu >= 1 && n_sigma >= 1, "pbx_grid_posterior2: sizes must be positive");
  PBX_CUDA(cudaSetDevice(ctx->device));
  {
    int rc0 = grid_init_exptab(ctx);
    if (rc0) return rc0;
  }
  const int ncb = (n_sigma + P2_COLS - 1) / P2_COLS;
  const int n_tiles = (n_mu + P2_RU - 1) / P2_RU;
  const bool full = (n_mu % P2_RU == 0) && (n_sigma % P2_COLS == 0) &&
                    ((((uintptr_t)prob) & 15) == 0) && (!post || (((uintptr_t)post) & 15) == 0);
  // persistent grid: as many CTAs as are resident at once (3 per SM for the interior variant
  // at 78 registers; capping at 64 registers for 4 spills), a whole number of row-CTAs per
  // column block
  int per_sm = 0;
  {
    cudaError_t oe;
    if (linear)
      oe = full ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(
                      &per_sm, grid_posterior2_kernel<true, true>, P2_THREADS, 0)
                : cudaOccupancyMaxActiveBlocksPerMultiprocessor(
                      &per_sm, grid_posterior2_kernel<true, false>, P2_THREADS, 0);
    else
      oe = full ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(
                      &per_sm, grid_posterior2_kernel<false, true>, P2_THREADS, 0)
                : cudaOccupancyMaxActiveBlocksPerMultiprocessor(
                      &per_sm, grid_posterior2_kernel<false, false>, P2_THREADS, 0);
    PBX_CUDA(oe);
    if (per_sm < 1) per_sm = 1;
  }
  int nrc = (per_sm * ctx->sm_count) / ncb;
  if (nrc < 1) nrc = 1;
  if (nrc > n_tiles) nrc = n_tiles;
  const int npr = ncb * P2_WARPS;                       // partial sums per row
  const size_t rp = ((size_t)n_mu * npr * 8 + 255) / 256 * 256;
  const size_t cp = (size_t)nrc * n_sigma * 8;
  int rc = pbx_ws_reserve(ctx, rp + cp);
  if (rc) return rc;
  double* row_partial = (double*)ctx->ws;
  double* col_partial = (double*)((char*)ctx->ws + rp);
  PBX_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
  const double qmin = (marg_log_flags & 4) ? 0.0 : PBX_TINY;
#define P2_LAUNCH(L, F)                                                                        \
  grid_posterior2_kernel<L, F><<<ncb * nrc, P2_THREADS, 0, ctx->stream>>>(                     \
      prob, n_mu, n_sigma, gmax, gsum, post, row_partial, col_partial, ncb, nrc, qmin)
  if (linear) {
    if (full) P2_LAUNCH(true, true); else P2_LAUNCH(true, false);
  } else {
    if (full) P2_LAUNCH(false, true); else P2_LAUNCH(false, false);
  }
#undef P2_LAUNCH
  PBX_LAUNCH_CHECK(ctx);
  if (marg_mu || marg_sigma) {
    const int rb = marg_mu ? (n_mu + 7) / 8 : 0, cbk = marg_sigma ? (n_sigma + 31) / 32 : 0;
    grid_marginal_finish2<<<rb + cbk, 256, 0, ctx->stream>>>(
        row_partial, n_mu, npr, col_partial, nrc, n_sigma, marg_mu, marg_sigma, marg_log_flags,
        rb);
    PBX_LAUNCH_CHECK(ctx);
  }
  PBX_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
  return PBX_OK;
}
