// pbx_mh_mvn.cu -- K1: batched-chain Metropolis-Hastings on a multivariate-normal
// target.  Restates (per chain) the reference step loop probayes/sp.py:221-258 with
// the accept rule of sp_utils.py:19-37 / pscales.py:219-236 and the scipy mvn
// density the reference calls at prob.py:347-360.
//
// Layout: state[D][C], outputs [..][D][C] / [..][C] -- chain-minor so a warp of 32
// chains reads/writes 256 contiguous bytes per dimension.
//
// Three kernels, one draw per (step, chain) and the same arithmetic on the state:
//  * mh_mvn_kernel     one thread = one chain, state + running sums in registers,
//                      Philox4x32-10 + Box-Muller in-thread or INJECTED streams (the
//                      bit-parity path), per-step accept/score outputs, bound=True.
//  * mh_mvn_ws_kernel  warp-specialised native-RNG path (reference rule, D >= 5,
//                      kernel_variant 2).  A CTA owns 32 chains: 12 (D <= 3) or 9 producer
//                      warps draw Philox blocks and turn them into proposal deltas and
//                      log-thresholds for batches of steps (that work does not depend on
//                      the chain state, so it parallelises over steps), hand them through
//                      a shared-memory ring guarded
//                      by mbarriers to ONE consumer warp that runs the inherently
//                      sequential part (propose, 2-D quadratic form, accept, record)
//                      for its 32 chains.  This takes a 4096-chain walk from one
//                      latency-bound warp per SM to ~16 busy warps per SM.
//  * mh_mvn_wd_kernel  whitened decisions (native RNG, log rule, D <= 4): the default.  The
//                      producers also whiten the deltas, so the decision warp's step is one
//                      D-term dot product and a compare (see the comment at the kernel).
// All three record bit-identical trajectories and densities for the same seed; the
// whitened decisions can differ only within the rounding of the tracked whitened state.
#include <math.h>
#include "pbx_common.cuh"

// ---------------------------------------------------------------------------
// Table-driven double-precision log / sincos(2 pi u) / exp for the RNG path.
// CUDA's libm versions cost ~75 / ~95 / ~45 SASS instructions each, a third of them
// constant materialisation (FP64 ops take no 64-bit immediates).  Here: one 16-byte
// table lookup + a short polynomial whose coefficients are constant-bank operands.
// Absolute error <= ~3e-16 (pinned by pbx_selftest_fastmath in the tests: <= 2 ulp of
// max(1, |value|), sin/cos <= 4e-16 against an extended-precision reference); inputs
// are the RNG's uniforms, so no special-case handling is needed.
// ---------------------------------------------------------------------------
// Shared-memory bank conflicts: a 128-bit shared load is served a quarter-warp (8 lanes) at
// a time, each lane touching one of the 8 sixteen-byte bank groups; with per-lane random
// table indices ~2.7 lanes collide per quarter and a lookup costs ~11 wavefronts instead of
// 4 (measured: 36 % of the kernel's shared-memory wavefronts were conflicts, and that pipe,
// not the FP64 pipe, was the busiest unit).  So every table is stored 8 (16 for the 8-byte
// exp table) times, interleaved, and lane l reads copy l % 8: entry j of copy g sits at
// index 8 j + g, i.e. always in bank group g -- conflict-free for any index pattern.  To
// keep the footprint the tables have 128 entries (polynomials two terms longer).
struct PbxTables {
  double2 lg[128 * 8];   // (1/c_j, -2 log c_j),         c_j = 1 + (j + 0.5)/128
  double2 sc[128 * 8];   // (cos, sin) of 2 pi (k + 0.5)/128
  double ex[64 * 16];    // 2^(j/64)
};
static __device__ PbxTables g_tables;
__constant__ double kSinP[3] = {-1.0 / 6.0, 1.0 / 120.0, -1.0 / 5040.0};
__constant__ double kCosP[3] = {-0.5, 1.0 / 24.0, -1.0 / 720.0};
__constant__ double kExpP[4] = {0.5, 1.0 / 6.0, 1.0 / 24.0, 1.0 / 120.0};

// -2 log(x) for positive normal x (what both Box-Muller and the accept threshold need):
// the same reduction with the factor -2 folded into the table value, the polynomial
// and the exponent term -- one multiply less than scaling a plain log afterwards
__constant__ double kN2LogP[5] = {1.0, -2.0 / 3.0, 0.5, -0.4, 1.0 / 3.0};
__device__ __forceinline__ double fast_neg2log(double x, const PbxTables* tb) {
  const int hi = __double2hiint(x), lo = __double2loint(x);
  const int e = (hi >> 20) - 1023;
  const double m = __hiloint2double((hi & 0x000FFFFF) | 0x3FF00000, lo);   // [1, 2)
  const double2 t = tb->lg[((hi >> 10) & 0x3F8) | (threadIdx.x & 7)];
  const double r = fma(m, t.x, -1.0);                                      // |r| < 2^-8
  // -2 log1p(r) = -2r + r^2 (1 - 2r/3 + r^2/2 - 2r^3/5 + r^4/3 - ...); the next term is
  // (2/7) r^7 < 0.3 * 2^-56
  double p = fma(r, kN2LogP[4], kN2LogP[3]);
  p = fma(r, p, kN2LogP[2]);
  p = fma(r, p, kN2LogP[1]);
  p = fma(r, p, kN2LogP[0]);
  p = fma(r * r, p, t.y);                        // -2 log c + r^2 (1 - 2r/3 + ...)
  p = fma(r, -2.0, p);                           // ... - 2r  = -2 log(c (1 + r))
  const double ed = __hiloint2double(0x43300000, e ^ (int)0x80000000) - 4503601774854144.0;
  return fma(ed, -1.386294361119890618835, p);   // -2 ln 2
}

// (sin, cos)(2 pi u), u = (w + 0.5) / 2^32
__device__ __forceinline__ void fast_sincos2pi(uint32_t w, const PbxTables* tb, double& s,
                                               double& c) {
  const double2 t = tb->sc[((w >> 22) & 0x3F8) | (threadIdx.x & 7)];
  // rho = 2 pi ((w & 0x1ffffff) + 0.5 - 2^24) / 2^32,  |rho| < pi/128.  The 25 bits go
  // into the mantissa of 2^51 (unit in the last place 1/2) doubled, so that 2^51 + k is
  // exact and one subtraction of 2^51 + 2^24 - 0.5 (representable) centres it
  const double v = __hiloint2double(0x43200000, (int)((w & 0x01FFFFFFu) << 1));
  const double rho = (v - 2251799830462463.5) * 1.4629180792671596e-9;    // 2 pi / 2^32
  const double q = rho * rho;
  // |rho| < 2.46e-2: the dropped terms are rho^9/9! < 1e-20 and rho^8/8! < 4e-18
  const double sr = fma(rho * q, fma(q, fma(q, kSinP[2], kSinP[1]), kSinP[0]), rho);   // sin(rho)
  const double cr = fma(q, fma(q, fma(q, kCosP[2], kCosP[1]), kCosP[0]), 1.0);         // cos(rho)
  c = fma(t.x, cr, -(t.y * sr));
  s = fma(t.y, cr, t.x * sr);
}

// exp(x) for x in [-700, 700]
__device__ __forceinline__ double fast_exp(double x, const PbxTables* tb) {
  const double fn = fma(x, 92.332482616893656877, 6755399441055744.0);     // 64/ln2, 1.5*2^52
  const int n = __double2loint(fn);
  const double k = fn - 6755399441055744.0;
  double r = fma(k, -0.01083042469326756, x);          // ln2/64 hi (32 bits: k*hi exact)
  r = fma(k, -2.9815858269852933e-12, r);              // ln2/64 lo
  double p = fma(r, kExpP[3], kExpP[2]);
  p = fma(r, p, kExpP[1]);
  p = fma(r, p, kExpP[0]);
  p = fma(r * r, p, r);                                                    // expm1(r)
  const double tj = tb->ex[((n & 63) << 4) | (threadIdx.x & 15)];
  const double y = fma(tj, p, tj);
  return __hiloint2double(__double2hiint(y) + ((n >> 6) << 20), __double2loint(y));
}

// sqrt(v) for positive normal v: hardware rsqrt seed (relative error < 2^-22), ONE
// Newton step on 1/sqrt (-> 2^-43) and one correction of the root (-> < 2^-80, i.e.
// the rounding of the last fma decides: faithfully rounded).  Branch-free (libm's
// sqrt carries a special-case branch that stops ptxas from interleaving independent
// steps).
__device__ __forceinline__ double fast_sqrt(double v) {
  double y;                                  // MUFU.RSQ64H
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(v));
  const double hv = 0.5 * v;
  y = y * fma(-hv * y, y, 1.5);
  double s = v * y;
  s = fma(fma(-s, s, v), 0.5 * y, s);
  return s;
}

// linear-pscale output density exp(logpdf): table exp in its safe range, libm beyond
// (out of line: the unrolled writers carry one call site each instead of libm's body)
__device__ __noinline__ double out_exp_slow(double l) { return exp(l); }
__device__ __forceinline__ double out_exp(double l, const PbxTables* tb) {
  return (l > -700.0 && l < 700.0) ? fast_exp(l, tb) : out_exp_slow(l);
}
// Density recorded for a retained state of log-density lp: lp itself under the log pscale,
// else pdf = exp(logpdf) as scipy does -- libm's under the reference rule (bit-equal to the
// linear density that rule decides with), the table exp under the log rule
__device__ __forceinline__ double rec_density(double lp, bool log_pscale, bool ref,
                                              const PbxTables* tb) {
  return log_pscale ? lp : (ref ? exp(lp) : out_exp(lp, tb));
}

// The warp-specialised kernels read the tables from a copy in shared memory, made by all
// kThreads threads of the CTA (the caller synchronises before the first use)
template <int kThreads>
__device__ __forceinline__ void stage_tables(PbxTables& s_tb) {
  const double* src = reinterpret_cast<const double*>(&g_tables);
  double* dst = reinterpret_cast<double*>(&s_tb);
  for (int i = threadIdx.x; i < (int)(sizeof(PbxTables) / sizeof(double)); i += kThreads)
    dst[i] = src[i];
}

static int init_tables(pbx_ctx* ctx) {
  // per context (one per device and process; a context is not thread-safe): no process-wide
  // flags that would go stale after a device reset or race between threads
  if (ctx->tables_ready) return PBX_OK;
  PbxTables* hp = new PbxTables();
  PbxTables& h = *hp;
  for (int j = 0; j < 128; ++j) {
    const long double c = 1.0L + (j + 0.5L) / 128.0L;
    const double inv = (double)(1.0L / c);
    // log c_j must pair with the ROUNDED reciprocal: log(1/inv) keeps r = m*inv - 1 exact
    const double n2l = (double)(2.0L * logl((long double)inv));        // = -2 log c_j
    for (int g = 0; g < 8; ++g) {
      h.lg[8 * j + g].x = inv;
      h.lg[8 * j + g].y = n2l;
    }
  }
  const long double two_pi = 6.283185307179586476925286766559L;
  for (int k = 0; k < 128; ++k) {
    const long double th = two_pi * (k + 0.5L) / 128.0L;
    for (int g = 0; g < 8; ++g) {
      h.sc[8 * k + g].x = (double)cosl(th);
      h.sc[8 * k + g].y = (double)sinl(th);
    }
  }
  for (int j = 0; j < 64; ++j)
    for (int g = 0; g < 16; ++g) h.ex[16 * j + g] = (double)exp2l(j / 64.0L);
  cudaError_t e = cudaMemcpyToSymbolAsync(g_tables, &h, sizeof(h), 0, cudaMemcpyHostToDevice,
                                          ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  delete hp;
  PBX_CUDA(e);
  ctx->tables_ready = true;
  return PBX_OK;
}

struct MhMvnConst {
  double mean[PBX_MAX_DIMS];
  double W[PBX_MAX_DIMS * PBX_MAX_DIMS];
  double L[PBX_MAX_DIMS * PBX_MAX_DIMS];
  double scale[PBX_MAX_DIMS];
  double norm_c;
  double radius;
  pbx_round_keys rk;         // Philox round keys of the walk's seed
  int bound;                 // set_delta(..., bound=True)
  double lims[PBX_MAX_DIMS][2];
  int open_end[PBX_MAX_DIMS][2];
};

struct MhMvnArgs {
  int C, T, thin;
  int64_t step0, chain0;
  uint64_t seed;
  int log_pscale, accept_mode, prop_kind, has_L;
  double* state;
  double* state_lp;
  const double* inj_delta;
  const double* inj_thresh;
  double* out_x;
  double* out_prob;
  uint8_t* out_accept;
  double* out_score;
  int64_t* accept_count;
  double* stat_sum;
  double* stat_sumsq;
  double* out_xprop;
  double* out_pprop;
};

// Whitening y = W^T (v - mean) (dev @ U in scipy's terms), handed to emit(k, y_k) one
// component at a time in dimension order, so that a caller that only sums y_k^2 never holds
// the whole vector (which costs the D = 7 per-thread kernel 21 registers).
// kZeroMean: the target mean is exactly 0 in every dimension; v - 0.0 == v bit for
// bit, so the subtraction is dropped (one FP64 op per dimension off the consumer's
// instruction budget).  A displacement is whitened without the mean: kZeroMean = true.
template <int D, bool kZeroMean, class Emit>
__device__ __forceinline__ void whiten(const double (&v)[D], const MhMvnConst& m, Emit emit) {
  double dev[D];
#pragma unroll
  for (int j = 0; j < D; ++j) dev[j] = kZeroMean ? v[j] : v[j] - m.mean[j];
#pragma unroll
  for (int k = 0; k < D; ++k) {
    double e = 0.0;
#pragma unroll
    for (int j = 0; j < D; ++j) e = fma(dev[j], m.W[j * D + k], e);
    emit(k, e);
  }
}
// scipy multivariate_normal_gen._logpdf: -0.5*(rank*log(2pi) + log_pdet + maha),
// maha = sum(square(dev @ U)).
template <int D, bool kZeroMean = false>
__device__ __forceinline__ double mvn_maha(const double (&x)[D], const MhMvnConst& m) {
  double maha = 0.0;
  whiten<D, kZeroMean>(x, m, [&](int, double y) { maha = fma(y, y, maha); });
  return maha;
}

template <int D, bool kNormalOnly = false>
__device__ __forceinline__ void draw_step(uint64_t seed, uint64_t gstep, uint32_t gchain,
                                          int prop_kind, const MhMvnConst& m,
                                          const PbxTables* tb, double (&dl)[D], double& t) {
  if (kNormalOnly) prop_kind = PBX_PROP_NORMAL;          // compile-time: no kind branches
#pragma unroll
  for (int s = 0; s < (D + 1) / 2; ++s) {
    pbx_u4 w = pbx_philox_rk((uint32_t)gstep, (uint32_t)(gstep >> 32), gchain, (uint32_t)s, m.rk);
    if (s == 0) t = pbx_t44(w.w, w.y);
    double d0, d1;
    if (prop_kind == PBX_PROP_NORMAL) {
      // Box-Muller: r = sqrt(-2 log u52), angle = 2 pi u32
      // (the table log is accurate to ~1e-16 ABSOLUTE: for u within a few ulp of 1 it may
      // return 0 or -1e-16, which the rsqrt-based root would turn into NaN -- clamp)
      const double rad = fast_sqrt(fmax(fast_neg2log(pbx_u52(w.x, w.y), tb), PBX_TINY));
      double sn, cs;
      fast_sincos2pi(w.z, tb, sn, cs);
      d0 = (rad * cs) * m.scale[2 * s];
      d1 = (2 * s + 1 < D) ? (rad * sn) * m.scale[2 * s + 1] : 0.0;
    } else if (prop_kind == PBX_PROP_UNIFORM) {
      double r0 = pbx_u52(w.x, w.y), r1 = pbx_u32(w.z);
      d0 = -m.scale[2 * s] + (2.0 * m.scale[2 * s]) * r0;
      d1 = (2 * s + 1 < D) ? -m.scale[2 * s + 1] + (2.0 * m.scale[2 * s + 1]) * r1 : 0.0;
    } else {                       // spherical: cube sample, rescaled below
      d0 = -m.radius + (2.0 * m.radius) * pbx_u52(w.x, w.y);
      d1 = (2 * s + 1 < D) ? -m.radius + (2.0 * m.radius) * pbx_u32(w.z) : 0.0;
    }
    dl[2 * s] = d0;
    if (2 * s + 1 < D) dl[2 * s + 1] = d1;
  }
  if (prop_kind == PBX_PROP_SPHERICAL) {   // field.py:509-531
    double ss = 0.0;
#pragma unroll
    for (int j = 0; j < D; ++j) ss += dl[j] * dl[j];
    const double nrm = (ss >= PBX_TINY) ? sqrt(ss) : 0.0;
#pragma unroll
    for (int j = 0; j < D; ++j) dl[j] = ((dl[j] * m.radius) / nrm) * m.scale[j];
  }
}

// delta -> proposal displacement (optional Cholesky colouring: rf.py:346-348)
template <int D>
__device__ __forceinline__ void colour_delta(int has_L, const MhMvnConst& m, const double (&dl)[D],
                                             double (&v)[D]) {
  if (has_L) {
#pragma unroll
    for (int i = 0; i < D; ++i) {
      double acc = 0.0;
#pragma unroll
      for (int j = 0; j < D; ++j) acc = fma(m.L[i * D + j], dl[j], acc);
      v[i] = acc;
    }
  } else {
#pragma unroll
    for (int j = 0; j < D; ++j) v[j] = dl[j];
  }
}

// End of a walk for chain c: the retained state, its log-density and the accept count, and
// the chain's running sums added to the caller's (ssum / ssq null: the caller adds them)
template <int D>
__device__ __forceinline__ void write_back(const MhMvnArgs& a, int c, const double (&x)[D],
                                           double lp, int64_t nacc, const double* ssum,
                                           const double* ssq) {
  const int64_t C = a.C;
#pragma unroll
  for (int j = 0; j < D; ++j) {
    a.state[j * C + c] = x[j];
    if (ssum && a.stat_sum) a.stat_sum[j * C + c] += ssum[j];
    if (ssq && a.stat_sumsq) a.stat_sumsq[j * C + c] += ssq[j];
  }
  a.state_lp[c] = lp;
  if (a.accept_count) a.accept_count[c] += nacc;
}

template <int D, bool kInjected>
__global__ void __launch_bounds__(128) mh_mvn_kernel(const MhMvnArgs a,
                                                     const __grid_constant__ MhMvnConst m) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= a.C) return;
  const int64_t C = a.C;
  const uint32_t gchain = (uint32_t)(a.chain0 + c);

  double x[D], ssum[D], ssq[D];
#pragma unroll
  for (int j = 0; j < D; ++j) {
    x[j] = a.state[j * C + c];
    ssum[j] = 0.0;
    ssq[j] = 0.0;
  }
  double lp = (a.step0 > 0) ? a.state_lp[c] : 0.0;
  // Mahalanobis distance of the retained state, recomputed from x (bit-identical to
  // the value obtained when that state was proposed, so resumed walks decide alike)
  double mcur = mvn_maha<D>(x, m);
  // linear density of the retained state (what the reference's opqr.o.prob holds)
  double lin = (a.step0 > 0) ? (a.log_pscale ? pbx_exp_logp(lp) : exp(lp)) : 0.0;
  int64_t nacc = 0;
  const bool ref_mode = (a.accept_mode == PBX_ACCEPT_REFERENCE);

  for (int k = 0; k < a.T; ++k) {
    const int64_t gstep = a.step0 + k;
    double dl[D];
    double t;
    // ---- draws: proposal first, then the threshold (sp.py:231-249) ----------
    if (kInjected) {
#pragma unroll
      for (int j = 0; j < D; ++j) dl[j] = a.inj_delta[((int64_t)k * D + j) * C + c];
      t = a.inj_thresh[(int64_t)k * C + c];
    } else {
      draw_step<D>(a.seed, (uint64_t)gstep, gchain, a.prop_kind, m, &g_tables, dl, t);
    }
    // ---- propose: x' = x + delta  (or + L delta: rf.py:346-348) -------------
    double xp[D], dv[D];
    colour_delta<D>(a.has_L, m, dl, dv);
#pragma unroll
    for (int j = 0; j < D; ++j) xp[j] = x[j] + dv[j];
    if (m.bound) {
#pragma unroll
      for (int j = 0; j < D; ++j)
        xp[j] = pbx_bound(xp[j], x[j], m.lims[j][0], m.lims[j][1], m.open_end[j][0] != 0,
                          m.open_end[j][1] != 0);
    }
    // ---- evaluate target ----------------------------------------------------
    const double maha = mvn_maha<D>(xp, m);
    const double lpp = -0.5 * (m.norm_c + maha);
    // ---- score / threshold / update (sp_utils.py:19-37) ---------------------
    bool acc;
    double s = nan("");
    double linp = 0.0;
    if (ref_mode) {
      linp = a.log_pscale ? pbx_exp_logp(lpp) : exp(lpp);
      if (gstep == 0) {
        acc = true;
      } else {
        s = fmin(1.0, linp / fmax(PBX_TINY, lin));
        acc = (s >= t);
      }
    } else {
      // Log-space accept test on the Mahalanobis distance: logp' - logp >= log t with
      // logp = -0.5 (c + maha)  <=>  maha' <= maha - 2 log t.  The right-hand side depends
      // only on the CURRENT state and the threshold draw, so it is off the sequential
      // critical path (the chain per step is add, sub, mul, fma, mul, fma, setp, select)
      // and the chain never needs logp itself (the writer derives it from maha).
      if (gstep == 0) {
        acc = true;
      } else {
        // injected thresholds go through libm's log (bit-parity with the oracle);
        // native ones through the same table log as the warp-specialised kernel
        const double th2 = kInjected ? -2.0 * log(t) : fast_neg2log(t, &g_tables);
        acc = (maha <= mcur + th2);
        if (a.out_score) s = fmin(1.0, exp(fmin(lpp - lp, 0.0)));
      }
    }
    if (acc) {
#pragma unroll
      for (int j = 0; j < D; ++j) x[j] = xp[j];
      lp = lpp;
      mcur = maha;
      lin = linp;
      ++nacc;
    }
    // ---- record -------------------------------------------------------------
#pragma unroll
    for (int j = 0; j < D; ++j) {
      ssum[j] += x[j];
      ssq[j] = fma(x[j], x[j], ssq[j]);
    }
    if (a.out_accept) a.out_accept[(int64_t)k * C + c] = acc ? 1 : 0;
    if (a.out_score) a.out_score[(int64_t)k * C + c] = s;
    if (a.out_xprop) {
#pragma unroll
      for (int j = 0; j < D; ++j) a.out_xprop[((int64_t)k * D + j) * C + c] = xp[j];
    }
    if (a.out_pprop)
      a.out_pprop[(int64_t)k * C + c] = a.log_pscale ? lpp : (ref_mode ? linp : exp(lpp));
    if ((k + 1) % a.thin == 0) {
      const int64_t r = (k + 1) / a.thin - 1;
      if (a.out_x) {
#pragma unroll
        for (int j = 0; j < D; ++j) a.out_x[(r * D + j) * C + c] = x[j];
      }
      if (a.out_prob) a.out_prob[r * C + c] = rec_density(lp, a.log_pscale, ref_mode, &g_tables);
    }
  }
  write_back(a, c, x, lp, nacc, ssum, ssq);
}

// ---------------------------------------------------------------------------
// Warp-specialised native-RNG kernel.  One CTA = 32 chains (lane = chain).
//   warp 0       consumer: the sequential chain only (propose, quadratic form,
//                accept, select, running sums) -- ~30 instructions per step, no
//                global traffic.  It overwrites the ring slot it just consumed
//                with the retained states (x, logp) of that batch.
//   12 or 9 producer/writer warps (every warp with warp % 4 != 0; warps 4, 8, 12 exit
//                at once so that the consumer has SM sub-partition 0 -- scheduler and
//                FP64 pipe -- to itself): each owns TWO ring slots.  Per use: drain the
//                consumer's results of the slot's previous batch (thinning, logp and
//                exp() for linear-pscale output, coalesced global stores), then refill
//                it with Philox + Box-Muller deltas and -2 log(threshold) for the next
//                batch of G steps.  Both jobs are independent of the chain state
//                and therefore parallel over steps.
// One mbarrier pair per slot: in_full (producer -> consumer), out_full (consumer
// -> owning producer).
// ---------------------------------------------------------------------------
template <int D> struct WsCfg {
  // steps per ring slot: G*(D+1) doubles per lane per slot, <= 6 KB per slot
  static constexpr int G = (D <= 2) ? 8 : (D == 3 ? 6 : (D <= 5 ? 4 : (D <= 7 ? 3 : 2)));
  static constexpr int SLOT_DOUBLES = G * (D + 1) * 32;
  // CTA shape (measured, 4096 chains x 10^4 steps): 12 producer warps in a 512-thread CTA
  // (128 registers per thread) for D <= 3 -- 0.546 ms at D = 2 against 0.559 with 15
  // producers / 96 registers and 0.598 with 9; the producer count must be a multiple of 3
  // so that the three producer sub-partitions carry equal load (11 or 13 are 7-14 % slower).
  // From D = 4 on the consumer's state + D x D quadratic form dominate and want registers:
  // 9 producers / 384 threads (up to 168 registers; D = 6: 1.70 -> 1.39 ms, D = 8: 6.5 ->
  // 3.9 ms against the 15-producer shape).
  // The producers are the warps with warp % 4 != 0 (see above): 12 of 16 warps, 9 of 12.
  static constexpr int NPROD = (D <= 3) ? 12 : 9;
  static constexpr int NSLOT = 2 * NPROD;                 // two ring slots per producer warp
  static constexpr int THREADS = 32 * (NPROD + 1 + (NPROD - 1) / 3);
  static constexpr size_t SMEM = (size_t)NSLOT * SLOT_DOUBLES * sizeof(double);
};

// kFast: normal proposal without Cholesky colouring -> branch-free producer body
// kZeroMean: see mvn_maha
template <int D, bool kRefAccept, bool kFast, bool kZeroMean = false>
__global__ void __launch_bounds__(WsCfg<D>::THREADS, 1)
    mh_mvn_ws_kernel(const MhMvnArgs a, const __grid_constant__ MhMvnConst m) {
  constexpr int G = WsCfg<D>::G;
  constexpr int SD = WsCfg<D>::SLOT_DOUBLES;
  constexpr int NP = WsCfg<D>::NPROD, NS = WsCfg<D>::NSLOT;
  extern __shared__ __align__(16) double ring[];          // [NS][G][D+1][32]
  __shared__ __align__(8) unsigned long long in_full[NS], out_full[NS];
  __shared__ __align__(16) PbxTables s_tb;                // 40 KB of math tables
  stage_tables<WsCfg<D>::THREADS>(s_tb);
  const PbxTables* tb = &s_tb;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t C = a.C;
  const int c = blockIdx.x * 32 + lane;
  const bool valid = c < a.C;
  const uint32_t gchain = (uint32_t)(a.chain0 + (valid ? c : 0));
  const int nb = (a.T + G - 1) / G;                       // batches of G steps

  if (threadIdx.x == 0) {
    for (int i = 0; i < NS; ++i) {
      pbx_mbar_init(&in_full[i], 1);
      pbx_mbar_init(&out_full[i], 1);
    }
  }
  __syncthreads();

  if (warp >= 1) {
    // ================= producer / writer: owns ring slots p and p + NP ===========
    if ((warp & 3) == 0) return;                          // keep sub-partition 0 for the consumer
    const int p = warp - 1 - (warp >> 2);
    const int n_mine = (nb > p) ? (nb - p + NP - 1) / NP : 0;
    for (int n = 0; n < n_mine + 2; ++n) {
      const int si = p + NP * (n & 1);
      double* slot = ring + (size_t)si * SD + lane;
      if (n >= 2 && n - 2 < n_mine) {
        // ---- drain the results of my batch n-2 (it used this slot) --------------
        const int bd = p + NP * (n - 2);
        pbx_mbar_wait(&out_full[si], (uint32_t)((n - 2) >> 1) & 1);
        const int k0 = bd * G;
        const int ng = min(G, a.T - k0);
        if (a.thin == 1 && ng == G && a.out_x != nullptr && a.out_prob != nullptr) {
          // common case (every step recorded, full batch): straight-line code, record
          // index = step index, addresses as base + compile-time multiples of C
          if (valid) {
            double* ox = a.out_x + ((int64_t)k0 * D) * C + c;
            double* op = a.out_prob + (int64_t)k0 * C + c;
            // the consumer leaves logp (reference rule) or the Mahalanobis distance (log
            // rule) of the retained state in the slot
            if (a.log_pscale) {
#pragma unroll
              for (int g = 0; g < G; ++g) {
#pragma unroll
                for (int j = 0; j < D; ++j) ox[(g * D + j) * C] = slot[(g * (D + 1) + j) * 32];
                const double sv = slot[(g * (D + 1) + D) * 32];
                const double lpv = kRefAccept ? sv : -0.5 * (m.norm_c + sv);
                op[g * C] = rec_density(lpv, true, kRefAccept, tb);
              }
            } else {
#pragma unroll
              for (int g = 0; g < G; ++g) {
#pragma unroll
                for (int j = 0; j < D; ++j) ox[(g * D + j) * C] = slot[(g * (D + 1) + j) * 32];
                const double sv = slot[(g * (D + 1) + D) * 32];
                const double lpv = kRefAccept ? sv : -0.5 * (m.norm_c + sv);
                op[g * C] = rec_density(lpv, false, kRefAccept, tb);
              }
            }
          }
        } else {
          int rem = (k0 + 1) % a.thin;                    // (k+1) % thin of step k0
          const int64_t rec0 = (k0 + 1) / a.thin - 1 + (rem != 0);   // first record index
          double* ox = a.out_x ? a.out_x + (rec0 * D) * C + c : nullptr;
          double* op = a.out_prob ? a.out_prob + rec0 * C + c : nullptr;
          if (rem == 0) rem = a.thin;                     // countdown form: record when == thin
          for (int g = 0; g < ng; ++g) {
            if (rem == a.thin) {
              rem = 0;
              if (valid) {
                if (ox) {
#pragma unroll
                  for (int j = 0; j < D; ++j) ox[j * C] = slot[(g * (D + 1) + j) * 32];
                  ox += D * C;
                }
                if (op) {
                  const double sv = slot[(g * (D + 1) + D) * 32];
                  const double lpv = kRefAccept ? sv : -0.5 * (m.norm_c + sv);
                  *op = rec_density(lpv, a.log_pscale, kRefAccept, tb);
                  op += C;
                }
              }
            }
            ++rem;
          }
        }
      }
      if (n >= n_mine) continue;
      const int b = p + NP * n;
      auto produce = [&](int g) {
        const int64_t gstep = a.step0 + (int64_t)b * G + g;
        double dl[D], dv[D], t;
        draw_step<D, kFast>(a.seed, (uint64_t)gstep, gchain, a.prop_kind, m, tb, dl, t);
        colour_delta<D>(kFast ? 0 : a.has_L, m, dl, dv);
#pragma unroll
        for (int j = 0; j < D; ++j) slot[(g * (D + 1) + j) * 32] = dv[j];
        // log rule: -2 log t (added to the current Mahalanobis distance by the consumer)
        slot[(g * (D + 1) + D) * 32] = kRefAccept ? t : fast_neg2log(t, tb);
      };
      if ((b + 1) * G <= a.T) {
        // full batch: kUnroll independent steps in flight per thread (ILP), since a
        // producer warp is otherwise a single chain of dependent instructions
        // (D <= 3: four independent steps in flight in the 128-register shape -- 0.547 ->
        // 0.532 ms at D = 2; D = 4: two; beyond that one, the draws of a step fill the file)
        constexpr int kUnroll = (D <= 3) ? (kRefAccept ? 2 : 4) : (D == 4 ? 2 : 1);
#pragma unroll kUnroll
        for (int g = 0; g < G; ++g) produce(g);
      } else {
#pragma unroll 1
        for (int g = 0; g < a.T - b * G; ++g) produce(g);
      }
      // global step 0 accepts unconditionally (sp.py:253): a threshold that always passes
      if (b == 0 && a.step0 == 0) slot[D * 32] = kRefAccept ? 0.0 : INFINITY;
      __syncwarp();
      if (lane == 0) pbx_mbar_arrive(&in_full[si]);
    }
    return;
  }

  // ======================= consumer: the sequential chain =====================
  double x[D], ssum[D], ssq[D];
#pragma unroll
  for (int j = 0; j < D; ++j) {
    x[j] = valid ? a.state[j * C + c] : 0.0;
    ssum[j] = ssq[j] = 0.0;
  }
  double lp = (a.step0 > 0 && valid) ? a.state_lp[c] : 0.0;
  double mcur = mvn_maha<D, kZeroMean>(x, m);   // log rule state: maha of the retained state
  double lin = 0.0;
  if (kRefAccept && a.step0 > 0) lin = a.log_pscale ? pbx_exp_logp(lp) : exp(lp);
  int64_t nacc = 0;

  for (int b = 0; b < nb; ++b) {
    const int s = b % NS;
    double* slot = ring + (size_t)s * SD + lane;
    pbx_mbar_wait(&in_full[s], (uint32_t)(b / NS) & 1);
    const int ng = min(G, a.T - b * G);
    // D <= 4: the whole batch is loaded into registers up front; beyond that G * (D + 1)
    // doubles no longer fit next to the state and each step loads its own inputs
    constexpr bool kPreload = D <= 4;
    constexpr int GP = kPreload ? G : 1;
    double dl[GP][D], th[GP];
    if (kPreload) {
#pragma unroll
      for (int g = 0; g < G; ++g) {
#pragma unroll
        for (int j = 0; j < D; ++j) dl[g][j] = slot[(g * (D + 1) + j) * 32];
        th[g] = slot[(g * (D + 1) + D) * 32];
      }
    }
    // every lane only ever touches its own column of the slot, so the results can
    // overwrite the inputs as soon as they are in registers
    auto step = [&](int g) {
      double xp[D];
#pragma unroll
      for (int j = 0; j < D; ++j)
        xp[j] = x[j] + (kPreload ? dl[kPreload ? g : 0][j] : slot[(g * (D + 1) + j) * 32]);
      const double thg = kPreload ? th[kPreload ? g : 0] : slot[(g * (D + 1) + D) * 32];
      const double maha = mvn_maha<D, kZeroMean>(xp, m);
      bool acc;
      if (kRefAccept) {
        const double lpp = -0.5 * (m.norm_c + maha);
        const double linp = a.log_pscale ? pbx_exp_logp(lpp) : exp(lpp);
        acc = fmin(1.0, linp / fmax(PBX_TINY, lin)) >= thg;
        if (acc) {
          lp = lpp;
          lin = linp;
        }
      } else {
        acc = maha <= mcur + thg;
      }
      if (acc) {
#pragma unroll
        for (int j = 0; j < D; ++j) x[j] = xp[j];
        mcur = maha;
        ++nacc;
      }
#pragma unroll
      for (int j = 0; j < D; ++j) {
        ssum[j] += x[j];
        ssq[j] = fma(x[j], x[j], ssq[j]);
        slot[(g * (D + 1) + j) * 32] = x[j];
      }
      slot[(g * (D + 1) + D) * 32] = kRefAccept ? lp : mcur;
    };
    // Two steps at a time with the second one speculated on both outcomes of the
    // first (log rule only): the distances of PA = S + dA, PB0 = S + dB and
    // PB1 = PA + dB are independent, so the dependent chain per PAIR is
    // add, add, sub, mul, fma, mul, fma, select, setp, select (10 ops instead of 16),
    // with bit-identical arithmetic (the same operations on the same operands).
    auto pair = [&](int g) {
      double pa[D], pb0[D], pb1[D];
#pragma unroll
      for (int j = 0; j < D; ++j) {
        pa[j] = x[j] + dl[g][j];
        pb0[j] = x[j] + dl[g + 1][j];
        pb1[j] = pa[j] + dl[g + 1][j];
      }
      const double ma = mvn_maha<D, kZeroMean>(pa, m), mb0 = mvn_maha<D, kZeroMean>(pb0, m),
                   mb1 = mvn_maha<D, kZeroMean>(pb1, m);
      const bool aa = ma <= mcur + th[g];
      const bool ab = aa ? (mb1 <= ma + th[g + 1]) : (mb0 <= mcur + th[g + 1]);
      double s1[D];
#pragma unroll
      for (int j = 0; j < D; ++j) s1[j] = aa ? pa[j] : x[j];
      const double m1 = aa ? ma : mcur;
#pragma unroll
      for (int j = 0; j < D; ++j) x[j] = ab ? (aa ? pb1[j] : pb0[j]) : s1[j];
      mcur = ab ? (aa ? mb1 : mb0) : m1;
      nacc += (int)aa + (int)ab;
#pragma unroll
      for (int j = 0; j < D; ++j) {
        ssum[j] += s1[j];
        ssq[j] = fma(s1[j], s1[j], ssq[j]);
        ssum[j] += x[j];
        ssq[j] = fma(x[j], x[j], ssq[j]);
        slot[(g * (D + 1) + j) * 32] = s1[j];
        slot[((g + 1) * (D + 1) + j) * 32] = x[j];
      }
      slot[(g * (D + 1) + D) * 32] = m1;
      slot[((g + 1) * (D + 1) + D) * 32] = mcur;
    };
    if (ng == G) {                       // full batch: straight-line code, no predicates
      if (!kRefAccept && (G % 2 == 0) && D <= 4) {   // speculation needs 3 states in registers
#pragma unroll
        for (int g = 0; g < G; g += 2) pair(g);
      } else {
#pragma unroll
        for (int g = 0; g < G; ++g) step(g);
      }
    } else {
#pragma unroll
      for (int g = 0; g < G; ++g)
        if (g < ng) step(g);
    }
    __syncwarp();
    if (lane == 0) pbx_mbar_arrive(&out_full[s]);
  }
  // written out rather than through write_back: with the helper ptxas schedules the consumer
  // loop differently, and the D = 6 walk of scripts/bench_k1_dims.py ran 3 % slower (B200)
  if (valid) {
#pragma unroll
    for (int j = 0; j < D; ++j) {
      a.state[j * C + c] = x[j];
      if (a.stat_sum) a.stat_sum[j * C + c] += ssum[j];
      if (a.stat_sumsq) a.stat_sumsq[j * C + c] += ssq[j];
    }
    a.state_lp[c] = kRefAccept ? lp : -0.5 * (m.norm_c + mcur);
    if (a.accept_count) a.accept_count[c] += nacc;
  }
}


// ---------------------------------------------------------------------------
// "Whitened-decision" kernel (log accept rule, D <= 4): the default native-RNG path.
//
// The accept test of the log rule, maha(x + d) <= maha(x) - 2 log t, is quadratic in the
// WHITENED state y = W^T (x - mean):  |y + e|^2 <= |y|^2 + th  with e = W^T d, i.e.
//         y . e  <=  (th - |e|^2) / 2  =: kappa
// and kappa, like e, does not depend on the chain state.  So the producers (parallel over
// steps) ship e, kappa and d, and the inherently sequential part shrinks to one D-term dot
// product, one compare and predicated adds (y += e, x += d): ~13 instructions per step
// instead of ~39, with a dependent chain of ~23 cycles per step instead of ~100.  Steps are
// taken in pairs (A, B): both dots use the state before A, and B's threshold is picked
// between kappa_B (A rejected) and kappa_B - e_A . e_B (A accepted), also state-free.
// x is still advanced by exactly x + d (the reference's arithmetic, sp.py:231-239 /
// variable.py:693-697), and the recorded density is recomputed from the recorded x by the
// writers with the same quadratic form as everywhere else, so trajectories and densities
// are bit-identical to the exact-arithmetic kernels as long as the decisions agree; a
// decision can only differ where the margin |y . e - kappa| is below the rounding of the
// incrementally tracked y (~1e-14 relative): ~1e-14 per step.
//
// CTA = `cpc` chains (<= 32, chosen by the host so that the grid fills all SMs: 28 for
// 4096 chains on 148 SMs), 15 warps:
//   warp 0        decisions: lane = chain
//   warps 1..14   producers / writers, parallel over a flat list of 448 (pair, chain)
//                 items per batch (batch = 448 / cpc pairs of steps); each thread owns one
//                 item of every batch: drains its previous result (record x, density,
//                 running sums), then draws the next pair of steps.  No lane is idle
//                 whatever cpc is.
// Ring of NSLOT batches in shared memory, [field pair][item] as double2 (128-bit
// conflict-free accesses on both sides), one mbarrier pair per slot.
// ---------------------------------------------------------------------------
constexpr int kWdMaxD = 4;
// shared-memory accesses of the decision warp by 32-bit shared-space address (a generic
// pointer makes the compiler rebuild the shared window base -- S2UR SR_CgaCtaId, ~100 cycles
// -- in front of every access of the loop); volatile keeps fetches and stores in program order
__device__ __forceinline__ double2 pbx_lds_v2(uint32_t addr) {
  double2 v;
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr));
  return v;
}
__device__ __forceinline__ void pbx_sts_v2(uint32_t addr, double a, double b) {
  asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(addr), "d"(a), "d"(b) : "memory");
}
template <int D> struct WdCfg {
  static constexpr int THREADS = 512;   // 16 warps: decisions, 14 producers, one idle (see below)
  static constexpr int NPROD = 14;
  // one item per producer thread and batch (two, i.e. four steps in flight per thread,
  // measured no gain)
  static constexpr int ITEMS = NPROD * 32;
  static constexpr int NF2 = 2 * D + 2;   // double2 per item: eA[D] eB[D] kA kB0 kB1 pad dA[D] dB[D]
  static constexpr int NSLOT = (D <= 2) ? 3 : 2;          // ring depth in batches
  static constexpr size_t SMEM = (size_t)NSLOT * NF2 * ITEMS * sizeof(double2);
};

template <int D, bool kFast, bool kZeroMean>
__global__ void __launch_bounds__(WdCfg<D>::THREADS, 1)
    mh_mvn_wd_kernel(const MhMvnArgs a, const __grid_constant__ MhMvnConst m, const int cpc) {
  constexpr int NF2 = WdCfg<D>::NF2;
  constexpr int NS = WdCfg<D>::NSLOT;
  constexpr int ITEMS = WdCfg<D>::ITEMS;
  extern __shared__ __align__(16) double2 ring2[];        // [NS][NF2][ITEMS]
  __shared__ __align__(8) unsigned long long in_full[NS], out_full[NS];
  __shared__ __align__(16) PbxTables s_tb;
  stage_tables<WdCfg<D>::THREADS>(s_tb);
  const PbxTables* tb = &s_tb;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t C = a.C;
  const int P = ITEMS / cpc;                    // pairs of steps per batch
  const int S = 2 * P;                          // steps per batch
  const int nb = (a.T + S - 1) / S;
  const int cbase = blockIdx.x * cpc;
  if (threadIdx.x == 0) {
    for (int i = 0; i < NS; ++i) {
      pbx_mbar_init(&in_full[i], WdCfg<D>::NPROD);
      pbx_mbar_init(&out_full[i], 1);
    }
  }
  __syncthreads();

  double ssum[D], ssq[D];                       // producers: running sums of their items
#pragma unroll
  for (int j = 0; j < D; ++j) ssum[j] = ssq[j] = 0.0;
  // Warp w runs on SM sub-partition w % 4.  The decision warp (0) is latency-critical:
  // it shares sub-partition 0 with only TWO producers (warps 4 and 8; warp 12 idles), the
  // other three sub-partitions run four producers each.  Producer index pi = 0..13.
  const int pi = (warp & 3) ? (warp - 1 - (warp >> 2)) : (warp == 4 ? 12 : (warp == 8 ? 13 : -1));
  const int item = (pi >= 0) ? pi * 32 + lane : 0;

  if (pi >= 0) {
    // ===================== producer / writer: one (pair, chain) item per batch ==========
    const int pr = item / cpc, ch = item - pr * cpc;
    const int c = cbase + ch;
    const bool valid = c < a.C;
    const uint32_t gchain = (uint32_t)(a.chain0 + (valid ? c : 0));
    const bool rec_all = a.thin == 1 && a.out_x != nullptr && a.out_prob != nullptr;
    // My item of a batch: pair pr of chain ch.  Records of the batch being drained
    // (thin == 1: record index = step index) through running pointers.
    double* px = rec_all ? a.out_x + ((int64_t)(2 * pr) * D) * C + c : nullptr;
    double* pp = rec_all ? a.out_prob + (int64_t)(2 * pr) * C + c : nullptr;
    for (int b = 0; b < nb + NS; ++b) {
      const int s = b % NS;
      double2* slot = ring2 + (size_t)s * NF2 * ITEMS + item;
      if (b >= NS) {
        // ---- drain my item of batch b - NS: the states after steps A and B --------------
        const int bd = b - NS;
        pbx_mbar_wait(&out_full[s], (uint32_t)(bd / NS) & 1);
        const bool whole = rec_all && (bd + 1) * S <= a.T;
        double r[2 * D];
#pragma unroll
        for (int q = 0; q < D; ++q) {
          const double2 t2 = slot[(D + 2 + q) * ITEMS];
          r[2 * q] = t2.x;
          r[2 * q + 1] = t2.y;
        }
        const int kA = bd * S + 2 * pr;
        if (valid && whole) {
          // common case (every step recorded, whole batch live): straight-line code
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            double xs[D];
#pragma unroll
            for (int j = 0; j < D; ++j) {
              xs[j] = r[h * D + j];
              ssum[j] += xs[j];
              ssq[j] = fma(xs[j], xs[j], ssq[j]);
              px[(h * D + j) * C] = xs[j];
            }
            const double lpv = -0.5 * (m.norm_c + mvn_maha<D, kZeroMean>(xs, m));
            pp[h * C] = rec_density(lpv, a.log_pscale, false, tb);
          }
        } else if (valid) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int kk = kA + h;
            if (kk < a.T) {
              double xs[D];
#pragma unroll
              for (int j = 0; j < D; ++j) {
                xs[j] = r[h * D + j];
                ssum[j] += xs[j];
                ssq[j] = fma(xs[j], xs[j], ssq[j]);
              }
              const bool keep = ((kk + 1) % a.thin) == 0;
              const int64_t rec = (kk + 1) / a.thin - 1;
              if (keep) {
                if (a.out_x) {
#pragma unroll
                  for (int j = 0; j < D; ++j) a.out_x[(rec * D + j) * C + c] = xs[j];
                }
                if (a.out_prob) {
                  const double lpv = -0.5 * (m.norm_c + mvn_maha<D, kZeroMean>(xs, m));
                  a.out_prob[rec * C + c] = rec_density(lpv, a.log_pscale, false, tb);
                }
              }
            }
          }
        }
        if (rec_all) {
          px += (int64_t)S * D * C;
          pp += (int64_t)S * C;
        }
      }
      if (b >= nb) continue;
      // ---- draw my pair of steps of batch b --------------------------------------------------
      const int64_t gA = a.step0 + (int64_t)b * S + 2 * pr;
      double eA[D], eB[D], dA_[D], dB_[D], kA_, kB_;
      auto gen = [&](int64_t gstep, double (&eta)[D], double (&dv)[D], double& kap) {
        double dl[D], t;
        draw_step<D, kFast>(a.seed, (uint64_t)gstep, gchain, a.prop_kind, m, tb, dl, t);
        colour_delta<D>(kFast ? 0 : a.has_L, m, dl, dv);
        const double th = fast_neg2log(t, tb);
        double n2 = 0.0;                         // |e|^2
        whiten<D, true>(dv, m, [&](int k, double e) {
          eta[k] = e;
          n2 = fma(e, e, n2);
        });
        kap = 0.5 * (th - n2);
      };
      gen(gA, eA, dA_, kA_);
      gen(gA + 1, eB, dB_, kB_);
      double cross = 0.0;
#pragma unroll
      for (int kk = 0; kk < D; ++kk) cross = fma(eA[kk], eB[kk], cross);
      double v[4 * D + 4];
#pragma unroll
      for (int j = 0; j < D; ++j) {
        v[j] = eA[j];
        v[D + j] = eB[j];
        v[2 * D + 4 + j] = dA_[j];
        v[3 * D + 4 + j] = dB_[j];
      }
      v[2 * D] = kA_;
      v[2 * D + 1] = kB_;
      v[2 * D + 2] = kB_ - cross;
      v[2 * D + 3] = 0.0;
      if (gA == 0) v[2 * D] = INFINITY;          // global step 0 accepts unconditionally (sp.py:253)
#pragma unroll
      for (int q = 0; q < NF2; ++q) slot[q * ITEMS] = make_double2(v[2 * q], v[2 * q + 1]);
      __syncwarp();
      if (lane == 0) pbx_mbar_arrive(&in_full[s]);
    }
  } else if (warp == 0) {
    // ======================= decisions: lane = chain ======================================
    const bool active = lane < cpc;
    const int c = cbase + lane;
    const bool valid = active && c < a.C;
    const int li = active ? lane : cpc - 1;      // idle lanes shadow the last chain (no stores)
    double x[D], y[D];
#pragma unroll
    for (int j = 0; j < D; ++j) x[j] = valid ? a.state[j * C + c] : 0.0;
    whiten<D, kZeroMean>(x, m, [&](int k, double e) { y[k] = e; });
    int nacc = 0;
    // (laundered through an opaque move so that the compiler keeps the base in a register
    // instead of rematerialising it -- S2UR SR_CgaCtaId and friends -- at every use)
    uint32_t ring_base = pbx_smem_u32(ring2);
    asm volatile("mov.u32 %0, %0;" : "+r"(ring_base));
    // one pair of steps; v = the item's fields (see WdCfg), results overwrite dA / dB
    auto process = [&](uint32_t it, const double (&v)[4 * D + 4], bool liveB) {
      double dA = y[0] * v[0], dB = y[0] * v[D];
#pragma unroll
      for (int j = 1; j < D; ++j) {
        dA = fma(y[j], v[j], dA);
        dB = fma(y[j], v[D + j], dB);
      }
      const bool aA = dA <= v[2 * D];
      const double kB = aA ? v[2 * D + 2] : v[2 * D + 1];
      const bool aB = liveB && (dB <= kB);
      // y (on the dependent chain): speculative add + select.  x (off the chain): one
      // fma with a 0.0 / 1.0 mask per component -- fma(1, d, x) rounds x + d exactly as the
      // add does, fma(0, d, x) returns x -- instead of an add and two 32-bit selects.
      const double mA = __hiloint2double(aA ? 0x3FF00000 : 0, 0);
      const double mB = __hiloint2double(aB ? 0x3FF00000 : 0, 0);
      double r[2 * D];
#pragma unroll
      for (int j = 0; j < D; ++j) {
        const double ya = y[j] + v[j];
        y[j] = aA ? ya : y[j];
        x[j] = fma(mA, v[2 * D + 4 + j], x[j]);
        r[j] = x[j];
      }
#pragma unroll
      for (int j = 0; j < D; ++j) {
        const double yb = y[j] + v[D + j];
        y[j] = aB ? yb : y[j];
        x[j] = fma(mB, v[3 * D + 4 + j], x[j]);
        r[D + j] = x[j];
      }
      nacc += (int)aA + (int)aB;
      if (active) {
#pragma unroll
        for (int q = 0; q < D; ++q)
          pbx_sts_v2(it + (D + 2 + q) * ITEMS * 16, r[2 * q], r[2 * q + 1]);
      }
    };
    auto fetch = [&](uint32_t it, double (&v)[4 * D + 4]) {
#pragma unroll
      for (int q = 0; q < NF2; ++q) {
        const double2 t2 = pbx_lds_v2(it + q * ITEMS * 16);
        v[2 * q] = t2.x;
        v[2 * q + 1] = t2.y;
      }
    };
#pragma unroll 1
    for (int b = 0; b < nb; ++b) {
      const int s = b % NS;
      const uint32_t slot = ring_base + (uint32_t)((s * NF2 * ITEMS + li) * 16);
      pbx_mbar_wait(&in_full[s], (uint32_t)(b / NS) & 1);
      const int kb = b * S;
      const int np = min(P, (a.T - kb + 1) / 2);            // pairs with a live step
      const bool tail = kb + S > a.T;                       // only the last batch can be short
      // A pair's fields are fetched three pairs before they are used (register ring of four
      // pairs), so that the shared-memory latency -- long under the producers' traffic --
      // stays off the chain; the fetches are volatile, i.e. issued exactly here.  Whole
      // batches run as straight-line groups of four pairs (one backward branch per group:
      // every branch costs the single decision warp a predicate + fetch bubble).
      int p = 0;
      if (!tail) {
        const int last = (np - 1) * cpc * 16;
        const int step16 = cpc * 16;
        uint32_t it = slot;
        int off = 0;                                       // byte offset of pair p
        if constexpr (D <= 2) {
          const int nfull = np & ~3;
          double v0[4 * D + 4], v1[4 * D + 4], v2[4 * D + 4], v3[4 * D + 4];
          fetch(slot, v0);
          fetch(slot + min(step16, last), v1);
          fetch(slot + min(2 * step16, last), v2);
#pragma unroll 1
          for (; p < nfull; p += 4) {
            fetch(slot + min(off + 3 * step16, last), v3);
            process(it, v0, true);
            fetch(slot + min(off + 4 * step16, last), v0);
            process(it + step16, v1, true);
            fetch(slot + min(off + 5 * step16, last), v1);
            process(it + 2 * step16, v2, true);
            fetch(slot + min(off + 6 * step16, last), v2);
            process(it + 3 * step16, v3, true);
            it += 4 * step16;
            off += 4 * step16;
          }
        } else {                                           // fewer registers to spare: ring of two
          const int nfull = np & ~1;
          double v0[4 * D + 4], v1[4 * D + 4];
          fetch(slot, v0);
#pragma unroll 1
          for (; p < nfull; p += 2) {
            fetch(slot + min(off + step16, last), v1);
            process(it, v0, true);
            fetch(slot + min(off + 2 * step16, last), v0);
            process(it + step16, v1, true);
            it += 2 * step16;
            off += 2 * step16;
          }
        }
      }
#pragma unroll 1
      for (; p < np; ++p) {                                // tail batch / remainder pairs
        double v[4 * D + 4];
        fetch(slot + p * cpc * 16, v);
        process(slot + p * cpc * 16, v, kb + 2 * p + 1 < a.T);
      }
      __syncwarp();
      if (lane == 0) pbx_mbar_arrive(&out_full[s]);
    }
    // the running sums are the producers' (reduced below)
    if (valid)
      write_back(a, c, x, -0.5 * (m.norm_c + mvn_maha<D, kZeroMean>(x, m)), nacc, nullptr,
                 nullptr);
  }
  // ---- running sums: fixed-order reduction of the per-item partials (deterministic) -------
  if (a.stat_sum == nullptr && a.stat_sumsq == nullptr) return;
  __syncthreads();                               // every slot is drained: reuse the ring
  double* part = reinterpret_cast<double*>(ring2);           // [2 D][ITEMS]
  if (pi >= 0) {
#pragma unroll
    for (int j = 0; j < D; ++j) {
      part[(2 * j) * ITEMS + item] = ssum[j];
      part[(2 * j + 1) * ITEMS + item] = ssq[j];
    }
  }
  __syncthreads();
  for (int t = threadIdx.x; t < cpc * D; t += WdCfg<D>::THREADS) {
    const int j = t / cpc, ch = t - j * cpc;
    const int c = cbase + ch;
    if (c >= a.C) continue;
    double s1 = 0.0, s2 = 0.0;
    for (int p = 0; p < P; ++p) {
      s1 += part[(2 * j) * ITEMS + p * cpc + ch];
      s2 += part[(2 * j + 1) * ITEMS + p * cpc + ch];
    }
    if (a.stat_sum) a.stat_sum[j * C + c] += s1;
    if (a.stat_sumsq) a.stat_sumsq[j * C + c] += s2;
  }
}

// chains per CTA of the whitened-decision kernel: 448 / cpc must be an even integer or 14;
// the grid should fill whole waves of SMs with as few chains per CTA as possible (the CTA's
// time is proportional to cpc: its producers work on cpc chains)
static int wd_pick_cpc(int C, int sms) {
  const int cand[5] = {32, 28, 16, 8, 4};
  int best = 32;
  long best_cost = -1;
  for (int i = 0; i < 5; ++i) {
    const long ctas = (C + cand[i] - 1) / cand[i];
    const long cost = ((ctas + sms - 1) / sms) * cand[i];
    if (best_cost < 0 || cost < best_cost) {
      best_cost = cost;
      best = cand[i];
    }
  }
  return best;
}

template <int D>
static int launch_mh_mvn(pbx_ctx* ctx, const MhMvnArgs& a, const MhMvnConst& m, int kernel_variant) {
  const bool injected = a.inj_delta != nullptr;
  const bool per_step = a.out_accept != nullptr || a.out_score != nullptr ||
                        a.out_xprop != nullptr || a.out_pprop != nullptr;
  const bool use_ws = !injected && !per_step && kernel_variant != 1 && !m.bound;
  const bool wd_ok = use_ws && D <= kWdMaxD && a.accept_mode == PBX_ACCEPT_LOG;
  if (kernel_variant == 4 && !wd_ok) {
    pbx_set_error("pbx_mh_mvn_run: kernel_variant 4 (whitened-decision kernel) needs the native "
                  "RNG, the log accept rule, no per-step outputs and n_dims <= %d", kWdMaxD);
    return PBX_ERR_UNSUPPORTED;
  }
  const bool fast = a.prop_kind == PBX_PROP_NORMAL && !a.has_L;      // kFast
  bool zero_mean = true;                                               // kZeroMean
  for (int j = 0; j < D; ++j) zero_mean = zero_mean && m.mean[j] == 0.0;
  if constexpr (D <= kWdMaxD) {
    if (wd_ok && kernel_variant != 2) {
      const int cpc = wd_pick_cpc(a.C, ctx->sm_count);
      auto* k = fast ? (zero_mean ? mh_mvn_wd_kernel<D, true, true> : mh_mvn_wd_kernel<D, true, false>)
                     : (zero_mean ? mh_mvn_wd_kernel<D, false, true> : mh_mvn_wd_kernel<D, false, false>);
      return launch_smem(ctx, k, (a.C + cpc - 1) / cpc, WdCfg<D>::THREADS, WdCfg<D>::SMEM, a, m, cpc);
    }
  }
  if (use_ws) {
    auto* k = mh_mvn_ws_kernel<D, false, false, false>;
    if (a.accept_mode == PBX_ACCEPT_REFERENCE)
      k = fast ? mh_mvn_ws_kernel<D, true, true, false> : mh_mvn_ws_kernel<D, true, false, false>;
    else if (fast)
      k = zero_mean ? mh_mvn_ws_kernel<D, false, true, true> : mh_mvn_ws_kernel<D, false, true, false>;
    return launch_smem(ctx, k, (a.C + 31) / 32, WsCfg<D>::THREADS, WsCfg<D>::SMEM, a, m);
  }
  const int warps = (a.C + 31) / 32;
  // few chains: one warp per CTA so the warps spread over all SMs
  const int block = (warps <= ctx->sm_count * 8) ? 32 : 128;
  const int grid = (a.C + block - 1) / block;
  if (injected)
    mh_mvn_kernel<D, true><<<grid, block, 0, ctx->stream>>>(a, m);
  else
    mh_mvn_kernel<D, false><<<grid, block, 0, ctx->stream>>>(a, m);
  PBX_LAUNCH_CHECK(ctx);
  return PBX_OK;
}

static int validate(const pbx_mh_mvn_params* p, const char* who) {
  PBX_REQUIRE(p != nullptr, "%s: null params", who);
  PBX_REQUIRE(p->n_chains >= 1, "%s: n_chains must be >= 1 (got %d)", who, p->n_chains);
  PBX_REQUIRE(p->n_dims >= 1 && p->n_dims <= PBX_MAX_DIMS, "%s: n_dims must be in 1..%d (got %d)",
              who, PBX_MAX_DIMS, p->n_dims);
  PBX_REQUIRE(p->n_steps >= 0, "%s: n_steps must be >= 0", who);
  PBX_REQUIRE(p->thin >= 1, "%s: thin must be >= 1", who);
  PBX_REQUIRE(p->step0 >= 0 && p->chain0 >= 0, "%s: step0/chain0 must be >= 0", who);
  PBX_REQUIRE(p->accept_mode == PBX_ACCEPT_REFERENCE || p->accept_mode == PBX_ACCEPT_LOG,
              "%s: unknown accept_mode %d", who, p->accept_mode);
  PBX_REQUIRE(p->prop_kind >= PBX_PROP_NORMAL && p->prop_kind <= PBX_PROP_SPHERICAL,
              "%s: unknown prop_kind %d", who, p->prop_kind);
  PBX_REQUIRE(p->state && p->state_lp, "%s: state/state_lp are mandatory", who);
  PBX_REQUIRE((p->inj_delta == nullptr) == (p->inj_thresh == nullptr),
              "%s: inj_delta and inj_thresh must be given together", who);
  return PBX_OK;
}

static void fill_const(const pbx_mh_mvn_params* p, MhMvnConst& m) {
  const int D = p->n_dims;
  for (int j = 0; j < PBX_MAX_DIMS; ++j) {
    m.mean[j] = j < D ? p->mean[j] : 0.0;
    m.scale[j] = j < D ? p->prop_scale[j] : 0.0;
  }
  for (int i = 0; i < PBX_MAX_DIMS * PBX_MAX_DIMS; ++i) {
    m.W[i] = i < D * D ? p->whiten[i] : 0.0;
    m.L[i] = i < D * D ? p->prop_mat[i] : 0.0;
  }
  m.norm_c = p->norm_c;
  m.radius = p->prop_radius;
  pbx_make_round_keys(p->seed, m.rk);
  m.bound = p->prop_bound ? 1 : 0;
  for (int j = 0; j < PBX_MAX_DIMS; ++j)
    for (int e = 0; e < 2; ++e) {
      m.lims[j][e] = p->lims[j][e];
      m.open_end[j][e] = p->open_end[j][e];
    }
}

static int run_device(pbx_ctx* ctx, const pbx_mh_mvn_params* p) {
  MhMvnConst m;
  fill_const(p, m);
  MhMvnArgs a;
  a.C = p->n_chains; a.T = p->n_steps; a.thin = p->thin;
  a.step0 = p->step0; a.chain0 = p->chain0; a.seed = p->seed;
  a.log_pscale = p->log_pscale; a.accept_mode = p->accept_mode;
  a.prop_kind = p->prop_kind; a.has_L = p->has_prop_mat;
  a.state = p->state; a.state_lp = p->state_lp;
  a.inj_delta = p->inj_delta; a.inj_thresh = p->inj_thresh;
  a.out_x = p->out_x; a.out_prob = p->out_prob;
  a.out_accept = p->out_accept; a.out_score = p->out_score;
  a.out_xprop = p->out_xprop; a.out_pprop = p->out_pprop;
  a.accept_count = p->accept_count; a.stat_sum = p->stat_sum; a.stat_sumsq = p->stat_sumsq;
  if (a.T == 0) return PBX_OK;
  {
    int rc = init_tables(ctx);
    if (rc) return rc;
  }
  switch (p->n_dims) {
    case 1: return launch_mh_mvn<1>(ctx, a, m, p->kernel_variant);
    case 2: return launch_mh_mvn<2>(ctx, a, m, p->kernel_variant);
    case 3: return launch_mh_mvn<3>(ctx, a, m, p->kernel_variant);
    case 4: return launch_mh_mvn<4>(ctx, a, m, p->kernel_variant);
    case 5: return launch_mh_mvn<5>(ctx, a, m, p->kernel_variant);
    case 6: return launch_mh_mvn<6>(ctx, a, m, p->kernel_variant);
    case 7: return launch_mh_mvn<7>(ctx, a, m, p->kernel_variant);
    case 8: return launch_mh_mvn<8>(ctx, a, m, p->kernel_variant);
  }
  pbx_set_error("pbx_mh_mvn_run: unsupported n_dims %d", p->n_dims);
  return PBX_ERR_UNSUPPORTED;
}

extern "C" int pbx_mh_mvn_run(pbx_ctx* ctx, const pbx_mh_mvn_params* p) {
  PBX_REQUIRE(ctx != nullptr, "pbx_mh_mvn_run: null ctx");
  int rc = validate(p, "pbx_mh_mvn_run");
  if (rc) return rc;
  PBX_CUDA(cudaSetDevice(ctx->device));
  PBX_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
  rc = run_device(ctx, p);
  if (rc) return rc;
  PBX_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
  return PBX_OK;
}

// Whole walk with host buffers: chunks of steps, double-buffered device staging,
// D2H on the copy stream overlapped with the next chunk's kernel.
extern "C" int pbx_mh_mvn_walk_host(pbx_ctx* ctx, const pbx_mh_mvn_params* p,
                                    int32_t chunk_steps) {
  PBX_REQUIRE(ctx != nullptr, "pbx_mh_mvn_walk_host: null ctx");
  int rc = validate(p, "pbx_mh_mvn_walk_host");
  if (rc) return rc;
  PBX_REQUIRE(!p->inj_delta && !p->out_accept && !p->out_score && !p->out_xprop && !p->out_pprop,
              "pbx_mh_mvn_walk_host: injected streams / per-step accept+score outputs are "
              "device-only (use pbx_mh_mvn_run)");
  PBX_CUDA(cudaSetDevice(ctx->device));
  const int64_t C = p->n_chains, D = p->n_dims, T = p->n_steps;
  const int thin = p->thin;
  if (chunk_steps <= 0) chunk_steps = 1024;
  chunk_steps = (chunk_steps + thin - 1) / thin * thin;   // chunk boundaries on record boundaries
  const int64_t rec_per_chunk = chunk_steps / thin;
  const size_t xbytes = p->out_x ? (size_t)rec_per_chunk * D * C * 8 : 0;
  const size_t pbytes = p->out_prob ? (size_t)rec_per_chunk * C * 8 : 0;
  const size_t sbytes = (size_t)D * C * 8;
  // workspace: state, lp, acc, sum, sumsq, 2 x (x chunk, prob chunk)
  size_t off = 0;
  auto take = [&](size_t b) { size_t o = off; off += (b + 255) / 256 * 256; return o; };
  const size_t o_state = take(sbytes), o_lp = take(C * 8), o_acc = take(C * 8),
               o_sum = take(sbytes), o_sq = take(sbytes);
  size_t o_x[2], o_p[2];
  for (int b = 0; b < 2; ++b) { o_x[b] = take(xbytes); o_p[b] = take(pbytes); }
  rc = pbx_ws_reserve(ctx, off);
  if (rc) return rc;
  char* ws = (char*)ctx->ws;
  cudaStream_t st = ctx->stream, cs = ctx->copy_stream;
  PBX_CUDA(cudaMemcpyAsync(ws + o_state, p->state, sbytes, cudaMemcpyHostToDevice, st));
  if (p->step0 > 0)
    PBX_CUDA(cudaMemcpyAsync(ws + o_lp, p->state_lp, C * 8, cudaMemcpyHostToDevice, st));
  PBX_CUDA(cudaMemsetAsync(ws + o_acc, 0, C * 8, st));
  PBX_CUDA(cudaMemsetAsync(ws + o_sum, 0, sbytes, st));
  PBX_CUDA(cudaMemsetAsync(ws + o_sq, 0, sbytes, st));

  cudaEvent_t done[2] = {nullptr, nullptr}, copied[2] = {nullptr, nullptr};
  // every failure below goes through ONE exit that drains both streams (no D2H copy may
  // still be writing into the caller's buffers when we return) and destroys the events
  int status = PBX_OK;
#define PBX_WH(call)                                                              \
  do {                                                                            \
    cudaError_t _e = (call);                                                      \
    if (_e != cudaSuccess && status == PBX_OK) {                                  \
      pbx_set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #call,            \
                    cudaGetErrorString(_e));                                      \
      status = PBX_ERR_CUDA;                                                      \
    }                                                                             \
  } while (0)
  for (int b = 0; b < 2; ++b) {
    PBX_WH(cudaEventCreateWithFlags(&done[b], cudaEventDisableTiming));
    PBX_WH(cudaEventCreateWithFlags(&copied[b], cudaEventDisableTiming));
  }
  PBX_WH(cudaEventRecord(ctx->ev0, st));
  int64_t rec_done = 0;
  int chunk = 0;
  for (int64_t t0 = 0; t0 < T && status == PBX_OK; t0 += chunk_steps, ++chunk) {
    const int b = chunk & 1;
    const int64_t nt = (T - t0 < chunk_steps) ? (T - t0) : chunk_steps;
    const int64_t nrec = nt / thin;
    if (chunk >= 2) PBX_WH(cudaStreamWaitEvent(st, copied[b], 0));
    pbx_mh_mvn_params q = *p;
    q.n_steps = (int32_t)nt;
    q.step0 = p->step0 + t0;
    q.state = (double*)(ws + o_state);
    q.state_lp = (double*)(ws + o_lp);
    q.out_x = p->out_x ? (double*)(ws + o_x[b]) : nullptr;
    q.out_prob = p->out_prob ? (double*)(ws + o_p[b]) : nullptr;
    q.accept_count = (int64_t*)(ws + o_acc);
    q.stat_sum = (double*)(ws + o_sum);
    q.stat_sumsq = (double*)(ws + o_sq);
    if (status == PBX_OK) status = run_device(ctx, &q);
    if (status != PBX_OK) break;
    PBX_WH(cudaEventRecord(done[b], st));
    PBX_WH(cudaStreamWaitEvent(cs, done[b], 0));
    if (p->out_x && nrec)
      PBX_WH(cudaMemcpyAsync(p->out_x + rec_done * D * C, ws + o_x[b], (size_t)nrec * D * C * 8,
                             cudaMemcpyDeviceToHost, cs));
    if (p->out_prob && nrec)
      PBX_WH(cudaMemcpyAsync(p->out_prob + rec_done * C, ws + o_p[b], (size_t)nrec * C * 8,
                             cudaMemcpyDeviceToHost, cs));
    PBX_WH(cudaEventRecord(copied[b], cs));
    rec_done += nrec;
  }
  if (status == PBX_OK) {
    PBX_WH(cudaEventRecord(ctx->ev1, st));
    PBX_WH(cudaMemcpyAsync(p->state, ws + o_state, sbytes, cudaMemcpyDeviceToHost, st));
    PBX_WH(cudaMemcpyAsync(p->state_lp, ws + o_lp, C * 8, cudaMemcpyDeviceToHost, st));
    if (p->accept_count)
      PBX_WH(cudaMemcpyAsync(p->accept_count, ws + o_acc, C * 8, cudaMemcpyDeviceToHost, st));
    if (p->stat_sum)
      PBX_WH(cudaMemcpyAsync(p->stat_sum, ws + o_sum, sbytes, cudaMemcpyDeviceToHost, st));
    if (p->stat_sumsq)
      PBX_WH(cudaMemcpyAsync(p->stat_sumsq, ws + o_sq, sbytes, cudaMemcpyDeviceToHost, st));
  }
  {
    cudaError_t e1 = cudaStreamSynchronize(st), e2 = cudaStreamSynchronize(cs);
    if (status == PBX_OK && (e1 != cudaSuccess || e2 != cudaSuccess)) {
      pbx_set_error("pbx_mh_mvn_walk_host: stream synchronisation failed: %s",
                    cudaGetErrorString(e1 != cudaSuccess ? e1 : e2));
      status = PBX_ERR_CUDA;
    }
  }
#undef PBX_WH
  for (int b = 0; b < 2; ++b) {
    if (done[b]) cudaEventDestroy(done[b]);
    if (copied[b]) cudaEventDestroy(copied[b]);
  }
  return status;
}


// ---------------------------------------------------------------------------
// Self-test hook for the table-driven math of the RNG path (tests/test_gpu_mh_mvn.py
// checks it against libm to a few ulp): u[n] in (0, 1), w[n] raw 32-bit words ->
// out[0][n] = -2 log(u), out[1][n] = sqrt(-2 log u), out[2][n] = sin(2 pi (w + .5)/2^32),
// out[3][n] = cos(same), out[4][n] = exp(-700 u).
// ---------------------------------------------------------------------------
__global__ void fastmath_selftest_kernel(const double* __restrict__ u, const uint32_t* __restrict__ w,
                                         int64_t n, double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double l = fast_neg2log(u[i], &g_tables);
  double sn, cs;
  fast_sincos2pi(w[i], &g_tables, sn, cs);
  out[i] = l;
  out[n + i] = fast_sqrt(fmax(l, PBX_TINY));
  out[2 * n + i] = sn;
  out[3 * n + i] = cs;
  out[4 * n + i] = fast_exp(-700.0 * u[i], &g_tables);
}

extern "C" int pbx_selftest_fastmath(pbx_ctx* ctx, const double* u, const uint32_t* w, int64_t n,
                                     double* out) {
  PBX_REQUIRE(ctx && u && w && out && n >= 0, "pbx_selftest_fastmath: bad argument");
  if (n == 0) return PBX_OK;
  PBX_CUDA(cudaSetDevice(ctx->device));
  int rc = init_tables(ctx);
  if (rc) return rc;
  fastmath_selftest_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(u, w, n, out);
  PBX_LAUNCH_CHECK(ctx);
  return PBX_OK;
}
