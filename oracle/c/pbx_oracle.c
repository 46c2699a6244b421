/*
 * pbx_oracle.c -- plain C (+OpenMP) restatement of the probayes hot path.
 * TEST INFRASTRUCTURE, NOT PRODUCT: only tests/, __graft_entry__.smoke() and the
 * cpu_baseline / --impl reference legs of bench.py may load this.  It exists to
 * (a) time the reference's algorithm on all host cores and (b) give a second,
 * independent opinion on oracle/np_oracle.py.  Paths cited are relative to the
 * reference checkout.
 *
 * RNG: Philox4x32-10 with the stream layout of oracle/philox.py.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define TINY 2.2250738585072014e-308
#define HUGE_P 1.7976931348623158e+308
#define LOG_HUGE 709.782712893384
#define LOG_SQRT_2PI 0.91893853320467274178

/* probayes/pscales.py:44-65 */
static inline double log_prob(double p) { return p >= TINY ? log(p) : -HUGE_P; }
static inline double exp_logp(double l) { return l <= LOG_HUGE ? exp(l) : HUGE_P; }

static inline void philox(uint32_t c[4], uint32_t k0, uint32_t k1) {
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c[0], p1 = (uint64_t)0xCD9E8D57u * c[2];
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1;
    c[1] = (uint32_t)p1; c[3] = (uint32_t)p0; c[0] = n0; c[2] = n2;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
}
static inline void block(uint64_t seed, uint64_t step, uint32_t chain, uint32_t slot,
                         uint32_t w[4]) {
  w[0] = (uint32_t)step; w[1] = (uint32_t)(step >> 32); w[2] = chain; w[3] = slot;
  philox(w, (uint32_t)seed, (uint32_t)(seed >> 32));
}
/* stream layout of oracle/philox.py: u52 / u32 / t44 */
static inline double u52(uint32_t w0, uint32_t w1) {
  uint64_t k = ((uint64_t)w0 << 20) | (uint64_t)(w1 >> 12);
  return (double)(2 * k + 1) * 1.1102230246251565e-16;          /* 2^-53 */
}
static inline double u32(uint32_t w2) {
  return (double)(2 * (uint64_t)w2 + 1) * 1.1641532182693481e-10; /* 2^-33 */
}
static inline double t44(uint32_t w3, uint32_t w1) {
  uint64_t k = ((uint64_t)w3 << 12) | (uint64_t)(w1 & 0xfffu);
  return (double)(2 * k + 1) * 2.8421709430404007e-14;           /* 2^-45 */
}
static inline void sincospi_(double x, double* s, double* c) {   /* x in (0, 2) */
  double n = rint(2.0 * x);
  double r = (x - 0.5 * n) * M_PI;
  double sr = sin(r), cr = cos(r);
  switch (((long)n) & 3) {
    case 0: *s = sr; *c = cr; break;
    case 1: *s = cr; *c = -sr; break;
    case 2: *s = -sr; *c = -cr; break;
    default: *s = -cr; *c = sr; break;
  }
}
static inline void normal_pair(const uint32_t w[4], double* z0, double* z1) {
  double u1 = u52(w[0], w[1]), u2 = u32(w[2]);
  double r = sqrt(-2.0 * log(u1)), s, c;
  sincospi_(2.0 * u2, &s, &c);
  *z0 = r * c; *z1 = r * s;
}

void orc_set_num_threads(int n) {
#ifdef _OPENMP
  if (n > 0) omp_set_num_threads(n);
#else
  (void)n;
#endif
}

int orc_num_threads(void) {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}

/* scipy multivariate_normal_gen._logpdf: -0.5*(d log 2pi + log_pdet + |dev U|^2) */
static inline double mvn_logpdf(const double* x, int D, const double* mean, const double* W,
                                double norm_c) {
  double maha = 0.0;
  for (int k = 0; k < D; ++k) {
    double y = 0.0;
    for (int j = 0; j < D; ++j) y += (x[j] - mean[j]) * W[j * D + k];
    maha += y * y;
  }
  return -0.5 * (norm_c + maha);
}

/*
 * MH step loop on an mvn target (probayes/sp.py:221-258, sp_utils.py:19-37,
 * pscales.py:219-236), native Philox draws, normal additive proposal with
 * per-dimension scale.  mean/W are in natural variable order with the value
 * permutation of prob.py:349-358 already folded in by the caller.
 * init [C][D]; out_x [T][D][C] / out_prob [T][C] (chain-minor, like the device) or NULL.
 * accept_mode 0 = reference linear ratio, 1 = log space.
 */
void orc_mh_mvn_walk(int C, int D, int T, const double* init, const double* mean,
                     const double* W, double norm_c, const double* scale, uint64_t seed,
                     int64_t step0, int64_t chain0, int log_pscale, int accept_mode,
                     double* out_x, double* out_prob, uint8_t* out_accept, double* final_x,
                     int64_t* accept_count) {
#pragma omp parallel for schedule(static)
  for (int c = 0; c < C; ++c) {
    double x[8], xp[8], dl[8];
    for (int j = 0; j < D; ++j) x[j] = init[(size_t)c * D + j];
    double lp = 0.0, lin = 0.0;
    int64_t nacc = 0;
    uint32_t gchain = (uint32_t)(chain0 + c);
    for (int k = 0; k < T; ++k) {
      uint64_t gstep = (uint64_t)(step0 + k);
      uint32_t w[4];
      double t = 0.0;
      for (int s = 0; s < (D + 1) / 2; ++s) {
        double z0, z1;
        block(seed, gstep, gchain, (uint32_t)s, w);
        normal_pair(w, &z0, &z1);
        if (s == 0) t = t44(w[3], w[1]);
        dl[2 * s] = z0 * scale[2 * s];
        if (2 * s + 1 < D) dl[2 * s + 1] = z1 * scale[2 * s + 1];
      }
      for (int j = 0; j < D; ++j) xp[j] = x[j] + dl[j];
      double lpp = mvn_logpdf(xp, D, mean, W, norm_c);
      int acc;
      double linp = 0.0;
      if (accept_mode == 0) {
        linp = log_pscale ? exp_logp(lpp) : exp(lpp);
        if (gstep == 0) acc = 1;
        else {
          double s = fmin(1.0, linp / fmax(TINY, lin));
          acc = s >= t;
        }
      } else {
        acc = (gstep == 0) ? 1 : ((lpp - lp) >= log(t));
      }
      if (acc) {
        for (int j = 0; j < D; ++j) x[j] = xp[j];
        lp = lpp; lin = linp; ++nacc;
      }
      if (out_accept) out_accept[(size_t)k * C + c] = (uint8_t)acc;
      if (out_x)
        for (int j = 0; j < D; ++j) out_x[((size_t)k * D + j) * C + c] = x[j];
      if (out_prob)
        out_prob[(size_t)k * C + c] = log_pscale ? lp : (accept_mode == 0 ? lin : exp(lp));
    }
    if (final_x)
      for (int j = 0; j < D; ++j) final_x[(size_t)c * D + j] = x[j];
    if (accept_count) accept_count[c] = nacc;
  }
}

/*
 * iid normal log-likelihood + box priors (probayes/rf.py:541-581, pd.py:332-370,
 * sd.py:154-161, rv_utils.py:8-47), scipy.stats.norm.logpdf per term:
 *   -(z*z)/2 - log(sqrt(2 pi)) - log(sigma),   z = (y - loc)/sigma
 * theta [C][P] (P = 2: mu, sigma; P = 3: b0, b1, sigma).  out [C].
 */
void orc_normreg_logjoint(int C, int P, const double* theta, int64_t N, const double* x_obs,
                          const double* y_obs, const double* lims, const int32_t* open_end,
                          const int32_t* log_ufun, double* out) {
#pragma omp parallel for schedule(dynamic, 1)
  for (int c = 0; c < C; ++c) {
    const double* th = theta + (size_t)c * P;
    double b0 = th[0], b1 = (P == 3) ? th[1] : 0.0, sg = th[P - 1];
    double lsg = log(sg), acc = 0.0;
    for (int64_t i = 0; i < N; ++i) {
      double loc = (P == 3) ? b0 + b1 * x_obs[i] : b0;
      double z = (y_obs[i] - loc) / sg;
      acc += -(z * z) / 2.0 - LOG_SQRT_2PI - lsg;
    }
    double prior = 0.0;
    for (int j = 0; j < P; ++j) {
      double lo = lims[2 * j], hi = lims[2 * j + 1], v = th[j];
      int in_lo = open_end[2 * j] ? (v > lo) : (v >= lo);
      int in_hi = open_end[2 * j + 1] ? (v < hi) : (v <= hi);
      double len = log_ufun[j] ? log(hi) - log(lo) : hi - lo;
      prior += (in_lo && in_hi) ? -log(len) : -HUGE_P;
    }
    out[c] = prior + acc;
  }
}

/*
 * DGEI log-joint [M][S] (probayes/rf.py:565-581, pd.py:368, pd_utils.py:85-328):
 * sequential sum over observations of norm.logpdf, then + priors.
 */
void orc_grid_norm_logjoint(int64_t N, const double* x_obs, int M, const double* mu, int S,
                            const double* sigma, const double* lp_mu, const double* lp_sigma,
                            double* out) {
#pragma omp parallel for schedule(static)
  for (int m = 0; m < M; ++m) {
    for (int s = 0; s < S; ++s) {
      double sg = sigma[s], lsg = log(sg), acc = 0.0;
      for (int64_t i = 0; i < N; ++i) {
        double z = (x_obs[i] - mu[m]) / sg;
        acc += -(z * z) / 2.0 - LOG_SQRT_2PI - lsg;
      }
      out[(size_t)m * S + s] = (lp_mu[m] + lp_sigma[s]) + acc;
    }
  }
}

/* PD.conditionalise + PD.marginal in log pscale (probayes/pd.py:285-295,162-164) */
void orc_grid_posterior(int M, int S, const double* lj, double* post, double* marg_mu,
                        double* marg_sigma) {
  size_t n = (size_t)M * S;
  double mx = lj[0];
  for (size_t i = 1; i < n; ++i) mx = lj[i] > mx ? lj[i] : mx;
  double sum = 0.0;
  for (size_t i = 0; i < n; ++i) sum += exp_logp(lj[i] - mx);
  double den = fmax(TINY, sum);
  for (size_t i = 0; i < n; ++i) post[i] = log_prob(exp_logp(lj[i] - mx) / den);
  for (int m = 0; m < M; ++m) {
    double a = 0.0;
    for (int s = 0; s < S; ++s) a += exp_logp(post[(size_t)m * S + s]);
    marg_mu[m] = log_prob(a);
  }
  for (int s = 0; s < S; ++s) {
    double a = 0.0;
    for (int m = 0; m < M; ++m) a += exp_logp(post[(size_t)m * S + s]);
    marg_sigma[s] = log_prob(a);
  }
}

/* inverse normal cdf: Acklam's rational start + two Halley steps on erfc => ~1 ulp.  Upper half
 * by symmetry: 1 - p is exact there, while a Halley residual formed against p itself keeps only
 * the absolute precision of p (~1e-16), i.e. ~1e-16 / pdf(x) in x (1e-10 at x = 5). */
static double ndtri_(double p) {
  if (p > 0.5) return -ndtri_(1.0 - p);
  static const double a[] = {-3.969683028665376e+01, 2.209460984245205e+02, -2.759285104469687e+02,
                             1.383577518672690e+02, -3.066479806614716e+01, 2.506628277459239e+00};
  static const double b[] = {-5.447609879822406e+01, 1.615858368580409e+02, -1.556989798598866e+02,
                             6.680131188771972e+01, -1.328068155288572e+01};
  static const double c[] = {-7.784894002430293e-03, -3.223964580411365e-01, -2.400758277161838e+00,
                             -2.549732539343734e+00, 4.374664141464968e+00, 2.938163982698783e+00};
  static const double d[] = {7.784695709041462e-03, 3.224671290700398e-01, 2.445134137142996e+00,
                             3.754408661907416e+00};
  double q, r, x;
  if (p <= 0.0) return -INFINITY;
  if (p >= 1.0) return INFINITY;
  if (p < 0.02425) {
    q = sqrt(-2 * log(p));
    x = (((((c[0] * q + c[1]) * q + c[2]) * q + c[3]) * q + c[4]) * q + c[5]) /
        ((((d[0] * q + d[1]) * q + d[2]) * q + d[3]) * q + 1);
  } else if (p > 1 - 0.02425) {
    q = sqrt(-2 * log(1 - p));
    x = -(((((c[0] * q + c[1]) * q + c[2]) * q + c[3]) * q + c[4]) * q + c[5]) /
        ((((d[0] * q + d[1]) * q + d[2]) * q + d[3]) * q + 1);
  } else {
    q = p - 0.5; r = q * q;
    x = (((((a[0] * r + a[1]) * r + a[2]) * r + a[3]) * r + a[4]) * r + a[5]) * q /
        (((((b[0] * r + b[1]) * r + b[2]) * r + b[3]) * r + b[4]) * r + 1);
  }
  for (int it = 0; it < 2; ++it) {
    double e = 0.5 * erfc(-x / M_SQRT2) - p;
    double u = e * sqrt(2 * M_PI) * exp(x * x / 2);
    x = x - u / (1 + x * u / 2);
  }
  return x;
}

/*
 * CondCov Gibbs (probayes/cond_cov.py:42-65 via rf.py:446-462): one coordinate
 * per step, coordinate = (step0 + k) mod d, native Philox uniforms (slot 0, two steps per
 * block).
 * x [C][d] in/out; coef [d][d] with zero diagonal.
 */
void orc_gibbs_mvn_walk(int C, int d, int T, double* x, const double* mean, const double* coef,
                        const double* stdv, const double* cdf_lo, const double* cdf_hi,
                        uint64_t seed, int64_t step0, int64_t chain0, const double* inj_runif) {
#pragma omp parallel for schedule(static)
  for (int c = 0; c < C; ++c) {
    double* xc = x + (size_t)c * d;
    for (int k = 0; k < T; ++k) {
      int i = (int)((step0 + k) % d);
      double r;
      if (inj_runif) r = inj_runif[(size_t)k * C + c];
      else {
        /* steps g and g + 4 share Philox block (seed, g & ~4, chain, 0): words (0, 1) when
         * bit 2 of g is clear, (2, 3) when it is set (pbx_gibbs.cu header) */
        uint32_t w[4];
        const uint64_t g = (uint64_t)(step0 + k);
        block(seed, g & ~(uint64_t)4, (uint32_t)(chain0 + c), 0u, w);
        r = (g & 4) ? u52(w[2], w[3]) : u52(w[0], w[1]);
      }
      double u = cdf_lo[i] + (cdf_hi[i] - cdf_lo[i]) * r;
      double cm = mean[i];
      for (int j = 0; j < d; ++j) cm += coef[(size_t)i * d + j] * (xc[j] - mean[j]);
      xc[i] = ndtri_(u) * stdv[i] + cm;
    }
  }
}
