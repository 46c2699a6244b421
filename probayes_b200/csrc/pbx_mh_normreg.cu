// pbx_mh_normreg.cu -- K2: streaming normal log-likelihood Metropolis-Hastings.
//
// Target (log pscale, iid=True, joint=True):
//   log p(theta, data) = sum_j boxprior_j(theta_j) + sum_i lik.logpdf(y_i; loc_i, sigma)
//   loc_i = b0 + b1 x_i (has_slope, theta = (b0, b1, sigma)) or mu (theta = (mu, sigma))
//   lik = norm, or t with nu degrees of freedom (kLik; cauchy = t with nu = 1), whose sum is
//   N logc - N log sigma - (nu+1)/2 sum_i log1p(r_i^2 / (nu sigma^2)), logc from the host;
//   or that t with nu sampled (PBX_LIK_STUDENT_T_NU, theta = (mu, sigma, nu)), logc(nu) on
//   the device (nr_t_logc)
// following probayes/rf.py:541-581, pd.py:332-370 (iid product = sum over the
// observation axis), sd.py:154-161 + rf_utils.py:10-22 + rv_utils.py:8-47 (product
// with the independent box priors, prior first), scipy.stats.norm.logpdf per term,
// proposals in ufun space (variable.py:693-697) and the accept rule of
// sp_utils.py:19-64 / pscales.py:219-236.
//
// One MH step = ONE kernel launch:
//   phase A  every CTA accumulates S_c = sum_i (y_i - loc_i)^2 (Student-t: the log1p sum)
//            over its slice of the observations for its chains and writes a partial sum;
//   phase B  the last CTA to finish (per chain group) reduces the partials in a
//            fixed order, adds -N(log sqrt(2pi) + log sigma) and the priors, runs
//            the accept test, records the sample and draws the NEXT proposal.
// Two phase-A kernels:
//   tiles  (many chains)  chains live in registers (KC per thread); observation
//          tiles are staged into shared memory with 1-D TMA bulk copies behind a
//          3-stage mbarrier pipeline and read back as 128-bit broadcast loads, so
//          every observation byte is fetched once per CTA and used by 128*KC chains.
//   stream (<= 8 chains)  one pass over HBM: every thread reads observations with
//          128-bit coalesced loads, updates all chains' sums, warp-shuffle + block
//          reduce.  This is the HBM-roofline regime (16 B per observation per step).
#include <math.h>
#include <string.h>
#include <algorithm>
#include "pbx_common.cuh"

#define NR_TILE 1024          // observations per shared-memory tile (tiles kernel: 48 KB/CTA)
#define NR_STAGES 3
#define NRS_TILE 2048         // stream kernel tile (96 KB/CTA -> ~190 KB in flight per SM)
#define NR_THREADS 128
#define NR_SMAX 8             // chains per pass of the streaming kernel

struct NrModel {
  int P, has_slope, accept_mode, prop_kind, bound;
  double coef;
  double lims[PBX_MAX_PARAMS][2];
  int open_end[PBX_MAX_PARAMS][2];
  int log_ufun[PBX_MAX_PARAMS];
  double scale[PBX_MAX_PARAMS];
  double nlhv[PBX_MAX_PARAMS];      // -log(length in ufun space): rv.py:153-166
  double radius;
  int has_L;                        // colour the delta with L (set_tran(covariance))
  double L[PBX_MAX_PARAMS][PBX_MAX_PARAMS];   // lower-triangular, zero outside [P][P]
};

// the Student-t likelihood of a call (PBX_LIK_STUDENT_T; unread by the normal and the
// sampled-nu instantiations).
// A kernel argument of its own, after the others, so that the normal kernels' argument
// offsets -- and with them their SASS -- are those of the normal-only build
struct NrLik {
  double df;                   // nu
  double logc;                 // log(poch(nu/2, 1/2)) - (log nu + log pi)/2, from the host
};

struct NrArgs {
  int C;
  int64_t N;
  const double* x;
  const double* y;
  int n_slices;                // partial sums per chain
  double* partial;             // [n_slices][C]
  unsigned int* counters;      // one per chain group, zero between launches
  const double* theta_in;      // [P][C] parameters to evaluate (the proposal)
  // ---- phase B (MH) ----
  int mode;                    // 0 = MH step, 1 = evaluate only (write logjoint to eval_out)
  double* eval_out;            // [C]
  double* prop;                // [P][C] next proposal (written by phase B)
  double* state;               // [P][C]
  double* state_lp;            // [C]
  int64_t gstep;               // global index of THIS step
  int64_t step0;
  int k;                       // index of this step within the call
  int T, thin;
  int64_t chain0;
  uint64_t seed;
  const double* inj_delta;     // [T][P][C]
  const double* inj_thresh;    // [T][C]
  double* out_x;
  double* out_prob;
  uint8_t* out_accept;
  double* out_score;
  double* out_xprop;
  double* out_pprop;
  int64_t* accept_count;
  double* stat_sum;
  double* stat_sumsq;
};

// ----------------------------------------------------------------------------
// proposal: theta' = ufun^-1(ufun(theta) + L delta)  (variable.py:693-697, rf.py:346-348)
// ----------------------------------------------------------------------------
// delta <- L delta for a lower-triangular L, in place: row i reads entries j <= i only, so
// the rows are taken from the last to the first
__device__ __forceinline__ void nr_colour(const NrModel& m, int P, double (&dl)[PBX_MAX_PARAMS]) {
#pragma unroll
  for (int i = PBX_MAX_PARAMS - 1; i >= 0; --i) {
    if (i >= P) continue;
    double acc = 0.0;
#pragma unroll
    for (int j = 0; j <= i; ++j) acc = fma(m.L[i][j], dl[j], acc);
    dl[i] = acc;
  }
}

// kP: the parameter count at compile time (0 = read m.P): with it every index below is a
// constant and the arrays stay in registers (runtime bounds put them into local memory, which
// only the one-launch walk kernel -- a latency-bound chain per warp -- cares about).
// The raw draw (injected, or Philox scaled / spherically rescaled) is coloured last, as the
// reference multiplies its delta draw by the Cholesky factor of set_tran(covariance).
// kColour = false compiles the colouring out (see nr_move for why the kernels care)
template <int kP = 0, bool kColour = true>
__device__ __forceinline__ void nr_draw_delta(const NrArgs& a, const NrModel& m, int64_t gstep,
                                              int kk, int c, double (&dl)[PBX_MAX_PARAMS]) {
  const int64_t C = a.C;
  const int P = kP ? kP : m.P;
  if (a.inj_delta) {
#pragma unroll
    for (int j = 0; j < PBX_MAX_PARAMS; ++j)
      if (j < P) dl[j] = a.inj_delta[((int64_t)kk * P + j) * C + c];
  } else {
    const uint32_t gchain = (uint32_t)(a.chain0 + c);
#pragma unroll
    for (int s = 0; s < (PBX_MAX_PARAMS + 1) / 2; ++s) {
      if (s >= (P + 1) / 2) break;
      pbx_u4 w = pbx_block(a.seed, (uint64_t)gstep, gchain, (uint32_t)s);
      double d0, d1;
      if (m.prop_kind == PBX_PROP_NORMAL) {
        pbx_normal_pair(w, d0, d1);
        d0 *= m.scale[2 * s];
        if (2 * s + 1 < P) d1 *= m.scale[2 * s + 1];
      } else if (m.prop_kind == PBX_PROP_UNIFORM) {
        d0 = -m.scale[2 * s] + (2.0 * m.scale[2 * s]) * pbx_u52(w.x, w.y);
        d1 = (2 * s + 1 < P) ? -m.scale[2 * s + 1] + (2.0 * m.scale[2 * s + 1]) * pbx_u32(w.z)
                               : 0.0;
      } else {                       // spherical: cube sample, rescaled below
        d0 = -m.radius + (2.0 * m.radius) * pbx_u52(w.x, w.y);
        d1 = (2 * s + 1 < P) ? -m.radius + (2.0 * m.radius) * pbx_u32(w.z) : 0.0;
      }
      dl[2 * s] = d0;
      if (2 * s + 1 < P) dl[2 * s + 1] = d1;
    }
    if (m.prop_kind == PBX_PROP_SPHERICAL) {   // field.py:509-531
      double ss = 0.0;
#pragma unroll
      for (int j = 0; j < PBX_MAX_PARAMS; ++j)
        if (j < P) ss += dl[j] * dl[j];
      const double nrm = (ss >= PBX_TINY) ? sqrt(ss) : 0.0;
#pragma unroll
      for (int j = 0; j < PBX_MAX_PARAMS; ++j)
        if (j < P) dl[j] = ((dl[j] * m.radius) / nrm) * m.scale[j];
    }
  }
  if (kColour && m.has_L) nr_colour(m, P, dl);
}

__device__ __forceinline__ double nr_threshold(const NrArgs& a, int64_t gstep, int kk, int c) {
  if (a.inj_thresh) return a.inj_thresh[(int64_t)kk * a.C + c];
  pbx_u4 w = pbx_block(a.seed, (uint64_t)gstep, (uint32_t)(a.chain0 + c), 0u);
  return pbx_t44(w.w, w.y);
}

// ----------------------------------------------------------------------------
// one MH step, shared by every walk path: only the likelihood sum differs between them
// ----------------------------------------------------------------------------
// coordinate j of the proposal: ufun^-1(ufun(th) + dl) (variable.py:693-697), then the bound
// rule.  kBound = false compiles the bound rule out: the one-launch-per-step kernels pass their
// kExtras there (and to nr_draw_delta's kColour), so that the rarely used per-step extras
// (bounded or coloured deltas, proposal outputs) never perturb the register allocation of the
// hot likelihood loops of the common configuration (a 9 % effect when it happened)
template <bool kBound>
__device__ __forceinline__ double nr_move(const NrModel& m, int j, double th, double dl) {
  const double v = m.log_ufun[j] ? exp(log(th) + dl) : th + dl;
  if (!kBound || !m.bound) return v;
  return pbx_bound(v, th, m.lims[j][0], m.lims[j][1], m.open_end[j][0] != 0,
                   m.open_end[j][1] != 0);
}

// accept decision for the proposal's log-joint lpp against the current lp and threshold t
// (sp_utils.py:19-64 / pscales.py:219-236); logt() gives log(t) and is called under the log
// rule only.  Global step 0 always accepts (sp.py:253, sp_utils.py:24-25), with score NaN;
// the log rule computes its score only when want_score
template <class LogT>
__device__ __forceinline__ bool nr_decide(const NrModel& m, double lpp, double lp, double t,
                                          LogT logt, int64_t gstep, bool want_score, double& s) {
  bool acc;
  s = nan("");
  if (gstep == 0) {
    acc = true;
  } else if (m.accept_mode == PBX_ACCEPT_REFERENCE) {
    // hastings_scores multiplies the linear proposal density into the LOG target
    // (sp_utils.py:62-64); coef = 1 for metropolis
    const double num = pbx_exp_logp(lpp * m.coef), den = pbx_exp_logp(lp * m.coef);
    s = fmin(1.0, num / fmax(PBX_TINY, den));
    acc = (s >= t);
  } else {
    const double d = m.coef * (lpp - lp);
    acc = (d >= logt());
    if (want_score) s = fmin(1.0, exp(fmin(d, 0.0)));
  }
  return acc;
}

// per-step outputs of step k (decision, score, proposal thp and its lpp) and, every thin-th
// step, the record of the state th / lp after it; kExtras = false leaves out the proposal
template <bool kExtras, int kP = 0>
__device__ __forceinline__ void nr_record(const NrArgs& a, const NrModel& m, int k, int c,
                                          bool acc, double s, const double* thp, double lpp,
                                          const double* th, double lp) {
  const int64_t C = a.C;
  const int P = kP ? kP : m.P;
  if (a.out_accept) a.out_accept[(int64_t)k * C + c] = acc ? 1 : 0;
  if (a.out_score) a.out_score[(int64_t)k * C + c] = s;
  if (kExtras && a.out_xprop)
    for (int j = 0; j < P; ++j) a.out_xprop[((int64_t)k * P + j) * C + c] = thp[j];
  if (kExtras && a.out_pprop) a.out_pprop[(int64_t)k * C + c] = lpp;
  if ((k + 1) % a.thin == 0) {
    const int64_t r = (k + 1) / a.thin - 1;
    if (a.out_x)
      for (int j = 0; j < P; ++j) a.out_x[(r * P + j) * C + c] = th[j];
    if (a.out_prob) a.out_prob[r * C + c] = lp;
  }
}

// end of a one-launch walk: the state, its log-joint, the running sums and the accept count
template <int kP = 0>
__device__ __forceinline__ void nr_write_back(const NrArgs& a, const NrModel& m, int c,
                                              const double* th, double lp, const double* ssum,
                                              const double* ssq, int64_t nacc) {
  const int64_t C = a.C;
  const int P = kP ? kP : m.P;
  for (int j = 0; j < P; ++j) {
    a.state[(int64_t)j * C + c] = th[j];
    if (a.stat_sum) a.stat_sum[(int64_t)j * C + c] += ssum[j];
    if (a.stat_sumsq) a.stat_sumsq[(int64_t)j * C + c] += ssq[j];
  }
  a.state_lp[c] = lp;
  if (a.accept_count) a.accept_count[c] += nacc;
}

// proposal of step kk (global step gstep) of chain c from its state th, into a.prop
template <bool kExtras>
__device__ __forceinline__ void nr_propose(const NrArgs& a, const NrModel& m, int64_t gstep,
                                           int kk, int c, const double* th) {
  double dl[PBX_MAX_PARAMS];
  nr_draw_delta<0, kExtras>(a, m, gstep, kk, c, dl);
  for (int j = 0; j < m.P; ++j)
    a.prop[(int64_t)j * a.C + c] = nr_move<kExtras>(m, j, th[j], dl[j]);
}

// one observation's term of the likelihood sum, residual r: r^2 (normal), or
// log1p(r^2 q) with q = 1/(nu sigma^2) (Student-t, nu fixed or sampled)
template <int kLik>
__device__ __forceinline__ double nr_term(double acc, double r, double q) {
  if (kLik != PBX_LIK_NORMAL) return acc + log1p((r * r) * q);
  return fma(r, r, acc);
}

// q of nr_term for scale sg and nu degrees of freedom
__device__ __forceinline__ double nr_q(double sg, double nu) { return 1.0 / (nu * (sg * sg)); }

// theta index of sigma: the last parameter, but for the sampled-nu t's (mu, sigma, nu)
template <int kLik, bool kSlope>
constexpr int nr_isg() { return kLik == PBX_LIK_STUDENT_T_NU ? 1 : (kSlope ? 2 : 1); }

// logc(nu) = lgamma((nu+1)/2) - lgamma(nu/2) - log(nu pi)/2, the per-observation constant of
// the t density, for a sampled nu, as R(z) - log sqrt(2 pi) with z = nu/2 and
// R(z) = lgamma(z + 1/2) - lgamma(z) - log(z)/2.  Below z = 8 the lgamma difference (both
// terms < 10 there); from z = 8 on the asymptotic series R(z) = sum_k c_k z^-k over odd k,
// c_k = -(2 - 2^-k) B_{k+1} / (k (k+1)) (B: Bernoulli), up to k = 17 (the first term left out
// is < 2e-17 at z = 8).  The series never cancels, where the lgamma difference would at large nu
// (which is why the host's t_logc uses poch), and R -> -1/(8z) -> 0 gives the normal's constant
// as nu -> inf.  Within 1.2e-15 absolute of mpmath over nu in [1e-3, 1e12], measured on a B200
// (tests/test_gpu_studentt_nu.py).  nu <= 0 gives NaN, as scipy's t.logpdf does.
// Once per chain and step.  __noinline__: inlined, the lgamma calls kept the epilogue's state
// live across libm's subroutine calls and spilled it in the tiles and stream kernels.
__device__ __noinline__ double nr_t_logc(double nu) {
  const double z = 0.5 * nu;
  double R;
  if (z < 8.0) {
    R = lgamma(z + 0.5) - lgamma(z) - 0.5 * log(z);
  } else {
    const double w = 1.0 / (z * z);
    double s = -3202291.0 / 8912896.0;                    // c_17
    s = fma(s, w, 929569.0 / 15728640.0);                 // c_15
    s = fma(s, w, -5461.0 / 425984.0);                    // c_13
    s = fma(s, w, 691.0 / 180224.0);                      // c_11
    s = fma(s, w, -31.0 / 18432.0);                       // c_9
    s = fma(s, w, 17.0 / 14336.0);                        // c_7
    s = fma(s, w, -1.0 / 640.0);                          // c_5
    s = fma(s, w, 1.0 / 192.0);                           // c_3
    s = fma(s, w, -0.125);                                // c_1
    R = s / z;
  }
  return R - PBX_LOG_SQRT_2PI;
}

// log-joint from the likelihood sum S (see file header; for Student-t S = sum log1p(z^2/nu))
template <int kP = 0, int kLik = PBX_LIK_NORMAL>
__device__ __forceinline__ double nr_logjoint(const NrArgs& a, const NrModel& m, const double* th,
                                              double S, const NrLik& lik = NrLik{}) {
  const int P = kP ? kP : m.P;
  const double sg = kLik == PBX_LIK_STUDENT_T_NU ? th[1] : th[P - 1];
  const double n = (double)a.N;
  double ll;
  if constexpr (kLik == PBX_LIK_STUDENT_T_NU) {
    const double nu = th[2];
    ll = -(0.5 * (nu + 1.0)) * S + n * (nr_t_logc(nu) - log(sg));
  } else if (kLik == PBX_LIK_STUDENT_T)
    ll = -(0.5 * (lik.df + 1.0)) * S + n * (lik.logc - log(sg));
  else
    ll = -(S / (sg * sg)) * 0.5 - n * (PBX_LOG_SQRT_2PI + log(sg));
  double prior = 0.0;
#pragma unroll
  for (int j = 0; j < PBX_MAX_PARAMS; ++j) {
    if (j >= P) break;
    const double v = th[j];
    const bool in_lo = m.open_end[j][0] ? (v > m.lims[j][0]) : (v >= m.lims[j][0]);
    const bool in_hi = m.open_end[j][1] ? (v < m.lims[j][1]) : (v <= m.lims[j][1]);
    prior += (in_lo && in_hi) ? m.nlhv[j] : -PBX_HUGE;
  }
  return prior + ll;
}

// phase B for one chain: S is the complete residual sum of squares of the proposal
template <bool kExtras, int kLik>
__device__ void nr_phase_b(const NrArgs& a, const NrModel& m, int c, double S, const NrLik& lik) {
  const int64_t C = a.C;
  double thp[PBX_MAX_PARAMS];
  for (int j = 0; j < m.P; ++j) thp[j] = a.theta_in[(int64_t)j * C + c];
  const double lpp = nr_logjoint<0, kLik>(a, m, thp, S, lik);
  if (a.mode == 1) {
    a.eval_out[c] = lpp;
    return;
  }
  double th[PBX_MAX_PARAMS];
  for (int j = 0; j < m.P; ++j) th[j] = a.state[(int64_t)j * C + c];
  double lp = a.state_lp[c];
  const double t = nr_threshold(a, a.gstep, a.k, c);
  double s;
  const bool acc = nr_decide(m, lpp, lp, t, [&] { return log(t); }, a.gstep,
                             a.out_score != nullptr, s);
  if (acc) {
    for (int j = 0; j < m.P; ++j) {
      th[j] = thp[j];
      a.state[(int64_t)j * C + c] = thp[j];
    }
    lp = lpp;
    a.state_lp[c] = lpp;
    if (a.accept_count) a.accept_count[c] += 1;
  }
  for (int j = 0; j < m.P; ++j) {
    if (a.stat_sum) a.stat_sum[(int64_t)j * C + c] += th[j];
    if (a.stat_sumsq) a.stat_sumsq[(int64_t)j * C + c] = fma(th[j], th[j], a.stat_sumsq[(int64_t)j * C + c]);
  }
  nr_record<kExtras>(a, m, a.k, c, acc, s, thp, lpp, th, lp);
  // draw the proposal of the NEXT step (none after the last step of the call)
  if (a.k + 1 < a.T) nr_propose<kExtras>(a, m, a.gstep + 1, a.k + 1, c, th);
}

// first proposal of a call, from the current state
template <bool kExtras>
__global__ void __launch_bounds__(256) nr_init_kernel(const NrArgs a, const __grid_constant__ NrModel m) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= a.C) return;
  double th[PBX_MAX_PARAMS];
  for (int j = 0; j < m.P; ++j) th[j] = a.state[(int64_t)j * a.C + c];
  nr_propose<kExtras>(a, m, a.step0, 0, c, th);
}

// "last CTA of the group" election; returns true in the CTA that arrives last
__device__ __forceinline__ bool nr_arrive_last(unsigned int* counter, unsigned int expected) {
  __shared__ int s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int old = atomicAdd(counter, 1u);
    s_last = (old == expected - 1);
    if (s_last) *counter = 0;                              // ready for the next launch
  }
  __syncthreads();
  if (s_last) __threadfence();
  return s_last != 0;
}

// ----------------------------------------------------------------------------
// phase A, "tiles": chains in registers, observation tiles via TMA bulk copies
// grid = (n_slices, n_groups); group = NR_THREADS*KC chains
// ----------------------------------------------------------------------------
template <int KC, bool kSlope, bool kExtras, int kLik>
__global__ void __launch_bounds__(NR_THREADS)
    nr_tiles_kernel(const NrArgs a, const __grid_constant__ NrModel m, int use_tma,
                    const NrLik lik) {
  extern __shared__ __align__(128) double sm[];            // [NR_STAGES][2][NR_TILE]
  __shared__ __align__(8) unsigned long long full_bar[NR_STAGES];
  const int slice = blockIdx.x, group = blockIdx.y;
  const int64_t C = a.C;
  const int cbase = group * (NR_THREADS * KC) + threadIdx.x;

  double b0[KC], b1[KC], q[KC], acc[KC];
#pragma unroll
  for (int k = 0; k < KC; ++k) {
    const int c = cbase + k * NR_THREADS;
    const bool v = c < a.C;
    b0[k] = v ? a.theta_in[c] : 0.0;
    b1[k] = (v && kSlope) ? a.theta_in[C + c] : 0.0;
    if constexpr (kLik == PBX_LIK_STUDENT_T_NU)
      q[k] = v ? nr_q(a.theta_in[C + c], a.theta_in[2 * C + c]) : 0.0;
    else
      q[k] = (kLik && v) ? nr_q(a.theta_in[nr_isg<kLik, kSlope>() * C + c], lik.df) : 0.0;
    acc[k] = 0.0;
  }

  // this CTA's range of full tiles
  const int64_t n_full = a.N / NR_TILE;
  const int64_t per = (n_full + a.n_slices - 1) / a.n_slices;
  const int64_t t_begin = (int64_t)slice * per;
  const int64_t t_end = (t_begin + per < n_full) ? t_begin + per : n_full;
  const int64_t nt = t_end > t_begin ? t_end - t_begin : 0;
  constexpr uint32_t kTileBytes = NR_TILE * sizeof(double);

  if (threadIdx.x == 0) {
    for (int s = 0; s < NR_STAGES; ++s) pbx_mbar_init(&full_bar[s], 1);
    pbx_fence_barrier_init();
  }
  __syncthreads();

  auto issue = [&](int64_t t) {                            // thread 0 only
    const int s = (int)(t % NR_STAGES);
    double* dx = sm + (size_t)s * 2 * NR_TILE;
    double* dy = dx + NR_TILE;
    const int64_t o = (t_begin + t) * NR_TILE;
    pbx_mbar_expect_tx(&full_bar[s], kSlope ? 2 * kTileBytes : kTileBytes);
    if (kSlope) pbx_bulk_g2s(dx, a.x + o, kTileBytes, &full_bar[s]);
    pbx_bulk_g2s(dy, a.y + o, kTileBytes, &full_bar[s]);
  };
  double acc1[KC];                                         // odd observations: breaks the
#pragma unroll                                             // dependent fma pair per iteration
  for (int k = 0; k < KC; ++k) acc1[k] = 0.0;
  auto tile_math = [&](const double* sx, const double* sy, int cnt) {
#pragma unroll 2
    for (int i = 0; i < cnt; i += 2) {
      const double2 yv = *reinterpret_cast<const double2*>(sy + i);
      double2 xv = make_double2(0.0, 0.0);
      if (kSlope) xv = *reinterpret_cast<const double2*>(sx + i);
#pragma unroll
      for (int k = 0; k < KC; ++k) {
        const double r0 = yv.x - (kSlope ? fma(b1[k], xv.x, b0[k]) : b0[k]);
        const double r1 = yv.y - (kSlope ? fma(b1[k], xv.y, b0[k]) : b0[k]);
        acc[k] = nr_term<kLik>(acc[k], r0, q[k]);
        acc1[k] = nr_term<kLik>(acc1[k], r1, q[k]);
      }
    }
  };

  if (use_tma) {
    if (threadIdx.x == 0)
      for (int64_t t = 0; t < nt && t < NR_STAGES; ++t) issue(t);
    for (int64_t t = 0; t < nt; ++t) {
      const int s = (int)(t % NR_STAGES);
      pbx_mbar_wait(&full_bar[s], (uint32_t)(t / NR_STAGES) & 1);
      const double* sx = sm + (size_t)s * 2 * NR_TILE;
      tile_math(sx, sx + NR_TILE, NR_TILE);
      __syncthreads();                                     // everyone is done with stage s
      if (threadIdx.x == 0 && t + NR_STAGES < nt) issue(t + NR_STAGES);
    }
  } else {
    // unaligned base pointers: cooperative copy instead of bulk copies
    for (int64_t t = 0; t < nt; ++t) {
      const int64_t o = (t_begin + t) * NR_TILE;
      for (int i = threadIdx.x; i < NR_TILE; i += NR_THREADS) {
        if (kSlope) sm[i] = a.x[o + i];
        sm[NR_TILE + i] = a.y[o + i];
      }
      __syncthreads();
      tile_math(sm, sm + NR_TILE, NR_TILE);
      __syncthreads();
    }
  }
  // ragged tail (< NR_TILE observations): handled by the last slice
  if (slice == a.n_slices - 1) {
    const int64_t o = n_full * NR_TILE;
    const int rem = (int)(a.N - o);
    if (rem > 0) {
      __syncthreads();
      for (int i = threadIdx.x; i < NR_TILE; i += NR_THREADS) {
        // pad with (x = 0, y = b0-independent) handled by counting: zero-pad and fix below
        sm[i] = (kSlope && i < rem) ? a.x[o + i] : 0.0;
        sm[NR_TILE + i] = (i < rem) ? a.y[o + i] : 0.0;
      }
      __syncthreads();
      const int even = rem & ~1;
      tile_math(sm, sm + NR_TILE, even);
      if (rem & 1) {
        const double yv = sm[NR_TILE + even], xv = sm[even];
#pragma unroll
        for (int k = 0; k < KC; ++k) {
          const double r0 = yv - (kSlope ? fma(b1[k], xv, b0[k]) : b0[k]);
          acc[k] = nr_term<kLik>(acc[k], r0, q[k]);
        }
      }
    }
  }
#pragma unroll
  for (int k = 0; k < KC; ++k) {
    const int c = cbase + k * NR_THREADS;
    if (c < a.C) a.partial[(int64_t)slice * C + c] = acc[k] + acc1[k];
  }
  if (!nr_arrive_last(&a.counters[group], (unsigned int)a.n_slices)) return;
  // ---- phase B: this CTA is the last of its chain group ----------------------
#pragma unroll 1
  for (int k = 0; k < KC; ++k) {
    const int c = cbase + k * NR_THREADS;
    if (c >= a.C) continue;
    double S = 0.0;
    for (int s = 0; s < a.n_slices; ++s) S += __ldcg(&a.partial[(int64_t)s * C + c]);
    nr_phase_b<kExtras, kLik>(a, m, c, S, lik);
  }
}

// ----------------------------------------------------------------------------
// phase A, "stream": <= NR_SMAX chains, ONE pass over HBM.
// grid = 2 CTAs per SM, 256 threads; CTA b owns tiles b, b + grid, ... of 2048
// observations.  The tiles are fetched by 1-D TMA bulk copies into a 3-stage
// shared-memory ring (96 KB per CTA -> ~190 KB of loads in flight per SM, which is
// what it takes to cover HBM latency at ~6.5 TB/s) and consumed with conflict-free
// 128-bit shared loads, every thread updating all KS chains' sums; warp-shuffle +
// block reduction; phase B in the last CTA.
// ----------------------------------------------------------------------------
#define NRS_THREADS 256
template <int KS, bool kSlope, bool kExtras, int kLik>
__global__ void __launch_bounds__(NRS_THREADS)
    nr_stream_kernel(const NrArgs a, const __grid_constant__ NrModel m, int use_tma,
                     const NrLik lik) {
  extern __shared__ __align__(128) double sm[];            // [NR_STAGES][2][NRS_TILE]
  __shared__ __align__(8) unsigned long long full_bar[NR_STAGES];
  __shared__ double s_red[NRS_THREADS / 32][KS];
  double b0[KS], b1[KS], q[KS], acc[KS];
#pragma unroll
  for (int k = 0; k < KS; ++k) {
    b0[k] = (k < a.C) ? a.theta_in[k] : 0.0;
    b1[k] = (k < a.C && kSlope) ? a.theta_in[(int64_t)a.C + k] : 0.0;
    if constexpr (kLik == PBX_LIK_STUDENT_T_NU)
      q[k] = k < a.C ? nr_q(a.theta_in[(int64_t)a.C + k], a.theta_in[2 * (int64_t)a.C + k]) : 0.0;
    else
      q[k] = (kLik && k < a.C)
                 ? nr_q(a.theta_in[(int64_t)nr_isg<kLik, kSlope>() * a.C + k], lik.df)
                 : 0.0;
    acc[k] = 0.0;
  }
  const int64_t n_full = a.N / NRS_TILE;
  // tiles of this CTA: blockIdx.x + j * gridDim.x
  const int64_t nt = (n_full > blockIdx.x) ? (n_full - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  constexpr uint32_t kTileBytes = NRS_TILE * sizeof(double);
  if (threadIdx.x == 0) {
    for (int s = 0; s < NR_STAGES; ++s) pbx_mbar_init(&full_bar[s], 1);
    pbx_fence_barrier_init();
  }
  __syncthreads();
  auto issue = [&](int64_t j) {                            // thread 0 only
    const int s = (int)(j % NR_STAGES);
    double* dx = sm + (size_t)s * 2 * NRS_TILE;
    const int64_t o = ((int64_t)blockIdx.x + j * gridDim.x) * NRS_TILE;
    pbx_mbar_expect_tx(&full_bar[s], kSlope ? 2 * kTileBytes : kTileBytes);
    if (kSlope) pbx_bulk_g2s(dx, a.x + o, kTileBytes, &full_bar[s]);
    pbx_bulk_g2s(dx + NRS_TILE, a.y + o, kTileBytes, &full_bar[s]);
  };
  auto tile_math = [&](const double* sx, const double* sy, int cnt) {
#pragma unroll 2
    for (int i = 2 * threadIdx.x; i < cnt; i += 2 * NRS_THREADS) {
      const double2 yv = *reinterpret_cast<const double2*>(sy + i);
      double2 xv = make_double2(0.0, 0.0);
      if (kSlope) xv = *reinterpret_cast<const double2*>(sx + i);
#pragma unroll
      for (int k = 0; k < KS; ++k) {
        const double r0 = yv.x - (kSlope ? fma(b1[k], xv.x, b0[k]) : b0[k]);
        const double r1 = yv.y - (kSlope ? fma(b1[k], xv.y, b0[k]) : b0[k]);
        acc[k] = nr_term<kLik>(acc[k], r0, q[k]);
        acc[k] = nr_term<kLik>(acc[k], r1, q[k]);
      }
    }
  };
  if (use_tma) {
    if (threadIdx.x == 0)
      for (int64_t j = 0; j < nt && j < NR_STAGES; ++j) issue(j);
    for (int64_t j = 0; j < nt; ++j) {
      const int s = (int)(j % NR_STAGES);
      pbx_mbar_wait(&full_bar[s], (uint32_t)(j / NR_STAGES) & 1);
      const double* sx = sm + (size_t)s * 2 * NRS_TILE;
      tile_math(sx, sx + NRS_TILE, NRS_TILE);
      __syncthreads();
      if (threadIdx.x == 0 && j + NR_STAGES < nt) issue(j + NR_STAGES);
    }
  } else {
    for (int64_t j = 0; j < nt; ++j) {
      const int64_t o = ((int64_t)blockIdx.x + j * gridDim.x) * NRS_TILE;
      for (int i = threadIdx.x; i < NRS_TILE; i += NRS_THREADS) {
        if (kSlope) sm[i] = a.x[o + i];
        sm[NRS_TILE + i] = a.y[o + i];
      }
      __syncthreads();
      tile_math(sm, sm + NRS_TILE, NRS_TILE);
      __syncthreads();
    }
  }
  // ragged tail (< NRS_TILE observations): CTA 0, straight from global memory
  if (blockIdx.x == 0) {
    for (int64_t i = n_full * NRS_TILE + threadIdx.x; i < a.N; i += NRS_THREADS) {
      const double yv = a.y[i], xv = kSlope ? a.x[i] : 0.0;
#pragma unroll
      for (int k = 0; k < KS; ++k) {
        const double r0 = yv - (kSlope ? fma(b1[k], xv, b0[k]) : b0[k]);
        acc[k] = nr_term<kLik>(acc[k], r0, q[k]);
      }
    }
  }
  // warp-shuffle reduction, then across the warps through shared memory
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < KS; ++k) {
    double v = acc[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) s_red[warp][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < KS && threadIdx.x < a.C) {
    double v = 0.0;
#pragma unroll
    for (int w = 0; w < NRS_THREADS / 32; ++w) v += s_red[w][threadIdx.x];
    a.partial[(int64_t)blockIdx.x * a.C + threadIdx.x] = v;
  }
  if (!nr_arrive_last(&a.counters[0], gridDim.x)) return;
  if (threadIdx.x < a.C && threadIdx.x < KS) {
    const int c = threadIdx.x;
    double S = 0.0;
    for (int s = 0; s < (int)gridDim.x; ++s) S += __ldcg(&a.partial[(int64_t)s * a.C + c]);
    nr_phase_b<kExtras, kLik>(a, m, c, S, lik);
  }
}

// ----------------------------------------------------------------------------
// host side
// ----------------------------------------------------------------------------
struct NrPlan {
  int variant;       // 1 tiles, 2 stream
  int kc;            // chains per thread (tiles)
  int n_groups, n_slices;
  int use_tma;
  size_t smem;
};

static NrPlan nr_plan(pbx_ctx* ctx, const pbx_mh_normreg_params* p) {
  NrPlan pl;
  const int C = p->n_chains;
  int variant = p->variant;
  if (variant == 0) variant = (C <= NR_SMAX) ? 2 : 1;
  if (variant == 2 && C > NR_SMAX) variant = 1;
  const bool aligned = (((uintptr_t)p->y_obs) % 16 == 0) &&
                       (!p->has_slope || ((uintptr_t)p->x_obs) % 16 == 0);
  pl.variant = variant;
  pl.use_tma = aligned ? 1 : 0;
  pl.smem = 0;
  if (variant == 1) {
    pl.kc = (C >= 4 * NR_THREADS * 8) ? 4 : ((C >= 2 * NR_THREADS * 8) ? 2 : 1);
    pl.n_groups = (C + NR_THREADS * pl.kc - 1) / (NR_THREADS * pl.kc);
    pl.smem = (size_t)NR_STAGES * 2 * NR_TILE * sizeof(double);     // 48 KB -> 4 CTAs / SM
    const int64_t n_full = p->n_obs / NR_TILE;
    const int concurrent = ctx->sm_count * 4;
    int64_t slices = (2 * (int64_t)concurrent) / pl.n_groups;       // ~2 full waves
    if (slices > n_full) slices = n_full;
    if (slices < 1) slices = 1;
    pl.n_slices = (int)slices;
  } else {
    pl.kc = (C <= 1) ? 1 : (C <= 2 ? 2 : (C <= 4 ? 4 : 8));    // KS: chains per thread
    pl.n_groups = 1;
    pl.smem = (size_t)NR_STAGES * 2 * NRS_TILE * sizeof(double);    // 96 KB -> 2 CTAs / SM
    int64_t want = p->n_obs / NRS_TILE;
    int64_t cap = (int64_t)ctx->sm_count * 2;
    pl.n_slices = (int)(want < 1 ? 1 : (want > cap ? cap : want));
  }
  return pl;
}

static int nr_validate(const pbx_mh_normreg_params* p, const char* who, bool need_state) {
  PBX_REQUIRE(p != nullptr, "%s: null params", who);
  PBX_REQUIRE(p->n_chains >= 1, "%s: n_chains must be >= 1", who);
  PBX_REQUIRE(p->n_params == 2 || p->n_params == 3, "%s: n_params must be 2 or 3", who);
  PBX_REQUIRE(p->lik_kind == PBX_LIK_NORMAL || p->lik_kind == PBX_LIK_STUDENT_T ||
                  p->lik_kind == PBX_LIK_STUDENT_T_NU,
              "%s: unknown lik_kind %d", who, p->lik_kind);
  if (p->lik_kind == PBX_LIK_STUDENT_T_NU) {
    PBX_REQUIRE(p->n_params == 3 && p->has_slope == 0,
                "%s: the sampled-nu Student-t needs 3 params (mu, sigma, nu) and no slope", who);
    PBX_REQUIRE(p->lik_df == 0.0 && p->lik_logc == 0.0,
                "%s: the sampled-nu Student-t reads nu from theta: lik_df and lik_logc must be 0",
                who);
    PBX_REQUIRE(p->lims[2][0] > 0.0 || (p->lims[2][0] == 0.0 && p->open_end[2][0]),
                "%s: nu's prior box must admit nu > 0 only (got lower limit %g, %s)", who,
                p->lims[2][0], p->open_end[2][0] ? "open" : "closed");
  } else {
    PBX_REQUIRE((p->has_slope != 0) == (p->n_params == 3),
                "%s: has_slope needs 3 params (b0, b1, sigma), otherwise 2 (mu, sigma)", who);
  }
  PBX_REQUIRE(p->n_obs >= 1, "%s: n_obs must be >= 1", who);
  PBX_REQUIRE(p->y_obs != nullptr && (!p->has_slope || p->x_obs != nullptr),
              "%s: observation arrays missing", who);
  PBX_REQUIRE(p->accept_mode == PBX_ACCEPT_REFERENCE || p->accept_mode == PBX_ACCEPT_LOG,
              "%s: unknown accept_mode", who);
  PBX_REQUIRE(p->prop_kind >= PBX_PROP_NORMAL && p->prop_kind <= PBX_PROP_SPHERICAL,
              "%s: unknown prop_kind", who);
  if (p->lik_kind == PBX_LIK_STUDENT_T) {
    PBX_REQUIRE(p->lik_df > 0.0 && isfinite(p->lik_df),
                "%s: the Student-t likelihood needs 0 < lik_df < inf (got %g)", who, p->lik_df);
    PBX_REQUIRE(isfinite(p->lik_logc), "%s: lik_logc is not finite", who);
  }
  PBX_REQUIRE(p->lik_kind == PBX_LIK_NORMAL || p->variant != 3,
              "%s: variant 3 (sufficient statistics) needs the normal likelihood", who);
  for (int j = 0; j < p->n_params; ++j) {
    PBX_REQUIRE(p->lims[j][1] > p->lims[j][0], "%s: empty prior box for parameter %d", who, j);
    PBX_REQUIRE(!p->log_ufun[j] || p->lims[j][0] > 0.0,
                "%s: log ufun needs positive limits (parameter %d)", who, j);
  }
  if (need_state) {
    PBX_REQUIRE(p->n_steps >= 0 && p->thin >= 1, "%s: n_steps >= 0 and thin >= 1 required", who);
    PBX_REQUIRE(p->step0 >= 0 && p->chain0 >= 0, "%s: step0/chain0 must be >= 0", who);
    PBX_REQUIRE(p->state && p->state_lp, "%s: state/state_lp are mandatory", who);
    PBX_REQUIRE((p->inj_delta == nullptr) == (p->inj_thresh == nullptr),
                "%s: inj_delta and inj_thresh must be given together", who);
    if (p->has_prop_mat) {
      const int P = p->n_params;
      for (int i = 0; i < P; ++i)
        for (int j = 0; j < P; ++j) {
          const double v = p->prop_mat[i * P + j];
          PBX_REQUIRE(isfinite(v), "%s: prop_mat[%d][%d] is not finite", who, i, j);
          PBX_REQUIRE(j <= i || v == 0.0,
                      "%s: prop_mat must be lower-triangular (entry [%d][%d] = %g)", who, i, j, v);
          PBX_REQUIRE(j != i || v > 0.0,
                      "%s: prop_mat needs a positive diagonal (entry [%d][%d] = %g)", who, i, i, v);
        }
    }
  }
  return PBX_OK;
}

static void nr_fill_model(const pbx_mh_normreg_params* p, NrModel& m) {
  m.P = p->n_params;
  m.has_slope = p->has_slope;
  m.bound = p->prop_bound != 0;
  m.accept_mode = p->accept_mode;
  m.prop_kind = p->prop_kind;
  m.coef = p->accept_coef;
  m.radius = p->prop_radius;
  for (int j = 0; j < PBX_MAX_PARAMS; ++j) {
    m.lims[j][0] = p->lims[j][0];
    m.lims[j][1] = p->lims[j][1];
    m.open_end[j][0] = p->open_end[j][0];
    m.open_end[j][1] = p->open_end[j][1];
    m.log_ufun[j] = p->log_ufun[j];
    m.scale[j] = p->prop_scale[j];
    double len = 1.0;
    if (j < p->n_params)
      len = p->log_ufun[j] ? log(p->lims[j][1]) - log(p->lims[j][0]) : p->lims[j][1] - p->lims[j][0];
    m.nlhv[j] = -log(len);
  }
  // the factor is read by pbx_mh_normreg_run only (pbx_normreg_logjoint draws no proposal)
  m.has_L = p->has_prop_mat != 0;
  for (int i = 0; i < PBX_MAX_PARAMS; ++i)
    for (int j = 0; j < PBX_MAX_PARAMS; ++j)
      m.L[i][j] = (m.has_L && i < p->n_params && j <= i) ? p->prop_mat[i * p->n_params + j] : 0.0;
}

static bool nr_extras(const NrArgs& a, const NrModel& m) {
  return m.bound != 0 || m.has_L != 0 || a.out_xprop != nullptr || a.out_pprop != nullptr;
}

template <int KC, int kLik>
static int nr_launch_tiles(pbx_ctx* ctx, const NrPlan& pl, const NrArgs& a, const NrModel& m,
                           const NrLik& lik) {
  dim3 grid(pl.n_slices, pl.n_groups);
#define NR_TILES_GO(S, E)                                                                      \
  do {                                                                                         \
    PBX_CUDA(cudaFuncSetAttribute(nr_tiles_kernel<KC, S, E, kLik>,                             \
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem)); \
    nr_tiles_kernel<KC, S, E, kLik><<<grid, NR_THREADS, pl.smem, ctx->stream>>>(a, m,          \
                                                                               pl.use_tma, lik); \
  } while (0)
  const bool ex = nr_extras(a, m);
  if constexpr (kLik == PBX_LIK_STUDENT_T_NU) {         // (mu, sigma, nu): never a slope
    if (ex) NR_TILES_GO(false, true);
    else NR_TILES_GO(false, false);
  } else {
    if (m.has_slope && ex) NR_TILES_GO(true, true);
    else if (m.has_slope) NR_TILES_GO(true, false);
    else if (ex) NR_TILES_GO(false, true);
    else NR_TILES_GO(false, false);
  }
#undef NR_TILES_GO
  PBX_LAUNCH_CHECK(ctx);
  return PBX_OK;
}

template <int KS, int kLik>
static int nr_launch_stream(pbx_ctx* ctx, const NrPlan& pl, const NrArgs& a, const NrModel& m,
                            const NrLik& lik) {
#define NR_STREAM_GO(S, E)                                                                     \
  do {                                                                                         \
    PBX_CUDA(cudaFuncSetAttribute(nr_stream_kernel<KS, S, E, kLik>,                            \
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem)); \
    nr_stream_kernel<KS, S, E, kLik><<<pl.n_slices, NRS_THREADS, pl.smem, ctx->stream>>>(      \
        a, m, pl.use_tma, lik);                                                                \
  } while (0)
  const bool ex = nr_extras(a, m);
  if constexpr (kLik == PBX_LIK_STUDENT_T_NU) {
    if (ex) NR_STREAM_GO(false, true);
    else NR_STREAM_GO(false, false);
  } else {
    if (m.has_slope && ex) NR_STREAM_GO(true, true);
    else if (m.has_slope) NR_STREAM_GO(true, false);
    else if (ex) NR_STREAM_GO(false, true);
    else NR_STREAM_GO(false, false);
  }
#undef NR_STREAM_GO
  PBX_LAUNCH_CHECK(ctx);
  return PBX_OK;
}

template <int kLik>
static int nr_launch_step_lik(pbx_ctx* ctx, const NrPlan& pl, const NrArgs& a, const NrModel& m,
                              const NrLik& lik) {
  if (pl.variant == 1) {
    switch (pl.kc) {
      case 4: return nr_launch_tiles<4, kLik>(ctx, pl, a, m, lik);
      case 2: return nr_launch_tiles<2, kLik>(ctx, pl, a, m, lik);
      default: return nr_launch_tiles<1, kLik>(ctx, pl, a, m, lik);
    }
  }
  switch (pl.kc) {
    case 1: return nr_launch_stream<1, kLik>(ctx, pl, a, m, lik);
    case 2: return nr_launch_stream<2, kLik>(ctx, pl, a, m, lik);
    case 4: return nr_launch_stream<4, kLik>(ctx, pl, a, m, lik);
    default: return nr_launch_stream<8, kLik>(ctx, pl, a, m, lik);
  }
}

static int nr_launch_step(pbx_ctx* ctx, const NrPlan& pl, const NrArgs& a, const NrModel& m,
                          int lik_kind, const NrLik& lik) {
  switch (lik_kind) {
    case PBX_LIK_STUDENT_T: return nr_launch_step_lik<PBX_LIK_STUDENT_T>(ctx, pl, a, m, lik);
    case PBX_LIK_STUDENT_T_NU: return nr_launch_step_lik<PBX_LIK_STUDENT_T_NU>(ctx, pl, a, m, lik);
    default: return nr_launch_step_lik<PBX_LIK_NORMAL>(ctx, pl, a, m, lik);
  }
}

// ============================================================================
// variant 3: sufficient statistics.  For a NORMAL likelihood the residual sum of squares
// of any (b0, b1) is a quadratic form in a few sums over the observations, so after a
// one-time reduction every likelihood evaluation is O(1) instead of O(N) and a whole
// walk is ONE launch.  To stay at the accuracy of the per-observation sum (<= 3e-16
// relative against a long-double evaluation, the same as the streaming kernels) the
// statistics are centred -- three deterministic passes over the data:
//   1. cx = mean x, cy = mean y
//   2. u = x - cx, v = y - cy:  Sxx = sum u^2, Sxy = sum u v, Su = sum u  -> b1* = Sxy / Sxx
//   3. e = v - b1* u:           RSS = sum e^2, Se = sum e, Seu = sum e u
// and with D = b1 - b1*, a = b0 + b1 cx - cy every term of
//   sum (y - b0 - b1 x)^2 = RSS + D^2 Sxx + N a^2 - 2 D Seu - 2 a Se + 2 a D Su
// is either non-negative or a rounding residual: no cancellation, whatever the fit.
// (Without a slope: u = 0, b1 = 0, e = v.)  Opt-in: the default variants evaluate the
// likelihood term by term as the reference does.
// ============================================================================

#define SS_THREADS 256
#define SS_MAXCTA 1024
// pass 1: (sum x, sum y);  pass 2: (Sxx, Sxy, Su, -);  pass 3: (RSS, Se, Seu, -)
template <int PASS>
__global__ void __launch_bounds__(SS_THREADS) ss_partial_kernel(const double* __restrict__ x,
                                                                const double* __restrict__ y,
                                                                long long n, long long per_cta,
                                                                const NrStats* __restrict__ st,
                                                                double* __restrict__ part) {
  __shared__ double s_red[SS_THREADS / 32][4];
  const long long e0 = (long long)blockIdx.x * per_cta, e1 = min(n, e0 + per_cta);
  const double cx = PASS > 1 ? st->cx : 0.0, cy = PASS > 1 ? st->cy : 0.0;
  const double b1 = PASS > 2 ? st->b1s : 0.0;
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  for (long long e = e0 + threadIdx.x; e < e1; e += SS_THREADS) {
    const double xv = x ? x[e] : 0.0, yv = y[e];
    if (PASS == 1) {
      acc[0] += xv;
      acc[1] += yv;
    } else if (PASS == 2) {
      const double u = xv - cx, v = yv - cy;
      acc[0] = fma(u, u, acc[0]);
      acc[1] = fma(u, v, acc[1]);
      acc[2] += u;
    } else {
      const double u = xv - cx, ee = (yv - cy) - b1 * u;
      acc[0] = fma(ee, ee, acc[0]);
      acc[1] += ee;
      acc[2] = fma(ee, u, acc[2]);
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    double v = acc[k];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
    if (lane == 0) s_red[warp][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    double v = 0.0;
#pragma unroll
    for (int w = 0; w < SS_THREADS / 32; ++w) v += s_red[w][threadIdx.x];
    part[(size_t)blockIdx.x * 4 + threadIdx.x] = v;
  }
}

// one warp: adds the partials in index order and updates the statistics
template <int PASS>
__global__ void ss_final_kernel(const double* __restrict__ part, int nparts, long long n,
                                int has_x, NrStats* st) {
  const int k = threadIdx.x;
  double v = 0.0;
  if (k < 4)
    for (int p = 0; p < nparts; ++p) v += part[(size_t)p * 4 + k];
  const double v0 = __shfl_sync(0xffffffffu, v, 0), v1 = __shfl_sync(0xffffffffu, v, 1);
  const double v2 = __shfl_sync(0xffffffffu, v, 2);
  if (k != 0) return;
  if (PASS == 1) {
    st->N = (double)n;
    st->cx = has_x ? v0 / (double)n : 0.0;
    st->cy = v1 / (double)n;
  } else if (PASS == 2) {
    st->Sxx = v0;
    st->b1s = (has_x && v0 > 0.0) ? v1 / v0 : 0.0;
    st->Su = v2;
  } else {
    st->RSS = v0;
    st->Se = v1;
    st->Seu = v2;
  }
}

__device__ __forceinline__ double ss_rss(const NrStats& st, const NrModel& m, const double* th) {
  const double b0 = th[0], b1 = m.has_slope ? th[1] : 0.0;
  const double D = b1 - st.b1s;
  const double a = fma(b1, st.cx, b0) - st.cy;
  double S = st.RSS;
  S = fma(D * D, st.Sxx, S);
  S = fma(st.N * a, a, S);
  S = fma(-2.0 * D, st.Seu, S);
  S = fma(-2.0 * a, st.Se, S);
  S = fma(2.0 * a * D, st.Su, S);
  return S;
}

// evaluate-only: log-joint of theta[P][C] from the statistics
__global__ void __launch_bounds__(256) ss_eval_kernel(const NrArgs a, const __grid_constant__ NrModel m,
                                                      const NrStats* __restrict__ stp) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= a.C) return;
  const NrStats st = *stp;
  double th[PBX_MAX_PARAMS];
  for (int j = 0; j < m.P; ++j) th[j] = a.theta_in[(int64_t)j * a.C + c];
  a.eval_out[c] = nr_logjoint(a, m, th, ss_rss(st, m, th));
}

// log(t) for nr_decide where a lambda cannot be used: nvcc 12.9's front end aborts on the
// [&] { return log(t); } of nr_phase_b inside the templated ss_walk_kernel
struct NrLogOf {
  double t;
  __device__ double operator()() const { return log(t); }
};

// the whole walk of one chain in one thread (the same draws, accept rule and records as
// nr_phase_b, with the O(1) likelihood); kColour as nr_draw_delta's (the runtime test alone
// slows the uncoloured walk by 4 %)
template <bool kColour>
__global__ void __launch_bounds__(128) ss_walk_kernel(const NrArgs a, const __grid_constant__ NrModel m,
                                                      const NrStats* __restrict__ stp) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= a.C) return;
  const int64_t C = a.C;
  const NrStats st = *stp;
  double th[PBX_MAX_PARAMS], ssum[PBX_MAX_PARAMS], ssq[PBX_MAX_PARAMS];
  for (int j = 0; j < m.P; ++j) {
    th[j] = a.state[(int64_t)j * C + c];
    ssum[j] = ssq[j] = 0.0;
  }
  double lp = a.state_lp[c];
  int64_t nacc = 0;
  for (int k = 0; k < a.T; ++k) {
    const int64_t gstep = a.step0 + k;
    double dl[PBX_MAX_PARAMS], thp[PBX_MAX_PARAMS];
    nr_draw_delta<0, kColour>(a, m, gstep, k, c, dl);
    for (int j = 0; j < m.P; ++j) thp[j] = nr_move<true>(m, j, th[j], dl[j]);
    const double lpp = nr_logjoint(a, m, thp, ss_rss(st, m, thp));
    const double t = nr_threshold(a, gstep, k, c);
    double s;
    const bool acc = nr_decide(m, lpp, lp, t, NrLogOf{t}, gstep, a.out_score != nullptr, s);
    if (acc) {
      for (int j = 0; j < m.P; ++j) th[j] = thp[j];
      lp = lpp;
      ++nacc;
    }
    for (int j = 0; j < m.P; ++j) {
      ssum[j] += th[j];
      ssq[j] = fma(th[j], th[j], ssq[j]);
    }
    nr_record<true>(a, m, k, c, acc, s, thp, lpp, th, lp);
  }
  nr_write_back(a, m, c, th, lp, ssum, ssq, nacc);
}


// ---------------------------------------------------------------------------
// variant 4: SMALL problems (N <= RW_MAXN observations, C * N <= 2^24 terms per step) --
// the whole walk in ONE launch.  The per-step kernels above cost a launch (~3-4 us) per MH
// step, which is all the time there is at the reference-feasible sizes (N = 60 ... 10^4, a
// handful of chains).  Here a WARP owns one chain for the whole walk: the observations are
// staged into shared memory once per CTA, lane l takes observations l, l + 32, ..., the
// residual sum of squares finishes with a fixed xor-shuffle tree (every lane ends up with the
// same bits, so all 32 lanes carry the chain state redundantly and no broadcast is needed),
// then proposal, priors, accept test and records exactly as nr_phase_b.  Term-by-term
// arithmetic as the other variants (the reference's array density path), not sufficient
// statistics.
// ---------------------------------------------------------------------------
#define RW_WARPS 4
#define RW_MAXN 8192
// kColour: as nr_draw_delta's (the colouring costs this kernel registers)
template <bool kSlope, bool kColour, int kLik>
__global__ void __launch_bounds__(32 * RW_WARPS)
    rw_walk_kernel(const NrArgs a, const __grid_constant__ NrModel m, const NrLik lik) {
  extern __shared__ __align__(16) double rw_sm[];       // y[N], then x[N] (kSlope)
  double* sy = rw_sm;
  double* sx = rw_sm + a.N;
  for (int64_t i = threadIdx.x; i < a.N; i += blockDim.x) {
    sy[i] = a.y[i];
    if (kSlope) sx[i] = a.x[i];
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (c >= a.C) return;
  const int64_t C = a.C;
  const int n = (int)a.N;
  // (b0, b1, sigma) with a slope, (mu, sigma, nu) for the sampled-nu t, else (mu, sigma)
  constexpr int P = (kSlope || kLik == PBX_LIK_STUDENT_T_NU) ? 3 : 2;
  double th[PBX_MAX_PARAMS], ssum[PBX_MAX_PARAMS], ssq[PBX_MAX_PARAMS];
  _Pragma("unroll") for (int j = 0; j < P; ++j) {
    th[j] = a.state[(int64_t)j * C + c];
    ssum[j] = ssq[j] = 0.0;
  }
  auto rss = [&](const double* t) {
    const double b0 = t[0], b1 = kSlope ? t[1] : 0.0;
    // four independent partial sums per lane (a fixed association: the result depends on n
    // only), so that the dependent-FMA latency is hidden at large n
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    auto term = [&](int i) {
      const double r = kSlope ? (sy[i] - b0) - b1 * sx[i] : sy[i] - b0;
      // if constexpr: the normal instantiation captures no more than the normal-only kernel
      // did, which keeps its SASS byte-identical (a runtime-dead capture reorders registers)
      if constexpr (kLik == PBX_LIK_STUDENT_T_NU) return log1p((r * r) * nr_q(t[1], t[2]));
      else if constexpr (kLik == PBX_LIK_STUDENT_T) return log1p((r * r) * nr_q(t[P - 1], lik.df));
      else return r * r;
    };
    int i = lane;
    for (; i + 96 < n; i += 128) {
      s0 += term(i);
      s1 += term(i + 32);
      s2 += term(i + 64);
      s3 += term(i + 96);
    }
    if (i < n) s0 += term(i);
    if (i + 32 < n) s1 += term(i + 32);
    if (i + 64 < n) s2 += term(i + 64);
    double s = (s0 + s1) + (s2 + s3);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    return s;
  };
  double lp = (a.step0 > 0) ? a.state_lp[c] : 0.0;
  int64_t nacc = 0;
  // the state-independent part of a step -- Philox, the proposal delta, the threshold and its
  // log -- is produced for 32 steps at a time, one step per lane, and handed out by shuffles:
  // all lanes carry the chain redundantly, so doing it per step would put ~150 dependent
  // instructions on every step's critical path
  double dlv[PBX_MAX_PARAMS], tv = 0.5, ltv = 0.0;
  _Pragma("unroll") for (int j = 0; j < PBX_MAX_PARAMS; ++j) dlv[j] = 0.0;
  for (int k = 0; k < a.T; ++k) {
    const int64_t gstep = a.step0 + k;
    if ((k & 31) == 0) {
      const int mine = k + lane;
      if (mine < a.T) {
        nr_draw_delta<P, kColour>(a, m, a.step0 + mine, mine, c, dlv);
        tv = nr_threshold(a, a.step0 + mine, mine, c);
        ltv = log(tv);
      }
    }
    double dl[PBX_MAX_PARAMS], thp[PBX_MAX_PARAMS];
    _Pragma("unroll") for (int j = 0; j < P; ++j) dl[j] = __shfl_sync(0xffffffffu, dlv[j], k & 31);
    const double t = __shfl_sync(0xffffffffu, tv, k & 31);
    const double logt = __shfl_sync(0xffffffffu, ltv, k & 31);
    _Pragma("unroll") for (int j = 0; j < P; ++j) thp[j] = nr_move<true>(m, j, th[j], dl[j]);
    const double lpp = nr_logjoint<P, kLik>(a, m, thp, rss(thp), lik);
    double s;
    const bool acc = nr_decide(m, lpp, lp, t, [&] { return logt; }, gstep,
                               a.out_score != nullptr, s);
    if (acc) {
      _Pragma("unroll") for (int j = 0; j < P; ++j) th[j] = thp[j];
      lp = lpp;
      ++nacc;
    }
    _Pragma("unroll") for (int j = 0; j < P; ++j) {
      ssum[j] += th[j];
      ssq[j] = fma(th[j], th[j], ssq[j]);
    }
    if (lane == 0) nr_record<true, P>(a, m, k, c, acc, s, thp, lpp, th, lp);
  }
  if (lane == 0) nr_write_back<P>(a, m, c, th, lp, ssum, ssq, nacc);
}

static bool rw_applies(const pbx_mh_normreg_params* p) {
  if (p->variant == 4) return true;
  return p->variant == 0 && p->n_obs <= RW_MAXN && p->n_steps >= 2 &&
         (int64_t)p->n_chains * p->n_obs <= ((int64_t)1 << 24);
}

// computes the statistics into the context workspace; *out points at them
int pbx_ss_compute(pbx_ctx* ctx, const double* x, const double* y, int64_t n, NrStats** out) {
  const int64_t chunk = 8192;
  int64_t grid = std::min<int64_t>((n + chunk - 1) / chunk, SS_MAXCTA);
  if (grid < 1) grid = 1;
  int64_t per_cta = ((n + grid - 1) / grid + chunk - 1) / chunk * chunk;
  grid = (n + per_cta - 1) / per_cta;
  const size_t part_bytes = ((size_t)SS_MAXCTA * 4 * 8 + 255) / 256 * 256;
  int rc = pbx_ws_reserve(ctx, part_bytes + 256);
  if (rc) return rc;
  double* part = (double*)ctx->ws;
  NrStats* st = (NrStats*)((char*)ctx->ws + part_bytes);
  const int has_x = x != nullptr;
  ss_partial_kernel<1><<<(int)grid, SS_THREADS, 0, ctx->stream>>>(x, y, n, per_cta, st, part);
  PBX_LAUNCH_CHECK(ctx);
  ss_final_kernel<1><<<1, 32, 0, ctx->stream>>>(part, (int)grid, n, has_x, st);
  PBX_LAUNCH_CHECK(ctx);
  ss_partial_kernel<2><<<(int)grid, SS_THREADS, 0, ctx->stream>>>(x, y, n, per_cta, st, part);
  PBX_LAUNCH_CHECK(ctx);
  ss_final_kernel<2><<<1, 32, 0, ctx->stream>>>(part, (int)grid, n, has_x, st);
  PBX_LAUNCH_CHECK(ctx);
  ss_partial_kernel<3><<<(int)grid, SS_THREADS, 0, ctx->stream>>>(x, y, n, per_cta, st, part);
  PBX_LAUNCH_CHECK(ctx);
  ss_final_kernel<3><<<1, 32, 0, ctx->stream>>>(part, (int)grid, n, has_x, st);
  PBX_LAUNCH_CHECK(ctx);
  *out = st;
  return PBX_OK;
}

// workspace: partial [n_slices][C] | counters [n_groups] | prop [P][C]
static int nr_workspace(pbx_ctx* ctx, const NrPlan& pl, int C, int P, double** partial,
                        unsigned int** counters, double** prop) {
  size_t off = 0;
  auto take = [&](size_t b) { size_t o = off; off += (b + 255) / 256 * 256; return o; };
  const size_t o_part = take((size_t)pl.n_slices * C * 8);
  const size_t o_cnt = take((size_t)pl.n_groups * 4);
  const size_t o_prop = take((size_t)P * C * 8);
  int rc = pbx_ws_reserve(ctx, off);
  if (rc) return rc;
  char* ws = (char*)ctx->ws;
  *partial = (double*)(ws + o_part);
  *counters = (unsigned int*)(ws + o_cnt);
  *prop = (double*)(ws + o_prop);
  PBX_CUDA(cudaMemsetAsync(*counters, 0, (size_t)pl.n_groups * 4, ctx->stream));
  return PBX_OK;
}

// the kernel arguments of a call, without the workspace of the one-launch-per-step kernels
static NrArgs nr_args(const pbx_mh_normreg_params* p) {
  NrArgs a;
  memset(&a, 0, sizeof(a));
  a.C = p->n_chains; a.N = p->n_obs; a.x = p->x_obs; a.y = p->y_obs;
  a.state = p->state; a.state_lp = p->state_lp;
  a.step0 = p->step0; a.T = p->n_steps; a.thin = p->thin;
  a.chain0 = p->chain0; a.seed = p->seed;
  a.inj_delta = p->inj_delta; a.inj_thresh = p->inj_thresh;
  a.out_x = p->out_x; a.out_prob = p->out_prob;
  a.out_accept = p->out_accept; a.out_score = p->out_score;
  a.out_xprop = p->out_xprop; a.out_pprop = p->out_pprop;
  a.accept_count = p->accept_count; a.stat_sum = p->stat_sum; a.stat_sumsq = p->stat_sumsq;
  return a;
}

static int nr_walk_suffstat(pbx_ctx* ctx, const NrArgs& a, const NrModel& m) {
  NrStats* st = nullptr;
  int rc = pbx_ss_compute(ctx, m.has_slope ? a.x : nullptr, a.y, a.N, &st);
  if (rc) return rc;
  if (m.has_L) ss_walk_kernel<true><<<(a.C + 127) / 128, 128, 0, ctx->stream>>>(a, m, st);
  else ss_walk_kernel<false><<<(a.C + 127) / 128, 128, 0, ctx->stream>>>(a, m, st);
  PBX_LAUNCH_CHECK(ctx);
  return PBX_OK;
}

template <int kLik>
static int nr_walk_small(pbx_ctx* ctx, const NrArgs& a, const NrModel& m, const NrLik& lik) {
  const size_t smem = (size_t)a.N * 8 * (m.has_slope ? 2 : 1);
  // warps (chains) per CTA: up to RW_WARPS, fewer when there are few chains, so that they
  // spread over the SMs (every warp re-reads the resident observations each step: four
  // warps on one SM share its 128 B/clk of shared-memory bandwidth)
  int wpc = (a.C + 2 * ctx->sm_count - 1) / (2 * ctx->sm_count);
  wpc = wpc < 1 ? 1 : (wpc > RW_WARPS ? RW_WARPS : wpc);
  const int grid = (a.C + wpc - 1) / wpc;
#define RW_GO(S, L)                                                                            \
  do {                                                                                         \
    PBX_CUDA(cudaFuncSetAttribute(rw_walk_kernel<S, L, kLik>,                                  \
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));    \
    rw_walk_kernel<S, L, kLik><<<grid, 32 * wpc, smem, ctx->stream>>>(a, m, lik);              \
  } while (0)
  if constexpr (kLik == PBX_LIK_STUDENT_T_NU) {
    if (m.has_L) RW_GO(false, true);
    else RW_GO(false, false);
  } else {
    if (m.has_slope && m.has_L) RW_GO(true, true);
    else if (m.has_slope) RW_GO(true, false);
    else if (m.has_L) RW_GO(false, true);
    else RW_GO(false, false);
  }
#undef RW_GO
  PBX_LAUNCH_CHECK(ctx);
  return PBX_OK;
}

static int nr_walk_per_step(pbx_ctx* ctx, const NrPlan& pl, NrArgs a, const NrModel& m,
                            int lik_kind, const NrLik& lik) {
  if (nr_extras(a, m)) nr_init_kernel<true><<<(a.C + 255) / 256, 256, 0, ctx->stream>>>(a, m);
  else nr_init_kernel<false><<<(a.C + 255) / 256, 256, 0, ctx->stream>>>(a, m);
  PBX_LAUNCH_CHECK(ctx);
  for (int k = 0; k < a.T; ++k) {
    a.k = k;
    a.gstep = a.step0 + k;
    int rc = nr_launch_step(ctx, pl, a, m, lik_kind, lik);
    if (rc) return rc;
  }
  return PBX_OK;
}

extern "C" int pbx_mh_normreg_run(pbx_ctx* ctx, const pbx_mh_normreg_params* p) {
  PBX_REQUIRE(ctx != nullptr, "pbx_mh_normreg_run: null ctx");
  int rc = nr_validate(p, "pbx_mh_normreg_run", true);
  if (rc) return rc;
  PBX_CUDA(cudaSetDevice(ctx->device));
  NrModel m;
  nr_fill_model(p, m);
  NrArgs a = nr_args(p);
  const NrLik lik{p->lik_df, p->lik_logc};
  // variant 3: sufficient statistics, else a small problem: the walk in one launch;
  // otherwise one launch per step
  const bool suffstat = p->variant == 3, small = !suffstat && rw_applies(p);
  NrPlan pl{};
  if (small) {
    PBX_REQUIRE(p->n_obs <= RW_MAXN, "pbx_mh_normreg_run: variant 4 needs n_obs <= %d", RW_MAXN);
  } else if (!suffstat) {
    pl = nr_plan(ctx, p);
    a.n_slices = pl.n_slices;
    rc = nr_workspace(ctx, pl, a.C, m.P, &a.partial, &a.counters, &a.prop);
    if (rc) return rc;
    a.theta_in = a.prop;
  }
  PBX_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
  if (a.T > 0) {
    if (suffstat) rc = nr_walk_suffstat(ctx, a, m);
    else if (small)
      rc = p->lik_kind == PBX_LIK_STUDENT_T      ? nr_walk_small<PBX_LIK_STUDENT_T>(ctx, a, m, lik)
           : p->lik_kind == PBX_LIK_STUDENT_T_NU ? nr_walk_small<PBX_LIK_STUDENT_T_NU>(ctx, a, m, lik)
                                                 : nr_walk_small<PBX_LIK_NORMAL>(ctx, a, m, lik);
    else rc = nr_walk_per_step(ctx, pl, a, m, p->lik_kind, lik);
    if (rc) return rc;
  }
  PBX_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
  return PBX_OK;
}

extern "C" int pbx_normreg_logjoint(pbx_ctx* ctx, const pbx_mh_normreg_params* p,
                                    const double* theta, double* out) {
  PBX_REQUIRE(ctx != nullptr && theta != nullptr && out != nullptr,
              "pbx_normreg_logjoint: null argument");
  int rc = nr_validate(p, "pbx_normreg_logjoint", false);
  if (rc) return rc;
  PBX_CUDA(cudaSetDevice(ctx->device));
  NrModel m;
  nr_fill_model(p, m);
  NrArgs a = nr_args(p);
  a.theta_in = theta;
  a.eval_out = out;
  if (p->variant == 3) {
    PBX_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
    NrStats* st = nullptr;
    rc = pbx_ss_compute(ctx, m.has_slope ? p->x_obs : nullptr, p->y_obs, p->n_obs, &st);
    if (rc) return rc;
    ss_eval_kernel<<<(a.C + 255) / 256, 256, 0, ctx->stream>>>(a, m, st);
    PBX_LAUNCH_CHECK(ctx);
    PBX_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
    return PBX_OK;
  }
  const NrPlan pl = nr_plan(ctx, p);
  a.n_slices = pl.n_slices;
  rc = nr_workspace(ctx, pl, a.C, m.P, &a.partial, &a.counters, &a.prop);
  if (rc) return rc;
  a.mode = 1;
  a.T = 1; a.thin = 1;
  PBX_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
  rc = nr_launch_step(ctx, pl, a, m, p->lik_kind, NrLik{p->lik_df, p->lik_logc});
  if (rc) return rc;
  PBX_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
  return PBX_OK;
}
