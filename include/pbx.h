/*
 * pbx.h -- C ABI of libpbx, the B200 (sm_100a) drop-in for the probayes hot path.
 *
 * The reference (Bhumbra/probayes) is pure Python and has no FFI of its own; the
 * seams this ABI sits behind are the reference's Python entry points for the
 * path (cited per function below, paths relative to the reference checkout).
 * The Python host mirror (probayes_b200/) binds these with ctypes; INTEGRATION.md
 * shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - plain C, no exceptions / Python objects / torch types cross the boundary;
 *   - every function returns PBX_OK (0) or a negative pbx_status; the message of
 *     the last failure on the calling thread is at pbx_last_error();
 *   - the CALLER allocates every buffer.  Pointers documented "device" are CUDA
 *     device pointers valid on the context's device (e.g. torch data_ptr()),
 *     "host" are ordinary host pointers read before the call returns;
 *   - calls are asynchronous on the context's stream unless named *_host or
 *     *_sync; buffers must stay alive until the stream is synchronised;
 *   - a context is bound to one GPU and is not thread-safe (the reference is
 *     single-threaded with global RNG state); use one context per GPU/process;
 *   - all arithmetic is fp64 (probayes/constants.py:7), chain-minor layouts
 *     ([.., C]) so that warps read/write coalesced.
 */
#ifndef PBX_H
#define PBX_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define PBX_API __attribute__((visibility("default")))
#else
#define PBX_API
#endif

#define PBX_VERSION 100            /* 0.1.0 */
#define PBX_MAX_DIMS 8             /* max state dimension of the small-target MH kernel */
#define PBX_MAX_PARAMS 3           /* (b0, b1, sigma) */

typedef enum {
  PBX_OK = 0,
  PBX_ERR_INVALID = -1,            /* bad argument */
  PBX_ERR_CUDA = -2,               /* CUDA runtime error (message has the string) */
  PBX_ERR_UNSUPPORTED = -3,        /* outside the catalogue (no CPU fallback by design) */
  PBX_ERR_NOMEM = -4
} pbx_status;

/* accept rule ---------------------------------------------------------------
 * REFERENCE: s = min(1, lin(p')/max(tiny, lin(p))), accept iff s >= t, with the
 *   clamped exp of probayes/pscales.py:56-65,219-236 (sp_utils.py:19-37).
 * LOG: accept iff coef*(logp' - logp) >= log(t); identical decisions wherever the
 *   reference's linear ratio does not underflow, and the only usable rule for
 *   N >~ 200 observations (SURVEY.md section 0.3). */
#define PBX_ACCEPT_REFERENCE 0
#define PBX_ACCEPT_LOG 1
/* proposal draw kind (probayes/field.py:469-531, variable.py:600-638) */
#define PBX_PROP_NORMAL 0          /* delta_j = scale_j * z_j,  z ~ N(0,1) (then optional L) */
#define PBX_PROP_UNIFORM 1         /* delta_j = -scale_j + 2 scale_j r_j, r ~ U(0,1)  ([delta] lists) */
#define PBX_PROP_SPHERICAL 2       /* u_j ~ U(-R, R); delta_j = (u_j R / |u|) scale_j  ((delta,) tuples,
                                      field.py:509-531; R = prop_radius) */
/* iid likelihood family of K2 / K3 (pbx_mh_normreg_params.lik_kind) */
#define PBX_LIK_NORMAL 0           /* scipy.stats.norm.logpdf */
#define PBX_LIK_STUDENT_T 1        /* scipy.stats.t.logpdf (cauchy.logpdf: df = 1) */
#define PBX_LIK_STUDENT_T_NU 2     /* scipy.stats.t.logpdf with df = nu a model parameter:
                                      params (mu, sigma, nu) */

typedef struct pbx_ctx pbx_ctx;

typedef struct {
  int32_t device;
  int32_t cc_major, cc_minor;
  int32_t sm_count;
  int32_t l2_bytes_mb;
  int32_t smem_per_block_optin;
  int64_t global_mem_bytes;
  char name[64];
} pbx_devinfo;

PBX_API int pbx_version(void);
PBX_API const char* pbx_last_error(void);
PBX_API int pbx_device_count(int* n);
PBX_API int pbx_device_info(int device, pbx_devinfo* out);

/* own_stream != 0: the context creates (and later destroys) its own non-blocking
 * stream and `stream` is ignored.  own_stream == 0: run on the caller's
 * cudaStream_t `stream` (passed as void*; NULL is the default stream), e.g. torch's
 * current stream so that kernels are ordered with the caller's allocations/copies. */
PBX_API int pbx_ctx_create(int device, void* stream, int32_t own_stream, pbx_ctx** out);
PBX_API int pbx_ctx_destroy(pbx_ctx* ctx);
PBX_API int pbx_ctx_sync(pbx_ctx* ctx);
/* number of kernels this context has launched since creation (bench: gpu_launches) */
PBX_API int64_t pbx_ctx_launch_count(pbx_ctx* ctx);
/* device time in ms of the kernels launched by the most recent *_run call on this
 * context, measured with CUDA events on the context's stream; syncs the stream. */
PBX_API int pbx_ctx_last_kernel_ms(pbx_ctx* ctx, float* ms);

/* pinned host memory for the *_host entry points */
PBX_API int pbx_host_alloc(size_t bytes, void** out);
PBX_API int pbx_host_free(void* p);

/* ---------------------------------------------------------------------------
 * K1  batched-chain Metropolis-Hastings on a multivariate-normal target.
 * Replaces the SP.next loop (probayes/sp.py:221-258, sp_utils.py:8-37) when the
 * target is scipy.stats.multivariate_normal (probayes/prob.py:347-360) and the
 * proposal is an additive delta (field.py:534-552, rf.py:340-354), e.g.
 * examples/mcmc/mcmc_prob4a.py:38-51.  One chain per reference sampler.
 * ------------------------------------------------------------------------- */
typedef struct {
  int32_t n_chains;        /* C (local to this GPU) */
  int32_t n_dims;          /* D, 1..PBX_MAX_DIMS */
  int32_t n_steps;         /* T steps in this call */
  int32_t thin;            /* record every thin-th step (step index % thin == thin-1) */
  int64_t step0;           /* global index of this call's first step; step 0 accepts
                              unconditionally (sp.py:253, sp_utils.py:24-25) */
  int64_t chain0;          /* global id of local chain 0 (Philox stream is keyed on
                              the global chain id => results invariant to sharding) */
  uint64_t seed;
  int32_t log_pscale;      /* recorded prob: 0 = pdf (linear pscale), 1 = logpdf */
  int32_t accept_mode;     /* PBX_ACCEPT_* */
  int32_t prop_kind;       /* PBX_PROP_* */
  int32_t has_prop_mat;    /* delta = prop_mat @ (scaled draw)  (rf.py:346-348) */
  int32_t kernel_variant;  /* 0 auto; 1 one thread per chain; 2 warp-specialised, exact reference
                              arithmetic in the decision; 4 warp-specialised, decisions on the
                              whitened state (the auto choice for the log rule, n_dims <= 4) */
  int32_t reserved0;
  double mean[PBX_MAX_DIMS];
  /* whitening matrix U (row-major [D][D]) of scipy's _PSD with the value
   * permutation of prob.py:349-358 folded into its rows: maha = |(x-mean') U'|^2 */
  double whiten[PBX_MAX_DIMS * PBX_MAX_DIMS];
  double norm_c;           /* D log 2pi + log_pdet;  logpdf = -0.5*(norm_c + maha), scipy's form */
  double prop_scale[PBX_MAX_DIMS];
  double prop_mat[PBX_MAX_DIMS * PBX_MAX_DIMS];   /* row-major lower-triangular L */
  double prop_radius;      /* PBX_PROP_SPHERICAL only */
  /* device buffers */
  double* state;           /* [D][C] in/out: current state */
  double* state_lp;        /* [C]    in/out: log-density of state (ignored on input when step0 == 0) */
  const double* inj_delta; /* [T][D][C] injected raw proposal draws, or NULL = Philox */
  const double* inj_thresh;/* [T][C] injected thresholds, or NULL = Philox */
  double* out_x;           /* [T/thin][D][C] or NULL */
  double* out_prob;        /* [T/thin][C] or NULL */
  uint8_t* out_accept;     /* [T][C] or NULL (u: 1 = True, 0 = None) */
  double* out_score;       /* [T][C] or NULL (s; NaN on the unconditional first step) */
  int64_t* accept_count;   /* [C] accumulated, or NULL */
  double* stat_sum;        /* [D][C] accumulated sum of the retained state, or NULL */
  double* stat_sumsq;      /* [D][C] accumulated sum of squares, or NULL */
  double* out_xprop;       /* [T][D][C] or NULL: the proposal of every step (opqr.p values) */
  double* out_pprop;       /* [T][C] or NULL: the target density at the proposal (opqr.p.prob) */
  /* set_delta(..., bound=True) (probayes/variable.py:700-739): a proposal beyond a CLOSED
   * limit is clipped to it, beyond an OPEN limit it bounces back to the current value.  The
   * proposal then depends on the state, so these walks run the one-thread-per-chain kernel. */
  int32_t prop_bound;      /* 0 / 1 */
  int32_t reserved1;
  double lims[PBX_MAX_DIMS][2];
  int32_t open_end[PBX_MAX_DIMS][2];
} pbx_mh_mvn_params;

PBX_API int pbx_mh_mvn_run(pbx_ctx* ctx, const pbx_mh_mvn_params* p);

/* Whole-walk call with HOST output buffers: runs the walk in chunks of
 * chunk_steps on the device and streams out_x/out_prob back to (pinned) host
 * memory on a copy stream, overlapped with the next chunk.  state/state_lp are
 * HOST [D][C]/[C] in/out; out_x/out_prob HOST; the inj_*, out_accept, out_score
 * pointers must be NULL; accept_count/stat_* are HOST or NULL.  Synchronous. */
PBX_API int pbx_mh_mvn_walk_host(pbx_ctx* ctx, const pbx_mh_mvn_params* p, int32_t chunk_steps);

/* ---------------------------------------------------------------------------
 * K2  streaming normal log-likelihood MH (iid=True, joint=True, log pscale).
 *   y_i ~ N(b0 + b1 x_i, sigma)   params (b0, b1, sigma)   has_slope = 1
 *   y_i ~ N(mu, sigma)            params (mu, sigma)       has_slope = 0
 *   y_i ~ t_nu(mu, sigma)         params (mu, sigma, nu)   has_slope = 0  (PBX_LIK_STUDENT_T_NU)
 * Replaces RF.__call__(iid=True) + SD.__call__(joint=True) evaluated every step
 * (probayes/rf.py:541-581, pd.py:332-370, sd.py:148-161) with scipy.stats.norm
 * .logpdf as the likelihood (examples/mcmc/metrohast_norm1d.py:30-31,
 * gibbs_linreg.py:35-36), box-uniform priors in ufun space (rv.py:153-166,
 * rv_utils.py:8-47) and ufun-space proposals (variable.py:693-697), optionally coloured by
 * the Cholesky factor of a covariance-matrix transition (has_prop_mat, rf.py:346-348).
 * ------------------------------------------------------------------------- */
typedef struct {
  int32_t n_chains;
  int32_t n_params;        /* 2 or 3 (3: has_slope, or PBX_LIK_STUDENT_T_NU) */
  int32_t n_steps;
  int32_t thin;
  int64_t step0;
  int64_t chain0;
  uint64_t seed;
  int32_t has_slope;
  int32_t accept_mode;
  double accept_coef;      /* linear proposal density multiplied into the log target by
                              hastings_scores (sp_utils.py:62-64); 1.0 for metropolis */
  int32_t prop_kind;
  int32_t variant;         /* 0 auto; 1 chains-in-registers + TMA-staged obs tiles;
                              2 obs-per-thread streaming + warp-shuffle reduction;
                              3 (opt-in) centred sufficient statistics: one reduction over
                              the observations, then O(1) per likelihood evaluation and the
                              whole walk in one launch -- same values to <= 1e-15;
                              4 resident observations: a warp per chain, observations in
                              shared memory, the whole walk in one launch, term-by-term
                              arithmetic -- the auto choice for small problems (n_obs <= 8192
                              and n_chains * n_obs <= 2^24), where a kernel launch per MH step
                              would be all the time there is */
  int64_t n_obs;
  const double* x_obs;     /* device [N] (unused when !has_slope) */
  const double* y_obs;     /* device [N] */
  double lims[PBX_MAX_PARAMS][2];        /* vlims */
  int32_t open_end[PBX_MAX_PARAMS][2];   /* 1 = exclusive end (tuple in vset) */
  int32_t log_ufun[PBX_MAX_PARAMS];      /* 1 = (np.log, np.exp) ufun */
  int32_t prop_bound;      /* set_delta(..., bound=True): proposals are constrained to the
                              vset (variable.py:700-739) -- closed ends clip, a proposal
                              beyond an open end bounces back to the current value */
  double prop_scale[PBX_MAX_PARAMS];
  double prop_radius;      /* PBX_PROP_SPHERICAL only */
  double* state;           /* [P][C] in/out */
  double* state_lp;        /* [C] in/out */
  const double* inj_delta; /* [T][P][C] or NULL */
  const double* inj_thresh;/* [T][C] or NULL */
  double* out_x;           /* [T/thin][P][C] or NULL */
  double* out_prob;        /* [T/thin][C] (log-joint) or NULL */
  uint8_t* out_accept;     /* [T][C] or NULL */
  double* out_score;       /* [T][C] or NULL */
  int64_t* accept_count;   /* [C] or NULL */
  double* stat_sum;        /* [P][C] or NULL */
  double* stat_sumsq;      /* [P][C] or NULL */
  double* out_xprop;       /* [T][P][C] or NULL: the proposal of every step (opqr.p values) */
  double* out_pprop;       /* [T][C] or NULL: the log-joint at the proposal (opqr.p.prob) */
  /* set_tran(covariance) (rf.py:209-220,346-348), as K1's has_prop_mat: the delta of every
   * step -- drawn, scaled or spherically rescaled, or injected -- is multiplied by prop_mat
   * before the ufun move and the bound rule.  prop_mat is row-major [P][P] in its first P*P
   * entries, lower-triangular with a positive diagonal and finite (pbx_mh_normreg_run returns
   * PBX_ERR_INVALID otherwise); pbx_normreg_logjoint ignores both fields. */
  int32_t has_prop_mat;
  int32_t reserved0;
  double prop_mat[PBX_MAX_PARAMS * PBX_MAX_PARAMS];
  /* the iid likelihood of every observation, y_i ~ family(loc_i, sigma).  PBX_LIK_NORMAL (a
   * zeroed tail) is scipy.stats.norm.logpdf; PBX_LIK_STUDENT_T is scipy.stats.t.logpdf with
   * df = lik_df (cauchy.logpdf: lik_df = 1), per observation
   *   lik_logc - (lik_df + 1)/2 log1p(z^2 / lik_df) - log sigma,   z = (y_i - loc_i) / sigma,
   * where the caller computes lik_logc = log(poch(df/2, 1/2)) - (log df + log pi)/2 as scipy
   * does (lgamma((df+1)/2) - lgamma(df/2) cancels: 9e-7 relative at df = 1e9).  Student-t needs
   * 0 < lik_df < inf and a finite lik_logc, and refuses variant 3 (the t likelihood has no
   * sufficient statistics); both entry points return PBX_ERR_INVALID otherwise.
   * PBX_LIK_STUDENT_T_NU is the same density with df = nu sampled as the model's third
   * parameter, theta = (mu, sigma, nu): n_params = 3, has_slope = 0, lik_df = lik_logc = 0
   * (unread: the kernels compute logc(nu) of every chain and step, as
   * lgamma((nu+1)/2) - lgamma(nu/2) - log(nu pi)/2 below nu = 16 and an asymptotic series
   * above, which does not cancel), nu's prior box admitting nu > 0 only (lims[2][0] > 0, or
   * lims[2][0] = 0 with an open lower end), and no variant 3. */
  int32_t lik_kind;        /* PBX_LIK_* */
  int32_t reserved1;
  double lik_df;
  double lik_logc;
} pbx_mh_normreg_params;

PBX_API int pbx_mh_normreg_run(pbx_ctx* ctx, const pbx_mh_normreg_params* p);

/* log-joint (likelihood + box priors) of theta[P][C] -> out[C]; the array density
 * evaluation on its own ("log-likelihood evals"). Uses the same kernels as K2. */
PBX_API int pbx_normreg_logjoint(pbx_ctx* ctx, const pbx_mh_normreg_params* model,
                         const double* theta, double* out);

/* ---------------------------------------------------------------------------
 * K3/K4  discrete grid exact inference of a normal (mu, sigma) posterior.
 * Replaces SD.__call__({x: data, mu: {M}, sigma: {S}}, iid=True, joint=True)
 * (probayes/sd.py:148-161, rf.py:565-581, pd.py:332-370, pd_utils.py:85-328)
 * and PD.conditionalise / PD.marginal (pd.py:136-165,168-211,214-295), as in
 * examples/dgei/dgei_norm1d_improved.py:36-43.
 * ------------------------------------------------------------------------- */
/* out[m][s] = logprior_mu[m] + logprior_sigma[s] + sum_i norm.logpdf(x_i; mu_m, sigma_s) */
PBX_API int pbx_grid_norm_logjoint(pbx_ctx* ctx, const double* x_obs, int64_t n_obs,
                           const double* mu, int32_t n_mu,
                           const double* sigma, int32_t n_sigma,
                           const double* logprior_mu, const double* logprior_sigma,
                           double* out);
/* the same grid with a Student-t likelihood: out[m][s] = logprior_mu[m] + logprior_sigma[s]
 * + sum_i t.logpdf(x_i; df, mu_m, sigma_s), logc as pbx_mh_normreg_params.lik_logc
 * (0 < df < inf, logc finite; PBX_ERR_INVALID otherwise) */
PBX_API int pbx_grid_t_logjoint(pbx_ctx* ctx, const double* x_obs, int64_t n_obs,
                                const double* mu, int32_t n_mu, const double* sigma,
                                int32_t n_sigma, const double* logprior_mu,
                                const double* logprior_sigma, double* out, double df,
                                double logc);
/* opt-in: the same values (<= 1e-15) from centred sufficient statistics of the
 * observations: one reduction over x_obs, then O(1) per cell instead of O(N) */
PBX_API int pbx_grid_norm_logjoint_ss(pbx_ctx* ctx, const double* x_obs, int64_t n_obs,
                                      const double* mu, int32_t n_mu, const double* sigma,
                                      int32_t n_sigma, const double* logprior_mu,
                                      const double* logprior_sigma, double* out);
/* The PD normalise / marginal algebra (PD.conditionalise + both PD.marginal calls,
 * pd.py:214-295,136-165) in TWO passes over the grid, for log-pscale (linear = 0) or
 * linear-pscale (linear = 1) input.  First pass: out2[0] = max (0 for linear input),
 * out2[1] = sum exp_logp(v - max) (plain sum for linear input), from ONE read of v with
 * online rescaling (device scalars) */
PBX_API int pbx_grid_max_sumexp(pbx_ctx* ctx, const double* v, int64_t n, int32_t linear,
                                double* out2);
/* slab-sharded grids: sum_inout[0] *= exp(local_max[0] - global_max[0]) (device scalars), so
 * that per-rank sums taken against the local maxima can be all-reduced */
PBX_API int pbx_grid_rescale_sumexp(pbx_ctx* ctx, const double* local_max,
                                    const double* global_max, double* sum_inout);
/* Second pass over the grid prob [n_mu, n_sigma] (device):
 *   post[m][s] = log_prob( exp_logp(prob - gmax) / max(tiny, gsum) )   (pd.py:285-295)
 *   marg_mu[m]    = sum_s exp_logp(post[m][s])                          (pd.py:162-163)
 *   marg_sigma[s] = sum_m exp_logp(post[m][s])   (partial over this slab's rows)
 * linear = 1: post = prob / max(tiny, gsum) and the marginals are plain sums (gmax unused).
 * post may be NULL (marginals only) or alias prob (in place).  The marginals' clamped logs
 * are fused: marg_log_flags bit 0 -> marg_mu = log_prob(sum),
 * bit 1 -> marg_sigma likewise (leave a bit clear where the sum must be all-reduced first);
 * bit 2 -> PD.marginalise semantics (pd.py:162-164): the terms exp_logp(p) are summed as they
 * are, subnormals included, instead of conditionalise's clamp of q < tiny to zero */
PBX_API int pbx_grid_posterior2(pbx_ctx* ctx, const double* prob, int32_t n_mu, int32_t n_sigma,
                                const double* gmax, const double* gsum, int32_t linear,
                                double* post, double* marg_mu, double* marg_sigma,
                                int32_t marg_log_flags);
/* v[i] = log_prob(v[i]) in place (clamped log of pscales.py:44-53) */
PBX_API int pbx_log_prob_inplace(pbx_ctx* ctx, double* v, int64_t n);
/* v[i] = exp_logp(v[i]) in place (clamped exp of pscales.py:56-65; PD.rescaled) */
PBX_API int pbx_exp_logp_inplace(pbx_ctx* ctx, double* v, int64_t n);

/* ---------------------------------------------------------------------------
 * Ordinary Monte Carlo with rejection sampling: SP.next with a proposal DENSITY
 * (set_prop) and custom scores / thresh / update (probayes/sp.py:221-258, sd.py:228-250,
 * rf.py:146-161,584-602), as in examples/omc/omc_rejection_sp_circle.py:26-39.  Catalogue:
 * target = indicator of a ball; proposal density = product of normal pdfs or the box-uniform
 * density; score = p or the safe ratio p / q; threshold ~ U(thresh_lo, thresh_hi);
 * update = (s >= t).  One sample per reference step; samples shard like chains (global
 * sample id = sample0 + t).
 * ------------------------------------------------------------------------- */
typedef struct {
  int32_t n_params;        /* P variables, 1..8 */
  int32_t target_kind;     /* 0 = indicator( |x - centre|^2 <= radius^2 ) */
  int32_t prop_kind;       /* 0 = prod_j norm.pdf(x_j; loc_j, scale_j); 1 = prod_j 1 / length_j */
  int32_t score_mode;      /* 0 = p; 1 = p / max(tiny, q) */
  int64_t n_samples;       /* T */
  int64_t sample0;
  uint64_t seed;
  double lims[8][2];       /* box of every variable (finite) */
  int32_t log_ufun[8];     /* uniform in log space (the (np.log, np.exp) ufun) */
  double target_centre[8];
  double target_radius;
  double prop_loc[8];
  double prop_scale[8];
  double thresh_lo, thresh_hi;
  const double* inj_unif;  /* [T][P + 1] injected uniforms (draws, then threshold) or NULL */
  double* out_theta;       /* [P][T] the proposals */
  double* out_p;           /* [T] target at the proposal */
  double* out_q;           /* [T] proposal density at the proposal */
  double* out_s;           /* [T] score */
  double* out_t;           /* [T] threshold */
  uint8_t* out_u;          /* [T] update flag (1 = kept) */
} pbx_rejection_params;
PBX_API int pbx_rejection_sample(pbx_ctx* ctx, const pbx_rejection_params* p);

/* ---------------------------------------------------------------------------
 * K5  batched Gibbs sweep over the conditionals of a multivariate normal.
 * Replaces RF.eval_tfun -> sample_cond_cov -> CondCov.interp
 * (probayes/rf.py:413-462, rf_utils.py:50-65, cond_cov.py:22-65) with the
 * per-step evaluation of the mvn target (sd.py:286), as in
 * examples/mcmc/gibbs_norm2d.py:15-22.  One step = one coordinate update
 * (tsteps=1); coordinate = (step0 + k) mod d.
 * Calls covering whole sweeps (step0, n_steps and thin multiples of d; d >= 5) run the
 * conditional means on the FP64 tensor cores, 8 coordinates per block in closed form; any
 * other step range runs coordinate by coordinate.  Same results up to summation order.
 * Native uniforms: global step g uses the 52-bit uniform of words (0, 1) (bit 2 of g clear)
 * or (2, 3) (bit 2 set) of Philox block (seed, g & ~4, chain0 + c, slot 0); the inverse
 * normal cdf is the table-driven pbx_ndtri below.
 * ------------------------------------------------------------------------- */
typedef struct {
  int32_t n_chains;
  int32_t n_dims;          /* d, 1..128 */
  int32_t n_steps;         /* coordinate steps in this call */
  int32_t thin;
  int64_t step0;
  int64_t chain0;
  uint64_t seed;
  int32_t log_pscale;
  int32_t want_prob;       /* evaluate + record the target density */
  const double* mean;      /* device [d] */
  const double* coef;      /* device [d][d] CondCov regression rows (0 on the diagonal) */
  const double* stdv;      /* device [d] conditional stdv */
  const double* cdf_lo;    /* device [d] fixed cdf limits (cond_cov.py:38-39) */
  const double* cdf_hi;    /* device [d] */
  const double* whiten;    /* device [d][d] row-major, value permutation folded in */
  const double* dens_mean; /* device [d] mean of the density in natural order with the
                              permutation folded in (NULL = mean); see prob.py:349-358 */
  double norm_c;           /* d log 2pi + log_pdet */
  double* state;           /* [d][C] in/out */
  const double* inj_runif; /* [T][C] injected U(0,1) draws (row k = step step0 + k) or
                              NULL = Philox */
  double* out_x;           /* [T/thin][d][C] or NULL */
  double* out_prob;        /* [T/thin][C] or NULL */
  double* stat_sum;        /* [d][C] accumulated over the RECORDED states, or NULL */
  double* stat_sumsq;      /* [d][C] or NULL */
} pbx_gibbs_mvn_params;

PBX_API int pbx_gibbs_mvn_run(pbx_ctx* ctx, const pbx_gibbs_mvn_params* p);

/* batched mvn log-density: x[d][C] -> out[C] (logpdf, or pdf when !log_pscale);
 * d >= 64 routes the [C,d]x[d,d] whitening product through FP64 tensor-core MMA. */
PBX_API int pbx_mvn_logpdf(pbx_ctx* ctx, const double* x, int32_t n_dims, int64_t n_chains,
                   const double* mean, const double* whiten, double norm_c,
                   int32_t log_pscale, double* out);

/* Inverse normal CDF as the Gibbs draws evaluate it (the reference: scipy.stats.norm.ppf ==
 * ndtri, vtypes.py:186 / cond_cov.py:58-65): out[i] = ndtri(u[i]), table-driven degree-5
 * polynomials on 64 segments per binade of min(u, 1 - u) (pbx_ndtri.cuh; <= 7e-16 relative to
 * max(|x|, 1e-3)), CUDA's normcdfinv outside the table (p < 2^-64, u <= 0, u >= 1).
 * pbx_ndtri: device arrays.  pbx_ndtri_host: host arrays, the same table and arithmetic on
 * the CPU without touching a GPU (NaN outside the table) -- a self-test hook, not a compute
 * fallback. */
PBX_API int pbx_ndtri(pbx_ctx* ctx, const double* u, int64_t n, double* out);
PBX_API int pbx_ndtri_host(const double* u, int64_t n, double* out);

/* ---------------------------------------------------------------------------
 * Chain summaries for R-hat: from per-chain sums over n_steps retained states,
 * out[j][0..3] = ( sum_c mean_cj, sum_c mean_cj^2, sum_c var_cj, C ) per dim j;
 * these are what the ranks all-reduce (SURVEY.md section 8e).  out: device [D][4].
 * ------------------------------------------------------------------------- */
PBX_API int pbx_reduce_chain_stats(pbx_ctx* ctx, const double* stat_sum, const double* stat_sumsq,
                           int32_t n_dims, int64_t n_chains, int64_t n_steps, double* out);

/* ---------------------------------------------------------------------------
 * K6: PD post-processing on large grids / sample sets -- SURVEY.md section 8f rank 2.
 * Replaces the numpy passes of PD.sorted (np.argsort + fancy indexing,
 * probayes/pd.py:464-493), PD.quantile (rescale + np.cumsum + div_prob + np.digitize,
 * pd.py:408-461) and PD.expectation (rescale + np.sum(prob*val), pd.py:373-405).
 * All HBM-bound; deterministic (fixed reduction / scan order, no atomics on doubles).
 * ------------------------------------------------------------------------- */

/* bytes of device workspace pbx_argsort_f64 needs for n keys */
PBX_API int pbx_argsort_workspace_bytes(int64_t n, size_t* bytes);
/* Ascending STABLE argsort of n doubles (np.argsort(kind='stable') order; -0.0 sorts
 * before +0.0, NaNs last): LSD radix sort, 8-bit digits, passes whose digit is constant
 * over all keys are skipped.  keys: device [n] (not modified); order: device int32 [n]
 * out; keys_sorted: device [n] out or NULL.  n < 2^31. */
PBX_API int pbx_argsort_f64(pbx_ctx* ctx, const double* keys, int64_t n, int32_t* order,
                            double* keys_sorted, void* workspace, size_t workspace_bytes);
/* dst[i] = src[idx[i]]  (values / probabilities re-ordered by a sort: pd.py:478-492) */
PBX_API int pbx_gather_f64(pbx_ctx* ctx, const double* src, const int32_t* idx, int64_t n,
                           double* dst);
/* 2-D take along an axis: axis 0: dst[i][j] = src[idx[i]][j]; axis 1: dst[i][j] = src[i][idx[j]]
 * (prob[tuple(slices)] of pd.py:476-478 for a grid PD) */
PBX_API int pbx_take_axis_f64(pbx_ctx* ctx, const double* src, int64_t rows, int64_t cols,
                              int32_t axis, const int32_t* idx, double* dst);
/* bytes of device workspace for pbx_cumprob_f64 / pbx_expectation_f64 */
PBX_API int pbx_scan_workspace_bytes(int64_t n, size_t* bytes);
/* cum[i] = (sum_{k<=i} lin(prob[k])) / max(tiny, sum_k lin(prob[k])), lin = clamped exp
 * when log_pscale (pscales.py:56-65,100-131,219-236); total (device, 1 double, may be NULL)
 * receives the un-normalised sum.  cum may alias prob.  Three-phase reduce-then-scan:
 * 24 B of traffic per element, bit-reproducible. */
PBX_API int pbx_cumprob_f64(pbx_ctx* ctx, const double* prob, int64_t n, int32_t log_pscale,
                            double* cum, double* total, void* workspace, size_t workspace_bytes);
/* np.maximum(0, np.digitize(q, cum) - 1) for nq quantiles (pd.py:430): idx_out device
 * int64 [nq]; q host [nq]; cum device [n] non-decreasing. nq <= 64. */
PBX_API int pbx_digitize_f64(pbx_ctx* ctx, const double* cum, int64_t n, const double* q,
                             int32_t nq, int64_t* idx_out);
/* Sums for PD.expectation over a [rows][cols] prob array (rows = 1 for sample sets):
 * out[0] = sum lin(p); out[1+k] = sum_ij lin(p_ij) row_vals[k][i], k < n_row_vals;
 * out[1+n_row_vals+k] = sum_ij lin(p_ij) col_vals[k][j].  row_vals: device
 * [n_row_vals][rows], col_vals: device [n_col_vals][cols] (either may be NULL with count 0;
 * counts <= 4).  out: device [1 + n_row_vals + n_col_vals].  The quotient
 * div_prob(numerator, total) is left to the caller (2 scalars). */
PBX_API int pbx_expectation_f64(pbx_ctx* ctx, const double* prob, int64_t rows, int64_t cols,
                                int32_t log_pscale, const double* row_vals, int32_t n_row_vals,
                                const double* col_vals, int32_t n_col_vals, double* out,
                                void* workspace, size_t workspace_bytes);

/* Binary PD algebra with broadcasting (SURVEY.md rows a14-a16, a19): op 0 = product rule
 * (PD.__mul__ -> pd_utils.product -> pscales.prod_rule, probayes/pd.py:564-565,
 * pd_utils.py:85-328, pscales.py:160-216), op 1 = safe division (PD.__truediv__ ->
 * pscales.div_prob, pd.py:572-615, pscales.py:219-236).  a: device [a_rows][a_cols] with
 * a_rows in {1, rows}, a_cols in {1, cols}; b likewise; *_log: 1 = log pscale, 0 = linear;
 * out: device [rows][cols].  Product: out_log must be (a_log || b_log). */
PBX_API int pbx_pd_binary_f64(pbx_ctx* ctx, int32_t op, const double* a, int64_t a_rows,
                              int64_t a_cols, int32_t a_log, const double* b, int64_t b_rows,
                              int64_t b_cols, int32_t b_log, int64_t rows, int64_t cols,
                              int32_t out_log, double* out);

/* ---------------------------------------------------------------------------
 * Ordinary Monte Carlo random sampling of box-bounded parameters -- SURVEY.md section 8f
 * rank 3.  Replaces Variable.evaluate({0}) -> vtypes.uniform(ulims, n=0) -> ufun^-1
 * (probayes/variable.py:558-583, vtypes.py:186) called once per sampler step by
 * SP.next's no-proposal branch (sp.py:229-234), as in examples/omc/omc_rs_sp_norm1d.py:
 * theta[j][t] = ufun_j^-1( ulo_j + (uhi_j - ulo_j) r ),  r ~ U(0,1); the log-joint of
 * the samples is then pbx_normreg_logjoint.  Draws: injected uniforms inj_unif
 * [n_samples][n_params] (reference draw order: parameters in field order per step), or
 * Philox block (seed, step = sample0 + t, chain = 0, slot j/2) -> (u52, u32).
 * lims host [n_params][2] (value space), log_ufun host [n_params]; out device
 * [n_params][n_samples]. n_params <= 8.
 * ------------------------------------------------------------------------- */
PBX_API int pbx_box_sample(pbx_ctx* ctx, int32_t n_params, int64_t n_samples, const double* lims,
                           const int32_t* log_ufun, uint64_t seed, int64_t sample0,
                           const double* inj_unif, double* out);

/* FP64 FMA peak micro-benchmark (roofline denominator for the compute-bound
 * kernels; MEASURED_PEAKS.json has no FP64 figure). Returns TFLOP/s. */
PBX_API int pbx_fp64_peak(pbx_ctx* ctx, double* tflops);
/* Dependent-issue latency of DFMA / DADD in SM cycles (one warp, one dependent chain):
 * the constant that bounds the sequential part of a Markov chain step. */
PBX_API int pbx_fp64_dep_latency(pbx_ctx* ctx, double* dfma_cycles, double* dadd_cycles);

/* Self-test of the table-driven math K1's RNG path uses instead of libm (-2 log u,
 * sqrt, sincos(2 pi .), exp): u device [n] in (0,1), w device uint32 [n], out device
 * [5][n] = (-2 log u, sqrt(-2 log u), sin, cos of 2 pi (w + 0.5)/2^32, exp(-700 u)). */
PBX_API int pbx_selftest_fastmath(pbx_ctx* ctx, const double* u, const uint32_t* w, int64_t n,
                                  double* out);

#ifdef __cplusplus
}
#endif
#endif /* PBX_H */
