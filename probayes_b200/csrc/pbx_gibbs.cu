// pbx_gibbs.cu -- K5: batched Gibbs over the conditionals of a multivariate normal
// and the batched mvn density.
//
// Gibbs step (probayes/rf.py:446-462 -> rf_utils.py:50-65 -> cond_cov.py:42-65),
// one coordinate i = step mod d per step (tsteps=1), with the truncation limits fixed at
// construction (cond_cov.py:38-39):
//     u   = cdf_lo_i + (cdf_hi_i - cdf_lo_i) * r          r ~ U(0,1)  (vtypes.py:186)
//     x_i = ndtri(u) * stdv_i + mean_i + coef_i . (x_-i - mean_-i)
// The dot product is evaluated as c0_i + coef_i . x with c0_i = mean_i - coef_i . mean
// folded on the host (coef_ii = 0).  ndtri is the table-driven pbx_ndtri.cuh.
// Native uniforms: global step g takes the 52-bit uniform of words (0, 1) (bit 2 of g clear)
// or (2, 3) (bit 2 set) of Philox block (seed, g & ~4, chain, slot 0): steps g and g + 4 --
// consecutive coordinates of the same lane below -- share one block (oracle/philox.py
// gibbs_uniforms replays it).
//
// Two Gibbs kernels, both with four lanes per chain and the state vector in REGISTERS (lane q
// of a chain holds coordinates 4m + q):
//   gibbs_mvn_kernel      any step range, one coordinate at a time: the coefficient rows come
//                         from shared memory with 128-bit loads, the dot product finishes with
//                         two shuffle-adds;
//   gibbs_mvn_mma_kernel  whole sweeps, d >= 5: blocks of 8 coordinates in closed form on the
//                         FP64 tensor cores; at d = 64 it also evaluates the density of every
//                         recorded state.
//
// Density (probayes/prob.py:347-360 -> scipy multivariate_normal): maha = |(x - mean) W|^2.
// At d = 64 the [chains, d] x [d, d] whitening product runs on the FP64 tensor cores
// (mma.sync.m8n8k4.f64 -- tcgen05 has no FP64 kind), 8 chains per MMA row block, with the same
// code as the fused density; other d use a plain FMA kernel.
#include <math.h>
#include <vector>
#include "pbx_common.cuh"
#include "pbx_ndtri.cuh"

// threads per CTA of both Gibbs kernels when there are enough chains (gibbs_launch); measured
// on gibbs_mvn_kernel: 0.137 / 0.116 / 0.108 ms per sweep at 64 / 128 / 256
constexpr int kGbThreads = 256;
// minimum resident CTAs of 256 threads per SM for the tensor-core kernel at d <= 64 (124
// registers); capping at 80 registers for 3 CTAs was measured slower
constexpr int kGmMinBlocks = 2;

struct GibbsArgs {
  int C, d, T, thin;
  int64_t step0, chain0;
  uint64_t seed;
  const double* coef;     // [d][d]
  const double* c0;       // [d] (workspace: mean_i - coef_i . mean)
  const double* stdv;
  const double* cdf_lo;
  const double* cdf_hi;
  double* state;          // [d][C]
  const double* inj_runif;
  double* out_x;
  double* stat_sum;
  double* stat_sumsq;
  // fused target density of the recorded states (whole-sweep kernel, d = 64 only; else null)
  double* out_prob;
  const double* whiten;   // [64][64]
  const double* dens_mean;
  double norm_c;
  int log_pscale;
};

__global__ void gibbs_c0_kernel(const double* coef, const double* mean, int d, double* c0) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= d) return;
  double acc = 0.0;
  for (int j = 0; j < d; ++j) acc = fma(coef[(int64_t)i * d + j], mean[j], acc);
  c0[i] = mean[i] - acc;
}

static __device__ __align__(16) double g_ndtab[NDT_ROWS * NDT_NCOEF];   // 192 KB, read through L1
// the rows of the 10 binades nearest 0.5 (p >= 2^-11: all but 0.1 % of the draws),
// TRANSPOSED [coefficient][row] for the tensor-core kernel's shared-memory copy: a lane's
// six 64-bit loads then fall on banks that are uniform in its (random) row index
#define NDT_HOT_BINADES 10
#define NDT_HOT_ROWS (NDT_HOT_BINADES * NDT_SEGS)
#define NDT_HOT0 (NDT_ROWS - NDT_HOT_ROWS)
static __device__ __align__(16) double g_ndhot[NDT_NCOEF * NDT_HOT_ROWS];   // 30 KB

// outside the table (p < 2^-64, u <= 0, u >= 1, NaN): practically never taken, out of line
__device__ __noinline__ double gibbs_ndtri_cold(double u) { return normcdfinv(u); }

__device__ __forceinline__ double gibbs_ndtri(double u) {
  const bool upper = u > 0.5;
  const double p = upper ? 1.0 - u : u;                  // exact for u > 0.5
  const unsigned seg = ndt_segment(p);
  if (seg >= (unsigned)NDT_ROWS) return gibbs_ndtri_cold(u);
  const double2* row = reinterpret_cast<const double2*>(g_ndtab + (size_t)seg * NDT_NCOEF);
  double c[NDT_NCOEF];
#pragma unroll
  for (int j = 0; j < NDT_NCOEF / 2; ++j) {
    const double2 t = __ldg(row + j);
    c[2 * j] = t.x;
    c[2 * j + 1] = t.y;
  }
  const double x = ndt_poly(c, p);
  return upper ? -x : x;
}

// the uniform of global step gk from its (shared) Philox block
__device__ __forceinline__ double gibbs_uniform(const pbx_u4& b, int64_t gk) {
  return (gk & 4) ? pbx_u52(b.z, b.w) : pbx_u52(b.x, b.y);
}

__device__ __forceinline__ void dmma_m8n8k4(double& d0, double& d1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
}

// ---------------------------------------------------------------------------
// the d = 64 density on the FP64 tensor cores: the fused density of gibbs_mvn_mma_kernel and
// mvn_logpdf_mma64_kernel.  One warp = 8 points.  D[8 x 8] += A[8 x 4] * B[4 x 8] with
//   A[r][k] = x[k] - mean[k] of point r   (lane T: r = T/4, k = 4 ks + T%4)
//   B[k][n] = W[k][n]                     (lane T: k = 4 ks + T%4, n = 8 nb + T/4)
//   D[r][n]: lane T holds (r = T/4, n = 8 nb + 2*(T%4) + {0,1})
// ---------------------------------------------------------------------------
// row stride of W in shared memory: 68 doubles = 4 mod 16 double-banks, so the B-fragment
// loads are bank-conflict free per half-warp
constexpr int kWStride = 68;

__device__ __forceinline__ void stage_whiten64(double* s_W, double* s_m, const double* W,
                                               const double* mean, int nthreads) {
  for (int i = threadIdx.x; i < 64 * 64; i += nthreads) s_W[(i >> 6) * kWStride + (i & 63)] = W[i];
  for (int i = threadIdx.x; i < 64; i += nthreads) s_m[i] = mean[i];
}

// |(x - mean) W|^2 of the 8 points of a warp, x[ks] = coordinate 4 ks + lane % 4 of point
// lane / 4; the sum is returned in all four lanes of the point
__device__ __forceinline__ double dmma_maha64(const double (&x)[16], const double* s_W,
                                              const double* s_m, int lane) {
  const int r = lane >> 2, q = lane & 3;
  double av[16];
#pragma unroll
  for (int ks = 0; ks < 16; ++ks) av[ks] = x[ks] - s_m[4 * ks + q];
  double maha = 0.0;
#pragma unroll
  for (int nb = 0; nb < 8; ++nb) {
    double d0 = 0.0, d1 = 0.0;
#pragma unroll
    for (int ks = 0; ks < 16; ++ks)
      dmma_m8n8k4(d0, d1, av[ks], s_W[(4 * ks + q) * kWStride + nb * 8 + r]);
    maha = fma(d0, d0, maha);
    maha = fma(d1, d1, maha);
  }
  maha += __shfl_xor_sync(0xffffffffu, maha, 1);
  maha += __shfl_xor_sync(0xffffffffu, maha, 2);
  return maha;
}

// the recorded density in log or linear pscale
__device__ __forceinline__ double mvn_density(double norm_c, double maha, int log_pscale) {
  const double lp = -0.5 * (norm_c + maha);
  return log_pscale ? lp : exp(lp);
}

// ---------------------------------------------------------------------------
// Per-coordinate Gibbs (any step range).
//
// One chain = FOUR lanes (a warp = 8 chains): lane q of a chain keeps coordinates
// j = 4m + q in registers (DQ = DP/4 doubles instead of DP, so the kernel fits ~64
// registers instead of 255 + local-memory spills), the dot product coef_i . x is DQ
// FMAs per lane + two shuffle-adds, and the expensive state-independent part of a
// coordinate update -- Philox, ndtri(u) * stdv -- is computed by each lane for ITS OWN
// next coordinate, i.e. four coordinates' worth in parallel with no redundancy.
// kSweepRec: records fall on sweep boundaries only (thin % d == 0, call aligned to
// sweeps) -> one copy of the record code per sweep instead of one per coordinate.
// NT threads per CTA (kGbThreads, or 128 when there are too few chains to give every SM a CTA
// of 64 chains: strong-scaled shards)
template <int DQ, bool kSweepRec, int NT>
__global__ void __launch_bounds__(NT)
    gibbs_mvn_kernel(const GibbsArgs a) {
  constexpr int DP = 4 * DQ;
  constexpr int RS = DQ + 2;                // padded row stride: the 4 sub-lane rows of a
                                            // coordinate land in distinct shared-memory banks
  extern __shared__ __align__(16) double sm[];
  double* s_coef = sm;                      // [DP][4][RS]: s_coef[i][q][m] = coef[i][4m + q]
  double* s_c0 = sm + DP * 4 * RS;          // [DP]
  double* s_sd = s_c0 + DP;
  double* s_lo = s_sd + DP;
  double* s_w = s_lo + DP;                  // hi - lo
  const int d = a.d;
  for (int idx = threadIdx.x; idx < DP * 4 * RS; idx += NT) {
    const int i = idx / (4 * RS), r = idx % (4 * RS), q = r / RS, mm = r % RS;
    const int j = 4 * mm + q;
    s_coef[idx] = (i < d && mm < DQ && j < d) ? a.coef[(int64_t)i * d + j] : 0.0;
  }
  for (int i = threadIdx.x; i < DP; i += NT) {
    const bool v = i < d;
    s_c0[i] = v ? a.c0[i] : 0.0;
    s_sd[i] = v ? a.stdv[i] : 0.0;
    s_lo[i] = v ? a.cdf_lo[i] : 0.0;
    s_w[i] = v ? a.cdf_hi[i] - a.cdf_lo[i] : 0.0;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, q = lane & 3;
  const int64_t C = a.C;
  const int64_t c_raw = ((int64_t)blockIdx.x * (NT / 32) + (threadIdx.x >> 5)) * 8 + (lane >> 2);
  const bool valid = c_raw < C;
  const int64_t c = valid ? c_raw : C - 1;          // clamp: idle lanes stay in the shuffles
  const uint32_t gchain = (uint32_t)(a.chain0 + c);

  double x[DQ];
#pragma unroll
  for (int mm = 0; mm < DQ; ++mm) {
    const int j = 4 * mm + q;
    x[mm] = (j < d) ? a.state[(int64_t)j * C + c] : 0.0;
  }
  const bool stats = a.stat_sum != nullptr;
  const int64_t k_begin = a.step0, k_end = a.step0 + a.T;
  int until_rec = a.thin;
  int64_t rec = 0;
  auto record = [&]() {
    if (valid) {
#pragma unroll
      for (int mm = 0; mm < DQ; ++mm) {
        const int j = 4 * mm + q;
        if (j < d) {
          if (a.out_x) a.out_x[(rec * d + j) * C + c] = x[mm];
          if (stats) {                              // running sums over RECORDED states
            a.stat_sum[(int64_t)j * C + c] += x[mm];
            a.stat_sumsq[(int64_t)j * C + c] =
                fma(x[mm], x[mm], a.stat_sumsq[(int64_t)j * C + c]);
          }
        }
      }
    }
    ++rec;
  };
  pbx_u4 blk;
  blk.x = blk.y = blk.z = blk.w = 0u;
  for (int64_t sweep = k_begin / d; sweep * d < k_end; ++sweep) {
#pragma unroll
    for (int l = 0; l < DQ; ++l) {
      // ---- my own next coordinate i = 4l + q: draw and transform (state independent)
      double z = 0.0;
      {
        const int i = 4 * l + q;
        const int64_t gk = sweep * d + i;
        if (i < d && gk >= k_begin && gk < k_end) {
          double r;
          if (a.inj_runif) {
            r = a.inj_runif[(gk - k_begin) * C + c];
          } else {
            blk = pbx_block(a.seed, (uint64_t)gk & ~(uint64_t)4, gchain, 0u);
            r = gibbs_uniform(blk, gk);
          }
          z = gibbs_ndtri(s_lo[i] + s_w[i] * r) * s_sd[i] + s_c0[i];
        }
      }
#pragma unroll
      for (int o = 0; o < 4; ++o) {
        const int i = 4 * l + o;
        const int64_t gk = sweep * d + i;
        if (i < d && gk >= k_begin && gk < k_end) {        // warp-uniform
          // conditional mean: coef_i . x  (my DQ coordinates, then the 4 sub-lanes)
          const double2* row = reinterpret_cast<const double2*>(s_coef + (i * 4 + q) * RS);
          double p0 = 0.0, p1 = 0.0;
          if (DQ >= 2) {
#pragma unroll
            for (int mm = 0; mm < DQ; mm += 2) {
              const double2 cf = row[mm / 2];
              p0 = fma(cf.x, x[mm], p0);
              p1 = fma(cf.y, x[mm + 1], p1);
            }
          } else {
            p0 = s_coef[(i * 4 + q) * RS] * x[0];
          }
          double dot = p0 + p1;
          dot += __shfl_xor_sync(0xffffffffu, dot, 1);
          dot += __shfl_xor_sync(0xffffffffu, dot, 2);
          if (q == o) x[l] = z + dot;                      // owner lane: x_i = ndtri*sd + c0 + dot
          if (!kSweepRec && --until_rec == 0) {
            until_rec = a.thin;
            record();
          }
        }
      }
    }
    if (kSweepRec) {
      until_rec -= d;
      if (until_rec == 0) {
        until_rec = a.thin;
        record();
      }
    }
  }
  if (valid) {
#pragma unroll
    for (int mm = 0; mm < DQ; ++mm) {
      const int j = 4 * mm + q;
      if (j < d) a.state[(int64_t)j * C + c] = x[mm];
    }
  }
}

// ---------------------------------------------------------------------------
// Whole-sweep Gibbs with the conditional means on the FP64 tensor cores (d >= 5).
//
// The per-coordinate kernel above reads 8 x 128-bit of coefficients from shared memory per
// lane per coordinate; ncu showed it bound by exactly that (50 % of the stall samples on the
// short scoreboard, 29 % issue utilisation, FP64 pipe 17 %): 4 shared-memory wavefronts per
// 64 useful FMAs.  Here the coordinates are taken in BLOCKS of 8 and a block's eight
// sequential updates are solved in closed form.  With C_b the block's 8 rows of the
// coefficient matrix, split into E (columns outside the block), L / U (strictly lower /
// upper part of its 8 x 8 diagonal block; the diagonal is 0), the Gauss-Seidel updates
//     x_t' = z_t + E_t x_out + sum_{s < t} L_ts x_s' + sum_{s > t} U_ts x_s     t = 0..7
// read (I - L) x' = z + E x_out + U x_blk, i.e. with M = (I - L)^-1 (unit lower triangular)
//     x' = (M [E | U]) x + M z  =  B'_b x + M_b z
// -- the same sweep order and the same result as the coordinate-by-coordinate recursion, up
// to rounding.  B'_b (8 x d) and M_b (8 x 8) are built once per launch (gibbs_mma_prep_kernel),
// so a block costs DQ + 2 tensor-core MMAs (mma.sync.m8n8k4.f64: D[chain][n] += A[chain][k]
// B[k][n]) and nothing sequential:
//   * A = the register-resident state: lane (r, q) holds x[4 ks + q] of chain r, which IS the
//     A-fragment layout, and z in the same ownership for the two M_b steps;
//   * B = B'_b / M_b pre-swizzled in shared memory, one conflict-free 64-bit load per MMA
//     (256 FMAs).  The column permutation pi(2j) = j, pi(2j + 1) = j + 4 makes the D
//     fragment of lane (r, q) hold exactly the two block coordinates it owns (8b + q and
//     8b + 4 + q), so the result is written straight back into the state registers;
//   * only the two k-steps holding the previous block's coordinates depend on it; they are
//     issued last, so consecutive blocks overlap.
// Draws: lane (r, q) draws for its own two coordinates of the block from ONE Philox block
// (steps g and g + 4), table ndtri from shared memory, one block ahead of the MMAs.
// ---------------------------------------------------------------------------
// the model in the kernel's shared-memory layout:
//   [NB][DQ][32] B'_b fragments | [NB][2][32] M_b fragments | c0, sd, lo, w [DP] each
template <int DQ>
__host__ __device__ constexpr size_t gibbs_mma_model_doubles() {
  return (size_t)(DQ / 2) * DQ * 32 + (size_t)(DQ / 2) * 64 + 4 * (4 * DQ);
}

// builds that image once per launch in the workspace: one CTA per block of 8 coordinates
template <int DQ>
__global__ void __launch_bounds__(256) gibbs_mma_prep_kernel(const GibbsArgs a,
                                                             double* __restrict__ img) {
  constexpr int DP = 4 * DQ, NB = DQ / 2;
  const int d = a.d, b = blockIdx.x, tid = threadIdx.x;
  __shared__ double sM[8][8];
  auto coef = [&](int row, int col) -> double {
    return (row < d && col < d) ? a.coef[(int64_t)row * d + col] : 0.0;
  };
  if (tid < 8) {                       // column tid of M = (I - L)^-1 by forward substitution
    for (int i = 0; i < 8; ++i) {
      double v = (i == tid) ? 1.0 : 0.0;
      for (int k = 0; k < i; ++k) v = fma(coef(8 * b + i, 8 * b + k), sM[k][tid], v);
      sM[i][tid] = v;
    }
  }
  __syncthreads();
  double* imgB = img + (size_t)b * DQ * 32;
  for (int idx = tid; idx < DQ * 32; idx += 256) {
    const int T = idx & 31, ks = idx >> 5, n = T >> 2;
    const int i = (n >> 1) + 4 * (n & 1), col = 4 * ks + (T & 3);
    const int jb = col - 8 * b;                           // position inside the block, if any
    double v = 0.0;
    for (int k = 0; k < 8; ++k) {
      const bool lower_or_diag = jb >= 0 && jb < 8 && jb <= k;    // L and the diagonal: dropped
      if (!lower_or_diag) v = fma(sM[i][k], coef(8 * b + k, col), v);
    }
    imgB[idx] = v;
  }
  double* imgM = img + (size_t)NB * DQ * 32 + (size_t)b * 64;
  for (int idx = tid; idx < 64; idx += 256) {
    const int T = idx & 31, ks = idx >> 5, n = T >> 2;
    const int i = (n >> 1) + 4 * (n & 1), k = 4 * ks + (T & 3);
    imgM[idx] = sM[i][k];
  }
  if (b == 0) {
    double* par = img + (size_t)NB * DQ * 32 + (size_t)NB * 64;
    for (int j = tid; j < 4 * DP; j += 256) {
      const int which = j / DP, i = j % DP;
      double v = 0.0;
      if (i < d)
        v = which == 0 ? a.c0[i] : which == 1 ? a.stdv[i] : which == 2 ? a.cdf_lo[i]
                                                          : a.cdf_hi[i] - a.cdf_lo[i];
      par[j] = v;
    }
  }
}

// kPair (d % 8 == 0): the two draws of a lane in a block, steps g and g + 4 with bit 2 of g
// clear, come from one Philox block.
// kDens (d = 64): the target density of every recorded state -- |(x - mean) W|^2 on the tensor
// cores, straight from the state registers (they are the A fragment of that product too) --
// instead of a second kernel re-reading the recorded states
template <int DQ, bool kPair, int NT, bool kDens = false>
__global__ void __launch_bounds__(NT, (DQ <= 16 ? (NT <= 128 ? 2 * kGmMinBlocks : kGmMinBlocks) : 1))
    gibbs_mvn_mma_kernel(const GibbsArgs a, const double* __restrict__ img) {
  static_assert(!kDens || (DQ == 16 && kPair), "the fused density is the d = 64 case, a kPair one");
  constexpr int DP = 4 * DQ, NB = DQ / 2;
  extern __shared__ __align__(16) double sm[];
  double* s_B = sm;                          // [NB][DQ][32]   B'_b fragments
  double* s_M = s_B + NB * DQ * 32;          // [NB][2][32]    M_b fragments
  double* s_c0 = s_M + NB * 64;              // [DP]
  double* s_sd = s_c0 + DP;
  double* s_lo = s_sd + DP;
  double* s_w = s_lo + DP;                   // hi - lo
  double* s_nd = s_w + DP;                   // [NDT_NCOEF][NDT_HOT_ROWS]  hot ndtri rows, transposed
  {
    constexpr int n2 = (int)(gibbs_mma_model_doubles<DQ>() / 2);
    const double2* src = reinterpret_cast<const double2*>(img);
    double2* dst = reinterpret_cast<double2*>(sm);
    for (int i = threadIdx.x; i < n2; i += NT) dst[i] = src[i];
    const double2* hsrc = reinterpret_cast<const double2*>(g_ndhot);
    double2* hdst = reinterpret_cast<double2*>(s_nd);
    for (int i = threadIdx.x; i < NDT_NCOEF * NDT_HOT_ROWS / 2; i += NT) hdst[i] = hsrc[i];
  }
  double* s_Wd = s_nd + NDT_NCOEF * NDT_HOT_ROWS;   // [64][kWStride]  whitening matrix (kDens)
  double* s_md = s_Wd + 64 * kWStride;              // [64]            density mean
  if (kDens) stage_whiten64(s_Wd, s_md, a.whiten, a.dens_mean, NT);
  __syncthreads();
  const int d = a.d;
  const int lane = threadIdx.x & 31, q = lane & 3;
  const int64_t C = a.C;
  const int64_t c_raw = ((int64_t)blockIdx.x * (NT / 32) + (threadIdx.x >> 5)) * 8 + (lane >> 2);
  const bool valid = c_raw < C;
  const int64_t c = valid ? c_raw : C - 1;          // clamp: idle lanes stay in the MMAs
  const uint32_t gchain = (uint32_t)(a.chain0 + c);

  double x[DQ];
#pragma unroll
  for (int mm = 0; mm < DQ; ++mm) {
    const int j = 4 * mm + q;
    x[mm] = (j < d) ? a.state[(int64_t)j * C + c] : 0.0;
  }
  const bool stats = a.stat_sum != nullptr;
  const int64_t k_begin = a.step0, k_end = a.step0 + a.T;
  int until_rec = a.thin;
  int64_t rec = 0;

  // The two draws of this lane for block b of sweep sw (coordinates 8b + q and 8b + 4 + q):
  // state independent and BRANCH-FREE.  The table rows come from the shared-memory copy of
  // the 10 binades nearest 0.5 with a clamped index (a first version gathered the 64-byte
  // rows from global memory: 27 L1 sectors per request made the L1 the bottleneck); for the
  // 0.1 % of arguments outside them the draw returns u itself and a flag bit, and the caller
  // finishes it with draw_fix (full table or, outside it, normcdfinv).
  auto draw_pair = [&](int64_t sw, int b, double& z0, double& z1) -> unsigned {
    const int i0 = 8 * b + q, i1 = i0 + 4;
    const int64_t g0 = sw * d + i0, g1 = g0 + 4;
    double r0, r1;
    if (a.inj_runif) {
      r0 = (i0 < d && g0 < k_end) ? a.inj_runif[(g0 - k_begin) * C + c] : 0.5;
      r1 = (i1 < d && g1 < k_end) ? a.inj_runif[(g1 - k_begin) * C + c] : 0.5;
    } else if (kPair) {
      const pbx_u4 blk = pbx_block(a.seed, (uint64_t)g0, gchain, 0u);       // bit 2 of g0 clear
      r0 = pbx_u52(blk.x, blk.y);
      r1 = pbx_u52(blk.z, blk.w);
    } else {
      const pbx_u4 b0 = pbx_block(a.seed, (uint64_t)g0 & ~(uint64_t)4, gchain, 0u);
      const pbx_u4 b1 = pbx_block(a.seed, (uint64_t)g1 & ~(uint64_t)4, gchain, 0u);
      r0 = gibbs_uniform(b0, g0);
      r1 = gibbs_uniform(b1, g1);
    }
    unsigned bad = 0u;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int i = h ? i1 : i0;
      const double u = s_lo[i] + s_w[i] * (h ? r1 : r0);
      const bool upper = u > 0.5;
      const double p = upper ? 1.0 - u : u;                    // exact for u > 0.5
      const unsigned seg = ndt_segment(p) - (unsigned)NDT_HOT0;     // wraps below the hot rows
      const bool cold = seg >= (unsigned)NDT_HOT_ROWS;
      if (cold && i < d) bad |= 1u << h;
      const double* row = s_nd + min(seg, (unsigned)(NDT_HOT_ROWS - 1));
      double cf[NDT_NCOEF];
#pragma unroll
      for (int j = 0; j < NDT_NCOEF; ++j) cf[j] = row[j * NDT_HOT_ROWS];
      const double xn = ndt_poly(cf, p);
      const double z = (upper ? -xn : xn) * s_sd[i] + s_c0[i];
      (h ? z1 : z0) = (i < d) ? (cold ? u : z) : 0.0;
    }
    return bad;
  };
  auto draw_fix = [&](unsigned bad, int b, double& z0, double& z1) {
    const int i0 = 8 * b + q, i1 = i0 + 4;
    if (bad & 1u) z0 = gibbs_ndtri(z0) * s_sd[i0] + s_c0[i0];
    if (bad & 2u) z1 = gibbs_ndtri(z1) * s_sd[i1] + s_c0[i1];
  };

  // Software pipeline: the draws of the NEXT block (of the next sweep after the last block)
  // are computed in the same basic block as the current block's MMAs and 8-step chain, whose
  // dependency stalls they fill -- 4 warps per scheduler do not hide them otherwise.
  double z0, z1;
  unsigned bad = draw_pair(k_begin / d, 0, z0, z1);
  for (int64_t sweep = k_begin / d; sweep * d < k_end; ++sweep) {
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      if (bad) draw_fix(bad, b, z0, z1);                         // practically never
      double zn0, zn1;
      const unsigned badn = (b + 1 < NB) ? draw_pair(sweep, b + 1, zn0, zn1)
                                         : draw_pair(sweep + 1, 0, zn0, zn1);
      // x'_blk = B'_b x + M_b z on the tensor cores: M_b z first (state independent), then two
      // accumulator chains over the state, the k-steps of the previous block's coordinates last
      double m0 = 0.0, m1 = 0.0, e0 = 0.0, e1 = 0.0;
      const double* mf = s_M + b * 64 + lane;
      dmma_m8n8k4(m0, m1, z0, mf[0]);
      dmma_m8n8k4(m0, m1, z1, mf[32]);
      const double* bf = s_B + (b * DQ) * 32 + lane;
#pragma unroll
      for (int kk = 0; kk < DQ; kk += 2) {
        const int ks = (b == 0) ? kk : (kk + 2 * b) % DQ;
        dmma_m8n8k4(m0, m1, x[ks], bf[ks * 32]);
        dmma_m8n8k4(e0, e1, x[ks + 1], bf[(ks + 1) * 32]);
      }
      x[2 * b] = m0 + e0;
      x[2 * b + 1] = m1 + e1;
      z0 = zn0;
      z1 = zn1;
      bad = badn;
    }
    until_rec -= d;
    if (until_rec == 0) {
      until_rec = a.thin;
      if (valid) {
#pragma unroll
        for (int mm = 0; mm < DQ; ++mm) {
          const int j = 4 * mm + q;
          if (j < d) {
            if (a.out_x) a.out_x[(rec * d + j) * C + c] = x[mm];
            if (stats) {                              // running sums over RECORDED states
              a.stat_sum[(int64_t)j * C + c] += x[mm];
              a.stat_sumsq[(int64_t)j * C + c] =
                  fma(x[mm], x[mm], a.stat_sumsq[(int64_t)j * C + c]);
            }
          }
        }
      }
      if constexpr (kDens) {
        const double maha = dmma_maha64(x, s_Wd, s_md, lane);
        if (q == 0 && valid) a.out_prob[rec * C + c] = mvn_density(a.norm_c, maha, a.log_pscale);
      }
      ++rec;
    }
  }
  if (valid) {
#pragma unroll
    for (int mm = 0; mm < DQ; ++mm) {
      const int j = 4 * mm + q;
      if (j < d) a.state[(int64_t)j * C + c] = x[mm];
    }
  }
}

// ---------------------------------------------------------------------------
// batched mvn density, plain FMA version: one thread per point, W from smem
// ---------------------------------------------------------------------------
// points: R blocks of [d][C]; point (r, c) -> x[(r*d + j)*C + c], out[r*C + c]
__global__ void __launch_bounds__(128)
    mvn_logpdf_kernel(const double* __restrict__ x, int d, int64_t C, int64_t R,
                      const double* __restrict__ mean, const double* __restrict__ W, double norm_c,
                      int log_pscale, double* __restrict__ out) {
  extern __shared__ __align__(16) double sm[];
  double* s_W = sm;            // [d][d]
  double* s_m = sm + d * d;    // [d]
  for (int i = threadIdx.x; i < d * d; i += blockDim.x) s_W[i] = W[i];
  for (int i = threadIdx.x; i < d; i += blockDim.x) s_m[i] = mean[i];
  __syncthreads();
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= C * R) return;
  const int64_t r = p / C, c = p % C;
  const double* xb = x + r * d * C + c;
  double maha = 0.0;
  for (int k = 0; k < d; ++k) {
    double y = 0.0;
    for (int j = 0; j < d; ++j) y = fma(xb[(int64_t)j * C] - s_m[j], s_W[j * d + k], y);
    maha = fma(y, y, maha);
  }
  out[p] = mvn_density(norm_c, maha, log_pscale);
}

// batched mvn density on the FP64 tensor cores, d = 64: one warp per 8-point row block
__global__ void __launch_bounds__(128)
    mvn_logpdf_mma64_kernel(const double* __restrict__ x, int64_t C, int64_t R,
                            const double* __restrict__ mean, const double* __restrict__ W,
                            double norm_c, int log_pscale, double* __restrict__ out) {
  __shared__ double s_W[64 * kWStride];
  __shared__ double s_m[64];
  stage_whiten64(s_W, s_m, W, mean, blockDim.x);
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int r = lane >> 2, q = lane & 3;
  const int64_t bpr = (C + 7) / 8, n_blocks = bpr * R;       // 8-point blocks per record
  for (int64_t blk = (int64_t)blockIdx.x * 4 + warp; blk < n_blocks; blk += (int64_t)gridDim.x * 4) {
    const int64_t rr = blk / bpr;
    const int64_t c = (blk % bpr) * 8 + r;
    const bool valid = c < C;
    const double* xb = x + rr * 64 * C;
    // this lane's A elements for the 16 k-steps: k = 4*ks + q (rows past C: any finite value)
    double xv[16];
#pragma unroll
    for (int ks = 0; ks < 16; ++ks) xv[ks] = valid ? xb[(int64_t)(4 * ks + q) * C + c] : 0.0;
    const double maha = dmma_maha64(xv, s_W, s_m, lane);
    if (q == 0 && valid) out[rr * C + c] = mvn_density(norm_c, maha, log_pscale);
  }
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
static int mvn_logpdf_launch(pbx_ctx* ctx, const double* x, int d, int64_t C, int64_t R,
                             const double* mean, const double* W, double norm_c, int log_pscale,
                             double* out) {
  if (C * R == 0) return PBX_OK;
  if (d == 64) {
    int64_t want = ((C + 7) / 8 * R + 3) / 4;
    int grid = (int)(want > (int64_t)ctx->sm_count * 6 ? (int64_t)ctx->sm_count * 6 : want);
    mvn_logpdf_mma64_kernel<<<grid, 128, 0, ctx->stream>>>(x, C, R, mean, W, norm_c, log_pscale,
                                                          out);
  } else {
    const size_t smem = ((size_t)d * d + d) * sizeof(double);
    const int64_t grid = (C * R + 127) / 128;
    if (smem > 48 * 1024)
      PBX_CUDA(cudaFuncSetAttribute(mvn_logpdf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)smem));
    mvn_logpdf_kernel<<<(unsigned)grid, 128, smem, ctx->stream>>>(x, d, C, R, mean, W, norm_c,
                                                                 log_pscale, out);
  }
  PBX_LAUNCH_CHECK(ctx);
  return PBX_OK;
}

extern "C" int pbx_mvn_logpdf(pbx_ctx* ctx, const double* x, int32_t n_dims, int64_t n_chains,
                              const double* mean, const double* whiten, double norm_c,
                              int32_t log_pscale, double* out) {
  PBX_REQUIRE(ctx && x && mean && whiten && out, "pbx_mvn_logpdf: null argument");
  PBX_REQUIRE(n_dims >= 1 && n_dims <= 128, "pbx_mvn_logpdf: n_dims must be in 1..128");
  PBX_REQUIRE(n_chains >= 0, "pbx_mvn_logpdf: negative point count");
  PBX_CUDA(cudaSetDevice(ctx->device));
  PBX_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
  int rc = mvn_logpdf_launch(ctx, x, n_dims, n_chains, 1, mean, whiten, norm_c, log_pscale, out);
  if (rc) return rc;
  PBX_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
  return PBX_OK;
}

// the host copies of the table, built once per process (19 ms; function-local statics:
// thread-safe initialisation)
static const double* ndt_host_table() {
  static const std::vector<double> tab = [] {
    std::vector<double> t((size_t)NDT_ROWS * NDT_NCOEF);
    ndt_build_table(t.data());
    return t;
  }();
  return tab.data();
}
static const double* ndt_host_hot_table() {
  static const std::vector<double> hot = [] {
    const double* h_tab = ndt_host_table();
    std::vector<double> t((size_t)NDT_NCOEF * NDT_HOT_ROWS);
    for (int r = 0; r < NDT_HOT_ROWS; ++r)
      for (int j = 0; j < NDT_NCOEF; ++j)
        t[(size_t)j * NDT_HOT_ROWS + r] = h_tab[(size_t)(NDT_HOT0 + r) * NDT_NCOEF + j];
    return t;
  }();
  return hot.data();
}

static int gibbs_init_ndtab(pbx_ctx* ctx) {
  if (ctx->ndtab_ready) return PBX_OK;
  const double* h_tab = ndt_host_table();
  const double* h_hot = ndt_host_hot_table();
  PBX_CUDA(cudaMemcpyToSymbolAsync(g_ndtab, h_tab, sizeof(double) * NDT_ROWS * NDT_NCOEF, 0,
                                   cudaMemcpyHostToDevice, ctx->stream));
  PBX_CUDA(cudaMemcpyToSymbolAsync(g_ndhot, h_hot, sizeof(double) * NDT_NCOEF * NDT_HOT_ROWS, 0,
                                   cudaMemcpyHostToDevice, ctx->stream));
  PBX_CUDA(cudaStreamSynchronize(ctx->stream));
  ctx->ndtab_ready = true;
  return PBX_OK;
}

// whole: the call is whole sweeps (step0, T and thin multiples of d); dens: the density of the
// recorded states is fused into the tensor-core kernel (whole sweeps at d = 64)
template <int DQ, int NT>
static int gibbs_launch_nt(pbx_ctx* ctx, const GibbsArgs& a, double* img, bool whole, bool dens) {
  constexpr int DP = 4 * DQ;
  const int chains_per_cta = (NT / 32) * 8;
  const int grid = (a.C + chains_per_cta - 1) / chains_per_cta;
  if constexpr (DQ >= 2) {
    if (whole) {                           // whole sweeps: conditional means on the tensor cores
      const size_t smem = (gibbs_mma_model_doubles<DQ>() + NDT_NCOEF * NDT_HOT_ROWS +
                           (dens ? 64 * kWStride + 64 : 0)) * sizeof(double);
      gibbs_mma_prep_kernel<DQ><<<DQ / 2, 256, 0, ctx->stream>>>(a, img);
      PBX_LAUNCH_CHECK(ctx);
      if constexpr (DQ == 16)
        if (dens) return launch_smem(ctx, gibbs_mvn_mma_kernel<DQ, true, NT, true>, grid, NT, smem, a, img);
      auto* k = a.d % 8 == 0 ? gibbs_mvn_mma_kernel<DQ, true, NT> : gibbs_mvn_mma_kernel<DQ, false, NT>;
      return launch_smem(ctx, k, grid, NT, smem, a, img);
    }
  }
  auto* k = gibbs_mvn_kernel<DQ, false, NT>;
  if constexpr (DQ == 1)
    if (whole) k = gibbs_mvn_kernel<DQ, true, NT>;
  return launch_smem(ctx, k, grid, NT, ((size_t)DP * 4 * (DQ + 2) + 4 * DP) * sizeof(double), a);
}

template <int DQ>
static int gibbs_launch(pbx_ctx* ctx, const GibbsArgs& a, double* img, bool whole, bool dens) {
  // fewer than ~3 CTAs of 64 chains per SM: halve the CTA so that the grid covers the chip
  // (a strong-scaled shard of 8192 chains is 128 CTAs of 64 on 148 SMs)
  if ((int64_t)a.C < (int64_t)ctx->sm_count * 64 * 3)
    return gibbs_launch_nt<DQ, 128>(ctx, a, img, whole, dens);
  return gibbs_launch_nt<DQ, kGbThreads>(ctx, a, img, whole, dens);
}

// workspace: c0 [d <= 128] at 0, the tensor-core kernel's model image at this offset
constexpr size_t kGibbsImageOffset = 128 * sizeof(double);

extern "C" int pbx_gibbs_mvn_run(pbx_ctx* ctx, const pbx_gibbs_mvn_params* p) {
  PBX_REQUIRE(ctx != nullptr && p != nullptr, "pbx_gibbs_mvn_run: null argument");
  PBX_REQUIRE(p->n_chains >= 1, "pbx_gibbs_mvn_run: n_chains must be >= 1");
  PBX_REQUIRE(p->n_dims >= 1 && p->n_dims <= 128, "pbx_gibbs_mvn_run: n_dims must be in 1..128");
  PBX_REQUIRE(p->n_steps >= 0 && p->thin >= 1, "pbx_gibbs_mvn_run: n_steps >= 0, thin >= 1");
  PBX_REQUIRE(p->step0 >= 0 && p->chain0 >= 0, "pbx_gibbs_mvn_run: step0/chain0 must be >= 0");
  PBX_REQUIRE(p->mean && p->coef && p->stdv && p->cdf_lo && p->cdf_hi && p->state,
              "pbx_gibbs_mvn_run: model/state pointers are mandatory");
  PBX_REQUIRE(!p->out_prob || (p->out_x && p->whiten),
              "pbx_gibbs_mvn_run: out_prob needs out_x and the whitening matrix");
  PBX_CUDA(cudaSetDevice(ctx->device));
  const int d = p->n_dims;
  int rc = gibbs_init_ndtab(ctx);
  if (rc) return rc;
  rc = pbx_ws_reserve(ctx, kGibbsImageOffset + gibbs_mma_model_doubles<32>() * sizeof(double));
  if (rc) return rc;
  double* c0 = (double*)ctx->ws;
  double* img = (double*)((char*)ctx->ws + kGibbsImageOffset);
  GibbsArgs a;
  a.C = p->n_chains; a.d = d; a.T = p->n_steps; a.thin = p->thin;
  a.step0 = p->step0; a.chain0 = p->chain0; a.seed = p->seed;
  a.coef = p->coef; a.c0 = c0; a.stdv = p->stdv; a.cdf_lo = p->cdf_lo; a.cdf_hi = p->cdf_hi;
  a.state = p->state; a.inj_runif = p->inj_runif; a.out_x = p->out_x;
  a.stat_sum = p->stat_sum; a.stat_sumsq = p->stat_sumsq;
  // whole sweeps at d = 64: the density of the recorded states is evaluated inside the Gibbs
  // kernel; otherwise by a second launch over the recorded states (below)
  const bool whole = (p->thin % d == 0) && (p->step0 % d == 0) && (p->n_steps % d == 0);
  const bool want_dens = p->out_prob && p->want_prob;
  const bool fused_dens = want_dens && d == 64 && whole;
  a.out_prob = fused_dens ? p->out_prob : nullptr;
  a.whiten = p->whiten;
  a.dens_mean = p->dens_mean ? p->dens_mean : p->mean;
  a.norm_c = p->norm_c;
  a.log_pscale = p->log_pscale;
  PBX_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
  if (a.T > 0) {
    gibbs_c0_kernel<<<1, 128, 0, ctx->stream>>>(p->coef, p->mean, d, c0);
    PBX_LAUNCH_CHECK(ctx);
    if (d <= 4) rc = gibbs_launch<1>(ctx, a, img, whole, fused_dens);
    else if (d <= 8) rc = gibbs_launch<2>(ctx, a, img, whole, fused_dens);
    else if (d <= 16) rc = gibbs_launch<4>(ctx, a, img, whole, fused_dens);
    else if (d <= 32) rc = gibbs_launch<8>(ctx, a, img, whole, fused_dens);
    else if (d <= 64) rc = gibbs_launch<16>(ctx, a, img, whole, fused_dens);
    else rc = gibbs_launch<32>(ctx, a, img, whole, fused_dens);
    if (rc) return rc;
    if (want_dens && !fused_dens) {
      // the target is evaluated and recorded on every kept step (sd.py:286)
      rc = mvn_logpdf_launch(ctx, p->out_x, d, p->n_chains, p->n_steps / p->thin, a.dens_mean,
                             p->whiten, p->norm_c, p->log_pscale, p->out_prob);
      if (rc) return rc;
    }
  }
  PBX_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
  return PBX_OK;
}

// ---------------------------------------------------------------------------
// the table-driven ndtri on its own: device evaluation over an array (accuracy tests) and the
// host mirror of the same arithmetic (usable without a GPU)
// ---------------------------------------------------------------------------
__global__ void ndtri_array_kernel(const double* __restrict__ u, int64_t n, double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = gibbs_ndtri(u[i]);
}

extern "C" int pbx_ndtri(pbx_ctx* ctx, const double* u, int64_t n, double* out) {
  PBX_REQUIRE(ctx && u && out && n >= 0, "pbx_ndtri: bad argument");
  PBX_CUDA(cudaSetDevice(ctx->device));
  int rc = gibbs_init_ndtab(ctx);
  if (rc) return rc;
  PBX_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
  if (n > 0) {
    ndtri_array_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(u, n, out);
    PBX_LAUNCH_CHECK(ctx);
  }
  PBX_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
  return PBX_OK;
}

extern "C" int pbx_ndtri_host(const double* u, int64_t n, double* out) {
  if (!u || !out || n < 0) {
    pbx_set_error("pbx_ndtri_host: bad argument");
    return PBX_ERR_INVALID;
  }
  const double* h_tab = ndt_host_table();
  for (int64_t i = 0; i < n; ++i) out[i] = ndt_eval_host(h_tab, u[i]);
  return PBX_OK;
}
