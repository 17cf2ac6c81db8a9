// K4: batched trust-region projection of a diagonal Gaussian policy, forward and backward.
// Replaces (all under geometry_rl/algorithms/trust_region_projections/):
//   projections/base_projection_layer.py:71-100   mean_projection (closed form, autograd through maha)
//   projections/kl_projection_layer.py:15-111     KL projection, diag branch; the ITPAL op
//       cpp_projection.BatchedDiagCovOnlyProjection (:162-204: numpy round trip, OpenMP + NLopt on the
//       CPU, float64) becomes an in-register safeguarded Newton solve of the 1-D dual, also float64
//   projections/w2_projection_layer.py:15-68      commuting W2 projection (scale_prec = True)
// "v" is the diagonal of the matrix the reference calls std (numerically the variance, SURVEY 0).
// One thread per sample, k <= GRL_MAX_ACTION_DIM values in registers.
#include "grl_common.cuh"

namespace grl {

constexpr int kMaxK = GRL_MAX_ACTION_DIM;
constexpr double kLog2Pi = 1.8378770664093454835606594728112;

// Entropy projection of one sample (base_projection_layer.py:14-68): alpha = exp((beta - H(v)) / k) with
// H(v) = 0.5 (k (1 + log 2pi) + 2 sum log v) ("std := v"), where H < beta (inequality) or always (equality); 1 elsewhere.
__device__ __forceinline__ double entropy_alpha(const float* v, int k, int mode, double beta) {
  double slog = 0.0;
#pragma unroll
  for (int i = 0; i < kMaxK; ++i)
    if (i < k) slog += log((double)v[i]);
  const double H = 0.5 * (k * (1.0 + kLog2Pi) + 2.0 * slog);
  return (mode == GRL_ENTROPY_EQ || H < beta) ? exp((beta - H) / k) : 1.0;
}

// Vector-Jacobian product of v' = alpha(v) v: g_j <- alpha (g_j - sum_i g_i x_i / (k x_j)).  With x = v this is
// alpha g_j - alpha / (k v_j) sum_i g_i v_i; x = v' gives the same value (alpha cancels).  beta is a constant.
__device__ __forceinline__ void entropy_vjp(double* g, const double* x, int k, double alpha) {
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < kMaxK; ++i)
    if (i < k) s += g[i] * x[i];
#pragma unroll
  for (int i = 0; i < kMaxK; ++i)
    if (i < k) g[i] = alpha * (g[i] - s / (k * x[i]));
}

struct KlEval {
  double kl, dkl;
};

// KL(eta) of c~(eta) = (eta + 1) / (eta / o + 1 / c) against o, and d KL / d eta, from the per-dimension invariants
// io = 1 / o, ic = 1 / c, lo = log o (formed once per sample): one division and one logarithm per dimension and
// evaluation instead of five and two - the solve is a serial chain of fp64 operations in ONE thread, so its length is
// the kernel's duration whatever the batch size.
struct KlInv {
  double io[kMaxK], ic[kMaxK], lo[kMaxK];
};
__device__ __forceinline__ KlEval kl_eval(const KlInv& q, int k, double eta) {
  KlEval r{0.0, 0.0};
  const double e1 = eta + 1.0, ie1 = 1.0 / e1;
#pragma unroll
  for (int i = 0; i < kMaxK; ++i) {
    if (i < k) {
      const double D = fma(eta, q.io[i], q.ic[i]);
      const double rD = 1.0 / D;
      const double ct = e1 * rD;                       // c~(eta)
      r.kl += fma(ct, q.io[i], -1.0) + q.lo[i] - log(ct);
      const double dct = (q.ic[i] - q.io[i]) * rD * rD;
      r.dkl += (q.io[i] - D * ie1) * dct;              // 1 / ct = D / (eta + 1)
    }
  }
  r.kl *= 0.5;
  r.dkl *= 0.5;
  return r;
}

// ENT: entropy control (d.entropy_mode != 0); the <false> instantiation is the plain trust-region projection.
template <bool ENT>
__global__ void __launch_bounds__(128) trpl_fwd_kernel(const GrlProjDesc d) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= d.batch) return;
  const int k = d.k;
  float m[kMaxK], v[kMaxK], mo[kMaxK], vo[kMaxK];
#pragma unroll
  for (int i = 0; i < kMaxK; ++i) {
    if (i < k) {
      m[i] = d.mean[(size_t)b * k + i];
      v[i] = d.v[(size_t)b * k + i];
      mo[i] = d.old_mean[(size_t)b * k + i];
      vo[i] = d.old_v[(size_t)b * k + i];
    } else {
      m[i] = mo[i] = 0.f;
      v[i] = vo[i] = 1.f;
    }
  }
  double alpha = 1.0;
  if constexpr (ENT) {
    if (d.entropy_first) {  // the trust-region projection then starts from the entropy-projected v
      alpha = entropy_alpha(v, k, d.entropy_mode, *d.entropy_beta);
#pragma unroll
      for (int i = 0; i < kMaxK; ++i)
        if (i < k) v[i] = (float)(alpha * (double)v[i]);
    }
  }
  // ---- mean part ---------------------------------------------------------------------------
  float maha = 0.f;
#pragma unroll
  for (int i = 0; i < kMaxK; ++i)
    if (i < k) { const float t = (m[i] - mo[i]) / vo[i]; maha += t * t; }
  const float mean_part = d.proj_type == 0 ? 0.5f * maha : maha;
  float omega = 0.f;
  const bool mean_active = mean_part > d.eps_mean;
  if (mean_active) omega = fabsf(sqrtf(mean_part / d.eps_mean) - 1.0f);
#pragma unroll
  for (int i = 0; i < kMaxK; ++i)
    if (i < k) d.proj_mean[(size_t)b * k + i] = mean_active ? (m[i] + omega * mo[i]) / (1.0f + omega + 1e-16f) : m[i];

  d.eta[2 * (size_t)b + 1] = mean_active ? (double)omega : 0.0;  // branch flag for the backward pass

  // ---- covariance part -----------------------------------------------------------------------
  if (d.proj_type == 0) {
    double c[kMaxK], o[kMaxK];
    KlInv q;
#pragma unroll
    for (int i = 0; i < kMaxK; ++i) {
      c[i] = (double)(v[i] * v[i]);
      o[i] = (double)(vo[i] * vo[i]);
      q.io[i] = 1.0 / o[i];
      q.ic[i] = 1.0 / c[i];
      q.lo[i] = i < k ? log(o[i]) : 0.0;
    }
    const double eps = (double)d.eps_cov;
    double eta = 0.0;
    KlEval f = kl_eval(q, k, 0.0);
    if (f.kl > eps) {
      double lo = 0.0, hi = 1.0;
      for (int it = 0; it < 200; ++it) {  // bracket: KL is decreasing in eta
        if (kl_eval(q, k, hi).kl <= eps) break;
        lo = hi;
        hi *= 2.0;
      }
      eta = 0.5 * (lo + hi);
      for (int it = 0; it < 100; ++it) {  // safeguarded Newton on KL(eta) - eps
        f = kl_eval(q, k, eta);
        const double res = f.kl - eps;
        if (res > 0.0) lo = eta; else hi = eta;
        if (fabs(res) <= 1e-14 * eps || (hi - lo) <= 1e-15 * hi) break;
        double nxt = eta - res / f.dkl;
        if (!(nxt > lo && nxt < hi)) nxt = 0.5 * (lo + hi);
        eta = nxt;
      }
    }
    d.eta[2 * (size_t)b] = eta;
#pragma unroll
    for (int i = 0; i < kMaxK; ++i) {
      if (i < k) {
        // reference: cov.new(float64 result) -> fp32, then .sqrt() in fp32 (kl_projection_layer.py:72)
        const float ct = eta > 0.0 ? (float)((eta + 1.0) / (eta / o[i] + 1.0 / c[i])) : v[i] * v[i];
        d.proj_v[(size_t)b * k + i] = sqrtf(ct);
      }
    }
  } else {
    float cov_part = 0.f;
#pragma unroll
    for (int i = 0; i < kMaxK; ++i)
      if (i < k) { const float inv = 1.0f / vo[i]; cov_part += 1.0f + inv * (v[i] * v[i]) * inv - 2.0f * inv * v[i]; }
    float eta = 0.f;
    const bool active = cov_part > d.eps_cov;
    if (active) eta = fabsf(sqrtf(cov_part / d.eps_cov) - 1.0f);
    d.eta[2 * (size_t)b] = active ? (double)eta : 0.0;
#pragma unroll
    for (int i = 0; i < kMaxK; ++i)
      if (i < k) d.proj_v[(size_t)b * k + i] = active ? (v[i] + eta * vo[i]) / (1.0f + eta + 1e-16f) : v[i];
  }
  if constexpr (ENT) {
    if (!d.entropy_first) {  // entropy projection of the trust-region output (this thread's own stores)
      float pv[kMaxK];
#pragma unroll
      for (int i = 0; i < kMaxK; ++i) pv[i] = i < k ? d.proj_v[(size_t)b * k + i] : 1.f;
      alpha = entropy_alpha(pv, k, d.entropy_mode, *d.entropy_beta);
#pragma unroll
      for (int i = 0; i < kMaxK; ++i)
        if (i < k) d.proj_v[(size_t)b * k + i] = (float)(alpha * (double)pv[i]);
    }
    d.entropy_alpha[b] = alpha;
  }
}

template <bool ENT>
__global__ void __launch_bounds__(128) trpl_bwd_kernel(const GrlProjDesc d) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= d.batch) return;
  const int k = d.k;
  double m[kMaxK], v[kMaxK], mo[kMaxK], vo[kMaxK], gm[kMaxK], gv[kMaxK];
  double am[kMaxK], av[kMaxK];  // gradients that reach (mean, v) directly (grad_mean_add / grad_v_add)
#pragma unroll
  for (int i = 0; i < kMaxK; ++i) {
    am[i] = (i < k && d.grad_mean_add) ? (double)d.grad_mean_add[(size_t)b * k + i] : 0.0;
    av[i] = (i < k && d.grad_v_add) ? (double)d.grad_v_add[(size_t)b * k + i] : 0.0;
  }
#pragma unroll
  for (int i = 0; i < kMaxK; ++i) {
    if (i < k) {
      m[i] = d.mean[(size_t)b * k + i];
      v[i] = d.v[(size_t)b * k + i];
      mo[i] = d.old_mean[(size_t)b * k + i];
      vo[i] = d.old_v[(size_t)b * k + i];
      gm[i] = d.grad_proj_mean[(size_t)b * k + i];
      gv[i] = d.grad_proj_v[(size_t)b * k + i];
    } else {
      m[i] = mo[i] = gm[i] = gv[i] = 0.0;
      v[i] = vo[i] = 1.0;
    }
  }
  // ENT: gq = gradient w.r.t. the trust-region projection's input v, before grad_v_add
  double alpha = 1.0, v_in[kMaxK], gq[kMaxK];
  bool ent_active = false;
  if constexpr (ENT) {
    alpha = d.entropy_alpha[b];
    ent_active = d.entropy_mode == GRL_ENTROPY_EQ || alpha > 1.0;  // inequality: alpha > 1 exactly where H < beta
#pragma unroll
    for (int i = 0; i < kMaxK; ++i) {
      v_in[i] = v[i];
      gq[i] = 0.0;
    }
    if (d.entropy_first) {
      // the trust-region projection saw v' = alpha v, rounded as the forward rounded it
#pragma unroll
      for (int i = 0; i < kMaxK; ++i)
        if (i < k) v[i] = (double)(float)(alpha * v[i]);
    } else if (ent_active) {
      // gradient reaching the trust-region output pv0 through pv = alpha(pv0) pv0 (evaluated at pv)
      double pv[kMaxK];
#pragma unroll
      for (int i = 0; i < kMaxK; ++i) pv[i] = i < k ? (double)d.proj_v[(size_t)b * k + i] : 1.0;
      entropy_vjp(gv, pv, k, alpha);
    }
  }
  // ---- mean: pm = (m + w mo) / (1 + w), w = sqrt(M / eps) - 1, M = scale * sum ((m - mo) / vo)^2
  const double scale = d.proj_type == 0 ? 0.5 : 1.0;
  double M = 0.0;
#pragma unroll
  for (int i = 0; i < kMaxK; ++i)
    if (i < k) { const double t = (m[i] - mo[i]) / vo[i]; M += t * t; }
  M *= scale;
  const double eps_m = (double)d.eps_mean;
  if (d.eta[2 * (size_t)b + 1] > 0.0) {
    const double w = sqrt(M / eps_m) - 1.0;
    double dot = 0.0;  // sum_i g_i d pm_i / d w
#pragma unroll
    for (int i = 0; i < kMaxK; ++i)
      if (i < k) dot += gm[i] * (mo[i] - m[i]) / ((1.0 + w) * (1.0 + w));
    const double dw_dM = 1.0 / (2.0 * eps_m * (1.0 + w));
#pragma unroll
    for (int i = 0; i < kMaxK; ++i)
      if (i < k)
        d.grad_mean[(size_t)b * k + i] =
            (float)(gm[i] / (1.0 + w) + dot * dw_dM * scale * 2.0 * (m[i] - mo[i]) / (vo[i] * vo[i]) + am[i]);
  } else {
#pragma unroll
    for (int i = 0; i < kMaxK; ++i)
      if (i < k) d.grad_mean[(size_t)b * k + i] = (float)(gm[i] + am[i]);
  }
  // ---- covariance
  const double eta = d.eta[2 * (size_t)b];
  if (d.proj_type == 0) {
    // pv = sqrt(c~), c~ = (eta+1)/(eta/o + 1/c), c = v^2, o = vo^2; implicit gradient through eta(c)
    if (eta > 0.0) {
      double num = 0.0, den = 0.0;
      double gct[kMaxK], dct_dc[kMaxK], dkl_dct[kMaxK];
#pragma unroll
      for (int i = 0; i < kMaxK; ++i) {
        gct[i] = dct_dc[i] = dkl_dct[i] = 0.0;
        if (i < k) {
          const double c = v[i] * v[i], o = vo[i] * vo[i];
          const double D = eta / o + 1.0 / c;
          const double ct = (eta + 1.0) / D;
          gct[i] = gv[i] / (2.0 * sqrt(ct));
          dct_dc[i] = (eta + 1.0) / (D * D * c * c);
          const double dct_deta = (1.0 / c - 1.0 / o) / (D * D);
          dkl_dct[i] = 0.5 * (1.0 / o - 1.0 / ct);
          num += gct[i] * dct_deta;
          den += dkl_dct[i] * dct_deta;
        }
      }
#pragma unroll
      for (int i = 0; i < kMaxK; ++i)
        if (i < k) {
          const double gc = gct[i] * dct_dc[i] - num * (dkl_dct[i] * dct_dc[i]) / den;
          if constexpr (ENT) gq[i] = gc * 2.0 * v[i];
          else d.grad_v[(size_t)b * k + i] = (float)(gc * 2.0 * v[i] + av[i]);
        }
    } else {
      // identity: pv = sqrt(v^2) = v
#pragma unroll
      for (int i = 0; i < kMaxK; ++i)
        if (i < k) {
          if constexpr (ENT) gq[i] = gv[i];
          else d.grad_v[(size_t)b * k + i] = (float)(gv[i] + av[i]);
        }
    }
  } else {
    if (eta > 0.0) {
      // nv = (v + eta vo) / (1 + eta), eta = sqrt(S / eps) - 1, S = sum (v/vo - 1)^2
      double dot = 0.0;
#pragma unroll
      for (int i = 0; i < kMaxK; ++i)
        if (i < k) dot += gv[i] * (vo[i] - v[i]) / ((1.0 + eta) * (1.0 + eta));
      const double deta_dS = 1.0 / (2.0 * (double)d.eps_cov * (1.0 + eta));
#pragma unroll
      for (int i = 0; i < kMaxK; ++i)
        if (i < k) {
          if constexpr (ENT) gq[i] = gv[i] / (1.0 + eta) + dot * deta_dS * 2.0 * (v[i] / vo[i] - 1.0) / vo[i];
          else
            d.grad_v[(size_t)b * k + i] =
                (float)(gv[i] / (1.0 + eta) + dot * deta_dS * 2.0 * (v[i] / vo[i] - 1.0) / vo[i] + av[i]);
        }
    } else {
#pragma unroll
      for (int i = 0; i < kMaxK; ++i)
        if (i < k) {
          if constexpr (ENT) gq[i] = gv[i];
          else d.grad_v[(size_t)b * k + i] = (float)(gv[i] + av[i]);
        }
    }
  }
  if constexpr (ENT) {
    // entropy first: chain through v' = alpha(v) v at the original v; grad_v_add reaches the original v after it
    if (d.entropy_first && ent_active) entropy_vjp(gq, v_in, k, alpha);
#pragma unroll
    for (int i = 0; i < kMaxK; ++i)
      if (i < k) d.grad_v[(size_t)b * k + i] = (float)(gq[i] + av[i]);
  }
}


// ---------------------------------------------------------------------------------------------------
// Loss terms around the projection (objectives/trpl.py:231-321, base_projection_layer.py:292-384).
// terms[b] = { log_w, tr_mean, tr_cov, kl_mean + kl_cov, H_dist(proj), H_policy(p), H_policy(proj), advantage }
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) trpl_loss_terms_kernel(const GrlLossDesc d) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= d.batch) return;
  const int k = d.k;
  double maha_a = 0.0, logdet_pv = 0.0, log_pv = 0.0, log_v = 0.0, maha_m = 0.0, trace = 0.0, w2_cov = 0.0;
#pragma unroll
  for (int i = 0; i < kMaxK; ++i) {
    if (i < k) {
      const size_t j = (size_t)b * k + i;
      const double m = d.mean[j], v = d.v[j], pm = d.proj_mean[j], pv = d.proj_v[j], a = d.action[j];
      maha_a += (a - pm) * (a - pm) / pv;          // MultivariateNormal(proj_mean, covariance = diag(proj_v)).log_prob
      logdet_pv += log(pv);
      log_pv += log(pv);
      log_v += log(v);
      const double t = (m - pm) / pv;              // "std" convention: distances divide by the matrix itself
      maha_m += t * t;
      trace += (v / pv) * (v / pv);
      w2_cov += 1.0 + v * v / (pv * pv) - 2.0 * v / pv;
    }
  }
  const double log_prob = -0.5 * (maha_a + k * kLog2Pi + logdet_pv);
  const double kl_mean = 0.5 * maha_m;                                         // projection_utils.py:34-67
  const double kl_cov = 0.5 * (trace - k + 2.0 * log_pv - 2.0 * log_v);
  const double tr_mean = d.proj_type == 0 ? kl_mean : maha_m;                  // projection_utils.py:107-149
  const double tr_cov = d.proj_type == 0 ? kl_cov : w2_cov;
  double* T = d.terms + (size_t)b * GRL_LOSS_TERMS;
  T[0] = log_prob - (double)d.prev_log_prob[b];
  T[1] = tr_mean;
  T[2] = tr_cov;
  T[3] = kl_mean + kl_cov;
  T[4] = 0.5 * (k * (1.0 + kLog2Pi) + logdet_pv);                              // dist.entropy()
  T[5] = 0.5 * (k * (1.0 + kLog2Pi) + 2.0 * log_v);                            // policy.entropy(p): log_determinant = 2 sum log
  T[6] = 0.5 * (k * (1.0 + kLog2Pi) + 2.0 * log_pv);                           // policy.entropy(proj)
  T[7] = (double)d.advantage[b];
}

constexpr int kLossThreads = 1024;

// fixed-order block reductions (deterministic): warp shuffles, then one warp over the 32 partials
__device__ __forceinline__ double block_sum(double x, double* sh) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = x;
  __syncthreads();
  x = sh[threadIdx.x & 31];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}
__device__ __forceinline__ double block_max(double x, double* sh) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x = fmax(x, __shfl_xor_sync(0xffffffffu, x, o));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = x;
  __syncthreads();
  x = sh[threadIdx.x & 31];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x = fmax(x, __shfl_xor_sync(0xffffffffu, x, o));
  return x;
}

// Scheduled entropy bound (see grl_trpl_entropy_bound in grl_b200.h).  Stage 1 needs the whole CTA (block_sum);
// stage 2 is one thread.  The sum runs over samples in a fixed order, so the bound is bit-reproducible.
__global__ void __launch_bounds__(kLossThreads) trpl_entropy_bound_kernel(const GrlEntropyBoundDesc d) {
  __shared__ double sh[32];
  const int B = d.batch, k = d.k, tid = threadIdx.x;
  if (d.stage != 2) {
    double s = 0.0;
    for (int b = tid; b < B; b += blockDim.x) {
      double slog = 0.0;
      for (int i = 0; i < k; ++i) slog += log((double)d.old_v[(size_t)b * k + i]);
      s += 0.5 * (k * (1.0 + kLog2Pi) + 2.0 * slog);  // policy.entropy(q), gnn_gaussian_policy_diag.py:116-122
    }
    s = block_sum(s, sh);
    if (tid == 0) { d.sums[0] = s; d.sums[1] = (double)B; }
  }
  if (d.stage != 1 && tid == 0) {
    double* S = d.state;
    if (S[1] == 0.0) {  // base_projection_layer.py:202-203: latched on the first call, detached
      S[0] = d.sums[0] / d.sums[1];
      S[1] = 1.0;
    }
    const double ie = S[0], te = d.target_entropy, step = (double)*d.step, T = (double)d.total_train_steps;
    S[2] = d.schedule == GRL_ENTROPY_LINEAR ? step * (te - ie) / T + ie
                                            : k * te + (ie - k * te) * pow(d.temperature, 10.0 * step / T);
  }
}

// Data parallel: out[i] = sum_r gathered[r][i] (i < n_sum) | max_r gathered[r][i] (i >= n_sum), ranks visited in rank
// order, so every rank computes bit-identical statistics from ONE all-gather per loss stage.
__global__ void dp_combine_kernel(const double* __restrict__ gathered, int world, int n, int n_sum, double* __restrict__ out) {
  const int i = threadIdx.x;
  if (i >= n) return;
  double acc = gathered[i];
  for (int r = 1; r < world; ++r) {
    const double v = gathered[(size_t)r * n + i];
    acc = i < n_sum ? acc + v : fmax(acc, v);
  }
  out[i] = acc;
}

// stats  = { sum A, sum A^2, n, max log_w, loc, 1 / scale }          (entries 0-3: stage 1; 4-5: stage 2)
// sums   = { [0] sum exp(lw) A_hat, [1] sum (tr_mean + tr_cov), [2] sum H_dist      -> this rank's share of the losses
//            [3] sum e, [4] sum e^2 (e = exp(lw - max)), [5] sum tr_mean, [6] sum tr_cov, [7] sum kl, [8] sum H_p,
//            [9] sum (H_proj - H_p)                                                   -> summed over ranks
//            [10] max tr_mean, [11] max tr_cov }                                      -> max over ranks
// Between the stages a data-parallel caller makes stats[0:3] (sum), stats[3] (max), sums[3:10] (sum) and sums[10:12] (max)
// global: one all-gather of stats[0:4] resp. sums[3:12] + grl_dp_combine per stage; a single process runs the three
// stages back to back.
__global__ void __launch_bounds__(kLossThreads) trpl_loss_stats_kernel(const GrlLossDesc d) {
  __shared__ double sh[32];
  const int B = d.batch, tid = threadIdx.x;
  const double* T = d.terms;
  double s = 0.0, q = 0.0, mx = -1e300;
  for (int b = tid; b < B; b += kLossThreads) {
    const double a = T[(size_t)b * GRL_LOSS_TERMS + 7];
    s += a;
    q += a * a;
    mx = fmax(mx, T[(size_t)b * GRL_LOSS_TERMS]);
  }
  s = block_sum(s, sh);
  q = block_sum(q, sh);
  mx = block_max(mx, sh);
  if (tid == 0) { d.stats[0] = s; d.stats[1] = q; d.stats[2] = (double)B; d.stats[3] = mx; }
}

__global__ void __launch_bounds__(kLossThreads) trpl_loss_sums_kernel(const GrlLossDesc d) {
  __shared__ double sh[32];
  const int B = d.batch, tid = threadIdx.x;
  const double* T = d.terms;
  // advantage standardisation (trpl.py:286-289): mean, unbiased std clamped at 1e-6, over the GLOBAL minibatch
  const double n = d.stats[2];
  double loc = 0.0, inv_scale = 1.0;
  if (d.normalize_advantage && n > 1.0) {
    loc = d.stats[0] / n;
    const double var = fmax((d.stats[1] - n * loc * loc) / (n - 1.0), 0.0);
    inv_scale = 1.0 / fmax(sqrt(var), 1e-6);
  }
  const double mx = d.stats[3];
  double s_obj = 0.0, s_e1 = 0.0, s_e2 = 0.0, s_trm = 0.0, s_trc = 0.0, s_kl = 0.0, s_hd = 0.0, s_hp = 0.0, s_hq = 0.0;
  double m_trm = -1e300, m_trc = -1e300;
  for (int b = tid; b < B; b += kLossThreads) {
    const double* t = T + (size_t)b * GRL_LOSS_TERMS;
    const double lw = t[0];
    s_obj += exp(lw) * ((t[7] - loc) * inv_scale);
    const double e = exp(lw - mx);
    s_e1 += e;
    s_e2 += e * e;
    s_trm += t[1]; s_trc += t[2]; s_kl += t[3]; s_hd += t[4]; s_hp += t[5]; s_hq += t[6];
    m_trm = fmax(m_trm, t[1]);
    m_trc = fmax(m_trc, t[2]);
  }
  s_obj = block_sum(s_obj, sh); s_e1 = block_sum(s_e1, sh); s_e2 = block_sum(s_e2, sh);
  s_trm = block_sum(s_trm, sh); s_trc = block_sum(s_trc, sh); s_kl = block_sum(s_kl, sh);
  s_hd = block_sum(s_hd, sh); s_hp = block_sum(s_hp, sh); s_hq = block_sum(s_hq, sh);
  m_trm = block_max(m_trm, sh); m_trc = block_max(m_trc, sh);
  if (tid == 0) {
    double* S = d.sums;
    S[0] = s_obj; S[1] = s_trm + s_trc; S[2] = s_hd;
    S[3] = s_e1; S[4] = s_e2; S[5] = s_trm; S[6] = s_trc; S[7] = s_kl; S[8] = s_hp; S[9] = s_hq - s_hp;
    S[10] = m_trm; S[11] = m_trc;
    d.stats[4] = loc;
    d.stats[5] = inv_scale;
  }
}

__global__ void trpl_loss_finalize_kernel(const GrlLossDesc d) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const double n = d.stats[2];  // global sample count
  const double* G = d.sums;
  float* S = d.scalars;
  // losses: this rank's share (local sum / global count); summed gradients are then the global-mean gradients
  S[GRL_LS_LOSS_OBJECTIVE] = (float)(-G[0] / n);
  S[GRL_LS_LOSS_TRUST_REGION] = (float)(G[1] / n * (double)d.trust_region_coeff);
  S[GRL_LS_LOSS_ENTROPY] = (float)(-(double)d.entropy_coef * G[2] / n);
  S[GRL_LS_DIST_ENTROPY] = (float)(G[2] / n);
  // exp(2 lse(lw) - lse(2 lw)) / B with both log-sum-exps shifted by max(lw)
  S[GRL_LS_ESS] = (float)(G[3] * G[3] / G[4] / n);
  S[GRL_LS_KL] = (float)(G[7] / n);
  S[GRL_LS_CONSTRAINT] = (float)((G[5] + G[6]) / n);
  S[GRL_LS_MEAN_CONSTRAINT] = (float)(G[5] / n);
  S[GRL_LS_MEAN_CONSTRAINT_MAX] = (float)G[10];
  S[GRL_LS_COV_CONSTRAINT] = (float)(G[6] / n);
  S[GRL_LS_COV_CONSTRAINT_MAX] = (float)G[11];
  S[GRL_LS_ENTROPY] = (float)(G[8] / n);
  S[GRL_LS_ENTROPY_DIFF] = (float)(G[9] / n);
  for (int i = GRL_LS_ENTROPY_DIFF + 1; i < GRL_LOSS_SCALARS; ++i) S[i] = 0.f;
}

__global__ void __launch_bounds__(128) trpl_loss_bwd_kernel(const GrlLossDesc d) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= d.batch) return;
  const int k = d.k;
  const double n = d.stats[2];  // global sample count
  const double g_obj = d.grad_losses[0], g_tr = d.grad_losses[1], g_ent = d.grad_losses[2];
  const double* T = d.terms + (size_t)b * GRL_LOSS_TERMS;
  const double adv = (T[7] - d.stats[4]) * d.stats[5];
  const double g_lw = -g_obj / n * exp(T[0]) * adv;           // d loss_objective / d log_prob
  const double c_ent = -g_ent * (double)d.entropy_coef / n;   // d loss_entropy / d H_dist
  const double c_tr = g_tr * (double)d.trust_region_coeff / n;
#pragma unroll
  for (int i = 0; i < kMaxK; ++i) {
    if (i < k) {
      const size_t j = (size_t)b * k + i;
      const double m = d.mean[j], v = d.v[j], pm = d.proj_mean[j], pv = d.proj_v[j], a = d.action[j];
      const double r = a - pm;
      // log_prob = -0.5 (sum r^2 / pv + k log 2pi + sum log pv);  H_dist = 0.5 (k (1 + log 2pi) + sum log pv)
      d.grad_proj_mean[j] = (float)(g_lw * r / pv);
      d.grad_proj_v[j] = (float)(g_lw * 0.5 * (r * r / (pv * pv) - 1.0 / pv) + c_ent * 0.5 / pv);
      // trust-region value of p against the DETACHED projection
      double gm, gv;
      if (d.proj_type == 0) {
        gm = (m - pm) / (pv * pv);
        gv = v / (pv * pv) - 1.0 / v;
      } else {
        gm = 2.0 * (m - pm) / (pv * pv);
        gv = 2.0 * v / (pv * pv) - 2.0 / pv;
      }
      d.grad_mean_direct[j] = (float)(c_tr * gm);
      d.grad_v_direct[j] = (float)(c_tr * gv);
    }
  }
}

}  // namespace grl

extern "C" {

static int check_proj(const GrlProjDesc* d, const char* who, bool bwd) {
  GRL_REQUIRE(d, GRL_EINVAL, "%s: null descriptor", who);
  GRL_REQUIRE(d->batch > 0 && d->k > 0, GRL_EINVAL, "%s: batch=%d k=%d", who, d->batch, d->k);
  GRL_REQUIRE(d->k <= GRL_MAX_ACTION_DIM, GRL_EUNSUPPORTED, "%s: k=%d > %d", who, d->k, GRL_MAX_ACTION_DIM);
  GRL_REQUIRE(d->proj_type == 0 || d->proj_type == 1, GRL_EUNSUPPORTED, "%s: proj_type=%d", who, d->proj_type);
  GRL_REQUIRE(d->eps_mean > 0.f && d->eps_cov > 0.f, GRL_EINVAL, "%s: bounds must be positive", who);
  GRL_REQUIRE(d->mean && d->v && d->old_mean && d->old_v && d->eta, GRL_EINVAL, "%s: null pointer", who);
  if (bwd) GRL_REQUIRE(d->grad_proj_mean && d->grad_proj_v && d->grad_mean && d->grad_v, GRL_EINVAL, "%s: null grad pointer", who);
  else GRL_REQUIRE(d->proj_mean && d->proj_v, GRL_EINVAL, "%s: null output pointer", who);
  GRL_REQUIRE(d->entropy_mode >= GRL_ENTROPY_OFF && d->entropy_mode <= GRL_ENTROPY_EQ, GRL_EUNSUPPORTED,
              "%s: entropy_mode=%d", who, d->entropy_mode);
  GRL_REQUIRE(d->entropy_first == 0 || (d->entropy_first == 1 && d->entropy_mode != GRL_ENTROPY_OFF), GRL_EINVAL,
              "%s: entropy_first=%d with entropy_mode=%d", who, d->entropy_first, d->entropy_mode);
  if (d->entropy_mode != GRL_ENTROPY_OFF) {
    GRL_REQUIRE(d->entropy_alpha && (bwd || d->entropy_beta), GRL_EINVAL, "%s: null entropy pointer", who);
    if (bwd && !d->entropy_first) GRL_REQUIRE(d->proj_v, GRL_EINVAL, "%s: entropy projection after: null proj_v", who);
  }
  return GRL_OK;
}

int grl_trpl_fwd(const GrlProjDesc* d, grl_stream_t stream) {
  const int rc = check_proj(d, "grl_trpl_fwd", false);
  if (rc != GRL_OK) return rc;
  if (d->entropy_mode == GRL_ENTROPY_OFF)
    grl::trpl_fwd_kernel<false><<<(d->batch + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*d);
  else
    grl::trpl_fwd_kernel<true><<<(d->batch + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*d);
  return grl::check_launch("grl_trpl_fwd");
}

int grl_trpl_bwd(const GrlProjDesc* d, grl_stream_t stream) {
  const int rc = check_proj(d, "grl_trpl_bwd", true);
  if (rc != GRL_OK) return rc;
  if (d->entropy_mode == GRL_ENTROPY_OFF)
    grl::trpl_bwd_kernel<false><<<(d->batch + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*d);
  else
    grl::trpl_bwd_kernel<true><<<(d->batch + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*d);
  return grl::check_launch("grl_trpl_bwd");
}

int grl_trpl_entropy_bound(const GrlEntropyBoundDesc* d, grl_stream_t stream) {
  const char* who = "grl_trpl_entropy_bound";
  GRL_REQUIRE(d, GRL_EINVAL, "%s: null descriptor", who);
  GRL_REQUIRE(d->batch > 0 && d->k > 0, GRL_EINVAL, "%s: batch=%d k=%d", who, d->batch, d->k);
  GRL_REQUIRE(d->k <= GRL_MAX_ACTION_DIM, GRL_EUNSUPPORTED, "%s: k=%d > %d", who, d->k, GRL_MAX_ACTION_DIM);
  GRL_REQUIRE(d->schedule == GRL_ENTROPY_LINEAR || d->schedule == GRL_ENTROPY_EXP, GRL_EUNSUPPORTED,
              "%s: schedule=%d", who, d->schedule);
  GRL_REQUIRE(d->stage >= 0 && d->stage <= 2, GRL_EINVAL, "%s: stage=%d", who, d->stage);
  GRL_REQUIRE(d->total_train_steps > 0, GRL_EINVAL, "%s: total_train_steps=%lld", who, (long long)d->total_train_steps);
  GRL_REQUIRE(d->schedule != GRL_ENTROPY_EXP || d->temperature > 0.0, GRL_EINVAL, "%s: temperature=%g for exp", who,
              d->temperature);
  GRL_REQUIRE(d->step && d->sums && d->state && (d->stage == 2 || d->old_v), GRL_EINVAL, "%s: null pointer", who);
  const int threads = d->stage == 2 ? 32 : grl::kLossThreads;
  grl::trpl_entropy_bound_kernel<<<1, threads, 0, (cudaStream_t)stream>>>(*d);
  return grl::check_launch(who);
}

static int check_loss(const GrlLossDesc* d, const char* who, bool bwd) {
  GRL_REQUIRE(d, GRL_EINVAL, "%s: null descriptor", who);
  GRL_REQUIRE(d->batch > 0 && d->k > 0, GRL_EINVAL, "%s: batch=%d k=%d", who, d->batch, d->k);
  GRL_REQUIRE(d->k <= GRL_MAX_ACTION_DIM, GRL_EUNSUPPORTED, "%s: k=%d > %d", who, d->k, GRL_MAX_ACTION_DIM);
  GRL_REQUIRE(d->proj_type == 0 || d->proj_type == 1, GRL_EUNSUPPORTED, "%s: proj_type=%d", who, d->proj_type);
  GRL_REQUIRE(d->mean && d->v && d->proj_mean && d->proj_v && d->action && d->terms && d->stats, GRL_EINVAL,
              "%s: null pointer", who);
  if (bwd) GRL_REQUIRE(d->grad_losses && d->grad_proj_mean && d->grad_proj_v && d->grad_mean_direct && d->grad_v_direct,
                       GRL_EINVAL, "%s: null grad pointer", who);
  else GRL_REQUIRE(d->prev_log_prob && d->advantage && d->scalars && d->sums, GRL_EINVAL, "%s: null input / output pointer", who);
  return GRL_OK;
}

int grl_trpl_loss_fwd(const GrlLossDesc* d, grl_stream_t stream) {
  const int rc = check_loss(d, "grl_trpl_loss_fwd", false);
  if (rc != GRL_OK) return rc;
  GRL_REQUIRE(d->stage >= 0 && d->stage <= 3, GRL_EINVAL, "grl_trpl_loss_fwd: stage=%d", d->stage);
  cudaStream_t st = (cudaStream_t)stream;
  if (d->stage == 0 || d->stage == 1) {
    grl::trpl_loss_terms_kernel<<<(d->batch + 127) / 128, 128, 0, st>>>(*d);
    grl::trpl_loss_stats_kernel<<<1, grl::kLossThreads, 0, st>>>(*d);
  }
  if (d->stage == 0 || d->stage == 2) grl::trpl_loss_sums_kernel<<<1, grl::kLossThreads, 0, st>>>(*d);
  if (d->stage == 0 || d->stage == 3) grl::trpl_loss_finalize_kernel<<<1, 32, 0, st>>>(*d);
  return grl::check_launch("grl_trpl_loss_fwd");
}

int grl_dp_combine(const double* gathered, int world, int n, int n_sum, double* out, grl_stream_t stream) {
  GRL_REQUIRE(gathered && out && world > 0 && n > 0 && n <= 32 && n_sum >= 0 && n_sum <= n, GRL_EINVAL,
              "grl_dp_combine: world=%d n=%d n_sum=%d", world, n, n_sum);
  grl::dp_combine_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(gathered, world, n, n_sum, out);
  return grl::check_launch("grl_dp_combine");
}

int grl_trpl_loss_bwd(const GrlLossDesc* d, grl_stream_t stream) {
  const int rc = check_loss(d, "grl_trpl_loss_bwd", true);
  if (rc != GRL_OK) return rc;
  grl::trpl_loss_bwd_kernel<<<(d->batch + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*d);
  return grl::check_launch("grl_trpl_loss_bwd");
}

}  // extern "C"
