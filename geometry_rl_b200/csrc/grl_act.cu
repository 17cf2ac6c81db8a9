// A1: rollout-time Gaussian head and on-device sampling (the acting side of the train loop: ProbabilisticActor(td) once
// per environment step, examples/torchrl/train.py).  One launch turns the body's output into every key the collector
// writes: loc, covariance_matrix (diagonal), action and sample_log_prob.  Arithmetic of
// GNNGaussianPolicyDiag.forward_diag:
//   pre  = hidden W_std^T + b_std  (contextual std)  |  the shared _pre_std vector
//   std  = softplus(pre + shift) + minimal_std        (torch Softplus: the input passes through above 20)
//   var  = std^2,  loc = mean  (tanh(mean) with use_tanh_mean),  mean = hidden W_mean^T + b_mean when post_fc
//   action = loc + eps * std,  log_prob = -0.5 (sum (action - loc)^2 / var + k log(2 pi) + sum log var)
// The head is evaluated in fp64 and rounded once to fp32 (loc, var); log_prob is summed in fp64 from the fp32 outputs.
//
// Noise: counter-based Philox4x32-10 (Salmon et al., SC'11; the Random123 constants), computed inline.
//   key     = (seed & 0xffffffff, (seed >> 32) ^ rank)
//   counter = (component block q, sample index s, call & 0xffffffff, call >> 32)
// Block q yields the four words x0..x3 for components 4q..4q+3 by Box-Muller on two pairs of uniforms:
//   u_i = (x_i + 0.5) * 2^-32 in (0, 1), computed in fp64 (exact)
//   z_{4q+0} = sqrt(-2 ln u_0) cos(2 pi u_1),  z_{4q+1} = sqrt(-2 ln u_0) sin(2 pi u_1)
//   z_{4q+2} = sqrt(-2 ln u_2) cos(2 pi u_3),  z_{4q+3} = sqrt(-2 ln u_2) sin(2 pi u_3)
// evaluated in fp64 and rounded to fp32.  A draw therefore depends on (seed, rank, call, sample, component) only: not
// on the grid, on grl_reserve_sms, or on how the k components split into actuator rows.  `call` is the counter word of
// the state buffer, advanced by grl_act_advance (a separate one-thread launch: no atomics, and a CUDA-graph replay of
// draw + advance takes fresh noise with no host involvement).
#include <math.h>

#include "grl_common.cuh"

namespace grl {

constexpr int kActMaxK = GRL_ACT_MAX_K;  // 32: one lane per component, one warp per sample
constexpr int kActWarps = 8;
constexpr int kActLdw = kC + 1;          // padded row stride of the staged weights (lanes of one step read one column)

struct Philox4 {
  uint32_t x[4];
};

__device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                                 uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t lo0 = 0xD2511F53u * c0, hi0 = __umulhi(0xD2511F53u, c0);
    const uint32_t lo1 = 0xCD9E8D57u * c2, hi1 = __umulhi(0xCD9E8D57u, c2);
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return Philox4{{c0, c1, c2, c3}};
}

// Standard normal of component `c` of sample `s` (see the mapping above).
__device__ __forceinline__ float act_normal(uint32_t k0, uint32_t k1, uint64_t call, uint32_t s, int c) {
  const Philox4 w = philox4x32_10((uint32_t)(c >> 2), s, (uint32_t)call, (uint32_t)(call >> 32), k0, k1);
  const int pair = (c >> 1) & 1;
  const double u_r = ((double)w.x[2 * pair] + 0.5) * 0x1p-32;
  const double u_t = ((double)w.x[2 * pair + 1] + 0.5) * 0x1p-32;
  const double r = sqrt(-2.0 * log(u_r));
  double sn, cs;
  sincospi(2.0 * u_t, &sn, &cs);
  return (float)(r * ((c & 1) ? sn : cs));
}

__device__ __forceinline__ double dot64(const float* __restrict__ w, const float* __restrict__ h) {
  double acc = 0.0;
#pragma unroll 16
  for (int i = 0; i < kC; ++i) acc = fma((double)w[i], (double)__ldg(h + i), acc);
  return acc;
}

__global__ void __launch_bounds__(32 * kActWarps) gaussian_act_kernel(GrlActDesc d) {
  __shared__ float s_wm[kActMaxK * kActLdw];  // _mean.weight   [a][64] (post_fc)
  __shared__ float s_ws[kActMaxK * kActLdw];  // _pre_std.weight [a][64] (contextual std)
  const int a = d.action_dim, A = d.num_rows, k = A * a;
  for (int i = threadIdx.x; i < a * kC; i += blockDim.x) {
    const int j = i / kC, h = i - j * kC;
    if (d.post_fc) s_wm[j * kActLdw + h] = d.mean_weight[i];
    if (d.contextual_std) s_ws[j * kActLdw + h] = d.std_weight[i];
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const bool active = lane < k;
  const int row = active ? lane / a : 0, j = active ? lane - row * a : 0;
  const uint64_t seed = (uint64_t)d.state[0], call = (uint64_t)d.state[1];
  const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32) ^ (uint32_t)d.rank;
  constexpr double kLog2Pi = 1.8378770664093454836;
  for (int s = blockIdx.x * kActWarps + (threadIdx.x >> 5); s < d.batch; s += gridDim.x * kActWarps) {
    float loc = 0.f, var = 1.f, act = 0.f, eps = 0.f;
    double lp = 0.0;
    if (active) {
      const float* h = d.hidden ? d.hidden + ((size_t)s * A + row) * kC : nullptr;
      double mean = d.post_fc ? (double)d.mean_bias[j] + dot64(s_wm + j * kActLdw, h) : (double)d.mean[(size_t)s * k + lane];
      if (d.use_tanh_mean) mean = tanh(mean);
      const double pre = d.contextual_std ? (double)d.std_bias[j] + dot64(s_ws + j * kActLdw, h) : (double)d.std_weight[j];
      const double x = pre + (double)d.pre_shift;
      const double sd = (x > 20.0 ? x : log1p(exp(x))) + (double)d.minimal_std;
      loc = (float)mean;
      var = (float)(sd * sd);
      if (!d.deterministic) {
        eps = act_normal(k0, k1, call, (uint32_t)s, lane);
        act = __fadd_rn(loc, __fmul_rn(eps, (float)sd));
      } else {
        act = loc;
      }
      const double diff = (double)act - (double)loc;
      lp = diff * diff / (double)var + log((double)var);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lp += __shfl_xor_sync(0xffffffffu, lp, o);
    if (active) {
      const size_t base = (size_t)s * k + lane;
      d.loc[base] = loc;
      d.action[base] = act;
      if (d.eps) d.eps[base] = eps;
    }
    if (lane == 0) d.log_prob[s] = (float)(-0.5 * (lp + k * kLog2Pi));
    // covariance_matrix[s]: k x k contiguous floats, diagonal = var, every other entry an exact 0 (coalesced rows).
    // The trip count is warp-uniform: every lane takes part in each shuffle, including lanes past the last entry.
    float* cov = d.cov + (size_t)s * k * k;
    for (int base = 0; base < k * k; base += 32) {
      const int i = base + lane, r = i / k;
      const float v = __shfl_sync(0xffffffffu, var, r & 31);
      if (i < k * k) cov[i] = (i - r * k == r) ? v : 0.f;
    }
  }
}

__global__ void act_advance_kernel(int64_t* state) { state[1] += 1; }

}  // namespace grl

extern "C" int grl_gaussian_act(const GrlActDesc* d, grl_stream_t stream) {
  GRL_REQUIRE(d, GRL_EINVAL, "grl_gaussian_act: null descriptor");
  GRL_REQUIRE(d->hidden_dim == GRL_CHANNELS, GRL_EUNSUPPORTED, "grl_gaussian_act: hidden_dim=%d (only 64)", d->hidden_dim);
  GRL_REQUIRE(d->batch > 0 && d->num_rows > 0 && d->action_dim > 0, GRL_EINVAL,
              "grl_gaussian_act: batch=%d num_rows=%d action_dim=%d", d->batch, d->num_rows, d->action_dim);
  GRL_REQUIRE((int64_t)d->num_rows * d->action_dim <= GRL_ACT_MAX_K, GRL_EUNSUPPORTED,
              "grl_gaussian_act: k = num_rows * action_dim = %lld > %d",
              (long long)d->num_rows * d->action_dim, GRL_ACT_MAX_K);
  GRL_REQUIRE(d->state && d->loc && d->cov && d->action && d->log_prob && d->std_weight, GRL_EINVAL,
              "grl_gaussian_act: null state, output or std pointer");
  GRL_REQUIRE(d->post_fc ? (d->hidden && d->mean_weight && d->mean_bias) : d->mean != nullptr, GRL_EINVAL,
              "grl_gaussian_act: post_fc=%d needs %s", d->post_fc, d->post_fc ? "hidden, mean_weight, mean_bias" : "mean");
  GRL_REQUIRE(!d->contextual_std || (d->hidden && d->std_bias), GRL_EINVAL,
              "grl_gaussian_act: contextual std needs hidden and std_bias");
  int grid = (d->batch + grl::kActWarps - 1) / grl::kActWarps;
  const int cap = 8 * grl::sm_count();
  if (grid > cap) grid = cap;
  grl::gaussian_act_kernel<<<grid, 32 * grl::kActWarps, 0, (cudaStream_t)stream>>>(*d);
  return grl::check_launch("grl_gaussian_act");
}

extern "C" int grl_act_advance(int64_t* state, grl_stream_t stream) {
  GRL_REQUIRE(state, GRL_EINVAL, "grl_act_advance: null state");
  grl::act_advance_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(state);
  return grl::check_launch("grl_act_advance");
}
