// DeepSets critic, inner per-token MLP up to the pooled sum (deepsets.py:34-53 with PyG MLP / LayerNorm(mode='graph')):
//   h    = x W1^T + b1                                  x: [B][N][F] tokens (F <= 16), W1: [64][F]
//   y    = relu((h - mean) / (std + eps) * gamma + beta)  mean / biased std over the WHOLE [B][N][64] tensor, or per group
//                                                        of Bg = B / n_groups consecutive graphs (forward only)
//   ysum = sum_n y[b][n]                                  [B][64]
// (the second Linear of the inner MLP commutes with the token sum: sum_n (y W2^T + b2) = ysum W2^T + N b2, a [B][64] GEMM the
// host applies with torch.)
//
// Nothing of size [B * N][64] ever touches HBM: every pass recomputes h from the 4 F bytes per token of x, so the whole
// critic body costs four streaming reads of x (forward: statistics, then output; backward: LayerNorm gradient sums, then
// weight gradients) instead of ~180 library launches over [B N, 64] activations (round 1: 6.7 ms of side-stream GPU time at
// 8192 graphs x 97 tokens, slowing the actor's kernels by ~20 % through contention).
//
// One CTA works on one graph at a time (persistent, contiguous graph ranges): 256 threads = 16 token lanes x 16 channel
// groups of 4; token lane p owns tokens p, p + 16, ...  Cross-thread sums use fixed-order shared-memory trees; cross-CTA sums
// are per-CTA partial slots reduced in slot order: deterministic, no atomics.  Statistics are accumulated in fp64.
//
// Groups (the time steps of the advantage phase, whose per-step statistics the reference computes in a Python loop): graphs
// are group-major, group g = graphs [g Bg, (g + 1) Bg).  The n_partials CTAs split into S = n_partials / n_groups slots per
// group, so a CTA never spans two groups and its partial slot c = g S + s belongs to group g alone.  With one group this is
// the plain contiguous split of the graphs over the grid.
#include "grl_common.cuh"

namespace grl {

constexpr int kCrThreads = 256;
constexpr int kCrMaxTokens = 256;  // tokens per graph staged at once (cloth critic: 239)

struct CriticSmem {
  float x[kCrMaxTokens * 16];  // [token][16] (F padded with zeros)
  float w1[16 * kC];           // [f][64]
  float red[16 * kC];          // cross-token-lane reduction scratch [lane p][channel]
  double dred[kCrThreads / 32 * 4];
};

__device__ __forceinline__ void critic_stage_w1(float* __restrict__ w1s, const GrlCriticDesc& d) {
  for (int i = threadIdx.x; i < 16 * kC; i += kCrThreads) {
    const int f = i >> 6, c = i & 63;
    w1s[i] = f < d.n_feat ? __ldg(d.w1 + c * d.n_feat + f) : 0.f;
  }
}

// tokens [t0, t0 + cnt) of graph b -> smem rows, zero-padded to 16 features
__device__ __forceinline__ void critic_stage_x(float* __restrict__ xs, const GrlCriticDesc& d, int b, int t0, int cnt) {
  const float* src = d.x + ((size_t)b * d.n_tokens + t0) * d.n_feat;
  for (int i = threadIdx.x; i < cnt * 16; i += kCrThreads) {
    const int t = i >> 4, f = i & 15;
    xs[i] = f < d.n_feat ? __ldg(src + t * d.n_feat + f) : 0.f;
  }
}

__device__ __forceinline__ float4 critic_h(const float* __restrict__ xrow, const float* __restrict__ w1s, int cg, float4 b1) {
  float4 h = b1;
#pragma unroll
  for (int f = 0; f < 16; ++f) {
    const float xv = xrow[f];
    const float4 w = *reinterpret_cast<const float4*>(w1s + f * kC + 4 * cg);
    h.x = fmaf(xv, w.x, h.x); h.y = fmaf(xv, w.y, h.y); h.z = fmaf(xv, w.z, h.z); h.w = fmaf(xv, w.w, h.w);
  }
  return h;
}

// block-wide sum of up to 4 doubles per thread, fixed order; result valid in thread 0
template <int NV>
__device__ __forceinline__ void block_sum_d(double (&v)[NV], double* __restrict__ scratch) {
#pragma unroll
  for (int i = 0; i < NV; ++i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[i] += __shfl_xor_sync(0xffffffffu, v[i], o);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) scratch[warp * 4 + i] = v[i];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      double s = 0.0;
      for (int w = 0; w < kCrThreads / 32; ++w) s += scratch[w * 4 + i];
      v[i] = s;
    }
  }
}

// graphs [g_lo, g_hi) of this CTA: slot s of group g (n_groups == 1: the contiguous split over the whole grid)
__device__ __forceinline__ void critic_range(const GrlCriticDesc& d, int& g_lo, int& g_hi) {
  const int S = d.n_partials / d.n_groups, g = blockIdx.x / S, s = blockIdx.x % S;
  const long long bg = d.n_graphs / d.n_groups;
  g_lo = (int)(g * bg + bg * s / S);
  g_hi = (int)(g * bg + bg * (s + 1) / S);
}

// ---- forward pass 1: partial (sum h, sum h^2) per CTA --------------------------------------------------------------------
__global__ void __launch_bounds__(kCrThreads) critic_stats_kernel(const GrlCriticDesc d) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  CriticSmem& s = *reinterpret_cast<CriticSmem*>(smem_raw);
  const int p = threadIdx.x >> 4, cg = threadIdx.x & 15;
  critic_stage_w1(s.w1, d);
  const float4 b1 = __ldg(reinterpret_cast<const float4*>(d.b1) + cg);
  int g_lo, g_hi;
  critic_range(d, g_lo, g_hi);
  double acc[2] = {0.0, 0.0};
  for (int b = g_lo; b < g_hi; ++b) {
    for (int t0 = 0; t0 < d.n_tokens; t0 += kCrMaxTokens) {
      const int cnt = min(kCrMaxTokens, d.n_tokens - t0);
      __syncthreads();
      critic_stage_x(s.x, d, b, t0, cnt);
      __syncthreads();
      float sm = 0.f, sq = 0.f;
      for (int t = p; t < cnt; t += 16) {
        const float4 h = critic_h(s.x + t * 16, s.w1, cg, b1);
        sm += (h.x + h.y) + (h.z + h.w);
        sq += (h.x * h.x + h.y * h.y) + (h.z * h.z + h.w * h.w);
      }
      acc[0] += (double)sm;
      acc[1] += (double)sq;
    }
  }
  block_sum_d<2>(acc, s.dred);
  if (threadIdx.x == 0) {
    d.stat_partials[2 * blockIdx.x] = acc[0];
    d.stat_partials[2 * blockIdx.x + 1] = acc[1];
  }
}

// out[g][i] = sum over the group's slots of partials[g][slot][i] in slot order (n doubles per slot)
constexpr int kCrCombineThreads = 128;
__global__ void critic_combine_kernel(const double* __restrict__ partials, int n_groups, int n_slots, int n,
                                      double* __restrict__ out) {
  const int j = blockIdx.x * kCrCombineThreads + threadIdx.x;
  if (j >= n_groups * n) return;
  const int g = j / n, i = j % n;
  const double* p = partials + (size_t)g * n_slots * n + i;
  double s = 0.0;
  for (int k = 0; k < n_slots; ++k) s += p[(size_t)k * n];
  out[j] = s;
}

struct CriticNorm {
  float mean, inv, r;  // inv = 1 / (std + eps), r = std / (std + eps)
};
// statistics of this CTA's group (`count` = elements of one group over all ranks)
__device__ __forceinline__ CriticNorm critic_norm(const GrlCriticDesc& d) {
  const double* st = d.stats + 2 * (blockIdx.x / (d.n_partials / d.n_groups));
  const double n = d.count;
  const double mean = st[0] / n;
  double var = st[1] / n - mean * mean;
  var = var > 0.0 ? var : 0.0;
  const double sd = sqrt(var);
  CriticNorm c;
  c.mean = (float)mean;
  c.inv = (float)(1.0 / (sd + (double)d.eps));
  c.r = (float)(sd / (sd + (double)d.eps));
  return c;
}

// ---- forward pass 2: ysum[b] = sum_n relu(LN(h)) ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kCrThreads) critic_fwd_kernel(const GrlCriticDesc d) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  CriticSmem& s = *reinterpret_cast<CriticSmem*>(smem_raw);
  const int p = threadIdx.x >> 4, cg = threadIdx.x & 15;
  critic_stage_w1(s.w1, d);
  const float4 b1 = __ldg(reinterpret_cast<const float4*>(d.b1) + cg);
  const float4 ga = __ldg(reinterpret_cast<const float4*>(d.gamma) + cg);
  const float4 be = __ldg(reinterpret_cast<const float4*>(d.beta) + cg);
  const CriticNorm nm = critic_norm(d);
  int g_lo, g_hi;
  critic_range(d, g_lo, g_hi);
  for (int b = g_lo; b < g_hi; ++b) {
    float4 ys = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int t0 = 0; t0 < d.n_tokens; t0 += kCrMaxTokens) {
      const int cnt = min(kCrMaxTokens, d.n_tokens - t0);
      __syncthreads();
      critic_stage_x(s.x, d, b, t0, cnt);
      __syncthreads();
      for (int t = p; t < cnt; t += 16) {
        const float4 h = critic_h(s.x + t * 16, s.w1, cg, b1);
        ys.x += fmaxf(fmaf((h.x - nm.mean) * nm.inv, ga.x, be.x), 0.f);
        ys.y += fmaxf(fmaf((h.y - nm.mean) * nm.inv, ga.y, be.y), 0.f);
        ys.z += fmaxf(fmaf((h.z - nm.mean) * nm.inv, ga.z, be.z), 0.f);
        ys.w += fmaxf(fmaf((h.w - nm.mean) * nm.inv, ga.w, be.w), 0.f);
      }
    }
    __syncthreads();
    *reinterpret_cast<float4*>(s.red + p * kC + 4 * cg) = ys;
    __syncthreads();
    if (threadIdx.x < kC) {  // token lanes combined in lane order
      float a = 0.f;
#pragma unroll
      for (int k = 0; k < 16; ++k) a += s.red[k * kC + threadIdx.x];
      d.ysum[(size_t)b * kC + threadIdx.x] = a;
    }
  }
}

// ---- backward pass 1: S1 = sum g_xhat, S2 = sum g_xhat * xhat (LayerNorm gradient sums), g_gamma, g_beta ----------------------
// per-CTA slot of stat_partials: [S1, S2]; per-CTA slot of grad_partials: [g_gamma[64] | g_beta[64] | ...]
__global__ void __launch_bounds__(kCrThreads) critic_bwd_stats_kernel(const GrlCriticDesc d) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  CriticSmem& s = *reinterpret_cast<CriticSmem*>(smem_raw);
  const int p = threadIdx.x >> 4, cg = threadIdx.x & 15;
  critic_stage_w1(s.w1, d);
  const float4 b1 = __ldg(reinterpret_cast<const float4*>(d.b1) + cg);
  const float4 ga = __ldg(reinterpret_cast<const float4*>(d.gamma) + cg);
  const float4 be = __ldg(reinterpret_cast<const float4*>(d.beta) + cg);
  const CriticNorm nm = critic_norm(d);
  int g_lo, g_hi;
  critic_range(d, g_lo, g_hi);
  double acc[2] = {0.0, 0.0};
  float4 gg = make_float4(0.f, 0.f, 0.f, 0.f), gb = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int b = g_lo; b < g_hi; ++b) {
    const float4 gy = __ldg(reinterpret_cast<const float4*>(d.grad_ysum + (size_t)b * kC) + cg);
    for (int t0 = 0; t0 < d.n_tokens; t0 += kCrMaxTokens) {
      const int cnt = min(kCrMaxTokens, d.n_tokens - t0);
      __syncthreads();
      critic_stage_x(s.x, d, b, t0, cnt);
      __syncthreads();
      float s1 = 0.f, s2 = 0.f;
      for (int t = p; t < cnt; t += 16) {
        const float4 h = critic_h(s.x + t * 16, s.w1, cg, b1);
        const float xh[4] = {(h.x - nm.mean) * nm.inv, (h.y - nm.mean) * nm.inv, (h.z - nm.mean) * nm.inv, (h.w - nm.mean) * nm.inv};
        const float g[4] = {gy.x, gy.y, gy.z, gy.w}, gam[4] = {ga.x, ga.y, ga.z, ga.w}, bet[4] = {be.x, be.y, be.z, be.w};
        float* ggp = &gg.x;
        float* gbp = &gb.x;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float go = fmaf(xh[k], gam[k], bet[k]) > 0.f ? g[k] : 0.f;  // gradient at the LayerNorm output
          ggp[k] += go * xh[k];
          gbp[k] += go;
          const float gx = go * gam[k];
          s1 += gx;
          s2 += gx * xh[k];
        }
      }
      acc[0] += (double)s1;
      acc[1] += (double)s2;
    }
  }
  block_sum_d<2>(acc, s.dred);
  if (threadIdx.x == 0) {
    d.stat_partials[2 * blockIdx.x] = acc[0];
    d.stat_partials[2 * blockIdx.x + 1] = acc[1];
  }
  float* P = d.grad_partials + (size_t)blockIdx.x * GRL_CRITIC_GRAD_FLOATS;
  __syncthreads();
  *reinterpret_cast<float4*>(s.red + p * kC + 4 * cg) = gg;
  __syncthreads();
  if (threadIdx.x < kC) {
    float a = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k) a += s.red[k * kC + threadIdx.x];
    P[threadIdx.x] = a;
  }
  __syncthreads();
  *reinterpret_cast<float4*>(s.red + p * kC + 4 * cg) = gb;
  __syncthreads();
  if (threadIdx.x < kC) {
    float a = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k) a += s.red[k * kC + threadIdx.x];
    P[kC + threadIdx.x] = a;
  }
}

// ---- backward pass 2: g_h, then g_W1[c][f] = sum g_h[c] x[f], g_b1[c] = sum g_h[c] ---------------------------------------------
// slot layout (GRL_CRITIC_GRAD_FLOATS): g_gamma[64] | g_beta[64] | g_b1[64] | g_W1[64][16]
__global__ void __launch_bounds__(kCrThreads) critic_bwd_kernel(const GrlCriticDesc d) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  CriticSmem& s = *reinterpret_cast<CriticSmem*>(smem_raw);
  const int p = threadIdx.x >> 4, cg = threadIdx.x & 15;
  critic_stage_w1(s.w1, d);
  const float4 b1 = __ldg(reinterpret_cast<const float4*>(d.b1) + cg);
  const float4 ga = __ldg(reinterpret_cast<const float4*>(d.gamma) + cg);
  const float4 be = __ldg(reinterpret_cast<const float4*>(d.beta) + cg);
  const CriticNorm nm = critic_norm(d);
  const float c1 = (float)(d.bstats[0] / d.count);                        // S1 / n
  const float c2 = (float)(d.bstats[1] / (d.count * (double)nm.r));       // S2 / (n r)
  int g_lo, g_hi;
  critic_range(d, g_lo, g_hi);
  float gw[4][16];
  float gb1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int k = 0; k < 4; ++k)
#pragma unroll
    for (int f = 0; f < 16; ++f) gw[k][f] = 0.f;
  for (int b = g_lo; b < g_hi; ++b) {
    const float4 gy = __ldg(reinterpret_cast<const float4*>(d.grad_ysum + (size_t)b * kC) + cg);
    for (int t0 = 0; t0 < d.n_tokens; t0 += kCrMaxTokens) {
      const int cnt = min(kCrMaxTokens, d.n_tokens - t0);
      __syncthreads();
      critic_stage_x(s.x, d, b, t0, cnt);
      __syncthreads();
      for (int t = p; t < cnt; t += 16) {
        const float* xr = s.x + t * 16;
        const float4 h = critic_h(xr, s.w1, cg, b1);
        const float hv[4] = {h.x, h.y, h.z, h.w}, g[4] = {gy.x, gy.y, gy.z, gy.w};
        const float gam[4] = {ga.x, ga.y, ga.z, ga.w}, bet[4] = {be.x, be.y, be.z, be.w};
        float gh[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float xh = (hv[k] - nm.mean) * nm.inv;
          const float gx = fmaf(xh, gam[k], bet[k]) > 0.f ? g[k] * gam[k] : 0.f;
          gh[k] = nm.inv * (gx - c1 - xh * c2);
          gb1[k] += gh[k];
        }
#pragma unroll
        for (int f = 0; f < 16; ++f) {
          const float xv = xr[f];
#pragma unroll
          for (int k = 0; k < 4; ++k) gw[k][f] = fmaf(gh[k], xv, gw[k][f]);
        }
      }
    }
  }
  // combine the 16 token lanes in lane order, one 64-float plane at a time
  float* P = d.grad_partials + (size_t)blockIdx.x * GRL_CRITIC_GRAD_FLOATS;
  auto combine = [&](float v0, float v1, float v2, float v3, float* dst, int stride) {
    __syncthreads();
    *reinterpret_cast<float4*>(s.red + p * kC + 4 * cg) = make_float4(v0, v1, v2, v3);
    __syncthreads();
    if (threadIdx.x < kC) {
      float a = 0.f;
#pragma unroll
      for (int k = 0; k < 16; ++k) a += s.red[k * kC + threadIdx.x];
      dst[(size_t)threadIdx.x * stride] = a;
    }
  };
  combine(gb1[0], gb1[1], gb1[2], gb1[3], P + 2 * kC, 1);
#pragma unroll
  for (int f = 0; f < 16; ++f) combine(gw[0][f], gw[1][f], gw[2][f], gw[3][f], P + 3 * kC + f, 16);
}

}  // namespace grl

extern "C" {

static int critic_check(const GrlCriticDesc* d, const char* who) {
  GRL_REQUIRE(d, GRL_EINVAL, "%s: null descriptor", who);
  GRL_REQUIRE(d->n_graphs > 0 && d->n_tokens > 0 && d->n_feat > 0 && d->n_feat <= 16, GRL_EINVAL,
              "%s: n_graphs=%d n_tokens=%d n_feat=%d (n_feat <= 16)", who, d->n_graphs, d->n_tokens, d->n_feat);
  GRL_REQUIRE(d->x && d->w1 && d->b1 && d->gamma && d->beta && d->stats && d->stat_partials, GRL_EINVAL, "%s: null pointer", who);
  GRL_REQUIRE(d->n_partials > 0 && d->n_partials <= d->n_graphs, GRL_EINVAL, "%s: n_partials=%d must be in [1, n_graphs]", who,
              d->n_partials);
  GRL_REQUIRE(d->n_groups > 0 && d->n_graphs % d->n_groups == 0 && d->n_partials % d->n_groups == 0, GRL_EINVAL,
              "%s: n_groups=%d must be >= 1 and divide n_graphs=%d and n_partials=%d", who, d->n_groups, d->n_graphs,
              d->n_partials);
  return GRL_OK;
}

// the backward pass has no grouped statistics (the advantage phase that uses groups takes no gradients)
static int critic_check_bwd(const GrlCriticDesc* d, const char* who) {
  const int rc = critic_check(d, who);
  if (rc != GRL_OK) return rc;
  GRL_REQUIRE(d->n_groups == 1, GRL_EUNSUPPORTED, "%s: n_groups=%d (the backward pass takes one group)", who, d->n_groups);
  GRL_REQUIRE(d->grad_ysum && d->bstats && d->grad_partials && d->count > 0, GRL_EINVAL, "%s: null pointer", who);
  return GRL_OK;
}

static int critic_grid(const GrlCriticDesc* d) { return d->n_partials; }

static void critic_combine(const GrlCriticDesc* d, double* out, cudaStream_t stream) {
  const int n = d->n_groups * 2;
  grl::critic_combine_kernel<<<(n + grl::kCrCombineThreads - 1) / grl::kCrCombineThreads, grl::kCrCombineThreads, 0, stream>>>(
      d->stat_partials, d->n_groups, d->n_partials / d->n_groups, 2, out);
}

int grl_critic_inner_stats(const GrlCriticDesc* d, grl_stream_t stream) {
  const int rc = critic_check(d, "grl_critic_inner_stats");
  if (rc != GRL_OK) return rc;
  const int smem = (int)sizeof(grl::CriticSmem);
  if (grl::ensure_dynamic_smem((const void*)grl::critic_stats_kernel, smem) != GRL_OK) return GRL_ECUDA;
  const int grid = critic_grid(d);
  grl::critic_stats_kernel<<<grid, grl::kCrThreads, smem, (cudaStream_t)stream>>>(*d);
  critic_combine(d, d->stats, (cudaStream_t)stream);
  return grl::check_launch("grl_critic_inner_stats");
}

int grl_critic_inner_fwd(const GrlCriticDesc* d, grl_stream_t stream) {
  const int rc = critic_check(d, "grl_critic_inner_fwd");
  if (rc != GRL_OK) return rc;
  GRL_REQUIRE(d->ysum && d->count > 0, GRL_EINVAL, "grl_critic_inner_fwd: ysum / count");
  const int smem = (int)sizeof(grl::CriticSmem);
  if (grl::ensure_dynamic_smem((const void*)grl::critic_fwd_kernel, smem) != GRL_OK) return GRL_ECUDA;
  grl::critic_fwd_kernel<<<critic_grid(d), grl::kCrThreads, smem, (cudaStream_t)stream>>>(*d);
  return grl::check_launch("grl_critic_inner_fwd");
}

int grl_critic_inner_bwd_stats(const GrlCriticDesc* d, grl_stream_t stream) {
  const int rc = critic_check_bwd(d, "grl_critic_inner_bwd_stats");
  if (rc != GRL_OK) return rc;
  const int smem = (int)sizeof(grl::CriticSmem);
  if (grl::ensure_dynamic_smem((const void*)grl::critic_bwd_stats_kernel, smem) != GRL_OK) return GRL_ECUDA;
  const int grid = critic_grid(d);
  grl::critic_bwd_stats_kernel<<<grid, grl::kCrThreads, smem, (cudaStream_t)stream>>>(*d);
  critic_combine(d, d->bstats, (cudaStream_t)stream);
  return grl::check_launch("grl_critic_inner_bwd_stats");
}

int grl_critic_inner_bwd(const GrlCriticDesc* d, grl_stream_t stream) {
  const int rc = critic_check_bwd(d, "grl_critic_inner_bwd");
  if (rc != GRL_OK) return rc;
  const int smem = (int)sizeof(grl::CriticSmem);
  if (grl::ensure_dynamic_smem((const void*)grl::critic_bwd_kernel, smem) != GRL_OK) return GRL_ECUDA;
  grl::critic_bwd_kernel<<<critic_grid(d), grl::kCrThreads, smem, (cudaStream_t)stream>>>(*d);
  return grl::check_launch("grl_critic_inner_bwd");
}

}  // extern "C"
