// Orientation lift + node encoder, forward and weight-gradient backward.
//   x[n][o][c] = sum_s scal[n][s] W[c][s] + sum_v <vec[n][v][:dim], ori[o]> W[c][S+v]
// Reference: geometry_rl/modules/pyg_models/ponita/utils/to_from_sphere.py:4-9 (scalar_to_sphere,
// vec_to_sphere) + hepi.py:136-143 (node_encoder, bias-free Linear) / ponita/ponita.py:358 (x_embedder).
#include "grl_common.cuh"

namespace grl {

constexpr int kMaxF = 16;

constexpr int kEmbTile = 16;  // nodes staged per CTA iteration

// Stage scalars [T][S] and vectors [T][V][3] of `cnt` consecutive nodes into shared memory (coalesced).
__device__ __forceinline__ void embed_stage(const GrlEmbedDesc& d, int n0, int cnt, float* __restrict__ sc, float* __restrict__ vc) {
  const int S = d.n_scalars, V3 = 3 * d.n_vectors;
  if (d.node_ids == nullptr) {
    for (int i = threadIdx.x; i < cnt * S; i += kThreads) sc[i] = d.scalars[(size_t)n0 * S + i];
    for (int i = threadIdx.x; i < cnt * V3; i += kThreads) vc[i] = d.vectors[(size_t)n0 * V3 + i];
  } else {  // live-row evaluation: node n0 + j of the compact batch is row node_ids[n0 + j] of the padded feature arrays
    for (int i = threadIdx.x; i < cnt * S; i += kThreads) sc[i] = d.scalars[(size_t)__ldg(d.node_ids + n0 + i / S) * S + i % S];
    for (int i = threadIdx.x; i < cnt * V3; i += kThreads) vc[i] = d.vectors[(size_t)__ldg(d.node_ids + n0 + i / V3) * V3 + i % V3];
  }
}

// Features of (staged node j, orientation o) -> feat[j][o][0..15] in shared memory (entries >= S + V are zero).
// One (j, o) pair per thread: the 16 channel-group threads of an orientation then share the row by broadcast
// loads instead of each recomputing it.
__device__ __forceinline__ void embed_features(const GrlEmbedDesc& d, const float* __restrict__ sc, const float* __restrict__ vc,
                                               int cnt, float* __restrict__ feat) {
  const int S = d.n_scalars, V = d.n_vectors;
  const int j = threadIdx.x >> 4, o = threadIdx.x & 15;
  const float ox = d.ori[3 * o], oy = d.ori[3 * o + 1], oz = (d.dim == 3) ? d.ori[3 * o + 2] : 0.f;
  float f[kMaxF];
#pragma unroll
  for (int i = 0; i < kMaxF; ++i) {
    float v = 0.f;
    if (j < cnt) {
      if (i < S) {
        v = sc[j * S + i];
      } else if (i < S + V) {
        const float* p = vc + (j * V + (i - S)) * 3;
        v = (p[0] * ox + p[1] * oy) + ((d.dim == 3) ? p[2] * oz : 0.f);
      }
    }
    f[i] = v;
  }
  float* dst = feat + (j * kO + o) * kMaxF;
#pragma unroll
  for (int i = 0; i < kMaxF; i += 4) st4(dst + i, make_float4(f[i], f[i + 1], f[i + 2], f[i + 3]));
}

// FQ = ceil((S + V) / 4): the feature count is a launch constant, so the weight slice of a thread is FQ * 16 registers
// (HEPi: 7 features -> 32 registers -> four CTAs per SM instead of two).  The channel pairs of a thread ride in packed
// FFMA2 (two fused multiply-adds per fma-pipe issue slot, each lane rounded like fmaf).
template <int FQ>
__global__ void __launch_bounds__(kThreads, FQ <= 2 ? 4 : 2) embed_fwd_kernel(const GrlEmbedDesc d) {
  __shared__ __align__(16) float feat[kEmbTile * kO * kMaxF];
  __shared__ float sc[kEmbTile * kMaxF], vc[kEmbTile * kMaxF * 3];
  const int tid = threadIdx.x, o = tid >> 4, cg = tid & 15;
  const int F = d.n_scalars + d.n_vectors;
  unsigned long long w01[4 * FQ], w23[4 * FQ];  // (W[4 cg][f], W[4 cg + 1][f]), (W[4 cg + 2][f], W[4 cg + 3][f])
#pragma unroll
  for (int f = 0; f < 4 * FQ; ++f) {
    float w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) w[i] = (f < F) ? __ldg(d.weight + (size_t)(4 * cg + i) * F + f) : 0.f;
    w01[f] = pack2(w[0], w[1]);
    w23[f] = pack2(w[2], w[3]);
  }
  const int n_tiles = (d.n_nodes + kEmbTile - 1) / kEmbTile;
  for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const int n0 = t * kEmbTile, cnt = min(kEmbTile, d.n_nodes - n0);
    __syncthreads();
    embed_stage(d, n0, cnt, sc, vc);
    __syncthreads();
    embed_features(d, sc, vc, cnt, feat);
    __syncthreads();
#pragma unroll 4
    for (int j = 0; j < cnt; ++j) {
      const float* fr = feat + (j * kO + o) * kMaxF;
      unsigned long long a01 = pack2(0.f, 0.f), a23 = a01;
#pragma unroll
      for (int qd = 0; qd < FQ; ++qd) {
        const float4 fv = ld4(fr + 4 * qd);
        const float fe[4] = {fv.x, fv.y, fv.z, fv.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const unsigned long long ff = pack2(fe[e], fe[e]);
          a01 = ffma2(ff, w01[4 * qd + e], a01);
          a23 = ffma2(ff, w23[4 * qd + e], a23);
        }
      }
      float4 a;
      unpack2(a01, a.x, a.y);
      unpack2(a23, a.z, a.w);
      st4(d.x + (size_t)(n0 + j) * kRow + o * kC + 4 * cg, a);
    }
  }
}

// gW[c][f] = sum_{n,o} grad_x[n][o][c] feat[n][o][f]; per-CTA partial, cross-o reduction through smem.
template <int FQ>
__global__ void __launch_bounds__(kThreads, FQ <= 2 ? 4 : 2) embed_bwd_kernel(const GrlEmbedDesc d) {
  __shared__ __align__(16) float feat[kEmbTile * kO * kMaxF];  // re-used as the reduction buffer at the end
  __shared__ float sc[kEmbTile * kMaxF], vc[kEmbTile * kMaxF * 3];
  const int tid = threadIdx.x, o = tid >> 4, cg = tid & 15;
  const int F = d.n_scalars + d.n_vectors;
  unsigned long long g01[4 * FQ], g23[4 * FQ];
#pragma unroll
  for (int f = 0; f < 4 * FQ; ++f) g01[f] = g23[f] = pack2(0.f, 0.f);
  const int n_tiles = (d.n_nodes + kEmbTile - 1) / kEmbTile;
  for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const int n0 = t * kEmbTile, cnt = min(kEmbTile, d.n_nodes - n0);
    __syncthreads();
    embed_stage(d, n0, cnt, sc, vc);
    __syncthreads();
    embed_features(d, sc, vc, cnt, feat);
    __syncthreads();
#pragma unroll 8
    for (int j = 0; j < cnt; ++j) {
      const float4 gx = ldg4(d.grad_x + (size_t)(n0 + j) * kRow + o * kC + 4 * cg);
      const unsigned long long gx01 = pack2(gx.x, gx.y), gx23 = pack2(gx.z, gx.w);
      const float* fr = feat + (j * kO + o) * kMaxF;
#pragma unroll
      for (int qd = 0; qd < FQ; ++qd) {
        const float4 fv = ld4(fr + 4 * qd);
        const float fe[4] = {fv.x, fv.y, fv.z, fv.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const unsigned long long ff = pack2(fe[e], fe[e]);
          g01[4 * qd + e] = ffma2(gx01, ff, g01[4 * qd + e]);
          g23[4 * qd + e] = ffma2(gx23, ff, g23[4 * qd + e]);
        }
      }
    }
  }
  float* P = d.grad_weight_partials + (size_t)blockIdx.x * kC * F;
  float* red = feat;  // [16 o][64 c]
#pragma unroll
  for (int f = 0; f < 4 * FQ; ++f) {
    if (f < F) {
      float4 g;
      unpack2(g01[f], g.x, g.y);
      unpack2(g23[f], g.z, g.w);
      __syncthreads();
      st4(red + o * kC + 4 * cg, g);
      __syncthreads();
      if (tid < kC) {
        float t = 0.f;
#pragma unroll
        for (int oo = 0; oo < kO; ++oo) t += red[oo * kC + tid];
        P[tid * F + f] = t;
      }
    }
  }
}

}  // namespace grl

extern "C" {

static int check_embed(const GrlEmbedDesc* d, const char* who) {
  GRL_REQUIRE(d, GRL_EINVAL, "%s: null descriptor", who);
  GRL_REQUIRE(d->n_nodes > 0 && (d->dim == 2 || d->dim == 3), GRL_EINVAL, "%s: n_nodes=%d dim=%d", who, d->n_nodes, d->dim);
  GRL_REQUIRE(d->n_scalars >= 0 && d->n_vectors >= 0 && d->n_scalars + d->n_vectors >= 1 &&
                  d->n_scalars + d->n_vectors <= grl::kMaxF, GRL_EUNSUPPORTED, "%s: S+V=%d not in [1,16]", who,
              d->n_scalars + d->n_vectors);
  GRL_REQUIRE((d->n_scalars == 0 || d->scalars) && (d->n_vectors == 0 || d->vectors) && d->ori, GRL_EINVAL,
              "%s: null pointer", who);
  return GRL_OK;
}

int grl_embed_fwd(const GrlEmbedDesc* d, grl_stream_t stream) {
  const int rc = check_embed(d, "grl_embed_fwd");
  if (rc != GRL_OK) return rc;
  GRL_REQUIRE(d->weight && d->x, GRL_EINVAL, "grl_embed_fwd: null pointer");
  const int n_tiles = (d->n_nodes + grl::kEmbTile - 1) / grl::kEmbTile;
  const int fq = (d->n_scalars + d->n_vectors + 3) / 4;
  int grid = (fq <= 2 ? 8 : 6) * grl::sm_count();
  if (grid > n_tiles) grid = n_tiles;
  cudaStream_t st = (cudaStream_t)stream;
  if (fq == 1) grl::embed_fwd_kernel<1><<<grid, grl::kThreads, 0, st>>>(*d);
  else if (fq == 2) grl::embed_fwd_kernel<2><<<grid, grl::kThreads, 0, st>>>(*d);
  else if (fq == 3) grl::embed_fwd_kernel<3><<<grid, grl::kThreads, 0, st>>>(*d);
  else grl::embed_fwd_kernel<4><<<grid, grl::kThreads, 0, st>>>(*d);
  return grl::check_launch("grl_embed_fwd");
}

int grl_embed_bwd(const GrlEmbedDesc* d, grl_stream_t stream) {
  const int rc = check_embed(d, "grl_embed_bwd");
  if (rc != GRL_OK) return rc;
  GRL_REQUIRE(d->grad_x && d->grad_weight_partials && d->n_partials > 0, GRL_EINVAL,
              "grl_embed_bwd: null pointer or n_partials=%d", d->n_partials);
  const int fq = (d->n_scalars + d->n_vectors + 3) / 4;
  cudaStream_t st = (cudaStream_t)stream;
  if (fq == 1) grl::embed_bwd_kernel<1><<<d->n_partials, grl::kThreads, 0, st>>>(*d);
  else if (fq == 2) grl::embed_bwd_kernel<2><<<d->n_partials, grl::kThreads, 0, st>>>(*d);
  else if (fq == 3) grl::embed_bwd_kernel<3><<<d->n_partials, grl::kThreads, 0, st>>>(*d);
  else grl::embed_bwd_kernel<4><<<d->n_partials, grl::kThreads, 0, st>>>(*d);
  return grl::check_launch("grl_embed_bwd");
}

}  // extern "C"
