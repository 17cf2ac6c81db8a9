// N4: observation normalisation of the collector (NDVecNorm, geometry_rl_b200/torchrl/envs/transforms.py), every key of
// one call in the same launches.  Key i is x[M_i][C_i] fp32 (M = B F / C rows), its running state the fp32 sum / ssq /
// count tensors of NDVecNorm._stats.
//   vecnorm_partials_kernel  CTA (key, slot s) sums x and x^2 of its rows per component in fp64 (the product of two
//                            floats is exact in fp64); thread t owns component t % C for its whole life, and the CTA's
//                            per-thread sums are added per component in thread order.  No atomics.
//   vecnorm_reduce_kernel    one CTA per key adds the S(M) slots per component in a fixed order -> inc[key][c][2].
//   vecnorm_update_kernel    one CTA per key: the state update with torch's two fp32 roundings (__fmul_rn / __fadd_rn:
//                            build.py does not forbid contraction, and an FMA would round once).
//   vecnorm_apply_kernel     every CTA derives (mean, clamped std) of its key from the state with torch's op order,
//                            then standardises its chunk of elements.
// The slot split depends on M only (not on the SM count or grl_reserve_sms), so the sums do not change with the
// reservation; the update reads the state only after every CTA of the previous launch has finished with it.
#include <math.h>

#include "grl_common.cuh"

namespace grl {

constexpr int kVnThreads = 256;
constexpr int kVnApplyElems = kVnThreads * 8;  // elements per CTA of the standardising launch

__host__ __device__ __forceinline__ int64_t vn_rows(const GrlVecNormKey& k) { return k.batch * k.feat / k.comps; }

__host__ __device__ __forceinline__ int vn_slots(int64_t M) {
  int64_t s = (M + GRL_VECNORM_ROWS_PER_SLOT - 1) / GRL_VECNORM_ROWS_PER_SLOT;
  if (s > GRL_VECNORM_MAX_SLOTS) s = GRL_VECNORM_MAX_SLOTS;
  return s < 1 ? 1 : (int)s;
}

__host__ __device__ __forceinline__ int64_t vn_apply_blocks(const GrlVecNormKey& k) {
  return (vn_rows(k) * k.comps + kVnApplyElems - 1) / kVnApplyElems;
}

// torch.clamp_min(v, lo): a NaN passes through
__device__ __forceinline__ float vn_clamp_min(float v, float lo) { return v < lo ? lo : v; }

__global__ void __launch_bounds__(kVnThreads) vecnorm_partials_kernel(GrlVecNormDesc d) {
  __shared__ double s_red[2][kVnThreads];
  int b = blockIdx.x, i = 0;
  int64_t poff = 0;
  for (; i < d.n_keys; ++i) {
    const int S = vn_slots(vn_rows(d.key[i]));
    if (b < S) break;
    b -= S;
    poff += (int64_t)S * d.key[i].comps * 2;
  }
  const GrlVecNormKey k = d.key[i];
  const int C = k.comps, lanes = (kVnThreads / C) * C;
  const int64_t M = vn_rows(k);
  const int S = vn_slots(M);
  const int64_t per = (M + S - 1) / S;
  const int64_t lo = b * per < M ? b * per : M, hi = lo + per < M ? lo + per : M;
  double s1 = 0.0, s2 = 0.0;
  if (threadIdx.x < lanes) {
    for (int64_t e = lo * C + threadIdx.x; e < hi * C; e += lanes) {
      const double v = (double)__ldg(k.x + e);
      s1 += v;
      s2 += v * v;
    }
  }
  s_red[0][threadIdx.x] = s1;
  s_red[1][threadIdx.x] = s2;
  __syncthreads();
  if (threadIdx.x < C) {
    double a1 = 0.0, a2 = 0.0;
    for (int t = threadIdx.x; t < lanes; t += C) {
      a1 += s_red[0][t];
      a2 += s_red[1][t];
    }
    double* p = d.partials + poff + ((int64_t)b * C + threadIdx.x) * 2;
    p[0] = a1;
    p[1] = a2;
  }
}

__global__ void __launch_bounds__(kVnThreads) vecnorm_reduce_kernel(GrlVecNormDesc d) {
  __shared__ double s_red[2][kVnThreads];
  int64_t poff = 0, ioff = 0;
  for (int j = 0; j < (int)blockIdx.x; ++j) {
    poff += (int64_t)vn_slots(vn_rows(d.key[j])) * d.key[j].comps * 2;
    ioff += (int64_t)d.key[j].comps * 2;
  }
  const GrlVecNormKey k = d.key[blockIdx.x];
  const int C = k.comps, lanes = (kVnThreads / C) * C, S = vn_slots(vn_rows(k));
  // thread t: component t % C of slots t / C, t / C + lanes / C, ...; then per component in thread order
  double s1 = 0.0, s2 = 0.0;
  if (threadIdx.x < lanes) {
    const int c = threadIdx.x % C;
    for (int s = threadIdx.x / C; s < S; s += lanes / C) {
      const double* p = d.partials + poff + ((int64_t)s * C + c) * 2;
      s1 += p[0];
      s2 += p[1];
    }
  }
  s_red[0][threadIdx.x] = s1;
  s_red[1][threadIdx.x] = s2;
  __syncthreads();
  if (threadIdx.x < C) {
    double a1 = 0.0, a2 = 0.0;
    for (int t = threadIdx.x; t < lanes; t += C) {
      a1 += s_red[0][t];
      a2 += s_red[1][t];
    }
    d.inc[ioff + 2 * threadIdx.x] = a1;
    d.inc[ioff + 2 * threadIdx.x + 1] = a2;
  }
}

__global__ void vecnorm_update_kernel(GrlVecNormDesc d) {
  int64_t ioff = 0;
  for (int j = 0; j < (int)blockIdx.x; ++j) ioff += (int64_t)d.key[j].comps * 2;
  const GrlVecNormKey k = d.key[blockIdx.x];
  const int c = threadIdx.x;
  if (c < k.comps) {
    k.sum[c] = __fadd_rn(__fmul_rn(k.sum[c], d.decay), (float)d.inc[ioff + 2 * c]);
    k.ssq[c] = __fadd_rn(__fmul_rn(k.ssq[c], d.decay), (float)d.inc[ioff + 2 * c + 1]);
  }
  if (c == 0) {
    const int64_t M = vn_rows(k);
    const float n = (float)((M > 1 ? M : (int64_t)1) * d.world);
    k.count[0] = __fadd_rn(__fmul_rn(k.count[0], d.decay), n);
  }
}

__global__ void __launch_bounds__(kVnThreads) vecnorm_apply_kernel(GrlVecNormDesc d) {
  __shared__ float s_mean[GRL_VECNORM_MAX_COMPS], s_std[GRL_VECNORM_MAX_COMPS];
  int64_t b = blockIdx.x;
  int i = 0;
  for (; i < d.n_keys; ++i) {
    const int64_t nb = vn_apply_blocks(d.key[i]);
    if (b < nb) break;
    b -= nb;
  }
  const GrlVecNormKey k = d.key[i];
  const int C = k.comps;
  if (threadIdx.x < C) {  // transforms.py:86-88, one rounding per torch op
    const float cnt = k.count[0];
    const float mean = __fdiv_rn(k.sum[threadIdx.x], cnt);
    const float var = __fsub_rn(__fdiv_rn(k.ssq[threadIdx.x], cnt), __fmul_rn(mean, mean));
    s_mean[threadIdx.x] = mean;
    s_std[threadIdx.x] = vn_clamp_min(__fsqrt_rn(vn_clamp_min(var, d.eps)), d.eps);
  }
  __syncthreads();
  const int64_t n = vn_rows(k) * C, e0 = b * kVnApplyElems;
  const int64_t e1 = e0 + kVnApplyElems < n ? e0 + kVnApplyElems : n;
  for (int64_t e = e0 + threadIdx.x; e < e1; e += kVnThreads) {
    const int c = (int)(e % C);
    k.out[e] = __fdiv_rn(__fsub_rn(__ldg(k.x + e), s_mean[c]), s_std[c]);
  }
}

static int vn_check(const GrlVecNormDesc* d, const char* what, bool stats, bool state, bool apply) {
  GRL_REQUIRE(d, GRL_EINVAL, "%s: null descriptor", what);
  GRL_REQUIRE(d->n_keys >= 1 && d->n_keys <= GRL_VECNORM_MAX_KEYS, GRL_EINVAL, "%s: n_keys=%d (1..%d)", what, d->n_keys,
              GRL_VECNORM_MAX_KEYS);
  GRL_REQUIRE(d->world >= 1, GRL_EINVAL, "%s: world=%d", what, d->world);
  GRL_REQUIRE(!stats || (d->partials && d->inc), GRL_EINVAL, "%s: null partials or inc workspace", what);
  GRL_REQUIRE(!state || d->inc, GRL_EINVAL, "%s: null inc", what);
  for (int i = 0; i < d->n_keys; ++i) {
    const GrlVecNormKey& k = d->key[i];
    GRL_REQUIRE(k.comps >= 1, GRL_EINVAL, "%s: key %d: comps=%d", what, i, k.comps);
    GRL_REQUIRE(k.comps <= GRL_VECNORM_MAX_COMPS, GRL_EUNSUPPORTED, "%s: key %d: comps=%d > %d", what, i, k.comps,
                GRL_VECNORM_MAX_COMPS);
    GRL_REQUIRE(k.batch >= 0 && k.feat >= 0, GRL_EINVAL, "%s: key %d: batch=%lld feat=%d (negative rows)", what, i,
                (long long)k.batch, k.feat);
    GRL_REQUIRE(k.feat % k.comps == 0, GRL_EINVAL, "%s: key %d: feat=%d is not a multiple of comps=%d", what, i, k.feat,
                k.comps);
    GRL_REQUIRE(k.x || !(stats || apply), GRL_EINVAL, "%s: key %d: null x", what, i);
    GRL_REQUIRE(k.out || !apply, GRL_EINVAL, "%s: key %d: null out", what, i);
    GRL_REQUIRE((k.sum && k.ssq && k.count) || !(state || apply), GRL_EINVAL, "%s: key %d: null sum, ssq or count", what,
                i);
  }
  return GRL_OK;
}

}  // namespace grl

extern "C" int grl_vecnorm_stats(const GrlVecNormDesc* d, grl_stream_t stream) {
  if (int rc = grl::vn_check(d, "grl_vecnorm_stats", true, false, false)) return rc;
  int64_t grid = 0;
  for (int i = 0; i < d->n_keys; ++i) grid += grl::vn_slots(grl::vn_rows(d->key[i]));
  grl::vecnorm_partials_kernel<<<(unsigned)grid, grl::kVnThreads, 0, (cudaStream_t)stream>>>(*d);
  if (int rc = grl::check_launch("grl_vecnorm_stats")) return rc;
  grl::vecnorm_reduce_kernel<<<d->n_keys, grl::kVnThreads, 0, (cudaStream_t)stream>>>(*d);
  return grl::check_launch("grl_vecnorm_stats");
}

extern "C" int grl_vecnorm_update(const GrlVecNormDesc* d, grl_stream_t stream) {
  if (int rc = grl::vn_check(d, "grl_vecnorm_update", false, true, false)) return rc;
  grl::vecnorm_update_kernel<<<d->n_keys, GRL_VECNORM_MAX_COMPS, 0, (cudaStream_t)stream>>>(*d);
  return grl::check_launch("grl_vecnorm_update");
}

extern "C" int grl_vecnorm_apply(const GrlVecNormDesc* d, grl_stream_t stream) {
  if (int rc = grl::vn_check(d, "grl_vecnorm_apply", false, false, true)) return rc;
  int64_t grid = 0;
  for (int i = 0; i < d->n_keys; ++i) grid += grl::vn_apply_blocks(d->key[i]);
  if (grid == 0) return GRL_OK;
  grl::vecnorm_apply_kernel<<<(unsigned)grid, grl::kVnThreads, 0, (cudaStream_t)stream>>>(*d);
  return grl::check_launch("grl_vecnorm_apply");
}
