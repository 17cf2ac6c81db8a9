// M4: equivariant readout of the actuator latents, forward and backward.
// Replaces hepi.py:173-190 / ponita_gcn.py:132-146 with to_from_sphere.py:12-17 (sphere_to_scalar, sphere_to_vec):
//   y[o][j]       = sum_c latent[o][c] W[j][c] + b[j]                         decoder Linear(64 -> od + odv)
//   out_scalar[s] = mean_o y[o][s]
//   out_vec[v][d] = mean_o y[o][od + v] ori[o][d]
//   out[v][d]     = out_vec[v][d] * out_scalar[v]            (od == odv, or od == 1 broadcast)
//   hidden[c]     = mean_o latent[o][c]
// Both means commute with the Linear, so the kernel first reduces the row over the 16 orientations
//   hidden[c] = 1/16 sum_o latent[o][c],   V[c][d] = 1/16 sum_o latent[o][c] ori[o][d]
// (per lane, no communication) and then takes od + 3 odv dot products over the 64 channels (warp shuffles):
//   out_scalar[s] = W[s] . hidden + b[s],   out_vec[v][d] = W[od + v] . V[:, d] + b[od + v] mean_o ori[o][d].
// One warp per node; lane l owns channels 2l, 2l + 1.  The torch formulation needed ~40 launches forward + backward,
// among them a [J x 65536] x [65536 x 64] weight-gradient GEMM that cuBLAS runs without split-K (105 us).
#include "grl_common.cuh"

namespace grl {

constexpr int kMaxJ = GRL_READOUT_MAX_OUT;  // od + odv

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// mean_o ori[o][d], the factor of b_j in the vector readout.  On a symmetric grid (the 2-D circle) the mean is ~1e-8
// while the partial sums of an fp32 loop reach ~5 and leave ~1e-7 of rounding, which b_j * mean would add to every
// output and bias gradient; summed in double, the mean is the float nearest the exact one.
__device__ __forceinline__ float orientation_mean(const float (&ori)[kO][3], int d) {
  double a = 0.0;
  for (int o = 0; o < kO; ++o) a += ori[o][d];
  return (float)(a / kO);
}

struct ReadoutRow {
  float2 hid;     // hidden of channels 2l, 2l+1
  float2 V[3];    // V[c][d]
};

__device__ __forceinline__ ReadoutRow reduce_row(const float* __restrict__ row, const float (&ori)[kO][3], int lane) {
  ReadoutRow r;
  r.hid = make_float2(0.f, 0.f);
  r.V[0] = r.V[1] = r.V[2] = make_float2(0.f, 0.f);
#pragma unroll
  for (int o = 0; o < kO; ++o) {
    const float2 x = __ldg(reinterpret_cast<const float2*>(row + o * kC) + lane);
    r.hid.x += x.x; r.hid.y += x.y;
#pragma unroll
    for (int dd = 0; dd < 3; ++dd) { r.V[dd].x = fmaf(x.x, ori[o][dd], r.V[dd].x); r.V[dd].y = fmaf(x.y, ori[o][dd], r.V[dd].y); }
  }
  const float s = 1.0f / kO;
  r.hid.x *= s; r.hid.y *= s;
#pragma unroll
  for (int dd = 0; dd < 3; ++dd) { r.V[dd].x *= s; r.V[dd].y *= s; }
  return r;
}

__global__ void __launch_bounds__(256) readout_fwd_kernel(const GrlReadoutDesc d) {
  __shared__ float s_ori[kO][3];
  __shared__ float s_obar[3];
  if (threadIdx.x < kO * 3) s_ori[threadIdx.x / 3][threadIdx.x % 3] = d.ori[threadIdx.x];
  __syncthreads();
  if (threadIdx.x < 3) s_obar[threadIdx.x] = orientation_mean(s_ori, threadIdx.x);
  __syncthreads();
  float ori[kO][3];
#pragma unroll
  for (int o = 0; o < kO; ++o) { ori[o][0] = s_ori[o][0]; ori[o][1] = s_ori[o][1]; ori[o][2] = s_ori[o][2]; }
  const int lane = threadIdx.x & 31, od = d.od, odv = d.odv;
  const int warps_per_grid = gridDim.x * (blockDim.x >> 5);
  for (int n = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); n < d.n_nodes; n += warps_per_grid) {
    const ReadoutRow r = reduce_row(d.latent + (size_t)n * kRow, ori, lane);
    reinterpret_cast<float2*>(d.hidden + (size_t)n * kC)[lane] = r.hid;
    float os[kMaxJ];  // out_scalar
#pragma unroll
    for (int s = 0; s < kMaxJ; ++s) {
      os[s] = 0.f;
      if (s < od) {
        const float2 w = __ldg(reinterpret_cast<const float2*>(d.weight + s * kC) + lane);
        os[s] = warp_sum(w.x * r.hid.x + w.y * r.hid.y) + __ldg(d.bias + s);
      }
    }
#pragma unroll
    for (int v = 0; v < kMaxJ; ++v) {
      if (v < odv) {
        const float2 w = __ldg(reinterpret_cast<const float2*>(d.weight + (od + v) * kC) + lane);
        const float bj = __ldg(d.bias + od + v);
        const float gate = os[od == 1 ? 0 : v];
#pragma unroll
        for (int dd = 0; dd < 3; ++dd) {
          const float ov = warp_sum(w.x * r.V[dd].x + w.y * r.V[dd].y) + bj * s_obar[dd];
          if (lane == 0) d.out[((size_t)n * odv + v) * 3 + dd] = dd < d.dim ? ov * gate : 0.f;  // z = 0 padding in 2-D
        }
      }
    }
  }
}

// Backward: g_latent[o][c] = 1/16 (g_hid_tot[c] + sum_d gV[c][d] ori[o][d]); decoder gradients into per-CTA partials
// laid out gW[J][64] | gb[J].
__global__ void __launch_bounds__(256) readout_bwd_kernel(const GrlReadoutDesc d) {
  __shared__ float s_ori[kO][3];
  __shared__ float s_obar[3];
  __shared__ float s_gw[8][kMaxJ * kC + kMaxJ];  // one slice per warp, summed in fixed order at the end
  if (threadIdx.x < kO * 3) s_ori[threadIdx.x / 3][threadIdx.x % 3] = d.ori[threadIdx.x];
  for (int i = threadIdx.x; i < 8 * (kMaxJ * kC + kMaxJ); i += blockDim.x) (&s_gw[0][0])[i] = 0.f;
  __syncthreads();
  if (threadIdx.x < 3) s_obar[threadIdx.x] = orientation_mean(s_ori, threadIdx.x);
  __syncthreads();
  float ori[kO][3];
#pragma unroll
  for (int o = 0; o < kO; ++o) { ori[o][0] = s_ori[o][0]; ori[o][1] = s_ori[o][1]; ori[o][2] = s_ori[o][2]; }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, od = d.od, odv = d.odv, J = od + odv;
  float* gw = s_gw[warp];
  const int warps_per_grid = gridDim.x * (blockDim.x >> 5);
  for (int n = blockIdx.x * (blockDim.x >> 5) + warp; n < d.n_nodes; n += warps_per_grid) {
    const ReadoutRow r = reduce_row(d.latent + (size_t)n * kRow, ori, lane);
    // recompute the gates and the un-gated vectors (cheaper than saving them)
    float os[kMaxJ], g_os[kMaxJ];
#pragma unroll
    for (int s = 0; s < kMaxJ; ++s) {
      os[s] = 0.f; g_os[s] = 0.f;
      if (s < od) {
        const float2 w = __ldg(reinterpret_cast<const float2*>(d.weight + s * kC) + lane);
        os[s] = warp_sum(w.x * r.hid.x + w.y * r.hid.y) + __ldg(d.bias + s);
      }
    }
    float2 g_hid = d.grad_hidden ? reinterpret_cast<const float2*>(d.grad_hidden + (size_t)n * kC)[lane] : make_float2(0.f, 0.f);
    float2 gV[3] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
#pragma unroll
    for (int v = 0; v < kMaxJ; ++v) {
      if (v < odv) {
        const int j = od + v, sidx = od == 1 ? 0 : v;
        const float2 w = __ldg(reinterpret_cast<const float2*>(d.weight + j * kC) + lane);
        const float bj = __ldg(d.bias + j);
        float gb = 0.f;
        float2 gwj = make_float2(0.f, 0.f);
#pragma unroll
        for (int dd = 0; dd < 3; ++dd) {
          if (dd < d.dim) {
            const float go = __ldg(d.grad_out + ((size_t)n * odv + v) * 3 + dd);
            const float ov = warp_sum(w.x * r.V[dd].x + w.y * r.V[dd].y) + bj * s_obar[dd];
            const float g_ov = go * os[sidx];
            g_os[sidx] += go * ov;
            gV[dd].x = fmaf(g_ov, w.x, gV[dd].x); gV[dd].y = fmaf(g_ov, w.y, gV[dd].y);
            gwj.x = fmaf(g_ov, r.V[dd].x, gwj.x); gwj.y = fmaf(g_ov, r.V[dd].y, gwj.y);
            gb = fmaf(g_ov, s_obar[dd], gb);
          }
        }
        gw[j * kC + 2 * lane] += gwj.x;
        gw[j * kC + 2 * lane + 1] += gwj.y;
        if (lane == 0) gw[J * kC + j] += gb;
      }
    }
#pragma unroll
    for (int s = 0; s < kMaxJ; ++s) {
      if (s < od) {
        const float2 w = __ldg(reinterpret_cast<const float2*>(d.weight + s * kC) + lane);
        g_hid.x = fmaf(g_os[s], w.x, g_hid.x); g_hid.y = fmaf(g_os[s], w.y, g_hid.y);
        gw[s * kC + 2 * lane] += g_os[s] * r.hid.x;
        gw[s * kC + 2 * lane + 1] += g_os[s] * r.hid.y;
        if (lane == 0) gw[J * kC + s] += g_os[s];
      }
    }
    const float sc = 1.0f / kO;
    float* gl = d.grad_latent + (size_t)n * kRow;
#pragma unroll
    for (int o = 0; o < kO; ++o) {
      float2 g;
      g.x = sc * (g_hid.x + gV[0].x * ori[o][0] + gV[1].x * ori[o][1] + gV[2].x * ori[o][2]);
      g.y = sc * (g_hid.y + gV[0].y * ori[o][0] + gV[1].y * ori[o][1] + gV[2].y * ori[o][2]);
      reinterpret_cast<float2*>(gl + o * kC)[lane] = g;
    }
  }
  __syncthreads();
  float* P = d.grad_partials + (size_t)blockIdx.x * (J * kC + J);
  for (int i = threadIdx.x; i < J * kC + J; i += blockDim.x) {
    float a = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) a += s_gw[w][i];
    P[i] = a;
  }
}

}  // namespace grl

extern "C" {

static int check_readout(const GrlReadoutDesc* d, const char* who, bool bwd) {
  GRL_REQUIRE(d, GRL_EINVAL, "%s: null descriptor", who);
  GRL_REQUIRE(d->n_nodes > 0 && (d->dim == 2 || d->dim == 3), GRL_EINVAL, "%s: n_nodes=%d dim=%d", who, d->n_nodes, d->dim);
  GRL_REQUIRE(d->od >= 1 && d->odv >= 1 && d->od + d->odv <= GRL_READOUT_MAX_OUT && (d->od == d->odv || d->od == 1),
              GRL_EUNSUPPORTED, "%s: od=%d odv=%d (need od == odv or od == 1, od + odv <= %d)", who, d->od, d->odv,
              GRL_READOUT_MAX_OUT);
  GRL_REQUIRE(d->latent && d->weight && d->bias && d->ori, GRL_EINVAL, "%s: null pointer", who);
  if (bwd)
    GRL_REQUIRE(d->grad_out && d->grad_latent && d->grad_partials && d->n_partials > 0, GRL_EINVAL,
                "%s: null grad pointer or n_partials=%d", who, d->n_partials);
  else GRL_REQUIRE(d->out && d->hidden, GRL_EINVAL, "%s: null output pointer", who);
  return GRL_OK;
}

int grl_readout_fwd(const GrlReadoutDesc* d, grl_stream_t stream) {
  const int rc = check_readout(d, "grl_readout_fwd", false);
  if (rc != GRL_OK) return rc;
  int grid = (d->n_nodes + 7) / 8;
  const int cap = 4 * grl::sm_count();
  if (grid > cap) grid = cap;
  grl::readout_fwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(*d);
  return grl::check_launch("grl_readout_fwd");
}

int grl_readout_bwd(const GrlReadoutDesc* d, grl_stream_t stream) {
  const int rc = check_readout(d, "grl_readout_bwd", true);
  if (rc != GRL_OK) return rc;
  grl::readout_bwd_kernel<<<d->n_partials, 256, 0, (cudaStream_t)stream>>>(*d);
  return grl::check_launch("grl_readout_bwd");
}

}  // extern "C"
