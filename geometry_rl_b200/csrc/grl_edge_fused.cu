// Fused edge side of the message passing, 16-bit tensor-core path: the edge basis is RECOMPUTED inside the kernels
// that consume it, so no [E][16][64] basis / basis-gradient tensor ever exists in HBM (SURVEY 8(d) traffic model:
// "edge basis recomputed on the fly").
//
//   forward  (key = dst, entries sorted by dst, CSR order = the reference's scatter order):
//     F      = 14 polynomial invariants of (i1, i2) per (edge, orientation)          hepi.py:109-123, ponita.py:233-244
//     basis  = GELU(GELU(F W1^T + b1) W2^T + b2)                                     hepi.py:76-82
//     kern   = basis Wk^T                                                            ponita/conv.py:84-87
//     x1[d]  = sum_{e in in(d)} kern[e] * x_src[src(e)]                              ponita/conv.py:116-149
//   backward (key = src, entries sorted by src): recompute F, H1, basis, kern, then
//     g_xsrc[s] = init[s] + sum_{e in out(s)} g_x1[dst(e)] * kern[e]
//     g_kern = g_x1[dst(e)] * x_src[src(e)];  gWk += g_kern^T basis;  g_basis = g_kern Wk
//     gP2 = g_basis * GELU'(pre2);  gW2 += gP2^T H1;  gb2 += colsum gP2;  gH1 = gP2 W2
//     gP1 = gH1 * GELU'(pre1);      [gW1 | gb1] += gP1^T [F | 1]
//
// A tile is 8 edges x 16 orientations = 128 rows = the 128 TMEM lanes.  All five contractions of a tile run on
// tcgen05 (16-bit operands produced by the threads straight into the no-swizzle core-matrix layout of grl_tc.cuh,
// fp32 accumulators in TMEM); invariants, GELU, the message products and the CSR-ordered segmented sums are fp32.
// Weight gradients stay in TMEM for the whole persistent CTA and leave once, as one partial slot per CTA
// (summed in fixed order by grl_reduce_partials): deterministic, no atomics.
//
// Forward: 256 threads, 74 KB shared memory, 128 TMEM columns -> three CTAs per SM overlap each other's MMA round
// trips and epilogues.  The x_src rows of a tile are requested through the bulk-copy engine at the START of the tile
// and land under its two MLP stages.
// Backward: one 800-thread CTA per SM, a four-stage pipeline (producer warp, recompute role, message-product role,
// gradient-epilogue role) over double-buffered operand sets; see the banner above edge_fused_bwd_ws3_kernel.
#include <cuda.h>

#include <cstdlib>

#include "grl_common.cuh"
#include "grl_tc.cuh"

namespace grl {


// first key node n in [0, n_nodes] with cost(n) = 8 * rowptr[n] + n >= target (a tile of 8 edges costs a few
// microseconds of MLP work, a node's flush one 4 KB row)
__device__ __forceinline__ int fused_lower_bound(const int32_t* __restrict__ rowptr, int n_nodes, long long target) {
  int lo = 0, hi = n_nodes;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (8ll * __ldg(rowptr + mid) + mid < target) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// positions of one (edge, orientation) row, loaded one tile ahead
struct RowPos {
  float p[6];
  bool valid;
  __device__ __forceinline__ void load(const GrlFusedEdgeDesc& d, int es, int ed, bool v) {
    valid = v;
    if (v) {
      const float* ps = d.pos_src + 3 * (size_t)es;
      const float* pd = d.pos_dst + 3 * (size_t)ed;
      p[0] = __ldg(ps); p[1] = __ldg(ps + 1); p[2] = __ldg(ps + 2);
      p[3] = __ldg(pd); p[4] = __ldg(pd + 1); p[5] = __ldg(pd + 2);
    }
  }
  // 14 invariant features + (1, 1) against the (hi, lo) split of b1 -> row r of the F image [2 chunks][128][8] bf16
  __device__ __forceinline__ void emit(const GrlFusedEdgeDesc& d, __nv_bfloat16* __restrict__ F, int r) const {
    const int o = r & 15;
    float f[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) f[i] = 0.f;
    if (valid) {
      const float rx = p[0] - p[3], ry = p[1] - p[4], rz = (d.dim == 3) ? p[2] - p[5] : 0.f;
      const float ox = __ldg(d.ori + 3 * o), oy = __ldg(d.ori + 3 * o + 1), oz = (d.dim == 3) ? __ldg(d.ori + 3 * o + 2) : 0.f;
      const float i1 = (rx * ox + ry * oy) + rz * oz;
      const float tx = rx - i1 * ox, ty = ry - i1 * oy, tz = rz - i1 * oz;
      const float i2 = sqrtf((tx * tx + ty * ty) + tz * tz);
      f[0] = i1; f[1] = i2;
      f[2] = i1 * i1; f[3] = i1 * i2; f[4] = i2 * i1; f[5] = i2 * i2;
      f[6] = f[2] * i1; f[7] = f[2] * i2; f[8] = f[3] * i1; f[9] = f[3] * i2;
      f[10] = f[4] * i1; f[11] = f[4] * i2; f[12] = f[5] * i1; f[13] = f[5] * i2;
      f[14] = 1.0f; f[15] = 1.0f;
    }
    *reinterpret_cast<uint4*>(F + ((size_t)0 * kTM + r) * 8) = tc::pack8(f);
    *reinterpret_cast<uint4*>(F + ((size_t)1 * kTM + r) * 8) = tc::pack8(f + 8);
  }
};

// W1 [64][14] row-major + b1 -> bf16 operand image [2 chunks][64 rows n][8 f]; f = 14, 15 hold the (hi, lo) split of b1
__device__ __forceinline__ void stage_w1_bias(__nv_bfloat16* __restrict__ img, const float* __restrict__ w1,
                                              const float* __restrict__ b1) {
  for (int i = threadIdx.x; i < kC * 16; i += blockDim.x) {
    const int n = i >> 4, f = i & 15;
    float w;
    if (f < GRL_BASIS_FEATS) {
      w = __ldg(w1 + n * GRL_BASIS_FEATS + f);
    } else {
      const float b = __ldg(b1 + n);
      const float hi = __bfloat162float(__float2bfloat16_rn(b));
      w = f == GRL_BASIS_FEATS ? hi : b - hi;
    }
    img[tc::op_index(kC, n, f)] = __float2bfloat16_rn(w);
  }
}

// forward only: rows 64..127 of a 128-row B image carry b2 against the same two ones columns, so that the pre1 MMA
// (N = 128) also lays a plane of b2 into the TMEM columns the pre2 MMA then ACCUMULATES onto: no bias adds in the epilogue
__device__ __forceinline__ void stage_w1_b1_b2(__nv_bfloat16* __restrict__ img, const float* __restrict__ w1,
                                               const float* __restrict__ b1, const float* __restrict__ b2) {
  for (int i = threadIdx.x; i < 2 * kC * 16; i += blockDim.x) {
    const int n = i >> 4, f = i & 15;
    float w = 0.f;
    if (f < GRL_BASIS_FEATS) {
      if (n < kC) w = __ldg(w1 + n * GRL_BASIS_FEATS + f);
    } else {
      const float b = n < kC ? __ldg(b1 + n) : __ldg(b2 + n - kC);
      const float hi = __bfloat162float(__float2bfloat16_rn(b));
      w = f == GRL_BASIS_FEATS ? hi : b - hi;
    }
    img[tc::op_index(2 * kC, n, f)] = __float2bfloat16_rn(w);
  }
}

// ---------------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------------
// float offset of the 16-byte chunk k (channels 4k..4k+3 of the half) of row (entry j, orientation o) in a swizzled row tile
__device__ __forceinline__ int swz_off(int j, int half, int o, int k) {
  return (((j * 2 + half) * kO + o) << 5) + ((k ^ (o & 7)) << 2);
}

struct FusedFwdSmem {
  __nv_bfloat16 F[kTM * 16];          // [2 chunks][128][8]
  __half HB[kTM * kC];                // H1 = GELU(pre1), then (same bytes) the basis tile; [8 chunks][128][8] fp16
  float XS[kTM * kC];                 // gathered x_src rows ([8 entries][2 halves][16 rows][32 floats]: 2 KB TMA boxes,
                                      // 128-byte swizzled, at 1024-byte multiples), then the messages in place
  __nv_bfloat16 W1b[2 * kC * 16];     // [2 chunks][128 rows][8 f]: rows 0..63 = [W1 | b1], rows 64..127 = [0 | b2]
  __half W2h[kC * kC];                // [8 chunks][64 rows n][8 k]
  __half Wkh[kC * kC];                // [8 chunks][64 rows c][8 j]
  int src[4][kTE], dst[4][kTE];       // 4-deep index ring: slot (t & 3) holds the entries of tile t
  uint64_t bar[3];                    // MMA completions (pre1, pre2, kern)
  uint64_t bar_x;                     // transaction barrier of the bulk x_src row gather
  uint32_t tmem_base;
};

__global__ void __launch_bounds__(kThreads, 3) edge_fused_fwd_kernel(const GrlFusedEdgeDesc d, const __grid_constant__ CUtensorMap tm_xs) {
  extern __shared__ unsigned char smem_raw[];
  FusedFwdSmem& s = *reinterpret_cast<FusedFwdSmem*>(
      smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u));  // the swizzle atoms want a 1024-byte aligned base
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q = warp & 3, ch = warp >> 2, row = 32 * q + lane;
  const int o = tid >> 4, cg = tid & 15;  // mapping of the segmented-sum phase
  if (tid == 0) {
    tc::mbar_init(&s.bar[0], 1);
    tc::mbar_init(&s.bar[1], 1);
    tc::mbar_init(&s.bar[2], 1);
    tc::mbar_init(&s.bar_x, 1);
    tc::fence_mbar_init();
  }
  if (warp == 0) tc::tmem_alloc(&s.tmem_base, 128);
  stage_w1_b1_b2(s.W1b, d.w1, d.b1, d.b2);
  tc::stage_weight_f16(s.W2h, d.w2, kC, kC, kC);
  tc::stage_weight_f16(s.Wkh, d.wk, kC, kC, kC);
  // this CTA's key (dst) node range: equal cost shares.  The edge count is read from rowptr[n_key], not n_edges: an edge
  // set of fixed capacity (refreshed in place on the device) has n_edges = capacity and its real count only there.
  const long long W = 8ll * __ldg(d.rowptr + d.n_key) + d.n_key;
  const int n_lo = blockIdx.x == 0 ? 0 : fused_lower_bound(d.rowptr, d.n_key, W * blockIdx.x / gridDim.x);
  const int n_hi = blockIdx.x + 1 == gridDim.x ? d.n_key : fused_lower_bound(d.rowptr, d.n_key, W * (blockIdx.x + 1) / gridDim.x);
  const int p0 = d.rowptr[n_lo], p1 = d.rowptr[n_hi];
  const int n_tiles = (p1 - p0 + kTE - 1) / kTE;

  auto load_idx = [&](int t, int& es, int& ed) {
    es = 0; ed = 0;
    const int e = p0 + t * kTE + tid;
    if (tid < kTE && t < n_tiles && e < p1) { es = __ldg(d.e_src + e); ed = __ldg(d.e_dst + e); }
  };
  int es_a, ed_a, es_b, ed_b;  // a: tile t+2 (published in iteration t), b: tile t+3
  load_idx(0, es_a, ed_a);
  if (tid < kTE) { s.src[0][tid] = es_a; s.dst[0][tid] = ed_a; }
  load_idx(1, es_a, ed_a);
  if (tid < kTE) { s.src[1][tid] = es_a; s.dst[1][tid] = ed_a; }
  load_idx(2, es_a, ed_a);
  load_idx(3, es_b, ed_b);
  tc::fence_async_smem();
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = s.tmem_base, lane_addr = tmem + ((uint32_t)(32 * q) << 16);
  const uint32_t fa = tc::smem_u32(s.F), hb = tc::smem_u32(s.HB);
  const uint32_t w1 = tc::smem_u32(s.W1b), w2 = tc::smem_u32(s.W2h), wk = tc::smem_u32(s.Wkh);
  constexpr uint32_t kIdF16 = tc::idesc_f16_ex(128, kC, 0, 0, 0, 0);

  RowPos pos;  // positions of tile t's rows (threads 0..127), loaded during tile t-1
  pos.valid = false;
  if (tid < kTM && n_tiles > 0) {
    const int j = tid >> 4;
    pos.load(d, s.src[0][j], s.dst[0][j], p0 + j < p1);
  }

  int cur = n_lo;
  float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int t = 0; t < n_tiles; ++t) {
    const int slot = t & 3;
    const uint32_t par = (uint32_t)t & 1u;
    const int cnt = min(kTE, p1 - (p0 + t * kTE));
    // publish the indices of tile t+2: slot (t+2)&3 was last read by tile t-2, two barriers ago
    if (tid < kTE) { s.src[(t + 2) & 3][tid] = es_a; s.dst[(t + 2) & 3][tid] = ed_a; }
    es_a = es_b; ed_a = ed_b;
    load_idx(t + 4, es_b, ed_b);
    tc::fence_async_smem();  // generic-proxy accesses to XS (tile t-1) before the bulk engine rewrites it
    __syncthreads();         // (A) everyone is done with tile t-1
    // x_src rows of this tile through tensor-map TMA: lane j < cnt of warp 4 requests the two 16-row x 32-channel boxes of
    // entry j (16 copies per tile instead of 128 per-row bulk copies, whose elect-and-broadcast issue loops were 17 % of
    // the kernel's instructions); they land under the two MLP stages below
    if (tid >= kTM && tid < kTM + kTE) {
      const int j = tid - kTM;
      if (j < cnt) {
        const int srow = s.src[slot][j] * kO;
        tc::tma_load_2d(s.XS + (j * 2 + 0) * 512, &tm_xs, 0, srow, &s.bar_x);
        tc::tma_load_2d(s.XS + (j * 2 + 1) * 512, &tm_xs, 32, srow, &s.bar_x);
      }
      if (j == 0) tc::mbar_expect_tx(&s.bar_x, (uint32_t)cnt * kO * kC * 4u);
    }
    if (cnt < kTE) {  // rows past the end of the list: zeros
      for (int i = tid; i < (kTE - cnt) * kRow / 4; i += kThreads)
        reinterpret_cast<float4*>(s.XS + cnt * kRow)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (tid < kTM) {
      const int j = tid >> 4;
      pos.emit(d, s.F, tid);
      // positions of tile t+1 (its indices were published one iteration ago)
      const int nb = p0 + (t + 1) * kTE + j;
      pos.load(d, s.src[(t + 1) & 3][j], s.dst[(t + 1) & 3][j], t + 1 < n_tiles && nb < p1);
    }
    if (tid >= kTM && tid < kTM + kTE && t + 1 < n_tiles) {  // next tile's x_src rows -> L2
      const int j = tid - kTM;
      if (p0 + (t + 1) * kTE + j < p1) tc::prefetch_l2(d.x_src + (size_t)s.src[(t + 1) & 3][j] * kRow, kRow * 4u);
    }
    tc::fence_async_smem();
    tc::tc_fence_before();
    __syncthreads();  // (B)
    if (tid == 0) {   // [pre1 | b2 plane] = [F | 1 1] [[W1 | b1] ; [0 | b2]]^T   (N = 128: TMEM columns 0..127)
      tc::tc_fence_after();
      tc::issue_mma(tmem, tc::view_k(fa, kTM), tc::view_k(w1, 2 * kC), tc::idesc_bf16(128, 2 * kC), 1, false);
      tc::mma_commit(&s.bar[0]);
    }
    tc::mbar_wait(&s.bar[0], par);
    tc::tc_fence_after();
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int c0 = 32 * ch + 16 * i;
      float v[16];
      tc::tmem_ld16(lane_addr + c0, v);
      __half2 h0[4], h1[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        h0[e] = tc::gelu_h2(__floats2half2_rn(v[2 * e], v[2 * e + 1]));
        h1[e] = tc::gelu_h2(__floats2half2_rn(v[8 + 2 * e], v[8 + 2 * e + 1]));
      }
      *reinterpret_cast<uint4*>(s.HB + ((size_t)(c0 >> 3) * kTM + row) * 8) = tc::pack_h8(h0);
      *reinterpret_cast<uint4*>(s.HB + ((size_t)((c0 >> 3) + 1) * kTM + row) * 8) = tc::pack_h8(h1);
    }
    tc::fence_async_smem();
    tc::tc_fence_before();
    __syncthreads();  // (C)
    if (tid == 0) {   // pre2 = b2 plane + H1 W2^T
      tc::tc_fence_after();
      tc::issue_mma(tmem + kC, tc::view_k(hb, kTM), tc::view_k(w2, kC), kIdF16, kC / 16, true);
      tc::mma_commit(&s.bar[1]);
    }
    tc::mbar_wait(&s.bar[1], par);
    tc::tc_fence_after();
#pragma unroll
    for (int i = 0; i < 2; ++i) {  // basis = GELU(pre2) over the H1 bytes (the MMA that read them has completed)
      const int c0 = 32 * ch + 16 * i;
      float v[16];
      tc::tmem_ld16(lane_addr + kC + c0, v);
      __half2 h0[4], h1[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        h0[e] = tc::gelu_h2(__floats2half2_rn(v[2 * e], v[2 * e + 1]));
        h1[e] = tc::gelu_h2(__floats2half2_rn(v[8 + 2 * e], v[8 + 2 * e + 1]));
      }
      *reinterpret_cast<uint4*>(s.HB + ((size_t)(c0 >> 3) * kTM + row) * 8) = tc::pack_h8(h0);
      *reinterpret_cast<uint4*>(s.HB + ((size_t)((c0 >> 3) + 1) * kTM + row) * 8) = tc::pack_h8(h1);
    }
    tc::fence_async_smem();
    tc::tc_fence_before();
    __syncthreads();  // (D)
    if (tid == 0) {   // kern = basis Wk^T   (pre1's columns are free again)
      tc::tc_fence_after();
      tc::issue_mma(tmem, tc::view_k(hb, kTM), tc::view_k(wk, kC), kIdF16, kC / 16, false);
      tc::mma_commit(&s.bar[2]);
    }
    tc::mbar_wait(&s.bar_x, par);  // the x_src rows have landed
    tc::mbar_wait(&s.bar[2], par);
    tc::tc_fence_after();
#pragma unroll
    for (int i = 0; i < 2; ++i) {  // messages in place: XS[row][c] *= kern[row][c]
      const int c0 = 32 * ch + 16 * i;
      float v[16];
      tc::tmem_ld16(lane_addr + c0, v);
      float* xs = s.XS + ((((row >> 4) * 2 + ch) * kO + (row & 15)) << 5);
#pragma unroll
      for (int e4 = 0; e4 < 4; ++e4) {
        float* px = xs + (((4 * i + e4) ^ (row & 7)) << 2);
        const int e = 4 * e4;
        float4 x = ld4(px);
        x.x *= v[e]; x.y *= v[e + 1]; x.z *= v[e + 2]; x.w *= v[e + 3];
        st4(px, x);
      }
    }
    tc::tc_fence_before();
    __syncthreads();  // (E)
    // CSR-ordered segmented sum: thread (o, 4 channels) adds the edges of the tile sequentially
#pragma unroll
    for (int j = 0; j < kTE; ++j) {
      if (j < cnt) {
        const int dn = s.dst[slot][j];
        while (cur < dn) {
          st4(d.x1 + (size_t)cur * kRow + o * kC + 4 * cg, sum);
          sum = make_float4(0.f, 0.f, 0.f, 0.f);
          ++cur;
        }
        const float4 m = ld4(s.XS + swz_off(j, cg >> 3, o, cg & 7));
        sum.x += m.x; sum.y += m.y; sum.z += m.z; sum.w += m.w;
      }
    }
  }
  while (cur < n_hi) {
    st4(d.x1 + (size_t)cur * kRow + o * kC + 4 * cg, sum);
    sum = make_float4(0.f, 0.f, 0.f, 0.f);
    ++cur;
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tmem, 128);
}

// ---------------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------------
// sum over the 32 lanes of a warp of 16 per-lane values by recursive halving; on return lane l holds in v[0] the
// total of original index l >> 1 (lanes l and l ^ 1 hold the same total).  Fixed exchange pattern -> deterministic.
__device__ __forceinline__ void warp_colsum16(float (&v)[16], int lane) {
#pragma unroll
  for (int step = 0; step < 4; ++step) {
    const int half = 8 >> step;
    const int bit = 16 >> step;
    const bool upper = (lane & bit) != 0;
#pragma unroll
    for (int i = 0; i < half; ++i) {
      const float keep = upper ? v[i + half] : v[i];
      const float send = upper ? v[i] : v[i + half];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, bit);
    }
  }
  v[0] += __shfl_xor_sync(0xffffffffu, v[0], 1);
}


// ---------------------------------------------------------------------------------------------------
// backward: a four-stage pipeline inside one CTA per SM.
// A tile's work is a serial chain of tensor-core round trips (pre1 -> pre2 -> kern -> products -> g_basis -> gP2 -> gH1 -> gP1)
// that no prefetching shortens (the lock-step and two-role generations of this kernel spent 16 k and 10.6 k cycles per tile in
// it: profiles/r02_*).  The chain is therefore cut into roles that work on consecutive tiles:
//   producer (warp 24)  owns the index stream and the row gathers, one tile ahead.  Rows arrive through tensor maps
//                          (cp.async.bulk.tensor.2d, SASS UTMALDG): one 16-row x 32-channel box per (edge, channel half),
//                          128-byte swizzled, so the row tiles need no padding; (src, dst, leader) of the tile are published
//                          under the same transaction barrier as the data
//   role R  (warps 0..7)   features -> pre1 -> H1, GELU' -> pre2 -> basis, GELU' (packed fp16)   into operand set t & 1
//   role C1 (warps 8..15)  kern MMA, message products (g_x1 * kern in place, g_kern image), issues the g_basis / gWk
//                          MMAs, src-CSR segmented sum -> grad_x_src
//   role C2 (warps 16..23) gP2 = g_basis * GELU'(pre2), gb2, issues the gH1 / gW2 MMAs, gP1 = gH1 * GELU'(pre1), issues
//                          the [gW1 | gb1] MMA whose commit frees the operand set
// TMEM (464 columns): one 64-column scratch for pre1 / pre2 (role R works on one tile at a time), 64 columns per operand
// set for the two packed fp16 derivative planes, 64 for kern (C1), 64 for g_basis / gH1 (C2), 144 for the weight gradients.
// Hand-offs: full[b] (R -> C1, C2), bar_c[1] = the g_basis MMA's commit (C1 -> C2), b2_free (C2 -> C1: the g_basis / gH1
// columns may be overwritten), empty[b] = the last MMA's commit (C2 -> R, C1: operand set b and gradient image b are free).
// ---------------------------------------------------------------------------------------------------
constexpr int kWs3Threads = 800;

struct FusedBwdWs3Smem {
  float GX[kTM * kC];            // [8 entries][2 halves][16 rows][32 floats]: 2 KB boxes at 1024-byte multiples, swizzled by TMA
  float XS[kTM * kC];
  float IN[kTM * kC];            // residual rows (grad_x_src_init) of the nodes whose run STARTS in this tile, same layout
  __nv_bfloat16 F[2][kTM * 16];
  __nv_bfloat16 H1[2][kTM * kC];
  __nv_bfloat16 BZ[2][kTM * kC];
  __nv_bfloat16 W1b[kC * 16];
  __nv_bfloat16 Wkb[kC * kC];    // [Wkb | W2b] and G[0] are the ignored X halves of the [X | G] images of G[0] and G[1]
  __nv_bfloat16 W2b[kC * kC];
  __nv_bfloat16 G[2][kTM * kC];  // MUST directly follow W2b
  float b2[kC];
  float acc_gb2[4][kC];
  int src[4][kTE], dst[4][kTE], lead[4][kTE];
  int adv[4][kTE];               // key nodes to advance before adding entry j: 0 = same node as the previous entry
  uint64_t bar_r[2], bar_c[3], full[2], empty[2];
  uint64_t bar_g, xs_free, gx_free, b2_free;
  uint32_t tmem_base;
};

__global__ void __launch_bounds__(kWs3Threads, 1)
edge_fused_bwd_ws3_kernel(const GrlFusedEdgeDesc d, const __grid_constant__ CUtensorMap tm_gx, const __grid_constant__ CUtensorMap tm_xs,
                          const __grid_constant__ CUtensorMap tm_in) {
  extern __shared__ unsigned char smem_dyn[];
  FusedBwdWs3Smem& s = *reinterpret_cast<FusedBwdWs3Smem*>(
      smem_dyn + ((1024u - (tc::smem_u32(smem_dyn) & 1023u)) & 1023u));  // the swizzle atoms want a 1024-byte aligned base
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int role = warp < 8 ? 0 : (warp < 16 ? 1 : (warp < 24 ? 2 : 3));  // R, C1, C2, producer
  const int rw = warp & 7;                                                // warp index inside the role
  const int rt = rw * 32 + lane;
  const int q = rw & 3, ch = rw >> 2, row = 32 * q + lane;
  if (tid == 0) {
    tc::mbar_init(&s.bar_r[0], 1);
    tc::mbar_init(&s.bar_r[1], 1);
    for (int i = 0; i < 3; ++i) tc::mbar_init(&s.bar_c[i], 1);
    tc::mbar_init(&s.full[0], 256);
    tc::mbar_init(&s.full[1], 256);
    tc::mbar_init(&s.empty[0], 1);
    tc::mbar_init(&s.empty[1], 1);
    tc::mbar_init(&s.bar_g, 1);
    tc::mbar_init(&s.xs_free, 256);
    tc::mbar_init(&s.gx_free, 256);
    tc::mbar_init(&s.b2_free, 1);
    tc::fence_mbar_init();
  }
  if (warp == 0) tc::tmem_alloc(&s.tmem_base, 512);
  stage_w1_bias(s.W1b, d.w1, d.b1);
  tc::stage_weight_bf16(s.W2b, d.w2, kC, kC, kC);
  tc::stage_weight_bf16(s.Wkb, d.wk, kC, kC, kC);
  if (tid < kC) s.b2[tid] = __ldg(d.b2 + tid);
  if (tid < 4 * kC) (&s.acc_gb2[0][0])[tid] = 0.f;
  const long long W = 8ll * __ldg(d.rowptr + d.n_key) + d.n_key;  // real edge count, as in the forward
  const int n_lo = blockIdx.x == 0 ? 0 : fused_lower_bound(d.rowptr, d.n_key, W * blockIdx.x / gridDim.x);
  const int n_hi = blockIdx.x + 1 == gridDim.x ? d.n_key : fused_lower_bound(d.rowptr, d.n_key, W * (blockIdx.x + 1) / gridDim.x);
  const int p0 = d.rowptr[n_lo], p1 = d.rowptr[n_hi];
  const int n_tiles = (p1 - p0 + kTE - 1) / kTE;
  tc::fence_async_smem();
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = s.tmem_base, lane_addr = tmem + ((uint32_t)(32 * q) << 16);
  const uint32_t w1 = tc::smem_u32(s.W1b), w2 = tc::smem_u32(s.W2b), wk = tc::smem_u32(s.Wkb);
  // TMEM columns: [0,64) pre1 / pre2 scratch   set b: [64 + 64 b, +32) packed GELU'(pre1), [+32, +64) packed GELU'(pre2)
  //               [192,256) kern   [256,320) g_basis -> gH1   [320,384) gWk   [384,448) gW2   [448,464) [gW1 | gb1]
  constexpr uint32_t kScr = 0, kKern = 192, kGB = 256, kGWk = 320, kGW2 = 384, kGW1 = 448;

  if (role == 3) {
    // =========================================== producer warp =====================================================
    if (lane == 0) {
      tc::tma_prefetch_desc(&tm_gx);
      tc::tma_prefetch_desc(&tm_xs);
    }
    if (lane == 0) tc::tma_prefetch_desc(&tm_in);
    int es = 0, ed = 0, es_n = 0, ed_n = 0;
    int last_key = n_lo;  // key node of the previous entry (the segmented sum starts at node n_lo)
    auto load_idx = [&](int t_, int& a, int& b_) {
      a = 0; b_ = 0;
      const int e = p0 + t_ * kTE + lane;
      if (lane < kTE && t_ < n_tiles && e < p1) { a = __ldg(d.e_src + e); b_ = __ldg(d.e_dst + e); }
    };
    load_idx(0, es, ed);
    for (int t = 0; t < n_tiles; ++t) {
      const int slot = t & 3;
      const int cnt = min(kTE, p1 - (p0 + t * kTE));
      load_idx(t + 1, es_n, ed_n);
      // src-sorted list: equal sources are adjacent, so a run inside the tile shares one staged x_src row tile
      int prev = __shfl_up_sync(0xffffffffu, es, 1);
      const bool valid = lane < cnt;
      const bool starts = lane == 0 || !valid || es != prev;
      const unsigned heads = __ballot_sync(0xffffffffu, starts);
      const int ld = 31 - __clz(heads & ((2u << lane) - 1u));
      const unsigned leaders = __ballot_sync(0xffffffffu, valid && ld == lane);
      if (lane == 0) prev = last_key;
      const int adv = valid ? es - prev : 0;  // > 0: entry j starts the run of a new key node (adv - 1 edge-less nodes skipped)
      const unsigned run_starts = d.grad_x_src_init ? __ballot_sync(0xffffffffu, adv > 0) : 0u;
      last_key = __shfl_sync(0xffffffffu, es, cnt - 1);
      if (lane < kTE) { s.src[slot][lane] = es; s.dst[slot][lane] = ed; s.lead[slot][lane] = ld; s.adv[slot][lane] = adv; }
      if (lane < kTE && t + 1 < n_tiles && p0 + (t + 1) * kTE + lane < p1) {  // next tile's rows -> L2
        tc::prefetch_l2(d.grad_x1 + (size_t)ed_n * kRow, kRow * 4u);
        tc::prefetch_l2(d.x_src + (size_t)es_n * kRow, kRow * 4u);
        if (d.grad_x_src_init) tc::prefetch_l2(d.grad_x_src_init + (size_t)es_n * kRow, kRow * 4u);
      }
      if (t > 0) tc::mbar_wait(&s.xs_free, (uint32_t)(t - 1) & 1u);  // role C1 has multiplied tile t-1's x_src rows
      if (cnt < kTE) {  // rows past the end of the list: zeros (they meet finite rows in the products)
        for (int i = lane; i < (kTE - cnt) * kRow / 4; i += 32) {
          reinterpret_cast<float4*>(s.XS + cnt * kRow)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
      if (valid && ld == lane) {
        tc::tma_load_2d(s.XS + (lane * 2 + 0) * 512, &tm_xs, 0, es * kO, &s.bar_g);
        tc::tma_load_2d(s.XS + (lane * 2 + 1) * 512, &tm_xs, 32, es * kO, &s.bar_g);
      }
      if (t > 0) tc::mbar_wait(&s.gx_free, (uint32_t)(t - 1) & 1u);  // ... and summed its g_x1 * kern rows
      if (cnt < kTE) {
        for (int i = lane; i < (kTE - cnt) * kRow / 4; i += 32) {
          reinterpret_cast<float4*>(s.GX + cnt * kRow)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
      if (valid) {
        tc::tma_load_2d(s.GX + (lane * 2 + 0) * 512, &tm_gx, 0, ed * kO, &s.bar_g);
        tc::tma_load_2d(s.GX + (lane * 2 + 1) * 512, &tm_gx, 32, ed * kO, &s.bar_g);
      }
      if ((run_starts >> lane) & 1u) {  // residual row of a node whose run starts here (read by the segmented sum)
        tc::tma_load_2d(s.IN + (lane * 2 + 0) * 512, &tm_in, 0, es * kO, &s.bar_g);
        tc::tma_load_2d(s.IN + (lane * 2 + 1) * 512, &tm_in, 32, es * kO, &s.bar_g);
      }
      __syncwarp();
      // one arrival + the byte count: completes when every box has landed; release also publishes the ring slot
      if (lane == 0) tc::mbar_expect_tx(&s.bar_g, (uint32_t)(cnt + __popc(leaders) + __popc(run_starts)) * kRow * 4u);
      es = es_n; ed = ed_n;
    }
  } else if (role == 0) {
    // =========================================== role R ===========================================================
    RowPos pos;
    int es_n = 0, ed_n = 0;
    bool v_n = false;
    auto load_ids = [&](int t_) {
      const int e = p0 + t_ * kTE + (rt >> 4);
      v_n = rt < kTM && t_ < n_tiles && e < p1;
      if (v_n) { es_n = __ldg(d.e_src + e); ed_n = __ldg(d.e_dst + e); }
    };
    pos.valid = false;
    load_ids(0);
    pos.load(d, es_n, ed_n, v_n);
    load_ids(1);
    for (int t = 0; t < n_tiles; ++t) {
      const int b = t & 1;
      const uint32_t par = (uint32_t)t & 1u, parb = (uint32_t)(t >> 1) & 1u;
      const uint32_t fa = tc::smem_u32(s.F[b]), ha = tc::smem_u32(s.H1[b]);
      const uint32_t kSet = 64u + 64u * b;
      tc::mbar_wait(&s.empty[b], parb ^ 1u);  // roles C1 / C2 are done with set b (tile t-2); passes at once for t < 2
      tc::tc_fence_after();
      if (rt < kTM) {
        pos.emit(d, s.F[b], rt);
        pos.load(d, es_n, ed_n, v_n);
        load_ids(t + 2);
      }
      tc::fence_async_smem();
      tc::tc_fence_before();
      tc::group_sync(1, 256);  // also: every thread has read tile t-1's pre2 from the scratch columns
      if (rt == 0) {  // pre1 = [F | 1 1] [W1 | b1]^T
        tc::tc_fence_after();
        tc::issue_mma(tmem + kScr, tc::view_k(fa, kTM), tc::view_k(w1, kC), tc::idesc_bf16(128, kC), 1, false);
        tc::mma_commit(&s.bar_r[0]);
      }
      tc::mbar_wait(&s.bar_r[0], par);
      tc::tc_fence_after();
#pragma unroll
      for (int layer = 0; layer < 2; ++layer) {
        __nv_bfloat16* img = layer == 0 ? s.H1[b] : s.BZ[b];
        if (layer == 1) {
          tc::fence_async_smem();
          tc::tc_fence_before();
          tc::group_sync(1, 256);  // H1 is complete and every thread has read pre1: the scratch columns may be rewritten
          if (rt == 0) {  // pre2 = H1 W2^T
            tc::tc_fence_after();
            tc::issue_mma(tmem + kScr, tc::view_k(ha, kTM), tc::view_k(w2, kC), tc::idesc_bf16(128, kC), kC / 16, false);
            tc::mma_commit(&s.bar_r[1]);
          }
          tc::mbar_wait(&s.bar_r[1], par);
          tc::tc_fence_after();
        }
        uint32_t dpk[16];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int c0 = 32 * ch + 16 * i;
          float v[16];
          tc::tmem_ld16(lane_addr + kScr + c0, v);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            float x0 = v[2 * e], x1 = v[2 * e + 1];
            if (layer == 1) { x0 += s.b2[c0 + 2 * e]; x1 += s.b2[c0 + 2 * e + 1]; }
            __half2 y, dy;
            tc::gelu_h2(__floats2half2_rn(x0, x1), y, dy);
            const float2 yf = __half22float2(y);
            v[2 * e] = yf.x; v[2 * e + 1] = yf.y;
            dpk[8 * i + e] = *reinterpret_cast<const uint32_t*>(&dy);
          }
          *reinterpret_cast<uint4*>(img + ((size_t)(c0 >> 3) * kTM + row) * 8) = tc::pack8(v);
          *reinterpret_cast<uint4*>(img + ((size_t)((c0 >> 3) + 1) * kTM + row) * 8) = tc::pack8(v + 8);
        }
        // packed GELU' of this thread's 32 columns -> 16 columns of the set's derivative plane `layer`
        tc::tmem_st16(lane_addr + kSet + 32 * layer + 16 * ch, dpk);
      }
      tc::tmem_st_wait();
      tc::fence_async_smem();
      tc::tc_fence_before();
      tc::mbar_arrive(&s.full[b]);
    }
  } else if (role == 1) {
    // =========================================== role C1 ==========================================================
    const int o = rt >> 4, cg = rt & 15;  // mapping of the segmented-sum phase
    int cur = n_lo;
    const size_t toff = (size_t)o * kC + 4 * cg;
    const bool has_init = d.grad_x_src_init != nullptr;
    float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
    // residual row of node `cur`: from global memory for the first node of the range, from the IN tile (TMA, one tile
    // ahead of its use) for every node whose run starts later
    float4 init = has_init && cur < n_hi ? ldg4(d.grad_x_src_init + (size_t)cur * kRow + toff) : make_float4(0.f, 0.f, 0.f, 0.f);
    // rows of the edge-less nodes [lo, hi): the residual rows alone (rare: kNN graphs have a few nodes nobody points to)
    auto fill_gap = [&](int lo, int hi) {
      for (int n = lo; n < hi; ++n)
        st4(d.grad_x_src + (size_t)n * kRow + toff,
            has_init ? ldg4(d.grad_x_src_init + (size_t)n * kRow + toff) : make_float4(0.f, 0.f, 0.f, 0.f));
    };
    const int rj = row >> 4, ro = row & 15;

    for (int t = 0; t < n_tiles; ++t) {
      const int slot = t & 3, b = t & 1;
      const uint32_t par = (uint32_t)t & 1u, parb = (uint32_t)(t >> 1) & 1u;
      const int cnt = min(kTE, p1 - (p0 + t * kTE));
      const bool acc = t > 0;
      const uint32_t bz = tc::smem_u32(s.BZ[b]);
      const uint32_t ga = tc::smem_u32(s.G[b]), xa = ga - kTM * kC * 2;  // xa: the 16 KB in front of G[b]
      __nv_bfloat16* G = s.G[b];
      if (t >= 2) {  // G[b] was last read by the [gW1 | gb1] MMA of tile t-2
        tc::mbar_wait(&s.empty[b], parb ^ 1u);
        tc::tc_fence_after();
      }
      tc::mbar_wait(&s.full[b], parb);  // role R has finished set b
      tc::tc_fence_after();
      if (rt == 0) {  // kern = basis Wk^T  (the kern columns are free: every C1 thread passed barrier (E) of tile t-1)
        tc::issue_mma(tmem + kKern, tc::view_k(bz, kTM), tc::view_k(wk, kC), tc::idesc_bf16(128, kC), kC / 16, false);
        tc::mma_commit(&s.bar_c[0]);
      }
      tc::mbar_wait(&s.bar_g, par);  // the producer's rows have landed; its ring slot is visible
      tc::mbar_wait(&s.bar_c[0], par);
      tc::tc_fence_after();
      {
        float* gxb = s.GX + (((rj * 2 + ch) * kO + ro) << 5);
        const float* xsb = s.XS + (((s.lead[slot][rj] * 2 + ch) * kO + ro) << 5);
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int c0 = 32 * ch + 16 * i;
          float v[16], gkv[16];
          tc::tmem_ld16(lane_addr + kKern + c0, v);
#pragma unroll
          for (int e4 = 0; e4 < 4; ++e4) {
            const int off = ((4 * i + e4) ^ (ro & 7)) << 2;
            const float4 gm = ld4(gxb + off), x = ld4(xsb + off);
            const int e = 4 * e4;
            st4(gxb + off, make_float4(gm.x * v[e], gm.y * v[e + 1], gm.z * v[e + 2], gm.w * v[e + 3]));
            gkv[e] = gm.x * x.x; gkv[e + 1] = gm.y * x.y; gkv[e + 2] = gm.z * x.z; gkv[e + 3] = gm.w * x.w;
          }
          *reinterpret_cast<uint4*>(G + ((size_t)(c0 >> 3) * kTM + row) * 8) = tc::pack8(gkv);
          *reinterpret_cast<uint4*>(G + ((size_t)((c0 >> 3) + 1) * kTM + row) * 8) = tc::pack8(gkv + 8);
        }
      }
      tc::fence_async_smem();
      tc::mbar_arrive(&s.xs_free);  // this thread is done with the x_src tile
      tc::tc_fence_before();
      tc::group_sync(2, 256);  // (E)
      if (rt == 0) {
        if (t > 0) tc::mbar_wait(&s.b2_free, (uint32_t)(t - 1) & 1u);  // role C2 has read gH1 of tile t-1
        tc::tc_fence_after();
        // g_basis = g_kern Wk (Wk image read MN-major: K = c, N = j)
        tc::issue_mma(tmem + kGB, tc::view_k(ga, kTM), tc::view_mn(wk, kC), tc::idesc_bf16_ex(128, 64, 0, 1), kC / 16, false);
        // lanes 64..127: gWk[c][j] += sum_rows g_kern[row][c] basis[row][j]   ([X | G] as one 128-column image)
        tc::issue_mma(tmem + kGWk, tc::view_mn(xa, kTM), tc::view_mn(bz, kTM), tc::idesc_bf16_ex(128, 64, 1, 1), kTM / 16, acc);
        tc::mma_commit(&s.bar_c[1]);  // role C2 takes over from here
      }
      // src-CSR segmented sum of g_x1 * kern.  Everything a step needs is in registers before the chain starts: the run
      // flags (producer), the messages and the residual rows of the runs that start in this tile (IN tile, shared memory)
      {
        const int4 a_lo = *reinterpret_cast<const int4*>(&s.adv[slot][0]), a_hi = *reinterpret_cast<const int4*>(&s.adv[slot][4]);
        const int adv[kTE] = {a_lo.x, a_lo.y, a_lo.z, a_lo.w, a_hi.x, a_hi.y, a_hi.z, a_hi.w};
        float4 m[kTE];
#pragma unroll
        for (int j = 0; j < kTE; ++j) m[j] = ld4(s.GX + swz_off(j, cg >> 3, o, cg & 7));
#pragma unroll
        for (int j = 0; j < kTE; ++j) {
          if (adv[j] > 0) {  // warp-uniform: node `cur` is complete (adv is 0 past the end of the list)
            st4(d.grad_x_src + (size_t)cur * kRow + toff,
                make_float4(sum.x + init.x, sum.y + init.y, sum.z + init.z, sum.w + init.w));
            if (adv[j] > 1) fill_gap(cur + 1, cur + adv[j]);
            cur += adv[j];
            sum = make_float4(0.f, 0.f, 0.f, 0.f);
            init = has_init ? ld4(s.IN + swz_off(j, cg >> 3, o, cg & 7)) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
          sum.x += m[j].x; sum.y += m[j].y; sum.z += m[j].z; sum.w += m[j].w;
        }
      }
      tc::fence_async_smem();
      tc::mbar_arrive(&s.gx_free);  // ... and with the g_x1 / residual tiles
    }
    if (cur < n_hi) {  // the last node of the range and the edge-less nodes behind it
      st4(d.grad_x_src + (size_t)cur * kRow + toff, make_float4(sum.x + init.x, sum.y + init.y, sum.z + init.z, sum.w + init.w));
      fill_gap(cur + 1, n_hi);
    }
  } else {
    // =========================================== role C2 ==========================================================
    for (int t = 0; t < n_tiles; ++t) {
      const int b = t & 1;
      const uint32_t par = (uint32_t)t & 1u, parb = (uint32_t)(t >> 1) & 1u;
      const bool acc = t > 0;
      const uint32_t fa = tc::smem_u32(s.F[b]), ha = tc::smem_u32(s.H1[b]);
      const uint32_t ga = tc::smem_u32(s.G[b]), xa = ga - kTM * kC * 2;
      __nv_bfloat16* G = s.G[b];
      const uint32_t kSet = 64u + 64u * b;
      tc::mbar_wait(&s.full[b], parb);      // the derivative planes of set b are in TMEM
      tc::mbar_wait(&s.bar_c[1], par);      // g_basis is complete (and the MMAs that read g_kern from G[b] are done)
      tc::tc_fence_after();
      {
        const int h = ch;  // this warp's 32 columns
        uint32_t dpk[16];
        tc::tmem_ld16_raw(lane_addr + kSet + 32 + 16 * h, dpk);  // GELU'(pre2), columns 32 h .. 32 h + 31
        float gp2[32];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int c0 = 32 * h + 16 * i;
          float v[16];
          tc::tmem_ld16(lane_addr + kGB + c0, v);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float2 dg = __half22float2(*reinterpret_cast<const __half2*>(&dpk[8 * i + e]));
            gp2[16 * i + 2 * e] = v[2 * e] * dg.x;
            gp2[16 * i + 2 * e + 1] = v[2 * e + 1] * dg.y;
          }
          *reinterpret_cast<uint4*>(G + ((size_t)(c0 >> 3) * kTM + row) * 8) = tc::pack8(gp2 + 16 * i);
          *reinterpret_cast<uint4*>(G + ((size_t)((c0 >> 3) + 1) * kTM + row) * 8) = tc::pack8(gp2 + 16 * i + 8);
        }
        tc::warp_colsum<32>(gp2, lane);
        s.acc_gb2[q][32 * h + lane] += gp2[0];
      }
      tc::fence_async_smem();
      tc::tc_fence_before();
      tc::group_sync(3, 256);  // (F)
      if (rt == 0) {
        tc::tc_fence_after();
        // gH1 = gP2 W2 (W2 image read MN-major: K = n, N = k) over the g_basis columns
        tc::issue_mma(tmem + kGB, tc::view_k(ga, kTM), tc::view_mn(w2, kC), tc::idesc_bf16_ex(128, 64, 0, 1), kC / 16, false);
        // lanes 64..127: gW2[n][k] += sum_rows gP2[row][n] H1[row][k]
        tc::issue_mma(tmem + kGW2, tc::view_mn(xa, kTM), tc::view_mn(ha, kTM), tc::idesc_bf16_ex(128, 64, 1, 1), kTM / 16, acc);
        tc::mma_commit(&s.bar_c[2]);
      }
      tc::mbar_wait(&s.bar_c[2], par);
      tc::tc_fence_after();
      {
        const int h = ch;
        uint32_t dpk[16];
        tc::tmem_ld16_raw(lane_addr + kSet + 16 * h, dpk);  // GELU'(pre1)
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int c0 = 32 * h + 16 * i;
          float v[16];
          tc::tmem_ld16(lane_addr + kGB + c0, v);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float2 dg = __half22float2(*reinterpret_cast<const __half2*>(&dpk[8 * i + e]));
            v[2 * e] *= dg.x;
            v[2 * e + 1] *= dg.y;
          }
          *reinterpret_cast<uint4*>(G + ((size_t)(c0 >> 3) * kTM + row) * 8) = tc::pack8(v);
          *reinterpret_cast<uint4*>(G + ((size_t)((c0 >> 3) + 1) * kTM + row) * 8) = tc::pack8(v + 8);
        }
      }
      tc::fence_async_smem();
      tc::tc_fence_before();
      tc::group_sync(3, 256);  // (G)
      if (rt == 0) {
        tc::mbar_arrive(&s.b2_free);  // every C2 thread has read gH1: role C1 may issue the next g_basis MMA
        tc::tc_fence_after();
        // [gW1 | gb1] += gP1^T [F | 1 1]; its completion frees operand set b (role R) and G[b] (role C1, tile t+2)
        tc::issue_mma(tmem + kGW1, tc::view_mn(xa, kTM), tc::view_mn(fa, kTM), tc::idesc_bf16_ex(128, 16, 1, 1), kTM / 16, acc);
        tc::mma_commit(&s.empty[b]);
      }
    }
    for (int t = max(0, n_tiles - 2); t < n_tiles; ++t) {  // the last MMAs on both operand sets
      tc::mbar_wait(&s.empty[t & 1], (uint32_t)(t >> 1) & 1u);
    }
    tc::tc_fence_after();
  }
  // partial slot of this CTA: gWk[64][64] | gW1b[64][16] (columns 14, 15 = gb1) | gW2[64][64] | gb2[64]
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  float* P = d.grad_partials + (size_t)blockIdx.x * GRL_FUSED_EDGE_GRAD_FLOATS;
  if (warp < 16) {
    const int q4 = warp & 3, cq = warp >> 2, row4 = 32 * q4 + lane, c0 = 16 * cq;  // 16 warps: 16 columns per thread
    const uint32_t la = tmem + ((uint32_t)(32 * q4) << 16);
    float v[16];
    auto read = [&](uint32_t col) {
      if (n_tiles > 0) {
        tc::tmem_ld16(la + col, v);
      } else {
#pragma unroll
        for (int e = 0; e < 16; ++e) v[e] = 0.f;
      }
    };
    read(kGWk + c0);
    if (row4 >= 64) {
      float* p = P + (size_t)(row4 - 64) * kC + c0;
#pragma unroll
      for (int e = 0; e < 16; e += 4) st4(p + e, make_float4(v[e], v[e + 1], v[e + 2], v[e + 3]));
    }
    read(kGW2 + c0);
    if (row4 >= 64) {
      float* p = P + kWFloats + 64 * 16 + (size_t)(row4 - 64) * kC + c0;
#pragma unroll
      for (int e = 0; e < 16; e += 4) st4(p + e, make_float4(v[e], v[e + 1], v[e + 2], v[e + 3]));
    }
    read(kGW1);
    if (row4 >= 64 && cq == 0) {
      float* p = P + kWFloats + (size_t)(row4 - 64) * 16;
#pragma unroll
      for (int e = 0; e < 16; e += 4) st4(p + e, make_float4(v[e], v[e + 1], v[e + 2], v[e + 3]));
    }
  }
  if (tid < kC)
    P[2 * kWFloats + 64 * 16 + tid] = ((s.acc_gb2[0][tid] + s.acc_gb2[1][tid]) + s.acc_gb2[2][tid]) + s.acc_gb2[3][tid];
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 0) tc::tmem_dealloc(tmem, 512);
}

}  // namespace grl

extern "C" {

static int fused_check(const GrlFusedEdgeDesc* d, const char* what) {
  GRL_REQUIRE(d, GRL_EINVAL, "%s: null descriptor", what);
  GRL_REQUIRE(d->n_key > 0 && d->n_edges >= 0 && (d->dim == 2 || d->dim == 3), GRL_EINVAL, "%s: n_key=%d n_edges=%d dim=%d",
              what, d->n_key, d->n_edges, d->dim);
  GRL_REQUIRE(d->rowptr && d->pos_src && d->pos_dst && d->ori && d->w1 && d->b1 && d->w2 && d->b2 && d->wk && d->x_src &&
                  (d->n_edges == 0 || (d->e_src && d->e_dst)), GRL_EINVAL, "%s: null pointer", what);
  return GRL_OK;
}

int grl_fbconv_edge_fused_fwd(const GrlFusedEdgeDesc* d, grl_stream_t stream) {
  const int rc = fused_check(d, "grl_fbconv_edge_fused_fwd");
  if (rc != GRL_OK) return rc;
  GRL_REQUIRE(d->x1, GRL_EINVAL, "grl_fbconv_edge_fused_fwd: x1 is null");
  GRL_REQUIRE(d->n_other > 0, GRL_EINVAL, "grl_fbconv_edge_fused_fwd: n_other=%d (rows of x_src) must be set", d->n_other);
  alignas(64) CUtensorMap tm_xs;
  if (grl::make_row_tensor_map(&tm_xs, d->x_src, d->n_other) != GRL_OK) return GRL_ECUDA;
  const int smem = (int)sizeof(grl::FusedFwdSmem) + 1024;
  if (grl::ensure_dynamic_smem((const void*)grl::edge_fused_fwd_kernel, smem) != GRL_OK) return GRL_ECUDA;
  int grid = 3 * grl::sm_count();
  if (grid > d->n_key) grid = d->n_key;
  grl::edge_fused_fwd_kernel<<<grid, grl::kThreads, smem, (cudaStream_t)stream>>>(*d, tm_xs);
  return grl::check_launch("grl_fbconv_edge_fused_fwd");
}

int grl_fbconv_edge_fused_bwd(const GrlFusedEdgeDesc* d, grl_stream_t stream) {
  const int rc = fused_check(d, "grl_fbconv_edge_fused_bwd");
  if (rc != GRL_OK) return rc;
  GRL_REQUIRE(d->grad_x1 && d->grad_x_src && d->grad_partials, GRL_EINVAL, "grl_fbconv_edge_fused_bwd: null pointer");
  GRL_REQUIRE(d->n_partials > 0 && d->n_partials <= d->n_key, GRL_EINVAL,
              "grl_fbconv_edge_fused_bwd: n_partials=%d must be in [1, n_key]", d->n_partials);
  GRL_REQUIRE(d->n_other > 0, GRL_EINVAL, "grl_fbconv_edge_fused_bwd: n_other=%d (rows of grad_x1) must be set", d->n_other);
  alignas(64) CUtensorMap tm_gx, tm_xs, tm_in;
  if (grl::make_row_tensor_map(&tm_gx, d->grad_x1, d->n_other) != GRL_OK) return GRL_ECUDA;
  if (grl::make_row_tensor_map(&tm_xs, d->x_src, d->n_key) != GRL_OK) return GRL_ECUDA;
  // residual rows (optional): an unused map over x_src keeps the kernel signature fixed when there are none
  if (grl::make_row_tensor_map(&tm_in, d->grad_x_src_init ? d->grad_x_src_init : d->x_src, d->n_key) != GRL_OK) return GRL_ECUDA;
  const int smem = (int)sizeof(grl::FusedBwdWs3Smem) + 1024;
  if (grl::ensure_dynamic_smem((const void*)grl::edge_fused_bwd_ws3_kernel, smem) != GRL_OK) return GRL_ECUDA;
  grl::edge_fused_bwd_ws3_kernel<<<d->n_partials, grl::kWs3Threads, smem, (cudaStream_t)stream>>>(*d, tm_gx, tm_xs, tm_in);
  return grl::check_launch("grl_fbconv_edge_fused_bwd");
}

}  // extern "C"
