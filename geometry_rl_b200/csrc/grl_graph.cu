// K1: batched edge construction (kNN / radius / dense) and stable CSR build.
// Replaces the per-graph Python loop of geometry_rl/modules/pyg_data/rigid_tasks_data.py:275-321
// (torch_geometric.nn.knn_graph per graph, nested loops for AGENT / TASK edges, coalesce()) and
// rope_tasks_data.py:238-278, cloth_tasks_data.py:236-286; plus the graph-major batching of
// Batch.from_data_list (rigid_tasks_data.py:324).  One CTA per graph; graphs have <= a few hundred
// nodes, so everything is brute force in shared memory.  Integer outputs are bit-exact by construction.
#include <algorithm>

#include "grl_common.cuh"

namespace grl {

constexpr int kMaxP = 512;  // points per graph held in shared memory

__device__ __forceinline__ int valid_points(const int32_t* num_valid, int b, int P) {
  if (!num_valid) return P;
  const int v = num_valid[b];
  return v < 0 ? 0 : (v > P ? P : v);
}

// count[b] = P_b * min(k, P_b - 1); edge_ptr = exclusive prefix sum (single CTA, sequential chunks).
__global__ void knn_edge_ptr_kernel(const int32_t* __restrict__ num_valid, int B, int P, int k, int64_t* __restrict__ edge_ptr) {
  __shared__ long long part[1024];
  const int tid = threadIdx.x, nt = blockDim.x;
  const int per = (B + nt - 1) / nt;
  const int b0 = tid * per, b1 = min(b0 + per, B);
  long long s = 0;
  for (int b = b0; b < b1; ++b) {
    const int pv = valid_points(num_valid, b, P);
    s += (long long)pv * max(0, min(k, pv - 1));
  }
  part[tid] = s;
  __syncthreads();
  if (tid == 0) {
    long long run = 0;
    for (int i = 0; i < nt; ++i) { const long long t = part[i]; part[i] = run; run += t; }
    edge_ptr[B] = run;
  }
  __syncthreads();
  long long run = part[tid];
  for (int b = b0; b < b1; ++b) {
    edge_ptr[b] = run;
    const int pv = valid_points(num_valid, b, P);
    run += (long long)pv * max(0, min(k, pv - 1));
  }
}

// squared distance with the oracle's exact rounding sequence: (dx*dx + dy*dy) + dz*dz, no FMA contraction
__device__ __forceinline__ float sqdist(const float* a, const float* b) {
  const float dx = __fsub_rn(a[0], b[0]), dy = __fsub_rn(a[1], b[1]), dz = __fsub_rn(a[2], b[2]);
  return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

__global__ void __launch_bounds__(128) knn_graph_kernel(const float* __restrict__ pos, const int32_t* __restrict__ num_valid,
                                                       const int64_t* __restrict__ edge_ptr, int B, int P, int k,
                                                       int64_t* __restrict__ coo, int64_t row_stride) {
  __shared__ float sp[kMaxP * 3];
  __shared__ short nbr[kMaxP * GRL_MAX_KNN];
  __shared__ int off[kMaxP + 1];
  const int tid = threadIdx.x;
  for (int g = blockIdx.x; g < B; g += gridDim.x) {
    const int pv = valid_points(num_valid, g, P);
    const int kk = max(0, min(k, pv - 1));
    __syncthreads();
    for (int i = tid; i < pv * 3; i += blockDim.x) sp[i] = pos[(size_t)g * P * 3 + i];
    __syncthreads();
    // k nearest of every centre i (self excluded); ascending distance, ties -> lower index
    for (int i = tid; i < pv; i += blockDim.x) {
      float bd[GRL_MAX_KNN];
      int bj[GRL_MAX_KNN];
#pragma unroll
      for (int s = 0; s < GRL_MAX_KNN; ++s) { bd[s] = __int_as_float(0x7f800000); bj[s] = -1; }
      for (int j = 0; j < pv; ++j) {
        if (j == i) continue;
        const float dd = sqdist(sp + 3 * i, sp + 3 * j);
        if (kk > 0 && dd < bd[kk - 1]) {
          int s = kk - 1;
#pragma unroll
          for (int u = GRL_MAX_KNN - 1; u > 0; --u) {
            if (u <= s && bd[u - 1] > dd) { bd[u] = bd[u - 1]; bj[u] = bj[u - 1]; s = u - 1; }
          }
          bd[s] = dd; bj[s] = j;
        }
      }
#pragma unroll
      for (int s = 0; s < GRL_MAX_KNN; ++s) if (s < kk) nbr[i * GRL_MAX_KNN + s] = (short)bj[s];
    }
    __syncthreads();
    // coalesced COO: sorted by (source = neighbour j, target = centre i)
    for (int j = tid; j < pv; j += blockDim.x) {
      int c = 0;
      for (int i = 0; i < pv; ++i)
        for (int s = 0; s < kk; ++s) c += (nbr[i * GRL_MAX_KNN + s] == j);
      off[j + 1] = c;
    }
    __syncthreads();
    if (tid == 0) {
      off[0] = 0;
      for (int j = 0; j < pv; ++j) off[j + 1] += off[j];
    }
    __syncthreads();
    const int64_t base = edge_ptr[g];
    for (int j = tid; j < pv; j += blockDim.x) {
      int64_t w = base + off[j];
      for (int i = 0; i < pv; ++i) {
        bool hit = false;
        for (int s = 0; s < kk; ++s) hit |= (nbr[i * GRL_MAX_KNN + s] == j);
        if (hit) {
          coo[w] = (int64_t)g * P + j;
          coo[row_stride + w] = (int64_t)g * P + i;
          ++w;
        }
      }
    }
  }
}

// Rank key of a squared distance: a sum of squares is +0, positive, +inf or NaN, and the bits of a non-negative float
// order like the float.  NaN ranks as +inf, so the order (key, index) is total whatever the positions hold.
__device__ __forceinline__ uint32_t dist_key(float d) { return d != d ? 0x7f800000u : __float_as_uint(d); }

// The kk nearest neighbours of every valid centre of graph g (self excluded), ranked by (dist_key, index), written to
// nbr[i * GRL_MAX_KNN + s], s < kk, in ascending INDEX order.  Every centre gets exactly kk neighbours; for finite
// distances the set is the one knn_graph_kernel picks.  Ends with a block barrier.
__device__ void knn_sorted_lists(const float* __restrict__ pos, int g, int P, int pv, int kk, float* sp, short* nbr) {
  const int tid = threadIdx.x;
  for (int i = tid; i < pv * 3; i += blockDim.x) sp[i] = pos[(size_t)g * P * 3 + i];
  __syncthreads();
  for (int i = tid; i < pv; i += blockDim.x) {
    uint32_t bk[GRL_MAX_KNN];
    int bj[GRL_MAX_KNN];
#pragma unroll
    for (int s = 0; s < GRL_MAX_KNN; ++s) { bk[s] = 0xffffffffu; bj[s] = 0x7fffffff; }  // empty: after every candidate
    uint32_t worst = 0xffffffffu;  // bk[kk - 1]
    for (int j = 0; j < pv; ++j) {
      if (j == i) continue;
      const uint32_t key = dist_key(sqdist(sp + 3 * i, sp + 3 * j));
      if (key >= worst) continue;  // a tie keeps the lower index, which came first
#pragma unroll
      for (int u = GRL_MAX_KNN - 1; u >= 0; --u) {
        if (u >= kk) continue;
        if (u > 0 && bk[u - 1] > key) { bk[u] = bk[u - 1]; bj[u] = bj[u - 1]; }
        else if (bk[u] > key) { bk[u] = key; bj[u] = j; }
      }
#pragma unroll
      for (int s = 0; s < GRL_MAX_KNN; ++s) if (s == kk - 1) worst = bk[s];
    }
    // ascending index (odd-even transposition; the empty slots past kk sort last)
#pragma unroll
    for (int r = 0; r < GRL_MAX_KNN; ++r) {
#pragma unroll
      for (int s = r & 1; s + 1 < GRL_MAX_KNN; s += 2) {
        const int a = bj[s], b = bj[s + 1];
        bj[s] = min(a, b);
        bj[s + 1] = max(a, b);
      }
    }
#pragma unroll
    for (int s = 0; s < GRL_MAX_KNN; ++s) if (s < kk) nbr[i * GRL_MAX_KNN + s] = (short)bj[s];
  }
  __syncthreads();
}

struct KnnTopoOut {
  int64_t* coo;
  int64_t row_stride;
  int32_t *rowptr_dst, *edge_src, *edge_dst, *eid_coo, *rowptr_src, *src_eid, *s_src, *s_dst;
};

// Every layout of the kNN edge set in one pass (see grl_knn_topology).  CTAs [0, n_graph_ctas) own the graphs; the
// others write the tail [edge_ptr[B], capacity).
__global__ void __launch_bounds__(128) knn_topology_kernel(const float* __restrict__ pos,
                                                          const int32_t* __restrict__ num_valid,
                                                          const int64_t* __restrict__ edge_ptr, int B, int P, int k,
                                                          int64_t capacity, int n_graph_ctas, KnnTopoOut o) {
  __shared__ float sp[kMaxP * 3];
  __shared__ short nbr[kMaxP * GRL_MAX_KNN];
  __shared__ int cnt[kMaxP];
  __shared__ int off[kMaxP + 1];
  __shared__ int first_edge;
  const int tid = threadIdx.x;
  if ((int)blockIdx.x < n_graph_ctas) {
    for (int g = blockIdx.x; g < B; g += n_graph_ctas) {
      const int pv = valid_points(num_valid, g, P);
      const int kk = max(0, min(k, pv - 1));
      __syncthreads();  // the previous graph's shared arrays are no longer read
      for (int j = tid; j < pv; j += blockDim.x) cnt[j] = 0;
      knn_sorted_lists(pos, g, P, pv, kk, sp, nbr);
      for (int q = tid; q < pv * kk; q += blockDim.x) atomicAdd(&cnt[nbr[(q / kk) * GRL_MAX_KNN + q % kk]], 1);
      __syncthreads();
      if (tid < 32) {  // off = exclusive prefix sum of cnt (off[j] = edges of the neighbours before j)
        int carry = 0;
        for (int b = 0; b < pv; b += 32) {
          const int j = b + tid;
          int v = j < pv ? cnt[j] : 0;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, v, d);
            if (tid >= d) v += t;
          }
          if (j < pv) off[j + 1] = carry + v;
          carry += __shfl_sync(0xffffffffu, v, 31);
        }
        if (tid == 0) off[0] = 0;
      }
      __syncthreads();
      const int64_t e0 = edge_ptr[g], e1 = edge_ptr[g + 1];
      const int64_t node0 = (int64_t)g * P;
      // edge order = dst-sorted CSR: centre i, then its neighbours ascending
      for (int i = tid; i < P; i += blockDim.x) {
        if (i >= pv) {
          o.rowptr_dst[node0 + i] = (int32_t)e1;
          continue;
        }
        const int64_t e = e0 + (int64_t)i * kk;
        o.rowptr_dst[node0 + i] = (int32_t)e;
        for (int s = 0; s < kk; ++s) {
          o.edge_src[e + s] = (int32_t)(node0 + nbr[i * GRL_MAX_KNN + s]);
          o.edge_dst[e + s] = (int32_t)(node0 + i);
        }
      }
      // COO order = src-sorted CSR: neighbour j, then the centres that chose it ascending
      for (int j = tid; j < P; j += blockDim.x) {
        if (j >= pv) {
          o.rowptr_src[node0 + j] = (int32_t)e1;
          continue;
        }
        int64_t w = e0 + off[j];
        const int64_t w1 = e0 + off[j + 1];
        o.rowptr_src[node0 + j] = (int32_t)w;
        for (int i = 0; i < pv && w < w1; ++i) {
          for (int s = 0; s < kk; ++s) {
            if (nbr[i * GRL_MAX_KNN + s] != j) continue;
            const int64_t e = e0 + (int64_t)i * kk + s;
            o.coo[w] = node0 + j;
            o.coo[o.row_stride + w] = node0 + i;
            o.eid_coo[e] = (int32_t)w;
            o.src_eid[w] = (int32_t)e;
            if (o.s_src) {
              o.s_src[w] = (int32_t)(node0 + j);
              o.s_dst[w] = (int32_t)(node0 + i);
            }
            ++w;
            break;  // a centre lists j at most once
          }
        }
      }
      if (g == B - 1 && tid == 0) {
        o.rowptr_dst[(size_t)B * P] = (int32_t)e1;
        o.rowptr_src[(size_t)B * P] = (int32_t)e1;
      }
    }
    return;
  }
  // Tail: coo, edge_src, eid_coo and src_eid hold 0; edge_dst, s_src and s_dst hold what a gather through those zeros
  // reads: coo[1][0], edge_src[0] and edge_dst[0].  They come from the first graph with edges, g0, whose kNN lists this
  // CTA recomputes: edge 0 of the edge order is (nbr[0][0] -> centre 0), and COO entry 0 is the smallest (j, i).
  const int64_t e_end = edge_ptr[B];
  if (e_end >= capacity) return;
  int v_dst = 0, v_ssrc = 0, v_sdst = 0;
  if (e_end > 0) {
    int lo = 0, hi = B - 1;  // smallest g with edge_ptr[g + 1] > 0 (edge_ptr is non-decreasing and edge_ptr[0] = 0)
    while (lo < hi) {
      const int mid = (lo + hi) / 2;
      if (edge_ptr[mid + 1] > 0) hi = mid; else lo = mid + 1;
    }
    const int g0 = lo, pv = valid_points(num_valid, g0, P), kk = max(0, min(k, pv - 1));
    if (tid == 0) first_edge = 0x7fffffff;
    knn_sorted_lists(pos, g0, P, pv, kk, sp, nbr);
    for (int i = tid; i < pv; i += blockDim.x) atomicMin(&first_edge, nbr[i * GRL_MAX_KNN] * kMaxP + i);
    __syncthreads();
    v_dst = (int)((int64_t)g0 * P + first_edge % kMaxP);
    v_ssrc = (int)((int64_t)g0 * P + nbr[0]);
    v_sdst = (int)((int64_t)g0 * P);
  }
  const int64_t n_tail = gridDim.x - n_graph_ctas;
  for (int64_t e = e_end + (int64_t)(blockIdx.x - n_graph_ctas) * blockDim.x + tid; e < capacity;
       e += n_tail * blockDim.x) {
    o.coo[e] = 0;
    o.coo[o.row_stride + e] = 0;
    o.edge_src[e] = 0;
    o.eid_coo[e] = 0;
    o.src_eid[e] = 0;
    o.edge_dst[e] = v_dst;
    if (o.s_src) {
      o.s_src[e] = v_ssrc;
      o.s_dst[e] = v_sdst;
    }
  }
}

__global__ void __launch_bounds__(128) radius_neighbors_kernel(const float* __restrict__ pos, const int32_t* __restrict__ num_valid,
                                                              int B, int P, float r2, int max_nb, int32_t* __restrict__ nbr,
                                                              int32_t* __restrict__ cnt) {
  __shared__ float sp[kMaxP * 3];
  const int tid = threadIdx.x;
  for (int g = blockIdx.x; g < B; g += gridDim.x) {
    const int pv = valid_points(num_valid, g, P);
    __syncthreads();
    for (int i = tid; i < pv * 3; i += blockDim.x) sp[i] = pos[(size_t)g * P * 3 + i];
    __syncthreads();
    for (int i = tid; i < P; i += blockDim.x) {
      float bd[GRL_MAX_KNN];
      int bj[GRL_MAX_KNN];
      int n = 0;
#pragma unroll
      for (int s = 0; s < GRL_MAX_KNN; ++s) { bd[s] = __int_as_float(0x7f800000); bj[s] = -1; }
      if (i < pv) {
        for (int j = 0; j < pv; ++j) {
          if (j == i) continue;
          const float dd = sqdist(sp + 3 * i, sp + 3 * j);
          if (dd <= r2 && dd < bd[max_nb - 1]) {
            int s = max_nb - 1;
#pragma unroll
            for (int u = GRL_MAX_KNN - 1; u > 0; --u) {
              if (u <= s && bd[u - 1] > dd) { bd[u] = bd[u - 1]; bj[u] = bj[u - 1]; s = u - 1; }
            }
            bd[s] = dd; bj[s] = j;
            if (n < max_nb) ++n;
          }
        }
      }
      for (int s = 0; s < max_nb; ++s) nbr[((size_t)g * P + i) * max_nb + s] = (s < n) ? bj[s] : -1;
      cnt[(size_t)g * P + i] = n;
    }
  }
}

// edge_ptr of a radius graph: count[b] = sum of cnt over graph b's P rows (rows past num_valid[b] hold 0), exclusive
// prefix sum, every entry clamped to `capacity` (the edges of the COO buffer; the last graphs lose what does not fit).
__global__ void radius_edge_ptr_kernel(const int32_t* __restrict__ cnt, int B, int P, int64_t capacity,
                                       int64_t* __restrict__ edge_ptr) {
  __shared__ long long part[1024];
  const int tid = threadIdx.x, nt = blockDim.x;
  const int per = (B + nt - 1) / nt;
  const int b0 = tid * per, b1 = min(b0 + per, B);
  long long s = 0;
  for (int b = b0; b < b1; ++b)
    for (int i = 0; i < P; ++i) s += cnt[(size_t)b * P + i];
  part[tid] = s;
  __syncthreads();
  if (tid == 0) {
    long long run = 0;
    for (int i = 0; i < nt; ++i) { const long long t = part[i]; part[i] = run; run += t; }
    edge_ptr[B] = min(run, (long long)capacity);
  }
  __syncthreads();
  long long run = part[tid];
  for (int b = b0; b < b1; ++b) {
    edge_ptr[b] = min(run, (long long)capacity);
    for (int i = 0; i < P; ++i) run += cnt[(size_t)b * P + i];
  }
}

// Coalesced COO of a radius graph from the padded neighbour lists of radius_neighbors_kernel: per graph, sorted by
// (source = neighbour j, target = centre i), like knn_graph_kernel.  Entries [edge_ptr[B], capacity) are set to 0, so
// a gather over the whole buffer stays in bounds.
__global__ void __launch_bounds__(128) radius_graph_kernel(const int32_t* __restrict__ nbr, const int32_t* __restrict__ cnt,
                                                          const int64_t* __restrict__ edge_ptr, int B, int P, int max_nb,
                                                          int64_t* __restrict__ coo, int64_t row_stride, int64_t capacity) {
  __shared__ short snb[kMaxP * GRL_MAX_KNN];
  __shared__ int off[kMaxP + 1];
  const int tid = threadIdx.x;
  for (int g = blockIdx.x; g < B; g += gridDim.x) {
    __syncthreads();
    for (int q = tid; q < P * max_nb; q += blockDim.x) {
      const int i = q / max_nb, s = q - i * max_nb;
      snb[q] = (short)(s < cnt[(size_t)g * P + i] ? nbr[(size_t)g * P * max_nb + q] : -1);
    }
    __syncthreads();
    for (int j = tid; j < P; j += blockDim.x) {
      int c = 0;
      for (int q = 0; q < P * max_nb; ++q) c += (snb[q] == j);
      off[j + 1] = c;
    }
    __syncthreads();
    if (tid == 0) {
      off[0] = 0;
      for (int j = 0; j < P; ++j) off[j + 1] += off[j];
    }
    __syncthreads();
    const int64_t base = edge_ptr[g], end = edge_ptr[g + 1];
    for (int j = tid; j < P; j += blockDim.x) {
      int64_t w = base + off[j];
      for (int i = 0; i < P && w < end; ++i) {
        bool hit = false;
        for (int s = 0; s < max_nb; ++s) hit |= (snb[i * max_nb + s] == j);
        if (hit) {
          coo[w] = (int64_t)g * P + j;
          coo[row_stride + w] = (int64_t)g * P + i;
          ++w;
        }
      }
    }
  }
  for (int64_t e = edge_ptr[B] + (int64_t)blockIdx.x * blockDim.x + tid; e < capacity; e += (int64_t)gridDim.x * blockDim.x) {
    coo[e] = 0;
    coo[row_stride + e] = 0;
  }
}

__global__ void __launch_bounds__(128) dense_edges_kernel(int mode, const int32_t* __restrict__ num_valid,
                                                         const int64_t* __restrict__ edge_ptr, int B, int n_src, int n_dst,
                                                         int64_t* __restrict__ coo, int64_t row_stride) {
  for (int g = blockIdx.x; g < B; g += gridDim.x) {
    const int64_t base = edge_ptr[g];
    const int n = (int)(edge_ptr[g + 1] - base);
    for (int e = threadIdx.x; e < n; e += blockDim.x) {
      int j, k;
      if (mode == 0) {  // ordered pairs j != k
        j = e / (n_src - 1);
        const int r = e % (n_src - 1);
        k = r < j ? r : r + 1;
        coo[base + e] = (int64_t)g * n_src + j;
        coo[row_stride + base + e] = (int64_t)g * n_src + k;
      } else {  // every valid source -> every destination
        j = e / n_dst;
        k = e % n_dst;
        coo[base + e] = (int64_t)g * n_src + j;
        coo[row_stride + base + e] = (int64_t)g * n_dst + k;
      }
    }
  }
}

// Stable counting sort of graph g's edges by key node; one thread per key node walks the graph's
// edge list in input order (<= a few hundred edges), so equal keys keep their relative order.
__global__ void __launch_bounds__(128) csr_build_kernel(const int64_t* __restrict__ coo, int64_t row_stride,
                                                       const int64_t* __restrict__ edge_ptr, int B, int n_key, int key_row,
                                                       int32_t* __restrict__ rowptr, int32_t* __restrict__ other,
                                                       int32_t* __restrict__ eid) {
  extern __shared__ int deg[];  // [n_key + 1]
  const int64_t* keys = coo + (key_row ? row_stride : 0);
  const int64_t* oth = coo + (key_row ? 0 : row_stride);
  for (int g = blockIdx.x; g < B; g += gridDim.x) {
    const int64_t e0 = edge_ptr[g], e1 = edge_ptr[g + 1];
    __syncthreads();
    for (int d = threadIdx.x; d < n_key; d += blockDim.x) {
      const int64_t key = (int64_t)g * n_key + d;
      int c = 0;
      for (int64_t e = e0; e < e1; ++e) c += (keys[e] == key);
      deg[d + 1] = c;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      deg[0] = 0;
      for (int d = 0; d < n_key; ++d) deg[d + 1] += deg[d];
    }
    __syncthreads();
    for (int d = threadIdx.x; d < n_key; d += blockDim.x) {
      const int64_t key = (int64_t)g * n_key + d;
      int64_t w = e0 + deg[d];
      rowptr[(size_t)g * n_key + d] = (int32_t)w;
      for (int64_t e = e0; e < e1; ++e) {
        if (keys[e] == key) {
          other[w] = (int32_t)oth[e];
          eid[w] = (int32_t)e;
          ++w;
        }
      }
    }
    if (g == B - 1 && threadIdx.x == 0) rowptr[(size_t)B * n_key] = (int32_t)e1;
  }
}

struct HomoParts {
  GrlHomoPart p[GRL_MAX_HOMO_PARTS];
  int n;
};

__device__ __forceinline__ int64_t homo_ptr(const HomoParts& hp, int b) {
  int64_t s = 0;
  for (int t = 0; t < hp.n; ++t) s += hp.p[t].edge_ptr[b];
  return s;
}

// One thread per output position p of the merged COO (grid-stride): the graph b owning p is found by a binary search
// over the merged edge_ptr (summed from the parts on the fly), then the part and the edge inside it by walking the
// parts' counts of graph b.  Threads p <= B also write edge_ptr[p].
__global__ void __launch_bounds__(256) homo_merge_kernel(HomoParts hp, int B, int n_tot, int64_t capacity,
                                                         int64_t* __restrict__ edge_ptr, int64_t* __restrict__ coo,
                                                         int64_t row_stride) {
  const int64_t e_end = homo_ptr(hp, B);
  const int64_t n = capacity > (int64_t)B + 1 ? capacity : (int64_t)B + 1;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (int64_t)gridDim.x * blockDim.x) {
    if (p <= B) edge_ptr[p] = homo_ptr(hp, (int)p);
    if (p >= capacity) continue;
    if (p >= e_end) {
      coo[p] = 0;
      coo[row_stride + p] = 0;
      continue;
    }
    int lo = 0, hi = B - 1;  // largest b with homo_ptr(b) <= p
    while (lo < hi) {
      const int mid = (lo + hi + 1) / 2;
      if (homo_ptr(hp, mid) <= p) lo = mid; else hi = mid - 1;
    }
    const int b = lo;
    int64_t r = p - homo_ptr(hp, b);
    for (int t = 0; t < hp.n; ++t) {
      const GrlHomoPart& q = hp.p[t];
      const int64_t e0 = q.edge_ptr[b], c = q.edge_ptr[b + 1] - e0;
      if (r >= c) {
        r -= c;
        continue;
      }
      const int64_t e = e0 + r, base = (int64_t)b * n_tot;
      coo[p] = base + q.off_src + (q.coo[e] - (int64_t)b * q.n_src);
      coo[row_stride + p] = base + q.off_dst + (q.coo[q.coo_row_stride + e] - (int64_t)b * q.n_dst);
      break;
    }
  }
}

// sub_edge_ptr / sub_rowptr_dst of grl_sub_edge_set: the output rows of graph b are contiguous in the parent, so their
// edges are the parent's edge range [rowptr_dst[b*n_tot+out_off], rowptr_dst[b*n_tot+out_off+n_out]).  One CTA,
// sequential chunks of graphs per thread, like knn_edge_ptr_kernel.
__global__ void sub_edge_ptr_kernel(const int32_t* __restrict__ rowptr_dst, int B, int n_tot, int out_off, int n_out,
                                    int64_t* __restrict__ sub_edge_ptr, int32_t* __restrict__ sub_rowptr_dst) {
  __shared__ long long part[1024];
  const int tid = threadIdx.x, nt = blockDim.x;
  const int per = (B + nt - 1) / nt;
  const int b0 = tid * per, b1 = min(b0 + per, B);
  auto row = [&](int b, int a) { return (long long)rowptr_dst[(size_t)b * n_tot + out_off + a]; };
  long long s = 0;
  for (int b = b0; b < b1; ++b) s += row(b, n_out) - row(b, 0);
  part[tid] = s;
  __syncthreads();
  if (tid == 0) {
    long long run = 0;
    for (int i = 0; i < nt; ++i) { const long long t = part[i]; part[i] = run; run += t; }
    sub_edge_ptr[B] = run;
    sub_rowptr_dst[(size_t)B * n_out] = (int32_t)run;
  }
  __syncthreads();
  long long run = part[tid];
  for (int b = b0; b < b1; ++b) {
    sub_edge_ptr[b] = run;
    const long long base = row(b, 0);
    for (int a = 0; a < n_out; ++a) sub_rowptr_dst[(size_t)b * n_out + a] = (int32_t)(run + row(b, a) - base);
    run += row(b, n_out) - base;
  }
}

struct SubEdgeOut {
  int64_t* eids;
  int32_t *eids32, *edge_src, *edge_dst, *edge_dst_parent;
  int64_t* pairs;
  int64_t pairs_row_stride;
};

__device__ __forceinline__ int out_rank(int32_t node, int n_tot, int out_off, int n_out) {
  const int g = node / n_tot, l = node - g * n_tot - out_off;
  return (l >= 0 && l < n_out) ? g * n_out + l : -1;
}

// Per-edge arrays of grl_sub_edge_set, one thread per sub edge q and per parent edge (grid-stride over the larger).
__global__ void __launch_bounds__(256) sub_edges_kernel(const int32_t* __restrict__ rowptr_dst,
                                                        const int32_t* __restrict__ edge_src,
                                                        const int32_t* __restrict__ edge_dst, int64_t n_edges, int B,
                                                        int n_tot, int out_off, int n_out, int64_t capacity,
                                                        const int64_t* __restrict__ sub_edge_ptr, SubEdgeOut o) {
  const int64_t e_par = rowptr_dst[(size_t)B * n_tot], e_sub = sub_edge_ptr[B];
  const int64_t n = capacity > n_edges ? capacity : n_edges;
  auto rank = [&](int64_t e) { return e < e_par ? out_rank(edge_dst[e], n_tot, out_off, n_out) : -1; };
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += (int64_t)gridDim.x * blockDim.x) {
    if (q < n_edges) o.edge_dst_parent[q] = rank(q);
    if (q >= capacity) continue;
    int64_t e = 0;
    int32_t src = 0;
    if (q < e_sub) {
      int lo = 0, hi = B - 1;  // largest b with sub_edge_ptr[b] <= q
      while (lo < hi) {
        const int mid = (lo + hi + 1) / 2;
        if (sub_edge_ptr[mid] <= q) lo = mid; else hi = mid - 1;
      }
      e = rowptr_dst[(size_t)lo * n_tot + out_off] + (q - sub_edge_ptr[lo]);
      src = edge_src[e];
    }
    const int dst = rank(e);
    o.eids[q] = e;
    o.eids32[q] = (int32_t)e;
    o.edge_src[q] = src;
    o.edge_dst[q] = dst;
    o.pairs[q] = src;
    o.pairs[o.pairs_row_stride + q] = dst;
  }
}

}  // namespace grl

extern "C" {

int grl_knn_edge_ptr(const int32_t* num_valid, int B, int P, int k, int64_t* edge_ptr, grl_stream_t stream) {
  GRL_REQUIRE(edge_ptr && B > 0 && P > 0, GRL_EINVAL, "grl_knn_edge_ptr: bad arguments");
  GRL_REQUIRE(k >= 1 && k <= GRL_MAX_KNN, GRL_EUNSUPPORTED, "grl_knn_edge_ptr: k=%d not in [1,%d]", k, GRL_MAX_KNN);
  grl::knn_edge_ptr_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(num_valid, B, P, k, edge_ptr);
  return grl::check_launch("grl_knn_edge_ptr");
}

int grl_knn_graph(const float* pos, const int32_t* num_valid, const int64_t* edge_ptr, int B, int P, int k, int64_t* coo,
                  int64_t coo_row_stride, grl_stream_t stream) {
  GRL_REQUIRE(pos && edge_ptr && coo && B > 0 && P > 0, GRL_EINVAL, "grl_knn_graph: bad arguments");
  GRL_REQUIRE(k >= 1 && k <= GRL_MAX_KNN, GRL_EUNSUPPORTED, "grl_knn_graph: k=%d not in [1,%d]", k, GRL_MAX_KNN);
  GRL_REQUIRE(P <= grl::kMaxP, GRL_EUNSUPPORTED, "grl_knn_graph: P=%d > %d", P, grl::kMaxP);
  int grid = B < 16 * grl::sm_count() ? B : 16 * grl::sm_count();
  grl::knn_graph_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(pos, num_valid, edge_ptr, B, P, k, coo, coo_row_stride);
  return grl::check_launch("grl_knn_graph");
}

int grl_knn_topology(const float* pos, const int32_t* num_valid, const int64_t* edge_ptr, int B, int P, int k,
                     int64_t capacity, int64_t* coo, int64_t coo_row_stride, int32_t* rowptr_dst, int32_t* edge_src,
                     int32_t* edge_dst, int32_t* eid_coo, int32_t* rowptr_src, int32_t* src_eid, int32_t* s_src,
                     int32_t* s_dst, grl_stream_t stream) {
  // the per-edge arrays may be NULL for a set of no edges (capacity 0): nothing is written to them then
  GRL_REQUIRE(pos && edge_ptr && rowptr_dst && rowptr_src && B > 0 && P > 0 && (s_src == nullptr) == (s_dst == nullptr) &&
                  (capacity == 0 || (coo && edge_src && edge_dst && eid_coo && src_eid)),
              GRL_EINVAL, "grl_knn_topology: bad arguments");
  GRL_REQUIRE(k >= 1 && k <= GRL_MAX_KNN, GRL_EUNSUPPORTED, "grl_knn_topology: k=%d not in [1,%d]", k, GRL_MAX_KNN);
  GRL_REQUIRE(P <= grl::kMaxP, GRL_EUNSUPPORTED, "grl_knn_topology: P=%d > %d", P, grl::kMaxP);
  const int64_t bound = (int64_t)B * P * std::max(0, std::min(k, P - 1));  // edges of B graphs with every point valid
  GRL_REQUIRE(capacity >= bound && coo_row_stride >= capacity, GRL_EINVAL,
              "grl_knn_topology: capacity=%lld (row stride %lld) below the %lld edges B*P*min(k,P-1)",
              (long long)capacity, (long long)coo_row_stride, (long long)bound);
  GRL_REQUIRE(capacity <= INT32_MAX && (int64_t)B * P < INT32_MAX, GRL_EUNSUPPORTED,
              "grl_knn_topology: capacity=%lld or B*P=%lld exceeds the int32 edge / node ids", (long long)capacity,
              (long long)B * P);
  const int graph_ctas = B < 16 * grl::sm_count() ? B : 16 * grl::sm_count();
  // a tail can only exist when some graph has fewer than P valid points or the buffer is larger than every edge
  const bool tail = num_valid != nullptr || capacity > bound;
  const int tail_ctas = tail ? (int)std::min<int64_t>(grl::sm_count(), (capacity + 4095) / 4096) : 0;
  grl::KnnTopoOut o{coo, coo_row_stride, rowptr_dst, edge_src, edge_dst, eid_coo, rowptr_src, src_eid, s_src, s_dst};
  grl::knn_topology_kernel<<<graph_ctas + tail_ctas, 128, 0, (cudaStream_t)stream>>>(pos, num_valid, edge_ptr, B, P, k,
                                                                                    capacity, graph_ctas, o);
  return grl::check_launch("grl_knn_topology");
}

int grl_radius_neighbors(const float* pos, const int32_t* num_valid, int B, int P, float radius, int max_neighbors,
                         int32_t* nbr, int32_t* cnt, grl_stream_t stream) {
  GRL_REQUIRE(pos && nbr && cnt && B > 0 && P > 0 && radius > 0.f, GRL_EINVAL, "grl_radius_neighbors: bad arguments");
  GRL_REQUIRE(max_neighbors >= 1 && max_neighbors <= GRL_MAX_KNN, GRL_EUNSUPPORTED,
              "grl_radius_neighbors: max_neighbors=%d not in [1,%d]", max_neighbors, GRL_MAX_KNN);
  GRL_REQUIRE(P <= grl::kMaxP, GRL_EUNSUPPORTED, "grl_radius_neighbors: P=%d > %d", P, grl::kMaxP);
  int grid = B < 16 * grl::sm_count() ? B : 16 * grl::sm_count();
  grl::radius_neighbors_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(pos, num_valid, B, P, radius * radius,
                                                                       max_neighbors, nbr, cnt);
  return grl::check_launch("grl_radius_neighbors");
}

int grl_radius_edge_ptr(const int32_t* cnt, int B, int P, int64_t capacity, int64_t* edge_ptr, grl_stream_t stream) {
  GRL_REQUIRE(cnt && edge_ptr && B > 0 && P > 0 && capacity >= 0, GRL_EINVAL, "grl_radius_edge_ptr: bad arguments");
  grl::radius_edge_ptr_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(cnt, B, P, capacity, edge_ptr);
  return grl::check_launch("grl_radius_edge_ptr");
}

int grl_radius_graph(const int32_t* nbr, const int32_t* cnt, const int64_t* edge_ptr, int B, int P, int max_neighbors,
                     int64_t* coo, int64_t coo_row_stride, int64_t capacity, grl_stream_t stream) {
  GRL_REQUIRE(nbr && cnt && edge_ptr && coo && B > 0 && P > 0 && capacity >= 1 && coo_row_stride >= capacity, GRL_EINVAL,
              "grl_radius_graph: bad arguments");
  GRL_REQUIRE(max_neighbors >= 1 && max_neighbors <= GRL_MAX_KNN, GRL_EUNSUPPORTED,
              "grl_radius_graph: max_neighbors=%d not in [1,%d]", max_neighbors, GRL_MAX_KNN);
  GRL_REQUIRE(P <= grl::kMaxP, GRL_EUNSUPPORTED, "grl_radius_graph: P=%d > %d", P, grl::kMaxP);
  int grid = B < 16 * grl::sm_count() ? B : 16 * grl::sm_count();
  grl::radius_graph_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(nbr, cnt, edge_ptr, B, P, max_neighbors, coo,
                                                                   coo_row_stride, capacity);
  return grl::check_launch("grl_radius_graph");
}

int grl_dense_edges(int mode, const int32_t* num_valid, const int64_t* edge_ptr, int B, int n_src, int n_dst, int64_t* coo,
                    int64_t coo_row_stride, grl_stream_t stream) {
  GRL_REQUIRE((mode == 0 || mode == 1) && edge_ptr && coo && B > 0 && n_src > 0 && n_dst > 0, GRL_EINVAL,
              "grl_dense_edges: bad arguments");
  GRL_REQUIRE(mode == 1 || n_src > 1, GRL_EINVAL, "grl_dense_edges: mode 0 needs n_src > 1");
  (void)num_valid;
  int grid = B < 16 * grl::sm_count() ? B : 16 * grl::sm_count();
  grl::dense_edges_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(mode, num_valid, edge_ptr, B, n_src, n_dst, coo,
                                                                  coo_row_stride);
  return grl::check_launch("grl_dense_edges");
}

int grl_csr_build(const int64_t* coo, int64_t coo_row_stride, const int64_t* edge_ptr, int B, int n_key, int key_row,
                  int32_t* rowptr, int32_t* other, int32_t* eid, grl_stream_t stream) {
  GRL_REQUIRE(coo && edge_ptr && rowptr && other && eid && B > 0 && n_key > 0 && (key_row == 0 || key_row == 1),
              GRL_EINVAL, "grl_csr_build: bad arguments");
  GRL_REQUIRE(n_key <= 8192, GRL_EUNSUPPORTED, "grl_csr_build: n_key=%d > 8192", n_key);
  int grid = B < 16 * grl::sm_count() ? B : 16 * grl::sm_count();
  grl::csr_build_kernel<<<grid, 128, (n_key + 1) * sizeof(int), (cudaStream_t)stream>>>(coo, coo_row_stride, edge_ptr, B,
                                                                                       n_key, key_row, rowptr, other, eid);
  return grl::check_launch("grl_csr_build");
}

int grl_homo_merge(const GrlHomoPart* parts, int n_parts, int B, int n_tot, int64_t capacity, int64_t* edge_ptr,
                   int64_t* coo, int64_t coo_row_stride, grl_stream_t stream) {
  GRL_REQUIRE(parts && edge_ptr && B > 0 && n_tot > 0 && capacity >= 0 && (capacity == 0 || coo) &&
                  coo_row_stride >= capacity,
              GRL_EINVAL, "grl_homo_merge: bad arguments");
  GRL_REQUIRE(n_parts >= 0 && n_parts <= GRL_MAX_HOMO_PARTS, GRL_EUNSUPPORTED, "grl_homo_merge: n_parts=%d not in [0,%d]",
              n_parts, GRL_MAX_HOMO_PARTS);
  grl::HomoParts hp{};
  hp.n = n_parts;
  for (int t = 0; t < n_parts; ++t) {
    const GrlHomoPart& q = parts[t];
    GRL_REQUIRE(q.edge_ptr && q.n_src > 0 && q.n_dst > 0 && q.off_src >= 0 && q.off_dst >= 0 &&
                    q.off_src + q.n_src <= n_tot && q.off_dst + q.n_dst <= n_tot,
                GRL_EINVAL, "grl_homo_merge: bad part %d", t);
    hp.p[t] = q;
  }
  const int64_t n = std::max<int64_t>(capacity, (int64_t)B + 1);
  const int grid = (int)std::min<int64_t>((n + 255) / 256, 16LL * grl::sm_count());
  grl::homo_merge_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(hp, B, n_tot, capacity, edge_ptr, coo, coo_row_stride);
  return grl::check_launch("grl_homo_merge");
}

int grl_sub_edge_set(const int32_t* rowptr_dst, const int32_t* edge_src, const int32_t* edge_dst, int64_t n_edges, int B,
                     int n_tot, int out_off, int n_out, int64_t capacity, int64_t* sub_edge_ptr, int32_t* sub_rowptr_dst,
                     int64_t* eids, int32_t* eids32, int32_t* sub_edge_src, int32_t* sub_edge_dst,
                     int32_t* edge_dst_parent, int64_t* pairs, int64_t pairs_row_stride, grl_stream_t stream) {
  GRL_REQUIRE(rowptr_dst && sub_edge_ptr && sub_rowptr_dst && B > 0 && n_tot > 0 && n_out > 0 && out_off >= 0 &&
                  out_off + n_out <= n_tot && n_edges >= 0 && capacity >= 0 && pairs_row_stride >= capacity &&
                  (n_edges == 0 || (edge_src && edge_dst && edge_dst_parent)) &&
                  (capacity == 0 || (eids && eids32 && sub_edge_src && sub_edge_dst && pairs)),
              GRL_EINVAL, "grl_sub_edge_set: bad arguments");
  GRL_REQUIRE((int64_t)B * n_tot < INT32_MAX && n_edges <= INT32_MAX && capacity <= INT32_MAX, GRL_EUNSUPPORTED,
              "grl_sub_edge_set: sizes exceed the int32 node / edge ids");
  grl::sub_edge_ptr_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(rowptr_dst, B, n_tot, out_off, n_out, sub_edge_ptr,
                                                                 sub_rowptr_dst);
  int rc = grl::check_launch("grl_sub_edge_set");
  if (rc != GRL_OK) return rc;
  const int64_t n = std::max(capacity, n_edges);
  if (n == 0) return GRL_OK;
  const int grid = (int)std::min<int64_t>((n + 255) / 256, 16LL * grl::sm_count());
  grl::SubEdgeOut o{eids, eids32, sub_edge_src, sub_edge_dst, edge_dst_parent, pairs, pairs_row_stride};
  grl::sub_edges_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(rowptr_dst, edge_src, edge_dst, n_edges, B, n_tot, out_off,
                                                                n_out, capacity, sub_edge_ptr, o);
  return grl::check_launch("grl_sub_edge_set");
}

}  // extern "C"
