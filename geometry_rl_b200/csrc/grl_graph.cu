// K1: batched edge construction (kNN / radius / dense) and stable CSR build.
// Replaces the per-graph Python loop of geometry_rl/modules/pyg_data/rigid_tasks_data.py:275-321
// (torch_geometric.nn.knn_graph per graph, nested loops for AGENT / TASK edges, coalesce()) and
// rope_tasks_data.py:238-278, cloth_tasks_data.py:236-286; plus the graph-major batching of
// Batch.from_data_list (rigid_tasks_data.py:324).  One CTA per graph; graphs have <= a few hundred
// nodes, so everything is brute force in shared memory.  Integer outputs are bit-exact by construction.
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

}  // extern "C"
