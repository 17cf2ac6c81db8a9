/*
 * grl_b200.h — C ABI of the B200-native (sm_100a) GeometryRL policy-training hot path.
 *
 * The reference (thobotics/geometry_rl) has no FFI of its own: its hot path is Python calling
 * third-party wheels.  Each entry point below replaces one such call site (cited as
 * reference-file:line, paths relative to the reference checkout).  The Python host layer
 * (geometry_rl_b200/_lib.py, ops.py) binds these with ctypes; INTEGRATION.md shows the stub.
 *
 * Conventions
 *  - All pointers are DEVICE pointers unless a parameter name ends in `_host`.
 *  - Buffers (inputs, outputs, workspaces) are allocated and owned by the caller; nothing is
 *    allocated or freed behind the ABI.
 *  - Every function is stream-ordered on `stream` (a cudaStream_t), never synchronises, keeps no
 *    mutable global state and is safe to capture in a CUDA graph.
 *  - Return value: GRL_OK or a negative GRL_E* code; grl_last_error() returns a thread-local
 *    message.  No exceptions cross the ABI.
 *  - Latent rows are [O=16][C=64] fp32 (4096 B per node); "edge order" is the dst-sorted CSR
 *    order produced by grl_csr_build.
 */
#ifndef GRL_B200_H_
#define GRL_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GRL_OK 0
#define GRL_EINVAL (-1)      /* bad shape / null pointer / inconsistent sizes            */
#define GRL_EUNSUPPORTED (-2) /* O != 16, C != 64, hidden != 256, k > GRL_MAX_ACTION_DIM … */
#define GRL_ECUDA (-3)       /* cudaGetLastError() != cudaSuccess after a launch          */

#define GRL_NUM_ORI 16
#define GRL_CHANNELS 64
#define GRL_HIDDEN 256
#define GRL_BASIS_FEATS 14   /* PolynomialFeatures(2) of (i1, i2): 2 + 4 + 8               */
#define GRL_MAX_ACTION_DIM 16
#define GRL_MAX_KNN 8

typedef void* grl_stream_t; /* cudaStream_t */

int grl_abi_version(void);
const char* grl_last_error(void);
/* Number of SMs of the current device (grid sizing for the persistent kernels). */
int grl_sm_count(void);
/* Launch policy for jobs that run collectives CONCURRENTLY with the kernels (data parallelism with the critic branch on its
 * own stream): every persistent kernel of this library sizes its grid to fill all SMs, so a CTA of a collective that is
 * spinning on an SM (waiting for its peers) keeps one CTA of the kernel from starting until the collective ends - and a
 * late CTA of a persistent grid doubles the kernel's duration.  With n SMs reserved the grids are sized for
 * (SMs - n) and both kinds of CTA always find a free SM.  Process-wide; grl_sm_count() reports the reduced number. */
int grl_reserve_sms(int n);

/* ------------------------------------------------------------------------------------------
 * K1  edge construction -> sorted CSR
 * replaces torch_geometric.nn.knn_graph(points[:P_i], k) + HeteroData.coalesce() per graph in a
 * Python loop: geometry_rl/modules/pyg_data/rigid_tasks_data.py:275-321, rope_tasks_data.py:251.
 * ------------------------------------------------------------------------------------------ */

/* Per-graph edge counts of a kNN graph: count[b] = P_b * min(k, P_b - 1), and their exclusive
 * prefix sum edge_ptr[B+1].  num_valid may be NULL (all P points valid). */
int grl_knn_edge_ptr(const int32_t* num_valid, int B, int P, int k, int64_t* edge_ptr, grl_stream_t stream);

/* Batched brute-force kNN (loop=False) over pos[B][P][3] (first num_valid[b] points of graph b),
 * emitted as the COALESCED COO the reference ends up with: row0 = neighbour (source), row1 =
 * centre (target), sorted by (row0,row1), global node index = b*P + local.  coo is [2][E_total]
 * int64 with E_total = edge_ptr[B].  Squared distances are (dx*dx + dy*dy) + dz*dz with separate
 * fp32 roundings; ties -> lower index. */
int grl_knn_graph(const float* pos, const int32_t* num_valid, const int64_t* edge_ptr, int B, int P, int k,
                  int64_t* coo, int64_t coo_row_stride, grl_stream_t stream);

/* Radius graph (extension, no reference counterpart; SURVEY §3.4): neighbours within `radius`,
 * at most max_neighbors nearest, same output convention but into a PADDED buffer:
 * nbr[B][P][max_neighbors] (local index or -1), cnt[B][P]. */
int grl_radius_neighbors(const float* pos, const int32_t* num_valid, int B, int P, float radius, int max_neighbors,
                         int32_t* nbr, int32_t* cnt, grl_stream_t stream);

/* Per-graph edge counts of a radius graph (the sum of cnt[b][0..P) from grl_radius_neighbors) and their exclusive
 * prefix sum edge_ptr[B+1], every entry clamped to `capacity`.  Reads nothing on the host: usable inside a CUDA graph. */
int grl_radius_edge_ptr(const int32_t* cnt, int B, int P, int64_t capacity, int64_t* edge_ptr, grl_stream_t stream);

/* Coalesced COO of the radius graph given by nbr / cnt (grl_radius_neighbors) and edge_ptr (grl_radius_edge_ptr), in
 * the convention of grl_knn_graph: row0 = neighbour (source), row1 = centre (target), sorted by (row0,row1) per graph,
 * graph-major.  coo is [2][capacity] int64 (coo_row_stride >= capacity); entries [edge_ptr[B], capacity) are written
 * with 0, so a gather over the whole buffer stays in bounds.  A point with a non-finite coordinate has no edges (a NaN
 * distance never passes sqdist <= radius^2). */
int grl_radius_graph(const int32_t* nbr, const int32_t* cnt, const int64_t* edge_ptr, int B, int P, int max_neighbors,
                     int64_t* coo, int64_t coo_row_stride, int64_t capacity, grl_stream_t stream);

/* Dense edge sets the reference builds with nested Python loops
 * (rigid_tasks_data.py:289-300,313-319): write the coalesced batched COO for
 *   mode 0: all ordered pairs j != k among n_src nodes per graph      (AGENT / cloth INTERNAL)
 *   mode 1: every valid source j < num_valid[b] -> every destination k (TASK)
 * edge_ptr[B+1] must hold the exclusive prefix sum of the per-graph counts. */
int grl_dense_edges(int mode, const int32_t* num_valid, const int64_t* edge_ptr, int B, int n_src, int n_dst,
                    int64_t* coo, int64_t coo_row_stride, grl_stream_t stream);

/* Stable counting sort of a batched COO (graph-major, graph b owns edges [edge_ptr[b],
 * edge_ptr[b+1]) and key nodes [b*n_key, (b+1)*n_key)) by row `key_row` (1 = dst, 0 = src):
 *   rowptr[B*n_key + 1], other[E] (the non-key endpoint), eid[E] (position in the input COO).
 * Relative order of edges with equal key is preserved (== summation order of a sequential
 * scatter over the coalesced COO). */
int grl_csr_build(const int64_t* coo, int64_t coo_row_stride, const int64_t* edge_ptr, int B, int n_key, int key_row,
                  int32_t* rowptr, int32_t* other, int32_t* eid, grl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K2  fused equivariant message passing (forward and backward)
 * replaces hepi.py:109-123,136-171 / ponita/conv.py:71-149 / ponita/ponita.py:149-185,219-230:
 * PolynomialFeatures+basis_fn, kernel Linear, gather*mul, torch_scatter.scatter (conv.py:141),
 * fibre einsum (conv.py:90), LayerNorm+Linear+GELU+Linear node update (conv.py:64-69,112).
 * ------------------------------------------------------------------------------------------ */

/* Lift + node encoder (to_from_sphere.py:4-9, hepi.py:136-143):
 *   x[n][o][c] = sum_s scal[n][s] W[c][s] + sum_v <vec[n][v][:dim], ori[o]> W[c][S+v]          */
typedef struct {
  int32_t n_nodes, n_scalars, n_vectors, dim; /* dim = 2 | 3 */
  const float* scalars;                        /* [N][S]                                        */
  const float* vectors;                        /* [N][V][3]                                     */
  const float* ori;                            /* [16][3] (z = 0 when dim == 2)                 */
  const float* weight;                         /* [64][S+V] row-major (nn.Linear.weight)        */
  float* x;                                    /* [N][16][64]                                   */
  /* backward */
  const float* grad_x;                         /* [N][16][64]                                   */
  float* grad_weight_partials;                 /* [n_partials][64][S+V]                         */
  int32_t n_partials;
  const int32_t* node_ids;                     /* optional [N]: row of node n in scalars / vectors (NULL = n); lets a
                                                  compacted batch read the padded feature arrays in place      */
} GrlEmbedDesc;
int grl_embed_fwd(const GrlEmbedDesc* d, grl_stream_t stream);
int grl_embed_bwd(const GrlEmbedDesc* d, grl_stream_t stream);

/* Edge basis (hepi.py:109-123 + basis_fn hepi.py:76-82): per edge (edge order) and orientation
 * invariants (i1,i2) -> 14 polynomial features -> Linear(14,64) GELU Linear(64,64) GELU.       */
typedef struct {
  int32_t n_edges, dim;
  const int32_t* edge_src;   /* [E] index into pos_src                                          */
  const int32_t* edge_dst;   /* [E] index into pos_dst                                          */
  const float* pos_src;      /* [Ns][3]                                                         */
  const float* pos_dst;      /* [Nd][3]                                                         */
  const float* ori;          /* [16][3]                                                         */
  const float* w1t;          /* [16][64]: w1t[f][n] = W1[n][f], rows 14,15 zero                 */
  const float* b1;           /* [64]                                                            */
  const float* w2t;          /* [64][64]: w2t[k][n] = W2[n][k]                                  */
  const float* b2;           /* [64]                                                            */
  float* basis;              /* [E][16][64]                                                     */
  /* backward */
  const float* w2;           /* [64][64] row-major W2[n][k]                                     */
  const float* grad_basis;   /* [E][16][64]                                                     */
  float* grad_partials;      /* [n_partials][GRL_BASIS_GRAD_FLOATS]                             */
  int32_t n_partials;
  /* bf16 tensor-core path: the basis and its gradient are stored as bf16 [E][16][64] (2 KB per edge) */
  void* basis_bf16;
  const void* grad_basis_bf16;
} GrlBasisDesc;
/* partial layout: gW1[64][16] | gb1[64] | gW2[64][64] | gb2[64] */
#define GRL_BASIS_GRAD_FLOATS (64 * 16 + 64 + 64 * 64 + 64)
int grl_edge_basis_fwd(const GrlBasisDesc* d, grl_stream_t stream);
int grl_edge_basis_bwd(const GrlBasisDesc* d, grl_stream_t stream);

/* One separable fibre-bundle convolution + ConvNeXt node update. */
typedef struct {
  int32_t n_src, n_dst, n_edges;
  /* dst-sorted CSR (edge order) */
  const int32_t* rowptr_dst; /* [n_dst+1]                                                       */
  const int32_t* edge_src;   /* [E]                                                             */
  const int32_t* edge_dst;   /* [E]                                                             */
  /* src-sorted CSR: entries reference edge-order positions */
  const int32_t* rowptr_src; /* [n_src+1]                                                       */
  const int32_t* src_eid;    /* [E] edge-order position of the q-th src-sorted entry            */
  const float* x_src;        /* [n_src][16][64]                                                 */
  const float* x_dst;        /* [n_dst][16][64]                                                 */
  const float* basis;        /* [E][16][64]                                                     */
  const float* fiber_kernel; /* [16(o)][16(p)][64]: x2[p] = 1/16 sum_o x1[o] * fk[o][p]         */
  const float* wk_t;         /* [64][64]: wk_t[j][c] = kernel.weight[c][j]                      */
  const float* wk;           /* [64][64] kernel.weight[c][j]                                    */
  const float* bias;         /* [64]                                                            */
  const float* ln_g;         /* [64]                                                            */
  const float* ln_b;         /* [64]                                                            */
  const float* w1_t;         /* [4][64(k)][64(n)]: w1_t[q][k][n] = W1[q*64+n][k]                */
  const float* w1;           /* [256][64] row-major                                             */
  const float* b1;           /* [256]                                                           */
  const float* w2_t;         /* [4][64(k)][64(n)]: w2_t[q][k][n] = W2[n][q*64+k]                */
  const float* w2_c;         /* [4][64(n)][64(m)]: w2_c[q][n][m] = W2[n][q*64+m]                */
  const float* b2;           /* [64]                                                            */
  float* x1;                 /* [n_dst][16][64] aggregated messages (saved for backward)        */
  float* out;                /* [n_dst][16][64]                                                 */
  int32_t accumulate_out;    /* out += x_dst + mlp(...) (HeteroConv group "sum")                */
  /* backward */
  const float* grad_out;     /* [n_dst][16][64]                                                 */
  float* grad_x1;            /* [n_dst][16][64] workspace                                       */
  float* grad_x_src;         /* [n_src][16][64]                                                 */
  const float* grad_x_src_init; /* optional [n_src][16][64] added in (may alias nothing)        */
  float* grad_basis;         /* [E][16][64]                                                     */
  int32_t accumulate_grad_basis; /* 0 overwrite, 1 add (fp32 sum, rounded once), 2 per edge (grad_basis_acc_mask; *_tc only) */
  float* node_grad_partials; /* [n_partials_node][GRL_NODE_GRAD_FLOATS]                         */
  int32_t n_partials_node;
  float* edge_grad_partials; /* [n_partials_edge][64*64] (kernel.weight)                        */
  int32_t n_partials_edge;
  /* bf16 tensor-core path (the *_tc entry points): plain row-major weights, staged as bf16 operands */
  const float* w2;           /* [64][256] row-major (nn.Linear.weight of the second node-MLP layer) */
  const void* basis_bf16;    /* [E][16][64] bf16 (edge order)                                       */
  void* grad_basis_bf16;     /* [E][16][64] bf16                                                    */
  float* grad_x2;            /* [n_dst][16][64] workspace: gradient w.r.t. the pre-LayerNorm tensor   */
  float* x2;                 /* optional [n_dst][16][64]: pre-LayerNorm tensor fibre(x1) + bias, written by
                                grl_fbconv_node_fwd_tc and read by grl_fbconv_node_bwd_tc instead of recomputing it     */
  const uint32_t* grad_amax; /* grl_absmax(grad_out): the tensor-core backward stages gradients as fp16 scaled by a
                                power of two derived from it (max |g| -> [32, 64)); NULL = scale 1          */
  /* sub layers (a layer evaluated at a subset of dst nodes that shares the PARENT graph's per-edge tensors):         */
  const int32_t* basis_row;  /* optional [E], grl_fbconv_edge_fwd_tc: row of edge e in basis_bf16 (NULL = e)          */
  const int32_t* grad_basis_acc_mask; /* accumulate_grad_basis == 2, grl_fbconv_edge_bwd_tc: [E_parent], indexed like
                                basis_bf16; edge e ADDS to its grad_basis_bf16 row iff mask[e] >= 0 (a sub layer wrote
                                that row earlier in this backward pass) and overwrites it otherwise                    */
} GrlConvDesc;
/* node partial layout: gW1[256][64] | gb1[256] | gW2[64][256] | gb2[64] | g_ln_g[64] | g_ln_b[64]
 *                      | g_bias[64] | g_fk[16][16][64] */
#define GRL_NODE_GRAD_FLOATS (256 * 64 + 256 + 64 * 256 + 64 + 64 + 64 + 64 + 16 * 16 * 64)
int grl_fbconv_edge_fwd(const GrlConvDesc* d, grl_stream_t stream); /* basis,x_src -> x1            */
int grl_fbconv_node_fwd(const GrlConvDesc* d, grl_stream_t stream); /* x1,x_dst -> out             */
int grl_fbconv_node_bwd(const GrlConvDesc* d, grl_stream_t stream); /* grad_out -> grad_x1, node partials */
int grl_fbconv_edge_bwd(const GrlConvDesc* d, grl_stream_t stream); /* grad_x1 -> grad_x_src, grad_basis, edge partials */
/* bf16 MLP path (north_star: "bf16 MLP path within 1e-2"): the same operators with the nn.Linear contractions
 * on the 5th-generation tensor cores (tcgen05.mma kind::f16, bf16 operands, fp32 accumulators in TMEM);
 * fibre convolution, LayerNorm, GELU, residuals and all segmented sums stay fp32. */
int grl_edge_basis_fwd_tc(const GrlBasisDesc* d, grl_stream_t stream);   /* positions -> basis_bf16        */
int grl_fbconv_edge_fwd_tc(const GrlConvDesc* d, grl_stream_t stream);   /* basis_bf16, x_src -> x1        */
int grl_fbconv_node_fwd_tc(const GrlConvDesc* d, grl_stream_t stream);
int grl_fbconv_edge_bwd_tc(const GrlConvDesc* d, grl_stream_t stream);   /* grad_x1 -> grad_x_src, grad_basis_bf16, edge partials */
int grl_edge_basis_bwd_tc(const GrlBasisDesc* d, grl_stream_t stream);   /* grad_basis_bf16 -> basis_fn partials */
/* grad_out -> grad_x1 + node partials (two launches: tensor-core MLP/LayerNorm backward, fp32 fibre backward) */
int grl_fbconv_node_bwd_tc(const GrlConvDesc* d, grl_stream_t stream);

/* Fused edge side of one convolution on the 16-bit tensor-core path (round 2): invariants -> basis MLP -> `kernel`
 * Linear -> gather * mul -> CSR-ordered segmented sum in ONE kernel, and the mirrored backward.  The edge basis is
 * recomputed per tile in shared memory; no [E][16][64] basis or basis-gradient tensor exists in HBM (SURVEY 8(d)).
 * Replaces hepi.py:76-82,109-123 + ponita/conv.py:84-87,116-149 (forward) and their autograd (backward); supersedes
 * grl_edge_basis_{fwd,bwd}_tc + grl_fbconv_edge_{fwd,bwd}_tc on the product path.
 *   forward : entries sorted by DST (edge order), rowptr = dst CSR, n_key = n_dst:
 *             x1[d] = sum_{e in in(d)} (basis(e) Wk^T) * x_src[src(e)]
 *   backward: entries sorted by SRC (ties in edge order), rowptr = src CSR, n_key = n_src:
 *             grad_x_src[s] = grad_x_src_init[s] + sum_{e in out(s)} (basis(e) Wk^T) * grad_x1[dst(e)]
 *             + one partial slot per CTA with the gradients of kernel.weight and of the basis MLP.
 * Both directions take the entry list as two plain arrays (e_src[p], e_dst[p]): no dependent index loads.       */
typedef struct {
  int32_t n_key, n_edges, dim, n_partials;
  const int32_t* rowptr;      /* [n_key+1] CSR over the key-sorted entry list                                  */
  const int32_t* e_src;       /* [E] source node of entry p (row of x_src / pos_src)                           */
  const int32_t* e_dst;       /* [E] destination node of entry p (row of x1 / grad_x1 / pos_dst)               */
  const float* pos_src;       /* [n_src][3]                                                                    */
  const float* pos_dst;       /* [n_dst][3]                                                                    */
  const float* ori;           /* [16][3] (z = 0 when dim == 2)                                                 */
  const float* w1;            /* [64][14] basis_fn[1].weight, row-major                                        */
  const float* b1;            /* [64]                                                                          */
  const float* w2;            /* [64][64] basis_fn[3].weight, row-major                                        */
  const float* b2;            /* [64]                                                                          */
  const float* wk;            /* [64][64] kernel.weight, row-major                                             */
  const float* x_src;         /* [n_src][16][64]                                                               */
  float* x1;                  /* forward out: [n_dst][16][64]                                                  */
  const float* grad_x1;       /* backward in: [n_dst][16][64]                                                  */
  float* grad_x_src;          /* backward out: [n_src][16][64]                                                 */
  const float* grad_x_src_init; /* optional [n_src][16][64] added in                                           */
  float* grad_partials;       /* [n_partials][GRL_FUSED_EDGE_GRAD_FLOATS]; the backward launches n_partials CTAs */
  int32_t n_other;            /* rows on the non-key side (n_src in the forward, n_dst in the backward): extent of the
                                 tensor maps the backward builds over x_src / grad_x1                              */
} GrlFusedEdgeDesc;
/* partial layout: gWk[64][64] | gW1b[64][16] (columns 0..13 = gW1, column 14 = gb1) | gW2[64][64] | gb2[64] */
#define GRL_FUSED_EDGE_GRAD_FLOATS (64 * 64 + 64 * 16 + 64 * 64 + 64)
int grl_fbconv_edge_fused_fwd(const GrlFusedEdgeDesc* d, grl_stream_t stream);
int grl_fbconv_edge_fused_bwd(const GrlFusedEdgeDesc* d, grl_stream_t stream);

/* *out_bits = bit pattern of max_i |x[i]| (NaNs ignored); feeds GrlConvDesc.grad_amax.  x must be 16-byte aligned. */
int grl_absmax(const float* x, int64_t n, uint32_t* out_bits, grl_stream_t stream);

/* out[i] = sum_p partials[p][i], fixed order (deterministic cross-CTA reduction). */
int grl_reduce_partials(const float* partials, int n_partials, int64_t n_floats, float* out, int accumulate,
                        grl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * V1  DeepSets critic, inner per-token MLP up to the pooled sum: replaces the first Linear, PyG LayerNorm(mode='graph'),
 * ReLU and the token sum of geometry_rl/modules/pyg_models/deepsets.py:34-53 (mlp_inner.lins.0, mlp_inner.norms.0,
 * x.sum(dim=1)).  The inner MLP's second Linear commutes with the sum and is applied by the caller on [B][64]:
 *   ysum[b] = sum_n relu(((x[b][n] W1^T + b1) - mean) / (std + eps) * gamma + beta)
 * with mean / biased std over the WHOLE [B][N][64] pre-activation tensor (LayerNorm mode 'graph', batch=None) — of all
 * ranks under data parallelism: `stats` / `bstats` are two doubles the caller all-reduces between the two passes of
 * each direction, `count` is the GLOBAL element count.  No [B N][64] activation is ever written: every pass recomputes
 * the pre-activations from x (4 F bytes per token).
 *   forward : grl_critic_inner_stats (-> stats = (sum h, sum h^2)), [all-reduce], grl_critic_inner_fwd (-> ysum)
 *   backward: grl_critic_inner_bwd_stats (-> bstats = (sum g_xhat, sum g_xhat xhat), g_gamma, g_beta partials),
 *             [all-reduce], grl_critic_inner_bwd (-> g_b1, g_W1 partials)
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t n_graphs, n_tokens, n_feat, n_partials; /* n_feat <= 16; n_partials <= n_graphs CTAs, one partial slot each    */
  float eps;
  double count;            /* number of elements of the [B][N][64] tensor over ALL ranks                              */
  const float* x;          /* [B][N][F]                                                                                */
  const float* w1;         /* [64][F] row-major (mlp_inner.lins.0.weight)                                              */
  const float* b1;         /* [64]                                                                                     */
  const float* gamma;      /* [64] mlp_inner.norms.0.weight                                                            */
  const float* beta;       /* [64] mlp_inner.norms.0.bias                                                              */
  double* stats;           /* [2] (sum h, sum h^2): written by _stats for this rank's rows, read by the other passes   */
  double* stat_partials;   /* [n_partials][2] workspace                                                                */
  float* ysum;             /* [B][64]                                                                                  */
  const float* grad_ysum;  /* [B][64]                                                                                  */
  double* bstats;          /* [2] (S1, S2): written by _bwd_stats, read by _bwd                                        */
  float* grad_partials;    /* [n_partials][GRL_CRITIC_GRAD_FLOATS]                                                     */
} GrlCriticDesc;
/* partial layout: g_gamma[64] | g_beta[64] | g_b1[64] | g_W1[64][16] (columns >= F are zero) */
#define GRL_CRITIC_GRAD_FLOATS (3 * 64 + 64 * 16)
int grl_critic_inner_stats(const GrlCriticDesc* d, grl_stream_t stream);
int grl_critic_inner_fwd(const GrlCriticDesc* d, grl_stream_t stream);
int grl_critic_inner_bwd_stats(const GrlCriticDesc* d, grl_stream_t stream);
int grl_critic_inner_bwd(const GrlCriticDesc* d, grl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * M4  Equivariant readout of the output-node latents: replaces hepi.py:173-190 / ponita_gcn.py:132-146 with
 * ponita/utils/to_from_sphere.py:12-17: decoder Linear(64 -> od + odv) per orientation, orientation means,
 * vector readout against the orientation grid, gating by the scalar readout, z = 0 padding in 2-D.
 * ------------------------------------------------------------------------------------------ */
#define GRL_READOUT_MAX_OUT 8 /* od + odv */
typedef struct {
  int32_t n_nodes, od, odv, dim;
  const float* latent;     /* [n][16][64]                                                         */
  const float* weight;     /* [od + odv][64] decoder nn.Linear.weight                             */
  const float* bias;       /* [od + odv]                                                          */
  const float* ori;        /* [16][3] (z = 0 when dim == 2)                                       */
  float* out;              /* [n][odv][3]                                                         */
  float* hidden;           /* [n][64] mean over orientations                                      */
  /* backward */
  const float* grad_out;   /* [n][odv][3]                                                         */
  const float* grad_hidden;/* optional [n][64]                                                    */
  float* grad_latent;      /* [n][16][64]                                                         */
  float* grad_partials;    /* [n_partials][(od + odv) * 64 + od + odv]: gW | gb per CTA           */
  int32_t n_partials;
} GrlReadoutDesc;
int grl_readout_fwd(const GrlReadoutDesc* d, grl_stream_t stream);
int grl_readout_bwd(const GrlReadoutDesc* d, grl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K5  One post-LN transformer encoder layer over the tokens of a graph (transformer baseline, M6): replaces the
 * nn.TransformerEncoderLayer(d_model = 64, nhead = 2, dim_feedforward = 64, dropout = 0, ReLU) call of
 * modules/pyg_models/transformer_vanilla.py:30-36,76-92 — ~30 library launches per layer and direction (in/out
 * projections, batched QK^T, softmax, PV, two LayerNorms, the feed-forward pair, residual adds) — by one kernel per
 * direction.  Tokens are batch-major [n_graphs][n_tokens][64]; parameters in torch's layouts.  The backward
 * recomputes the layer's forward from x and leaves the parameter gradients in one partial slot per CTA.
 * ------------------------------------------------------------------------------------------ */
#define GRL_ENCODER_MAX_TOKENS 56
/* partial layout: gWqkv[192][64] | gbqkv[192] | gWo[64][64] | gbo[64] | gW1[64][64] | gb1[64] | gW2[64][64] | gb2[64] |
 *                 g_norm1.weight[64] | g_norm1.bias[64] | g_norm2.weight[64] | g_norm2.bias[64]                        */
#define GRL_ENCODER_GRAD_FLOATS (192 * 64 + 192 + 3 * (64 * 64 + 64) + 4 * 64)
typedef struct {
  int32_t n_graphs, n_tokens, n_partials;
  const float* x;                /* [n_graphs][n_tokens][64] layer input                                          */
  const float* in_proj_weight;   /* [192][64] self_attn.in_proj_weight (q | k | v rows)                           */
  const float* in_proj_bias;     /* [192]                                                                         */
  const float* out_proj_weight;  /* [64][64]  self_attn.out_proj.weight                                           */
  const float* out_proj_bias;    /* [64]                                                                          */
  const float* linear1_weight;   /* [64][64]                                                                      */
  const float* linear1_bias;     /* [64]                                                                          */
  const float* linear2_weight;   /* [64][64]                                                                      */
  const float* linear2_bias;     /* [64]                                                                          */
  const float* norm1_weight;     /* [64]                                                                          */
  const float* norm1_bias;
  const float* norm2_weight;
  const float* norm2_bias;
  float* out;                    /* forward out: [n_graphs][n_tokens][64]                                         */
  const float* grad_out;         /* backward in                                                                   */
  float* grad_x;                 /* backward out                                                                  */
  float* grad_partials;          /* [n_partials][GRL_ENCODER_GRAD_FLOATS]; the backward launches n_partials CTAs   */
} GrlEncoderDesc;
int grl_encoder_layer_fwd(const GrlEncoderDesc* d, grl_stream_t stream);
int grl_encoder_layer_bwd(const GrlEncoderDesc* d, grl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K3  GAE: replaces torchrl.objectives.value.GAE(...)(data) at examples/torchrl/train.py:134-140,
 * 249-252 (the advantage arithmetic; the critic call stays with the caller).
 * reward/done/terminated [B][T], value [B][T+1] (shifted=True layout) -> adv, value_target [B][T].
 * ------------------------------------------------------------------------------------------ */
int grl_gae_scan(const float* reward, const float* value_T1, const uint8_t* done, const uint8_t* terminated,
                 float gamma, float lmbda, int B, int T, float* advantage, float* value_target, grl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * A1  Rollout-time Gaussian head + sampling: replaces the eager ProbabilisticActor call of the collector
 * (examples/torchrl/train.py, SyncDataCollector(policy=actor)): the head of
 * models/policy/gnn_gaussian_policy_diag.py:26-87 (_mean, _pre_std, softplus, square), torch.randn, log_prob and
 * diag_embed, one warp per sample.  Noise is counter-based Philox4x32-10 keyed by state[0] (seed) and the rank, with
 * state[1] (the call counter) in the counter; grl_act_advance increments state[1].  The draw of a component depends
 * on (seed, rank, call, sample, component) only.  Bit-level mapping: geometry_rl_b200/csrc/grl_act.cu.
 * ------------------------------------------------------------------------------------------ */
#define GRL_ACT_MAX_K 32 /* k = num_rows * action_dim components per sample */
typedef struct {
  int32_t batch;           /* B samples                                                                          */
  int32_t num_rows;        /* A actuator rows per sample                                                         */
  int32_t action_dim;      /* a components per row (k = A a <= GRL_ACT_MAX_K)                                     */
  int32_t hidden_dim;      /* must be 64                                                                         */
  int32_t post_fc;         /* 1: mean = hidden _mean.weight^T + _mean.bias; 0: mean given                          */
  int32_t contextual_std;  /* 1: pre = hidden _pre_std.weight^T + _pre_std.bias; 0: pre = std_weight (shared)        */
  int32_t use_tanh_mean;   /* loc = tanh(mean)                                                                   */
  int32_t deterministic;   /* action = loc, eps = 0 (evaluation / play); draws nothing                             */
  int32_t rank;            /* data-parallel rank: enters the Philox key                                           */
  float pre_shift;         /* _pre_activation_shift                                                              */
  float minimal_std;
  const float* hidden;     /* [B*A][64] (post_fc or contextual std; else may be NULL)                              */
  const float* mean;       /* [B][k] body mean rows (post_fc == 0)                                               */
  const float* mean_weight;/* [a][64] (post_fc)                                                                  */
  const float* mean_bias;  /* [a]     (post_fc)                                                                  */
  const float* std_weight; /* [a][64] contextual, [a] shared _pre_std                                             */
  const float* std_bias;   /* [a] (contextual)                                                                   */
  const int64_t* state;    /* [2] {seed, call counter}                                                            */
  float* loc;              /* [B][k]                                                                             */
  float* cov;              /* [B][k][k]: diagonal var, off-diagonal entries exact zeros                            */
  float* action;           /* [B][k]                                                                             */
  float* log_prob;         /* [B]                                                                                */
  float* eps;              /* optional [B][k]: the standard normals drawn                                          */
} GrlActDesc;
int grl_gaussian_act(const GrlActDesc* d, grl_stream_t stream);
/* state[1] += 1 (one thread). */
int grl_act_advance(int64_t* state, grl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * K4  TRPL projection of a diagonal Gaussian (mean + "std := cov" diagonal v):
 * replaces projections/kl_projection_layer.py:15-111,162-204 (ITPAL cpp_projection on the CPU),
 * projections/w2_projection_layer.py:15-68, base_projection_layer.py:71-100.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t batch, k;
  int32_t proj_type;      /* 0 = KL, 1 = W2 (commuting, scale_prec = True)                      */
  float eps_mean, eps_cov;
  const float* mean;      /* [B][k]                                                             */
  const float* v;         /* [B][k] diagonal of the matrix the reference calls "std"            */
  const float* old_mean;  /* [B][k]                                                             */
  const float* old_v;     /* [B][k]                                                             */
  float* proj_mean;       /* [B][k]                                                             */
  float* proj_v;          /* [B][k]                                                             */
  double* eta;            /* [B][2] saved (cov dual eta | W2 weight, mean omega); 0 = inactive  */
  /* backward */
  const float* grad_proj_mean; /* [B][k]                                                        */
  const float* grad_proj_v;    /* [B][k]                                                        */
  float* grad_mean;            /* [B][k]                                                        */
  float* grad_v;               /* [B][k]                                                        */
  const float* grad_mean_add;  /* optional [B][k]: added to grad_mean (gradient reaching `mean` directly)   */
  const float* grad_v_add;     /* optional [B][k]: added to grad_v                                          */
} GrlProjDesc;
int grl_trpl_fwd(const GrlProjDesc* d, grl_stream_t stream);
int grl_trpl_bwd(const GrlProjDesc* d, grl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * L1/P3  TRPL loss terms around the projection: replaces the ~170 elementwise / reduction launches of
 * objectives/trpl.py:231-321 (advantage standardisation :286-289, log-weight :246-251, surrogate :303,
 * entropy bonus :310-312, ESS :294-300, log_tr_metrics :255-273) and of
 * projections/base_projection_layer.py:292-327 (get_trust_region_loss), :332-384 (compute_metrics) with
 * utils/projection_utils.py:34-67,107-149 (gaussian_kl / gaussian_wasserstein_commutative) and the policy's
 * entropy (gnn_gaussian_policy_diag.py:117-137), for diagonal Gaussians under "std := covariance diagonal".
 * Per-sample terms are evaluated in fp64 and summed in a fixed order by one CTA (deterministic).
 * Data parallel (SURVEY 8(e)): the cross-sample reductions must be global.  grl_trpl_loss_fwd runs in three stages
 * (GrlLossDesc.stage: 0 = all, single process) between which the caller all-reduces a few doubles:
 *   stage 1  per-sample terms; stats[0:3] = (sum A, sum A^2, n), stats[3] = max log_w     -> SUM stats[0:3], MAX stats[3]
 *   stage 2  sums[0:3] this rank's loss sums, sums[3:10] metric sums, sums[10:12] maxima   -> SUM sums[3:10], MAX sums[10:12]
 *   stage 3  scalars (losses = local sum / global count, metrics global)
 * ------------------------------------------------------------------------------------------ */
#define GRL_LOSS_TERMS 8    /* doubles per sample in GrlLossDesc.terms */
#define GRL_LOSS_SCALARS 16 /* floats in GrlLossDesc.scalars */
#define GRL_LOSS_STATS 8    /* doubles in GrlLossDesc.stats */
#define GRL_LOSS_SUMS 16    /* doubles in GrlLossDesc.sums */
enum {
  GRL_LS_LOSS_OBJECTIVE = 0, /* -mean(exp(log_w) * A_hat)                                   trpl.py:303      */
  GRL_LS_LOSS_TRUST_REGION,  /* coeff * mean(mean_part + cov_part)(p || proj.detach())      base:292-327     */
  GRL_LS_LOSS_ENTROPY,       /* -entropy_coef * mean(H[N(proj)])                            trpl.py:310-312  */
  GRL_LS_DIST_ENTROPY,       /* mean(H[N(proj_mean, diag(proj_v))])                                          */
  GRL_LS_ESS,                /* exp(2 lse(log_w) - lse(2 log_w)) / B                        trpl.py:294-300  */
  GRL_LS_KL,                 /* mean gaussian_kl(p, proj) (mean + cov part)                 base:355-369     */
  GRL_LS_CONSTRAINT,         /* mean trust_region_value(p, proj) (mean + cov part)                           */
  GRL_LS_MEAN_CONSTRAINT, GRL_LS_MEAN_CONSTRAINT_MAX, GRL_LS_COV_CONSTRAINT, GRL_LS_COV_CONSTRAINT_MAX,
  GRL_LS_ENTROPY,            /* mean policy.entropy(p)                                                        */
  GRL_LS_ENTROPY_DIFF        /* mean(policy.entropy(proj) - policy.entropy(p))                                */
};
typedef struct {
  int32_t batch, k;
  int32_t proj_type;          /* trust_region_value: 0 = gaussian_kl, 1 = commuting W2 with scale_prec       */
  int32_t normalize_advantage;
  float entropy_coef, trust_region_coeff;
  const float* mean;          /* [B][k] current policy p                                                     */
  const float* v;             /* [B][k]                                                                      */
  const float* proj_mean;     /* [B][k] grl_trpl_fwd outputs                                                 */
  const float* proj_v;        /* [B][k]                                                                      */
  const float* action;        /* [B][k]                                                                      */
  const float* prev_log_prob; /* [B]                                                                         */
  const float* advantage;     /* [B] un-normalised                                                           */
  double* terms;              /* [B][GRL_LOSS_TERMS] workspace: written by fwd, read by bwd                  */
  double* stats;              /* [GRL_LOSS_STATS] (sum A, sum A^2, n, max log_w, loc, 1/scale): fwd writes, bwd reads */
  float* scalars;             /* [GRL_LOSS_SCALARS] outputs, GRL_LS_* order                                  */
  /* backward */
  const float* grad_losses;   /* [3] upstream gradients of (loss_objective, loss_trust_region, loss_entropy) */
  float* grad_proj_mean;      /* [B][k] -> GrlProjDesc.grad_proj_mean                                        */
  float* grad_proj_v;         /* [B][k] -> GrlProjDesc.grad_proj_v                                           */
  float* grad_mean_direct;    /* [B][k] -> GrlProjDesc.grad_mean_add (trust-region loss reaches p directly)  */
  float* grad_v_direct;       /* [B][k] -> GrlProjDesc.grad_v_add                                            */
  /* staged forward (data parallel) */
  double* sums;               /* [GRL_LOSS_SUMS] workspace between stages 2 and 3                            */
  int32_t stage;              /* 0 = stages 1-3 in one call, else 1 | 2 | 3                                  */
} GrlLossDesc;
int grl_trpl_loss_fwd(const GrlLossDesc* d, grl_stream_t stream);
int grl_trpl_loss_bwd(const GrlLossDesc* d, grl_stream_t stream);
/* Data-parallel glue of the staged forward: `gathered` is the all-gather [world][n] (n <= 32 doubles per rank) of a
 * statistics slice; out[i] = sum over ranks for i < n_sum, max over ranks for i >= n_sum, ranks visited in rank order
 * (bit-identical on every rank).  ONE all-gather + this per stage replaces a SUM and a MAX all-reduce. */
int grl_dp_combine(const double* gathered, int world, int n, int n_sum, double* out, grl_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Tensor-core building-block self-test: D[128][N] = bf16(A[128][K]) * bf16(B[N][K])^T, fp32 accumulate in
 * TMEM (tcgen05.mma kind::f16).  (N,K) in {(64,16),(64,64),(256,64),(64,256)}.  Test hook only.
 * ------------------------------------------------------------------------------------------ */
int grl_tc_selftest_gemm(const float* A, const float* B, float* D, int N, int K, grl_stream_t stream);
/* The same with the A operand fed from tensor memory (TS mode: tcgen05.st of packed fp16 pairs, lane = row), N = 64,
 * K in {64, 256}.  Pins the TMEM operand layout the kernels rely on. */
int grl_tc_selftest_gemm_ts(const float* A, const float* B, float* D, int K, grl_stream_t stream);
/* Raw hook behind tests/test_gpu_tc.py's layout probes: the caller supplies the bf16 shared-memory images of
 * both operands and every descriptor field (byte offsets, per-K-step advance, instruction descriptor). */
int grl_tc_debug_mma(const void* a_img, int a_bytes, const void* b_img, int b_bytes, float* D, int N, int n_ksteps,
                     uint32_t lbo_a, uint32_t sbo_a, uint32_t adv_a, uint32_t lbo_b, uint32_t sbo_b, uint32_t adv_b,
                     uint32_t idesc, uint32_t desc_hi_bits, grl_stream_t stream);
/* Hand-off latency probe (SM clock cycles): out64[2 i], out64[2 i + 1] = min, mean of measurement i, 9 measurements
 * (MMA + commit -> wait for 1/4/8/16 MMAs, fence.proxy.async, mbarrier arrive -> wait, tcgen05.ld, epilogue <-> MMA-warp
 * round trips); out64 must hold 64 entries.  Measurement hook only (tools/tc_latency_probe.py, DESIGN.md). */
int grl_tc_latency_probe(long long* out64, grl_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GRL_B200_H_ */
