"""torch.autograd wrappers around the C-ABI kernels (host side of the hot path).

Everything here is plumbing: tensor allocation, weight re-packing, descriptor filling and the
autograd graph.  All arithmetic on latents / edges happens inside libgrl_b200.so; there is no
eager fallback — tensors must live on a CUDA device.
"""
import ctypes as C
import os
from dataclasses import dataclass
from typing import Optional

import torch

from . import _lib as L

ROW = 16 * 64

# Precision of the nn.Linear contractions inside the message-passing kernels (north_star):
#   "fp32": FFMA kernels, parity 1e-5 against the reference's fp32 CPU results (default)
#   "bf16": tcgen05 tensor-core kernels, bf16 operands / fp32 accumulation, parity 1e-2
_PRECISION = "fp32"
# debugging aid for error attribution: which halves of the bf16 path use the tensor-core kernels ("node", "edge")
_TC_PARTS = set(os.environ.get("GRL_TC_PARTS", "node,edge").split(","))
# 16-bit path: recompute the edge basis inside the edge kernels (grl_fbconv_edge_fused_*) instead of materialising an
# [E,16,64] basis and its gradient in HBM.  GRL_FUSED_EDGE=0 (or set_fused_edge(False)) selects the round-1 kernels
# (grl_edge_basis_*_tc + grl_fbconv_edge_*_tc), kept as the parity partner of the fused ones in the tests.
_FUSED_EDGE = os.environ.get("GRL_FUSED_EDGE", "1") != "0"


def set_precision(mode: str):
    global _PRECISION
    if mode not in ("fp32", "bf16"):
        raise ValueError("precision must be 'fp32' or 'bf16'")
    _PRECISION = mode


def get_precision() -> str:
    return _PRECISION


def set_fused_edge(on: bool):
    global _FUSED_EDGE
    _FUSED_EDGE = bool(on)


def fused_edge_enabled() -> bool:
    return _PRECISION == "bf16" and _FUSED_EDGE and "edge" in _TC_PARTS and "node" in _TC_PARTS


# std() used by the one-time kernel calibration (conv.py:151-157, ponita.py:178-192).  Single process: torch's own
# Tensor.std(), exactly like the reference.  Data parallel: DataParallel.attach installs a global version (moments
# all-reduced over the ranks), so every replica derives the same scaling factors from the whole minibatch.
_CALIBRATION_STD = None


def set_calibration_std(fn):
    global _CALIBRATION_STD
    _CALIBRATION_STD = fn


def calibration_std(x: torch.Tensor) -> torch.Tensor:
    return x.std() if _CALIBRATION_STD is None else _CALIBRATION_STD(x)


def _f32c(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


# ------------------------------------------------------------------------------------------------
# K1: edge construction and CSR
# ------------------------------------------------------------------------------------------------
@dataclass
class EdgeSet:
    """One edge type of a batched graph, in the layouts the kernels consume.

    `coo` keeps the reference's coalesced [2, E] int64 edge_index (parity artefact, rows = source,
    target); everything else is in "edge order" = dst-sorted CSR order with ties in COO order."""
    n_src: int
    n_dst: int
    n_edges: int
    coo: torch.Tensor
    edge_ptr: torch.Tensor  # [B+1] int64
    rowptr_dst: torch.Tensor  # [n_dst+1] int32
    edge_src: torch.Tensor  # [E] int32
    edge_dst: torch.Tensor  # [E] int32
    eid_coo: torch.Tensor  # [E] int32: edge order -> COO position
    rowptr_src: torch.Tensor  # [n_src+1] int32
    src_eid: torch.Tensor  # [E] int32: src-sorted entry -> edge-order position
    s_src: Optional[torch.Tensor] = None  # [E] int32: source of the q-th src-sorted entry (lazy, see src_sorted_pairs)
    s_dst: Optional[torch.Tensor] = None  # [E] int32: destination of the q-th src-sorted entry
    # False: a fixed-capacity set (refresh_edge_set rewrites it in place on the device, no host sync).  Every array is
    # sized for `n_edges` = capacity; the real count is rowptr_dst[-1] (device only), and past it coo, edge_src, eid_coo and
    # src_eid hold 0 (edge_dst, s_src, s_dst the node ids those zeros point at), so every gather stays in bounds.  Only
    # the fused 16-bit kernels, which walk the CSR row pointers, accept such a set (`require_exact` guards the others).
    exact: bool = True


def require_exact(es: "EdgeSet", what: str) -> None:
    """Refuse a fixed-capacity edge set in a consumer that visits all `n_edges` rows (strict fp32 kernels, the
    materialised basis, the homogeneous view): the padding rows would enter its sums."""
    if not es.exact:
        raise ValueError(f"{what} needs an exact-size edge set; fixed-capacity (in-place refreshed) topology is consumed "
                         "by the fused 16-bit edge kernels only (ops.set_precision('bf16'), fused edge path)")


def exact_edge_set(es: "EdgeSet") -> "EdgeSet":
    """The real-count prefix of a fixed-capacity edge set as an exact one (reads the count: one host sync).  Edges
    [0, rowptr_dst[-1]) of the edge order are exactly the real ones, and the src-sorted entries point into them."""
    if es.exact:
        return es
    E = int(es.rowptr_dst[-1].item())
    return EdgeSet(es.n_src, es.n_dst, E, es.coo[:, :E], es.edge_ptr, es.rowptr_dst, es.edge_src[:E], es.edge_dst[:E],
                   es.eid_coo[:E], es.rowptr_src, es.src_eid[:E])


@dataclass
class SubEdgeSet:
    """The edges of a homogeneous `EdgeSet` that END in a given set of nodes (`out_ids`), as a bipartite set
    "all nodes -> those nodes" for a layer whose result is only read there (the last EMPN layer).

    Forward arrays are contiguous in sub-edge order (= the parent's dst-sorted order restricted to the subset, so the
    segmented sums add the same edges in the same order); the backward walks the subset in src-sorted order and
    addresses the PARENT's per-edge arrays (basis, basis gradient, edge_src) through `src_eid_parent`."""
    n_src: int
    n_dst: int  # = len(out_ids)
    n_edges: int
    out_ids: torch.Tensor  # [n_dst] int64, ascending: row of the parent's node tensor behind every dst row
    eids: torch.Tensor  # [E_sub] int64, ascending: position of every sub-edge in the parent's edge order
    eids32: torch.Tensor  # the same as int32 (GrlConvDesc.basis_row of the tensor-core forward)
    rowptr_dst: torch.Tensor  # [n_dst+1] int32
    edge_src: torch.Tensor  # [E_sub] int32 (parent node ids)
    edge_dst: torch.Tensor  # [E_sub] int32 (0..n_dst-1)
    rowptr_src: torch.Tensor  # [n_src+1] int32
    src_eid_parent: torch.Tensor  # [E_sub] int32: src-sorted entry -> position in the PARENT's edge order
    edge_dst_parent: torch.Tensor  # [E_parent] int32: dst rank (0..n_dst-1) of every parent edge, -1 outside the subset
    s_src: Optional[torch.Tensor] = None  # [E_sub] int32: source (parent node id) of the q-th src-sorted sub-edge (lazy)
    s_dst: Optional[torch.Tensor] = None  # [E_sub] int32: destination rank of the q-th src-sorted sub-edge


def src_sorted_pairs(es: "EdgeSet", sub: Optional[SubEdgeSet] = None):
    """(s_src, s_dst): endpoints of the src-sorted entry list as two plain arrays, so the fused backward kernel walks it
    without dependent index loads.  Derived once per topology and cached on the edge set."""
    top = sub if sub is not None else es
    if top.s_src is None:
        if sub is None:
            idx = es.src_eid.long()
            top.s_src, top.s_dst = es.edge_src[idx].contiguous(), es.edge_dst[idx].contiguous()
        else:
            idx = sub.src_eid_parent.long()
            top.s_src, top.s_dst = es.edge_src[idx].contiguous(), sub.edge_dst_parent[idx].contiguous()
    return top.s_src, top.s_dst


def build_sub_edge_set(es: "EdgeSet", out_ids: torch.Tensor) -> SubEdgeSet:
    assert es.n_src == es.n_dst, "sub edge sets are derived from homogeneous graphs"
    require_exact(es, "build_sub_edge_set")
    dev = es.edge_src.device
    n_out = int(out_ids.numel())
    rank = torch.full((es.n_dst,), -1, dtype=torch.int64, device=dev)
    rank[out_ids] = torch.arange(n_out, device=dev)
    dst_rank = rank[es.edge_dst.long()]
    eids = (dst_rank >= 0).nonzero().squeeze(1)
    edge_src = es.edge_src[eids].contiguous()
    edge_dst = dst_rank[eids].to(torch.int32).contiguous()

    def rowptr(keys, n):
        rp = torch.zeros(n + 1, dtype=torch.int64, device=dev)
        rp[1:] = torch.cumsum(torch.bincount(keys.long(), minlength=n), 0)
        return rp.to(torch.int32).contiguous()

    order = torch.sort(edge_src.long(), stable=True).indices  # ties keep edge order, like grl_csr_build
    return SubEdgeSet(es.n_src, n_out, int(eids.numel()), out_ids.contiguous(), eids.contiguous(),
                      eids.to(torch.int32).contiguous(), rowptr(edge_dst, n_out), edge_src, edge_dst,
                      rowptr(edge_src, es.n_src), eids[order].to(torch.int32).contiguous(),
                      dst_rank.to(torch.int32).contiguous())


def knn_edge_ptr(num_valid: Optional[torch.Tensor], B: int, P: int, k: int, device) -> torch.Tensor:
    edge_ptr = torch.empty(B + 1, dtype=torch.int64, device=device)
    L.call("grl_knn_edge_ptr", L.ptr(num_valid), B, P, k, L.ptr(edge_ptr))
    return edge_ptr


def knn_graph(pos: torch.Tensor, num_valid: Optional[torch.Tensor], k: int):
    """pos [B,P,3] fp32 -> (coo [2,E] int64 coalesced, edge_ptr [B+1])."""
    pos = _f32c(pos)
    B, P, _ = pos.shape
    if num_valid is not None:
        num_valid = num_valid.to(torch.int32).clamp(0, P).contiguous()  # the kernels clamp too: keep the edge counts in step
    if not bool(torch.isfinite(pos).all()):  # a NaN distance never wins a comparison: edge_ptr would count edges that are not written
        raise ValueError("knn_graph: non-finite positions (topology is built off the step path, so this check is free)")
    edge_ptr = knn_edge_ptr(num_valid, B, P, k, pos.device)
    E = int(edge_ptr[-1].item())  # topology is built once per batch size; this sync is off the step path
    coo = torch.empty(2, max(E, 1), dtype=torch.int64, device=pos.device)
    if E > 0:
        L.call("grl_knn_graph", L.ptr(pos), L.ptr(num_valid), L.ptr(edge_ptr), B, P, k, L.ptr(coo), coo.stride(0))
    return coo[:, :E], edge_ptr


def radius_neighbors(pos: torch.Tensor, num_valid: Optional[torch.Tensor], radius: float, max_neighbors: int):
    pos = _f32c(pos)
    B, P, _ = pos.shape
    if num_valid is not None:
        num_valid = num_valid.to(torch.int32).contiguous()
    nbr = torch.empty(B, P, max_neighbors, dtype=torch.int32, device=pos.device)
    cnt = torch.empty(B, P, dtype=torch.int32, device=pos.device)
    L.call("grl_radius_neighbors", L.ptr(pos), L.ptr(num_valid), B, P, float(radius), max_neighbors, L.ptr(nbr),
           L.ptr(cnt))
    return nbr, cnt


def radius_graph(pos: torch.Tensor, num_valid: Optional[torch.Tensor], radius: float, max_num_neighbors: int,
                 capacity: Optional[int] = None):
    """pos [B,P,3] fp32 -> (coo [2,E] int64 coalesced, edge_ptr [B+1]): the radius graph of every point set.

    Neighbours of centre i are the points j != i of the first num_valid[b] with sqdist <= radius^2 (the rounding of
    knn_graph), at most `max_num_neighbors` nearest, ties to the lower index; row 0 = neighbour j (source), row 1 =
    centre i (target), sorted by (j, i) per graph.  A point with a non-finite coordinate has no edges.
    `capacity=None`: exact size (reads the count once, like knn_graph).  Otherwise no host sync: coo is
    [2, capacity] with the entries past edge_ptr[B] set to 0, and edges that do not fit are dropped (edge_ptr is
    clamped); `capacity=B * P * max_num_neighbors` can never drop one."""
    pos = _f32c(pos)
    B, P, _ = pos.shape
    nbr, cnt = radius_neighbors(pos, num_valid, radius, max_num_neighbors)
    edge_ptr = torch.empty(B + 1, dtype=torch.int64, device=pos.device)
    bound = B * P * max_num_neighbors
    L.call("grl_radius_edge_ptr", L.ptr(cnt), B, P, bound if capacity is None else int(capacity), L.ptr(edge_ptr))
    E = int(edge_ptr[-1].item()) if capacity is None else int(capacity)
    coo = torch.empty(2, max(E, 1), dtype=torch.int64, device=pos.device)
    L.call("grl_radius_graph", L.ptr(nbr), L.ptr(cnt), L.ptr(edge_ptr), B, P, max_num_neighbors, L.ptr(coo),
           coo.stride(0), coo.shape[1])
    return coo[:, :E], edge_ptr


def dense_edges(mode: int, B: int, n_src: int, n_dst: int, device, num_valid: Optional[torch.Tensor] = None,
                capacity: bool = False):
    """mode 0: ordered pairs j != k among n_src; mode 1: valid sources x all destinations.
    `capacity` (mode 1): no host sync; coo is [2, B * n_src * n_dst] with the entries past edge_ptr[B] set to 0."""
    if mode == 0:
        counts = torch.full((B,), n_src * (n_src - 1), dtype=torch.int64, device=device)
    else:
        nv = (num_valid.to(torch.int64).clamp(0, n_src) if num_valid is not None  # the kernel clamps to [0, n_src] as well
              else torch.full((B,), n_src, dtype=torch.int64, device=device))
        counts = nv * n_dst
    edge_ptr = torch.zeros(B + 1, dtype=torch.int64, device=device)
    edge_ptr[1:] = torch.cumsum(counts, 0)
    if capacity:
        assert mode == 1, "fixed-capacity dense edges are the TASK edges (mode 1)"
        E = B * n_src * n_dst
        coo = torch.zeros(2, E, dtype=torch.int64, device=device)
    else:
        E = int(edge_ptr[-1].item())
        coo = torch.empty(2, max(E, 1), dtype=torch.int64, device=device)
    if E > 0:
        nvp = num_valid.to(torch.int32).clamp(0, n_src).contiguous() if num_valid is not None else None
        L.call("grl_dense_edges", mode, L.ptr(nvp), L.ptr(edge_ptr), B, n_src, n_dst, L.ptr(coo), coo.stride(0))
    return coo[:, :E], edge_ptr


def _csr(coo: torch.Tensor, edge_ptr: torch.Tensor, B: int, n_key: int, key_row: int, out=None):
    """`out` = (rowptr, other, eid) to rewrite in place; their entries past edge_ptr[B] are zeroed first (the kernel
    writes the real edges only), so a gather through `other` / `eid` over the whole capacity stays in bounds."""
    E = coo.shape[1]
    dev = coo.device
    if out is None:
        rowptr = torch.zeros(B * n_key + 1, dtype=torch.int32, device=dev)
        other = torch.empty(max(E, 1), dtype=torch.int32, device=dev)
        eid = torch.empty(max(E, 1), dtype=torch.int32, device=dev)
    else:
        rowptr, other, eid = out
        other.zero_()
        eid.zero_()
    if E > 0:
        assert coo.stride(1) == 1
        L.call("grl_csr_build", L.ptr_any(coo), coo.stride(0), L.ptr(edge_ptr), B, n_key, key_row, L.ptr(rowptr),
               L.ptr(other), L.ptr(eid))
    return rowptr, other[:E], eid[:E]


def build_edge_set(coo: torch.Tensor, edge_ptr: torch.Tensor, B: int, n_src_per_graph: int,
                   n_dst_per_graph: int, exact: bool = True) -> EdgeSet:
    """dst-sorted CSR (edge order) and src-sorted CSR of a batched, graph-major COO.
    `exact=False`: `coo` is a fixed-capacity buffer (radius_graph / dense_edges with a capacity); the set's `n_edges` is
    the capacity, its real count rowptr_dst[-1], and it can be refreshed in place by `refresh_edge_set`."""
    E = coo.shape[1]
    if coo.stride(1) != 1:
        coo = coo.contiguous()

    def buffers(n_key):  # a capacity set gets zero tails (see _csr); a capacity is never 0
        if exact:
            return None
        z = lambda n: torch.zeros(n, dtype=torch.int32, device=coo.device)  # noqa: E731
        return z(B * n_key + 1), z(E), z(E)

    rowptr_dst, edge_src, eid_coo = _csr(coo, edge_ptr, B, n_dst_per_graph, 1, buffers(n_dst_per_graph))
    edge_dst = coo[1][eid_coo.long()].to(torch.int32) if E > 0 else edge_src.clone()
    coo2 = torch.stack([edge_src.long(), edge_dst.long()]) if E > 0 else coo
    rowptr_src, _, src_eid = _csr(coo2, edge_ptr, B, n_src_per_graph, 0, buffers(n_src_per_graph))
    return EdgeSet(B * n_src_per_graph, B * n_dst_per_graph, E, coo, edge_ptr, rowptr_dst, edge_src.contiguous(),
                   edge_dst.contiguous(), eid_coo.contiguous(), rowptr_src, src_eid.contiguous(), exact=exact)


def refresh_edge_set(es: EdgeSet, coo: torch.Tensor, edge_ptr: torch.Tensor) -> None:
    """Rewrite a fixed-capacity `EdgeSet` in place (same tensors, same addresses) from a new capacity COO / edge_ptr of
    the same shape, cached src-sorted pairs included.  Device work only (no host sync): valid inside a CUDA-graph
    capture, whose replays then rebuild the topology from whatever the inputs hold."""
    assert not es.exact and tuple(coo.shape) == tuple(es.coo.shape) and edge_ptr.shape == es.edge_ptr.shape
    B = es.edge_ptr.numel() - 1
    es.coo.copy_(coo)
    es.edge_ptr.copy_(edge_ptr)
    _csr(es.coo, es.edge_ptr, B, es.n_dst // B, 1, (es.rowptr_dst, es.edge_src, es.eid_coo))
    torch.index_select(es.coo[1], 0, es.eid_coo.long(), out=coo[1])  # coo is a scratch buffer from here on
    es.edge_dst.copy_(coo[1])
    coo[0].copy_(es.edge_src)
    _csr(coo, es.edge_ptr, B, es.n_src // B, 0,
         (es.rowptr_src, torch.empty_like(es.src_eid), es.src_eid))
    if es.s_src is not None:
        idx = es.src_eid.long()
        torch.index_select(es.edge_src, 0, idx, out=es.s_src)
        torch.index_select(es.edge_dst, 0, idx, out=es.s_dst)


# ------------------------------------------------------------------------------------------------
# partial-gradient helpers
# ------------------------------------------------------------------------------------------------
def _reduce(partials: torch.Tensor) -> torch.Tensor:
    n_p, n = partials.shape
    out = torch.empty(n, dtype=torch.float32, device=partials.device)
    L.call("grl_reduce_partials", L.ptr(partials), n_p, n, L.ptr(out), 0)
    return out


def _n_partials(n_units: int, per_sm: int = 1) -> int:
    return max(1, min(n_units, per_sm * L.sm_count()))


# ------------------------------------------------------------------------------------------------
# lift + node encoder
# ------------------------------------------------------------------------------------------------
class EmbedFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, scalars, vectors, weight, ori3, dim, node_ids=None):
        """`node_ids` (int32 [N]): embed rows node_ids[n] of the (padded) feature arrays as node n of a compact batch."""
        scalars, vectors, weight = _f32c(scalars), _f32c(vectors), _f32c(weight)
        N, S = (scalars.shape[0] if node_ids is None else int(node_ids.numel())), scalars.shape[1]
        V = vectors.shape[1] // 3
        assert weight.shape == (64, S + V), f"node encoder weight {tuple(weight.shape)} vs S+V={S + V}"
        x = torch.empty(N, 16, 64, dtype=torch.float32, device=scalars.device)
        d = L.GrlEmbedDesc(n_nodes=N, n_scalars=S, n_vectors=V, dim=dim, scalars=L.ptr(scalars), vectors=L.ptr(vectors),
                           ori=L.ptr(ori3), weight=L.ptr(weight), x=L.ptr(x), node_ids=L.ptr(node_ids))
        L.call("grl_embed_fwd", C.byref(d))
        ctx.save_for_backward(scalars, vectors, ori3)
        ctx.meta, ctx.node_ids = (N, S, V, dim), node_ids
        return x

    @staticmethod
    def backward(ctx, gx):
        scalars, vectors, ori3 = ctx.saved_tensors
        N, S, V, dim = ctx.meta
        gx = _f32c(gx)
        n_p = _n_partials((N + 15) // 16, 4 if S + V <= 8 else 2)  # resident CTAs per SM of grl_embed_bwd
        partials = torch.empty(n_p, 64 * (S + V), dtype=torch.float32, device=gx.device)
        d = L.GrlEmbedDesc(n_nodes=N, n_scalars=S, n_vectors=V, dim=dim, scalars=L.ptr(scalars), vectors=L.ptr(vectors),
                           ori=L.ptr(ori3), grad_x=L.ptr(gx), grad_weight_partials=L.ptr(partials), n_partials=n_p,
                           node_ids=L.ptr(ctx.node_ids))
        L.call("grl_embed_bwd", C.byref(d))
        return None, None, _reduce(partials).view(64, S + V), None, None, None


# ------------------------------------------------------------------------------------------------
# edge basis
# ------------------------------------------------------------------------------------------------
class EdgeBasisFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pos_src, pos_dst, w1, b1, w2, b2, ori3, dim, es: EdgeSet):
        require_exact(es, "the materialised edge basis")
        pos_src, pos_dst = _f32c(pos_src), _f32c(pos_dst)
        dev = pos_src.device
        w1t = torch.zeros(16, 64, dtype=torch.float32, device=dev)
        w1t[:14] = w1.detach().t()
        w2t = w2.detach().t().contiguous()
        b1c, b2c = _f32c(b1.detach()), _f32c(b2.detach())
        bf16 = _PRECISION == "bf16" and "edge" in _TC_PARTS
        basis = torch.empty(es.n_edges, 16, 64, dtype=torch.bfloat16 if bf16 else torch.float32, device=dev)
        d = L.GrlBasisDesc(n_edges=es.n_edges, dim=dim, edge_src=L.ptr(es.edge_src), edge_dst=L.ptr(es.edge_dst),
                           pos_src=L.ptr(pos_src), pos_dst=L.ptr(pos_dst), ori=L.ptr(ori3), w1t=L.ptr(w1t), b1=L.ptr(b1c),
                           w2t=L.ptr(w2t), b2=L.ptr(b2c), basis=None if bf16 else L.ptr(basis),
                           basis_bf16=L.ptr(basis) if bf16 else None)
        if es.n_edges > 0:
            L.call("grl_edge_basis_fwd_tc" if bf16 else "grl_edge_basis_fwd", C.byref(d),
                   shape=(es.n_src, es.n_dst, es.n_edges))
        ctx.save_for_backward(pos_src, pos_dst, w1t, b1c, w2t, b2c, _f32c(w2.detach()), ori3)
        ctx.es, ctx.dim = es, dim
        # One basis feeds every layer of the model.  Instead of letting autograd add the layers' [E,16,64] gradients
        # with a separate kernel, the first FiberConvFn.backward to run returns its gradient buffer and the later ones
        # accumulate into that same buffer inside the edge kernel (and return None).  This function's backward runs
        # after all of them (topological order), so it sees the complete sum whichever subset of consumers ran.
        ctx.gacc = {"buf": None, "mask": None}
        if bf16:
            basis._grl_gacc = ctx.gacc
        return basis

    @staticmethod
    def backward(ctx, g_basis):
        pos_src, pos_dst, w1t, b1c, w2t, b2c, w2, ori3 = ctx.saved_tensors
        es, dim = ctx.es, ctx.dim
        dev = pos_src.device
        pending_mask = ctx.gacc.get("mask")
        ctx.gacc["buf"], ctx.gacc["mask"] = None, None  # a later backward through the same graph starts a fresh accumulation
        if pending_mask is not None and g_basis is not None and es.n_edges > 0:
            # the only consumer was a sub layer: rows of the other edges were never written
            g_basis = g_basis.masked_fill((pending_mask < 0).view(-1, 1, 1), 0)
        if es.n_edges == 0:
            z = torch.zeros
            return (None, None, z(64, 14, device=dev), z(64, device=dev), z(64, 64, device=dev), z(64, device=dev),
                    None, None, None)
        bf16 = g_basis.dtype == torch.bfloat16
        g_basis = g_basis.contiguous() if bf16 else _f32c(g_basis)
        n_p = _n_partials((es.n_edges + 7) // 8, 2 if bf16 else 1)
        partials = torch.empty(n_p, L.BASIS_GRAD_FLOATS, dtype=torch.float32, device=dev)
        d = L.GrlBasisDesc(n_edges=es.n_edges, dim=dim, edge_src=L.ptr(es.edge_src), edge_dst=L.ptr(es.edge_dst),
                           pos_src=L.ptr(pos_src), pos_dst=L.ptr(pos_dst), ori=L.ptr(ori3), w1t=L.ptr(w1t), b1=L.ptr(b1c),
                           w2t=L.ptr(w2t), b2=L.ptr(b2c), w2=L.ptr(w2), grad_basis=None if bf16 else L.ptr(g_basis),
                           grad_basis_bf16=L.ptr(g_basis) if bf16 else None, grad_partials=L.ptr(partials), n_partials=n_p)
        L.call("grl_edge_basis_bwd_tc" if bf16 else "grl_edge_basis_bwd", C.byref(d), shape=(es.n_src, es.n_dst, es.n_edges))
        g = _reduce(partials)
        gw1 = g[:1024].view(64, 16)[:, :14].contiguous()
        gb1 = g[1024:1088]
        gw2 = g[1088:1088 + 4096].view(64, 64)
        gb2 = g[1088 + 4096:]
        return None, None, gw1, gb1, gw2, gb2, None, None, None


class BasisSpec:
    """What a fused convolution needs to recompute its edge basis per tile: positions of both endpoint sets and the
    `basis_fn` parameters (hepi.py:76-82).  Stands in for the [E,16,64] `kernel_basis` tensor on the fused path."""

    def __init__(self, pos_src, pos_dst, w1, b1, w2, b2, ori3, dim, es: EdgeSet):
        self.pos_src, self.pos_dst = _f32c(pos_src.detach()), _f32c(pos_dst.detach())
        self.w1, self.b1, self.w2, self.b2 = w1, b1, w2, b2
        self.ori3, self.dim, self.es = ori3, dim, es

    def on(self, es: EdgeSet) -> "BasisSpec":
        """The same basis over another edge set (the exact view of a fixed-capacity one, see exact_edge_set)."""
        return BasisSpec(self.pos_src, self.pos_dst, self.w1, self.b1, self.w2, self.b2, self.ori3, self.dim, es)

    def materialize(self) -> torch.Tensor:
        """The basis as a tensor (one-time calibration only, conv.py:151-157)."""
        return EdgeBasisFn.apply(self.pos_src, self.pos_dst, self.w1, self.b1, self.w2, self.b2, self.ori3, self.dim,
                                 self.es)


def edge_basis(pos_src, pos_dst, w1, b1, w2, b2, ori3, dim, es: EdgeSet):
    """kernel_basis of one edge type: a `BasisSpec` on the fused 16-bit path, the [E,16,64] tensor otherwise."""
    if fused_edge_enabled():
        return BasisSpec(pos_src, pos_dst, w1, b1, w2, b2, ori3, dim, es)
    return EdgeBasisFn.apply(pos_src, pos_dst, w1, b1, w2, b2, ori3, dim, es)


# ------------------------------------------------------------------------------------------------
# separable fibre-bundle convolution + ConvNeXt update
# ------------------------------------------------------------------------------------------------
class FusedFiberConvFn(torch.autograd.Function):
    """FiberConvFn with the edge basis recomputed inside the edge kernels (16-bit path): no basis tensor, no basis
    gradient tensor; the gradients of the basis MLP leave the edge backward kernel directly."""

    @staticmethod
    def forward(ctx, x_src, x_dst, pos_src, pos_dst, bw1, bb1, bw2, bb2, fk, wk, bias, ln_g, ln_b, w1, b1, w2, b2, ori3,
                dim, es: EdgeSet, sub: Optional[SubEdgeSet]):
        homo = x_dst is None
        x_src = _f32c(x_src)
        if sub is not None:
            assert homo and sub.n_src == es.n_src
            xd = x_src.index_select(0, sub.out_ids)
            pos_dst = pos_dst.index_select(0, sub.out_ids)
        else:
            xd = x_src if homo else _f32c(x_dst)
        top = sub if sub is not None else es
        assert x_src.shape[0] == top.n_src and xd.shape[0] == top.n_dst, "latent rows do not match the edge set"
        assert tuple(x_src.shape[1:]) == (16, 64) and tuple(w1.shape) == (256, 64) and tuple(w2.shape) == (64, 256)
        assert tuple(bw1.shape) == (64, 14) and tuple(bw2.shape) == (64, 64)
        dev = x_src.device
        pos_src, pos_dst = _f32c(pos_src), _f32c(pos_dst)
        bw1_c, bb1_c, bw2_c, bb2_c = _f32c(bw1.detach()), _f32c(bb1.detach()), _f32c(bw2.detach()), _f32c(bb2.detach())
        fk = _f32c(fk)
        wk_c, w1_c, w2_rm = _f32c(wk.detach()), _f32c(w1.detach()), _f32c(w2.detach())
        bias_c, lng_c, lnb_c = _f32c(bias.detach()), _f32c(ln_g.detach()), _f32c(ln_b.detach())
        b1_c, b2_c = _f32c(b1.detach()), _f32c(b2.detach())
        x1 = torch.empty(top.n_dst, 16, 64, dtype=torch.float32, device=dev)
        out = torch.empty(top.n_dst, 16, 64, dtype=torch.float32, device=dev)
        shape = (top.n_src, top.n_dst, top.n_edges)
        fd = L.GrlFusedEdgeDesc(n_key=top.n_dst, n_other=top.n_src, n_edges=top.n_edges, dim=dim, n_partials=0, rowptr=L.ptr(top.rowptr_dst),
                                e_src=L.ptr(top.edge_src), e_dst=L.ptr(top.edge_dst), pos_src=L.ptr(pos_src),
                                pos_dst=L.ptr(pos_dst), ori=L.ptr(ori3), w1=L.ptr(bw1_c), b1=L.ptr(bb1_c), w2=L.ptr(bw2_c),
                                b2=L.ptr(bb2_c), wk=L.ptr(wk_c), x_src=L.ptr(x_src), x1=L.ptr(x1))
        L.call("grl_fbconv_edge_fused_fwd", C.byref(fd), shape=shape)
        # the tensor-core node backward reads the pre-LayerNorm tensor instead of recomputing the fibre convolution
        x2 = torch.empty_like(x1) if any(ctx.needs_input_grad) else None
        d = L.GrlConvDesc(n_src=top.n_src, n_dst=top.n_dst, n_edges=top.n_edges, rowptr_dst=L.ptr(top.rowptr_dst),
                          x_src=L.ptr(x_src), x_dst=L.ptr(xd), fiber_kernel=L.ptr(fk), wk=L.ptr(wk_c), bias=L.ptr(bias_c),
                          ln_g=L.ptr(lng_c), ln_b=L.ptr(lnb_c), w1=L.ptr(w1_c), b1=L.ptr(b1_c), w2=L.ptr(w2_rm),
                          b2=L.ptr(b2_c), x1=L.ptr(x1), out=L.ptr(out), accumulate_out=0, x2=L.ptr(x2),
                          # operands of the strict kernels only; the descriptor check wants them non-null
                          wk_t=L.ptr(wk_c), w1_t=L.ptr(w1_c), w2_t=L.ptr(w1_c), w2_c=L.ptr(w1_c))
        L.call("grl_fbconv_node_fwd_tc", C.byref(d), shape=shape)
        ctx.save_for_backward(x_src, pos_src, pos_dst, bw1_c, bb1_c, bw2_c, bb2_c, fk, wk_c, bias_c, lng_c, lnb_c, w1_c,
                              b1_c, w2_rm, b2_c, x1, x2 if x2 is not None else x1, ori3)
        ctx.es, ctx.sub, ctx.homo, ctx.dim = es, sub, homo, dim
        return out

    @staticmethod
    def backward(ctx, g_out):
        (x_src, pos_src, pos_dst, bw1_c, bb1_c, bw2_c, bb2_c, fk, wk_c, bias_c, lng_c, lnb_c, w1_c, b1_c, w2_rm, b2_c, x1,
         x2, ori3) = ctx.saved_tensors
        es, sub, homo, dim = ctx.es, ctx.sub, ctx.homo, ctx.dim
        top = sub if sub is not None else es
        dev = x_src.device
        g_out = _f32c(g_out)
        g_x1, g_x2 = torch.empty_like(x1), torch.empty_like(x1)
        g_xsrc = torch.empty_like(x_src)
        shape = (top.n_src, top.n_dst, top.n_edges)
        n_pn = _n_partials((top.n_dst + 7) // 8)
        node_part = torch.empty(n_pn, L.NODE_GRAD_FLOATS, dtype=torch.float32, device=dev)
        amax = torch.empty(1, dtype=torch.int32, device=dev)  # bit pattern of max |grad_out| (fp16 gradient scale)
        L.call("grl_absmax", L.ptr(g_out), g_out.numel(), L.ptr(amax), shape=shape)
        d = L.GrlConvDesc(n_src=top.n_src, n_dst=top.n_dst, n_edges=top.n_edges, rowptr_dst=L.ptr(top.rowptr_dst),
                          x_src=L.ptr(x_src), fiber_kernel=L.ptr(fk), wk=L.ptr(wk_c), bias=L.ptr(bias_c), ln_g=L.ptr(lng_c),
                          ln_b=L.ptr(lnb_c), w1=L.ptr(w1_c), b1=L.ptr(b1_c), w2=L.ptr(w2_rm), x1=L.ptr(x1), x2=L.ptr(x2),
                          grad_out=L.ptr(g_out), grad_x1=L.ptr(g_x1), grad_x2=L.ptr(g_x2), grad_amax=L.ptr(amax),
                          node_grad_partials=L.ptr(node_part), n_partials_node=n_pn,
                          wk_t=L.ptr(wk_c), w1_t=L.ptr(w1_c), w2_c=L.ptr(w1_c))
        L.call("grl_fbconv_node_bwd_tc", C.byref(d), shape=shape)
        s_src, s_dst = src_sorted_pairs(es, sub)
        n_pe = _n_partials(top.n_src)
        edge_part = torch.empty(n_pe, L.FUSED_EDGE_GRAD_FLOATS, dtype=torch.float32, device=dev)
        fd = L.GrlFusedEdgeDesc(n_key=top.n_src, n_other=top.n_dst, n_edges=top.n_edges, dim=dim, n_partials=n_pe, rowptr=L.ptr(top.rowptr_src),
                                e_src=L.ptr(s_src), e_dst=L.ptr(s_dst), pos_src=L.ptr(pos_src), pos_dst=L.ptr(pos_dst),
                                ori=L.ptr(ori3), w1=L.ptr(bw1_c), b1=L.ptr(bb1_c), w2=L.ptr(bw2_c), b2=L.ptr(bb2_c),
                                wk=L.ptr(wk_c), x_src=L.ptr(x_src), grad_x1=L.ptr(g_x1), grad_x_src=L.ptr(g_xsrc),
                                grad_x_src_init=L.ptr(g_out) if (homo and sub is None) else None,
                                grad_partials=L.ptr(edge_part))
        L.call("grl_fbconv_edge_fused_bwd", C.byref(fd), shape=shape)
        g = _reduce(node_part)
        o = 0
        gw1 = g[o:o + 256 * 64].view(256, 64); o += 256 * 64
        gb1 = g[o:o + 256]; o += 256
        gw2 = g[o:o + 64 * 256].view(64, 256); o += 64 * 256
        gb2 = g[o:o + 64]; o += 64
        glng = g[o:o + 64]; o += 64
        glnb = g[o:o + 64]; o += 64
        gbias = g[o:o + 64]; o += 64
        gfk = g[o:o + 16 * 16 * 64].view(16, 16, 64)
        ge = _reduce(edge_part)
        gwk = ge[:4096].view(64, 64)
        gw1b = ge[4096:4096 + 1024].view(64, 16)
        g_bw1, g_bb1 = gw1b[:, :14].contiguous(), gw1b[:, 14].contiguous()
        g_bw2 = ge[5120:5120 + 4096].view(64, 64)
        g_bb2 = ge[9216:9280]
        g_xdst = None if homo else g_out
        if sub is not None:  # residual path of the output rows (out_ids are unique: plain read-modify-write)
            g_xsrc.index_copy_(0, sub.out_ids, g_xsrc.index_select(0, sub.out_ids) + g_out)
        return (g_xsrc, g_xdst, None, None, g_bw1, g_bb1, g_bw2, g_bb2, gfk, gwk, gbias, glng, glnb, gw1, gb1, gw2, gb2,
                None, None, None, None)


class FiberConvFn(torch.autograd.Function):
    """out = x_dst + MLP(LN(fibre(scatter(kernel(basis) * x_src[src])) + bias)).

    `x_dst is None` means a homogeneous graph (source and destination nodes are the same tensor).  With `sub`
    (homogeneous graphs only) the layer is evaluated at the rows `sub.out_ids` alone: `out` is [len(out_ids), 16, 64],
    only the edges ending there are visited, `basis` stays the parent's full [E, 16, 64] tensor."""

    @staticmethod
    def forward(ctx, x_src, x_dst, basis, fk, wk, bias, ln_g, ln_b, w1, b1, w2, b2, es: EdgeSet,
                sub: Optional[SubEdgeSet] = None):
        require_exact(es, "FiberConvFn (strict fp32 / materialised-basis convolution)")
        homo = x_dst is None
        x_src = _f32c(x_src)
        if sub is not None:
            assert homo and sub.n_src == es.n_src
            xd = x_src.index_select(0, sub.out_ids)
        else:
            xd = x_src if homo else _f32c(x_dst)
        precision = _PRECISION if "node" in _TC_PARTS else "fp32"
        basis_in_dtype = basis.dtype
        basis = basis.contiguous() if (precision == "bf16" and basis.dtype == torch.bfloat16) else _f32c(basis)
        fk = _f32c(fk)
        dev = x_src.device
        basis_full = basis
        # the tensor-core edge kernel reads the parent's basis rows in place (GrlConvDesc.basis_row); the strict fp32
        # kernel reads the basis contiguously in edge order and gets a compact copy of the subset's rows
        basis_row = sub.eids32 if (sub is not None and basis.dtype == torch.bfloat16) else None
        if sub is not None and basis_row is None:
            basis = basis.index_select(0, sub.eids)
        top = sub if sub is not None else es  # topology of the forward kernels
        assert x_src.shape[0] == top.n_src and xd.shape[0] == top.n_dst, "latent rows do not match the edge set"
        assert tuple(x_src.shape[1:]) == (16, 64) and tuple(w1.shape) == (256, 64) and tuple(w2.shape) == (64, 256)
        wk_d, w1_d, w2_d = wk.detach(), w1.detach(), w2.detach()
        wk_c = _f32c(wk_d)
        w1_c = _f32c(w1_d)
        tc_edge, tc_node = basis.dtype == torch.bfloat16, precision == "bf16"
        # transposed / chunked copies are operands of the strict FFMA kernels only (the tensor-core kernels stage the
        # row-major weights themselves)
        wk_t = wk_c if tc_edge else wk_d.t().contiguous()
        w1_t = w1_c if tc_node else w1_d.view(4, 64, 64).transpose(1, 2).contiguous()
        w2_t = w1_c if tc_node else w2_d.view(64, 4, 64).permute(1, 2, 0).contiguous()
        w2_c = w1_c if tc_node else w2_d.view(64, 4, 64).permute(1, 0, 2).contiguous()
        bias_c, lng_c, lnb_c = _f32c(bias.detach()), _f32c(ln_g.detach()), _f32c(ln_b.detach())
        b1_c, b2_c = _f32c(b1.detach()), _f32c(b2.detach())
        x1 = torch.empty(top.n_dst, 16, 64, dtype=torch.float32, device=dev)
        out = torch.empty(top.n_dst, 16, 64, dtype=torch.float32, device=dev)
        d = L.GrlConvDesc(n_src=top.n_src, n_dst=top.n_dst, n_edges=top.n_edges, rowptr_dst=L.ptr(top.rowptr_dst),
                          edge_src=L.ptr(top.edge_src), edge_dst=L.ptr(top.edge_dst), rowptr_src=L.ptr(top.rowptr_src),
                          src_eid=None if sub is not None else L.ptr(es.src_eid), x_src=L.ptr(x_src), x_dst=L.ptr(xd),
                          basis=L.ptr(basis) if basis.dtype == torch.float32 else None,
                          basis_bf16=L.ptr(basis) if basis.dtype == torch.bfloat16 else None,
                          fiber_kernel=L.ptr(fk), wk_t=L.ptr(wk_t), wk=L.ptr(wk_c), bias=L.ptr(bias_c), ln_g=L.ptr(lng_c),
                          ln_b=L.ptr(lnb_c), w1_t=L.ptr(w1_t), w1=L.ptr(w1_c), b1=L.ptr(b1_c), w2_t=L.ptr(w2_t),
                          w2_c=L.ptr(w2_c), b2=L.ptr(b2_c), x1=L.ptr(x1), out=L.ptr(out), accumulate_out=0,
                          basis_row=L.ptr(basis_row))
        shape = (top.n_src, top.n_dst, top.n_edges)
        L.call("grl_fbconv_edge_fwd_tc" if basis.dtype == torch.bfloat16 else "grl_fbconv_edge_fwd", C.byref(d), shape=shape)
        x2 = x1  # placeholder so that save_for_backward has a tensor in the strict path
        if precision == "bf16":
            w2_rm = _f32c(w2_d)
            # the tensor-core backward reads the pre-LayerNorm tensor instead of recomputing the fibre convolution
            x2 = torch.empty_like(x1) if any(ctx.needs_input_grad) else None
            d.w2, d.x2 = L.ptr(w2_rm), L.ptr(x2)
            L.call("grl_fbconv_node_fwd_tc", C.byref(d), shape=shape)
        else:
            L.call("grl_fbconv_node_fwd", C.byref(d), shape=shape)
        ctx.save_for_backward(x_src, basis_full if sub is not None else basis, fk, wk_t, wk_c, bias_c, lng_c, lnb_c, w1_t,
                              w1_c, b1_c, w2_c, x1, _f32c(w2_d) if precision == "bf16" else w2_c, x2)
        ctx.es, ctx.sub, ctx.homo, ctx.precision, ctx.basis_in_dtype = es, sub, homo, precision, basis_in_dtype
        ctx.gacc = getattr(basis_full, "_grl_gacc", None) if tc_edge else None
        return out

    @staticmethod
    def backward(ctx, g_out):
        x_src, basis, fk, wk_t, wk_c, bias_c, lng_c, lnb_c, w1_t, w1_c, b1_c, w2_c, x1, w2_rm, x2 = ctx.saved_tensors
        es, sub, homo = ctx.es, ctx.sub, ctx.homo
        top = sub if sub is not None else es
        dev = x_src.device
        g_out = _f32c(g_out)
        g_x1 = torch.empty_like(x1)
        g_xsrc = torch.empty_like(x_src)
        basis_bf16 = basis.dtype == torch.bfloat16
        gacc = ctx.gacc
        acc_basis = gacc is not None and gacc["buf"] is not None
        acc_mode, acc_mask = int(acc_basis), None
        if acc_basis:
            g_basis = gacc["buf"]
            if gacc.get("mask") is not None:  # only the rows a sub layer wrote are valid so far: add there, overwrite the rest
                assert sub is None, "two sub layers on one basis are not supported"
                acc_mode, acc_mask = 2, gacc["mask"]
                gacc["mask"] = None  # after this launch every row is valid
        elif sub is not None and gacc is not None:
            # first consumer is a sub layer: it writes the rows of its own edges into an uninitialised buffer and leaves
            # a mask behind; the next (full) layer overwrites the other rows, EdgeBasisFn.backward zeroes them otherwise
            g_basis = torch.empty_like(basis)
            gacc["buf"], gacc["mask"] = g_basis, sub.edge_dst_parent
        else:
            # strict path (autograd sums the layers' gradients): rows outside a sub layer's edges must read as zero
            g_basis = torch.zeros_like(basis) if sub is not None else torch.empty_like(basis)
            if gacc is not None:
                gacc["buf"] = g_basis
        n_pn = _n_partials((top.n_dst + 7) // 8)
        n_pe = _n_partials((top.n_src + 15) // 16, 2 if basis_bf16 else 1)
        node_part = torch.empty(n_pn, L.NODE_GRAD_FLOATS, dtype=torch.float32, device=dev)
        edge_part = torch.empty(n_pe, L.EDGE_GRAD_FLOATS, dtype=torch.float32, device=dev)
        # the edge backward reaches per-edge data through src_eid: for a sub layer that is the parent's edge order, so
        # basis / grad_basis / edge_src are the parent's arrays and edge_dst the parent-order dst ranks
        d = L.GrlConvDesc(n_src=top.n_src, n_dst=top.n_dst, n_edges=top.n_edges, rowptr_dst=L.ptr(top.rowptr_dst),
                          edge_src=L.ptr(es.edge_src), edge_dst=L.ptr(sub.edge_dst_parent if sub is not None else es.edge_dst),
                          rowptr_src=L.ptr(top.rowptr_src),
                          src_eid=L.ptr(sub.src_eid_parent if sub is not None else es.src_eid), x_src=L.ptr(x_src),
                          basis=None if basis_bf16 else L.ptr(basis),
                          basis_bf16=L.ptr(basis) if basis_bf16 else None, fiber_kernel=L.ptr(fk),
                          wk_t=L.ptr(wk_t), wk=L.ptr(wk_c), bias=L.ptr(bias_c), ln_g=L.ptr(lng_c), ln_b=L.ptr(lnb_c),
                          w1_t=L.ptr(w1_t), w1=L.ptr(w1_c), b1=L.ptr(b1_c), w2_c=L.ptr(w2_c), x1=L.ptr(x1),
                          grad_out=L.ptr(g_out), grad_x1=L.ptr(g_x1), grad_x_src=L.ptr(g_xsrc),
                          grad_x_src_init=L.ptr(g_out) if (homo and sub is None) else None,
                          grad_basis=None if basis_bf16 else L.ptr(g_basis),
                          grad_basis_bf16=L.ptr(g_basis) if basis_bf16 else None,
                          accumulate_grad_basis=acc_mode, grad_basis_acc_mask=L.ptr(acc_mask),
                          node_grad_partials=L.ptr(node_part), n_partials_node=n_pn,
                          edge_grad_partials=L.ptr(edge_part), n_partials_edge=n_pe)
        shape = (top.n_src, top.n_dst, top.n_edges)
        if ctx.precision == "bf16":
            g_x2 = torch.empty_like(x1)
            amax = torch.empty(1, dtype=torch.int32, device=dev)  # bit pattern of max |grad_out| (fp16 gradient scale)
            L.call("grl_absmax", L.ptr(g_out), g_out.numel(), L.ptr(amax), shape=shape)
            d.w2, d.grad_x2, d.grad_amax, d.x2 = L.ptr(w2_rm), L.ptr(g_x2), L.ptr(amax), L.ptr(x2)
            L.call("grl_fbconv_node_bwd_tc", C.byref(d), shape=shape)
        else:
            L.call("grl_fbconv_node_bwd", C.byref(d), shape=shape)
        L.call("grl_fbconv_edge_bwd_tc" if basis_bf16 else "grl_fbconv_edge_bwd", C.byref(d), shape=shape)
        g = _reduce(node_part)
        o = 0
        gw1 = g[o:o + 256 * 64].view(256, 64); o += 256 * 64
        gb1 = g[o:o + 256]; o += 256
        gw2 = g[o:o + 64 * 256].view(64, 256); o += 64 * 256
        gb2 = g[o:o + 64]; o += 64
        glng = g[o:o + 64]; o += 64
        glnb = g[o:o + 64]; o += 64
        gbias = g[o:o + 64]; o += 64
        gfk = g[o:o + 16 * 16 * 64].view(16, 16, 64)
        gwk = _reduce(edge_part).view(64, 64)
        g_xdst = None if homo else g_out
        if sub is not None:  # residual path of the output rows (out_ids are unique: plain read-modify-write)
            g_xsrc.index_copy_(0, sub.out_ids, g_xsrc.index_select(0, sub.out_ids) + g_out)
        if acc_basis:
            g_basis = None  # already inside the buffer the first consumer handed to autograd
        elif g_basis.dtype != ctx.basis_in_dtype:
            g_basis = g_basis.to(ctx.basis_in_dtype)
        return g_xsrc, g_xdst, g_basis, gfk, gwk, gbias, glng, glnb, gw1, gb1, gw2, gb2, None, None


def fiber_conv(x_src, x_dst, basis, fk, wk, bias, ln_g, ln_b, w1, b1, w2, b2, es: EdgeSet,
               sub: Optional[SubEdgeSet] = None):
    """`basis`: the [E,16,64] kernel_basis tensor, or a `BasisSpec` (fused 16-bit path: recomputed inside the kernels)."""
    if isinstance(basis, BasisSpec):
        assert basis.es is es, "the BasisSpec belongs to another edge set"
        return FusedFiberConvFn.apply(x_src, x_dst, basis.pos_src, basis.pos_dst, basis.w1, basis.b1, basis.w2, basis.b2,
                                      fk, wk, bias, ln_g, ln_b, w1, b1, w2, b2, basis.ori3, basis.dim, es, sub)
    return FiberConvFn.apply(x_src, x_dst, basis, fk, wk, bias, ln_g, ln_b, w1, b1, w2, b2, es, sub)


def aggregate_messages(x_src, basis, wk, es: EdgeSet) -> torch.Tensor:
    """x1 only (no grad): used by the one-time calibration of conv.py:104-105,151-157."""
    require_exact(es, "aggregate_messages")
    if isinstance(basis, BasisSpec):
        basis = basis.materialize()
    x_src, basis = _f32c(x_src.detach()), _f32c(basis.detach())
    wk_t = wk.detach().t().contiguous()
    x1 = torch.empty(es.n_dst, 16, 64, dtype=torch.float32, device=x_src.device)
    d = L.GrlConvDesc(n_src=es.n_src, n_dst=es.n_dst, n_edges=es.n_edges, rowptr_dst=L.ptr(es.rowptr_dst),
                      edge_src=L.ptr(es.edge_src), edge_dst=L.ptr(es.edge_dst), x_src=L.ptr(x_src), basis=L.ptr(basis),
                      wk_t=L.ptr(wk_t), x1=L.ptr(x1))
    L.call("grl_fbconv_edge_fwd", C.byref(d), shape=(es.n_src, es.n_dst, es.n_edges))
    return x1


# ------------------------------------------------------------------------------------------------
# V1: DeepSets critic, inner per-token MLP up to the pooled sum
# ------------------------------------------------------------------------------------------------
class CriticInnerFn(torch.autograd.Function):
    """x [B,N,F] -> ysum [B,64] = sum_n relu(graph_layer_norm(x W1^T + b1) * gamma + beta)  (deepsets.py:34-53 up to the
    token sum; PyG LayerNorm(mode='graph') statistics over the whole tensor).  Four launches forward + backward, no
    [B N, 64] activation in HBM.  `all_reduce(double[2])` (data parallel) makes the statistics global."""

    @staticmethod
    def forward(ctx, x, w1, b1, gamma, beta, eps, all_reduce=None, world_size=1):
        x, w1c, b1c = _f32c(x), _f32c(w1.detach()), _f32c(b1.detach())
        gc, bc = _f32c(gamma.detach()), _f32c(beta.detach())
        B, N, Fdim = x.shape
        assert tuple(w1c.shape) == (64, Fdim) and Fdim <= 16, f"critic inner layer {tuple(w1c.shape)} on {Fdim} features"
        dev = x.device
        n_p = _n_partials(B, 2)
        stats = torch.empty(2, dtype=torch.float64, device=dev)
        sp = torch.empty(n_p, 2, dtype=torch.float64, device=dev)
        ysum = torch.empty(B, 64, dtype=torch.float32, device=dev)
        d = L.GrlCriticDesc(n_graphs=B, n_tokens=N, n_feat=Fdim, n_partials=n_p, eps=float(eps),
                            count=float(B) * N * 64 * world_size, x=L.ptr(x), w1=L.ptr(w1c), b1=L.ptr(b1c), gamma=L.ptr(gc),
                            beta=L.ptr(bc), stats=L.ptr_any(stats), stat_partials=L.ptr_any(sp), ysum=L.ptr(ysum))
        L.call("grl_critic_inner_stats", C.byref(d), shape=(B * N, B, 0))
        if all_reduce is not None:
            all_reduce(stats)
        L.call("grl_critic_inner_fwd", C.byref(d), shape=(B * N, B, 0))
        ctx.save_for_backward(x, w1c, b1c, gc, bc, stats)
        ctx.meta = (float(eps), all_reduce, world_size, n_p)
        return ysum

    @staticmethod
    def backward(ctx, g_ysum):
        x, w1c, b1c, gc, bc, stats = ctx.saved_tensors
        eps, all_reduce, world_size, n_p = ctx.meta
        B, N, Fdim = x.shape
        dev = x.device
        g_ysum = _f32c(g_ysum)
        bstats = torch.empty(2, dtype=torch.float64, device=dev)
        sp = torch.empty(n_p, 2, dtype=torch.float64, device=dev)
        part = torch.empty(n_p, L.CRITIC_GRAD_FLOATS, dtype=torch.float32, device=dev)
        d = L.GrlCriticDesc(n_graphs=B, n_tokens=N, n_feat=Fdim, n_partials=n_p, eps=eps, count=float(B) * N * 64 * world_size,
                            x=L.ptr(x), w1=L.ptr(w1c), b1=L.ptr(b1c), gamma=L.ptr(gc), beta=L.ptr(bc), stats=L.ptr_any(stats),
                            stat_partials=L.ptr_any(sp), grad_ysum=L.ptr(g_ysum), bstats=L.ptr_any(bstats),
                            grad_partials=L.ptr(part))
        L.call("grl_critic_inner_bwd_stats", C.byref(d), shape=(B * N, B, 0))
        if all_reduce is not None:
            all_reduce(bstats)
        L.call("grl_critic_inner_bwd", C.byref(d), shape=(B * N, B, 0))
        g = _reduce(part)
        g_w1 = g[192:].view(64, 16)[:, :Fdim].contiguous()
        return None, g_w1, g[128:192], g[0:64], g[64:128], None, None, None


def critic_inner(x, w1, b1, gamma, beta, eps, all_reduce=None, world_size=1):
    return CriticInnerFn.apply(x, w1, b1, gamma, beta, eps, all_reduce, world_size)


# ------------------------------------------------------------------------------------------------
# K3: GAE
# ------------------------------------------------------------------------------------------------
# ------------------------------------------------------------------------------------------------
# K5: transformer encoder layer (M6 baseline)
# ------------------------------------------------------------------------------------------------
ENCODER_MAX_TOKENS = L.ENCODER_MAX_TOKENS


class EncoderLayerFn(torch.autograd.Function):
    """x [B,S,64] -> nn.TransformerEncoderLayer(64, 2, 64, dropout 0, post-LN, ReLU)(x) with the module's own parameter
    tensors (transformer_vanilla.py:30-36): one kernel forward, one backward (recomputes from x)."""

    @staticmethod
    def forward(ctx, x, in_w, in_b, out_w, out_b, w1, b1, w2, b2, n1w, n1b, n2w, n2b):
        x = _f32c(x)
        B, S, D = x.shape
        assert D == 64 and tuple(in_w.shape) == (192, 64) and tuple(w1.shape) == (64, 64) and tuple(w2.shape) == (64, 64)
        params = [_f32c(t.detach()) for t in (in_w, in_b, out_w, out_b, w1, b1, w2, b2, n1w, n1b, n2w, n2b)]
        out = torch.empty_like(x)
        d = EncoderLayerFn._desc(x, params, B, S)
        d.out = L.ptr(out)
        L.call("grl_encoder_layer_fwd", C.byref(d), shape=(B * S, B * S, 0))
        ctx.save_for_backward(x, *params)
        return out

    @staticmethod
    def _desc(x, p, B, S):
        return L.GrlEncoderDesc(n_graphs=B, n_tokens=S, n_partials=0, x=L.ptr(x), in_proj_weight=L.ptr(p[0]),
                                in_proj_bias=L.ptr(p[1]), out_proj_weight=L.ptr(p[2]), out_proj_bias=L.ptr(p[3]),
                                linear1_weight=L.ptr(p[4]), linear1_bias=L.ptr(p[5]), linear2_weight=L.ptr(p[6]),
                                linear2_bias=L.ptr(p[7]), norm1_weight=L.ptr(p[8]), norm1_bias=L.ptr(p[9]),
                                norm2_weight=L.ptr(p[10]), norm2_bias=L.ptr(p[11]))

    @staticmethod
    def backward(ctx, g_out):
        x, *params = ctx.saved_tensors
        B, S, _ = x.shape
        g_out = _f32c(g_out)
        g_x = torch.empty_like(x)
        n_p = _n_partials(B)
        part = torch.empty(n_p, L.ENCODER_GRAD_FLOATS, dtype=torch.float32, device=x.device)
        d = EncoderLayerFn._desc(x, params, B, S)
        d.n_partials, d.grad_out, d.grad_x, d.grad_partials = n_p, L.ptr(g_out), L.ptr(g_x), L.ptr(part)
        L.call("grl_encoder_layer_bwd", C.byref(d), shape=(B * S, B * S, 0))
        g = _reduce(part)
        o = 0
        grads = []
        for shape in ((192, 64), (192,), (64, 64), (64,), (64, 64), (64,), (64, 64), (64,), (64,), (64,), (64,), (64,)):
            n = 1
            for v in shape:
                n *= v
            grads.append(g[o:o + n].view(*shape))
            o += n
        return (g_x, *grads)


def encoder_layer(x: torch.Tensor, layer: "torch.nn.TransformerEncoderLayer") -> torch.Tensor:
    """`layer(x.transpose(0, 1)).transpose(0, 1)` for a batch-major x [B,S,64]."""
    a = layer.self_attn
    return EncoderLayerFn.apply(x, a.in_proj_weight, a.in_proj_bias, a.out_proj.weight, a.out_proj.bias, layer.linear1.weight,
                                layer.linear1.bias, layer.linear2.weight, layer.linear2.bias, layer.norm1.weight,
                                layer.norm1.bias, layer.norm2.weight, layer.norm2.bias)


def encoder_layer_supported(x: torch.Tensor, layer) -> bool:
    """The kernel covers what the shipped transformer config builds (transformer.yaml + transformer_vanilla.py:30-36):
    width 64, 2 heads, feed-forward 64, ReLU, post-LN, no active dropout, at most ENCODER_MAX_TOKENS tokens per graph."""
    a = layer.self_attn
    drop = layer.training and (layer.dropout.p > 0 or layer.dropout1.p > 0 or layer.dropout2.p > 0 or a.dropout > 0)
    return (x.is_cuda and x.dim() == 3 and x.shape[-1] == 64 and x.shape[1] <= ENCODER_MAX_TOKENS and a.embed_dim == 64
            and a.num_heads == 2 and a.in_proj_weight is not None and layer.linear1.out_features == 64
            and not layer.norm_first and layer.activation is torch.nn.functional.relu and not drop
            and layer.norm1.eps == 1e-5 and layer.norm2.eps == 1e-5)


def gae(reward, value_T1, done, terminated, gamma: float, lmbda: float):
    """reward/done/terminated [B,T], value_T1 [B,T+1] -> (advantage, value_target) [B,T]."""
    reward, value_T1 = _f32c(reward), _f32c(value_T1)
    B, T = reward.shape
    assert value_T1.shape == (B, T + 1)
    done_u8 = done.to(torch.uint8).contiguous()
    term_u8 = terminated.to(torch.uint8).contiguous()
    adv = torch.empty_like(reward)
    vt = torch.empty_like(reward)
    L.call("grl_gae_scan", L.ptr(reward), L.ptr(value_T1), L.ptr(done_u8), L.ptr(term_u8), float(gamma), float(lmbda), B,
           T, L.ptr(adv), L.ptr(vt))
    return adv, vt


# ------------------------------------------------------------------------------------------------
# A1: rollout-time Gaussian head + on-device sampling
# ------------------------------------------------------------------------------------------------
def gaussian_act(state, *, batch: int, num_rows: int, action_dim: int, pre_shift: float, minimal_std: float,
                 std_weight, std_bias=None, hidden=None, mean=None, mean_weight=None, mean_bias=None,
                 use_tanh_mean: bool = False, deterministic: bool = False, rank: int = 0, return_eps: bool = False):
    """One grl_gaussian_act launch (no autograd: acting only).  `state` is the int64 [2] {seed, call counter} buffer the
    draw reads; it is not advanced here (`act_advance`).  post_fc is implied by `mean is None` (the head's `_mean`
    Linear is applied to `hidden`), contextual std by `std_bias is not None` (`_pre_std` is a Linear).
    -> loc [B,k], covariance_matrix [B,k,k], action [B,k], sample_log_prob [B], eps [B,k] (or None)."""
    if state.dtype != torch.int64 or state.numel() != 2:
        raise ValueError("gaussian_act: state must be an int64 tensor {seed, counter}")
    post_fc, contextual = mean is None, std_bias is not None
    B, A, a = int(batch), int(num_rows), int(action_dim)
    k = A * a
    dev = state.device
    hidden = _f32c(hidden) if hidden is not None else None
    mean = _f32c(mean) if mean is not None else None
    if (post_fc or contextual) and (hidden is None or hidden.shape[0] != B * A):
        raise ValueError(f"gaussian_act: hidden must have batch * num_rows = {B * A} rows")
    if not post_fc and mean.numel() != B * k:
        raise ValueError(f"gaussian_act: mean must hold batch * k = {B * k} values, got {mean.numel()}")
    ws = [None if w is None else _f32c(w.detach()) for w in (mean_weight, mean_bias, std_weight, std_bias)]
    loc = torch.empty(B, k, dtype=torch.float32, device=dev)
    cov = torch.empty(B, k, k, dtype=torch.float32, device=dev)
    action = torch.empty(B, k, dtype=torch.float32, device=dev)
    log_prob = torch.empty(B, dtype=torch.float32, device=dev)
    eps = torch.empty(B, k, dtype=torch.float32, device=dev) if return_eps else None
    d = L.GrlActDesc(batch=B, num_rows=A, action_dim=a, hidden_dim=hidden.shape[-1] if hidden is not None else 64,
                     post_fc=int(post_fc), contextual_std=int(contextual), use_tanh_mean=int(bool(use_tanh_mean)),
                     deterministic=int(bool(deterministic)), rank=int(rank), pre_shift=float(pre_shift),
                     minimal_std=float(minimal_std), hidden=L.ptr(hidden), mean=L.ptr(mean), mean_weight=L.ptr(ws[0]),
                     mean_bias=L.ptr(ws[1]), std_weight=L.ptr(ws[2]), std_bias=L.ptr(ws[3]), state=L.ptr(state),
                     loc=L.ptr(loc), cov=L.ptr(cov), action=L.ptr(action), log_prob=L.ptr(log_prob), eps=L.ptr(eps))
    L.call("grl_gaussian_act", C.byref(d), shape=(B, k, 0))
    return loc, cov, action, log_prob, eps


def act_advance(state) -> None:
    """state[1] += 1 on the device (the call counter of gaussian_act's noise stream)."""
    L.call("grl_act_advance", L.ptr(state))


# ------------------------------------------------------------------------------------------------
# K4: trust-region projection
# ------------------------------------------------------------------------------------------------
class TrplProjectFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mean, v, old_mean, old_v, eps_mean, eps_cov, proj_type):
        mean, v, old_mean, old_v = _f32c(mean), _f32c(v), _f32c(old_mean), _f32c(old_v)
        B, k = mean.shape
        pm, pv = torch.empty_like(mean), torch.empty_like(v)
        eta = torch.empty(B, 2, dtype=torch.float64, device=mean.device)
        d = L.GrlProjDesc(batch=B, k=k, proj_type=proj_type, eps_mean=float(eps_mean), eps_cov=float(eps_cov),
                          mean=L.ptr(mean), v=L.ptr(v), old_mean=L.ptr(old_mean), old_v=L.ptr(old_v), proj_mean=L.ptr(pm),
                          proj_v=L.ptr(pv), eta=L.ptr_any(eta))
        L.call("grl_trpl_fwd", C.byref(d))
        ctx.save_for_backward(mean, v, old_mean, old_v, eta)
        ctx.meta = (float(eps_mean), float(eps_cov), proj_type)
        return pm, pv

    @staticmethod
    def backward(ctx, g_pm, g_pv):
        mean, v, old_mean, old_v, eta = ctx.saved_tensors
        eps_mean, eps_cov, proj_type = ctx.meta
        B, k = mean.shape
        g_pm = _f32c(g_pm) if g_pm is not None else torch.zeros_like(mean)
        g_pv = _f32c(g_pv) if g_pv is not None else torch.zeros_like(v)
        gm, gv = torch.empty_like(mean), torch.empty_like(v)
        d = L.GrlProjDesc(batch=B, k=k, proj_type=proj_type, eps_mean=eps_mean, eps_cov=eps_cov, mean=L.ptr(mean),
                          v=L.ptr(v), old_mean=L.ptr(old_mean), old_v=L.ptr(old_v), eta=L.ptr_any(eta),
                          grad_proj_mean=L.ptr(g_pm), grad_proj_v=L.ptr(g_pv), grad_mean=L.ptr(gm), grad_v=L.ptr(gv))
        L.call("grl_trpl_bwd", C.byref(d))
        return gm, gv, None, None, None, None, None


def trpl_project(mean, v, old_mean, old_v, eps_mean, eps_cov, proj_type="kl"):
    """Projected (mean, v) of a diagonal Gaussian; v is the diagonal of the reference's "std" matrix."""
    code = {"kl": 0, "w2": 1}[proj_type]
    return TrplProjectFn.apply(mean, v, old_mean, old_v, eps_mean, eps_cov, code)


# ------------------------------------------------------------------------------------------------
# M4: equivariant readout
# ------------------------------------------------------------------------------------------------
class ReadoutFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, latent, weight, bias, ori3, od, odv, dim):
        latent, w, b = _f32c(latent), _f32c(weight.detach()), _f32c(bias.detach())
        n = latent.shape[0]
        assert tuple(latent.shape[1:]) == (16, 64) and tuple(w.shape) == (od + odv, 64)
        out = torch.empty(n, odv, 3, dtype=torch.float32, device=latent.device)
        hidden = torch.empty(n, 64, dtype=torch.float32, device=latent.device)
        d = L.GrlReadoutDesc(n_nodes=n, od=od, odv=odv, dim=dim, latent=L.ptr(latent), weight=L.ptr(w), bias=L.ptr(b),
                             ori=L.ptr(ori3), out=L.ptr(out), hidden=L.ptr(hidden))
        L.call("grl_readout_fwd", C.byref(d))
        ctx.save_for_backward(latent, w, b, ori3)
        ctx.meta = (od, odv, dim)
        return out, hidden

    @staticmethod
    def backward(ctx, g_out, g_hidden):
        latent, w, b, ori3 = ctx.saved_tensors
        od, odv, dim = ctx.meta
        n, J = latent.shape[0], od + odv
        dev = latent.device
        g_out = _f32c(g_out) if g_out is not None else torch.zeros(n, odv, 3, dtype=torch.float32, device=dev)
        g_hidden = _f32c(g_hidden) if g_hidden is not None else None
        g_latent = torch.empty_like(latent)
        n_p = _n_partials((n + 7) // 8, 2)
        partials = torch.empty(n_p, J * 64 + J, dtype=torch.float32, device=dev)
        d = L.GrlReadoutDesc(n_nodes=n, od=od, odv=odv, dim=dim, latent=L.ptr(latent), weight=L.ptr(w), bias=L.ptr(b),
                             ori=L.ptr(ori3), grad_out=L.ptr(g_out), grad_hidden=L.ptr(g_hidden),
                             grad_latent=L.ptr(g_latent), grad_partials=L.ptr(partials), n_partials=n_p)
        L.call("grl_readout_bwd", C.byref(d))
        g = _reduce(partials)
        return g_latent, g[:J * 64].view(J, 64), g[J * 64:], None, None, None, None


def equivariant_readout(latent, weight, bias, ori3, od, odv, dim):
    """-> (out [n * odv, 3], hidden [n, 64]): hepi.py:173-190 on the output-node latents."""
    out, hidden = ReadoutFn.apply(latent, weight, bias, ori3, od, odv, dim)
    return out.reshape(-1, 3), hidden


# ------------------------------------------------------------------------------------------------
# L1 / P3: projection + every loss term around it in five launches
# ------------------------------------------------------------------------------------------------
class TrplLossFn(torch.autograd.Function):
    """(mean, v) of the current policy -> (loss_objective, loss_trust_region, loss_entropy, scalars[16]).

    grl_trpl_fwd projects, grl_trpl_loss_fwd evaluates log-weights, the standardised-advantage surrogate, the
    trust-region value against the detached projection, entropies, ESS and the trust-region metrics; the backward
    is grl_trpl_loss_bwd (gradients w.r.t. the projected parameters and the direct trust-region gradients) followed
    by grl_trpl_bwd (implicit differentiation of the projection).  `scalars` is not differentiable."""

    @staticmethod
    def forward(ctx, mean, v, old_mean, old_v, action, prev_log_prob, advantage, eps_mean, eps_cov, proj_type,
                entropy_coef, trust_region_coeff, normalize_advantage, all_reduce=None):
        mean, v, old_mean, old_v = _f32c(mean), _f32c(v), _f32c(old_mean), _f32c(old_v)
        action, prev_log_prob, advantage = _f32c(action), _f32c(prev_log_prob).reshape(-1), _f32c(advantage).reshape(-1)
        B, k = mean.shape
        assert action.shape == (B, k) and prev_log_prob.numel() == B and advantage.numel() == B
        dev = mean.device
        pm, pv = torch.empty_like(mean), torch.empty_like(v)
        eta = torch.empty(B, 2, dtype=torch.float64, device=dev)
        d = L.GrlProjDesc(batch=B, k=k, proj_type=proj_type, eps_mean=float(eps_mean), eps_cov=float(eps_cov),
                          mean=L.ptr(mean), v=L.ptr(v), old_mean=L.ptr(old_mean), old_v=L.ptr(old_v), proj_mean=L.ptr(pm),
                          proj_v=L.ptr(pv), eta=L.ptr_any(eta))
        L.call("grl_trpl_fwd", C.byref(d))
        terms = torch.empty(B, L.LOSS_TERMS, dtype=torch.float64, device=dev)
        stats = torch.empty(L.LOSS_STATS, dtype=torch.float64, device=dev)
        sums = torch.empty(L.LOSS_SUMS, dtype=torch.float64, device=dev)
        scalars = torch.empty(L.LOSS_SCALARS, dtype=torch.float32, device=dev)
        ld = L.GrlLossDesc(batch=B, k=k, proj_type=proj_type, normalize_advantage=int(bool(normalize_advantage)),
                           entropy_coef=float(entropy_coef), trust_region_coeff=float(trust_region_coeff),
                           mean=L.ptr(mean), v=L.ptr(v), proj_mean=L.ptr(pm), proj_v=L.ptr(pv), action=L.ptr(action),
                           prev_log_prob=L.ptr(prev_log_prob), advantage=L.ptr(advantage), terms=L.ptr_any(terms),
                           stats=L.ptr_any(stats), scalars=L.ptr(scalars), sums=L.ptr_any(sums), stage=0)
        if all_reduce is None:
            L.call("grl_trpl_loss_fwd", C.byref(ld))
        else:
            # data parallel: `all_reduce` is the hook `gather(tensor[n]) -> [world, n]` (one all-gather); the slice is then
            # combined in rank order by grl_dp_combine (sums first, maxima last): ONE collective per stage, deterministic
            def make_global(buf, lo, hi, n_sum):
                g = all_reduce(buf[lo:hi])
                L.call("grl_dp_combine", L.ptr_any(g), g.shape[0], hi - lo, n_sum, buf[lo:hi].data_ptr())
            ld.stage = 1
            L.call("grl_trpl_loss_fwd", C.byref(ld))
            make_global(stats, 0, 4, 3)
            ld.stage = 2
            L.call("grl_trpl_loss_fwd", C.byref(ld))
            make_global(sums, 3, 12, 7)
            ld.stage = 3
            L.call("grl_trpl_loss_fwd", C.byref(ld))
        ctx.save_for_backward(mean, v, old_mean, old_v, action, pm, pv, eta, terms, stats)
        ctx.meta = (float(eps_mean), float(eps_cov), proj_type, float(entropy_coef), float(trust_region_coeff))
        ctx.mark_non_differentiable(scalars)
        return scalars[0].clone(), scalars[1].clone(), scalars[2].clone(), scalars

    @staticmethod
    def backward(ctx, g_obj, g_tr, g_ent, _g_scalars):
        mean, v, old_mean, old_v, action, pm, pv, eta, terms, stats = ctx.saved_tensors
        eps_mean, eps_cov, proj_type, entropy_coef, trust_region_coeff = ctx.meta
        B, k = mean.shape
        dev = mean.device
        zero = torch.zeros((), dtype=torch.float32, device=dev)
        g3 = torch.stack([zero if g is None else g.reshape(()).float() for g in (g_obj, g_tr, g_ent)])
        g_pm, g_pv = torch.empty_like(mean), torch.empty_like(v)
        g_md, g_vd = torch.empty_like(mean), torch.empty_like(v)
        ld = L.GrlLossDesc(batch=B, k=k, proj_type=proj_type, normalize_advantage=0, entropy_coef=entropy_coef,
                           trust_region_coeff=trust_region_coeff, mean=L.ptr(mean), v=L.ptr(v), proj_mean=L.ptr(pm),
                           proj_v=L.ptr(pv), action=L.ptr(action), terms=L.ptr_any(terms), stats=L.ptr_any(stats),
                           grad_losses=L.ptr(g3), grad_proj_mean=L.ptr(g_pm), grad_proj_v=L.ptr(g_pv),
                           grad_mean_direct=L.ptr(g_md), grad_v_direct=L.ptr(g_vd))
        L.call("grl_trpl_loss_bwd", C.byref(ld))
        gm, gv = torch.empty_like(mean), torch.empty_like(v)
        d = L.GrlProjDesc(batch=B, k=k, proj_type=proj_type, eps_mean=eps_mean, eps_cov=eps_cov, mean=L.ptr(mean),
                          v=L.ptr(v), old_mean=L.ptr(old_mean), old_v=L.ptr(old_v), eta=L.ptr_any(eta),
                          grad_proj_mean=L.ptr(g_pm), grad_proj_v=L.ptr(g_pv), grad_mean=L.ptr(gm), grad_v=L.ptr(gv),
                          grad_mean_add=L.ptr(g_md), grad_v_add=L.ptr(g_vd))
        L.call("grl_trpl_bwd", C.byref(d))
        return (gm, gv) + (None,) * 12


def trpl_loss(mean, v, old_mean, old_v, action, prev_log_prob, advantage, eps_mean, eps_cov, proj_type, entropy_coef,
              trust_region_coeff, normalize_advantage=True, all_reduce=None):
    """-> (loss_objective, loss_trust_region, loss_entropy, scalars) with scalars indexed by _lib.LOSS_SCALAR_INDEX.
    `all_reduce` (data parallel, equal shards) = the hook `gather(tensor[n]) -> [world, n]`: advantage statistics, ESS and
    metrics become global, the three losses are this rank's share (local sum / global count)."""
    code = {"kl": 0, "w2": 1}[proj_type]
    return TrplLossFn.apply(mean, v, old_mean, old_v, action, prev_log_prob, advantage, eps_mean, eps_cov, code,
                            entropy_coef, trust_region_coeff, normalize_advantage, all_reduce)
