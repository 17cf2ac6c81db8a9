"""numpy references of the homogeneous views EMPN reads, as ops.homogeneous_edge_set / ops.sub_edge_set write them on the
device (grl_homo_merge, grl_sub_edge_set, then grl_csr_build and gathers).

merge_layout: the merge rule restated per output position (graph by the merged edge_ptr, then the edge type and the edge
inside it by walking the types' counts of that graph).
edge_set_layouts: the CSRs of an EdgeSet from a graph-major COO, the long way (stable counting sorts per graph, zero tails
and the gathers through them), as build_edge_set / refresh_edge_set compute them.
sub_layout: the sub-set rule restated (the output rows of graph b own one contiguous range of the parent's edge order).
sub_long_way: masking and a stable sort by source, as build_sub_edge_set computes them.
All arrays are numpy, named like the EdgeSet / SubEdgeSet fields."""
import numpy as np


def merge_layout(parts, B: int, n_tot: int, capacity: int):
    """parts: dicts with coo [2, >= edge_ptr[B]], edge_ptr [B+1], n_src, n_dst, off_src, off_dst (per graph)."""
    ptr = np.zeros(B + 1, np.int64)
    for p in parts:
        ptr += np.asarray(p["edge_ptr"], np.int64)
    coo = np.zeros((2, capacity), np.int64)
    for q in range(int(ptr[B])):
        b = int(np.searchsorted(ptr, q, side="right")) - 1
        r = q - int(ptr[b])
        for p in parts:
            e0 = int(p["edge_ptr"][b])
            c = int(p["edge_ptr"][b + 1]) - e0
            if r >= c:
                r -= c
                continue
            s, d = int(p["coo"][0, e0 + r]) - b * p["n_src"], int(p["coo"][1, e0 + r]) - b * p["n_dst"]
            coo[:, q] = (b * n_tot + p["off_src"] + s, b * n_tot + p["off_dst"] + d)
            break
    return {"edge_ptr": ptr, "coo": coo}


def _stable_csr(keys, other, edge_ptr, B, n_key, capacity):
    rowptr = np.zeros(B * n_key + 1, np.int32)
    oth, eid = np.zeros(capacity, np.int32), np.zeros(capacity, np.int32)
    E = int(edge_ptr[B])
    order = np.argsort(keys[:E], kind="stable")  # keys are graph-major, so this is the per-graph sort
    oth[:E], eid[:E] = other[:E][order], order
    rowptr[:] = np.searchsorted(keys[:E][order], np.arange(B * n_key + 1), side="left")
    return rowptr, oth, eid


def edge_set_layouts(coo, edge_ptr, B: int, n_tot: int):
    cap = coo.shape[1]
    o = {"coo": coo, "edge_ptr": edge_ptr}
    o["rowptr_dst"], o["edge_src"], o["eid_coo"] = _stable_csr(coo[1], coo[0], edge_ptr, B, n_tot, cap)
    o["edge_dst"] = coo[1][o["eid_coo"]].astype(np.int32) if cap else np.zeros(0, np.int32)
    o["rowptr_src"], _, o["src_eid"] = _stable_csr(o["edge_src"].astype(np.int64), o["edge_dst"], edge_ptr, B, n_tot, cap)
    o["s_src"], o["s_dst"] = o["edge_src"][o["src_eid"]], o["edge_dst"][o["src_eid"]]
    return o


def _rank(node, n_tot, out_off, n_out):
    g, l = node // n_tot, node % n_tot - out_off
    return g * n_out + l if 0 <= l < n_out else -1


def sub_layout(parent, B: int, n_tot: int, out_off: int, n_out: int, capacity: int):
    rp, E_par = parent["rowptr_dst"], int(parent["rowptr_dst"][B * n_tot])
    n_par = parent["edge_src"].shape[0]
    rank = lambda e: _rank(int(parent["edge_dst"][e]), n_tot, out_off, n_out) if e < E_par else -1  # noqa: E731
    o = {"edge_dst_parent": np.array([rank(e) for e in range(n_par)], np.int32).reshape(n_par)}
    o["edge_ptr"] = np.zeros(B + 1, np.int64)
    o["rowptr_dst"] = np.zeros(B * n_out + 1, np.int32)
    for b in range(B):
        base = int(rp[b * n_tot + out_off])
        o["edge_ptr"][b + 1] = o["edge_ptr"][b] + int(rp[b * n_tot + out_off + n_out]) - base
        for a in range(n_out):
            o["rowptr_dst"][b * n_out + a] = o["edge_ptr"][b] + int(rp[b * n_tot + out_off + a]) - base
    o["rowptr_dst"][B * n_out] = o["edge_ptr"][B]
    eids = np.zeros(capacity, np.int64)
    for q in range(int(o["edge_ptr"][B])):
        b = int(np.searchsorted(o["edge_ptr"], q, side="right")) - 1
        eids[q] = int(rp[b * n_tot + out_off]) + q - int(o["edge_ptr"][b])
    E_sub = int(o["edge_ptr"][B])
    o["eids"], o["eids32"] = eids, eids.astype(np.int32)
    o["edge_src"] = np.where(np.arange(capacity) < E_sub, parent["edge_src"][eids] if n_par else 0, 0).astype(np.int32)
    o["edge_dst"] = np.array([rank(int(e)) for e in eids], np.int32).reshape(capacity)
    o["rowptr_src"], _, eid = _stable_csr(o["edge_src"].astype(np.int64), o["edge_dst"], o["edge_ptr"], B, n_tot, capacity)
    o["src_eid_parent"], o["s_src"], o["s_dst"] = o["eids32"][eid], o["edge_src"][eid], o["edge_dst"][eid]
    return o


def sub_long_way(parent, out_ids, n_nodes: int):
    """build_sub_edge_set of an exact parent: mask the edges ending in out_ids, stable sort by source."""
    rank = np.full(n_nodes, -1, np.int64)
    rank[out_ids] = np.arange(len(out_ids))
    dst_rank = rank[parent["edge_dst"].astype(np.int64)]
    eids = np.nonzero(dst_rank >= 0)[0].astype(np.int64)
    edge_src, edge_dst = parent["edge_src"][eids], dst_rank[eids].astype(np.int32)
    order = np.argsort(edge_src, kind="stable")
    rp = lambda keys, n: np.concatenate([[0], np.cumsum(np.bincount(keys, minlength=n))]).astype(np.int32)  # noqa: E731
    return {"eids": eids, "eids32": eids.astype(np.int32), "rowptr_dst": rp(edge_dst, len(out_ids)), "edge_src": edge_src,
            "edge_dst": edge_dst, "rowptr_src": rp(edge_src, n_nodes), "src_eid_parent": eids[order].astype(np.int32),
            "edge_dst_parent": dst_rank.astype(np.int32), "s_src": edge_src[order], "s_dst": edge_dst[order]}
