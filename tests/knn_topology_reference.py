"""numpy references of the kNN edge set that ops.knn_edge_set writes with one kernel (grl_knn_topology).

neighbour_lists: the min(k, P-1) nearest of every centre (self excluded), ranked by (fp32 squared distance
(dx*dx + dy*dy) + dz*dz with NaN ranked as +inf, index), in ascending index order.
one_pass_layouts: the kernel's layout rules restated - every position follows from the per-centre lists, no sort.
chain_layouts: the same arrays the long way, as knn_graph -> build_edge_set -> src_sorted_pairs compute them: a coalesced
COO per graph, a stable counting sort of each graph's edges by destination and then by source (grl_csr_build), and the
gathers, with the zero tails of a fixed-capacity set.
Both return a dict of numpy arrays named like the EdgeSet fields (s_src / s_dst included)."""
import numpy as np


def neighbour_lists(pts: np.ndarray, k: int):
    pts = np.asarray(pts, dtype=np.float32)
    P = pts.shape[0]
    kk = max(0, min(k, P - 1))
    with np.errstate(invalid="ignore", over="ignore"):
        diff = pts[:, None, :] - pts[None, :, :]
        sq = diff * diff
        d = (sq[..., 0] + sq[..., 1]) + sq[..., 2]
    d = np.where(np.isnan(d), np.float32(np.inf), d)
    return [sorted(j for _, j in sorted((float(d[i, j]), j) for j in range(P) if j != i)[:kk]) for i in range(P)]


def _shape(pos, num_valid, k):
    B, P, _ = pos.shape
    nvs = [P if num_valid is None else min(max(int(num_valid[b]), 0), P) for b in range(B)]
    kks = [max(0, min(k, v - 1)) for v in nvs]
    edge_ptr = np.zeros(B + 1, np.int64)
    edge_ptr[1:] = np.cumsum([v * kk for v, kk in zip(nvs, kks)])
    return B, P, nvs, kks, edge_ptr


def one_pass_layouts(pos: np.ndarray, num_valid, k: int, capacity: int):
    B, P, nvs, kks, edge_ptr = _shape(pos, num_valid, k)
    E = capacity
    i32 = lambda n: np.zeros(n, np.int32)  # noqa: E731
    o = dict(coo=np.zeros((2, E), np.int64), edge_ptr=edge_ptr, rowptr_dst=i32(B * P + 1), edge_src=i32(E),
             edge_dst=i32(E), eid_coo=i32(E), rowptr_src=i32(B * P + 1), src_eid=i32(E), s_src=i32(E), s_dst=i32(E))
    for g in range(B):
        pv, kk, e0, e1, n0 = nvs[g], kks[g], int(edge_ptr[g]), int(edge_ptr[g + 1]), g * P
        lists = neighbour_lists(pos[g, :pv], k)
        cnt = np.bincount(np.array([j for lst in lists for j in lst], np.int64), minlength=pv)
        off = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)
        taken = np.zeros(pv, np.int64)
        for i in range(pv):  # edge order: centre i, then its neighbours ascending
            o["rowptr_dst"][n0 + i] = e0 + i * kk
            for s, j in enumerate(lists[i]):
                e = e0 + i * kk + s
                w = e0 + off[j] + taken[j]  # COO / src-sorted position: neighbour j, then rank of i among its centres
                taken[j] += 1
                o["edge_src"][e], o["edge_dst"][e] = n0 + j, n0 + i
                o["coo"][:, w] = (n0 + j, n0 + i)
                o["eid_coo"][e], o["src_eid"][w] = w, e
                o["s_src"][w], o["s_dst"][w] = n0 + j, n0 + i
        for j in range(pv):
            o["rowptr_src"][n0 + j] = e0 + off[j]
        o["rowptr_dst"][n0 + pv:n0 + P] = e1
        o["rowptr_src"][n0 + pv:n0 + P] = e1
    o["rowptr_dst"][B * P] = o["rowptr_src"][B * P] = edge_ptr[B]
    tail = int(edge_ptr[B])
    if tail < E and tail > 0:  # gathers through the zero tails read coo[1][0], edge_src[0], edge_dst[0]
        g0 = int(np.argmax(edge_ptr[1:] > 0))
        lists = neighbour_lists(pos[g0, :nvs[g0]], k)
        _, i_min = min((lst[0], i) for i, lst in enumerate(lists))
        o["edge_dst"][tail:] = g0 * P + i_min
        o["s_src"][tail:] = g0 * P + lists[0][0]
        o["s_dst"][tail:] = g0 * P
    return o


def _csr(coo, edge_ptr, B, n_key, key_row, E):
    rowptr, other, eid = np.zeros(B * n_key + 1, np.int32), np.zeros(E, np.int32), np.zeros(E, np.int32)
    for g in range(B):
        e0, e1 = int(edge_ptr[g]), int(edge_ptr[g + 1])
        keys = coo[key_row, e0:e1] - g * n_key
        order = np.argsort(keys, kind="stable")
        rowptr[g * n_key:(g + 1) * n_key] = e0 + np.concatenate([[0], np.cumsum(np.bincount(keys, minlength=n_key))])[:-1]
        other[e0:e1] = coo[1 - key_row, e0 + order]
        eid[e0:e1] = e0 + order
    rowptr[B * n_key] = edge_ptr[B]
    return rowptr, other, eid


def chain_layouts(pos: np.ndarray, num_valid, k: int, capacity: int):
    B, P, nvs, kks, edge_ptr = _shape(pos, num_valid, k)
    E = capacity
    coo = np.zeros((2, E), np.int64)
    for g in range(B):
        lists = neighbour_lists(pos[g, :nvs[g]], k)
        pairs = sorted((j, i) for i, lst in enumerate(lists) for j in lst)  # coalesce: sorted by (source, target)
        if pairs:
            coo[:, edge_ptr[g]:edge_ptr[g + 1]] = np.array(pairs, np.int64).T + g * P
    rowptr_dst, edge_src, eid_coo = _csr(coo, edge_ptr, B, P, 1, E)
    edge_dst = coo[1][eid_coo].astype(np.int32)
    rowptr_src, _, src_eid = _csr(np.stack([edge_src, edge_dst]).astype(np.int64), edge_ptr, B, P, 0, E)
    return dict(coo=coo, edge_ptr=edge_ptr, rowptr_dst=rowptr_dst, edge_src=edge_src, edge_dst=edge_dst,
                eid_coo=eid_coo, rowptr_src=rowptr_src, src_eid=src_eid, s_src=edge_src[src_eid], s_dst=edge_dst[src_eid])
