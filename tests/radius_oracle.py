"""CPU brute-force radius graph for the tests (built on oracle/graph.py's kNN restatement and its rounding).

radius_edges: every j != i with sqdist <= r*r (fp32, (dx*dx + dy*dy) + dz*dz as in oracle.graph.sqdist_matrix, r*r
rounded to fp32), at most the m nearest, ties -> lower index; a NaN distance never passes the test, so a point with a
non-finite coordinate has no edges.  radius_topology: oracle.graph.build_topology with the INTERNAL edges of the kNN
tasks replaced by the radius graph of every point set (first num_points[b] points)."""
from typing import Dict, Optional

import torch

from oracle import graph as og


def radius_edges(points: torch.Tensor, r: float, m: int) -> torch.Tensor:
    """Coalesced [2,E] int64: row0 = neighbour j (source), row1 = centre i (target), sorted by (j, i)."""
    P = points.shape[0]
    if P == 0:
        return torch.empty(2, 0, dtype=torch.long)
    d = og.sqdist_matrix(points.float())
    r2 = torch.tensor(r, dtype=torch.float32) * torch.tensor(r, dtype=torch.float32)
    rows, cols = [], []
    for i in range(P):
        order = torch.argsort(d[i], stable=True)
        picked = [int(j) for j in order if int(j) != i and bool(d[i, j] <= r2)][:m]
        rows += picked
        cols += [i] * len(picked)
    return og.coalesce(torch.tensor([rows, cols], dtype=torch.long).reshape(2, -1))


def radius_topology(task: og.TaskSpec, position_vectors: Dict[str, torch.Tensor], *, full_graph_obs: bool,
                    output_mask_key: Optional[str], radius: float, max_num_neighbors: int,
                    num_points: Optional[torch.Tensor] = None) -> og.OGraph:
    assert task.internal_mode == "knn", "radius INTERNAL edges apply to the kNN tasks"
    g = og.build_topology(task, position_vectors, full_graph_obs=full_graph_obs, output_mask_key=output_mask_key,
                          num_points=num_points)
    e_int = task.edge_types[0]
    if e_int in g.edge_index_dict:
        pts = position_vectors[task.particle_type]
        B, P = pts.shape[0], pts.shape[1]
        per_graph = [radius_edges(pts[b, : int(num_points[b]) if num_points is not None else P], radius,
                                  max_num_neighbors) + b * P for b in range(B)]
        g.edge_index_dict[e_int] = torch.cat(per_graph, dim=1)
        g.edge_counts[e_int] = torch.tensor([e.shape[1] for e in per_graph], dtype=torch.long)
    return g
