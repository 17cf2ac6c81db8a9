"""Device-resident batched heterogeneous graph: the stand-in for the `HeteroData` batch the
reference's data builders return (geometry_rl/modules/pyg_data/rigid_tasks_data.py:324-343).

It exposes the attributes the reference's models read (`node_types`, `edge_types`,
`edge_index_dict`, `graph[node_type].pos`, `output_mask_key`, `output_mask`, `len(graph)`) and, in
addition, the sorted-CSR `EdgeSet`s the CUDA kernels consume.  Topology lives on the GPU and is built
by the K1 kernels (ops.knn_graph / dense_edges / build_edge_set); it is constructed once per batch
size and re-used, exactly like the reference's cached placeholder (rigid_tasks_data.py:254-255).
"""
from dataclasses import dataclass
from typing import Dict, List, Optional, Tuple

import torch

from ... import ops

EdgeType = Tuple[str, str, str]


class NodeStore:
    """Attribute bag of one node type (pos, norm_pos, properties)."""

    def __init__(self, num_nodes: int):
        self.num_nodes = num_nodes
        self.pos: Optional[torch.Tensor] = None
        self.norm_pos: Optional[torch.Tensor] = None
        self.properties: Optional[torch.Tensor] = None


@dataclass
class PrunedHomo:
    """Homogeneous topology restricted to the rows that can influence the readout (built once per topology).

    `es` is the homogeneous edge set over the LIVE nodes only: a node is dropped when it has no edge at all and is
    not an output node (the zero-padded object points of rigid_tasks_data.py:272-300, isolated target nodes) — its
    latent row never reaches an output, so neither the forward values read by anybody nor any gradient change.
    The edge order (dst-sorted, ties in COO order) is that of the full set: the renumbering is monotone.
    `sub` is the bipartite set "live nodes -> output nodes" of the LAST layer, whose result is only read at the
    output nodes (ponita_gcn.py:132-146 slices `output_mask` out of the last latent).
    With refreshed edge types (see `homogeneous`) every row is live: `es` is the full homogeneous set, `live_ids` and
    `live_ids32` are None (identity renumbering), and only `sub` restricts the last layer; both follow every refresh."""
    live_ids: Optional[torch.Tensor]  # [n_live] int64: full (padded) node index of every live node, ascending
    live_ids32: Optional[torch.Tensor]  # the same as int32 (GrlEmbedDesc.node_ids)
    es: ops.EdgeSet  # n_src = n_dst = n_live, all E edges, compact node ids
    sub: ops.SubEdgeSet


@dataclass
class PrunedHetero:
    """Heterogeneous topology without the nodes that cannot influence the readout: a node is kept when it has an edge
    of any type (as source or destination) or belongs to the output node type.  Per node type the renumbering is
    monotone, so every edge set keeps its edge order; node types left without nodes (isolated target nodes) vanish."""
    live_ids: Dict[str, torch.Tensor]  # node type -> [n_live] int64 indices into the padded per-type node order
    live_ids32: Dict[str, torch.Tensor]  # the same as int32 (GrlEmbedDesc.node_ids)
    edge_sets: Dict[EdgeType, ops.EdgeSet]  # compact node ids; edge types whose endpoints vanished are omitted
    num_nodes: int  # total live nodes


class GraphBatch:
    def __init__(self, num_graphs: int, nodes_per_graph: Dict[str, int], device):
        self.num_graphs = num_graphs
        self.nodes_per_graph = dict(nodes_per_graph)
        self.node_types: List[str] = list(nodes_per_graph.keys())
        self.device = device
        self._stores = {t: NodeStore(num_graphs * n) for t, n in nodes_per_graph.items()}
        self.edge_types: List[EdgeType] = []
        self.edge_sets: Dict[EdgeType, ops.EdgeSet] = {}
        self.output_mask_key: Optional[str] = None
        self.output_mask: slice = slice(None)
        self.homo_batch = None
        # edge types whose sets the data builder refreshes in place from every batch's positions (BaseData.refresh_in_place:
        # radius edges, or kNN edges with knn_in_place); their row sets never enter pruning
        self.refreshed_edge_types: set = set()
        self._homo_cache: Dict[str, ops.EdgeSet] = {}  # shared by every shallow copy of this topology

    # -- HeteroData-like surface ---------------------------------------------------------------
    def __len__(self):
        return self.num_graphs

    def __getitem__(self, key) -> NodeStore:
        return self._stores[str.__str__(key) if isinstance(key, str) else key]

    @property
    def edge_index_dict(self) -> Dict[EdgeType, torch.Tensor]:
        return {et: es.coo for et, es in self.edge_sets.items()}

    @property
    def num_nodes(self) -> int:
        return self.num_graphs * sum(self.nodes_per_graph.values())

    @property
    def node_offsets(self) -> Dict[str, int]:
        out, off = {}, 0
        for t in self.node_types:
            out[t] = off
            off += self.nodes_per_graph[t]
        return out

    def add_edge_type(self, et: EdgeType, coo: torch.Tensor, edge_ptr: torch.Tensor, refreshed: bool = False,
                      exact: bool = True):
        """`exact=False`: `coo` is a fixed-capacity buffer.  `refreshed`: see `add_edge_set`."""
        src, _, dst = et
        self.add_edge_set(et, ops.build_edge_set(coo, edge_ptr, self.num_graphs, self.nodes_per_graph[src],
                                                 self.nodes_per_graph[dst], exact=exact), refreshed)

    def add_edge_set(self, et: EdgeType, es: ops.EdgeSet, refreshed: bool = False):
        """`refreshed`: the data builder rewrites `es` in place from every batch (exact-size or fixed-capacity)."""
        self.edge_types.append(et)
        self.edge_sets[et] = es
        if refreshed:
            self.refreshed_edge_types.add(et)

    def shallow_copy(self) -> "GraphBatch":
        """`example_data.clone()` of the reference without copying the (immutable) topology."""
        g = GraphBatch.__new__(GraphBatch)
        g.__dict__.update(self.__dict__)
        g._stores = {}
        for t, s in self._stores.items():
            ns = NodeStore(s.num_nodes)
            ns.properties = s.properties
            g._stores[t] = ns
        return g

    # -- homogeneous view (ponita_gcn.py:65-83) ----------------------------------------------------
    def homogeneous(self) -> ops.EdgeSet:
        """All edge types merged into one graph whose nodes are the node types concatenated per graph
        (node_types order); per graph the edges keep edge-type insertion order, as to_homogeneous()
        yields them, so the segmented sums see the same edge order as the reference.

        With refreshed edge types the view is merged on the device (ops.homogeneous_edge_set, no host read): sized for
        the sum of the edge types' capacities, exact only when every edge type is, and rewritten in place by
        `refresh_homogeneous` after each refresh of the edge types."""
        if "homo" not in self._homo_cache and self.refreshed_edge_types:
            self._homo_cache["homo"] = ops.homogeneous_edge_set(self._homo_parts(), self.num_graphs,
                                                                sum(self.nodes_per_graph.values()))
        if "homo" not in self._homo_cache:
            for es in self.edge_sets.values():
                ops.require_exact(es, "GraphBatch.homogeneous")
            B, dev = self.num_graphs, self.device
            n_tot = sum(self.nodes_per_graph.values())
            offs = self.node_offsets
            counts = [self.edge_sets[et].edge_ptr[1:] - self.edge_sets[et].edge_ptr[:-1] for et in self.edge_types]
            total = torch.stack(counts).sum(0) if counts else torch.zeros(B, dtype=torch.int64, device=dev)
            homo_ptr = torch.zeros(B + 1, dtype=torch.int64, device=dev)
            homo_ptr[1:] = torch.cumsum(total, 0)
            E = int(homo_ptr[-1].item())
            coo = torch.empty(2, max(E, 1), dtype=torch.int64, device=dev)
            before = torch.zeros(B, dtype=torch.int64, device=dev)
            for et, cnt in zip(self.edge_types, counts):
                es = self.edge_sets[et]
                if es.n_edges > 0:
                    src, _, dst = et
                    g = torch.repeat_interleave(torch.arange(B, device=dev), cnt)
                    r = torch.arange(es.n_edges, device=dev) - es.edge_ptr[:-1][g]
                    dest = homo_ptr[:-1][g] + before[g] + r
                    ls = es.coo[0] - g * self.nodes_per_graph[src]
                    ld = es.coo[1] - g * self.nodes_per_graph[dst]
                    coo[0, dest] = g * n_tot + offs[src] + ls
                    coo[1, dest] = g * n_tot + offs[dst] + ld
                before = before + cnt
            self._homo_cache["homo"] = ops.build_edge_set(coo[:, :E], homo_ptr, B, n_tot, n_tot)
        return self._homo_cache["homo"]

    def _homo_parts(self):
        offs = self.node_offsets
        return [(self.edge_sets[et], offs[et[0]], offs[et[2]]) for et in self.edge_types]

    def _output_rows(self):
        """(first output row, output rows, sub-edge capacity) per graph: output rows are one contiguous range of the
        concatenated node types, and the capacity sums the edge types that end in it."""
        n_tot = sum(self.nodes_per_graph.values())
        start, stop, _ = self.output_mask.indices(n_tot)
        offs = self.node_offsets
        cap = sum(es.n_edges for (_, _, dst), es in self.edge_sets.items() if start <= offs[dst] < stop)
        return start, stop - start, cap

    def homogeneous_pruned(self) -> PrunedHomo:
        """See PrunedHomo.  Derived from `homogeneous()` with a handful of torch index ops, once per topology; with
        refreshed edge types, every row is kept and the last layer's sub set is derived on the device."""
        if "pruned" not in self._homo_cache and self.refreshed_edge_types:
            es = self.homogeneous()
            start, n_out, cap = self._output_rows()
            self._homo_cache["pruned"] = PrunedHomo(None, None, es, ops.sub_edge_set(es, start, n_out, cap))
        if "pruned" not in self._homo_cache:
            es = self.homogeneous()
            B, dev = self.num_graphs, self.device
            n_tot = sum(self.nodes_per_graph.values())
            is_out = torch.zeros(n_tot, dtype=torch.bool, device=dev)
            is_out[self.output_mask] = True
            is_out = is_out.repeat(B)
            deg_in = es.rowptr_dst[1:] - es.rowptr_dst[:-1]
            deg_out = es.rowptr_src[1:] - es.rowptr_src[:-1]
            live = (deg_in > 0) | (deg_out > 0) | is_out
            live_ids = live.nonzero().squeeze(1)
            n_live = int(live_ids.numel())
            new_id = torch.cumsum(live.to(torch.int64), 0) - 1
            edge_src = new_id[es.edge_src.long()].to(torch.int32).contiguous()
            edge_dst = new_id[es.edge_dst.long()].to(torch.int32).contiguous()
            # dropped nodes own no edges, so their CSR rows are empty and can simply be removed
            rowptr_dst = torch.cat([es.rowptr_dst[:-1][live_ids], es.rowptr_dst[-1:]]).contiguous()
            rowptr_src = torch.cat([es.rowptr_src[:-1][live_ids], es.rowptr_src[-1:]]).contiguous()
            compact = ops.EdgeSet(n_live, n_live, es.n_edges, es.coo, es.edge_ptr, rowptr_dst, edge_src, edge_dst,
                                  es.eid_coo, rowptr_src, es.src_eid)
            out_ids = new_id[is_out.nonzero().squeeze(1)]
            sub = ops.build_sub_edge_set(compact, out_ids)
            self._homo_cache["pruned"] = PrunedHomo(live_ids, live_ids.to(torch.int32).contiguous(), compact, sub)
        return self._homo_cache["pruned"]

    def refresh_homogeneous(self) -> None:
        """Rewrite the homogeneous views built so far (`homogeneous`, `homogeneous_pruned`) from the refreshed edge
        types, in place, on the device.  The data builder calls it after every in-place refresh of the edge types."""
        homo = self._homo_cache.get("homo")
        if homo is None or not self.refreshed_edge_types:
            return
        ops.refresh_homogeneous_edge_set(homo, self._homo_parts())
        pruned = self._homo_cache.get("pruned")
        if pruned is not None:
            ops.refresh_sub_edge_set(pruned.sub, homo, self._output_rows()[0])

    # -- heterogeneous view without dead rows (HEPi) ---------------------------------------------------
    def hetero_pruned(self) -> PrunedHetero:
        """Derived once per topology.  Every row of a node type that carries a refreshed edge type is live, so the live
        set does not depend on edges that change from batch to batch; the pruned set of a refreshed edge type is then the
        full `EdgeSet` itself (identity renumbering) and follows every in-place refresh."""
        if "hetero_pruned" not in self._homo_cache:
            dev = self.device
            touched = {t: torch.zeros(self._stores[t].num_nodes, dtype=torch.bool, device=dev) for t in self.node_types}
            for (src, _, dst), es in self.edge_sets.items():
                if (src, _, dst) in self.refreshed_edge_types:
                    touched[src][:] = True
                    touched[dst][:] = True
                elif es.n_edges > 0:
                    touched[src] |= (es.rowptr_src[1:] - es.rowptr_src[:-1]) > 0
                    touched[dst] |= (es.rowptr_dst[1:] - es.rowptr_dst[:-1]) > 0
            if self.output_mask_key is not None:
                touched[self.output_mask_key][:] = True
            else:  # no readout restriction: every node is an output
                for t in touched:
                    touched[t][:] = True
            live_ids, new_id = {}, {}
            for t, m in touched.items():
                ids = m.nonzero().squeeze(1)
                if ids.numel() > 0:
                    live_ids[t] = ids
                    new_id[t] = torch.cumsum(m.to(torch.int64), 0) - 1
            edge_sets = {}
            for et, es in self.edge_sets.items():
                src, _, dst = et
                if et in self.refreshed_edge_types:
                    edge_sets[et] = es
                    continue
                if es.n_edges == 0 or src not in live_ids or dst not in live_ids:
                    continue
                edge_sets[et] = ops.EdgeSet(
                    int(live_ids[src].numel()), int(live_ids[dst].numel()), es.n_edges, es.coo, es.edge_ptr,
                    torch.cat([es.rowptr_dst[:-1][live_ids[dst]], es.rowptr_dst[-1:]]).contiguous(),
                    new_id[src][es.edge_src.long()].to(torch.int32).contiguous(),
                    new_id[dst][es.edge_dst.long()].to(torch.int32).contiguous(), es.eid_coo,
                    torch.cat([es.rowptr_src[:-1][live_ids[src]], es.rowptr_src[-1:]]).contiguous(), es.src_eid)
            self._homo_cache["hetero_pruned"] = PrunedHetero(
                live_ids, {t: v.to(torch.int32).contiguous() for t, v in live_ids.items()}, edge_sets,
                sum(int(v.numel()) for v in live_ids.values()))
        return self._homo_cache["hetero_pruned"]
