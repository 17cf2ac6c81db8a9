"""EMPN (`PonitaGCN`): drop-in for geometry_rl/modules/pyg_models/ponita_gcn.py."""
from typing import Dict

import torch
from torch.nn import Linear

from .hepi import equivariant_readout
from .ponita.ponita import Ponita


class PonitaGCN(torch.nn.Module):
    # reads only GraphBatch.homogeneous() / homogeneous_pruned(), which are derived on the device from fixed-capacity,
    # in-place refreshed edge sets (BaseData.refresh_in_place)
    accepts_capacity_homogeneous_view = True

    def __init__(self, input_dim_node, output_dim, output_dim_vec, num_layers=2, hidden_dim=64, dropout=0.1, num_ori=20,
                 degree=2, widening_factor=4, attention=False, ponita_dim=3, only_upper_hemisphere=False, **ignored):
        super().__init__()
        self.input_dim = input_dim_node
        self._device = None
        self.dim = ponita_dim
        self.output_dim, self.output_dim_vec = output_dim, output_dim_vec
        self.ponita = Ponita(input_dim=input_dim_node, dim=ponita_dim, hidden_dim=hidden_dim, output_dim=output_dim,
                             num_layers=num_layers, output_dim_vec=output_dim_vec, num_ori=num_ori, basis_dim=None,
                             degree=degree, widening_factor=widening_factor, layer_scale=None, multiple_readouts=False,
                             last_feature_conditioning=False, task_level="node", attention=attention,
                             only_upper_hemisphere=only_upper_hemisphere)
        self.linear = Linear(hidden_dim, output_dim + output_dim_vec)
        # Evaluate only the latent rows that can reach the readout: nodes without any edge that are not output nodes
        # (zero-padded object points) are dropped from every layer, and the last layer is computed at the output nodes
        # alone.  The reference computes those rows and then discards them (ponita_gcn.py:132-146 masks the last
        # latent); outputs and every parameter gradient are unchanged.  False = dense evaluation of all B*n rows.
        self.prune_dead_rows = True

    @property
    def device(self):
        if self._device is None:
            self._device = next(self.parameters()).device
        return self._device

    def forward(self, data, input_vector, **kwargs):
        return self.one_step(data, input_vector, **kwargs)

    def one_step(self, graph, u_dict, **ignored):
        scalar_dict, vector_dict = u_dict
        B = len(graph)
        with torch.no_grad():  # ponita_gcn.py:94-125: per-graph concatenation of the node types
            sc = torch.cat([scalar_dict[t].reshape(B, -1, scalar_dict[t].shape[-1]) for t in graph.node_types], dim=1)
            vc = torch.cat([vector_dict[t].reshape(B, -1, vector_dict[t].shape[-1]) for t in graph.node_types], dim=1)
            pos = torch.cat([graph[t].pos.reshape(B, -1, 3) for t in graph.node_types], dim=1)
            n_per_graph = sc.shape[1]
            sc, vc, pos = sc.reshape(B * n_per_graph, -1), vc.reshape(B * n_per_graph, -1), pos.reshape(-1, 3)
            # the one-time calibration (ponita.py:178-192) takes statistics over ALL rows: that call runs dense
            pruned = graph.homogeneous_pruned() if (self.prune_dead_rows and not self.ponita.calibration_pending()) else None
            if pruned is not None and pruned.live_ids is not None:
                pos = pos[pruned.live_ids]  # the embed kernel reads sc / vc rows in place through live_ids32
            else:
                edge_set = graph.homogeneous()
        if pruned is not None:
            # [B*A, 16, 64]: rows of the output nodes, graph-major like the masked slice below
            latent = self.ponita(sc, vc, pos, pruned.es, last_sub=pruned.sub, node_ids=pruned.live_ids32)
        else:
            hidden = self.ponita(sc, vc, pos, edge_set)  # [B*n, 16, 64]
            # ponita_gcn.py:132-146 reads out every node and then masks; reading out the masked nodes is the same
            m = graph.output_mask
            latent = hidden.reshape(B, n_per_graph, 16, -1)[:, m].reshape(-1, 16, hidden.shape[-1])
        return equivariant_readout(latent, self.linear, self.ponita.ori_grid, self.output_dim, self.output_dim_vec,
                                   self.dim)
