"""HEPi: heterogeneous equivariant message-passing policy body, drop-in for
geometry_rl/modules/pyg_models/hepi.py (same class name, constructor kwargs, `one_step` contract and
state_dict keys), executed by the sm_100a kernels of libgrl_b200."""
from typing import Dict

import torch
import torch.nn as nn

from ... import ops
from .ponita.hetero_fiber_conv import HeteroFiberConv
from .ponita.ponita import _check_supported, make_basis_fn, make_ori_grid, pad_ori3


def _plain(s) -> str:
    return str.__str__(s.value if hasattr(s, "value") and isinstance(s.value, str) else s)


class HEPi(nn.Module):
    # On the fused 16-bit path every convolution walks the CSR row pointers, so it runs on fixed-capacity edge sets
    # (ops.EdgeSet.exact False) as well; the other paths refuse them (ops.require_exact).
    accepts_capacity_edge_sets = True

    def __init__(self, input_dim_node, input_dim_edge, hidden_dim, latent_dim, output_dim, output_dim_vec,
                 node_encoder_layers, edge_encoder_layers, node_decoder_layers, node_type_mapping, edge_type_mapping,
                 edge_level_mapping, message_passing, num_messages, concat_global=False, shared_processor=False,
                 shared_node_encoder=True, shared_edge_encoder=True, device="cuda", num_ori=16, basis_dim=None, degree=2,
                 ponita_dim=3, only_upper_hemisphere=False, **ignored):
        super().__init__()
        basis_dim = hidden_dim if basis_dim is None else basis_dim
        _check_supported(latent_dim, basis_dim, num_ori, 4, degree)
        if hidden_dim != 64:
            raise NotImplementedError("hidden_dim must be 64")
        if concat_global:
            raise NotImplementedError("concat_global is False in every shipped config (hepi.yaml:15)")
        self.input_dim_node = input_dim_node
        self.output_dim, self.output_dim_vec = output_dim, output_dim_vec
        self.latent_dim, self.hidden_dim = latent_dim, hidden_dim
        self.num_messages = num_messages
        self.shared_processor = shared_processor
        self.node_type_mapping, self.edge_type_mapping = node_type_mapping, edge_type_mapping
        self.device = device
        self.concat_global = concat_global
        self.dim, self.num_ori = ponita_dim, num_ori

        self.register_buffer("ori_grid", make_ori_grid(self.dim, num_ori, only_upper_hemisphere))
        self.basis_fn = make_basis_fn(sum(2 ** i for i in range(1, degree + 2)), hidden_dim, basis_dim, degree)
        self.fiber_basis_fn = make_basis_fn(sum(1 ** i for i in range(1, degree + 2)), hidden_dim, basis_dim, degree)
        self.node_encoder = nn.Linear(self.input_dim_node, latent_dim, False)

        # hepi.py:93-104: one conv instance per (level, step); every edge type of that level shares it
        self.processor = nn.ModuleList()
        for k in range(num_messages):
            level_processor = {}
            for l, edge_level in enumerate(edge_level_mapping):
                pl = message_passing[l][k]
                if pl is None:
                    continue
                for et in edge_type_mapping:
                    src, level, dest = et.value if hasattr(et, "value") else et
                    if _plain(level) == _plain(edge_level):
                        level_processor[(_plain(src), _plain(level), _plain(dest))] = pl.to(device)
            self.processor.append(HeteroFiberConv(level_processor))
        self.decoder = nn.Linear(latent_dim, output_dim + output_dim_vec)
        # Skip the rows that cannot reach the readout: nodes without any edge outside the output node type (zero-padded
        # object points, isolated target nodes) are neither embedded nor convolved.  The reference computes and then
        # never reads them; outputs and every parameter gradient are unchanged.  False = all padded rows.
        self.prune_dead_rows = True

    def fiber_basis(self) -> torch.Tensor:
        g = self.ori_grid
        inv3 = (g[None, :, :] * g[:, None, :]).sum(-1, keepdim=True)  # hepi.py:119
        return self.fiber_basis_fn(inv3)

    def calibration_pending(self, graph) -> bool:
        """True until every convolution that runs on this graph did its one-time calibration (conv.py:104-105,151-157),
        which takes statistics over ALL rows of its inputs: those calls are evaluated densely.  Convolutions of edge
        types without edges never run (hetero_fiber_conv.py:48-49) and never calibrate."""
        if not self.training:
            return False
        from .ponita.hetero_fiber_conv import key_edge_type
        procs = [self.processor] if self.shared_processor else list(self.processor)
        for p in procs:
            for key, c in p.convs.items():
                es = graph.edge_sets.get(key_edge_type(key))
                if es is not None and es.n_edges > 0 and not c._is_callibrated():
                    return True
        return False

    def one_step(self, graph, u_dict, u: torch.Tensor = None, u_properties: torch.Tensor = None):
        scalar_dict, vector_dict = u_dict
        ori3 = pad_ori3(self.ori_grid)
        node_types, edge_sets = list(graph.node_types), graph.edge_sets
        pos = {nt: graph[nt].pos for nt in node_types}
        if self.prune_dead_rows and graph.output_mask_key is not None and not self.calibration_pending(graph):
            pr = graph.hetero_pruned()
            node_types = [nt for nt in node_types if nt in pr.live_ids]
            edge_sets = {et: pr.edge_sets.get(et, graph.edge_sets[et]) for et in graph.edge_types}
            with torch.no_grad():
                pos = {nt: pos[nt][pr.live_ids[nt]] for nt in node_types}
            node_ids = pr.live_ids32  # the embed kernel reads the padded feature rows in place
            live_edge_types = [et for et in graph.edge_types if et in pr.edge_sets]
        else:
            node_ids = {}
            live_edge_types = list(graph.edge_types)
        latent_dict = {nt: ops.EmbedFn.apply(scalar_dict[nt], vector_dict[nt], self.node_encoder.weight, ori3, self.dim,
                                             node_ids.get(nt))
                       for nt in node_types}
        bf = self.basis_fn
        fiber = self.fiber_basis()
        kernel_basis_dict, fiber_dict = {}, {}
        for et in live_edge_types:
            src, _, dst = et
            es = edge_sets[et]
            kernel_basis_dict[et] = ops.edge_basis(pos[src], pos[dst], bf[1].weight, bf[1].bias,
                                                   bf[3].weight, bf[3].bias, ori3, self.dim, es)
            fiber_dict[et] = fiber
        for i in range(self.num_messages):
            processor = self.processor if self.shared_processor else self.processor[i]
            latent_dict = processor(latent_dict=latent_dict, edge_index_dict=graph.edge_index_dict,
                                    edge_attr_dict=kernel_basis_dict, fiber_attr_dict=fiber_dict,
                                    edge_set_dict=edge_sets)
        latent = latent_dict[graph.output_mask_key]
        return equivariant_readout(latent, self.decoder, self.ori_grid, self.output_dim, self.output_dim_vec, self.dim)


def equivariant_readout(latent, decoder, ori_grid, output_dim, output_dim_vec, dim):
    """hepi.py:180-190 on the actuator nodes only ([B*A, 16, 64]): gate the orientation-averaged vector readout with
    the scalar readout.  One kernel forward, one backward (ops.equivariant_readout) when the shapes allow it."""
    if (latent.is_cuda and latent.shape[-1] == 64 and latent.shape[-2] == 16 and decoder.bias is not None
            and output_dim + output_dim_vec <= 8 and (output_dim == output_dim_vec or output_dim == 1)):
        return ops.equivariant_readout(latent, decoder.weight, decoder.bias, pad_ori3(ori_grid), output_dim,
                                       output_dim_vec, dim)
    return equivariant_readout_torch(latent, decoder, ori_grid, output_dim, output_dim_vec, dim)


def equivariant_readout_torch(latent, decoder, ori_grid, output_dim, output_dim_vec, dim):
    """The same readout written with torch ops (reference formulation; parity partner of the kernel in the tests)."""
    output = decoder(latent)
    out_scalar, out_vec = output.split([output_dim, output_dim_vec], dim=-1)
    hidden = latent.mean(dim=-2)
    out_scalar = out_scalar.mean(dim=-2)
    out_vec = torch.einsum("boc,od->bcd", out_vec, ori_grid) / ori_grid.shape[0]
    out = out_vec * out_scalar.unsqueeze(-1)
    if dim == 2:
        out = torch.cat([out, torch.zeros_like(out[..., :1])], dim=-1)
    return out.reshape(-1, out.shape[-1]), hidden.reshape(-1, hidden.shape[-1])
