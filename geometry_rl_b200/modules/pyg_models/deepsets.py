"""DeepSets critic body: drop-in for geometry_rl/modules/pyg_models/deepsets.py (class name,
constructor, `one_step`, parameter names).

The per-token half (first Linear, whole-tensor LayerNorm, ReLU, token sum: all of the [B N, 64] work) runs in the
grl_critic_inner_* kernels, which recompute the pre-activations from x in every pass and never write a per-token
activation.  The inner MLP's second Linear commutes with the token sum (sum_n (y W2^T + b2) = (sum_n y) W2^T + N b2), so
it and the outer MLP are [B, 64] library GEMMs.  Time-batched calls of the advantage phase (`norm_groups` > 1, no
gradients) keep the plain torch formulation with per-step statistics by default (`adv_module(td)`); with `fused_groups`
(`GAE.advantage` / `capture`) the per-token half runs in the same kernels with one set of statistics per time step.  The
outer MLP works on [B, 64] and stays in torch with GraphLayerNorm(norm_groups) either way."""
from typing import Dict, List

import torch
from torch import nn

from ... import ops
from .pyg_compat import GraphLayerNorm, MLP


class DeepSets(nn.Module):
    def __init__(self, input_dim_node, output_dim, hidden_dim=64, norm: List[str] = [None, None], **ignored):
        super().__init__()
        self.input_dim = input_dim_node
        self._device = None
        self.mlp_inner = MLP([input_dim_node, hidden_dim, hidden_dim], norm=norm[0])
        self.mlp_outer = MLP([hidden_dim, hidden_dim, output_dim], norm=norm[1])
        self.fused_inner = True  # False: the torch formulation of the per-token half (parity partner in the tests)

    @property
    def device(self):
        if self._device is None:
            self._device = next(self.parameters()).device
        return self._device

    def forward(self, data, input_vector, **kwargs):
        return self.one_step(data, input_vector, **kwargs)

    def one_step(self, graph, u_dict: Dict[str, torch.Tensor], norm_groups: int = 1, fused_groups: bool = False,
                 **ignored):
        """`fused_groups`: run a time-batched call (`norm_groups` > 1) on the fused kernels too (forward only)."""
        B = len(graph)
        with torch.no_grad():
            x = torch.cat([u_dict[t].reshape(B, -1, u_dict[t].shape[-1]) for t in graph.node_types], dim=1)
        inner = self.mlp_inner
        norm = inner.norms[0] if len(inner.norms) == 1 else None
        if (x.is_cuda and (norm_groups == 1 or fused_groups) and isinstance(norm, GraphLayerNorm) and len(inner.lins) == 2
                and inner.lins[0].out_channels == 64 and x.shape[-1] <= 16 and self.fused_inner):
            hook = norm.fused_all_reduce
            ysum = ops.critic_inner(x, inner.lins[0].weight, inner.lins[0].bias, norm.weight, norm.bias, norm.eps,
                                    None if hook is None else hook[0], 1 if hook is None else hook[1], groups=norm_groups)
            x = torch.nn.functional.linear(ysum, inner.lins[1].weight) + x.shape[1] * inner.lins[1].bias
        else:
            x = self.mlp_inner(x, norm_groups)
            x = x.sum(dim=1)
        return self.mlp_outer(x, norm_groups)
