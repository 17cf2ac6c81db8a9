"""Critic wrapper: drop-in for models/value/gnn_vf_net.py:8-102 (`forward(*obs, train=)` -> [B,1] or
[B,T,1] for 3-D observations; parameter names `gnn.*`, `final.*`).

The reference evaluates 3-D inputs with a Python loop over time (gnn_vf_net.py:72-78), i.e. T+1
independent critic calls whose whole-batch LayerNorm statistics are PER TIME STEP.  Here all T+1 steps go
through the body as ONE [T*B] batch; `GraphLayerNorm` is told the number of independent groups so the
statistics (and therefore the values) are those of the loop (SURVEY 8(f) N2).  `fused_groups=True` (GAE.advantage)
runs that per-step normalisation of the per-token half on the fused critic kernels (DeepSets.one_step)."""
import torch
import torch.nn as nn


class GNNVFNet(nn.Module):
    def __init__(self, gnn, hyper_data, init="orthogonal", hidden_sizes=(64, 64), activation: str = "tanh",
                 layer_norm: bool = False, mesh_pos_obs: bool = False, actuator_vel_obs: bool = False, **kwargs):
        super().__init__()
        self.mesh_pos_obs = mesh_pos_obs
        self.actuator_vel_obs = actuator_vel_obs
        self.hyper_data = hyper_data
        self.gnn = gnn
        self.final = nn.Linear(hidden_sizes[-1], 1)

    def forward(self, *args, train=True, fused_groups: bool = False):
        self.train(train)
        if args[0].dim() == 3:
            B, T, _ = args[0].shape
            # time-major flattening: group t = rows [t*B, (t+1)*B) = one iteration of the reference's loop
            flat = [a.transpose(0, 1).reshape(T * B, a.shape[-1]) for a in args]
            c = self.gnn_forward(*flat, train=train, norm_groups=T, fused_groups=fused_groups)
            return self.final(c.reshape(T, B, -1).transpose(0, 1))
        return self.final(self.gnn_forward(*args, train=train))

    def gnn_forward(self, *args, train=True, norm_groups: int = 1, fused_groups: bool = False):
        data, input_vector = self.hyper_data.build_data(*args, train=train)
        if norm_groups > 1:
            return self.gnn.one_step(data, input_vector, norm_groups=norm_groups, fused_groups=fused_groups)
        return self.gnn.one_step(data, input_vector)
