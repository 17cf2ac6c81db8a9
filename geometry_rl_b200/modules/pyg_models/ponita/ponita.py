"""EMPN body: orientation grids, polynomial features and the `Ponita` network with the reference's
parameter names (geometry_rl/modules/pyg_models/ponita/ponita.py), executed by the CUDA kernels.

Only the configuration the shipped configs reach is supported (separable depth-wise convolution,
64 channels, 16 orientations, widening 4, no attention, layer_scale None, degree 2); anything else
raises instead of silently running a different code path."""
import math
from typing import Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from .... import ops


def make_ori_grid(dim: int, n: int, only_upper_hemisphere: bool = False) -> torch.Tensor:
    """S1: n equispaced angles starting at 0.  S2: Fibonacci spiral, polar angle from
    acos(1 - s (i + 1/2) / n) with s = 2 (sphere) or 1 (upper hemisphere).  (ponita.py:53-97)"""
    if dim == 2:
        ang = torch.linspace(0, 2 * torch.pi - (2 * torch.pi / n), n)
        return torch.stack((ang.cos(), ang.sin()), dim=1)
    if dim != 3:
        raise ValueError("Only S1 and S2 are supported.")
    if n < 1:
        raise ValueError("n must be greater than 0.")
    idx = torch.arange(n)
    golden = (math.pi * idx * (1 + math.sqrt(5))) % (2 * math.pi)
    s = 1 if only_upper_hemisphere else 2
    polar = torch.acos(1 - s * (idx + 0.5) / (n - 1 + 1.0))
    return torch.stack((golden.cos() * polar.sin(), golden.sin() * polar.sin(), polar.cos()), dim=-1)


class GridGenerator(nn.Module):
    def __init__(self, dim: int, n: int, steps: int = 200, step_size: float = 0.01, device=None,
                 only_upper_hemisphere: bool = False):
        super().__init__()
        self.dim, self.n, self.only_upper_hemisphere = dim, n, only_upper_hemisphere

    def forward(self) -> torch.Tensor:
        return make_ori_grid(self.dim, self.n, self.only_upper_hemisphere)


class PolynomialFeatures(nn.Module):
    """[x, x (x) x, (x (x) x) (x) x, ...] flattened (ponita.py:233-244); used on the 16 x 16 fibre
    invariants only — the per-edge spatial features are generated inside grl_edge_basis_fwd."""

    def __init__(self, degree):
        super().__init__()
        self.degree = degree

    def forward(self, x):
        feats = [x]
        for _ in range(self.degree):
            feats.append((feats[-1].unsqueeze(-1) * x.unsqueeze(-2)).flatten(-2, -1))
        return torch.cat(feats, -1)


def make_basis_fn(in_feats: int, hidden_dim: int, basis_dim: int, degree: int) -> nn.Sequential:
    act = nn.GELU()
    return nn.Sequential(PolynomialFeatures(degree), nn.Linear(in_feats, hidden_dim), act,
                         nn.Linear(hidden_dim, basis_dim), act)


def pad_ori3(grid: torch.Tensor) -> torch.Tensor:
    """[16, dim] -> contiguous [16, 3] fp32 with z = 0 for S1 (kernel-side layout)."""
    g3 = torch.zeros(grid.shape[0], 3, dtype=torch.float32, device=grid.device)
    g3[:, : grid.shape[1]] = grid
    return g3.contiguous()


def _check_supported(channels, kernel_dim, num_ori, widening_factor, degree):
    if not (channels == 64 and kernel_dim == 64 and num_ori == 16 and widening_factor == 4 and degree == 2):
        raise NotImplementedError(
            "libgrl_b200 kernels are specialised for hidden=basis=64, num_ori=16, widening_factor=4, degree=2 "
            f"(got hidden={channels}, basis={kernel_dim}, num_ori={num_ori}, widening={widening_factor}, "
            f"degree={degree})")


class SeparableFiberBundleConv(nn.Module):
    """Parameter container of ponita.py:100-192 (depth-wise separable variant)."""

    def __init__(self, in_channels, out_channels, kernel_dim, bias=True, groups=1, attention=False):
        super().__init__()
        if not (groups == in_channels == out_channels) or attention or not bias:
            raise NotImplementedError("only the depth-wise separable, attention-free convolution with bias is built")
        self.depthwise = True
        self.in_channels, self.out_channels = in_channels, out_channels
        self.kernel = nn.Linear(kernel_dim, in_channels, bias=False)
        self.fiber_kernel = nn.Linear(kernel_dim, int(in_channels * out_channels / groups), bias=False)
        self.attention = attention
        self.bias = nn.Parameter(torch.zeros(out_channels))
        self.register_buffer("callibrated", torch.tensor(False))
        # host-side latch of `callibrated` (reading the device buffer every forward would be a GPU sync per layer)
        self._cal_latch = False
        self._register_load_state_dict_pre_hook(lambda *a, **k: setattr(self, "_cal_latch", False))

    def is_callibrated(self) -> bool:
        if not self._cal_latch:
            self._cal_latch = bool(self.callibrated)
        return self._cal_latch


class SeparableFiberBundleConvNext(nn.Module):
    """ponita.py:195-230: conv -> LayerNorm -> Linear -> GELU -> Linear -> + input, run as ONE fused call."""

    def __init__(self, channels, kernel_dim, act=nn.GELU(), layer_scale=1e-6, widening_factor=4, attention=False):
        super().__init__()
        if layer_scale is not None:
            raise NotImplementedError("layer_scale is None in every shipped config (ponita_gcn.py:48)")
        self.conv = SeparableFiberBundleConv(channels, channels, kernel_dim, groups=channels, attention=attention)
        self.act_fn = act
        self.linear_1 = nn.Linear(channels, widening_factor * channels)
        self.linear_2 = nn.Linear(widening_factor * channels, channels)
        self.register_buffer("layer_scale", None)
        self.norm = nn.LayerNorm(channels)

    def forward(self, x, kernel_basis, fiber_kernel_basis, edge_set: ops.EdgeSet, sub: Optional[ops.SubEdgeSet] = None):
        """`sub`: evaluate the layer at the rows `sub.out_ids` only (returns [len(out_ids), 16, 64])."""
        c = self.conv
        fk = F.linear(fiber_kernel_basis, c.fiber_kernel.weight)  # [p, o, c] (ponita.py:166 "boc,poc->bpc")
        fk_op = fk.transpose(0, 1).contiguous()  # kernel layout [o][p][c]
        pending = None
        if self.training and not c.is_callibrated():
            assert sub is None, "the one-time calibration needs the statistics of ALL rows (ponita.py:178-192)"
            pending = self._callibration_factors(x, kernel_basis, fk_op, edge_set)
        out = ops.fiber_conv(x, None, kernel_basis, fk_op, c.kernel.weight, c.bias, self.norm.weight, self.norm.bias,
                             self.linear_1.weight, self.linear_1.bias, self.linear_2.weight, self.linear_2.bias, edge_set,
                             sub)
        if pending is not None:
            # ponita.py:178-192: the kernels are re-scaled after this forward consumed the un-calibrated ones
            c.kernel.weight.data = c.kernel.weight.data * pending[0]
            c.fiber_kernel.weight.data = c.fiber_kernel.weight.data * pending[1]
            c.callibrated = ~c.callibrated
        return out

    @torch.no_grad()
    def _callibration_factors(self, x, kernel_basis, fk_op, edge_set):
        if not edge_set.exact:  # fixed-capacity topology: statistics over the real edges only (one count read)
            edge_set = ops.exact_edge_set(edge_set)
            kernel_basis = kernel_basis.on(edge_set) if isinstance(kernel_basis, ops.BasisSpec) else kernel_basis
        x1 = ops.aggregate_messages(x, kernel_basis, self.conv.kernel.weight, edge_set)
        x2 = torch.einsum("boc,opc->bpc", x1, fk_op) / 16
        std_in, std_1, std_2 = ops.calibration_std(x), ops.calibration_std(x1), ops.calibration_std(x2)
        return std_in / std_1, std_1 / std_2


class Ponita(nn.Module):
    def __init__(self, input_dim, hidden_dim, output_dim, num_layers, output_dim_vec=0, dim=3, num_ori=20,
                 basis_dim=None, degree=2, widening_factor=4, layer_scale=None, task_level="graph",
                 multiple_readouts=False, last_feature_conditioning=False, attention=False,
                 only_upper_hemisphere=False, **kwargs):
        super().__init__()
        basis_dim = hidden_dim if basis_dim is None else basis_dim
        _check_supported(hidden_dim, basis_dim, num_ori, widening_factor, degree)
        if last_feature_conditioning:
            raise NotImplementedError("last_feature_conditioning is False in every shipped config")
        self.dim, self.num_ori = dim, num_ori
        self.output_dim, self.output_dim_vec = output_dim, output_dim_vec
        self.last_feature_conditioning = last_feature_conditioning
        self.global_pooling = task_level == "graph"
        self.register_buffer("ori_grid", make_ori_grid(dim, num_ori, only_upper_hemisphere))
        self.basis_fn = make_basis_fn(sum(2 ** i for i in range(1, degree + 2)), hidden_dim, basis_dim, degree)
        self.fiber_basis_fn = make_basis_fn(sum(1 ** i for i in range(1, degree + 2)), hidden_dim, basis_dim, degree)
        self.x_embedder = nn.Linear(input_dim, hidden_dim, False)
        self.interaction_layers = nn.ModuleList()
        self.read_out_layers = nn.ModuleList()
        for i in range(num_layers):
            self.interaction_layers.append(
                SeparableFiberBundleConvNext(hidden_dim, basis_dim, act=nn.GELU(), layer_scale=layer_scale,
                                             widening_factor=widening_factor, attention=attention))
            if multiple_readouts or i == (num_layers - 1):
                self.read_out_layers.append(nn.Linear(hidden_dim, output_dim + output_dim_vec))
            else:
                self.read_out_layers.append(None)

    def fiber_basis(self) -> torch.Tensor:
        g = self.ori_grid
        inv3 = (g[None, :, :] * g[:, None, :]).sum(-1, keepdim=True)  # [16,16,1]
        return self.fiber_basis_fn(inv3)

    def calibration_pending(self) -> bool:
        return self.training and any(not l.conv.is_callibrated() for l in self.interaction_layers)

    def forward(self, scalars, vectors, pos, edge_set: ops.EdgeSet, batch=None, last_sub: Optional[ops.SubEdgeSet] = None,
                node_ids: Optional[torch.Tensor] = None):
        """scalars [N,S], vectors [N,3V] (un-lifted), pos [N,3] -> latent [N,16,64]; with `last_sub` the last layer is
        evaluated at `last_sub.out_ids` only and the result is [len(out_ids),16,64].  `node_ids` (int32): scalars / vectors
        are the PADDED arrays and node n of the (compact) graph is their row node_ids[n]; pos is already compact."""
        ori3 = pad_ori3(self.ori_grid)
        bf = self.basis_fn
        kernel_basis = ops.edge_basis(pos, pos, bf[1].weight, bf[1].bias, bf[3].weight, bf[3].bias, ori3, self.dim,
                                      edge_set)
        fiber_kernel_basis = self.fiber_basis()
        x = ops.EmbedFn.apply(scalars, vectors, self.x_embedder.weight, ori3, self.dim, node_ids)
        n_layers = len(self.interaction_layers)
        for i, layer in enumerate(self.interaction_layers):
            x = layer(x, kernel_basis, fiber_kernel_basis, edge_set, last_sub if i == n_layers - 1 else None)
        return x
