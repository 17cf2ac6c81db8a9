"""HEPi's convolution module with the reference's name, constructor and parameter names
(geometry_rl/modules/pyg_models/ponita/conv.py:7-157); forward = two fused CUDA kernels."""
import torch
import torch.nn.functional as F
from torch.nn import LayerNorm, Linear, Sequential

from .... import ops


class FiberBundleConv(torch.nn.Module):
    def __init__(self, in_channels, out_channels, attr_dim, bias=True, aggr="add", separable=True, groups=1,
                 widening_factor=4):
        super().__init__()
        if aggr != "add" or not separable or not bias:
            raise NotImplementedError("only aggr='add', separable=True, bias=True is built (no shipped config "
                                      "selects AttentionalAggregation: configs/algorithm/pyg_agent/model/hepi.yaml)")
        if not (groups == in_channels == out_channels == 64 and attr_dim == 64 and widening_factor == 4):
            raise NotImplementedError("libgrl_b200 kernels are specialised for the depth-wise separable 64-channel "
                                      "convolution with widening_factor=4")
        self.depthwise = True
        self.separable = True
        self.in_channels, self.out_channels = in_channels, out_channels
        self.kernel = Linear(attr_dim, in_channels, bias=False)
        self.fiber_kernel = Linear(attr_dim, int(in_channels * out_channels / groups), bias=False)
        self.bias = torch.nn.Parameter(torch.zeros(out_channels))
        self.register_buffer("callibrated", torch.tensor(False))
        # host-side latch of `callibrated` (reading the device buffer every forward would be a GPU sync per conv)
        self._cal_latch = False
        self._register_load_state_dict_pre_hook(lambda *a, **k: setattr(self, "_cal_latch", False))
        self.vmap_aggr = None
        self.args = "sum"
        self.node_mlp = Sequential(LayerNorm(in_channels), Linear(in_channels, out_channels * widening_factor),
                                   torch.nn.GELU(), Linear(out_channels * widening_factor, out_channels))

    def forward(self, x, edge_index=None, edge_attr=None, fiber_attr=None, size=None, edge_set: ops.EdgeSet = None,
                **kwargs):
        if edge_set is None:
            raise RuntimeError("FiberBundleConv needs the sorted-CSR EdgeSet of the edge type (graph.edge_sets[et]); "
                               "a bare edge_index is not enough for the CUDA path")
        if isinstance(x, tuple):
            x_src, x_dst = x
            homo = x_src is x_dst
        else:
            x_src = x_dst = x
            homo = True
        fk = F.linear(fiber_attr, self.fiber_kernel.weight)  # [o, p, c]  (conv.py:88-90 "boc,opc->bpc")
        pending = None
        if self.training and not self._is_callibrated():
            pending = self._callibration_factors(x_src, x_dst, edge_attr, fk, edge_set)
        mlp = self.node_mlp
        out = ops.fiber_conv(x_src, None if homo else x_dst, edge_attr, fk, self.kernel.weight, self.bias, mlp[0].weight,
                             mlp[0].bias, mlp[1].weight, mlp[1].bias, mlp[3].weight, mlp[3].bias, edge_set)
        if pending is not None:
            # conv.py:151-157: weights are re-scaled after this forward consumed the un-calibrated ones
            self.kernel.weight.data = self.kernel.weight.data * pending[0]
            self.fiber_kernel.weight.data = self.fiber_kernel.weight.data * pending[1]
            self.callibrated = ~self.callibrated
        return (x_src, out)

    def _is_callibrated(self) -> bool:
        if not self._cal_latch:
            self._cal_latch = bool(self.callibrated)
        return self._cal_latch

    @torch.no_grad()
    def _callibration_factors(self, x_src, x_dst, edge_attr, fk, edge_set):
        if not edge_set.exact:
            # fixed-capacity topology: statistics over the real edges only (one count read; the calibration is eager).
            # A batch without any edge of this type leaves the convolution uncalibrated: the first batch with edges
            # calibrates it, as with exact topology, where such a batch skips the convolution.
            edge_set = ops.exact_edge_set(edge_set)
            if edge_set.n_edges == 0:
                return None
            edge_attr = edge_attr.on(edge_set) if isinstance(edge_attr, ops.BasisSpec) else edge_attr
        x1 = ops.aggregate_messages(x_src, edge_attr, self.kernel.weight, edge_set)
        x2 = torch.einsum("boc,opc->bpc", x1, fk) / fk.shape[-2]
        std_in, std_1, std_2 = ops.calibration_std(x_dst), ops.calibration_std(x1), ops.calibration_std(x2)
        return std_in / std_1, std_1 / std_2
