"""fp64 references of the pieces of the strict fp32 convolution path that conv16_reference does not restate alone.

`basis_reference`: the edge basis of grl_edge_basis_fwd (invariants -> polynomial features -> Linear GELU Linear GELU)
and, given `grad_basis`, the gradients of the four basis-MLP tensors (grl_edge_basis_bwd).
`spatial_reference`: the spatial half of grl_fbconv_edge_fwd / _bwd fed a given basis: x1 and the gradients of x_src,
the basis and kernel.weight.
`node_reference`: the node half (fibre convolution, bias, LayerNorm, MLP, residual) fed a given x1, through the
identity-message trick: one message per node with kernel.weight = I and a basis of ones reproduces x1 exactly.
`calibration_reference`: the one-time calibration factors (std_in / std_1, std_1 / std_2) of conv.py and ponita.py.

All of them are compositions of `oracle.models` evaluated in the dtype of their inputs; tests/test_conv_reference_cpu.py
pins each to the oracle in fp32."""
import torch

from oracle import models as om
from tests import conv16_reference as R

BASIS = ("bw1", "bb1", "bw2", "bb2")


def _basis_sd(leaves):
    return {"basis_fn.1.weight": leaves["bw1"], "basis_fn.1.bias": leaves["bb1"], "basis_fn.3.weight": leaves["bw2"],
            "basis_fn.3.bias": leaves["bb2"]}


def basis_reference(pos_src, pos_dst, params, ori3, dim, edge_index, grad_basis=None):
    """basis [E,16,64] of the edges `edge_index` (row 0 source, row 1 destination) in the dtype of `pos_src`, and with
    `grad_basis` grad[name] for bw1 [64,14], bb1, bw2, bb2.  Positions carry no gradient (as in the model)."""
    dt = pos_src.dtype
    leaves = {k: params[k].detach().to(dt).requires_grad_(grad_basis is not None) for k in BASIS}
    src, dst = edge_index[0].long(), edge_index[1].long()
    sp, _ = om.invariants(ori3[:, :dim].to(dt), pos_src[src][:, :dim].to(dt), pos_dst[dst][:, :dim].to(dt))
    basis = om.basis_mlp(sp, _basis_sd(leaves), "basis_fn")
    res = {"basis": basis.detach()}
    if grad_basis is not None:
        gs = torch.autograd.grad(basis, [leaves[k] for k in BASIS], grad_basis.to(dt))
        res["grad"] = dict(zip(BASIS, gs))
    return res


def spatial_reference(x_src, basis, wk, edge_index, n_dst, grad_x1=None):
    """x1[d] = sum over edges (s, d) of (basis[e] wk^T) * x_src[s], in the dtype of `x_src`; with `grad_x1` the gradients
    of x_src, basis and wk."""
    dt = x_src.dtype
    xs = x_src.detach().to(dt).requires_grad_(grad_x1 is not None)
    b = basis.detach().to(dt).requires_grad_(grad_x1 is not None)
    w = wk.detach().to(dt).requires_grad_(grad_x1 is not None)
    zeros = torch.zeros(n_dst, 16, 64, dtype=dt, device=xs.device)
    sd = {"c.kernel.weight": w, "c.fiber_kernel.weight": torch.zeros(64, 64, dtype=dt, device=xs.device),
          "c.bias": zeros[0, 0]}
    inter = {}
    om.fiber_bundle_conv(xs, zeros, torch.stack([edge_index[0].long(), edge_index[1].long()]), b,
                         torch.zeros(16, 16, 64, dtype=dt, device=xs.device), sd, "c", intermediates=inter)
    res = {"x1": inter["x1"].detach()}
    if grad_x1 is not None:
        gs = torch.autograd.grad(inter["x1"], [xs, b, w], grad_x1.to(dt))
        res["grad"] = dict(zip(("x_src", "basis", "wk"), gs))
    return res


def node_reference(x1, x_dst, params, grad_out=None):
    """The layer's node half fed x1 [N,16,64]: dict(x2, out) and, with `grad_out`, grad[name] for x_src (= grad_x1),
    x_dst and the node parameters (fk, bias, ln_g, ln_b, w1, b1, w2, b2).  `params` as conv16_reference.PARAM_NAMES; the
    basis MLP and kernel.weight are replaced by the identity message."""
    dt = x1.dtype
    n = x1.shape[0]
    pr = dict(params, wk=torch.eye(64, dtype=dt, device=x1.device))
    ei = torch.arange(n, device=x1.device).expand(2, -1)
    ori3 = torch.zeros(16, 3, dtype=dt, device=x1.device)
    return R.layer_reference(x1, x_dst.to(dt), x1[:, 0, :3], x1[:, 0, :3], pr, ori3, 3, ei, grad_out=grad_out,
                             kernel_basis=torch.ones(n, 16, 64, dtype=dt, device=x1.device))


def calibration_reference(x_dst, x1, fk):
    """(std(x_dst) / std(x1), std(x1) / std(x2)) with x2 = einsum("boc,opc->bpc", x1, fk) / 16, the factors that
    FiberBundleConv._callibration_factors (conv.py) and SeparableFiberBundleConvNext._callibration_factors (ponita.py,
    fk already in [o][p][c] layout) multiply kernel.weight and fiber_kernel.weight by.  torch.std: unbiased, over every
    element."""
    dt = x1.dtype
    x2 = torch.einsum("boc,opc->bpc", x1, fk.to(dt)) / fk.shape[-2]
    s_in, s1, s2 = x_dst.to(dt).std(), x1.std(), x2.std()
    return s_in / s1, s1 / s2
