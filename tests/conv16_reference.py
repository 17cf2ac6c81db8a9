"""fp64 reference of one fused 16-bit convolution layer (FusedFiberConvFn) and a per-row error metric.

`layer_reference` composes the dtype-generic pieces of `oracle.models` (invariants, basis_mlp, fiber_bundle_conv,
convnext_update) in whatever dtype its inputs have (float64 in the tests) on whatever device they sit on, and returns
x1, x2 (before LayerNorm), the layer output and, through autograd, the gradient of every input.  It takes the argument
set of `ops.fiber_conv` plus an explicit COO edge list, so homogeneous, bipartite and sub-layer cases all go through it.

`row_rel` is the per-row error the 16-bit tests use next to the global `max|a-b| / max|b|`: a row is one node at one
orientation (64 channels), and a single misrouted or dropped message shows up in its row even when the global ratio of a
large tensor stays small.  `perturbed` builds the reference of a deliberately wrong edge list, so that every test can
show that its own tolerance catches one dropped or misrouted edge.

The kernels evaluate GELU with the tanh approximation in fp16; this reference uses F.gelu (erf).  The difference
between the two GELUs in exact arithmetic is at most 4.7e-4 absolute (measured over [-8, 8]: `gelu_gap`), well
below the 16-bit tolerances, so the reference keeps the erf form of the model it restates."""
from typing import Dict, Optional

import torch
import torch.nn.functional as F

from oracle import models as om

PARAM_NAMES = ("bw1", "bb1", "bw2", "bb2", "fk", "wk", "bias", "ln_g", "ln_b", "w1", "b1", "w2", "b2")
_P = "conv"  # state-dict prefix of the one layer

# max |pos_src - pos_dst| (first `ponita_dim` coordinates) over every edge of the policy graphs of the four
# message-passing configs, 64 synthetic observations each: measured 1.8141 (test_conv_reference_cpu.py checks it)
LONGEST_EDGE = 1.82


def random_params(gen: torch.Generator, dtype=torch.float32, wk_scale: float = 0.12, bw2_scale: float = 0.15):
    """The 13 layer parameters of PARAM_NAMES at the scales of an initialised layer, drawn in fp64 from `gen`."""
    r = lambda *s, scale=1.0: torch.randn(*s, generator=gen, dtype=torch.float64).to(dtype) * scale  # noqa: E731
    return dict(bw1=r(64, 14, scale=0.25), bb1=r(64, scale=0.2), bw2=r(64, 64, scale=bw2_scale), bb2=r(64, scale=0.2),
                fk=r(16, 16, 64, scale=0.3), wk=r(64, 64, scale=wk_scale), bias=r(64, scale=0.1),
                ln_g=1 + r(64, scale=0.1), ln_b=r(64, scale=0.1), w1=r(256, 64, scale=0.12), b1=r(256, scale=0.1),
                w2=r(64, 256, scale=0.06), b2=r(64, scale=0.1))


def _state_dict(p: Dict[str, torch.Tensor], fk_identity: torch.Tensor) -> Dict[str, torch.Tensor]:
    """The layer's parameters under the oracle's key names.  `fiber_bundle_conv` forms fk = F.linear(fiber_basis, W);
    the ABI takes fk itself, so fk is fed as the fibre basis and W is the identity (F.linear(fk, I) == fk, exactly)."""
    return {"basis_fn.1.weight": p["bw1"], "basis_fn.1.bias": p["bb1"], "basis_fn.3.weight": p["bw2"],
            "basis_fn.3.bias": p["bb2"], f"{_P}.kernel.weight": p["wk"], f"{_P}.fiber_kernel.weight": fk_identity,
            f"{_P}.bias": p["bias"], f"{_P}.node_mlp.0.weight": p["ln_g"], f"{_P}.node_mlp.0.bias": p["ln_b"],
            f"{_P}.node_mlp.1.weight": p["w1"], f"{_P}.node_mlp.1.bias": p["b1"], f"{_P}.node_mlp.3.weight": p["w2"],
            f"{_P}.node_mlp.3.bias": p["b2"]}


def layer_reference(x_src, x_dst, pos_src, pos_dst, params: Dict[str, torch.Tensor], ori3, dim: int,
                    edge_index: torch.Tensor, out_ids: Optional[torch.Tensor] = None,
                    grad_out: Optional[torch.Tensor] = None, kernel_basis: Optional[torch.Tensor] = None):
    """One layer, out = x_dst + MLP(LN(fibre(scatter(kernel(basis) * x_src[src])) + bias)), in the dtype of `x_src`.

    x_src [n_src,16,64]; x_dst [n_dst,16,64] (bipartite) or None (homogeneous: x_dst is x_src); pos_* [n,3]; params: the
    13 tensors of PARAM_NAMES (fk [16,16,64] as the ABI takes it); ori3 [16,3] (z = 0 for dim 2); edge_index [2,E]
    (row 0 source, row 1 destination, node ids of x_src / x_dst).  `out_ids` (homogeneous only): evaluate the layer at
    those nodes alone, over the edges that end there (ops.build_sub_edge_set).  `kernel_basis` replaces the basis MLP
    (used by the node-kernel tests, which feed x1 directly).  Returns dict(x1, x2, out) and, with `grad_out`,
    grad[name] for x_src, x_dst (bipartite) and every parameter."""
    dt = x_src.dtype
    homo = x_dst is None
    leaves = {k: params[k].detach().to(dt).requires_grad_(True) for k in PARAM_NAMES}
    leaves["x_src"] = x_src.detach().to(dt).requires_grad_(True)
    if not homo:
        leaves["x_dst"] = x_dst.detach().to(dt).requires_grad_(True)
    xs = leaves["x_src"]
    src, dst = edge_index[0].long(), edge_index[1].long()
    pd_all = pos_dst
    if out_ids is not None:
        assert homo
        rank = torch.full((xs.shape[0],), -1, dtype=torch.long, device=xs.device)
        rank[out_ids.long()] = torch.arange(out_ids.numel(), device=xs.device)
        keep = rank[dst] >= 0
        src, dst = src[keep], rank[dst[keep]]
        xd = xs[out_ids.long()]
        pd_all = pos_dst[out_ids.long()]
    else:
        xd = xs if homo else leaves["x_dst"]
    sd = _state_dict(leaves, torch.eye(64, dtype=dt, device=xs.device))
    if kernel_basis is None:
        grid = ori3[:, :dim].to(dt)
        sp, _ = om.invariants(grid, pos_src[src][:, :dim].to(dt), pd_all[dst][:, :dim].to(dt))
        kernel_basis = om.basis_mlp(sp, sd, "basis_fn")
    inter = {}
    x2 = om.fiber_bundle_conv(xs, xd, torch.stack([src, dst]), kernel_basis, leaves["fk"], sd, _P, intermediates=inter)
    out = om.convnext_update(xd, x2, sd, f"{_P}.node_mlp.0", f"{_P}.node_mlp.1", f"{_P}.node_mlp.3")
    res = {"x1": inter["x1"].detach(), "x2": x2.detach(), "out": out.detach()}
    if grad_out is not None:
        names = [k for k in leaves if leaves[k].requires_grad]
        gs = torch.autograd.grad(out, [leaves[k] for k in names], grad_out.to(dt), allow_unused=True)
        res["grad"] = {k: (torch.zeros_like(leaves[k]) if g is None else g) for k, g in zip(names, gs)}
    return res


def edge_reference(x_src, pos_src, pos_dst, params, ori3, dim, edge_index, n_dst, grad_x1=None):
    """The edge half alone (what grl_fbconv_edge_fused_fwd / _bwd compute): x1 and, with `grad_x1`, the gradients of
    x_src, wk and the four basis-MLP tensors.  The layer reference with x_dst = 0; only x1 and its backward are used."""
    dt = x_src.dtype
    leaves = {k: params[k].detach().to(dt).requires_grad_(True) for k in ("bw1", "bb1", "bw2", "bb2", "wk")}
    xs = x_src.detach().to(dt).requires_grad_(True)
    zeros = torch.zeros(n_dst, 16, 64, dtype=dt, device=xs.device)
    sd = _state_dict(dict(leaves, bias=zeros[0, 0], ln_g=None, ln_b=None, w1=None, b1=None, w2=None, b2=None),
                     torch.eye(64, dtype=dt, device=xs.device))
    src, dst = edge_index[0].long(), edge_index[1].long()
    grid = ori3[:, :dim].to(dt)
    sp, _ = om.invariants(grid, pos_src[src][:, :dim].to(dt), pos_dst[dst][:, :dim].to(dt))
    kb = om.basis_mlp(sp, sd, "basis_fn")
    inter = {}
    om.fiber_bundle_conv(xs, zeros, torch.stack([src, dst]), kb, torch.zeros(16, 16, 64, dtype=dt, device=xs.device),
                         sd, _P, intermediates=inter)
    x1 = inter["x1"]
    res = {"x1": x1.detach()}
    if grad_x1 is not None:
        names = ["x_src", "wk", "bw1", "bb1", "bw2", "bb2"]
        gs = torch.autograd.grad(x1, [xs] + [leaves[k] for k in names[1:]], grad_x1.to(dt))
        res["grad"] = dict(zip(names, gs))
    return res


def row_rel(a: torch.Tensor, b: torch.Tensor, floor: float = 1e-2) -> float:
    """max over rows r of max|a_r - b_r| / (max|b_r| + floor * max|b|); a row is the last dimension (one node at one
    orientation for [N,16,64] tensors).  NaN or inf in `a` gives inf, so that no `row_rel(...) < tol` passes on them."""
    a = a.detach().double().reshape(-1, a.shape[-1] if a.dim() else 1)
    b = b.detach().double().to(a.device).reshape(a.shape)
    if not bool(torch.isfinite(a).all()):
        return float("inf")
    den = b.abs().amax(1) + floor * float(b.abs().max()) + 1e-300
    return float(((a - b).abs().amax(1) / den).max())


def global_rel(a: torch.Tensor, b: torch.Tensor) -> float:
    """max|a - b| / max|b| (north_star's bound for the 16-bit path); NaN or inf in `a` gives inf."""
    a, b = a.detach().double(), b.detach().double().to(a.device)
    if not bool(torch.isfinite(a).all()):
        return float("inf")
    return float((a - b).abs().max()) / (float(b.abs().max()) + 1e-300)


def perturbation(edge_index: torch.Tensor, kind: str, n_src: int) -> torch.Tensor:
    """A copy of `edge_index` with one edge wrong.  "drop": the last in-edge of a destination of the smallest degree
    >= 2, among those preferably one whose last edge ends a tile of 8 entries of the dst-sorted order (the kernels' tile
    boundary).  "swap": that same edge keeps its destination but takes another source."""
    src, dst = edge_index[0].long().cpu(), edge_index[1].long().cpu()
    order = torch.sort(dst, stable=True).indices
    d_sorted = dst[order]
    deg = torch.bincount(dst)
    last = torch.ones_like(d_sorted, dtype=torch.bool)
    last[:-1] = d_sorted[1:] != d_sorted[:-1]
    pos = torch.arange(d_sorted.numel())
    cand = last & (deg[d_sorted] >= 2)
    assert bool(cand.any()), "perturbation needs a destination of degree >= 2"
    idx = pos[cand]
    # smallest degree first (the row it changes is then dominated by few messages), a tile end before other entries
    score = 2 * deg[d_sorted[idx]] - (idx % 8 == 7).long()
    q = int(idx[torch.argmin(score)])
    e = int(order[q])
    if kind == "drop":
        keep = torch.ones(src.numel(), dtype=torch.bool)
        keep[e] = False
        return edge_index[:, keep.to(edge_index.device)]
    assert kind == "swap" and n_src >= 2
    out = edge_index.clone()
    out[0, e] = (int(src[e]) + 1 + n_src // 2) % n_src if n_src > 2 else 1 - int(src[e])
    return out


def perturbed(fn, edge_index: torch.Tensor, n_src: int, **kw):
    """{"drop": fn(edge_index=<one edge dropped>, **kw), "swap": fn(edge_index=<one source swapped>, **kw)}, where fn
    is layer_reference or edge_reference."""
    return {kind: fn(edge_index=perturbation(edge_index, kind, n_src), **kw) for kind in ("drop", "swap")}


def gelu_gap(lo: float = -8.0, hi: float = 8.0, n: int = 200001) -> float:
    """max |gelu_erf(x) - gelu_tanh(x)| over [lo, hi] in fp64: the part of the kernels' error that is the GELU form."""
    x = torch.linspace(lo, hi, n, dtype=torch.float64)
    return float((F.gelu(x) - F.gelu(x, approximate="tanh")).abs().max())
