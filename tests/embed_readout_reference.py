"""fp64 references of the two ends of every message-passing body, restated with plain torch ops.

`embed_reference`: the orientation lift and bias-free node encoder of grl_embed_fwd (scalar_to_sphere / vec_to_sphere of
to_from_sphere.py, then hepi.py's node_encoder): x[n][o][c] = sum_s scal[n][s] W[c][s] + sum_v <vec[n][v][:dim], ori[o]>
W[c][S + v], optionally over rows `node_ids` of padded feature arrays; and, given `grad_x`, the weight gradient of
grl_embed_bwd.  `readout_reference`: hepi.py's equivariant readout (decoder Linear, orientation means, the `od == 1`
broadcast gate, z = 0 in 2-D) and, through fp64 autograd, the gradients of grl_readout_bwd.

Both compute in the dtype of their inputs (float64 in the tests).  tests/test_embed_readout_reference_cpu.py pins the
first to oracle.models.lift + F.linear and the second to hepi.equivariant_readout_torch, both in fp32."""
from typing import Optional

import torch


def embed_features(scalars, vectors, ori3, dim: int, node_ids: Optional[torch.Tensor] = None) -> torch.Tensor:
    """[N,16,S+V]: the S scalars repeated over the 16 orientations, then <vec[v][:dim], ori[o][:dim]> per vector."""
    if node_ids is not None:
        scalars, vectors = scalars[node_ids.long()], vectors[node_ids.long()]
    n, S = scalars.shape
    vec = vectors.reshape(n, -1, 3)[..., :dim]
    sv = scalars[:, None, :].expand(n, ori3.shape[0], S)
    vv = torch.einsum("nvd,od->nov", vec, ori3[:, :dim].to(vec.dtype))
    return torch.cat([sv, vv], -1)


def embed_reference(scalars, vectors, weight, ori3, dim: int, node_ids: Optional[torch.Tensor] = None,
                    grad_x: Optional[torch.Tensor] = None):
    """dict(x [N,16,64]) and, with `grad_x`, grad_weight [64, S+V] = sum over nodes and orientations of
    grad_x[n][o][c] feat[n][o][f].  scalars [N',S], vectors [N',3V] (z ignored in 2-D), weight [64, S+V], ori3 [16,3];
    `node_ids` (int [N]) selects the rows of the padded arrays that form the batch, in that order."""
    feat = embed_features(scalars, vectors, ori3, dim, node_ids)
    w = weight.to(feat.dtype)
    res = {"x": torch.einsum("nof,cf->noc", feat, w)}
    if grad_x is not None:
        res["grad_weight"] = torch.einsum("noc,nof->cf", grad_x.to(feat.dtype), feat)
    return res


def readout_reference(latent, W, b, ori3, od: int, odv: int, dim: int, grad_out: Optional[torch.Tensor] = None,
                      grad_hidden: Optional[torch.Tensor] = None):
    """dict(out [n,odv,3], hidden [n,64]) of hepi.equivariant_readout_torch in the dtype of `latent`, with z = 0 in 2-D;
    with `grad_out` ([n,odv,3]) and / or `grad_hidden` ([n,64]) also grad = dict(latent, weight, bias).  A null
    upstream gradient contributes nothing, as in autograd; the z column of `grad_out` reaches nothing in 2-D."""
    dt = latent.dtype
    need = grad_out is not None or grad_hidden is not None
    lat = latent.detach().to(dt).requires_grad_(need)
    w = W.detach().to(dt).requires_grad_(need)
    bb = b.detach().to(dt).requires_grad_(need)
    grid = ori3[:, :dim].to(dt)
    y = torch.einsum("noc,jc->noj", lat, w) + bb            # decoder Linear(64 -> od + odv) per orientation
    scal = y[..., :od].mean(1)                               # [n, od]
    vec = torch.einsum("nov,od->nvd", y[..., od:], grid) / grid.shape[0]  # [n, odv, dim]
    out = vec * scal[:, :, None]                             # od == odv: vector v gated by scalar v; od == 1: broadcast
    if dim == 2:
        out = torch.cat([out, torch.zeros_like(out[..., :1])], -1)
    hidden = lat.mean(1)
    res = {"out": out.detach(), "hidden": hidden.detach()}
    if need:
        outs, grads = [], []
        if grad_out is not None:
            outs.append(out)
            grads.append(grad_out.to(dt))
        if grad_hidden is not None:
            outs.append(hidden)
            grads.append(grad_hidden.to(dt))
        g = torch.autograd.grad(outs, [lat, w, bb], grads)
        res["grad"] = dict(zip(("latent", "weight", "bias"), g))
    return res
