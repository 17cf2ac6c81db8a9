"""Restatements of TRPL entropy control (base_projection_layer.py:14-68,199-273, projection_utils.py:252-280) that the
entropy-control tests check the kernels against: the scheduled bound in fp64 numpy, and the entropy projection chained
with the oracle's trust-region projections in fp64 torch (differentiable)."""
import math

import numpy as np
import torch


def schedule(kind, ie, te, temperature, step, total_train_steps, k):
    """The bound grl_trpl_entropy_bound writes: projection_utils.get_entropy_schedule in fp64, the same operation order."""
    ie, te, step, T = np.float64(ie), np.float64(te), np.float64(step), np.float64(total_train_steps)
    if kind == "linear":
        return step * (te - ie) / T + ie
    if kind == "exp":
        return k * te + (ie - k * te) * np.power(np.float64(temperature), 10.0 * step / T)
    raise ValueError(kind)


def entropy(v):
    """policy.entropy((., v)) under "std := v": 0.5 (k (1 + log 2 pi) + 2 sum log v)."""
    k = v.shape[-1]
    return 0.5 * (k * (1.0 + math.log(2 * math.pi)) + 2.0 * v.log().sum(-1))


def entropy_projection(v, beta, equality):
    h = entropy(v)
    alpha = torch.exp((beta - h) / v.shape[-1])
    if not equality:
        alpha = torch.where(h < beta, alpha, torch.ones_like(alpha))
    return v * alpha[..., None]


def project(mean, v, old_mean, old_v, eps_mean, eps_cov, proj_type, beta, equality, first):
    """(proj_mean, proj_v) of base_projection_layer._projection with the oracle's KL / W2 (scale_prec) projections."""
    from oracle.projection import kl_projection, w2_projection
    tr = kl_projection if proj_type == "kl" else w2_projection
    if first:
        v = entropy_projection(v, beta, equality)
    pm, pv = tr(mean, v, old_mean, old_v, eps_mean, eps_cov)
    return pm, (pv if first else entropy_projection(pv, beta, equality))
