"""Trust-region projection layers: drop-in for
geometry_rl/algorithms/trust_region_projections/projections/base_projection_layer.py:126-384
(`projection(policy, p, q, step)`, `get_trust_region_loss`, `compute_metrics`, `initial_entropy`).

Differences in mechanism only: everything stays on the policy's CUDA device (the reference moves p and q
to the CPU, objectives/trpl.py:241-245) and the mean + covariance projection of a minibatch is ONE
kernel launch (grl_trpl_fwd / grl_trpl_bwd) instead of torch ops + numpy + ITPAL/NLopt on the host."""
from collections import OrderedDict
from typing import Tuple, Union

import torch

from .... import ops
from ..utils.projection_utils import diag_of, gaussian_kl, get_entropy_schedule


def _like(template: torch.Tensor, diag: torch.Tensor) -> torch.Tensor:
    """Return `diag` in the layout of `template` ([B,k] stays, [B,k,k] -> diag_embed)."""
    return torch.diag_embed(diag) if template.dim() == 3 else diag


def entropy_inequality_projection(policy, p, beta):
    """base_projection_layer.py:14-44."""
    mean, std = p
    d = diag_of(std)
    k = d.shape[-1]
    ent = policy.entropy(p)
    mask = ent < beta
    alpha = torch.where(mask, torch.exp((beta - ent) / k), torch.ones_like(ent))
    return mean, _like(std, d * alpha[..., None])


def entropy_equality_projection(policy, p, beta):
    """base_projection_layer.py:47-68."""
    mean, std = p
    d = diag_of(std)
    alpha = torch.exp((beta - policy.entropy(p)) / d.shape[-1])
    return mean, _like(std, d * alpha[..., None])


class BaseProjectionLayer(object):
    KERNEL_TYPE = None  # "kl" | "w2" for the layers the CUDA kernel implements

    def __init__(self, proj_type: str = "", mean_bound: float = 0.0, cov_bound: float = 0.0,
                 trust_region_coeff: float = 0.0, scale_prec: bool = False, mean_eq: bool = False,
                 entropy_schedule: Union[None, str] = None, action_dim: Union[None, int] = None,
                 total_train_steps: Union[None, int] = None, target_entropy: float = 0.0, temperature: float = 0.0,
                 entropy_eq: bool = False, entropy_first: bool = False, do_regression: bool = False,
                 regression_iters: int = 1000, lr_regression: float = 3e-4, optimizer_regression: str = "adam",
                 cpu: bool = True, dtype: torch.dtype = torch.float32):
        if do_regression:
            raise NotImplementedError("trust_region_regression is not used by the train loop (SURVEY 2 row 9)")
        self.proj_type = proj_type
        # kept as python floats: the bounds are kernel arguments, not tensors that need a device
        self.mean_bound = float(mean_bound)
        self.cov_bound = float(cov_bound)
        self.mean_eq = mean_eq
        self.trust_region_coeff = trust_region_coeff
        self.scale_prec = scale_prec
        assert (action_dim and total_train_steps) if entropy_schedule else True
        self._entropy_proj = entropy_equality_projection if entropy_eq else entropy_inequality_projection
        self._entropy_schedule_type = entropy_schedule
        self._entropy_schedule = get_entropy_schedule(entropy_schedule, total_train_steps, dim=action_dim)
        self.target_entropy = torch.tensor(float(target_entropy), dtype=dtype)
        self.entropy_first = entropy_first
        self.entropy_eq = entropy_eq
        self.temperature = temperature
        self.total_train_steps = total_train_steps
        self._initial_entropy = None
        self._entropy_state = None  # fused path: float64 [4] (initial_entropy, latched flag, bound, unused) on the device

    # ---- call protocol (base_projection_layer.py:199-273) ------------------------------------------
    def __call__(self, policy, p: Tuple[torch.Tensor, torch.Tensor], q, step, **kwargs):
        if self.initial_entropy is None:
            self.initial_entropy = policy.entropy(q).mean().detach()
        if not self.has_entropy_control:
            # schedule None -> bound -inf -> the entropy projection is the identity (kl.yaml:9-12)
            return self._trust_region_projection(policy, p, q, self.mean_bound, self.cov_bound, **kwargs)
        m = p[0]
        entropy_bound = self.get_entropy_bound(step).to(m.device) * m.new_ones(m.shape[0])
        return self._projection(policy, p, q, self.mean_bound, self.cov_bound, entropy_bound, **kwargs)

    def _trust_region_projection(self, policy, p, q, eps, eps_cov, **kwargs):
        if self.KERNEL_TYPE is None:
            return p
        if self.KERNEL_TYPE == "w2" and not self.scale_prec:
            raise NotImplementedError("the W2 kernel implements scale_prec=True (configs/algorithm/projection/w2.yaml)")
        if not getattr(policy, "contextual_std", True):
            raise NotImplementedError("non-contextual std is not reachable with the shipped configs")
        mean, std = p
        pm, pv = ops.trpl_project(mean, diag_of(std), q[0], diag_of(q[1]), eps, eps_cov, self.KERNEL_TYPE)
        return pm, _like(std, pv)

    def _projection(self, policy, p, q, eps, eps_cov, beta, **kwargs):
        if self.entropy_first:
            p = self._entropy_proj(policy, p, beta)
        proj = self._trust_region_projection(policy, p, q, eps, eps_cov, **kwargs)
        if self.entropy_first:
            return proj
        return self._entropy_proj(policy, proj, beta)

    @property
    def initial_entropy(self):
        return self._initial_entropy

    @initial_entropy.setter
    def initial_entropy(self, entropy):
        if self.initial_entropy is None:
            self._initial_entropy = entropy

    def entropy_state(self, device) -> torch.Tensor:
        """The fused path's entropy-control state, created on first use.  An initial entropy the torch formulation has
        already latched is carried over; from then on `initial_entropy` is a 0-dim view of the state."""
        if self._entropy_state is None:
            s = torch.zeros(4, dtype=torch.float64, device=device)
            if self._initial_entropy is not None:
                s[0] = self._initial_entropy.detach().to(device=device, dtype=torch.float64)
                s[1] = 1.0
            self._entropy_state = s
            self._initial_entropy = s[0]
        return self._entropy_state

    def entropy_control(self, step: torch.Tensor) -> ops.EntropyControl:
        """Arguments of ops.trpl_loss's entropy control; `step` is the int64 device step counter."""
        return ops.EntropyControl(self.entropy_state(step.device), step, self._entropy_schedule_type, self.total_train_steps,
                                  float(self.target_entropy), float(self.temperature), self.entropy_eq, self.entropy_first)

    @property
    def entropy_bound(self):
        """Entropy bound of the latest fused call (0-dim device view, for logging); None before one has run."""
        return None if self._entropy_state is None else self._entropy_state[2]

    def trust_region_value(self, policy, p, q):
        return gaussian_kl(policy, p, q)

    def get_trust_region_loss(self, policy, p, proj_p):
        """base_projection_layer.py:292-327."""
        p_target = (proj_p[0].detach(), proj_p[1].detach())
        mean_diff, cov_diff = self.trust_region_value(policy, p, p_target)
        return (mean_diff + cov_diff).mean() * self.trust_region_coeff

    def get_entropy_bound(self, step):
        return self._entropy_schedule(self.initial_entropy, self.target_entropy, self.temperature, step)

    def compute_metrics(self, policy, p, q, step=None, aggregate=True) -> dict:
        """base_projection_layer.py:332-384."""
        with torch.no_grad():
            entropy_old = policy.entropy(q)
            entropy = policy.entropy(p)
            mean_kl, cov_kl = gaussian_kl(policy, p, q)
            kl = mean_kl + cov_kl
            mean_diff, cov_diff = self.trust_region_value(policy, p, q)
            combined = mean_diff + cov_diff
            entropy_diff = entropy_old - entropy
        if aggregate:
            d = OrderedDict(kl=kl.mean(), constraint=combined.mean(), mean_constraint=mean_diff.mean(),
                            cov_constraint=cov_diff.mean(), entropy=entropy.mean(), entropy_diff=entropy_diff.mean(),
                            kl_max=kl.max(), constraint_max=combined.max(), mean_constraint_max=mean_diff.max(),
                            cov_constraint_max=cov_diff.max(), entropy_max=entropy.max(),
                            entropy_diff_max=entropy_diff.max())
        else:
            d = OrderedDict(kl=kl, constraint=combined, mean_constraint=mean_diff, cov_constraint=cov_diff,
                            entropy=entropy, entropy_diff=entropy_diff)
        if self.has_entropy_control:
            assert step is not None
            d.update(OrderedDict(entropy_constraint=(entropy - self.get_entropy_bound(step).to(entropy.device)).mean()))
        return d

    @property
    def has_entropy_control(self):
        return bool(self._entropy_schedule_type)
