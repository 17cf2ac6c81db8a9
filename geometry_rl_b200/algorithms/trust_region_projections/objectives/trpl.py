"""TRPL loss: drop-in for objectives/trpl.py:19-321 (constructor keywords, `loss_module(batch) -> dict` with
the keys train.py:275-301 reads, `_global_steps`, `clip_epsilon`, `projection`).

What changed in mechanism, not in results: no `.cpu()` round trip of (mean, cov) (trpl.py:241-245), no
`.item()` host syncs (trpl.py:264-271,287-288: outputs stay 0-dim device tensors), diagonal Gaussians are
handled as `[B,k]` diagonals instead of `[B,k,k]` matrices + Cholesky, and the projection is one CUDA
kernel.  `stats_reduce` hooks make the cross-sample reductions global under data parallelism (SURVEY 8(e))."""
import math
from typing import Optional

import torch
from torch import nn

from .operators import td_get


def td_is_cuda(module) -> bool:
    p = next(module.parameters(), None)
    return p is not None and p.is_cuda
from .utils import _clip_value_loss, distance_loss


class TRPLLoss(nn.Module):
    def __init__(self, actor_network, critic_network, *, projection=None, clip_epsilon: float = 0.2,
                 entropy_bonus: bool = True, samples_mc_entropy: int = 1, entropy_coef: float = 0.01,
                 critic_coef: float = 1.0, trust_region_coef: float = 1.0, loss_critic_type: str = "smooth_l1",
                 normalize_advantage: bool = True, gamma: float = None, separate_losses: bool = False,
                 clip_value: float = None, **kwargs):
        super().__init__()
        self.actor_network = actor_network
        self.critic_network = critic_network
        self.entropy_bonus = entropy_bonus
        self.samples_mc_entropy = samples_mc_entropy
        self.entropy_coef = entropy_coef
        self.critic_coef = critic_coef
        self.loss_critic_type = loss_critic_type
        self.normalize_advantage = normalize_advantage
        self.separate_losses = separate_losses
        # plain float (the reference registers a 0-dim buffer and moves it to the device on every call, trpl.py:219)
        self.clip_value = None if clip_value is None else float(clip_value)
        self.trust_region_coef = trust_region_coef
        self.register_buffer("clip_epsilon", torch.tensor(clip_epsilon))
        self.projection = projection
        self._global_steps = 0
        # entropy control on the fused path reads the step from this int64 device tensor.  A Learner owns and advances it
        # on the device (`steps_on_device`), so captured updates see the right step; otherwise every call writes
        # `_global_steps` into it.
        self.step_counter = None
        self.steps_on_device = False
        # data-parallel hooks (None = single process): see geometry_rl_b200/parallel.py
        self.dp = None
        # projection + every actor-side loss term and metric in a handful of kernel launches (ops.trpl_loss) instead
        # of ~170 elementwise / reduction launches; False = the torch formulation below
        self.fused = True

    @property
    def _clip_bounds(self):
        return math.log1p(-self.clip_epsilon), math.log1p(self.clip_epsilon)

    # ---- critic (trpl.py:176-229) ------------------------------------------------------------------
    def loss_critic(self, td) -> torch.Tensor:
        target_return = td_get(td, "value_target")
        old_state_value = td_get(td, "state_value") if self.clip_value is not None else None
        state_value = self.critic_network.module(*[td_get(td, k) for k in self.critic_network.in_keys])
        loss_value = distance_loss(target_return, state_value, loss_function=self.loss_critic_type)
        if self.clip_value is not None:
            loss_value, _ = _clip_value_loss(old_state_value, state_value, self.clip_value, target_return, loss_value,
                                             self.loss_critic_type)
        return self.critic_coef * loss_value

    # ---- actor (trpl.py:231-253) ---------------------------------------------------------------------
    def _log_weight_and_projection(self, td):
        action = td_get(td, "action")
        previous_dist = self.actor_network.build_dist_from_params(td)
        current_dist = self.actor_network.get_dist(td)
        # diagonals only: p[1] is the VARIANCE handed over as "std" (trpl.py:241, SURVEY 0 quirk)
        p = (current_dist.mean, current_dist.var_diag)
        q = (previous_dist.mean, previous_dist.var_diag)
        policy = self.actor_network.get_submodule("0").module
        proj_p = self.projection(policy, p, q, self._global_steps)
        dist = current_dist.__class__(proj_p[0], var_diag=proj_p[1])
        log_prob = dist.log_prob(action)
        prev_log_prob = td_get(td, "sample_log_prob")
        log_weight = (log_prob - prev_log_prob).unsqueeze(-1)
        return log_weight, dist, policy, p, proj_p

    def _mean(self, x: torch.Tensor) -> torch.Tensor:
        """Mean over the GLOBAL minibatch: local sum / global count (gradients are summed by the all-reduce)."""
        if self.dp is None:
            return x.mean()
        return x.sum() / (x.numel() * self.dp.world_size)

    def critic_term(self, td) -> torch.Tensor:
        """`loss_critic` entry of forward(): the critic branch shares nothing with the actor branch, so the learner
        may evaluate (and differentiate) it on a second CUDA stream."""
        return self._mean(self.loss_critic(td))

    def _can_fuse(self, policy) -> bool:
        pr = self.projection
        return (self.fused and getattr(pr, "KERNEL_TYPE", None) in ("kl", "w2")
                and (pr.KERNEL_TYPE != "w2" or pr.scale_prec)
                and getattr(policy, "contextual_std", True) and td_is_cuda(policy))

    def _forward_fused(self, td, with_critic: bool) -> dict:
        from .... import _lib, ops
        policy = self.actor_network.get_submodule("0").module
        previous_dist = self.actor_network.build_dist_from_params(td)
        current_dist = self.actor_network.get_dist(td)
        pr = self.projection
        entropy = None
        if pr.has_entropy_control:  # the initial entropy is latched on the device, with the bound
            if self.step_counter is None:
                self.step_counter = torch.zeros((), dtype=torch.int64, device=current_dist.mean.device)
            if not self.steps_on_device:
                self.step_counter.fill_(self._global_steps)
            entropy = pr.entropy_control(self.step_counter)
        elif pr.initial_entropy is None:  # base_projection_layer.py:202-203
            pr.initial_entropy = policy.entropy((previous_dist.mean, previous_dist.var_diag)).mean().detach()
        advantage = td_get(td, "advantage")
        l_obj, l_tr, l_ent, sc = ops.trpl_loss(
            current_dist.mean, current_dist.var_diag, previous_dist.mean, previous_dist.var_diag, td_get(td, "action"),
            td_get(td, "sample_log_prob"), advantage, pr.mean_bound, pr.cov_bound, pr.KERNEL_TYPE,
            self.entropy_coef if self.entropy_bonus else 0.0, pr.trust_region_coeff,
            self.normalize_advantage and advantage.numel() * (1 if self.dp is None else self.dp.world_size) > 1,
            None if self.dp is None else self.dp.all_gather_small, entropy)
        ix = _lib.LOSS_SCALAR_INDEX
        out = {"loss_objective": l_obj, "loss_trust_region": l_tr}
        if self.entropy_bonus:
            out["loss_entropy"] = l_ent
        if self.critic_coef and with_critic:
            out["loss_critic"] = self.critic_term(td)
        for key in ("ESS", "kl", "constraint", "mean_constraint", "mean_constraint_max", "cov_constraint",
                    "cov_constraint_max", "entropy", "entropy_diff"):
            out[key] = sc[ix[key]]
        return out

    def forward(self, td, with_critic: bool = True) -> dict:
        if self._can_fuse(self.actor_network.get_submodule("0").module):
            return self._forward_fused(td, with_critic)
        advantage = td_get(td, "advantage")
        if self.normalize_advantage and advantage.numel() > 1:
            if self.dp is None:
                loc, scale = advantage.mean(), advantage.std().clamp_min(1e-6)
            else:
                loc, scale = self.dp.mean_std_unbiased(advantage)
                scale = scale.clamp_min(1e-6)
            advantage = (advantage - loc) / scale
        log_weight, dist, policy, p, proj_p = self._log_weight_and_projection(td)
        with torch.no_grad():
            lw = log_weight.squeeze(-1)
            if self.dp is None:
                ess = (2 * lw.logsumexp(0) - (2 * lw).logsumexp(0)).exp()
                batch = log_weight.shape[0]
            else:
                ess = (2 * self.dp.logsumexp(lw) - self.dp.logsumexp(2 * lw)).exp()
                batch = log_weight.shape[0] * self.dp.world_size
        out = {"loss_objective": -self._mean(log_weight.exp() * advantage)}
        p_target = (proj_p[0].detach(), proj_p[1].detach())
        mean_diff, cov_diff = self.projection.trust_region_value(policy, p, p_target)
        out["loss_trust_region"] = self._mean(mean_diff + cov_diff) * self.projection.trust_region_coeff
        if self.entropy_bonus:
            entropy = dist.entropy()
            out["entropy"] = self._mean(entropy).detach()
            out["loss_entropy"] = -self.entropy_coef * self._mean(entropy)
        if self.critic_coef and with_critic:
            out["loss_critic"] = self.critic_term(td)
        out["ESS"] = ess.mean() / batch
        # trpl.py:318-320: metrics compare p with the PROJECTED distribution (log_tr_metrics(..., p, proj_p))
        m = self.projection.compute_metrics(policy, (p[0].detach(), p[1].detach()), p_target, step=self._global_steps,
                                            aggregate=self.dp is None)
        if self.dp is not None:
            m = self.dp.aggregate_metrics(m)
        for k in ("kl", "constraint", "mean_constraint", "mean_constraint_max", "cov_constraint", "cov_constraint_max",
                  "entropy", "entropy_diff"):
            out[k] = m[k]
        return out
