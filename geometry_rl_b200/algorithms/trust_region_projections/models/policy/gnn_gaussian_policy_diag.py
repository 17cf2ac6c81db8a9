"""Diagonal Gaussian policy head around a GNN body: drop-in for
models/policy/gnn_gaussian_policy_diag.py:11-148 + abstract_gnn_gaussian_policy.py:16-121 +
abstract_gaussian_policy.py:124-134 (same constructor keywords, `forward(*obs, train=) ->
(mean [B,k], covariance [B,k,k])`, parameter names `_mean`, `_pre_std`, `gnn.*`).

`forward_diag` is the same computation without materialising the k x k matrices; TRPLLoss uses it."""
from typing import Tuple

import numpy as np
import torch
import torch.nn as nn

from ..... import ops
from ...utils.network_utils import initialize_weights
from ...utils.torch_utils import inverse_softplus
from ...utils.projection_utils import diag_of


class GNNGaussianPolicyDiag(nn.Module):
    def __init__(self, gnn, hyper_data, action_dim, num_actuators, init, hidden_sizes=(64, 64), activation: str = "tanh",
                 layer_norm: bool = False, contextual_std: bool = False, trainable_std: bool = True,
                 init_std: float = 1.0, use_tanh_mean: bool = False, share_weights=False, vf_model=None,
                 minimal_std: float = 1e-5, scale: float = 1e-4, gain: float = 0.01, share_action_dim: bool = True,
                 post_fc: bool = True, **kwargs):
        super().__init__()
        if isinstance(action_dim, list):
            raise NotImplementedError("per-actuator action_dim lists are not used by the shipped configs")
        self.action_dim = action_dim
        self.contextual_std = contextual_std
        self.share_weights = share_weights
        self.minimal_std = torch.tensor(minimal_std)
        self.init_std = torch.tensor(init_std)
        self.use_tanh_mean = use_tanh_mean
        self.post_fc = post_fc
        prev_size = hidden_sizes[-1]
        self.diag_activation = nn.Softplus()
        self.diag_activation_inv = inverse_softplus
        action_dim_shared = action_dim // num_actuators if share_action_dim else action_dim
        self._pre_activation_shift = self.diag_activation_inv(self.init_std - self.minimal_std)
        self._mean = nn.Linear(prev_size, action_dim_shared)
        initialize_weights(self._mean, init, gain=gain, scale=scale)
        if contextual_std:
            self._pre_std = nn.Linear(prev_size, action_dim_shared)
            initialize_weights(self._pre_std, init, gain=gain, scale=scale)
        else:
            self._pre_std = nn.Parameter(torch.normal(0, 0.01, (action_dim_shared,)))
            if not trainable_std:
                self._pre_std.requires_grad_(False)
        self.num_actuators = num_actuators
        self.hyper_data = hyper_data
        self.gnn = gnn
        # fixed-capacity, in-place refreshed topology (BaseData.refresh_in_place) only for a model that consumes it
        hyper_data.consumer_accepts_capacity = bool(getattr(gnn, "accepts_capacity_edge_sets", False))

    # ---- forward ---------------------------------------------------------------------------------
    def gnn_forward(self, *args, train=True):
        data, input_vector = self.hyper_data.build_data(*args, train=train)
        return self.gnn.one_step(data, input_vector)

    def forward_diag(self, *args, train=True) -> Tuple[torch.Tensor, torch.Tensor]:
        """(mean [B,k], variance diagonal [B,k]) — gnn_gaussian_policy_diag.py:26-87 without diag_embed."""
        self.train(train)
        batch_size = args[0].shape[0]
        a_out = self.gnn_forward(*args, train=train)
        if self.post_fc:
            hidden = a_out
        else:
            mean, hidden = a_out
        std = self._pre_std(hidden) if self.contextual_std else self._pre_std
        std = self.diag_activation(std + self._pre_activation_shift) + self.minimal_std
        if not self.contextual_std:
            std = std.tile((hidden.shape[0], 1))
        std = std.reshape(batch_size, -1)
        if self.post_fc:
            mean = self._mean(hidden)
            if self.use_tanh_mean:
                mean = torch.tanh(mean)
        return mean.reshape(batch_size, -1), std ** 2

    def forward(self, *args, train=True):
        mean, var = self.forward_diag(*args, train=train)
        return mean, torch.diag_embed(var)

    @torch.no_grad()
    def act(self, *args, state, deterministic=False, rank=0, return_eps=False, train=True):
        """`forward_diag`'s body call, then the head and the draw in one kernel (ops.gaussian_act) on the noise stream
        `state` (not advanced here).  -> loc, covariance_matrix, action, sample_log_prob, eps (or None)."""
        self.train(train)
        batch_size = args[0].shape[0]
        a_out = self.gnn_forward(*args, train=train)
        mean, hidden = (None, a_out) if self.post_fc else a_out
        std_w, std_b = (self._pre_std.weight, self._pre_std.bias) if self.contextual_std else (self._pre_std, None)
        return ops.gaussian_act(state, batch=batch_size, num_rows=self.num_actuators, action_dim=self._mean.out_features,
                                pre_shift=float(self._pre_activation_shift), minimal_std=float(self.minimal_std),
                                std_weight=std_w, std_bias=std_b, hidden=hidden, mean=mean,
                                mean_weight=self._mean.weight if self.post_fc else None,
                                mean_bias=self._mean.bias if self.post_fc else None,
                                use_tanh_mean=self.use_tanh_mean and self.post_fc, deterministic=deterministic,
                                rank=rank, return_eps=return_eps)

    # ---- distribution helpers (std := second tuple element; diagonal or full layout) ----------------
    def sample(self, p, n=1):
        return self.rsample(p, n).detach()

    def rsample(self, p, n=1):
        means, std = p[0], diag_of(p[1])
        eps = torch.randn((n,) + means.shape, dtype=std.dtype, device=std.device)
        return (means + eps * std).squeeze(0)

    def log_probability(self, p, x, **kwargs):
        mean, std = p
        k = x.shape[-1]
        return -0.5 * (self.maha(x, mean, std) + np.log(2.0 * np.pi) * k + self.log_determinant(std))

    def entropy(self, p):
        _, std = p
        k = std.shape[-1]
        return 0.5 * (k * np.log(2 * np.e * np.pi) + self.log_determinant(std))

    def log_determinant(self, std):
        return 2 * diag_of(std).log().sum(-1)

    def maha(self, mean, mean_other, std):
        return ((mean - mean_other) / diag_of(std)).pow(2).sum(-1)

    def precision(self, std):
        return (1 / diag_of(std).pow(2)).diag_embed()

    def covariance(self, std):
        return std.pow(2)

    @property
    def is_diag(self):
        return True
