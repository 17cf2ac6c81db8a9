"""The learner side of examples/torchrl/train.py:134-146,249-316 without Hydra / collectors / logging:
model assembly from a PathConfig (what AgentBuilder + make_ppo_models produce,
examples/torchrl/builders/utils_algo_graph.py:208-276), the advantage phase and one minibatch update."""
from typing import Dict, Optional

import torch

from .algorithms.trust_region_projections.models.policy.gnn_gaussian_policy_diag import GNNGaussianPolicyDiag
from .algorithms.trust_region_projections.models.value.critic import BaseCritic
from .algorithms.trust_region_projections.models.value.gnn_vf_net import GNNVFNet
from .algorithms.trust_region_projections.objectives.operators import PolicyOperator, ValueOperator
from .algorithms.trust_region_projections.objectives.trpl import TRPLLoss
from .algorithms.trust_region_projections.objectives.value import GAE
from .algorithms.trust_region_projections.projections.projection_factory import get_projection_layer
from .synthetic import PathConfig, observation_layout, obs_keys


def _task_module(cfg: PathConfig):
    if cfg.task == "rigid":
        from .modules.pyg_data import rigid_tasks_data as m
        return m, m.RigidTasksData
    if cfg.task == "rope":
        from .modules.pyg_data import rope_tasks_data as m
        return m, m.RopeTasksData
    from .modules.pyg_data import cloth_tasks_data as m
    return m, m.ClothTasksData


def make_data(cfg: PathConfig, *, policy: bool):
    """configs/algorithm/pyg_agent/data/*.yaml + the per-experiment overrides (policy: dist_as_pos,
    output_mask_key=grippers, no full graph; critic: full_graph_obs, concat features)."""
    dims, names = observation_layout(cfg)
    _, D = _task_module(cfg)
    concat = (not policy) or cfg.model == "transformer"
    return D(observation_dim=dims, observation_names=names, full_graph_obs=not policy, dist_as_pos=policy,
             output_mask_key="grippers" if policy else None, concat_input_vector=concat,
             angular_velocity=cfg.angular_velocity, build_edges=policy and cfg.model != "transformer")


def make_policy_body(cfg: PathConfig, device):
    m, _ = _task_module(cfg)
    NodeType, EdgeType, EdgeLevel = m.NodeType, m.EdgeType, m.EdgeLevel
    if cfg.model == "hepi":
        from .modules.pyg_models.hepi import HEPi
        from .modules.pyg_models.ponita.conv import FiberBundleConv
        # configs/algorithm/pyg_agent/model/hepi.yaml:17-48: INTERNAL at step 0, TASK + AGENT at step 1
        codes = [[1, 0], [0, 1], [0, 1]]
        mp = [[FiberBundleConv(64, 64, 64, groups=64, separable=True, widening_factor=4) if c else None for c in code]
              for code in codes]
        net = HEPi(input_dim_node=len(NodeType) + cfg.policy_aux_dim, input_dim_edge=len(EdgeType) + 4, hidden_dim=64,
                   latent_dim=64, output_dim=cfg.output_dim, output_dim_vec=cfg.output_dim_vec, node_encoder_layers=2,
                   edge_encoder_layers=2, node_decoder_layers=2, node_type_mapping=NodeType, edge_type_mapping=EdgeType,
                   edge_level_mapping=EdgeLevel, message_passing=mp, num_messages=2, device=device, num_ori=16,
                   degree=2, ponita_dim=cfg.ponita_dim, only_upper_hemisphere=cfg.only_upper_hemisphere)
    elif cfg.model == "empn":
        from .modules.pyg_models.ponita_gcn import PonitaGCN
        net = PonitaGCN(input_dim_node=len(NodeType) + cfg.policy_aux_dim, output_dim=cfg.output_dim,
                        output_dim_vec=cfg.output_dim_vec, num_layers=2, hidden_dim=64, dropout=0.0, num_ori=16,
                        degree=2, widening_factor=4, attention=False, ponita_dim=cfg.ponita_dim)
    else:
        from .modules.pyg_models.transformer_vanilla import TransformerVanilla
        net = TransformerVanilla(input_dim_node=len(NodeType) + 12, output_dim=64, num_layers=2, num_heads=2,
                                 hidden_dim=64, dropout=0.0, concat_global=False)
    return net.to(device)


def policy_in_keys(cfg: PathConfig):
    keys = obs_keys(cfg)
    if cfg.policy_pos_is_norm:  # transformer cfg feeds the norm_* groups into the position / velocity slots
        keys = ["norm_position_vectors" if k == "position_vectors" else
                "norm_velocity_vectors" if k == "velocity_vectors" else k for k in keys]
    return keys


def build_agent(cfg: PathConfig, device, proj_type: str = "kl", seed: int = 0, projection_kwargs=None):
    """-> (actor PolicyOperator, critic ValueOperator, projection, loss_module, adv_module).  `projection_kwargs` override
    the projection layer's keywords, e.g. dict(entropy_schedule="linear", target_entropy=-2.0) for entropy control."""
    torch.manual_seed(seed)
    m, _ = _task_module(cfg)
    body = make_policy_body(cfg, device)
    policy = GNNGaussianPolicyDiag(gnn=body, hyper_data=make_data(cfg, policy=True),
                                   action_dim=cfg.total_action_dim, num_actuators=cfg.num_actuators, init="orthogonal",
                                   hidden_sizes=(64, 64), contextual_std=True, init_std=1.0, minimal_std=1e-5,
                                   share_action_dim=True, post_fc=cfg.post_fc).to(device)
    from .modules.pyg_models.deepsets import DeepSets
    n_feat = len(m.NodeType) + (12 if cfg.task == "rigid" else 9)
    vf = GNNVFNet(gnn=DeepSets(input_dim_node=n_feat, output_dim=64, hidden_dim=64, norm=["layer_norm", "layer_norm"]),
                  hyper_data=make_data(cfg, policy=False), init="orthogonal", hidden_sizes=(64, 64))
    torch.nn.init.orthogonal_(vf.final.weight, 0.01)  # builders/utils_algo_graph.py:195-198 (only nn.Linear)
    vf.final.bias.data.zero_()
    critic_net = BaseCritic(vf).to(device)
    actor = PolicyOperator(policy, policy_in_keys(cfg))
    critic = ValueOperator(critic_net, obs_keys(cfg))
    pkw = dict(mean_bound=cfg.mean_bound, cov_bound=cfg.cov_bound, trust_region_coeff=cfg.trust_region_coeff,
               scale_prec=True, entropy_schedule=False, target_entropy=0.0, temperature=0.5, entropy_eq=False,
               entropy_first=False, action_dim=cfg.total_action_dim, total_train_steps=1000, cpu=False,
               dtype=torch.float32)
    pkw.update(projection_kwargs or {})
    projection = get_projection_layer(proj_type=proj_type, **pkw)
    loss_module = TRPLLoss(actor, critic, projection=projection, clip_epsilon=0.2, entropy_bonus=True,
                           entropy_coef=cfg.entropy_coef, critic_coef=cfg.critic_coef, loss_critic_type="l2",
                           normalize_advantage=True, clip_value=cfg.clip_value)
    adv_module = GAE(gamma=cfg.gamma, lmbda=cfg.gae_lambda, value_network=critic, average_gae=False, shifted=True)
    return actor, critic, projection, loss_module, adv_module


class Learner:
    """train.py:145-146 (two Adam optimisers, eps=1e-5) + one iteration of the minibatch loop (:275-316)."""

    def __init__(self, cfg: PathConfig, actor, critic, loss_module, dp=None, fused_adam: bool = True,
                 overlap_critic: bool = True):
        self.cfg, self.actor, self.critic, self.loss_module, self.dp = cfg, actor, critic, loss_module, dp
        fused = fused_adam and next(actor.parameters()).is_cuda
        # The critic branch (DeepSets forward, clipped value loss, backward: ~100 small launches) is independent of the
        # actor branch until the optimiser steps: it runs on a second stream, under the actor's large kernels.
        # Data parallel: its graph-LayerNorm statistics are collectives, so it needs its own communicator
        # (DataParallel(side_group=True)); without one the step stays on a single stream.
        self._critic_stream = (torch.cuda.Stream() if overlap_critic and (dp is None or dp.side is not None)
                               and loss_module.critic_coef and next(actor.parameters()).is_cuda else None)
        # capturable: the step counter lives on the device, so the whole update can be replayed from a CUDA graph
        self.actor_optim = torch.optim.Adam(actor.parameters(), lr=cfg.lr, eps=1e-5, fused=fused, capturable=fused)
        self.critic_optim = torch.optim.Adam(critic.parameters(), lr=cfg.lr, eps=1e-5, fused=fused, capturable=fused)
        self.num_network_updates = 0
        self._graph = None
        # ONE persistent flat fp32 gradient bucket (actor | critic); after `_finish_grads` every parameter's .grad is a
        # view into it, so the data-parallel exchange is one all-reduce of this buffer with no copy back, and the
        # gradients of the last update stay readable (`flat_grads`) after the optimisers have zeroed the .grad fields.
        self._params = [p for p in list(actor.parameters()) + list(critic.parameters()) if p.requires_grad]
        self._flat = torch.zeros(sum(p.numel() for p in self._params), dtype=torch.float32, device=self._params[0].device)
        self._views, off = [], 0
        for p in self._params:
            self._views.append(self._flat[off:off + p.numel()].view_as(p))
            off += p.numel()
        if dp is not None:
            dp.attach(loss_module)
            dp.sync_module_state(actor, critic)  # replicas start bit-identical whatever each rank's RNG did
        # entropy control: the step the bound is scheduled on lives on the device and every update advances it there, so
        # a captured update replays with the right step; `num_network_updates` is its host mirror
        self._step = None
        if getattr(loss_module.projection, "has_entropy_control", False):
            self._step = torch.zeros((), dtype=torch.int64, device=self._params[0].device)
            loss_module.step_counter, loss_module.steps_on_device = self._step, True

    def set_step(self, n: int):
        """Resume at `n` network updates (host counter and the device step of the entropy bound)."""
        self.num_network_updates = int(n)
        if self._step is not None:
            self._step.fill_(int(n))

    def compute_losses(self, batch) -> Dict[str, torch.Tensor]:
        self.loss_module._global_steps = self.num_network_updates
        loss = self.loss_module(batch)
        loss["actor_loss"] = loss["loss_objective"] + loss["loss_entropy"] + loss["loss_trust_region"]
        return loss

    def _finish_grads(self):
        """Move this step's gradients into the flat bucket (one multi-tensor copy; parameters that took no part in the
        step, e.g. the AGENT convolution when A == 1, contribute zeros so the layout is identical on every rank),
        all-reduce it under data parallelism, and point every .grad at its view."""
        have = [i for i, p in enumerate(self._params) if p.grad is not None]
        if len(have) != len(self._params):
            self._flat.zero_()
        torch._foreach_copy_([self._views[i] for i in have], [self._params[i].grad for i in have])
        if self.dp is not None:
            self.dp.all_reduce(self._flat)  # summed: the losses already divide by the global count
        for p, v in zip(self._params, self._views):
            p.grad = v

    def flat_grads(self) -> Dict[str, torch.Tensor]:
        """Gradients of the most recent update (after the data-parallel all-reduce), keyed like `named_parameters()` of
        the actor ("actor.<name>") and the critic ("critic.<name>"); views into the flat bucket."""
        names = [f"actor.{n}" for n, p in self.actor.named_parameters() if p.requires_grad] + \
                [f"critic.{n}" for n, p in self.critic.named_parameters() if p.requires_grad]
        return dict(zip(names, self._views))

    @torch.no_grad()
    def calibrate(self, batch):
        """The one-time calibration forward of train.py:72-74 (FiberBundleConv rescales its kernels from the statistics of
        the first training-mode forward, conv.py:104-105,151-157).  Under data parallelism the statistics are global
        (every rank must call this with its shard), so replicas stay identical."""
        self.actor.get_dist(batch)

    def update(self, batch) -> Dict[str, torch.Tensor]:
        if self._critic_stream is not None:
            return self._update_two_streams(batch)
        loss = self.compute_losses(batch)
        self.num_network_updates += 1
        loss["actor_loss"].backward()
        loss["loss_critic"].backward()
        self._finish_grads()
        if self.cfg.clip_grad_norm:
            torch.nn.utils.clip_grad_norm_(self.actor.parameters(), self.cfg.max_grad_norm)
            torch.nn.utils.clip_grad_norm_(self.critic.parameters(), self.cfg.max_grad_norm)
        self.actor_optim.step()
        self.critic_optim.step()
        self.actor_optim.zero_grad()
        self.critic_optim.zero_grad()
        if self._step is not None:
            self._step.add_(1)
        return loss


    def _update_two_streams(self, batch) -> Dict[str, torch.Tensor]:
        """Same arithmetic as `update`; the critic loss and its backward are enqueued on `_critic_stream` (forked from
        and joined to the current stream, so the pattern is also valid inside a CUDA-graph capture)."""
        main, side = torch.cuda.current_stream(), self._critic_stream
        # The critic branch forks from the START of the step but is enqueued AFTER the actor's forward: in a graph replay
        # the device picks nodes up in creation order, and with the ~120 small critic nodes first the actor's first
        # kernel started 0.47 ms late (tools/step_timeline.py); now they run under the actor's large kernels.
        fork = torch.cuda.Event()
        fork.record(main)
        self.loss_module._global_steps = self.num_network_updates
        loss = self.loss_module(batch, with_critic=False)
        loss["actor_loss"] = loss["loss_objective"] + loss["loss_entropy"] + loss["loss_trust_region"]
        side.wait_event(fork)
        with torch.cuda.stream(side):
            loss_critic = self.loss_module.critic_term(batch)
            loss_critic.backward()  # autograd runs these nodes on the stream of their forward: `side`
        loss["loss_critic"] = loss_critic.detach()
        self.num_network_updates += 1
        loss["actor_loss"].backward()
        main.wait_stream(side)
        self._finish_grads()
        if self.cfg.clip_grad_norm:
            torch.nn.utils.clip_grad_norm_(self.actor.parameters(), self.cfg.max_grad_norm)
            torch.nn.utils.clip_grad_norm_(self.critic.parameters(), self.cfg.max_grad_norm)
        self.actor_optim.step()
        self.critic_optim.step()
        self.actor_optim.zero_grad()
        self.critic_optim.zero_grad()
        if self._step is not None:
            self._step.add_(1)
        return loss

    # ---- CUDA-graph replay of the whole update (launch-bound glue: ~500 launches per step) -----------------------
    def capture(self, example_batch, warmup: int = 3, restore: bool = True):
        """Capture `update` on static copies of `example_batch` (same shapes for every later batch).

        The warm-up iterations (allocator / NCCL / topology-cache warm-up) run real updates; with `restore` (default)
        parameters and optimiser state are put back afterwards, so the first replayed minibatch is the first update the
        networks see, as in the reference loop (train.py:259-316).  The one-time calibration runs BEFORE the snapshot:
        it belongs to the first forward, not to the warm-up.  The captured graph bakes in Python-side scalars (Adam's lr,
        `loss_module._global_steps`): lr annealing would be frozen.  An entropy schedule is captured on the fused loss
        path, which reads the step from the learner's device counter; `restore` then also puts back that counter and the
        projection's latched initial entropy, so the first replayed minibatch latches it.  The torch formulation reads the
        host step and is refused.
        The graph also holds the topology tensors of this batch size: re-capture after `hyper_data.invalidate()`.  With
        `hyper_data.rebuild_every_call` the data builder must refresh its topology in place (`refresh_in_place()`): every
        replay then rebuilds the kNN or radius graph from the static inputs' positions; any other rebuild mode is refused."""
        for net in (self.actor, self.critic):
            for m in net.modules():
                hd = getattr(m, "hyper_data", None)
                if hd is not None and hd.rebuild_every_call and not hd.refresh_in_place():
                    raise ValueError(
                        "capture: the data builder rebuilds its topology eagerly on every call (rebuild_every_call with "
                        "kNN edges without knn_in_place, a task with num_valid or an EMPN policy on the fp32 or unfused "
                        "path, radius edges with EMPN, or a model other than HEPi and EMPN), which reads sizes on the "
                        "host and cannot be replayed; a captured update rebuilds kNN INTERNAL edges with "
                        "`hyper_data.knn_in_place = True` (HEPi rope: any precision; HEPi rigid and EMPN: fused 16-bit "
                        "path) and, for HEPi, radius INTERNAL edges on the fused 16-bit path (internal_edges='radius', "
                        "ops.set_precision('bf16')) - otherwise use `update`")
        proj = self.loss_module.projection
        if self._step is not None and not self.loss_module._can_fuse(self.actor.get_submodule("0").module):
            raise NotImplementedError("an entropy schedule on the torch loss formulation depends on the host-side step "
                                      "counter, which a captured graph freezes; use the fused loss or the eager `update`")
        # data-parallel: the NCCL all-reduces of the step are captured too (torch's ProcessGroupNCCL records them on the
        # capture stream); every rank must capture and replay in lock-step
        self._static = {k: v.clone() for k, v in example_batch.items() if torch.is_tensor(v)}
        self.calibrate(self._static)
        modules = [self.actor, self.critic]
        if restore:
            saved = [[t.detach().clone() for t in list(m.parameters()) + list(m.buffers())] for m in modules]
            import copy
            saved_opt = [copy.deepcopy(o.state_dict()) for o in (self.actor_optim, self.critic_optim)]
            saved_n = self.num_network_updates
            if self._step is not None:
                saved_ent = [t.clone() for t in (self._step, proj.entropy_state(self._step.device))]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self.update(self._static)
        torch.cuda.current_stream().wait_stream(side)
        if restore:
            with torch.no_grad():
                for m, ts in zip(modules, saved):
                    for t, s_ in zip(list(m.parameters()) + list(m.buffers()), ts):
                        t.copy_(s_)
            if saved_opt[0]["state"]:
                self.actor_optim.load_state_dict(saved_opt[0])
                self.critic_optim.load_state_dict(saved_opt[1])
            else:  # fresh optimisers: zero the moments / step counters the warm-up created, keep their (static) tensors
                for o in (self.actor_optim, self.critic_optim):
                    for st in o.state.values():
                        for v in st.values():
                            if torch.is_tensor(v):
                                v.zero_()
            self.num_network_updates = saved_n
            if self._step is not None:
                for t, s_ in zip((self._step, proj.entropy_state(self._step.device)), saved_ent):
                    t.copy_(s_)
        self._graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._graph):
            self._graph_out = self.update(self._static)
        self.num_network_updates -= 1  # the capture pass did not execute
        # the graph replays kernels that read the topology tensors of THIS batch size: keep them alive even if the data
        # builders later drop their placeholder (batch-size change, invalidate())
        self._captured_topology = [m.hyper_data.example_data for net in modules for m in net.modules()
                                   if getattr(m, "hyper_data", None) is not None]
        return self

    def update_static(self):
        """Replay the captured update on whatever the static inputs (`self._static`) hold right now."""
        self._graph.replay()
        self.num_network_updates += 1
        return self._graph_out

    # ---- the epoch loop of train.py:255-316 over a device-resident rollout buffer (SURVEY 8(f) N3) ---------------
    def fit(self, buffer, epochs: Optional[int] = None, graphed: bool = True):
        """`epochs` passes (default cfg.ppo_epochs) over a `DeviceRolloutBuffer`; one update per minibatch of each pass's
        permutation.  `graphed`: full-size minibatches are gathered straight into the static inputs of the captured
        update and replayed (captured on the first call from the first minibatch — the buffer should be built with
        `drop_last=True`, a short tail chunk falls back to the eager update).  Returns the per-update loss dicts (for a
        replayed update these are the graph's output tensors, overwritten by the next replay: read them before it)."""
        from .rollout import run_minibatch_epochs
        epochs = self.cfg.ppo_epochs if epochs is None else epochs
        if not graphed:
            return run_minibatch_epochs(self.update, buffer, epochs)
        if self._graph is None:
            if len(buffer) < buffer.batch_size:
                raise ValueError("the buffer holds less than one full minibatch; use graphed=False")
            # example batch = the first stored frames (shapes and topology slots only; capture() undoes its warm-up
            # updates, and the sampler's random stream is left untouched)
            self.capture({k: v[:buffer.batch_size] for k, v in buffer._storage.items()})

        def step(mb):
            return self.update_static() if mb is self._static else self.update(mb)
        return run_minibatch_epochs(step, buffer, epochs, static_inputs=self._static)

    def update_graphed(self, batch):
        for k, v in self._static.items():
            v.copy_(batch[k], non_blocking=True)
        self._graph.replay()
        self.num_network_updates += 1
        return self._graph_out

    # ---- input pipeline: the NEXT minibatch crosses PCIe while the current update runs (SURVEY 8(f) N3) ----------
    def prefetch(self, host_batch):
        """Start the host -> device copy of a (pinned) minibatch into staging buffers on a copy stream."""
        if getattr(self, "_staging", None) is None:
            self._staging = {k: torch.empty_like(v) for k, v in self._static.items()}
            self._copy_stream = torch.cuda.Stream()
            self._staged = torch.cuda.Event()
            self._consumed = torch.cuda.Event()
            self._consumed.record()
        self._copy_stream.wait_event(self._consumed)  # the previous contents have been moved into the graph's inputs
        with torch.cuda.stream(self._copy_stream):
            for k, v in self._staging.items():
                v.copy_(host_batch[k], non_blocking=True)
            self._staged.record()

    def update_prefetched(self, next_host_batch=None):
        """Replay the captured update on the minibatch handed to `prefetch`, then start fetching `next_host_batch`."""
        main = torch.cuda.current_stream()
        main.wait_event(self._staged)
        for k, v in self._static.items():
            v.copy_(self._staging[k], non_blocking=True)  # device -> device, a few microseconds
        self._consumed.record(main)
        self._graph.replay()
        self.num_network_updates += 1
        if next_host_batch is not None:
            self.prefetch(next_host_batch)
        return self._graph_out
