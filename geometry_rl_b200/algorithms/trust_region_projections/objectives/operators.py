"""TensorDict-free stand-ins for the three torchrl wrappers the train loop builds around the networks
(examples/torchrl/builders/utils_algo_graph.py:146-158,200-203): `ProbabilisticActor(TensorDictModule(policy))`,
`ValueOperator(critic)`.  torchrl / tensordict are not installed offline; these expose exactly the methods
TRPLLoss and GAE call (`get_dist`, `build_dist_from_params`, `get_submodule("0").module`, `__call__(td)`) and
accept any mapping with `.get` (a TensorDict works unchanged)."""
import math
from typing import Mapping, Sequence

import torch
from torch import nn

from .... import ops
from ....parallel import SegmentedGraph

LOG_2PI = math.log(2.0 * math.pi)


def td_get(td, key, default=None):
    """`td.get(key)` for nested keys given as tuples (TensorDict semantics) on plain nested dicts."""
    if isinstance(key, tuple):
        cur = td
        for k in key:
            if cur is None:
                return default
            cur = cur.get(k, None) if hasattr(cur, "get") else None
        return default if cur is None else cur
    v = td.get(key, None)
    return default if v is None else v


class DiagMultivariateNormal:
    """torch.distributions.MultivariateNormal(loc, covariance_matrix=diag(var)) restricted to what the loss
    reads (objectives/trpl.py:237-246,310): mean, covariance_matrix, log_prob, entropy, sample."""

    def __init__(self, loc: torch.Tensor, covariance_matrix: torch.Tensor = None, var_diag: torch.Tensor = None):
        self.loc = loc
        if var_diag is None:
            var_diag = covariance_matrix.diagonal(dim1=-2, dim2=-1) if covariance_matrix.dim() == loc.dim() + 1 \
                else covariance_matrix
        self.var_diag = var_diag
        self._cov = covariance_matrix if (covariance_matrix is not None and covariance_matrix.dim() == loc.dim() + 1) \
            else None

    @property
    def mean(self):
        return self.loc

    @property
    def covariance_matrix(self):
        if self._cov is None:
            self._cov = torch.diag_embed(self.var_diag)
        return self._cov

    def log_prob(self, x):
        k = x.shape[-1]
        return -0.5 * (((x - self.loc) ** 2 / self.var_diag).sum(-1) + k * LOG_2PI + self.var_diag.log().sum(-1))

    def entropy(self):
        k = self.loc.shape[-1]
        return 0.5 * (k * (1.0 + LOG_2PI) + self.var_diag.log().sum(-1))

    def sample(self, generator=None):
        eps = torch.randn(self.loc.shape, dtype=self.loc.dtype, device=self.loc.device, generator=generator)
        return self.loc + eps * self.var_diag.sqrt()


class _Holder(nn.Module):
    def __init__(self, module):
        super().__init__()
        self.module = module


class PolicyOperator(nn.Module):
    """ProbabilisticActor equivalent: in_keys -> policy -> (loc, covariance_matrix) -> MultivariateNormal."""

    def __init__(self, policy: nn.Module, in_keys: Sequence[str], distribution_class=DiagMultivariateNormal):
        super().__init__()
        self.add_module("0", _Holder(policy))
        self.in_keys = list(in_keys)
        self.out_keys = ["loc", "covariance_matrix", "action", "sample_log_prob"]
        self.distribution_class = distribution_class

    @property
    def policy(self):
        return self.get_submodule("0").module

    def get_dist(self, td: Mapping):
        mean, var = self.policy.forward_diag(*[td_get(td, k) for k in self.in_keys])
        return DiagMultivariateNormal(mean, var_diag=var)

    def build_dist_from_params(self, td: Mapping):
        return DiagMultivariateNormal(td_get(td, "loc"), covariance_matrix=td_get(td, "covariance_matrix"))

    @torch.no_grad()
    def forward(self, td, generator=None):
        dist = self.get_dist(td)
        action = dist.sample(generator)
        td["loc"], td["covariance_matrix"] = dist.mean, dist.covariance_matrix
        td["action"], td["sample_log_prob"] = action, dist.log_prob(action)
        return td

    # ---- rollout-time acting: fused head + on-device Philox noise (grl_gaussian_act), optionally one CUDA graph -----
    # Opt-in path for the collector (`SyncDataCollector(policy=actor.act_graphed)`); `forward` and its torch RNG stay as
    # they are.  The noise stream is an int64 device buffer {seed, call counter}: each sampling call draws from it and
    # advances the counter on the device, so eager and replayed calls continue one stream.  Under data parallelism
    # `act_rank` (set by DataParallel.attach) enters the key and ranks draw different noise.
    act_rank = 0

    def _act_state_buffer(self) -> torch.Tensor:
        st = getattr(self, "_act_state", None)
        if st is None:
            st = torch.zeros(2, dtype=torch.int64, device=next(self.policy.parameters()).device)
            self._act_state = st
        return st

    def act_state(self):
        """(seed, call counter) of the acting noise stream (reads the device)."""
        seed, counter = self._act_state_buffer().tolist()
        return seed, counter

    def set_act_state(self, seed: int, counter: int = 0) -> None:
        """Restore the noise stream (in place: a captured act graph keeps reading the same buffer)."""
        self._act_state_buffer().copy_(torch.tensor([int(seed), int(counter)], dtype=torch.int64))

    def _act(self, obs, deterministic: bool, return_eps: bool = False):
        state = self._act_state_buffer()
        out = self.policy.act(*obs, state=state, deterministic=deterministic, rank=self.act_rank, return_eps=return_eps)
        if not deterministic:
            ops.act_advance(state)
        return out

    @staticmethod
    def _write_act(td, out, copy: bool):
        loc, cov, action, log_prob = out[:4]
        if copy:
            loc, cov, action, log_prob = loc.clone(), cov.clone(), action.clone(), log_prob.clone()
        td["loc"], td["covariance_matrix"], td["action"], td["sample_log_prob"] = loc, cov, action, log_prob
        return td

    @torch.no_grad()
    def act(self, td, *, deterministic: bool = False):
        """The keys `forward` writes (loc, covariance_matrix, action, sample_log_prob), computed by one kernel after the
        body, with noise from the device stream (`deterministic`: action = loc, nothing drawn)."""
        return self._write_act(td, self._act([td_get(td, k) for k in self.in_keys], deterministic), copy=False)

    def capture_act(self, example_td, *, seed: int, deterministic: bool = False, warmup: int = 2, obs_norm=None):
        """Record `build_data -> body -> grl_gaussian_act -> advance` into one CUDA graph on static copies of the
        example's observation keys (the batch size of every later `act_graphed` call), and start the noise stream at
        (seed, 0).  A pending one-time FiberBundleConv calibration runs eagerly on the example first.  The graph holds the
        topology of this batch size: re-capture after `hyper_data.invalidate()`.  With `hyper_data.rebuild_every_call`
        the data builder must refresh its topology in place (`refresh_in_place()`): every replay then rebuilds the kNN or
        radius graph from the static positions; any other rebuild mode is refused.

        `obs_norm` (an `NDVecNorm`): the graph starts from the RAW observation groups the normaliser reads and runs its
        device kernels (`NDVecNorm.apply_device`) into the static `norm_*` tensors the body reads; `act_graphed` then also
        writes copies of the `norm_*` keys.  Capture leaves the statistics as they were.  A normaliser frozen at capture
        gives a graph with no update (and no collective); replaying after its `frozen` flag changed raises.  Under data
        parallelism (`obs_norm.dp`) the graph is split at the statistics all-reduce (`parallel.SegmentedGraph`)."""
        hd = self.policy.hyper_data
        if hd.rebuild_every_call and not hd.refresh_in_place():
            raise ValueError(
                "capture_act: the data builder rebuilds its topology eagerly on every call (rebuild_every_call with kNN "
                "edges without knn_in_place, a task with num_valid or an EMPN policy on the fp32 or unfused path, radius "
                "edges with EMPN, or a model other than HEPi and EMPN), which reads sizes on the host and cannot be "
                "replayed; a captured act rebuilds kNN INTERNAL edges with `hyper_data.knn_in_place = True` (HEPi rope: "
                "any precision; HEPi rigid and EMPN: fused 16-bit path) and, for HEPi, radius INTERNAL edges on the "
                "fused 16-bit path (internal_edges='radius', ops.set_precision('bf16')) - otherwise use `act`")
        if obs_norm is not None:
            return self._capture_act_norm(example_td, seed, deterministic, warmup, obs_norm)
        self._act_norm = None
        self._act_static = [td_get(example_td, k).clone() for k in self.in_keys]
        with torch.no_grad():
            self.get_dist(dict(zip(self.in_keys, self._act_static)))  # the one-time calibration, if still pending
        self.set_act_state(seed, 0)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(warmup):  # draws without advancing: the stream is where set_act_state left it
                self.policy.act(*self._act_static, state=self._act_state, deterministic=deterministic, rank=self.act_rank)
        torch.cuda.current_stream().wait_stream(side)
        self._act_graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._act_graph), torch.no_grad():
            self._act_graph_out = self._act(self._act_static, deterministic)
        # the replayed kernels read this batch size's topology tensors: keep them alive if the builder drops them
        self._captured_topology = hd.example_data
        return self

    def _capture_act_norm(self, example_td, seed, deterministic, warmup, obs_norm):
        raw = {k: td_get(example_td, k).clone() for k in obs_norm.in_keys if td_get(example_td, k) is not None}
        if not raw:
            raise ValueError(f"capture_act: the example holds none of the normaliser's keys {obs_norm.in_keys}")
        normed = {ok: torch.empty_like(raw[k]) for k, ok in zip(obs_norm.in_keys, obs_norm.out_keys) if k in raw}
        static = {**raw, **normed}
        self._act_static = [static[k] if k in static else td_get(example_td, k).clone() for k in self.in_keys]
        # what act_graphed copies in: the raw groups and every policy input the normaliser does not write
        self._act_copy_in = list(raw.items()) + [(k, s) for k, s in zip(self.in_keys, self._act_static)
                                                 if k not in static]
        self._act_norm, self._act_norm_out, self._act_norm_frozen = obs_norm, normed, obs_norm.frozen

        def normalise():
            obs_norm.apply_device(dict(raw), out=normed)

        obs_norm.ensure_stats(raw)  # no allocation or memset of the state inside the graph
        saved = obs_norm.state_dict()
        with torch.no_grad():
            normalise()
            self.get_dist(dict(zip(self.in_keys, self._act_static)))  # the one-time calibration, if still pending
        self.set_act_state(seed, 0)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(warmup):  # draws without advancing; the statistics are restored below
                normalise()
                self.policy.act(*self._act_static, state=self._act_state, deterministic=deterministic, rank=self.act_rank)
        torch.cuda.current_stream().wait_stream(side)
        obs_norm.load_state_dict(saved)  # in place: the graph reads these tensors

        def step():
            normalise()
            return self._act(self._act_static, deterministic)

        self._act_graph = SegmentedGraph()
        with torch.no_grad():
            self._act_graph_out = self._act_graph.capture(step)
        self._captured_topology = self.policy.hyper_data.example_data
        return self

    def _check_act_norm(self):
        norm = getattr(self, "_act_norm", None)
        if norm is not None and norm.frozen != self._act_norm_frozen:
            raise RuntimeError(
                f"act_graphed: the observation normaliser was {'frozen' if self._act_norm_frozen else 'updating'} at "
                "capture and has changed since; re-capture with capture_act(obs_norm=...)")

    def act_static(self, td=None):
        """Replay the captured act on whatever the static inputs hold; with `td`, write the graph's own output tensors
        into it (no copy: the next replay overwrites them).  Returns the outputs keyed like `forward`'s."""
        self._check_act_norm()
        self._act_graph.replay()
        out = dict(zip(self.out_keys, self._act_graph_out[:4]))
        if td is not None:
            self._write_act(td, self._act_graph_out, copy=False)
        return out

    def act_graphed(self, td):
        """Copy td's observation keys into the static inputs, replay the captured act and write copies of its outputs
        (and, with a captured `obs_norm`, copies of the `norm_*` keys it computed from td's raw groups)."""
        if self._act_norm is None:
            for s, k in zip(self._act_static, self.in_keys):
                s.copy_(td_get(td, k), non_blocking=True)
            self._act_graph.replay()
            return self._write_act(td, self._act_graph_out, copy=True)
        self._check_act_norm()
        for k, s in self._act_copy_in:
            s.copy_(td_get(td, k), non_blocking=True)
        self._act_graph.replay()
        for ok, t in self._act_norm_out.items():
            td[ok] = t.clone()
        return self._write_act(td, self._act_graph_out, copy=True)


class ValueOperator(nn.Module):
    def __init__(self, module: nn.Module, in_keys: Sequence[str], out_keys=("state_value",)):
        super().__init__()
        self.module = module
        self.in_keys = list(in_keys)
        self.out_keys = list(out_keys)

    def forward(self, td):
        td[self.out_keys[0]] = self.module(*[td_get(td, k) for k in self.in_keys])
        return td
