"""Advantage module: replaces `torchrl.objectives.value.GAE(gamma, lmbda, value_network, average_gae=False,
shifted=True)` as constructed and called at examples/torchrl/train.py:134-140,249-252.

`adv_module(td[B_env, T])` runs ONE critic call over the T+1 observations of every env (shifted=True: the
rollout's obs plus the last `next` obs) and the reverse-time warp-scan kernel grl_gae_scan, then writes
`advantage`, `value_target`, `state_value` ([B_env, T, 1]) back.

`forward` keeps the torch formulation of the critic's per-token half for this time-batched call.  `advantage` computes
the same keys with that half on the fused critic kernels (one set of LayerNorm statistics per time step, no per-token
activation in HBM); `capture` / `advantage_graphed` / `advantage_static` replay it from one CUDA graph."""
import torch
from torch import nn

from .... import ops
from ....parallel import SegmentedGraph
from .operators import td_get


class GAE(nn.Module):
    def __init__(self, *, gamma: float, lmbda: float, value_network: nn.Module, average_gae: bool = False,
                 shifted: bool = True, **kwargs):
        super().__init__()
        if not shifted:
            raise NotImplementedError("the reference train loop uses shifted=True (train.py:139)")
        self.gamma, self.lmbda = float(gamma), float(lmbda)
        self.average_gae = average_gae
        self.value_network = value_network

    def _phase(self, obs, reward, done, terminated, fused: bool):
        """obs [B, T+1, F] per in_key, reward / done / terminated [B, T] -> (advantage, value_target, state_value,
        next state_value), [B, T, 1] each."""
        value = self.value_network.module(*obs, fused_groups=True) if fused else self.value_network.module(*obs)
        B, T1 = value.shape[:2]
        adv, vt = ops.gae(reward.reshape(B, T1 - 1), value.reshape(B, T1), done.reshape(B, T1 - 1),
                          terminated.reshape(B, T1 - 1), self.gamma, self.lmbda)
        if self.average_gae:
            adv = (adv - adv.mean()) / adv.std().clamp_min(1e-4)
        return adv.unsqueeze(-1), vt.unsqueeze(-1), value[:, :-1], value[:, 1:]

    @staticmethod
    def _inputs(td, keys):
        nxt = td_get(td, "next")
        done = td_get(nxt, "done")
        return ([td_get(td, k) for k in keys], [td_get(nxt, k)[:, -1:] for k in keys], td_get(nxt, "reward"), done,
                td_get(nxt, "terminated", done))

    @staticmethod
    def _write(td, out, copy: bool):
        if copy:
            out = [t.clone() for t in out]
        td["advantage"], td["value_target"], td["state_value"] = out[:3]
        td_get(td, "next")["state_value"] = out[3]
        return td

    @torch.no_grad()
    def forward(self, td):
        obs, last, reward, done, terminated = self._inputs(td, self.value_network.in_keys)
        obs = [torch.cat([o, l], dim=1) for o, l in zip(obs, last)]  # [B, T+1, F]
        return self._write(td, self._phase(obs, reward, done, terminated, fused=False), copy=False)

    @torch.no_grad()
    def advantage(self, td):
        """The keys `forward` writes, with the critic's per-token half on the fused kernels (per-time-step statistics)."""
        obs, last, reward, done, terminated = self._inputs(td, self.value_network.in_keys)
        obs = [torch.cat([o, l], dim=1) for o, l in zip(obs, last)]
        return self._write(td, self._phase(obs, reward, done, terminated, fused=True), copy=False)

    # ---- the advantage phase replayed from one CUDA graph ---------------------------------------------------------
    def _data_builders(self):
        return [m.hyper_data for m in self.value_network.modules() if getattr(m, "hyper_data", None) is not None]

    def capture(self, example_td, warmup: int = 2):
        """Record `advantage` (critic build_data -> fused critic -> final Linear -> grl_gae_scan) into one CUDA graph on
        static inputs of the example's [B_env, T] shape, the shape of every later `advantage_graphed` call.  The static
        observations are held as [B_env, T+1, F] (`_adv_static`), so a replay needs no concatenation.  Replays read the
        critic's parameters in place: after an update they evaluate the updated critic.  The graph holds the critic
        builder's placeholder for B_env (T+1) graphs; it is kept alive here when an update at another batch size drops it
        from the builder's cache.  A builder that rebuilds its topology eagerly on every call is refused."""
        for hd in self._data_builders():
            if hd.rebuild_every_call and not hd.refresh_in_place():
                raise ValueError(
                    "capture: the critic's data builder rebuilds its topology eagerly on every call (rebuild_every_call "
                    "without an in-place refresh), which reads sizes on the host and cannot be replayed - use `advantage`")
        keys = self.value_network.in_keys
        obs, last, reward, done, terminated = self._inputs(example_td, keys)
        B, T = obs[0].shape[:2]
        st = {k: torch.cat([o, l], dim=1).contiguous() for k, o, l in zip(keys, obs, last)}
        st["reward"] = reward.reshape(B, T).clone()
        st["done"] = done.reshape(B, T).clone()
        st["terminated"] = terminated.reshape(B, T).clone()
        self._adv_static, self._adv_T = st, T
        args = ([st[k] for k in keys], st["reward"], st["done"], st["terminated"])
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(warmup):
                self._phase(*args, fused=True)
        torch.cuda.current_stream().wait_stream(side)
        # under data parallelism the graph is split at the statistics all-reduces, which run between its segments
        self._adv_graph = SegmentedGraph()
        with torch.no_grad():
            self._adv_graph_out = self._adv_graph.capture(lambda: self._phase(*args, fused=True))
        # the replayed kernels read the placeholder of THIS batch size: keep it alive if the builder drops it
        self._adv_captured_topology = [hd.example_data for hd in self._data_builders()]
        return self

    def advantage_static(self):
        """Replay the captured phase on whatever the static inputs hold; returns the graph's own output tensors
        (advantage, value_target, state_value, next state_value; the next replay overwrites them)."""
        self._adv_graph.replay()
        return self._adv_graph_out

    def advantage_graphed(self, td):
        """Copy td's observations (`td[k]` -> [:, :T], `td["next"][k][:, -1:]` -> [:, T:]), reward, done and terminated
        into the static inputs, replay the captured phase and write copies of its outputs, as `forward` does."""
        st, T = self._adv_static, self._adv_T
        keys = self.value_network.in_keys
        obs, last, reward, done, terminated = self._inputs(td, keys)
        for k, o, l in zip(keys, obs, last):
            st[k][:, :T].copy_(o, non_blocking=True)
            st[k][:, T:].copy_(l, non_blocking=True)
        for k, v in (("reward", reward), ("done", done), ("terminated", terminated)):
            st[k].copy_(v.reshape(st[k].shape), non_blocking=True)
        self._adv_graph.replay()
        return self._write(td, self._adv_graph_out, copy=True)
